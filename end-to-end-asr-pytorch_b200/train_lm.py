"""RNN-LM training Solver with the reference's interface (the reference's bin/train_lm.py): Solver(config, paras,
"train").load_data() / .set_model() / .exec(), the same batches, loss, logging names, validation and checkpoints.
The model is lm.RNNLM (embedding / LSTM / head kernels), the loss the fused log-softmax + NLL kernel, and the update
BaseSolver.backward (grad-norm, clip 5, NaN skip and Adam fused on flat buffers, norm kept on the device)."""
import os

import torch

from . import ops
from .data import load_textset
from .lm import RNNLM
from .optim import Optimizer
from .solver import BaseSolver
from .util import human_format


class Solver(BaseSolver):
    def __init__(self, config, paras, mode):
        world = int(os.environ.get("WORLD_SIZE", "1"))
        if world > 1:           # checked before BaseSolver would join a process group
            raise NotImplementedError("RNN-LM training runs on one GPU; data-parallel LM training (WORLD_SIZE=%d) is "
                                      "not supported" % world)
        super().__init__(config, paras, mode)
        self.best_loss = 10

    def fetch_data(self, data):
        """txt [B, L] (host) -> (<sos>=0 prepended, on the device; token counts [B] on the host)."""
        txt = torch.cat((torch.zeros((data.shape[0], 1), dtype=torch.long), data), dim=1).to(self.device)
        txt_len = torch.sum(data != 0, dim=-1)
        return txt, txt_len

    def load_data(self):
        self.tr_set, self.dv_set, self.vocab_size, self.tokenizer, msg = load_textset(
            self.paras.njobs, self.paras.gpu, self.paras.pin_memory, **self.config["data"])
        self.verbose(msg)

    def set_model(self):
        self.model = RNNLM(self.vocab_size, **self.config["model"]).to(self.device)
        self.verbose(self.model.create_msg())
        self.seq_loss = lambda logits, target: ops.cross_entropy(logits, target, ignore_index=0)
        self.optimizer = Optimizer(self.model.parameters(), **self.config["hparas"])
        self.verbose(self.optimizer.create_msg())
        self.load_ckpt()

    def exec(self):
        self.verbose("Total training steps {}.".format(human_format(self.max_step)))
        self.timer.set()
        while self.step < self.max_step:
            for data in self.tr_set:
                self.optimizer.pre_step(self.step)
                txt, txt_len = self.fetch_data(data)
                self.timer.cnt("rd")
                pred, _ = self.model(txt[:, :-1], txt_len)
                lm_loss = self.seq_loss(pred.view(-1, self.vocab_size), txt[:, 1:].reshape(-1))
                self.timer.cnt("fw")
                grad_norm = self.backward(lm_loss)
                self.step += 1
                if self.step % self.PROGRESS_STEP == 0:
                    self.progress("Tr stat | Loss - {:.2f} | Grad. Norm - {:.2f} | {}".format(
                        lm_loss.cpu().item(), grad_norm.item(), self.timer.show()))
                    self.write_log("entropy", {"tr": lm_loss})
                    self.write_log("perplexity", {"tr": torch.exp(lm_loss).cpu().item()})
                if (self.step == 1) or (self.step % self.valid_step == 0):
                    self.validate()
                self.timer.set()
                if self.step > self.max_step:
                    break
        self.log.close()

    def validate(self):
        self.model.eval()
        dev_loss = []
        for i, data in enumerate(self.dv_set):
            self.progress("Valid step - {}/{}".format(i + 1, len(self.dv_set)))
            txt, txt_len = self.fetch_data(data)
            with torch.no_grad():
                pred, _ = self.model(txt[:, :-1], txt_len)
                dev_loss.append(self.seq_loss(pred.view(-1, self.vocab_size), txt[:, 1:].reshape(-1)))
        dev_loss = sum(dev_loss) / len(dev_loss)
        dev_ppx = torch.exp(dev_loss).cpu().item()
        if dev_loss < self.best_loss:
            self.best_loss = dev_loss
            self.save_checkpoint("best_ppx.pth", "perplexity", dev_ppx)
        self.write_log("entropy", {"dv": dev_loss})
        self.write_log("perplexity", {"dv": dev_ppx})
        for i in range(min(len(txt), self.DEV_N_EXAMPLE)):
            if self.step == 1:
                self.write_log("true_text{}".format(i), self.tokenizer.decode(txt[i].tolist()))
            self.write_log("pred_text{}".format(i), self.tokenizer.decode(pred[i].argmax(dim=-1).tolist()))
        self.model.train()
