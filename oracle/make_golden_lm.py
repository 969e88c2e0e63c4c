"""Generate the RNN-LM golden files tests/golden/lm_*.npz by RUNNING the unmodified reference (CPU):

    B200ASR_REFERENCE=<checkout of the original project> python -m oracle.make_golden_lm        # from the repo root

  lm_model_{lstm,tied,gru}.npz   the reference's RNNLM (src/lm.py) on a ragged batch: outputs, (h_n, c_n), the
                                 CE loss (ignore_index 0), every parameter gradient, the initial state_dict
  lm_plumbing.npz                the reference's own bin/train_lm.Solver (--cpu) for 2 steps on a LibriSpeech-shaped
                                 text fixture: each step's batch, loss and grad-norm, and the step-1 dev perplexity

The fixture helpers (lm_plumbing_tree / lm_plumbing_config) are shared with tests/test_gpu_lm.py.  Sizes are tiny;
every file stays far below 1 MB.  The ASR goldens (oracle/make_golden.py) are not touched by this script.
"""
import os
import sys

import numpy as np
import torch

from . import ref_shim

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
VOCAB_FILE = os.path.join(OUT, "character.vocab")

# kind -> (seed, RNNLM keyword arguments); character vocabulary (31 ids), 2 layers, no dropout
LM_KINDS = {
    "lstm": (101, dict(emb_tying=False, emb_dim=32, module="LSTM", dim=32, n_layers=2, dropout=0.0)),
    "tied": (102, dict(emb_tying=True, emb_dim=32, module="LSTM", dim=32, n_layers=2, dropout=0.0)),
    "gru": (103, dict(emb_tying=False, emb_dim=32, module="GRU", dim=32, n_layers=2, dropout=0.0)),
}
LM_VOCAB = 31
LM_LENS = [5, 1, 8, 3]          # unsorted, one row of <eos> only and one full-length row


def lm_batch(seed, lens, V):
    """Ragged token rows (ids in [2, V), <eos> = 1 last, zero padded) -> (x = <sos> + row without its last column, lens)
    exactly as bin/train_lm.py:fetch_data forms the model input."""
    g = torch.Generator().manual_seed(seed)
    data = torch.zeros(len(lens), max(lens), dtype=torch.long)
    for b, n in enumerate(lens):
        data[b, :n - 1] = torch.randint(2, V, (n - 1,), generator=g)
        data[b, n - 1] = 1
    txt = torch.cat((torch.zeros((data.shape[0], 1), dtype=torch.long), data), dim=1)
    return txt, (data != 0).sum(-1)


def golden_lm_model(kind):
    from src.lm import RNNLM                                                  # the reference's
    seed, cfg = LM_KINDS[kind]
    torch.manual_seed(seed)
    model = RNNLM(LM_VOCAB, **cfg)
    model.train()
    out = {"seed": np.int64(seed), "vocab": np.int64(LM_VOCAB)}
    for k, v in model.state_dict().items():
        out["sd." + k] = v.numpy().copy()
    txt, lens = lm_batch(seed + 1, LM_LENS, LM_VOCAB)
    pred, hidden = model(txt[:, :-1], lens)
    loss = torch.nn.CrossEntropyLoss(ignore_index=0)(pred.reshape(-1, LM_VOCAB), txt[:, 1:].reshape(-1))
    loss.backward()
    out.update(txt=txt.numpy(), lens=lens.numpy(), outputs=pred.detach().numpy(), loss=loss.detach().numpy())
    if cfg["module"] == "LSTM":
        out["h_n"], out["c_n"] = hidden[0].detach().numpy(), hidden[1].detach().numpy()
    else:
        out["h_n"] = hidden.detach().numpy()
    sq = 0.0
    for k, p in model.named_parameters():
        out["grad." + k] = p.grad.numpy().copy()
        sq += float((p.grad.double() ** 2).sum())
    out["grad_norm"] = np.float64(np.sqrt(sq))
    np.savez_compressed(os.path.join(OUT, "lm_model_%s.npz" % kind), **out)
    print("lm_model_%s.npz" % kind, "loss", float(loss.detach()), "grad_norm", np.sqrt(sq))


# LibriSpeech-shaped text fixture: distinct transcript lengths (the length sort has no ties, so the order does not
# depend on directory listing order); one transcript is longer than 150 characters (the half-batch rule)
LM_PLUMBING_TRAIN = {
    ("19", "198"): ["NORTHANGER ABBEY", "IT WAS A DARK AND STORMY NIGHT",
                    "SHE HAD A THIN AWKWARD FIGURE A SALLOW SKIN WITHOUT COLOUR DARK LANK HAIR AND STRONG FEATURES "
                    "SO MUCH FOR HER PERSON AND NOT LESS UNPROPITIOUS FOR HEROISM SEEMED HER MIND",
                    "NO ONE WHO HAD EVER SEEN CATHERINE"],
    ("26", "495"): ["THE QUICK BROWN FOX", "A B", "WHAT IS THE USE OF A BOOK THOUGHT ALICE",
                    "DOWN THE RABBIT HOLE SHE WENT WITHOUT A MOMENT'S THOUGHT"],
}
LM_PLUMBING_DEV = {("84", "121"): ["HELLO WORLD", "THE LAZY DOG SLEEPS IN THE SUN", "SPEECH"]}


def _write_split(root, split, table):
    for (spk, chap), lines in table.items():
        d = os.path.join(root, split, spk, chap)
        os.makedirs(d, exist_ok=True)
        with open(os.path.join(d, "%s-%s.trans.txt" % (spk, chap)), "w") as f:
            for i, line in enumerate(lines):
                utt = "%s-%s-%04d" % (spk, chap, i)
                f.write("%s %s\n" % (utt, line))
                open(os.path.join(d, utt + ".flac"), "wb").close()   # globbed only, never read


def lm_plumbing_tree(root):
    path = os.path.join(root, "LibriSpeech")
    _write_split(path, "train-clean-100", LM_PLUMBING_TRAIN)
    _write_split(path, "dev-clean", LM_PLUMBING_DEV)
    return path


def lm_plumbing_config(cfg, path):
    """The edits lm_example.yaml needs to run on the fixture (the same for the reference's and config/b200/'s)."""
    cfg["data"]["corpus"].update(path=path, train_split=["train-clean-100"], dev_split=["dev-clean"], batch_size=2)
    cfg["data"]["text"] = {"mode": "character", "vocab_file": VOCAB_FILE}
    cfg["hparas"].update(max_step=2)
    cfg["model"].update(emb_dim=32, dim=32, dropout=0)
    return cfg


def golden_lm_plumbing():
    import argparse
    import tempfile
    import yaml
    from bin.train_lm import Solver                                            # the reference's
    tmp = tempfile.mkdtemp(prefix="b200asr_lm_plumbing_")
    path = lm_plumbing_tree(tmp)
    cfg = yaml.load(open(os.path.join(ref_shim.REF_ROOT, "config", "libri", "lm_example.yaml")), Loader=yaml.FullLoader)
    own = yaml.load(open(os.path.join(os.path.dirname(OUT), "..", "config", "b200", "lm_example.yaml")),
                    Loader=yaml.FullLoader)
    assert own == cfg, "config/b200/lm_example.yaml drifted from the reference's lm_example.yaml"
    cfg = lm_plumbing_config(cfg, path)
    paras = argparse.Namespace(config="lm_example.yaml", name="lm_plumbing", logdir=os.path.join(tmp, "log"),
                               ckpdir=os.path.join(tmp, "ckpt"), outdir=os.path.join(tmp, "out"), load=None, seed=0,
                               cudnn_ctc=False, njobs=0, cpu=True, no_pin=True, test=False, no_msg=True, lm=True,
                               amp=False, reserve_gpu=0, jit=False, gpu=False, pin_memory=False, verbose=False)
    torch.set_num_threads(8)
    np.random.seed(0)
    torch.manual_seed(0)
    solver = Solver(cfg, paras, "train")
    solver.load_data()
    torch.manual_seed(0)                     # the weights and the shuffle are a function of this seed alone
    solver.set_model()
    losses, norms, batches, dev_ppx = [], [], [], []
    real_backward, real_fetch, real_log = solver.backward, solver.fetch_data, solver.write_log

    def backward(loss):
        losses.append(float(loss))
        n = real_backward(loss)
        norms.append(float(n))
        return n

    def fetch(data):
        if solver.model.training:
            batches.append(data.numpy().copy())
        return real_fetch(data)

    def write_log(name, d):
        if name == "perplexity" and isinstance(d, dict) and "dv" in d:
            dev_ppx.append(float(d["dv"]))
        return real_log(name, d)

    solver.backward, solver.fetch_data, solver.write_log = backward, fetch, write_log
    solver.exec()
    out = {"loss": np.asarray(losses, np.float64), "grad_norm": np.asarray(norms, np.float64),
           "dev_ppx": np.asarray(dev_ppx, np.float64), "n_steps": np.int64(len(batches))}
    for i, b in enumerate(batches):
        out["batch%d" % i] = b.astype(np.int64)
    ckpt = torch.load(os.path.join(solver.ckpdir, "best_ppx.pth"), map_location="cpu")
    for k, v in ckpt["model"].items():
        out["ckpt_shape." + k] = np.asarray(v.shape, np.int64)
    np.savez_compressed(os.path.join(OUT, "lm_plumbing.npz"), **out)
    print("lm_plumbing.npz", losses, norms, dev_ppx, [b.shape for b in batches])


def main():
    ref_shim.install()
    torch.set_num_threads(1)
    for kind in LM_KINDS:
        golden_lm_model(kind)
    golden_lm_plumbing()


if __name__ == "__main__":
    main()
