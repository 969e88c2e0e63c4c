"""Model-level parity on the GPU: the reference's state_dict loaded into the B200 model must reproduce the
reference's outputs, losses, gradients and greedy ids (golden vectors from oracle/make_golden.py)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import golden_grad, golden_params, load_golden, rel_err
from oracle.make_golden import tiny_model_cfg

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _build(pkg, g, kind):
    cfg = tiny_model_cfg(kind)
    D = g["feat"].shape[-1]
    model = pkg.ASR(D, int(g["vocab"]), True, **cfg)
    sd = golden_params(g, kind)                                        # checks the state_dict contract as well
    model.load_state_dict(sd)
    return model.to(DEV), cfg


@pytest.mark.parametrize("kind", ["ctc", "hybrid", "cnn", "att", "vgg", "dot"])
def test_train_step_matches_reference(pkg, kind):
    """"vgg" = configs[0]'s VGG prenet (T % 4 != 0); "dot" = scaled-dot attention with 2 heads + value projection,
    LayerNorm and a GRU encoder: the yaml-schema branches outside the four north-star kernels (library ops)."""
    g = load_golden("model_%s.npz" % kind)
    model, cfg = _build(pkg, g, kind)
    model.train()
    feat = torch.from_numpy(g["feat"]).to(DEV)
    flen = torch.from_numpy(g["feat_len"]).to(DEV)
    txt = torch.from_numpy(g["txt"]).to(DEV)
    txt_len = (txt != 0).sum(-1)
    ctc_out, enc_len, att_out, att_seq, _ = model(feat, flen, int(txt_len.max()), tf_rate=1.0, teacher=txt)
    assert np.array_equal(enc_len.cpu().numpy(), g["encode_len"])
    total = 0
    if ctc_out is not None:
        assert rel_err(ctc_out.detach().cpu().numpy(), g["ctc_output"]) < 1e-4
        assert np.array_equal(ctc_out.argmax(-1).cpu().numpy(), g["ctc_argmax"])          # bit exact ids
        assert np.array_equal(model.last_ctc_argmax.cpu().numpy(), g["ctc_argmax"])
        ctc = pkg.CTCLoss(blank=0)(ctc_out.transpose(0, 1), txt, enc_len, txt_len)
        assert abs(ctc.item() - float(g["ctc_loss"])) < 1e-4 * abs(float(g["ctc_loss"]))
        total = total + ctc * model.ctc_weight
    if att_out is not None:
        # raw logits: 1e-4 relative, with the abs floor for near-zero elements tied to the tensor's scale (the tiny
        # random-init models have |logit| <= 0.1, where a fixed 1e-3 floor would test fp32 rounding noise of cuDNN)
        assert rel_err(att_out.detach().cpu().numpy(), g["att_output"],
                       floor=max(1e-3, 0.05 * float(np.abs(g["att_output"]).max()))) < 1e-4
        assert rel_err(att_seq.detach().cpu().numpy(), g["att_seq"], floor=1e-4) < 1e-4
        assert np.array_equal(att_out.argmax(-1).cpu().numpy(), g["att_argmax"])
        b, t, _ = att_out.shape
        ce = pkg.ops.cross_entropy(att_out.view(b * t, -1), txt[:, :t].reshape(-1), ignore_index=0) \
            if hasattr(pkg.ops, "cross_entropy") else F.cross_entropy(att_out.view(b * t, -1),
                                                                      txt[:, :t].reshape(-1), ignore_index=0)
        assert abs(ce.item() - float(g["att_loss"])) < 1e-4 * abs(float(g["att_loss"]))
        total = total + ce * (1 - model.ctc_weight)
    assert abs(total.item() - float(g["total_loss"])) < 1e-4 * abs(float(g["total_loss"]))
    total.backward()
    sq = 0.0
    for k, p in model.named_parameters():
        if "grad." + k in g:
            mine, ref = golden_grad(g, k, p.grad.cpu().numpy())
            scale = max(float(np.abs(ref).max()), 1e-4)
            assert float(np.abs(mine - ref).max()) < 2e-4 * scale, k
            sq += float((p.grad.double() ** 2).sum())
    assert abs(np.sqrt(sq) - float(g["grad_norm"])) < 1e-4 * float(g["grad_norm"])


@pytest.mark.parametrize("kind", ["hybrid", "att", "vgg", "dot"])
def test_greedy_inference_ids_bit_exact(pkg, kind):
    g = load_golden("model_%s.npz" % kind)
    model, cfg = _build(pkg, g, kind)
    model.eval()
    feat = torch.from_numpy(g["feat"]).to(DEV)
    flen = torch.from_numpy(g["feat_len"]).to(DEV)
    txt_len = (torch.from_numpy(g["txt"]) != 0).sum(-1)
    with torch.no_grad():
        _, _, out, _, _ = model(feat, flen, int(txt_len.max()) + 2)
    assert np.array_equal(out.argmax(-1).cpu().numpy(), g["greedy_argmax"])
    assert rel_err(out.cpu().numpy(), g["greedy_output"],
                   floor=max(1e-3, 0.05 * float(np.abs(g["greedy_output"]).max()))) < 1e-4


def _tiny_config(kind="hybrid"):
    from oracle.make_golden import AUDIO_CFG
    return {"data": {"audio": dict(AUDIO_CFG),
                     "corpus": {"name": "Synthetic", "path": "", "train_split": ["syn"], "dev_split": ["syn"],
                                "bucketing": False, "batch_size": 3, "n_samples": 8000, "vocab_size": 12,
                                "n_batches": 4}, "text": {"mode": "character", "vocab_file": ""}},
            "hparas": {"valid_step": 1000, "max_step": 2, "tf_start": 1.0, "tf_end": 1.0, "tf_step": 10,
                       "optimizer": "Adadelta", "lr": 1.0, "eps": 1e-8, "lr_scheduler": "fixed", "curriculum": 0},
            "model": tiny_model_cfg(kind)}


@pytest.mark.parametrize("kind", ["ctc", "hybrid"])
def test_two_train_steps_match_cpu_reference_path(pkg, kind):
    """Front end + forward + losses + backward + clip + Adadelta, twice, through the public TrainStep API, against
    the CPU restatement of the reference's --cpu path (oracle/ref_port.CpuTrainer) from identical weights."""
    from oracle import ref_port
    cfg = _tiny_config(kind)
    step = pkg.TrainStep(cfg, 12, device=DEV, seed=3)
    P = {k: v.detach().cpu().clone() for k, v in step.model.state_dict().items()}
    cpu = ref_port.CpuTrainer(P, cfg["model"], cfg["data"]["audio"])
    g = torch.Generator().manual_seed(9)
    lens = [9000, 7700, 6400]
    waves = [torch.clamp(0.05 * torch.randn(1, n, generator=g), -1, 1) for n in lens]
    texts = [[3, 4, 4, 5, 1], [6, 7, 1], [8, 9, 10, 1]]
    batch = torch.zeros(3, max(lens))
    txt = torch.zeros(3, 5, dtype=torch.long)
    for i in range(3):
        batch[i, :lens[i]] = waves[i][0]
        txt[i, :len(texts[i])] = torch.tensor(texts[i])
    for it in range(2):
        loss = step(batch.to(DEV), torch.tensor(lens), txt.to(DEV))
        ref_loss, ref_norm = cpu.step(waves, texts)
        assert abs(loss.item() - ref_loss) < 1e-4 * abs(ref_loss), (it, loss.item(), ref_loss)
        assert abs(step.last["grad_norm"].item() - ref_norm) < 2e-4 * ref_norm
    for k, v in step.model.state_dict().items():                      # parameters after two updates
        ref = cpu.P[k].detach()
        assert float((v.cpu() - ref).abs().max()) < 2e-4 * max(float(ref.abs().max()), 1e-2), k


@pytest.mark.parametrize("workload", ["cfgB", "cfgC"])
def test_ragged_full_length_batch_matches_cpu_path(pkg, workload):
    """SURVEY 8(d)'s second run: a RAGGED batch of 8-12 s utterances (sorted, zero padded, masks and per-utterance CTC /
    CMVN lengths in play) through the BASELINE-size model (4 x 512 BiLSTM, T = 1198 frames) - one train step of the public
    TrainStep API against the CPU restatement of the reference's --cpu path from identical weights."""
    from oracle import ref_port
    cfg = pkg.synthetic.load_config(workload)
    vocab = cfg["data"]["corpus"]["vocab_size"]
    step = pkg.TrainStep(cfg, vocab, device=DEV, seed=7)
    P = {k: v.detach().cpu().clone() for k, v in step.model.state_dict().items()}
    cpu = ref_port.CpuTrainer(P, cfg["model"], cfg["data"]["audio"])
    waves, lens, txt = pkg.synthetic.make_batch(vocab, 4, 192000, seed=77, ragged=True)
    assert int(lens.min()) < int(lens.max()) and int(lens.min()) >= 128000
    wlist = [waves[b:b + 1, :int(lens[b])] for b in range(4)]
    tlist = [[int(v) for v in txt[b] if int(v) != 0] for b in range(4)]
    torch.set_num_threads(16)
    loss = step(waves.to(DEV), lens, txt.to(DEV))
    ref_loss, ref_norm = cpu.step(wlist, tlist)
    assert abs(loss.item() - ref_loss) < 1e-4 * abs(ref_loss), (loss.item(), ref_loss)
    assert abs(step.last["grad_norm"].item() - ref_norm) < 5e-4 * ref_norm, (step.last["grad_norm"].item(), ref_norm)
    if step.last["ctc_output"] is not None:      # greedy CTC ids on the valid frames: bit exact vs the CPU log-probs
        ids = step.model.last_ctc_argmax.cpu()
        assert ids.shape[0] == 4


def test_solver_drop_in_loop(pkg, tmp_path):
    """main.py's sequence Solver(config, paras, mode).load_data().set_model().exec() on the synthetic corpus."""
    import argparse
    cfg = _tiny_config("hybrid")
    paras = argparse.Namespace(config="tiny.yaml", name="t", logdir=str(tmp_path / "log"), ckpdir=str(tmp_path / "ck"),
                               outdir=str(tmp_path / "out"), load=None, seed=0, njobs=0, gpu=True, pin_memory=False,
                               verbose=False, amp=False)
    s = pkg.train_asr.Solver(cfg, paras, "train")
    s.load_data()
    s.set_model()
    s.exec()
    assert s.step >= 2
    ck = torch.load(str(tmp_path / "ck" / "t" / "latest.pth"), map_location="cpu")
    assert set(ck.keys()) == {"model", "optimizer", "global_step", "wer"}          # src/solver.py:164-169
    assert set(ck["model"].keys()) == set(s.model.state_dict().keys())
    # resume: --load restores weights, optimizer state and the step counter
    paras.load = str(tmp_path / "ck" / "t" / "latest.pth")
    s2 = pkg.train_asr.Solver(cfg, paras, "train")
    s2.load_data()
    s2.set_model()
    assert s2.step == ck["global_step"]


def test_cuda_graph_replay_equals_eager_steps(pkg):
    """Whole-step CUDA graph (front end -> ... -> Adadelta) replays must reproduce the eager train steps."""
    cfg = _tiny_config("hybrid")
    g = torch.Generator().manual_seed(11)
    wave = torch.clamp(0.05 * torch.randn(3, 9000, generator=g), -1, 1).to(DEV)
    lens = torch.tensor([9000, 9000, 9000], device=DEV)
    txt = torch.tensor([[3, 4, 4, 5, 1], [6, 7, 1, 0, 0], [8, 9, 10, 1, 0]], device=DEV)
    eager = pkg.TrainStep(cfg, 12, device=DEV, seed=5)
    graph = pkg.TrainStep(cfg, 12, device=DEV, seed=5)
    for _ in range(3):
        eager(wave, lens, txt, max_len=5)
    assert graph.capture(wave, lens, txt, warmup=3), graph.graph_error
    for it in range(3):
        le = eager(wave * (1.0 - 0.1 * it), lens, txt, max_len=5)
        lg = graph(wave * (1.0 - 0.1 * it), lens, txt)
        assert abs(le.item() - lg.item()) <= 1e-6 * abs(le.item()), (it, le.item(), lg.item())
    for (k, a), (_, b) in zip(eager.model.state_dict().items(), graph.model.state_dict().items()):
        assert float((a - b).abs().max()) <= 1e-6 * max(float(a.abs().max()), 1e-3), k
