"""RNN-LM on the GPU: the embedding kernels against ATen, the package's RNNLM against the reference's (golden vectors
from oracle/make_golden_lm.py), the LM Solver against the reference's own short run, and main.py --lm end to end."""
import argparse
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F
import yaml

from conftest import load_golden, rel_err
from oracle.make_golden_lm import LM_KINDS, lm_plumbing_config, lm_plumbing_tree

pytestmark = pytest.mark.gpu
DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ids(V, shape, seed):
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(0, V // 2, shape, generator=g)        # the upper half of the table receives no id
    ids.view(-1)[::7] = 0                                      # id 0 repeated (the LM's <sos> / padding)
    return ids.to(DEV)


@pytest.mark.parametrize("V,E", [(16000, 1024), (31, 32), (50, 30)])
def test_embedding_forward_exact(pkg, V, E):
    w = torch.randn(V, E, device=DEV)
    ids = _ids(V, (5, 13), V + E)
    out = pkg.ops.embedding(ids, w)
    assert out.shape == (5, 13, E)
    assert torch.equal(out, F.embedding(ids, w))


@pytest.mark.parametrize("V,E", [(16000, 1024), (31, 32), (50, 30)])
def test_embedding_backward_matches_index_add(pkg, V, E):
    w = torch.randn(V, E, device=DEV, requires_grad=True)
    ids = _ids(V, (32, 41), 2 * V + E)
    dy = torch.randn(32, 41, E, device=DEV)
    pkg.ops.embedding(ids, w).backward(dy)
    ref = torch.zeros(V, E, dtype=torch.float64, device=DEV).index_add_(0, ids.view(-1), dy.view(-1, E).double())
    scale = float(ref.abs().max())
    assert float((w.grad.double() - ref).abs().max()) < 1e-5 * scale
    assert torch.count_nonzero(w.grad[V // 2:]) == 0           # rows that receive no id: exactly 0
    # accumulate: add onto an existing gradient, leave unused rows as they are
    base = torch.randn(V, E, device=DEV)
    acc = pkg.ops.embedding_backward(ids, dy, base.clone(), accumulate=True)
    assert float((acc.double() - (base.double() + ref)).abs().max()) < 1e-5 * (scale + float(base.abs().max()))
    assert torch.equal(acc[V // 2:], base[V // 2:])


def test_embedding_backward_bit_identical(pkg):
    V, E = 16000, 1024
    ids = _ids(V, (32, 40), 9)
    dy = torch.randn(32, 40, E, device=DEV)
    a = pkg.ops.embedding_backward(ids, dy, torch.empty(V, E, device=DEV))
    b = pkg.ops.embedding_backward(ids, dy, torch.empty(V, E, device=DEV))
    assert torch.equal(a, b)


def test_embedding_rejects_out_of_range_ids(pkg):
    w = torch.randn(10, 8, device=DEV)
    for bad in ([0, 10], [-1, 3]):
        with pytest.raises(pkg.B200AsrError, match="ids must lie"):
            pkg.ops.embedding(torch.tensor(bad, device=DEV), w)
        with pytest.raises(pkg.B200AsrError, match="ids must lie"):
            pkg.ops.embedding_backward(torch.tensor(bad, device=DEV), torch.ones(2, 8, device=DEV), w.clone())


def _golden_model(pkg, kind):
    g = load_golden("lm_model_%s.npz" % kind)
    _, cfg = LM_KINDS[kind]
    model = pkg.lm.RNNLM(int(g["vocab"]), **cfg)
    model.load_state_dict({k[3:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("sd.")})
    return g, cfg, model.to(DEV)


@pytest.mark.parametrize("kind", sorted(LM_KINDS))
def test_rnnlm_matches_reference(pkg, kind):
    """Same tolerances as the ASR model goldens (tests/test_gpu_model.py)."""
    g, cfg, model = _golden_model(pkg, kind)
    model.train()
    V = int(g["vocab"])
    txt = torch.from_numpy(g["txt"]).to(DEV)
    lens = torch.from_numpy(g["lens"])
    pred, hidden = model(txt[:, :-1], lens)
    out = pred.detach().cpu().numpy()
    assert out.shape == g["outputs"].shape
    assert rel_err(out, g["outputs"], floor=max(1e-3, 0.05 * float(np.abs(g["outputs"]).max()))) < 1e-4
    # padded steps: the head sees exactly 0, so their logits are exactly the bias (0 with tied weights)
    pad_logit = model.trans.bias.detach() if not cfg["emb_tying"] else torch.zeros(V, device=DEV)
    for b, n in enumerate(g["lens"]):
        assert torch.equal(pred[b, int(n):].detach(), pad_logit.expand(pred.shape[1] - int(n), V))
    h_n = hidden[0] if cfg["module"] == "LSTM" else hidden
    assert h_n.shape == g["h_n"].shape
    assert rel_err(h_n.detach().cpu().numpy(), g["h_n"], floor=1e-2) < 1e-4
    if cfg["module"] == "LSTM":
        assert rel_err(hidden[1].cpu().numpy(), g["c_n"], floor=1e-2) < 1e-4
    loss = pkg.ops.cross_entropy(pred.reshape(-1, V), txt[:, 1:].reshape(-1), ignore_index=0)
    assert abs(loss.item() - float(g["loss"])) < 1e-4 * abs(float(g["loss"]))
    loss.backward()
    sq = 0.0
    for k, p in model.named_parameters():
        ref = g["grad." + k]
        scale = max(float(np.abs(ref).max()), 1e-4)
        assert float(np.abs(p.grad.cpu().numpy() - ref).max()) < 2e-4 * scale, k
        sq += float((p.grad.double() ** 2).sum())
    assert abs(np.sqrt(sq) - float(g["grad_norm"])) < 1e-4 * float(g["grad_norm"])


def test_rnnlm_lstm_matches_packed_cudnn_at_width_256(pkg):
    """Packed-sequence semantics at a non-toy width: outputs, h_n and c_n against the library's packed nn.LSTM."""
    torch.manual_seed(5)
    V, H, B = 500, 256, 16
    model = pkg.lm.RNNLM(V, False, H, "LSTM", H, 2, 0.0).to(DEV).eval()
    lens = torch.randint(1, 30, (B,))
    lens[3] = 30
    x = torch.randint(0, V, (B, 30), device=DEV)
    with torch.no_grad():
        pred, (h_n, c_n) = model(x, lens)
        packed = torch.nn.utils.rnn.pack_padded_sequence(model.emb(x), lens, batch_first=True, enforce_sorted=False)
        ref, (rh, rc) = model.rnn(packed)
        ref, _ = torch.nn.utils.rnn.pad_packed_sequence(ref, batch_first=True)
        ref_pred = model.trans(ref)
    assert rel_err(pred.cpu(), ref_pred.cpu(), floor=0.05 * float(ref_pred.abs().max())) < 1e-4
    assert rel_err(h_n.cpu(), rh.cpu(), floor=1e-2) < 1e-4
    assert rel_err(c_n.cpu(), rc.cpu(), floor=1e-2) < 1e-4


def test_rnnlm_dropout_train_vs_eval(pkg):
    torch.manual_seed(0)
    model = pkg.lm.RNNLM(200, False, 64, "LSTM", 64, 2, 0.5).to(DEV)
    x = torch.randint(0, 200, (4, 12), device=DEV)
    lens = torch.tensor([12, 9, 5, 1])
    model.train()
    a, _ = model(x, lens)
    b, _ = model(x, lens)
    assert not torch.equal(a, b)
    model.eval()
    with torch.no_grad():
        c, _ = model(x, lens)
        d, _ = model(x, lens)
    assert torch.equal(c, d)


def test_lm_solver_plumbing_matches_reference(pkg, tmp_path):
    g = load_golden("lm_plumbing.npz")
    path = lm_plumbing_tree(str(tmp_path))
    cfg = yaml.load(open(os.path.join(ROOT, "config", "b200", "lm_example.yaml")), Loader=yaml.FullLoader)
    cfg = lm_plumbing_config(cfg, path)
    paras = argparse.Namespace(config="lm_example.yaml", name="lm_plumbing", logdir=str(tmp_path / "log"),
                               ckpdir=str(tmp_path / "ck"), outdir=str(tmp_path / "out"), load=None, seed=0, njobs=0,
                               gpu=True, pin_memory=False, verbose=False, amp=False)
    torch.manual_seed(0)
    s = pkg.train_lm.Solver(cfg, paras, "train")
    s.load_data()
    torch.manual_seed(0)                     # the reference's weights and shuffle order follow from this seed
    s.set_model()
    losses, norms, batches, dev_ppx = [], [], [], []
    real_backward, real_fetch, real_log = s.backward, s.fetch_data, s.write_log

    def backward(loss):
        losses.append(loss.item())
        n = real_backward(loss)
        norms.append(float(n))
        return n

    def fetch(data):
        if s.model.training:
            batches.append(data.numpy().copy())
        return real_fetch(data)

    def write_log(name, d):
        if name == "perplexity" and isinstance(d, dict) and "dv" in d:
            dev_ppx.append(float(d["dv"]))
        return real_log(name, d)

    s.backward, s.fetch_data, s.write_log = backward, fetch, write_log
    s.exec()
    n = int(g["n_steps"])
    assert len(batches) == n and len(losses) == n
    for i in range(n):
        assert np.array_equal(batches[i], g["batch%d" % i]), i
        assert abs(losses[i] - float(g["loss"][i])) < 1e-4 * abs(float(g["loss"][i])), (i, losses, g["loss"])
        assert abs(norms[i] - float(g["grad_norm"][i])) < 1e-4 * float(g["grad_norm"][i]), (i, norms, g["grad_norm"])
    assert len(dev_ppx) == len(g["dev_ppx"])
    assert abs(dev_ppx[0] - float(g["dev_ppx"][0])) < 1e-4 * float(g["dev_ppx"][0])
    ckpt = torch.load(str(tmp_path / "ck" / "lm_plumbing" / "best_ppx.pth"), map_location="cpu")
    shapes = {k[len("ckpt_shape."):]: tuple(int(x) for x in v) for k, v in g.items() if k.startswith("ckpt_shape.")}
    assert {k: tuple(v.shape) for k, v in ckpt["model"].items()} == shapes
    assert set(ckpt) == {"model", "optimizer", "global_step", "perplexity"}
    fresh = pkg.lm.RNNLM(31, **cfg["model"])
    fresh.load_state_dict(ckpt["model"])


def test_main_lm_synthetic_end_to_end(tmp_path):
    cmd = [sys.executable, os.path.join(ROOT, "main.py"), "--lm", "--config",
           os.path.join(ROOT, "config", "b200", "lm_synthetic.yaml"), "--njobs", "0", "--no-msg",
           "--ckpdir", str(tmp_path / "ck"), "--logdir", str(tmp_path / "log")]
    r = subprocess.run(cmd, cwd=str(tmp_path), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    ckpt = torch.load(str(tmp_path / "ck" / "lm_synthetic_sd0" / "best_ppx.pth"), map_location="cpu")
    assert ckpt["global_step"] >= 1 and "emb.weight" in ckpt["model"]
