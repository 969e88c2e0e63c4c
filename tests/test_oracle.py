"""Pin the CPU oracle (oracle/oracle_np.py, oracle/ref_port.py) against golden vectors produced by running the
unmodified reference (oracle/make_golden.py).  CPU only."""
import numpy as np
import pytest
import torch

from conftest import golden_grad, golden_params, load_golden, rel_err
from oracle import oracle_np as onp
from oracle import ref_port
from oracle.make_golden import AUDIO_CFG, tiny_model_cfg


# ------------------------------------------------------------------------------------------- front end
def test_fbank_np_matches_reference_sample_wav():
    g = load_golden("frontend.npz")
    wave = g["sample_pcm"].astype(np.float32) / 32768.0
    fb = onp.fbank(wave, dtype=np.float64)
    assert fb.shape == (392, 40)                       # reference tests/test_audio.py:24
    assert rel_err(fb, g["sample_fbank_raw"], floor=1.0) < 2e-5
    for order in (0, 1, 2):
        y = onp.delta_cmvn(fb, order=order, dtype=np.float64)
        ref = g["sample_feat_d%d" % order]
        assert y.shape == ref.shape == (392, 40 * (order + 1))   # tests/test_audio.py:53-55,72,87
        assert np.max(np.abs(y - ref)) < 2e-4


def test_frontend_properties_the_reference_tests_pin():
    g = load_golden("frontend.npz")
    wave = g["sample_pcm"].astype(np.float32) / 32768.0
    fb = onp.fbank(wave)
    y2 = onp.delta_cmvn(fb, order=2)
    # tests/test_audio.py:103 - CMVN: mean ~ 0 (atol 5e-5), std ~ 1 (atol 1e-6), per (channel, bin) over time
    assert np.allclose(y2.mean(0), 0.0, atol=5e-5)
    assert np.allclose(y2.std(0, ddof=1), 1.0, atol=1e-6)
    # tests/test_audio.py:87 - the first 40 dims of the delta-order-1 output equal the no-delta output
    y1 = onp.delta_cmvn(fb, order=1)
    y0 = onp.delta_cmvn(fb, order=0)
    assert np.allclose(y1[:, :40], y0, rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("i", [0, 1, 2, 3])
def test_fbank_np_synthetic(i):
    g = load_golden("frontend.npz")
    fb = onp.fbank(g["syn%d_wave" % i])
    assert fb.shape == g["syn%d_raw" % i].shape
    assert rel_err(fb, g["syn%d_raw" % i], floor=1.0) < 2e-5
    if i > 0:
        y = onp.delta_cmvn(fb, order=2)
        assert np.max(np.abs(y - g["syn%d_feat" % i])) < 5e-4


def test_ref_port_frontend_is_bit_identical():
    g = load_golden("frontend.npz")
    for i in (1, 2, 3):
        w = torch.from_numpy(g["syn%d_wave" % i])[None]
        y = ref_port.frontend(w, AUDIO_CFG)
        assert np.array_equal(y.numpy(), g["syn%d_feat" % i])


def test_delta_filters():
    f = onp.delta_filters(2, 2)
    assert f.shape == (3, 9)
    assert np.allclose(f[1, 2:7], np.array([-2, -1, 0, 1, 2]) / 10.0)
    assert np.allclose(f[2], [.04, .04, .01, -.04, -.1, -.04, .01, .04, .04])


# ------------------------------------------------------------------------------------------- CTC
def test_ctc_np_matches_aten_cases():
    g = load_golden("ctc_cases.npz")
    for i in range(int(g["n_cases"])):
        lp, tgt, tl, il = g["c%d_lp" % i], g["c%d_tgt" % i], int(g["c%d_tl" % i][0]), int(g["c%d_il" % i][0])
        nll, alpha, beta, grad = onp.ctc_single(lp[:il].astype(np.float64), list(tgt[:tl]))
        ref_nll = float(g["c%d_nll" % i][0])
        if np.isinf(ref_nll):
            assert np.isinf(nll)
            continue
        assert abs(nll - ref_nll) < 1e-5 * max(1.0, abs(ref_nll))
        ra = g["c%d_alpha" % i][:il, :2 * tl + 1]
        fin = np.isfinite(ra)
        assert np.array_equal(fin, np.isfinite(alpha))
        assert np.max(np.abs(alpha[fin] - ra[fin])) < 1e-4
        assert np.max(np.abs(grad - g["c%d_grad" % i][:il])) < 1e-5
        assert np.all(g["c%d_grad" % i][il:] == 0)


# ------------------------------------------------------------------------------------------- model
@pytest.mark.parametrize("kind", ["ctc", "hybrid", "cnn", "att", "vgg"])
def test_ref_port_matches_reference_model(kind):
    g = load_golden("model_%s.npz" % kind)
    P = {k: v.requires_grad_(True) for k, v in golden_params(g, kind).items()}
    cfg = tiny_model_cfg(kind)
    res = ref_port.forward_losses(P, cfg, torch.from_numpy(g["feat"]), torch.from_numpy(g["feat_len"]),
                                  torch.from_numpy(g["txt"]))
    tol = 1e-4 if kind == "vgg" else 1e-5     # oneDNN's conv2d picks thread-count dependent algorithms
    assert np.array_equal(res["encode_len"].numpy(), g["encode_len"])
    if "ctc_output" in g:
        assert rel_err(res["ctc_output"].detach().numpy(), g["ctc_output"]) < 1e-5
        assert np.array_equal(res["ctc_output"].argmax(-1).numpy(), g["ctc_argmax"])
        assert abs(float(res["ctc_loss"]) - float(g["ctc_loss"])) < 1e-5
    if "att_output" in g:
        assert rel_err(res["att_output"].detach().numpy(), g["att_output"]) < tol
        assert rel_err(res["att_seq"].detach().numpy(), g["att_seq"]) < tol
        assert np.array_equal(res["att_output"].argmax(-1).numpy(), g["att_argmax"])
    res["total_loss"].backward()
    assert abs(float(res["total_loss"]) - float(g["total_loss"])) < tol
    for k, p in P.items():
        if ("grad." + k) in g:
            assert rel_err(*golden_grad(g, k, p.grad.numpy()), floor=1e-4) < 1e-3, k
    norm, _ = ref_port.grad_norm_clip([p.grad for p in P.values() if p.grad is not None])
    assert abs(float(norm) - float(g["grad_norm"])) < tol


def test_lstm_np_matches_reference_layer():
    g = load_golden("model_ctc.npz")
    Pt = golden_params(g, "ctc")
    pre = "encoder.layers.0.layer."
    params = {k[len(pre):]: v.numpy() for k, v in Pt.items() if k.startswith(pre)}
    out = onp.bilstm(g["feat"], params)
    ref, _ = ref_port._lstm(Pt, pre, torch.from_numpy(g["feat"]), True)
    assert np.max(np.abs(out - ref.numpy())) < 1e-6      # fp64 restatement vs ATen fp32


def test_attention_step_np_matches_port():
    g = load_golden("model_hybrid.npz")
    P = golden_params(g, "hybrid")
    cfg = tiny_model_cfg("hybrid")
    enc, enc_len = ref_port.encoder(P, cfg["encoder"], torch.from_numpy(g["feat"]), torch.from_numpy(g["feat_len"]))
    key = torch.tanh(torch.nn.functional.linear(enc, P["attention.proj_k.weight"], P["attention.proj_k.bias"]))
    B, T, _ = enc.shape
    q = torch.tanh(torch.nn.functional.linear(torch.zeros(B, 32), P["attention.proj_q.weight"],
                                              P["attention.proj_q.bias"]))
    prev = (torch.arange(T)[None] < enc_len[:, None]).float() / enc_len[:, None].float()
    ctx, a = onp.loc_attention_step(q.numpy().astype(np.float64), key.numpy().astype(np.float64),
                                    enc.numpy().astype(np.float64), prev.numpy().astype(np.float64), enc_len.numpy(),
                                    P["attention.att_layer.loc_conv.weight"].numpy(),
                                    P["attention.att_layer.loc_proj.weight"].numpy(),
                                    P["attention.att_layer.gen_energy.weight"].numpy(),
                                    P["attention.att_layer.gen_energy.bias"].numpy(), 0.5)
    assert rel_err(a, g["att_seq"][:, 0, 0, :]) < 1e-4     # first decode step of the reference run


def test_cross_entropy_np():
    rng = np.random.default_rng(0)
    x = rng.standard_normal((10, 7))
    t = np.array([0, 3, 2, 0, 6, 1, 1, 0, 5, 4])
    loss, grad = onp.cross_entropy(x, t)
    xt = torch.tensor(x, requires_grad=True)
    ref = torch.nn.functional.cross_entropy(xt, torch.tensor(t), ignore_index=0)
    ref.backward()
    assert abs(loss - float(ref)) < 1e-10
    assert np.max(np.abs(grad - xt.grad.numpy())) < 1e-12


def test_ctc_prefix_oracle_matches_reference_scorer():
    """oracle_np.ctc_prefix_* against the reference's CTCPrefixScore run by oracle/make_golden.py (src/ctc.py:12-116)."""
    g = load_golden("ctc_prefix.npz")
    x = g["x"][0]
    assert rel_err(onp.ctc_prefix_init(x), g["r_init"]) < 1e-6
    for s in range(int(g["n_steps"])):
        psi, r = onp.ctc_prefix_cheap(x, list(g["s%d_prefix" % s]), g["s%d_rprev" % s], list(g["s%d_cands" % s]))
        assert rel_err(psi, g["s%d_psi" % s]) < 1e-6
        assert rel_err(r, g["s%d_r" % s]) < 1e-6
