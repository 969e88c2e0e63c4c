"""CPU-only checks of the host side: the C-ABI library builds, loads and exports every symbol the header declares;
the host-side tables are bit-identical to the reference's; the LSTM planner; the API mirror's contracts."""
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT, load_golden


def test_library_exports_every_declared_symbol(pkg):
    import __graft_entry__ as ge
    ge.build()
    lib = pkg.load_library()
    header = open(os.path.join(ROOT, "include", "b200asr.h")).read()
    public = set(re.findall(r"\b(b200asr_[a-z0-9_]+)\s*\(", header))
    assert not any("debug" in n for n in public)          # test / measurement switches live in b200asr_debug.h
    header += open(os.path.join(ROOT, "include", "b200asr_debug.h")).read()
    declared = set(re.findall(r"\b(b200asr_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(lib, name), name
    assert declared == set(pkg.lib.SIGNATURES.keys())
    assert lib.b200asr_version() == 100
    assert lib.b200asr_grad_norm_scratch_bytes() > 0


def test_error_convention_without_gpu(pkg):
    lib = pkg.load_library()
    # invalid arguments are rejected before any CUDA call: rc < 0 and a message, never a crash
    rc = lib.b200asr_log_softmax_fwd(None, None, None, None, 4, 8, None)
    assert rc == -1 and "null pointer" in pkg.lib.last_error()
    rc = lib.b200asr_bilstm_plan(8, 20, 2, None, None, None)
    assert rc == -1 and "multiple of 16" in pkg.lib.last_error()
    with pytest.raises(pkg.B200AsrError):
        pkg.lib.ptr(torch.zeros(3))            # host tensors are refused: no CPU fallback


@pytest.mark.parametrize("B,H,ndir,mode,exp", [
    (64, 512, 2, 0, (16, 32, 128)), (32, 640, 2, 0, (10, 32, 128)),
    (32, 512, 2, 0, (8, 32, 128)),          # tensor-core plan: 16-row halves, 8 units per CTA
    (32, 512, 2, 1, (16, 16, 128)),         # forced fp32-FMA kernels keep the old decomposition
    (8, 320, 2, 0, (10, 4, 128)),           # tiny batch: the FMA kernels stay cheaper than a padded MMA tile
    (130, 512, 2, 0, (16, 32, 128)),        # too many CTAs for one launch: three launches of 44 rows
    (64, 640, 2, 0, (10, 32, 128)),         # cfg D at batch 64: two launches of 32 rows
])
def test_lstm_plan_fills_the_sms(pkg, B, H, ndir, mode, exp):
    from ctypes import c_int, byref
    lib = pkg.load_library()
    ub, bc, n = c_int(), c_int(), c_int()
    lib.b200asr_debug_set_lstm_mode(mode)
    try:
        assert lib.b200asr_bilstm_plan(B, H, ndir, byref(ub), byref(bc), byref(n)) == 0
        assert (ub.value, bc.value, n.value) == exp
        assert n.value <= 148 and H % ub.value == 0
        assert lib.b200asr_bilstm_workspace_bytes(B, 100, H, ndir) > 0
    finally:
        lib.b200asr_debug_set_lstm_mode(0)


def test_host_tables_bit_identical_to_torchaudio(pkg):
    from torchaudio.compliance import kaldi
    d = pkg.audio.mel_filterbank(40, 512, 16000.0, 20.0, 0.0)
    ref, _ = kaldi.get_mel_banks(40, 512, 16000.0, 20.0, 0.0, 100.0, -500.0, 1.0)
    assert torch.equal(d[:, :256], ref) and float(d[:, 256].abs().max()) == 0
    w = pkg.audio.window_function("povey", 400)
    assert torch.equal(w, kaldi._feature_window_function("povey", 400, 0.42, torch.device("cpu"), torch.float32))
    s, c, o, ww = pkg.audio.sparsify_mel(d)
    dense = np.zeros((40, 257), np.float32)
    for i in range(40):
        dense[i, s[i]:s[i] + c[i]] = ww[o[i]:o[i] + c[i]]
    assert np.array_equal(dense, d.numpy())


def test_create_transform_contract(pkg):
    cfg = dict(feat_type="fbank", feat_dim=40, frame_length=25, frame_shift=10, dither=0, apply_cmvn=True,
               delta_order=2, delta_window_size=2)
    tr, dim = pkg.create_transform(cfg, device="cpu")
    assert dim == 120 and cfg["feat_type"] == "fbank"          # caller's dict untouched
    assert tr.frontend.num_frames(63040) == 392 and tr.frontend.num_frames(399) == 0
    with pytest.raises(NotImplementedError):
        pkg.create_transform(dict(cfg, dither=1.0))
    with pytest.raises(TypeError):
        pkg.create_transform(dict(cfg, not_an_option=3))


def test_state_dict_contract_matches_reference_goldens(pkg):
    from oracle.make_golden import tiny_model_cfg
    for kind in ("ctc", "hybrid", "cnn", "att"):
        g = load_golden("model_%s.npz" % kind)
        cfg = tiny_model_cfg(kind)
        model = pkg.ASR(8, 12, True, **cfg)
        ref_keys = {k[len("sd_shape."):]: v for k, v in g.items() if k.startswith("sd_shape.")}
        mine = {k: tuple(v.shape) for k, v in model.state_dict().items()}
        assert mine == {k: tuple(s) for k, s in ref_keys.items()}
        assert model.enable_ctc == (cfg["ctc_weight"] > 0) and model.enable_att == (cfg["ctc_weight"] != 1)
        assert model.encoder.sample_rate == (4 if kind == "cnn" else (1 if kind == "att" else 2))
        assert len(model.create_msg()) >= 2


def test_init_adadelta_matches_reference_quirks(pkg):
    """SURVEY F10: root-level re-init overrides the embedding special case; decoder forget-gate bias_ih = 1."""
    from oracle.make_golden import tiny_model_cfg
    torch.manual_seed(0)
    model = pkg.ASR(8, 500, True, **tiny_model_cfg("hybrid"))
    assert abs(float(model.pre_embed.weight.std()) - 1 / np.sqrt(32)) < 0.02
    b = model.decoder.layers.bias_ih_l0
    assert float(b[32:64].min()) == 1.0 and float(b[:32].abs().max()) == 0 and float(b[64:].abs().max()) == 0
    assert float(model.decoder.layers.bias_hh_l0.abs().max()) == 0


def test_lstm_planner_sweep_is_consistent(pkg):
    """Every (B, H, ndir) either has a plan that fits the machine (<= 148 co-resident CTAs, unit block divides H,
    a workspace size, tensor-core flag in {0,1}) or is refused with rc < 0 and a message - never a crash or a zero."""
    from ctypes import c_int, byref
    lib = pkg.load_library()
    ub, bc, n = c_int(), c_int(), c_int()
    seen_tc, seen_fma, refused = 0, 0, 0
    for H in (16, 32, 48, 64, 96, 128, 160, 256, 320, 512, 640, 768, 1024):
        for B in (1, 2, 3, 8, 16, 17, 32, 40, 64, 100, 130, 256):
            for ndir in (1, 2):
                rc = lib.b200asr_bilstm_plan(B, H, ndir, byref(ub), byref(bc), byref(n))
                tc = lib.b200asr_bilstm_uses_tensor_cores(B, H, ndir)
                ws = lib.b200asr_bilstm_workspace_bytes(B, 50, H, ndir)
                if rc != 0:
                    refused += 1
                    assert rc < 0 and tc == -1 and ws == 0 and "no feasible decomposition" in pkg.lib.last_error()
                    continue
                assert 1 <= n.value <= 148 and H % ub.value == 0 and 4 <= bc.value <= 64 and ws > 0
                assert tc in (0, 1)
                if tc:
                    assert bc.value == 32 and ub.value % 2 == 0 and ub.value <= 16 and H % 32 == 0
                    seen_tc += 1
                else:
                    seen_fma += 1
    assert seen_tc > 20 and seen_fma > 20
    assert lib.b200asr_bilstm_uses_tensor_cores(64, 512, 2) == 1 and lib.b200asr_bilstm_uses_tensor_cores(3, 16, 2) == 0
    lib.b200asr_debug_set_lstm_mode(1)
    try:
        assert lib.b200asr_bilstm_uses_tensor_cores(64, 512, 2) == 0
    finally:
        lib.b200asr_debug_set_lstm_mode(0)
