"""Generate tests/golden/*.npz by RUNNING the unmodified reference (CPU) in the build container.

    B200ASR_REFERENCE=<checkout of the original project> python -m oracle.make_golden     # from the repo root

The vectors pin the oracle (oracle_np.py, ref_port.py) and are the committed authority the GPU parity tests compare
against on the GPU box, where /root/reference does not exist.  Everything is seeded; sizes are tiny on purpose.
"""
import os
import sys
import zlib

import numpy as np
import torch

from . import ref_shim

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
GRAD_FULL_MAX = 32768       # gradients with more elements are stored as a sample of GRAD_SAMPLE of them (files < 1 MB)
GRAD_SAMPLE = 8192

AUDIO_CFG = dict(feat_type="fbank", feat_dim=40, frame_length=25, frame_shift=10, dither=0, apply_cmvn=True,
                 delta_order=2, delta_window_size=2)


def tiny_model_cfg(kind):
    enc = dict(prenet="", module="LSTM", bidirection=True, dim=[32, 32], dropout=[0, 0], layer_norm=[False, False],
               proj=[False, False], sample_rate=[1, 2], sample_style="concat")
    att = dict(mode="loc", dim=16, num_head=1, v_proj=False, temperature=0.5, loc_kernel_size=5, loc_kernel_num=4)
    dec = dict(module="LSTM", dim=32, layer=1, dropout=0)
    if kind == "ctc":
        return dict(ctc_weight=1.0, encoder=enc, attention=att, decoder=dec)
    if kind == "hybrid":
        return dict(ctc_weight=0.3, encoder=enc, attention=att, decoder=dec)
    if kind == "cnn":
        enc = dict(prenet="cnn", module="LSTM", bidirection=True, dim=[48, 48], dropout=[0, 0],
                   layer_norm=[False, False], proj=[True, True], sample_rate=[1, 1], sample_style="drop")
        return dict(ctc_weight=0.3, encoder=enc, attention=att, decoder=dec)
    if kind == "att":
        enc = dict(enc, sample_rate=[1, 1], proj=[True, False], sample_style="drop")
        dec = dict(dec, layer=2)
        return dict(ctc_weight=0.0, encoder=enc, attention=att, decoder=dec)
    if kind == "vgg":      # configs[0]'s prenet (config/libri/asr_example.yaml): VGG extractor, T not a multiple of 4
        enc = dict(prenet="vgg", module="LSTM", bidirection=True, dim=[32], dropout=[0], layer_norm=[False],
                   proj=[True], sample_rate=[1], sample_style="drop")
        return dict(ctc_weight=0.0, encoder=enc, attention=att, decoder=dec)
    if kind == "dot":      # scaled-dot attention, 2 heads, value projection, layer norm, GRU encoder layer
        enc = dict(prenet="", module="GRU", bidirection=True, dim=[32, 32], dropout=[0, 0],
                   layer_norm=[True, False], proj=[False, True], sample_rate=[1, 2], sample_style="drop")
        att = dict(mode="dot", dim=16, num_head=2, v_proj=True, temperature=0.5, loc_kernel_size=5, loc_kernel_num=4)
        return dict(ctc_weight=0.5, encoder=enc, attention=att, decoder=dec)
    raise KeyError(kind)


def synth_batch(seed, B, T, D, V, Lmax, ragged=True):
    g = torch.Generator().manual_seed(seed)
    feat_len = torch.full((B,), T, dtype=torch.long)
    if ragged:
        feat_len = torch.sort(torch.randint(max(T // 2, 8), T + 1, (B,), generator=g), descending=True)[0]
        feat_len[0] = T
    feat = torch.randn(B, T, D, generator=g)
    for b in range(B):
        feat[b, feat_len[b]:] = 0
    txt = torch.zeros(B, Lmax, dtype=torch.long)
    for b in range(B):
        L = int(torch.randint(2, Lmax, (1,), generator=g))
        ids = torch.randint(3, V, (L,), generator=g)
        if L > 3:
            ids[2] = ids[1]                      # force a repeated label (CTC needs the blank between them)
        txt[b, :L] = ids
        txt[b, L] = 1                            # <eos>
    return feat, feat_len, txt


def golden_frontend():
    from src.audio import create_transform                                    # the reference's
    from scipy.io import wavfile
    wav = os.path.join(ref_shim.REF_ROOT, "tests", "sample_data", "3830-12529-0005.wav")
    sr, pcm = wavfile.read(wav)
    out = {"sample_pcm": pcm.astype(np.int16), "sample_rate": np.int64(sr)}
    for order in (0, 1, 2):
        cfg = dict(AUDIO_CFG, delta_order=order)
        tr, dim = create_transform(cfg.copy())
        y = tr(wav)
        out["sample_feat_d%d" % order] = y.numpy().astype(np.float32)
    cfg = dict(AUDIO_CFG, delta_order=0, apply_cmvn=False)
    tr, _ = create_transform(cfg.copy())
    out["sample_fbank_raw"] = tr(wav).numpy().astype(np.float32)
    # synthetic, different lengths (incl. one exactly one frame long and one with a remainder)
    import torchaudio
    g = torch.Generator().manual_seed(1234)
    real_load = torchaudio.load
    for i, n in enumerate([400, 4000, 7013, 16000]):
        w = torch.clamp(0.05 * torch.randn(1, n, generator=g) + 0.02 * torch.sin(torch.arange(n) * 0.05 * (i + 1)),
                        -1, 1)
        torchaudio.load = lambda path, _w=w: (_w, 16000)
        tr, _ = create_transform(dict(AUDIO_CFG).copy())
        raw, _ = create_transform(dict(AUDIO_CFG, delta_order=0, apply_cmvn=False).copy())
        out["syn%d_wave" % i] = w[0].numpy()
        out["syn%d_raw" % i] = raw("x").numpy().astype(np.float32)
        if n > 400:
            out["syn%d_feat" % i] = tr("x").numpy().astype(np.float32)
    torchaudio.load = real_load
    np.savez_compressed(os.path.join(OUT, "frontend.npz"), **out)
    print("frontend.npz", {k: v.shape for k, v in out.items() if hasattr(v, "shape")})


def golden_model(kind, seed, B, T, D, V, Lmax):
    from src.asr import ASR                                                   # the reference's
    cfg = tiny_model_cfg(kind)
    torch.manual_seed(seed)
    model = ASR(D, V, True, **cfg)
    model.train()
    feat, feat_len, txt = synth_batch(seed + 1, B, T, D, V, Lmax)
    txt_len = (txt != 0).sum(-1)
    ctc_out, enc_len, att_out, att_seq, _ = model(feat, feat_len, int(txt_len.max()), tf_rate=1.0, teacher=txt)
    out = {"feat": feat.numpy(), "feat_len": feat_len.numpy(), "txt": txt.numpy(), "encode_len": enc_len.numpy()}
    total = 0
    if ctc_out is not None:
        ctc = torch.nn.CTCLoss(blank=0, zero_infinity=False)(ctc_out.transpose(0, 1), txt, enc_len, txt_len)
        total = total + ctc * model.ctc_weight
        out["ctc_output"] = ctc_out.detach().numpy()
        out["ctc_loss"] = ctc.detach().numpy()
        out["ctc_argmax"] = ctc_out.argmax(-1).numpy()
    if att_out is not None:
        b, t, _ = att_out.shape
        ce = torch.nn.CrossEntropyLoss(ignore_index=0)(att_out.view(b * t, -1), txt[:, :t].reshape(-1))
        total = total + ce * (1 - model.ctc_weight)
        out["att_output"] = att_out.detach().numpy()
        out["att_seq"] = att_seq.detach().numpy()
        out["att_loss"] = ce.detach().numpy()
        out["att_argmax"] = att_out.argmax(-1).numpy()
    total.backward()
    out["total_loss"] = total.detach().numpy()
    gn = torch.nn.utils.clip_grad_norm_(model.parameters(), 5.0)
    out["grad_norm"] = np.float32(gn)
    # The initial weights are the seeded init_adadelta initialisation, which the package's ASR reproduces bit for bit:
    # keep the seed and each tensor's shape and CRC-32 instead of the values (tests/conftest.py: golden_params).
    out["seed"], out["vocab"] = np.int64(seed), np.int64(V)
    for k, v in model.state_dict().items():
        out["sd_shape." + k] = np.asarray(v.shape, np.int64)
        out["sd_crc32." + k] = np.int64(zlib.crc32(np.ascontiguousarray(v.numpy()).tobytes()))
    rng = np.random.default_rng(seed)
    for k, p in model.named_parameters():
        if p.grad is not None:
            # clip_grad_norm_ scaled the grads in place: undo so the vectors hold the raw gradients
            coef = min(1.0, 5.0 / (float(gn) + 1e-6))
            grad = (p.grad / coef).numpy()
            if grad.size > GRAD_FULL_MAX:       # large gradients: a fixed random sample of their elements
                idx = np.sort(rng.choice(grad.size, GRAD_SAMPLE, replace=False)).astype(np.int32)
                out["grad_idx." + k] = idx
                grad = grad.reshape(-1)[idx]
            out["grad." + k] = grad
    # greedy inference outputs as well (teacher=None, argmax feedback), src/asr.py:137-142
    if att_out is not None:
        model.eval()
        with torch.no_grad():
            _, _, g_out, g_seq, _ = model(feat, feat_len, int(txt_len.max()) + 2)
        out["greedy_argmax"] = g_out.argmax(-1).numpy()
        out["greedy_output"] = g_out.numpy()
    np.savez_compressed(os.path.join(OUT, "model_%s.npz" % kind), **out)
    print("model_%s.npz" % kind, "loss", float(total), "grad_norm", float(gn))


def golden_ctc():
    """torch.nn.functional.ctc_loss + torch._ctc_loss (log_alpha) on adversarial small cases."""
    g = torch.Generator().manual_seed(7)
    cases = []
    # (T, V, targets, input_len)
    specs = [
        (12, 6, [1, 2, 2, 3], 12),       # repeated label
        (10, 5, [], 10),                 # empty target
        (7, 5, [1, 1, 1, 1], 7),         # exactly feasible (needs 4 + 3 blanks = 7)
        (6, 5, [1, 1, 1, 1], 6),         # infeasible -> inf
        (15, 8, [3, 4, 5, 3, 4, 5, 6], 9),   # input shorter than T
        (1, 4, [2], 1),                  # single frame
    ]
    out = {}
    for i, (T, V, tgt, il) in enumerate(specs):
        lp = torch.randn(T, 1, V, generator=g).log_softmax(-1).requires_grad_(True)
        t = torch.tensor([tgt + [0]], dtype=torch.long) if tgt else torch.zeros(1, 1, dtype=torch.long)
        tl = torch.tensor([len(tgt)])
        ilt = torch.tensor([il])
        nll, log_alpha = torch._ctc_loss(lp, t, ilt, tl, 0, False)
        loss = torch.nn.functional.ctc_loss(lp, t, ilt, tl, blank=0, reduction="sum", zero_infinity=False)
        loss.backward()
        out["c%d_lp" % i] = lp.detach()[:, 0].numpy()
        out["c%d_tgt" % i] = t[0].numpy()
        out["c%d_tl" % i] = tl.numpy()
        out["c%d_il" % i] = ilt.numpy()
        out["c%d_nll" % i] = nll.detach().numpy()
        out["c%d_alpha" % i] = log_alpha.detach()[0].numpy()
        out["c%d_grad" % i] = lp.grad[:, 0].numpy()
    out["n_cases"] = np.int64(len(specs))
    np.savez_compressed(os.path.join(OUT, "ctc_cases.npz"), **out)
    print("ctc_cases.npz", len(specs), "cases")


def golden_prefix():
    """CTCPrefixScore (src/ctc.py:12-116) driven like src/decode.py:93-131: empty prefix, then three extensions, each
    with a candidate list that contains <eos> and the prefix's last token."""
    from src.ctc import CTCPrefixScore                                          # the reference's numpy scorer
    g = torch.Generator().manual_seed(77)
    T, V = 37, 12
    x = torch.randn(1, T, V, generator=g).log_softmax(-1)
    sc = CTCPrefixScore(x)
    out = {"x": x.numpy()}
    r_prev = sc.init_state()
    out["r_init"] = r_prev.copy()
    prefix = []
    for step, (cands, pick) in enumerate([([3, 1, 5, 7], 0), ([3, 5, 1, 9, 2], 1), ([5, 1, 4, 11], 0),
                                          ([1, 5, 6, 10, 8, 3], 3)]):
        psi, r = sc.cheap_compute(prefix, r_prev, cands)
        out["s%d_prefix" % step] = np.asarray(prefix, np.int64)
        out["s%d_cands" % step] = np.asarray(cands, np.int64)
        out["s%d_rprev" % step] = r_prev.copy()
        out["s%d_psi" % step] = psi.copy()
        out["s%d_r" % step] = r.copy()
        prefix = prefix + [cands[pick]]
        r_prev = r[pick]
    out["n_steps"] = np.int64(4)
    np.savez_compressed(os.path.join(OUT, "ctc_prefix.npz"), **out)
    print("ctc_prefix.npz")


PLUMBING_UTTS = [("3830-12529-0005", 63040, "THE QUICK BROWN FOX JUMPS OVER"), ("3830-12529-0006", 56000, "THE LAZY DOG SLEEPS"),
                 ("3830-12529-0007", 48000, "HELLO WORLD"), ("3830-12529-0008", 40000, "SPEECH")]


def plumbing_tree(root, pcm, ext="flac"):
    """LibriSpeech-shaped tree (corpus/librispeech.py:19-25,37) of 4 utterances cut from the sample wav: 16-bit PCM wav
    data under the extension the dataset class globs for (SURVEY.md 8(c) shim 3) + a made-up transcript file."""
    from scipy.io import wavfile
    d = os.path.join(root, "LibriSpeech", "dev-clean", "3830", "12529")
    os.makedirs(d, exist_ok=True)
    with open(os.path.join(d, "3830-12529.trans.txt"), "w") as f:
        for name, n, text in PLUMBING_UTTS:
            f.write("%s %s\n" % (name, text))
            with open(os.path.join(d, "%s.%s" % (name, ext)), "wb") as w:
                wavfile.write(w, 16000, np.asarray(pcm[:n], dtype=np.int16))
    return os.path.join(root, "LibriSpeech")


def plumbing_config(cfg, path, vocab_file):
    """The edits configs[0] needs on asr_example.yaml to run on the fixture (the same for the reference and for the
    repo's config/b200/cfgA_example_vgg.yaml)."""
    cfg["data"]["corpus"].update(path=path, train_split=["dev-clean"], dev_split=["dev-clean"], batch_size=2)
    cfg["data"]["text"] = {"mode": "character", "vocab_file": vocab_file}
    cfg["hparas"].update(max_step=2, curriculum=1)
    return cfg


def golden_plumbing():
    """BASELINE configs[0]: the reference's own Solver (main.py:76-79 with --cpu) on the fixture, 2 train steps from
    seed-0 weights; the attention loss and grad-norm of each step are the golden values."""
    import argparse
    import tempfile
    import yaml
    import bin.train_asr as ref_train
    from bin.train_asr import Solver
    # validation (step 1) draws attention maps through matplotlib, which is not installed: a blank image instead
    ref_train.feat_to_fig = lambda feat: (torch.zeros(8, 8, 3), "HWC")
    pcm = np.load(os.path.join(OUT, "frontend.npz"))["sample_pcm"]
    tmp = tempfile.mkdtemp(prefix="b200asr_plumbing_")
    path = plumbing_tree(tmp, pcm, "flac")
    cfg = yaml.load(open(os.path.join(ref_shim.REF_ROOT, "config", "libri", "asr_example.yaml")), Loader=yaml.FullLoader)
    cfg = plumbing_config(cfg, path, os.path.join(OUT, "character.vocab"))
    own = yaml.load(open(os.path.join(os.path.dirname(OUT), "..", "config", "b200", "cfgA_example_vgg.yaml")),
                    Loader=yaml.FullLoader)
    own = plumbing_config(own, path, os.path.join(OUT, "character.vocab"))
    assert own == cfg, "config/b200/cfgA_example_vgg.yaml drifted from the reference's asr_example.yaml"
    paras = argparse.Namespace(config="asr_example.yaml", name="plumbing", logdir=os.path.join(tmp, "log"),
                               ckpdir=os.path.join(tmp, "ckpt"), outdir=os.path.join(tmp, "out"), load=None, seed=0,
                               cudnn_ctc=False, njobs=0, cpu=True, no_pin=True, test=False, no_msg=True, lm=False,
                               amp=False, reserve_gpu=0, jit=False, gpu=False, pin_memory=False, verbose=False)
    torch.set_num_threads(8)
    np.random.seed(0)
    solver = Solver(cfg, paras, "train")
    solver.load_data()
    torch.manual_seed(0)                     # the weights are a function of this seed alone (tests re-seed the same way)
    solver.set_model()
    losses, norms, names = [], [], []
    real_backward, real_fetch = solver.backward, solver.fetch_data

    def backward(loss):
        losses.append(float(loss))
        n = real_backward(loss)
        norms.append(float(n))
        return n

    def fetch(data):
        names.append(list(data[0]))
        return real_fetch(data)

    solver.backward, solver.fetch_data = backward, fetch
    solver.exec()
    out = {"loss": np.asarray(losses, np.float64), "grad_norm": np.asarray(norms, np.float64),
           "names": np.asarray([",".join(n) for n in names]), "n_params": np.int64(sum(p.numel() for p in solver.model.parameters()))}
    np.savez_compressed(os.path.join(OUT, "plumbing.npz"), **out)
    print("plumbing.npz", losses, norms, names)


def main():
    ref_shim.install()
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(1)
    golden_frontend()
    golden_ctc()
    golden_prefix()
    golden_model("ctc", 11, 3, 24, 8, 12, 5)
    golden_model("hybrid", 21, 3, 24, 8, 12, 5)
    golden_model("cnn", 31, 2, 40, 8, 12, 5)
    golden_model("att", 41, 3, 16, 8, 12, 6)
    golden_model("vgg", 51, 2, 26, 40, 12, 5)
    golden_model("dot", 61, 3, 20, 8, 12, 5)
    golden_plumbing()


if __name__ == "__main__":
    main()
