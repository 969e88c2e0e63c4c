#!/usr/bin/env python
"""Benchmark of the ASR train-step hot path (BASELINE.json metric: utterances/sec, ~12 s @ 16 kHz synthetic).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfgB|cfgC|cfgD] [--impl b200|reference]
                    [--dump-outputs DIR]

One "step" = one full train step over one synthetic batch: fused front end (STFT+mel+log, delta, CMVN) -> encoder ->
CTC (+ attention decoder + CE) -> backward -> [NCCL grad all-reduce] -> grad-norm / clip / Adadelta.
  value : whole-job utt/s with the waveforms already resident in HBM (device-timed, CUDA events, max over ranks);
  e2e   : the same step driven from pinned HOST buffers: H2D of the waveforms + targets and D2H of the loss inside
          the timed region, through the package's public TrainStep API;
  roofline     : the dominant hand-written kernel (by device time inside the timed region, CUDA events on the
                 launching stream), algorithmic bytes per SURVEY.md 8(d) over its mean launch duration, against
                 the measured HBM peak of MEASURED_PEAKS.json;
  cpu_baseline : the reference's CPU path (oracle/ref_port.py = the same ATen/torchaudio CPU kernels the reference
                 calls) on a bounded sample of the same workload, on this box's host cores.
--impl reference prints the CPU arm alone (rank 0 only under torchrun).
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

PKG = "end-to-end-asr-pytorch_b200"
METRIC = "utterances/sec (train step, ~12s@16kHz synthetic)"
UNIT = "utt/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfgB", choices=["cfgB", "cfgC", "cfgD"])
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the workload's)")
    ap.add_argument("--n-samples", type=int, default=192000)
    ap.add_argument("--cpu-batch", type=int, default=0, help="utterances per CPU-baseline step (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="time the eager step instead of the CUDA-graph replay")
    ap.add_argument("--no-parity-fp64", action="store_true",
                    help="parity block of the benchmarked workload: skip the extra fp64 CPU pass (both fp32 sides - the "
                         "reference's CPU path and these kernels - against the exact gradient)")
    ap.add_argument("--parity-diagnose", action="store_true",
                    help="parity block: also compare d(loss)/d(layer outputs, CTC logits) of both fp32 sides with fp64")
    ap.add_argument("--graph-dp", action="store_true",
                    help="N > 1: capture the data-parallel step (NCCL all-reduces included) into the CUDA graph as well")
    ap.add_argument("--no-micro", action="store_true", help="skip the fbank/CTC micro-benchmark (BASELINE configs[4])")
    ap.add_argument("--no-also", action="store_true", help="multi-GPU runs: skip the extra cfgD (BASELINE configs[3]) timing")
    ap.add_argument("--no-parity", action="store_true", help="skip the same-run parity check against the CPU path")
    ap.add_argument("--parity-workloads", default="auto",
                    help="comma list of workloads parity-checked at full size after the timed regions "
                         "(auto = the benchmarked one, plus cfgB,cfgC,cfgD on a default 1-GPU run)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy: loss, grad_norm, and a fixed "
                         "sample of the updated parameters and of the gradient (params, grad), so that two builds can "
                         "be compared output for output on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 train step")
    return args


T0 = time.time()


def log(msg):
    """progress on stderr (stdout carries exactly one JSON line)"""
    sys.stderr.write("[bench %6.1fs] %s\n" % (time.time() - T0, msg))
    sys.stderr.flush()


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for n, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


DUMP_SAMPLE = 4 << 20       # elements kept of each flat buffer: 2 x 16 MB of float32


def step_outputs(step_fn, loss):
    """What a caller of the train step holds after it, as float arrays: the loss it returned, the gradient norm, and
    the model's flat parameter buffer (after the update) and gradient buffer.  A buffer larger than DUMP_SAMPLE
    elements is cut to a fixed random sample of that many (seed 0, ascending indices)."""
    import numpy as np
    buf = step_fn.optimizer.buf
    idx = None
    if buf.total > DUMP_SAMPLE:
        idx = np.sort(np.random.default_rng(0).choice(buf.total, DUMP_SAMPLE, replace=False))
        idx = torch.from_numpy(idx).to(buf.flat.device)
    pick = (lambda t: t) if idx is None else (lambda t: t[idx])
    return {"loss": np.array([loss], np.float32),
            "grad_norm": step_fn.optimizer.grad_norm.detach().cpu().numpy().astype(np.float32),
            "params": pick(buf.flat).cpu().numpy(), "grad": pick(buf.grad).cpu().numpy()}


def build_cpu_reference(cfg, vocab, seed=0):
    """Parameter dict initialised like the reference (init_adadelta) for the CPU arm."""
    pkg = importlib.import_module(PKG)
    torch.manual_seed(seed)
    audio = cfg["data"]["audio"]
    feat_dim = audio["feat_dim"] * (audio.get("delta_order", 0) + 1)
    model = pkg.ASR(feat_dim, vocab, True, **cfg["model"])        # parameters only; never run on the CPU
    return {k: v.detach().clone() for k, v in model.state_dict().items()}


def calibrate_threads(cfg, vocab):
    """The reference would run with torch's default (= all cores).  On a many-core host the small per-step LSTM
    GEMMs get slower with more threads, so give the CPU arm its best thread count: time one short step at
    8, 16, 32, ... cores and stop as soon as it gets slower."""
    from oracle import ref_port
    pkg = importlib.import_module(PKG)
    ncpu = os.cpu_count() or 1
    cands = [c for c in (8, 16, 32, 64) if c < ncpu] + [ncpu]
    P = build_cpu_reference(cfg, vocab)
    waves, lens, txt = pkg.synthetic.make_batch(vocab, 2, 32000, seed=7)
    wl = [waves[b:b + 1] for b in range(2)]
    tl = [[int(v) for v in txt[b] if int(v) != 0] for b in range(2)]
    best, best_t = cands[0], None
    for c in cands:
        torch.set_num_threads(c)
        tr = ref_port.CpuTrainer(P, cfg["model"], cfg["data"]["audio"])
        tr.step(wl, tl)
        t0 = time.perf_counter()
        tr.step(wl, tl)
        dt = time.perf_counter() - t0
        log("cpu calibration: %d threads -> %.2f s" % (c, dt))
        if best_t is None or dt < best_t:
            best, best_t = c, dt
        elif dt > 1.15 * best_t:
            break
    return best


def cpu_arm(cfg, vocab, n_samples, batch, steps, warmup):
    """Time the reference's CPU path (oracle port) for `steps` steps of `batch` utterances."""
    from oracle import ref_port
    pkg = importlib.import_module(PKG)
    torch.set_num_threads(calibrate_threads(cfg, vocab))
    P = build_cpu_reference(cfg, vocab)
    trainer = ref_port.CpuTrainer(P, cfg["model"], cfg["data"]["audio"], lr=cfg["hparas"]["lr"],
                                  eps=cfg["hparas"]["eps"])
    waves, lens, txt = pkg.synthetic.make_batch(vocab, batch, n_samples, seed=1000)
    wl = [waves[b:b + 1, :int(lens[b])] for b in range(batch)]
    tl = [[int(v) for v in txt[b] if int(v) != 0] for b in range(batch)]
    times = []
    loss = None
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        loss, _ = trainer.step(wl, tl)
        dt = time.perf_counter() - t0
        log("cpu step %d: %.2f s (%d threads)" % (i, dt, torch.get_num_threads()))
        if i >= warmup:
            times.append(dt)
    total = sum(times)
    return {"value": batch * len(times) / total, "ms_per_step": 1000.0 * total / len(times), "batch": batch,
            "cores": torch.get_num_threads(), "loss": loss}


def parity_check(pkg, step_fn, cfg, waves, lens, txt, dev, n_ref=8, fp64=False, diagnose=False):
    """Same-run, full-size parity (BASELINE metric, second half): the product path on the FULL per-GPU batch - front
    end, encoder, CTC head / decoder, both losses, backward, all through the CUDA kernels at the benchmark's shapes -
    against the reference's CPU path (oracle/ref_port.py: kaldi.fbank per utterance, ATen LSTM / CTC / CE) on the
    first `n_ref` utterances, from the SAME state_dict and the SAME waveforms.  The GPU loss is restricted to those
    utterances (CTC weights 0 and CE targets ignored for the others), so losses and every parameter gradient are
    directly comparable while all B rows run through the kernels.  Utterances are independent given the global T_max
    (SURVEY.md F5), which both sides share.  Mirrors /root/reference/bin/train_asr.py:104-137."""
    from oracle import ref_port
    import numpy as np
    model, opt = step_fn.model, step_fn.optimizer
    lam = model.ctc_weight
    B = waves.shape[0]
    n = min(n_ref, B)
    P = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}
    # ---- product path
    model.train()
    opt.pre_step(step_fn.step_id)                      # zero the flat gradient buffer
    wave_dev, txt_dev = waves.to(dev), txt.to(dev)
    feat, feat_len = step_fn.front_end(wave_dev, lens.to(dev))
    txt_len = (txt_dev != 0).sum(-1)
    taps, hooks = {}, []
    if diagnose:        # gradient of the loss with respect to every encoder layer's output (and the CTC logits below)
        def tap(i):
            def hook(mod, inp, outp):
                if isinstance(outp[0], torch.Tensor) and outp[0].requires_grad:
                    outp[0].retain_grad()
                    taps["layer%d_out" % i] = outp[0]
            return hook
        hooks = [layer.register_forward_hook(tap(i)) for i, layer in enumerate(model.encoder.layers)]
    ctc_out, enc_len, att_out, _, _ = model(feat, feat_len, int(txt.shape[1]), tf_rate=1.0, teacher=txt_dev)
    for h in hooks:
        h.remove()
    if diagnose and isinstance(ctc_out, pkg.ops.CTCHeadOutput):
        ctc_out.logits.retain_grad()
        taps["ctc_logits"] = ctc_out.logits
    total = 0
    g = {}
    if ctc_out is not None:
        w = torch.zeros(B, device=dev)
        w[:n] = 1.0 / (txt_len[:n].clamp_min(1).float() * n)
        if isinstance(ctc_out, pkg.ops.CTCHeadOutput):     # fused CTC head (the train step's path): logits + row lse
            ctc, nll = pkg.ops.CTCLossFn.apply(ctc_out.logits.transpose(0, 1), txt_dev, enc_len, txt_len, 0, w, ctc_out.lse)
            lp_dev = ctc_out.materialize()
        else:
            ctc, nll = pkg.ops.CTCLossFn.apply(ctc_out.transpose(0, 1), txt_dev, enc_len, txt_len, 0, w)
            lp_dev = ctc_out
        total = total + ctc * lam
        g.update(ctc_loss=float(ctc), nll=nll[:n].detach().cpu().double().numpy(),
                 ctc_output=lp_dev[:n].detach().cpu(), ctc_argmax=model.last_ctc_argmax[:n].cpu())
    if att_out is not None:
        b, t, v = att_out.shape
        tgt = txt_dev[:, :t].clone()
        tgt[n:] = 0
        ce = pkg.ops.cross_entropy(att_out.reshape(b * t, v), tgt.reshape(-1), ignore_index=0)
        total = total + ce * (1 - lam)
        g.update(att_loss=float(ce), att_output=att_out[:n].detach().cpu())
    total.backward()
    if model.enable_att:
        model.attention.reset_mem()
        model.decoder.hidden_state = None
    opt.buf.rebind_grads()
    torch.cuda.synchronize()
    g_grads = {k: p.grad.detach().cpu().clone() for k, p in model.named_parameters() if p.grad is not None}
    g_feat = feat[:n].detach().cpu()
    # ---- reference CPU path
    torch.set_num_threads(min(16, os.cpu_count() or 1))
    Pr = {k: v.clone().requires_grad_(True) for k, v in P.items()}
    wl = [waves[b:b + 1, :int(lens[b])] for b in range(n)]
    tl = [[int(x) for x in txt[b] if int(x) != 0] for b in range(n)]
    f_ref, l_ref, t_ref, order = ref_port.collate(wl, cfg["data"]["audio"], tl)
    assert order == list(range(n)), "synthetic batch must already be sorted by length"
    if f_ref.shape[1] < feat.shape[1]:                 # the encoder computes through padding: share the global T_max
        f_ref = torch.nn.functional.pad(f_ref, (0, 0, 0, feat.shape[1] - f_ref.shape[1]))
    col32 = [] if diagnose else None
    res = ref_port.forward_losses(Pr, cfg["model"], f_ref, l_ref, t_ref, collect=col32)
    if diagnose:
        for t in col32 + [res["ctc_output"]]:
            t.retain_grad()
    res["total_loss"].backward()

    def rel(a, b, floor):
        a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
        return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), floor)))

    out = {"utterances_compared": n, "batch_through_kernels": B, "frames": int(feat.shape[1]),
           "feat_max_abs_err": float((g_feat - f_ref).abs().max()),
           "total_loss_rel_err": abs(float(total) - float(res["total_loss"])) / abs(float(res["total_loss"]))}
    if ctc_out is not None:
        lp_ref = res["ctc_output"].detach()
        lp = g["ctc_output"][:, :lp_ref.shape[1]]
        nll_ref = torch.nn.functional.ctc_loss(lp_ref.transpose(0, 1), t_ref, res["encode_len"], (t_ref != 0).sum(-1),
                                               blank=0, reduction="none").double().numpy()
        am_ref = lp_ref.argmax(-1)
        mism = (g["ctc_argmax"][:, :am_ref.shape[1]] != am_ref)
        top2 = lp_ref.topk(2, dim=-1).values
        margin = (top2[..., 0] - top2[..., 1])
        out.update(ctc_loss_rel_err=abs(g["ctc_loss"] - float(res["ctc_loss"])) / abs(float(res["ctc_loss"])),
                   ctc_nll_rel_err=rel(g["nll"], nll_ref, 1e-3),
                   logits_rel_err=rel(lp.numpy(), lp_ref.numpy(), 1.0),
                   logits_max_abs_err=float((lp - lp_ref).abs().max()),
                   ctc_argmax_equal=bool(not mism.any()), ctc_argmax_mismatches=int(mism.sum()),
                   ctc_argmax_frames=int(mism.numel()),
                   ctc_argmax_mismatch_max_ref_margin=float(margin[mism].max()) if mism.any() else 0.0)
    if att_out is not None:
        a_ref = res["att_output"].detach()
        a = g["att_output"][:, :a_ref.shape[1]]
        mism = a.argmax(-1) != a_ref.argmax(-1)
        top2 = a_ref.topk(2, dim=-1).values
        margin = (top2[..., 0] - top2[..., 1])
        out.update(att_loss_rel_err=abs(g["att_loss"] - float(res["att_loss"])) / abs(float(res["att_loss"])),
                   att_logits_rel_err=rel(a.numpy(), a_ref.numpy(), 1.0),
                   att_logits_max_abs_err=float((a - a_ref).abs().max()),
                   att_argmax_equal=bool(not mism.any()), att_argmax_mismatches=int(mism.sum()),
                   att_argmax_tokens=int(mism.numel()),
                   att_argmax_mismatch_max_ref_margin=float(margin[mism].max()) if mism.any() else 0.0)
    sq_g = sq_r = 0.0
    worst, worst_key = 0.0, None
    errs = []
    for k, ref in Pr.items():
        if ref.grad is None or k not in g_grads:
            continue
        r = ref.grad.double()
        d = g_grads[k].double()
        sq_g += float((d ** 2).sum())
        sq_r += float((r ** 2).sum())
        errs.append((k, float((d - r).abs().max()), float(r.abs().max())))
    gmax = max(m for _, _, m in errs)
    for k, e, m in errs:
        # error relative to the tensor's own scale; tensors whose true gradient is zero up to rounding (e.g. the
        # softmax-invariant energy bias) are measured against 1e-6 of the largest gradient instead
        e = e / max(m, 1e-6 * gmax)
        if e > worst:
            worst, worst_key = e, k
    out.update(grad_norm_rel_err=abs(sq_g ** 0.5 - sq_r ** 0.5) / sq_r ** 0.5, grad_norm_ref=sq_r ** 0.5,
               grad_max_scaled_err=worst, grad_worst_tensor=worst_key)
    if fp64:
        # The same CPU path once more in fp64: how far is EACH fp32 implementation (the reference's ATen path and these
        # kernels) from the exact gradient?  The step back-propagates through thousands of recurrent steps; the fp32
        # reference itself only holds ~4e-5 here, which is the floor of any fp32-vs-fp32 gradient comparison.
        P64 = {k: (v.double() if v.is_floating_point() else v).clone().requires_grad_(v.is_floating_point())
               for k, v in P.items()}
        col64 = [] if diagnose else None
        r64 = ref_port.forward_losses(P64, cfg["model"], f_ref.double(), l_ref, t_ref, collect=col64)
        if diagnose:
            for t in col64 + [r64["ctc_output"]]:
                t.retain_grad()
        r64["total_loss"].backward()
        sq = {"x": 0.0, "ref": 0.0, "own": 0.0}
        w = {"ref": (0.0, None), "own": (0.0, None)}
        g64 = {k: v.grad for k, v in P64.items() if v.requires_grad and v.grad is not None and k in g_grads
               and Pr[k].grad is not None}
        gmax64 = max(float(v.abs().max()) for v in g64.values())
        for k, x in g64.items():
            sq["x"] += float((x ** 2).sum())
            for name, t in (("ref", Pr[k].grad.double()), ("own", g_grads[k].double())):
                sq[name] += float((t ** 2).sum())
                e = float((t - x).abs().max()) / max(float(x.abs().max()), 1e-6 * gmax64)
                if e > w[name][0]:
                    w[name] = (e, k)
        nx = sq["x"] ** 0.5
        out["vs_fp64"] = {
            "reference_fp32": {"grad_norm_rel_err": abs(sq["ref"] ** 0.5 - nx) / nx, "grad_max_scaled_err": w["ref"][0],
                               "grad_worst_tensor": w["ref"][1],
                               "loss_rel_err": abs(float(res["total_loss"]) - float(r64["total_loss"])) / abs(float(r64["total_loss"]))},
            "these_kernels": {"grad_norm_rel_err": abs(sq["own"] ** 0.5 - nx) / nx, "grad_max_scaled_err": w["own"][0],
                              "grad_worst_tensor": w["own"][1],
                              "loss_rel_err": abs(float(total) - float(r64["total_loss"])) / abs(float(r64["total_loss"]))}}
    if fp64 and diagnose:
        # where does the gradient noise enter?  d(loss)/d(boundary) of both fp32 sides against fp64, top of the network
        # first (the CTC head's log-prob gradient equals the logit gradient: SURVEY F9), max error / max |exact|
        rows = {}
        names = ["ctc_logits"] + ["layer%d_out" % i for i in reversed(range(len(col64)))]
        exact = [r64["ctc_output"].grad] + [t.grad for t in reversed(col64)]
        ref32 = [res["ctc_output"].grad] + [t.grad for t in reversed(col32)]
        for name, x, r in zip(names, exact, ref32):
            if name not in taps or taps[name].grad is None:
                continue
            o = taps[name].grad[:n].detach().cpu().double()
            if o.shape != x.shape:       # this package's encoder tensors keep the pre-subsampling time axis / full T_max
                if o.numel() == x.numel():
                    o = o.reshape(x.shape)
                else:
                    rows[name] = {"shape_own": list(o.shape), "shape_ref": list(x.shape)}
                    continue
            sc = float(x.abs().max())
            rows[name] = {"own_vs_fp64": float((o - x).abs().max()) / sc, "ref32_vs_fp64": float((r.double() - x).abs().max()) / sc,
                          "own_norm_rel_err": abs(float(o.norm()) - float(x.norm())) / float(x.norm()),
                          "ref32_norm_rel_err": abs(float(r.double().norm()) - float(x.norm())) / float(x.norm())}
        out["vs_fp64"]["boundaries"] = rows
    opt.buf.grad.zero_()
    return out


def micro_bench(pkg, dev, peak):
    """BASELINE.json configs[4]: mel-fbank (+delta+CMVN) and the CTC kernels on 1000 synthetic utterances of 2-30 s
    (front end: batches of 100; CTC: batches of 250 = 500 lattice warps per launch, enough to occupy the 148 SMs of the
    T'-long latency chain - the train step's batch of 64 is reported by the `kernels` table instead; zero padded to the
    batch maximum), L2 flushed (256 MB write) before every timed launch, CUDA
    events per C-ABI launch.  Algorithmic bytes per SURVEY.md 8(d): fbank 4N + 160m, delta+CMVN 4m(40+120), CTC
    2*4*T'*V (+4*T'*V logits read for the log-softmax that feeds it).  Returns {kernel: {ms, GB/s, frac of HBM peak}}."""
    cfg = pkg.synthetic.load_config("cfgB")
    tr, _ = pkg.create_transform(dict(cfg["data"]["audio"]), device=dev)
    fe = tr.frontend
    g = torch.Generator().manual_seed(0)
    lens = torch.randint(32000, 480001, (1000,), generator=g).sort(descending=True)[0]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    T = pkg.lib.TIMER
    acc = {}

    def run(fn, names):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        for _ in range(3):
            flush.zero_()
            T.reset()
            T.enabled = True
            fn()
            torch.cuda.synchronize()
            T.enabled = False
            for k, d in T.summary().items():
                if k in names:
                    acc.setdefault(k, []).append((d["ms"], d["bytes"]))

    for i in range(0, 1000, 100):
        l = lens[i:i + 100]
        wave = torch.zeros(100, int(l[0]), device=dev)
        for b in range(100):
            wave[b, :int(l[b])] = 0.05 * torch.randn(int(l[b]), device=dev)
        run(lambda: fe(wave, l), ("fbank_fwd", "delta_cmvn_fwd"))
        del wave
    out = {}
    for V, Lr in ((31, (20, 130)), (5000, (6, 45))):
        CB = 250
        for i in range(0, 1000, CB):
            l = lens[i:i + CB]
            Tp = ((l - 400) // 160 + 1) // 4
            Tm = int(Tp.max())
            logits = torch.randn(CB, Tm, V, device=dev, requires_grad=True)
            tl = torch.minimum(torch.randint(Lr[0], Lr[1], (CB,), generator=g), (Tp // 3).clamp(min=1))
            txt = torch.zeros(CB, int(tl.max()), dtype=torch.long)
            for b in range(CB):
                txt[b, :tl[b]] = torch.randint(1, V, (int(tl[b]),), generator=g)
            txt, Td, tld = txt.to(dev), Tp.to(dev), tl.to(dev)
            crit = pkg.CTCLoss(blank=0)

            def step():
                logits.grad = None
                head = pkg.ops.ctc_head(logits)                 # fused CTC head: row lse + arg-max, no V-wide output
                crit(head.transpose(0, 1), txt, Td, tld).backward()
            run(step, ("log_softmax_fwd", "ctc_alpha_beta", "ctc_grad"))
            del logits
        for k in ("log_softmax_fwd", "ctc_alpha_beta", "ctc_grad"):
            acc["%s_V%d" % (k, V)] = acc.pop(k, [])
    for k, rows in acc.items():
        if not rows:
            continue
        # per batch: median of its 3 timed launches; totals over the 10 batches
        n = len(rows) // 3
        ms = sum(sorted(r[0] for r in rows[3 * j:3 * j + 3])[1] for j in range(n))
        by = sum(rows[3 * j][1] for j in range(n))
        out[k] = {"ms_per_1000_utt": ms, "algorithmic_gbs": by / (ms * 1e-3) / 1e9, "frac_hbm": by / (ms * 1e-3) / 1e9 / peak}
    for V in (31, 5000):
        ks = ["log_softmax_fwd_V%d" % V, "ctc_alpha_beta_V%d" % V, "ctc_grad_V%d" % V]
        if all(k in out for k in ks):
            ms = sum(out[k]["ms_per_1000_utt"] for k in ks)
            by = out[ks[0]]["algorithmic_gbs"] * out[ks[0]]["ms_per_1000_utt"] * 1e6 + \
                out[ks[2]]["algorithmic_gbs"] * out[ks[2]]["ms_per_1000_utt"] * 1e6      # 4T'V (logits) + 8T'V
            out["ctc_total_V%d" % V] = {"ms_per_1000_utt": ms, "algorithmic_gbs": by / (ms * 1e-3) / 1e9,
                                        "frac_hbm": by / (ms * 1e-3) / 1e9 / peak,
                                        "note": "fused CTC head: logits -> row lse + arg-max -> alpha/beta on logits - lse -> logit gradient; "
                                                "12*T'*V bytes, no V-wide log-prob tensor"}
    return out


def main():
    args = parse_args()
    pkg = importlib.import_module(PKG)
    cfg = pkg.synthetic.load_config(args.workload)
    vocab = cfg["data"]["corpus"]["vocab_size"]
    per_gpu = args.batch or cfg["data"]["corpus"]["batch_size"]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    config = {"workload": "%s: %s" % (args.workload, pkg.synthetic.WORKLOADS[args.workload]),
              "global_batch": per_gpu * world, "per_gpu_batch": per_gpu, "n_samples": args.n_samples,
              "frames": 1 + (args.n_samples - 400) // 160, "vocab": vocab,
              "parallelism": "dp%d (utterance shards; per-layer NCCL grad all-reduce buckets overlapped with backward)" % world,
              "l2": "inputs+activations per step (>1 GB) exceed the 126 MB L2; no explicit flush",
              "gemm": "own tcgen05 3xTF32 kernel in three operand forms (x.W^T, dY.W, dY^T.X incl. shifted h_prev reads, split-K, "
                      "gate permutation in the epilogue), weight residuals (and the wide operand of the weight gradients) pre-split once per step, two-level accumulation (TMEM "
                      "chunks of 128 k summed in fp32 registers); B200ASR_GEMM=tf32x3 selects the cuBLAS 3xTF32 composition; fp32-accurate",
              "lstm": "tcgen05 fp16 hi/lo 2x2-block split product, forward and backward (H = 256 ... 768; backward exchange: data-is-the-flag polling)"}

    # ------------------------------------------------------------------------------- reference (CPU) arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        nsteps = args.steps + args.warmup
        cb = args.cpu_batch or (8 if nsteps <= 25 else (4 if nsteps <= 60 else 2))
        r = cpu_arm(cfg, vocab, args.n_samples, cb, args.steps, args.warmup)
        sample = "%d-utterance steps of the same workload (reference CPU path via oracle/ref_port.py)" % cb
        line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": dict(config, cpu_batch=cb),
                "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                                 "sample": sample + "; thread count calibrated (best of 8/16/32/64/all cores)"},
                "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------------------- B200 arm
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    dp = pkg.dist.DataParallel()
    local = dp.local_rank if dp.enabled else 0
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    lib = pkg.load_library()
    log("building model %s on %s" % (args.workload, dev))
    step_fn = pkg.trainer.TrainStep(cfg, vocab, device=dev, dp=dp, seed=0)
    log("model built; generating the synthetic batch")
    # identical initial weights on every rank
    if dp.enabled:
        torch.distributed.broadcast(step_fn.optimizer.buf.flat, 0)
    waves, lens, txt = pkg.synthetic.make_batch(vocab, per_gpu, args.n_samples, seed=1000 + rank)
    gb = per_gpu * world
    ntok = None
    if dp.enabled:
        ntok = dp.all_reduce_scalar(float((txt != 0).sum()), dev)
        # pad targets to the global max length so every rank decodes the same number of steps
        t = torch.tensor([txt.shape[1]], device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        if int(t) > txt.shape[1]:
            txt = torch.nn.functional.pad(txt, (0, int(t) - txt.shape[1]))
    waves_pin, txt_pin = waves.pin_memory(), txt.pin_memory()
    wave_dev = waves.to(dev)
    txt_dev = txt.to(dev)
    lens_dev = lens.to(dev)
    loss_pin = torch.zeros(1).pin_memory()
    gbatch = gb if dp.enabled else None

    def step_resident():
        return step_fn(wave_dev, lens_dev, txt_dev, global_batch=gbatch, global_tokens=ntok)

    def step_e2e():
        wave_dev.copy_(waves_pin, non_blocking=True)
        txt_dev.copy_(txt_pin, non_blocking=True)
        loss = step_fn(wave_dev, lens_dev, txt_dev, global_batch=gbatch, global_tokens=ntok)
        loss_pin.copy_(loss.reshape(1), non_blocking=True)
        return loss

    def timed(fn, steps, profile=False):
        dp.barrier()
        torch.cuda.synchronize()
        pkg.lib.TIMER.reset()
        pkg.lib.TIMER.enabled = profile
        pkg.lib.launch_count_reset()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            loss = fn()
        b.record()
        torch.cuda.synchronize()
        dp.barrier()
        pkg.lib.TIMER.enabled = False
        ms = dp.max_time(a.elapsed_time(b), dev)
        return ms, float(loss), pkg.lib.launch_count()

    log("warm-up")
    for i in range(max(args.warmup, 3)):
        step_resident()
        torch.cuda.synchronize()
        log("warm-up step %d done" % i)
    # (1) eager pass with per-kernel CUDA events -> kernel table / roofline
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    eager_ms, loss, launches = timed(step_resident, args.steps, profile=True)
    dump = step_outputs(step_fn, loss) if args.dump_outputs else None
    summary = pkg.lib.TIMER.summary()
    launches_per_step = launches / args.steps
    log("eager timed region done: %.1f ms/step" % (eager_ms / args.steps))
    # (2) whole-step CUDA graph (fixed shapes) -> the reported value / e2e
    use_graph = False
    # multi-GPU runs stay eager: the captured graph would contain the NCCL all-reduce, whose teardown at process exit
    # was seen to hang (the eager data-parallel path is the validated one; the graph is worth ~1 % on cfg B)
    if not args.no_graph and (world == 1 or args.graph_dp):
        use_graph = step_fn.capture(wave_dev, lens_dev, txt_dev, global_batch=gbatch, global_tokens=ntok)
        if world > 1:      # every rank replays the graph or none does (the collectives inside must pair up)
            ok = torch.tensor([1.0 if use_graph else 0.0], device=dev)
            torch.distributed.all_reduce(ok, op=torch.distributed.ReduceOp.MIN)
            if use_graph and float(ok) == 0.0:
                step_fn.release_graph()
                use_graph = False
                step_fn.graph_error = "capture failed on another rank"
        log("CUDA graph capture: %s" % ("ok" if use_graph else "not used (%s)" % step_fn.graph_error))
    if use_graph:
        for _ in range(3):
            step_resident()
        ms, loss, _ = timed(step_resident, args.steps)
        dump = step_outputs(step_fn, loss) if args.dump_outputs else None
    else:
        ms = eager_ms
    clocks = sampler.stop() if rank == 0 else None
    if dump is not None and rank == 0:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        log("outputs of the last timed step written to %s" % args.dump_outputs)
    log("timed region done: %.1f ms/step" % (ms / args.steps))
    value = gb * args.steps / (ms / 1000.0)
    e2e = None
    if not args.no_e2e:
        log("e2e (pinned host -> device each step)")
        step_e2e()
        ems, _, _ = timed(step_e2e, args.steps)
        log("e2e done: %.1f ms/step" % (ems / args.steps))
        e2e = {"value": gb * args.steps / (ems / 1000.0), "unit": UNIT,
               "h2d_bytes_per_step": int(waves_pin.numel() * 4 + txt_pin.numel() * 8) * world,
               "d2h_bytes_per_step": 4 * world, "ms_per_step": ems / args.steps}

    # ---- BASELINE configs[3] (CNN + BiLSTM 5x640, global batch 32 x N) measured in the same multi-GPU launch ----
    also = None
    if world > 1 and args.workload == "cfgB" and not args.batch and not args.no_also:
        log("also: cfgD (BASELINE configs[3]), 32 utterances per GPU")
        cfg_d = pkg.synthetic.load_config("cfgD")
        vocab_d = cfg_d["data"]["corpus"]["vocab_size"]
        bs_d = cfg_d["data"]["corpus"]["batch_size"]
        st = pkg.trainer.TrainStep(cfg_d, vocab_d, device=dev, dp=dp, seed=0)
        torch.distributed.broadcast(st.optimizer.buf.flat, 0)
        wv, ln, tx = pkg.synthetic.make_batch(vocab_d, bs_d, args.n_samples, seed=2000 + rank)
        nt = dp.all_reduce_scalar(float((tx != 0).sum()), dev)
        tmx = torch.tensor([tx.shape[1]], device=dev)
        torch.distributed.all_reduce(tmx, op=torch.distributed.ReduceOp.MAX)
        if int(tmx) > tx.shape[1]:
            tx = torch.nn.functional.pad(tx, (0, int(tmx) - tx.shape[1]))
        wv, ln, tx = wv.to(dev), ln.to(dev), tx.to(dev)
        fn_d = lambda: st(wv, ln, tx, global_batch=bs_d * world, global_tokens=nt)
        for _ in range(3):
            fn_d()
        nd = max(3, min(args.steps, 10))
        ms_d, loss_d, _ = timed(fn_d, nd)
        also = {"cfgD": {"workload": "cfgD: " + pkg.synthetic.WORKLOADS["cfgD"], "value": bs_d * world * nd / (ms_d / 1e3),
                         "unit": UNIT, "ms_per_step": ms_d / nd, "global_batch": bs_d * world, "steps": nd,
                         "loss": loss_d}}
        del st
        torch.cuda.empty_cache()
    if world > 1:
        step_fn.release_graph()          # the graph holds this communicator's NCCL kernels: drop it first
    dp.close()
    if rank != 0:
        return 0
    # ---- same-run parity at the benchmark's full size (CTC-loss rel-err is half of BASELINE.json's metric) ----
    parity = None
    if not args.no_parity:
        names = [args.workload]
        if args.parity_workloads == "auto":
            if world == 1 and not args.batch and args.n_samples == 192000:
                names += [w for w in ("cfgB", "cfgC", "cfgD") if w != args.workload]
        else:
            names = [w for w in args.parity_workloads.split(",") if w]
        parity = {}
        for w in names:
            log("parity check %s (full batch through the kernels vs the CPU path on 8 utterances)" % w)
            if w == args.workload:
                parity[w] = parity_check(pkg, step_fn, cfg, waves, lens, txt, dev, fp64=not args.no_parity_fp64,
                                         diagnose=args.parity_diagnose)
            else:
                cfg_w = pkg.synthetic.load_config(w)
                vocab_w = cfg_w["data"]["corpus"]["vocab_size"]
                st = pkg.trainer.TrainStep(cfg_w, vocab_w, device=dev, dp=dp, seed=0)
                wv, ln, tx = pkg.synthetic.make_batch(vocab_w, cfg_w["data"]["corpus"]["batch_size"], args.n_samples,
                                                      seed=1000)
                parity[w] = parity_check(pkg, st, cfg_w, wv, ln, tx, dev)
                del st
                torch.cuda.empty_cache()
            log("parity %s: %s" % (w, json.dumps(parity[w])))
    peak, peak_src = peaks()
    micro = None
    if world == 1 and not args.no_micro:
        log("micro-benchmark (BASELINE configs[4]: fbank + CTC on 1000 utterances of 2-30 s)")
        try:
            del step_fn
        except NameError:
            pass
        torch.cuda.empty_cache()
        micro = micro_bench(pkg, dev, peak)
    kernels = {}
    top, top_ms = None, -1.0
    for name, d in summary.items():
        per_launch_ms = d["ms"] / d["launches"]
        gbs = (d["bytes"] / d["launches"]) / (per_launch_ms * 1e-3) / 1e9 if per_launch_ms > 0 else 0.0
        kernels[name] = {"ms_per_step": d["ms"] / args.steps, "launches_per_step": d["launches"] / args.steps,
                         "algorithmic_gbs": gbs, "frac_hbm": gbs / peak}
        if d["ms"] > top_ms:
            top, top_ms = name, d["ms"]
    own_ms = sum(d["ms"] for d in summary.values()) / args.steps
    roofline = None
    if top is not None:
        k = kernels[top]
        d = summary[top]
        # DRAM traffic per launch = (dram bytes / algorithmic bytes) measured with `ncu --set full` on the SHIPPED kernels
        # (profiles/r02_ncu_traffic.json, written from this round's captures by tools/ncu_summary.py) x this launch's
        # algorithmic bytes; null when no capture of that kernel is committed
        ratios = {}
        try:
            with open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")) as f:
                ratios = json.load(f)
        except Exception:
            pass
        ratio = (ratios.get(top) or {}).get("dram_over_algorithmic")
        alg_per_launch = d["bytes"] / d["launches"]
        roofline = {"kernel": top, "bound": "hbm", "achieved": k["algorithmic_gbs"], "peak": peak, "unit": "GB/s",
                    "frac": k["frac_hbm"], "traffic": (ratio * alg_per_launch) if ratio else None,
                    "algorithmic_bytes_per_launch": alg_per_launch, "peak_source": peak_src,
                    "traffic_source": (ratios.get(top) or {}).get("source"),
                    "note": "The LSTM step kernels are bound by the per-step latency chain (gpu-scope fence -> flag -> "
                            "poll -> bulk copy -> tcgen05 MMAs -> TMEM load -> pointwise), not by HBM (SURVEY.md 7, "
                            "AI ~ 170 FLOP/B): see binding_bound"}
        if top.startswith("bilstm"):
            H = cfg["model"]["encoder"]["dim"][0]
            nbytes_per_step_dir = 24 * per_gpu * H
            steps_dirs = d["bytes"] / ((2 if top.endswith("bwd") else 1) * nbytes_per_step_dir)
            flops = steps_dirs * 2.0 * per_gpu * H * 4 * H
            tf = flops / (d["ms"] * 1e-3) / 1e12
            us_step = 1e3 * d["ms"] / (steps_dirs / 2.0)
            if lib.b200asr_bilstm_uses_tcgen05(per_gpu, H, 2) == 1:
                # tensor floor of one step: H/16 MMAs (M 64, N 128) x 64 cycles, measured by tools/micro/umma_probe.cu
                # (2192 cycles for 32 MMAs incl. completion latency) at the SM clock of this run
                mhz = (clocks or {}).get("sm_mhz") or 1965.0
                floor_us = (H / 16.0) * 68.5 / mhz
                roofline["binding_bound"] = {"bound": "tcgen05 step latency chain", "us_per_recurrent_step": us_step,
                                             "tensor_floor_us_per_step": floor_us, "frac": floor_us / us_step,
                                             "achieved": tf, "unit": "TFLOP/s (fp32-equivalent recurrent flops)"}
            else:
                on_tc = lib.b200asr_bilstm_uses_tensor_cores(per_gpu, H, 2) == 1
                pk = 92.7 if on_tc else 58.0
                roofline["binding_bound"] = {"bound": "mma_sync_3xtf32" if on_tc else "fp32_fma", "achieved": tf,
                                             "peak": pk, "unit": "TFLOP/s (fp32-equivalent)", "frac": tf / pk,
                                             "us_per_recurrent_step": us_step}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "loss": loss, "gpu_launches": int(round(launches_per_step * args.steps)), "clocks": clocks, "e2e": e2e,
            "roofline": roofline, "kernels": kernels, "cuda_graph": bool(use_graph),
            "eager_ms_per_step": eager_ms / args.steps, "own_kernel_ms_per_step": own_ms,
            "library_ms_per_step": eager_ms / args.steps - own_ms, "parity": parity, "also": also, "micro": micro,
            "note": "kernels/roofline come from the eager pass (CUDA events around each C-ABI launch); value and "
                    "e2e replay the same step as one CUDA graph when cuda_graph is true; gpu_launches counts this "
                    "library's kernels per step x steps"}
    if world == 1 and not args.no_cpu_baseline:
        cb = args.cpu_batch or 8
        log("cpu baseline (%d utterances/step)" % cb)
        r = cpu_arm(cfg, vocab, args.n_samples, cb, 2, 1)
        log("cpu baseline done")
        line["cpu_baseline"] = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                                "sample": "1 warm-up + 2 timed steps of %d utterances of the same workload "
                                          "(reference CPU path: kaldi.fbank per utterance + ATen LSTM/CTC + "
                                          "clip + Adadelta, oracle/ref_port.py); thread count calibrated (best of 8/16/32/"
                                          "64/all cores)" % cb,
                                "ms_per_step": r["ms_per_step"]}
    print(json.dumps(line))
    sys.stdout.flush()
    return 0


if __name__ == "__main__":
    sys.exit(main())
