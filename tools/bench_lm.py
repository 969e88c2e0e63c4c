"""RNN-LM train step: this package against a torch-native fp32 step, alternated in one process on the same batches.

    python tools/bench_lm.py [--seconds 4] [--rounds 6] [--parity-steps 5] [--out lm_bench.json]
    python tools/bench_lm.py --profile DIR          # one torch.profiler kernel table per arm (separate run)

Sizes are config/b200/lm_example.yaml's (B = 32, V = 16000, emb = dim = 1024, 2 LSTM layers, dropout 0.5, Adam 1e-4).
Batches: data.SyntheticTextDataset buckets, lengths U[20, 60] tokens including <eos> (mean 40), ids in [2, V) - the
same 8 seeded buckets, cycled, for both arms.
  (a) package   lm.RNNLM + ops.cross_entropy + optim.Optimizer (grad-norm, clip 5, Adam fused on flat buffers)
  (b) torch     nn.Embedding, cuDNN nn.LSTM on packed input, nn.Linear, CrossEntropyLoss(ignore_index=0),
                clip_grad_norm_(5), torch.optim.Adam; TF32 off (fp32 like the reference)
Each round times one arm for --seconds with CUDA events around the whole window, then the other arm; ms/step is the
median over rounds.  Target tokens/s counts the non-ignored targets (the <eos>-terminated rows' lengths).
Parity: both arms from identical weights with dropout 0 for --parity-steps steps on the same batches.
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pkg = importlib.import_module("end-to-end-asr-pytorch_b200")

B, V, E, H, LAYERS, DROPOUT, LR, EPS = 32, 16000, 1024, 1024, 2, 0.5, 1e-4, 1e-8
MIN_LEN, MAX_LEN, N_BATCHES = 20, 60, 8


class TorchLM(nn.Module):
    """The reference model's computation in plain torch modules (same parameter names)."""

    def __init__(self, dropout):
        super().__init__()
        self.emb = nn.Embedding(V, E)
        self.dp1 = nn.Dropout(dropout)
        self.dp2 = nn.Dropout(dropout)
        self.rnn = nn.LSTM(E, H, num_layers=LAYERS, dropout=dropout, batch_first=True)
        self.trans = nn.Linear(H, V)

    def forward(self, x, lens):
        packed = nn.utils.rnn.pack_padded_sequence(self.dp1(self.emb(x)), lens, batch_first=True, enforce_sorted=False)
        out, _ = self.rnn(packed)
        out, _ = nn.utils.rnn.pad_packed_sequence(out, batch_first=True)
        return self.trans(self.dp2(out))


def batches():
    ds = pkg.data.SyntheticTextDataset(V, B, N_BATCHES, seed=0, min_len=MIN_LEN, max_len=MAX_LEN)
    out = []
    for i in range(N_BATCHES):
        data = pkg.data.collect_text_batch([ds[i]], mode="train")
        txt = torch.cat((torch.zeros((B, 1), dtype=torch.long), data), dim=1).cuda()
        out.append((txt, (data != 0).sum(-1)))
    return out


def make_arms(dropout, seed=0):
    torch.manual_seed(seed)
    mine = pkg.lm.RNNLM(V, False, E, "LSTM", H, LAYERS, dropout).cuda()
    ref = TorchLM(dropout).cuda()
    ref.load_state_dict(mine.state_dict())
    opt = pkg.optim.Optimizer(mine.parameters(), "Adam", LR, EPS, "fixed")
    opt.grad_clip = 5.0
    ref_opt = torch.optim.Adam(ref.parameters(), lr=LR, eps=EPS)
    ce = nn.CrossEntropyLoss(ignore_index=0)

    def step_pkg(batch, step):
        txt, lens = batch
        opt.pre_step(step)
        pred, _ = mine(txt[:, :-1], lens)
        loss = pkg.ops.cross_entropy(pred.view(-1, V), txt[:, 1:].reshape(-1), ignore_index=0)
        loss.backward()
        opt.step()
        return loss

    def step_torch(batch, step):
        txt, lens = batch
        ref_opt.zero_grad(set_to_none=False)
        pred = ref(txt[:, :-1], lens)
        loss = ce(pred.reshape(-1, V), txt[:, 1:].reshape(-1))
        loss.backward()
        torch.nn.utils.clip_grad_norm_(ref.parameters(), 5.0)
        ref_opt.step()
        return loss

    return step_pkg, step_torch


def timed_window(step, data, seconds, start):
    """Steps until `seconds` of device time have passed; returns (steps, ms, target tokens)."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n, toks, ms = 0, 0, 0.0
    a.record()
    while True:
        for _ in range(4):
            batch = data[(start + n) % len(data)]
            step(batch, start + n)
            toks += int(batch[1].sum())
            n += 1
        b.record()
        b.synchronize()
        ms = a.elapsed_time(b)
        if ms >= 1000 * seconds:
            return n, ms, toks


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:          # the card name alone is still worth reporting
        q = "unavailable (%s)" % e
    return name, q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=4.0)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--parity-steps", type=int, default=5)
    ap.add_argument("--profile", default=None)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_lm.py measures on a CUDA device; there is no CPU mode"
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    data = batches()
    name, power = card()
    lib = pkg.lib.load()

    # parity: identical weights, dropout 0, the same batches
    p_pkg, p_torch = make_arms(0.0, seed=1)
    la = [p_pkg(data[i % len(data)], i).item() for i in range(args.parity_steps)]
    lb = [p_torch(data[i % len(data)], i).item() for i in range(args.parity_steps)]
    del p_pkg, p_torch
    torch.cuda.empty_cache()

    step_pkg, step_torch = make_arms(DROPOUT)
    arms = {"package": step_pkg, "torch": step_torch}
    for arm in arms.values():
        for i in range(args.warmup):
            arm(data[i % len(data)], i)
    torch.cuda.synchronize()

    if args.profile:
        os.makedirs(args.profile, exist_ok=True)
        from torch.profiler import ProfilerActivity, profile
        for label, arm in arms.items():
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for i in range(8):
                    arm(data[i % len(data)], i)
                torch.cuda.synchronize()
            with open(os.path.join(args.profile, "lm_profile_%s.txt" % label), "w") as f:
                f.write("%s, %s; 8 steps of the %s arm\n" % (name, power, label))
                f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=25, max_name_column_width=90))
        print(json.dumps({"profile": args.profile, "gpu": name, "power_limit_max_sm_clock": power}))
        return

    per = {k: [] for k in arms}
    tok = {k: [] for k in arms}
    start = args.warmup
    for r in range(args.rounds):
        for label in (("package", "torch") if r % 2 == 0 else ("torch", "package")):
            n, ms, toks = timed_window(arms[label], data, args.seconds, start)
            start += n
            per[label].append(ms / n)
            tok[label].append(toks / (ms / 1000.0))
    rec = {
        "workload": "RNN-LM train step, lm_example.yaml sizes",
        "B": B, "V": V, "emb_dim": E, "dim": H, "n_layers": LAYERS, "dropout": DROPOUT,
        "lengths": "U[%d, %d] tokens incl. <eos> (8 seeded buckets, cycled)" % (MIN_LEN, MAX_LEN),
        "gpu": name, "power_limit_max_sm_clock": power,
        "recurrence_tcgen05": int(lib.b200asr_bilstm_uses_tcgen05(B, H, 1)),
        "rounds": args.rounds, "seconds_per_window": args.seconds,
        "package_ms_per_step": statistics.median(per["package"]),
        "torch_ms_per_step": statistics.median(per["torch"]),
        "package_ms_per_step_rounds": [round(v, 3) for v in per["package"]],
        "torch_ms_per_step_rounds": [round(v, 3) for v in per["torch"]],
        "package_target_tokens_per_s": statistics.median(tok["package"]),
        "torch_target_tokens_per_s": statistics.median(tok["torch"]),
        "parity_steps": args.parity_steps,
        "parity_loss_package": la, "parity_loss_torch": lb,
        "parity_max_rel_loss_diff": max(abs(x - y) / abs(y) for x, y in zip(la, lb)),
    }
    rec["speedup_vs_torch"] = rec["torch_ms_per_step"] / rec["package_ms_per_step"]
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
