#!/usr/bin/env python
# coding: utf-8
"""Same command line as the reference's main.py (/root/reference/main.py:13-47), driving the B200-native Solver.
    python main.py --config config/b200/cfgB_ctc_char.yaml [--njobs 0] [--seed 0] [--load ckpt]
    torchrun --nproc-per-node 8 --master-addr 127.0.0.1 main.py --config ...      (data parallel, one process per GPU)
--test runs greedy decoding (decode.beam_size 1); --lm trains the RNN language model (config/b200/lm_example.yaml,
one GPU) and takes precedence over --test as in the reference; --cpu hands the whole command line to the reference
checkout (B200ASR_REFERENCE, default /root/reference) - this package has no CPU path."""
import argparse
import importlib
import os
import sys

import numpy as np
import torch
import yaml

parser = argparse.ArgumentParser(description="Training E2E asr (B200-native hot path).")
parser.add_argument("--config", type=str, help="Path to experiment config.")
parser.add_argument("--name", default=None, type=str, help="Name for logging.")
parser.add_argument("--logdir", default="log/", type=str, help="Logging path.")
parser.add_argument("--ckpdir", default="ckpt/", type=str, help="Checkpoint path.")
parser.add_argument("--outdir", default="result/", type=str, help="Decode output path.")
parser.add_argument("--load", default=None, type=str, help="Load pre-trained model (for training only)")
parser.add_argument("--seed", default=0, type=int, help="Random seed for reproducable results.")
parser.add_argument("--cudnn-ctc", action="store_true", help="(reference flag) unsupported: the CTC kernel is ours")
parser.add_argument("--njobs", default=6, type=int, help="Number of DataLoader worker processes.")
parser.add_argument("--cpu", action="store_true", help="(reference flag) use the reference itself for CPU runs")
parser.add_argument("--no-pin", action="store_true", help="Disable pin-memory for dataloader")
parser.add_argument("--test", action="store_true", help="Test the model (greedy decoding, decode.beam_size: 1).")
parser.add_argument("--no-msg", action="store_true", help="Hide all messages.")
parser.add_argument("--lm", action="store_true", help="Train the RNN language model (single GPU).")
parser.add_argument("--amp", action="store_true", help="(reference flag) unsupported")
parser.add_argument("--reserve-gpu", default=0, type=float)
parser.add_argument("--jit", action="store_true")


def main():
    paras = parser.parse_args()
    setattr(paras, "gpu", not paras.cpu)
    setattr(paras, "pin_memory", not paras.no_pin)
    setattr(paras, "verbose", not paras.no_msg)
    if paras.cpu:
        # SURVEY.md 8(b): `--cpu` keeps routing to the REFERENCE implementation (the baseline run, main.py:30,45 there).
        # It is not part of this repository: point B200ASR_REFERENCE at a checkout (default /root/reference).
        ref = os.environ.get("B200ASR_REFERENCE", "/root/reference")
        if not os.path.isfile(os.path.join(ref, "main.py")):
            raise SystemExit("--cpu runs the reference's own CPU path, but no reference checkout was found at %s "
                             "(set B200ASR_REFERENCE); this package has no CPU fallback" % ref)
        import runpy
        sys.path.insert(0, ref)
        os.chdir(ref)
        sys.argv[0] = os.path.join(ref, "main.py")
        return runpy.run_path(sys.argv[0], run_name="__main__")
    if paras.cudnn_ctc:
        raise SystemExit("--cudnn-ctc selects a reference path outside the B200 hot path")
    config = yaml.load(open(paras.config, "r"), Loader=yaml.FullLoader)
    np.random.seed(paras.seed)
    torch.manual_seed(paras.seed)
    torch.cuda.manual_seed_all(paras.seed)
    pkg = importlib.import_module("end-to-end-asr-pytorch_b200")
    if paras.lm:
        solver = pkg.train_lm.Solver(config, paras, "train")
    elif paras.test:        # greedy decoding (decode.beam_size: 1); beam search stays the reference's CPU path
        assert paras.load is None, "Load option is mutually exclusive to --test"
        solver = pkg.test_asr.Solver(config, paras, "test")
    else:
        solver = pkg.train_asr.Solver(config, paras, "train")
    solver.load_data()
    solver.set_model()
    solver.exec()


if __name__ == "__main__":
    main()
