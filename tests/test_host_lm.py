"""RNN-LM host side: text datasets and batches, the synthetic text corpus, main.py's --lm routing, and the contract
between the package's RNNLM constructor and the reference's (the seeded initial weights in tests/golden/lm_*.npz)."""
import importlib
import os
import sys

import numpy as np
import pytest
import torch
import yaml
from torch.utils.data import RandomSampler, SequentialSampler

from conftest import load_golden
from oracle.make_golden_lm import LM_KINDS, LM_PLUMBING_DEV, LM_PLUMBING_TRAIN, lm_batch, lm_plumbing_config, \
    lm_plumbing_tree

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _char_tokenizer(pkg):
    return pkg.text.load_text_encoder("character", os.path.join(ROOT, "tests", "golden", "character.vocab"))


def test_libri_text_dataset_sorts_and_buckets(pkg, tmp_path):
    path = lm_plumbing_tree(str(tmp_path))
    tok = _char_tokenizer(pkg)
    ds = pkg.corpus.LibriTextDataset(path, ["train-clean-100"], tok, 1)
    lines = [s for v in LM_PLUMBING_TRAIN.values() for s in v]
    assert len(ds) == len(lines)
    want = sorted((tok.encode(s) for s in lines), key=len, reverse=True)
    assert [ds[i] for i in range(len(ds))] == want
    assert all(t[-1] == 1 for t in want)
    b = pkg.corpus.LibriTextDataset(path, ["train-clean-100"], tok, 3)
    assert b[0] == want[0:3]
    assert b[len(b) - 1] == want[-3:]                       # a bucket never runs past the end
    dv = pkg.corpus.LibriTextDataset(path, ["dev-clean"], tok, 1)
    assert len(dv) == len(LM_PLUMBING_DEV[("84", "121")])


def test_official_text_split_is_emptied_by_remove_top_n(pkg, tmp_path):
    path = lm_plumbing_tree(str(tmp_path))
    with open(os.path.join(path, "librispeech-lm-norm.txt"), "w") as f:
        f.write("A SHORT LINE\nANOTHER LINE\n")
    tok = _char_tokenizer(pkg)
    ds = pkg.corpus.LibriTextDataset(path, ["librispeech-lm-norm.txt", "dev-clean"], tok, 1)
    assert pkg.corpus.REMOVE_TOP_N_TXT == 5000000 and len(ds) == 0


def test_collect_text_batch_pads_and_halves(pkg):
    short = [[5, 6, 1], [7, 1]]
    t = pkg.data.collect_text_batch([short], mode="train")
    assert t.tolist() == [[5, 6, 1], [7, 1, 0]]
    long_ = [[3] * 151 + [1], [4] * 10 + [1], [5, 1], [6, 1]]
    assert pkg.data.collect_text_batch([long_], mode="train").shape == (2, 152)
    assert pkg.data.collect_text_batch([long_], mode="dev").shape == (4, 152)
    edge = [[3] * 149 + [1], [4, 1]]                         # exactly 150 tokens: not halved
    assert pkg.data.collect_text_batch([edge], mode="train").shape == (2, 150)
    assert pkg.data.collect_text_batch(short, mode="dev").shape == (2, 3)   # unbucketed list of sequences


def test_synthetic_text_set_is_seeded(pkg):
    a = pkg.data.SyntheticTextDataset(100, 8, 4, seed=3, min_len=5, max_len=9)
    b = pkg.data.SyntheticTextDataset(100, 8, 4, seed=3, min_len=5, max_len=9)
    assert len(a) == 4
    for i in range(4):
        assert a[i] == b[i]
        lens = [len(s) for s in a[i]]
        assert lens == sorted(lens, reverse=True) and min(lens) >= 5 and max(lens) <= 9
        for s in a[i]:
            assert s[-1] == 1 and all(2 <= v < 100 for v in s[:-1])
    assert a[0] != a[1]


def test_load_textset_loaders_match_reference(pkg, tmp_path):
    path = lm_plumbing_tree(str(tmp_path))
    cfg = yaml.safe_load(open(os.path.join(ROOT, "config", "b200", "lm_example.yaml")))
    cfg = lm_plumbing_config(cfg, path)
    tr, dv, V, tok, msg = pkg.data.load_textset(0, False, False, **cfg["data"])
    assert V == 31 and tok.token_type == "character"
    assert isinstance(tr.sampler, RandomSampler) and tr.drop_last and tr.batch_size == 1
    assert isinstance(dv.sampler, SequentialSampler) and not dv.drop_last and dv.batch_size == 2
    syn = yaml.safe_load(open(os.path.join(ROOT, "config", "b200", "lm_synthetic.yaml")))
    tr, dv, V, tok, msg = pkg.data.load_textset(0, False, False, **syn["data"])
    batch = next(iter(tr))
    assert V == 1000 and batch.shape[0] == 32 and batch.dtype == torch.int64


@pytest.mark.parametrize("kind", sorted(LM_KINDS))
def test_rnnlm_init_and_keys_match_reference(pkg, kind):
    g = load_golden("lm_model_%s.npz" % kind)
    seed, cfg = LM_KINDS[kind]
    assert int(g["seed"]) == seed
    torch.manual_seed(seed)
    sd = pkg.lm.RNNLM(int(g["vocab"]), **cfg).state_dict()
    ref = {k[3:]: v for k, v in g.items() if k.startswith("sd.")}
    assert list(sd) == list(ref)
    for k, v in sd.items():
        assert np.array_equal(v.numpy(), ref[k]), k
    txt, lens = lm_batch(seed + 1, [int(n) for n in g["lens"]], int(g["vocab"]))
    assert np.array_equal(txt.numpy(), g["txt"])


def test_rnnlm_refuses_initial_state(pkg):
    m = pkg.lm.RNNLM(31, False, 16, "LSTM", 16, 1, 0.0)
    with pytest.raises(NotImplementedError, match="beam search"):
        m(torch.zeros(1, 2, dtype=torch.long), torch.tensor([2]), hidden=(torch.zeros(1, 1, 16),) * 2)


class _FakeSolver:
    made = []

    def __init__(self, config, paras, mode):
        _FakeSolver.made.append((self.kind, mode))

    def load_data(self):
        pass

    def set_model(self):
        pass

    def exec(self):
        pass


def _run_main(monkeypatch, pkg, argv):
    main = importlib.import_module("main")
    for mod, kind in ((pkg.train_lm, "lm"), (pkg.train_asr, "asr"), (pkg.test_asr, "test")):
        monkeypatch.setattr(mod, "Solver", type("S_" + kind, (_FakeSolver,), {"kind": kind}))
    monkeypatch.setattr(sys, "argv", ["main.py"] + argv)
    _FakeSolver.made = []
    main.main()
    return _FakeSolver.made


def test_main_routes_lm_before_test(monkeypatch, pkg):
    cfg = os.path.join(ROOT, "config", "b200", "lm_synthetic.yaml")
    assert _run_main(monkeypatch, pkg, ["--config", cfg, "--lm"]) == [("lm", "train")]
    assert _run_main(monkeypatch, pkg, ["--config", cfg, "--lm", "--test"]) == [("lm", "train")]
    assert _run_main(monkeypatch, pkg, ["--config", cfg, "--test"]) == [("test", "test")]
    with pytest.raises(SystemExit, match="cudnn-ctc"):
        _run_main(monkeypatch, pkg, ["--config", cfg, "--lm", "--cudnn-ctc"])


def test_lm_solver_refuses_data_parallel(monkeypatch, pkg, tmp_path):
    import argparse
    monkeypatch.setenv("WORLD_SIZE", "2")
    cfg = yaml.safe_load(open(os.path.join(ROOT, "config", "b200", "lm_synthetic.yaml")))
    paras = argparse.Namespace(config="lm_synthetic.yaml", name=None, seed=0, gpu=True, verbose=False,
                               ckpdir=str(tmp_path), logdir=str(tmp_path))
    with pytest.raises(NotImplementedError, match="data-parallel"):
        pkg.train_lm.Solver(cfg, paras, "train")
