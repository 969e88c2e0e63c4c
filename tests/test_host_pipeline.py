"""CPU-only tests of the host-side mirror: text codecs (the reference's own known-answer ids), batching rules,
optimizer wrapper schedule logic, and the data-parallel rules with a world_size-2 gloo group."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from conftest import GOLDEN, ROOT, golden_params, load_golden


def test_character_encoder_known_answers(pkg):
    """/root/reference/tests/test_text.py:26-27: 'SPEECH LAB!' -> [22,19,8,8,6,11,3,15,4,5,2,1], vocab 31."""
    enc = pkg.text.load_text_encoder("character", os.path.join(GOLDEN, "character.vocab"))
    assert enc.vocab_size == 31 and enc.token_type == "character"
    ids = enc.encode("SPEECH LAB!")
    assert ids == [22, 19, 8, 8, 6, 11, 3, 15, 4, 5, 2, 1]
    assert enc.decode(ids) == "SPEECH LAB<unk>"
    assert enc.decode([22, 22, 0, 19, 19, 1, 8], ignore_repeat=True) == "SP"      # CTC collapse, stop at <eos>
    assert (enc.pad_idx, enc.eos_idx, enc.unk_idx) == (0, 1, 2)


def test_collate_sorts_pads_and_halves(pkg):
    fe = pkg.audio.FbankFrontEnd(feat_dim=40)
    g = torch.Generator().manual_seed(0)
    items = [(torch.randn(n, generator=g), [3, 4, 1][:k]) for n, k in [(8000, 2), (16000, 3), (12000, 1), (4000, 3)]]
    names, wave, wl, txt = pkg.data.collect_wave_batch(items, fe.num_frames, "train")
    assert wl.tolist() == [16000, 12000, 8000, 4000] and wave.shape == (4, 16000)      # longest first, zero padded
    assert float(wave[3, 4000:].abs().max()) == 0 and txt.shape == (4, 3) and txt[1].tolist() == [3, 0, 0]
    # first utterance longer than 800 frames (~8 s): the training batch is halved (src/data.py:9,23-24)
    long_items = [(torch.randn(140000, generator=g), [3, 1])] + items
    _, wave2, wl2, _ = pkg.data.collect_wave_batch(long_items, fe.num_frames, "train")
    assert wave2.shape[0] == 2
    _, wave3, _, _ = pkg.data.collect_wave_batch(long_items, fe.num_frames, "test")
    assert wave3.shape[0] == 5


def test_synthetic_workload_shapes(pkg):
    cfg = pkg.synthetic.load_config("cfgB")
    assert cfg["model"]["ctc_weight"] == 1.0 and cfg["model"]["encoder"]["sample_rate"] == [1, 2, 2, 1]
    w, l, t = pkg.synthetic.make_batch(31, 4, 32000, seed=3)
    assert w.shape == (4, 32000) and l.tolist() == [32000] * 4 and float(w.abs().max()) <= 1.0
    lens = (t != 0).sum(1)
    assert int(t.max()) < 31 and all(int(t[b, lens[b] - 1]) == 1 for b in range(4))      # <eos> terminated
    w2, _, t2 = pkg.synthetic.make_batch(31, 4, 32000, seed=3)
    assert torch.equal(w, w2) and torch.equal(t, t2)                                      # seeded
    model = pkg.ASR(120, 31, True, **cfg["model"])
    assert sum(p.numel() for p in model.parameters()) == 29916191                        # SURVEY.md 8(a) cfg B
    cfgc = pkg.synthetic.load_config("cfgC")
    assert sum(p.numel() for p in pkg.ASR(120, 5000, True, **cfgc["model"]).parameters()) == 52323879
    cfgd = pkg.synthetic.load_config("cfgD")
    assert sum(p.numel() for p in pkg.ASR(120, 5000, True, **cfgd["model"]).parameters()) == 72867879


def test_optimizer_schedules(pkg):
    sched = pkg.optim.speech_aug_scheduler
    assert sched(0, 500, 20000, 80000, 1.0) == pytest.approx(1 / 500)
    assert sched(1000, 500, 20000, 80000, 1.0) == 1.0
    assert sched(10 ** 6, 500, 20000, 80000, 1.0) == pytest.approx(0.01)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _dp_worker(rank, world, port, out):
    import importlib
    import sys
    sys.path.insert(0, ROOT)
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1",
                      MASTER_PORT=str(port))
    torch.set_num_threads(1)
    pkg = importlib.import_module("end-to-end-asr-pytorch_b200")
    from oracle import ref_port
    from oracle.make_golden import tiny_model_cfg
    dp = pkg.dist.DataParallel(backend="gloo")
    g = dict(np.load(os.path.join(GOLDEN, "model_hybrid.npz")))
    cfg = tiny_model_cfg("hybrid")
    P = {k: v.requires_grad_(True) for k, v in golden_params(g, "hybrid").items()}
    feat, flen, txt = torch.from_numpy(g["feat"]), torch.from_numpy(g["feat_len"]), torch.from_numpy(g["txt"])
    B = feat.shape[0]
    ntok = float((txt != 0).sum())
    # rank r takes rows r::world of the globally padded batch (SURVEY.md 8(e))
    f, l, t = dp.shard(feat, flen, txt)
    enc, enc_len = ref_port.encoder(P, cfg["encoder"], f, l)
    lp = torch.log_softmax(torch.nn.functional.linear(enc, P["ctc_layer.weight"], P["ctc_layer.bias"]), -1)
    tl = (t != 0).sum(-1)
    nll = torch.nn.functional.ctc_loss(lp.transpose(0, 1), t, enc_len, tl, blank=0, reduction="none")
    ctc = (nll / tl.clamp_min(1)).sum() / B                                   # global batch normalisation
    L = int((txt != 0).sum(-1).max())                                       # decode to the GLOBAL max length
    att, _ = ref_port.loc_attention_decode(P, cfg["attention"], cfg["decoder"], enc, enc_len, t, L)
    ce = torch.nn.functional.cross_entropy(att.reshape(-1, att.shape[-1]), t[:, :L].reshape(-1), ignore_index=0,
                                           reduction="sum") / ntok          # global token normalisation
    (0.3 * ctc + 0.7 * ce).backward()
    names = sorted(k for k in P if P[k].grad is not None)
    flat = torch.cat([P[k].grad.reshape(-1) for k in names])
    dp.all_reduce_(flat, n_buckets=3)                                         # SUM, not mean
    tmax = dp.max_time(10.0 * (rank + 1), "cpu")
    if rank == 0:
        ref = np.concatenate([g["grad." + k].reshape(-1) for k in names])
        out.put((float(np.abs(flat.numpy() - ref).max() / np.abs(ref).max()), tmax, dp.world))
    dp.barrier()
    torch.distributed.destroy_process_group()


def test_data_parallel_rules_match_single_process_gloo():
    """world_size 2 over gloo: sharded losses with global normalisation + SUM all-reduce of the flat gradient
    reproduce the single-process (reference) gradient of the full batch."""
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    err, tmax, world = out.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert world == 2 and tmax == 20.0
    assert err < 1e-4, err


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (CPU arm) prints one JSON line with the contract's keys; tiny sample here."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--cpu-batch", "1", "--n-samples", "16000"], capture_output=True, text=True,
                         timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "utt/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["e2e"]["value"] == line["value"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["cpu_baseline"]["kind"] == "port"
    assert line["config"]["workload"].startswith("cfgB")


def test_greedy_decode_rows_and_synthetic_decode_split(pkg):
    """Host side of the `--test` greedy path (bin/test_asr.py:199-217): csv rows, empty hypothesis -> one blank,
    the reference's un-collapsed CTC hypotheses by default, and the (dev, test) split of the synthetic corpus."""
    tok = pkg.data._VocabOnly(12)
    res = [("0", [[3, 3, 0, 4, 1, 7]], [3, 4, 1, 0]), ("1", [[1, 5]], [6, 1])]
    rows = pkg.test_asr.format_hyp_rows(tok, res)
    assert rows == ["0\t3 3 4\t3 4", "1\t \t6"]
    assert pkg.test_asr.format_hyp_rows(tok, res, collapse_repeats=True)[0] == "0\t3 4\t3 4"
    dv, tt, bs_a, bs_b, mode, msg = pkg.data.create_dataset(tok, False, name="Synthetic", path="", bucketing=False,
                                                            batch_size=3, dev_split=["a"], test_split=["b"],
                                                            n_samples=8000, vocab_size=12)
    assert mode == "test" and (bs_a, bs_b) == (1, 1) and len(dv) == 2 and len(tt) == 2
    assert any("Test sets" in m for m in msg)
    names, wave, wave_len, txt = pkg.data.collect_wave_batch([dv[0]], lambda n: 1 + (n - 400) // 160, "test")
    assert wave.shape[0] == 3 and txt.shape[0] == 3 and list(wave_len) == sorted(wave_len, reverse=True)


def test_greedy_decode_exec_with_stub_model(pkg, tmp_path):
    """exec()/greedy_decode() of the `--test` Solver on stand-ins for the front end and the model: utterance
    numbering across batches, arg-max feedback ids -> csv, CTC-only models read the kernel's arg-max ids."""
    import argparse
    S = pkg.test_asr.Solver
    tok = pkg.data._VocabOnly(8)

    class FrontEnd:
        def batch(self, wave, wave_len, t_max=None):
            return wave.unsqueeze(-1), torch.tensor([10, 8])

    class Model:
        def __init__(self, att):
            self.enable_att, self.last_ctc_argmax, self.steps = att, None, []

        def __call__(self, feat, feat_len, steps, emb_decoder=None):
            self.steps.append(steps)
            ids = torch.tensor([[3, 4, 1, 0, 0], [5, 5, 6, 1, 0]])
            if self.enable_att:
                return None, None, torch.nn.functional.one_hot(ids, 8).float(), None, None
            self.last_ctc_argmax = ids
            return torch.zeros(2, 5, 8), None, None, None, None

    def batch(seed):
        return (["a", "b"], torch.zeros(2, 16), torch.tensor([16, 12]), torch.tensor([[3, 4, 1], [5, 6, 1]]) + 0 * seed)

    for att, collapse, want in ((True, False, "5 5 6"), (False, False, "5 5 6"), (False, True, "5 6")):
        s = object.__new__(S)
        s.config = {"decode": {"beam_size": 1, "max_len_ratio": 0.5, "ctc_collapse": collapse},
                    "data": {"corpus": {"batch_size": 2}}}
        s.paras = argparse.Namespace(verbose=False)
        s.dp = argparse.Namespace(rank=0)
        s.device, s.step, s.emb_decoder, s.tokenizer = "cpu", 0, None, tok
        s.audio_transform, s.decoder = FrontEnd(), Model(att)
        s.dv_set, s.tt_set = [batch(0), batch(1)], [batch(2)]
        s.output_file = str(tmp_path / ("o%d%d" % (att, collapse))) + "_{}_{}.csv"
        s.exec()
        dev = open(s.output_file.format("dev", "output")).read().splitlines()
        assert dev == ["idx\thyp\ttruth", "0\t3 4\t3 4", "1\t%s\t5 6" % want, "2\t3 4\t3 4", "3\t%s\t5 6" % want]
        assert len(open(s.output_file.format("test", "output")).read().splitlines()) == 3
        assert s.decoder.steps == [5, 5, 5]            # int(max feature length 10 * max_len_ratio 0.5)
