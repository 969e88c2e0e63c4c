"""Data pipeline around the GPU front end (/root/reference/src/data.py:14-43,129-156).

The reference runs fbank+delta+CMVN on the CPU inside the DataLoader workers' collate_fn, one file at a time
(src/data.py:22,31).  Here the workers only LOAD waveforms (they must never touch CUDA); collate pads them into a
[B, N_max] batch sorted by length (descending, same order as the reference's sort by feature length) and the main
process runs the fused front-end kernels on the GPU (Solver.fetch_data).  The half-batch rule
(HALF_BATCHSIZE_AUDIO_LEN = 800 frames, src/data.py:9,23-24) is applied on the frame count implied by the sample
count."""
from functools import partial

import numpy as np
import torch
from torch.nn.utils.rnn import pad_sequence
from torch.utils.data import DataLoader, Dataset

from .audio import create_transform, load_wav
from .synthetic import make_batch
from .text import load_text_encoder

HALF_BATCHSIZE_AUDIO_LEN = 800
HALF_BATCHSIZE_TEXT_LEN = 150


def read_waveform(path):
    """[N] waveform of one file.  16-bit PCM wav files are returned AS int16 (half the pinned-host and H2D bytes; the
    fbank kernel converts sample / 32768 on the fly - bit-identical to the fp32 path); anything else as fp32 in
    [-1, 1] through soundfile (flac) / scipy."""
    if str(path).lower().endswith(".wav"):
        try:
            from scipy.io import wavfile
            _, data = wavfile.read(str(path))
            if data.dtype == np.int16:
                return torch.from_numpy(np.ascontiguousarray(data if data.ndim == 1 else data[:, 0]))
        except Exception:
            pass
    try:
        import soundfile as sf
        x, _ = sf.read(str(path), dtype="float32")
        return torch.from_numpy(x if x.ndim == 1 else x[:, 0].copy())
    except Exception:
        wave, _ = load_wav(str(path))
        return wave[0]


def collect_wave_batch(batch, num_frames, mode):
    """[(path, tokens), ...] -> (names, wave [B,N] fp32, wave_len [B] i64, txt [B,L] i64), longest first."""
    if type(batch[0]) is not tuple:
        batch = batch[0]                                   # bucketed: [[(file, txt), ...]]
    waves = [read_waveform(b[0]) if not torch.is_tensor(b[0]) else b[0] for b in batch]
    if any(w.dtype != torch.int16 for w in waves):         # mixed sources: everything as fp32 in [-1, 1]
        waves = [w.to(torch.float32) / 32768.0 if w.dtype == torch.int16 else w for w in waves]
    if num_frames(len(waves[0])) > HALF_BATCHSIZE_AUDIO_LEN and mode == "train":
        batch, waves = batch[:len(batch) // 2], waves[:len(batch) // 2]
    names = [str(b[0]).split("/")[-1].split(".")[0] if not torch.is_tensor(b[0]) else "syn%d" % i
             for i, b in enumerate(batch)]
    texts = [torch.LongTensor(b[1]) for b in batch]
    order = sorted(range(len(waves)), key=lambda i: num_frames(len(waves[i])), reverse=True)
    waves, names, texts = [waves[i] for i in order], [names[i] for i in order], [texts[i] for i in order]
    wave_len = torch.LongTensor([len(w) for w in waves])
    return names, pad_sequence(waves, batch_first=True), wave_len, pad_sequence(texts, batch_first=True)


class SyntheticDataset(Dataset):
    """Seeded LibriSpeech-shaped batches (SURVEY.md 8(d)); one item = one ready batch."""

    def __init__(self, vocab_size, batch_size, n_samples=192000, n_batches=64, seed=0, ragged=True):
        self.args = (vocab_size, batch_size, n_samples)
        self.n_batches, self.seed, self.ragged = n_batches, seed, ragged

    def __len__(self):
        return self.n_batches

    def __getitem__(self, i):
        waves, lens, txt = make_batch(*self.args, seed=self.seed + i, ragged=self.ragged)
        return [(waves[b, :int(lens[b])], [int(v) for v in txt[b] if int(v) != 0]) for b in range(waves.shape[0])]


def create_dataset(tokenizer, ascending, name, path, bucketing, batch_size, train_split=None, dev_split=None,
                   test_split=None, **extra):
    """Same roles as src/data.py:65-104: returns (tr_set, dv_set, tr_loader_bs, dv_loader_bs, mode, msg)."""
    if name.lower() == "synthetic":
        n = extra.get("n_samples", 192000)
        v = extra.get("vocab_size", tokenizer.vocab_size if tokenizer is not None else 31)
        dv = SyntheticDataset(v, batch_size, n, 2, seed=10 ** 6)
        if train_split is None:            # decoding: (dev, test) like the LibriSpeech branch below
            tt = SyntheticDataset(v, batch_size, n, 2, seed=2 * 10 ** 6)
            msg = _data_msg(name, path, str(dev_split), len(dv), str(test_split), len(tt), batch_size, False)
            msg = [m.replace("Dev", "Test").replace("Train", "Dev") for m in msg]
            return dv, tt, 1, 1, "test", msg
        tr = SyntheticDataset(v, batch_size, n, extra.get("n_batches", 64), seed=0)
        msg = _data_msg(name, path, str(train_split), len(tr), str(dev_split), len(dv), batch_size, False)
        return tr, dv, 1, 1, "train", msg
    if name.lower() != "librispeech":
        raise NotImplementedError(name)
    from .corpus import LibriDataset as Dataset_
    if train_split is not None:
        mode = "train"
        tr_loader_bs = 1 if bucketing and (not ascending) else batch_size
        bucket_size = batch_size if bucketing and (not ascending) else 1
        dv_set = Dataset_(path, dev_split, tokenizer, 1)
        tr_set = Dataset_(path, train_split, tokenizer, bucket_size, ascending=ascending)
        msg = _data_msg(name, path, str(train_split), len(tr_set), str(dev_split), len(dv_set), batch_size, bucketing)
        return tr_set, dv_set, tr_loader_bs, batch_size, mode, msg
    mode = "test"
    dv_set = Dataset_(path, dev_split, tokenizer, 1)
    tt_set = Dataset_(path, test_split, tokenizer, 1)
    msg = _data_msg(name, path, str(dev_split), len(dv_set), str(test_split), len(tt_set), batch_size, False)
    msg = [m.replace("Dev", "Test").replace("Train", "Dev") for m in msg]
    return dv_set, tt_set, batch_size, batch_size, mode, msg


class _VocabOnly:
    """Stand-in tokenizer for synthetic corpora: ids <-> space separated numbers."""
    token_type = "synthetic"

    def __init__(self, vocab_size):
        self.vocab_size = vocab_size

    def encode(self, s):
        return [int(x) for x in s.split()] + [1]

    def decode(self, ids, ignore_repeat=False):
        out = []
        for t, i in enumerate(ids):
            if i == 1:
                break
            if i == 0 or (ignore_repeat and t > 0 and i == ids[t - 1]):
                continue
            out.append(str(i))
        return " ".join(out)


def load_dataset(n_jobs, use_gpu, pin_memory, ascending, corpus, audio, text, device="cuda"):
    """Same signature and 6-tuple as src/data.py:129-156.  The returned loaders yield
    (names, wave [B,N], wave_len [B], txt [B,L]) - raw audio; features are made on the GPU by the Solver."""
    audio_transform, feat_dim = create_transform(audio.copy(), device=device)
    synthetic = corpus["name"].lower() == "synthetic"
    tokenizer = _VocabOnly(corpus.get("vocab_size", 31)) if synthetic else load_text_encoder(**text)
    tr_set, dv_set, tr_bs, dv_bs, mode, msg = create_dataset(tokenizer, ascending, **corpus)
    nf = audio_transform.frontend.num_frames
    collect_tr = partial(collect_wave_batch, num_frames=nf, mode=mode)
    collect_dv = partial(collect_wave_batch, num_frames=nf, mode="test")
    shuffle = (mode == "train" and not ascending) and not synthetic
    tr_loader = DataLoader(tr_set, batch_size=tr_bs, shuffle=shuffle, drop_last=shuffle, collate_fn=collect_tr,
                           num_workers=n_jobs, pin_memory=use_gpu)
    dv_loader = DataLoader(dv_set, batch_size=dv_bs, shuffle=False, drop_last=False, collate_fn=collect_dv,
                           num_workers=n_jobs, pin_memory=pin_memory)
    msg.append("I/O spec.  | Audio feature = {}\t| feature dim = {}\t| Token type = {}\t| Vocab size = {}".format(
        audio["feat_type"], feat_dim, tokenizer.token_type, tokenizer.vocab_size))
    tr_loader.audio_transform = audio_transform
    return tr_loader, dv_loader, feat_dim, tokenizer.vocab_size, tokenizer, msg


def _data_msg(name, path, train_split, tr_set, dev_split, dv_set, batch_size, bucketing):
    return ["Data spec. | Corpus = {} (from {})".format(name, path),
            "           | Train sets = {}\t| Number of utts = {}".format(train_split, tr_set),
            "           | Dev sets = {}\t| Number of utts = {}".format(dev_split, dv_set),
            "           | Batch size = {}\t\t| Bucketing = {}".format(batch_size, bucketing)]


# ---- text data of the RNN language model (the reference's src/data.py:46-61,107-126,159-177)--------------------
def collect_text_batch(batch, mode):
    """[[tokens, ...]] (one bucket) or [tokens, ...] -> txt [B, L] int64, zero padded; in train mode the batch is
    halved when its first sequence is longer than HALF_BATCHSIZE_TEXT_LEN tokens."""
    if type(batch[0][0]) is list:
        batch = batch[0]
    if len(batch[0]) > HALF_BATCHSIZE_TEXT_LEN and mode == "train":
        batch = batch[:len(batch) // 2]
    return pad_sequence([torch.LongTensor(b) for b in batch], batch_first=True)


class SyntheticTextDataset(Dataset):
    """Seeded text buckets for runs without a corpus: item i is a bucket of `batch_size` token lists, longest first,
    with lengths ~ U[min_len, max_len] (<eos> included), ids in [2, V) and <eos> = 1 last."""

    def __init__(self, vocab_size, batch_size, n_batches, seed, min_len=20, max_len=60):
        self.vocab_size, self.batch_size, self.n_batches, self.seed = vocab_size, batch_size, n_batches, seed
        self.min_len, self.max_len = min_len, max_len

    def __len__(self):
        return self.n_batches

    def __getitem__(self, i):
        g = torch.Generator().manual_seed(self.seed + i)
        lens = torch.sort(torch.randint(self.min_len, self.max_len + 1, (self.batch_size,), generator=g),
                          descending=True)[0]
        return [torch.randint(2, self.vocab_size, (int(n) - 1,), generator=g).tolist() + [1] for n in lens]


def create_textset(tokenizer, train_split, dev_split, name, path, bucketing, batch_size, **extra):
    """(tr_set, dv_set, tr_loader_bs, dv_loader_bs, msg) as src/data.py:107-126; the dev set is never bucketed."""
    if name.lower() == "synthetic":
        tr_set = SyntheticTextDataset(tokenizer.vocab_size, batch_size, extra.get("n_batches", 64), 0,
                                      extra.get("min_len", 20), extra.get("max_len", 60))
        dv_set = SyntheticTextDataset(tokenizer.vocab_size, batch_size, 2, 10 ** 6,
                                      extra.get("min_len", 20), extra.get("max_len", 60))
        msg = _data_msg(name, path, str(train_split), len(tr_set), str(dev_split), len(dv_set), batch_size, True)
        return tr_set, dv_set, 1, 1, msg
    if name.lower() != "librispeech":
        raise NotImplementedError(name)
    from .corpus import LibriTextDataset
    bucket_size = batch_size if bucketing else 1
    tr_loader_bs = 1 if bucketing else batch_size
    dv_set = LibriTextDataset(path, dev_split, tokenizer, 1)
    tr_set = LibriTextDataset(path, train_split, tokenizer, bucket_size)
    msg = _data_msg(name, path, str(train_split), len(tr_set), str(dev_split), len(dv_set), batch_size, bucketing)
    return tr_set, dv_set, tr_loader_bs, batch_size, msg


def load_textset(n_jobs, use_gpu, pin_memory, corpus, text):
    """(tr_loader, dv_loader, vocab_size, tokenizer, msg) as src/data.py:159-177.  The text lives in host memory, so
    the loaders use no worker processes (n_jobs is accepted for the reference's signature)."""
    synthetic = corpus["name"].lower() == "synthetic"
    tokenizer = _VocabOnly(corpus.get("vocab_size", 31)) if synthetic else load_text_encoder(**text)
    tr_set, dv_set, tr_bs, dv_bs, msg = create_textset(tokenizer, **corpus)
    tr_loader = DataLoader(tr_set, batch_size=tr_bs, shuffle=True, drop_last=True,
                           collate_fn=partial(collect_text_batch, mode="train"), num_workers=0, pin_memory=use_gpu)
    dv_loader = DataLoader(dv_set, batch_size=dv_bs, shuffle=False, drop_last=False,
                           collate_fn=partial(collect_text_batch, mode="dev"), num_workers=0, pin_memory=pin_memory)
    msg.append("I/O spec.  | Token type = {}\t| Vocab size = {}".format(tokenizer.token_type, tokenizer.vocab_size))
    return tr_loader, dv_loader, tokenizer.vocab_size, tokenizer, msg
