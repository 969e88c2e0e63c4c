"""LibriSpeech file listing (/root/reference/corpus/librispeech.py:28-61): glob the audio files of the splits, read
`<spk>-<chap>.trans.txt`, sort by token length, serve single items or buckets.  Out of the accelerated path; kept so
that `main.py --config <libri yaml>` is a drop-in."""
from pathlib import Path

from torch.utils.data import Dataset


def _transcripts(directory):
    table = {}
    for f in Path(directory).glob("*.trans.txt"):
        for line in open(f, "r"):
            utt, _, txt = line.rstrip("\n").partition(" ")
            table[utt] = txt
    return table


class LibriDataset(Dataset):
    def __init__(self, path, split, tokenizer, bucket_size, ascending=False):
        self.path, self.bucket_size = path, bucket_size
        files = []
        for s in split:
            found = sorted(list(Path(path, s).rglob("*.flac")) + list(Path(path, s).rglob("*.wav")))
            assert len(found) > 0, "No data found @ {}".format(Path(path, s))
            files += found
        cache = {}
        texts = []
        for f in files:
            d = str(f.parent)
            if d not in cache:
                cache[d] = _transcripts(d)
            texts.append(tokenizer.encode(cache[d][f.name.split(".")[0]]))
        pairs = sorted(zip(files, texts), reverse=not ascending, key=lambda x: len(x[1]))
        self.file_list, self.text = [p[0] for p in pairs], [p[1] for p in pairs]

    def __getitem__(self, index):
        if self.bucket_size > 1:
            index = min(len(self.file_list) - self.bucket_size, index)
            return list(zip(self.file_list[index:index + self.bucket_size], self.text[index:index + self.bucket_size]))
        return self.file_list[index], self.text[index]

    def __len__(self):
        return len(self.file_list)


# the official LM text of LibriSpeech; a split with this name is a text file, encoded lazily on first access
OFFICIAL_TXT_SRC = ["librispeech-lm-norm.txt"]
# The longest N sentences of the combined, length-sorted text are dropped whenever the official text is among the
# splits, as in the reference.  N is 5,000,000 there (and here), so a small official-text file - or a small
# corpus that merely includes one - is emptied entirely; the quirk is kept for identical sampling on the full corpus.
REMOVE_TOP_N_TXT = 5000000


class LibriTextDataset(Dataset):
    """Text-only LibriSpeech (the reference's corpus/librispeech.py:64-117): the transcripts next to the globbed
    `*.flac` files of each split (the audio is never read) plus, for OFFICIAL_TXT_SRC splits, the lines of that file.
    Sorted by length, longest first; serves single token lists or buckets of `bucket_size` consecutive ones."""

    def __init__(self, path, split, tokenizer, bucket_size):
        self.path, self.bucket_size = path, bucket_size
        self.encode_on_fly = False
        files, sentences = [], []
        for s in split:
            if s in OFFICIAL_TXT_SRC:
                self.encode_on_fly = True
                with open(Path(path, s), "r") as f:
                    sentences += f.readlines()
            files += sorted(Path(path, s).rglob("*.flac"))
        assert len(files) > 0 or len(sentences) > 0, "No data found @ {}".format(path)
        cache = {}
        for f in files:
            d = str(f.parent)
            if d not in cache:
                cache[d] = _transcripts(d)
            sentences.append(cache[d][f.name.split(".")[0]])
        if self.encode_on_fly:
            # strings until first served: the sort below is by character count, as in the reference
            self.tokenizer = tokenizer
            self.text = sentences
        else:
            self.text = [tokenizer.encode(t) for t in sentences]
        self.text = sorted(self.text, reverse=True, key=len)
        if self.encode_on_fly:
            del self.text[:REMOVE_TOP_N_TXT]

    def _tokens(self, i):
        if type(self.text[i]) is str:
            self.text[i] = self.tokenizer.encode(self.text[i])
        return self.text[i]

    def __getitem__(self, index):
        if self.bucket_size > 1:
            index = min(len(self.text) - self.bucket_size, index)
            return [self._tokens(i) for i in range(index, index + self.bucket_size)]
        return self._tokens(index)

    def __len__(self):
        return len(self.text)
