"""RNN language model with the reference's constructor, state_dict keys and forward contract (the reference's src/lm.py),
computing through the b200asr kernels.

  emb            ops.embedding (csrc/embedding.cu): row gather, deterministic segmented-sum weight gradient
  rnn (LSTM)     one persistent unidirectional LSTM layer per layer (ops.lstm_last_state); `self.rnn` is an nn.LSTM
                 used purely as the parameter container, so seeding + construction reproduce the reference's weights
  trans / tying  ops.dense3x (3xTF32 tensor-core GEMM) against trans.weight or, tied, emb.weight
  rnn (GRU)      the library's packed nn.GRU, as the ASR encoder's GRU branch (module.RNNLayer)

Packed-sequence semantics without packing: the recurrence is unidirectional and starts from a zero state, so running
it through the padding cannot change any valid step.  The outputs at t >= lens[b] are set to exactly 0 before the
head (pad_packed_sequence's zeros), so those logits equal trans.bias like the reference's, and (h_n, c_n) are read at
each row's last valid step.  The zeroed outputs also make the gradient of every padded step exactly 0.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops


class RNNLM(nn.Module):
    """RNN language model: (B, T) token ids -> (B, max(lens), vocab) logits and the final (h_n, c_n)."""

    def __init__(self, vocab_size, emb_tying, emb_dim, module, dim, n_layers, dropout):
        super().__init__()
        self.dim = dim
        self.n_layers = n_layers
        self.emb_tying = emb_tying
        if emb_tying:
            assert emb_dim == dim, "Output dim of RNN should be identical to embedding if using weight tying."
        self.vocab_size = vocab_size
        self.module = module.upper()
        if self.module not in ("LSTM", "GRU"):
            raise NotImplementedError("RNN module %s (the reference accepts LSTM and GRU)" % module)
        self.dropout = dropout
        # creation order = the reference's, so torch.manual_seed(s); RNNLM(...) draws the same initial weights
        self.emb = nn.Embedding(vocab_size, emb_dim)
        self.dp1 = nn.Dropout(dropout)
        self.dp2 = nn.Dropout(dropout)
        self.rnn = getattr(nn, self.module)(emb_dim, dim, num_layers=n_layers, dropout=dropout, batch_first=True)
        if not self.emb_tying:
            self.trans = nn.Linear(dim, vocab_size)

    def create_msg(self):
        return ["Model spec.| RNNLM weight tying = {}, # of layers = {}, dim = {}".format(
            self.emb_tying, self.n_layers, self.dim)]

    def layer_params(self, k):
        return [getattr(self.rnn, "%s_l%d" % (n, k)) for n in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")]

    def forward(self, x, lens, hidden=None):
        """x [B, T] int64 (device), lens [B] (host or device) -> (outputs [B, max(lens), V], hidden); hidden is
        (h_n, c_n) for LSTM and h_n for GRU, [n_layers, B, dim] each."""
        if hidden is not None:
            raise NotImplementedError("RNNLM.forward with an initial state (one-step decoding for LM-fused beam search) "
                                      "is not implemented yet")
        t_out = int(lens.max())
        x = x[:, :t_out]
        emb_x = self.dp1(ops.embedding(x, self.emb.weight))
        if self.module == "LSTM":
            outputs, hidden = self._lstm(emb_x, lens)
        else:
            packed = nn.utils.rnn.pack_padded_sequence(emb_x, lens.cpu(), batch_first=True, enforce_sorted=False)
            outputs, hidden = self.rnn(packed)
            outputs, _ = nn.utils.rnn.pad_packed_sequence(outputs, batch_first=True)
        head_w = self.emb.weight if self.emb_tying else self.trans.weight
        head_b = None if self.emb_tying else self.trans.bias
        return ops.dense3x(self.dp2(outputs), head_w, head_b), hidden

    def _lstm(self, h, lens):
        B, T, _ = h.shape
        lens = lens.to(h.device)
        last = (lens - 1).clamp_min(0)
        rows = torch.arange(B, device=h.device)
        h_n, c_n = [], []
        for k in range(self.n_layers):
            if k > 0:
                h = F.dropout(h, self.dropout, self.training)      # nn.LSTM(dropout=...): between layers, training only
            h, c_last = ops.lstm_last_state(h, self.layer_params(k), last)
            h_n.append(h[rows, last].detach())
            c_n.append(c_last)
        valid = torch.arange(T, device=h.device).unsqueeze(0) < lens.unsqueeze(1)
        outputs = h.masked_fill(~valid.unsqueeze(-1), 0.0)
        return outputs, (torch.stack(h_n), torch.stack(c_n))
