"""torch.autograd wrappers around the C-ABI kernels (host-side plumbing; the arithmetic is in csrc/)."""
import ctypes
import os

import torch
from torch.autograd import Function

from . import lib as L


def _f32c(t):
    if t.dtype != torch.float32:
        raise L.B200AsrError("b200asr kernels compute in fp32 (got %s)" % t.dtype)
    return t if t.is_contiguous() else t.contiguous()


def _gemm_exact():
    """Plain library GEMMs (cuBLAS through torch) must run in true fp32 for the 1e-4 parity budget."""
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False


_gemm_exact()

_perm_cache = {}


def gate_perm(H, device):
    """Row permutation from PyTorch's gate-major [i|f|g|o] layout to the kernels' unit-major layout:
    new row j*4+g  <-  old row g*H+j."""
    key = (H, str(device))
    p = _perm_cache.get(key)
    if p is None:
        p = torch.arange(4 * H, device=device).view(4, H).t().reshape(-1).contiguous()
        _perm_cache[key] = p
    return p


# ----------------------------------------------------------------------------------------------------------
# Dense contractions of the step (K6 / K9 / K11 and their autograd backward).  fp32 parity (1e-4 on logits after 4
# recurrent layers) rules out single-pass TF32/BF16, so every product is error-compensated "3xTF32" (fp32 class).
# GEMM_MODE "umma" (default): this library's own tcgen05 kernel (csrc/gemm.cu) in its three operand forms -
#   gemm_tn  x . W^T (+ bias)   forward;   gemm_nn  dY . W   input gradient (W in place);   gemm_nt  dY^T . X   weight
#   gradient (contraction over the B*T rows, h_prev read shifted from the layer output, gate permutation in the epilogue).
#   Raw fp32 tiles are the TF32 hi operands, residual tiles are made on the fly in shared memory, and the TMEM
#   accumulation chain is cut every 128 k and summed in fp32 registers (the tensor core's own adds truncate).
# GEMM_MODE "tf32x3": the same arithmetic as three cuBLAS TF32 GEMMs on operands split by b200asr_split_tf32 (kept as a
#   cross-check and for shapes whose row pitch is not a multiple of 4 floats); "fp32": cuBLAS SGEMM on the CUDA cores.
GEMM_MODE = os.environ.get("B200ASR_GEMM", "umma")


# Pre-split activations too (B200ASR_GEMM_PRESPLIT):
#   "x" (default)  only the wide operand of the weight-gradient products (the layer input x for dW_ih, the layer output
#                  for dW_hh: small next to dG): nt 188 -> 204 TFLOP/s, cfg B weight gradients 13.5 -> 12.8 ms for 0.5 ms of
#                  residual passes
#   "1"            every activation / gradient operand (no in-kernel split pass at all): measured SLOWER (cfg B 66.1 ->
#                  68.4 ms/step; tn 248 -> 232, nn 233 -> 208 TFLOP/s) - the extra residual tiles arrive through the same
#                  L2 -> SM path that already runs at ~2/3 of its measured rate
#   "0"            weights only
_PRESPLIT = os.environ.get("B200ASR_GEMM_PRESPLIT", "x")
PRESPLIT_ACTIVATIONS = _PRESPLIT == "1"
PRESPLIT_NT_B = _PRESPLIT == "x"


def tf32_residual(w):
    """w - trunc_tf32(w): the part of a weight matrix the tensor core does not see in the raw fp32 bit pattern.  Computed
    once per step and weight (instead of once per tile by every CTA) for the `_pre` GEMM forms."""
    lib = L.load()
    w = _f32c(w)
    lo = torch.empty_like(w)
    with L.timed("tf32_residual", 8 * w.numel()):
        L.check(lib.b200asr_tf32_residual(L.ptr(w), L.ptr(lo), w.numel(), L.stream()), "tf32_residual")
    return lo


def gemm_tn(a, w, bias=None, out=None, accumulate=False, w_lo=None, a_lo=None):
    """out[M,N] (= or +=) a[M,K] @ w[N,K]^T (+ bias[N]) on the tensor cores at fp32-class accuracy (csrc/gemm.cu).
    w_lo = tf32_residual(w) selects the pre-split form; a_lo = tf32_residual(a) in addition the form without any
    in-kernel split pass."""
    lib = L.load()
    a, w = _f32c(a), _f32c(w)
    M, K = a.shape
    N = w.shape[0]
    if out is None:
        out = torch.empty((M, N), device=a.device, dtype=torch.float32)
        accumulate = False
    assert out.stride(1) == 1 and out.shape == (M, N)
    b = _f32c(bias) if bias is not None else None
    # algorithmic bytes: both operands and the result once; flops 2*M*N*K (x3 tensor-core products)
    with L.timed("gemm3x_tn", 4 * (M * K + N * K + M * N * (2 if accumulate else 1))):
        if w_lo is not None and a_lo is not None:
            ws_bytes = lib.b200asr_gemm3x_workspace_bytes(M, N)
            ws = torch.empty(max(ws_bytes, 16), device=a.device, dtype=torch.uint8)
            L.check(lib.b200asr_gemm3x_tn_pre2(L.ptr(a), L.ptr(a_lo), K, L.ptr(w), L.ptr(w_lo), L.ptr(b), L.ptr(out), M, N, K,
                                               out.stride(0), int(bool(accumulate)), L.ptr(ws), ws_bytes, L.stream()),
                    "gemm3x_tn_pre2")
        elif w_lo is not None:
            ws_bytes = lib.b200asr_gemm3x_workspace_bytes(M, N)
            ws = torch.empty(max(ws_bytes, 16), device=a.device, dtype=torch.uint8)
            L.check(lib.b200asr_gemm3x_tn_pre(L.ptr(a), K, L.ptr(w), L.ptr(w_lo), L.ptr(b), L.ptr(out), M, N, K,
                                              out.stride(0), int(bool(accumulate)), L.ptr(ws), ws_bytes, L.stream()),
                    "gemm3x_tn_pre")
        elif M <= 256:          # skinny (the decoder's per-step products): split-K over all SMs
            ws_bytes = lib.b200asr_gemm3x_workspace_bytes(M, N)
            ws = torch.empty(max(ws_bytes, 16), device=a.device, dtype=torch.uint8)
            L.check(lib.b200asr_gemm3x_tn_ws(L.ptr(a), K, L.ptr(w), L.ptr(b), L.ptr(out), M, N, K, out.stride(0),
                                             int(bool(accumulate)), L.ptr(ws), ws_bytes, L.stream()), "gemm3x_tn_ws")
        else:
            L.check(lib.b200asr_gemm3x_tn(L.ptr(a), L.ptr(w), L.ptr(b), L.ptr(out), M, N, K, out.stride(0),
                                          int(bool(accumulate)), L.stream()), "gemm3x_tn")
    return out


def _use_umma(K):
    return GEMM_MODE == "umma" and K % 4 == 0


def gemm_tn_ld(a_base, lda, M, K, w, bias=None):
    """Like gemm_tn but A is given as (base tensor, row pitch lda in floats, M rows of K floats): rows may overlap."""
    lib = L.load()
    w = _f32c(w)
    N = w.shape[0]
    out = torch.empty((M, N), device=w.device, dtype=torch.float32)
    b = _f32c(bias) if bias is not None else None
    with L.timed("gemm3x_tn", 4 * (M * lda + N * K + M * N)):
        L.check(lib.b200asr_gemm3x_tn_ld(L.ptr(a_base), lda, L.ptr(w), L.ptr(b), L.ptr(out), M, N, K, N, 0, L.stream()),
                "gemm3x_tn_ld")
    return out


def gemm_nn(a, w, out=None, accumulate=False, w_lo=None, a_lo=None):
    """out[M,N] (= or +=) a[M,K] @ w[K,N]: the input gradient dY . W with W read in place (MN-major operand)."""
    lib = L.load()
    a, w = _f32c(a), _f32c(w)
    M, K = a.shape
    N = w.shape[1]
    if out is None:
        out = torch.empty((M, N), device=a.device, dtype=torch.float32)
        accumulate = False
    assert out.stride(1) == 1 and out.shape == (M, N)
    with L.timed("gemm3x_nn", 4 * (M * K + N * K + M * N * (2 if accumulate else 1))):
        if w_lo is not None and a_lo is not None:
            ws_bytes = lib.b200asr_gemm3x_workspace_bytes(M, N)
            ws = torch.empty(max(ws_bytes, 16), device=a.device, dtype=torch.uint8)
            L.check(lib.b200asr_gemm3x_nn_pre2(L.ptr(a), L.ptr(a_lo), K, L.ptr(w), L.ptr(w_lo), N, None, L.ptr(out), M, N, K,
                                               out.stride(0), int(bool(accumulate)), L.ptr(ws), ws_bytes, L.stream()),
                    "gemm3x_nn_pre2")
        elif w_lo is not None:
            ws_bytes = lib.b200asr_gemm3x_workspace_bytes(M, N)
            ws = torch.empty(max(ws_bytes, 16), device=a.device, dtype=torch.uint8)
            L.check(lib.b200asr_gemm3x_nn_pre(L.ptr(a), K, L.ptr(w), L.ptr(w_lo), N, None, L.ptr(out), M, N, K,
                                              out.stride(0), int(bool(accumulate)), L.ptr(ws), ws_bytes, L.stream()),
                    "gemm3x_nn_pre")
        elif M <= 256:
            ws_bytes = lib.b200asr_gemm3x_workspace_bytes(M, N)
            ws = torch.empty(max(ws_bytes, 16), device=a.device, dtype=torch.uint8)
            L.check(lib.b200asr_gemm3x_nn_ws(L.ptr(a), K, L.ptr(w), N, None, L.ptr(out), M, N, K, out.stride(0),
                                             int(bool(accumulate)), L.ptr(ws), ws_bytes, L.stream()), "gemm3x_nn_ws")
        else:
            L.check(lib.b200asr_gemm3x_nn(L.ptr(a), K, L.ptr(w), N, None, L.ptr(out), M, N, K, out.stride(0),
                                          int(bool(accumulate)), L.stream()), "gemm3x_nn")
    return out


def gemm_nt(a, b, M, N, T, batches=1, lda=None, a_bstride=0, ldb=None, b_bstride=0, b_shift=0, permute_rows=False,
            a_lo=None, b_lo=None):
    """out[M,N] = sum over (batch, t) of a[batch, t, :M]^T b[batch, t + b_shift, :N]: the weight gradient dY^T . X.
    `a` / `b` are tensors whose data pointer is element (0, 0, 0); pitches are in floats (default: dense [T, M] / [T, N]).
    b_lo (+ optionally a_lo): tf32_residual of the operands, same layout - their tiles are not split in the kernel."""
    lib = L.load()
    lda = M if lda is None else lda
    ldb = N if ldb is None else ldb
    out = torch.empty((M, N), device=a.device, dtype=torch.float32)
    ws_bytes = lib.b200asr_gemm3x_workspace_bytes(M, N)
    ws = torch.empty(max(ws_bytes, 16), device=a.device, dtype=torch.uint8)
    with L.timed("gemm3x_nt", 4 * (batches * T * (M + N) + M * N)):
        if b_lo is not None:
            L.check(lib.b200asr_gemm3x_nt_pre(L.ptr(a), L.ptr(a_lo), lda, a_bstride, 0, L.ptr(b), L.ptr(b_lo), ldb, b_bstride,
                                              b_shift, L.ptr(out), M, N, T, batches, N, 0, int(bool(permute_rows)),
                                              L.ptr(ws), ws_bytes, L.stream()), "gemm3x_nt_pre")
        else:
            L.check(lib.b200asr_gemm3x_nt(L.ptr(a), lda, a_bstride, 0, L.ptr(b), ldb, b_bstride, b_shift, L.ptr(out), M, N,
                                          T, batches, N, 0, int(bool(permute_rows)), L.ptr(ws), ws_bytes, L.stream()),
                    "gemm3x_nt")
    return out


class Conv1dK4S2Fn(Function):
    """Conv1d(C -> O, kernel 4, stride 2, padding 1) over [B, T, C] (CNNExtractor, src/module.py:75-78) as ONE
    tensor-core GEMM: with one zero row in front of every utterance, output frame t reads the 4*C CONTIGUOUS floats that
    start at padded row 2t, so the im2col matrix is just the padded buffer viewed with row pitch 2*C (overlapping rows)
    and the TMA tensor map reads it in place.  Input gradient = GEMM + an overlap-add of the two window halves."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        x = _f32c(x)
        B, T, C = x.shape
        O = weight.shape[0]
        Tout = T // 2
        Tp = 2 * (Tout + 1)                                   # padded rows per utterance (even)
        xp = torch.zeros((B, Tp, C), device=x.device, dtype=torch.float32)
        xp[:, 1:T + 1] = x
        wm = weight.detach().permute(0, 2, 1).reshape(O, 4 * C).contiguous()    # K index = tap * C + channel
        M = B * (Tp // 2) - 1                                 # the last row of the view would read past the buffer
        yf = torch.empty((B * (Tp // 2), O), device=x.device, dtype=torch.float32)
        yf[M:] = 0
        yf[:M] = gemm_tn_ld(xp, 2 * C, M, 4 * C, wm, bias.detach() if bias is not None else None)
        ctx.save_for_backward(xp, wm)
        ctx.dims = (B, T, C, O, Tout, Tp, M)
        ctx.has_bias = bias is not None
        return yf.view(B, Tp // 2, O)[:, :Tout]

    @staticmethod
    def backward(ctx, dy):
        xp, wm = ctx.saved_tensors
        B, T, C, O, Tout, Tp, M = ctx.dims
        half = Tp // 2
        dyf = torch.zeros((B, half, O), device=dy.device, dtype=torch.float32)
        dyf[:, :Tout] = dy
        dy2 = dyf.view(B * half, O)
        dx = None
        if ctx.needs_input_grad[0]:
            dcols = gemm_nn(dy2, wm).view(B, half, 2, 2 * C)      # [.., 0]: rows 2t,2t+1  [.., 1]: 2t+2,2t+3
            dxp = torch.zeros((B, half + 1, 2 * C), device=dy.device, dtype=torch.float32)
            dxp[:, :half] += dcols[:, :, 0]
            dxp[:, 1:] += dcols[:, :, 1]
            dx = dxp.view(B, Tp + 2, C)[:, 1:T + 1].contiguous()
        dw = db = None
        if ctx.needs_input_grad[1]:
            dwm = gemm_nt(dy2, xp, O, 4 * C, M, ldb=2 * C)                          # [O, 4C], windows read in place
            dw = dwm.view(O, 4, C).permute(0, 2, 1).contiguous()
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = dy.reshape(-1, O).sum(0)
        return dx, dw, db


def conv1d_k4s2p1(x, conv):
    """[B,T,C] -> [B,T//2,O] through the tensor-core GEMM when available, else the library convolution."""
    C = x.shape[-1]
    if (x.is_cuda and _use_umma(4 * C) and conv.kernel_size == (4,) and conv.stride == (2,) and conv.padding == (1,)
            and x.shape[1] >= 2 and (2 * C) % 4 == 0):
        return Conv1dK4S2Fn.apply(x, conv.weight, conv.bias)
    return conv(x.transpose(1, 2)).transpose(1, 2)


class Split:
    """fp32 matrix as (hi, lo) with hi exactly representable in TF32."""

    def __init__(self, x):
        lib = L.load()
        x = _f32c(x)
        self.hi = torch.empty_like(x)
        self.lo = torch.empty_like(x)
        with L.timed("split_tf32", 12 * x.numel()):
            L.check(lib.b200asr_split_tf32(L.ptr(x), L.ptr(self.hi), L.ptr(self.lo), x.numel(), L.stream()),
                    "split_tf32")

    def t(self):
        o = object.__new__(Split)
        o.hi, o.lo = self.hi.t(), self.lo.t()
        return o

    def view(self, *shape):
        o = object.__new__(Split)
        o.hi, o.lo = self.hi.view(*shape), self.lo.view(*shape)
        return o


def mm3(a, b, out=None, bias=None, accumulate=False):
    """out (= or +=) a @ b (+ bias) for Split operands: three error-compensated TF32 tensor-core GEMMs."""
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        if out is None:
            out = torch.empty((a.hi.shape[0], b.hi.shape[1]), device=a.hi.device, dtype=torch.float32)
            accumulate = False
        if accumulate:
            out.addmm_(a.lo, b.hi)
        elif bias is not None:
            torch.addmm(bias, a.lo, b.hi, out=out)
        else:
            torch.mm(a.lo, b.hi, out=out)
        out.addmm_(a.hi, b.lo)
        out.addmm_(a.hi, b.hi)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    return out


class Plain:
    """Same interface as Split for the exact-fp32 SGEMM mode."""

    def __init__(self, x):
        self.x = _f32c(x)

    def t(self):
        o = object.__new__(Plain)
        o.x = self.x.t()
        return o

    def view(self, *shape):
        o = object.__new__(Plain)
        o.x = self.x.view(*shape)
        return o


def mm1(a, b, out=None, bias=None, accumulate=False):
    if out is None:
        return torch.mm(a.x, b.x) if bias is None else torch.addmm(bias, a.x, b.x)
    if accumulate:
        return out.addmm_(a.x, b.x)
    if bias is not None:
        return torch.addmm(bias, a.x, b.x, out=out)
    return torch.mm(a.x, b.x, out=out)


def _gemm_ops():
    return (Split, mm3) if GEMM_MODE in ("tf32x3", "umma") else (Plain, mm1)


def _bilstm_forward(ctx, x, ndir, params):
    """BiLSTMFn.forward; also returns the cell states cst [ndir, B, T, H] (saved for the backward, which reads them)."""
    lib = L.load()
    assert len(params) == 4 * ndir
    Op, mm = _gemm_ops()
    x = _f32c(x)
    B, T, I = x.shape
    H = params[1].shape[1]
    dev = x.device
    perm = gate_perm(H, dev)
    umma = _use_umma(I)
    xs = None if umma else Op(x.view(B * T, I))
    gates = torch.empty((ndir, B, T, H, 4), device=dev, dtype=torch.float32)
    w_ih_p, w_ih_lo = [], []
    # the layer input enters the forward projection of both directions and both dW_ih products: split it once
    x_lo = tf32_residual(x) if (umma and PRESPLIT_ACTIVATIONS) else None
    for d in range(ndir):
        w_ih, w_hh, b_ih, b_hh = params[4 * d:4 * d + 4]
        wp = w_ih.detach().index_select(0, perm)
        bp = (b_ih.detach() + b_hh.detach()).index_select(0, perm)
        if umma:
            wlo = tf32_residual(wp)            # once per step: shared by the forward product and the input gradient
            gemm_tn(x.view(B * T, I), wp, bias=bp, out=gates[d].view(B * T, 4 * H), w_lo=wlo,
                    a_lo=x_lo.view(B * T, I) if x_lo is not None else None)
            w_ih_lo.append(wlo)
        else:
            mm(xs, Op(wp).t(), out=gates[d].view(B * T, 4 * H), bias=bp)
        w_ih_p.append(wp)
    del xs
    w_hh = torch.stack([_f32c(params[4 * d + 1].detach()) for d in range(ndir)]).contiguous()
    cst = torch.empty((ndir, B, T, H), device=dev, dtype=torch.float32)
    out = torch.empty((B, T, ndir * H), device=dev, dtype=torch.float32)
    ws_bytes = lib.b200asr_bilstm_workspace_bytes(B, T, H, ndir)
    if ws_bytes == 0:
        raise L.B200AsrError("bilstm: no feasible decomposition for B=%d H=%d (H must be a multiple of 16)" % (B, H))
    ws = torch.empty(ws_bytes, device=dev, dtype=torch.uint8)
    # algorithmic bytes (SURVEY.md 8(d)): per step and direction read Gx[t] (16BH) + write h,c (8BH); W_hh once
    with L.timed("bilstm_fwd", ndir * (24 * B * H * T + 16 * H * H)):
        L.check(lib.b200asr_bilstm_fwd(L.ptr(gates), L.ptr(w_hh), L.ptr(cst), L.ptr(out), B, T, H, ndir,
                                       L.ptr(ws), ws_bytes, L.stream()), "bilstm_fwd")
    ctx.ndir = ndir
    ctx.dims = (B, T, I, H)
    ctx.consumed = False
    ctx.has_x_lo = x_lo is not None
    ctx.save_for_backward(x, gates, cst, out, w_hh, *w_ih_p, *w_ih_lo, *([x_lo] if x_lo is not None else []))
    return out, cst


class BiLSTMFn(Function):
    """One (bi)directional LSTM layer over zero-padded frames, zero initial state (src/module.py:129-132).

    forward(x[B,T,I], ndir, w_ih_0, w_hh_0, b_ih_0, b_hh_0 [, w_ih_1, w_hh_1, b_ih_1, b_hh_1]) -> out[B,T,ndir*H]
    The input projection and the weight-gradient contractions are tensor-core GEMMs (see GEMM_MODE); the recurrence
    (forward and BPTT) is the persistent kernel pair b200asr_bilstm_fwd / b200asr_bilstm_bwd.
    """

    @staticmethod
    def forward(ctx, x, ndir, *params):
        return _bilstm_forward(ctx, x, ndir, params)[0]

    @staticmethod
    def backward(ctx, dout):
        lib = L.load()
        if ctx.consumed:
            raise L.B200AsrError("BiLSTMFn.backward ran twice: the gate stash is overwritten in place")
        ctx.consumed = True
        Op, mm = _gemm_ops()
        ndir = ctx.ndir
        B, T, I, H = ctx.dims
        x, gates, cst, out, w_hh = ctx.saved_tensors[:5]
        w_ih_p = ctx.saved_tensors[5:5 + ndir]
        rest = ctx.saved_tensors[5 + ndir:]
        x_lo = rest[-1] if ctx.has_x_lo else None
        w_ih_lo = rest[:-1] if ctx.has_x_lo else rest
        dev = x.device
        dout = _f32c(dout)
        ws_bytes = lib.b200asr_bilstm_workspace_bytes(B, T, H, ndir)
        ws = torch.empty(ws_bytes, device=dev, dtype=torch.uint8)
        with L.timed("bilstm_bwd", 2 * ndir * (24 * B * H * T + 16 * H * H)):
            L.check(lib.b200asr_bilstm_bwd(L.ptr(gates), L.ptr(w_hh), L.ptr(cst), L.ptr(dout), B, T, H, ndir,
                                           L.ptr(ws), ws_bytes, L.stream()), "bilstm_bwd")
        perm = gate_perm(H, dev)
        need_dx = ctx.needs_input_grad[0]
        dx2 = torch.empty((B * T, I), device=dev, dtype=torch.float32) if need_dx else None
        grads = []
        if _use_umma(I) and H % 4 == 0:
            # own tensor-core kernels throughout: dX = dG . W (W in place), dW_ih = dG^T . X, dW_hh = dG^T . h_prev with
            # h_prev read from the layer output shifted by one step (never materialised); rows written through the gate
            # permutation by the epilogue.
            # Residuals made once per step (B200ASR_GEMM_PRESPLIT): "x" = the wide operand of the two weight-gradient
            # products (layer input for dW_ih, layer output for dW_hh); "1" = the gate gradient as well (it enters
            # dX, dW_ih and dW_hh), so that none of these kernels splits a tile - measured slower, see the switch above
            pre = x_lo is not None and len(w_ih_lo) == ndir
            g_lo = tf32_residual(gates) if pre else None
            pre_b = pre or PRESPLIT_NT_B
            if PRESPLIT_NT_B:
                x_lo = tf32_residual(x)
            out_lo = tf32_residual(out) if pre_b else None
            for d in range(ndir):
                g2 = gates[d].view(B * T, 4 * H)
                gl2 = g_lo[d].view(B * T, 4 * H) if pre else None
                if need_dx:
                    gemm_nn(g2, w_ih_p[d], out=dx2, accumulate=(d > 0), w_lo=w_ih_lo[d] if len(w_ih_lo) == ndir else None,
                            a_lo=gl2)
                dw_ih = gemm_nt(g2, x, 4 * H, I, B * T, permute_rows=True, a_lo=gl2, b_lo=x_lo)
                hd = out[:, :, d * H:(d + 1) * H]
                dw_hh = gemm_nt(g2, hd, 4 * H, H, T, batches=B, a_bstride=T * 4 * H, ldb=ndir * H,
                                b_bstride=T * ndir * H, b_shift=(-1 if d == 0 else 1), permute_rows=True,
                                a_lo=gl2, b_lo=out_lo[:, :, d * H:(d + 1) * H] if pre_b else None)
                db = torch.empty((4 * H,), device=dev, dtype=torch.float32)
                db.index_copy_(0, perm, g2.sum(0))
                grads += [dw_ih, dw_hh, db, db.clone()]
            return (dx2.view(B, T, I) if need_dx else None, None, *grads)
        xs = Op(x.view(B * T, I))
        for d in range(ndir):
            dG = Op(gates[d].view(B * T, 4 * H))  # d(loss)/d(pre-activation), unit-major columns
            if need_dx:
                mm(dG, Op(w_ih_p[d]), out=dx2, accumulate=(d > 0))
            dw_ih = torch.empty((4 * H, I), device=dev, dtype=torch.float32)
            dw_ih.index_copy_(0, perm, mm(dG.t(), xs))
            db = torch.empty((4 * H,), device=dev, dtype=torch.float32)
            db.index_copy_(0, perm, gates[d].view(B * T, 4 * H).sum(0))
            # h_{prev}: the hidden state of the previous step of this direction (zero at its first step)
            hprev = torch.zeros((B, T, H), device=dev, dtype=torch.float32)
            hd = out[:, :, d * H:(d + 1) * H]
            if T > 1:
                if d == 0:
                    hprev[:, 1:] = hd[:, :-1]
                else:
                    hprev[:, :-1] = hd[:, 1:]
            dw_hh = torch.empty((4 * H, H), device=dev, dtype=torch.float32)
            dw_hh.index_copy_(0, perm, mm(dG.t(), Op(hprev.view(B * T, H))))
            del dG, hprev
            grads += [dw_ih, dw_hh, db, db.clone()]
        return (dx2.view(B, T, I) if need_dx else None, None, *grads)


def bilstm(x, lstm_params, ndir):
    return BiLSTMFn.apply(x, ndir, *lstm_params)


class LSTMLastStateFn(Function):
    """A unidirectional BiLSTMFn layer that also returns each row's cell state at its step last[b]: the c_n of a
    packed nn.LSTM.  forward(x[B,T,I], last[B] int64 (device), w_ih, w_hh, b_ih, b_hh) -> (out[B,T,H], c_last[B,H]).
    c_last is a copy that carries no gradient (the RNN-LM's training loss does not depend on it)."""

    @staticmethod
    def forward(ctx, x, last, *params):
        out, cst = _bilstm_forward(ctx, x, 1, params)
        c_last = cst[0, torch.arange(x.shape[0], device=x.device), last]
        ctx.mark_non_differentiable(c_last)
        return out, c_last

    @staticmethod
    def backward(ctx, dout, _dc_last):
        dx, _, *grads = BiLSTMFn.backward(ctx, dout)
        return (dx, None, *grads)


def lstm_last_state(x, lstm_params, last):
    return LSTMLastStateFn.apply(x, last, *lstm_params)


# ----------------------------------------------------------------------------------------------------------
class EmbeddingFn(Function):
    """nn.Embedding without padding_idx (the RNN-LM's `emb`): row gather forward, deterministic segmented-sum weight
    gradient (csrc/embedding.cu).  forward(ids int64 [...], weight [V,E]) -> [..., E]."""

    @staticmethod
    def forward(ctx, ids, weight):
        lib = L.load()
        w = _f32c(weight.detach())
        V, E = w.shape
        ids = _check_ids(ids, V)
        out = torch.empty((ids.numel(), E), device=w.device, dtype=torch.float32)
        with L.timed("embedding_fwd", 8 * ids.numel() + 8 * ids.numel() * E):
            L.check(lib.b200asr_embedding_fwd(L.ptr(ids), ids.numel(), L.ptr(w), V, E, L.ptr(out), L.stream()),
                    "embedding_fwd")
        ctx.save_for_backward(ids)
        ctx.V = V
        return out.view(*ids.shape, E)

    @staticmethod
    def backward(ctx, dy):
        (ids,) = ctx.saved_tensors
        E = dy.shape[-1]
        dw = torch.empty((ctx.V, E), device=dy.device, dtype=torch.float32)
        embedding_backward(ids, dy, dw, accumulate=False, checked=True)
        return None, dw


def _check_ids(ids, V):
    """int64, contiguous, on the device, every id in [0, V) - else B200AsrError (one 16-byte read-back)."""
    if not ids.is_cuda:
        raise L.B200AsrError("embedding: ids must be a CUDA tensor (got %s); there is no CPU fallback" % ids.device)
    ids = ids.to(torch.int64).contiguous()
    if ids.numel():
        lo, hi = torch.stack(torch.aminmax(ids)).tolist()
        if lo < 0 or hi >= V:
            raise L.B200AsrError("embedding: ids must lie in [0, %d) (got min %d, max %d)" % (V, lo, hi))
    return ids


def embedding_backward(ids, dy, dw, accumulate=False, checked=False):
    """dw[V,E] (= or +=) the weight gradient of the gather `table[ids]`, given its output gradient dy [..., E].  Rows
    that receive no id are zeroed (or left as they are with accumulate).  The ids are stably sorted (torch.sort) so that every row
    sums its contributions in ascending position: bit-identical across runs."""
    lib = L.load()
    V, E = dw.shape
    assert dw.dtype == torch.float32 and dw.is_contiguous() and dy.shape[-1] == E
    if not checked:
        ids = _check_ids(ids, V)
    flat = ids.reshape(-1)
    dy = _f32c(dy).reshape(-1, E)
    assert dy.shape[0] == flat.numel()
    sorted_ids, order = torch.sort(flat, stable=True)
    with L.timed("embedding_bwd", 4 * dy.numel() + 16 * flat.numel() + 4 * V * E * (2 if accumulate else 1)):
        L.check(lib.b200asr_embedding_bwd(L.ptr(sorted_ids), L.ptr(order), flat.numel(), L.ptr(dy), V, E, L.ptr(dw),
                                          int(bool(accumulate)), L.stream()), "embedding_bwd")
    return dw


def embedding(ids, weight):
    return EmbeddingFn.apply(ids, weight)


# ----------------------------------------------------------------------------------------------------------
class LogSoftmaxFn(Function):
    """log_softmax over the last dim (src/asr.py:96) + greedy argmax ids as a by-product.

    `ctc_head=True` declares that the ONLY differentiable consumer of the result is the CTC loss (ops.CTCLoss), as in
    the reference's train step (bin/train_asr.py:123-124).  ATen's CTC backward - and ours - returns
    exp(lp) - occupancy, whose class sum is zero, i.e. it already IS the logit gradient (SURVEY.md F9): the
    log-softmax backward  dx = g - exp(lp) * sum_c g  is then the identity and its 12*T*V-byte pass is skipped.
    B200ASR_CHECK_CTC_HEAD=1 runs the full backward and checks the claim."""

    @staticmethod
    def forward(ctx, logits, ctc_head=False):
        lib = L.load()
        x = _f32c(logits)
        V = x.shape[-1]
        n = x.numel() // V
        y = torch.empty_like(x)
        am = torch.empty(x.shape[:-1], device=x.device, dtype=torch.int64)
        with L.timed("log_softmax_fwd", 8 * n * V):
            L.check(lib.b200asr_log_softmax_fwd(L.ptr(x), L.ptr(y), None, L.ptr(am), n, V, L.stream()),
                    "log_softmax_fwd")
        ctx.ctc_head = bool(ctc_head)
        ctx.save_for_backward(y)
        ctx.mark_non_differentiable(am)
        return y, am

    @staticmethod
    def backward(ctx, g, _gam):
        (y,) = ctx.saved_tensors
        if ctx.ctc_head and not _CHECK_CTC_HEAD:
            return g, None
        lib = L.load()
        g = _f32c(g)
        V = y.shape[-1]
        n = y.numel() // V
        dx = torch.empty_like(y)
        with L.timed("log_softmax_bwd", 12 * n * V):
            L.check(lib.b200asr_log_softmax_bwd(L.ptr(y), L.ptr(g), L.ptr(dx), n, V, L.stream()), "log_softmax_bwd")
        if ctx.ctc_head:
            err = float((dx - g).abs().max()) / max(float(g.abs().max()), 1e-30)
            if err > 1e-4:
                raise L.B200AsrError("log_softmax(ctc_head=True): upstream gradient is not a CTC gradient "
                                     "(identity-backward error %.2e)" % err)
        return dx, None


_CHECK_CTC_HEAD = os.environ.get("B200ASR_CHECK_CTC_HEAD", "0") == "1"


def log_softmax(logits, ctc_head=False):
    return LogSoftmaxFn.apply(logits, ctc_head)


class CTCHeadOutput:
    """`ctc_output` of ASR.forward when the CTC head is fused into the loss (train step): the logits [B, T, V], their
    per-row log-sum-exp [B, T] and the arg-max ids [B, T] instead of the V-wide log-prob tensor, which the train step
    never reads except through CTCLoss (bin/train_asr.py:123-124) and arg-max (cal_er, util.py:113-127).  Quacks
    like the tensor for exactly those uses; `materialize()` gives the log-probs [B, T, V] (detached) on demand."""

    def __init__(self, logits, lse, ids, time_major=False):
        self.logits, self.lse, self.ids, self.time_major = logits, lse, ids, time_major

    @property
    def shape(self):
        s = self.logits.shape
        return torch.Size((s[1], s[0], s[2])) if self.time_major else s

    @property
    def device(self):
        return self.logits.device

    def transpose(self, a, b):
        if {a % 3, b % 3} != {0, 1}:
            raise L.B200AsrError("CTCHeadOutput only swaps batch and time")
        return CTCHeadOutput(self.logits, self.lse, self.ids, not self.time_major)

    def argmax(self, dim=-1):
        if dim not in (-1, 2):
            raise L.B200AsrError("CTCHeadOutput.argmax is over the classes")
        return self.ids.transpose(0, 1) if self.time_major else self.ids

    def detach(self):
        return CTCHeadOutput(self.logits.detach(), self.lse, self.ids, self.time_major)

    def materialize(self):
        lp = self.logits.detach() - self.lse.unsqueeze(-1)
        return lp.transpose(0, 1) if self.time_major else lp


def ctc_head(logits):
    """logits [B, T, V] -> CTCHeadOutput: one pass over the logits for the row statistics (lse + arg-max), nothing
    V-wide written."""
    lib = L.load()
    x = _f32c(logits)
    B, T, V = x.shape
    lse = torch.empty((B, T), device=x.device, dtype=torch.float32)
    am = torch.empty((B, T), device=x.device, dtype=torch.int64)
    with L.timed("log_softmax_fwd", 4 * B * T * V):
        L.check(lib.b200asr_log_softmax_fwd(L.ptr(x), None, L.ptr(lse), L.ptr(am), B * T, V, L.stream()),
                "log_softmax_fwd(stats)")
    return CTCHeadOutput(x, lse, am)


class CTCLossFn(Function):
    """sum_b weight_b * nll_b.  Forward = the alpha/beta lattice kernels (nll); backward = ONE gradient kernel that
    already multiplies by weight_b and by the upstream scalar, so no scaling pass over [T,B,V] follows.

    log_probs: [T,B,V] view of [B,T,V] memory (or any layout with unit class stride), like the reference passes
    `ctc_output.transpose(0,1)` (bin/train_asr.py:123-124).
    """

    @staticmethod
    def forward(ctx, log_probs, targets, input_lengths, target_lengths, blank, weights, row_lse=None):
        """row_lse [B, T] given: `log_probs` holds the LOGITS of the CTC head and the log-softmax is fused into the
        lattice / gradient kernels (b200asr_ctc_*_logits); the returned gradient is then the logit gradient."""
        lib = L.load()
        if log_probs.dtype != torch.float32 or log_probs.stride(2) != 1:
            if row_lse is not None:
                raise L.B200AsrError("fused CTC head: logits must be fp32 with unit class stride")
            log_probs = log_probs.float().contiguous()
        T, B, V = log_probs.shape
        dev = log_probs.device
        targets = targets.to(device=dev, dtype=torch.int64).contiguous()
        if targets.dim() != 2:
            raise L.B200AsrError("CTC targets must be a padded [B, L] tensor (cudnn-style 1-D targets unsupported)")
        Lmax = targets.shape[1]
        il = torch.as_tensor(input_lengths, dtype=torch.int64).to(dev).contiguous()
        tl = torch.as_tensor(target_lengths, dtype=torch.int64).to(dev).contiguous()
        w = _f32c(weights.to(dev))
        nll = torch.empty(B, device=dev, dtype=torch.float32)
        ws_bytes = lib.b200asr_ctc_workspace_bytes(B, T, Lmax)
        ws = torch.empty(ws_bytes, device=dev, dtype=torch.uint8)
        if row_lse is not None:
            row_lse = _f32c(row_lse)
            assert tuple(row_lse.shape) == (B, T)
        with L.timed("ctc_alpha_beta", 4 * B):
            if row_lse is None:
                L.check(lib.b200asr_ctc_fwd_bwd(L.ptr(log_probs), log_probs.stride(1), log_probs.stride(0),
                                                L.ptr(targets), L.ptr(il), L.ptr(tl), B, T, V, Lmax, blank, L.ptr(nll),
                                                L.ptr(w), None, L.ptr(ws), ws_bytes, L.stream()), "ctc_fwd_bwd")
            else:
                L.check(lib.b200asr_ctc_fwd_bwd_logits(L.ptr(log_probs), L.ptr(row_lse), log_probs.stride(1),
                                                       log_probs.stride(0), L.ptr(targets), L.ptr(il), L.ptr(tl), B, T,
                                                       V, Lmax, blank, L.ptr(nll), L.ptr(w), None, L.ptr(ws), ws_bytes,
                                                       L.stream()), "ctc_fwd_bwd_logits")
        ctx.save_for_backward(log_probs, targets, il, tl, w, nll, ws)
        ctx.row_lse = row_lse
        ctx.blank = blank
        ctx.mark_non_differentiable(nll)
        loss = (nll * w).sum()
        return loss, nll

    @staticmethod
    def backward(ctx, gloss, _gnll):
        lib = L.load()
        log_probs, targets, il, tl, w, nll, ws = ctx.saved_tensors
        T, B, V = log_probs.shape
        # gradient buffer laid out like log_probs' memory
        grad = torch.empty_strided(log_probs.shape, log_probs.stride(), device=log_probs.device, dtype=torch.float32)
        up = _f32c(gloss.reshape(1))
        # algorithmic bytes (SURVEY.md 8(d)): read the log-probs and write the gradient once each
        with L.timed("ctc_grad", 8 * T * V * B):
            if ctx.row_lse is None:
                L.check(lib.b200asr_ctc_grad(L.ptr(log_probs), log_probs.stride(1), log_probs.stride(0),
                                             L.ptr(targets), L.ptr(il), L.ptr(tl), B, T, V, targets.shape[1], ctx.blank,
                                             L.ptr(nll), L.ptr(w), L.ptr(up), L.ptr(grad), L.ptr(ws), ws.numel(),
                                             L.stream()), "ctc_grad")
            else:
                L.check(lib.b200asr_ctc_grad_logits(L.ptr(log_probs), L.ptr(ctx.row_lse), log_probs.stride(1),
                                                    log_probs.stride(0), L.ptr(targets), L.ptr(il), L.ptr(tl), B, T, V,
                                                    targets.shape[1], ctx.blank, L.ptr(nll), L.ptr(w), L.ptr(up),
                                                    L.ptr(grad), L.ptr(ws), ws.numel(), L.stream()), "ctc_grad_logits")
        return grad, None, None, None, None, None, None


class CTCLoss(torch.nn.Module):
    """Drop-in for torch.nn.CTCLoss(blank, reduction, zero_infinity=False) at bin/train_asr.py:49.

    `global_batch` lets a data-parallel rank normalise by the global batch size (SURVEY.md 8(e))."""

    def __init__(self, blank=0, reduction="mean", zero_infinity=False):
        super().__init__()
        if zero_infinity:
            raise NotImplementedError("zero_infinity=True is not part of the reference path")
        self.blank = blank
        self.reduction = reduction
        self.global_batch = None

    def forward(self, log_probs, targets, input_lengths, target_lengths):
        row_lse = None
        if isinstance(log_probs, CTCHeadOutput):       # fused head: logits + row lse instead of V-wide log-probs
            if not log_probs.time_major:
                raise L.B200AsrError("CTCLoss expects [T, B, V] (pass ctc_output.transpose(0, 1))")
            row_lse = log_probs.lse
            log_probs = log_probs.logits.transpose(0, 1)
        B = log_probs.shape[1]
        dev = log_probs.device
        tl = torch.as_tensor(target_lengths, dtype=torch.int64).to(dev)
        if self.reduction == "mean":
            denom = float(self.global_batch or B)
            w = 1.0 / (tl.clamp_min(1).to(torch.float32) * denom)
        elif self.reduction == "sum":
            w = torch.ones(B, device=dev, dtype=torch.float32)
        else:
            raise NotImplementedError("reduction=%s" % self.reduction)
        loss, nll = CTCLossFn.apply(log_probs, targets, input_lengths, tl, self.blank, w, row_lse)
        self.last_nll = nll
        return loss


# ----------------------------------------------------------------------------------------------------------
class LSTMCellFn(Function):
    """Pointwise part of one LSTM step (decoder, src/asr.py:214-221): pre[B,4H] (i,f,g,o) , c_prev -> h, c."""

    @staticmethod
    def forward(ctx, pre, c_prev):
        lib = L.load()
        pre = _f32c(pre)
        c_prev = _f32c(c_prev)
        B, H4 = pre.shape
        H = H4 // 4
        gates = torch.empty_like(pre)
        c = torch.empty_like(c_prev)
        h = torch.empty_like(c_prev)
        L.check(lib.b200asr_lstm_cell_fwd(L.ptr(pre), L.ptr(c_prev), L.ptr(gates), L.ptr(c), L.ptr(h), B, H,
                                          L.stream()), "lstm_cell_fwd")
        ctx.save_for_backward(gates, c_prev, c)
        return h, c

    @staticmethod
    def backward(ctx, dh, dc):
        lib = L.load()
        gates, c_prev, c = ctx.saved_tensors
        B, H4 = gates.shape
        H = H4 // 4
        dh = _f32c(dh) if dh is not None else torch.zeros_like(c)
        dcn = _f32c(dc) if dc is not None else None
        dpre = torch.empty_like(gates)
        dcp = torch.empty_like(c)
        L.check(lib.b200asr_lstm_cell_bwd(L.ptr(gates), L.ptr(c_prev), L.ptr(c), L.ptr(dh), L.ptr(dcn), L.ptr(dpre),
                                          L.ptr(dcp), B, H, L.stream()), "lstm_cell_bwd")
        return dpre, dcp


def lstm_cell(pre, c_prev):
    return LSTMCellFn.apply(pre, c_prev)


# ----------------------------------------------------------------------------------------------------------
# Decoder LSTM step (src/asr.py:214-221): the two per-step projections  x . W_ih^T + h . W_hh^T + b  are ONE skinny
# tensor-core GEMM on [x | h] . [W_ih | W_hh]^T (split-K, csrc/gemm.cu), the backward's input gradient is one more, and
# the weight gradients of all L steps are ONE  dPre^T . [x | h]  contraction over the L*B stacked rows at the end of the
# loop (same accumulator-node idea as the attention memory above) instead of 2 L library SGEMMs + 2 L accumulations.
class DecMem:
    def __init__(self):
        self.dpre, self.x = [], []


class DecWeightsFn(Function):
    @staticmethod
    def forward(ctx, mem, w_ih, w_hh, b_ih, b_hh):
        ctx.set_materialize_grads(False)
        ctx.mem = mem
        ctx.I = w_ih.shape[1]
        token = torch.zeros(1, device=w_ih.device, dtype=torch.float32)
        wcat = torch.cat([w_ih, w_hh], 1).contiguous()
        wlo = tf32_residual(wcat)
        ctx.mark_non_differentiable(wlo)
        return wcat, (b_ih + b_hh).contiguous(), token, wlo

    @staticmethod
    def backward(ctx, gW, gb, _gtoken, _gwlo=None):
        mem, I = ctx.mem, ctx.I
        dW = gW
        db = gb
        if mem.dpre:
            dpre_all = torch.cat(mem.dpre, 0)
            x_all = torch.cat(mem.x, 0)
            d = gemm_nt(dpre_all, x_all, dpre_all.shape[1], x_all.shape[1], dpre_all.shape[0])
            dW = d if gW is None else d + gW
            s = dpre_all.sum(0)
            db = s if gb is None else s + gb
            mem.dpre, mem.x = [], []
        if dW is None:
            return None, None, None, None, None
        return None, dW[:, :I], dW[:, I:], db, db


class DecStepFn(Function):
    @staticmethod
    def forward(ctx, mem, token, x, h, wcat, bias, wlo):
        ctx.set_materialize_grads(False)
        xcat = torch.cat([x, h], 1).contiguous()
        pre = gemm_tn(xcat, wcat, bias=bias, w_lo=wlo)
        ctx.save_for_backward(xcat, wcat, wlo)
        ctx.mem = mem
        ctx.I = x.shape[1]
        return pre

    @staticmethod
    def backward(ctx, dpre):
        xcat, wcat, wlo = ctx.saved_tensors
        if dpre is None:
            return None, None, None, None, None, None, None
        dpre = _f32c(dpre)
        dx = gemm_nn(dpre, wcat, w_lo=wlo)
        ctx.mem.dpre.append(dpre)
        ctx.mem.x.append(xcat)
        return None, torch.zeros(1, device=dpre.device), dx[:, :ctx.I], dx[:, ctx.I:], None, None, None


def decoder_weights(w_ih, w_hh, b_ih, b_hh):
    """-> (mem, wcat [4H, I+H], bias [4H], token) for decoder_step(); once per batch and decoder layer."""
    mem = DecMem()
    return (mem,) + tuple(DecWeightsFn.apply(mem, w_ih, w_hh, b_ih, b_hh))


def decoder_step(dw, x, h):
    """pre-activations [B, 4H] of one decoder LSTM step from decoder_weights()' handle."""
    mem, wcat, bias, token, wlo = dw
    return DecStepFn.apply(mem, token, x, h, wcat, bias, wlo)


def decoder_gemm_supported(I, H):
    return GEMM_MODE == "umma" and (I + H) % 4 == 0 and (4 * H) % 4 == 0


# ----------------------------------------------------------------------------------------------------------
class CrossEntropyFn(Function):
    """CrossEntropyLoss(ignore_index) with the logit gradient produced by the same launch."""

    @staticmethod
    def forward(ctx, logits, target, ignore_index, reduction):
        lib = L.load()
        x = _f32c(logits)
        N, V = x.shape
        target = target.to(device=x.device, dtype=torch.int64).contiguous()
        if reduction == "mean":
            scale = 1.0 / (target != ignore_index).sum().to(torch.float32)
        elif reduction == "sum":
            scale = torch.ones((), device=x.device, dtype=torch.float32)
        else:
            raise NotImplementedError("reduction=%s" % reduction)
        scale = scale.reshape(1).contiguous()
        row = torch.empty(N, device=x.device, dtype=torch.float32)
        grad = torch.empty_like(x)
        with L.timed("ce_fwd_bwd", 8 * N * V):
            L.check(lib.b200asr_ce_fwd_bwd(L.ptr(x), L.ptr(target), ignore_index, N, V, L.ptr(scale), L.ptr(row),
                                           L.ptr(grad), L.stream()), "ce_fwd_bwd")
        ctx.save_for_backward(grad)
        return row.sum() * scale[0]

    @staticmethod
    def backward(ctx, gloss):
        (grad,) = ctx.saved_tensors
        return grad.mul_(gloss), None, None, None


def cross_entropy(logits, target, ignore_index=0, reduction="mean"):
    return CrossEntropyFn.apply(logits, target, ignore_index, reduction)


# ----------------------------------------------------------------------------------------------------------
class LocAttnStepFn(Function):
    """One location-aware attention step (src/module.py:234-258 + 189-195, single head) in one kernel launch;
    its backward is one launch too (+ a [B*CS, P] -> [P] reduction of the small weight-gradient partials)."""

    @staticmethod
    def forward(ctx, q, key, value, prev_att, enc_len, conv_w, proj_w, e_w, e_b, temperature):
        lib = L.load()
        q, key, value, prev_att = _f32c(q), _f32c(key), _f32c(value), _f32c(prev_att)
        B, T, D = key.shape
        E = value.shape[2]
        K, _, W = conv_w.shape
        R = (W - 1) // 2
        dev = key.device
        enc_len = enc_len.to(device=dev, dtype=torch.int64).contiguous()
        cw, pw = _f32c(conv_w.detach()), _f32c(proj_w.detach())
        ew, eb = _f32c(e_w.detach()).view(-1), _f32c(e_b.detach()).view(-1)
        attn = torch.empty((B, T), device=dev, dtype=torch.float32)
        cvec = torch.empty((B, E), device=dev, dtype=torch.float32)
        # algorithmic bytes (SURVEY.md 8(d)): key + value read once per step
        with L.timed("locattn_fwd", 4 * B * T * (D + E)):
            L.check(lib.b200asr_locattn_fwd(L.ptr(q), L.ptr(key), L.ptr(value), L.ptr(prev_att), L.ptr(enc_len),
                                            L.ptr(cw), L.ptr(pw), L.ptr(ew), L.ptr(eb), float(temperature), B, T, D, E,
                                            K, R, L.ptr(attn), L.ptr(cvec), L.stream()), "locattn_fwd")
        ctx.save_for_backward(q, key, value, prev_att, enc_len, cw, pw, ew, attn)
        ctx.dims = (B, T, D, E, K, R)
        ctx.temperature = float(temperature)
        ctx.w_shapes = (conv_w.shape, proj_w.shape, e_w.shape, e_b.shape)
        return cvec, attn

    @staticmethod
    def backward(ctx, dctx, dattn):
        lib = L.load()
        q, key, value, prev_att, enc_len, cw, pw, ew, attn = ctx.saved_tensors
        B, T, D, E, K, R = ctx.dims
        dev = key.device
        CS = lib.b200asr_locattn_cluster_size(T, E)
        P = lib.b200asr_locattn_wpart_floats(D, K, R)
        dctx = _f32c(dctx) if dctx is not None else torch.zeros((B, E), device=dev)
        dattn = _f32c(dattn) if dattn is not None else None
        dq_part = torch.empty((B, CS, D), device=dev, dtype=torch.float32)
        dkey = torch.empty((B, T, D), device=dev, dtype=torch.float32)
        dvalue = torch.empty((B, T, E), device=dev, dtype=torch.float32)
        dprev = torch.empty((B, T), device=dev, dtype=torch.float32)
        wpart = torch.empty((B * CS, P), device=dev, dtype=torch.float32)
        with L.timed("locattn_bwd", 4 * B * T * (2 * D + 2 * E)):
            L.check(lib.b200asr_locattn_bwd(L.ptr(q), L.ptr(key), L.ptr(value), L.ptr(prev_att), L.ptr(enc_len),
                                            L.ptr(cw), L.ptr(pw), L.ptr(ew), ctx.temperature, L.ptr(attn), L.ptr(dctx),
                                            L.ptr(dattn), B, T, D, E, K, R, L.ptr(dq_part), L.ptr(dkey), L.ptr(dvalue),
                                            L.ptr(dprev), L.ptr(wpart), L.stream()), "locattn_bwd")
        wsum = wpart.sum(0)
        W = 2 * R + 1
        s_conv, s_proj, s_ew, s_eb = ctx.w_shapes
        d_proj = wsum[:D * K].view(s_proj)
        d_conv = wsum[D * K:D * K + K * W].view(s_conv)
        d_ew = wsum[D * K + K * W:D * K + K * W + D].view(s_ew)
        d_eb = wsum[D * K + K * W + D:].view(s_eb)
        return dq_part.sum(1), dkey, dvalue, dprev, None, d_conv, d_proj, d_ew, d_eb, None


def loc_attention_step(q, key, value, prev_att, enc_len, conv_w, proj_w, e_w, e_b, temperature):
    """-> (context [B,E], attn [B,T])"""
    return LocAttnStepFn.apply(q, key, value, prev_att, enc_len, conv_w, proj_w, e_w, e_b, temperature)


# ----------------------------------------------------------------------------------------------------------
# The decode loop calls the attention L times on the SAME key / value / weights (src/asr.py:112-151).  Left to autograd,
# every step's backward writes a [B,T,D] and a [B,T,E] gradient that the engine then re-adds L-1 times (cfg C: 46 x
# (78 + 11) MB written and ~3x that re-read and re-written by ATen adds).  Instead the per-batch gradients live in ONE
# accumulator node:  AttnMemFn  hands key / value / the four small weights to the steps (plus a 1-element token whose
# only job is to make the engine run AttnMemFn.backward after the LAST step);  LocAttnMemStepFn.backward  adds d(key) and
# the weight-gradient partials in place (b200asr_locattn_bwd_acc) and records (attn_l, dctx_l);  AttnMemFn.backward
# forms d(value) = sum_l attn_l (x) dctx_l once (b200asr_attn_dvalue) and reduces the weight partials once.
class AttnMem:
    def __init__(self):
        self.dkey = None
        self.wpart = None
        self.attn, self.dctx = [], []
        self.meta = None


class AttnMemFn(Function):
    @staticmethod
    def forward(ctx, mem, key, value, conv_w, proj_w, e_w, e_b):
        ctx.set_materialize_grads(False)        # undefined output gradients arrive as None, not as [B,T,E] zeros
        ctx.mem = mem
        ctx.shapes = (key.shape, value.shape, conv_w.shape, proj_w.shape, e_w.shape, e_b.shape)
        token = torch.zeros(1, device=key.device, dtype=torch.float32)
        return (key.view_as(key), value.view_as(value), conv_w.view_as(conv_w), proj_w.view_as(proj_w),
                e_w.view_as(e_w), e_b.view_as(e_b), token)

    @staticmethod
    def backward(ctx, gkey, gvalue, gcw, gpw, gew, geb, _gtoken):
        lib = L.load()
        mem = ctx.mem
        s_key, s_value, s_conv, s_proj, s_ew, s_eb = ctx.shapes
        B, T, D = s_key
        E = s_value[2]
        dev = _gtoken.device
        dkey = mem.dkey if mem.dkey is not None else torch.zeros(s_key, device=dev)
        if gkey is not None:
            dkey = dkey + gkey
        if mem.attn:
            attn_all = torch.stack(mem.attn, 1).contiguous()          # [B, L, T]
            dctx_all = torch.stack(mem.dctx, 1).contiguous()          # [B, L, E]
            Lsteps = attn_all.shape[1]
            acc = gvalue is not None
            dvalue = _f32c(gvalue).clone() if acc else torch.empty(s_value, device=dev, dtype=torch.float32)
            with L.timed("attn_dvalue", 4 * B * (T * E + Lsteps * (T + E))):
                L.check(lib.b200asr_attn_dvalue(L.ptr(attn_all), L.ptr(dctx_all), B, Lsteps, T, E, L.ptr(dvalue),
                                                int(acc), L.stream()), "attn_dvalue")
        else:
            dvalue = gvalue
        d_conv = d_proj = d_ew = d_eb = None
        if mem.wpart is not None:
            K, _, W = s_conv
            wsum = mem.wpart.sum(0)
            d_proj = wsum[:D * K].view(s_proj)
            d_conv = wsum[D * K:D * K + K * W].view(s_conv)
            d_ew = wsum[D * K + K * W:D * K + K * W + D].view(s_ew)
            d_eb = wsum[D * K + K * W + D:].view(s_eb)
        add = lambda a, b: a if b is None else (b if a is None else a + b)
        mem.dkey = mem.wpart = None
        mem.attn, mem.dctx = [], []
        return None, dkey, dvalue, add(d_conv, gcw), add(d_proj, gpw), add(d_ew, gew), add(d_eb, geb)


def attention_memory(key, value, conv_w, proj_w, e_w, e_b):
    """-> (mem, key, value, conv_w, proj_w, e_w, e_b, token) for loc_attention_mem_step."""
    mem = AttnMem()
    return (mem,) + tuple(AttnMemFn.apply(mem, _f32c(key), _f32c(value), conv_w, proj_w, e_w, e_b))


class LocAttnMemStepFn(Function):
    """One decode step on an attention memory: forward = the same single-launch kernel as LocAttnStepFn; backward =
    b200asr_locattn_bwd_acc (d(key) / weight partials added into the memory, no d(value) write)."""

    @staticmethod
    def forward(ctx, mem, token, q, key, value, prev_att, enc_len, conv_w, proj_w, e_w, e_b, temperature):
        ctx.set_materialize_grads(False)
        lib = L.load()
        q, prev_att = _f32c(q), _f32c(prev_att)
        B, T, D = key.shape
        E = value.shape[2]
        K, _, W = conv_w.shape
        R = (W - 1) // 2
        dev = key.device
        enc_len = enc_len.to(device=dev, dtype=torch.int64).contiguous()
        cw, pw = _f32c(conv_w.detach()), _f32c(proj_w.detach())
        ew, eb = _f32c(e_w.detach()).view(-1), _f32c(e_b.detach()).view(-1)
        attn = torch.empty((B, T), device=dev, dtype=torch.float32)
        cvec = torch.empty((B, E), device=dev, dtype=torch.float32)
        with L.timed("locattn_fwd", 4 * B * T * (D + E)):
            L.check(lib.b200asr_locattn_fwd(L.ptr(q), L.ptr(key), L.ptr(value), L.ptr(prev_att), L.ptr(enc_len),
                                            L.ptr(cw), L.ptr(pw), L.ptr(ew), L.ptr(eb), float(temperature), B, T, D, E,
                                            K, R, L.ptr(attn), L.ptr(cvec), L.stream()), "locattn_fwd")
        ctx.save_for_backward(q, key, value, prev_att, enc_len, cw, pw, ew, attn)
        ctx.mem = mem
        ctx.dims = (B, T, D, E, K, R)
        ctx.temperature = float(temperature)
        return cvec, attn

    @staticmethod
    def backward(ctx, dctx, dattn):
        lib = L.load()
        q, key, value, prev_att, enc_len, cw, pw, ew, attn = ctx.saved_tensors
        B, T, D, E, K, R = ctx.dims
        mem = ctx.mem
        dev = key.device
        CS = lib.b200asr_locattn_cluster_size(T, E)
        P = lib.b200asr_locattn_wpart_floats(D, K, R)
        if mem.dkey is None:
            mem.dkey = torch.zeros((B, T, D), device=dev, dtype=torch.float32)
            mem.wpart = torch.zeros((B * CS, P), device=dev, dtype=torch.float32)
        dctx = _f32c(dctx) if dctx is not None else torch.zeros((B, E), device=dev)
        dattn = _f32c(dattn) if dattn is not None else None
        dq_part = torch.empty((B, CS, D), device=dev, dtype=torch.float32)
        dprev = torch.empty((B, T), device=dev, dtype=torch.float32)
        with L.timed("locattn_bwd", 4 * B * T * (2 * D + E)):
            L.check(lib.b200asr_locattn_bwd_acc(L.ptr(q), L.ptr(key), L.ptr(value), L.ptr(prev_att), L.ptr(enc_len),
                                                L.ptr(cw), L.ptr(pw), L.ptr(ew), ctx.temperature, L.ptr(attn),
                                                L.ptr(dctx), L.ptr(dattn), B, T, D, E, K, R, L.ptr(dq_part),
                                                L.ptr(mem.dkey), L.ptr(dprev), L.ptr(mem.wpart), L.stream()),
                    "locattn_bwd_acc")
        mem.attn.append(attn)
        mem.dctx.append(dctx)
        token_grad = torch.zeros(1, device=dev, dtype=torch.float32)
        return None, token_grad, dq_part.sum(1), None, None, dprev, None, None, None, None, None, None


def loc_attention_mem_step(mem, token, q, key, value, prev_att, enc_len, conv_w, proj_w, e_w, e_b, temperature):
    """-> (context [B,E], attn [B,T]); key ... e_b and token come from attention_memory()."""
    return LocAttnMemStepFn.apply(mem, token, q, key, value, prev_att, enc_len, conv_w, proj_w, e_w, e_b, temperature)


# ----------------------------------------------------------------------------------------------------------
class Linear3xFn(Function):
    """y = x W^T + b for the large dense layers of the step (CTC head, key projection, vocabulary projection) on
    the tensor cores with the same error-compensated 3xTF32 scheme as the LSTM input projection (fp32-class)."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        Op, mm = _gemm_ops()
        shp = x.shape
        x2 = _f32c(x).reshape(-1, shp[-1])
        wlo = None
        if _use_umma(x2.shape[1]):
            wlo = tf32_residual(weight.detach())
            y = gemm_tn(x2, weight.detach(), bias=bias.detach() if bias is not None else None, w_lo=wlo)
        else:
            y = mm(Op(x2), Op(weight.detach()).t(), bias=bias.detach() if bias is not None else None,
                   out=torch.empty((x2.shape[0], weight.shape[0]), device=x.device, dtype=torch.float32))
        ctx.save_for_backward(x2, weight, *([wlo] if wlo is not None else []))
        ctx.shp = shp
        ctx.has_bias = bias is not None
        return y.view(*shp[:-1], weight.shape[0])

    @staticmethod
    def backward(ctx, gy):
        Op, mm = _gemm_ops()
        x2, weight = ctx.saved_tensors[:2]
        wlo = ctx.saved_tensors[2] if len(ctx.saved_tensors) > 2 else None
        gy2 = _f32c(gy).reshape(-1, weight.shape[0])
        dx = None
        umma = _use_umma(weight.shape[0]) and _use_umma(weight.shape[1])
        if ctx.needs_input_grad[0]:
            if umma:
                dx = gemm_nn(gy2, weight.detach(), w_lo=wlo).view(ctx.shp)
            else:
                dx = mm(Op(gy2), Op(weight.detach())).view(ctx.shp)
        dw = None
        if ctx.needs_input_grad[1]:
            if umma:
                dw = gemm_nt(gy2, x2, weight.shape[0], weight.shape[1], gy2.shape[0])
            else:
                dw = mm(Op(gy2).t(), Op(x2))
        db = gy.reshape(-1, weight.shape[0]).sum(0) if ctx.has_bias and ctx.needs_input_grad[2] else None
        return dx, dw, db


def linear3x(x, layer):
    """Apply an nn.Linear through the 3xTF32 tensor-core path when the problem is large enough to matter."""
    return dense3x(x, layer.weight, layer.bias)


def dense3x(x, weight, bias=None):
    """linear3x for a bare weight (e.g. a tied embedding matrix as the output projection)."""
    rows = x.numel() // x.shape[-1]
    if x.is_cuda and rows * weight.shape[1] * weight.shape[0] >= (1 << 24):
        return Linear3xFn.apply(x, weight, bias)
    return torch.nn.functional.linear(x, weight, bias)
