"""ctypes binding of libb200asr.so (the C ABI declared in include/b200asr.h).

PyTorch is used only as the owner of device memory and streams: every call passes raw device pointers and the
current CUDA stream. There is no CPU fallback - a missing library or a non-CUDA tensor is an error.
"""
import ctypes
import os
from ctypes import c_int, c_float, c_longlong, c_size_t, c_void_p, c_char_p, c_ulonglong, POINTER

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200asr.so")

_lib = None

# name -> (restype, argtypes); mirrors include/b200asr.h one to one
_P = c_void_p
SIGNATURES = {
    "b200asr_version": (c_int, []),
    "b200asr_last_error": (c_char_p, []),
    "b200asr_launch_count": (c_ulonglong, []),
    "b200asr_launch_count_reset": (None, []),
    "b200asr_device_sm_count": (c_int, []),
    "b200asr_fbank_fwd": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, c_float, c_int, _P, c_int, _P, _P, _P, _P,
                                  c_int, c_int, c_float, _P, c_int, _P, _P]),
    "b200asr_fbank_fwd_pcm16": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, c_float, c_int, _P, c_int, _P, _P, _P, _P,
                                  c_int, c_int, c_float, _P, c_int, _P, _P]),
    "b200asr_delta_cmvn_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "b200asr_delta_cmvn_fwd": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, c_int, c_float, _P, _P, c_size_t,
                                       _P]),
    "b200asr_log_softmax_fwd": (c_int, [_P, _P, _P, _P, c_longlong, c_int, _P]),
    "b200asr_log_softmax_bwd": (c_int, [_P, _P, _P, c_longlong, c_int, _P]),
    "b200asr_ctc_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "b200asr_ctc_fwd_bwd": (c_int, [_P, c_longlong, c_longlong, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P,
                                    _P, _P, c_size_t, _P]),
    "b200asr_ctc_grad": (c_int, [_P, c_longlong, c_longlong, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, _P,
                                 _P, _P, c_size_t, _P]),
    "b200asr_ctc_fwd_bwd_logits": (c_int, [_P, _P, c_longlong, c_longlong, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P,
                                           _P, _P, _P, c_size_t, _P]),
    "b200asr_ctc_grad_logits": (c_int, [_P, _P, c_longlong, c_longlong, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P,
                                        _P, _P, _P, _P, c_size_t, _P]),
    "b200asr_ctc_prefix_score": (c_int, [_P, c_int, c_int, _P, _P, _P, _P, c_int, c_int, c_int, c_int, _P, _P, _P]),
    "b200asr_bilstm_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "b200asr_bilstm_plan": (c_int, [c_int, c_int, c_int, POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "b200asr_bilstm_uses_tensor_cores": (c_int, [c_int, c_int, c_int]),
    "b200asr_bilstm_uses_tcgen05": (c_int, [c_int, c_int, c_int]),
    "b200asr_bilstm_fwd": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, _P, c_size_t, _P]),
    "b200asr_bilstm_bwd": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, _P, c_size_t, _P]),
    "b200asr_debug_set_lstm_trace": (None, [_P]),
    "b200asr_debug_set_lstm_mode": (None, [c_int]),
    "b200asr_lstm_cell_fwd": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, _P]),
    "b200asr_lstm_cell_bwd": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int, c_int, _P]),
    "b200asr_locattn_cluster_size": (c_int, [c_int, c_int]),
    "b200asr_locattn_wpart_floats": (c_size_t, [c_int, c_int, c_int]),
    "b200asr_locattn_fwd": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, c_float, c_int, c_int, c_int, c_int, c_int,
                                    c_int, _P, _P, _P]),
    "b200asr_locattn_bwd": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, c_float, _P, _P, _P, c_int, c_int, c_int, c_int,
                                    c_int, c_int, _P, _P, _P, _P, _P, _P]),
    "b200asr_locattn_bwd_acc": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, c_float, _P, _P, _P, c_int, c_int, c_int, c_int,
                                        c_int, c_int, _P, _P, _P, _P, _P]),
    "b200asr_attn_dvalue": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P, c_int, _P]),
    "b200asr_ce_fwd_bwd": (c_int, [_P, _P, c_longlong, c_longlong, c_int, _P, _P, _P, _P]),
    "b200asr_gemm3x_supported": (c_int, [c_int, c_int, c_int]),
    "b200asr_gemm3x_tn": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P]),
    "b200asr_gemm3x_tn_ld": (c_int, [_P, c_int, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P]),
    "b200asr_gemm3x_nn": (c_int, [_P, c_int, _P, c_int, _P, _P, c_int, c_int, c_int, c_int, c_int, _P]),
    "b200asr_gemm3x_workspace_bytes": (c_size_t, [c_int, c_int]),
    "b200asr_gemm3x_tn_ws": (c_int, [_P, c_int, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, c_size_t, _P]),
    "b200asr_gemm3x_nn_ws": (c_int, [_P, c_int, _P, c_int, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, c_size_t, _P]),
    "b200asr_gemm3x_nt": (c_int, [_P, c_longlong, c_longlong, c_int, _P, c_longlong, c_longlong, c_int, _P, c_int, c_int,
                                  c_int, c_int, c_int, c_int, c_int, _P, c_size_t, _P]),
    "b200asr_tf32_residual": (c_int, [_P, _P, c_longlong, _P]),
    "b200asr_gemm3x_tn_pre": (c_int, [_P, c_int, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, c_size_t, _P]),
    "b200asr_gemm3x_nn_pre": (c_int, [_P, c_int, _P, _P, c_int, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, c_size_t,
                                      _P]),
    "b200asr_gemm3x_tn_pre2": (c_int, [_P, _P, c_int, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, c_size_t, _P]),
    "b200asr_gemm3x_nn_pre2": (c_int, [_P, _P, c_int, _P, _P, c_int, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, c_size_t,
                                       _P]),
    "b200asr_gemm3x_nt_pre": (c_int, [_P, _P, c_longlong, c_longlong, c_int, _P, _P, c_longlong, c_longlong, c_int, _P, c_int,
                                      c_int, c_int, c_int, c_int, c_int, c_int, _P, c_size_t, _P]),
    "b200asr_split_tf32": (c_int, [_P, _P, _P, c_longlong, _P]),
    "b200asr_embedding_fwd": (c_int, [_P, c_longlong, _P, c_longlong, c_int, _P, _P]),
    "b200asr_embedding_bwd": (c_int, [_P, _P, c_longlong, _P, c_longlong, c_int, _P, c_int, _P]),
    "b200asr_grad_norm_scratch_bytes": (c_size_t, []),
    "b200asr_grad_norm": (c_int, [_P, c_longlong, _P, _P, _P]),
    "b200asr_adadelta_step": (c_int, [_P, _P, _P, _P, c_longlong, c_float, c_float, c_float, c_float, _P, c_float, _P]),
    "b200asr_adam_step": (c_int, [_P, _P, _P, _P, c_longlong, c_float, c_float, c_float, c_float, c_float, c_int, _P,
                                  c_float, _P]),
}


class B200AsrError(RuntimeError):
    pass


def load(build_if_missing=False):
    """dlopen the in-tree library (optionally building it first) and set the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        if build_if_missing:
            from . import _build
            _build.build()
        else:
            raise B200AsrError(
                "libb200asr.so is missing (%s): run `python -c 'import __graft_entry__ as g; g.build()'`; "
                "there is no CPU fallback" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    return load().b200asr_last_error().decode("utf-8", "replace")


def check(rc, what=""):
    if rc != 0:
        raise B200AsrError("%s failed (rc=%d): %s" % (what or "b200asr call", rc, last_error()))


def ptr(t):
    """Device pointer of a CUDA tensor (None -> NULL). Refuses host tensors: there is no CPU path."""
    if t is None:
        return None
    if not t.is_cuda:
        raise B200AsrError("b200asr kernels need CUDA tensors (got a %s tensor); there is no CPU fallback" % t.device)
    return c_void_p(t.data_ptr())


def stream():
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def launch_count():
    return int(load().b200asr_launch_count())


def launch_count_reset():
    load().b200asr_launch_count_reset()


# ---- optional per-kernel CUDA-event timing (bench.py's roofline numbers) -----------------------------------
class KernelTimer:
    """When enabled, every C-ABI kernel call is bracketed by CUDA events on the launching stream and tagged with
    its algorithmic byte count (SURVEY.md 8(d)); durations are read after the timed region, never inside it."""

    def __init__(self):
        self.enabled = False
        self.records = []        # (name, start_event, end_event, algorithmic_bytes)

    def reset(self):
        self.records = []

    def summary(self):
        out = {}
        for name, a, b, nbytes in self.records:
            d = out.setdefault(name, {"launches": 0, "ms": 0.0, "bytes": 0})
            d["launches"] += 1
            d["ms"] += a.elapsed_time(b)
            d["bytes"] += nbytes
        return out


TIMER = KernelTimer()


class timed:
    def __init__(self, name, nbytes=0):
        self.name, self.nbytes = name, nbytes

    def __enter__(self):
        if TIMER.enabled:
            self.a = torch.cuda.Event(enable_timing=True)
            self.b = torch.cuda.Event(enable_timing=True)
            self.a.record()
        return self

    def __exit__(self, *exc):
        if TIMER.enabled:
            self.b.record()
            TIMER.records.append((self.name, self.a, self.b, self.nbytes))
        return False
