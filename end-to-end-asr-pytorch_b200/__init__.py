"""b200asr - B200-native (sm_100a) implementation of the End-to-end-ASR-Pytorch train-step hot path.

The directory name follows the reference repository; import it with
    importlib.import_module("end-to-end-asr-pytorch_b200")
(or `import b200asr`, the alias module at the repo root).  Layout:
    csrc/      hand-written CUDA kernels + the C ABI (include/b200asr.h) -> libb200asr.so
    lib.py     ctypes binding;  ops.py  autograd wrappers
    audio.py / module.py / asr.py / lm.py / optim.py / solver.py / train_asr.py / test_asr.py / train_lm.py / data.py /
    text.py    host-side mirror of the reference's src/ + bin/train_{asr,lm}.py API (same names and signatures)
"""
from . import lib
from . import ops
from .lib import B200AsrError, load as load_library
from .audio import create_transform, FbankFrontEnd
from .asr import ASR, Encoder, Decoder, Attention
from .ops import CTCLoss
from . import audio, module, asr, optim, dist, synthetic, trainer, util, text, data, corpus, option, solver, train_asr, test_asr, ctc, lm, train_lm
from .optim import Optimizer
from .trainer import TrainStep

__all__ = ["lib", "B200AsrError", "load_library", "create_transform", "FbankFrontEnd", "ASR", "Encoder", "Decoder",
           "Attention", "CTCLoss"]
