import importlib
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


@pytest.fixture(scope="session")
def pkg():
    """The product package (its directory name is not a Python identifier, hence importlib)."""
    return importlib.import_module("end-to-end-asr-pytorch_b200")


def load_golden(name):
    return dict(np.load(os.path.join(GOLDEN, name), allow_pickle=False))


def golden_params(g, kind):
    """The initial state_dict of a golden model run (model_<kind>.npz).  It is the reference's seeded init_adadelta
    initialisation, which the package's ASR reproduces bit for bit, so the file keeps the seed and each tensor's shape
    and CRC-32 rather than the values; both are checked here."""
    import zlib
    import torch
    from oracle.make_golden import tiny_model_cfg
    pkg = importlib.import_module("end-to-end-asr-pytorch_b200")
    torch.manual_seed(int(g["seed"]))
    sd = pkg.ASR(g["feat"].shape[-1], int(g["vocab"]), True, **tiny_model_cfg(kind)).state_dict()
    shapes = {k[len("sd_shape."):]: tuple(v) for k, v in g.items() if k.startswith("sd_shape.")}
    assert {k: tuple(v.shape) for k, v in sd.items()} == shapes, "state_dict keys / shapes differ from the reference's"
    for k, v in sd.items():
        assert zlib.crc32(v.numpy().tobytes()) == int(g["sd_crc32." + k]), \
            "%s: the package's initialisation no longer reproduces the reference's" % k
    return {k: v.detach().clone() for k, v in sd.items()}


def golden_grad(g, k, grad):
    """(grad, golden gradient of parameter k) on the elements the golden file keeps: large gradients are stored as a
    fixed sample of their elements, whose flat indices are grad_idx.<k>."""
    grad = np.asarray(grad)
    idx = g.get("grad_idx." + k)
    return (grad if idx is None else grad.reshape(-1)[idx]), g["grad." + k]


def rel_err(a, b, floor=1e-3):
    """max |a-b| / max(|b|, floor) - the tolerance form of SURVEY.md 8(c)."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), floor))) if a.size else 0.0


def scaled_err(a, b):
    """max |a-b| / max |b|: error relative to the tensor's scale (for gradients with near-zero elements)."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b)) / max(float(np.max(np.abs(b))), 1e-30)) if a.size else 0.0
