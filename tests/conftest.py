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
    """GPU tests are selected with -m gpu; without a device they are skipped, never run on a fallback."""
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:  # pragma: no cover
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session", autouse=True)
def _built_library():
    """Make sure the C-ABI library exists (nvcc cross-compiles without a GPU)."""
    import __graft_entry__ as ge
    ge.build(verbose=False)


def load_golden(name):
    return dict(np.load(os.path.join(GOLDEN, name), allow_pickle=False))


def state_dict_from(g, prefix="sd/", dtype=None):
    out = {k[len(prefix):]: v for k, v in g.items() if k.startswith(prefix)}
    if dtype is not None:
        out = {k: (v.astype(dtype) if np.issubdtype(v.dtype, np.floating) else v) for k, v in out.items()}
    return out


def golden_grad(g, name, grad):
    """(grad, golden gradient of parameter `name`).  A fixture may store a weight matrix's gradient as every
    g["grad_stride"]-th element of the flattened matrix (keeps the file small); `grad` is then sampled the same way.
    The stride is coprime with the row lengths, so every row and every column of the matrix is compared."""
    ref = g["grad/" + name]
    if tuple(ref.shape) == tuple(grad.shape):
        return grad, ref
    stride, numel = int(g["grad_stride"]), grad.reshape(-1).shape[0]
    assert grad.ndim > 1 and ref.ndim == 1 and ref.size == -(-numel // stride), \
        f"grad {name}: shape {tuple(grad.shape)} is neither the stored {ref.shape} nor a matrix it was sampled from"
    return grad.reshape(-1)[::stride], ref
