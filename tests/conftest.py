import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


class _Arrays(dict):
    """A golden file's arrays by name, with the `files` list of the NpzFile that np.load returns."""

    @property
    def files(self):
        return list(self)


def _with_synth_1d_inputs(npz):
    """synth_1d.npz stores every SYNTH_1D_SAMPLE-th input point only: the full inputs k*_x, k*_y are regenerated from their
    seed and must match those samples."""
    import numpy as np

    if os.path.join(ROOT, "tests") not in sys.path:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
    import scale_cases as SC

    out = _Arrays((name, npz[name]) for name in npz.files)
    for k, (x, y, xs) in SC.synth_1d_inputs().items():
        key = "k%d" % k
        np.testing.assert_array_equal(x[::SC.SYNTH_1D_SAMPLE], out[key + "_x_sample"])
        np.testing.assert_allclose(y[::SC.SYNTH_1D_SAMPLE], out[key + "_y_sample"], rtol=0, atol=1e-14)   # np.sin may differ by an ulp
        np.testing.assert_array_equal(xs, out[key + "_xs"])
        out[key + "_x"], out[key + "_y"] = x, y
    return out


@pytest.fixture(scope="session")
def golden():
    import numpy as np

    def load(name):
        npz = np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)
        return _with_synth_1d_inputs(npz) if name == "synth_1d" else npz

    return load


@pytest.fixture(scope="session")
def cuda():
    import torch

    if not torch.cuda.is_available():
        pytest.fail("this test is marked gpu but no CUDA device is visible")
    # the native library must be the thing that runs: fail loudly if it is missing
    from asvgp_b200 import _lib

    _lib.load()
    return torch.device("cuda", 0)


@pytest.fixture(autouse=True)
def _poison_shared_memory(request):
    """Before every GPU test: NaN bit patterns into every SM's shared memory (asvgp_debug_poison_smem), so that a kernel reading
    a shared-memory slot it never wrote fails here, not once in ten runs on whatever the previous test left behind."""
    if request.node.get_closest_marker("gpu") is None:
        yield
        return
    import ctypes

    import torch

    from asvgp_b200 import _lib

    if torch.cuda.is_available():
        _lib.call("asvgp_debug_poison_smem", ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    yield


@pytest.fixture(scope="session", autouse=True)
def _poison_device_allocations():
    """ASVGP_POISON_SMEM=1 also NaN-fills (0xFF bytes for integer types) every CUDA tensor that torch.empty / empty_like hands
    out for the duration of the run: scratch and output buffers must not be read before the kernels write them."""
    if os.environ.get("ASVGP_POISON_SMEM") is None:
        yield
        return
    import torch

    orig_empty, orig_like = torch.empty, torch.empty_like

    def poison(t):
        if isinstance(t, torch.Tensor) and t.is_cuda and t.numel() > 0:
            if t.dtype.is_floating_point:
                t.fill_(float("nan"))
            elif t.dtype in (torch.uint8, torch.int8, torch.int16, torch.int32, torch.int64):
                t.fill_(-1 if t.dtype != torch.uint8 else 255)
        return t

    torch.empty = lambda *a, **k: poison(orig_empty(*a, **k))
    torch.empty_like = lambda *a, **k: poison(orig_like(*a, **k))
    try:
        yield
    finally:
        torch.empty, torch.empty_like = orig_empty, orig_like
