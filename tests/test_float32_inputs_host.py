"""Host-side parts of float32 training data: the typed C entry points reject unknown element types before any CUDA call, and
the io loaders honour `dtype` (default float64, unchanged).  Runs without a GPU."""
import numpy as np
import pytest

TYPED = {
    "asvgp_accum_1d_typed": lambda xt, yt: (None, xt, None, yt, 10, None, 5, 3, None, None),
    "asvgp_accum_1d_binned_typed": lambda xt, yt: (None, xt, None, yt, 10, None, 5, 3, None, None, 0, None),
    "asvgp_order_probe_1d_typed": lambda xt, yt: (None, xt, 10, None, 5, None, None),
    "asvgp_accum_2d_typed": lambda xt, yt: (None, xt, None, yt, 10, None, 5, None, 5, 3, None, None, None),
    "asvgp_accum_2d_raster_typed": lambda xt, yt: (None, xt, None, yt, 10, 5, None, 5, None, 5, 3, None, None, None),
    "asvgp_accum_2d_binned_typed": lambda xt, yt: (None, xt, None, yt, 10, None, 5, None, 5, 3, None, None, None, 0, None),
    "asvgp_order_probe_2d_typed": lambda xt, yt: (None, xt, 10, None, 5, None, 5, None, None),
}


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__

    __graft_entry__.build()
    from asvgp_b200 import _lib

    return _lib


@pytest.mark.parametrize("name", sorted(TYPED))
@pytest.mark.parametrize("xt,yt", [(2, 0), (0, -1), (7, 1)])
def test_unknown_element_type_fails_loudly(lib, name, xt, yt):
    import threading

    if "probe" in name and xt in (0, 1):
        xt = 5                                   # the probes take one array: make its type the bad one
    caught = []

    def run():                                   # on a thread of its own: the library's last-error text is per thread
        try:
            lib.call(name, *TYPED[name](xt, yt))
        except lib.AsvgpNativeError as exc:
            caught.append(str(exc))

    t = threading.Thread(target=run)
    t.start()
    t.join()
    assert caught and "element type" in caught[0], caught


def test_type_codes_match_the_header():
    import os
    import re

    from asvgp_b200 import ops

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    text = open(os.path.join(root, "include", "asvgp_b200.h")).read()
    codes = dict((m.group(1), int(m.group(2))) for m in re.finditer(r"#define ASVGP_(F64|F32) (\d+)", text))
    import torch

    assert ops.ELEM_TYPES == {torch.float64: codes["F64"], torch.float32: codes["F32"]}
    assert ops.point_dtype(torch.float16) == torch.float64 and ops.point_dtype(torch.int32) == torch.float64
    assert ops.points_to_host(np.arange(5, dtype=np.int64)).dtype == torch.float64
    h = ops.points_to_host(np.arange(5, dtype=np.float32))
    assert h.dtype == torch.float32


def test_text_loader_dtype(tmp_path):
    import torch

    from asvgp_b200 import io

    x = np.random.default_rng(0).uniform(0, 6, (200, 2))
    p = tmp_path / "train"
    np.savetxt(p, x)
    t64 = io.load_text(p)
    assert t64.dtype == torch.float64
    np.testing.assert_array_equal(t64.numpy(), np.loadtxt(p))
    t32 = io.load_text(p, dtype=np.float32)
    assert t32.dtype == torch.float32
    np.testing.assert_array_equal(t32.numpy(), np.loadtxt(p).astype(np.float32))
    with pytest.raises(ValueError):
        io.load_text(p, dtype=np.float16)


def test_pickle_loader_dtype(tmp_path):
    import pandas as pd
    import torch

    from asvgp_b200 import io

    rng = np.random.default_rng(1)
    df = pd.DataFrame({"t": np.arange(50.0) * 60, "v": rng.uniform(0, 5, 50)})
    p = tmp_path / "frame.pkl"
    df.to_pickle(p)
    X64, y64 = io.load_pickle(p, "t", "v", rescale_x_to=1000)
    X32, y32 = io.load_pickle(p, "t", "v", rescale_x_to=1000, dtype=np.float32)
    assert X64.dtype == y64.dtype == torch.float64 and X32.dtype == y32.dtype == torch.float32
    xr = df[["t"]].to_numpy()
    xr = (xr - xr.min(0)) / (xr.max(0) - xr.min(0)) * 1000.0
    np.testing.assert_array_equal(X64.numpy(), xr)
    np.testing.assert_array_equal(X32.numpy(), X64.numpy().astype(np.float32))
    np.testing.assert_array_equal(y32.numpy(), y64.numpy().astype(np.float32))


def test_netcdf_loader_and_split_dtype(tmp_path):
    import torch
    from scipy.io import netcdf_file

    from asvgp_b200 import io

    p = str(tmp_path / "ssh.nc")
    ny, nx = 12, 15
    lon2, lat2 = np.meshgrid(np.linspace(-80, -25, nx), np.linspace(15, 55, ny))
    raw = np.round(np.sin(lon2 / 9) * np.cos(lat2 / 7) * 10000).astype(np.int16)
    raw[2, 3] = -32767
    with netcdf_file(p, "w") as nc:
        nc.createDimension("t", 1); nc.createDimension("y", ny); nc.createDimension("x", nx)
        v = nc.createVariable("sossheig", "i2", ("t", "y", "x")); v[0] = raw
        v._FillValue = np.int16(-32767); v.scale_factor = 1e-4; v.add_offset = 0.25
        nc.createVariable("nav_lon", "f4", ("y", "x"))[:] = lon2.astype(np.float32)
        nc.createVariable("nav_lat", "f4", ("y", "x"))[:] = lat2.astype(np.float32)
    X64, y64 = io.load_netcdf(p, "sossheig")
    X32, y32 = io.load_netcdf(p, "sossheig", dtype=np.float32)
    assert X64.dtype == y64.dtype == torch.float64 and X32.dtype == y32.dtype == torch.float32
    with netcdf_file(p, "r", mmap=False) as nc:                           # the attributes as the file stores them
        scale, offset = nc.variables["sossheig"].scale_factor, nc.variables["sossheig"].add_offset
    ok = raw.reshape(-1) != -32767
    want = raw.reshape(-1)[ok].astype(np.float64) * scale + offset          # scale and offset in float64 ...
    np.testing.assert_array_equal(y64.numpy().ravel(), want)
    np.testing.assert_array_equal(y32.numpy().ravel(), want.astype(np.float32))   # ... then one rounding
    np.testing.assert_array_equal(X32.numpy(), X64.numpy().astype(np.float32))
    (a, b), (c, d) = io.train_test_split(X64, y64, 40, 10, seed=5)
    (a32, b32), (c32, d32) = io.train_test_split(X64, y64, 40, 10, seed=5, dtype=np.float32)
    assert a.dtype == torch.float64 and a32.dtype == d32.dtype == torch.float32
    np.testing.assert_array_equal(a32.numpy(), a.numpy().astype(np.float32))
    np.testing.assert_array_equal(d32.numpy(), d.numpy().astype(np.float32))
