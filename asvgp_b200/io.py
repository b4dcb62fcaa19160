"""Ingestion of the data formats the reference's experiments read, into PINNED host memory, so that the models' host path
(`GPR_1d((X, y), ...)`, `GPR_kron`, `GPR_additive` with numpy / CPU-tensor data: double-buffered asynchronous H2D staging,
ops.accum_1d_host / accum_2d_host) streams them to the GPU at PCIe speed without an extra pageable->pinned copy.

    whitespace text      experiments/snelson/example.py:12-14        (np.loadtxt)
    pandas pickle        experiments/large_regression/electricity.py:30-31
    NetCDF               experiments/eNATL60/eNATL60.py:42-56         (xarray there; scipy.io.netcdf_file here: NetCDF-3 classic /
                                                                       64-bit offset files; NetCDF-4 needs a converter, no HDF5
                                                                       library ships in this image)

Every loader takes dtype=np.float64 (the default) or np.float32: the accumulate kernels read float32 training data as it is,
which halves the host memory and the PCIe bytes of the host path.

Host-side plumbing only (numpy / pandas / SciPy + torch for the pinned allocation); no arithmetic of the hot path."""
import numpy as np
import torch


def pin(a, dtype=torch.float64):
    """numpy array / tensor -> contiguous CPU tensor in page-locked memory (a plain CPU tensor when no CUDA driver is present,
    e.g. on a build machine)."""
    t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))
    t = t.to(dtype=dtype, device="cpu").contiguous()
    if torch.cuda.is_available() and not t.is_pinned():
        t = t.pin_memory()
    return t


def _torch_dtype(dtype):
    dt = np.dtype(dtype)
    if dt not in (np.dtype(np.float64), np.dtype(np.float32)):
        raise ValueError("dtype must be float64 or float32, not %s" % dt)
    return torch.float64 if dt == np.float64 else torch.float32


def load_text(path, dtype=np.float64, **loadtxt_kwargs):
    """Whitespace-separated numbers (the Snelson files): [n] or [n, columns] of `dtype`, pinned (parsed as float64, then
    rounded once)."""
    return pin(np.loadtxt(path, **loadtxt_kwargs), dtype=_torch_dtype(dtype))


def load_pickle(path, x_columns, y_column, dropna=True, rescale_x_to=None, dtype=np.float64):
    """pandas DataFrame pickle (electricity.py:30): (X[n, d], y[n, 1]) of `dtype`, pinned.  rescale_x_to = m rescales every
    input column to [0, m] as electricity.py:31 does with `Date_seq` (in float64, before the rounding to `dtype`)."""
    import pandas as pd

    df = pd.read_pickle(path)
    cols = [x_columns] if isinstance(x_columns, str) else list(x_columns)
    df = df[cols + [y_column]]
    if dropna:
        df = df.dropna()
    X = df[cols].to_numpy(dtype=np.float64)
    if rescale_x_to is not None:
        lo, hi = X.min(0), X.max(0)
        X = (X - lo) / (hi - lo) * float(rescale_x_to)
    td = _torch_dtype(dtype)
    return pin(X, dtype=td), pin(df[y_column].to_numpy(dtype=np.float64).reshape(-1, 1), dtype=td)


def load_netcdf(path, field, lon="nav_lon", lat="nav_lat", time_index=0, bbox=None, dtype=np.float64):
    """One time slice of a gridded field with 2-D coordinate variables (eNATL60.py:42-56): flattened, masked to finite values
    (and to bbox = (lon_min, lon_max, lat_min, lat_max) when given) -> (X[n, 2] = (lon, lat), y[n, 1]) of `dtype`, pinned.
    The scale factor and offset are applied in float64; the result is rounded to `dtype` once."""
    from scipy.io import netcdf_file

    try:
        nc = netcdf_file(path, "r", mmap=False)
    except Exception as exc:
        raise ValueError("%s is not a NetCDF-3 (classic / 64-bit offset) file: %s.  NetCDF-4 files are HDF5; convert them "
                         "with `nccopy -k classic`" % (path, exc))
    try:
        var = nc.variables[field]
        data = np.array(var[time_index] if var.data.ndim == 3 else var[:], dtype=np.float64)
        fill = getattr(var, "_FillValue", None)
        scale, offset = getattr(var, "scale_factor", 1.0), getattr(var, "add_offset", 0.0)
        if fill is not None:            # (the attribute may be stored in a narrower type than the data: compare loosely)
            data[np.isclose(data, float(np.asarray(fill).ravel()[0]), rtol=1e-6, atol=0.0)] = np.nan
        data = data * scale + offset
        lo = np.array(nc.variables[lon][:], dtype=np.float64)
        la = np.array(nc.variables[lat][:], dtype=np.float64)
        if lo.ndim == 1 and la.ndim == 1:                       # 1-D coordinate axes: make the 2-D coordinate fields
            lo, la = np.meshgrid(lo, la)
    finally:
        nc.close()
    z, lo, la = data.reshape(-1), lo.reshape(-1), la.reshape(-1)
    ok = np.isfinite(z)
    if bbox is not None:
        ok &= (lo > bbox[0]) & (lo < bbox[1]) & (la > bbox[2]) & (la < bbox[3])
    td = _torch_dtype(dtype)
    return pin(np.stack([lo[ok], la[ok]], 1), dtype=td), pin(z[ok].reshape(-1, 1), dtype=td)


def train_test_split(X, y, num_train, num_test, seed=1997, dtype=np.float64):
    """Random disjoint train / test subsets as the experiment scripts draw them (eNATL60.py:58-70): pinned tensors of
    `dtype`."""
    n = X.shape[0]
    if num_train + num_test > n:
        raise ValueError("num_train + num_test exceeds the %d available points" % n)
    perm = torch.from_numpy(np.random.default_rng(seed).permutation(n))
    tr, te = perm[:num_train], perm[num_train: num_train + num_test]
    td = _torch_dtype(dtype)
    return (pin(X[tr], dtype=td), pin(y[tr], dtype=td)), (pin(X[te], dtype=td), pin(y[te], dtype=td))
