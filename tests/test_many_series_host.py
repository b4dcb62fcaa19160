"""Host-side parts of many-series regression (GPR_1d_many): offsets validation, the argument checks of the segmented and
per-row C entry points (all before any CUDA call), and lockstep_minimize(pass_ids=True) against serial runs.  Runs without a
GPU."""
import ctypes
import threading

import numpy as np
import pytest
import scipy.optimize

from asvgp_b200 import optimizers


# ---- offsets ---------------------------------------------------------------------------------------------------------------
def test_validate_offsets_accepts_ragged_series_with_empty_ones():
    from asvgp_b200 import ops

    out = ops.validate_offsets([0, 0, 3, 3, 10], 10)
    assert out.dtype == np.int64 and out.tolist() == [0, 0, 3, 3, 10]
    import torch

    assert ops.validate_offsets(torch.tensor([0, 5], dtype=torch.int32), 5).tolist() == [0, 5]


@pytest.mark.parametrize("offsets,n,err,what", [
    ([0, 4, 2, 10], 10, ValueError, "non-decreasing"),
    ([0, 3, 9], 10, ValueError, "end at"),
    ([1, 3, 10], 10, ValueError, "start at 0"),
    (np.array([0.0, 3.0, 10.0]), 10, TypeError, "integers"),
    ([0], 0, ValueError, "S \\+ 1 >= 2"),
    (np.zeros((2, 2), dtype=np.int64), 0, ValueError, "1-D"),
])
def test_validate_offsets_rejects(offsets, n, err, what):
    from asvgp_b200 import ops

    with pytest.raises(err, match=what):
        ops.validate_offsets(offsets, n)


def test_float_tensor_offsets_rejected():
    import torch

    from asvgp_b200 import ops

    with pytest.raises(TypeError, match="integers"):
        ops.validate_offsets(torch.tensor([0.0, 2.0]), 2)


def test_model_rejects_bad_offsets_before_device_work():
    """GPR_1d_many validates offsets on the host before it touches the device."""
    from asvgp_b200 import basis as B, kernels as Kn
    from asvgp_b200.gpr import GPR_1d_many

    x = np.linspace(0.5, 9.5, 20).reshape(-1, 1)
    y = np.sin(x).reshape(-1)
    basis = B.B3Spline(0, 10, 10)
    for offsets in ([0, 12, 8, 20], [0, 19], np.array([0, 20], dtype=np.float64), [0]):
        with pytest.raises((ValueError, TypeError)):
            GPR_1d_many((x, y), offsets, Kn.Matern32(), basis)
    with pytest.raises(NotImplementedError):
        GPR_1d_many((x, np.zeros((20, 2))), [0, 20], Kn.Matern32(), basis)


# ---- lockstep with per-run objectives ----------------------------------------------------------------------------------------
def _f(u, i):
    """A different objective per run id i: a shifted bowl with ripples, and its gradient."""
    c = np.array([0.3 * i, -0.2 * i, 0.1])
    w = np.array([1.0, 1.3 + 0.1 * i, 0.7])
    f = 0.2 * np.sum((u - c) ** 2) - np.sum(np.cos(w * 2.0 * (u - c)))
    g = 0.4 * (u - c) + w * 2.0 * np.sin(w * 2.0 * (u - c))
    return float(f), g


def test_lockstep_pass_ids_matches_serial_runs_id_by_id():
    rng = np.random.default_rng(7)
    starts = rng.uniform(-2.0, 2.0, (6, 3))
    seen = []

    def fun_batch(U, ids):
        seen.append(np.array(ids))
        vals = [_f(u, int(i)) for u, i in zip(U, ids)]
        return np.array([v[0] for v in vals]), np.array([v[1] for v in vals]), np.zeros(len(ids), dtype=np.int64)

    results = optimizers.lockstep_minimize(fun_batch, starts, pass_ids=True)
    for i, (u0, res) in enumerate(zip(starts, results)):
        ref = scipy.optimize.minimize(lambda u, i=i: _f(u, i), u0, jac=True, method="L-BFGS-B")
        np.testing.assert_array_equal(res.x, ref.x)
        assert (res.nit, res.nfev, res.fun) == (ref.nit, ref.nfev, ref.fun)
    assert seen[0].tolist() == list(range(6))
    assert all(set(s) <= set(range(6)) for s in seen)


def test_lockstep_default_passes_points_only():
    calls = []

    def fun_batch(U):
        calls.append(U.shape)
        return np.sum(U * U, 1), 2 * U, np.zeros(U.shape[0], dtype=np.int64)

    res = optimizers.lockstep_minimize(fun_batch, np.ones((2, 3)))
    assert calls and all(r.fun < 1e-10 for r in res)


# ---- C entry points ----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    import __graft_entry__

    __graft_entry__.build()
    from asvgp_b200 import _lib

    return _lib


def _error_of(lib, name, *args):
    """The error text of a failing call, run on a thread of its own (the library's last-error text is per thread)."""
    out = []

    def run():
        try:
            lib.call(name, *args)
            out.append(None)
        except lib.AsvgpNativeError as exc:
            out.append(str(exc))

    t = threading.Thread(target=run)
    t.start()
    t.join()
    return out[0]


def _host(vals, ctype=ctypes.c_double):
    arr = (ctype * len(vals))(*vals)
    return ctypes.cast(arr, ctypes.c_void_p), arr


def test_segmented_accumulate_rejects_bad_arguments(lib):
    fake = ctypes.c_void_p(16)              # never dereferenced: every case fails before any CUDA call
    for args, what in (((fake, 0, fake, 0, 10, fake, 0, fake, 12, 3, fake, None), "S=0"),
                       ((fake, 0, fake, 0, 10, fake, -2, fake, 12, 3, fake, None), "S=-2"),
                       ((fake, 2, fake, 0, 10, fake, 3, fake, 12, 3, fake, None), "element type"),
                       ((fake, 0, fake, 7, 10, fake, 3, fake, 12, 3, fake, None), "element type"),
                       ((fake, 0, fake, 0, 10, fake, 3, fake, 12, 9, fake, None), "order"),
                       ((fake, 0, fake, 0, 10, None, 3, fake, 12, 3, fake, None), "NULL")):
        msg = _error_of(lib, "asvgp_accum_1d_segmented_typed", *args)
        assert msg is not None and what in msg, (args, msg)


def _rows_call(lib, B=2, R=3, rows=(0, 2), D=1, h_rows=True, M=1000):
    pv, _kv = _host([1.0] * max(B, 1))
    ps, _ks = _host([0.1] * max(B, 1))
    pr, _kr = _host(list(rows), ctypes.c_int64)
    work = max(lib.load().asvgp_workspace_bytes_1d_batched(M, 3, 0, max(1, min(B, 64)), max(1, min(D, 64))), 1)
    return _error_of(lib, "asvgp_elbo_grad_1d_batched_rows", None, None, None, R, pr if h_rows else None, M, 3, B, D, pv, ps, 0,
                     None, None, work, None)


def test_rows_bound_rejects_bad_arguments(lib):
    for kw, what in ((dict(rows=(0, 3)), "slot 1: row 3"), (dict(rows=(-1, 0)), "slot 0: row -1"), (dict(h_rows=False), "h_row"),
                     (dict(R=0, rows=(0, 0)), "R=0"), (dict(B=0), "B=0"), (dict(B=65, rows=[0] * 65), "B=65"),
                     (dict(D=65), "D=65")):
        msg = _rows_call(lib, **kw)
        assert msg is not None and what in msg, (kw, msg)


def test_batched_posterior_rejects_bad_arguments(lib):
    h = lib.load()
    assert h.asvgp_workspace_bytes_posterior_1d_batched(1000, 3, 0, 1) > 0
    assert h.asvgp_workspace_bytes_posterior_1d_batched(1000, 3, 0, 64) > 60 * h.asvgp_workspace_bytes_posterior_1d_batched(1000, 3, 0, 1)
    for args in ((1000, 3, 0, 0), (1000, 3, 0, 65), (0, 3, 0, 1), (1000, 7, 0, 1)):
        assert h.asvgp_workspace_bytes_posterior_1d_batched(*args) == -1, args
    ps, _ks = _host([0.1, 0.2])
    bad_s, _kb = _host([0.1, -1.0])
    pr, _kr = _host([0, 1], ctypes.c_int64)
    out_of_range, _ko = _host([0, 2], ctypes.c_int64)
    big = 1 << 40
    for args, what in (((None, None, 2, pr, 1000, 3, 0, ps, 0, None, None, None, None, big, None), "B=0"),
                       ((None, None, 2, pr, 1000, 3, 65, ps, 0, None, None, None, None, big, None), "B=65"),
                       ((None, None, 2, out_of_range, 1000, 3, 2, ps, 0, None, None, None, None, big, None), "slot 1: row 2"),
                       ((None, None, 2, None, 1000, 3, 2, ps, 0, None, None, None, None, big, None), "h_row"),
                       ((None, None, 2, pr, 1000, 3, 2, None, 0, None, None, None, None, big, None), "h_sigma2"),
                       ((None, None, 2, pr, 1000, 3, 2, bad_s, 0, None, None, None, None, big, None), "slot 1: sigma2"),
                       ((None, None, 2, pr, 1000, 3, 2, ps, 0, None, None, None, None, 1024, None), "workspace"),
                       ((None, None, 2, pr, 6, 3, 2, ps, 0, None, None, None, None, big, None), "M=6")):
        msg = _error_of(lib, "asvgp_posterior_1d_batched", *args)
        assert msg is not None and what in msg, (args, msg)


def test_segmented_predictor_rejects_bad_arguments(lib):
    fake = ctypes.c_void_p(16)
    for args, what in (((fake, 10, fake, 0, fake, 12, 3, fake, fake, fake, fake, fake, None), "S=0"),
                       ((fake, 10, None, 2, fake, 12, 3, fake, fake, fake, fake, fake, None), "NULL"),
                       ((fake, 10, fake, 2, fake, 12, 0, fake, fake, fake, fake, fake, None), "order")):
        msg = _error_of(lib, "asvgp_predict_1d_segmented", *args)
        assert msg is not None and what in msg, (args, msg)
