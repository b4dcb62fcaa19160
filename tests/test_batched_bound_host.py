"""Host-side parts of batched hyper-parameter evaluation: the lockstep multi-start driver against serial scipy runs (with a
fake batched objective), Scipy.minimize(starts=...) on a model stand-in, and the argument checks of the batched C entry points
and of GPR_1d.training_loss_and_gradients_batch.  Runs without a GPU."""
import ctypes
import threading

import numpy as np
import pytest
import scipy.optimize

from asvgp_b200 import optimizers
from asvgp_b200.kernels import Parameter

N_VARS = 3
FAIL_ABOVE = 2.2          # the fake objective "fails" (info != 0) where u[0] exceeds this


def _f(u):
    """A seeded multimodal objective with its gradient: a bowl with cosine ripples, several local minima per axis."""
    w = np.array([1.0, 1.7, 0.6])
    f = 0.1 * np.sum(u * u) - np.sum(np.cos(w * 3.0 * u + 0.3))
    g = 0.2 * u + w * 3.0 * np.sin(w * 3.0 * u + 0.3)
    return float(f), g


def _info(u):
    return 7 if u[0] > FAIL_ABOVE else 0


def _serial(u0):
    def fun(u):
        if _info(u):
            raise np.linalg.LinAlgError("pivot")
        return _f(u)

    return scipy.optimize.minimize(fun, u0, jac=True, method="L-BFGS-B")


class _Counter:
    def __init__(self):
        self.rounds, self.sizes = 0, []

    def __call__(self, U):
        self.rounds += 1
        self.sizes.append(U.shape[0])
        vals = [_f(u) for u in U]
        return (np.array([v[0] for v in vals]), np.array([v[1] for v in vals]), np.array([_info(u) for u in U]))


def _starts():
    rng = np.random.default_rng(20261021)
    starts = rng.uniform(-4.0, 4.0, (9, N_VARS))
    starts[0] = 0.0                      # near a minimum: finishes in few iterations
    starts[1] = [1.9, 0.0, 0.0]          # walks into the failing region
    starts[2] = [3.5, 1.0, -1.0]         # fails on its first evaluation
    return starts


def test_lockstep_iterates_equal_serial_runs():
    starts = _starts()
    ev = _Counter()
    results = optimizers.lockstep_minimize(ev, starts)
    assert len(results) == len(starts)
    n_failed = 0
    for u0, res in zip(starts, results):
        try:
            ref = _serial(u0)
        except np.linalg.LinAlgError:
            n_failed += 1
            assert not res.success and res.fun == np.inf and res.nit == -1
            assert _info(res.x) != 0
            continue
        np.testing.assert_array_equal(res.x, ref.x)
        assert (res.nit, res.nfev, res.fun, res.status) == (ref.nit, ref.nfev, ref.fun, ref.status)
    assert n_failed >= 2
    # one evaluation per round; a finished or failed run leaves the rounds, so the slowest run sets their number
    finished = [r.nfev for r in results if r.nit >= 0]
    assert ev.rounds >= max(finished) and sum(ev.sizes) >= sum(finished)
    assert ev.sizes[0] == len(starts) and ev.sizes[-1] < len(starts)
    assert all(a >= b for a, b in zip(ev.sizes, ev.sizes[1:]))


def test_lockstep_evaluation_error_stops_every_run():
    def broken(U):
        raise RuntimeError("device lost")

    with pytest.raises(RuntimeError, match="device lost"):
        optimizers.lockstep_minimize(broken, _starts())


class _FakeModel:
    """The slice of a model the optimiser uses, on the fake objective over all three unconstrained values."""

    def __init__(self, batch=True):
        self.a, self.b, self.c = Parameter(1.0, name="a"), Parameter(1.0, name="b"), Parameter(1.0, lower=1e-6, name="c")
        if not batch:
            self.training_loss_and_gradients_batch = None

    @property
    def trainable_variables(self):
        return [self.a, self.b, self.c]

    def training_loss(self):
        return self.training_loss_and_gradients()[0]

    def training_loss_and_gradients(self):
        u = np.array([p.unconstrained for p in self.trainable_variables])
        if _info(u):
            raise np.linalg.LinAlgError("pivot")
        return _f(u)

    def training_loss_and_gradients_batch(self, U):
        before = [p.unconstrained for p in self.trainable_variables]
        loss, grad, info = _Counter()(U)
        assert [p.unconstrained for p in self.trainable_variables] == before
        loss[info != 0], grad[info != 0] = np.inf, np.nan
        return loss, grad, info


def test_scipy_multi_start_matches_serial_and_keeps_the_best():
    starts = _starts()
    model = _FakeModel()
    res = optimizers.Scipy().minimize(model.training_loss, model.trainable_variables, starts=starts)
    assert len(res.results) == len(starts)
    for u0, r in zip(starts, res.results):
        ref_model = _FakeModel()
        for p, u in zip(ref_model.trainable_variables, u0):
            p.unconstrained = float(u)
        try:
            ref = optimizers.Scipy().minimize(ref_model.training_loss, ref_model.trainable_variables)
        except np.linalg.LinAlgError:
            assert r.fun == np.inf and not r.success
            continue
        np.testing.assert_array_equal(r.x, ref.x)
        assert r.nit == ref.nit
    funs = [r.fun for r in res.results]
    assert res.best == int(np.argmin(funs)) and res.fun == min(funs)
    np.testing.assert_array_equal([p.unconstrained for p in model.trainable_variables], res.results[res.best].x)


def test_scipy_multi_start_over_a_subset_of_variables():
    model = _FakeModel()
    model.c.unconstrained = 0.25
    starts = np.array([[0.5, -1.0], [-2.0, 2.0]])
    res = optimizers.Scipy().minimize(model.training_loss, [model.a, model.b], starts=starts)
    assert model.c.unconstrained == 0.25
    ref_model = _FakeModel()
    ref_model.c.unconstrained = 0.25
    ref_model.a.unconstrained, ref_model.b.unconstrained = starts[res.best]
    ref = optimizers.Scipy().minimize(ref_model.training_loss, [ref_model.a, ref_model.b])
    np.testing.assert_array_equal(res.x, ref.x)


def test_scipy_multi_start_argument_checks():
    model = _FakeModel()
    before = [p.unconstrained for p in model.trainable_variables]
    with pytest.raises(ValueError, match="starts"):
        optimizers.Scipy().minimize(model.training_loss, model.trainable_variables, starts=np.zeros((2, 2)))
    with pytest.raises(ValueError, match="finite"):
        optimizers.Scipy().minimize(model.training_loss, model.trainable_variables, starts=np.full((1, 3), np.nan))
    with pytest.raises(NotImplementedError):
        no_batch = _FakeModel(batch=False)
        optimizers.Scipy().minimize(no_batch.training_loss, no_batch.trainable_variables, starts=np.zeros((2, 3)))
    assert [p.unconstrained for p in model.trainable_variables] == before


def test_gpr_1d_batch_argument_checks():
    """Malformed U is rejected before any device work (the model is assembled without data)."""
    from asvgp_b200 import kernels as Kn
    from asvgp_b200.gpr import GPR_1d

    model = GPR_1d.__new__(GPR_1d)
    model.kernel, model.likelihood = Kn.Matern32(), Kn.Gaussian()
    for U, what in ((np.zeros(3), "shape"), (np.zeros((2, 2)), "shape"), (np.zeros((65, 3)), "1..64"),
                    (np.zeros((0, 3)), "1..64"), (np.array([[0.0, np.inf, 0.0]]), "finite")):
        with pytest.raises(ValueError, match=what):
            model.training_loss_and_gradients_batch(U)


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


def _host(vals):
    arr = (ctypes.c_double * len(vals))(*vals)
    return ctypes.cast(arr, ctypes.c_void_p), arr


def test_workspace_query_ranges(lib):
    h = lib.load()
    assert lib.MAX_BATCH == 64 and lib.MAX_BATCH_COLUMNS == 64
    one = h.asvgp_workspace_bytes_1d_batched(10_000, 3, 0, 1, 1)
    assert one > 0
    assert h.asvgp_workspace_bytes_1d_batched(10_000, 3, 0, 64, 3) > 64 * one
    for args in ((10_000, 3, 0, 0, 1), (10_000, 3, 0, 65, 1), (10_000, 3, 0, 1, 0), (10_000, 3, 0, 1, 65), (0, 3, 0, 1, 1),
                 (10_000, 7, 0, 1, 1)):
        assert h.asvgp_workspace_bytes_1d_batched(*args) == -1, args


def _elbo_batched(lib, B=2, D=1, v=None, s2=None, work_bytes=None, M=1000):
    v = v if v is not None else [1.0] * B
    s2 = s2 if s2 is not None else [0.1] * B
    pv, _kv = _host(v)
    ps, _ks = _host(s2)
    if work_bytes is None:
        work_bytes = max(lib.load().asvgp_workspace_bytes_1d_batched(M, 3, 0, max(1, min(B, 64)), max(1, min(D, 64))), 1)
    return _error_of(lib, "asvgp_elbo_grad_1d_batched", None, None, None, M, 3, B, D, pv, ps, 0, None, None, work_bytes, None)


def test_elbo_batched_rejects_bad_arguments_before_any_cuda_call(lib):
    for kw, what in ((dict(B=0), "B=0"), (dict(B=65, v=[1.0] * 65, s2=[0.1] * 65), "B=65"), (dict(D=0), "D=0"),
                     (dict(D=65), "D=65"), (dict(v=[1.0, -1.0]), "slot 1"), (dict(s2=[0.1, 0.0]), "slot 1"),
                     (dict(s2=[float("nan"), 0.1]), "slot 0"), (dict(work_bytes=1024), "workspace"), (dict(M=6), "M=6")):
        msg = _elbo_batched(lib, **kw)
        assert msg is not None and what in msg, (kw, msg)
    msg = _error_of(lib, "asvgp_elbo_grad_1d_batched", None, None, None, 1000, 3, 2, 1, None, None, 0, None, None, 1 << 40, None)
    assert msg is not None and "NULL" in msg


def test_kuu_assemble_batched_rejects_bad_arguments(lib):
    pc, _k = _host([1.0] * 4 * 65)
    for args, what in (((None, 4, 0, pc, None, 100, 3, None, None, None), "B=0"),
                       ((None, 4, 65, pc, None, 100, 3, None, None, None), "B=65"),
                       ((None, 0, 2, pc, None, 100, 3, None, None, None), "n_terms"),
                       ((None, 4, 2, pc, None, 100, 9, None, None, None), "order"),
                       ((None, 4, 2, None, None, 100, 3, None, None, None), "NULL")):
        msg = _error_of(lib, "asvgp_kuu_assemble_batched", *args)
        assert msg is not None and what in msg, (args, msg)
