"""Host-side parts of the model layer: the multi-output column combination of the three models, the scal layouts of the
factorisation workspaces, the batched rows -> (loss, grad, info) step and the constructors' input checks.  The combination
is compared bit for bit with the per-model formulas it replaced (frozen copies below).  Runs without a GPU."""
import numpy as np
import pytest
import torch

from asvgp_b200 import basis as B, gpr, kernels as Kn, ops
from asvgp_b200.gpr import GPR_1d, GPR_1d_many, GPR_additive, GPR_kron


# ---- frozen copies of the per-model combinations this layer replaced -------------------------------------------------------
def _frozen_1d(outs, v, s2, n):
    out = outs[0].copy()
    extra = len(outs) - 1
    if extra:
        tr, dtr_dl = out[7], out[15]
        T = 0.5 * (-n * v + tr) / s2
        out[0:4] = outs[:, 0:4].sum(0) - extra * np.array([T, 0.5 * (-n + tr / v) / s2, 0.5 * dtr_dl / s2, -T / s2])
        out[6] = outs[:, 6].sum()
        bad = outs[:, 8][outs[:, 8] != 0]
        out[8] = bad[0] if bad.size else 0.0
    return out


def _frozen_kron(cols, Ts, N, v, s2, infos, want_grad):
    """cols[d] = (elbo_d, grad_d or None)."""
    info = infos[0] or infos[1] or infos[2]
    D = len(cols)
    if D == 1:
        return cols[0][0], cols[0][1], info
    tr = Ts[0][8]
    T0 = 0.5 * (-N * v[0] * v[1] + tr) / s2
    elbo = sum(c[0] for c in cols) - (D - 1) * T0
    g = None
    if want_grad:
        dT = np.array([0.5 * (-N * v[1] + tr / v[0]) / s2, 0.5 * Ts[0][9] / s2,
                       0.5 * (-N * v[0] + tr / v[1]) / s2, 0.5 * Ts[0][10] / s2, -T0 / s2])
        g = np.sum([c[1] for c in cols], 0) - (D - 1) * dT
    return elbo, g, info


def _frozen_additive(cols, N, v, s2, trn, infoP, sc, want_grad):
    info = infoP or next((s[2] for s in sc if s[2] != 0), 0.0)
    R, D = len(cols), len(v)
    vsum = float(np.sum(v))
    trace = float(trn[:, 0].sum())
    if R == 1:
        return cols[0][0], cols[0][1], info
    T0 = 0.5 * (-N * vsum + trace) / s2
    elbo = sum(c[0] for c in cols) - (R - 1) * T0
    g = None
    if want_grad:
        dT = []
        for i in range(D):
            dT += [0.5 * (-N + trn[i, 0] / v[i]) / s2, 0.5 * trn[i, 1] / s2]
        g = np.sum([c[1] for c in cols], 0) - (R - 1) * np.array(dT + [-T0 / s2])
    return elbo, g, info


def _same(got, want):
    assert np.array_equal(np.asarray(got[0]), np.asarray(want[0])), (got[0], want[0])
    if want[1] is not None:
        assert np.array_equal(np.asarray(got[1]), np.asarray(want[1])), (got[1], want[1])
    assert got[2] == want[2], (got[2], want[2])


def _infos(rng, n, fail):
    """n info values: all zero, or failing pivots (integers as float64) from position `fail` on (every later one too)."""
    out = np.zeros(n)
    if fail is not None:
        out[fail:] = rng.integers(1, 1000, n - fail)
    return out


CASES = [(D, fail) for D in (1, 2, 5) for fail in (None, 0, 1)] + [(5, 3)]


@pytest.mark.parametrize("D,fail", CASES)
def test_combination_matches_1d_formula(D, fail):
    rng = np.random.default_rng(10 * D + (fail or 0))
    for _ in range(50):
        outs = rng.standard_normal((D, 16)) * 10.0 ** rng.integers(-3, 4, (D, 16))
        outs[:, 8] = _infos(rng, D, fail if fail is None or fail < D else None)
        v, s2, n = rng.uniform(0.1, 3.0), rng.uniform(0.01, 1.0), float(rng.integers(1, 10**7))
        want = _frozen_1d(outs, v, s2, n)
        _same(GPR_1d._bound(outs, v, s2, lambda: n), (want[0], want[1:4], want[8]))


def _kron_inputs(rng, D):
    m1, m2 = 40, 30
    N = np.float64(rng.integers(1, 10**7))
    s2, v = rng.uniform(0.01, 1.0), [rng.uniform(0.1, 3.0), rng.uniform(0.1, 3.0)]
    sc1, sc2 = rng.standard_normal(4) * 100, rng.standard_normal(4) * 100
    logdetP = np.float64(rng.standard_normal() * 1e3)
    Qs, yys, Ts = rng.uniform(0, 1e4, D), rng.uniform(0, 1e4, D), rng.standard_normal((D, 11)) * 10.0 ** rng.integers(-2, 4, 11)
    return m1, m2, N, s2, v, sc1, sc2, logdetP, Qs, yys, Ts


@pytest.mark.parametrize("want_grad", [True, False])
@pytest.mark.parametrize("D,fail", CASES)
def test_combination_matches_kron_formula(D, fail, want_grad):
    rng = np.random.default_rng(100 + 10 * D + (fail or 0))
    for _ in range(50):
        m1, m2, N, s2, v, sc1, sc2, logdetP, Qs, yys, Ts = _kron_inputs(rng, D)
        infos = list(_infos(rng, 3, fail if fail is None or fail < 3 else None))
        rows = [gpr._kron_column_bound(N, s2, v, m1, m2, sc1, sc2, logdetP, Qs[d], yys[d], Ts[d], want_grad)[0]
                for d in range(D)]
        cols = [(r[0], r[1:] if want_grad else None) for r in rows]
        got = gpr._combine_columns(np.array(rows), infos, lambda: gpr._kron_shared(N, s2, v, Ts[0]))
        _same(got, _frozen_kron(cols, Ts, N, v, s2, infos, want_grad))


@pytest.mark.parametrize("want_grad", [True, False])
@pytest.mark.parametrize("D,fail", CASES)
def test_combination_matches_additive_formula(D, fail, want_grad):
    rng = np.random.default_rng(200 + 10 * D + (fail or 0))
    d = 3
    for _ in range(50):
        N, s2 = np.float64(rng.integers(1, 10**7)), rng.uniform(0.01, 1.0)
        v = list(rng.uniform(0.1, 3.0, d))
        ms = [50, 60, 70]
        sc = rng.standard_normal((d, 4)) * 100
        sc[:, 2] = 0.0
        infoP = 0.0
        if fail is not None and fail < d + 1:      # failing pivots in P (position 0) or in a dimension's factor
            if fail == 0:
                infoP = np.float64(rng.integers(1, 1000))
            sc[max(fail - 1, 0):, 2] = rng.integers(1, 1000, d - max(fail - 1, 0))
        trn = rng.standard_normal((d, 4)) * 100
        logdetP, logdetK, trace = np.float64(rng.standard_normal() * 1e3), float(sc[:, 0].sum()), float(trn[:, 0].sum())
        vsum = float(np.sum(v))
        Qs, yys = rng.uniform(0, 1e4, D), rng.uniform(0, 1e4, D)
        Tc, dn = rng.standard_normal((D, d, 4)) * 100, rng.standard_normal((D, 2)) * 100
        rows = [gpr._additive_column_bound(N, s2, v, vsum, ms, sc, logdetP, logdetK, trace, trn, Qs[c], yys[c], Tc[c], dn[c],
                                           want_grad) for c in range(D)]
        cols = [(r[0], r[1:] if want_grad else None) for r in rows]
        got = gpr._combine_columns(np.array(rows), [infoP] + list(sc[:, 2]),
                                   lambda: gpr._additive_shared(N, s2, v, vsum, trace, trn))
        _same(got, _frozen_additive(cols, N, v, s2, trn, infoP, sc, want_grad))


# ---- scal layouts ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cls", [ops.KronWorkspace, ops.DenseWorkspace])
def test_unpack_scal_reads_both_layouts(cls):
    logdet, info, Q = cls.unpack_scal(np.array([-12.5, 3.25, 7.0]))        # one right-hand side: {log|P|, Q, info}
    assert (logdet, info) == (-12.5, 7.0) and Q.tolist() == [3.25]
    logdet, info, Q = cls.unpack_scal(np.array([4.0, 0.0, 1.5, 2.5, 3.5]))  # three: {log|P|, info, Q_1, Q_2, Q_3}
    assert (logdet, info) == (4.0, 0.0) and Q.tolist() == [1.5, 2.5, 3.5]
    logdet, info, Q = cls.unpack_scal(np.array([4.0, 9.0, 1.5, 2.5]))
    assert (logdet, info) == (4.0, 9.0) and Q.tolist() == [1.5, 2.5]


# ---- rows -> (loss, grad, info) ----------------------------------------------------------------------------------------------
class _FakeFeatures:
    def make_Kuu_device_batched(self, kernel, ell, var, want_grad=True):
        return None, None


def _params():
    return [Kn.Parameter(1.3, name="variance"), Kn.Parameter(0.7, name="lengthscales"), Kn.Gaussian().variance]


def _rows(rng, B, D, failed):
    outs = rng.standard_normal((B, D, 16))
    outs[:, :, 8] = 0.0
    for b, d in failed:
        outs[b, d, 8] = float(rng.integers(1, 1000))
    return outs


@pytest.mark.parametrize("D", [1, 3])
def test_gpr_1d_batch_rows_match_inline_code(monkeypatch, D):
    rng = np.random.default_rng(D)
    B, n = 7, 12345.0
    outs = _rows(rng, B, D, [(2, D - 1), (5, 0)])
    monkeypatch.setattr(ops, "elbo_grad_1d_batched", lambda *a, **k: torch.from_numpy(outs.copy()))
    model = GPR_1d.__new__(GPR_1d)
    model.kernel, model.likelihood, model.inducing_features, model.basis, model._chunks = Kn.Matern32(), Kn.Gaussian(), \
        _FakeFeatures(), None, 0
    model._accs = [torch.zeros(10, dtype=torch.float64) for _ in range(D)]
    model._acc, model._scal = model._accs[0], torch.tensor([0.0, n], dtype=torch.float64)
    U = rng.standard_normal((B, 3))
    loss, grad, info = model.training_loss_and_gradients_batch(U)

    params = model.trainable_variables
    vals = np.array([[p.value_at(float(u)) for p, u in zip(params, row)] for row in U])
    for b in range(B):              # the loop of GPR_1d.training_loss_and_gradients_batch at d914e60
        out = _frozen_1d(outs[b], vals[b, 0], vals[b, 2], n)
        if out[8] != 0:
            assert loss[b] == np.inf and np.isnan(grad[b]).all() and info[b] == int(out[8])
            continue
        grads = gpr._grad_dict([(params[0], out[1]), (params[1], out[2]), (params[2], out[3])])
        assert info[b] == 0 and loss[b] == -float(out[0])
        assert np.array_equal(grad[b], [-(grads[id(p)] * p.dvalue_dunconstrained_at(float(u))) for p, u in zip(params, U[b])])
    assert info[2] != 0 and info[5] != 0


def test_many_series_rows_match_inline_code(monkeypatch):
    rng = np.random.default_rng(7)
    counts = np.array([5, 0, 3, 0, 0, 8, 2, 1])
    S = counts.size
    table = _rows(rng, S, 1, [(2, 0), (6, 0)])[:, 0]          # the bound row of every series
    calls = []

    def fake_batched(Kuu, dKuu, acc, basis, variances, sigma2s, chunks=0, rows=None):
        calls.append(np.asarray(rows).copy())
        return torch.from_numpy(table[np.asarray(rows)].copy()).view(-1, 1, 16)

    monkeypatch.setattr(ops, "elbo_grad_1d_batched", fake_batched)
    model = GPR_1d_many.__new__(GPR_1d_many)
    model._counts, model._params, model.inducing_features = counts, _params(), _FakeFeatures()
    model.kernel, model.basis, model._chunks, model._acc = Kn.Matern32(), None, 0, None
    ids = np.array([0, 1, 2, 3, 5, 6, 7, 4])
    U = rng.standard_normal((ids.size, 3))
    loss, grad, info = model._evaluate(U, ids)

    live = np.flatnonzero(counts[ids] > 0)
    assert np.array_equal(np.concatenate(calls), ids[live])
    want_loss, want_grad, want_info = np.zeros(ids.size), np.zeros((ids.size, 3)), np.zeros(ids.size, dtype=np.int64)
    for i, b in enumerate(live):    # the loop of GPR_1d_many._evaluate at d914e60
        o = table[ids[b]]
        if o[8] != 0:
            want_loss[b], want_grad[b], want_info[b] = np.inf, np.nan, int(o[8])
            continue
        want_loss[b] = -float(o[0])
        want_grad[b] = [-(o[1 + j] * p.dvalue_dunconstrained_at(float(u))) for j, (p, u) in enumerate(zip(model._params, U[b]))]
    assert np.array_equal(loss, want_loss) and np.array_equal(info, want_info)
    assert np.array_equal(grad, want_grad, equal_nan=True)
    assert (info != 0).sum() == 2 and (loss[counts[ids] == 0] == 0).all()


# ---- constructor input checks, all before any device work -------------------------------------------------------------------
def _data_2d(n=50, cols=1, outside=False):
    rng = np.random.default_rng(3)
    X = rng.uniform(0.5, 9.5, (n, 2))
    if outside:
        X[7, 1] = 10.5
    y = rng.standard_normal((n, cols)) if cols != 1 else rng.standard_normal(n)
    return X, y


def _bases(d):
    return [B.B3Spline(0, 10, 10) for _ in range(d)]


@pytest.mark.parametrize("make,err", [
    (lambda: GPR_1d((np.array([[0.5], [10.5]]), np.zeros(2)), Kn.Matern32(), _bases(1)[0]), AssertionError),
    (lambda: GPR_1d_many((np.array([[0.5], [10.5]]), np.zeros(2)), [0, 2], Kn.Matern32(), _bases(1)[0]), AssertionError),
    (lambda: GPR_1d_many((np.array([[0.5], [1.5]]), np.zeros((2, 2))), [0, 2], Kn.Matern32(), _bases(1)[0]), NotImplementedError),
    (lambda: GPR_kron(_data_2d(outside=True), [Kn.Matern32(), Kn.Matern32()], _bases(2)), AssertionError),
    (lambda: GPR_kron(_data_2d(cols=ops.MAX_RHS + 1), [Kn.Matern32(), Kn.Matern32()], _bases(2)), ValueError),
    (lambda: GPR_kron((_data_2d()[0], np.zeros((50, 0))), [Kn.Matern32(), Kn.Matern32()], _bases(2)), ValueError),
    (lambda: GPR_kron(_data_2d(cols=2), [Kn.Matern32(), Kn.Matern32()], _bases(2), method="band"), NotImplementedError),
    (lambda: GPR_additive(_data_2d(outside=True), [Kn.Matern32(), Kn.Matern12()], _bases(2)), AssertionError),
    (lambda: GPR_additive(_data_2d(cols=ops.MAX_RHS + 1), [Kn.Matern32(), Kn.Matern12()], _bases(2)), ValueError),
])
def test_constructor_checks_come_before_device_work(make, err):
    with pytest.raises(err):
        make()
