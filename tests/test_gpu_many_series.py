"""Many independent 1-D series on one basis (asvgp_accum_1d_segmented_typed, asvgp_elbo_grad_1d_batched_rows,
asvgp_posterior_1d_batched, asvgp_predict_1d_segmented, GPR_1d_many): every series gets what the single-series entry points and
GPR_1d give on its slice alone."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
CHECKED = list(range(9)) + [15]         # slots 9..14 are each evaluation's own clock diagnostics
TILE = 32 * 8 * 2                        # points of one float64 warp tile


def _series(sizes, m, seed, shuffle=False):
    """Concatenated ragged series on [0, m]: each sorted (or shuffled within itself), with its own signal."""
    rng = np.random.default_rng(seed)
    xs, ys = [], []
    for s, n in enumerate(sizes):
        x = np.sort(rng.uniform(0.0, m, n))
        if shuffle:
            x = rng.permutation(x)
        xs.append(x)
        ys.append(np.sin(x / (3.0 + s % 7)) + 0.3 * rng.standard_normal(n) + 0.1 * s)
    offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    return np.concatenate(xs) if xs else np.zeros(0), np.concatenate(ys) if ys else np.zeros(0), offsets


def _ragged_sizes(S, seed):
    rng = np.random.default_rng(seed)
    sizes = rng.integers(0, 3 * TILE, S)
    special = [0, 1, 0, 31, TILE - 1, 2 * TILE + 5, 1, 0]
    sizes[: min(S, len(special))] = special[:S] if S > 1 else [5000]
    return sizes


def _check_segmented(x, y, offsets, basis, acc):
    from asvgp_b200 import ops

    acc = acc.cpu().numpy()
    k, m = basis.order, basis.m
    for s in range(len(offsets) - 1):
        lo, hi = offsets[s], offsets[s + 1]
        ref = ops.accum_1d(x[lo:hi], y[lo:hi], basis).cpu().numpy() if hi > lo else np.zeros(acc.shape[1])
        G, G0 = acc[s, : (k + 2) * m], ref[: (k + 2) * m]
        scale = max(np.abs(G0).max(), 1.0)
        np.testing.assert_allclose(G, G0, rtol=1e-10, atol=1e-10 * scale, err_msg="series %d" % s)
        assert abs(acc[s, -2] - ref[-2]) <= 1e-10 * max(abs(ref[-2]), 1e-300), s
        assert acc[s, -1] == hi - lo, s


@pytest.mark.parametrize("S", [1, 3, 64, 1000])
def test_segmented_accumulate_ragged(cuda, S):
    from asvgp_b200 import basis as B, ops

    m = 200
    x, y, offsets = _series(_ragged_sizes(S, S), m, seed=S)
    basis = B.B3Spline(-1, m + 1, m)
    acc = ops.accum_1d_segmented(ops.to_device(x), ops.to_device(y), offsets, basis)
    _check_segmented(ops.to_device(x), ops.to_device(y), offsets, basis, acc)


@pytest.mark.parametrize("k", [1, 2, 3, 4, 5, 6])
@pytest.mark.parametrize("types", ["ff", "fs", "sf", "ss"])
def test_segmented_accumulate_orders_and_types(cuda, k, types):
    import torch

    from asvgp_b200 import basis as B, ops

    m = 300
    x, y, offsets = _series(_ragged_sizes(40, 7 * k), m, seed=11 * k)
    basis = getattr(B, "B%dSpline" % k)(-1, m + 1, m)
    dt = {"f": torch.float64, "s": torch.float32}
    xd, yd = ops.to_device(x).to(dt[types[0]]), ops.to_device(y).to(dt[types[1]])
    acc = ops.accum_1d_segmented(xd, yd, offsets, basis)
    _check_segmented(xd, yd, offsets, basis, acc)
    # misaligned views: the scalar-load path
    xm, ym = torch.cat([xd[:1], xd])[1:], torch.cat([yd[:1], yd])[1:]
    assert xm.data_ptr() % 16 and ym.data_ptr() % 16
    _check_segmented(xd, yd, offsets, basis, ops.accum_1d_segmented(xm, ym, offsets, basis))


def test_segmented_accumulate_shuffled_within_series(cuda):
    from asvgp_b200 import basis as B, ops

    m = 500
    x, y, offsets = _series(_ragged_sizes(64, 5), m, seed=5, shuffle=True)
    basis = B.B3Spline(-1, m + 1, m)
    acc = ops.accum_1d_segmented(ops.to_device(x), ops.to_device(y), offsets, basis)
    _check_segmented(ops.to_device(x), ops.to_device(y), offsets, basis, acc)


def test_segmented_accumulate_long_series_among_short_ones(cuda):
    from asvgp_b200 import basis as B, ops

    m = 1000
    sizes = np.array([3, 0, 100, 10_000_000, 1, 700, 0, 40_000])
    x, y, offsets = _series(sizes, m, seed=21)
    basis = B.B3Spline(-1, m + 1, m)
    acc = ops.accum_1d_segmented(ops.to_device(x), ops.to_device(y), offsets, basis)
    _check_segmented(ops.to_device(x), ops.to_device(y), offsets, basis, acc)


# ---- bound, posterior, predictor per row ---------------------------------------------------------------------------------
def _many(S=6, m=400, n_per=20_000, seed=3):
    from asvgp_b200 import basis as B, ops

    sizes = np.full(S, n_per)
    x, y, offsets = _series(sizes, m, seed)
    basis = B.B3Spline(-1, m + 1, m)
    return basis, ops.accum_1d_segmented(ops.to_device(x), ops.to_device(y), offsets, basis), (x, y, offsets)


def _settings(B, seed):
    rng = np.random.default_rng(seed)
    return rng.uniform(0.5, 2.0, B), rng.uniform(0.6, 4.0, B), rng.uniform(0.05, 0.6, B)


def _single(basis, kern, acc, v, l, s2):
    from asvgp_b200 import ops
    from asvgp_b200.inducing_features import SplineFeatures1D

    terms = SplineFeatures1D(kern, basis)._terms(kern, l, v)
    Kuu, dKuu = ops.kuu_assemble(basis, [t[0] for t in terms], [t[1] for t in terms], [t[2] for t in terms])
    return ops.elbo_grad_1d_single_stream(Kuu, dKuu, acc, basis, v, s2).cpu().numpy()


def test_rows_bound_bitwise_permuted_and_repeated(cuda):
    from asvgp_b200 import kernels as Kn, ops
    from asvgp_b200.inducing_features import SplineFeatures1D

    basis, acc, _ = _many()
    kern = Kn.Matern52()
    feats = SplineFeatures1D(kern, basis)
    rows = np.array([5, 0, 3, 3, 1, 5, 2, 4, 0, 2, 1])
    v, l, s2 = _settings(rows.size, 1)
    Kuu, dKuu = feats.make_Kuu_device_batched(kern, l, v)
    out = ops.elbo_grad_1d_batched(Kuu, dKuu, acc, basis, v, s2, rows=rows).cpu().numpy()
    for b, r in enumerate(rows):
        np.testing.assert_array_equal(out[b, 0, CHECKED], _single(basis, kern, acc[r], v[b], l[b], s2[b])[CHECKED], err_msg=str(b))
    # every row 0: the batched call of one accumulator
    zero = ops.elbo_grad_1d_batched(Kuu, dKuu, acc, basis, v, s2, rows=np.zeros(rows.size, dtype=np.int64)).cpu().numpy()
    ref = ops.elbo_grad_1d_batched(Kuu, dKuu, acc[0].contiguous(), basis, v, s2).cpu().numpy()
    np.testing.assert_array_equal(zero[:, :, CHECKED], ref[:, :, CHECKED])


def _snelson_with_others(golden):
    """Snelson as series 2 of five on the Snelson basis (others: shifted copies with noise)."""
    from asvgp_b200 import basis as B, ops

    g = golden("snelson")
    X, Y = g["X"].reshape(-1), g["y"].reshape(-1)
    rng = np.random.default_rng(4)
    xs = [X, X, X, X, X]
    ys = [Y + 0.2 * rng.standard_normal(Y.size), -Y, Y, 0.5 * Y, Y + 1.0]
    order = np.argsort(X, kind="stable")
    x = np.concatenate([xx[order] for xx in xs])
    y = np.concatenate([yy[order] for yy in ys])
    offsets = np.arange(6, dtype=np.int64) * X.size
    basis = B.B3Spline(-3.5, 10.5, 100)
    return basis, ops.accum_1d_segmented(ops.to_device(x), ops.to_device(y), offsets, basis), g


def _failing_setting(basis, acc):
    from asvgp_b200 import kernels as Kn

    for kind in ("Matern52", "Matern32"):
        kern = getattr(Kn, kind)()
        for ell in (1e2, 1e3, 1e4, 1e5, 1e6):
            if _single(basis, kern, acc, 1.0, ell, 0.1)[8] != 0:
                return kind, ell
    raise AssertionError("no failing setting found")


def test_rows_bound_failed_slot_keeps_the_others(cuda, golden):
    from asvgp_b200 import kernels as Kn, ops
    from asvgp_b200.inducing_features import SplineFeatures1D

    basis, acc, _ = _snelson_with_others(golden)
    kind, ell = _failing_setting(basis, acc[2])
    kern = getattr(Kn, kind)()
    feats = SplineFeatures1D(kern, basis)
    rows = np.array([0, 1, 2, 3, 4])
    v, l, s2 = _settings(5, 8)
    good = ops.elbo_grad_1d_batched(*feats.make_Kuu_device_batched(kern, l, v), acc, basis, v, s2, rows=rows).cpu().numpy()
    l[2], v[2], s2[2] = ell, 1.0, 0.1
    out = ops.elbo_grad_1d_batched(*feats.make_Kuu_device_batched(kern, l, v), acc, basis, v, s2, rows=rows).cpu().numpy()
    assert out[2, 0, 8] != 0 and out[2, 0, 8] == _single(basis, kern, acc[2], v[2], l[2], s2[2])[8]
    for b in (0, 1, 3, 4):
        np.testing.assert_array_equal(out[b, 0, CHECKED], good[b, 0, CHECKED])


def test_batched_posterior_bitwise_and_failed_slot(cuda, golden):
    from asvgp_b200 import kernels as Kn, ops
    from asvgp_b200.inducing_features import SplineFeatures1D

    basis, acc, _ = _snelson_with_others(golden)
    kind, ell = _failing_setting(basis, acc[2])
    kern = getattr(Kn, kind)()
    feats = SplineFeatures1D(kern, basis)
    rows = np.array([4, 2, 0, 2, 1, 3])
    v, l, s2 = _settings(rows.size, 9)
    l[3], v[3], s2[3] = ell, 1.0, 0.1
    Kuu, _ = feats.make_Kuu_device_batched(kern, l, v, want_grad=False)
    alpha, S, info = (t.cpu().numpy() for t in ops.posterior_1d_batched(Kuu, acc, basis, s2, rows))
    for b, r in enumerate(rows):
        a1, S1, i1 = (t.cpu().numpy() for t in ops.posterior_1d(Kuu[b].contiguous(), acc[r].contiguous(), basis, s2[b]))
        np.testing.assert_array_equal(info[b], i1)
        if b != 3:
            np.testing.assert_array_equal(alpha[b], a1, err_msg=str(b))
            np.testing.assert_array_equal(S[b], S1, err_msg=str(b))
    assert info[3].any() and not np.delete(info, 3, axis=0).any()


def test_segmented_predictor_matches_predict_1d(cuda):
    import torch

    from asvgp_b200 import ops
    from asvgp_b200.inducing_features import SplineFeatures1D
    from asvgp_b200 import kernels as Kn

    basis, acc, _ = _many(S=5)
    kern = Kn.Matern32()
    feats = SplineFeatures1D(kern, basis)
    v, l, s2 = _settings(5, 2)
    Kuu, _ = feats.make_Kuu_device_batched(kern, l, v, want_grad=False)
    alpha, S, info = ops.posterior_1d_batched(Kuu, acc, basis, s2, np.arange(5))
    assert not info.any().item()
    rng = np.random.default_rng(3)
    sizes = [1000, 0, 1, 2500, 37]              # an empty test segment and a single point
    xs = [np.sort(rng.uniform(-0.5, basis.m + 0.5, n)) for n in sizes]
    offsets = np.concatenate([[0], np.cumsum(sizes)])
    xnew = np.concatenate(xs)
    mean, var = (t.cpu().numpy() for t in ops.predict_1d_segmented(xnew, offsets, basis, alpha, S, torch.tensor(v)))
    for s in range(5):
        lo, hi = offsets[s], offsets[s + 1]
        if hi == lo:
            continue
        m1, v1 = (t.cpu().numpy() for t in ops.predict_1d(xs[s], basis, alpha[s], S[s], v[s]))
        np.testing.assert_allclose(mean[lo:hi], m1, rtol=1e-12, atol=1e-12 * np.abs(m1).max())
        np.testing.assert_allclose(var[lo:hi], v1, rtol=1e-12, atol=1e-12 * np.abs(v1).max())


# ---- the model -------------------------------------------------------------------------------------------------------------
def test_model_matches_gpr_1d_per_series(cuda):
    from asvgp_b200 import basis as B, kernels as Kn
    from asvgp_b200.gpr import GPR_1d, GPR_1d_many

    m = 300
    sizes = np.array([5000, 0, 800, 12_000, 1, 70])
    x, y, offsets = _series(sizes, m, seed=17)
    basis = B.B3Spline(-1, m + 1, m)
    U0 = np.random.default_rng(2).uniform(-1.0, 1.0, (sizes.size, 3))
    model = GPR_1d_many((x.reshape(-1, 1), y), offsets, Kn.Matern52(), basis, U0=U0)
    loss, grad, info = model.training_loss_and_gradients()
    assert (info == 0).all()
    np.testing.assert_array_equal(model.elbo(), -loss)
    xnew = np.linspace(-0.5, m + 0.5, 333)
    off_new = np.arange(sizes.size + 1) * xnew.size
    mean, var = model.predict_f(np.tile(xnew, sizes.size).reshape(-1, 1), off_new)
    for s in range(sizes.size):
        lo, hi = offsets[s], offsets[s + 1]
        sl = slice(s * xnew.size, (s + 1) * xnew.size)
        if hi == lo:
            assert loss[s] == 0 and (grad[s] == 0).all()
            assert (mean[sl] == 0).all() and np.allclose(var[sl], model.variance[s], rtol=1e-14)
            continue
        ref = GPR_1d((x[lo:hi].reshape(-1, 1), y[lo:hi].reshape(-1, 1)), Kn.Matern52(), basis)
        for p, u in zip(ref.trainable_variables, U0[s]):
            p.unconstrained = float(u)
        l1, g1 = ref.training_loss_and_gradients()
        assert abs(loss[s] - l1) <= 1e-10 * abs(l1), s
        np.testing.assert_allclose(grad[s], g1, rtol=1e-8, atol=1e-8 * np.abs(g1).max())
        m1, v1 = ref.predict_f(xnew.reshape(-1, 1))
        np.testing.assert_allclose(mean[sl], m1, rtol=1e-10, atol=1e-10 * np.abs(m1).max())
        np.testing.assert_allclose(var[sl], v1, rtol=1e-10, atol=1e-10 * np.abs(v1).max())
    np.testing.assert_allclose(model.variance, [Kn._softplus(u) for u in U0[:, 0]], rtol=1e-15)


def test_optimize_iterates_equal_serial_runs(cuda):
    import scipy.optimize

    from asvgp_b200 import kernels as Kn
    from asvgp_b200.gpr import GPR_1d_many
    from asvgp_b200.kernels import Gaussian, Parameter

    basis, _, (x, y, offsets) = _many(S=2, m=200, n_per=30_000, seed=8)
    U0 = np.array([[0.2, 1.0, -1.0], [-0.5, 0.5, 0.0]])
    model = GPR_1d_many((x, y), offsets, Kn.Matern32(), basis, U0=U0)
    results = model.optimize()
    params = [Parameter(1.0), Parameter(1.0), Gaussian().variance]
    kern = Kn.Matern32()
    for s in range(2):
        acc = model._acc[s]

        def fun(u):
            vals = [p.value_at(float(ui)) for p, ui in zip(params, u)]
            out = _single(basis, kern, acc, vals[0], vals[1], vals[2])
            return -float(out[0]), np.array([-(out[1 + j] * p.dvalue_dunconstrained_at(float(u[j]))) for j, p in enumerate(params)])

        ref = scipy.optimize.minimize(fun, U0[s], jac=True, method="L-BFGS-B")
        np.testing.assert_array_equal(results[s].x, ref.x)
        assert (results[s].nit, results[s].nfev, results[s].fun) == (ref.nit, ref.nfev, ref.fun)
        np.testing.assert_array_equal(model.U[s], ref.x)


def test_eight_snelsons_reach_the_notebook_optimum(cuda, golden):
    from asvgp_b200 import basis as B, kernels as Kn
    from asvgp_b200.gpr import GPR_1d_many

    g = golden("snelson")
    X, Y = g["X"].reshape(-1), g["y"].reshape(-1)
    order = np.argsort(X, kind="stable")
    x, y = np.tile(X[order], 8), np.tile(Y[order], 8)
    offsets = np.arange(9, dtype=np.int64) * X.size
    model = GPR_1d_many((x.reshape(-1, 1), y), offsets, Kn.Matern32(), B.B3Spline(-3.5, 10.5, 100))
    results = model.optimize(wave=5)
    assert all(r.success for r in results)
    elbo = model.elbo()
    assert np.abs(elbo - float(g["notebook_elbo"])).max() < 1e-6
    assert np.abs(np.array([-r.fun for r in results]) - float(g["notebook_elbo"])).max() < 1e-6
