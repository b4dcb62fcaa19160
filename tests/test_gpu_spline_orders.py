"""Every spline order k = 1..6 of the 2-D Kronecker, 1-D and additive kernels against the CPU oracle.

Each order is its own template instantiation (ASVGP_DISPATCH_ORDER) with its own registers, spills, shared-memory footprint
and table sizes, so an order the suite runs without a reference is an order that can be wrong unnoticed.  Covered here:
  * 2-D accumulate: every input class of the on-device probe (separable raster detected and stated, curvilinear raster with
    256-bit and per-point loads, x1 runs, scattered points, float32 data on the column sweep) vs O.precompute_kron;
  * 2-D bound: ELBO and five gradients vs the dense autograd oracle on a small mesh, and vs the LAPACK-band oracle plus
    4th-order differences on a 40 x 36 mesh with a multi-level front tree; the nested-dissection and scalar-band
    factorisations against each other;
  * 2-D predictor (table, column-sweep and per-point kernels): scattered points, detected and stated rasters with ragged
    row lengths and row counts, n = 1, 3, 5 (the 256-bit tail), knots and both domain ends vs O.predict_kron_banded;
  * 1-D: the k = 6 bound vs the dense autograd oracle; predict_1d at every order on sorted, shuffled and half-ordered
    points, knots, points outside [a, b], a misaligned device view (scalar path) and sizes around the CTA-range edges;
  * GPR_additive: Gram, projection, bound, 2 D + 1 gradients and predictions for D = 2 and 8, n = 1, 31, 33, 4097, with
    sorted and shuffled first coordinates.
Valid kernel / order pairs follow the reference tables: Matern12 for every order, Matern32 from k = 2, Matern52 for
k = 3, 4, 5 (B6Spline defines no BC_ggrad).  Length-scales are 1.5 to 2.5 knot spacings unless a case says otherwise."""
import functools

import numpy as np
import pytest
import scipy.linalg as sla

from oracle import asvgp_oracle as O

pytestmark = pytest.mark.gpu
ORDERS = (1, 2, 3, 4, 5, 6)
DOMAINS = ((-80, -25), (15, 55))


def _kinds(k):
    """Matern kinds the reference tables of order k support, lowest first."""
    return ["Matern12"] + (["Matern32"] if k >= 2 else []) + (["Matern52"] if 3 <= k <= 5 else [])


def _bases_2d(k, ms):
    from asvgp_b200 import basis as B

    cls = getattr(B, "B%dSpline" % k)
    return [cls(DOMAINS[0][0], DOMAINS[0][1], ms[0]), cls(DOMAINS[1][0], DOMAINS[1][1], ms[1])]


def _kron_model(X, y, k, ms, s2=0.05, **kw):
    """GPR_kron with the highest kernel order k allows in dimension 1 and the next lower one in dimension 2 (Matern12 twice
    at k = 1), length-scales 2 and 1.5 knot spacings.  Returns (model, kinds, hypers)."""
    from asvgp_b200 import kernels as Kn
    from asvgp_b200.gpr import GPR_kron

    bases = _bases_2d(k, ms)
    kinds = _kinds(k)
    kinds = (kinds[-1], kinds[-2] if len(kinds) > 1 else kinds[-1])
    hyp = [(0.9, 2.0 * bases[0].delta), (1.2, 1.5 * bases[1].delta)]
    kerns = [getattr(Kn, kind)(variance=v, lengthscales=l) for kind, (v, l) in zip(kinds, hyp)]
    model = GPR_kron((X, y.reshape(-1, 1)), kerns, bases, **kw)
    model.likelihood.variance.assign(s2)
    return model, kinds, hyp


def _target(X, rng):
    return np.sin(X[:, 0] / 4.0) * np.cos(X[:, 1] / 3.0) + 0.05 * rng.standard_normal(X.shape[0])


def _scattered_2d(n, rng):
    return np.stack([rng.uniform(-79.9, -25.1, n), rng.uniform(15.1, 54.9, n)], 1)


def _small_ms(k):
    """A small rectangular mesh for the dense oracles (M = m1 m2 <= 304); m >= 2 (k + 1) as the reference requires."""
    m1 = max(10, 2 * k + 4)
    return m1, m1 + 3


# ---------------------------------------------------------------------------------------------------------------------
# 2-D accumulate
# ---------------------------------------------------------------------------------------------------------------------
ACCUM_VARIANTS = {          # variant -> (n1, n2, path selected by the probe)
    "separable": (60, 131, (4,)),
    "separable-stated": (60, 131, None),
    "curvilinear-vec": (61, 132, (3,)),
    "curvilinear": (59, 131, (2,)),
    "x1-runs": (67, 129, (1,)),
    "scattered": (0, 0, (0,)),
    "float32-sweep": (60, 131, (4,)),
}


@pytest.mark.parametrize("variant", list(ACCUM_VARIANTS))
@pytest.mark.parametrize("k", ORDERS)
def test_accumulate_every_input_class(cuda, k, variant):
    import torch

    from asvgp_b200 import ops, utils

    n1, n2, want = ACCUM_VARIANTS[variant]
    rng = np.random.default_rng(100 * k + len(variant))
    ms = (19, 23)
    bases = _bases_2d(k, ms)
    if variant == "scattered":
        X = _scattered_2d(7919, rng)
    else:
        x1 = np.sort(rng.uniform(-79.9, -25.1, n1))
        x2 = np.sort(rng.uniform(15.1, 54.9, n2))
        X = np.stack(np.meshgrid(x1, x2, indexing="ij"), -1)
        if variant.startswith("curvilinear"):
            X[:, :, 1] += 0.01 * np.sin(np.arange(n1))[:, None]            # x2 depends on the row
        X = X.reshape(-1, 2)
        if variant == "x1-runs":
            X = X[rng.uniform(size=X.shape[0]) > 0.1]                      # rows of different lengths
    y = _target(X, rng)
    Xa, ya = X, y
    if variant == "float32-sweep":
        Xa, ya = X.astype(np.float32), y.astype(np.float32)
        X, y = Xa.astype(np.float64), ya.astype(np.float64)                # the model of the float64-converted data
    Xd, yd = torch.from_numpy(Xa).cuda(), torch.from_numpy(ya).cuda()
    acc = torch.zeros(ops.accum_size_2d(bases), dtype=torch.float64, device="cuda")
    cm = ops.moment_table_2d(bases)
    stated = n2 if variant == "separable-stated" else None
    ops.accum_2d(Xd, yd, bases, cm, ops.split_accum_2d(acc, bases)[2], raster_row_len=stated)
    if want is not None:
        select = int(cm[-1:].view(torch.int32)[0].item())
        assert select in want, "probe chose path %d for a %s input" % (select, variant)
    ops.expand_moments_2d(cm, bases, acc)
    Gs, b, scal = [t.cpu().numpy() for t in ops.split_accum_2d(acc, bases)]
    G0, b0, yy0 = O.precompute_kron([bb.mesh for bb in bases], [bb.delta for bb in bases], k, list(ms), X, y)
    scale = abs(G0).max()
    assert abs(utils.stencil_to_sparse(Gs, ms[0], ms[1], k) - G0).max() <= 1e-11 * scale
    np.testing.assert_allclose(b, b0.ravel(), rtol=0, atol=1e-11 * np.abs(b0).max())
    assert abs(scal[0] - yy0) <= 1e-12 * yy0 and scal[1] == X.shape[0]


# ---------------------------------------------------------------------------------------------------------------------
# 2-D bound and predictor on a small mesh (dense oracles)
# ---------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _small_kron_case(k):
    rng = np.random.default_rng(7 + k)
    ms = _small_ms(k)
    X = _scattered_2d(6000, rng)
    y = _target(X, rng)
    bases = _bases_2d(k, ms)
    meshes, deltas = [b.mesh for b in bases], [b.delta for b in bases]
    G0, b0, yy0 = O.precompute_kron(meshes, deltas, k, list(ms), X, y)
    return X, y, ms, meshes, deltas, G0, b0, yy0


@pytest.mark.parametrize("k", ORDERS)
def test_kron_bound_small_mesh_vs_dense_oracle(cuda, k):
    X, y, ms, meshes, deltas, G0, b0, yy0 = _small_kron_case(k)
    model, kinds, hyp = _kron_model(X, y, k, ms)
    assert abs(model.KufKfu_sparse - G0).max() <= 1e-10 * abs(G0).max()
    T = [O.static_bands(k, m, d) for m, d in zip(ms, deltas)]
    e0, g0 = O.elbo_grad_kron_dense(kinds, T, G0, b0, yy0, X.shape[0], hyp, 0.05)
    assert abs(model.elbo() - e0) <= 1e-10 * abs(e0)
    elbo, grads = model.elbo_and_grad()
    assert abs(elbo - e0) <= 1e-10 * abs(e0)
    got = np.array([grads[id(p)] for p in model.trainable_variables])
    np.testing.assert_allclose(got, g0, rtol=1e-8, atol=1e-8 * np.abs(g0).max())


def _predict_inputs_2d(bases, rng):
    """name -> (Xnew, raster_shape or None)."""
    (a1, b1), (a2, b2) = DOMAINS
    g1, g2 = np.linspace(a1 + 0.3, b1 - 0.3, 37), np.linspace(a2 + 0.3, b2 - 0.3, 53)
    h1, h2 = np.linspace(a1 + 0.7, b1 - 0.7, 29), np.linspace(a2 + 0.2, b2 - 0.2, 45)
    k1, k2 = np.asarray(bases[0].mesh), np.asarray(bases[1].mesh)
    knots = np.stack(np.meshgrid(k1, k2, indexing="ij"), -1).reshape(-1, 2)
    corners = np.array([[a1, a2], [a1, b2], [b1, a2], [b1, b2]], dtype=np.float64)
    edges = np.concatenate([np.stack([np.full(9, a1), rng.uniform(a2, b2, 9)], 1), np.stack([np.full(9, b1), rng.uniform(a2, b2, 9)], 1),
                            np.stack([rng.uniform(a1, b1, 9), np.full(9, a2)], 1), np.stack([rng.uniform(a1, b1, 9), np.full(9, b2)], 1)])
    return {
        "scattered": (_scattered_2d(300, rng), None),
        # detected raster: the column sweep, 37 rows = four 8-row blocks and a 5-row tail
        "raster-detected": (np.stack(np.meshgrid(g1, g2, indexing="ij"), -1).reshape(-1, 2), None),
        # stated raster: 45 columns (not a multiple of 32), 29 rows (not a multiple of 8)
        "raster-stated": (np.stack(np.meshgrid(h1, h2, indexing="ij"), -1).reshape(-1, 2), (29, 45)),
        "n1": (_scattered_2d(1, rng), None),
        "n3": (_scattered_2d(3, rng), None),
        "n5": (_scattered_2d(5, rng), None),
        "knots-raster": (knots, None),
        "knots-shuffled": (np.concatenate([knots[rng.permutation(knots.shape[0])], corners]), None),
        "domain-ends": (np.concatenate([corners, edges]), None),
    }


# absolute tolerance on the predictive variance of the small-mesh cases.  At k = 6 that mesh gives cond(P) = 6e14: moving
# the band entries of P by one ulp of max|P| (three draws) moves LAPACK's variance by 6e-7 ... 8e-7 and its mean by
# 4e-6 ... 1e-5, and the variance of one knot point has been seen 1.9e-9 from the oracle between runs whose fp64 atomic
# sums differ in the last bits.  1e-8 stays far below that sensitivity; every other order and every mean keeps 1e-9.
VAR_TOL_SMALL = {6: 1e-8}


@pytest.mark.parametrize("k", ORDERS)
def test_kron_predict_small_mesh_vs_banded_oracle(cuda, k):
    X, y, ms, meshes, deltas, G0, b0, yy0 = _small_kron_case(k)
    model, kinds, hyp = _kron_model(X, y, k, ms)
    T = [O.static_bands(k, m, d) for m, d in zip(ms, deltas)]
    Ks = [O.make_Kuu(kind, l, v, t) for kind, (v, l), t in zip(kinds, hyp, T)]
    rng = np.random.default_rng(k)
    for name, (Xs, shape) in _predict_inputs_2d(model.bases, rng).items():
        mean, var = model.predict_f(Xs, raster_shape=shape)
        mean0, var0 = O.predict_kron_banded(meshes, deltas, k, list(ms), Ks, G0, b0, [h[0] for h in hyp], 0.05, Xs)
        np.testing.assert_allclose(mean, mean0, atol=1e-9, rtol=0, err_msg=name)
        np.testing.assert_allclose(var, var0, atol=VAR_TOL_SMALL.get(k, 1e-9), rtol=0, err_msg=name)


# ---------------------------------------------------------------------------------------------------------------------
# 2-D on a mid-size rectangular mesh: multi-level front tree, banded oracle, both factorisations
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 5, 6])
def test_kron_midsize_rectangular_vs_banded_oracle(cuda, k):
    rng = np.random.default_rng(40 + k)
    ms = (40, 36)
    n1, n2 = 150, 120
    x1, x2 = np.linspace(-79.5, -25.5, n1), np.linspace(15.5, 54.5, n2)
    X = np.stack(np.meshgrid(x1, x2, indexing="ij"), -1).reshape(-1, 2)
    y = _target(X, rng)
    s2 = 0.01
    model, kinds, hyp = _kron_model(X, y, k, ms, s2=s2)
    from asvgp_b200 import ops

    assert int(ops.kron_plan_info(ms[0], ms[1], k)["levels"]) >= 3              # a multi-level front tree
    meshes, deltas = [b.mesh for b in model.bases], [b.delta for b in model.bases]
    G0, b0, yy0 = O.precompute_kron(meshes, deltas, k, list(ms), X, y)
    assert abs(model.KufKfu_sparse - G0).max() <= 1e-10 * abs(G0).max()
    np.testing.assert_allclose(model.Kuf_y, b0, rtol=1e-10, atol=1e-10 * np.abs(b0).max())
    T = [O.static_bands(k, m, d) for m, d in zip(ms, deltas)]

    def f(th):
        Ks = [O.make_Kuu(kinds[0], th[1], th[0], T[0]), O.make_Kuu(kinds[1], th[3], th[2], T[1])]
        return O.elbo_kron_banded(Ks, G0, b0, yy0, X.shape[0], [th[0], th[2]], th[4], k, list(ms))

    th0 = np.array([hyp[0][0], hyp[0][1], hyp[1][0], hyp[1][1], s2])
    want = f(th0)
    assert abs(model.elbo() - want) <= 1e-10 * abs(want)
    e, grads = model.elbo_and_grad()
    assert abs(e - want) <= 1e-10 * abs(want)
    got = np.array([grads[id(p)] for p in model.trainable_variables])
    for i in range(5):
        h = 1e-4 * th0[i]
        e_ = np.zeros(5); e_[i] = h
        fd = (-f(th0 + 2 * e_) + 8 * f(th0 + e_) - 8 * f(th0 - e_) + f(th0 - 2 * e_)) / (12 * h)
        assert abs(fd - got[i]) <= 1e-6 * max(1.0, abs(got[i])), (i, fd, got[i])
    Ks = [O.make_Kuu(kind, l, v, t) for kind, (v, l), t in zip(kinds, hyp, T)]
    for name, (Xs, shape) in _predict_inputs_2d(model.bases, rng).items():
        if name.startswith("knots"):
            continue                                 # 1440 x 1480 dense right-hand sides: covered on the small mesh
        mean, var = model.predict_f(Xs, raster_shape=shape)
        mean0, var0 = O.predict_kron_banded(meshes, deltas, k, list(ms), Ks, G0, b0, [h[0] for h in hyp], s2, Xs)
        np.testing.assert_allclose(mean, mean0, atol=1e-9, rtol=0, err_msg=name)
        np.testing.assert_allclose(var, var0, atol=1e-9, rtol=0, err_msg=name)


@pytest.mark.parametrize("k", [1, 6])
def test_nested_dissection_and_band_factorisations_agree(cuda, k):
    """The nested-dissection fronts (asvgp_kron_*) and the tile DAG over the scalar band (asvgp_kronband_*) at the lowest
    and highest order: bound, gradients, alpha and the stencil of P^-1."""
    import torch

    rng = np.random.default_rng(60 + k)
    X = _scattered_2d(30000, rng)
    y = _target(X, rng)
    Xd, yd = torch.from_numpy(X).cuda(), torch.from_numpy(y).cuda()
    nd, _, _ = _kron_model(Xd, yd, k, (40, 36), s2=0.01)
    band, _, _ = _kron_model(Xd, yd, k, (40, 36), s2=0.01, method="band")
    e1, g1 = nd.elbo_and_grad()
    e2, g2 = band.elbo_and_grad()
    assert abs(e1 - e2) <= 1e-11 * abs(e1), (e1, e2)
    a = np.array([g1[id(p)] for p in nd.trainable_variables])
    b = np.array([g2[id(p)] for p in band.trainable_variables])
    np.testing.assert_allclose(a, b, rtol=1e-8, atol=1e-9 * np.abs(a).max())
    al1, S1, *_ = nd.posterior_weights()
    al1, S1 = al1.cpu().numpy().copy(), S1.cpu().numpy().copy()
    al2, S2, *_ = band.posterior_weights()
    np.testing.assert_allclose(S1, S2.cpu().numpy(), rtol=0, atol=5e-8 * np.abs(S1).max())
    np.testing.assert_allclose(al1, al2.cpu().numpy(), rtol=0, atol=1e-6 * np.abs(al1).max())


# ---------------------------------------------------------------------------------------------------------------------
# 1-D model
# ---------------------------------------------------------------------------------------------------------------------
def _model_1d(x, y, kind, k, a, b, m, hyp, chunks=0):
    from asvgp_b200 import basis as B, kernels as Kn
    from asvgp_b200.gpr import GPR_1d

    kern = getattr(Kn, kind)(variance=hyp[0], lengthscales=hyp[1])
    model = GPR_1d((x.reshape(-1, 1), y.reshape(-1, 1)), kern, getattr(B, "B%dSpline" % k)(a, b, m), chunks=chunks)
    model.likelihood.variance.assign(hyp[2])
    return model


@pytest.mark.parametrize("kind", ["Matern12", "Matern32"])
@pytest.mark.parametrize("chunks", [0, 5])
def test_bound_1d_order6_vs_dense_oracle(cuda, kind, chunks):
    rng = np.random.default_rng(66)
    m, n = 200, 40000
    x = np.sort(rng.uniform(0.0, m, n))
    y = np.sin(x / 7.0) + 0.3 * np.cos(x / 2.3) + 0.2 * rng.standard_normal(n)
    from asvgp_b200 import basis as B

    delta = B.B6Spline(-1, m + 1, m).delta
    hyp = (1.1, 2.0 * delta, 0.3)
    model = _model_1d(x, y, kind, 6, -1, m + 1, m, hyp, chunks=chunks)
    G0, b0, yy0 = O.precompute_1d(model.basis.mesh, model.basis.delta, 6, m, x, y)
    np.testing.assert_allclose(model.KufKfu, G0, rtol=0, atol=1e-10 * np.abs(G0).max())
    e0, g0 = O.elbo_grad_1d_dense(kind, O.static_bands(6, m, model.basis.delta), G0, b0, yy0, n, *hyp)
    elbo, grads = model.elbo_and_grad()
    assert abs(elbo - e0) <= 1e-10 * abs(e0)
    got = np.array([grads[id(p)] for p in model.trainable_variables])
    np.testing.assert_allclose(got, g0, rtol=1e-8, atol=1e-8 * np.abs(g0).max())


def _predict_1d_reference(mesh, delta, k, Kuu, G, b, var, s2, xs):
    """Mean and variance of the 1-D posterior at any xs from the oracle's pieces and LAPACK band factors; a point outside
    [a, b] takes the polynomial of the end interval it lies beyond (what the kernel does; the reference's feature matrix
    has no row for it).  Inside [a, b] this equals O.predict_1d (checked in the test); it needs O(n k^2) memory, not the
    dense m x n right-hand side of O.predict_1d, so it reaches n ~ 1e6."""
    mesh = np.asarray(mesh)
    cP = sla.cholesky_banded(G / s2 + Kuu, lower=True)
    cK = sla.cholesky_banded(Kuu, lower=True)
    alpha = sla.cho_solve_banded((cP, True), b).ravel() / s2
    S = O.takahashi_band(cP) - O.takahashi_band(cK)         # band of P^-1 - Kuu^-1
    idx, _ = O.locate(mesh, xs)
    idx = np.minimum(idx, mesh.size - 2)
    w = O.pieces(k, xs - mesh[idx], delta)
    mean = sum(w[r] * alpha[idx + r] for r in range(k + 1))
    v = np.full(xs.shape, float(var))
    for r in range(k + 1):
        v += w[r] * w[r] * S[0, idx + r]
        for s in range(r):
            v += 2.0 * w[r] * w[s] * S[r - s, idx + s]
    return mean, v


@functools.lru_cache(maxsize=None)
def _posterior_1d(k):
    """A fitted 1-D model of order k (the highest kernel it allows, length-scale 2 knot spacings) and its oracle pieces."""
    rng = np.random.default_rng(600 + k)
    a, b, m = 0.0, 30.0, 40
    x = np.sort(rng.uniform(a, b, 5000))
    y = np.sin(x) + 0.2 * rng.standard_normal(x.size)
    from asvgp_b200 import basis as B

    delta = getattr(B, "B%dSpline" % k)(a, b, m).delta
    kind = _kinds(k)[-1]
    hyp = (1.3, 2.0 * delta, 0.1)
    model = _model_1d(x, y, kind, k, a, b, m, hyp)
    G0, b0, _ = O.precompute_1d(model.basis.mesh, model.basis.delta, k, m, x, y)
    Kuu = O.make_Kuu(kind, hyp[1], hyp[0], O.static_bands(k, m, model.basis.delta))
    alpha, S, info = model.posterior_weights()
    assert not info.any().item()
    return model, alpha.clone(), S.clone(), (model.basis.mesh, model.basis.delta, k, Kuu, G0, b0, hyp[0], hyp[2])


def _predict_1d_inputs(name, basis, rng):
    a, b, delta = basis.a, basis.b, basis.delta
    if name == "sorted":
        return np.sort(rng.uniform(a, b, 20000))
    if name == "shuffled":
        return rng.uniform(a, b, 20001)
    if name == "every-5th-random":                  # lanes toggle between the interval cache and the direct evaluation
        xs = np.sort(rng.uniform(a, b, 20000))
        xs[::5] = rng.uniform(a, b, xs[::5].size)
        return xs
    if name == "knots-and-outside":
        mesh = np.asarray(basis.mesh)
        out = np.array([a - 0.7 * delta, a - 0.2 * delta, b + 0.2 * delta, b + 0.7 * delta])
        return np.concatenate([mesh, out, mesh[::-1], np.sort(np.concatenate([mesh, out]))])
    n = int(name[2:])                                # "n=<size>": sorted points, ragged CTA ranges
    return np.sort(rng.uniform(a, b, n))


PREDICT_1D_INPUTS = ["sorted", "shuffled", "every-5th-random", "knots-and-outside", "misaligned-view",
                     "n=8191", "n=8192", "n=8193", "n=%d" % (2 * 4096 * 148 - 1), "n=%d" % (2 * 4096 * 148 + 1)]


@pytest.mark.parametrize("case", PREDICT_1D_INPUTS)
@pytest.mark.parametrize("k", ORDERS)
def test_predict_1d_every_order(cuda, k, case):
    import torch

    from asvgp_b200 import ops

    model, alpha, S, ref = _posterior_1d(k)
    rng = np.random.default_rng(k * 31 + len(case))
    if case == "misaligned-view":
        xs = _predict_1d_inputs("shuffled", model.basis, rng)[:4097]
        buf = torch.from_numpy(np.concatenate([[0.0], xs])).cuda()
        xd = buf[1:]                                  # 8 bytes past a 16-byte boundary: the scalar path
        assert xd.data_ptr() % 16 == 8
    else:
        xs = _predict_1d_inputs(case, model.basis, rng)
        xd = torch.from_numpy(xs).cuda()
    mean, var = ops.predict_1d(xd, model.basis, alpha, S, ref[6])
    mean, var = mean.cpu().numpy(), var.cpu().numpy()
    mean0, var0 = _predict_1d_reference(*ref[:6], ref[6], ref[7], xs)
    np.testing.assert_allclose(mean, mean0, atol=1e-9, rtol=0)
    np.testing.assert_allclose(var, var0, atol=1e-9, rtol=0)
    if case in ("shuffled", "knots-and-outside"):
        # the reference of this file against the oracle's own predictor, inside [a, b]
        inside = xs[(xs >= model.basis.a) & (xs <= model.basis.b)][:3000]
        m1, v1 = O.predict_1d(ref[0], ref[1], k, model.basis.m, ref[3], ref[4], ref[5], ref[6], ref[7], inside)
        m2, v2 = _predict_1d_reference(*ref[:6], ref[6], ref[7], inside)
        np.testing.assert_allclose(m2, m1.ravel(), rtol=0, atol=1e-12)
        np.testing.assert_allclose(v2, v1.ravel(), rtol=0, atol=1e-12)
        mf, vf = model.predict_f(inside.reshape(-1, 1))            # and through the model API
        np.testing.assert_allclose(mf.ravel(), m1.ravel(), atol=1e-9, rtol=0)
        np.testing.assert_allclose(vf.ravel(), v1.ravel(), atol=1e-9, rtol=0)


# ---------------------------------------------------------------------------------------------------------------------
# GPR_additive
# ---------------------------------------------------------------------------------------------------------------------
def _additive_cases():
    out = []
    for k in ORDERS:
        for D in (2, 8):
            for n in (1, 31, 33, 4097):
                for order in (("sorted",) if n == 1 else ("sorted", "shuffled")):
                    out.append((k, D, n, order))
    return out


@pytest.mark.parametrize("k,D,n,order", _additive_cases())
def test_additive_every_order(cuda, k, D, n, order):
    from asvgp_b200 import basis as B, kernels as Kn
    from asvgp_b200.gpr import GPR_additive

    rng = np.random.default_rng(1000 * k + 10 * D + n)
    cls = getattr(B, "B%dSpline" % k)
    ms = [2 * k + 4 + 3 * d for d in range(D)]                    # a different m in every dimension
    doms = [(-d, 4 + 2 * d) for d in range(D)]
    bases = [cls(a, b, m) for (a, b), m in zip(doms, ms)]
    allowed = _kinds(k)
    kinds = [allowed[-1 - d % len(allowed)] for d in range(D)]     # the highest kernel in dimension 0
    hyp = [(0.5 + 0.1 * d, (1.5 + 0.125 * d) * bb.delta) for d, bb in enumerate(bases)]
    s2 = 0.05
    X = np.stack([rng.uniform(a + 1e-3, b - 1e-3, n) for a, b in doms], 1)
    if order == "sorted":
        X = X[np.argsort(X[:, 0])]                                 # long runs of the first coordinate's intervals
    y = np.sin(X).sum(1) + 0.1 * rng.standard_normal(n)
    kerns = [getattr(Kn, kind)(variance=v, lengthscales=l) for kind, (v, l) in zip(kinds, hyp)]
    model = GPR_additive((X, y.reshape(-1, 1)), kerns, bases)
    model.likelihood.variance.assign(s2)

    meshes, deltas = [bb.mesh for bb in bases], [bb.delta for bb in bases]
    G0, b0, yy0 = O.precompute_additive(meshes, deltas, k, ms, X, y)
    np.testing.assert_allclose(model.KufKfu, G0, rtol=0, atol=1e-10 * np.abs(G0).max())
    np.testing.assert_allclose(np.ravel(model.Kuf_y), b0.ravel(), rtol=0, atol=1e-10 * np.abs(b0).max())
    assert abs(model.tr_yTy - yy0) <= 1e-12 * yy0 and model.num_data == n
    T = [O.static_bands(k, m, d) for m, d in zip(ms, deltas)]
    e0, g0 = O.elbo_grad_additive_dense(kinds, T, G0, b0, yy0, n, hyp, s2)
    assert abs(model.elbo() - e0) <= 1e-10 * abs(e0)
    elbo, grads = model.elbo_and_grad()
    assert abs(elbo - e0) <= 1e-10 * abs(e0)
    got = np.array([grads[id(p)] for p in model.trainable_variables])
    assert got.size == 2 * D + 1
    np.testing.assert_allclose(got, g0, rtol=1e-8, atol=1e-8 * np.abs(g0).max())

    Xs = np.concatenate([np.stack([rng.uniform(a, b, 97) for a, b in doms], 1),
                         np.array([[a for a, _ in doms], [b for _, b in doms]], dtype=np.float64),
                         np.stack([np.asarray(bb.mesh)[rng.integers(0, len(bb.mesh), 16)] for bb in bases], 1)])
    Ks = [O.make_Kuu(kind, l, v, t) for kind, (v, l), t in zip(kinds, hyp, T)]
    mean, var = model.predict_f(Xs)
    mean0, var0 = O.predict_additive_dense(meshes, deltas, k, ms, Ks, G0, b0, [h[0] for h in hyp], s2, Xs)
    np.testing.assert_allclose(mean, mean0, atol=1e-9, rtol=0)
    np.testing.assert_allclose(var, var0, atol=1e-9, rtol=0)
