"""GPU parity of multi-output targets y[N, D] in GPR_kron and GPR_additive: one factorisation of P with D right-hand sides
(asvgp_kron_*_multi / asvgp_dense_*_multi) against D single-column models combined by the reference's multi-output bound,
ELBO_D = sum_d ELBO(y_d) - (D - 1) T with T = (-N prior + trace) / (2 sigma2) (reference gpr.py:78-87), against a D-column
torch-autograd dense oracle and the LAPACK-band oracle, at the ops level against D single-rhs calls and numpy, and across the
input variants (host, device, raster, float32, shuffled, strided)."""
import numpy as np
import pytest
import scipy.sparse as sp

from oracle import asvgp_oracle as O

pytestmark = pytest.mark.gpu
DOMAINS = ((0, 1), (0, 2))
HYP, S2 = [(.7, .3), (1.3, .5)], .05


def _kron(X, Y, k, ms, hyp=HYP, s2=S2, domains=DOMAINS, kinds=("Matern32", "Matern32"), **kw):
    from asvgp_b200 import basis as B, kernels as Kn
    from asvgp_b200.gpr import GPR_kron

    cls = getattr(B, "B%dSpline" % k)
    bases = [cls(domains[0][0], domains[0][1], ms[0]), cls(domains[1][0], domains[1][1], ms[1])]
    kerns = [getattr(Kn, kind)(variance=v, lengthscales=l) for kind, (v, l) in zip(kinds, hyp)]
    model = GPR_kron((X, Y), kerns, bases, **kw)
    model.likelihood.variance.assign(s2)
    return model


def _widen(X, y, seed=11):
    """y and two more columns: a second seeded smooth field and -0.5 y + noise."""
    rng = np.random.default_rng(seed)
    y = np.asarray(y).reshape(-1)
    second = np.cos(3.0 * X[:, 0] + 0.5) * np.sin(2.0 * X[:, 1]) + 0.1 * rng.standard_normal(y.size)
    return np.stack([y, second, -0.5 * y + 0.05 * rng.standard_normal(y.size)], 1)


def _grads(model):
    e, g = model.elbo_and_grad()
    return e, np.array([g[id(p)] for p in model.trainable_variables])


def _combine(elbos, grads, T, dT):
    D = len(elbos)
    return float(np.sum(elbos) - (D - 1) * T), np.sum(grads, 0) - (D - 1) * np.asarray(dT)


def _kron_T(kinds, tables, G, n, hyp, s2):
    """T = (-N v1 v2 + trace((K1 (x) K2)^-1 G)) / (2 s2) and its gradient in (v1, l1, v2, l2, s2), by torch autograd."""
    import torch

    th = torch.tensor([hyp[0][0], hyp[0][1], hyp[1][0], hyp[1][1], s2], dtype=torch.float64, requires_grad=True)
    Ls = []
    for i in range(2):
        dense = {nme: torch.from_numpy(O.band_to_dense_sym(t)) for nme, t in tables[i].items()}
        K = sum(c * dense[nme] for nme, c in O._kuu_coefficients_torch(kinds[i], th[2 * i + 1], th[2 * i]).items())
        Ls.append(torch.linalg.cholesky(K))
    Gd = torch.from_numpy(np.asarray(G.toarray() if sp.issparse(G) else G, dtype=np.float64))
    tr = torch.trace(torch.cholesky_solve(Gd, torch.kron(Ls[0], Ls[1])))
    T = 0.5 * (-n * th[0] * th[2] + tr) / th[4]
    T.backward()
    return float(T.detach()), th.grad.numpy().copy()


def _kron_dense_multi(kinds, tables, G, B, yy_total, n, hyp, s2):
    """The D-column bound of the dense reference algebra (oracle.elbo_grad_kron_dense with B [M, D] in place of b): the
    log-dets and the log(2 pi s2) term count D times, -N v1 v2 / 2 s2 and trace / 2 s2 once; torch autograd."""
    import torch

    D = B.shape[1]
    th = torch.tensor([hyp[0][0], hyp[0][1], hyp[1][0], hyp[1][1], s2], dtype=torch.float64, requires_grad=True)
    Ks = []
    for i in range(2):
        dense = {nme: torch.from_numpy(O.band_to_dense_sym(t)) for nme, t in tables[i].items()}
        Ks.append(sum(c * dense[nme] for nme, c in O._kuu_coefficients_torch(kinds[i], th[2 * i + 1], th[2 * i]).items()))
    s2t = th[4]
    Kuu = torch.kron(Ks[0], Ks[1])
    L_Kuu = torch.kron(torch.linalg.cholesky(Ks[0]), torch.linalg.cholesky(Ks[1]))
    Gd = torch.from_numpy(np.asarray(G.toarray(), dtype=np.float64))
    Bt = torch.from_numpy(np.asarray(B, dtype=np.float64))
    L_P = torch.linalg.cholesky(Kuu + Gd / s2t)
    C = torch.linalg.solve_triangular(L_P, Bt, upper=False) / s2t
    elbo = (-0.5 * n * D * torch.log(2 * np.pi * s2t) - D * torch.log(torch.diagonal(L_P)).sum()
            + D * torch.log(torch.diagonal(L_Kuu)).sum() - 0.5 * yy_total / s2t + 0.5 * (C**2).sum()
            - 0.5 * n * th[0] * th[2] / s2t + 0.5 * torch.trace(torch.cholesky_solve(Gd, L_Kuu)) / s2t)
    elbo.backward()
    return float(elbo.detach()), th.grad.numpy().copy()


# ---- GPR_kron against D single-column models --------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [2, 3, 4])
def test_kron_matches_single_column_models(cuda, golden, k):
    g = golden("kron_2d")
    m = int(g["k%d_m" % k])
    X, Y = g["X"], _widen(g["X"], g["y"])
    multi = _kron(X, Y, k, (m, m))
    singles = [_kron(X, Y[:, d].copy(), k, (m, m)) for d in range(3)]
    e, gr = _grads(multi)
    eg = [_grads(s) for s in singles]
    tables = [O.static_bands(k, m, b.delta) for b in multi.bases]
    T, dT = _kron_T(("Matern32", "Matern32"), tables, multi.KufKfu_sparse, X.shape[0], HYP, S2)
    e0, g0 = _combine([a for a, _ in eg], [b for _, b in eg], T, dT)
    assert abs(e - e0) <= 1e-10 * abs(e0)
    np.testing.assert_allclose(gr, g0, rtol=1e-8, atol=1e-8 * np.abs(g0).max())
    assert abs(multi.elbo() - e0) <= 1e-10 * abs(e0)
    assert multi.Kuf_y.shape == (m * m, 3)
    for d, s in enumerate(singles):
        np.testing.assert_allclose(multi.Kuf_y[:, d], s.Kuf_y[:, 0], rtol=1e-12, atol=1e-12 * np.abs(s.Kuf_y).max())
    assert abs(multi.tr_yTy - sum(s.tr_yTy for s in singles)) <= 1e-12 * multi.tr_yTy
    assert multi.num_data == X.shape[0]
    Xs = g["k%d_Xs" % k]
    mean, var = multi.predict_f(Xs)
    assert mean.shape == (Xs.shape[0], 3) and var.shape == (Xs.shape[0], 1)
    for d, s in enumerate(singles):
        m_d, v_d = s.predict_f(Xs)
        np.testing.assert_allclose(mean[:, d], m_d[:, 0], atol=1e-12, rtol=0)
        np.testing.assert_allclose(var, v_d, atol=1e-12, rtol=0)
    # device test points give device results of the same shapes
    import torch

    md, vd = multi.predict_f(torch.from_numpy(Xs).cuda())
    assert md.is_cuda and tuple(md.shape) == (Xs.shape[0], 3) and tuple(vd.shape) == (Xs.shape[0], 1)
    np.testing.assert_allclose(md.cpu().numpy(), mean, atol=1e-13, rtol=0)


@pytest.mark.parametrize("k,kinds", [(3, ("Matern32", "Matern32")), (4, ("Matern32", "Matern52")), (2, ("Matern12", "Matern32"))])
def test_kron_gradients_match_multi_column_autograd_oracle(cuda, golden, k, kinds):
    g = golden("kron_2d")
    m = int(g["k%d_m" % k])
    X, Y = g["X"], _widen(g["X"], g["y"])
    model = _kron(X, Y, k, (m, m), kinds=kinds)
    e, gr = _grads(model)
    tables = [O.static_bands(k, m, b.delta) for b in model.bases]
    e0, g0 = _kron_dense_multi(kinds, tables, model.KufKfu_sparse, model.Kuf_y, model.tr_yTy, X.shape[0], HYP, S2)
    assert abs(e - e0) <= 1e-10 * abs(e0)
    np.testing.assert_allclose(gr, g0, rtol=1e-8, atol=1e-8 * np.abs(g0).max())


def _raster(n1, n2, rng, inner=((-75, -30), (20, 50))):
    x1 = np.linspace(inner[0][0], inner[0][1], n1)
    x2 = np.linspace(inner[1][0], inner[1][1], n2)
    return np.stack(np.meshgrid(x1, x2, indexing="ij"), -1).reshape(-1, 2)


def _fields(X, D, rng):
    cols = [np.sin(X[:, 0] / (3.0 + d)) * np.cos(X[:, 1] / (2.5 + 0.5 * d)) + 0.05 * rng.standard_normal(X.shape[0])
            for d in range(D)]
    return np.stack(cols, 1)


def test_kron_midsize_vs_banded_oracle(cuda):
    """40 x 36, k = 3, 500 x 400 raster points, D = 4: per-column LAPACK-band oracle combined."""
    rng = np.random.default_rng(5)
    k, ms, D = 3, (40, 36), 4
    domains = ((-80, -25), (15, 55))
    X = _raster(500, 400, rng)
    Y = _fields(X, D, rng)
    hyp, s2 = [(1.0, 6.0), (0.8, 5.0)], 0.01
    model = _kron(X, Y, k, ms, hyp=hyp, s2=s2, domains=domains)
    meshes = [b.mesh for b in model.bases]
    deltas = [b.delta for b in model.bases]
    pre = [O.precompute_kron(meshes, deltas, k, list(ms), X, Y[:, d]) for d in range(D)]
    G0 = pre[0][0]
    for d in range(D):
        np.testing.assert_allclose(model.Kuf_y[:, d], np.asarray(pre[d][1]).ravel(), rtol=1e-10,
                                   atol=1e-10 * np.abs(pre[d][1]).max())
    T = [O.static_bands(k, m, dl) for m, dl in zip(ms, deltas)]
    Gc = sp.coo_matrix(G0)

    def f(th):
        Ks = [O.make_Kuu("Matern32", th[1], th[0], T[0]), O.make_Kuu("Matern32", th[3], th[2], T[1])]
        tot = sum(O.elbo_kron_banded(Ks, G0, b0, yy0, X.shape[0], [th[0], th[2]], th[4], k, list(ms)) for _, b0, yy0 in pre)
        Kinv = [np.linalg.inv(O.band_to_dense_sym(K)) for K in Ks]
        tr = np.sum(Gc.data * Kinv[0][Gc.row // ms[1], Gc.col // ms[1]] * Kinv[1][Gc.row % ms[1], Gc.col % ms[1]])
        return tot - (D - 1) * 0.5 * (-X.shape[0] * th[0] * th[2] + tr) / th[4]

    th0 = np.array([hyp[0][0], hyp[0][1], hyp[1][0], hyp[1][1], s2])
    want = f(th0)
    e, got = _grads(model)
    assert abs(e - want) <= 1e-10 * abs(want)
    assert abs(model.elbo() - want) <= 1e-10 * abs(want)
    for i in range(5):
        h = 1e-4 * th0[i]
        e_ = np.zeros(5); e_[i] = h
        fd = (-f(th0 + 2 * e_) + 8 * f(th0 + e_) - 8 * f(th0 - e_) + f(th0 - 2 * e_)) / (12 * h)
        assert abs(fd - got[i]) <= 1e-6 * max(1.0, abs(got[i])), (i, fd, got[i])
    Ks = [O.make_Kuu("Matern32", l, v, t) for (v, l), t in zip(hyp, T)]
    Xs = np.stack([rng.uniform(-74, -31, 300), rng.uniform(21, 49, 300)], 1)
    mean, var = model.predict_f(Xs)
    for d in range(D):
        mean0, var0 = O.predict_kron_banded(meshes, deltas, k, list(ms), Ks, G0, pre[d][1], [h[0] for h in hyp], s2, Xs)
        np.testing.assert_allclose(mean[:, d], np.asarray(mean0).ravel(), atol=1e-9, rtol=0)
        if d == 0:
            np.testing.assert_allclose(var, var0, atol=1e-9, rtol=0)


def test_kron_full_size_plan(cuda):
    """200 x 200, k = 3, D = 4: the full multi-level tree with four rhs nodes, against four single-column models."""
    import torch

    rng = np.random.default_rng(8)
    k, ms, D = 3, (200, 200), 4
    domains = ((-80, -25), (15, 55))
    X = _raster(700, 600, rng)
    Y = _fields(X, D, rng)
    hyp, s2 = [(1.0, 6.0), (0.8, 5.0)], 0.01
    Xd, Yd = torch.from_numpy(X).cuda(), torch.from_numpy(Y).cuda()
    multi = _kron(Xd, Yd, k, ms, hyp=hyp, s2=s2, domains=domains, raster_shape=(700, 600))
    singles = [_kron(Xd, Yd[:, d].contiguous(), k, ms, hyp=hyp, s2=s2, domains=domains, raster_shape=(700, 600)) for d in range(D)]
    e, gr = _grads(multi)
    eg = [_grads(s) for s in singles]
    # T and its derivatives from the single-column model's terms: T = (-N v1 v2 + tr) / (2 s2)
    tr = singles[0].last_terms["trace"]
    n = X.shape[0]
    T = 0.5 * (-n * hyp[0][0] * hyp[1][0] + tr) / s2
    e0 = float(np.sum([a for a, _ in eg]) - (D - 1) * T)
    assert abs(e - e0) <= 1e-10 * abs(e0)
    assert abs(multi.last_terms["trace"] - tr) <= 1e-12 * abs(tr)
    # the v and s2 derivatives of T are closed-form; l1, l2 come from the difference, which must then agree column-wise
    dT = np.array([0.5 * (-n * hyp[1][0] + tr / hyp[0][0]) / s2, np.nan, 0.5 * (-n * hyp[0][0] + tr / hyp[1][0]) / s2, np.nan, -T / s2])
    gsum = np.sum([b for _, b in eg], 0)
    for i in (0, 2, 4):
        want = gsum[i] - (D - 1) * dT[i]
        assert abs(gr[i] - want) <= 1e-8 * max(abs(want), 1.0), (i, gr[i], want)
    # lengthscale derivatives of T, as the D = 4 model implies them, must also account for a D = 2 model of the first columns
    _, g2 = _grads(_kron(Xd, Yd[:, :2].contiguous(), k, ms, hyp=hyp, s2=s2, domains=domains, raster_shape=(700, 600)))
    for i in (1, 3):
        dT_l = (gsum[i] - gr[i]) / (D - 1)
        want = eg[0][1][i] + eg[1][1][i] - dT_l
        assert abs(g2[i] - want) <= 1e-8 * max(abs(want), 1.0), (i, g2[i], want)
    for d, s in enumerate(singles):
        np.testing.assert_allclose(multi.Kuf_y[:, d], s.Kuf_y[:, 0], rtol=1e-12, atol=1e-12 * np.abs(s.Kuf_y).max())
    Xs = np.stack([rng.uniform(-74, -31, 2000), rng.uniform(21, 49, 2000)], 1)
    mean, var = multi.predict_f(Xs)
    for d, s in enumerate(singles):
        m_d, v_d = s.predict_f(Xs)
        np.testing.assert_allclose(mean[:, d], m_d[:, 0], atol=1e-10 * max(1.0, np.abs(m_d).max()), rtol=0)
        np.testing.assert_allclose(var, v_d, atol=1e-10 * max(1.0, np.abs(v_d).max()), rtol=0)


# ---- ops level --------------------------------------------------------------------------------------------------------------
def _kron_inputs(golden, k):
    g = golden("kron_2d")
    m = int(g["k%d_m" % k])
    model = _kron(g["X"], g["y"].reshape(-1), k, (m, m))
    Ks, _, _, _, _ = model._factors(False)
    return model, Ks, m


@pytest.mark.parametrize("D", [2, 5, 32])
def test_kron_ops_multi_vs_single_rhs(cuda, golden, D):
    import torch

    from asvgp_b200 import ops

    model, Ks, m = _kron_inputs(golden, 3)
    M = m * m
    rng = np.random.default_rng(D)
    b = model._b.cpu().numpy()
    B = np.stack([b * (1 + 0.3 * d) + rng.standard_normal(M) * np.abs(b).max() * 0.2 * (d > 0) for d in range(D)])
    Bd = torch.from_numpy(B).cuda()
    wsm = ops.kron_workspace(m, m, 3, "nd", n_rhs=D)
    ops.kron_factor(Ks[0], Ks[1], model._acc, model.bases, S2, wsm, b=Bd)
    SigM, XM = ops.kron_selinv(model.bases, wsm)
    scal = wsm.scal.cpu().numpy()
    SigM, XM = SigM.cpu().numpy(), XM.cpu().numpy()
    assert XM.shape == (D, M) and scal[1] == 0
    ws1 = ops.kron_workspace(m, m, 3, "nd")
    for d in range(D):
        ops.kron_factor(Ks[0], Ks[1], model._acc, model.bases, S2, ws1, b=Bd[d])
        Sig1, x1 = ops.kron_selinv(model.bases, ws1)
        s1 = ws1.scal.cpu().numpy()
        assert abs(scal[0] - s1[0]) <= 1e-12 * abs(s1[0])
        assert abs(scal[2 + d] - s1[1]) <= 1e-12 * abs(s1[1])
        x1 = x1.cpu().numpy()
        np.testing.assert_allclose(XM[d], x1, rtol=0, atol=1e-10 * np.abs(x1).max())
        S1 = Sig1.cpu().numpy()
        np.testing.assert_allclose(SigM, S1, rtol=0, atol=1e-12 * np.abs(S1).max())


def test_multi_entry_points_with_one_rhs_equal_the_single_rhs_ones(cuda, golden):
    """n_rhs = 1 through the _multi entry points runs the single-rhs plan and arithmetic: the outputs agree with those of
    asvgp_kron_factor / _selinv and asvgp_dense_factor / _selinv as closely as two runs of the latter agree with each other
    (the extend-add and the selected inverse add into shared entries with fp64 REDs, whose order varies from run to run)."""
    import torch

    from asvgp_b200 import ops

    model, Ks, m = _kron_inputs(golden, 4)
    ws = ops.kron_workspace(m, m, 4, "nd")
    Gs, b, _ = ops.split_accum_2d(model._acc, model.bases)

    def run(multi):
        rhs = b.clone()
        scal = torch.zeros(3, dtype=torch.float64, device="cuda")
        sig = torch.empty(ws.n_sig, dtype=torch.float64, device="cuda")
        st = torch.zeros_like(ws.sigma_stencil)
        if multi:
            ops._lib.call("asvgp_kron_factor_multi", ops._p(Ks[0]), ops._p(Ks[1]), ops._p(Gs), m, m, 4, 1, S2, ops._p(ws.band),
                          ops._p(rhs), ops._p(scal), ops._stream())
            ops._lib.call("asvgp_kron_selinv_multi", ops._p(ws.band), m, m, 4, 1, ops._p(sig), ops._p(rhs), ops._p(st),
                          ops._p(ws.work), ops._stream())
            s = scal.cpu().numpy()[[0, 2, 1]]                   # {log|P|, info, Q} -> {log|P|, Q, info}
        else:
            ops._lib.call("asvgp_kron_factor", ops._p(Ks[0]), ops._p(Ks[1]), ops._p(Gs), m, m, 4, S2, ops._p(ws.band),
                          ops._p(rhs), ops._p(scal), ops._stream())
            ops._lib.call("asvgp_kron_selinv", ops._p(ws.band), m, m, 4, ops._p(sig), ops._p(rhs), ops._p(st), ops._p(ws.work),
                          ops._stream())
            s = scal.cpu().numpy()
        return [s, rhs.cpu().numpy(), st.cpu().numpy()]

    _same_as_reproducible(run)

    n = 300
    rng = np.random.default_rng(2)
    A_ = rng.standard_normal((n, n))
    A = torch.from_numpy(np.tril(A_ @ A_.T + n * np.eye(n))).cuda()
    r = torch.from_numpy(rng.standard_normal(n)).cuda()
    wd = ops.dense_workspace(n)

    def run_dense(multi):
        scal = torch.zeros(3, dtype=torch.float64, device="cuda")
        x = torch.empty(n, dtype=torch.float64, device="cuda")
        inv = torch.empty((n, n), dtype=torch.float64, device="cuda")
        if multi:
            ops._lib.call("asvgp_dense_factor_multi", ops._p(A), n, 1, ops._p(r), ops._p(wd.band), ops._p(scal), ops._stream())
            ops._lib.call("asvgp_dense_selinv_multi", ops._p(wd.band), n, 1, ops._p(wd.sig_band), ops._p(x), ops._p(inv),
                          ops._p(wd.work), ops._stream())
            s = scal.cpu().numpy()[[0, 2, 1]]
        else:
            ops._lib.call("asvgp_dense_factor", ops._p(A), n, ops._p(r), ops._p(wd.band), ops._p(scal), ops._stream())
            ops._lib.call("asvgp_dense_selinv", ops._p(wd.band), n, ops._p(wd.sig_band), ops._p(x), ops._p(inv), ops._p(wd.work),
                          ops._stream())
            s = scal.cpu().numpy()
        return [s, x.cpu().numpy(), inv.cpu().numpy()]

    _same_as_reproducible(run_dense)


def _same_as_reproducible(run):
    a, a2, b = run(False), run(False), run(True)
    for u, u2, v in zip(a, a2, b):
        spread = np.abs(u - u2).max()            # run-to-run spread of the single-rhs function itself
        assert np.abs(v - u).max() <= 4 * spread + 1e-13 * np.abs(u).max(), (np.abs(v - u).max(), spread)


@pytest.mark.parametrize("n", [1, 63, 64, 65, 300])
@pytest.mark.parametrize("D", [1, 2, 5, 32])
def test_dense_multi_matches_numpy(cuda, n, D):
    import torch

    from asvgp_b200 import ops

    rng = np.random.default_rng(100 * n + D)
    A_ = rng.standard_normal((n, n))
    A = A_ @ A_.T + n * np.eye(n)
    B = rng.standard_normal((D, n))
    ws = ops.dense_workspace(n, D)
    ops.dense_factor(torch.from_numpy(np.tril(A)).cuda(), torch.from_numpy(B).cuda(), ws)
    x, inv = ops.dense_selinv(ws)
    scal = ws.scal.cpu().numpy()
    X0 = np.linalg.solve(A, B.T).T
    Q0 = np.einsum("dn,dn->d", B, X0)
    if D == 1:
        logdet, info, Q = scal[0], scal[2], scal[1:2]
    else:
        logdet, info, Q = scal[0], scal[1], scal[2:]
    assert info == 0
    assert abs(logdet - np.linalg.slogdet(A)[1]) <= 1e-12 * abs(logdet) + 1e-12
    np.testing.assert_allclose(Q, Q0, rtol=1e-12, atol=0)
    np.testing.assert_allclose(x.cpu().numpy().reshape(D, n), X0, rtol=0, atol=1e-12 * np.abs(X0).max())
    inv0 = np.linalg.inv(A)
    np.testing.assert_allclose(inv.cpu().numpy(), inv0, rtol=0, atol=1e-12 * np.abs(inv0).max())


# ---- input variants ---------------------------------------------------------------------------------------------------------
def _same_model(a, b, rtol=1e-12):
    np.testing.assert_allclose(a.Kuf_y, b.Kuf_y, rtol=0, atol=rtol * np.abs(b.Kuf_y).max())
    assert abs(a.tr_yTy - b.tr_yTy) <= rtol * b.tr_yTy and a.num_data == b.num_data
    ea, ga = _grads(a)
    eb, gb = _grads(b)
    assert abs(ea - eb) <= 1e-10 * abs(eb)
    np.testing.assert_allclose(ga, gb, rtol=1e-8, atol=1e-8 * np.abs(gb).max())


def test_input_variants_give_the_same_model(cuda):
    import torch

    rng = np.random.default_rng(21)
    k, ms, D = 3, (40, 36), 3
    domains = ((-80, -25), (15, 55))
    hyp, s2 = [(1.0, 6.0), (0.8, 5.0)], 0.01
    X = _raster(600, 500, rng)                    # 300 000 points: enough for the binned path
    Y = _fields(X, 2 * D, rng)
    Yc = np.ascontiguousarray(Y[:, ::2])
    Xd, Ycd = torch.from_numpy(X).cuda(), torch.from_numpy(Yc).cuda()
    kw = dict(hyp=hyp, s2=s2, domains=domains)
    ref = _kron(Xd, Ycd, k, ms, **kw)
    _same_model(_kron(X, Yc, k, ms, **kw), ref)                                            # host numpy
    _same_model(_kron(X, Yc, k, ms, raster_shape=(600, 500), **kw), ref)                   # host, stated raster
    _same_model(_kron(Xd, Ycd, k, ms, raster_shape=(600, 500), **kw), ref)                 # device, stated raster
    _same_model(_kron(Xd, torch.from_numpy(Y).cuda()[:, ::2], k, ms, **kw), ref)           # strided device columns
    _same_model(_kron(X, Y[:, ::2], k, ms, **kw), ref)                                     # strided host columns
    # float32 targets: the same model as the float64-converted ones
    Y32 = Yc.astype(np.float32)
    ref32 = _kron(Xd, torch.from_numpy(Y32.astype(np.float64)).cuda(), k, ms, **kw)
    _same_model(_kron(Xd, torch.from_numpy(Y32).cuda(), k, ms, **kw), ref32)
    _same_model(_kron(X, Y32, k, ms, **kw), ref32)
    # shuffled points: the binned path, probed once for all columns
    from asvgp_b200 import ops

    perm = rng.permutation(X.shape[0])
    Xs_d = torch.from_numpy(X[perm]).cuda()
    assert ops.choose_binned_2d(Xs_d, ref.bases)
    _same_model(_kron(Xs_d, torch.from_numpy(Yc[perm]).cuda(), k, ms, **kw), ref, rtol=1e-11)


def test_band_method_refuses_several_columns(cuda, golden):
    g = golden("kron_2d")
    m = int(g["k3_m"])
    with pytest.raises(NotImplementedError):
        _kron(g["X"], _widen(g["X"], g["y"]), 3, (m, m), method="band")
    model = _kron(g["X"], g["y"].reshape(-1), 3, (m, m), method="band")      # one column: unchanged
    assert np.isfinite(model.elbo())


# ---- GPR_additive -----------------------------------------------------------------------------------------------------------
def _additive(g, Y, kinds=("Matern52", "Matern12", "Matern32"), hypers=((.7, .3), (1.3, .5), (.9, .8)), s2=.05):
    from asvgp_b200 import basis as B, kernels as Kn
    from asvgp_b200.gpr import GPR_additive

    m = int(g["m"])
    bases = [B.B3Spline(int(a), int(b), m) for a, b in g["doms"]]
    kerns = [getattr(Kn, kind)(variance=v, lengthscales=l) for kind, (v, l) in zip(kinds, hypers)]
    model = GPR_additive((g["X"], Y), kerns, bases)
    model.likelihood.variance.assign(s2)
    return model


def _additive_T(kinds, tables, G, offsets, n, hypers, s2):
    import torch

    th = torch.tensor([h for vl in hypers for h in vl] + [s2], dtype=torch.float64, requires_grad=True)
    tr = 0.0
    for i in range(len(kinds)):
        dense = {nme: torch.from_numpy(O.band_to_dense_sym(t)) for nme, t in tables[i].items()}
        K = sum(c * dense[nme] for nme, c in O._kuu_coefficients_torch(kinds[i], th[2 * i + 1], th[2 * i]).items())
        o0, o1 = offsets[i], offsets[i + 1]
        tr = tr + torch.trace(torch.linalg.solve(K, torch.from_numpy(np.ascontiguousarray(G[o0:o1, o0:o1]))))
    vsum = sum(th[2 * i] for i in range(len(kinds)))
    T = 0.5 * (-n * vsum + tr) / th[-1]
    T.backward()
    return float(T.detach()), th.grad.numpy().copy()


def test_additive_matches_single_column_models(cuda, golden):
    g = golden("additive_3d")
    Y = _widen(g["X"], g["y"])
    multi = _additive(g, Y)
    singles = [_additive(g, Y[:, d:d + 1].copy()) for d in range(3)]
    e, gr = _grads(multi)
    eg = [_grads(s) for s in singles]
    kinds, hypers, s2 = ("Matern52", "Matern12", "Matern32"), ((.7, .3), (1.3, .5), (.9, .8)), .05
    tables = [O.static_bands(3, b.m, b.delta) for b in multi.bases]
    T, dT = _additive_T(kinds, tables, multi.KufKfu, multi._offsets, g["X"].shape[0], hypers, s2)
    e0, g0 = _combine([a for a, _ in eg], [b for _, b in eg], T, dT)
    assert abs(e - e0) <= 1e-10 * abs(e0)
    assert abs(multi.elbo() - e0) <= 1e-10 * abs(e0)
    np.testing.assert_allclose(gr, g0, rtol=1e-8, atol=1e-8 * np.abs(g0).max())
    assert multi.Kuf_y.shape == (multi.M, 3)
    for d, s in enumerate(singles):
        np.testing.assert_allclose(multi.Kuf_y[:, d], s.Kuf_y[:, 0], rtol=1e-12, atol=1e-12 * np.abs(s.Kuf_y).max())
    mean, var = multi.predict_f(g["Xs"])
    assert mean.shape == (g["Xs"].shape[0], 3) and var.shape == (g["Xs"].shape[0], 1)
    for d, s in enumerate(singles):
        m_d, v_d = s.predict_f(g["Xs"])
        np.testing.assert_allclose(mean[:, d], m_d[:, 0], atol=1e-12, rtol=0)
        np.testing.assert_allclose(var, v_d, atol=1e-12, rtol=0)
