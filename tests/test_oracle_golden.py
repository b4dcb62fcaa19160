"""Pins the CPU oracle (oracle/asvgp_oracle.py) to the golden vectors produced by the UNMODIFIED reference run
under numpy stand-ins (oracle/make_golden.py), and to the reference's own stored known answer."""
import numpy as np
import pytest
import scipy.sparse as sp

from oracle import asvgp_oracle as O

KINDS = ("Matern12", "Matern32", "Matern52")


def test_snelson_tables_precompute_and_elbo(golden):
    g = golden("snelson")
    mesh, delta = O.make_mesh(-3.5, 10.5, 100, 3)
    np.testing.assert_array_equal(mesh, g["mesh"])
    assert delta == float(g["delta"])
    T = O.static_bands(3, 100, delta)
    for name in ("A", "B", "C", "D", "BC", "BC_grad", "BC_ggrad"):
        np.testing.assert_allclose(T[name], g["tab_" + name], rtol=1e-13, atol=1e-13 * np.abs(g["tab_" + name]).max())
    assert not g["tab_BC_ggrad_none"].any() and not g["tab_BC_none_ggrad"].any()        # SURVEY quirk Q5
    G, b, yy = O.precompute_1d(mesh, delta, 3, 100, g["X"], g["y"])
    np.testing.assert_allclose(G, g["G"], rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(b, g["Kuf_y"], rtol=1e-12, atol=1e-14)
    assert abs(yy - float(g["tr_yTy"])) < 1e-12
    for kind in KINDS:
        Kuu = O.make_Kuu(kind, 1.0, 1.0, T)
        np.testing.assert_allclose(Kuu, g["Kuu111_" + kind], rtol=1e-12, atol=1e-12)
        e = O.elbo_1d(Kuu, G, b, yy, 200, 1.0, 1.0)
        assert abs(e - float(g["elbo111_" + kind])) <= 1e-10 * abs(e)
        e = O.elbo_1d(O.make_Kuu(kind, 1.03, 0.8, T), G, b, yy, 200, 0.8, 0.08)
        assert abs(e - float(g["elbo_b_" + kind])) <= 1e-10 * abs(e)


def test_snelson_known_answer_and_predictions(golden):
    g = golden("snelson")
    mesh, delta = O.make_mesh(-3.5, 10.5, 100, 3)
    T = O.static_bands(3, 100, delta)
    G, b, yy = O.precompute_1d(mesh, delta, 3, 100, g["X"], g["y"])
    v, l, s2 = g["opt_hypers"]
    Kuu = O.make_Kuu("Matern32", l, v, T)
    e = O.elbo_1d(Kuu, G, b, yy, 200, v, s2)
    # at the (10-digit) stored optimum the ELBO equals the reference notebook's printed value to ~1e-8
    assert abs(e - float(g["notebook_elbo"])) < 5e-8
    assert abs(e - float(g["elbo_opt"])) <= 1e-10 * abs(e)
    assert e < float(g["notebook_exact_gp"])
    mean, var = O.predict_1d(mesh, delta, 3, 100, Kuu, G, b, v, s2, g["Xtest"])
    np.testing.assert_allclose(mean, g["pred_mean"], atol=1e-9)
    np.testing.assert_allclose(var, g["pred_var"], atol=1e-9)


def test_snelson_optimum_is_stationary(golden):
    g = golden("snelson")
    mesh, delta = O.make_mesh(-3.5, 10.5, 100, 3)
    T = O.static_bands(3, 100, delta)
    G, b, yy = O.precompute_1d(mesh, delta, 3, 100, g["X"], g["y"])
    v, l, s2 = g["opt_hypers"]
    _, grad = O.elbo_grad_1d_dense("Matern32", T, G, b, yy, 200, v, l, s2)
    assert np.abs(grad).max() < 5e-2          # constrained-space gradient at the 10-digit stored optimum


@pytest.mark.parametrize("k", [1, 2, 3, 4, 5, 6])
def test_basis_eval_golden(golden, k):
    g = golden("basis_eval")
    for tag, a, b in (("f32", -3.5, 10.5), ("f64", -1, 41)):
        key = "k%d_%s" % (k, tag)
        mesh, delta = O.make_mesh(a, b, 40, k)
        np.testing.assert_array_equal(mesh, g[key + "_mesh"])
        for dx in range(4):
            name = key + "_dx%d" % dx
            if name in g.files:
                got = O.make_Kuf(mesh, delta, k, 40, g[key + "_x"], dx).toarray()
                np.testing.assert_allclose(got, g[name], rtol=1e-12, atol=1e-12 * np.abs(g[name]).max())
        T = O.static_bands(k, 40, delta)
        for name in ("A", "B", "C", "D", "BC", "BC_grad", "BC_ggrad"):
            if key + "_" + name in g.files:
                want = g[key + "_" + name]
                np.testing.assert_allclose(T[name], want, rtol=1e-12, atol=1e-12 * np.abs(want).max())


@pytest.mark.parametrize("k", [1, 2, 3, 4, 5])
def test_synth_1d_golden(golden, k):
    g = golden("synth_1d")
    key = "k%d" % k
    m = int(g[key + "_m"])
    mesh, delta = O.make_mesh(-1, m + 1, m, k)
    T = O.static_bands(k, m, delta)
    x, y = g[key + "_x"], g[key + "_y"]
    G, b, yy = O.precompute_1d(mesh, delta, k, m, x, y)
    np.testing.assert_allclose(G, g[key + "_G"], rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(b, g[key + "_Kuf_y"], rtol=1e-12, atol=1e-12)
    G2, b2, yy2 = O.precompute_1d_chunked(mesh, delta, k, m, x, y, chunk=3000)
    np.testing.assert_allclose(G2, G, rtol=1e-12, atol=1e-12)
    for kind in KINDS:
        for tag, (v, l, s2) in (("a", (1.0, 1.0, 0.1)), ("b", (1.3, 2.5, 0.7))):
            name = "%s_%s_elbo_%s" % (key, kind, tag)
            if name in g.files:
                e = O.elbo_1d(O.make_Kuu(kind, l, v, T), G, b, yy, x.shape[0], v, s2)
                assert abs(e - float(g[name])) <= 1e-10 * abs(e), name
    v, l, s2 = g[key + "_pred_hypers"]
    Kuu = O.make_Kuu(str(g[key + "_pred_kind"]), l, v, T)
    mean, var = O.predict_1d(mesh, delta, k, m, Kuu, G, b, v, s2, g[key + "_xs"])
    np.testing.assert_allclose(mean, g[key + "_mean"], atol=1e-9)
    np.testing.assert_allclose(var, g[key + "_var"], atol=1e-9)


def test_autograd_oracle_matches_finite_differences(golden):
    g = golden("synth_1d")
    m = int(g["k3_m"])
    mesh, delta = O.make_mesh(-1, m + 1, m, 3)
    T = O.static_bands(3, m, delta)
    G, b, yy, n = g["k3_G"], g["k3_Kuf_y"], float(g["k3_tr_yTy"]), g["k3_x"].shape[0]
    th = np.array([1.3, 2.5, 0.7])
    _, grad = O.elbo_grad_1d_dense("Matern52", T, G, b, yy, n, *th)

    def f(t):
        return O.elbo_1d(O.make_Kuu("Matern52", t[1], t[0], T), G, b, yy, n, t[0], t[2])

    for i in range(3):
        h = 1e-4 * th[i]
        e = np.zeros(3); e[i] = h
        fd = (-f(th + 2 * e) + 8 * f(th + e) - 8 * f(th - e) + f(th - 2 * e)) / (12 * h)
        assert abs(fd - grad[i]) <= 1e-6 * max(1.0, abs(grad[i]))


@pytest.mark.parametrize("k", [2, 3, 4])
def test_kron_golden(golden, k):
    g = golden("kron_2d")
    key = "k%d" % k
    m = int(g[key + "_m"])
    X, y = g["X"], g["y"]
    meshes, deltas = zip(*[O.make_mesh(0, 1, m, k), O.make_mesh(0, 2, m, k)])
    G, b, yy = O.precompute_kron(meshes, deltas, k, [m, m], X, y, chunk=1000)
    Gref = sp.coo_matrix((g[key + "_G_val"], (g[key + "_G_row"], g[key + "_G_col"])), shape=(m * m, m * m)).toarray()
    np.testing.assert_allclose(G.toarray(), Gref, rtol=1e-11, atol=1e-13)
    np.testing.assert_allclose(b, g[key + "_Kuf_y"], rtol=1e-11, atol=1e-13)
    T = [O.static_bands(k, m, d) for d in deltas]
    Ks = [O.make_Kuu("Matern32", .3, .7, T[0]), O.make_Kuu("Matern32", .5, 1.3, T[1])]
    e = O.elbo_kron_dense(Ks, G, b, yy, X.shape[0], [.7, 1.3], .05)
    assert abs(e - float(g[key + "_elbo"])) <= 1e-10 * abs(e)
    assert int(g[key + "_bandwidth"]) == k * (m + 1)
    mean, var = O.predict_kron_dense(meshes, deltas, k, [m, m], Ks, G, b, [.7, 1.3], .05, g[key + "_Xs"])
    np.testing.assert_allclose(mean, g[key + "_mean"], atol=1e-9)
    np.testing.assert_allclose(var, g[key + "_var"], atol=1e-9)
    if key + "_elbo_m52_m12" in g.files:
        Ks = [O.make_Kuu("Matern52", .4, .9, T[0]), O.make_Kuu("Matern12", .6, 1.1, T[1])]
        e = O.elbo_kron_dense(Ks, G, b, yy, X.shape[0], [.9, 1.1], .2)
        assert abs(e - float(g[key + "_elbo_m52_m12"])) <= 1e-10 * abs(e)


def test_multi_output_1d_golden(golden):
    """D = 3 output columns: Kuf_y is M x D, the log-dets count D times, the K_diag and trace terms once (gpr.py:78-87)."""
    g = golden("multi_output_1d")
    m, k = int(g["m"]), int(g["order"])
    mesh, delta = O.make_mesh(-1, m + 1, m, k)
    T = O.static_bands(k, m, delta)
    x, y = g["x"], g["y"]
    G, b, yy = O.precompute_1d(mesh, delta, k, m, x, y)
    assert b.shape == (m, 3)
    np.testing.assert_allclose(b, g["Kuf_y"], rtol=1e-12, atol=1e-12)
    assert abs(yy - float(g["tr_yTy"])) <= 1e-12 * yy
    for kind in KINDS:
        for tag, (v, l, s2) in (("a", (1.0, 1.0, 0.1)), ("b", (0.6, 3.5, 0.3))):
            want = float(g["elbo_%s_%s" % (kind, tag)])
            e = O.elbo_1d(O.make_Kuu(kind, l, v, T), G, b, yy, x.shape[0], v, s2)
            assert abs(e - want) <= 1e-10 * abs(want), (kind, tag)
    v, l, s2 = g["pred_hypers"]
    mean, var = O.predict_1d(mesh, delta, k, m, O.make_Kuu("Matern52", l, v, T), G, b, v, s2, g["xs"])
    np.testing.assert_allclose(mean, g["mean"], atol=1e-9)
    np.testing.assert_allclose(var, g["var"], atol=1e-9)


@pytest.mark.parametrize("kind,k", [("Matern12", 2), ("Matern32", 3), ("Matern52", 3), ("Matern52", 4)])
def test_closed_form_banded_gradient_oracle_matches_autograd(kind, k):
    """elbo_grad_1d_banded (the gradient oracle of the M = 1e4 fixtures) vs torch autograd through the dense algebra."""
    rng = np.random.default_rng(1)
    m, n = 60, 5000
    mesh, delta = O.make_mesh(-1, m + 1, m, k)
    x = np.sort(rng.uniform(0, m, n))
    y = np.sin(x / 3) + 0.2 * rng.standard_normal(n)
    G, b, yy = O.precompute_1d(mesh, delta, k, m, x, y)
    T = O.static_bands(k, m, delta)
    e0, g0 = O.elbo_grad_1d_dense(kind, T, G, b, yy, n, 1.1, 2.3, 0.15)
    e1, g1 = O.elbo_grad_1d_banded(kind, T, G, b, yy, n, 1.1, 2.3, 0.15, block=17)
    assert abs(e0 - e1) <= 1e-12 * abs(e0)
    np.testing.assert_allclose(g1, g0, rtol=1e-11, atol=1e-11 * np.abs(g0).max())


def test_large_size_kron_oracle_helpers_match_dense(golden):
    """predict_kron_banded_cells and stencil_columns_of_inverse (used for the 200 x 200 fixtures) vs the dense algebra."""
    g = golden("kron_2d")
    k, m = 3, int(g["k3_m"])
    ms = [m, m]
    meshes, deltas = zip(*[O.make_mesh(0, 1 + i, m, k) for i in range(2)])
    G = sp.coo_matrix((g["k3_G_val"], (g["k3_G_row"], g["k3_G_col"])), shape=(m * m, m * m)).tocsr()
    T = [O.static_bands(k, m, d) for d in deltas]
    Ks = [O.make_Kuu("Matern32", .3, .7, T[0]), O.make_Kuu("Matern32", .5, 1.3, T[1])]
    Xs = g["k3_Xs"]
    mean0, var0 = O.predict_kron_dense(meshes, deltas, k, ms, Ks, G, g["k3_Kuf_y"], [.7, 1.3], .05, Xs)
    mean1, var1 = O.predict_kron_banded_cells(meshes, deltas, k, ms, Ks, G, g["k3_Kuf_y"], [.7, 1.3], .05, Xs)
    np.testing.assert_allclose(mean1, mean0.reshape(-1, 1), atol=1e-11, rtol=0)
    np.testing.assert_allclose(var1, var0, atol=1e-11, rtol=0)
    np.testing.assert_allclose(mean1, g["k3_mean"], atol=1e-10, rtol=0)           # reference-under-shim
    P = (sp.kron(sp.csr_matrix(O.band_to_dense_sym(Ks[0])), sp.csr_matrix(O.band_to_dense_sym(Ks[1]))) + G / .05).toarray()
    Pinv = np.linalg.inv(P)
    cols = [0, 5, 77, m * m - 1]
    S = O.stencil_columns_of_inverse(Ks, G, .05, k, ms, cols)
    for c, j in enumerate(cols):
        j1, j2 = divmod(j, m)
        for d1 in range(k + 1):
            for d2 in range(-k, k + 1):
                inside = not (d1 == 0 and d2 < 0) and j1 + d1 < m and 0 <= j2 + d2 < m
                want = Pinv[(j1 + d1) * m + j2 + d2, j] if inside else 0.0
                assert abs(S[d1 * 7 + d2 + 3, c] - want) <= 1e-11 * np.abs(Pinv).max()


def test_scale_fixtures_are_self_consistent(golden):
    """The committed BASELINE-sized fixtures: closed-form and finite-difference gradients of the oracle agree, inputs
    regenerate with the recorded sizes."""
    import os
    import sys

    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import scale_cases as SC

    g = golden("scale_1d")
    assert int(g["n"]) == SC.C3_N and g["G"].shape == (SC.C3_ORDER + 1, SC.C3_M)
    for name in SC.C3_HYPERS:
        scale = np.abs(g[name + "_grad"]).max()
        assert np.abs(g[name + "_grad"] - g[name + "_grad_fd"]).max() <= 1e-6 * scale
        assert g[name + "_mean"].shape == (500, 1)
    c4 = golden("scale_kron_c4")
    assert int(c4["n"]) == SC.C4["raster"][0] * SC.C4["raster"][1]
    assert np.abs(c4["grad"] - c4["grad_h2"]).max() <= 1e-6 * np.abs(c4["grad"]).max()
    assert c4["Xs"].shape[0] == c4["mean"].shape[0] == 64 * 157


def test_additive_golden(golden):
    """GPR_additive restatement (precompute, bound, predictor) vs the unmodified reference under the shim, and its autograd
    gradient vs central differences."""
    g = golden("additive_3d")
    m, k = int(g["m"]), int(g["order"])
    md = [O.make_mesh(int(a), int(b), m, k) for a, b in g["doms"]]
    meshes, deltas = [x[0] for x in md], [x[1] for x in md]
    n = g["X"].shape[0]
    G, b, yy = O.precompute_additive(meshes, deltas, k, [m] * 3, g["X"], g["y"])
    np.testing.assert_allclose(G, g["KufKfu"], rtol=1e-11, atol=1e-11 * np.abs(G).max())
    np.testing.assert_allclose(b, g["Kuf_y"], rtol=1e-11, atol=1e-11)
    T = [O.static_bands(k, m, d) for d in deltas]
    for tag, kinds, hyp, s2 in (("a", ("Matern32",) * 3, [(1., 1.)] * 3, 1.0),
                                ("b", ("Matern52", "Matern12", "Matern32"), [(.7, .3), (1.3, .5), (.9, .8)], .05)):
        Ks = [O.make_Kuu(kd, l, v, t) for kd, (v, l), t in zip(kinds, hyp, T)]
        e = O.elbo_additive_dense(Ks, G, b, yy, n, [h[0] for h in hyp], s2)
        assert abs(e - float(g["elbo_" + tag])) <= 1e-10 * abs(e)
        mean, var = O.predict_additive_dense(meshes, deltas, k, [m] * 3, Ks, G, b, [h[0] for h in hyp], s2, g["Xs"])
        np.testing.assert_allclose(mean, g["mean_" + tag], atol=1e-10, rtol=0)
        np.testing.assert_allclose(var, g["var_" + tag], atol=1e-10, rtol=0)
    e2, grad = O.elbo_grad_additive_dense(kinds, T, G, b, yy, n, hyp, s2)
    assert abs(e2 - e) <= 1e-11 * abs(e)
    th0 = np.array([h for vl in hyp for h in vl] + [s2])

    def f(th):
        Ks = [O.make_Kuu(kd, th[2 * i + 1], th[2 * i], T[i]) for i, kd in enumerate(kinds)]
        return O.elbo_additive_dense(Ks, G, b, yy, n, [th[0], th[2], th[4]], th[6])

    for i in (1, 2, 6):
        h = 1e-5 * th0[i]
        e_ = np.zeros(7); e_[i] = h
        fd = (f(th0 + e_) - f(th0 - e_)) / (2 * h)
        assert abs(fd - grad[i]) <= 1e-5 * max(1.0, abs(grad[i]))
