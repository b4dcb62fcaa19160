"""Generates tests/golden/*.npz by running the UNMODIFIED reference (/root/reference/asvgp) under the
numpy/SciPy stand-ins of oracle/shim ("reference-under-shim").  Build-container only; the committed .npz files
are what travels.  Usage:  python oracle/make_golden.py

TEST INFRASTRUCTURE ONLY.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import scale_cases as SC  # noqa: E402
from oracle import ref_under_shim  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
KINDS = ("Matern12", "Matern32", "Matern52")


def set_hypers(ns, model, kernels, hypers, sigma2):
    for kern, (v, l) in zip(kernels, hypers):
        kern.variance = kern.variance * 0 + v
        kern.lengthscales = kern.lengthscales * 0 + l
    model.likelihood.variance = model.likelihood.variance * 0 + sigma2


def snelson(ns):
    d = os.path.join(ref_under_shim.REFERENCE_ROOT, "experiments", "snelson", "data")
    X = np.loadtxt(os.path.join(d, "train_inputs")).reshape(-1, 1)
    y = np.loadtxt(os.path.join(d, "train_outputs")).reshape(-1, 1)
    Xt = np.loadtxt(os.path.join(d, "test_inputs")).reshape(-1, 1)
    out = dict(X=X, y=y, Xtest=Xt, a=-3.5, b=10.5, m=100, order=3,
               notebook_elbo=-60.8356263428725, notebook_exact_gp=-60.573988814770104,
               opt_hypers=np.array([0.7981456786, 1.0268804385, 0.0800658741]))
    basis = ns.basis.B3Spline(-3.5, 10.5, 100)
    out["mesh"] = np.asarray(basis.mesh)
    out["delta"] = float(basis.delta)
    for name in ("A", "B", "C", "D", "BC", "BC_grad", "BC_ggrad", "BC_ggrad_none", "BC_none_ggrad"):
        out["tab_" + name] = np.asarray(getattr(basis, name))
    for kind in KINDS:
        kern = getattr(ns.gpflow.kernels, kind)()
        model = ns.gpr.GPR_1d((X, y), kern, basis)
        out["elbo111_" + kind] = float(model.elbo())
        out["Kuu111_" + kind] = np.asarray(model.inducing_features.make_Kuu(kern))
        set_hypers(ns, model, [kern], [(0.8, 1.03)], 0.08)
        out["elbo_b_" + kind] = float(model.elbo())
    out["G"] = np.asarray(model.KufKfu)
    out["Kuf_y"] = np.asarray(model.Kuf_y)
    out["tr_yTy"] = float(model.tr_yTy)
    kern = ns.gpflow.kernels.Matern32()
    model = ns.gpr.GPR_1d((X, y), kern, basis)
    v, l, s2 = out["opt_hypers"]
    set_hypers(ns, model, [kern], [(v, l)], s2)
    out["elbo_opt"] = float(model.elbo())
    mu, var = model.predict_f(Xt)
    out["pred_mean"], out["pred_var"] = np.asarray(mu), np.asarray(var)
    np.savez_compressed(os.path.join(OUT, "snelson.npz"), **out)
    print("snelson: elbo_opt", out["elbo_opt"], "M32(1,1,1)", out["elbo111_Matern32"])


def basis_eval(ns):
    rng = np.random.default_rng(7)
    out = {}
    for k in range(1, 7):
        for (a, b, m, tag) in ((-3.5, 10.5, 40, "f32"), (-1, 41, 40, "f64")):
            basis = getattr(ns.basis, "B%dSpline" % k)(a, b, m)
            lo, hi = float(a), float(b)
            x = rng.uniform(lo + 1e-3, hi - 1e-3, 257)
            x[:5] = np.asarray(basis.mesh)[[1, 2, 5, 7, 11]]          # points exactly on knots (Q2)
            key = "k%d_%s" % (k, tag)
            out[key + "_x"] = x
            out[key + "_mesh"] = np.asarray(basis.mesh)
            for dx in range(0, 4):
                if dx > k or (k == 1 and dx == 1) or (k == 2 and dx == 2) or (k == 6 and dx > 0):
                    continue                                         # Q10/Q11: broken or inaccurate upstream
                out[key + "_dx%d" % dx] = basis.evaluate_basis(x.reshape(-1, 1), dx=dx).toarray()
            for name in ("A", "B", "C", "D", "BC", "BC_grad", "BC_ggrad"):
                if hasattr(basis, name) and not (k == 6 and name == "BC_grad"):
                    out[key + "_" + name] = np.asarray(getattr(basis, name))
    np.savez_compressed(os.path.join(OUT, "basis_eval.npz"), **out)
    print("basis_eval:", len(out), "arrays")


def synth_1d(ns):
    """C2-shaped small case: x ~ U(0, m) on (a,b)=(-1, m+1) (int endpoints -> f64 mesh), random order.  The inputs come
    from tests/scale_cases.py (seeded numpy); the tests regenerate them, so only every SYNTH_1D_SAMPLE-th point is stored."""
    out = {}
    inputs = SC.synth_1d_inputs()
    for k, m in SC.SYNTH_1D:
        x, y, xs = inputs[k]
        basis = getattr(ns.basis, "B%dSpline" % k)(-1, m + 1, m)
        key = "k%d" % k
        out[key + "_x_sample"], out[key + "_y_sample"] = x[::SC.SYNTH_1D_SAMPLE], y[::SC.SYNTH_1D_SAMPLE]
        out[key + "_m"] = m
        for kind in KINDS:
            need = {"Matern12": 1, "Matern32": 2, "Matern52": 3}[kind]
            if k < need:
                continue
            kern = getattr(ns.gpflow.kernels, kind)()
            last_kind = kind
            model = ns.gpr.GPR_1d((x.reshape(-1, 1), y.reshape(-1, 1)), kern, basis)
            for tag, (v, l, s2) in (("a", (1.0, 1.0, 0.1)), ("b", (1.3, 2.5, 0.7))):
                set_hypers(ns, model, [kern], [(v, l)], s2)
                out["%s_%s_elbo_%s" % (key, kind, tag)] = float(model.elbo())
        out[key + "_G"] = np.asarray(model.KufKfu)
        out[key + "_Kuf_y"] = np.asarray(model.Kuf_y)
        out[key + "_tr_yTy"] = float(model.tr_yTy)
        mu, var = model.predict_f(xs)
        out[key + "_xs"], out[key + "_mean"], out[key + "_var"] = xs, np.asarray(mu), np.asarray(var)
        out[key + "_pred_hypers"] = np.array([1.3, 2.5, 0.7])
        out[key + "_pred_kind"] = last_kind
    np.savez_compressed(os.path.join(OUT, "synth_1d.npz"), **out)
    print("synth_1d:", len(out), "arrays")


def kron_2d(ns):
    out = {}
    rng = np.random.default_rng(0)
    N = 3000
    x1 = rng.uniform(.01, .99, N)
    x2 = rng.uniform(.01, 1.99, N)
    y = (np.sin(6 * x1) * np.cos(3 * x2) + 0.1 * rng.standard_normal(N)).reshape(-1, 1)
    X = np.stack([x1, x2], 1)
    out.update(X=X, y=y)
    for k, m in ((3, 14), (4, 14), (2, 10)):
        B = getattr(ns.basis, "B%dSpline" % k)
        bases = [B(0, 1, m), B(0, 2, m)]
        ks = [ns.gpflow.kernels.Matern32(), ns.gpflow.kernels.Matern32()]
        import contextlib, io
        with contextlib.redirect_stdout(io.StringIO()):
            model = ns.gpr.GPR_kron((X, y), ks, bases)
        set_hypers(ns, model, ks, [(.7, .3), (1.3, .5)], .05)
        key = "k%d" % k
        out[key + "_m"] = m
        out[key + "_elbo"] = float(model.elbo())
        out[key + "_bandwidth"] = model.bandwidth
        G = model.KufKfu_sparse.tocoo()
        out[key + "_G_row"], out[key + "_G_col"], out[key + "_G_val"] = G.row, G.col, G.data
        out[key + "_Kuf_y"] = np.asarray(model.Kuf_y)
        out[key + "_tr_yTy"] = float(model.tr_yTy)
        Xs = np.stack([rng.uniform(.02, .98, 40), rng.uniform(.02, 1.98, 40)], 1)
        mu, var = model.predict_f(Xs)
        mu2, var2 = model.predict_f_sparse(Xs)
        assert np.allclose(np.asarray(mu), np.asarray(mu2), atol=1e-11) and np.allclose(np.asarray(var), np.asarray(var2), atol=1e-11)
        out[key + "_Xs"], out[key + "_mean"], out[key + "_var"] = Xs, np.asarray(mu), np.asarray(var)
        ks2 = [ns.gpflow.kernels.Matern52(), ns.gpflow.kernels.Matern12()]
        if k >= 3:
            with contextlib.redirect_stdout(io.StringIO()):
                model2 = ns.gpr.GPR_kron((X, y), ks2, bases)
            set_hypers(ns, model2, ks2, [(.9, .4), (1.1, .6)], .2)
            out[key + "_elbo_m52_m12"] = float(model2.elbo())
    np.savez_compressed(os.path.join(OUT, "kron_2d.npz"), **out)
    print("kron_2d:", {k: v for k, v in out.items() if k.endswith("elbo")})


def multi_output_1d(ns):
    """y with D = 3 columns (reference gpr.py:39-44,78-85 carry D through Kuf_y, tr_yTy and the bound)."""
    out = {}
    rng = np.random.default_rng(2024)
    n, m, k = 6000, 48, 3
    x = rng.uniform(0.0, m, n)
    f = np.stack([np.sin(2 * np.pi * x / 17), np.cos(2 * np.pi * x / 5.3), 0.02 * x], 1)
    y = f + 0.2 * rng.standard_normal((n, 3))
    basis = ns.basis.B3Spline(-1, m + 1, m)
    out.update(x=x, y=y, m=m, order=k)
    for kind in KINDS:
        kern = getattr(ns.gpflow.kernels, kind)()
        model = ns.gpr.GPR_1d((x.reshape(-1, 1), y), kern, basis)
        for tag, (v, l, s2) in (("a", (1.0, 1.0, 0.1)), ("b", (0.6, 3.5, 0.3))):
            set_hypers(ns, model, [kern], [(v, l)], s2)
            out["elbo_%s_%s" % (kind, tag)] = float(model.elbo())
    out["Kuf_y"] = np.asarray(model.Kuf_y)
    out["tr_yTy"] = float(model.tr_yTy)
    xs = rng.uniform(0.5, m - 0.5, 50).reshape(-1, 1)
    mu, var = model.predict_f(xs)
    out["xs"], out["mean"], out["var"] = xs, np.asarray(mu), np.asarray(var)
    out["pred_hypers"] = np.array([0.6, 3.5, 0.3])
    np.savez_compressed(os.path.join(OUT, "multi_output_1d.npz"), **out)
    print("multi_output_1d: Kuf_y", out["Kuf_y"].shape, "mean", out["mean"].shape, out["elbo_Matern52_b"])




def additive(ns):
    """GPR_additive (reference gpr.py:139-236) on a small 3-D synthetic set: Gram, projection, bound at two sets of
    hyper-parameters and kernel mixes, predictions."""
    rng = np.random.default_rng(12)
    n, m, k = 4000, 24, 3
    doms = [(0, 1), (0, 2), (-1, 1)]
    X = np.stack([rng.uniform(a + 0.01, b - 0.01, n) for a, b in doms], 1)
    y = (np.sin(5 * X[:, 0]) + np.cos(3 * X[:, 1]) + X[:, 2] ** 2 + 0.1 * rng.standard_normal(n)).reshape(-1, 1)
    Xs = np.stack([rng.uniform(a + 0.02, b - 0.02, 60) for a, b in doms], 1)
    out = dict(X=X, y=y, Xs=Xs, m=m, order=k, doms=np.array(doms, dtype=np.float64))
    for tag, kinds, hypers, s2 in (("a", ("Matern32",) * 3, [(1.0, 1.0)] * 3, 1.0),
                                   ("b", ("Matern52", "Matern12", "Matern32"), [(.7, .3), (1.3, .5), (.9, .8)], .05)):
        bases = [ns.basis.B3Spline(a, b, m) for a, b in doms]
        kerns = [getattr(ns.gpflow.kernels, kind)() for kind in kinds]
        model = ns.gpr.GPR_additive((X, y), kerns, bases)
        set_hypers(ns, model, kerns, hypers, s2)
        out["elbo_" + tag] = float(np.asarray(model.elbo()))
        mean, var = model.predict_f(Xs)
        out["mean_" + tag], out["var_" + tag] = np.asarray(mean), np.asarray(var)
    out["KufKfu"] = np.asarray(model.KufKfu)
    out["Kuf_y"] = np.asarray(model.Kuf_y)
    out["tr_yTy"] = float(np.asarray(model.tr_yTy))
    np.savez_compressed(os.path.join(OUT, "additive_3d.npz"), **out)
    print("additive: elbo", out["elbo_a"], out["elbo_b"], "mean", out["mean_b"].shape, "var", out["var_b"].shape)


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    ns = ref_under_shim.load()
    only = sys.argv[1:]
    for fn in (snelson, basis_eval, synth_1d, kron_2d, multi_output_1d, additive):
        if not only or fn.__name__ in only:
            fn(ns)
