"""Batched hyper-parameter evaluation of the 2-D Kronecker bound (asvgp_band_inverse_1d_batched, asvgp_kron_*_batched,
GPR_kron.training_loss_and_gradients_batch, Scipy.minimize(starts=...)).  The per-dimension pieces are deterministic and are
compared bit for bit; the factorisation of P adds children's updates into their parent front with fp64 REDs, so every slot is
compared with the single call at the project's 2-D tolerances (DESIGN §3): relative 1e-10 on the loss, 1e-8 on each gradient."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
DOMAINS = ((0, 1), (0, 2))
BENCH_DOMAINS = ((-80, -25), (15, 55))        # bench.py's 2-D workload (eNATL60 domains) and its hypers
BENCH_HYPERS = ((1.0, 5.0), (1.0, 4.0), 0.01)
GOLDEN_KINDS = {2: ("Matern12", "Matern32"), 3: ("Matern52", "Matern12"), 4: ("Matern32", "Matern52")}


def _model(X, y, k, ms, kinds, domains=DOMAINS, shared=False):
    from asvgp_b200 import basis as B, kernels as Kn
    from asvgp_b200.gpr import GPR_kron

    cls = getattr(B, "B%dSpline" % k)
    bases = [cls(domains[0][0], domains[0][1], ms[0]), cls(domains[1][0], domains[1][1], ms[1])]
    kerns = [getattr(Kn, kinds[0])()] * 2 if shared else [getattr(Kn, kind)() for kind in kinds]
    return GPR_kron((X, y.reshape(len(X), -1)), kerns, bases)


def _golden_model(golden, k, kinds=None, shared=False):
    g = golden("kron_2d")
    m = int(g["k%d_m" % k])
    return _model(g["X"], g["y"], k, (m, m), kinds or GOLDEN_KINDS[k], shared=shared)


def _synth(n, domains, seed=5, D=1):
    rng = np.random.default_rng(seed)
    lo, hi = np.array([d[0] for d in domains]), np.array([d[1] for d in domains])
    X = lo + (hi - lo) * rng.uniform(0.02, 0.98, (n, 2))
    u = (X - lo) / (hi - lo)
    cols = [np.sin(6 * u[:, 0] + d) * np.cos(4 * u[:, 1]) + 0.1 * rng.standard_normal(n) for d in range(D)]
    return X, np.stack(cols, 1)


def _settings(model, B, seed, scale=1.0):
    """U[B, G]: random unconstrained settings (variances 0.5..2, lengthscales scale * 0.2..0.8, sigma2 0.02..0.2)."""
    from asvgp_b200.kernels import _inv_softplus

    rng = np.random.default_rng(seed)
    lengths = {id(k.lengthscales) for k in model.kernels}
    cols = []
    for p in model.trainable_variables:
        if p is model.likelihood.variance:
            v = rng.uniform(0.02, 0.2, B)
        elif id(p) in lengths:
            v = scale * rng.uniform(0.2, 0.8, B)
        else:
            v = rng.uniform(0.5, 2.0, B)
        cols.append([_inv_softplus(x - p.lower) for x in v])
    return np.array(cols).T


def _serial(model, U):
    """training_loss_and_gradients at every row of U (the parameters are restored afterwards)."""
    params = model.trainable_variables
    before = [p.unconstrained for p in params]
    out = []
    for u in U:
        for p, ui in zip(params, u):
            p.unconstrained = float(ui)
        out.append(model.training_loss_and_gradients())
    for p, ui in zip(params, before):
        p.unconstrained = ui
    return np.array([o[0] for o in out]), np.array([o[1] for o in out])


def _assert_close(loss, grad, want_loss, want_grad):
    for b in range(len(loss)):
        assert abs(loss[b] - want_loss[b]) <= 1e-10 * abs(want_loss[b]), (b, loss[b], want_loss[b])
        np.testing.assert_allclose(grad[b], want_grad[b], rtol=1e-8, atol=1e-8 * np.abs(want_grad[b]).max())


def _check_batch(model, U, **kw):
    params = model.trainable_variables
    before = [p.unconstrained for p in params]
    loss, grad, info = model.training_loss_and_gradients_batch(U, **kw)
    assert [p.unconstrained for p in params] == before
    assert loss.shape == (len(U),) and grad.shape == (len(U), len(params)) and (info == 0).all()
    _assert_close(loss, grad, *_serial(model, U))
    return loss, grad


# ---- 1. deterministic per-dimension pieces, bit for bit ------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 2, 3, 4, 5, 6])
@pytest.mark.parametrize("m", [40, 200])
def test_band_inverse_batched_is_bitwise_single(cuda, k, m):
    import torch

    from asvgp_b200 import basis as B, kernels as Kn, ops
    from asvgp_b200.inducing_features import SplineFeatures1D, kuu_terms

    basis = getattr(B, "B%dSpline" % k)(0.0, 1.0, m)
    kinds = [kd for kd in ("Matern12", "Matern32", "Matern52") if all(hasattr(basis, n) for n, _, _ in kuu_terms(kd, 1.0, 1.0))]
    assert kinds
    for kind in kinds:
        kern = getattr(Kn, kind)()
        feats = SplineFeatures1D(kern, basis)
        rng = np.random.default_rng(k * 100 + m)
        ells, vs = rng.uniform(0.05, 0.5, 6), rng.uniform(0.5, 2.0, 6)
        K, dK = feats.make_Kuu_device_batched(kern, ells, vs)
        S, dS, sc = ops.band_inverse_1d_batched(K, dK, basis)
        torch.cuda.synchronize()
        for b in range(6):
            terms = feats._terms(kern, ells[b], vs[b])
            K1, dK1 = ops.kuu_assemble(basis, [t[0] for t in terms], [t[1] for t in terms], [t[2] for t in terms])
            assert torch.equal(K[b], K1) and torch.equal(dK[b], dK1)
            S1, dS1, sc1 = ops.band_inverse_1d(K1, dK1, basis)
            assert torch.equal(S[b], S1) and torch.equal(dS[b], dS1) and torch.equal(sc[b], sc1), (kind, b)
            assert sc1[2].item() == 0


# ---- 2. every slot equals the single call ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [2, 3, 4])
@pytest.mark.parametrize("B", [1, 7, 24])
def test_golden_slots_match_single(cuda, golden, k, B):
    model = _golden_model(golden, k)
    _check_batch(model, _settings(model, B, seed=10 * k + B))


def test_three_output_columns(cuda):
    X, y = _synth(6000, DOMAINS, D=3)
    model = _model(X, y, 3, (14, 14), ("Matern32", "Matern52"))
    assert model.n_outputs == 3
    _check_batch(model, _settings(model, 5, seed=3))


def test_unequal_grid(cuda):
    X, y = _synth(20000, DOMAINS, seed=7)
    model = _model(X, y, 3, (40, 36), ("Matern52", "Matern32"))
    _check_batch(model, _settings(model, 6, seed=4))


def test_shared_kernel_object(cuda, golden):
    model = _golden_model(golden, 3, kinds=("Matern32", "Matern32"), shared=True)
    assert len(model.trainable_variables) == 3
    _check_batch(model, _settings(model, 5, seed=5))


def test_bench_shape_200x200(cuda):
    from asvgp_b200.kernels import _inv_softplus

    X, y = _synth(400_000, BENCH_DOMAINS, seed=11)
    model = _model(X, y, 3, (200, 200), ("Matern32", "Matern32"), domains=BENCH_DOMAINS)
    (v1, l1), (v2, l2), s2 = BENCH_HYPERS
    base = np.array([v1, l1, v2, l2, s2])
    U = np.array([[_inv_softplus(x * f) for x in base] for f in (1.0, 0.9, 1.1, 1.25)])
    _check_batch(model, U)


# ---- 3. slots are independent ----------------------------------------------------------------------------------------------------
def test_permuted_repeated_and_grouped(cuda, golden):
    model = _golden_model(golden, 3)
    U = _settings(model, 9, seed=21)
    loss, grad, _ = model.training_loss_and_gradients_batch(U)
    perm = np.random.default_rng(0).permutation(9)
    lp, gp, ip = model.training_loss_and_gradients_batch(U[perm])
    assert (ip == 0).all()
    _assert_close(lp, gp, loss[perm], grad[perm])
    lr, gr, ir = model.training_loss_and_gradients_batch(np.repeat(U[4:5], 6, axis=0))
    assert (ir == 0).all()
    _assert_close(lr, gr, np.repeat(loss[4:5], 6), np.repeat(grad[4:5], 6, axis=0))
    lg, gg, ig = model.training_loss_and_gradients_batch(U, max_slots=2)
    assert (ig == 0).all()
    _assert_close(lg, gg, loss, grad)


# ---- 4. a failing slot ------------------------------------------------------------------------------------------------------------
def _failing_setting(model):
    """A lengthscale at which a factorisation fails (found by search, as the 1-D batch test does), as an unconstrained row."""
    from asvgp_b200.kernels import _inv_softplus

    params = model.trainable_variables
    base = _settings(model, 1, seed=1)[0]
    j = next(i for i, p in enumerate(params) if p is model.kernels[0].lengthscales)
    for ell in (1e2, 1e3, 1e4, 1e5, 1e6):
        u = base.copy()
        u[j] = _inv_softplus(ell)
        for p, ui in zip(params, u):
            p.unconstrained = float(ui)
        try:
            model.training_loss_and_gradients()
        except np.linalg.LinAlgError:
            return u
    return None


def test_failed_slot_keeps_the_others(cuda, golden):
    model = _golden_model(golden, 3, kinds=("Matern52", "Matern32"))
    before = [p.unconstrained for p in model.trainable_variables]
    bad = _failing_setting(model)
    for p, ui in zip(model.trainable_variables, before):
        p.unconstrained = ui
    assert bad is not None, "no failing setting found"
    U = _settings(model, 5, seed=31)
    U[2] = bad
    loss, grad, info = model.training_loss_and_gradients_batch(U)
    assert [p.unconstrained for p in model.trainable_variables] == before
    assert loss[2] == np.inf and np.isnan(grad[2]).all() and info[2] != 0
    ok = [0, 1, 3, 4]
    assert (info[ok] == 0).all() and np.isfinite(loss[ok]).all()
    _assert_close(loss[ok], grad[ok], *_serial(model, U[ok]))


# ---- 5. multi-start L-BFGS -----------------------------------------------------------------------------------------------------------
def test_multi_start_lbfgs(cuda, golden):
    from asvgp_b200.optimizers import Scipy

    model = _golden_model(golden, 3)
    before = [p.unconstrained for p in model.trainable_variables]
    bad = _failing_setting(model)
    assert bad is not None
    starts = _settings(model, 4, seed=41)
    starts[3] = bad
    opts = dict(options={"maxiter": 40})
    for p, ui in zip(model.trainable_variables, before):
        p.unconstrained = ui
    res = Scipy().minimize(model.training_loss, model.trainable_variables, starts=starts, **opts)
    assert res.results[3].fun == np.inf and not res.results[3].success
    finite = [b for b in range(3) if np.isfinite(res.results[b].fun)]
    assert len(finite) == 3
    best = min(finite, key=lambda b: res.results[b].fun)
    assert res.best == best
    np.testing.assert_array_equal([p.unconstrained for p in model.trainable_variables], res.results[best].x)
    for b in range(3):
        for p, ui in zip(model.trainable_variables, starts[b]):
            p.unconstrained = float(ui)
        serial = Scipy().minimize(model.training_loss, model.trainable_variables, **opts)
        assert abs(serial.fun - res.results[b].fun) <= 1e-6 * max(1.0, abs(serial.fun))
        np.testing.assert_allclose(res.results[b].x, serial.x, rtol=1e-6, atol=1e-6)
