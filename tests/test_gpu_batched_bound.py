"""Batched hyper-parameter evaluation of the 1-D bound (asvgp_kuu_assemble_batched, asvgp_elbo_grad_1d_batched,
GPR_1d.training_loss_and_gradients_batch, Scipy.minimize(starts=...)): every slot of a batch equals the single call at its
setting bit for bit, whatever B, the other slots, their order or their failure; multi-start L-BFGS takes each start's serial
iterates and reaches the notebook answer."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import scale_cases as SC  # noqa: E402

pytestmark = pytest.mark.gpu
KINDS = ("Matern12", "Matern32", "Matern52")
CHECKED = list(range(9)) + [15]         # slots 9..14 are each evaluation's own clock diagnostics


def _problem(k, m, n=200_000, D=1, seed=3):
    from asvgp_b200 import basis as B, ops

    if m == SC.C3_M:
        x, y, _ = SC.case_1d(n=n, m=m, seed=31, n_test=1)
        ys = [y] + [np.cos(x / (5.0 + d)) + 0.1 * y for d in range(1, D)]
    else:
        rng = np.random.default_rng(seed + 17 * k + m)
        x = np.sort(rng.uniform(0.0, m, n))
        ys = [np.sin(x / (7.0 + 2 * d)) + 0.2 * rng.standard_normal(n) for d in range(D)]
    basis = getattr(B, "B%dSpline" % k)(-1, m + 1, m)
    xd = ops.to_device(x)
    accs = [ops.accum_1d(xd, ops.to_device(y), basis) for y in ys]
    return basis, accs


def _settings(B, seed):
    rng = np.random.default_rng(seed)
    return rng.uniform(0.5, 2.0, B), rng.uniform(0.6, 4.0, B), rng.uniform(0.05, 0.6, B)     # v, l, sigma2


def _kind_ok(basis, kind):
    from asvgp_b200.inducing_features import kuu_terms

    return all(hasattr(basis, n) for n, _, _ in kuu_terms(kind, 1.0, 1.0))


def _single(feats, kern, basis, acc, v, l, s2, chunks):
    from asvgp_b200 import ops

    terms = feats._terms(kern, l, v)
    Kuu, dKuu = ops.kuu_assemble(basis, [t[0] for t in terms], [t[1] for t in terms], [t[2] for t in terms])
    out = ops.elbo_grad_1d_single_stream(Kuu, dKuu, acc, basis, v, s2, chunks=chunks)
    return Kuu.cpu().numpy(), dKuu.cpu().numpy(), out.cpu().numpy()


def _check_batch(basis, accs, kind, B, chunks, seed, settings=None):
    import torch

    from asvgp_b200 import kernels as Kn, ops
    from asvgp_b200.inducing_features import SplineFeatures1D

    kern = getattr(Kn, kind)()
    feats = SplineFeatures1D(kern, basis)
    v, l, s2 = settings if settings is not None else _settings(B, seed)
    Kuu, dKuu = feats.make_Kuu_device_batched(kern, l, v)
    stack = torch.stack(accs)
    out = ops.elbo_grad_1d_batched(Kuu, dKuu, stack, basis, v, s2, chunks=chunks).cpu().numpy()
    Kb, dKb = Kuu.cpu().numpy(), dKuu.cpu().numpy()
    singles = []
    for b in range(B):
        for d, acc in enumerate(accs):
            K1, dK1, o1 = _single(feats, kern, basis, acc, v[b], l[b], s2[b], chunks)
            if d == 0:
                np.testing.assert_array_equal(Kb[b], K1)
                np.testing.assert_array_equal(dKb[b], dK1)
            np.testing.assert_array_equal(out[b, d, CHECKED], o1[CHECKED], err_msg="slot %d column %d" % (b, d))
            singles.append(o1)
    return out, singles


@pytest.mark.parametrize("k", [1, 2, 3, 4, 5, 6])
def test_every_order_and_kernel_bitwise(cuda, k):
    basis, accs = _problem(k, 1000)
    kinds = [kind for kind in KINDS if _kind_ok(basis, kind)]
    assert kinds
    for i, kind in enumerate(kinds):
        out, _ = _check_batch(basis, accs, kind, 7, 0, seed=100 * k + i)
        assert (out[:, 0, 8] == 0).all()


@pytest.mark.parametrize("m,chunks,B", [(100, 0, 24), (100, 1, 2), (100, 3, 7), (1000, 0, 1), (1000, 3, 64), (1000, 256, 7),
                                        (SC.C3_M, 0, 64), (SC.C3_M, 1, 2), (SC.C3_M, 3, 7), (SC.C3_M, 256, 24),
                                        (SC.C3_M, 512, 7), (SC.C3_M, 1024, 2)])
def test_layouts_and_batch_sizes_bitwise(cuda, m, chunks, B):
    basis, accs = _problem(3, m)
    out, _ = _check_batch(basis, accs, "Matern52", B, chunks, seed=m + chunks + B)
    assert (out[:, 0, 8] == 0).all()


def test_multi_column_bitwise(cuda):
    basis, accs = _problem(3, SC.C3_M, D=3)
    _check_batch(basis, accs, "Matern32", 7, 0, seed=9)


def test_permuted_batch_permutes_outputs(cuda):
    import torch

    from asvgp_b200 import kernels as Kn, ops
    from asvgp_b200.inducing_features import SplineFeatures1D

    basis, accs = _problem(3, SC.C3_M, D=2)
    kern = Kn.Matern52()
    feats = SplineFeatures1D(kern, basis)
    v, l, s2 = _settings(24, 5)
    stack = torch.stack(accs)
    Kuu, dKuu = feats.make_Kuu_device_batched(kern, l, v)
    out = ops.elbo_grad_1d_batched(Kuu, dKuu, stack, basis, v, s2).cpu().numpy()
    perm = np.random.default_rng(6).permutation(24)
    Kp, dKp = feats.make_Kuu_device_batched(kern, l[perm], v[perm])
    outp = ops.elbo_grad_1d_batched(Kp, dKp, stack, basis, v[perm], s2[perm]).cpu().numpy()
    np.testing.assert_array_equal(outp[:, :, CHECKED], out[perm][:, :, CHECKED])
    # and a prefix of the batch (another B) gives the same bits
    out7 = ops.elbo_grad_1d_batched(Kuu[:7].contiguous(), dKuu[:7].contiguous(), stack, basis, v[:7], s2[:7]).cpu().numpy()
    np.testing.assert_array_equal(out7[:, :, CHECKED], out[:7][:, :, CHECKED])


def test_failed_slot_keeps_the_others(cuda, golden):
    from asvgp_b200 import basis as B, kernels as Kn, ops
    from asvgp_b200.inducing_features import SplineFeatures1D

    g = golden("snelson")
    basis = B.B3Spline(-3.5, 10.5, 100)
    acc = ops.accum_1d(ops.to_device(g["X"].reshape(-1)), ops.to_device(g["y"].reshape(-1)), basis)
    bad = None
    for kind in ("Matern52", "Matern32"):
        kern = getattr(Kn, kind)()
        feats = SplineFeatures1D(kern, basis)
        for ell in (1e2, 1e3, 1e4, 1e5, 1e6):
            info = _single(feats, kern, basis, acc, 1.0, ell, 0.1, 0)[2][8]
            if info != 0:
                bad = (kind, ell)
                break
        if bad:
            break
    assert bad is not None, "no failing setting found"
    kind, ell = bad
    v, l, s2 = _settings(5, 8)
    l[2] = ell
    v[2], s2[2] = 1.0, 0.1
    out, singles = _check_batch(basis, [acc], kind, 5, 0, seed=0, settings=(v, l, s2))
    assert out[2, 0, 8] != 0 and out[2, 0, 8] == singles[2][8]
    assert all(out[b, 0, 8] == 0 for b in (0, 1, 3, 4))
    # through the model: +inf loss, NaN gradients, the pivot in info; nothing raised, parameters untouched
    from asvgp_b200.gpr import GPR_1d

    kern = getattr(Kn, kind)()
    model = GPR_1d((g["X"].reshape(-1, 1), g["y"].reshape(-1, 1)), kern, basis)
    before = [p.unconstrained for p in model.trainable_variables]
    U = np.array([[Kn._inv_softplus(v[b]), Kn._inv_softplus(l[b]), Kn._inv_softplus(s2[b] - 1e-6)] for b in range(5)])
    loss, grad, info = model.training_loss_and_gradients_batch(U)
    assert [p.unconstrained for p in model.trainable_variables] == before
    assert loss[2] == np.inf and np.isnan(grad[2]).all() and info[2] != 0
    assert np.isfinite(loss[[0, 1, 3, 4]]).all() and (info[[0, 1, 3, 4]] == 0).all()


def _model_rows_equal_single(model, U):
    before = [p.unconstrained for p in model.trainable_variables]
    loss, grad, info = model.training_loss_and_gradients_batch(U)
    assert [p.unconstrained for p in model.trainable_variables] == before
    assert (info == 0).all()
    for b, u in enumerate(U):
        for p, ui in zip(model.trainable_variables, u):
            p.unconstrained = float(ui)
        l1, g1 = model.training_loss_and_gradients()
        assert loss[b] == l1, b
        np.testing.assert_array_equal(grad[b], g1)
    for p, ui in zip(model.trainable_variables, before):
        p.unconstrained = ui


def test_model_rows_equal_training_loss_and_gradients(cuda, golden):
    from asvgp_b200 import basis as B, kernels as Kn
    from asvgp_b200.gpr import GPR_1d

    g = golden("snelson")
    for kind in KINDS:
        model = GPR_1d((g["X"].reshape(-1, 1), g["y"].reshape(-1, 1)), getattr(Kn, kind)(), B.B3Spline(-3.5, 10.5, 100))
        U = np.random.default_rng(12).uniform(-1.5, 1.5, (24, 3))
        _model_rows_equal_single(model, U)
    model = GPR_1d((g["X"].reshape(-1, 1), g["y"].reshape(-1, 1)), Kn.Matern32(), B.B3Spline(-3.5, 10.5, 100), chunks=3)
    _model_rows_equal_single(model, np.random.default_rng(13).uniform(-1.0, 1.0, (64, 3)))


def test_multi_output_model_rows(cuda, golden):
    from asvgp_b200 import basis as B, kernels as Kn
    from asvgp_b200.gpr import GPR_1d

    g = golden("multi_output_1d")
    m = int(g["m"])
    model = GPR_1d((g["x"].reshape(-1, 1), g["y"]), Kn.Matern52(), B.B3Spline(-1, m + 1, m))
    assert g["y"].shape[1] == 3
    _model_rows_equal_single(model, np.random.default_rng(14).uniform(-1.0, 1.5, (7, 3)))


def test_multi_start_snelson(cuda, golden):
    from asvgp_b200 import basis as B, kernels as Kn
    from asvgp_b200.gpr import GPR_1d
    from asvgp_b200.optimizers import Scipy

    g = golden("snelson")

    def fresh():
        return GPR_1d((g["X"].reshape(-1, 1), g["y"].reshape(-1, 1)), Kn.Matern32(), B.B3Spline(-3.5, 10.5, 100))

    model = fresh()
    default = [p.unconstrained for p in model.trainable_variables]
    starts = np.vstack([default, np.random.default_rng(15).uniform(-1.5, 1.5, (5, 3))])
    res = Scipy().minimize(model.training_loss, model.trainable_variables, starts=starts)
    assert abs(model.elbo() - float(g["notebook_elbo"])) < 1e-6
    assert abs(-res.fun - float(g["notebook_elbo"])) < 1e-6
    for u0, r in zip(starts, res.results):
        ref_model = fresh()
        for p, u in zip(ref_model.trainable_variables, u0):
            p.unconstrained = float(u)
        try:
            ref = Scipy().minimize(ref_model.training_loss, ref_model.trainable_variables)
        except np.linalg.LinAlgError:
            assert r.fun == np.inf and not r.success
            continue
        np.testing.assert_array_equal(r.x, ref.x)
        assert r.nit == ref.nit and r.fun == ref.fun
