"""float32 training data read natively by the accumulate kernels (asvgp_*_typed): every result equals the same call on the
float64-converted data up to summation order (1e-11 x max |entry|, counts exact), for each of the four (x, y) dtype pairs,
on the device, binned, host-staged and through the models."""
import numpy as np
import pytest

from oracle import asvgp_oracle as O

pytestmark = pytest.mark.gpu

PAIRS = [("f64", "f64"), ("f64", "f32"), ("f32", "f64"), ("f32", "f32")]
TOL = 1e-11


def _dt(name):
    import torch

    return {"f64": torch.float64, "f32": torch.float32}[name]


def _basis(k, a, b, m):
    from asvgp_b200 import basis as B

    return getattr(B, "B%dSpline" % k)(a, b, m)


def _same(got, want, tol=TOL):
    """Equal up to summation order: |got - want| <= tol * max |want|, counts (the last entry) exact."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    scale = max(float(np.abs(want).max()) if want.size else 0.0, 1e-300)
    assert float(np.abs(got - want).max()) <= tol * scale if want.size else True
    assert got[-1] == want[-1]


def _acc1(x, y, basis, **kw):
    from asvgp_b200 import ops

    return ops.accum_1d(x, y, basis, **kw).cpu().numpy()


def _points_1d(rng, n, m, kind):
    x = rng.uniform(0.0, m, n)
    if kind == "sorted":
        x.sort()
    else:                                   # sorted, but every 5th point jumps to a random interval (the RED path)
        x.sort()
        jump = np.arange(n) % 5 == 3
        x[jump] = rng.uniform(0.0, m, int(jump.sum()))
    y = np.cos(x / 7.0) + 0.2 * rng.standard_normal(n)
    return x, y


# ---- 1-D streaming ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 2, 3, 4, 5, 6])
@pytest.mark.parametrize("xd,yd", PAIRS)
def test_accum_1d_streaming_dtype_pairs(cuda, k, xd, yd):
    import torch

    m = 300
    basis = _basis(k, -1, m + 1, m)
    rng = np.random.default_rng(10 * k + PAIRS.index((xd, yd)))
    for n in (0, 1, 3, 4 * 1031 + 1, 1_000_003):
        for kind in ("sorted", "jumps"):
            x, y = _points_1d(rng, n + 1, m, kind)
            xt = torch.from_numpy(x).to(cuda, _dt(xd))
            yt = torch.from_numpy(y).to(cuda, _dt(yd))
            for off in (0, 1):                          # off = 1: misaligned views, scalar loads
                xs, ys = xt[off:off + n], yt[off:off + n]
                assert xs.dtype == _dt(xd) and ys.dtype == _dt(yd)
                want = _acc1(xs.double(), ys.double(), basis)
                _same(_acc1(xs, ys, basis), want)
                if n == 4 * 1031 + 1 and kind == "sorted" and off == 0 and k == 3:
                    G0, b0, yy0 = O.precompute_1d(basis.mesh, basis.delta, k, m, xs.double().cpu().numpy(), ys.double().cpu().numpy())
                    G = want[: (k + 1) * m].reshape(k + 1, m)
                    np.testing.assert_allclose(G, G0, rtol=1e-10, atol=1e-10 * np.abs(G0).max())


@pytest.mark.parametrize("xd,yd", PAIRS)
def test_accum_1d_shards_add_up(cuda, xd, yd):
    import torch

    from asvgp_b200 import ops

    m, n = 500, 300_001
    basis = _basis(3, -1, m + 1, m)
    x, y = _points_1d(np.random.default_rng(3), n, m, "sorted")
    xt, yt = torch.from_numpy(x).to(cuda, _dt(xd)), torch.from_numpy(y).to(cuda, _dt(yd))
    acc = ops.accum_1d(xt[: n // 3], yt[: n // 3], basis)
    ops.accum_1d(xt[n // 3:], yt[n // 3:], basis, acc=acc)
    _same(acc.cpu().numpy(), _acc1(xt.double(), yt.double(), basis))


@pytest.mark.parametrize("xd,yd", [("f32", "f32"), ("f64", "f32")])
def test_accum_1d_binned_large(cuda, xd, yd):
    """2e7 shuffled points as test_accum_binned_large_matches_streaming, in float32: partition path, "auto" (which must
    choose as it does for the float64 copy) and the float64-converted data agree; partition of unity holds."""
    import torch

    from asvgp_b200 import ops

    m, n = 10_000, 20_000_000
    basis = _basis(3, -1, m + 1, m)
    g = torch.Generator(device="cuda"); g.manual_seed(7)
    x = (torch.rand(n, dtype=torch.float64, device="cuda", generator=g) * m).to(_dt(xd))
    y = (torch.sin(x.double() / 37.0) + 0.25).to(_dt(yd))
    want = ops.accum_1d(x.double(), y.double(), basis, binned=True)
    a_bin = ops.accum_1d(x, y, basis, binned=True)
    a_auto = ops.accum_1d(x, y, basis, binned="auto")
    assert ops.order_probe_1d(x, basis) == ops.order_probe_1d(x.double(), basis)
    for got in (a_bin, a_auto):
        _same(got.cpu().numpy(), want.cpu().numpy())
    G, b, scal = ops.split_accum_1d(a_bin, basis)
    assert scal[1].item() == n
    total = float(G[0].sum() + 2 * G[1:].sum())
    assert abs(total - n) <= 1e-10 * n
    assert abs(float(b.sum()) - float(y.double().sum())) <= 1e-10 * float(y.double().abs().sum())


@pytest.mark.parametrize("xd,yd", PAIRS)
def test_accum_1d_host_path(cuda, xd, yd):
    """numpy and pinned host arrays in their own dtypes, small chunks, odd n: the same sums as the device path."""
    import torch

    from asvgp_b200 import ops

    m, n = 200, 100_001
    basis = _basis(4, -1, m + 1, m)
    x, y = _points_1d(np.random.default_rng(5), n, m, "jumps")
    npx = x.astype(np.float32) if xd == "f32" else x
    npy = y.astype(np.float32) if yd == "f32" else y
    want = _acc1(torch.from_numpy(npx).cuda().double(), torch.from_numpy(npy).cuda().double(), basis)
    _same(ops.accum_1d_host(npx, npy, basis, chunk=7_777).cpu().numpy(), want)
    px, py = torch.from_numpy(npx).pin_memory(), torch.from_numpy(npy).pin_memory()
    _same(ops.accum_1d_host(px, py, basis, chunk=10_001).cpu().numpy(), want)
    _same(ops.accum_1d_host(px, py, basis).cpu().numpy(), want)


# ---- 2-D ----------------------------------------------------------------------------------------------------------------
def _acc2(X, y, bases, **kw):
    import torch

    from asvgp_b200 import ops

    acc = torch.zeros(ops.accum_size_2d(bases), dtype=torch.float64, device="cuda")
    cm = ops.moment_table_2d(bases)
    ops.accum_2d(X, y, bases, cm, ops.split_accum_2d(acc, bases)[2], **kw)
    select = int(cm[-1:].view(torch.int32)[0].item())
    ops.expand_moments_2d(cm, bases, acc)
    return acc.cpu().numpy(), select


def _acc2_host(X, y, bases, **kw):
    import torch

    from asvgp_b200 import ops

    acc = torch.zeros(ops.accum_size_2d(bases), dtype=torch.float64, device="cuda")
    cm = ops.moment_table_2d(bases)
    ops.accum_2d_host(X, y, bases, cm, ops.split_accum_2d(acc, bases)[2], **kw)
    ops.expand_moments_2d(cm, bases, acc)
    return acc.cpu().numpy()


def _raster(variant, n1, n2):
    rng = np.random.default_rng(n1 * 1000 + n2)
    x1 = np.sort(rng.uniform(-74.9, -30.1, n1))
    x2 = np.sort(rng.uniform(20.1, 49.9, n2))
    X = np.stack(np.meshgrid(x1, x2, indexing="ij"), -1)
    if variant == "curvilinear":
        X[:, :, 1] += 0.01 * np.sin(np.arange(n1))[:, None]
    if variant in ("separable-dirty", "separable-dirty-x1"):
        for r, c in ((3, 17), (50, 150), (51, 151), (129, 298)):
            X[r, c, 0] += 0.013
    if variant == "separable-dirty":
        for r, c in ((7, 5), (64, 200), (100, 31)):
            X[r, c, 1] -= 0.021
    X = X.reshape(-1, 2)
    if variant == "x1-runs":
        X = X[rng.uniform(size=X.shape[0]) > 0.1]
    y = np.sin(X[:, 0] / 4.0) * np.cos(X[:, 1] / 3.0) + 0.05 * rng.standard_normal(X.shape[0])
    return X.astype(np.float32), y


@pytest.mark.parametrize("k", [3, 4])
@pytest.mark.parametrize("yd", ["f32", "f64"])
@pytest.mark.parametrize("variant,n1,n2", [("separable", 130, 300), ("separable", 67, 301), ("curvilinear", 130, 300),
                                            ("curvilinear", 67, 301), ("x1-runs", 97, 211), ("separable-dirty", 130, 300),
                                            ("separable-dirty-x1", 130, 300)])
def test_accum_2d_raster_variants_float32(cuda, k, yd, variant, n1, n2):
    """float32 X through every path of asvgp_accum_2d's probe: the same path and sums as the float64-converted points."""
    import torch

    from asvgp_b200 import basis as B

    X, y = _raster(variant, n1, n2)
    cls = getattr(B, "B%dSpline" % k)
    bases = [cls(-80, -25, 19), cls(15, 55, 23)]
    Xt = torch.from_numpy(X).cuda()
    yt = torch.from_numpy(y).cuda().to(_dt(yd))
    want, sel64 = _acc2(Xt.double(), yt.double(), bases)
    got, sel = _acc2(Xt, yt, bases)
    assert sel == sel64
    if variant.startswith("separable"):
        assert sel == 4 or variant == "separable-dirty"
    _same(got, want)
    if k == 3 and yd == "f64":
        G0, b0, _ = O.precompute_kron([bb.mesh for bb in bases], [bb.delta for bb in bases], 3, [19, 23], X.astype(np.float64), y)
        from asvgp_b200 import ops, utils

        Gs, b, _ = ops.split_accum_2d(torch.from_numpy(got), bases)
        assert abs(utils.stencil_to_sparse(Gs.numpy(), 19, 23, 3) - G0).max() <= 1e-10 * abs(G0).max()
    if variant == "separable":
        _same(_acc2(Xt, yt, bases, raster_row_len=n2)[0], want)
        _same(_acc2_host(X, yt.cpu().numpy(), bases, chunk=3 * n2 + 1, raster_row_len=n2), want)
        _same(_acc2_host(torch.from_numpy(X).pin_memory(), yt.cpu().pin_memory(), bases, chunk=5 * n2), want)
        perm = torch.from_numpy(np.random.default_rng(1).permutation(X.shape[0])).cuda()
        Xs, ys = Xt[perm].contiguous(), yt[perm].contiguous()
        want_s = _acc2(Xs.double(), ys.double(), bases)[0]
        _same(_acc2(Xs, ys, bases, raster_row_len=n2)[0], want_s)     # a false raster statement: slow, never wrong
        _same(_acc2(Xs, ys, bases, binned=True)[0], want_s)
        _same(_acc2(Xs, ys, bases, binned="auto")[0], want_s)


@pytest.mark.parametrize("xd,yd", PAIRS)
def test_accum_2d_binned_large_and_misaligned(cuda, xd, yd):
    import torch

    from asvgp_b200 import basis as B, ops

    bases = [B.B3Spline(0, 1, 300), B.B3Spline(0, 2, 40)]
    g = torch.Generator(device="cuda"); g.manual_seed(11)
    n = 3_000_001
    X = torch.stack([torch.rand(n, device="cuda", dtype=torch.float64, generator=g) * 0.98 + 0.01,
                     torch.rand(n, device="cuda", dtype=torch.float64, generator=g) * 1.96 + 0.02], 1).to(_dt(xd))
    y = torch.cos(3 * X[:, 0].double()).to(_dt(yd))
    want = _acc2(X.double(), y.double(), bases, binned=True)[0]
    _same(_acc2(X, y, bases, binned=True)[0], want)
    assert ops.order_probe_2d(X, bases) == ops.order_probe_2d(X.double(), bases)
    Xm = torch.empty((n + 1, 2), dtype=X.dtype, device="cuda")[1:]        # misaligned by one point: cloned in its dtype
    Xm.copy_(X)
    ym = torch.empty(n + 1, dtype=y.dtype, device="cuda")[1:]
    ym.copy_(y)
    _same(_acc2(Xm, ym, bases)[0], _acc2(X.double(), y.double(), bases)[0])


# ---- models ---------------------------------------------------------------------------------------------------------------
def _loss_grad(model):
    loss, g = model.training_loss_and_gradients()
    return float(loss), np.asarray(g)


def _check_model(m32, m64):
    l32, g32 = _loss_grad(m32)
    l64, g64 = _loss_grad(m64)
    assert abs(l32 - l64) <= 1e-10 * abs(l64)
    np.testing.assert_allclose(g32, g64, rtol=1e-8, atol=1e-8 * np.abs(g64).max())


@pytest.mark.parametrize("where", ["device", "host"])
@pytest.mark.parametrize("outputs", [1, 3])
def test_gpr_1d_float32_data(cuda, where, outputs):
    import torch

    from asvgp_b200 import kernels as Kn
    from asvgp_b200.gpr import GPR_1d

    rng = np.random.default_rng(outputs)
    n, m = 200_001, 400
    x = np.sort(rng.uniform(0.5, m - 0.5, n)).astype(np.float32).reshape(-1, 1)
    y = (np.sin(x / 9.0) + 0.1 * rng.standard_normal((n, outputs))).astype(np.float32)

    def build(X, Y):
        kern = Kn.Matern32(variance=1.1, lengthscales=13.0)
        model = GPR_1d((X, Y), kern, _basis(3, 0, m, m))
        model.likelihood.variance.assign(0.05)
        return model

    if where == "device":
        Xd, Yd = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
        _check_model(build(Xd, Yd), build(Xd.double(), Yd.double()))
    else:
        _check_model(build(x, y), build(x.astype(np.float64), y.astype(np.float64)))


@pytest.mark.parametrize("where", ["device", "host"])
def test_gpr_kron_float32_data(cuda, where):
    import torch

    from asvgp_b200 import basis as B, kernels as Kn
    from asvgp_b200.gpr import GPR_kron

    X, y = _raster("separable", 130, 300)
    y = y.astype(np.float32).reshape(-1, 1)
    bases = [B.B4Spline(-80, -25, 19), B.B4Spline(15, 55, 23)]

    def build(Xa, ya, **kw):
        kerns = [Kn.Matern32(variance=1.0, lengthscales=6.0), Kn.Matern32(variance=0.8, lengthscales=5.0)]
        model = GPR_kron((Xa, ya), kerns, bases, **kw)
        model.likelihood.variance.assign(0.01)
        return model

    if where == "device":
        Xd, yd = torch.from_numpy(X).cuda(), torch.from_numpy(y).cuda()
        ref = build(Xd.double(), yd.double())
        _check_model(build(Xd, yd), ref)
        _check_model(build(Xd, yd, raster_shape=(130, 300)), ref)
    else:
        ref = build(X.astype(np.float64), y.astype(np.float64))
        _check_model(build(X, y), ref)
        _check_model(build(X, y, raster_shape=(130, 300)), ref)


# ---- no widened copy ----------------------------------------------------------------------------------------------------
def test_float32_inputs_allocate_no_float64_copy(cuda):
    import torch

    from asvgp_b200 import _lib, basis as B, ops

    n, m = 8_000_000, 1000
    basis = _basis(3, -1, m + 1, m)
    g = torch.Generator(device="cuda"); g.manual_seed(3)
    x = torch.sort(torch.rand(n, device="cuda", generator=g) * m)[0]          # float32
    y = torch.rand(n, device="cuda", generator=g)
    acc = torch.zeros(ops.accum_size_1d(basis), dtype=torch.float64, device="cuda")
    bound = 8 * n                                                              # one float64 copy of the smaller array
    for binned in (False, True, "auto"):
        torch.cuda.synchronize(); torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        ops.accum_1d(x, y, basis, acc=acc, binned=binned)
        torch.cuda.synchronize()
        extra = _lib.load().asvgp_accum_1d_binned_work_bytes(n) if binned is True else 0
        assert torch.cuda.max_memory_allocated() - base < bound + extra

    bases = [B.B3Spline(0, 1, 200), B.B3Spline(0, 1, 200)]
    X = torch.rand((n, 2), device="cuda", generator=g) * 0.98 + 0.01
    cm = ops.moment_table_2d(bases)
    scal = torch.zeros(2, dtype=torch.float64, device="cuda")
    for binned in (False, True):
        torch.cuda.synchronize(); torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        ops.accum_2d(X, y, bases, cm, scal, binned=binned)
        torch.cuda.synchronize()
        extra = _lib.load().asvgp_accum_2d_binned_work_bytes(n) if binned else 0
        assert torch.cuda.max_memory_allocated() - base < bound + extra
