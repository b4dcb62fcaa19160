"""Host-side checks of the batched Kronecker evaluation (no GPU needed): the argument checks of
GPR_kron.training_loss_and_gradients_batch, the C ABI's rejections before any CUDA call, the new exports, the size query and the
choice of groups for a memory budget."""
import ctypes
import math
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ("asvgp_kron_doubles_batched", "asvgp_kron_factor_batched", "asvgp_kron_selinv_batched", "asvgp_band_inverse_1d_batched",
       "asvgp_kron_terms_batched", "asvgp_workspace_bytes_band_inverse_1d_batched")
FAKE = ctypes.c_void_p(256)         # a non-NULL device address: every call below is rejected before it is used


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__

    __graft_entry__.build()
    from asvgp_b200 import _lib

    return _lib


def _bare_model(shared=False, method=None):
    from asvgp_b200 import kernels as Kn
    from asvgp_b200.gpr import GPR_kron

    model = GPR_kron.__new__(GPR_kron)
    k = Kn.Matern32()
    model.kernels = [k, k] if shared else [k, Kn.Matern52()]
    model.likelihood = Kn.Gaussian()
    model._method = method
    return model


def test_batch_method_checks_its_arguments():
    model = _bare_model()
    G = len(model.trainable_variables)
    assert G == 5 and len(_bare_model(shared=True).trainable_variables) == 3
    for bad in (np.zeros(G), np.zeros((2, G + 1)), np.zeros((0, G)), np.zeros((65, G))):
        with pytest.raises(ValueError):
            model.training_loss_and_gradients_batch(bad)
    U = np.zeros((2, G))
    U[1, 3] = np.nan
    with pytest.raises(ValueError, match="finite"):
        model.training_loss_and_gradients_batch(U)
    U[1, 3] = np.inf
    with pytest.raises(ValueError, match="finite"):
        model.training_loss_and_gradients_batch(U)
    with pytest.raises(NotImplementedError):
        _bare_model(method="band").training_loss_and_gradients_batch(np.zeros((2, G)))


def test_new_exports_match_the_header(lib):
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "asvgp_b200.h")).read(), flags=re.S)
    handle = lib.load()
    bound = dict(lib.SIGNATURES)
    bound.update({k: v[1] for k, v in lib.VALUE_FUNCTIONS.items()})
    for name in NEW:
        m = re.search(r"ASVGP_API[^;(]*\b%s\s*\(([^;]*?)\)\s*;" % name, text, flags=re.S)
        assert m, "%s is not declared" % name
        assert len(bound[name]) == m.group(1).count(",") + 1
        assert hasattr(handle, name)


def _sizes(lib, m1, m2, k, n_rhs, B):
    h = (ctypes.c_int64 * 6)()
    lib.call("asvgp_kron_doubles_batched", m1, m2, k, n_rhs, B, ctypes.cast(h, ctypes.c_void_p))
    return np.array(list(h), dtype=np.int64)


@pytest.mark.parametrize("shape", [(14, 14, 3, 1), (40, 36, 2, 3), (60, 60, 4, 1)])
def test_size_query_is_linear_in_B(lib, shape):
    one = _sizes(lib, *shape, 1)
    assert (one > 0).all() and one[0] % 32 == 0 and one[1] % 32 == 0 and one[2] % 32 == 0
    for B in (2, 7, 64):
        np.testing.assert_array_equal(_sizes(lib, *shape, B), B * one)
    m1, m2, k, n_rhs = shape
    assert one[3] == n_rhs * m1 * m2 and one[4] == 2 + n_rhs and one[5] == (k + 1) * (2 * k + 1) * m1 * m2
    handle = lib.load()
    w1 = handle.asvgp_workspace_bytes_band_inverse_1d_batched(m1, k, 0, 1)
    assert w1 > 0 and w1 % 256 == 0 and handle.asvgp_workspace_bytes_band_inverse_1d_batched(m1, k, 0, 5) == 5 * w1
    assert handle.asvgp_workspace_bytes_band_inverse_1d_batched(m1, k, 0, 0) == -1
    assert handle.asvgp_workspace_bytes_band_inverse_1d_batched(m1, k, 0, 65) == -1


def test_abi_rejects_bad_arguments_before_any_cuda_call(lib):
    sizes = (ctypes.c_int64 * 6)()
    sz = ctypes.cast(sizes, ctypes.c_void_p)
    for B, n_rhs in ((0, 1), (65, 1), (4, 0), (4, 33)):
        with pytest.raises(lib.AsvgpNativeError, match="B=|n_rhs="):
            lib.call("asvgp_kron_doubles_batched", 14, 14, 3, n_rhs, B, sz)
    with pytest.raises(lib.AsvgpNativeError, match="h_sizes is NULL"):
        lib.call("asvgp_kron_doubles_batched", 14, 14, 3, 1, 2, None)
    need = int(_sizes(lib, 14, 14, 3, 1, 3)[0])

    def factor(B=3, n_rhs=1, s2=(0.1, 0.2, 0.3), band_doubles=need, K1=FAKE):
        h = None if s2 is None else (ctypes.c_double * max(1, len(s2)))(*s2)
        lib.call("asvgp_kron_factor_batched", K1, FAKE, FAKE, FAKE, 14, 14, 3, n_rhs, B,
                 None if h is None else ctypes.cast(h, ctypes.c_void_p), FAKE, band_doubles, FAKE, None)

    for kw, msg in ((dict(B=0), "B=0"), (dict(B=65), "B=65"), (dict(n_rhs=0), "n_rhs=0"), (dict(n_rhs=33), "n_rhs=33"),
                    (dict(s2=None), "h_sigma2 is NULL"), (dict(K1=None), "NULL buffer"),
                    (dict(s2=(0.1, 0.0, 0.3)), "slot 1"), (dict(s2=(0.1, 0.2, -1.0)), "slot 2"),
                    (dict(s2=(math.nan, 0.2, 0.3)), "slot 0"), (dict(band_doubles=need - 1), "needed")):
        with pytest.raises(lib.AsvgpNativeError, match=msg):
            factor(**kw)
    s = _sizes(lib, 14, 14, 3, 2, 4)

    def selinv(B=4, n_rhs=2, band=s[0], sig=s[1], work=s[2], x=FAKE):
        lib.call("asvgp_kron_selinv_batched", FAKE, 14, 14, 3, n_rhs, B, int(band), FAKE, int(sig), FAKE, int(work), x, FAKE, None)

    for kw, msg in ((dict(B=0), "B=0"), (dict(B=65), "B=65"), (dict(n_rhs=33), "n_rhs=33"), (dict(x=None), "NULL buffer"),
                    (dict(band=s[0] - 1), "needed"), (dict(sig=s[1] - 1), "needed"), (dict(work=s[2] - 1), "needed")):
        with pytest.raises(lib.AsvgpNativeError, match=msg):
            selinv(**kw)
    handle = lib.load()
    wb = handle.asvgp_workspace_bytes_band_inverse_1d_batched(30, 3, 0, 4)
    for B, A, work_bytes, msg in ((0, FAKE, wb, "B=0"), (65, FAKE, wb, "B=65"), (4, None, wb, "NULL buffer"),
                                  (4, FAKE, wb - 1, "workspace too small")):
        with pytest.raises(lib.AsvgpNativeError, match=msg):
            lib.call("asvgp_band_inverse_1d_batched", A, FAKE, 30, 3, 0, B, FAKE, FAKE, FAKE, FAKE, work_bytes, None)
    for B, D, msg in ((0, 1, "B=0"), (65, 1, "B=65"), (2, 0, "D=0"), (2, 33, "D=33")):
        with pytest.raises(lib.AsvgpNativeError, match=msg):
            lib.call("asvgp_kron_terms_batched", *([FAKE] * 11), 14, 14, 3, B, D, FAKE, None)


def test_groups_for_a_memory_budget():
    from asvgp_b200 import ops

    GB = 1 << 30
    slot = int(1.34 * GB)
    assert ops.kron_batch_groups(64, slot, 180 * GB) == [(0, 64)]
    # 0.8 of 60 GB holds 35 slots of 1.34 GB
    assert ops.kron_batch_groups(64, slot, 60 * GB) == [(0, 35), (35, 29)]
    assert ops.kron_batch_groups(10, slot, 180 * GB) == [(0, 10)]
    assert ops.kron_batch_groups(5, slot, GB) == [(s, 1) for s in range(5)]          # less than one slot free: one at a time
    assert ops.kron_batch_groups(7, slot, 180 * GB, max_slots=2) == [(0, 2), (2, 2), (4, 2), (6, 1)]
    assert ops.kron_batch_groups(7, slot, 0, max_slots=3) == [(0, 3), (3, 3), (6, 1)]
    assert ops.kron_batch_groups(64, 1, 1 << 50) == [(0, 64)]
    for B in range(1, 65):
        groups = ops.kron_batch_groups(B, slot, 20 * GB)
        assert sum(n for _, n in groups) == B and all(n <= 11 for _, n in groups)
        assert [s for s, _ in groups] == list(np.cumsum([0] + [n for _, n in groups])[:-1])
