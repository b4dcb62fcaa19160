"""Host-side parts of multi-output targets: every *_multi entry point rejects a right-hand-side count outside
[1, ASVGP_MAX_RHS] before any CUDA call, and the nested-dissection plan for D right-hand sides carries them as the last D
boundary unknowns of every front.  Runs without a GPU."""
import ctypes
import threading

import numpy as np
import pytest

CAP = 32


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__

    __graft_entry__.build()
    from asvgp_b200 import _lib

    return _lib


def _sizes():
    return ctypes.cast((ctypes.c_int64 * 4)(), ctypes.c_void_p)


MULTI = {
    "asvgp_kron_doubles_multi": lambda r: (12, 10, 3, r, _sizes()),
    "asvgp_kron_factor_multi": lambda r: (None, None, None, 12, 10, 3, r, 0.5, None, None, None, None),
    "asvgp_kron_selinv_multi": lambda r: (None, 12, 10, 3, r, None, None, None, None, None),
    "asvgp_dense_doubles_multi": lambda r: (100, r, _sizes()),
    "asvgp_dense_factor_multi": lambda r: (None, 100, r, None, None, None, None),
    "asvgp_dense_selinv_multi": lambda r: (None, 100, r, None, None, None, None, None),
}


def _on_thread(fn):
    """Runs fn on a thread of its own (the library's last-error text is per thread) and returns what it returned."""
    out = []
    t = threading.Thread(target=lambda: out.append(fn()))
    t.start()
    t.join()
    return out[0]


@pytest.mark.parametrize("name", sorted(MULTI))
@pytest.mark.parametrize("n_rhs", [0, CAP + 1, -1, -40])
def test_bad_rhs_count_fails_loudly(lib, name, n_rhs):
    def run():
        try:
            lib.call(name, *MULTI[name](n_rhs))
        except lib.AsvgpNativeError as exc:
            return str(exc)
        return None

    msg = _on_thread(run)
    assert msg is not None and "n_rhs" in msg, msg


@pytest.mark.parametrize("n_rhs", [0, CAP + 1, -1])
def test_plan_info_multi_rejects_bad_rhs_count(lib, n_rhs):
    handle = lib.load()

    def run():
        out = (ctypes.c_double * 8)()
        need = handle.asvgp_kron_plan_info_multi(12, 10, 3, n_rhs, ctypes.cast(out, ctypes.c_void_p), None, 0)
        return need, handle.asvgp_last_error().decode()

    need, msg = _on_thread(run)
    assert need == -1 and "n_rhs" in msg, msg


def test_cap_matches_the_header(lib):
    import os
    import re

    from asvgp_b200 import ops

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    text = open(os.path.join(root, "include", "asvgp_b200.h")).read()
    assert int(re.search(r"#define ASVGP_MAX_RHS (\d+)", text).group(1)) == CAP == ops.MAX_RHS


@pytest.mark.parametrize("n_rhs", [1, CAP])
def test_sizes_grow_with_rhs_count(lib, n_rhs):
    h = (ctypes.c_int64 * 4)()
    lib.call("asvgp_kron_doubles_multi", 40, 36, 3, n_rhs, ctypes.cast(h, ctypes.c_void_p))
    handle = lib.load()
    single = [handle.asvgp_kron_band_doubles(40, 36, 3), handle.asvgp_kron_sig_doubles(40, 36, 3),
              handle.asvgp_kron_work_doubles(40, 36, 3)]
    assert h[3] == 40 * 36 * n_rhs
    if n_rhs == 1:
        assert list(h[:3]) == single
    else:
        assert all(a >= b for a, b in zip(h[:3], single))
    lib.call("asvgp_dense_doubles_multi", 130, n_rhs, ctypes.cast(h, ctypes.c_void_p))
    if n_rhs == 1:
        assert list(h[:3]) == [handle.asvgp_dense_band_doubles(130), handle.asvgp_dense_sig_doubles(130),
                               handle.asvgp_dense_work_doubles(130)]
    assert h[3] == 130 * n_rhs


@pytest.mark.parametrize("m1,m2,k", [(12, 10, 3), (40, 36, 3), (30, 30, 4), (60, 50, 2)])
@pytest.mark.parametrize("n_rhs", [1, 2, 5, CAP])
def test_plan_with_rhs_nodes(lib, m1, m2, k, n_rhs):
    from asvgp_b200 import ops

    M = m1 * m2
    rhs = np.arange(M, M + n_rhs)
    info = ops.kron_plan_info(m1, m2, k, with_fronts=True, n_rhs=n_rhs)
    fronts = info["front_list"]
    roots = [f for f in fronts if f[0] == 0]
    assert len(roots) == 1
    np.testing.assert_array_equal(roots[0][2], rhs)                # the root's boundary is exactly the D rhs ids
    seen = []
    for level, sep, bnd in fronts:
        assert len(bnd) >= n_rhs
        np.testing.assert_array_equal(bnd[-n_rhs:], rhs)         # every boundary ends with M ... M+D-1
        assert (bnd[:-n_rhs] < M).all() and (sep < M).all()
        seen.append(sep)
    np.testing.assert_array_equal(np.sort(np.concatenate(seen)), np.arange(M))
    # the same tree as with one rhs: separators and grid boundaries do not depend on D
    one = ops.kron_plan_info(m1, m2, k, with_fronts=True, n_rhs=1)["front_list"]
    assert len(one) == len(fronts)
    for (l1, s1, b1), (l2, s2, b2) in zip(one, fronts):
        assert l1 == l2
        np.testing.assert_array_equal(s1, s2)
        np.testing.assert_array_equal(b1[:-1], b2[:-n_rhs])


@pytest.mark.parametrize("m1,m2,k", [(12, 10, 3), (40, 36, 3), (200, 200, 3), (100, 100, 4)])
def test_single_rhs_plan_is_todays(lib, m1, m2, k):
    from asvgp_b200 import ops

    old = ops.kron_plan_info(m1, m2, k, with_fronts=True)
    new = ops.kron_plan_info(m1, m2, k, with_fronts=True, n_rhs=1)
    assert {a: b for a, b in old.items() if a != "front_list"} == {a: b for a, b in new.items() if a != "front_list"}
    assert len(old["front_list"]) == len(new["front_list"])
    for (l1, s1, b1), (l2, s2, b2) in zip(old["front_list"], new["front_list"]):
        assert l1 == l2
        np.testing.assert_array_equal(s1, s2)
        np.testing.assert_array_equal(b1, b2)
