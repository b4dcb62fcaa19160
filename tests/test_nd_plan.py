"""The nested-dissection plan of the 2-D factorisation (asvgp_b200/csrc/ndfront_2d.cu), checked on the CPU:
  * the C++ elimination tree (asvgp_kron_plan_info, a host-side query) equals the numpy prototype's (tools/nd_prototype.py)
    front by front and satisfies the structural invariants the multifrontal method relies on;
  * the prototype — the same algebra as the CUDA kernels, dense numpy per front — reproduces log|P|, ||L^-1 b||^2, P^-1 b
    and the stencil entries of P^-1 of the LAPACK-band oracle (reference gpr.py:292-307 on the band)."""
import os
import sys

import numpy as np
import pytest
import scipy.linalg as sla

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import nd_prototype as ND                      # noqa: E402
from oracle import asvgp_oracle as O           # noqa: E402


@pytest.fixture(scope="module")
def ops():
    import __graft_entry__

    __graft_entry__.build()
    from asvgp_b200 import ops as _ops

    return _ops


@pytest.mark.parametrize("m1,m2,k", [(14, 14, 3), (40, 36, 3), (100, 64, 3), (200, 200, 3), (100, 100, 4), (33, 57, 2), (12, 30, 1),
                                    (41, 23, 1), (40, 36, 5), (60, 44, 5), (44, 40, 6), (70, 52, 6)])
def test_cxx_plan_matches_prototype_and_invariants(ops, m1, m2, k):
    info = ops.kron_plan_info(m1, m2, k, with_fronts=True)
    fronts, root = ND.build_tree(m1, m2, k, leaf=12)
    got = info["front_list"]
    assert len(got) == len(fronts) == int(info["fronts"])
    M = m1 * m2
    seen = np.zeros(M, dtype=int)
    for (level, sep, bnd), f in zip(got, fronts):
        assert level == f.level
        np.testing.assert_array_equal(sep, f.sep)
        np.testing.assert_array_equal(bnd[:-1], f.bnd)          # same ancestors, same order
        assert bnd[-1] == M                                      # the right-hand-side row closes every boundary
        seen[sep] += 1
    assert (seen == 1).all()                                     # every basis function is eliminated in exactly one front
    # the boundary of a child lies inside its parent's front, and separators really separate: no stencil edge joins the
    # regions of two siblings
    by_id = {id(f): g for f, g in zip(fronts, got)}
    for f in fronts:
        _, sep, bnd = by_id[id(f)]
        if f.parent is not None:
            _, psep, pbnd = by_id[id(f.parent)]
            assert set(bnd.tolist()) <= set(psep.tolist()) | set(pbnd.tolist())
        if f.children:
            (a0, a1, b0, b1), (c0, c1, d0, d1) = f.children[0].region, f.children[1].region
            gap_rows = max(c0 - (a1 - 1), a0 - (c1 - 1))
            gap_cols = max(d0 - (b1 - 1), b0 - (d1 - 1))
            assert max(gap_rows, gap_cols) > k
    if (m1, m2, k) == (200, 200, 3):
        assert int(info["levels"]) == 9 and int(info["chain_columns"]) <= 1760 and int(info["chain_block_columns"]) <= 34


# relative tolerance on x = P^-1 b.  At k = 6 (44 x 40, cond(P) = 8e10) x is only defined to a few 1e-7 of max|x|: moving the
# band entries of P by one ulp of max|P| (uniform in [-1, 1] ulp, three draws) moves LAPACK's x by 3.5e-7 ... 2.7e-6 of
# max|x|; the prototype's elimination order lands 1.6e-7 from LAPACK's (iterative refinement in extended precision puts
# LAPACK itself within 4e-11).  At k <= 5 the same perturbation moves x by <= 1.1e-11.
X_TOL = {6: 3e-6}


@pytest.mark.parametrize("m1,m2,k,kind", [(14, 14, 3, "Matern32"), (40, 36, 3, "Matern32"), (30, 44, 2, "Matern12"), (36, 30, 4, "Matern52"),
                                         (41, 23, 1, "Matern12"), (40, 36, 5, "Matern52"), (44, 40, 6, "Matern32")])
def test_prototype_matches_band_oracle(m1, m2, k, kind):
    from asvgp_b200 import utils as U

    rng = np.random.default_rng(m1 * 100 + m2)
    n = 30 * m1 * m2
    meshes, deltas = zip(*[O.make_mesh(0, m, m, k) for m in (m1, m2)])
    X = np.stack([rng.uniform(0.01, m1 - 0.01, n), rng.uniform(0.01, m2 - 0.01, n)], 1)
    y = np.sin(X[:, 0] / 3) * np.cos(X[:, 1] / 4) + 0.1 * rng.standard_normal(n)
    G, b, _ = O.precompute_kron(meshes, deltas, k, [m1, m2], X, y)
    T = [O.static_bands(k, m, d) for m, d in zip((m1, m2), deltas)]
    Ks = [O.make_Kuu(kind, 6.0, 1.0, T[0]), O.make_Kuu(kind, 5.0, 0.9, T[1])]
    s2 = 0.05
    out = ND.factor_and_selinv(m1, m2, k, Ks[0], Ks[1], U.sparse_to_stencil(G, m1, m2, k), b[:, 0], s2)
    cP = sla.cholesky_banded(O.kron_band(Ks, G, s2, k, [m1, m2]), lower=True)
    ld = 2 * np.sum(np.log(cP[0]))
    x = sla.cho_solve_banded((cP, True), b)[:, 0]
    assert abs(out["logdet"] - ld) <= 1e-12 * abs(ld)
    assert abs(out["quad"] - b[:, 0] @ x) <= 1e-10 * abs(b[:, 0] @ x)
    np.testing.assert_allclose(out["x"], x, rtol=0, atol=X_TOL.get(k, 1e-11) * np.abs(x).max())
    cols = rng.choice(m1 * m2, 10, replace=False)
    want = O.stencil_columns_of_inverse(Ks, G, s2, k, [m1, m2], cols)
    np.testing.assert_allclose(out["sig"][:, cols], want, rtol=0, atol=1e-12 * np.abs(want).max())
