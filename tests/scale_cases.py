"""Seeded synthetic inputs of the BASELINE-sized parity cases (SURVEY §8(d) C3 / C4 / C5 shapes).  Pure numpy, shared by
the generator of the golden fixtures (oracle/make_golden_scale.py, run in the build container where the oracle's
LAPACK-band evaluations take minutes) and by the GPU tests that compare the CUDA path with those fixtures.
Also the inputs of tests/golden/synth_1d.npz (oracle/make_golden.py), which are too many to store."""
import numpy as np

# ---- 1-D, C2-shaped small case of synth_1d.npz: 20 000 points in random order per (spline order, M) --------------------------
SYNTH_1D = ((1, 50), (2, 50), (3, 60), (4, 60), (5, 64))
SYNTH_1D_SAMPLE = 97                # synth_1d.npz keeps every 97th input point to check the regenerated ones


def synth_1d_inputs(n=20_000, seed=1997):
    """{order: (x, y, xs)} drawn in sequence from one generator: x ~ U(0, M), standardised y, 64 test points xs."""
    rng = np.random.default_rng(seed)
    out = {}
    for k, m in SYNTH_1D:
        x = rng.uniform(0.0, m, n)
        y = np.sin(2 * np.pi * x / 37) + 0.5 * np.sin(2 * np.pi * x / 3.1) + 0.3 * rng.standard_normal(n)
        y = (y - y.mean()) / y.std()
        xs = rng.uniform(0.5, m - 0.5, 64).reshape(-1, 1)
        out[k] = x, y, xs
    return out

# ---- 1-D, C3-shaped: M = 1e4 cubic B-splines on (-1, M + 1), N = 2e7 sorted points ---------------------------------------
C3_M, C3_N, C3_ORDER = 10_000, 20_000_000, 3
C3_HYPERS = {                       # name: (kernel, variance, lengthscale, sigma2)
    "m52": ("Matern52", 1.0, 1.0, 0.1),            # bench.py HYPERS
    "m32": ("Matern32", 1.0, 1.0, 0.1),
    "m52_long": ("Matern52", 1.3, 10.0, 0.05),     # stress variant, lengthscale = 10 knot spacings (SURVEY §8(d) C2)
    "m32_long": ("Matern32", 0.7, 10.0, 0.2),
}


def case_1d(n=C3_N, m=C3_M, seed=31, n_test=500):
    rng = np.random.default_rng(seed)
    x = np.sort(rng.uniform(1e-9, m - 1e-9, n))
    y = np.sin(x * (2 * np.pi / 37.0)) + 0.5 * np.sin(x * (2 * np.pi / 3.1)) + 0.3 * rng.standard_normal(n)
    y = (y - y.mean()) / y.std()
    xs = rng.uniform(0.25, m - 0.25, n_test)
    return x, y, xs


# ---- 2-D, C4-shaped: eNATL60-like raster (x1 slow) on basis domains (-80, -25) x (15, 55) ------------------------------------
DOM_2D = ((-80, -25), (15, 55))
INNER_2D = ((-75.0, -30.0), (20.0, 50.0))
C4 = dict(m=(200, 200), order=3, raster=(2000, 2000), hypers=((1.0, 5.0), (1.0, 4.0)), sigma2=0.01, seed=41)   # bench.py HYPERS_2D
# more tiles than SMs (500 > 148: the persistent kernels' task loop wraps) and Kuu-dominated (l / delta ~ 18), in seconds
MID = dict(m=(100, 64), order=3, raster=(600, 500), hypers=((1.0, 10.0), (0.9, 11.5)), sigma2=0.01, seed=43)


def case_2d(raster, seed):
    n1, n2 = raster
    x1 = np.linspace(INNER_2D[0][0], INNER_2D[0][1], n1 + 2)[1:-1]
    x2 = np.linspace(INNER_2D[1][0], INNER_2D[1][1], n2)
    X = np.stack(np.meshgrid(x1, x2, indexing="ij"), -1).reshape(-1, 2)
    rng = np.random.default_rng(seed)
    y = np.zeros(X.shape[0])
    for _ in range(8):                                  # smooth field: 8 random 2-D sinusoids (SURVEY §8(d) C4)
        f1, f2, ph = rng.uniform(0, 1, 3) * np.array([0.6, 0.8, 6.28])
        y += np.sin(X[:, 0] * f1 + X[:, 1] * f2 + ph)
    y = y / 2.0 + 0.05 * rng.standard_normal(X.shape[0])
    return X, y


def points_in_cells_2d(n_cells, per_cell, ms, order, seed):
    """Test points clustered in `n_cells` random knot cells (so that the oracle needs (k+1)^2 band solves per cell, not
    per point), `per_cell` uniform points in each."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n_cells):
        lo, hi = [], []
        for d in range(2):
            knots = np.linspace(DOM_2D[d][0], DOM_2D[d][1], ms[d] - order + 1)
            inside = np.nonzero((knots[:-1] >= INNER_2D[d][0]) & (knots[1:] <= INNER_2D[d][1]))[0]
            c = rng.choice(inside)
            lo.append(knots[c]); hi.append(knots[c + 1])
        u = rng.uniform(0.02, 0.98, (per_cell, 2))
        out.append(np.array(lo) + u * (np.array(hi) - np.array(lo)))
    return np.concatenate(out)
