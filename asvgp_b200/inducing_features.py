"""`SplineFeatures1D` — same name and methods as reference asvgp/inducing_features.py:6-48."""
import math

import numpy as np

from . import ops
from .kernels import hyper_value, kernel_kind

SQRT3, SQRT5 = math.sqrt(3.0), math.sqrt(5.0)


def kuu_terms(kind, ell, var):
    """[(table name, coefficient, d coefficient / d lengthscale)] with Kuu = sum coefficient * basis.<name>.
    Coefficients of reference inducing_features.py:17-20 (Matern12), :23-30 (Matern32), :33-44 (Matern52; its
    BC_ggrad_none / BC_none_ggrad terms multiply identically-zero tables, SURVEY Q5, and are dropped)."""
    l, v = float(ell), float(var)
    if kind == "Matern12":
        return [("A", 1 / (2 * l * v), -1 / (2 * l * l * v)),
                ("B", l / (2 * v), 1 / (2 * v)),
                ("BC", 1 / (2 * v), 0.0)]
    if kind == "Matern32":
        return [("A", SQRT3 / (4 * l * v), -SQRT3 / (4 * l * l * v)),
                ("B", l / (2 * SQRT3 * v), 1 / (2 * SQRT3 * v)),
                ("C", l**3 / (12 * SQRT3 * v), l * l / (4 * SQRT3 * v)),
                ("BC", 1 / (2 * v), 0.0),
                ("BC_grad", l * l / (2 * v), l / v)]
    if kind == "Matern52":
        return [("A", 3 * SQRT5 / (16 * l * v), -3 * SQRT5 / (16 * l * l * v)),
                ("B", 9 * l / (16 * SQRT5 * v), 9 / (16 * SQRT5 * v)),
                ("C", 9 * l**3 / (80 * SQRT5 * v), 27 * l * l / (80 * SQRT5 * v)),
                ("D", 3 * l**5 / (400 * SQRT5 * v), 15 * l**4 / (400 * SQRT5 * v)),
                ("BC", 9 / (16 * v), 0.0),
                ("BC_grad", 3 * l * l / (10 * v), 6 * l / (10 * v)),
                ("BC_ggrad", 9 * l**4 / (400 * v), 36 * l**3 / (400 * v))]
    raise AssertionError(kind)


class SplineFeatures1D:
    def __init__(self, kernel, basis):
        self.kernel = kernel
        self.basis = basis

    def _terms(self, kernel, ell=None, var=None):
        kind = kernel_kind(kernel)
        if ell is None:
            ell, var = hyper_value(kernel.lengthscales), hyper_value(kernel.variance)
        terms = kuu_terms(kind, ell, var)
        missing = [n for n, _, _ in terms if not hasattr(self.basis, n)]
        if missing:
            raise AttributeError("B%dSpline has no table %s needed by %s (as in the reference)"
                                 % (self.basis.order, missing, kind))
        return terms

    def make_Kuu_device(self, kernel, want_grad=True):
        """(Kuu, dKuu/dlengthscale) lower bands (k+1, m) as CUDA tensors (asvgp_kuu_assemble)."""
        terms = self._terms(kernel)
        return ops.kuu_assemble(self.basis, [t[0] for t in terms], [t[1] for t in terms], [t[2] for t in terms],
                                want_grad=want_grad)

    def make_Kuu_device_batched(self, kernel, lengthscales, variances, want_grad=True):
        """make_Kuu_device of `kernel`'s family at B (lengthscale, variance) settings: bands [B, k+1, m], slot b equal to
        make_Kuu_device at that setting (asvgp_kuu_assemble_batched)."""
        sets = [self._terms(kernel, ell, var) for ell, var in zip(lengthscales, variances)]
        names = [t[0] for t in sets[0]]
        return ops.kuu_assemble_batched(self.basis, names, [[t[1] for t in s] for s in sets], [[t[2] for t in s] for s in sets],
                                        want_grad=want_grad)

    def make_Kuu(self, kernel):
        """Banded Kuu, (k+1) x m lower band, as the reference returns it (inducing_features.py:12-44)."""
        return self.make_Kuu_device(kernel, want_grad=False)[0].cpu().numpy()

    def make_Kuf(self, X, sparse=True):
        """Sparse (m, n) Kuf; like the reference the `sparse` argument is ignored (inducing_features.py:47-48)."""
        return self.basis.evaluate_basis(X, dx=0, sparse=True)
