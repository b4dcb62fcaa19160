"""Minimal stand-ins for the GPflow objects the reference's model API is written against
(`gpflow.kernels.Matern12/32/52`, `gpflow.likelihoods.Gaussian`, GPflow `Parameter`s): same attribute names
(`.variance`, `.lengthscales`, `.K_diag`) and the same parameterisation (softplus-positive, likelihood variance
bounded below by 1e-6, everything initialised to 1.0 — SURVEY App. A).  GPflow itself is not installable here;
real GPflow kernels are accepted by duck-typing (`kernel_kind`)."""
import math

import numpy as np


def _softplus(u):
    return u + math.log1p(math.exp(-u)) if u > 0 else math.log1p(math.exp(u))


def _inv_softplus(x):
    # log(exp(x) - 1), stable for large x
    return x + math.log(-math.expm1(-x))


class Parameter:
    """Positive scalar: value = lower + softplus(unconstrained)  (GPflow's `positive(lower=...)` bijector)."""

    def __init__(self, value, lower=0.0, trainable=True, name=""):
        self.lower = float(lower)
        self.trainable = trainable
        self.name = name
        self.assign(value)

    def assign(self, value):
        value = float(value)
        if not value > self.lower:
            raise ValueError("parameter %s must be > %g" % (self.name, self.lower))
        self.unconstrained = _inv_softplus(value - self.lower)

    @property
    def value(self):
        return self.value_at(self.unconstrained)

    def dvalue_dunconstrained(self):
        return self.dvalue_dunconstrained_at(self.unconstrained)

    def value_at(self, u):
        """The value at unconstrained value `u` (the parameter itself is not changed)."""
        return self.lower + _softplus(u)

    @staticmethod
    def dvalue_dunconstrained_at(u):
        return 1.0 / (1.0 + math.exp(-u))

    def numpy(self):
        return np.float64(self.value)

    def __float__(self):
        return self.value

    def __array__(self, dtype=None, copy=None):
        return np.asarray(self.value, dtype=dtype or np.float64)

    def __repr__(self):
        return "Parameter(%s=%r)" % (self.name, self.value)

    # arithmetic with plain numbers, as user scripts do with GPflow parameters (`variance * 1`, ...)
    def __mul__(self, o): return self.value * float(o)
    __rmul__ = __mul__
    def __add__(self, o): return self.value + float(o)
    __radd__ = __add__
    def __sub__(self, o): return self.value - float(o)
    def __rsub__(self, o): return float(o) - self.value
    def __truediv__(self, o): return self.value / float(o)
    def __rtruediv__(self, o): return float(o) / self.value
    def __pow__(self, o): return self.value ** float(o)
    def __neg__(self): return -self.value


class _Matern:
    kind = None

    def __init__(self, variance=1.0, lengthscales=1.0):
        self.variance = Parameter(variance, name="variance")
        self.lengthscales = Parameter(lengthscales, name="lengthscales")

    def K_diag(self, X):
        return np.full(np.shape(X)[0], float(self.variance))

    @property
    def trainable_variables(self):
        return [self.variance, self.lengthscales]


class Matern12(_Matern):
    kind = "Matern12"


class Matern32(_Matern):
    kind = "Matern32"


class Matern52(_Matern):
    kind = "Matern52"


class Gaussian:
    """gpflow.likelihoods.Gaussian: `.variance` with GPflow's default lower bound 1e-6."""

    def __init__(self, variance=1.0, variance_lower_bound=1e-6):
        self.variance = Parameter(variance, lower=variance_lower_bound, name="likelihood_variance")


def kernel_kind(kernel):
    """'Matern12' | 'Matern32' | 'Matern52' for our kernels and (by class name) for real GPflow ones —
    the reference dispatches with isinstance (inducing_features.py:16,22,32; gpr.py:22)."""
    for cls in type(kernel).__mro__:
        if cls.__name__ in ("Matern12", "Matern32", "Matern52"):
            return cls.__name__
    raise AssertionError("kernel must be Matern12, Matern32 or Matern52 (reference gpr.py:22)")


def hyper_value(p):
    """float value of our Parameter, a GPflow Parameter / tf.Variable (has .numpy()) or a plain number."""
    if isinstance(p, Parameter):
        return p.value
    if hasattr(p, "numpy"):
        return float(np.asarray(p.numpy()))
    return float(p)
