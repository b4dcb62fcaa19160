"""Import the UNMODIFIED reference package (a checkout of the original ASVGP sources at $ASVGP_REFERENCE_ROOT) under the
numpy/SciPy stand-ins of `oracle/shim/` ("reference-under-shim", SURVEY §8(c)).

TEST INFRASTRUCTURE ONLY: the reference sources are not part of this repository, so this module is used solely by
`oracle/make_golden.py`, which writes tests/golden/*.npz; the tests compare with those stored vectors.
"""
import importlib
import os
import sys

REFERENCE_ROOT = os.environ.get("ASVGP_REFERENCE_ROOT", "/root/reference")
SHIM_ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "shim")


def available():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "asvgp"))


def load():
    """Returns the namespace (basis, inducing_features, gpr, utils, kronecker, gpflow) of the reference."""
    if not available():
        raise RuntimeError("reference sources not found at %s" % REFERENCE_ROOT)
    for p in (REFERENCE_ROOT, SHIM_ROOT):
        if p not in sys.path:
            sys.path.insert(0, p)
    mods = {}
    for name in ("tensorflow", "gpflow"):
        mods[name] = importlib.import_module(name)
    assert mods["tensorflow"].__file__.startswith(SHIM_ROOT), "a real tensorflow is shadowing the shim"
    for name in ("basis", "inducing_features", "utils", "kronecker", "gpr"):
        mods[name] = importlib.import_module("asvgp." + name)
    return type("RefNS", (), mods)
