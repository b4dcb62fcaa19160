"""ctypes loader of libasvgp_sm100a.so (the C ABI declared in include/asvgp_b200.h).

There is deliberately no CPU fallback: if the library has not been built, or a call fails, this raises."""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libasvgp_sm100a.so")

_c_double_p = ctypes.c_void_p
_c_i64 = ctypes.c_int64
_c_int = ctypes.c_int
_c_dbl = ctypes.c_double
_vp = ctypes.c_void_p

# name -> argtypes; every function returns int except the two runtime queries.  Kept in sync with
# include/asvgp_b200.h by tests/test_c_abi.py.
SIGNATURES = {
    "asvgp_basis_eval_1d": [_vp, _c_i64, _vp, _c_int, _c_int, _c_int, _vp, _vp, _vp, _vp],
    "asvgp_accum_1d": [_vp, _vp, _c_i64, _vp, _c_int, _c_int, _vp, _vp],
    "asvgp_accum_1d_binned": [_vp, _vp, _c_i64, _vp, _c_int, _c_int, _vp, _vp, _c_i64, _vp],
    "asvgp_order_probe_1d": [_vp, _c_i64, _vp, _c_int, _vp, _vp],
    "asvgp_accum_1d_typed": [_vp, _c_int, _vp, _c_int, _c_i64, _vp, _c_int, _c_int, _vp, _vp],
    "asvgp_accum_1d_binned_typed": [_vp, _c_int, _vp, _c_int, _c_i64, _vp, _c_int, _c_int, _vp, _vp, _c_i64, _vp],
    "asvgp_order_probe_1d_typed": [_vp, _c_int, _c_i64, _vp, _c_int, _vp, _vp],
    "asvgp_predict_1d": [_vp, _c_i64, _vp, _c_int, _c_int, _vp, _vp, _c_dbl, _vp, _vp, _vp],
    "asvgp_kuu_assemble": [_vp, _c_int, _vp, _vp, _c_int, _c_int, _vp, _vp, _vp],
    "asvgp_elbo_grad_1d": [_vp, _vp, _vp, _c_int, _c_int, _c_dbl, _c_dbl, _c_int, _vp, _vp, _c_i64, _vp],
    "asvgp_debug_poison_smem": [_vp],
    "asvgp_kuu_chain_1d": [_vp, _vp, _c_int, _c_int, _c_int, _vp, _vp, _c_i64, _vp, _vp],
    "asvgp_elbo_grad_1d_prepared": [_vp, _vp, _vp, _vp, _c_int, _c_int, _c_dbl, _c_dbl, _c_int, _vp, _vp, _c_i64, _vp, _c_int, _vp],
    "asvgp_kuu_assemble_batched": [_vp, _c_int, _c_int, _vp, _vp, _c_int, _c_int, _vp, _vp, _vp],
    "asvgp_elbo_grad_1d_batched": [_vp, _vp, _vp, _c_int, _c_int, _c_int, _c_int, _vp, _vp, _c_int, _vp, _vp, _c_i64, _vp],
    "asvgp_posterior_1d": [_vp, _vp, _c_int, _c_int, _c_dbl, _c_int, _vp, _vp, _vp, _vp, _c_i64, _vp],
    "asvgp_accum_1d_segmented_typed": [_vp, _c_int, _vp, _c_int, _c_i64, _vp, _c_int, _vp, _c_int, _c_int, _vp, _vp],
    "asvgp_elbo_grad_1d_batched_rows": [_vp, _vp, _vp, _c_int, _vp, _c_int, _c_int, _c_int, _c_int, _vp, _vp, _c_int, _vp, _vp,
                                        _c_i64, _vp],
    "asvgp_posterior_1d_batched": [_vp, _vp, _c_int, _vp, _c_int, _c_int, _c_int, _vp, _c_int, _vp, _vp, _vp, _vp, _c_i64, _vp],
    "asvgp_predict_1d_segmented": [_vp, _c_i64, _vp, _c_int, _vp, _c_int, _c_int, _vp, _vp, _vp, _vp, _vp, _vp],
    "asvgp_band_inverse_1d": [_vp, _vp, _c_int, _c_int, _c_int, _vp, _vp, _vp, _vp, _c_i64, _vp],
    "asvgp_accum_2d": [_vp, _vp, _c_i64, _vp, _c_int, _vp, _c_int, _c_int, _vp, _vp, _vp],
    "asvgp_accum_2d_raster": [_vp, _vp, _c_i64, _c_i64, _vp, _c_int, _vp, _c_int, _c_int, _vp, _vp, _vp],
    "asvgp_predict_2d_prepare": [_c_int, _c_int, _c_int, _vp, _vp, _vp, _vp, _vp, _vp],
    "asvgp_predict_2d_apply": [_vp, _c_i64, _c_i64, _vp, _c_int, _vp, _c_int, _c_int, _c_dbl, _vp, _vp, _vp, _vp],
    "asvgp_accum_2d_binned": [_vp, _vp, _c_i64, _vp, _c_int, _vp, _c_int, _c_int, _vp, _vp, _vp, _c_i64, _vp],
    "asvgp_order_probe_2d": [_vp, _c_i64, _vp, _c_int, _vp, _c_int, _vp, _vp],
    "asvgp_accum_2d_typed": [_vp, _c_int, _vp, _c_int, _c_i64, _vp, _c_int, _vp, _c_int, _c_int, _vp, _vp, _vp],
    "asvgp_accum_2d_raster_typed": [_vp, _c_int, _vp, _c_int, _c_i64, _c_i64, _vp, _c_int, _vp, _c_int, _c_int, _vp, _vp, _vp],
    "asvgp_accum_2d_binned_typed": [_vp, _c_int, _vp, _c_int, _c_i64, _vp, _c_int, _vp, _c_int, _c_int, _vp, _vp, _vp, _c_i64,
                                    _vp],
    "asvgp_order_probe_2d_typed": [_vp, _c_int, _c_i64, _vp, _c_int, _vp, _c_int, _vp, _vp],
    "asvgp_expand_moments_2d": [_vp, _vp, _vp, _c_int, _c_int, _c_int, _vp, _vp, _vp],
    "asvgp_kron_factor": [_vp, _vp, _vp, _c_int, _c_int, _c_int, _c_dbl, _vp, _vp, _vp, _vp],
    "asvgp_kron_selinv": [_vp, _c_int, _c_int, _c_int, _vp, _vp, _vp, _vp, _vp],
    "asvgp_kron_doubles_multi": [_c_int, _c_int, _c_int, _c_int, _vp],
    "asvgp_kron_factor_multi": [_vp, _vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_dbl, _vp, _vp, _vp, _vp],
    "asvgp_kron_selinv_multi": [_vp, _c_int, _c_int, _c_int, _c_int, _vp, _vp, _vp, _vp, _vp],
    "asvgp_kronband_factor": [_vp, _vp, _vp, _c_int, _c_int, _c_int, _c_dbl, _vp, _vp, _vp, _vp],
    "asvgp_kronband_selinv": [_vp, _c_int, _c_int, _c_int, _vp, _vp, _vp, _vp, _vp],
    "asvgp_kron_terms": [_vp] * 11 + [_c_int, _c_int, _c_int, _vp, _vp],
    "asvgp_predict_2d": [_vp, _c_i64, _vp, _c_int, _vp, _c_int, _c_int, _vp, _vp, _vp, _vp, _c_dbl, _vp, _vp, _vp, _vp],
    "asvgp_allreduce_oneshot": [_vp, _vp, _c_int, _c_int, _c_i64, _c_i64, ctypes.c_uint, _c_int, _vp, _vp, _vp],
    "asvgp_dense_factor": [_vp, _c_int, _vp, _vp, _vp, _vp],
    "asvgp_dense_selinv": [_vp, _c_int, _vp, _vp, _vp, _vp, _vp],
    "asvgp_dense_doubles_multi": [_c_int, _c_int, _vp],
    "asvgp_dense_factor_multi": [_vp, _c_int, _c_int, _vp, _vp, _vp, _vp],
    "asvgp_dense_selinv_multi": [_vp, _c_int, _c_int, _vp, _vp, _vp, _vp, _vp],
    "asvgp_accum_cross": [_vp, _vp, _c_i64, _c_i64, _vp, _c_int, _vp, _c_int, _c_int, _vp, _vp],
    "asvgp_additive_put_band": [_vp, _c_int, _c_int, _c_int, _c_int, _c_dbl, _c_int, _vp, _vp],
    "asvgp_additive_put_cross": [_vp, _c_int, _c_int, _c_int, _c_int, _c_int, _vp, _vp],
    "asvgp_additive_scale": [_vp, _c_int, _c_dbl, _vp, _vp],
    "asvgp_additive_terms": [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _vp, _vp, _vp, _vp],
    "asvgp_dense_terms": [_vp, _vp, _vp, _c_int, _vp, _vp],
    "asvgp_predict_additive": [_vp, _c_i64, _c_int, _vp, _vp, _c_int, _c_int, _vp, _vp, _vp, _c_dbl, _vp, _vp, _vp],
    "asvgp_khatri_rao_csc": [_vp, _vp, _vp, _vp, _vp, _vp, _c_i64, _c_i64, _vp, _vp, _vp, _vp],
    "asvgp_kron_dense": [_vp, _c_int, _vp, _c_int, _vp, _vp],
    "asvgp_cholesky_dense": [_vp, _c_int, _vp, _vp, _vp],
}
# functions whose return value is not a status code
VALUE_FUNCTIONS = {
    "asvgp_launch_count": (_c_i64, []),
    "asvgp_workspace_bytes_1d": (_c_i64, [_c_int, _c_int, _c_int]),
    "asvgp_workspace_bytes_1d_batched": (_c_i64, [_c_int, _c_int, _c_int, _c_int, _c_int]),
    "asvgp_workspace_bytes_posterior_1d_batched": (_c_i64, [_c_int, _c_int, _c_int, _c_int]),
    "asvgp_kuu_state_doubles": (_c_i64, [_c_int, _c_int]),
    "asvgp_accum_1d_binned_work_bytes": (_c_i64, [_c_i64]),
    "asvgp_accum_2d_binned_work_bytes": (_c_i64, [_c_i64]),
    "asvgp_accum_2d_moment_doubles": (_c_i64, [_c_int, _c_int, _c_int]),
    "asvgp_kron_band_doubles": (_c_i64, [_c_int, _c_int, _c_int]),
    "asvgp_kron_work_doubles": (_c_i64, [_c_int, _c_int, _c_int]),
    "asvgp_kron_sig_doubles": (_c_i64, [_c_int, _c_int, _c_int]),
    "asvgp_kron_rhs_doubles": (_c_i64, [_c_int, _c_int, _c_int]),
    "asvgp_dense_band_doubles": (_c_i64, [_c_int]),
    "asvgp_dense_sig_doubles": (_c_i64, [_c_int]),
    "asvgp_dense_work_doubles": (_c_i64, [_c_int]),
    "asvgp_kron_plan_info": (_c_i64, [_c_int, _c_int, _c_int, _vp, _vp, _c_i64]),
    "asvgp_kron_plan_info_multi": (_c_i64, [_c_int, _c_int, _c_int, _c_int, _vp, _vp, _c_i64]),
    "asvgp_kronband_band_doubles": (_c_i64, [_c_int, _c_int, _c_int]),
    "asvgp_kronband_work_doubles": (_c_i64, [_c_int, _c_int, _c_int]),
    "asvgp_kronband_sig_doubles": (_c_i64, [_c_int, _c_int, _c_int]),
    "asvgp_kronband_rhs_doubles": (_c_i64, [_c_int, _c_int, _c_int]),
    "asvgp_kronband_colstat_offset": (_c_i64, [_c_int, _c_int, _c_int]),
    "asvgp_predict_2d_work_doubles": (_c_i64, [_c_int, _c_int, _c_int]),
}

_lib = None


class AsvgpNativeError(RuntimeError):
    pass


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AsvgpNativeError(
            "libasvgp_sm100a.so not found at %s — build it with `python -m asvgp_b200.build` "
            "(there is no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    lib.asvgp_abi_version.restype = ctypes.c_int
    lib.asvgp_abi_version.argtypes = []
    lib.asvgp_last_error.restype = ctypes.c_char_p
    lib.asvgp_last_error.argtypes = []
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = ctypes.c_int
        fn.argtypes = argtypes
    for name, (restype, argtypes) in VALUE_FUNCTIONS.items():
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


MAX_BATCH = 64              # ASVGP_MAX_BATCH / ASVGP_MAX_BATCH_COLUMNS in include/asvgp_b200.h
MAX_BATCH_COLUMNS = 64

_POISON_EVERY_CALL = os.environ.get("ASVGP_POISON_SMEM") is not None      # test aid: NaN-fill shared memory before EVERY native call


def call(name, *args):
    lib = load()
    if _POISON_EVERY_CALL and name != "asvgp_debug_poison_smem":
        lib.asvgp_debug_poison_smem(args[-1] if isinstance(args[-1], ctypes.c_void_p) else None)    # the call's own stream (always last)
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise AsvgpNativeError("%s failed (%d): %s" % (name, rc, lib.asvgp_last_error().decode()))
