"""ctypes binding of libppbo_b200.so (the C ABI declared in include/ppbo_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails, the product path raises.
PyTorch is used only for device memory, streams and torch.distributed (plumbing).
"""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_int, c_longlong, c_uint, c_ulonglong, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libppbo_b200.so")

FIT_G_READY, FIT_FACTOR_WARM, FIT_FACTOR_AT_MODE = 1, 2, 4
KERNEL_KINDS = {"SE_kernel": 0, "RQ_kernel": 1, "camphor_copper_kernel": 2, "Matern32_kernel": 4, "Matern52_kernel": 5}


class PPBOError(RuntimeError):
    pass


_lib = None
_P, _I, _L, _D = c_void_p, c_int, c_longlong, c_double
_PD, _PI = POINTER(c_double), POINTER(c_int)

# name: (restype, argtypes) -- mirrors include/ppbo_b200.h one to one
_SIGNATURES = {
    "ppbo_version": (_I, []),
    "ppbo_last_error": (c_char_p, []),
    "ppbo_device_sm_count": (_I, [_I]),
    "ppbo_launch_count": (_L, []),
    "ppbo_set_tuning": (_I, [_I, _I]),
    "ppbo_set_thread_background": (_I, [_I]),
    "ppbo_kernel_matrix": (_I, [_I, _P, _I, _P, _I, _I, _PD, _D, _P, _L, _P]),
    "ppbo_sqdist": (_I, [_P, _I, _P, _I, _I, _P, _L, _P]),
    "ppbo_gram_regularized": (_I, [_I, _P, _I, _I, _PD, _D, _D, _P, _L, _P]),
    "ppbo_kernel_se_grad": (_I, [_P, _I, _P, _I, _I, _PD, _D, _P, _L, _L, _P]),
    "ppbo_lik_terms": (_I, [_P, _I, _I, _D, _P, _P, _P, _P]),
    "ppbo_lik_set_sums": (_I, [_P, _I, _I, _D, _P, _P]),
    "ppbo_lambda_dense": (_I, [_P, _I, _I, _P, _L, _P]),
    "ppbo_diffspace_gram": (_I, [_P, _L, _I, _I, _P, _L, _P]),
    "ppbo_factor_doubles": (_L, [_I]),
    "ppbo_laplace_workspace_bytes": (_L, [_I, _I]),
    "ppbo_gram_append": (_I, [_I, _P, _I, _I, _I, _PD, _D, _D, _P, _L, _P]),
    "ppbo_diffspace_gram_append": (_I, [_P, _L, _I, _I, _I, _P, _L, _P]),
    "ppbo_laplace_fit": (_I, [_P, _L, _I, _I, _D, _P, _P, _I, _D, _I, _P, _L, _P, _I, _P, _I, _P, _PI, _P, _P, _P, _P, _L, _PD, _P]),
    "ppbo_laplace_refactor": (_I, [_P, _L, _I, _P, _P, _I, _P, _P]),
    "ppbo_factor_extend": (_I, [_P, _L, _I, _I, _P, _P, _I, _D, _P, _I, _P]),
    "ppbo_gemm_nt": (_I, [_P, _L, _P, _L, _P, _L, _I, _I, _I, _D, _D, _P]),
    "ppbo_gemm_nt_cfg": (_I, [_I, _P, _L, _P, _L, _P, _L, _I, _I, _I, _D, _D, _P]),
    "ppbo_gemm_nt_lower": (_I, [_P, _L, _P, _L, _P, _L, _I, _I, _D, _D, _P]),
    "ppbo_potrf_workspace_bytes": (_L, [_I]),
    "ppbo_potrf_lower": (_I, [_P, _L, _I, _P, _L, _PI, _P]),
    "ppbo_trsm_right_lower": (_I, [_P, _L, _I, _P, _L, _I, _I, _P, _L, _P]),
    "ppbo_potrs_vec": (_I, [_P, _L, _I, _P, _P, _L, _P]),
    "ppbo_blockinv_bytes": (_L, [_I]),
    "ppbo_blockinv_build": (_I, [_P, _L, _I, _P, _P, _L, _P]),
    "ppbo_potrs_vec_blockinv": (_I, [_P, _L, _I, _P, _L, _P, _P]),
    "ppbo_potri_lower": (_I, [_P, _L, _I, _P, _L, _P, _P, _L, _P]),
    "ppbo_shrink_inplace": (_I, [_P, _L, _I, _D, _P, _P]),
    "ppbo_evidence_matrix": (_I, [_P, _L, _I, _I, _P, _I, _P, _L, _P]),
    "ppbo_lu_workspace_bytes": (_L, [_I]),
    "ppbo_lu_logdet": (_I, [_P, _L, _I, _P, _L, _PD, _P]),
    "ppbo_gemv": (_I, [_P, _L, _I, _I, _P, _P, _P]),
    "ppbo_symv_lower": (_I, [_P, _L, _I, _P, _P, _P]),
    "ppbo_neg_count": (_I, [_P, _I, _PI, _I, _P]),
    "ppbo_neg_corr_doubles": (_L, [_I, _I]),
    "ppbo_neg_corr_build": (_I, [_P, _L, _I, _P, _P, _I, _PI, _I, _P, _P]),
    "ppbo_predict_workspace_bytes": (_L, [_I, _I, _I, _I, _I]),
    "ppbo_predict_mean_workspace_bytes": (_L, [_I, _I, _I, _I]),
    "ppbo_predict": (_I, [_I, _P, _I, _I, _PD, _D, _D, _I, _I, _P, _P, _P, _I, _P, _I, _P, _I, _I, _P, _P, _P, _L, _P]),
    "ppbo_mu_pred_point": (_I, [_I, _P, _I, _I, _PD, _D, _P, _PD, _PD, _P]),
    "ppbo_de_minimize": (_I, [_P, _P, _I, _P, _I, _PD, _PD, _I, _I, _D, _D, _D, _D, _D, POINTER(c_uint), _PI, _PD, _PD, _PI]),
    "ppbo_mu_star_de": (_I, [_I, _P, _I, _I, _PD, _D, _P, _PD, _PD, _I, _I, _D, _D, _D, _D, _D, _I, POINTER(c_uint), _PI, _PD, _PD,
                             _PI, _P]),
    "ppbo_mu_pred_points": (_I, [_I, _P, _I, _I, _PD, _D, _P, _PD, _I, _PD, _P]),
    "ppbo_mvn_rowmax": (_I, [_P, _L, _L, _P, _L, _L, _P, _L, _I, _I, _I, _I, _P, _P, _P]),
    "ppbo_acq_reduce": (_I, [_P, _I, _I, _D, _P, _P]),
    "ppbo_acq_reduce_dev": (_I, [_P, _I, _I, _P, _P, _P]),
    "ppbo_vec_max": (_I, [_P, _L, _I, _P, _P]),
    "ppbo_rff_features": (_I, [_P, _P, _I, _I, _P, _I, _D, _P, _L, _I, _P]),
    "ppbo_rff_jacobian": (_I, [_P, _P, _I, _I, _P, _D, _P, _P]),
    "ppbo_rff_value_grad": (_I, [_P, _P, _I, _I, _P, _P, _D, _P, _P]),
    "ppbo_rff_maximize": (_I, [_P, _P, _I, _I, _D, _P, _L, _I, _P, _I, _I, _D, _P, _P, _P, _P]),
    "ppbo_rff_workspace_bytes": (_L, [_I, _I, _I]),
    "ppbo_rff_objective": (_I, [_P, _L, _I, _I, _I, _D, _P, _PD, _P, _P, _P, _L, _P]),
    "ppbo_rff_factor_cache_doubles": (_L, [_I]),
    "ppbo_rff_fit": (_I, [_P, _L, _I, _I, _I, _D, _P, _I, _D, _P, _I, _P, _P, _P, _L, _PD, _P]),
    "ppbo_rff_refactor": (_I, [_P, _L, _I, _I, _I, _D, _P, _P, _P, _L, _P]),
    "ppbo_rff_hessian_factor_workspace_bytes": (_L, [_I, _I, _I]),
    "ppbo_rff_hessian_factor_doubles": (_L, [_I, _L]),
    "ppbo_rff_hessian_factor": (_I, [_P, _L, _I, _I, _I, _D, _P, _P, _L, _P, _L, _PI, _P]),
    "ppbo_normal_fill": (_I, [c_ulonglong, c_uint, _L, _P, _L, _P]),
    "ppbo_rff_sample_omega": (_I, [_P, _P, _P, _L, c_ulonglong, c_uint, _L, _I, _I, _P, _L, _P]),
    "ppbo_rff_sample_omega_full_workspace_bytes": (_L, [_I, _I]),
    "ppbo_rff_sample_omega_full": (_I, [_P, _P, _L, _P, _L, c_ulonglong, c_uint, _L, _I, _I, _P, _L, _P, _L, _P]),
    "ppbo_rff_eval_argmax": (_I, [_P, _L, _I, _I, _P, _L, _L, _I, _I, _P, _P, _P, _P]),
    "ppbo_ozaki_tile_rows": (_I, [_I]),
    "ppbo_ozaki_plane_bytes": (_L, [_I, _I, _I, _I, _I]),
    "ppbo_ozaki_scale_doubles": (_L, [_I, _I, _I]),
    "ppbo_ozaki_slice": (_I, [_P, _L, _L, _I, _I, _I, _I, _I, _P, _P, _P]),
    "ppbo_ozaki_sample_slice": (_I, [_P, _P, c_ulonglong, c_uint, _L, _I, _I, _I, _P, _P, _P]),
    "ppbo_ozaki_normal_slice": (_I, [c_ulonglong, c_uint, _L, _I, _I, _I, _P, _P, _P]),
    "ppbo_ozaki_mma_rate": (_I, [_I, _I, _I, _I, _I, _P, _P]),
    "ppbo_ozaki_rowmax_workspace_bytes": (_L, [_I, _I, _I]),
    "ppbo_ozaki_rowmax": (_I, [_P, _P, _I, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _L, _P, _P]),
    "ppbo_ozaki_rowmax_bias": (_I, [_P, _P, _I, _P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _L, _P, _P]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def load():
    """Load the shared library (once).  Raises PPBOError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PPBOError("libppbo_b200.so is missing (%s): run `python -m ppbo_b200.build` or "
                        "__graft_entry__.build(); there is no CPU fallback" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what):
    """0 -> ok; > 0 LAPACK-style info is returned to the caller; < 0 raises."""
    if rc < 0:
        raise PPBOError("%s failed (%d): %s" % (what, rc, load().ppbo_last_error().decode()))
    return rc


def last_error():
    return load().ppbo_last_error().decode()


def host_doubles(values):
    arr = (c_double * len(values))(*[float(v) for v in values])
    return arr
