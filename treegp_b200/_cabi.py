"""ctypes binding of include/treegp_b200.h (libtreegp_b200.so).

This is the only place the Python host code crosses into native code.  There is no CPU fallback: if
the library is missing, or a call returns a non-zero status, an exception is raised.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# TREEGP_B200_LIB: alternative build of the same library (kernel-tuning experiments only)
LIB_PATH = os.environ.get("TREEGP_B200_LIB") or os.path.join(_HERE, "libtreegp_b200.so")

ABI_VERSION = 1

# tgp_family / tgp_bintype (include/treegp_b200.h)
FAM_RBF, FAM_VONKARMAN, FAM_MATERN12, FAM_MATERN32, FAM_MATERN52 = range(5)
BIN_TWOD, BIN_LOG = 0, 1


class TgpKernel(ctypes.Structure):
    """POD kernel descriptor `tgp_kernel`."""
    _fields_ = [("family", ctypes.c_int32), ("ndim", ctypes.c_int32), ("amp", ctypes.c_double),
                ("m00", ctypes.c_double), ("m01", ctypes.c_double), ("m11", ctypes.c_double)]


MAX_TERMS = 4   # TGP_MAX_TERMS
MAX_RHS = 8     # TGP_MAX_RHS: outputs of the multi-output entries
BATCH_MAX_N = 4096   # TGP_BATCH_MAX_N: points per problem of the batch entries
GRAD_BATCH_OUT = 4 + 4 * MAX_TERMS   # TGP_GRAD_BATCH_OUT: outputs per problem of tgp_loglike_grad_batch


class TgpKernelSum(ctypes.Structure):
    """POD sum descriptor `tgp_kernel_sum`: nterms stationary terms plus a WhiteKernel level."""
    _fields_ = [("nterms", ctypes.c_int32), ("ndim", ctypes.c_int32), ("white", ctypes.c_double),
                ("term", TgpKernel * MAX_TERMS)]


class TgpError(RuntimeError):
    pass


_vp, _i64, _i32, _f64 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_double
_kp = ctypes.POINTER(TgpKernel)
_ksp = ctypes.POINTER(TgpKernelSum)

# name -> argtypes; every entry returns int (tgp_status) unless listed in _RESTYPES
SIGNATURES = {
    "tgp_abi_version": [],
    "tgp_last_error": [],
    "tgp_kmat_sym": [_vp, _i64, _kp, _vp, _vp, _i64, ctypes.c_int, _vp],
    "tgp_kmat_cross": [_vp, _i64, _vp, _i64, _kp, _vp, _i64, _vp],
    "tgp_potrf": [_vp, _i64, _i64, _vp, _vp],
    "tgp_potrf_rows": [_vp, _i64, _i64, _i64, _vp, _vp],
    "tgp_potrs_vec": [_vp, _i64, _i64, _vp, _vp],
    "tgp_trsm_rows": [_vp, _i64, _i64, _vp, _i64, _i64, _vp],
    "tgp_gemm_nt_sub": [_vp, _i64, _i64, _i64, _vp, _i64, _vp, _i64, _i64, ctypes.c_int, _vp],
    "tgp_logdet_chi2": [_vp, _i64, _i64, _vp, _vp, _vp, _vp],
    "tgp_loglike": [_vp, _vp, _vp, _i64, _kp, _vp, _i64, _vp, ctypes.c_int, _vp, _vp, _vp],
    "tgp_envelope_block": [],
    "tgp_potrf_env": [_vp, _i64, _i64, _vp, _i64, _i64, _vp, _vp],
    "tgp_trsm_rows_env": [_vp, _i64, _i64, _vp, _i64, _vp, _i64, _i64, _vp],
    "tgp_loglike_env": [_vp, _vp, _vp, _i64, _kp, _vp, _i64, _vp, ctypes.c_int, _vp, _vp, _vp, _i64, _vp],
    "tgp_selinv_work_doubles": [_i64],
    "tgp_selinv": [_vp, _i64, _i64, _vp, _i64, _vp, _vp],
    "tgp_loglike_grad": [_vp, _vp, _vp, _i64, _kp, _vp, _i64, _vp, _vp, _vp, _vp, _i64, _vp, _vp],
    "tgp_kmat_sym_sum": [_vp, _i64, _ksp, _vp, _vp, _i64, ctypes.c_int, _vp],
    "tgp_kmat_cross_sum": [_vp, _i64, _vp, _i64, _ksp, _vp, _i64, _vp],
    "tgp_loglike_sum": [_vp, _vp, _vp, _i64, _ksp, _vp, _i64, _vp, ctypes.c_int, _vp, _vp, _vp, _i64, _vp],
    "tgp_loglike_grad_sum_work_doubles": [_i64, _i32],
    "tgp_loglike_grad_sum": [_vp, _vp, _vp, _i64, _ksp, _vp, _i64, _vp, _vp, _vp, _vp, _i64, _vp, _vp],
    "tgp_predict_mean_sum": [_vp, _i64, _vp, _i64, _ksp, _vp, _vp, _vp],
    "tgp_predict_mean_trunc_sum": [_vp, _i64, _vp, _i64, _ksp, _vp, _vp, _vp, _vp],
    "tgp_predict_var_sum": [_vp, _i64, _vp, _i64, _ksp, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _vp],
    "tgp_loglike_multi": [_vp, _vp, _i32, _vp, _i64, _ksp, _vp, _i64, _vp, ctypes.c_int, _vp, _vp, _vp, _i64, _vp],
    "tgp_loglike_grad_multi_work_doubles": [_i64, _i32, _i32],
    "tgp_potrs_multi": [_vp, _i64, _i64, _vp, _i32, _vp],
    "tgp_loglike_grad_multi": [_vp, _vp, _i32, _vp, _i64, _ksp, _vp, _i64, _vp, _vp, _vp, _vp, _i64, _vp, _vp],
    "tgp_predict_mean_multi": [_vp, _i64, _vp, _i64, _ksp, _vp, _i32, _vp, _vp],
    "tgp_predict_mean_trunc_multi": [_vp, _i64, _vp, _i64, _ksp, _vp, _i32, _vp, _vp, _vp],
    "tgp_batch_work_doubles": [_vp, _i32],
    "tgp_loglike_batch": [_vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, ctypes.c_int, _vp, _vp, _vp],
    "tgp_predict_mean_batch": [_vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp],
    "tgp_loglike_grad_batch_work_doubles": [_vp, _i32],
    "tgp_loglike_grad_batch": [_vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "tgp_predict_var_batch_work_doubles": [_vp, _vp, _i32, _i64],
    "tgp_predict_var_batch": [_vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _i64, _vp, _vp],
    "tgp_loo_batch": [_vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "tgp_batch_multi_work_doubles": [_vp, _i32, _i32],
    "tgp_loglike_batch_multi": [_vp, _vp, _i32, _vp, _vp, _i32, _vp, _vp, _vp, ctypes.c_int, _vp, _vp, _vp],
    "tgp_loglike_grad_batch_multi": [_vp, _vp, _i32, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "tgp_predict_mean_batch_multi": [_vp, _vp, _vp, _vp, _i32, _vp, _vp, _i32, _vp, _vp],
    "tgp_loo_batch_multi": [_vp, _vp, _i32, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "tgp_predict_var_env": [_vp, _i64, _vp, _i64, _kp, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _vp],
    "tgp_predict_mean": [_vp, _i64, _vp, _i64, _kp, _vp, _vp, _vp],
    "tgp_predict_mean_trunc": [_vp, _i64, _vp, _i64, _kp, _vp, _vp, _vp, _vp],
    "tgp_predict_work_doubles": [_i64],
    "tgp_profile_qcut": [_i32],
    "tgp_knn_mean": [_vp, _i64, _vp, _vp, _i64, _i32, _i32, _vp, _vp],
    "tgp_predict_var": [_vp, _i64, _vp, _i64, _kp, _vp, _i64, _vp, _i64, _vp, _vp],
    "tgp_pairbin": [_vp, _vp, _vp, _vp, _vp, _i32, _i64, _i32, _vp, _i32, _f64, _f64, _i32, _i32,
                    _vp, _vp, _vp, _vp, _vp, _vp],
    "tgp_pairbin_work_doubles": [_i64, _i32],
    "tgp_hilbert_keys": [_vp, _vp, _i64, _f64, _f64, _f64, _i32, _vp, _vp],
    "tgp_hilbert_keys_auto": [_vp, _vp, _i64, _i32, _vp, _vp, _vp],
    "tgp_bootstrap_multiplicities": [_vp, _i64, _i64, _vp, _vp],
    "tgp_bootbin_twod": [_vp, _vp, _vp, _vp, _i64, _vp, _i32, _vp, _i32, _f64, _f64, _i32, _i32, _vp, _vp, _vp, _vp],
    "tgp_bootbin_xi": [_vp, _vp, _i32, _i32, _vp, _vp, _vp],
    "tgp_bootbin_work_bytes": [_i64, _i32],
    "tgp_bootbin_sums_doubles": [_i32, _i32],
    "tgp_bootbin_stats": [_vp, ctypes.c_int],
    "tgp_device_error": [_i32],
    "tgp_robust_chi2_batch": [_vp, _vp, _vp, _i32, _i32, _vp, _i32, _vp, _vp],
    "tgp_comm_unique_id": [_vp],
    "tgp_comm_init_rank": [_vp, _i32, _i32, _vp],
    "tgp_comm_destroy": [_vp],
    "tgp_allreduce_bins": [_vp, _vp, _i64, _i64, _vp],
    "tgp_vcorr": [_vp, _vp, _vp, _vp, _i64, _vp, _i32, _vp, _vp, _vp, _i32, _vp, _vp],
    "tgp_pairbin_tile": [],
    "tgp_pairbin_stats": [_vp, ctypes.c_int],
    "tgp_pairbin_super_leaves": [_vp, ctypes.c_int],
    "tgp_pairbin_super_rows": [_vp, ctypes.c_int],
    "tgp_pairbin_super_one_axis_rows": [_vp, ctypes.c_int],
    "tgp_set_option": [ctypes.c_char_p, ctypes.c_int],
    "tgp_microbench_fp64": [ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_double)],
}
_RESTYPES = {"tgp_last_error": ctypes.c_char_p, "tgp_pairbin_work_doubles": ctypes.c_int64,
             "tgp_selinv_work_doubles": ctypes.c_int64, "tgp_loglike_grad_sum_work_doubles": ctypes.c_int64,
             "tgp_loglike_grad_multi_work_doubles": ctypes.c_int64,
             "tgp_predict_work_doubles": ctypes.c_int64, "tgp_batch_work_doubles": ctypes.c_int64,
             "tgp_batch_multi_work_doubles": ctypes.c_int64,
             "tgp_loglike_grad_batch_work_doubles": ctypes.c_int64, "tgp_predict_var_batch_work_doubles": ctypes.c_int64,
             "tgp_bootbin_work_bytes": ctypes.c_int64, "tgp_bootbin_sums_doubles": ctypes.c_int64, "tgp_profile_qcut": ctypes.c_double}

_lib = None


def load():
    """Load (once) and return the ctypes handle.  Raises TgpError if the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise TgpError(
            "treegp_b200: %s not found -- build it with `make` (or __graft_entry__.build()). "
            "There is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here means header and library disagree
        fn.argtypes = argtypes
        fn.restype = _RESTYPES.get(name, ctypes.c_int)
    if lib.tgp_abi_version() != ABI_VERSION:
        raise TgpError("treegp_b200: ABI version mismatch (library %d, binding %d)"
                       % (lib.tgp_abi_version(), ABI_VERSION))
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().tgp_last_error()
        raise TgpError("treegp_b200 %s failed (status %d): %s"
                       % (what, rc, msg.decode() if msg else "?"))
