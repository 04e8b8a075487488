"""ctypes binding of libgegp.so (the C ABI declared in include/gegp.h).

There is NO CPU fallback: if the CUDA library has not been built, importing the compute path raises.
Build it with ``python -c "import __graft_entry__ as g; g.build()"`` (nvcc, sm_100a).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgegp.so")

# mirrors of the #defines in include/gegp.h
ABI_VERSION = 4
MODE_BASE, MODE_PRECON, MODE_PRECON_COV = 0, 1, 2
OUT_LML, OUT_SIGMA2, OUT_BETA, OUT_LOGDET, OUT_INFO, OUT_QUAD, OUT_DVARK, OUT_DVARF, OUT_DVARG, OUT_DKERN, OUT_GRAD = range(11)
KERNEL_SQEXP, KERNEL_MATERN52, KERNEL_RATQUAD = 0, 1, 2
KERNEL_IDS = {"SqExp": KERNEL_SQEXP, "Ma5f2": KERNEL_MATERN52, "RatQu": KERNEL_RATQUAD}   # names of kernel/Kernel.py:27-107
OP_LML, OP_LML_GRAD, OP_PREDICT = 0, 1, 2
OPT_TMA_MIN_TILES = 1
OPT_LOOKAHEAD = 2
OPT_SMALL_TILE_MAX = 3
OPT_CHAIN_CLUSTER = 4
OPT_INV_EARLY = 5

EXPORTS = (
    "gegp_abi_version", "gegp_set_option", "gegp_workspace_bytes", "gegp_ld", "gegp_build_cov", "gegp_cross_cov", "gegp_potrf",
    "gegp_trsm_rows", "gegp_dinv_doubles", "gegp_potri", "gegp_dgemm", "gegp_lml_eval", "gegp_predict_setup", "gegp_predict", "gegp_profile_begin", "gegp_profile_end",
    "gegp_predict_grad", "gegp_predict_hess", "gegp_predict_hess_batch", "gegp_lml_layout", "gegp_symv", "gegp_row_abs_sum", "gegp_row_sq_sum", "gegp_weighted_grad", "gegp_lanczos_step", "gegp_lincomb", "gegp_quad_grad_work_bytes", "gegp_quad_grad", "gegp_dmma_peak", "gegp_lml_direct_terms",
    "gegp_symv_batch", "gegp_lanczos_step_batch", "gegp_lincomb_batch", "gegp_quad_grad_batch_work_bytes",
    "gegp_quad_grad_batch", "gegp_build_cov_batch",
)


def out_len(d: int) -> int:
    return OUT_GRAD + d


_lib = None


def load():
    """Load libgegp.so once and declare every prototype. Raises if the library is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: the CUDA extension is not built and there is no CPU fallback. "
            "Run __graft_entry__.build() (needs nvcc).")
    lib = C.CDLL(LIB_PATH)
    vp, dp, ip = C.c_void_p, C.c_void_p, C.c_void_p   # device pointers travel as integers
    i, i64, dbl, sz = C.c_int, C.c_int64, C.c_double, C.c_size_t
    lib.gegp_abi_version.restype = i
    lib.gegp_abi_version.argtypes = []
    lib.gegp_set_option.restype = i
    lib.gegp_set_option.argtypes = [i, i]
    lib.gegp_workspace_bytes.restype = sz
    lib.gegp_workspace_bytes.argtypes = [i, i, i, i, i]
    lib.gegp_ld.restype = i64
    lib.gegp_ld.argtypes = [i]
    lib.gegp_build_cov.restype = i
    lib.gegp_build_cov.argtypes = [i, i, i, dp, ip, dp, i, dbl, dp, i, dbl, dbl, dp, i64, dp, i, vp]
    lib.gegp_cross_cov.restype = i
    lib.gegp_cross_cov.argtypes = [i, i, i, dp, ip, dp, i, dp, i, dbl, dp, dp, i64, vp]
    lib.gegp_potrf.restype = i
    lib.gegp_potrf.argtypes = [i, i, dp, i64, dp, ip, vp]
    lib.gegp_dinv_doubles.restype = i64
    lib.gegp_dinv_doubles.argtypes = [i]
    lib.gegp_trsm_rows.restype = i
    lib.gegp_trsm_rows.argtypes = [i, dp, i64, dp, dp, i64, i, vp]
    lib.gegp_potri.restype = i
    lib.gegp_potri.argtypes = [i, dp, i64, dp, dp, i64, dp, i64, vp]
    lib.gegp_dgemm.restype = i
    lib.gegp_dgemm.argtypes = [i, i, i, i, dbl, dp, i64, dp, i64, dbl, dp, i64, vp]
    lib.gegp_lml_eval.restype = i
    lib.gegp_lml_eval.argtypes = [i, dp, dp, i, dp, i, i, i, dp, ip, dp, dp, i, dbl, i, dbl, i, dp, dp, vp, sz, vp]
    lib.gegp_predict_setup.restype = i
    lib.gegp_predict_setup.argtypes = [i, i, i, dp, ip, dp, i, dbl, dp, i, dbl, dp, dbl, dp, i64, dp, dp, dp, ip, vp]
    lib.gegp_predict.restype = i
    lib.gegp_predict.argtypes = [i, i, i, dp, ip, dp, i, dbl, dp, i64, dp, dp, i, dbl, dbl, dp, i, dp, dp, dp, ip, vp, sz, vp]
    lib.gegp_predict_grad.restype = i
    lib.gegp_predict_grad.argtypes = [i, i, i, dp, ip, dp, i, dbl, dp, i64, dp, dp, i, dbl, dbl, dp, i, dp, dp, dp, dp, dp, ip, vp,
                                      sz, vp]
    lib.gegp_predict_hess.restype = i
    lib.gegp_predict_hess.argtypes = [i, i, i, dp, ip, dp, i, dbl, dp, i64, dp, dp, dp, i, dbl, dbl, dp, dp, dp, dp, dp, dp, dp, ip,
                                      vp, sz, vp]
    lib.gegp_predict_hess_batch.restype = i
    lib.gegp_predict_hess_batch.argtypes = [i, i, i, dp, ip, dp, i, dbl, dp, i64, dp, dp, dp, i, dbl, dbl, dp, i, dp, dp, dp, dp,
                                            dp, dp, ip, vp, sz, vp]
    lib.gegp_lml_layout.restype = i
    lib.gegp_lml_layout.argtypes = [i, i, i, i, i, C.POINTER(i64)]
    lib.gegp_symv.restype = i
    lib.gegp_symv.argtypes = [i, dp, i64, dp, dp, vp]
    lib.gegp_row_abs_sum.restype = i
    lib.gegp_row_abs_sum.argtypes = [i, dp, i64, dp, vp]
    lib.gegp_row_sq_sum.restype = i
    lib.gegp_row_sq_sum.argtypes = [i, dp, i64, dp, vp]
    lib.gegp_weighted_grad.restype = i
    lib.gegp_weighted_grad.argtypes = [i, i, i, dp, ip, dp, i, dbl, dp, i64, i, dbl, i, dp, dp, vp, sz, vp]
    lib.gegp_lanczos_step.restype = i
    lib.gegp_lanczos_step.argtypes = [i, i, dp, i64, dp, dp, dp, vp]
    lib.gegp_lincomb.restype = i
    lib.gegp_lincomb.argtypes = [i, i, dp, i64, dp, dp, vp]
    lib.gegp_quad_grad_work_bytes.restype = sz
    lib.gegp_quad_grad_work_bytes.argtypes = [i, i, i]
    lib.gegp_quad_grad.restype = i
    lib.gegp_quad_grad.argtypes = [i, i, i, dp, ip, dp, i, dbl, dp, i, dbl, i, dp, dp, vp, sz, vp]
    lib.gegp_symv_batch.restype = i
    lib.gegp_symv_batch.argtypes = [i, i, dp, i64, i64, dp, i64, dp, i64, ip, vp]
    lib.gegp_lanczos_step_batch.restype = i
    lib.gegp_lanczos_step_batch.argtypes = [i, i, i, dp, i64, i64, dp, i64, dp, dp, i64, ip, vp]
    lib.gegp_lincomb_batch.restype = i
    lib.gegp_lincomb_batch.argtypes = [i, i, i, ip, dp, i64, i64, dp, i64, dp, i64, ip, vp]
    lib.gegp_quad_grad_batch_work_bytes.restype = sz
    lib.gegp_quad_grad_batch_work_bytes.argtypes = [i, i, i, i]
    lib.gegp_quad_grad_batch.restype = i
    lib.gegp_quad_grad_batch.argtypes = [i, dp, dp, i, dp, i, i, i, dp, ip, dp, i64, i, dbl, i, dp, vp, sz, vp]
    lib.gegp_build_cov_batch.restype = i
    lib.gegp_build_cov_batch.argtypes = [i, dp, dp, i, dp, i, i, i, dp, ip, dp, i, dbl, dp, i64, i64, dp, i64, i, vp]
    lib.gegp_lml_direct_terms.restype = i
    lib.gegp_lml_direct_terms.argtypes = [i, i, i, dp, ip, dp, i, dbl, i, dbl, i, dp, vp, sz, dp, dp, vp]
    lib.gegp_dmma_peak.restype = i
    lib.gegp_dmma_peak.argtypes = [dp, sz, i, C.POINTER(dbl), vp]
    lib.gegp_profile_begin.restype = None
    lib.gegp_profile_begin.argtypes = [i]
    lib.gegp_profile_end.restype = i
    lib.gegp_profile_end.argtypes = [C.POINTER(C.c_long), C.POINTER(C.c_long), C.POINTER(dbl), C.POINTER(dbl)]
    if lib.gegp_abi_version() != ABI_VERSION:
        raise RuntimeError("libgegp.so ABI version mismatch; rebuild the extension")
    _lib = lib
    return lib


def profile_begin(time_gemm: bool = False):
    load().gegp_profile_begin(int(time_gemm))


def profile_end():
    """-> dict(launches, gemm_launches, gemm_ms, gemm_flops); synchronises the device when GEMM timing was on."""
    a, b, c, d = C.c_long(0), C.c_long(0), C.c_double(0), C.c_double(0)
    rc = load().gegp_profile_end(C.byref(a), C.byref(b), C.byref(c), C.byref(d))
    if rc != 0:
        raise RuntimeError("gegp_profile_end failed")
    return dict(launches=a.value, gemm_launches=b.value, gemm_ms=c.value, gemm_flops=d.value)
