"""ctypes binding of libbk200.so (include/bk200.h).  No fallback: if the shared library is
missing or a CUDA call fails, the error is raised -- the product path never routes through
NumPy or the oracle."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbk200.so")
CSRC = os.path.join(_HERE, "csrc")

BK_OK, BK_NOT_CONVERGED = 0, 1
BK_CHAN, BK_SH2D, BK_SH3D, BK_CGL2D, BK_POTRAP_CGL2D = 1, 2, 3, 4, 5
BK_SPARSE = 6  # the Jacobian is a caller-assembled sparse matrix (bk_sparse_set_pattern / bk_sparse_set_values)
BK_COMPLEX = 0x100  # OR-ed into the kind: complexified context, vectors [re; im]
BK_PC_NONE, BK_PC_SH_DCT, BK_PC_CHAN_TRIDIAG, BK_PC_CGL_DST, BK_PC_POTRAP_CIRC = 0, 1, 2, 3, 4
BK_PC_JACOBI = 5
BK_SPARSE_CSR, BK_SPARSE_CSC = 0, 1
BK_SIDE_NONE, BK_SIDE_LEFT, BK_SIDE_RIGHT = 0, 1, 2
BK_ORTH_CGS, BK_ORTH_CGS2 = 0, 1

SYMBOLS = [
    "bk_ctx_create", "bk_ctx_destroy", "bk_last_error", "bk_problem_size", "bk_state_size", "bk_set_params", "bk_get_stats",
    "bk_set_timing", "bk_sync", "bk_stream",
    "bk_vec_alloc", "bk_vec_free", "bk_host_alloc", "bk_host_free", "bk_vec_upload", "bk_vec_download", "bk_vec_copy", "bk_vec_zero", "bk_vec_scale",
    "bk_vec_axpby", "bk_vec_dot", "bk_vec_norm2", "bk_vec_norminf", "bk_vec_diffdot",
    "bk_residual", "bk_jac_set_state", "bk_jvp", "bk_jac_set_shift_imag", "bk_jac_set_transpose", "bk_precond_setup", "bk_precond_apply",
    "bk_gmres", "bk_gmres2", "bk_bls_bordering", "bk_bls_matrixfree", "bk_bls_map",
    "bk_bls_block_bordering", "bk_bls_block_matrixfree", "bk_bls_block_map",
    "bk_eigs_shift_invert", "bk_potrap_set_section", "bk_hessenberg_eig", "bk_palc_run",
    "bk_sparse_set_pattern", "bk_sparse_set_values",
]


class GmresOpts(C.Structure):
    _fields_ = [("reltol", C.c_double), ("abstol", C.c_double), ("restart", C.c_int32), ("maxiter", C.c_int32),
                ("pc_side", C.c_int32), ("orth", C.c_int32), ("fused", C.c_int32), ("reserved", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [("kernel_launches", C.c_int64), ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64),
                ("last_fused_ms", C.c_double), ("last_fused_bytes", C.c_int64), ("last_fused_launches", C.c_int64),
                ("total_fused_ms", C.c_double), ("total_fused_bytes", C.c_int64), ("total_fused_launches", C.c_int64),
                ("cgs_fallbacks", C.c_int64), ("total_precond_ms", C.c_double), ("total_precond_applies", C.c_int64)]


class PalcOpts(C.Structure):
    """bk_palc_opts (include/bk200.h)"""
    _fields_ = [(k, C.c_double) for k in ("ds", "dsmin", "dsmax", "a", "p_min", "p_max", "theta", "eta", "newton_tol", "fd_eps", "bls_tol")] + \
               [(k, C.c_int32) for k in ("max_steps", "newton_maxit", "lens", "tangent", "bls", "bls_check_precision", "bls_k", "normc")]


class PalcResult(C.Structure):
    """bk_palc_result"""
    _fields_ = [("nrows", C.c_int32), ("steps", C.c_int32), ("nfail", C.c_int32), ("stopped", C.c_int32),
                ("work_newton", C.c_int64), ("work_linear", C.c_int64), ("p_final", C.c_double), ("ds_final", C.c_double)]


BK_PALC_ROW = 6
# int32_t (*bk_palc_callback)(void* user, int32_t step, const double* row, const double* z_u /* device */, double z_p)
PalcCallback = C.CFUNCTYPE(C.c_int32, C.c_void_p, C.c_int32, C.POINTER(C.c_double), C.c_void_p, C.c_double)


class BK200Error(RuntimeError):
    pass


def build(verbose=False):
    """Compile libbk200.so for sm_100a with nvcc (works without a GPU)."""
    r = subprocess.run(["make", "-C", CSRC, "-j8"], capture_output=True, text=True)
    if r.returncode != 0:
        raise BK200Error("nvcc build of libbk200.so failed:\n" + r.stdout[-4000:] + r.stderr[-4000:])
    if verbose:
        print(r.stdout[-2000:])
    return LIB_PATH


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BK200Error(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                         "(no CPU fallback exists)")
    lib = C.CDLL(LIB_PATH)
    dp = C.POINTER(C.c_double)
    vp = C.c_void_p  # vectors: host or device addresses, passed as raw pointers
    i32, i64, dbl = C.c_int32, C.c_int64, C.c_double
    sig = {
        "bk_ctx_create": [i32, i32, C.POINTER(i64), dp, i32, C.POINTER(C.c_void_p)],
        "bk_ctx_destroy": [C.c_void_p],
        "bk_problem_size": [C.c_void_p],
        "bk_state_size": [C.c_void_p],
        "bk_set_params": [C.c_void_p, dp, i32],
        "bk_get_stats": [C.c_void_p, C.POINTER(Stats)],
        "bk_set_timing": [C.c_void_p, i32],
        "bk_sync": [C.c_void_p],
        "bk_stream": [C.c_void_p],
        "bk_vec_alloc": [C.c_void_p, i64, C.POINTER(C.c_void_p)],
        "bk_vec_free": [C.c_void_p, vp],
        "bk_host_alloc": [C.c_void_p, i64, C.POINTER(C.c_void_p)],
        "bk_host_free": [C.c_void_p, vp],
        "bk_vec_upload": [C.c_void_p, vp, vp, i64],
        "bk_vec_download": [C.c_void_p, vp, vp, i64],
        "bk_vec_copy": [C.c_void_p, vp, vp, i64],
        "bk_vec_zero": [C.c_void_p, vp, i64],
        "bk_vec_scale": [C.c_void_p, vp, dbl, i64],
        "bk_vec_axpby": [C.c_void_p, vp, dbl, vp, dbl, i64],
        "bk_vec_dot": [C.c_void_p, vp, vp, i64, dp],
        "bk_vec_norm2": [C.c_void_p, vp, i64, dp],
        "bk_vec_norminf": [C.c_void_p, vp, i64, dp],
        "bk_vec_diffdot": [C.c_void_p, vp, vp, vp, i64, dp],
        "bk_residual": [C.c_void_p, vp, vp],
        "bk_jac_set_state": [C.c_void_p, vp],
        "bk_jvp": [C.c_void_p, vp, vp, dbl, dbl],
        "bk_jac_set_shift_imag": [C.c_void_p, dbl],
        "bk_jac_set_transpose": [C.c_void_p, i32],
        "bk_precond_setup": [C.c_void_p, i32, dbl, dbl],
        "bk_precond_apply": [C.c_void_p, vp, vp],
        "bk_gmres": [C.c_void_p, vp, vp, dbl, dbl, C.POINTER(GmresOpts), C.POINTER(i32), C.POINTER(i32), dp],
        "bk_gmres2": [C.c_void_p, vp, vp, vp, vp, dbl, dbl, C.POINTER(GmresOpts), C.POINTER(i32), C.POINTER(i32)],
        "bk_bls_bordering": [C.c_void_p, vp, vp, dbl, vp, dbl, dbl, dbl, i32, dbl, dbl, C.POINTER(GmresOpts), i32, i32, dbl,
                             vp, dp, C.POINTER(i32), C.POINTER(i32)],
        "bk_bls_matrixfree": [C.c_void_p, vp, vp, dbl, vp, dbl, dbl, dbl, i32, dbl, dbl, C.POINTER(GmresOpts),
                              vp, dp, C.POINTER(i32), C.POINTER(i32)],
        "bk_bls_map": [C.c_void_p, vp, vp, dbl, i32, dbl, dbl, vp, vp],
        "bk_bls_block_bordering": [C.c_void_p, i32, C.POINTER(vp), C.POINTER(vp), dp, vp, dp, i32, dbl, C.POINTER(GmresOpts),
                                   vp, dp, C.POINTER(i32), C.POINTER(i32)],
        "bk_bls_block_matrixfree": [C.c_void_p, i32, C.POINTER(vp), C.POINTER(vp), dp, vp, dp, i32, dbl, dbl, C.POINTER(GmresOpts),
                                    vp, dp, C.POINTER(i32), C.POINTER(i32)],
        "bk_bls_block_map": [C.c_void_p, i32, C.POINTER(vp), C.POINTER(vp), dp, i32, dbl, dbl, vp, vp],
        "bk_eigs_shift_invert": [C.c_void_p, dbl, i32, i32, dbl, i32, C.POINTER(GmresOpts), vp, dp, dp, vp,
                                 C.POINTER(i32), C.POINTER(i32)],
        "bk_potrap_set_section": [C.c_void_p, vp, vp],
        "bk_hessenberg_eig": [dp, i32, i32, dp, dp, dp, dp],
        "bk_palc_run": [C.c_void_p, C.POINTER(PalcOpts), C.POINTER(GmresOpts), vp, dbl, vp, dbl, dp, i32, PalcCallback, C.c_void_p,
                        vp, C.POINTER(PalcResult)],
        "bk_sparse_set_pattern": [C.c_void_p, i32, i32, i64, C.POINTER(i64), C.POINTER(i64)],
        "bk_sparse_set_values": [C.c_void_p, vp],
    }
    for name, args in sig.items():
        f = getattr(lib, name)
        f.argtypes = args
        f.restype = i32
    lib.bk_problem_size.restype = i64
    lib.bk_state_size.restype = i64
    lib.bk_stream.restype = C.c_void_p
    lib.bk_last_error.argtypes = [C.c_void_p]
    lib.bk_last_error.restype = C.c_char_p
    _lib = lib
    return lib


def ptr(a):
    """Raw address of a NumPy array (host pointer) or of a DeviceVec / int (device pointer)."""
    if isinstance(a, np.ndarray):
        assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"], "vectors must be contiguous float64"
        return a.ctypes.data
    if hasattr(a, "dptr"):
        return a.dptr
    if a is None:
        return None
    return int(a)
