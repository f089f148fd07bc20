"""ctypes binding of libgsi_b200.so -- a mechanical transcription of
include/gsi_b200.h (the same table the Julia `ccall` shim uses).

The library is the only compute path: if it is missing or fails to load this
module raises; nothing here falls back to NumPy/torch/CPU.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GSI_B200_LIB") or os.path.join(_HERE, "lib", "libgsi_b200.so")   # same override as the Julia shim

# status codes (include/gsi_b200.h)
OK = 0
ERR_INVALID_ARGUMENT = 1
ERR_DIMENSION_MISMATCH = 2
ERR_SINGULAR = 3
ERR_NOT_POSDEF = 4
ERR_CUDA = 5
ERR_NCCL = 6
ERR_NO_DEVICE = 7
ERR_UNSUPPORTED = 8
ERR_NEGATIVE_ITERATIONS = 9
ERR_NO_CONVERGENCE = 10

LAYOUT_TALL = 0
LAYOUT_COLMAJOR = 1
KERNEL_EXPONENTIAL = 0
KERNEL_GAUSSIAN = 1
KERNEL_POWERLAW = 2
KERNEL_MATERN32 = 3
KERNEL_MATERN52 = 4
KERNEL_SPHERICAL = 5
MODEL_MAX_STRUCTURES = 4
NORMALISER_LU_REF = 0
NORMALISER_QR = 1

_i32, _i64, _f64 = C.c_int32, C.c_int64, C.c_double
_p = C.c_void_p
_pd = C.POINTER(C.c_double)
_pp = C.POINTER(C.c_void_p)
_pi64 = C.POINTER(C.c_int64)
_pi32 = C.POINTER(C.c_int32)

# name -> (restype, argtypes); one row per declaration in include/gsi_b200.h
SIGNATURES = {
    "gsi_version": (_i32, []),
    "gsi_last_error_string": (C.c_char_p, []),
    "gsi_comm_unique_id": (_i32, [_p]),
    "gsi_ctx_create": (_i32, [_i32, _i32, _i32, _p, _pp]),
    "gsi_ctx_destroy": (_i32, [_p]),
    "gsi_ctx_sync": (_i32, [_p]),
    "gsi_ctx_stream": (_i32, [_p, _pp]),
    "gsi_ctx_launch_count": (_i32, [_p, _pi64, _i32]),
    "gsi_ctx_gemm_timing": (_i32, [_p, _i32, _pd, _pi64, _pd]),
    "gsi_ctx_phase_timing": (_i32, [_p, _pd, _i32]),
    "gsi_ctx_set_option": (_i32, [_p, C.c_char_p, _i64]),
    "gsi_ctx_get_option": (_i32, [_p, C.c_char_p, _pi64]),
    "gsi_buf_alloc": (_i32, [_p, _i32, _i64, _i64, _pp]),
    "gsi_buf_free": (_i32, [_p]),
    "gsi_buf_dims": (_i32, [_p, _pi64, _pi64]),
    "gsi_buf_upload": (_i32, [_p, _pd, _i64]),
    "gsi_buf_download": (_i32, [_p, _pd, _i64]),
    "gsi_host_alloc": (_i32, [_p, _i64, _pp]),
    "gsi_host_free": (_i32, [_p, _p]),
    "gsi_buf_upload_rows": (_i32, [_p, _i64, _i64, _pd, _i64]),
    "gsi_buf_download_rows": (_i32, [_p, _i64, _i64, _pd, _i64]),
    "gsi_buf_copy": (_i32, [_p, _p]),
    "gsi_buf_zero": (_i32, [_p]),
    "gsi_op_dense": (_i32, [_p, _p, _i64, _i64, _pp]),
    "gsi_op_lowrankcov": (_i32, [_p, _p, _i32, _pp]),
    "gsi_op_lowrankcov_sharded": (_i32, [_p, _p, _i32, _i64, _i64, _pp]),
    "gsi_op_kernelcov": (_i32, [_p, _i32, _i32, _i64, _pd, _pd, _f64, _f64, _f64, _i64, _i64, _pp]),
    "gsi_op_kernelcov_grid": (_i32, [_p, _i32, _i32, _pi64, _pd, _pd, _f64, _f64, _f64, _i64, _i64, _pp]),
    "gsi_op_kernelcov_model": (_i32, [_p, _i32, _i64, _pd, _i32, _pi32, _pd, _pd, _pd, _pd, _f64, _i64, _i64, _pp]),
    "gsi_op_kernelcov_model_grid": (_i32, [_p, _i32, _pi64, _pd, _i32, _pi32, _pd, _pd, _pd, _pd, _f64, _i64, _i64,
                                           _pp]),
    "gsi_op_kernelcov_cross": (_i32, [_p, _i32, _i64, _pd, _i64, _pd, _i32, _pi32, _pd, _pd, _pd, _pd, _i64, _i64, _pp]),
    "gsi_op_kernelcov_cross_grid": (_i32, [_p, _i32, _pi64, _pd, _i64, _pi64, _i64, _pi64, _i32, _pi32, _pd, _pd, _pd,
                                           _pd, _i64, _i64, _pp]),
    "gsi_op_free": (_i32, [_p]),
    "gsi_op_size": (_i32, [_p, _pi64, _pi64]),
    "gsi_op_apply": (_i32, [_p, _i32, _p, _p]),
    "gsi_lu_L": (_i32, [_p, _p]),
    "gsi_qr_thinQ": (_i32, [_p, _p, _pd, _i64]),
    "gsi_svd_small": (_i32, [_p, _pd, _i64, _i64, _pd]),
    "gsi_rangefinder_fixed": (_i32, [_p, _p, _i64, _i32, _p]),
    "gsi_randsvd": (_i32, [_p, _p, _i64, _i64, _i64, _i32, _p, _pd]),
    "gsi_rangefinder_adaptive": (_i32, [_p, _p, _p, _f64, _i64, _p, _pi64]),
    "gsi_rangefinder_adaptive_blocked": (_i32, [_p, _p, _f64, _i64, _p, _pi64]),
    "gsi_eig_nystrom": (_i32, [_p, _p, _p, _pd]),
    "gsi_fftrf_powerlaw": (_i32, [_p, _i32, _pi64, _f64, _f64, _f64, _p, _p]),
    "gsi_pcga_lowrank_matvec": (_i32, [_p, _i64, _i64, _pd, _i64, _pd, _pd, _pd, _i64, _pd, _pd]),
    "gsi_pcga_lsqr_solve": (_i32, [_p, _i64, _i64, _pd, _i64, _pd, _pd, _pd, _i64, _pd, _f64, _f64, _f64,
                                   _i64, _pd, _pi64, _pi32]),
    "gsi_pcga_direct_solve": (_i32, [_p, _i64, _i64, _pd, _i64, _pd, _pd, _pd, _i64, _pd, _pd, _pi64]),
    "gsi_pcga_update": (_i32, [_p, _p, _i64, _pd, _pd, _i64, _i64, _pd, _pd]),
    "gsi_pcga_paramstorun": (_i32, [_p, _p, _i64, _pd, _pd, _f64, _p]),
    "gsi_sketch_apply": (_i32, [_p, _p, _p, _p]),
    "gsi_sketch_cov": (_i32, [_p, _p, _pd, _pd, _i64]),
}

_lib = None


class GsiError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"[gsi_b200 status {code}] {message}")
        self.code = code
        self.message = message


class SingularException(GsiError, ArithmeticError):
    """LinearAlgebra.SingularException (lu check=true, RandMatFact.jl:60,68,72)."""


class PosDefException(GsiError, ArithmeticError):
    """LinearAlgebra.PosDefException (eig_nystrom Cholesky, RandMatFact.jl:95)."""


class DimensionMismatch(GsiError, ValueError):
    pass


class NoDeviceError(GsiError):
    pass


def load():
    """dlopen libgsi_b200.so and type every entry point.  Raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python geostatinversion.jl_b200/build.py` "
            "(there is no CPU/NumPy fallback)")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status):
    if status == OK:
        return
    msg = load().gsi_last_error_string().decode("utf-8", "replace")
    if status == ERR_SINGULAR:
        raise SingularException(status, msg)
    if status == ERR_NOT_POSDEF:
        raise PosDefException(status, msg)
    if status == ERR_DIMENSION_MISMATCH:
        raise DimensionMismatch(status, msg)
    if status == ERR_NO_DEVICE:
        raise NoDeviceError(status, msg)
    if status == ERR_NEGATIVE_ITERATIONS:
        # the reference's `error(...)` text (src/RandMatFact.jl:63)
        raise GsiError(status, msg)
    raise GsiError(status, msg)
