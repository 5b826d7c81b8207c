"""ctypes binding of libihtb200.so (see include/ihtb200.h).

This is the Python twin of julia/MendelIHTB200.jl: the same C entry points, bound with ctypes instead of ccall.
There is deliberately no CPU fallback: if the shared library is missing this module raises, and every compute
entry point returns IHTB_ECUDA when no CUDA device is present.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libihtb200.so")

IHTB_OK, IHTB_EINVAL, IHTB_EDIM, IHTB_EDOMAIN, IHTB_ENUMERIC, IHTB_ECUDA, IHTB_ENOMEM, IHTB_EUNSUPPORTED = (
    0, -1, -2, -3, -4, -5, -6, -7)
SWEEP_FAST, SWEEP_EXACT, SWEEP_PAIR = 0, 1, 2
DENSE_F64, DENSE_F32, DENSE_FIX16 = 0, 1, 2
DOSAGE16_MISSING = 65535


class IHTBError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(msg)
        self.code = code


class DimensionMismatch(IHTBError, ValueError):
    pass


class NumericError(IHTBError, FloatingPointError):
    pass


class CudaError(IHTBError):
    pass


_EXC = {IHTB_EINVAL: IHTBError, IHTB_EDIM: DimensionMismatch, IHTB_EDOMAIN: IHTBError, IHTB_ENUMERIC: NumericError,
        IHTB_ECUDA: CudaError, IHTB_ENOMEM: IHTBError, IHTB_EUNSUPPORTED: IHTBError}


class Cfg(C.Structure):
    _fields_ = [("dist", C.c_int32), ("link", C.c_int32), ("k", C.c_int64), ("nb_r", C.c_double),
                ("tol", C.c_double), ("max_iter", C.c_int32), ("min_iter", C.c_int32), ("max_step", C.c_int32),
                ("sweep_mode", C.c_int32), ("est_r", C.c_int32), ("debias", C.c_int32)]


class Result(C.Structure):
    _fields_ = [("time", C.c_double), ("logl", C.c_double), ("iter", C.c_int64), ("sigma_g", C.c_double),
                ("n_sweeps", C.c_int64), ("n_backtracks", C.c_int64), ("sweep_seconds", C.c_double),
                ("n_launches", C.c_int64), ("n_steps", C.c_int64)]


class IterTrace(C.Structure):
    _fields_ = [("logl", C.c_double), ("tol", C.c_double), ("eta", C.c_double), ("backtracks", C.c_int32),
                ("n_candidates", C.c_int32)]


_p = C.c_void_p
_pp = C.POINTER(C.c_void_p)
_f64 = C.POINTER(C.c_double)
_i64 = C.POINTER(C.c_int64)
_u8 = C.POINTER(C.c_uint8)

# name -> (argtypes); every function returns int32 except ihtb_version
SIGNATURES = {
    "ihtb_version": [],
    "ihtb_last_error": [C.c_char_p, C.c_int64],
    "ihtb_device_count": [C.POINTER(C.c_int32)],
    "ihtb_set_device": [C.c_int32],
    "ihtb_launch_count": [_i64],
    "ihtb_geno_create": [_u8, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _pp],
    "ihtb_geno_create_empty": [C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _pp],
    "ihtb_geno_load_columns": [_p, _u8, C.c_int64, C.c_int64, C.c_int64],
    "ihtb_geno_finalize": [_p],
    "ihtb_geno_counts": [_p, _i64],
    "ihtb_geno_maf": [_p, _f64],
    "ihtb_geno_create_synthetic": [C.c_int64, C.c_int64, C.c_int64, C.c_uint64, C.c_double, _pp],
    "ihtb_synth_host": [C.c_int64, C.c_int64, C.c_int64, C.c_uint64, C.c_double, _u8],
    "ihtb_geno_dims": [_p, _i64, _i64],
    "ihtb_geno_stats": [_p, _f64, _f64, _i64],
    "ihtb_geno_decode": [_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, _f64],
    "ihtb_geno_packed": [_p, C.c_int64, C.c_int64, _u8],
    "ihtb_xt_v": [_p, _f64, C.c_int64, _f64, C.c_int32],
    "ihtb_x_support": [_p, _i64, C.c_int64, _f64, C.c_int64, _f64],
    "ihtb_sweep_bench": [_p, C.c_int32, C.c_int32, C.c_int32, _f64, _f64],
    "ihtb_geno_sweep_stream_bytes": [_p, C.POINTER(C.c_int64), C.POINTER(C.c_int32)],
    "ihtb_gather_bench": [_p, C.c_int64, C.c_int32, _f64, _f64],
    "ihtb_geno_ternary_tiles": [_p, _u8, C.c_int64],
    "ihtb_geno_destroy": [_p],
    "ihtb_geno_create_dense": [_p, C.c_int32, C.c_int64, C.c_int64, C.c_int64, C.c_int32, _pp],
    "ihtb_geno_create_dense_empty": [C.c_int64, C.c_int64, C.c_int32, C.c_int32, _pp],
    "ihtb_geno_load_dense_columns": [_p, _p, C.c_int64, C.c_int64, C.c_int64],
    "ihtb_geno_create_dosage16": [_p, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_int32, _pp],
    "ihtb_geno_create_dosage16_empty": [C.c_int64, C.c_int64, C.c_int32, C.c_int32, _pp],
    "ihtb_geno_load_bgen_columns": [_p, _u8, _i64, C.c_int64, C.c_int64, C.c_int32],
    "ihtb_bgen_set_batch_bytes": [C.c_int64],
    "ihtb_fit_create": [_p, _f64, _f64, C.c_int64, _u8, C.POINTER(Cfg), _pp],
    "ihtb_fit_create_sharded": [_p, _p, C.c_int64, _f64, _f64, C.c_int64, _u8, C.POINTER(Cfg), _pp],
    "ihtb_fit_set_weights": [_p, _f64],
    "ihtb_fit_set_groups": [_p, C.POINTER(C.c_int32), C.c_int32, _i64, C.c_int64],
    "ihtb_fit_set_k": [_p, C.c_int64],
    "ihtb_fit_init": [_p, _u8],
    "ihtb_fit_init_beta": [_p, _u8],
    "ihtb_fit_run": [_p, C.POINTER(Result), C.POINTER(IterTrace), C.c_int64],
    "ihtb_fit_get": [_p, _f64, _f64, _f64, _f64],
    "ihtb_fit_get_sparse": [_p, C.POINTER(C.c_int64), _f64, C.c_int64, C.POINTER(C.c_int64)],
    "ihtb_fit_predict": [_p, _u8, _f64],
    "ihtb_fit_timer": [_p, C.c_int32, _f64],
    "ihtb_fit_phase_times": [_p, _f64],
    "ihtb_fit_destroy": [_p],
    "ihtb_cv_run": [_p, _f64, _f64, C.c_int64, _u8, C.POINTER(Cfg), C.POINTER(C.c_int32), C.c_int32, _i64, C.c_int64,
                    _f64, _f64, _i64],
    "ihtb_mvfit_create": [_p, _f64, C.c_int64, _f64, C.c_int64, C.POINTER(Cfg), _pp],
    "ihtb_mvfit_create_sharded": [_p, _p, C.c_int64, _f64, C.c_int64, _f64, C.c_int64, C.POINTER(Cfg), _pp],
    "ihtb_mvfit_set_k": [_p, C.c_int64],
    "ihtb_mvfit_init": [_p, _u8],
    "ihtb_mvfit_init_beta": [_p, _u8],
    "ihtb_mvfit_run": [_p, C.POINTER(Result), C.POINTER(IterTrace), C.c_int64],
    "ihtb_mvfit_get": [_p, _f64, _f64, _f64, _f64],
    "ihtb_mvfit_predict": [_p, _u8, _f64],
    "ihtb_mvfit_destroy": [_p],
    "ihtb_comm_unique_id": [C.c_char_p, _u8],
    "ihtb_comm_create": [C.c_char_p, _u8, C.c_int32, C.c_int32, _pp],
    "ihtb_comm_destroy": [_p],
    "ihtb_comm_stats": [_p, _i64, _i64],
    "ihtb_comm_allreduce_bench": [_p, C.c_int64, C.c_int32, C.c_int32, _f64],
    "ihtb_geno_set_offset": [_p, C.c_int64],
    "ihtb_mgeno_create": [_u8, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                          C.POINTER(C.c_int32), C.c_int32, _pp],
    "ihtb_mgeno_create_synthetic": [C.c_int64, C.c_int64, C.c_uint64, C.c_double, C.c_int32, C.POINTER(C.c_int32),
                                    C.c_int32, _pp],
    "ihtb_mgeno_info": [_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), _i64, _i64],
    "ihtb_mgeno_part": [_p, C.c_int32, _pp, C.POINTER(C.c_int32), _i64],
    "ihtb_mgeno_destroy": [_p],
    "ihtb_mfit_create": [_p, _f64, _f64, C.c_int64, _u8, C.POINTER(Cfg), _pp],
    "ihtb_mfit_set_weights": [_p, _f64],
    "ihtb_mfit_set_groups": [_p, C.POINTER(C.c_int32), C.c_int32, _i64, C.c_int64],
    "ihtb_mfit_set_k": [_p, C.c_int64],
    "ihtb_mfit_init": [_p, _u8, C.c_int32],
    "ihtb_mfit_run": [_p, C.POINTER(Result), C.POINTER(IterTrace), C.c_int64],
    "ihtb_mfit_get": [_p, _f64, _f64, _f64, _f64],
    "ihtb_mfit_get_sparse": [_p, C.POINTER(C.c_int64), _f64, C.c_int64, C.POINTER(C.c_int64)],
    "ihtb_mfit_predict": [_p, _u8, _f64],
    "ihtb_mfit_timer": [_p, C.c_int32, _f64],
    "ihtb_mfit_destroy": [_p],
    "ihtb_mmvfit_create": [_p, _f64, C.c_int64, _f64, C.c_int64, C.POINTER(Cfg), _pp],
    "ihtb_mmvfit_set_k": [_p, C.c_int64],
    "ihtb_mmvfit_init": [_p, _u8, C.c_int32],
    "ihtb_mmvfit_run": [_p, C.POINTER(Result), C.POINTER(IterTrace), C.c_int64],
    "ihtb_mmvfit_get": [_p, _f64, _f64, _f64, _f64],
    "ihtb_mmvfit_predict": [_p, _u8, _f64],
    "ihtb_mmvfit_destroy": [_p],
    "ihtb_mcv_run": [_p, _f64, _f64, C.c_int64, _u8, C.POINTER(Cfg), C.POINTER(C.c_int32), C.c_int32, _i64, C.c_int64,
                     _f64, _f64, _i64, _f64],
}

_lib = None


def load() -> C.CDLL:
    """Load the CUDA library; fail loudly if it has not been built (no fallback path exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: the CUDA extension has not been built. "
                "Run `python -c 'import __graft_entry__ as g; g.build()'` (needs nvcc). "
                "mendeliht.jl_b200 has no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, args in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.argtypes = args
            fn.restype = C.c_int32
        _lib = lib
    return _lib


def last_error() -> str:
    buf = C.create_string_buffer(1024)
    load().ihtb_last_error(buf, 1024)
    return buf.value.decode("utf-8", "replace")


def check(status: int) -> None:
    if status != IHTB_OK:
        raise _EXC.get(status, IHTBError)(status, last_error())


def f64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float64)


def ptr(a: np.ndarray, ctype):
    return a.ctypes.data_as(C.POINTER(ctype)) if a is not None else None


def device_count() -> int:
    n = C.c_int32(0)
    load().ihtb_device_count(C.byref(n))
    return int(n.value)


def launch_count() -> int:
    n = C.c_int64(0)
    check(load().ihtb_launch_count(C.byref(n)))
    return int(n.value)
