"""ctypes binding of libssi.so (include/ssi.h).  No fallback: if the library is missing or
no sm_100 device is usable, every compute call raises."""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import os

PKG = Path(__file__).resolve().parent
# SSI_LIB_PATH: load another build of the same library (A-B measurements of two builds in one GPU session)
LIB_PATH = Path(os.environ["SSI_LIB_PATH"]).resolve() if os.environ.get("SSI_LIB_PATH") else PKG / "lib" / "libssi.so"

SSI_OK = 0
ERR_NAMES = {-1: "SSI_ERR_ARG", -2: "SSI_ERR_CUDA", -3: "SSI_ERR_STATE", -4: "SSI_ERR_RANK", -5: "SSI_ERR_UNSUPPORTED", -6: "SSI_ERR_RANGE"}

ACT_IDENTITY, ACT_RELU, ACT_TANH, ACT_SIGMOID = 0, 1, 2, 3
TERM_LL, TERM_PRIOR_W, TERM_PRIOR_Z = 1, 2, 4
PATH_AUTO, PATH_FUSED, PATH_LAYERED, PATH_TENSOR, PATH_BASIS = 0, 1, 2, 3, 4
PATH_NAMES = {0: "auto", 1: "fused", 2: "layered", 3: "tensor", 4: "basis"}


class SsiError(RuntimeError):
    """Raised for every non-zero return code of the C ABI (the Julia shim throws a String,
    as the reference does at src/space_inference.jl:42,103,162)."""

    def __init__(self, code: int, msg: str):
        super().__init__(f"{ERR_NAMES.get(code, code)}: {msg}")
        self.code = code


class Stats(C.Structure):
    _fields_ = [
        ("last_ms", C.c_double), ("last_flops", C.c_double), ("last_bytes", C.c_double), ("last_units", C.c_double),
        ("kernel_launches", C.c_int64), ("mh_accepts", C.c_int64), ("mh_proposals", C.c_int64),
        ("last_path", C.c_int32), ("sm_count", C.c_int32),
        ("gram_path", C.c_int32), ("jacobi_sweeps", C.c_int32), ("gram_risk", C.c_double),
        ("dominant_ms", C.c_double), ("dominant_launches", C.c_int64),
        ("finish_gram_ms", C.c_double), ("finish_eigen_ms", C.c_double), ("finish_p_ms", C.c_double),
        ("tc_range_fallbacks", C.c_int64), ("gemm_tc_launches", C.c_int64), ("gemm_skinny_launches", C.c_int64),
    ]


class HmcParams(C.Structure):
    """ssi_hmc_params_t."""
    _fields_ = [("step_size", C.c_double), ("n_leapfrog", C.c_int32), ("n_adapts", C.c_int64), ("target_accept", C.c_double),
                ("inv_metric", C.c_void_p)]


_p, _i64, _i32, _u32, _u64, _dbl = C.c_void_p, C.c_int64, C.c_int32, C.c_uint32, C.c_uint64, C.c_double

# name -> (restype, argtypes); kept in one table so tests can check it against include/ssi.h
SIGNATURES = {
    "ssi_version": (C.c_int, []),
    "ssi_ctx_create": (C.c_int, [C.c_int, C.POINTER(_p)]),
    "ssi_ctx_create_multi": (C.c_int, [_p, _i32, C.POINTER(_p)]),
    "ssi_ctx_devices": (C.c_int, [_p]),
    "ssi_ctx_destroy": (C.c_int, [_p]),
    "ssi_last_error": (C.c_char_p, [_p]),
    "ssi_set_stream": (C.c_int, [_p, _p]),
    "ssi_sync": (C.c_int, [_p]),
    "ssi_set_option": (C.c_int, [_p, C.c_char_p, _i64]),
    "ssi_stats": (C.c_int, [_p, C.POINTER(Stats)]),
    "ssi_set_model": (C.c_int, [_p, C.c_int, _p, _p]),
    "ssi_set_data": (C.c_int, [_p, _p, _p, _i64]),
    "ssi_set_subspace": (C.c_int, [_p, _p, _p, _i64, _i32]),
    "ssi_set_decoder": (C.c_int, [_p, _p, _i32, _p, _p, _p]),
    "ssi_logpost_batch": (C.c_int, [_p, _p, _i64, _dbl, _dbl, _dbl, _u32, _p, _p]),
    "ssi_logpost_batch_dev": (C.c_int, [_p, _p, _i64, _dbl, _dbl, _dbl, _u32, _p, _p]),
    "ssi_logpost_grad_batch": (C.c_int, [_p, _p, _i64, _dbl, _dbl, _dbl, _u32, _p, _p]),
    "ssi_logpost_grad_batch_dev": (C.c_int, [_p, _p, _i64, _dbl, _dbl, _dbl, _u32, _p, _p]),
    "ssi_mh_run": (C.c_int, [_p, _i64, _i64, _u64, _i64, _dbl, _dbl, _dbl, _u32, _p, _p, _p, _p]),
    "ssi_mh_run_dev": (C.c_int, [_p, _i64, _i64, _u64, _i64, _dbl, _dbl, _dbl, _u32, _p, _p, _p, _p]),
    "ssi_mala_run": (C.c_int, [_p, _i64, _i64, _u64, _i64, _dbl, _dbl, _dbl, _u32, _p, _p, _p, _p]),
    "ssi_mala_run_dev": (C.c_int, [_p, _i64, _i64, _u64, _i64, _dbl, _dbl, _dbl, _u32, _p, _p, _p, _p]),
    "ssi_mh_get_state": (C.c_int, [_p, _p, _p]),
    "ssi_mh_run_from": (C.c_int, [_p, _i32, _i64, _i64, _u64, _i64, _i64, _dbl, _dbl, _dbl, _u32, _p, _p, _p, _p]),
    "ssi_mh_run_from_dev": (C.c_int, [_p, _i32, _i64, _i64, _u64, _i64, _i64, _dbl, _dbl, _dbl, _u32, _p, _p, _p, _p]),
    "ssi_hmc_run": (C.c_int, [_p, _i64, _i64, _u64, _i64, _i64, C.POINTER(HmcParams), _dbl, _dbl, _dbl, _u32, _p, _p, _p, _p, _p, _p]),
    "ssi_hmc_run_dev": (C.c_int, [_p, _i64, _i64, _u64, _i64, _i64, C.POINTER(HmcParams), _dbl, _dbl, _dbl, _u32, _p, _p, _p, _p, _p, _p]),
    "ssi_hmc_get_adapt": (C.c_int, [_p, _p]),
    "ssi_rng_replay": (C.c_int, [_u64, _i64, _i64, _i32, _p, _p]),
    "ssi_project": (C.c_int, [_p, _p, _i64, _p]),
    "ssi_predict_batch": (C.c_int, [_p, _p, _i64, _p, _i64, _p, _p, _p]),
    "ssi_swa_begin": (C.c_int, [_p, _i64, _i64]),
    "ssi_swa_push": (C.c_int, [_p, _p, _dbl]),
    "ssi_swa_push_dev": (C.c_int, [_p, _p, _dbl]),
    "ssi_swa_finish": (C.c_int, [_p, _i32, _p, _p, _p, _i32]),
    "ssi_swa_columns": (_i64, [_p]),
    "ssi_swa_deviations": (C.c_int, [_p, _p]),
    "ssi_swa_mean": (C.c_int, [_p, _p]),
    "ssi_train_begin": (C.c_int, [_p, _p, C.c_int32, _dbl, _dbl, _dbl]),
    "ssi_train_step": (C.c_int, [_p, _p, _i64, _i64, _p]),
    "ssi_train_snapshot": (C.c_int, [_p, _dbl]),
    "ssi_train_get_weights": (C.c_int, [_p, _p]),
    "ssi_train_end": (C.c_int, [_p]),
    "ssi_swa_gram_dev": (C.c_int, [_p, _p, _i32]),
    "ssi_swa_finish_gram": (C.c_int, [_p, _i32, _p, _i32, _p, _p, _p, _i32]),
}
RETRY_EXACT = 1

_lib = None


def load() -> C.CDLL:
    """dlopen libssi.so and declare every prototype.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ImportError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback)")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)        # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
