"""ctypes binding of liblogreg_b200.so (include/logreg_b200.h).

Loading the library needs no GPU (so the symbol table can be checked on a CPU
box); every entry point that does work fails loudly with `LogregB200Error` when
there is no CUDA device. There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

LRB_OK = 0
E_NO_DEVICE, E_BAD_ARG, E_CUDA, E_NCCL, E_STATE, E_UNSUPPORTED = 1, 2, 3, 4, 5, 6
F32, F64, U8 = 0, 1, 2
ROW_MAJOR, COL_MAJOR = 0, 1
HOST, DEVICE = 0, 1
MODE_FP64, MODE_FP32 = 0, 1
RWMH, UL, MALA, HMC = 0, 1, 2, 3
RNG_PHILOX, RNG_REPLAY, RNG_KEYED = 0, 1, 2
RUN_REUSE_CACHE, RUN_SET_T0, RUN_MOMENTS, RUN_NO_SAMPLES = 1, 2, 4, 8
OPT_DETERMINISTIC, OPT_TC_MIN_CHAINS, OPT_P2P_TIMEOUT_MS, OPT_PDL, OPT_L2_PERSIST = 1, 2, 3, 4, 5


class LogregB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"liblogreg_b200 error {code}: {msg}")
        self.code = code


class SamplerParams(C.Structure):
    _fields_ = [("sampler", C.c_int32), ("l", C.c_int32), ("step", C.c_double),
                ("scale", C.POINTER(C.c_double)), ("seed", C.c_uint64),
                ("rng", C.c_int32), ("flags", C.c_int32), ("init_lpost", C.c_double), ("t0", C.c_int64)]


class MapInfo(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("converged", C.c_int32), ("halvings", C.c_int32), ("evals", C.c_int32),
                ("lpost", C.c_double), ("grad_norm", C.c_double)]


class Info(C.Structure):
    _fields_ = [("n", C.c_int64), ("p", C.c_int32), ("p_pad", C.c_int32), ("mode", C.c_int32),
                ("grid", C.c_int32), ("block", C.c_int32), ("world", C.c_int32), ("rank", C.c_int32),
                ("comm", C.c_int32), ("bytes_per_eval", C.c_int64), ("kernel_launches", C.c_int64),
                ("eval_launches", C.c_int64)]


class PredictiveTotals(C.Structure):
    _fields_ = [("n", C.c_int64), ("draws", C.c_int64), ("lppd", C.c_double), ("p_waic", C.c_double),
                ("elpd_waic", C.c_double), ("se_elpd_waic", C.c_double)]


class LooTotals(C.Structure):
    _fields_ = [("n", C.c_int64), ("draws", C.c_int64), ("elpd_loo", C.c_double), ("se_elpd_loo", C.c_double),
                ("p_loo", C.c_double), ("se_p_loo", C.c_double), ("looic", C.c_double),
                ("k_threshold", C.c_double), ("k_max", C.c_double), ("n_k_high", C.c_int64)]


_vp, _i, _i64, _u64 = C.c_void_p, C.c_int, C.c_int64, C.c_uint64
_dp = C.POINTER(C.c_double)

# name -> (restype, argtypes); must list every function include/logreg_b200.h declares
SIGNATURES = {
    "lrb_abi_version": (_i, []),
    "lrb_device_count": (_i, [C.POINTER(_i)]),
    "lrb_create": (_i, [_i, C.POINTER(_vp)]),
    "lrb_destroy": (_i, [_vp]),
    "lrb_last_error": (C.c_char_p, [_vp]),
    "lrb_set_stream": (_i, [_vp, _vp]),
    "lrb_synchronize": (_i, [_vp]),
    "lrb_set_option": (_i, [_vp, _i, _i64]),
    "lrb_get_info": (_i, [_vp, C.POINTER(Info)]),
    "lrb_bind_data": (_i, [_vp, _vp, _i, _i, _i64, _vp, _i, _i64, _i, _dp, _i, _i]),
    "lrb_gen_synthetic": (_i, [_vp, _i64, _i, _i, _u64, _dp, _dp, _i64]),
    "lrb_copy_rows": (_i, [_vp, _i64, _i64, _dp, C.POINTER(C.c_float)]),
    "lrb_eval": (_i, [_vp, _dp, _i, _i, _dp, _dp, _dp]),
    "lrb_eval_device": (_i, [_vp, _vp, _vp, _i]),
    "lrb_lprior": (_i, [_vp, _dp, _i, _dp]),
    "lrb_predictive": (_i, [_vp, _dp, _i64, _i, _vp, _vp, _vp, _vp, C.POINTER(PredictiveTotals)]),
    "lrb_loo": (_i, [_vp, _dp, _i64, _i, _vp, _vp, _vp, C.POINTER(LooTotals)]),
    "lrb_loglik": (_i, [_vp, _dp, _i64, _i64, _i64, _i, _vp]),
    "lrb_debug_psis": (_i, [_dp, _i64, _dp, _dp]),
    "lrb_map": (_i, [_vp, _dp, C.c_double, _i, _dp, C.POINTER(MapInfo)]),
    "lrb_hessian": (_i, [_vp, _dp, _dp]),
    "lrb_debug_chol_solve": (_i, [_dp, _i, _i, _dp, _dp, _dp]),
    "lrb_debug_tc_eta": (_i, [_vp, _dp, _i, C.POINTER(C.c_float)]),
    "lrb_tc_tile_rows": (_i, []),
    "lrb_debug_timeline": (_i, [_vp, _i]),
    "lrb_debug_timeline_read": (_i, [_vp, C.POINTER(_i64), _i64, C.POINTER(_i64)]),
    "lrb_run": (_i, [_vp, C.POINTER(SamplerParams), _dp, _i, _i64, _i64, _dp, _dp, _dp, C.POINTER(_i64)]),
    "lrb_run_begin": (_i, [_vp, C.POINTER(SamplerParams), _dp, _i64, _i64, _dp, _dp]),
    "lrb_run_launch": (_i, [_vp]),
    "lrb_run_finish": (_i, [_vp, _dp, C.POINTER(_i64)]),
    "lrb_chain_state": (_i, [_vp, _dp, _dp, C.POINTER(_i64)]),
    "lrb_run_evals_per_launch": (_i, [_vp, C.POINTER(_i64)]),
    "lrb_run_moments": (_i, [_vp, _i, C.POINTER(_i64), _dp, _dp]),
    "lrb_key_child": (_u64, [_u64, _u64]),
    "lrb_rng_dump": (_i, [_vp, _u64, _i64, _i64, _i, _dp, _dp]),
    "lrb_nccl_unique_id": (_i, [_vp, C.c_char_p]),
    "lrb_comm_init_nccl": (_i, [_vp, _i, _i, _vp, C.c_char_p]),
    "lrb_comm_p2p_export": (_i, [_vp, _vp]),
    "lrb_comm_p2p_connect": (_i, [_vp, _i, _i, _vp]),
}

_lib = None


def library_path() -> str:
    return os.environ.get("LRB_LIBRARY") or _build.LIB   # override: A/B a differently built library


def load(build_if_missing: bool = True):
    """dlopen the in-tree library (building it with nvcc first if it is absent)."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        if not build_if_missing:
            raise LogregB200Error(-1, f"{path} not built; run `python -m logreg_b200.build`")
        _build.build()
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError = missing export: fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error(handle=None) -> str:
    msg = load().lrb_last_error(handle)
    return msg.decode() if msg else ""


def check(rc: int, handle=None):
    if rc != LRB_OK:
        raise LogregB200Error(rc, last_error(handle))


def device_count() -> int:
    n = _i(0)
    check(load().lrb_device_count(C.byref(n)))
    return n.value


def as_dp(a):
    return a.ctypes.data_as(_dp)
