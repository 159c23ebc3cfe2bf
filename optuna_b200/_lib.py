"""ctypes binding of libtpe_b200.so (the C ABI declared in include/optuna_b200_tpe.h).

The library is built in-tree by ``__graft_entry__.build()`` (nvcc, sm_100a).  Loading fails loudly
when it is missing: there is no CPU fallback for the product path.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# TPE_LAB=1 loads the lab build (experimental kernels selectable by TPE_MMA_VARIANT etc., see profiles/r2_variants.md)
LIB_PATH = os.path.join(_HERE, "libtpe_b200_lab.so" if os.environ.get("TPE_LAB") == "1" else "libtpe_b200.so")

TPE_OK, TPE_E_INVALID, TPE_E_CUDA, TPE_E_STATE, TPE_E_NOMEM = 0, -1, -2, -3, -4
KIND_FLOAT, KIND_INT, KIND_CAT = 0, 1, 2
CAT_COMPLETE, CAT_PRUNED, CAT_INFEASIBLE, CAT_RUNNING, CAT_EXCLUDED = 0, 1, 2, 3, 4


class ParamDesc(C.Structure):
    _fields_ = [("kind", C.c_int32), ("log", C.c_int32), ("has_step", C.c_int32), ("n_choices", C.c_int32),
                ("low", C.c_double), ("high", C.c_double), ("step", C.c_double)]


class Cfg(C.Structure):
    _fields_ = [("prior_weight", C.c_double), ("magic_clip", C.c_int32), ("endpoints", C.c_int32),
                ("multivariate", C.c_int32), ("n_candidates", C.c_int32), ("n_below", C.c_int64)]


class SplitInfo(C.Structure):
    _fields_ = [("n_below_all", C.c_int64), ("n_below_obs", C.c_int64), ("n_above_obs", C.c_int64)]


class PedCfg(C.Structure):
    _fields_ = [("target_quantile", C.c_double), ("region_quantile", C.c_double), ("prior_weight", C.c_double),
                ("evaluate_on_local", C.c_int32), ("min_n_top", C.c_int32), ("n_steps", C.c_int32)]


# name -> (restype, argtypes); every symbol include/optuna_b200_tpe.h declares
_P = C.c_void_p
SYMBOLS = {
    "tpe_abi_version": (C.c_int, []),
    "tpe_ctx_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "tpe_ctx_destroy": (None, [_P]),
    "tpe_last_error": (C.c_char_p, [_P]),
    "tpe_space_set": (C.c_int, [_P, C.POINTER(ParamDesc), C.c_int32, _P, _P]),
    "tpe_history_set": (C.c_int, [_P, _P, _P, _P, C.c_int64]),
    "tpe_history_append": (C.c_int, [_P, _P, _P, _P, C.c_int64]),
    "tpe_history_update": (C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_int64]),
    "tpe_history_set_device": (C.c_int, [_P, _P, _P, _P, C.c_int64, _P]),
    "tpe_history_set_values": (C.c_int, [_P, _P, C.c_int64, C.c_int32, C.c_int64]),
    "tpe_history_size": (C.c_int64, [_P]),
    "tpe_history_device_ptrs": (C.c_int, [_P, C.POINTER(_P), C.POINTER(_P), C.POINTER(_P)]),
    "tpe_prepare": (C.c_int, [_P, C.POINTER(Cfg), _P, C.c_int32, C.POINTER(SplitInfo)]),
    "tpe_build": (C.c_int, [_P, _P, _P]),
    "tpe_sample_and_select": (C.c_int, [_P, _P, C.c_int64, _P, _P, _P]),
    "tpe_stage_uniforms": (C.c_int, [_P, _P, C.c_int64]),
    "tpe_stage_uniforms_mt19937": (C.c_int, [_P, _P, C.c_int32, C.c_int64, C.c_int64]),
    "tpe_rng_state": (C.c_int, [_P, _P, C.POINTER(C.c_int32)]),
    "tpe_rng_state_device": (C.c_int, [_P, C.POINTER(_P)]),
    "tpe_sample_and_select_async": (C.c_int, [_P, _P, C.c_int64]),
    "tpe_collect": (C.c_int, [_P, _P, _P, _P]),
    "tpe_set_kernel_shard": (C.c_int, [_P, C.c_int32, C.c_int32]),
    "tpe_sample_and_partial": (C.c_int, [_P, _P, C.c_int64, C.POINTER(_P), C.POINTER(C.c_int64)]),
    "tpe_finish_from_partials": (C.c_int, [_P, _P, C.c_int32, _P, _P, _P]),
    "tpe_result_device_ptrs": (C.c_int, [_P, C.POINTER(_P), C.POINTER(_P), C.POINTER(_P)]),
    "tpe_get_uniforms": (C.c_int, [_P, _P, C.c_int64]),
    "tpe_host_alloc": (C.c_int, [_P, C.c_size_t, C.POINTER(C.c_void_p)]),
    "tpe_host_free": (C.c_int, [_P, _P]),
    "tpe_suggest": (C.c_int, [_P, C.POINTER(Cfg), _P, C.c_int32, _P, _P, _P, C.c_int64, _P, _P, _P]),
    "tpe_suggest_univariate_batch": (C.c_int, [_P, C.POINTER(Cfg), _P, C.c_int32, _P, _P, _P, _P, _P, _P]),
    "tpe_suggest_univariate_batch_async": (C.c_int, [_P, C.POINTER(Cfg), _P, C.c_int32, _P, _P, _P]),
    "tpe_collect_univariate": (C.c_int, [_P, _P, _P, _P]),
    "tpe_get_split_info": (C.c_int, [_P, C.POINTER(SplitInfo)]),
    "tpe_get_split": (C.c_int, [_P, _P, _P]),
    "tpe_get_mixture": (C.c_int, [_P, C.c_int, _P, _P, _P]),
    "tpe_get_mo_weights": (C.c_int, [_P, _P]),
    "tpe_get_candidates": (C.c_int, [_P, _P, _P, _P]),
    "tpe_logpdf": (C.c_int, [_P, C.c_int, _P, C.c_int64, _P]),
    "tpe_last_timing": (C.c_int, [_P, _P, _P]),
    "tpe_probe_fp64_tflops": (C.c_int, [_P, C.POINTER(C.c_double)]),
    "tpe_last_logpdf_kernel": (C.c_char_p, [_P]),
    "tpe_ped_anova": (C.c_int, [_P, C.POINTER(PedCfg), _P, C.c_int32, _P, _P, _P, _P, _P, _P]),
}

_lib = None


ABI_VERSION = 7  # include/optuna_b200_tpe.h TPE_ABI_VERSION


def load() -> C.CDLL:
    """Load libtpe_b200.so and bind every declared symbol.  Raises if the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  optuna_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args
    if lib.tpe_abi_version() != ABI_VERSION:
        raise RuntimeError(f"libtpe_b200.so has ABI version {lib.tpe_abi_version()}, this package needs {ABI_VERSION}: "
                           "rebuild it (python -c 'import __graft_entry__ as g; g.build()')")
    _lib = lib
    return lib
