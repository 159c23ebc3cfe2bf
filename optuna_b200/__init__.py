"""optuna_b200 -- B200-native TPE suggestion engine (drop-in for optuna.samplers.TPESampler).

Host Python (this package) mirrors the reference's sampler plugin interface
(optuna/samplers/_base.py:31-228, optuna/samplers/_tpe/sampler.py:72) and calls hand-written
sm_100a CUDA through a C ABI (include/optuna_b200_tpe.h) bound with ctypes.
"""
from .engine import ParamSpec, TPEEngine  # noqa: F401

__all__ = ["ParamSpec", "TPEEngine", "B200TPESampler", "B200PedAnovaImportanceEvaluator"]


def __getattr__(name):
    if name == "B200TPESampler":
        from .sampler import B200TPESampler
        return B200TPESampler
    if name == "B200PedAnovaImportanceEvaluator":
        from .importance import B200PedAnovaImportanceEvaluator
        return B200PedAnovaImportanceEvaluator
    raise AttributeError(name)
