"""Time B200PedAnovaImportanceEvaluator against optuna's PedAnovaImportanceEvaluator on the benchmark's study.

Builds the config-2 study (bench.synthetic_history / bench.build_study: N trials x 32 FloatDistribution(0, 1), loss
sum (x - 0.5)^2) and times
  cold       the first get_param_importances with our evaluator (poll of every trial + history upload + device call),
  warm       one more trial added, then get_param_importances again (median over --warm-reps additions); `warm_call`
             is the library call alone (host clock around tpe_ped_anova, which returns after a device synchronise),
  reference  optuna.importance.PedAnovaImportanceEvaluator on the same study.
Checks that both evaluators give the same importances (within 1e-9 * max, same order) and prints one JSON line with
the device name and power limit beside the numbers.  Fails when no CUDA device is present.

    python tools/profile_importance.py [--trials 100000] [--warm-reps 5]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def device_info() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (s.strip() for s in out.split(","))
    return {"device": name, "power_limit": power}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--trials", type=int, default=100_000)
    ap.add_argument("--warm-reps", type=int, default=5)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("profile_importance: no CUDA device")
    import bench
    from oracle import ref
    if not ref.enable():
        sys.exit("profile_importance: optuna is not importable")
    import warnings

    import optuna
    from optuna_b200 import B200PedAnovaImportanceEvaluator
    warnings.simplefilter("ignore")

    X, loss = bench.synthetic_history(args.trials)
    t0 = time.perf_counter()
    study, space = bench.build_study(optuna, optuna.samplers.RandomSampler(seed=0), X, loss)
    build_s = time.perf_counter() - t0

    ev = B200PedAnovaImportanceEvaluator()
    t0 = time.perf_counter()
    ours = optuna.importance.get_param_importances(study, evaluator=ev, normalize=False)
    cold_s = time.perf_counter() - t0

    eng = ev._engine
    call_s = []
    inner = eng.ped_anova

    def timed(*a, **kw):
        t = time.perf_counter()
        r = inner(*a, **kw)
        call_s.append(time.perf_counter() - t)
        return r
    eng.ped_anova = timed

    rs = np.random.RandomState(1)
    warm_s = []
    for _ in range(args.warm_reps):
        x = rs.uniform(0, 1, len(bench.NAMES))
        study.add_trial(optuna.trial.create_trial(value=float(((x - 0.5) ** 2).sum()),
                                                  params=dict(zip(bench.NAMES, x.tolist())), distributions=space))
        t0 = time.perf_counter()
        ours = optuna.importance.get_param_importances(study, evaluator=ev, normalize=False)
        warm_s.append(time.perf_counter() - t0)
    ev.close()

    t0 = time.perf_counter()
    theirs = optuna.importance.get_param_importances(
        study, evaluator=optuna.importance.PedAnovaImportanceEvaluator(), normalize=False)
    ref_s = time.perf_counter() - t0

    tol = 1e-9 * max(abs(v) for v in theirs.values())
    diff = max(abs(ours[k] - theirs[k]) for k in theirs)
    names = list(theirs)
    order_ok = all(list(ours).index(a) < list(ours).index(b)
                   for i, a in enumerate(names) for b in names[i + 1:] if theirs[a] - theirs[b] > tol)
    match = set(ours) == set(theirs) and diff <= tol and order_ok
    print(json.dumps({**device_info(), "trials": len(study.trials), "params": len(space),
                      "study_build_s": round(build_s, 3), "cold_s": cold_s, "warm_s_median": float(np.median(warm_s)),
                      "warm_s": warm_s, "warm_call_s_median": float(np.median(call_s)), "reference_s": ref_s,
                      "max_abs_diff": diff, "tolerance": tol, "match": match}))
    if not match:
        sys.exit("profile_importance: importances differ from the reference")


if __name__ == "__main__":
    main()
