#!/usr/bin/env python
"""bench.py -- TPE suggestions/sec at a 100k-trial history (BASELINE.json metric).

Workload (config.workload "c2"): N = 100 000 COMPLETE trials x P = 32 FloatDistribution(0, 1)
params, X = RandomState(0).uniform, loss = sum((x - 0.5)^2), n_ei_candidates C = 4096,
multivariate TPE, default gamma (n_below = 25) -- SURVEY.md section 8d.  One *step* = one
suggestion = split + both Parzen-estimator builds + C candidate draws + log l(x) and log g(x) over
the C x K x P grid + argmax.  Nothing is cached between steps.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

``value``  device-resident throughput: the K timed steps go through the C ABI (tpe_suggest) with the
           history already in HBM; time = wall clock between device synchronisations around the K
           steps (each call ends with a stream sync), max over ranks; the CUDA-event time of the same
           steps is reported as ``device_ms_per_step``.
``e2e``    the same metric through the call a user makes: the UNMODIFIED optuna package (oracle/_ref,
           the reference itself) drives ``B200TPESampler`` -- ``optuna.create_study(sampler=...)`` with the
           100k trials added by ``study.add_trials``, then per step ``trial = study.ask()``, 32 x
           ``trial.suggest_float`` (the first one triggers infer_relative_search_space + sample_relative),
           ``study.tell(trial, value)``: every step appends a trial, so every step also ingests one.
           optuna's own per-trial bookkeeping is inside the timed region.  The sampler computes suggestions
           ahead of the ask where the call order allows it (DESIGN.md section 1b: queued when the previous
           suggestion has been handed out, confirmed at tell time); every step is still one full ask + tell and
           ``e2e.host`` reports the same loop with that switched off (``per_trial_ms_without_look_ahead``), the
           time the caller waits, and how many look-aheads / speculations were kept.
``extras`` (N = 1)  other shapes of the same path: the default n_ei_candidates = 24 and univariate TPE through
           optuna's Study, the batched univariate trial, config 3 (mixed, C = 24 / 4096), config 4 (MOTPE), batched asks.
``config5`` 8192 asks sharded over the ranks (strong scaling); ``kernel_sharded`` (N > 1): ONE suggestion evaluated
           by all ranks together (g(x) sharded over the kernels, one all-gather of per-candidate partials).
``--impl reference``  the reference ITSELF on the host cores: optuna's own ``_split_trials``,
           ``_ParzenEstimator`` and ``log_pdf`` (oracle/_ref, unmodified) on the same 100k-trial study;
           each step is a bounded sample (see run_reference).
``--dump-outputs DIR``  after the timed steps, rank 0 writes what the last timed step computed as float64 .npy files:
           what tpe_suggest returns (x, acq, best) and the candidates behind it (tpe_get_candidates: candidates,
           log_l, log_g; 1.1 MB in all).  The inputs are seeded, so two builds can be compared output for output.
           log_g is a sum over 100k kernels whose order varies from run to run: on a B200 two runs of the same build
           differ in its last bits (2.5e-15 relative); everything else is bit-identical.

The benchmark writes nothing into the source tree (no bytecode caches either): it may run from a read-only checkout.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_TRIALS, N_PARAMS, N_CAND = 100_000, 32, 4096
METRIC = "TPE suggestions/sec at 100k-trial history, 32 params"
UNIT = "suggestions/s"


def synthetic_history(n=None, p=N_PARAMS):
    n = N_TRIALS if n is None else n
    rs = np.random.RandomState(0)
    X = rs.uniform(0, 1, (n, p))
    loss = ((X - 0.5) ** 2).sum(1)
    return X, loss


def algorithmic_bytes(n=N_TRIALS, p=N_PARAMS, c=N_CAND, m=1) -> int:
    """SURVEY.md section 8d: every input read once, every output written once (multivariate)."""
    return 8 * (n * p + n * m + n) + 16 * c * p + 16 * c


def algorithmic_flops(n=N_TRIALS, p=N_PARAMS, c=N_CAND, n_below=25) -> float:
    """SURVEY.md section 8d: C * (K_below + K_above) * (4 P + 25)."""
    return float(c) * (n + 2) * (4 * p + 25)


def executed_flops(n=N_TRIALS, p=N_PARAMS, c=N_CAND) -> float:
    """fp64 flops the g(x) grid kernel issues: C x K_above x P fma on the tensor-core path."""
    return 2.0 * c * (n - 25) * p


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (NVML, ~1 kHz; nvidia-smi
    subprocesses are too slow for a 50 ms region and remain only as a fallback)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int) -> None:
        self.index = index
        self.sm: list[float] = []
        self.max_sm = None
        self.reasons: set[str] = set()
        self._stop = threading.Event()
        self._t: threading.Thread | None = None
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nvml = None

    def _poll_nvml(self) -> None:
        n = self._nvml
        bits = {"hw_slowdown": getattr(n, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                "hw_thermal_slowdown": getattr(n, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(n, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": getattr(n, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        while not self._stop.is_set():
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM)))
                r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for name, bit in bits.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.002)

    def _poll_smi(self) -> None:
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                for line in out.strip().splitlines():
                    c = [v.strip() for v in line.split(",")]
                    self.sm.append(float(c[0]))
                    self.max_sm = float(c[1])
                    for i, nm in enumerate(names):
                        if len(c) > 3 + i and c[3 + i].lower().startswith("active"):
                            self.reasons.add(nm)
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self) -> None:
        self._t = threading.Thread(target=self._poll_nvml if self._nvml else self._poll_smi, daemon=True)
        self._t.start()

    def stop(self) -> dict:
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_sm,
                "reasons": sorted(self.reasons), "samples": len(self.sm),
                "source": "nvml" if self._nvml else "nvidia-smi"}


def measured_peaks() -> tuple[float, str]:
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "MEASURED_PEAKS.json"
        except Exception:
            pass
    return 6650.0, "fallback"


# -------------------------------------------------------------------------------------------------
# the reference as the caller (e2e) and as the CPU baseline (unmodified optuna from oracle/_ref)
# -------------------------------------------------------------------------------------------------
WORKLOAD = "c2: N=100000 trials x P=32 float params, C=4096 candidates, multivariate TPE"
CONFIG = {"workload": WORKLOAD, "n_trials": N_TRIALS, "n_params": N_PARAMS, "n_ei_candidates": N_CAND,
          "l2": "inputs larger than L2: every step rebuilds the 51 MB g(x) kernel table (126 MB L2; the split / "
                "build kernels in between evict it)"}
NAMES = [f"x{j:02d}" for j in range(N_PARAMS)]


def import_optuna():
    """The reference package: an installed optuna, else the copy build() left under oracle/_ref (oracle/build_ref.py)."""
    from oracle import ref
    if not ref.enable():
        raise RuntimeError("optuna is not importable and oracle/_ref is absent (run `python oracle/build_ref.py`)")
    import optuna
    optuna.logging.set_verbosity(optuna.logging.ERROR)
    import warnings
    warnings.filterwarnings("ignore", category=optuna.exceptions.ExperimentalWarning)
    return optuna


def build_study(optuna, sampler, X, loss):
    """optuna.create_study + study.add_trials of the synthetic history (SURVEY.md section 8d)."""
    space = {name: optuna.distributions.FloatDistribution(0.0, 1.0) for name in NAMES}
    study = optuna.create_study(sampler=sampler)
    study.add_trials([optuna.trial.create_trial(value=float(loss[i]), params=dict(zip(NAMES, X[i].tolist())),
                                                distributions=space) for i in range(X.shape[0])])
    # 100k FrozenTrials = millions of long-lived Python objects: without this the cyclic GC re-scans them from time
    # to time in the middle of a timed step (10-20 ms pauses).  Both arms build their study here.
    import gc
    gc.collect()
    gc.freeze()
    return study, space


class ReferenceSuggestion:
    """One c2 suggestion by the reference's own code, cut into the pieces a bounded sample needs.

    `fixed()` runs, once and in full, what `TPESampler._sample` (sampler.py:523-553) does before the grid:
    study._get_trials, _split_trials, both _build_parzen_estimator calls and mpe_below.sample(rng, 4096).
    `chunk(lo, hi)` evaluates rows [lo, hi) of the 4096 candidates under both estimators with the reference's
    `_ParzenEstimator.log_pdf` -- the chunked-candidate driver BASELINE.md section 3 prescribes, because the
    un-chunked call needs a 105 GB (C, K, P) temporary.  The grid is linear in the candidate count, so
    full_s = fixed_s + chunk_s / rows * 4096 / processes."""

    def __init__(self, optuna, study, space):
        from optuna.samplers._tpe import sampler as ref_sampler
        self.optuna, self.mod, self.study, self.space = optuna, ref_sampler, study, space
        self.sampler = optuna.samplers.TPESampler(seed=1, n_ei_candidates=N_CAND, multivariate=True)

    def fixed(self) -> dict:
        s, st = self.sampler, self.optuna.trial.TrialState
        t0 = time.perf_counter()
        trials = self.study._get_trials(deepcopy=False, states=(st.COMPLETE, st.PRUNED), use_cache=False)
        below, above = self.mod._split_trials(self.study, trials, s._gamma(len(trials)), False)
        t1 = time.perf_counter()
        self.mpe_below = s._build_parzen_estimator(self.study, self.space, below, handle_below=True)
        self.mpe_above = s._build_parzen_estimator(self.study, self.space, above, handle_below=False)
        t2 = time.perf_counter()
        self.samples = self.mpe_below.sample(s._rng.rng, N_CAND)
        t3 = time.perf_counter()
        return {"split_s": t1 - t0, "build_s": t2 - t1, "sample_s": t3 - t2, "fixed_s": t3 - t0}

    def chunk(self, lo: int, hi: int) -> float:
        part = {k: v[lo:hi] for k, v in self.samples.items()}
        return float((self.mpe_below.log_pdf(part) - self.mpe_above.log_pdf(part)).sum())


_REF: ReferenceSuggestion | None = None


def _ref_chunk(args):
    return _REF.chunk(*args)


def run_reference(args) -> None:
    """`--impl reference`: the reference itself (oracle/_ref) on the host cores, c2.

    Setup (untimed): the 100k-trial study; one full run of the fixed part of a suggestion (split, both
    estimator builds, 4096 draws -- single process, like the reference).  Each STEP (timed) evaluates
    `rows` candidates per process under l(x) and g(x) with the reference's log_pdf in `procs` forked processes
    (NumPy's elementwise kernels are single-threaded: this is how the reference can use the host's cores at
    all).  ms_per_step is the wall time of that step; `value` is the suggestion rate this implies for the whole
    4096-candidate suggestion (formula in `extrapolation`) -- a full one takes hours, BASELINE.md section 2."""
    global _REF
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    optuna = import_optuna()
    X, loss = synthetic_history()
    t0 = time.perf_counter()
    study, space = build_study(optuna, optuna.samplers.RandomSampler(seed=0), X, loss)
    setup_s = time.perf_counter() - t0
    _REF = ReferenceSuggestion(optuna, study, space)
    fixed = _REF.fixed()
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, 32))
    rows = 4   # per process and step: 4 x 25.6 MB per (K, P) temporary; the per-call overhead is < 10 % of a chunk
    times = []
    with mp.get_context("fork").Pool(procs) as pool:
        for i in range(args.warmup + args.steps):
            base = (i * procs * rows) % (N_CAND - procs * rows)
            t0 = time.perf_counter()
            pool.map(_ref_chunk, [(base + q * rows, base + (q + 1) * rows) for q in range(procs)])
            if i >= args.warmup:
                times.append(time.perf_counter() - t0)
    step_s = float(np.mean(times))
    per_cand_s = step_s / (procs * rows)          # seconds per candidate with every process busy
    full_s = fixed["fixed_s"] + per_cand_s * N_CAND
    val = 1.0 / full_s
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_s * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": dict(CONFIG),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": procs, "kind": "reference",
                         "sample": (f"unmodified optuna (oracle/_ref): fixed part of one suggestion run once in full "
                                    f"({fixed['fixed_s']:.1f} s: _split_trials {fixed['split_s']:.1f}, two "
                                    f"_ParzenEstimator builds {fixed['build_s']:.1f}, 4096 draws {fixed['sample_s']:.1f}); "
                                    f"each step = _ParzenEstimator.log_pdf of {rows} candidate(s) x {procs} processes "
                                    f"under l(x) and g(x) ({step_s:.2f} s)")},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "measured": dict(fixed, step_s=step_s, candidates_per_step=procs * rows, processes=procs,
                         study_setup_s=setup_s, host_cores=cores),
        "extrapolation": {"full_suggestion_s": full_s,
                          "formula": "fixed_s + step_s / candidates_per_step * 4096 (the grid is linear in the "
                                     "candidate count; the un-chunked call needs a 105 GB temporary)",
                          "fraction_of_a_suggestion_per_step": procs * rows / N_CAND},
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_leg(optuna, study, space) -> dict:
    """The reference on ONE core (what a user of the reference gets: NumPy elementwise kernels are
    single-threaded, SURVEY.md section 6) -- bounded sample: fixed part once, log_pdf of 2 and then 6 candidates."""
    ref = ReferenceSuggestion(optuna, study, space)
    fixed = ref.fixed()
    ref.chunk(8, 9)  # first-touch / lazy-import cost of the first call is not the reference's steady state
    t0 = time.perf_counter()
    ref.chunk(0, 2)
    t1 = time.perf_counter()
    ref.chunk(2, 8)
    t2 = time.perf_counter()
    per = (t2 - t0) / 8.0
    full = fixed["fixed_s"] + per * N_CAND
    return {"value": 1.0 / full, "unit": UNIT, "cores": 1, "kind": "reference",
            "sample": (f"unmodified optuna (oracle/_ref), 1 process: _split_trials + both _ParzenEstimator builds + 4096 "
                       f"draws in full ({fixed['fixed_s']:.1f} s); log_pdf under l(x) and g(x) of 8 of the 4096 candidates "
                       f"({t2 - t0:.1f} s, {per:.2f} s per candidate) -> {full:.0f} s per suggestion")}


# -------------------------------------------------------------------------------------------------
# GPU arm
# -------------------------------------------------------------------------------------------------
def dump_outputs(out_dir: str, eng, x, acq, best) -> None:
    """The last timed suggestion as DIR/<name>.npy (float64): the returned point, acquisition value and candidate
    index, and the 4096 candidates with their log-densities under l(x) and g(x)."""
    os.makedirs(out_dir, exist_ok=True)
    smp, ll, lg = eng.get_candidates()
    for name, a in (("x", x), ("acq", acq), ("best", best), ("candidates", smp), ("log_l", ll), ("log_g", lg)):
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(a, dtype=np.float64))


def run_b200(args) -> None:
    import torch
    import torch.distributed as dist

    from optuna_b200 import ParamSpec, TPEEngine

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    X, loss = synthetic_history()
    cat = np.zeros(N_TRIALS, np.int8)
    key = np.stack([loss, np.zeros(N_TRIALS)], 1)
    eng = TPEEngine(local)
    eng.set_space([ParamSpec(kind=0, low=0.0, high=1.0) for _ in range(N_PARAMS)])
    if world > 1:
        # frozen history: rank 0 uploads, ONE NCCL broadcast over NVLink, every rank adopts the buffer
        dev = torch.device("cuda", local)
        tX = torch.empty((N_TRIALS, N_PARAMS), dtype=torch.float64, device=dev)
        tk = torch.empty((N_TRIALS, 2), dtype=torch.float64, device=dev)
        tc = torch.empty((N_TRIALS,), dtype=torch.int8, device=dev)
        if rank == 0:
            tX.copy_(torch.from_numpy(X))
            tk.copy_(torch.from_numpy(key))
            tc.copy_(torch.from_numpy(cat))
        flat = torch.cat([tX.view(-1), tk.view(-1)])
        dist.broadcast(torch.zeros(1, device=dev), 0)   # NCCL communicator set-up is not the broadcast
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        dist.broadcast(flat, 0)
        dist.broadcast(tc, 0)
        torch.cuda.synchronize()
        bcast_ms = (time.perf_counter() - t0) * 1e3
        tX = flat[: N_TRIALS * N_PARAMS].view(N_TRIALS, N_PARAMS).contiguous()
        tk = flat[N_TRIALS * N_PARAMS:].view(N_TRIALS, 2).contiguous()
        torch.cuda.synchronize()
        eng.set_history_device(tX.data_ptr(), tc.data_ptr(), tk.data_ptr(), N_TRIALS, np.zeros(N_PARAMS, np.uint8))
    else:
        eng.set_history(X, cat, key)
        bcast_ms = None

    cols = list(range(N_PARAMS))
    cfg = dict(n_below=min(math.ceil(0.1 * N_TRIALS), 25), n_candidates=N_CAND, multivariate=True)
    per_ask = N_CAND * (1 + N_PARAMS)
    rng = np.random.RandomState(1000 + rank)
    total = args.warmup + args.steps
    U = torch.empty((total, per_ask), dtype=torch.float64).pin_memory()
    U.numpy()[:] = rng.random_sample((total, per_ask))
    Unp = U.numpy()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        eng.suggest(cols, Unp[i], 1, **cfg)
    clocks = ClockSampler(local)
    barrier()
    if rank == 0:
        clocks.start()
    stage = np.zeros(9)
    launches = 0
    t0 = time.perf_counter()
    for i in range(args.warmup, total):
        x_last, acq_last, best_last = eng.suggest(cols, Unp[i], 1, **cfg)
        ms, nl = eng.last_timing()
        stage += ms
        launches += nl
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    barrier()
    clk = clocks.stop() if rank == 0 else {}
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, eng, x_last, acq_last, best_last)
    kernel_name = eng.last_logpdf_kernel()
    wall = t1 - t0
    dev_ms = float(stage[8])
    if world > 1:
        t = torch.tensor([wall, dev_ms], dtype=torch.float64, device=torch.device("cuda", local))
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        wall, dev_ms = float(t[0]), float(t[1])
    value = world * args.steps / wall

    # ---- end to end: optuna's own Study drives the plugin (host buffers, copies inside the timed region) ----
    optuna = import_optuna()
    from optuna_b200 import B200TPESampler
    sampler = B200TPESampler(seed=1 + rank, n_ei_candidates=N_CAND, multivariate=True, device=local)
    t0 = time.perf_counter()
    study, space = build_study(optuna, sampler, X, loss)
    study_setup_s = time.perf_counter() - t0

    def one_trial():
        trial = study.ask()
        x = [trial.suggest_float(name, 0.0, 1.0) for name in NAMES]
        study.tell(trial, sum((v - 0.5) ** 2 for v in x))
        return x

    e2e_steps = max(3, min(2 * args.steps, 50))
    t0 = time.perf_counter()
    one_trial()                      # first ask: the one-time walk + upload of the 100k-trial history
    first_ask_s = time.perf_counter() - t0
    for _ in range(max(2, min(args.warmup, 3))):
        one_trial()
    barrier()
    # the same loop with the sampler's look-ahead switched off (every ask then computes its suggestion while the
    # caller waits): reported beside the headline, not instead of it
    sampler.LOOK_AHEAD = False
    one_trial()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        one_trial()
    torch.cuda.synchronize()
    plain_wall = time.perf_counter() - t0
    sampler.LOOK_AHEAD = True
    one_trial()
    barrier()
    sync_s = dev_s = tell_s = spec_s = 0.0
    served0 = sampler.ahead_stats[0]
    spec0 = list(sampler.spec_stats)
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        out = one_trial()
        sync_s += sampler.last_ask_s[0]
        dev_s += sampler.last_ask_s[1]
        tell_s += sampler.last_tell_s
        spec_s += sampler.last_spec_s
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    barrier()
    e2e_wall = t1 - t0
    served = sampler.ahead_stats[0] - served0
    if world > 1:
        t = torch.tensor([e2e_wall], dtype=torch.float64, device=torch.device("cuda", local))
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_wall = float(t[0])
    e2e_value = world * e2e_steps / e2e_wall
    assert len(out) == N_PARAMS and all(0.0 <= v <= 1.0 for v in out)
    assert len(study.get_trials(deepcopy=False)) == N_TRIALS + 3 + max(2, min(args.warmup, 3)) + 2 * e2e_steps
    e2e_host = {"per_trial_ms": e2e_wall / e2e_steps * 1e3,
                "history_sync_ms": sync_s / e2e_steps * 1e3,       # in the ask: trial-log poll + row uploads (B200TPESampler._sync)
                # in the ask: waiting for the queued suggestion + read-back, then queueing the NEXT one (speculate_queue_ms)
                "wait_and_collect_ms": (dev_s - spec_s) / e2e_steps * 1e3,
                "speculate_queue_ms": spec_s / e2e_steps * 1e3,    # row upload (worst key) + prepare / build / uniforms / sample+select queued
                "tell_queue_ms": tell_s / e2e_steps * 1e3,         # in the tell: is the trial's outcome the assumed one? + its true row
                "optuna_ms": (e2e_wall - sync_s - dev_s - tell_s) / e2e_steps * 1e3,  # Study.ask / 32 x suggest_float / tell
                "look_ahead_served": served, "look_ahead_of": e2e_steps,
                "speculations_confirmed": sampler.spec_stats[0] - spec0[0],
                "speculations_abandoned": sampler.spec_stats[1] - spec0[1],
                "per_trial_ms_without_look_ahead": plain_wall / e2e_steps * 1e3,
                "first_ask_s": first_ask_s, "study_setup_s": study_setup_s}

    # ---- extras (rank 0, N=1 only): other shapes of the same path, not the headline ------------------
    extras = {}
    if rank == 0 and world == 1 and not args.no_extras:
        # cold suggestion: history upload (25.6 MB H2D) + everything else
        t0 = time.perf_counter()
        eng.set_history(X, cat, key)
        eng.suggest(cols, Unp[0], 1, **cfg)
        extras["cold_suggestion_ms"] = (time.perf_counter() - t0) * 1e3
        # univariate TPE (the reference default): the 32 sample_independent calls of a trial -- one by one, and
        # evaluated together as B200TPESampler does from the second trial on (tpe_suggest_univariate_batch)
        ucfg = dict(cfg, multivariate=False)
        ru = np.random.RandomState(5)
        for rep in range(2):
            # a new trial = a new history version (zero-row append): the split is shared by the 32 calls
            # of one trial, never across trials
            eng.append_history(np.zeros((0, N_PARAMS)), np.zeros(0, np.int8), np.zeros((0, 2)))
            t0 = time.perf_counter()
            for j in range(N_PARAMS):
                eng.suggest([j], ru.random_sample(N_CAND * 2), 1, **ucfg)
            uni = time.perf_counter() - t0
        extras["univariate_trial_one_by_one_ms"] = uni * 1e3
        for rep in range(4):
            # a trial has finished in between (one row more in the above set, as in a running study)
            eng.append_history(ru.uniform(0, 1, (1, N_PARAMS)), np.zeros(1, np.int8), np.array([[1e9, 0.0]]))
            uu = ru.random_sample(N_PARAMS * N_CAND * 2)
            t0 = time.perf_counter()
            eng.suggest_univariate_batch(cols, uu, **ucfg)
            unib = time.perf_counter() - t0
        extras["univariate_trial_ms"] = unib * 1e3
        extras["univariate_suggestions_per_s"] = 1.0 / unib
        extras["univariate_device_ms"] = float(eng.last_timing()[0][8])
        # config 2 with the DEFAULT n_ei_candidates = 24 through optuna's Study (what most studies run)
        try:
            dsampler = B200TPESampler(seed=12, n_ei_candidates=24, multivariate=True, device=local)
            study.sampler = dsampler
            for rep in range(4):
                one_trial()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            n_def = 40
            for rep in range(n_def):
                one_trial()
            torch.cuda.synchronize()
            de = (time.perf_counter() - t0) / n_def
            extras["default_candidates_e2e"] = {"n_ei_candidates": 24, "trial_ms": de * 1e3, "suggestions_per_s": 1.0 / de,
                                                "trials": n_def, "look_ahead": list(dsampler.ahead_stats),
                                                "speculations": list(dsampler.spec_stats)}
            study.sampler = sampler
            dsampler.close()
        except Exception as e:
            extras["default_candidates_e2e"] = {"error": repr(e)}
        # the same through optuna's Study: the reference's default sampler mode (multivariate=False), 32
        # sample_independent calls per trial answered from one batched device call (B200TPESampler._plan_trial)
        try:
            usampler = B200TPESampler(seed=11, n_ei_candidates=N_CAND, multivariate=False, device=local)
            study.sampler = usampler
            for rep in range(3):
                one_trial()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            n_uni = 20
            for rep in range(n_uni):
                one_trial()
            torch.cuda.synchronize()
            ue = (time.perf_counter() - t0) / n_uni
            extras["univariate_e2e"] = {"trial_ms": ue * 1e3, "trials_per_s": 1.0 / ue, "trials": n_uni,
                                        "look_ahead": list(usampler.ahead_stats),
                                        "path": "optuna Study.ask -> 32 x trial.suggest_float -> sample_independent "
                                                "(the first call of a trial collects the batch queued when the last "
                                                "trial was told: tpe_collect_univariate) -> study.tell [after_trial -> "
                                                "tpe_history_update / tpe_suggest_univariate_batch_async]"}
            study.sampler = sampler
            usampler.close()
        except Exception as e:
            extras["univariate_e2e"] = {"error": repr(e)}
        # config 4: MOTPE, 20 000 trials x 8 floats, 4 objectives, C = 24 -- with the default gamma (25 below trials)
        # and with gamma = ceil(0.1 n) (2000 below trials: rank peeling + HSSP over a 150-point tie rank + hypervolume
        # weights over the below set's Pareto front), next to the reference's own split + weights on the same values
        try:
            n4, p4 = 20_000, 8
            r4 = np.random.RandomState(4)
            X4 = r4.uniform(0, 1, (n4, p4))
            v4 = ((X4[:, None, :] - np.array([0.2, 0.4, 0.6, 0.8])[None, :, None]) ** 2).sum(2)
            e4 = TPEEngine(local)
            e4.set_space([ParamSpec(kind=0, low=0.0, high=1.0) for _ in range(p4)])
            e4.set_history(X4, np.zeros(n4, np.int8), np.zeros((n4, 2)))
            e4.set_values(v4, 0)
            mo = {}
            for tag, nb in (("default_gamma", 25), ("gamma_10pct", int(math.ceil(0.1 * n4)))):
                u4 = np.random.RandomState(7).random_sample(24 * (1 + p4))
                for rep in range(3):
                    t0 = time.perf_counter()
                    e4.suggest(list(range(p4)), u4, 1, n_below=nb, n_candidates=24, multivariate=True)
                    dt = time.perf_counter() - t0
                mo[tag] = {"n_below": nb, "suggestion_ms": dt * 1e3}
            e4.close()
            from optuna.samplers._tpe import sampler as ref_tpe
            from optuna.study._multi_objective import _fast_non_domination_rank

            class _S:  # what _calculate_weights_below_for_multi_objective reads from a study / a trial
                directions = [optuna.study.StudyDirection.MINIMIZE] * 4

            class _T:
                def __init__(self, v):
                    self.values = list(v)
            for tag in mo:
                nb = mo[tag]["n_below"]
                t0 = time.perf_counter()
                ranks = _fast_non_domination_rank(v4, n_below=nb)
                uq, cnts = np.unique(ranks, return_counts=True)
                last = int(np.max(uq[np.cumsum(cnts) <= nb], initial=-1))
                idx = np.arange(n4)
                bel = idx[ranks <= last]
                tie = ranks == last + 1
                if bel.size < nb:
                    sel = ref_tpe._solve_hssp_with_cache(tuple(v4[tie].ravel()), tuple(idx[tie]), nb - bel.size,
                                                         tuple(ref_tpe._get_reference_point(v4[tie])))
                    bel = np.sort(np.append(bel, sel))
                ref_tpe._calculate_weights_below_for_multi_objective(_S(), [_T(v) for v in v4[bel]], None)
                mo[tag]["reference_split_and_weights_ms"] = (time.perf_counter() - t0) * 1e3
            extras["motpe_c4"] = mo
        except Exception as e:  # an extra must never take the headline down
            extras["motpe_c4"] = {"error": repr(e)}
        # config 3: 64 mixed parameters (24 float, 8 log-float, 8 step-float, 8 int, 4 log-int, 12 categorical),
        # N = 50 000, multivariate -- with the default n_ei_candidates and with 4096 candidates (k_logpdf_mixed)
        try:
            n3 = 50_000
            r3 = np.random.RandomState(0)
            specs3, cols3 = [], []
            for _ in range(24):
                specs3.append(ParamSpec(kind=0, low=0.0, high=1.0)); cols3.append(r3.uniform(0, 1, n3))
            for _ in range(8):
                specs3.append(ParamSpec(kind=0, low=1e-5, high=1.0, log=True)); cols3.append(np.exp(r3.uniform(np.log(1e-5), 0, n3)))
            for _ in range(8):
                specs3.append(ParamSpec(kind=0, low=0.0, high=10.0, step=0.5)); cols3.append(r3.randint(0, 21, n3) * 0.5)
            for _ in range(8):
                specs3.append(ParamSpec(kind=1, low=0, high=100, step=1)); cols3.append(r3.randint(0, 101, n3).astype(float))
            for _ in range(4):
                specs3.append(ParamSpec(kind=1, low=1, high=1024, step=1, log=True))
                cols3.append(np.round(np.exp(r3.uniform(0, np.log(1024), n3))))
            for k in range(12):
                specs3.append(ParamSpec(kind=2, n_choices=4 + k % 5)); cols3.append(r3.randint(0, 4 + k % 5, n3).astype(float))
            e3 = TPEEngine(local)
            e3.set_space(specs3)
            e3.set_history(np.stack(cols3, 1), np.zeros(n3, np.int8), np.stack([r3.normal(size=n3), np.zeros(n3)], 1))
            c3 = {"n_trials": n3, "n_params": 64}
            for C3 in (24, 4096):
                for rep in range(3):
                    u3 = r3.random_sample(C3 * (1 + 64))
                    t0 = time.perf_counter()
                    e3.suggest(list(range(64)), u3, 1, n_below=25, n_candidates=C3, multivariate=True)
                    dt = time.perf_counter() - t0
                c3[f"c{C3}"] = {"suggestion_ms": dt * 1e3, "device_ms": float(e3.last_timing()[0][8]),
                                "kernel": e3.last_logpdf_kernel()}
            e3.close()
            extras["config3"] = c3
        except Exception as e:
            extras["config3"] = {"error": repr(e)}
        # config-5 shape: 8192 concurrent asks with the default n_ei_candidates = 24, one device call
        bcfg = dict(cfg, n_candidates=24)
        n_asks = 8192
        ub = np.random.RandomState(6).random_sample(n_asks * 24 * (1 + N_PARAMS))
        for rep in range(2):
            t0 = time.perf_counter()
            eng.suggest(cols, ub, n_asks, **bcfg)
            bt = time.perf_counter() - t0
        extras["batched_asks"] = {"n_asks": n_asks, "n_ei_candidates": 24, "ms": bt * 1e3,
                                  "suggestions_per_s": n_asks / bt,
                                  "note": "tpe_suggest with 52 MB of host-drawn uniforms uploaded inside the call"}
        # the same batch end to end through the plugin: uniforms generated on the device (MT19937 stream
        # of the sampler's RandomState), results converted to parameter dicts
        bs = B200TPESampler(seed=3, n_ei_candidates=24, multivariate=True, device=local)
        study.sampler = bs              # the same optuna study, asked through a fresh sampler
        for rep in range(2):
            t0 = time.perf_counter()
            res = bs.sample_relative_batch(study, space, n_asks)
            be = time.perf_counter() - t0
        assert len(res) == n_asks and len(res[0]) == N_PARAMS
        extras["batched_asks_e2e"] = {"n_asks": n_asks, "n_ei_candidates": 24, "ms": be * 1e3,
                                      "suggestions_per_s": n_asks / be,
                                      "path": "B200TPESampler.sample_relative_batch (device MT19937)"}
        bs.close()
        study.sampler = sampler
    # ---- config 5: 8192 concurrent asks (default n_ei_candidates = 24) sharded over the ranks -----------
    # every rank evaluates its block of asks on uniforms its GPU generates from the shared generator state
    # (MT19937 stream of one sampler consumed sequentially, the reference's semantics); results all-gathered
    config5 = None
    if not args.no_extras:
        from optuna_b200.dist import shard_asks, sharded_asks_device_rng
        n_asks5, c5 = 8192, 24
        per_ask5 = c5 * (1 + N_PARAMS)
        cfg5 = dict(cfg, n_candidates=c5)
        for rep in range(2):
            rng5 = np.random.RandomState(6)
            barrier()
            t0 = time.perf_counter()
            eng.prepare(cols, **cfg5)
            eng.build()
            if world > 1:
                tm5 = {}
                res5 = sharded_asks_device_rng(eng, rng5, n_asks5, per_ask5, gather=True, timing=tm5)
            else:
                eng.stage_rng(rng5, n_asks5 * per_ask5)
                res5, _, _ = eng.sample_and_select(None, n_asks5)
                eng.finish_rng(rng5)
            torch.cuda.synchronize()
            barrier()
            dt5 = time.perf_counter() - t0
        assert res5.shape == (n_asks5, N_PARAMS)
        if world > 1:
            t = torch.tensor([dt5], dtype=torch.float64, device=torch.device("cuda", local))
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt5 = float(t[0])
        config5 = {"n_asks": n_asks5, "n_ei_candidates": c5, "ms": dt5 * 1e3, "suggestions_per_s": n_asks5 / dt5,
                   "asks_per_rank": shard_asks(n_asks5, world, 0)[1], "scaling": "strong",
                   "path": "per rank: tpe_prepare / tpe_build / tpe_stage_uniforms_mt19937(skip: jump-ahead) / "
                           "tpe_sample_and_select(out_x = NULL); then ncclBroadcast of the generator end state and "
                           "ncclAllGather of the [8192, 32] results straight from the contexts' device buffers"}
        if world > 1:
            config5["rank0_compute_ms"] = tm5["compute_s"] * 1e3
            config5["rank0_collectives_ms"] = tm5["collectives_s"] * 1e3
    # ---- one suggestion over all GPUs: every rank evaluates g(x) over its slice of the above kernels, the
    # per-candidate (max, sum) partials are all-gathered (16 B per candidate and rank), every rank finishes ----
    kshard = None
    if world > 1 and not args.no_extras:
        from optuna_b200.dist import kernel_sharded_suggest
        ks_steps = 20
        uks = np.random.RandomState(77).random_sample((ks_steps + 3, per_ask))   # the same uniforms on every rank
        eng.set_kernel_shard(rank, world)
        for i in range(3):
            kernel_sharded_suggest(eng, cols, uks[i], 1, **cfg)
        barrier()
        t0 = time.perf_counter()
        for i in range(3, 3 + ks_steps):
            xk, _, _ = kernel_sharded_suggest(eng, cols, uks[i], 1, **cfg)
        torch.cuda.synchronize()
        barrier()
        dtk = (time.perf_counter() - t0) / ks_steps
        eng.set_kernel_shard(0, 1)
        xs, _, _ = eng.suggest(cols, uks[-1], 1, **cfg)
        t = torch.tensor([dtk, 0.0 if np.array_equal(xs, xk) else 1.0], dtype=torch.float64, device=torch.device("cuda", local))
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        kshard = {"ms_per_suggestion": float(t[0]) * 1e3, "suggestions_per_s": 1.0 / float(t[0]),
                  "equals_single_gpu_suggestion_on_every_rank": float(t[1]) == 0.0, "scaling": "strong",
                  "path": "per rank: tpe_prepare / tpe_build / tpe_sample_and_partial (g(x) over 1/N of the kernels) -> "
                          "ncclAllGather of the [N][4096] (max, sum) partials -> tpe_finish_from_partials"}
    if rank == 0:
        peak, peak_src = measured_peaks()
        k_ms = float(stage[5]) / args.steps  # main log-density kernel under g(x)
        ach = algorithmic_bytes() / (k_ms * 1e-3) / 1e9
        try:
            fp64_peak = eng.probe_fp64_tflops()
        except Exception:
            fp64_peak = None
        fl = algorithmic_flops()
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": wall / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": dict(CONFIG),
            "parallelism": f"{world} independent asks per step, history replicated by one NCCL broadcast",
            "device_ms_per_step": dev_ms / args.steps,
            "stage_ms": {k: float(v) / args.steps for k, v in zip(
                ["split", "build", "h2d", "sample", "logpdf_below", "logpdf_above_main", "logpdf_fixup", "select",
                 "span"], stage)},
            "gpu_launches": int(launches),
            "clocks": clk,
            # inputs of one ask: the generator state (624 words + position; the uniforms themselves are
            # produced on the device by the same MT19937), the column list and the config struct
            # inputs of one step: the row that changed, twice (with the assumed and with the true key: 32 params +
            # 2 key doubles + 1 category byte), the column list and the config struct; the
            # generator state travels only when somebody else drew from it
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 2 * (N_PARAMS * 8 + 16 + 1) + N_PARAMS * 4 + 32,
                    "d2h_bytes_per_step": N_PARAMS * 8 + 16 + 24 + 625 * 4, "steps": e2e_steps,
                    "path": "optuna.create_study(sampler=B200TPESampler) + study.add_trials(100k) ; per step study.ask() "
                            "[infer_relative_search_space, sample_relative -> ctypes -> tpe_collect, then "
                            "tpe_history_update (this trial's row, worst key) / tpe_prepare / tpe_build / "
                            "tpe_stage_uniforms_mt19937 / tpe_sample_and_select_async: the NEXT suggestion is queued "
                            "assuming the trial will not enter the below set] -> 32 x trial.suggest_float -> "
                            "study.tell [after_trial: assumption checked against the value, tpe_history_update (true "
                            "key); if it failed the suggestion is recomputed now]; every step is one full ask + tell, "
                            "nothing skipped",
                    "caller": f"optuna {optuna.__version__} ({os.path.relpath(os.path.dirname(optuna.__file__), ROOT)})",
                    "host": e2e_host},
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "traffic": 27560960, "traffic_source": "ncu --set full, profiles/r2_ncu_raw_logpdf_mma.txt "
                         "(dram__bytes_read.sum 27 523 328 + dram__bytes_write.sum 37 632 of this launch)",
                         "peak_source": peak_src, "kernel": kernel_name,
                         "kernel_ms": k_ms, "algorithmic_bytes": algorithmic_bytes(),
                         "note": "the C x K x P grid reuses every history byte C=4096 times from shared memory, so "
                                 "this kernel sits on the fp64 (DMMA) pipe, not on HBM (SURVEY.md section 8d); see fp64"},
            # algorithmic = the reference's operation count (SURVEY.md 8d: 4P + 25 flops per cell);
            # executed = what the tensor-core kernel issues after expanding the square: one fma per
            # cell on mma.m8n8k4.f64 (DMMA and DFMA share the 37 TFLOP/s fp64 peak on B200)
            "fp64": {"achieved_tflops": fl / (k_ms * 1e-3) / 1e12, "peak_tflops": fp64_peak,
                     "frac": (fl / (k_ms * 1e-3) / 1e12 / fp64_peak) if fp64_peak else None,
                     "algorithmic_flops": fl,
                     "executed_flops": executed_flops(),
                     "executed_tflops": executed_flops() / (k_ms * 1e-3) / 1e12,
                     "executed_frac": (executed_flops() / (k_ms * 1e-3) / 1e12 / fp64_peak) if fp64_peak else None,
                     "kernel": eng.last_logpdf_kernel(),
                     "peak_source": "tpe_probe_fp64_tflops (DFMA microbenchmark, this run; tools/probe_dmma.cu "
                                    "measures the same 37.1 TFLOP/s for DMMA.8x8x4)"},
        }
        if extras:
            line["extras"] = extras
        if config5:
            line["config5"] = config5
        if kshard:
            line["kernel_sharded"] = kshard
        if bcast_ms is not None:
            line["history_broadcast"] = {"ms": bcast_ms, "bytes": N_TRIALS * (N_PARAMS + 2) * 8 + N_TRIALS,
                                         "note": "one ncclBroadcast of the frozen history (X and keys as one fp64 buffer, "
                                                 "categories as int8), before the timed region"}
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_baseline_leg(optuna, study, space)
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extras", action="store_true", help="skip the univariate / batched / cold extras")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    ap.add_argument("--n-trials", type=int, default=N_TRIALS, help="development only: a shorter history (the line then "
                    "says so in config.n_trials); the benchmark is the default")
    args = ap.parse_args()
    if args.n_trials != N_TRIALS:
        globals()["N_TRIALS"] = args.n_trials
        CONFIG["n_trials"] = args.n_trials
        CONFIG["workload"] += f" [DEVELOPMENT RUN: n_trials={args.n_trials}]"
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
