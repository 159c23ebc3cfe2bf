"""B200TPESampler -- drop-in for optuna.samplers.TPESampler backed by libtpe_b200.so.

Mirrors the reference's plugin surface (optuna/samplers/_base.py:31-228) and constructor
(optuna/samplers/_tpe/sampler.py:305-385).  What stays on the host is exactly what the reference
can only do in Python: walking FrozenTrial objects once (incrementally) into arrays, evaluating the
user's callables (gamma, weights, constraints_func, categorical_distance_func), drawing the
uniforms from the sampler's own numpy RandomState in the reference's order
(probability_distributions.py:87,100,138-144) and converting the winner back with
``to_external_repr``.  Split, estimator build, candidate sampling, the log-density grid and the
argmax run on the GPU through the C ABI (include/optuna_b200_tpe.h).  There is no CPU fallback.
"""
from __future__ import annotations

import bisect
import json
import math
import threading
import time
from dataclasses import dataclass, field
from typing import Any, Callable, Sequence

import numpy as np

from . import _lib
from ._compat import (CONSTRAINTS_KEY, RELATIVE_PARAMS_KEY, SYSTEM_ATTR_MAX_LENGTH, _INDEPENDENT_SAMPLING_WARNING_TEMPLATE,
                      BaseDistribution, BaseSampler, CategoricalDistribution, FloatDistribution, InMemoryStorage,
                      IntDistribution, LazyRandomState, RandomSampler, StudyDirection, TrialState,
                      _process_constraints_after_trial, get_logger, optuna_warn, warn_experimental_argument)
from .engine import ParamSpec, TPEEngine

EPS = 1e-12
_logger = get_logger("optuna.samplers.optuna_b200")  # a child of optuna's root logger: same handlers / verbosity


def default_gamma(x: int) -> int:
    """sampler.py:53-54"""
    return min(math.ceil(0.1 * x), 25)


def hyperopt_default_gamma(x: int) -> int:
    """sampler.py:57-58"""
    return min(math.ceil(0.25 * x**0.5), 25)


def default_weights(x: int) -> np.ndarray:
    """sampler.py:61-69.  When this very function is the sampler's ``weights`` the library
    evaluates it on the device (k_weights); the host version serves custom compositions."""
    if x == 0:
        return np.asarray([])
    if x < 25:
        return np.ones(x)
    return np.concatenate([np.linspace(1.0 / x, 1.0, num=x - 25), np.ones(25)], axis=0)


def _checked_weights(func: Callable[[int], np.ndarray], n: int) -> np.ndarray:
    """parzen_estimator.py:88-109"""
    w = np.array(func(n))[:n]
    if np.any(w < 0):
        raise ValueError(f"The `weights` function is not allowed to return negative values {w}. "
                         f"The argument of the `weights` function is {n}.")
    if len(w) > 0 and np.sum(w) <= 0:
        raise ValueError(f"The `weight` function is not allowed to return all-zero values {w}."
                         f" The argument of the `weights` function is {n}.")
    if not np.all(np.isfinite(w)):
        raise ValueError("The `weights`function is not allowed to return infinite or NaN values "
                         f"{w}. The argument of the `weights` function is {n}.")
    return np.asarray(w, dtype=np.float64)


def _pruned_key(trial, sign: float) -> tuple[float, float]:
    """sampler.py:782-792"""
    if len(trial.intermediate_values) > 0:
        step, v = max(trial.intermediate_values.items())
        if math.isnan(v):
            return -step, float("inf")
        return -step, sign * v
    return 1, 0.0


def _infeasible_score(trial) -> float:
    """sampler.py:803-813"""
    con = trial.system_attrs.get(CONSTRAINTS_KEY)
    if con is None:
        optuna_warn(f"Trial {trial.number} does not have constraint values."
                    " It will be treated as a lower priority than other trials.")
        return float("inf")
    return sum(v for v in con if v > 0)


def _spec_of(name: str, d: BaseDistribution, dist_funcs: dict) -> ParamSpec:
    if isinstance(d, CategoricalDistribution):
        table = None
        if name in dist_funcs:
            f = dist_funcs[name]
            table = np.asarray([[f(a, b) for b in d.choices] for a in d.choices], dtype=np.float64)
        return ParamSpec(kind=_lib.KIND_CAT, n_choices=len(d.choices), dist_table=table)
    if isinstance(d, IntDistribution):
        return ParamSpec(kind=_lib.KIND_INT, low=float(d.low), high=float(d.high), step=float(d.step), log=bool(d.log))
    assert isinstance(d, FloatDistribution), d
    return ParamSpec(kind=_lib.KIND_FLOAT, low=d.low, high=d.high, step=d.step, log=bool(d.log))


class _Reset(Exception):
    """The study's trial list is not an extension of what the log has seen (another study behind the same ids)."""


class _History:
    """The study's trial list followed incrementally, and its mirror on the device.

    Replaces the per-call FrozenTrial walks of the reference -- ``study._get_trials(states=...)`` filters
    (study/study.py:269-287, O(N) each, three per ask in sampler.py:449-535), ``_get_internal_repr``
    (:511-521), ``_split_trials`` (:686-722), ``IntersectionSearchSpace._calculate``
    (search_space/intersection.py:14-55) and ``_GroupDecomposedSearchSpace.calculate``
    (search_space/group_decomposed.py:45-68) -- by O(#changes) work per ask (SURVEY.md section 8f rank 1).

    Row r of the log (and of the device history) is the r-th trial of the study's list, i.e. trial number r:
    COMPLETE / PRUNED trials carry their sort key, everything the sampler must not see (WAITING, FAIL, RUNNING
    without ``constant_liar``, the trial being sampled) is a TPE_CAT_EXCLUDED placeholder, so a trial that
    finishes later -- in any order -- is one in-place row update.

    Two ways to learn what changed since the last look:
      * ``InMemoryStorage`` (everything in this process): O(1) probes through the storage's public API --
        ``get_trial`` of the few unfinished trials (the storage replaces a FrozenTrial object whenever it changes:
        an unchanged object means an unchanged trial) and ``get_trial_id_from_study_id_trial_number`` for numbers
        not seen yet.  No O(N) list copy per ask.
      * any other storage: ``study._get_trials(deepcopy=False, use_cache=...)`` (all states -- the call is O(1) on
        the study's per-trial cache once the storage has answered) and the same scan of unfinished + new rows.
    """

    #: how many of the best sort keys are kept on the host (outcome speculation needs the n_below-th best)
    BEST_KEYS = 64

    def __init__(self) -> None:
        # ---- log (host only) ----
        self.storage = None            # strong reference: a recycled id() can never alias another storage
        self.token: tuple | None = None
        self.rows = 0
        self.numbers: list[int] = []
        self.pending: dict[int, list] = {}     # row -> [trial_id, FrozenTrial object at the last look]
        self.n_finished = 0                    # COMPLETE + PRUNED trials (sampler.py:449-456, :538)
        self.n_complete = 0                    # COMPLETE trials of a single-objective study ...
        self.best_keys: list[float] = []       # ... and the BEST_KEYS smallest of their sort keys, ascending
        self.all_dists: dict[str, BaseDistribution] = {}   # latest distribution of every parameter seen
        self.seen_params: set[str] = set()
        self.inter: dict[str, BaseDistribution] | None = None
        self.groups: list[dict[str, BaseDistribution]] = []
        self.group_backlog: list[tuple[int, dict]] = []
        self.last_list: list | None = None     # trial list of the last generic poll (valid during one sync)
        # ---- device mirror ----
        self.columns: dict[str, int] = {}
        self.dists: list[BaseDistribution] = []
        self.dev_token: tuple | None = None
        self.dev_rows = 0
        self.dev_cat: dict[int, int] = {}      # category uploaded for the rows still pending
        self.backlog: dict[int, Any] = {}      # row -> FrozenTrial: changes the log has seen, the device has not
        self.dev_pred: dict[int, Any] = {}     # row -> _Told: uploaded at `tell` time, before the storage showed it
        self.dev_version = 0                   # counts the uploads that change what the estimators see

    # -- log ---------------------------------------------------------------------------------------------
    def _account(self, t) -> None:
        """A trial seen finished for the first time."""
        if t.state != TrialState.COMPLETE and t.state != TrialState.PRUNED:
            return  # FAIL: in no estimator, in no search space
        self.n_finished += 1
        if t.state == TrialState.COMPLETE and len(self.token[1]) == 1 and t.values is not None:
            key = -t.values[0] if self.token[1][0] == StudyDirection.MAXIMIZE else t.values[0]
            self.n_complete += 1
            if len(self.best_keys) < self.BEST_KEYS or key < self.best_keys[-1]:
                bisect.insort(self.best_keys, key)
                del self.best_keys[self.BEST_KEYS:]
        d = t.distributions
        self.all_dists.update(d)
        self.seen_params.update(t.params)
        if self.inter is None:
            self.inter = dict(d)
        elif self.inter:
            inter = self.inter
            if not (len(d) == len(inter) and all(d.get(k) is v for k, v in inter.items())):
                self.inter = {k: v for k, v in inter.items() if d.get(k) == v}
        self.group_backlog.append((t.number, d))

    def poll(self, study, use_cache: bool) -> list[tuple[int, Any]]:
        """(row, FrozenTrial) of every row that is new or whose trial changed since the last poll, ascending."""
        st, sid = study._storage, study._study_id
        token = (sid, tuple(study.directions))
        if self.storage is not st or self.token != token:
            self.__init__()
            self.storage, self.token = st, token
        changed: list[tuple[int, Any]] = []
        fast = type(st) is InMemoryStorage and self.rows > 0
        trials = None
        if not fast:
            trials = study._get_trials(deepcopy=False, use_cache=use_cache)
            if len(trials) < self.rows or (self.rows and trials[self.rows - 1].number != self.numbers[-1]):
                raise _Reset()
        self.last_list = trials
        for row, slot in list(self.pending.items()):
            t = st.get_trial(slot[0]) if fast else trials[row]
            if t is slot[1]:
                continue
            if t.number != self.numbers[row]:
                raise _Reset()
            changed.append((row, t))
            if t.state.is_finished():
                del self.pending[row]
                self._account(t)
            else:
                slot[1] = t
        while True:
            row = self.rows
            if fast:
                try:
                    tid = st.get_trial_id_from_study_id_trial_number(sid, row)
                except KeyError:
                    break
                t = st.get_trial(tid)
            else:
                if row >= len(trials):
                    break
                t = trials[row]
                tid = t._trial_id
            self.rows += 1
            self.numbers.append(t.number)
            changed.append((row, t))
            if t.state.is_finished():
                self._account(t)
            else:
                self.pending[row] = [tid, t]
        return changed

    def all_trials(self, study, use_cache: bool) -> list:
        """Every trial the log has seen, as a list (device rebuilds only: O(N))."""
        trials = self.last_list
        if trials is None:  # fast polls keep no list; a fresh one (a cached one may be older than the log)
            trials = study._get_trials(deepcopy=False, use_cache=False)
        return trials[: self.rows]

    def intersection(self) -> dict[str, BaseDistribution]:
        return dict(sorted((self.inter or {}).items(), key=lambda kv: kv[0]))

    def group_spaces(self) -> list[dict[str, BaseDistribution]]:
        """_GroupDecomposedSearchSpace.calculate (group_decomposed.py:45-68).  The reference re-adds the
        distributions of every finished trial, in trial order, at each call; adding a trial twice changes nothing
        (its parameters already are a union of groups), so adding the trials that finished since the last call,
        in trial order, gives the same list of groups in the same order."""
        backlog, self.group_backlog = sorted(self.group_backlog, key=lambda e: e[0]), []
        for _, dist in backlog:
            left = set(dist)
            nxt: list[dict[str, BaseDistribution]] = []
            for sub in self.groups:
                keys = set(sub)
                nxt.append({name: sub[name] for name in keys & left})
                nxt.append({name: sub[name] for name in keys - left})
                left -= keys
            nxt.append({name: dist[name] for name in left})
            self.groups = [g for g in nxt if g]
        return [dict(g) for g in self.groups]


class _DeviceSyncedRng:
    """The sampler's ``LazyRandomState`` whose MT19937 state may temporarily be newer on the device.

    Large asks draw their uniforms on the GPU; instead of copying the generator state back into the host
    ``RandomState`` after every ask (get_state + set_state cost 80 us), the state stays on the device
    and the next ask continues from it.  Any access to ``.rng`` -- an ask drawn on the host, reseeding,
    pickling, somebody reading ``sampler._rng.rng`` -- first brings the host generator up to date.

    Work queued ahead of its ask `stage`s its draws without taking them: an undo armed with `arm` puts the generator
    back to the snapshot taken before them (or, for a plan served in part, where the calls served so far left it).
    Every staged draw is either adopted (`release(.., adopted=True)`) or undone -- by `release`, or by the next look
    at ``.rng``, whichever comes first."""

    def __init__(self, inner) -> None:
        self._inner = inner
        self._engine = None  # the engine holding a newer state, if any (never while an undo is pending)
        self._settle = None  # the pending undo: called before anyone looks

    @property
    def rng(self) -> np.random.RandomState:
        settle, self._settle = self._settle, None
        if settle is not None:
            settle()
        eng, self._engine = self._engine, None
        if eng is not None:
            eng.finish_rng(self._inner.rng)
        return self._inner.rng

    def on_device(self, eng) -> bool:
        return self._engine is not None and self._engine is eng

    def mark_device(self, eng) -> None:
        self._engine = eng

    def draw(self, eng, count: int, device: bool) -> np.ndarray | None:
        """The next `count` uniforms for `eng`, taken at once: generated on the device (returns None), continuing
        from the state `eng` holds if it holds one, or drawn on the host."""
        if not device:
            return self.rng.random_sample(count)
        eng.stage_rng(None if self._engine is eng else self.rng, count)
        self._engine = eng                            # from here on the device holds the newer state
        return None

    def stage(self, eng, count: int, device: bool) -> tuple[Any, np.ndarray | None]:
        """Snapshot the generator and stage its next `count` uniforms for `eng` without taking them: generated on the
        device, continuing from the state `eng` holds if it holds one, or drawn on the host (returned, else None).
        Returns (snapshot, host draws).  Until the draws are adopted the generator stands at the snapshot: a caller
        whose work fails `restore`s it, one whose work is queued `arm`s the undo."""
        if not device:
            r = self.rng                              # (a pending undo runs first)
            snap = r.get_state()
            return snap, r.random_sample(count)
        if self._engine is eng:
            snap = eng.rng_snapshot()                 # where the last ask left the generator (no device access)
            eng.stage_rng(None, count)
            self._engine = None
        else:
            r = self.rng
            snap = r.get_state()
            eng.stage_rng(r, count, state=snap)       # (the host object stays at the snapshot)
        return snap, None

    def restore(self, snap, advance: int = 0) -> None:
        """Put the generator at `snap`, `advance` draws on."""
        r = self._inner.rng
        r.set_state(snap)
        if advance:
            r.random_sample(advance)
        self._engine = None

    def arm(self, undo: Callable[[], None]) -> Callable[[], None]:
        """Make `undo` the pending undo of the draws just staged; returns it."""
        self._settle = undo
        return undo

    def armed(self, undo) -> bool:
        """Is `undo` still pending (nobody has looked at the generator since it was armed)?"""
        return self._settle is undo

    def release(self, undo, adopted: bool) -> None:
        """The draws `undo` belongs to are adopted (the generator stays where they left it) or undone.  Nothing
        happens when `undo` is no longer pending."""
        if self._settle is undo:
            self._settle = None
            if not adopted:
                undo()

    def __getstate__(self) -> dict:
        self.rng  # flush
        return {"_inner": self._inner, "_engine": None, "_settle": None}

    def __setstate__(self, state: dict) -> None:
        self.__dict__.update(state)


class _Told:
    """A trial as it will look once ``Study.tell`` has stored it: ``after_trial`` (samplers/_base.py:178-203) is
    handed the trial, its final state and values just BEFORE the storage records them (study/_tell.py:163-169).
    Quacks like the FrozenTrial ``_rows`` reads."""

    def __init__(self, trial, state, values) -> None:
        self.number = trial.number
        self.state = state
        self.values = None if values is None else [float(v) for v in values]
        self.value = self.values[0] if self.values is not None and len(self.values) == 1 else None
        self.params = dict(trial.params)
        self.distributions = dict(trial.distributions)
        self.intermediate_values = dict(trial.intermediate_values)
        self.system_attrs = dict(trial.system_attrs)
        self.confirmed = False
        self.threshold = None   # an outcome speculated by `_speculate`: the sort key the trial's value must not beat

    def matches(self, t) -> bool:
        """Is the stored trial exactly what was uploaded for it?"""
        return (t.state == self.state and t.values == self.values and t.params == self.params
                and t.distributions == self.distributions and t.intermediate_values == self.intermediate_values
                and t.system_attrs.get(CONSTRAINTS_KEY) == self.system_attrs.get(CONSTRAINTS_KEY))


@dataclass(eq=False)
class _Ahead:
    """A suggestion whose device work was queued before its ask (``B200TPESampler._look_ahead``, ``_speculate``)."""

    kind: str              # "joint": one sample_relative; "spec": the same, queued before the running trial ended;
                           # "uni": the per-parameter calls of a trial
    told: _Told            # the trial whose row was uploaded for it
    space: dict
    cols: list
    cfg: dict
    cfg_n_finished: int    # the count of finished trials `cfg` was made for ("spec" checks it at `tell` time)
    dev_version: int
    eng: Any
    dev_rng: bool          # its uniforms were generated on the device
    snap: Any              # the generator before its draws
    cancel: Callable       # the undo armed on the generator for them
    order: list = field(default_factory=list)  # "uni": the predicted calls, the user's weights of the two sets
    wb: Any = None
    wa: Any = None


class _UniPlan:
    """Univariate TPE asks every parameter of a trial separately (sampler.py:458-491), one `_sample` each; the P
    calls of a trial see the same history and differ only in the column and in the stretch of the generator they
    consume.  The plan evaluates all of them at the FIRST call -- in the order the previous trial asked, with the
    stretches of the stream in that order -- and the following calls are answered from it as long as they arrive
    exactly as predicted (same name, same distribution, same history, generator untouched).  Anything else settles
    the generator where the calls served so far would have left it and goes back to one call at a time."""

    def __init__(self) -> None:
        self.trial = None          # trial number the plan was made for
        self.order: list = []      # [(name, distribution)] predicted call sequence
        self.values: list = []     # external representation per call
        self.next = 0
        self.version = None        # history version the plan was computed on
        self.calls_trial = None    # recording of the running trial's actual calls (the next trial's prediction)
        self.calls: list = []
        self.prev: list = []       # calls of the last completed recording
        self.disabled = False      # the engine said "not batchable" for this space
        self.on_device = None      # the engine whose generator state is the one after the whole batch
        self.settle = None         # the undo armed on the generator until the whole batch is served


class B200TPESampler(BaseSampler):
    """``optuna.samplers.TPESampler`` (sampler.py:72-385) with the numeric path on a B200.  Same constructor
    arguments (+ ``device``), same plugin methods, same suggestions for the same seed.

    Where the reference's call order allows it the device work of an ask is queued BEFORE the ask (DESIGN.md
    section 1b): at `tell` time (``after_trial`` knows the finished trial before the storage does) and, for joint
    sampling, already when the previous suggestion has been handed out, on the assumption -- checked at `tell` time --
    that the running trial will not enter the below set.  An ask that is not the predicted one puts the generator
    back and computes as the reference does; ``LOOK_AHEAD`` / ``SPECULATE`` switch both off."""

    #: what answers the array-level calls -- the CUDA library; no fallback.  (The seam mirrors the reference's
    #: ``_parzen_estimator_cls``, sampler.py:358-359; tests plug the CPU oracle in here to check the host glue.)
    _engine_cls = TPEEngine
    #: test hook: called as _audit(trial, search_space, engine) after every device suggestion (the candidates and
    #: both log-densities of the ask are still on the engine: engine.get_candidates())
    _audit = None

    def __init__(
        self,
        *,
        consider_prior: bool = True,
        prior_weight: float = 1.0,
        consider_magic_clip: bool = True,
        consider_endpoints: bool = False,
        n_startup_trials: int = 10,
        n_ei_candidates: int = 24,
        gamma: Callable[[int], int] = default_gamma,
        weights: Callable[[int], np.ndarray] = default_weights,
        seed: int | None = None,
        multivariate: bool = False,
        group: bool = False,
        warn_independent_sampling: bool = True,
        constant_liar: bool = False,
        constraints_func: Callable[[Any], Sequence[float]] | None = None,
        categorical_distance_func: dict[str, Callable[[Any, Any], float]] | None = None,
        device: int = 0,
    ) -> None:
        if not consider_prior:
            optuna_warn("`consider_prior` has been deprecated in v4.3.0 and automatically falls back to `True`.",
                        FutureWarning)
        self._prior_weight = prior_weight
        self._magic_clip = consider_magic_clip
        self._endpoints = consider_endpoints
        self._n_startup_trials = n_startup_trials
        self._n_ei_candidates = n_ei_candidates
        self._gamma = gamma
        self._weights = weights
        self._multivariate = multivariate
        self._group = group
        self._warn_independent_sampling = warn_independent_sampling
        self._constant_liar = constant_liar
        self._constraints_func = constraints_func
        self._cat_dist_funcs = categorical_distance_func or {}
        self._rng = _DeviceSyncedRng(LazyRandomState(seed))
        self._random_sampler = RandomSampler(seed=seed)  # startup trials (sampler.py:348-349, :471-474)
        self._device = device
        self._engine: TPEEngine | None = None
        self._hist = _History()
        self._groups_now: list[dict[str, BaseDistribution]] = []
        self._lock = threading.RLock()
        self._uni = _UniPlan()
        self._ahead: _Ahead | None = None
        self._last_space: dict[str, BaseDistribution] | None = None
        self.ahead_stats = [0, 0]   # look-ahead suggestions [served, discarded]
        self.spec_stats = [0, 0]    # outcome speculations [confirmed at tell time, abandoned]
        self.last_spec_s = 0.0
        self.last_tell_s = 0.0
        if multivariate:
            warn_experimental_argument("multivariate")
        if group:
            if not multivariate:
                raise ValueError("``group`` option can only be enabled when ``multivariate`` is enabled.")
            warn_experimental_argument("group")
        if constant_liar:
            warn_experimental_argument("constant_liar")
        if constraints_func is not None:
            warn_experimental_argument("constraints_func")
        if categorical_distance_func is not None:
            warn_experimental_argument("categorical_distance_func")

    # -- pickling: device state is a cache re-creatable from the study (SURVEY.md section 5) ----------
    def __getstate__(self) -> dict:
        state = self.__dict__.copy()
        state["_engine"] = None
        state["_hist"] = _History()
        state["_groups_now"] = []
        state["_uni"] = _UniPlan()
        state["_ahead"] = None
        state["_last_space"] = None
        del state["_lock"]
        return state

    def __setstate__(self, state: dict) -> None:
        self.__dict__.update(state)
        self._lock = threading.RLock()

    def close(self) -> None:
        """Release the device context (re-created on demand)."""
        if getattr(self, "_ahead", None) is not None:
            self._drop_ahead()
        eng, self._engine = getattr(self, "_engine", None), None
        if eng is not None:
            rng = getattr(self, "_rng", None)
            if rng is not None:
                rng.rng  # bring the host generator up to date before the device state goes away
            eng.close()
        h = getattr(self, "_hist", None)
        if h is not None:
            h.dev_token, h.dev_rows, h.dev_cat = None, 0, {}

    def __del__(self) -> None:  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def hyperopt_parameters() -> dict[str, Any]:
        return {"consider_prior": True, "prior_weight": 1.0, "consider_magic_clip": True,
                "consider_endpoints": False, "n_startup_trials": 20, "n_ei_candidates": 24,
                "gamma": hyperopt_default_gamma, "weights": default_weights}

    def reseed_rng(self) -> None:
        self._rng.rng.seed()
        self._random_sampler.reseed_rng()

    # -- plugin surface -------------------------------------------------------------------------------
    def _poll(self, study) -> list[tuple[int, Any]]:
        """Bring the log up to date.  ``use_cache`` as the reference passes it (sampler.py:392, :528)."""
        h = self._hist
        use_cache = self._multivariate or not self._constant_liar
        try:
            return h.poll(study, use_cache)
        except _Reset:
            h.storage = None  # forget everything and read the list afresh
            return h.poll(study, use_cache)

    def infer_relative_search_space(self, study, trial) -> dict[str, BaseDistribution]:
        if not self._multivariate:
            return {}
        with self._lock:
            self._note_changes(self._poll(study))
            if self._group:
                self._groups_now = self._hist.group_spaces()
                out: dict[str, BaseDistribution] = {}
                for sub in self._groups_now:
                    for name, d in sorted(sub.items()):  # sorted: the reference's order (sampler.py:400-404)
                        if not d.single():
                            out[name] = d
                return out
            space = self._hist.intersection()
        return {k: d for k, d in space.items() if not d.single()}

    def sample_relative(self, study, trial, search_space: dict[str, BaseDistribution]) -> dict[str, Any]:
        if self._group:
            # one joint suggestion per group of parameters that always appear together (sampler.py:417-431);
            # the search space may be smaller than what was inferred (PartialFixedSampler, _partial_fixed.py:65-84)
            with self._lock:
                groups = [dict(g) for g in self._groups_now]
            params: dict[str, Any] = {}
            for sub in groups:
                part = {name: d for name, d in sorted(sub.items()) if not d.single() and name in search_space}
                params.update(self._sample_relative(study, trial, part))
        else:
            params = self._sample_relative(study, trial, search_space)
        if params != {} and self._constant_liar:
            # share the relative parameters with the other workers (sampler.py:435-443)
            text = json.dumps(params)
            for i in range(0, len(text), SYSTEM_ATTR_MAX_LENGTH):
                study._storage.set_trial_system_attr(trial._trial_id,
                                                     f"{RELATIVE_PARAMS_KEY}:{i // SYSTEM_ATTR_MAX_LENGTH}",
                                                     text[i: i + SYSTEM_ATTR_MAX_LENGTH])
        return params

    def _sample_relative(self, study, trial, search_space) -> dict[str, Any]:
        if search_space == {}:
            return {}
        with self._lock:
            self._note_changes(self._poll(study))
            if self._hist.n_finished < self._n_startup_trials:
                return {}
            return self._sample(study, trial, search_space, speculate=not self._group)

    def sample_independent(self, study, trial, param_name: str, param_distribution: BaseDistribution) -> Any:
        with self._lock:
            self._note_changes(self._poll(study))
            startup = self._hist.n_finished < self._n_startup_trials
            seen = param_name in self._hist.seen_params
        if startup:
            return self._random_sampler.sample_independent(study, trial, param_name, param_distribution)
        if self._warn_independent_sampling and self._multivariate and seen:
            # not at the first sampling of `param_name` (sampler.py:476-489)
            _logger.warning(_INDEPENDENT_SAMPLING_WARNING_TEMPLATE.format(
                param_name=param_name, trial_number=trial.number,
                independent_sampler_name=self._random_sampler.__class__.__name__,
                sampler_name=self.__class__.__name__,
                fallback_reason="dynamic search space is not supported for `multivariate=True`"))
        with self._lock:
            return self._sample_one(study, trial, param_name, param_distribution)

    def before_trial(self, study, trial) -> None:
        self._random_sampler.before_trial(study, trial)

    def after_trial(self, study, trial, state, values) -> None:
        """sampler.py:666-676: constraints are evaluated once, here, and stored with the trial."""
        assert state in (TrialState.COMPLETE, TrialState.FAIL, TrialState.PRUNED)
        if self._constraints_func is not None:
            _process_constraints_after_trial(self._constraints_func, study, trial, state)
        self._random_sampler.after_trial(study, trial, state, values)
        if self.LOOK_AHEAD and self._engine is not None:
            t0 = time.perf_counter()
            with self._lock:
                try:
                    if self._multivariate:
                        if self._last_space is not None:
                            self._look_ahead(study, trial, state, values)
                    else:
                        self._look_ahead_uni(study, trial, state, values)
                except Exception as e:               # computing ahead is an optimisation: it must never break a `tell`
                    _logger.debug(f"look-ahead abandoned: {e!r}")
                    self._abandon_ahead()
            self.last_tell_s = time.perf_counter() - t0   # row upload + queueing the next suggestion

    # -- host glue -------------------------------------------------------------------------------------
    def _eng(self) -> TPEEngine:
        if self._engine is None:
            self._engine = self._engine_cls(self._device)
        return self._engine

    def _get_params(self, trial) -> dict[str, Any]:
        """sampler.py:493-509"""
        if trial.state.is_finished() or not self._multivariate:
            return trial.params
        chunks = []
        i = 0
        while (c := trial.system_attrs.get(f"{RELATIVE_PARAMS_KEY}:{i}")):
            chunks.append(c)
            i += 1
        if not chunks:
            return trial.params
        params = json.loads("".join(chunks))
        params.update(trial.params)
        return params

    def sample_relative_batch(self, study, search_space: dict[str, BaseDistribution], n_asks: int) -> list[dict]:
        """`n_asks` joint suggestions against the current (frozen) history in ONE device call.

        Equivalent to calling ``sample_relative`` n_asks times without a ``tell`` in between
        (SURVEY.md section 3.3: the reference idiom is a Python loop of ``study.ask()``; with
        ``constant_liar=False`` every such ask sees the same split and the same two mixtures and
        only the RNG position differs).  The uniforms are drawn ask by ask from the sampler's own
        RandomState, so the results are those of the sequential loop."""
        if self._group or self._constant_liar:
            raise ValueError("sample_relative_batch needs group=False and constant_liar=False "
                             "(constant-liar asks depend on each other)")
        if search_space == {} or n_asks <= 0:
            return [{} for _ in range(max(n_asks, 0))]
        with self._lock:
            self._drop_ahead()
            self._note_changes(self._poll(study))
            if self._hist.n_finished < self._n_startup_trials:
                return [{} for _ in range(n_asks)]
            cols = self._sync(study, None, search_space)
            cfg = self._cfg(self._hist.n_finished)
            eng = self._eng()
            wb, wa = self._prepare(eng, cols, cfg, study)
            eng.build(wb, wa)
            # ask-by-ask draws are consecutive stretches of one stream: one generation yields the same numbers
            x = self._sample_and_select(eng, search_space, n_asks)
        # column-wise conversion (FloatDistribution.to_external_repr is the identity): 8192 x 32 values in
        # a few ms instead of one Python call per value
        names = list(search_space)
        columns = []
        for j, name in enumerate(names):
            d = search_space[name]
            col = x[:, j].tolist()
            columns.append(col if isinstance(d, FloatDistribution) else [d.to_external_repr(v) for v in col])
        return [dict(zip(names, row)) for row in zip(*columns)]

    def _rows(self, study, trials, names: list[str], dists: list[BaseDistribution], current: int | None):
        """History rows of `trials` (the arrays tpe_history_set / tpe_history_update take): internal
        representation of the parameters (NaN = absent), category and the reference's sort key inside it
        (sampler.py:686-722, :735-742, :782-821), objective values for multi-objective studies."""
        multi = study._is_multi_objective()
        sign = -1.0 if (not multi and study.direction == StudyDirection.MAXIMIZE) else 1.0
        n, p = len(trials), len(names)
        X = np.full((n, p), np.nan)
        cat = np.full(n, _lib.CAT_EXCLUDED, dtype=np.int8)
        key = np.zeros((n, 2))
        signs = np.asarray([-1.0 if d == StudyDirection.MAXIMIZE else 1.0 for d in study.directions])
        vals = np.full((n, len(signs)), np.inf) if multi else None
        index = names if isinstance(names, dict) else {name: j for j, name in enumerate(names)}
        complete, pruned, running = TrialState.COMPLETE, TrialState.PRUNED, TrialState.RUNNING
        constrained = self._constraints_func is not None
        for i, t in enumerate(trials):
            state = t.state
            if state == running:
                # constant liar: the other workers' trials sit in g(x) (sampler.py:526-535, :695-698)
                if not self._constant_liar or t.number == current:
                    continue
                cat[i] = _lib.CAT_RUNNING
            elif state != complete and state != pruned:
                continue  # WAITING, FAIL
            elif constrained and (score := _infeasible_score(t)) > 0:
                cat[i] = _lib.CAT_INFEASIBLE
                key[i, 0] = score
            elif state == complete:
                cat[i] = _lib.CAT_COMPLETE
                key[i, 0] = sign * t.value if not multi else 0.0
            else:
                cat[i] = _lib.CAT_PRUNED
                key[i] = _pruned_key(t, sign) if not multi else (1, 0.0)
            row = X[i]
            for name, value in self._get_params(t).items():
                j = index.get(name)
                if j is not None:
                    row[j] = dists[j].to_internal_repr(value)
            if multi and t.values is not None:
                vals[i] = signs * np.asarray(t.values, dtype=float)
        return X, cat, key, vals

    def _note_changes(self, changed: list[tuple[int, Any]]) -> None:
        """What a poll found goes to the device at the next sync (many polls never get there: startup
        trials, search-space queries)."""
        if changed:
            self._hist.backlog.update(changed)

    def _sync(self, study, trial, search_space: dict[str, BaseDistribution]) -> list[int]:
        """Bring the device history up to date with the log (the caller has polled); returns the device
        columns of `search_space`.  O(#rows that changed) unless a column is new: then the history is
        re-uploaded once with a column for every parameter the study has used so far."""
        h = self._hist
        eng = self._eng()
        current = None if trial is None else trial.number
        rebuild = h.dev_token != (id(h.storage), h.token) or h.dev_rows > h.rows
        for name, d in search_space.items():
            j = h.columns.get(name)
            if j is None or h.dists[j] != d:
                rebuild = True
        backlog = h.backlog
        if rebuild:
            names = list(h.columns) if h.dev_token == (id(h.storage), h.token) else []
            dists = list(h.dists) if names else []
            for name, d in list(h.all_dists.items()) + list(search_space.items()):
                if name in names:
                    dists[names.index(name)] = d
                else:
                    names.append(name)
                    dists.append(d)
            h.columns = {name: j for j, name in enumerate(names)}
            h.dists = dists
            h.dev_token = (id(h.storage), h.token)
            eng.set_space([_spec_of(nm, d, self._cat_dist_funcs) for nm, d in zip(names, dists)])
            trials = h.all_trials(study, self._multivariate or not self._constant_liar)
            X, cat, key, vals = self._rows(study, trials, names, dists, current)
            eng.set_history(X, cat, key)
            if vals is not None:
                eng.set_values(vals, 0, len(study.directions))
            h.dev_rows = len(trials)
            h.dev_cat = {row: int(cat[row]) for row in h.pending if row < h.dev_rows}
            h.dev_pred.clear()
            h.dev_version += 1
            backlog.clear()
            return [h.columns[name] for name in search_space]
        # rows uploaded at `tell` time: confirmed by what the storage shows now, or put back
        if h.dev_pred:
            for row, told in list(h.dev_pred.items()):
                t = backlog.get(row)
                if t is not None and told.matches(t):
                    del backlog[row]                 # the device holds exactly this row already
                    told.confirmed = True
                    h.dev_cat.pop(row, None)
                elif t is None and row in h.pending:
                    backlog[row] = h.pending[row][1]  # not stored (yet): the device gets back what the log shows
            h.dev_pred.clear()
        # constant liar: which unfinished rows sit in g(x) depends on who is asking
        if self._constant_liar:
            for row, slot in h.pending.items():
                if row in backlog:
                    continue
                t = slot[1]
                want = _lib.CAT_RUNNING if (t.state == TrialState.RUNNING and t.number != current) else _lib.CAT_EXCLUDED
                if h.dev_cat.get(row, _lib.CAT_EXCLUDED) != want:
                    backlog[row] = t
        # an unfinished trial nobody may see stays an EXCLUDED placeholder however often its object changes
        # (every suggest_* of a running trial replaces it): nothing to upload
        for row in [r for r in backlog if r < h.dev_rows and r in h.pending
                    and h.dev_cat.get(r, _lib.CAT_EXCLUDED) == _lib.CAT_EXCLUDED]:
            t = backlog[row]
            if not (self._constant_liar and t.state == TrialState.RUNNING and t.number != current):
                del backlog[row]
        if backlog:
            # unfinished trials nobody may see, past the end of the device history: nothing to upload -- a later row
            # that is written brings them along (_upload fills the gap from the log)
            for row in sorted(backlog, reverse=True):
                t = backlog[row]
                if row < h.dev_rows or t.state.is_finished() or (
                        self._constant_liar and t.state == TrialState.RUNNING and t.number != current):
                    break
                del backlog[row]
            self._upload(study, eng, backlog, current)
            backlog.clear()
        return [h.columns[name] for name in search_space]

    def _upload(self, study, eng, items: dict[int, Any], current: int | None) -> None:
        """Rows -> device, one tpe_history_update per contiguous run (a run may extend the history; rows between
        the device's end and the run are the placeholders of unfinished trials the log knows)."""
        h = self._hist
        if not items:
            return
        names = h.columns                            # (name -> column: _rows takes the mapping as it is)
        rows = sorted(items)
        if rows and rows[0] > h.dev_rows:
            gap = {r: h.pending[r][1] for r in range(h.dev_rows, rows[0])}  # KeyError: a finished row was skipped
            items = {**gap, **items}
            rows = sorted(items)
        i = 0
        while i < len(rows):
            j = i + 1
            while j < len(rows) and rows[j] == rows[j - 1] + 1:
                j += 1
            at = rows[i]
            run = [items[r] for r in rows[i:j]]
            X, cat, key, vals = self._rows(study, run, names, h.dists, current)
            if (cat != _lib.CAT_EXCLUDED).any() or any(
                    r < h.dev_rows and (r not in h.pending or h.dev_cat.get(r, _lib.CAT_EXCLUDED) != _lib.CAT_EXCLUDED)
                    for r in rows[i:j]):
                h.dev_version += 1                   # (placeholders coming and going change nothing anyone sees)
            eng.update_history(X, cat, key, at)
            if vals is not None:
                eng.set_values(vals, at, len(study.directions))
            for r, c in zip(rows[i:j], cat):
                if r in h.pending:
                    h.dev_cat[r] = int(c)
                else:
                    h.dev_cat.pop(r, None)
            h.dev_rows = max(h.dev_rows, at + len(run))
            i = j

    #: asks needing at least this many uniforms have them generated on the device
    DEVICE_RNG_MIN = 4096

    def _draw_uniforms(self, search_space: dict[str, BaseDistribution]) -> np.ndarray:
        """The uniforms one reference `_sample` consumes, in its order: C for `rng.choice`, C per
        categorical column, then an (n_numeric, C) block (probability_distributions.py:87,100,138-144).
        `rand`, `choice` and `uniform(0, 1)` all take consecutive `random_sample` outputs unchanged, so
        ONE call yields the identical stream (checked in tests/test_host_glue.py) at half the cost."""
        return self._rng.rng.random_sample(self._n_ei_candidates * (1 + len(search_space)))

    def _sample_and_select(self, eng: TPEEngine, search_space: dict[str, BaseDistribution], n_asks: int) -> np.ndarray:
        """Uniforms + stages 3-4, once the estimators are built.  Large asks: the library generates the generator's
        next outputs on the GPU (k_mt19937_uniform, the same MT19937 stream bit for bit) while the estimator builds
        run, and the host generator is moved to the state after the draws on demand; small asks draw on the host.
        The estimators are built (and validated) BEFORE the generator moves, as in the reference (sampler.py:544-553):
        an ask that fails in the build leaves the stream untouched."""
        n = n_asks * self._n_ei_candidates * (1 + len(search_space))
        x, _, _ = eng.sample_and_select(self._rng.draw(eng, n, n >= self.DEVICE_RNG_MIN), n_asks)
        return x

    def _cfg(self, n_finished: int) -> dict:
        """The configuration of every engine call, for a history of `n_finished` finished trials."""
        if self._prior_weight < 0:
            raise ValueError("A non-negative value must be specified for prior_weight,"
                             f" but got {self._prior_weight}.")
        return dict(n_below=int(self._gamma(n_finished)), n_candidates=self._n_ei_candidates,
                    multivariate=self._multivariate, prior_weight=self._prior_weight, magic_clip=self._magic_clip,
                    endpoints=self._endpoints)

    def _prepare(self, eng: TPEEngine, cols: list[int], cfg: dict, study=None) -> tuple:
        """``eng.prepare(cols)``, then the user's weights of the below and above sets as ``eng.build`` takes them --
        None for `default_weights`, which the library evaluates itself (k_weights).  In a multi-objective `study`
        l(x) is weighted by hypervolume contributions (computed by the library) and the user's function only
        shapes g(x) (sampler.py:570-584)."""
        _, nb, na = eng.prepare(cols, **cfg)
        if self._weights is default_weights:
            return None, None
        wb = None if study is not None and study._is_multi_objective() else _checked_weights(self._weights, nb)
        return wb, _checked_weights(self._weights, na)

    #: per-parameter asks of a univariate trial are evaluated together from this many parameters on
    UNI_BATCH_MIN = 2

    def _plannable(self, study, calls: list) -> bool:
        """Can the per-parameter `calls` of a trial be evaluated together (_UniPlan)?  Only for univariate TPE: the
        reference computes a multivariate sampler's independent parameters with multivariate bandwidths
        (sampler.py:335-341, :491), which the batched entry does not take."""
        return (not self._multivariate and not self._constant_liar and not self._uni.disabled
                and not study._is_multi_objective() and len(calls) >= self.UNI_BATCH_MIN
                and len({n for n, _ in calls}) == len(calls))

    def _sample_one(self, study, trial, name: str, dist: BaseDistribution) -> Any:
        """One `sample_independent` past the startup trials.  The caller holds the lock and has polled."""
        a = self._ahead
        if a is not None and a.kind != "uni":
            self._drop_ahead()
            a = None
        u = self._uni
        h = self._hist
        if u.calls_trial != trial.number:            # a new trial: the finished recording becomes the prediction
            if u.calls_trial is not None:
                u.prev = u.calls
            u.calls_trial, u.calls = trial.number, []
        u.calls.append((name, dist))
        version = (id(h.storage), h.token, h.n_finished, len(h.pending) if self._constant_liar else 0)
        if a is not None:                            # the batch of this trial was queued when the last one was told
            if len(u.calls) == 1 and self._adopt_uni_ahead(study, trial, a, name, dist, version):
                return u.values[0]
            self._drop_ahead()
        if u.trial == trial.number and u.next < len(u.order):
            if u.order[u.next] == (name, dist) and u.version == version and not self._finished_backlog():
                return self._serve_plan()
            self._rng.rng                            # not as predicted: settle the generator, then one at a time
            u.trial = None
        if len(u.calls) == 1 and u.prev and u.prev[0] == (name, dist) and self._plannable(study, u.prev):
            try:
                return self._plan_trial(study, trial, version)
            except RuntimeError as e:
                if "not batchable" not in str(e):
                    raise
                u.disabled, u.trial = True, None
        return self._sample(study, trial, {name: dist})[name]

    def _finished_backlog(self) -> bool:
        """Did a trial other than the running ones change since the plan was made?"""
        h = self._hist
        return any(r not in h.pending for r in h.backlog)

    def _uni_batch(self, eng: TPEEngine, cols: list[int], cfg: dict, run) -> tuple:
        """The user's weights and the uniforms of the per-parameter calls of `cols`, handed to `run`
        (``eng.suggest_univariate_batch`` or its async twin).  Returns (what `run` returned, wb, wa, the generator
        before the draws, whether they were generated on the device); if `run` fails, the generator is put back."""
        wb = wa = None
        if self._weights is not default_weights:   # the sizes of the two sets (the split does not depend on the column)
            wb, wa = self._prepare(eng, cols[:1], cfg)
        count = 2 * self._n_ei_candidates * len(cols)
        dev_rng = count >= self.DEVICE_RNG_MIN
        snap, uniforms = self._rng.stage(eng, count, dev_rng)
        try:
            out = run(cols, uniforms, wb, wa, **cfg)
        except Exception:
            self._rng.restore(snap)                 # nothing was served: the generator has not moved
            raise
        return out, wb, wa, snap, dev_rng

    def _plan_trial(self, study, trial, version) -> Any:
        """Evaluate every parameter of `self._uni.prev` for `trial` in one device call; returns the first value."""
        order = list(self._uni.prev)
        cols = self._sync(study, trial, dict(order))
        cfg = self._cfg(self._hist.n_finished)
        eng = self._eng()
        (x, _, _), wb, wa, st0, dev_rng = self._uni_batch(eng, cols, cfg, eng.suggest_univariate_batch)
        return self._install_plan(trial, version, order, cols, cfg, wb, wa, x, st0, eng if dev_rng else None)

    def _install_plan(self, trial, version, order, cols, cfg, wb, wa, x, st0, on_device) -> Any:
        """The batch has been evaluated (x: the winners per column, st0: the generator before its draws, on_device:
        the engine that generated them, None for host draws); returns the first value."""
        u = self._uni
        eng = self._eng()
        per = 2 * self._n_ei_candidates
        count = per * len(order)
        u.trial, u.order, u.version, u.on_device = trial.number, order, version, on_device
        u.values = [d.to_external_repr(float(v)) for (_, d), v in zip(order, x)]
        u.next = 0
        if self._audit is not None:
            # test hook: the candidates / log-densities of every column, re-evaluated one column at a time on the
            # same stretch of uniforms (the batched entry keeps only the winners)
            uu = eng.get_uniforms(count) if u.on_device is not None else np.random.RandomState()
            if u.on_device is None:
                uu.set_state(st0)
                uu = uu.random_sample(count)
            for j, (nm, d) in enumerate(order):
                eng.suggest(cols[j: j + 1], uu[j * per: (j + 1) * per], 1, wb, wa, **cfg)
                self._audit(trial, {nm: d}, eng)

        def settle() -> None:   # the generator after the calls served so far (and only those)
            self._rng.restore(st0, per * u.next)
            u.trial = None
        u.settle = self._rng.arm(settle)
        return self._serve_plan()

    def _serve_plan(self) -> Any:
        """The next value of the plan; once all are served the generator stands where the batch left it."""
        u = self._uni
        value = u.values[u.next]
        u.next += 1
        if u.next == len(u.order):
            self._rng.release(u.settle, adopted=True)
            if u.on_device is not None:
                self._rng.mark_device(u.on_device)
        return value

    def _look_ahead_uni(self, study, trial, state, values) -> None:
        """`_look_ahead` for univariate TPE: the per-parameter calls of the NEXT trial, predicted to repeat this
        trial's, are queued as one batch now (tpe_suggest_univariate_batch_async); the first `sample_independent` of
        the next trial adopts it if the trial was stored as uploaded, the call is the predicted one and nobody touched
        the generator (`_adopt_uni_ahead`)."""
        self._drop_ahead()
        u = self._uni
        if not (self._prior_weight >= 0 and (state == TrialState.COMPLETE or state == TrialState.PRUNED)
                and u.calls_trial == trial.number and self._plannable(study, u.calls)):
            return
        order = list(u.calls)
        space = dict(order)
        up = self._upload_told(study, trial, state, values, space)
        if up is None:
            return
        cols, told = up
        eng = self._eng()
        cfg = self._cfg(self._hist.n_finished + 1)
        try:
            _, wb, wa, snap, dev_rng = self._uni_batch(eng, cols, cfg, eng.suggest_univariate_batch_async)
        except Exception:                            # e.g. "not batchable asynchronously": the ask plans as before
            return
        cancel = self._rng.arm(lambda: self._rng.restore(snap))
        self._ahead = _Ahead("uni", told, space, cols, cfg, self._hist.n_finished + 1, self._hist.dev_version, eng,
                             dev_rng, snap, cancel, order=order, wb=wb, wa=wa)

    def _adopt_uni_ahead(self, study, trial, a, name, dist, version) -> bool:
        """First `sample_independent` of a trial with a batch queued at `tell` time: take it if it is this trial's."""
        h = self._hist
        cols = self._sync(study, trial, dict(a.order))
        cfg = self._cfg(h.n_finished)
        if not (a.told.confirmed and a.eng is self._engine and a.dev_version == h.dev_version and a.cols == cols
                and a.cfg == cfg and a.order[0] == (name, dist) and self._rng.armed(a.cancel)):
            self._drop_ahead()
            return False
        self._ahead = None
        self._rng.release(a.cancel, adopted=True)
        x, _, _ = a.eng.collect_univariate()
        # (host draws: the generator already stands after the batch)
        self._install_plan(trial, version, a.order, cols, cfg, a.wb, a.wa, x, a.snap, a.eng if a.dev_rng else None)
        self.ahead_stats[0] += 1
        return True

    def _sample(self, study, trial, search_space: dict[str, BaseDistribution], speculate: bool = False) -> dict[str, Any]:
        """TPESampler._sample (sampler.py:523-560).  The caller holds the lock and has polled."""
        t0 = time.perf_counter()
        cols = self._sync(study, trial, search_space)
        t1 = time.perf_counter()
        try:
            out = self._sample_synced(study, cols, search_space)
            if self._audit is not None:
                self._audit(trial, search_space, self._eng())
            if speculate and self.LOOK_AHEAD and self.SPECULATE:
                t2 = time.perf_counter()
                try:
                    self._speculate(study, trial, cols, search_space, out)
                except Exception as e:               # ... nor an `ask` whose suggestion is already computed
                    _logger.debug(f"speculation abandoned: {e!r}")
                    self._abandon_ahead()
                self.last_spec_s = time.perf_counter() - t2
            return out
        finally:
            # wall time of the last ask: history sync (host walk + row uploads) / everything after it
            # (prepare, build, uniforms, sampling + grids + argmax, read-back, to_external_repr)
            self.last_ask_s = (t1 - t0, time.perf_counter() - t1)

    def _sample_synced(self, study, cols: list[int], search_space: dict[str, BaseDistribution]) -> dict[str, Any]:
        cfg = self._cfg(self._hist.n_finished)
        eng = self._eng()
        x = self._take_ahead(eng, cols, search_space, cfg)
        if x is None:
            wb, wa = self._prepare(eng, cols, cfg, study)
            eng.build(wb, wa)
            x = self._sample_and_select(eng, search_space, 1)
        self._last_space = search_space
        out = {}
        for j, (name, d) in enumerate(search_space.items()):
            out[name] = d.to_external_repr(float(x[0, j]))
        return out

    # -- look-ahead: the next suggestion is computed while the study finishes `tell` and starts `ask` ----------
    #: queue the next joint suggestion at `tell` time (multivariate TPE; see _look_ahead)
    LOOK_AHEAD = True

    def _abandon_ahead(self) -> None:
        """Something went wrong while computing ahead: forget it, put the generator back, and let the next ask
        rebuild the device history from the study (nothing the device holds is trusted)."""
        try:
            self._drop_ahead()
        except Exception:                            # (the failed undo is no longer pending)
            pass
        h = self._hist
        h.dev_token = None
        h.dev_pred.clear()

    def _drop_ahead(self) -> None:
        """Discard the suggestion queued ahead, if any: nobody takes it, its draws are undone."""
        a, self._ahead = self._ahead, None
        if a is not None:
            self.ahead_stats[1] += 1
            self._rng.release(a.cancel, adopted=False)

    def _take_ahead(self, eng, cols, search_space, cfg):
        """The suggestion queued at `tell` time, if this ask is the one it was computed for: the very columns and
        configuration, the finished trial stored exactly as it was uploaded, nothing else the estimators see
        changed since, the generator untouched.  Otherwise the generator goes back to where it was."""
        a = self._ahead
        if a is None:
            return None
        if not (a.kind == "joint" and a.told.confirmed and a.eng is eng and a.dev_version == self._hist.dev_version
                and a.cols == cols and a.cfg == cfg and self._rng.armed(a.cancel)
                and list(a.space.items()) == list(search_space.items())):
            self._drop_ahead()
            return None
        self._ahead = None
        self._rng.release(a.cancel, adopted=True)
        x, _, _ = eng.collect()
        if a.dev_rng:
            self._rng.mark_device(eng)
        self.ahead_stats[0] += 1
        return x

    def _upload_told(self, study, trial, state, values, space) -> tuple[list[int], _Told] | None:
        """`tell` time, past the startup trials: the finished trial's row goes to the device before the storage
        shows it.  Returns the device columns of `space` and what was uploaded, or None when the trial's row is not
        the log's pending row of that trial (nothing is uploaded then)."""
        h = self._hist
        self._note_changes(self._poll(study))
        if h.n_finished + 1 < self._n_startup_trials:
            return None
        row = trial.number
        cols = self._sync(study, None, space)
        if row >= h.rows or row not in h.pending or h.numbers[row] != trial.number:
            return None
        told = _Told(trial, state, values)
        if self._constraints_func is not None:       # after_trial has just stored them (samplers/_base.py:241-267)
            told.system_attrs[CONSTRAINTS_KEY] = study._storage.get_trial_system_attrs(trial._trial_id).get(CONSTRAINTS_KEY)
        self._upload(study, self._eng(), {row: told}, None)
        h.dev_pred[row] = told                       # (_upload kept its category in dev_cat: the row is pending)
        return cols, told

    def _look_ahead(self, study, trial, state, values) -> None:
        """Called from `after_trial`: the trial, its final state and values are known, the storage records them
        right after (study/_tell.py:163-169).  In a sequential loop everything the next ask will compute is
        determined at this point -- the history plus this trial, the same search space, the generator where the
        last ask left it -- so the row is uploaded and the whole suggestion queued on the device now; it runs while
        optuna stores the trial and creates the next one, and `sample_relative` collects it after checking that the
        ask really is the predicted one (`_take_ahead`).  Joint sampling only; anything out of the ordinary (constant
        liar, groups, a failed trial, a changed space) just skips it."""
        if self._confirm_speculation(study, trial, state, values):
            return
        self._drop_ahead()
        if not (self._multivariate and not self._group and not self._constant_liar and self._prior_weight >= 0
                and (state == TrialState.COMPLETE or state == TrialState.PRUNED)):
            return
        space = self._last_space
        d = trial.distributions
        if any(d.get(k) != v for k, v in space.items()):
            return                                   # the intersection search space shrinks with this trial
        up = self._upload_told(study, trial, state, values, space)
        if up is not None:
            cols, told = up
            self._queue_ahead(study, cols, space, told, "joint")

    def _confirm_speculation(self, study, trial, state, values) -> bool:
        """`tell` time: did the trial end the way `_speculate` assumed?  Then the queued suggestion is the next one's;
        the row gets its true key (queued behind the suggestion's kernels: it changes nothing they read)."""
        a = self._ahead
        if a is None or a.kind != "spec":
            return False
        h = self._hist
        g = a.told
        ok = (g.number == trial.number and state == TrialState.COMPLETE and values is not None and len(values) == 1
              and self._rng.armed(a.cancel) and a.dev_version == h.dev_version and a.eng is self._engine
              and trial.params == g.params and trial.distributions == g.distributions)
        if ok:
            v = float(values[0])
            key = -v if h.token[1][0] == StudyDirection.MAXIMIZE else v
            ok = key >= g.threshold
        if ok:
            self._note_changes(self._poll(study))
            ok = (trial.number in h.pending and not any(r not in h.pending for r in h.backlog)
                  and h.n_finished + 1 == a.cfg_n_finished)
        if not ok:
            self.spec_stats[1] += 1
            return False                             # (the caller drops it: the generator goes back)
        told = _Told(trial, state, values)
        self._upload(study, a.eng, {trial.number: told}, None)
        h.dev_pred[trial.number] = told
        a.told, a.kind, a.dev_version = told, "joint", h.dev_version
        self.spec_stats[0] += 1
        return True

    def _queue_ahead(self, study, cols, space, told, kind) -> None:
        """Queue the joint suggestion of the ask after `told` (whose row is on the device) without waiting for it."""
        h = self._hist
        eng = self._eng()
        cfg = self._cfg(h.n_finished + 1)
        n = self._n_ei_candidates * (1 + len(space))
        dev_rng = n >= self.DEVICE_RNG_MIN
        snap = None
        try:
            if not dev_rng:                          # host draws: uploaded on the side stream before anything is queued
                snap, uniforms = self._rng.stage(eng, n, False)  # (a copy from pageable memory waits for the work
                uniforms = eng.stage_uniforms(uniforms)          # queued before it)
            wb, wa = self._prepare(eng, cols, cfg, study)        # as _sample_synced
            eng.build(wb, wa)
            if dev_rng:
                snap, uniforms = self._rng.stage(eng, n, True)
            eng.sample_and_select_async(uniforms, 1)
        except Exception:                            # the ask will run into it again, and report it
            if snap is not None:
                self._rng.restore(snap)
            return
        cancel = self._rng.arm(lambda: self._rng.restore(snap))   # nobody took the suggestion: the draws never happened
        self._ahead = _Ahead(kind, told, space, cols, cfg, h.n_finished + 1, h.dev_version, eng, dev_rng, snap, cancel)

    #: queue the NEXT suggestion already when a suggestion has been handed out, assuming the trial will end up in the
    #: above set (see _speculate)
    SPECULATE = True

    def _speculate(self, study, trial, cols, space, params) -> None:
        """Outcome speculation.  The estimators of the next ask depend on the running trial only through the SET it
        falls into: g(x) weights its kernels by position, not by value, and a trial whose value does not beat the
        n_below-th best leaves l(x) untouched (sampler.py:686-722).  With 100k trials that is how all but ~25 in
        100k trials end, so the next joint suggestion is queued right now -- the trial's row goes to the device as
        COMPLETE with the worst possible key -- and runs while the objective is evaluated.  `_look_ahead` (at `tell`
        time) keeps it only if the trial really ended that way: COMPLETE, exactly these parameters, a value that does
        not enter the below set (`_History.best_keys`), nothing else changed, the generator untouched; otherwise the
        generator goes back and the suggestion is computed with the true row.  Single-objective studies without
        constraints, joint sampling."""
        h = self._hist
        if (self._constant_liar or self._constraints_func is not None or study._is_multi_objective()
                or self._prior_weight < 0 or self._ahead is not None or trial is None):
            return
        n_below = int(self._gamma(h.n_finished + 1))
        row = trial.number
        if not (0 < n_below <= min(len(h.best_keys), h.n_complete) and row in h.pending and row < h.rows
                and h.numbers[row] == trial.number and h.n_finished + 1 >= self._n_startup_trials and not h.backlog):
            return
        worst = float("-inf") if h.token[1][0] == StudyDirection.MAXIMIZE else float("inf")
        guess = _Told(trial, TrialState.COMPLETE, [worst])
        guess.params = dict(params)
        guess.distributions = dict(space)
        guess.threshold = h.best_keys[n_below - 1]
        self._upload(study, self._eng(), {row: guess}, None)
        h.dev_pred[row] = guess
        self._queue_ahead(study, cols, space, guess, "spec")
