"""B200PedAnovaImportanceEvaluator -- optuna's PED-ANOVA importance evaluator on a B200.

Same constructor arguments as ``optuna.importance.PedAnovaImportanceEvaluator`` (optuna/importance/_ped_anova/
evaluator.py:141-172, + ``device``) and the same ``evaluate`` results, so
``optuna.importance.get_param_importances(study, evaluator=B200PedAnovaImportanceEvaluator())`` works unchanged.

The reference walks every FrozenTrial at every call: the intersection search space (importance/_base.py:72-77),
``_get_filtered_trials`` (:145-156), the quantile filters and one list comprehension per parameter for the binning
(scott_parzen_estimator.py:90-135).  Here the study's trial list is followed incrementally (``_History``, as the
sampler does) into a device history of this evaluator's own, and the rest -- row filter, the two order statistics,
the per-column histograms, the Scott estimators and the Pearson divergence -- is one call into libtpe_b200.so
(``tpe_ped_anova``, include/optuna_b200_tpe.h).  A second call on the same study costs O(trials changed since the
last call) of host work plus that one call.
"""
from __future__ import annotations

import threading
from typing import Any, Callable

import numpy as np

from . import _lib
from ._compat import (BaseDistribution, CategoricalDistribution, IntDistribution, StudyDirection, TrialState,
                      optuna_warn)
from .engine import TPEEngine
from .sampler import _History, _Reset, _spec_of

from optuna._deprecated import _DEPRECATION_WARNING_TEMPLATE  # noqa: I100 (optuna is importable: ._compat checked)
from optuna.importance._base import (BaseImportanceEvaluator, _get_distributions, _get_filtered_trials,
                                     _sort_dict_by_importance)


def _grid(d: BaseDistribution, n_steps: int) -> tuple[int, np.ndarray | None]:
    """Bins of one parameter and, for a numerical one, its grid (scott_parzen_estimator.py:96-105)."""
    if isinstance(d, CategoricalDistribution):
        return len(d.choices), None
    if isinstance(d, IntDistribution) and d.log:
        log2_domain_size = int(np.ceil(np.log(d.high - d.low + 1) / np.log(2))) + 1
        n_steps = min(log2_domain_size, n_steps)
    elif d.step is not None:
        n_steps = min(round((d.high - d.low) / d.step) + 1, n_steps)
    scaler = np.log if d.log else np.asarray
    return n_steps, np.linspace(scaler(d.low), scaler(d.high), n_steps)


class B200PedAnovaImportanceEvaluator(BaseImportanceEvaluator):
    """PED-ANOVA importance evaluator (``optuna.importance.PedAnovaImportanceEvaluator``) computed on a B200.

    Args:
        target_quantile, region_quantile, baseline_quantile, evaluate_on_local:
            As ``optuna.importance.PedAnovaImportanceEvaluator``; ``baseline_quantile`` is deprecated and ignored.
        device:
            CUDA device of the evaluator's history.

    The evaluator keeps a copy of the study's COMPLETE trials on the device and brings it up to date at each call, so
    calling it again after a few more trials costs little.  A ``target`` callable is evaluated on every COMPLETE trial
    that has the evaluated parameters at every call, as the reference does: O(trials) Python per call.
    """

    #: what answers the array-level call -- the CUDA library; tests plug the CPU oracle in here
    _engine_cls = TPEEngine

    def __init__(
        self,
        *,
        target_quantile: float = 0.1,
        region_quantile: float = 1.0,
        baseline_quantile: float | None = None,
        evaluate_on_local: bool = True,
        device: int = 0,
    ) -> None:
        assert 0.0 < target_quantile < region_quantile <= 1.0, (
            "condition 0.0 < `target_quantile` < `region_quantile` <= 1.0 must be satisfied"
        )
        if baseline_quantile is not None:
            msg = _DEPRECATION_WARNING_TEMPLATE.format(name="`baseline_quantile`", d_ver="4.7.0", r_ver="5.0.0")
            optuna_warn(f"{msg} `baseline_quantile` is currently ignored. Use `target_quantile` instead.")
        if region_quantile != 1.0 and not evaluate_on_local:
            optuna_warn("If `evaluate_on_local` is False, `region_quantile` has no effect.")
        self._target_quantile = target_quantile
        self._region_quantile = region_quantile
        self._evaluate_on_local = evaluate_on_local
        # the reference's fixed settings (evaluator.py:166-172)
        self._n_steps = 50
        self._prior_weight = 1.0
        self._min_n_top_trials = 2
        self._device = device
        self._engine: Any = None
        self._lock = threading.RLock()
        self._hist = _History()
        self._forget()

    def _forget(self) -> None:
        """Drop everything learnt from a study (another study, or a trial list that is not the one seen)."""
        self._n_complete = 0
        self._inter: dict[str, BaseDistribution] | None = None   # intersection over COMPLETE trials
        self._first: dict[str, BaseDistribution] = {}            # first distribution COMPLETE trials used, per name
        self._dynamic: set[str] = set()                          # names COMPLETE trials used with two distributions
        self._name_count: dict[str, int] = {}                    # COMPLETE trials holding each name
        self._columns: dict[str, int] = {}                       # device history column per name
        self._col_dists: list[BaseDistribution] = []
        self._dev_rows = -1                                      # -1: no device history
        self._backlog: dict[int, Any] = {}                       # row -> trial the device has not seen

    def close(self) -> None:
        """Release the device context (re-created on demand)."""
        eng, self._engine = self._engine, None
        if eng is not None:
            eng.close()
        self._dev_rows = -1

    def __del__(self) -> None:  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    # -- trial log ----------------------------------------------------------------------------------------------
    def _poll(self, study) -> None:
        h = self._hist
        seen = (h.storage, h.token)
        try:
            changed = h.poll(study, False)
        except _Reset:
            h.storage = None
            changed = h.poll(study, False)
            seen = None
        h.group_backlog.clear()   # (kept by _History for the sampler's group decomposition only)
        if seen is None or seen[0] is not h.storage or seen[1] != h.token:
            self._forget()
        for row, t in changed:
            self._backlog[row] = t
            if t.state == TrialState.COMPLETE:
                self._account(t)

    def _account(self, t) -> None:
        """A trial seen COMPLETE for the first time (a finished trial never changes again)."""
        self._n_complete += 1
        d = t.distributions
        for name, dist in d.items():
            first = self._first.setdefault(name, dist)
            if first is not dist and first != dist:
                self._dynamic.add(name)
            self._name_count[name] = self._name_count.get(name, 0) + 1
        if self._inter is None:
            self._inter = dict(d)
        elif self._inter and not (len(d) == len(self._inter) and all(d.get(k) is v for k, v in self._inter.items())):
            self._inter = {k: v for k, v in self._inter.items() if d.get(k) == v}

    # -- search space (importance/_base.py:72-142) ------------------------------------------------------------------
    def _distributions(self, study, params: list[str] | None) -> dict[str, BaseDistribution]:
        if self._n_complete == 0:
            raise ValueError("Cannot evaluate parameter importances without completed trials.")
        if self._n_complete == 1:
            raise ValueError("Cannot evaluate parameter importances with only a single trial.")
        if params is None:
            return dict(sorted((self._inter or {}).items(), key=lambda kv: kv[0]))
        if not isinstance(params, (list, tuple)):
            raise TypeError(f"Parameters must be specified as a list. Actual parameters: {params}.")
        if any(not isinstance(p, str) for p in params):
            raise TypeError(f"Parameters must be specified by their names with strings. Actual parameters: {params}.")
        if any(p in self._dynamic for p in params):
            return _get_distributions(study, params)   # the reference's walk: only here can it raise
        if len(params) > 0 and not all(self._name_count.get(p, 0) == self._n_complete for p in params):
            complete = study.get_trials(deepcopy=False, states=(TrialState.COMPLETE,))
            if not any(all(p in t.distributions for p in params) for t in complete):
                raise ValueError("Study must contain completed trials with all specified parameters. "
                                 f"Specified parameters: {params}.")
        return {name: self._first[name] for name in sorted(set(params))}

    # -- device history ---------------------------------------------------------------------------------------------
    def _eng(self):
        if self._engine is None:
            self._engine = self._engine_cls(self._device)
        return self._engine

    def _rows(self, study, trials):
        """History rows: COMPLETE trials as TPE_CAT_COMPLETE with key (sign * value, 0), everything else an
        excluded placeholder.  A parameter is stored in the internal representation of the trial's own distribution."""
        single = len(study.directions) == 1
        sign = -1.0 if single and study.direction == StudyDirection.MAXIMIZE else 1.0
        n, index = len(trials), self._columns
        X = np.full((n, len(index)), np.nan)
        cat = np.full(n, _lib.CAT_EXCLUDED, dtype=np.int8)
        key = np.zeros((n, 2))
        for i, t in enumerate(trials):
            if t.state != TrialState.COMPLETE:
                continue
            cat[i] = _lib.CAT_COMPLETE
            if single:
                key[i, 0] = sign * t.value
            dists, row = t.distributions, X[i]
            for name, value in t.params.items():
                j = index.get(name)
                if j is not None:
                    row[j] = dists[name].to_internal_repr(value)
        return X, cat, key

    def _sync(self, study, dists: dict[str, BaseDistribution]) -> list[int]:
        """Bring the device history up to date; returns the columns of `dists`.  O(#changed rows) unless a column is
        new or its distribution changed: then one re-upload with a column for every parameter seen so far."""
        eng = self._eng()
        if self._dev_rows < 0 or any(self._columns.get(n) is None or self._col_dists[self._columns[n]] != d
                                     for n, d in dists.items()):
            names = list(self._first)
            col_dists = [dists.get(n, self._first[n]) for n in names]
            self._columns = {n: j for j, n in enumerate(names)}
            self._col_dists = col_dists
            eng.set_space([_spec_of(n, d, {}) for n, d in zip(names, col_dists)])
            trials = self._hist.all_trials(study, False)
            eng.set_history(*self._rows(study, trials))
            self._dev_rows = len(trials)
            self._backlog.clear()
            return [self._columns[n] for n in dists]
        # rows the device must see: new ones (placeholders included, so that rows stay trial numbers) and those that
        # became COMPLETE; an unfinished trial that changed stays a placeholder
        rows = sorted(r for r, t in self._backlog.items() if r >= self._dev_rows or t.state == TrialState.COMPLETE)
        i = 0
        while i < len(rows):
            j = i + 1
            while j < len(rows) and rows[j] == rows[j - 1] + 1:
                j += 1
            eng.update_history(*self._rows(study, [self._backlog[r] for r in rows[i:j]]), rows[i])
            self._dev_rows = max(self._dev_rows, rows[j - 1] + 1)
            i = j
        self._backlog.clear()
        return [self._columns[n] for n in dists]

    # -- evaluate (evaluator.py:222-266) ------------------------------------------------------------------------------
    def evaluate(
        self,
        study,
        params: list[str] | None = None,
        *,
        target: Callable[[Any], float] | None = None,
    ) -> dict[str, float]:
        with self._lock:
            self._poll(study)
            dists = self._distributions(study, params)
            if params is None:
                params = list(dists.keys())
            non_single = {name: d for name, d in dists.items() if not d.single()}
            single = {name: d for name, d in dists.items() if d.single()}
            if len(non_single) == 0:
                return {}
            loss = None
            if target is not None:
                loss = self._target_loss(study, params, target)
            elif len(study.directions) > 1:
                _get_filtered_trials(study, params, None)   # FrozenTrial.value raises as in the reference
            cols = self._sync(study, dists)
            n_grid = np.zeros(len(dists), dtype=np.int32)
            grids = np.zeros((len(dists), self._n_steps))
            for j, d in enumerate(dists.values()):
                n_grid[j], g = _grid(d, self._n_steps)
                if g is not None:
                    grids[j, : g.size] = g
            imp, (n, n_target, n_region), _ = self._eng().ped_anova(
                cols, grids, n_grid, target_quantile=self._target_quantile, region_quantile=self._region_quantile,
                evaluate_on_local=self._evaluate_on_local, loss=loss, prior_weight=self._prior_weight,
                min_n_top=self._min_n_top_trials, n_steps=self._n_steps)
        if n <= self._min_n_top_trials:
            return {k: 0.0 for k in dists}
        if target is not None:
            for _ in range(1 if self._region_quantile == 1.0 else 2):   # once per quantile filter (evaluator.py:183)
                optuna_warn("PedAnovaImportanceEvaluator computes the importances of params to achieve "
                            "low `target` values. If this is not what you want, "
                            "please modify target, e.g., by multiplying the output by -1.")
        if n_target == n_region:
            optuna_warn("Target and region quantiles select the same set of trials. "
                        "Parameter importances will be equal.")
        pos = {name: j for j, name in enumerate(dists)}
        param_importances = {name: float(imp[pos[name]]) for name in non_single}
        param_importances.update({k: 0.0 for k in single})
        return _sort_dict_by_importance(param_importances)

    def _target_loss(self, study, params, target) -> np.ndarray:
        """target(t) of every COMPLETE trial holding all of `params` (the trials _get_filtered_trials evaluates it
        on, importance/_base.py:149-156), NaN elsewhere; one entry per trial of the study's list."""
        trials = self._hist.all_trials(study, False)
        need = set(params)
        loss = np.full(len(trials), np.nan)
        for i, t in enumerate(trials):
            if t.state == TrialState.COMPLETE and need <= set(t.params):
                loss[i] = target(t)
        return loss
