"""PED-ANOVA importance over arrays (TEST INFRASTRUCTURE ONLY -- see oracle/__init__.py).

NumPy restatement of the arithmetic of ``optuna.importance.PedAnovaImportanceEvaluator`` on the history arrays the
library keeps (X in internal representation, category, key; include/optuna_b200_tpe.h) instead of FrozenTrials:

* row filter            <- optuna/importance/_base.py:145-156 (COMPLETE, every selected parameter, finite loss)
* quantile cut-offs     <- optuna/importance/_ped_anova/evaluator.py:37-55 (two np.partition calls per quantile)
* binning               <- optuna/importance/_ped_anova/scott_parzen_estimator.py:90-135
* Scott estimator       <- scott_parzen_estimator.py:16-87 on top of parzen_estimator.py:39-78, :132-166,
                           evaluated with oracle.tpe_oracle.mixture_log_pdf (probability_distributions.py:154-223)
* Pearson divergence    <- evaluator.py:196-220, scaled by (n_target / n_region) ** 2 (:258-263)

Every expression keeps the reference's operation order and array shapes, so the results agree with it bit for bit
on the same NumPy / libm (tests/test_ped_anova.py).
"""
from __future__ import annotations

import numpy as np

from oracle import tpe_oracle as orc


def quantile_cutoff(loss: np.ndarray, quantile: float, min_n_top: int) -> float:
    """evaluator.py:44-53: the larger of the min_n_top-th smallest loss and the ceil(q n)-th smallest."""
    n = loss.size
    cutoff_index = int(np.ceil(quantile * n)) - 1
    return max(np.partition(loss, min_n_top - 1)[min_n_top - 1],
               float(np.partition(loss, cutoff_index)[cutoff_index]))


def bin_counts(values: np.ndarray, param: orc.Param, grid: np.ndarray | None, n_grid: int) -> np.ndarray:
    """scott_parzen_estimator.py:106-135: counts of the observed values per grid point (categorical: per choice)."""
    if param.is_cat:
        idx = values.astype(int)
    else:
        v = np.log(values) if param.log else values
        step_size = grid[1] - grid[0] if n_grid >= 2 else 0.0
        idx = np.searchsorted(grid[:n_grid], v - step_size / 2)
    unique_vals, counts_in_unique = np.unique(idx, return_counts=True)
    counts = np.zeros(n_grid, dtype=np.int32)
    counts[unique_vals] += counts_in_unique
    return counts


def scott_pdf(counts: np.ndarray, is_cat: bool, prior_weight: float) -> np.ndarray:
    """_ScottParzenEstimator(...).pdf(np.arange(n_steps)) + 1e-12 (scott_parzen_estimator.py:16-87,
    evaluator.py:209-210)."""
    counts = counts.astype(np.float64)
    n_steps = len(counts)
    obs = np.arange(n_steps)[counts > 0.0]
    cfg = orc.Config(prior_weight=prior_weight)
    if is_cat:
        param = orc.Param("cat", n_choices=n_steps)
        mix = orc.build_mixture(obs.astype(float), [param], cfg, counts[counts > 0.0])
    else:
        param = orc.Param("int", 0, n_steps - 1, 1.0)
        w = counts[counts > 0.0]
        w = np.append(w, [prior_weight]) if obs.size else np.array([1.0])
        mix = orc.Mixture(weights=w / w.sum(), params=[param])
        n_trials = np.sum(counts)
        counts_non_zero = counts[counts > 0]
        weights = counts_non_zero / n_trials
        mus = np.arange(n_steps)[counts > 0]
        mean_est = mus @ weights
        sigma_est = np.sqrt((mus - mean_est) ** 2 @ counts_non_zero / max(1, n_trials - 1))
        count_cum = np.cumsum(counts_non_zero)
        idx_q25 = np.searchsorted(count_cum, n_trials // 4, side="left")
        idx_q75 = np.searchsorted(count_cum, n_trials * 3 // 4, side="right")
        interquantile_range = mus[min(mus.size - 1, idx_q75)] - mus[idx_q25]
        sigma_est = 1.059 * min(interquantile_range / 1.34, sigma_est) * n_trials ** (-0.2)
        sigma_min = 0.5 / 1.64
        sigmas = np.full_like(mus, max(sigma_est, sigma_min), dtype=np.float64)
        mix.mu[0] = np.append(mus, [0.5 * (0 + n_steps - 1)])
        mix.sigma[0] = np.append(sigmas, [1.0 * (n_steps - 1 - 0 + 1)])
    grid = np.arange(n_steps)[:, np.newaxis]
    return np.exp(orc.mixture_log_pdf(mix, grid)) + 1e-12


def ped_anova(X: np.ndarray, category: np.ndarray, key: np.ndarray, params: list[orc.Param], cols: list[int],
              grids: np.ndarray, n_grid: np.ndarray, *, target_quantile: float, region_quantile: float,
              evaluate_on_local: bool, loss: np.ndarray | None = None, prior_weight: float = 1.0,
              min_n_top: int = 2):
    """Importance of every column of `cols`, the sizes (kept, target, region) and the per-column bin counts
    [n_cols, 2 (target, region), max(n_grid)].  Importances are zero and counts empty when at most min_n_top rows
    are kept (evaluator.py:244-245)."""
    X = np.asarray(X, dtype=np.float64)
    lv = key[:, 0] if loss is None else np.asarray(loss, dtype=np.float64)
    keep = (np.asarray(category) == orc.CAT_COMPLETE) & np.isfinite(lv)
    for c in cols:
        keep &= ~np.isnan(X[:, c])
    rows = np.nonzero(keep)[0]
    n = rows.size
    width = int(max(n_grid)) if len(cols) else 0
    counts = np.zeros((len(cols), 2, width), dtype=np.int32)
    imp = np.zeros(len(cols))
    if n <= min_n_top:
        return imp, (n, 0, 0), counts
    kept_loss = lv[rows]
    target = rows[kept_loss <= quantile_cutoff(kept_loss, target_quantile, min_n_top)]
    region = rows if region_quantile == 1.0 else rows[
        kept_loss <= quantile_cutoff(kept_loss, region_quantile, min_n_top)]
    quantile = len(target) / len(region)
    for j, c in enumerate(cols):
        p, g = params[c], int(n_grid[j])
        ct = bin_counts(X[target, c], p, None if p.is_cat else grids[j], g)
        cr = bin_counts(X[region, c], p, None if p.is_cat else grids[j], g)
        counts[j, 0, :g], counts[j, 1, :g] = ct, cr
        pdf_top = scott_pdf(ct, p.is_cat, prior_weight)
        if evaluate_on_local:
            pdf_local = scott_pdf(cr, p.is_cat, prior_weight)
        else:
            pdf_local = np.full(g, 1.0 / g)
        imp[j] = quantile**2 * float(pdf_local @ ((pdf_top / pdf_local - 1) ** 2))
    return imp, (n, len(target), len(region)), counts
