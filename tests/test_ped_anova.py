"""B200PedAnovaImportanceEvaluator against optuna.importance.PedAnovaImportanceEvaluator.

Every scenario builds a study from fixed trials and evaluates it with our evaluator on both engines: the CPU oracle
(oracle/ped_anova.py, host glue checked anywhere; it must equal the reference bit for bit) and libtpe_b200.so (GPU
box; importances within 1e-9 * max of the reference, counts exact).  The reference's results are stored in
tests/golden/ped_anova_runs.json.xz; with the reference importable, TPE_REGEN_REFERENCE=1 recomputes them:

    TPE_REGEN_REFERENCE=1 python -m pytest tests/test_ped_anova.py -m "not gpu"
"""
from __future__ import annotations

import atexit
import json
import lzma
import math
import os
import warnings

import numpy as np
import pytest

from tests.conftest import HAVE_OPTUNA

from tests._oracle_engine import OracleEngine

pytestmark = pytest.mark.skipif(not HAVE_OPTUNA, reason="optuna (oracle/_ref) is not available")

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ped_anova_runs.json.xz")
_golden: dict | None = None
_fresh: set[str] = set()


def recorded(key: str, compute):
    """The reference's stored result `key`; with TPE_REGEN_REFERENCE=1, `compute()` (a live reference run) replaces
    it and the file is rewritten at exit.  Values are plain JSON (floats round-trip exactly)."""
    global _golden
    if _golden is None:
        _golden = {}
        if os.path.exists(GOLDEN):
            with lzma.open(GOLDEN, "rt") as f:
                _golden = json.load(f)
    if os.environ.get("TPE_REGEN_REFERENCE") == "1" and key not in _fresh:
        if not _fresh:
            atexit.register(_save_golden)
        _golden[key] = json.loads(json.dumps(compute()))
        _fresh.add(key)
    if key not in _golden:
        raise KeyError(f"no stored reference result {key!r} in {GOLDEN} (see the module docstring)")
    return _golden[key]


def _save_golden() -> None:
    raw = json.dumps(_golden, sort_keys=True, separators=(",", ":")).encode()
    with open(GOLDEN, "wb") as f:
        f.write(lzma.compress(raw, preset=9 | lzma.PRESET_EXTREME))


class PedOracleEngine(OracleEngine):
    """The CPU oracle engine answering ``ped_anova`` with oracle/ped_anova.py (the TPEEngine call of the same name)."""

    def ped_anova(self, cols, grids, n_grid, *, target_quantile, region_quantile, evaluate_on_local, loss=None,
                  prior_weight=1.0, min_n_top=2, n_steps=50, counts=False):
        from oracle import ped_anova as ped
        self.calls.append(("ped_anova", len(cols)))
        g = np.asarray(grids, dtype=np.float64).reshape(len(cols), int(n_steps))
        imp, sizes, cnt = ped.ped_anova(self.X, self.cat, self.key, self.params, [int(c) for c in cols], g,
                                        np.asarray(n_grid), target_quantile=target_quantile,
                                        region_quantile=region_quantile, evaluate_on_local=evaluate_on_local,
                                        loss=loss, prior_weight=prior_weight, min_n_top=min_n_top)
        return imp, sizes, (cnt if counts else None)


@pytest.fixture(params=[pytest.param("oracle", id="oracle-engine"),
                        pytest.param("cuda", id="cuda-engine", marks=pytest.mark.gpu)])
def make_evaluator(request, monkeypatch):
    from optuna_b200 import B200PedAnovaImportanceEvaluator
    if request.param == "oracle":
        monkeypatch.setattr(B200PedAnovaImportanceEvaluator, "_engine_cls", PedOracleEngine)
    made = []

    def make(**kw):
        e = B200PedAnovaImportanceEvaluator(**kw)
        made.append(e)
        return e

    make.kind = request.param
    yield make
    for e in made:
        e.close()


# ---- studies ------------------------------------------------------------------------------------------------------
def _dists():
    from optuna.distributions import CategoricalDistribution as Cat
    from optuna.distributions import FloatDistribution as F
    from optuna.distributions import IntDistribution as I
    return {"f": F(-2.0, 3.0), "lf": F(1e-3, 10.0, log=True), "sf": F(0.0, 1.0, step=0.1), "i": I(0, 20),
            "li": I(1, 1000, log=True), "c": Cat(["red", "green", "blue", "cyan"])}


def _params(rs, d):
    from optuna.distributions import CategoricalDistribution, FloatDistribution, IntDistribution
    out = {}
    for name, dist in d.items():
        if isinstance(dist, CategoricalDistribution):
            out[name] = dist.choices[rs.randint(len(dist.choices))]
        elif isinstance(dist, IntDistribution):
            out[name] = int(round(math.exp(rs.uniform(math.log(dist.low), math.log(dist.high))))) if dist.log \
                else int(rs.randint(dist.low, dist.high + 1))
        elif dist.step is not None:
            out[name] = float(round(rs.randint(0, round((dist.high - dist.low) / dist.step) + 1) * dist.step
                                    + dist.low, 10))
        elif dist.log:
            out[name] = float(math.exp(rs.uniform(math.log(dist.low), math.log(dist.high))))
        else:
            out[name] = float(rs.uniform(dist.low, dist.high))
    return out


def _objective(p):
    v = (p.get("f", 0.0) - 0.5) ** 2 + 0.3 * abs(math.log10(p.get("lf", 1.0))) + 2.0 * (p.get("sf", 0.5) - 0.7) ** 2
    v += 0.05 * abs(p.get("i", 10) - 7) + 0.1 * math.log(p.get("li", 10)) + {"red": 0.0, "green": 0.4}.get(
        p.get("c", "red"), 0.8)
    return v


def _add(study, params, dists, value=None, state=None, values=None):
    import optuna
    from optuna.trial import TrialState
    state = TrialState.COMPLETE if state is None else state
    kw = {"params": params, "distributions": {k: dists[k] for k in params}, "state": state}
    if state == TrialState.COMPLETE:
        kw["values" if values is not None else "value"] = values if values is not None else value
    if state == TrialState.PRUNED:
        kw["intermediate_values"] = {0: value}
    study.add_trial(optuna.trial.create_trial(**kw))


def study_kinds(n=300, direction="minimize", seed=0, mixed_states=False):
    import optuna
    from optuna.trial import TrialState
    rs = np.random.RandomState(seed)
    d = _dists()
    study = optuna.create_study(direction=direction)
    for k in range(n):
        p = _params(rs, d)
        v = _objective(p) + 0.01 * rs.rand()
        if mixed_states and k % 7 == 3:
            _add(study, p, d, v, state=TrialState.PRUNED)
        elif mixed_states and k % 11 == 5:
            _add(study, p, d, state=TrialState.FAIL)
        else:
            _add(study, p, d, v)
    if mixed_states:
        for _ in range(3):
            study.enqueue_trial(_params(rs, d))
            study.ask(fixed_distributions=d)     # left RUNNING
    return study


def study_ties():
    """Many losses tie at the cut-offs; -0.0 and 0.0 among them."""
    import optuna
    rs = np.random.RandomState(3)
    d = {k: v for k, v in _dists().items() if k in ("f", "i", "c")}
    study = optuna.create_study()
    for k in range(200):
        _add(study, _params(rs, d), d, [-0.0, 0.0, 1.0, 2.0, 0.0, 3.0][k % 6] if k % 5 else float(rs.randint(4)))
    return study


def study_conditional_dynamic():
    """'cond' only in some trials, 'dyn' with two ranges, 'one' / 'k' / 'z' single-valued."""
    import optuna
    from optuna.distributions import CategoricalDistribution, FloatDistribution, IntDistribution
    rs = np.random.RandomState(5)
    d = {k: v for k, v in _dists().items() if k in ("f", "lf", "c")}
    study = optuna.create_study()
    for k in range(240):
        dk = dict(d, dyn=FloatDistribution(0.0, 1.0 if k < 120 else 2.0), one=FloatDistribution(1.5, 1.5),
                  k=IntDistribution(3, 3), z=CategoricalDistribution(["only"]))
        if k % 3 == 0:
            dk["cond"] = FloatDistribution(-1.0, 1.0)
        p = _params(rs, dk)
        _add(study, p, dk, _objective(p) + p.get("cond", 0.0) ** 2 + 0.2 * p["dyn"])
    return study


def study_multi():
    import optuna
    rs = np.random.RandomState(7)
    d = {k: v for k, v in _dists().items() if k in ("f", "sf", "c")}
    study = optuna.create_study(directions=["minimize", "maximize"])
    for _ in range(150):
        p = _params(rs, d)
        _add(study, p, d, values=[_objective(p), p["f"] * p["sf"]])
    return study


def study_small(n):
    import optuna
    rs = np.random.RandomState(11)
    d = {k: v for k, v in _dists().items() if k in ("f", "c")}
    study = optuna.create_study()
    for _ in range(n):
        p = _params(rs, d)
        _add(study, p, d, _objective(p))
    return study


def study_single_only():
    import optuna
    from optuna.distributions import FloatDistribution, IntDistribution
    d = {"a": FloatDistribution(2.0, 2.0), "b": IntDistribution(1, 1)}
    study = optuna.create_study()
    for k in range(10):
        _add(study, {"a": 2.0, "b": 1}, d, float(k))
    return study


def _target_sq(t):
    return t.params["f"] ** 2


def _target_nonfinite(t):
    k = t.number % 9
    return math.inf if k == 1 else (math.nan if k == 2 else (-math.inf if k == 4 else t.params["f"] - t.params["sf"]))


def _target_first(t):
    return t.values[0]


STUDIES = {"kinds": study_kinds, "max": lambda: study_kinds(250, "maximize", 1),
           "states": lambda: study_kinds(260, seed=2, mixed_states=True), "ties": study_ties,
           "cond": study_conditional_dynamic, "multi": study_multi, "zero": lambda: study_small(0),
           "one": lambda: study_small(1), "two": lambda: study_small(2), "three": lambda: study_small(3),
           "single": study_single_only}
TARGETS = {None: None, "sq": _target_sq, "nonfinite": _target_nonfinite, "first": _target_first}

# (id, study, evaluator kwargs, params, target)
SCENARIOS = [
    ("kinds", "kinds", {}, None, None),
    ("kinds-region05", "kinds", {"region_quantile": 0.5}, None, None),
    ("kinds-global", "kinds", {"evaluate_on_local": False}, None, None),
    ("kinds-global-region05", "kinds", {"evaluate_on_local": False, "region_quantile": 0.5}, None, None),
    ("kinds-q02", "kinds", {"target_quantile": 0.2, "region_quantile": 0.7}, None, None),
    ("kinds-subset", "kinds", {}, ["li", "c", "f"], None),
    ("kinds-target", "kinds", {}, None, "sq"),
    ("kinds-target-region05", "kinds", {"region_quantile": 0.5}, ["f", "i"], "sq"),
    ("kinds-target-nonfinite", "kinds", {}, None, "nonfinite"),
    ("kinds-baseline", "kinds", {"baseline_quantile": 0.2}, None, None),
    ("max", "max", {}, None, None),
    ("max-region05", "max", {"region_quantile": 0.5}, None, None),
    ("states", "states", {}, None, None),
    ("ties", "ties", {}, None, None),
    ("ties-region05", "ties", {"target_quantile": 0.3, "region_quantile": 0.5}, None, None),
    ("cond", "cond", {}, None, None),
    ("cond-params", "cond", {}, ["cond", "f", "one"], None),
    ("cond-dynamic-params", "cond", {}, ["dyn", "f"], None),
    ("cond-missing-param", "cond", {}, ["nope"], None),
    ("cond-params-tuple", "cond", {}, ("f", "c"), None),
    ("cond-params-type", "cond", {}, "f", None),
    ("cond-params-nonstr", "cond", {}, ["f", 1], None),
    ("cond-params-empty", "cond", {}, [], None),
    ("multi-target", "multi", {}, None, "first"),
    ("multi-no-target", "multi", {}, None, None),
    ("zero", "zero", {}, None, None),
    ("one", "one", {}, None, None),
    ("two", "two", {}, None, None),
    ("three-same-set", "three", {"target_quantile": 0.4, "region_quantile": 0.5}, None, None),
    ("three", "three", {}, None, None),
    ("single", "single", {}, None, None),
]


def _run(evaluator, study, params, target):
    """What evaluate reports: ("ok", [[name, importance], ...]) or ("error", type name, message), and the warnings
    (texts, in order) emitted by the constructor call that is already done and by evaluate."""
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        try:
            out = evaluator.evaluate(study, params=params, target=target)
            res = ["ok", [[k, float(v)] for k, v in out.items()]]
        except (ValueError, TypeError, RuntimeError) as e:
            res = ["error", type(e).__name__, str(e)]
    return {"result": res, "warnings": [str(w.message) for w in rec if "experimental" not in str(w.message)]}


def _make_with_warnings(factory, kw):
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        ev = factory(**kw)
    return ev, [str(w.message) for w in rec if "experimental" not in str(w.message)]


def _reference(key, build, kw, params, target):

    def compute():
        from optuna.importance import PedAnovaImportanceEvaluator
        ev, init_w = _make_with_warnings(PedAnovaImportanceEvaluator, kw)
        out = _run(ev, build(), params, target)
        out["init_warnings"] = init_w
        return out
    return recorded(f"{key}", compute)


def _compare(kind, got, want):
    assert got["warnings"] == want["warnings"]
    assert got["result"][0] == want["result"][0], (got["result"], want["result"])
    if got["result"][0] == "error":
        assert got["result"][1:] == want["result"][1:]
        return
    g, w = got["result"][1], want["result"][1]
    assert sorted(k for k, _ in g) == sorted(k for k, _ in w)
    if kind == "oracle":   # the NumPy restatement equals the reference bit for bit
        assert g == w
        return
    tol = 1e-9 * max([abs(v) for _, v in w] + [0.0])
    wd = dict(w)
    for k, v in g:
        assert abs(v - wd[k]) <= tol, (k, v, wd[k])
    # the order agrees wherever two importances differ by more than the tolerance
    pos = {k: i for i, (k, _) in enumerate(g)}
    for i, (a, va) in enumerate(w):
        for b, vb in w[i + 1:]:
            if va - vb > tol:
                assert pos[a] < pos[b], (a, b)


@pytest.mark.parametrize("sid,study,kw,params,target", SCENARIOS, ids=[s[0] for s in SCENARIOS])
def test_matches_reference(make_evaluator, sid, study, kw, params, target):
    want = _reference(sid, STUDIES[study], kw, params, TARGETS[target])
    ev, init_w = _make_with_warnings(make_evaluator, kw)
    assert init_w == want["init_warnings"]
    got = _run(ev, STUDIES[study](), params, TARGETS[target])
    _compare(make_evaluator.kind, got, want)


def test_constructor_checks_quantiles(make_evaluator):
    with pytest.raises(AssertionError, match="target_quantile"):
        make_evaluator(target_quantile=0.5, region_quantile=0.5)


def _incremental_steps():
    """A study that grows by asks and tells, trials finishing out of order, a parameter ('late') first used in trial 40;
    after each change the evaluation the test compares.  Yields (tag, study, params)."""
    import optuna
    rs = np.random.RandomState(13)
    d = {k: v for k, v in _dists().items() if k in ("f", "sf", "c", "i")}
    dl = dict(d, late=optuna.distributions.FloatDistribution(0.0, 4.0))
    study = optuna.create_study()
    running = []
    step = 0
    for k in range(70):
        dk = dl if k >= 40 else d
        study.enqueue_trial(_params(rs, dk))
        running.append(study.ask(fixed_distributions=dk))
        if rs.rand() < 0.6 and len(running) > 1:
            t = running.pop(rs.randint(len(running)))
            if rs.rand() < 0.15:
                study.tell(t, state=optuna.trial.TrialState.PRUNED)
            else:
                study.tell(t, _objective(t.params) + t.params.get("late", 0.0))
            if k >= 8 and k % 3 == 0:
                yield f"s{step}", study, None
                step += 1
                if k >= 45:
                    yield f"s{step}", study, ["late", "f"]
                    step += 1
    for t in running:
        study.tell(t, _objective(t.params))
    yield f"s{step}", study, None
    yield f"s{step + 1}", study, ["late", "c"]
    # the same evaluator moves to another study
    other = study_kinds(120, seed=4)
    yield "other", other, None


def test_incremental_growing_study(make_evaluator):
    ev = make_evaluator()
    for tag, study, params in _incremental_steps():
        def compute(study=study, params=params):
            from optuna.importance import PedAnovaImportanceEvaluator
            return _run(PedAnovaImportanceEvaluator(), study, params, None)
        want = recorded(f"incremental/{tag}", compute)
        _compare(make_evaluator.kind, _run(ev, study, params, None), want)


def test_incremental_uploads_only_changes():
    """Host glue: a second call after one more trial uploads that trial's row, not the history."""
    import optuna
    from optuna_b200 import B200PedAnovaImportanceEvaluator
    ev = B200PedAnovaImportanceEvaluator()
    ev._engine_cls = PedOracleEngine
    study = study_kinds(100)
    ev.evaluate(study)
    calls = ev._engine.calls
    assert [c[0] for c in calls] == ["set_space", "set_history", "ped_anova"]
    rs = np.random.RandomState(1)
    d = _dists()
    p = _params(rs, d)
    _add(study, p, d, _objective(p))
    ev.evaluate(study)
    assert calls[3:] == [("update_history", 1), ("ped_anova", 6)]


# ---- GPU only: bins and importances at scale against the oracle ----------------------------------------------------
def _engine_pair(specs, X, cat, key):
    from optuna_b200 import TPEEngine
    out = []
    for cls in (TPEEngine, PedOracleEngine):
        e = cls(0)
        e.set_space(specs)
        e.set_history(X, cat, key)
        out.append(e)
    return out


def _check_scale(specs, X, cat, key, cols, grids, n_grid, loss=None, **kw):
    cuda, orc = _engine_pair(specs, X, cat, key)
    try:
        for evaluate_on_local, rq in ((True, 1.0), (True, 0.5), (False, 1.0)):
            args = dict(target_quantile=0.1, region_quantile=rq, evaluate_on_local=evaluate_on_local, loss=loss,
                        counts=True, **kw)
            ic, nc, cc = cuda.ped_anova(cols, grids, n_grid, **args)
            io, no, co = orc.ped_anova(cols, grids, n_grid, **args)
            assert nc == no
            np.testing.assert_array_equal(cc, co)
            assert np.max(np.abs(ic - io)) <= 1e-9 * np.max(np.abs(io)), (ic, io)
    finally:
        cuda.close()


@pytest.mark.gpu
def test_counts_and_importances_config2_scale():
    """100k x 32 FloatDistribution(0, 1), loss sum (x - 0.5)^2 (the benchmark's history)."""
    from optuna_b200 import ParamSpec
    from optuna_b200.importance import _grid
    from optuna.distributions import FloatDistribution
    rs = np.random.RandomState(0)
    N, P = 100_000, 32
    X = rs.uniform(0, 1, (N, P))
    key = np.stack([((X - 0.5) ** 2).sum(1), np.zeros(N)], 1)
    cat = np.zeros(N, np.int8)
    cat[rs.rand(N) < 0.02] = 4
    ng, g = _grid(FloatDistribution(0.0, 1.0), 50)
    _check_scale([ParamSpec(kind=0, low=0.0, high=1.0)] * P, X, cat, key, list(range(P)),
                 np.tile(g, (P, 1)), np.full(P, ng))


@pytest.mark.gpu
def test_counts_and_importances_mixed_kinds_scale():
    """Config-3-like mixed kinds (log float, stepped float, int, log int, wide categorical), missing values, a target
    loss with non-finite entries."""
    from optuna_b200 import ParamSpec
    from optuna_b200.importance import _grid
    from optuna.distributions import CategoricalDistribution, FloatDistribution, IntDistribution
    rs = np.random.RandomState(1)
    N = 60_000
    dists = [FloatDistribution(-3.0, 5.0), FloatDistribution(1e-4, 1.0, log=True), FloatDistribution(0.0, 2.0, step=0.25),
             IntDistribution(-5, 40), IntDistribution(1, 4096, log=True), IntDistribution(0, 300, step=3),
             CategoricalDistribution(list(range(7))), CategoricalDistribution([str(i) for i in range(9000)])]
    cols = []
    for d in dists:
        if isinstance(d, CategoricalDistribution):
            cols.append(rs.randint(len(d.choices), size=N).astype(float))
        elif isinstance(d, IntDistribution):
            if d.log:
                cols.append(np.round(np.exp(rs.uniform(0, np.log(d.high), N))))
            else:
                cols.append(d.low + d.step * rs.randint(0, (d.high - d.low) // d.step + 1, N).astype(float))
        elif d.step is not None:
            cols.append(d.low + d.step * rs.randint(0, 9, N))
        elif d.log:
            cols.append(np.exp(rs.uniform(np.log(d.low), np.log(d.high), N)))
        else:
            cols.append(rs.uniform(d.low, d.high, N))
    X = np.stack(cols, 1)
    X[rs.rand(N) < 0.05, 1] = np.nan
    cat = rs.choice([0, 0, 0, 0, 1, 4], size=N).astype(np.int8)
    key = np.stack([rs.rand(N), np.zeros(N)], 1)
    loss = np.round(rs.rand(N) * 50) / 7.0
    loss[rs.rand(N) < 0.03] = np.inf
    specs = []
    for d in dists:
        if isinstance(d, CategoricalDistribution):
            specs.append(ParamSpec(kind=2, n_choices=len(d.choices)))
        else:
            specs.append(ParamSpec(kind=1 if isinstance(d, IntDistribution) else 0, low=float(d.low),
                                   high=float(d.high), step=None if d.step is None else float(d.step), log=d.log))
    grids = np.zeros((len(dists), 50))
    n_grid = np.zeros(len(dists), np.int32)
    for j, d in enumerate(dists):
        n_grid[j], g = _grid(d, 50)
        if g is not None:
            grids[j, : g.size] = g
    _check_scale(specs, X, cat, key, list(range(len(dists))), grids, n_grid, loss=loss)
    _check_scale(specs, X, cat, key, list(range(len(dists))), grids, n_grid)


def test_get_param_importances_normalized(make_evaluator):
    """The public path: optuna.importance.get_param_importances with normalize=True."""
    import optuna
    want = recorded("get_param_importances_normalized", lambda: [
        [k, v] for k, v in optuna.importance.get_param_importances(
            study_kinds(150, seed=9), evaluator=optuna.importance.PedAnovaImportanceEvaluator()).items()])
    got = optuna.importance.get_param_importances(study_kinds(150, seed=9), evaluator=make_evaluator())
    assert [k for k, _ in want] == list(got)
    assert abs(sum(got.values()) - 1.0) < 1e-12
    for k, v in want:
        if make_evaluator.kind == "oracle":
            assert got[k] == v
        else:
            assert abs(got[k] - v) <= 1e-9
