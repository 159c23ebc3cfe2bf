"""B200TPESampler behind the reference's OWN ``Study`` (unmodified optuna, oracle/_ref), compared with what
``optuna.samplers.TPESampler`` computed when driven through the same calls with the same seed (stored in
tests/golden/reference_runs.json.xz, see tests/_reference_golden.py).

Every scenario runs twice: with the CPU oracle answering the array-level calls (checks the host glue -- trial
log, device mirror, search spaces, RNG hand-over -- anywhere) and, marked ``gpu``, with libtpe_b200.so (the
product).  Reference behaviour: optuna/samplers/_tpe/sampler.py:386-560, the conformance suite
optuna/testing/pytest_samplers.py:81-540, boundary cases of SURVEY.md section 8b."""
import math
import pickle
import warnings

import numpy as np
import pytest

optuna = pytest.importorskip("optuna")
from optuna.samplers import TPESampler  # noqa: E402
from optuna.trial import TrialState  # noqa: E402

from tests._reference_golden import recorded, regenerating  # noqa: E402
from tests._util import load  # noqa: E402

warnings.filterwarnings("ignore", category=optuna.exceptions.ExperimentalWarning)


class Tie(Exception):
    """The two samplers picked different candidates whose acquisition values agree to rounding."""


def same(pa, pb, tol=1e-9):
    """Suggested parameter dicts: ints / categorical choices exact, floats to `tol` relative."""
    assert pa.keys() == pb.keys(), (pa, pb)
    for k in pa:
        a, b = pa[k], pb[k]
        if isinstance(b, float):
            assert type(a) is float and abs(a - b) <= tol * max(1.0, abs(b)), (k, a, b)
        else:
            assert type(a) is type(b) and a == b, (k, a, b)


class Audit:
    """Candidates and acquisition values of every device suggestion of a sampler (B200TPESampler._audit)."""

    def __init__(self, sampler):
        self.rec = {}
        sampler._audit = self

    def __call__(self, trial, space, eng):
        smp, ll, lg = eng.get_candidates()
        self.rec[(None if trial is None else trial.number, tuple(space))] = (np.array(smp), np.array(ll) - np.array(lg))


def same_trial(ta, tb, audit):
    """ta (ours) == tb (yardstick), or -- Tie -- ours is a different candidate of the same ask whose acquisition
    value equals the maximum to rounding: `argmax` over values that agree to ~1 ulp is decided by the summation
    order of the log-sum-exp (NumPy's pairwise sum vs the kernels' tiles), mostly two categorical choices with
    the same observation counts.  Anything else is a failure."""
    try:
        same(ta.params, tb.params)
        return
    except AssertionError:
        if audit is None:
            raise
        for (number, names), (smp, acq) in audit.rec.items():
            if number != ta.number or not all(n in tb.params for n in names):
                continue
            want = np.asarray([ta.distributions[n].to_internal_repr(tb.params[n]) for n in names], dtype=float)
            mine = np.asarray([ta.distributions[n].to_internal_repr(ta.params[n]) for n in names], dtype=float)
            if np.allclose(want, mine, rtol=1e-9, atol=0):
                continue  # this ask agrees; the difference is in another one
            hit = np.all(np.abs(smp - want) <= 1e-9 * np.maximum(1.0, np.abs(want)), axis=1)
            if hit.any() and acq[hit].max() >= np.nanmax(acq) - 1e-9:
                raise Tie(f"trial {ta.number} {names}: {ta.params} vs {tb.params}")
        raise


def same_trials(a, b, audit=None):
    assert len(a.trials) == len(b.trials)
    for ta, tb in zip(a.trials, b.trials):
        assert ta.state == tb.state
        same_trial(ta, tb, audit)


def over_seeds(scenario, make_sampler, ties, kw, seeds=(0, 1, 2, 3, 4, 5)):
    """Run `scenario(sampler) -> study` for our sampler and the yardstick, seed after seed, until a seed goes
    through without an acquisition tie; a difference that is not such a tie fails at once.  With the CPU oracle
    as the engine no tie is tolerated: glue + oracle must BE the reference."""
    base = kw.pop("seed", 0)
    run = next(make_sampler.runs)
    if regenerating():  # store the reference's run of every seed: the CUDA engine may need a later one
        for seed in seeds:
            make_sampler.yardstick(f"{run}/{base + seed}", scenario, ties, seed=base + seed, **kw)
    tied = []
    for seed in seeds:
        mine = make_sampler(seed=base + seed, **kw)
        audit = Audit(mine) if make_sampler.kind == "cuda" else None
        a = scenario(mine)
        b = make_sampler.yardstick(f"{run}/{base + seed}", scenario, ties, seed=base + seed, **kw)
        try:
            same_trials(a, b, audit)
            return a, b
        except Tie as t:
            tied.append(str(t))
    pytest.fail("every seed ran into an acquisition tie: " + "; ".join(tied))


def run_both(make_sampler, objective, n_trials, study_kw=None, ties=False, **kw):
    """study.optimize on both samplers; returns (ours, yardstick) studies after comparing every trial.
    ties: the scenario repeats numeric observations (see conftest.make_sampler.reference)."""
    study_kw = study_kw or {}

    def scenario(sampler):
        s = optuna.create_study(sampler=sampler, **study_kw)
        s.optimize(objective, n_trials=n_trials)
        return s

    return over_seeds(scenario, make_sampler, ties, kw)


def branin(t):
    x = t.suggest_float("x", -5, 10)
    y = t.suggest_float("y", 0, 15)
    return ((y - 5.1 / (4 * math.pi**2) * x * x + 5 / math.pi * x - 6) ** 2
            + 10 * (1 - 1 / (8 * math.pi)) * math.cos(x) + 10)


def mixed(t):
    a = t.suggest_float("a", -1.0, 1.0)
    b = t.suggest_float("b", 1e-3, 10.0, log=True)
    c = t.suggest_float("c", 0.0, 2.0, step=0.25)
    d = t.suggest_int("d", -3, 7)
    e = t.suggest_int("e", 1, 64, log=True)
    f = t.suggest_int("f", 0, 30, step=5)
    g = t.suggest_categorical("g", ["p", "q", None, 3])
    assert type(a) is float and type(b) is float and type(c) is float
    assert type(d) is int and type(e) is int and type(f) is int
    v = a * a + math.log(b) ** 2 + c + d * 0.1 + abs(e - 8) * 0.05 + f * 0.01 + (g == "p")
    if t.number % 7 == 3:
        t.report(v, 1)
        t.report(v * 0.9, 3)
        raise optuna.TrialPruned()
    return v


@pytest.mark.parametrize("mv", [False, True])
def test_branin_200_trials_is_the_reference_trajectory(make_sampler, mv):
    """BASELINE config 1: same seed => same 200-trial trajectory as optuna.samplers.TPESampler (the committed
    golden tests/golden/branin.npz, generated from the reference by oracle/gen_golden.py)."""
    study = optuna.create_study(sampler=make_sampler(seed=0, multivariate=mv))
    study.optimize(branin, n_trials=200)
    g = load("branin.npz")
    ref = g[f"branin_{'mv' if mv else 'uni'}/xy"]
    xy = np.asarray([[t.params["x"], t.params["y"]] for t in study.trials])
    assert np.array_equal(xy[:10], ref[:10])  # startup trials: RandomSampler's stream, bit-identical
    np.testing.assert_allclose(xy, ref, rtol=1e-9, atol=1e-9)
    # ... computed ahead: the joint suggestion / the batch of per-parameter suggestions is queued when a trial is told
    assert study.sampler.ahead_stats[0] >= 180, study.sampler.ahead_stats
    if not mv:
        assert abs(study.best_value - 0.4069652013131506) < 1e-9


@pytest.mark.parametrize("mv", [False, True])
@pytest.mark.parametrize("direction", ["minimize", "maximize"])
def test_mixed_space_with_pruned_trials(make_sampler, mv, direction):
    run_both(make_sampler, mixed, 45, {"direction": direction}, ties=True, seed=3, multivariate=mv, n_startup_trials=5)


def test_custom_gamma_weights_and_constraints(make_sampler):
    def obj(t):
        x = t.suggest_float("x", -3, 3)
        k = t.suggest_int("k", 0, 4)
        t.set_user_attr("c", x - 1.0)
        if t.number % 5 == 4:
            t.report(abs(x), 1)
            raise optuna.TrialPruned()
        return x * x + k

    kw = dict(seed=1, gamma=lambda n: max(1, n // 4), weights=lambda n: np.arange(1, n + 1) ** 0.5,
              constraints_func=lambda tr: (tr.user_attrs["c"], -1.0), n_startup_trials=5)
    a, b = run_both(make_sampler, obj, 40, ties=True, **kw)
    for ta, tb in zip(a.trials, b.trials):  # constraints are stored once, by after_trial (samplers/_base.py:242-268)
        np.testing.assert_allclose(ta.system_attrs["constraints"], tb.system_attrs["constraints"], rtol=1e-9)
    # joint sampling: the suggestions are queued at `tell` time also with constraints and custom weights (the
    # constraints of the trial being told are read back from the storage, the weights evaluated then)
    a, b = run_both(make_sampler, obj, 40, ties=True, multivariate=True, **dict(kw, seed=3))
    assert a.sampler.ahead_stats[0] >= 25, a.sampler.ahead_stats
    for ta, tb in zip(a.trials, b.trials):
        np.testing.assert_allclose(ta.system_attrs["constraints"], tb.system_attrs["constraints"], rtol=1e-9)
    with pytest.raises(ValueError):
        bad = optuna.create_study(sampler=make_sampler(seed=1, weights=lambda n: -np.ones(n), n_startup_trials=2))
        bad.optimize(lambda t: t.suggest_float("x", 0, 1), n_trials=5)
    with pytest.raises(ValueError):  # samplers/_base.py:253-254
        nan = optuna.create_study(sampler=make_sampler(seed=1, constraints_func=lambda tr: (float("nan"),)))
        nan.optimize(lambda t: t.suggest_float("x", 0, 1), n_trials=2)


def test_hyperopt_parameters_and_endpoints(make_sampler):
    from optuna_b200.sampler import B200TPESampler
    assert B200TPESampler.hyperopt_parameters().keys() == TPESampler.hyperopt_parameters().keys()
    kw = dict(TPESampler.hyperopt_parameters(), seed=9, consider_endpoints=True, consider_magic_clip=False,
              prior_weight=0.5)
    # hyperopt_parameters() of the reference holds the reference's gamma / weights functions: equally valid here
    run_both(make_sampler, mixed, 50, ties=True, **kw)


def test_constant_liar_batches_out_of_order_tells_and_failures(make_sampler):
    """constant_liar=True (sampler.py:435-443, :493-509, :526-535): RUNNING trials -- their relative parameters
    relayed through system attrs -- sit in g(x); tells arrive out of order; a trial fails."""
    def obj(t):
        x = t.suggest_float("x", -2, 2)
        k = t.suggest_int("k", 0, 6)
        c = t.suggest_categorical("c", ["u", "v", "w"])
        return x * x + (k - 3) ** 2 + (c == "v")

    def scenario(sampler):
        s = optuna.create_study(sampler=sampler)
        s.optimize(obj, n_trials=10)
        pending = [s.ask() for _ in range(5)]
        vals = [obj(t) for t in pending]
        s.tell(pending[3], vals[3])                        # out of order
        s.tell(pending[1], state=TrialState.FAIL)          # never counts
        more = [s.ask() for _ in range(3)]
        mv = [obj(t) for t in more]
        s.tell(pending[0], vals[0])
        last = [s.ask() for _ in range(2)]
        lv = [obj(t) for t in last]
        for t, v in zip([pending[2], pending[4]] + more + last, [vals[2], vals[4]] + mv + lv):
            s.tell(t, v)
        assert any("tpe:relative_params:0" in t.system_attrs for t in s.trials[10:]) == sampler._multivariate
        return s

    for mv in (True, False):
        a, _ = over_seeds(scenario, make_sampler, True, dict(seed=5, multivariate=mv, constant_liar=True, n_startup_trials=5))
        assert len(a.trials) == 20 and len({tuple(sorted(t.params.items())) for t in a.trials[10:]}) > 5


def test_group_decomposed_conditional_space(make_sampler):
    """group=True (sampler.py:394-405, :417-431; search_space/group_decomposed.py:14-68)."""
    def obj(t):
        kind = t.suggest_categorical("kind", ["a", "b"])
        x = t.suggest_float("x", -1, 1)
        if kind == "a":
            return x * x + t.suggest_float("ya", 0, 2)
        return x * x + (t.suggest_int("yb", 0, 5) - 2) ** 2 + t.suggest_float("zb", 1e-2, 1, log=True)

    a, b = run_both(make_sampler, obj, 50, seed=4, multivariate=True, group=True, n_startup_trials=6)
    names = sorted(sorted(g) for g in a.sampler._groups_now)
    assert names == [["kind", "x"], ["ya"], ["yb", "zb"]]
    assert [sorted(g) for g in a.sampler._groups_now] == b.groups
    from optuna_b200 import B200TPESampler
    with pytest.raises(ValueError):
        B200TPESampler(group=True)


def test_conditional_space_without_group_warns_and_matches(make_sampler):
    def obj(t):
        kind = t.suggest_categorical("kind", ["a", "b"])
        x = t.suggest_float("x", -1, 1)
        y = t.suggest_float("ya", 0, 2) if kind == "a" else t.suggest_int("yb", 0, 5)
        return x * x + y

    run_both(make_sampler, obj, 40, seed=8, multivariate=True, n_startup_trials=6)
    run_both(make_sampler, obj, 40, ties=True, seed=8, multivariate=False, n_startup_trials=6)

    # a multivariate sampler's independent parameters use multivariate bandwidths (sampler.py:335-341, :491), also
    # when two or more of them are asked in the same order in every trial
    def obj2(t):
        hi = 4.0 if t.number == 0 else 3.0   # trial 0 keeps x and y out of the intersection search space
        x = t.suggest_float("x", -3.0, hi)
        y = t.suggest_float("y", -3.0, hi)
        return (x - 1) ** 2 + (y + 0.5) ** 2

    run_both(make_sampler, obj2, 30, seed=3, multivariate=True, n_startup_trials=5)


def test_categorical_distance_func(make_sampler):
    def obj(t):
        a = t.suggest_categorical("a", [0, 1, 2, 3])
        x = t.suggest_float("x", -2, 2)
        return (a - 2) ** 2 + x * x

    run_both(make_sampler, obj, 35, seed=2, multivariate=True, n_startup_trials=4,
             categorical_distance_func={"a": lambda p, q: abs(p - q)})


@pytest.mark.parametrize("n_obj", [2, 3, 4])
def test_motpe_through_the_study(make_sampler, n_obj):
    """MOTPE (sampler.py:745-779, :824-863) with mixed directions; univariate and multivariate."""
    cs = [0.2, 0.4, 0.6, 0.8][:n_obj]
    dirs = ["minimize", "maximize", "minimize", "minimize"][:n_obj]

    def obj(t):
        xs = [t.suggest_float(f"x{j}", 0, 1) for j in range(3)]
        out = [sum((x - c) ** 2 for x in xs) for c in cs]
        out[1] = -out[1] if n_obj > 1 else out[1]
        return out

    for mv in (False, True):
        run_both(make_sampler, obj, 40, {"directions": dirs}, seed=5, multivariate=mv)


def test_motpe_with_conditional_parameters_and_constraints(make_sampler):
    """Multi-objective + a parameter only some trials have + constraints: the hypervolume weights are computed over
    ALL below trials and the trials lacking the parameter drop out afterwards (weights_below[param_mask_below],
    sampler.py:570-576); infeasible below trials weigh EPS (:829-833)."""
    def obj(t):
        x = t.suggest_float("x", 0, 1)
        y = t.suggest_float("y", 0, 1) if x > 0.4 else 0.5
        t.set_user_attr("c", x + y - 1.4)
        return (x - 0.2) ** 2 + (y - 0.7) ** 2, (x - 0.8) ** 2 + (y - 0.3) ** 2

    for mv in (False, True):
        run_both(make_sampler, obj, 45, {"directions": ["minimize", "minimize"]}, seed=3, multivariate=mv,
                 n_startup_trials=8, constraints_func=lambda tr: (tr.user_attrs["c"],))
    # a custom gamma puts most trials below: far more than the 25 of the default
    run_both(make_sampler, obj, 90, {"directions": ["minimize", "minimize"]}, seed=4, multivariate=True,
             n_startup_trials=8, gamma=lambda n: (3 * n) // 4)


def test_dynamic_range_and_single_distributions(make_sampler):
    """pytest_samplers.py:243-345: a parameter whose range changes between trials (independent sampling) and
    distributions holding a single value."""
    def obj(t):
        hi = 5 + t.number % 3
        x = t.suggest_int("x", -hi, hi)
        s = t.suggest_float("s", 1.0, 1.0)
        c = t.suggest_categorical("c", ["only"])
        return x * x + s + (c == "only")

    for mv in (False, True):
        run_both(make_sampler, obj, 30, ties=True, seed=6, multivariate=mv, n_startup_trials=4)


def test_enqueued_added_and_failed_trials(make_sampler):
    """WAITING trials (study.enqueue_trial), trials added from outside (study.add_trials) and exceptions in the
    objective: rows nobody may see yet / ever must not disturb the log."""
    def obj(t):
        x = t.suggest_float("x", -3, 3)
        y = t.suggest_int("y", 0, 9)
        if t.number % 6 == 5:
            raise RuntimeError("boom")
        return (x - 1) ** 2 + y

    def scenario(sampler):
        s = optuna.create_study(sampler=sampler)
        s.optimize(obj, n_trials=12, catch=(RuntimeError,))
        s.enqueue_trial({"x": 0.5, "y": 3})
        s.enqueue_trial({"x": -0.5})
        s.optimize(obj, n_trials=6, catch=(RuntimeError,))
        dist = {"x": optuna.distributions.FloatDistribution(-3, 3), "y": optuna.distributions.IntDistribution(0, 9)}
        s.add_trials([optuna.trial.create_trial(value=float(i), params={"x": 0.1 * i, "y": i}, distributions=dist)
                      for i in range(4)])
        s.optimize(obj, n_trials=10, catch=(RuntimeError,))
        return s

    for mv in (False, True):
        a, b = over_seeds(scenario, make_sampler, True, dict(seed=12, multivariate=mv, n_startup_trials=5))
        assert [t.state for t in a.trials] == [t.state for t in b.trials]


def test_partial_fixed_sampler_and_hyperband_wrapper(make_sampler):
    """PartialFixedSampler hands sample_relative a subset of the inferred space (_partial_fixed.py:65-84);
    HyperbandPruner hands the sampler a _BracketStudy that whitelists a few attributes
    (pruners/_hyperband.py:273-324) -- a fresh wrapper per call."""
    def obj(t):
        x = t.suggest_float("x", -2, 2)
        y = t.suggest_float("y", -2, 2)
        for step in range(4):
            t.report((x * x + y * y) * (1 + 0.1 * (3 - step)), step)
            if t.should_prune():
                raise optuna.TrialPruned()
        return x * x + y * y

    def scenario(base):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            fixed = optuna.samplers.PartialFixedSampler({"y": 0.25}, base)
        s = optuna.create_study(sampler=fixed, pruner=optuna.pruners.HyperbandPruner(min_resource=1, max_resource=4),
                                study_name="hb")
        s.optimize(obj, n_trials=40)
        return s

    for mv in (False, True):
        a, b = over_seeds(scenario, make_sampler, False, dict(seed=21, multivariate=mv, n_startup_trials=5))
        assert all(t.params.get("y", 0.25) == 0.25 for t in a.trials)


def test_one_sampler_shared_by_n_jobs_threads(make_sampler):
    """study/_optimize.py:87-121: one sampler object, n_jobs threads; reseed_rng per thread (:142-143)."""
    s = optuna.create_study(sampler=make_sampler(seed=2, multivariate=True, n_startup_trials=8))
    s.optimize(mixed, n_trials=60, n_jobs=4)
    done = [t for t in s.trials if t.state in (TrialState.COMPLETE, TrialState.PRUNED)]
    assert len(s.trials) == 60 and len(done) == 60
    h = s.sampler._hist
    s.sampler.sample_independent(s, optuna.trial.create_trial(value=0.0), "a", optuna.distributions.FloatDistribution(-1.0, 1.0))
    assert h.n_finished == 60 and not [r for r in h.pending if h.pending[r][1].state.is_finished()]


def test_pickled_study_and_sampler_continue_identically(make_sampler):
    """study/study.py:99-107: a study pickles with its sampler; the device state is a cache."""
    def obj(t):
        return (t.suggest_float("x", 0, 1) - 0.3) ** 2 + t.suggest_int("k", 0, 5) * 0.01

    engine_cls = type(make_sampler(seed=0))._engine_cls

    def scenario(sampler):
        s = optuna.create_study(sampler=sampler)
        s.optimize(obj, n_trials=20)
        if hasattr(sampler, "_engine_cls"):  # ours: continue in a pickled copy of the whole study
            audit, sampler._audit = sampler._audit, None
            clone = pickle.loads(pickle.dumps(s))
            assert clone.sampler._engine is None
            clone.sampler._engine_cls = sampler._engine_cls if "_engine_cls" in sampler.__dict__ else engine_cls
            clone.sampler._audit = sampler._audit = audit
            s.optimize(obj, n_trials=10)
            clone.optimize(obj, n_trials=10)
            assert [t.params for t in s.trials] == [t.params for t in clone.trials]
            clone.sampler.close()
            return s
        s.optimize(obj, n_trials=10)
        return s

    over_seeds(scenario, make_sampler, True, dict(seed=11))


def test_sync_cost_is_proportional_to_the_changes(make_sampler):
    """SURVEY.md 8f rank 1: per ask the history mirror receives the rows that changed, not the history."""
    if make_sampler.kind != "oracle":
        pytest.skip("call log of the stand-in engine")
    s = optuna.create_study(sampler=make_sampler(seed=0, multivariate=True, n_startup_trials=5))
    s.optimize(branin, n_trials=40)
    calls = s.sampler._engine.calls
    assert [c[0] for c in calls].count("set_history") == 1
    ups = [c[1] for c in calls if c[0] == "update_history"]
    # one row per trial: uploaded at `tell` time together with the look-ahead suggestion (the placeholder of the
    # running trial never travels on its own)
    # ... or two: the row goes up with the worst possible key when the trial's suggestion has been handed out (the
    # next suggestion is queued then, on the assumption that the trial will not enter the below set) and gets its
    # true key at `tell` time
    assert 40 - 5 <= len(ups) <= 3 * (40 - 5) + 1 and max(ups) <= 2, ups   # (three when the assumption fails)
    assert s.sampler.ahead_stats[0] >= 40 - 5 - 2, s.sampler.ahead_stats
    assert sum(s.sampler.spec_stats) >= 25 and s.sampler.spec_stats[0] >= 10, s.sampler.spec_stats
    eng = s.sampler._engine
    X, cat, key, _ = s.sampler._rows(s, s.get_trials(deepcopy=False), list(s.sampler._hist.columns),
                                     s.sampler._hist.dists, None)
    n = eng.history_size
    assert n >= 39 and np.array_equal(eng.cat[:39], cat[:39]) and np.array_equal(eng.key[:39], key[:39])
    assert np.array_equal(np.nan_to_num(eng.X[:39], nan=-7.0), np.nan_to_num(X[:39], nan=-7.0))


def test_look_ahead_suggestions_are_the_reference_suggestions(make_sampler):
    """B200TPESampler queues the next joint suggestion at `tell` time (after_trial knows the trial's final state
    before the storage does, study/_tell.py:163-169) and `sample_relative` collects it -- if and only if the ask is
    the predicted one.  One scenario walks through what can come between a tell and the next ask: nothing (served),
    a foreign draw from the sampler's generator, a second tell, asks without tells, a trial told to the sampler but
    never stored, a pruned and a failed trial, a trial with fewer parameters (the search space shrinks), and the
    MAXIMIZE direction; C is chosen so that the generator lives on the device for one half of the seeds' asks."""
    from optuna.trial import TrialState as TS

    def obj_params(t, small=False):
        x = t.suggest_float("x", -2.0, 2.0)
        k = t.suggest_int("k", 0, 6)
        if small:
            return -(x * x) - 0.1 * k
        y = t.suggest_float("y", 1e-2, 10.0, log=True)
        c = t.suggest_categorical("c", ["a", "b", "c"])
        return -(x * x) - 0.1 * k - math.log(y) ** 2 - (c == "b")

    served = []

    def scenario(sampler):
        s = optuna.create_study(sampler=sampler, direction="maximize")
        for _ in range(12):                               # startup + plain sequential loop
            t = s.ask()
            s.tell(t, obj_params(t))
        sampler._rng.rng.random_sample(5)                 # somebody else draws between a tell and the ask
        t = s.ask()
        s.tell(t, obj_params(t))
        t1, t2 = s.ask(), s.ask()                         # asks without tells, then two tells in a row
        v1, v2 = obj_params(t1), obj_params(t2)
        s.tell(t2, v2)
        s.tell(t1, v1)
        t = s.ask()
        obj_params(t)
        frozen = s._storage.get_trial(t._trial_id)
        sampler.after_trial(s, frozen, TS.COMPLETE, [123.0])   # told to the sampler, never stored (still RUNNING)
        u = s.ask()
        s.tell(u, obj_params(u))
        s.tell(t, state=TS.FAIL)
        t = s.ask()
        obj_params(t)
        t.report(0.5, 0)
        t.report(-0.25, 2)
        s.tell(t, state=TS.PRUNED)
        for _ in range(3):
            t = s.ask()
            s.tell(t, obj_params(t))
        t = s.ask()
        s.tell(t, obj_params(t, small=True))              # the intersection search space shrinks
        for _ in range(4):
            t = s.ask()
            s.tell(t, obj_params(t))
        if hasattr(sampler, "ahead_stats"):
            served.append(tuple(sampler.ahead_stats))
            specs.append(tuple(sampler.spec_stats))
        return s

    specs = []
    for C in (24, 2048):   # uniforms drawn on the host / on the device (>= DEVICE_RNG_MIN with 4 parameters)
        over_seeds(scenario, make_sampler, True, dict(seed=31, multivariate=True, n_startup_trials=6, n_ei_candidates=C))
    assert served and all(ok >= 8 and dropped >= 4 for ok, dropped in served), served
    # the suggestion after next is queued as soon as a suggestion has been handed out, on the assumption that the
    # trial will not enter the below set: kept when the value confirms it, recomputed at `tell` time when not (a good
    # value, a pruned or failed trial, a trial with other parameters, a tell that never came)
    assert all(kept >= 3 and dropped >= 3 for kept, dropped in specs), specs
    # univariate TPE: the batch of per-parameter suggestions of the next trial is queued at `tell` time (the CUDA
    # engine does so for all-continuous trials only; this scenario then simply plans at the first ask)
    del served[:]
    for C in (24, 1024):
        over_seeds(scenario, make_sampler, True, dict(seed=47, multivariate=False, n_startup_trials=6, n_ei_candidates=C))
    if make_sampler.kind == "oracle":
        assert served and all(ok >= 6 for ok, _ in served), served


def test_univariate_look_ahead_with_continuous_parameters(make_sampler):
    """All-continuous univariate trials (what the CUDA engine evaluates stage by stage and can queue at `tell` time):
    sequential loop, a foreign draw, two tells in a row, a trial told but never stored, a pruned trial, a trial that
    asks its parameters in another order, one that asks fewer -- against the reference sampler, with host-drawn and
    device-generated uniforms."""
    from optuna.trial import TrialState as TS

    def ask3(t, order=("x", "y", "z")):
        d = {"x": lambda: t.suggest_float("x", -2.0, 2.0), "y": lambda: t.suggest_float("y", 1e-2, 10.0, log=True),
             "z": lambda: t.suggest_float("z", 0.0, 1.0)}
        v = {k: d[k]() for k in order}
        return v.get("x", 0.0) ** 2 + math.log(v.get("y", 1.0)) ** 2 + (v.get("z", 0.3) - 0.3) ** 2

    stats = []

    def scenario(sampler):
        s = optuna.create_study(sampler=sampler)
        for _ in range(12):
            t = s.ask()
            s.tell(t, ask3(t))
        sampler._rng.rng.random_sample(3)
        t = s.ask()
        s.tell(t, ask3(t))
        t1, t2 = s.ask(), s.ask()
        v1, v2 = ask3(t1), ask3(t2)
        s.tell(t2, v2)
        s.tell(t1, v1)
        t = s.ask()
        ask3(t)
        sampler.after_trial(s, s._storage.get_trial(t._trial_id), TS.COMPLETE, [0.001])   # never stored
        u = s.ask()
        s.tell(u, ask3(u))
        s.tell(t, state=TS.FAIL)
        t = s.ask()
        ask3(t)
        t.report(0.5, 0)
        s.tell(t, state=TS.PRUNED)
        for _ in range(3):
            t = s.ask()
            s.tell(t, ask3(t))
        t = s.ask()
        s.tell(t, ask3(t, ("z", "x", "y")))                 # another order: the prediction fails at the first call
        t = s.ask()
        s.tell(t, ask3(t, ("z", "x", "y")))
        t = s.ask()
        s.tell(t, ask3(t, ("z", "x")))                      # fewer calls than predicted: the generator is settled
        for _ in range(4):
            t = s.ask()
            s.tell(t, ask3(t))
        if hasattr(sampler, "ahead_stats"):
            stats.append(tuple(sampler.ahead_stats))
        return s

    for C in (24, 1024):   # 3 x 2 x 1024 uniforms >= DEVICE_RNG_MIN: generated on the device
        over_seeds(scenario, make_sampler, True, dict(seed=5, multivariate=False, n_startup_trials=6, n_ei_candidates=C))
    assert stats and all(ok >= 10 and dropped >= 3 for ok, dropped in stats), stats


@pytest.mark.parametrize("mv", [True, False])
@pytest.mark.parametrize("events", [0, 1, 2, 5])
def test_random_event_sequences_match_the_reference(make_sampler, mv, events):
    """A random walk through what a caller can do between suggestions -- plain trials, batches of asks told in any
    order, failed and pruned trials, values that enter the below set, trials with fewer parameters, foreign draws
    from the sampler's generator, reseeding -- executed identically behind our sampler and the reference's.  Every
    suggestion computed ahead of its ask (look-ahead, outcome speculation, univariate plans) must be dropped or kept
    exactly when the reference's sequential computation says so."""
    from optuna.trial import TrialState as TS

    def run_trial(s, t, ev, short=False):
        x = t.suggest_float("x", -2.0, 2.0)
        y = t.suggest_float("y", 1e-2, 10.0, log=True)
        v = x * x + math.log(y) ** 2
        if not short:
            z = t.suggest_float("z", 0.0, 1.0)
            v += (z - 0.3) ** 2
        return v + 0.05 * ev.standard_normal()

    def scenario(sampler):
        ev = np.random.RandomState(1000 + events)          # the caller's own randomness: the same for both samplers
        sign = -1.0 if events % 2 else 1.0                  # odd event seeds: a study that maximises
        s = optuna.create_study(sampler=sampler, direction="maximize" if events % 2 else "minimize")
        tell = s.tell
        s.tell = lambda t, v=None, state=None: tell(t, None if v is None else sign * v, state=state)
        for _ in range(45):
            op = ev.choice(["trial", "trial", "trial", "trial", "batch", "fail", "prune", "good", "short", "draw"])
            if op == "trial":
                t = s.ask()
                s.tell(t, run_trial(s, t, ev))
            elif op == "batch":
                ts = [s.ask() for _ in range(int(ev.randint(2, 4)))]
                vs = [run_trial(s, t, ev) for t in ts]
                for i in ev.permutation(len(ts)):
                    s.tell(ts[i], vs[i])
            elif op == "fail":
                t = s.ask()
                run_trial(s, t, ev)
                s.tell(t, state=TS.FAIL)
            elif op == "prune":
                t = s.ask()
                v = run_trial(s, t, ev)
                t.report(v, 0)
                t.report(v * 0.9, 1)
                s.tell(t, state=TS.PRUNED)
            elif op == "good":
                t = s.ask()
                run_trial(s, t, ev)
                s.tell(t, -1.0 - ev.uniform())             # better than anything: enters the below set
            elif op == "short":
                t = s.ask()
                s.tell(t, run_trial(s, t, ev, short=True))
            else:
                sampler._rng.rng.random_sample(int(ev.randint(1, 7)))
        return s

    a, b = over_seeds(scenario, make_sampler, True, dict(seed=77 + events, multivariate=mv, n_startup_trials=5))
    assert [t.state for t in a.trials] == [t.state for t in b.trials]
    if mv:   # (univariate: a parameter absent from some trials switches the batched plans off for good)
        assert sum(a.sampler.ahead_stats) >= 10, (a.sampler.ahead_stats, a.sampler.spec_stats)


@pytest.mark.parametrize("kind", ["two_objectives", "constraints", "custom_gamma_weights", "endpoints_no_clip"])
@pytest.mark.parametrize("events", [3, 4])
def test_random_event_sequences_with_other_sampler_options(make_sampler, kind, events):
    """The random walk of test_random_event_sequences_match_the_reference (joint sampling) with the options that change
    what a suggestion computed ahead must respect: two objectives (look-ahead without outcome speculation, hypervolume
    weights), constraints (read back from the storage at `tell` time), a custom gamma that grows the below set and
    custom weights, endpoints without the magic clip.  Host glue only (the CPU oracle answers the engine calls)."""
    if make_sampler.kind != "oracle":
        pytest.skip("host-glue walk: the CPU oracle is the engine")
    from optuna.trial import TrialState as TS
    kw = dict(seed=300 + events, multivariate=True, n_startup_trials=5)
    study_kw = {}
    if kind == "two_objectives":
        study_kw["directions"] = ["minimize", "maximize"]
    elif kind == "constraints":
        kw["constraints_func"] = lambda tr: (tr.params["x"] - 1.0, -0.5)
    elif kind == "custom_gamma_weights":
        kw.update(gamma=lambda n: max(1, n // 3), weights=lambda n: np.linspace(0.2, 1.0, n) if n else np.asarray([]))
    else:
        kw.update(consider_endpoints=True, consider_magic_clip=False, prior_weight=0.3)

    def value(x, y, z, ev):
        v = x * x + math.log(y) ** 2 + (z - 0.3) ** 2 + 0.05 * ev.standard_normal()
        return [v, -abs(x) + z] if kind == "two_objectives" else v

    def run_trial(t, ev):
        return value(t.suggest_float("x", -2.0, 2.0), t.suggest_float("y", 1e-2, 10.0, log=True),
                     t.suggest_float("z", 0.0, 1.0), ev)

    def scenario(sampler):
        ev = np.random.RandomState(2000 + events)
        s = optuna.create_study(sampler=sampler, **study_kw)
        for _ in range(40):
            op = ev.choice(["trial", "trial", "trial", "batch", "fail", "good", "draw"] +
                           ([] if kind == "two_objectives" else ["prune"]))
            if op == "trial":
                t = s.ask()
                s.tell(t, run_trial(t, ev))
            elif op == "batch":
                ts = [s.ask() for _ in range(int(ev.randint(2, 4)))]
                vs = [run_trial(t, ev) for t in ts]
                for i in ev.permutation(len(ts)):
                    s.tell(ts[i], vs[i])
            elif op == "fail":
                t = s.ask()
                run_trial(t, ev)
                s.tell(t, state=TS.FAIL)
            elif op == "prune":
                t = s.ask()
                v = run_trial(t, ev)
                t.report(v, 0)
                s.tell(t, state=TS.PRUNED)
            elif op == "good":
                t = s.ask()
                run_trial(t, ev)
                g = -1.0 - ev.uniform()
                s.tell(t, [g, 3.0] if kind == "two_objectives" else g)
            else:
                sampler._rng.rng.random_sample(int(ev.randint(1, 7)))
        return s

    a, b = over_seeds(scenario, make_sampler, True, kw)
    assert [t.state for t in a.trials] == [t.state for t in b.trials]
    assert sum(a.sampler.ahead_stats) >= 8, (a.sampler.ahead_stats, a.sampler.spec_stats)


def test_batched_ask_equals_sequential_asks(make_sampler):
    """BASELINE config 5 semantics: ask_batch(n) == n sequential study.ask() with no tell between."""
    from optuna_b200.batch import ask_batch

    def obj(t):
        return sum((t.suggest_float(f"x{j}", 0, 1) - 0.3) ** 2 for j in range(5)) + t.suggest_int("k", 0, 9) * 0.01

    def warm(sampler):
        s = optuna.create_study(sampler=sampler)
        s.optimize(obj, n_trials=30)
        return s

    def params(trials):
        return [[t.suggest_float(f"x{j}", 0, 1) for j in range(5)] + [t.suggest_int("k", 0, 9)] for t in trials]

    def sequential():
        b = warm(make_sampler.reference(**kw))
        return params([b.ask() for _ in range(50)])

    kw = dict(seed=7, multivariate=True, n_ei_candidates=32)
    pa = params(ask_batch(warm(make_sampler(**kw)), 50))
    pb = recorded("test_batched_ask_equals_sequential_asks/sequential", sequential)
    np.testing.assert_allclose(pa, pb, rtol=1e-9, atol=0)
    assert len({tuple(p) for p in pa}) > 40  # different uniforms per ask


def test_device_generated_uniforms_give_the_reference_suggestions(make_sampler):
    """Asks large enough for the device MT19937 (>= DEVICE_RNG_MIN uniforms): consecutive asks, a foreign draw in
    between and close() must all reproduce what the reference computes from its host RandomState."""
    from optuna_b200 import B200TPESampler
    P, C, n = 16, 1024, 300
    assert C * (1 + P) >= B200TPESampler.DEVICE_RNG_MIN
    rs = np.random.RandomState(2)
    space = {f"x{j:02d}": optuna.distributions.FloatDistribution(0.0, 1.0) for j in range(P)}
    names = list(space)
    X = rs.uniform(0, 1, (n, P))
    loss = ((X - 0.4) ** 2).sum(1)
    hist = [optuna.trial.create_trial(value=float(loss[i]), params=dict(zip(names, X[i].tolist())), distributions=space)
            for i in range(n)]

    def run(sampler):
        study = optuna.create_study(sampler=sampler)
        study.add_trials(hist)
        got = []
        for it in range(6):
            t = study.ask()
            got.append([t.suggest_float(nm, 0.0, 1.0) for nm in names])
            if it == 2:
                sampler._rng.rng.random_sample(3)  # someone else consumes from the generator
            if it == 4 and hasattr(sampler, "close"):
                sampler.close()                    # engine re-created at the next ask
        return got, sampler._rng.rng.random_sample(4)

    def run_reference():
        want, tail = run(make_sampler.reference(**kw))
        return want, tail.tolist()

    kw = dict(seed=11, n_ei_candidates=C, multivariate=True)
    got, tail = run(make_sampler(**kw))
    want, tail_ref = recorded("test_device_generated_uniforms_give_the_reference_suggestions/run", run_reference)
    np.testing.assert_allclose(got, want, rtol=1e-9, atol=0)
    assert np.array_equal(tail, tail_ref)  # the generator ends in the reference's state


def test_univariate_plans_are_used_and_survive_surprises(make_sampler):
    """Univariate TPE: the per-parameter asks of a trial are evaluated together in the order the previous trial
    asked (B200TPESampler._plan_trial); the trajectory must stay the reference's when a trial asks in another
    order, fails half way, or somebody else draws from the sampler's generator in between -- and when parameters
    are missing from some trials (then the columns cannot share a split and nothing is batched)."""
    def obj(t, holes=False):
        n = t.number
        names = ["a", "b", "c", "d"]
        if n % 5 == 2:
            names = ["b", "a", "c", "d"]              # another order
        if holes and n % 7 == 3:
            names = names[:2]                          # a trial without c and d
        vals = {}
        for i, nm in enumerate(names):
            vals[nm] = t.suggest_float(nm, -1.0, 1.0) if nm != "d" else t.suggest_float(nm, 1e-3, 1.0, log=True)
            if n % 6 == 4 and i == 1:
                t.study.sampler._rng.rng.random_sample(3)   # a foreign draw in the middle of a trial
            if not holes and n % 7 == 3 and i == 1:
                raise RuntimeError("fails half way")   # FAIL: the rest of the plan is never asked for
        if holes and n % 11 == 5:
            vals["e"] = t.suggest_float("e", 0.0, 2.0)  # a parameter the plan did not expect
        return sum(v * v for v in vals.values())

    def scenario(holes, n_trials):
        def run(sampler):
            s = optuna.create_study(sampler=sampler)
            s.optimize(lambda t: obj(t, holes), n_trials=n_trials, catch=(RuntimeError,))
            return s
        return run

    a, _ = over_seeds(scenario(False, 60), make_sampler, False, dict(seed=17, n_startup_trials=6, n_ei_candidates=16))
    if make_sampler.kind == "oracle":
        batches = [c for c in a.sampler._engine.calls if c[0] == "univariate_batch"]
        assert len(batches) > 25 and max(c[1] for c in batches) == 4
    a, _ = over_seeds(scenario(True, 60), make_sampler, False, dict(seed=18, n_startup_trials=6, n_ei_candidates=16))
    if make_sampler.kind == "oracle":
        assert not [c for c in a.sampler._engine.calls if c[0] == "univariate_batch"] and a.sampler._uni.disabled
    # large asks: the plan's uniforms come from the device generator (2 * 2048 * 4 >= DEVICE_RNG_MIN)
    over_seeds(scenario(False, 24), make_sampler, False, dict(seed=3, n_startup_trials=6, n_ei_candidates=2048))
