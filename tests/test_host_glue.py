"""Host-side glue of the sampler plugin that needs no GPU."""
import pickle

import numpy as np
import pytest

from optuna_b200 import _lib
from tests._reference_golden import recorded
from tests._util import draw_uniforms


def test_library_loads_and_exports_every_declared_symbol():
    lib = _lib.load()
    assert lib.tpe_abi_version() == _lib.ABI_VERSION
    import os
    import re
    hdr = open(os.path.join(os.path.dirname(_lib.LIB_PATH), "..", "include", "optuna_b200_tpe.h")).read()
    assert int(re.search(r"#define TPE_ABI_VERSION (\d+)", hdr).group(1)) == _lib.ABI_VERSION
    declared = set(re.findall(r"\b(tpe_[a-z0-9_]+)\s*\(", hdr)) - {"tpe_ctx"}
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    for name in declared:
        assert hasattr(lib, name)


def test_no_cpu_fallback_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from optuna_b200 import TPEEngine
    with pytest.raises(RuntimeError):
        TPEEngine(0)
    # ... and the sampler's engine IS that class: nothing else can answer a suggestion in the product
    pytest.importorskip("optuna")
    from optuna_b200 import B200TPESampler
    assert B200TPESampler._engine_cls is TPEEngine


def test_single_random_sample_call_is_the_reference_stream():
    C = 24
    for ncat, nnum in ((0, 1), (2, 3), (12, 52), (1, 0)):
        a, b = np.random.RandomState(9), np.random.RandomState(9)
        assert np.array_equal(draw_uniforms(a, C, ncat, nnum), b.random_sample(C * (1 + ncat + nnum)))


def test_gamma_and_weights_mirror_reference_formulas():
    pytest.importorskip("optuna")
    from optuna_b200.sampler import default_gamma, default_weights, hyperopt_default_gamma
    ns = (0, 1, 10, 11, 24, 25, 26, 250, 100000)

    def sample(w):  # every weight of the short arrays, a fixed sample of the long one
        idx = np.unique(np.r_[0:300, 300:len(w):997, len(w) - 300:len(w)])
        return w[idx[(idx >= 0) & (idx < len(w))]]

    def reference():
        from optuna.samplers._tpe import sampler as ref
        return [[ref.default_gamma(n), ref.hyperopt_default_gamma(n), sample(ref.default_weights(n)).tolist()]
                for n in ns]

    for n, (gamma, hyperopt_gamma, weights) in zip(ns, recorded("test_gamma_and_weights_mirror_reference_formulas",
                                                                reference)):
        assert default_gamma(n) == gamma
        assert hyperopt_default_gamma(n) == hyperopt_gamma
        assert np.array_equal(sample(default_weights(n)), np.asarray(weights, dtype=float))


def test_sampler_constructor_contract():
    optuna = pytest.importorskip("optuna")
    import inspect
    import warnings
    from optuna_b200 import B200TPESampler
    ref = inspect.signature(optuna.samplers.TPESampler.__init__).parameters
    mine = inspect.signature(B200TPESampler.__init__).parameters
    assert [k for k in mine if k != "device"] == list(ref)          # same keyword arguments, same order
    for k in ref:
        if k not in ("self", "gamma", "weights"):
            assert mine[k].default == ref[k].default, k
    assert issubclass(B200TPESampler, optuna.samplers.BaseSampler)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        with pytest.raises(ValueError):
            B200TPESampler(group=True)  # needs multivariate
        B200TPESampler(seed=1, multivariate=True, group=True, constant_liar=True)
    with pytest.warns(optuna.exceptions.ExperimentalWarning):
        B200TPESampler(multivariate=True)
    with pytest.warns(FutureWarning):
        B200TPESampler(consider_prior=False)
    # startup trials never touch the device: they are optuna's RandomSampler (sampler.py:348-349, :471-474)
    def startup(sampler):
        s = optuna.create_study(sampler=sampler)
        s.optimize(lambda t: t.suggest_float("x", 0, 1) + t.suggest_int("k", 1, 3)
                   + (t.suggest_categorical("c", ["u", None]) is None), n_trials=5)
        return s

    a = startup(B200TPESampler(seed=0, n_startup_trials=5))
    want = recorded("test_sampler_constructor_contract/startup",
                    lambda: [t.params for t in startup(optuna.samplers.TPESampler(seed=0, n_startup_trials=5)).trials])
    assert [t.params for t in a.trials] == want and a.sampler._engine is None


def test_device_synced_rng_flushes_on_access_and_pickle():
    """sampler._DeviceSyncedRng: while the newer MT19937 state lives on the device, any access to
    `.rng` (and pickling) first copies it back -- here with a stand-in engine."""
    pytest.importorskip("optuna")
    from optuna.samplers._lazy_random_state import LazyRandomState
    from optuna_b200.sampler import _DeviceSyncedRng

    class FakeEngine:
        def __init__(self, end_state):
            self.end_state, self.calls = end_state, 0

        def finish_rng(self, rng):
            self.calls += 1
            rng.set_state(self.end_state)

    ahead = np.random.RandomState(3)
    ahead.random_sample(1000)                      # what the device would have drawn
    proxy = _DeviceSyncedRng(LazyRandomState(3))
    eng = FakeEngine(ahead.get_state())
    assert not proxy.on_device(eng)
    proxy.mark_device(eng)
    assert proxy.on_device(eng) and not proxy.on_device(object())
    clone = pickle.loads(pickle.dumps(proxy))      # pickling flushes
    assert eng.calls == 1 and not proxy.on_device(eng)
    want = ahead.random_sample(4)
    assert np.array_equal(clone.rng.random_sample(4), want)
    assert np.array_equal(proxy.rng.random_sample(4), want) and eng.calls == 1

    # draws staged ahead of their ask: an armed undo puts the generator back at the next look, a released one does not
    before = proxy.rng.get_state()
    snap, drawn = proxy.stage(eng, 6, device=False)
    assert np.array_equal(drawn, ahead.random_sample(6))
    undo = proxy.arm(lambda: proxy.restore(snap))
    assert proxy.armed(undo)
    assert np.array_equal(proxy.rng.random_sample(6), drawn) and not proxy.armed(undo)   # undone before the look
    proxy.rng.set_state(before)
    snap, drawn = proxy.stage(eng, 6, device=False)
    undo = proxy.arm(lambda: proxy.restore(snap))
    proxy.release(undo, adopted=True)
    assert not proxy.armed(undo)
    assert np.array_equal(proxy.rng.random_sample(4), ahead.random_sample(4))           # nothing restored
    undo = proxy.arm(lambda: proxy.restore(snap, 2))           # a plan served in part: restored `advance` draws on
    proxy.release(undo, adopted=False)
    assert np.array_equal(proxy.rng.random_sample(4), drawn[2:])
    assert not pickle.loads(pickle.dumps(proxy)).armed(undo) and eng.calls == 1


def test_trial_log_matches_optunas_search_spaces_under_out_of_order_finishes():
    """_History.poll / intersection / group_spaces vs optuna's IntersectionSearchSpace
    (search_space/intersection.py) and _GroupDecomposedSearchSpace (group_decomposed.py) on a study whose
    trials finish out of order, fail, wait in the queue and are added from outside."""
    optuna = pytest.importorskip("optuna")
    from optuna.search_space import IntersectionSearchSpace
    from optuna.search_space.group_decomposed import _GroupDecomposedSearchSpace
    from optuna.trial import TrialState
    from optuna_b200.sampler import _History

    rs = np.random.RandomState(0)
    study = optuna.create_study(sampler=optuna.samplers.RandomSampler(seed=0))
    log, inter, groups = _History(), IntersectionSearchSpace(include_pruned=True), _GroupDecomposedSearchSpace(True)
    open_trials = []

    def suggest(t):
        t.suggest_float("x", 0, 1)
        if rs.rand() < 0.5:
            t.suggest_int("k", 0, 3)
        if rs.rand() < 0.3:
            t.suggest_categorical("c", ["a", "b"])
        if rs.rand() < 0.2:
            t.suggest_float("x2", 0, 1 + (t.number % 2))  # dynamic range: drops out of the intersection

    for step in range(120):
        r = rs.rand()
        if r < 0.45 or not open_trials:
            t = study.ask()
            suggest(t)
            open_trials.append(t)
        elif r < 0.8:
            t = open_trials.pop(rs.randint(len(open_trials)))
            state = [TrialState.COMPLETE, TrialState.PRUNED, TrialState.FAIL][rs.choice(3, p=[0.7, 0.15, 0.15])]
            study.tell(t, rs.rand() if state == TrialState.COMPLETE else None, state=state)
        elif r < 0.9:
            study.enqueue_trial({"x": 0.5})
        else:
            study.add_trial(optuna.trial.create_trial(value=0.1, params={"x": 0.2, "k": 1}, distributions={
                "x": optuna.distributions.FloatDistribution(0, 1), "k": optuna.distributions.IntDistribution(0, 3)}))
        log.poll(study, use_cache=False)
        assert log.intersection() == inter.calculate(study)
        assert list(log.intersection()) == list(inter.calculate(study))
        got = [sorted(g) for g in log.group_spaces()]
        want = [sorted(g) for g in groups.calculate(study).search_spaces]
        assert got == want, (step, got, want)
        fin = [t for t in study.get_trials(deepcopy=False) if t.state in (TrialState.COMPLETE, TrialState.PRUNED)]
        assert log.n_finished == len(fin) and log.rows == len(study.get_trials(deepcopy=False))
        assert log.seen_params == {k for t in fin for k in t.params}
