import itertools
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# The reference itself (unmodified optuna, oracle/_ref -- built by oracle/build_ref.py where /root/reference exists,
# shipped to the GPU box with the snapshot) is the caller the plugin is tested behind.  Test infrastructure only.
from oracle import build_ref, ref  # noqa: E402

build_ref.build()
HAVE_OPTUNA = ref.enable()


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def has_gpu() -> bool:
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if has_gpu():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def _engine_params():
    return [pytest.param("oracle", id="oracle-engine"),
            pytest.param("cuda", id="cuda-engine", marks=pytest.mark.gpu)]


@pytest.fixture(params=_engine_params())
def make_sampler(request, monkeypatch):
    """Factory of B200TPESampler instances answered by the CPU oracle (host glue, runs anywhere) or by
    libtpe_b200.so (the product, GPU box)."""
    if not HAVE_OPTUNA:
        pytest.skip("optuna (oracle/_ref) is not available")
    from optuna_b200 import B200TPESampler
    if request.param == "oracle":
        from tests._oracle_engine import OracleEngine
        monkeypatch.setattr(B200TPESampler, "_engine_cls", OracleEngine)
    made = []

    def make(**kw):
        s = B200TPESampler(**kw)
        made.append(s)
        return s

    def reference(ties=False, **kw):
        """The sampler to compare with: the reference (run live only to store its results, see `yardstick`) -- except
        for the CUDA engine in univariate scenarios
        with repeated numeric observations, where the reference's bandwidths depend on the tie order of numpy's
        UNSTABLE argsort (parzen_estimator.py:200; CPU-dispatch dependent) while the CUDA path sorts stably
        (DESIGN.md section 4): there the yardstick is the same host glue answered by the stable-sort oracle.
        (The oracle-engine runs of the same scenarios pin glue + oracle to the live reference.)"""
        if request.param == "cuda" and ties and not kw.get("multivariate", False):
            from tests._oracle_engine import StableOracleEngine
            s = B200TPESampler(**kw)
            s._engine_cls = StableOracleEngine
            made.append(s)
            return s
        from optuna.samplers import TPESampler
        return TPESampler(**kw)

    def yardstick(tag, scenario, ties=False, **kw):
        """What the yardstick computed in `scenario(sampler) -> study`, as tests._reference_golden.stored_study: the
        stored result of the reference (run `tag` of this test) -- or, where `reference` names the stable-sort
        oracle, that oracle's run now."""
        from tests._reference_golden import node_key, recorded, stored_study, summarize
        if request.param == "cuda" and ties and not kw.get("multivariate", False):
            return stored_study(summarize(scenario(reference(ties, **kw))))
        return stored_study(recorded(f"{node_key(request.node.name)}/{tag}",
                                     lambda: summarize(scenario(reference(**kw)))))

    make.kind = request.param
    make.reference = reference
    make.yardstick = yardstick
    make.runs = itertools.count()
    yield make
    for s in made:
        s.close()
