"""What the reference sampler (optuna.samplers.TPESampler, unmodified) computed in the scenarios the plugin tests
drive, stored in tests/golden/reference_runs.json.xz: the tests compare with these results instead of running a
second, live copy of the reference next to ours.

Each entry is keyed by the test (its name without the engine parameter) and a tag of the run within it.  The
values are plain JSON: parameter dicts keep their Python types (int / float / str / None), floats round-trip
exactly.  To regenerate, with the reference importable (oracle/_ref):

    TPE_REGEN_REFERENCE=1 python -m pytest tests -k "not cuda-engine"

Univariate runs with repeated observations depend on the tie order of NumPy's unstable argsort inside the reference
(parzen_estimator.py:200), which follows the host's SIMD dispatch; the stored results come from an AVX-512 host.
"""
from __future__ import annotations

import atexit
import json
import lzma
import os
import re
from types import SimpleNamespace

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_runs.json.xz")
_data: dict | None = None
_save_registered = False
_fresh: set[str] = set()


def regenerating() -> bool:
    return os.environ.get("TPE_REGEN_REFERENCE") == "1"


def _load() -> dict:
    global _data
    if _data is None:
        _data = {}
        if os.path.exists(PATH):
            with lzma.open(PATH, "rt") as f:
                _data = json.load(f)
    return _data


def _save() -> None:
    raw = json.dumps(_data, sort_keys=True, separators=(",", ":")).encode()
    with open(PATH, "wb") as f:
        f.write(lzma.compress(raw, preset=9 | lzma.PRESET_EXTREME))


def node_key(node_name: str) -> str:
    """A test's node name without the engine parameter (the reference's result does not depend on it)."""
    name = re.sub(r"-?(oracle|cuda)-engine-?", "-", node_name)
    return name.replace("[-", "[").replace("-]", "]").replace("[]", "")


def recorded(key: str, compute):
    """The stored reference result `key`; when regenerating, `compute()` (a live reference run) replaces it."""
    global _save_registered
    data = _load()
    if regenerating() and key not in _fresh:
        data[key] = json.loads(json.dumps(compute()))
        _fresh.add(key)
        if not _save_registered:
            atexit.register(_save)
            _save_registered = True
    if key not in data:
        raise KeyError(f"no stored reference result {key!r} in {PATH} (see tests/_reference_golden.py)")
    return data[key]


def summarize(study) -> dict:
    """The parts of a finished study the tests compare: per trial its state, parameters and constraints, and the
    groups of a group-decomposed search space."""
    group = getattr(study.sampler, "_search_space_group", None)
    return {"trials": [[int(t.state), t.params, t.system_attrs.get("constraints")] for t in study.trials],
            "groups": None if group is None else [sorted(g) for g in group.search_spaces]}


def stored_study(summary: dict):
    """A summary as an object with the study attributes the tests read (trials[i].state / .params /
    .system_attrs, groups)."""
    from optuna.trial import TrialState
    trials = [SimpleNamespace(state=TrialState(s), params=p, system_attrs={} if c is None else {"constraints": c})
              for s, p, c in summary["trials"]]
    return SimpleNamespace(trials=trials, groups=summary["groups"])
