"""Array-level Python face of the C ABI: one ``TPEEngine`` = one ``tpe_ctx`` on one GPU.

This is the thin layer ``B200TPESampler`` (sampler.py) drives; it is also what the parity tests
call so that every check goes through the C ABI.  It holds no algorithmic logic: inputs are
validated and copied by the library (include/optuna_b200_tpe.h).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Sequence

import numpy as np

from . import _lib


@dataclass(frozen=True)
class ParamSpec:
    """One column of the search space (mirror of optuna.distributions.*Distribution fields)."""

    kind: int  # _lib.KIND_*
    low: float = 0.0
    high: float = 0.0
    step: float | None = None
    log: bool = False
    n_choices: int = 0
    dist_table: np.ndarray | None = None  # categorical_distance_func evaluated on all pairs


def _ptr(a: np.ndarray | None):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _f64(a, shape=None) -> np.ndarray:
    out = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        out = out.reshape(shape)
    return out


class TPEEngine:
    def __init__(self, device: int = 0) -> None:
        self._lib = _lib.load()
        handle = C.c_void_p()
        rc = self._lib.tpe_ctx_create(int(device), C.byref(handle))
        if rc != 0:
            raise RuntimeError(f"tpe_ctx_create(device={device}) failed with code {rc}: a CUDA device is required")
        self._h = handle
        self.device = int(device)
        self.n_params = 0
        self._cfg = None
        self._pc = 0
        self._ncat = self._nnum = 0
        self._specs: list[ParamSpec] = []
        self._cols: list[int] = []

    # -- lifecycle -----------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None):
            for p in getattr(self, "_pinned", []):
                self._lib.tpe_host_free(self._h, C.c_void_p(p))
            self._pinned = []
            self._lib.tpe_ctx_destroy(self._h)
            self._h = None

    def __del__(self) -> None:  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int) -> None:
        if rc == 0:
            return
        msg = self._lib.tpe_last_error(self._h).decode()
        if rc == _lib.TPE_E_INVALID:
            raise ValueError(msg)
        raise RuntimeError(f"libtpe_b200 error {rc}: {msg}")

    # -- space / history -------------------------------------------------------------------------
    def set_space(self, specs: Sequence[ParamSpec]) -> None:
        n = len(specs)
        arr = (_lib.ParamDesc * max(n, 1))()
        offs = np.full(max(n, 1), -1, dtype=np.int64)
        tables = []
        at = 0
        for i, s in enumerate(specs):
            arr[i].kind = s.kind
            arr[i].log = int(bool(s.log))
            arr[i].has_step = int(s.step is not None)
            arr[i].n_choices = int(s.n_choices)
            arr[i].low = float(s.low)
            arr[i].high = float(s.high)
            arr[i].step = float(s.step) if s.step is not None else 0.0
            if s.dist_table is not None:
                t = _f64(s.dist_table, (s.n_choices, s.n_choices))
                tables.append(t.ravel())
                offs[i] = at
                at += t.size
        flat = np.concatenate(tables) if tables else None
        self._check(self._lib.tpe_space_set(self._h, arr, n, _ptr(flat), _ptr(offs) if tables else None))
        self._specs = list(specs)
        self.n_params = n

    def set_history(self, X, category, key) -> None:
        X = _f64(X, (-1, self.n_params))
        cat = np.ascontiguousarray(category, dtype=np.int8)
        key = _f64(key, (-1, 2))
        assert X.shape[0] == cat.shape[0] == key.shape[0]
        self._check(self._lib.tpe_history_set(self._h, _ptr(X), _ptr(cat), _ptr(key), X.shape[0]))

    def append_history(self, X, category, key) -> None:
        X = _f64(X, (-1, self.n_params))
        cat = np.ascontiguousarray(category, dtype=np.int8).reshape(-1)
        key = _f64(key, (-1, 2))
        self._check(self._lib.tpe_history_append(self._h, _ptr(X), _ptr(cat), _ptr(key), X.shape[0]))

    def update_history(self, X, category, key, at_row: int) -> None:
        """Overwrite rows [at_row, at_row + n) in place (a trial that finished keeps its position); a write
        past the end extends the history."""
        X = _f64(X, (-1, self.n_params))
        cat = np.ascontiguousarray(category, dtype=np.int8).reshape(-1)
        key = _f64(key, (-1, 2))
        self._check(self._lib.tpe_history_update(self._h, _ptr(X), _ptr(cat), _ptr(key), X.shape[0], int(at_row)))

    def set_values(self, values, at_row: int = 0, n_objectives: int | None = None) -> None:
        """Sign-normalised objective values [n, M] of history rows [at_row, at_row + n) (MOTPE).  Pass
        `n_objectives` when n may be 0 (the shape of an empty array does not say)."""
        v = _f64(values)
        m = int(n_objectives) if n_objectives is not None else (v.shape[1] if v.ndim == 2 else 1)
        v = v.reshape(-1, m)
        self._check(self._lib.tpe_history_set_values(self._h, _ptr(v), v.shape[0], m, int(at_row)))

    def set_history_device(self, dX: int, dcat: int, dkey: int, n: int, col_has_missing=None) -> None:
        miss = None if col_has_missing is None else np.ascontiguousarray(col_has_missing, dtype=np.uint8)
        self._check(self._lib.tpe_history_set_device(self._h, C.c_void_p(dX), C.c_void_p(dcat), C.c_void_p(dkey),
                                                     int(n), _ptr(miss)))

    def history_device_ptrs(self) -> tuple[int, int, int]:
        a, b, c = C.c_void_p(), C.c_void_p(), C.c_void_p()
        self._check(self._lib.tpe_history_device_ptrs(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    @property
    def history_size(self) -> int:
        return int(self._lib.tpe_history_size(self._h))

    # -- stages ------------------------------------------------------------------------------------
    def _make_cfg(self, *, n_below: int, n_candidates: int, multivariate: bool, prior_weight: float = 1.0,
                  magic_clip: bool = True, endpoints: bool = False) -> _lib.Cfg:
        return _lib.Cfg(float(prior_weight), int(magic_clip), int(endpoints), int(multivariate),
                        int(n_candidates), int(n_below))

    def _note_cols(self, cols: Sequence[int], n_candidates: int) -> np.ndarray:
        self._cols = [int(c) for c in cols]
        self._pc = len(self._cols)
        self._ncat = sum(1 for c in self._cols if 0 <= c < self.n_params and self._specs[c].kind == _lib.KIND_CAT)
        self._nnum = self._pc - self._ncat
        self._C = int(n_candidates)
        return np.ascontiguousarray(self._cols, dtype=np.int32)

    def uniforms_per_ask(self) -> int:
        return self._C * (1 + self._ncat + self._nnum)

    def prepare(self, cols: Sequence[int], **cfg) -> tuple[int, int, int]:
        c = self._make_cfg(**cfg)
        cols_a = self._note_cols(cols, c.n_candidates)
        info = _lib.SplitInfo()
        self._check(self._lib.tpe_prepare(self._h, C.byref(c), _ptr(cols_a), len(cols_a), C.byref(info)))
        self._info = (int(info.n_below_all), int(info.n_below_obs), int(info.n_above_obs))
        return self._info

    def build(self, w_below=None, w_above=None) -> None:
        wb = None if w_below is None else _f64(w_below)
        wa = None if w_above is None else _f64(w_above)
        if wb is not None:
            assert wb.size == self._info[1], (wb.size, self._info)
        if wa is not None:
            assert wa.size == self._info[2], (wa.size, self._info)
        self._check(self._lib.tpe_build(self._h, _ptr(wb), _ptr(wa)))

    def sample_and_select(self, uniforms, n_asks: int = 1):
        """uniforms=None: consume the device-generated uniforms of ``stage_rng``."""
        u = None
        if uniforms is not None:
            u = _f64(uniforms).reshape(-1)
            assert u.size == n_asks * self.uniforms_per_ask(), (u.size, n_asks, self.uniforms_per_ask())
        x = np.empty((n_asks, self._pc), dtype=np.float64)
        acq = np.empty(n_asks, dtype=np.float64)
        best = np.empty(n_asks, dtype=np.int64)
        self._check(self._lib.tpe_sample_and_select(self._h, _ptr(u), int(n_asks), _ptr(x), _ptr(acq), _ptr(best)))
        self._last_asks = n_asks
        return x, acq, best

    def sample_and_select_async(self, uniforms, n_asks: int = 1) -> None:
        """Queue ``sample_and_select`` and return; ``collect()`` waits and returns the results."""
        u = None
        if uniforms is not None:
            u = _f64(uniforms).reshape(-1)
            assert u.size == n_asks * self.uniforms_per_ask(), (u.size, n_asks, self.uniforms_per_ask())
        self._check(self._lib.tpe_sample_and_select_async(self._h, _ptr(u), int(n_asks)))
        self._last_asks = n_asks

    def collect(self):
        n_asks = self._last_asks
        x = np.empty((n_asks, self._pc), dtype=np.float64)
        acq = np.empty(n_asks, dtype=np.float64)
        best = np.empty(n_asks, dtype=np.int64)
        self._check(self._lib.tpe_collect(self._h, _ptr(x), _ptr(acq), _ptr(best)))
        return x, acq, best

    def rng_snapshot(self) -> tuple:
        """The generator state the device holds (after the last staged draw) as ``RandomState.set_state`` takes it."""
        key = np.empty(624, dtype=np.uint32)
        pos = C.c_int32()
        self._check(self._lib.tpe_rng_state(self._h, _ptr(key), C.byref(pos)))
        name, has_gauss, cached = self._rng_tail
        return (name, key, int(pos.value), has_gauss, cached)

    def set_kernel_shard(self, rank: int, world: int) -> None:
        """This engine evaluates g(x) over slice `rank` of `world` of the above kernels (world = 1: off)."""
        self._check(self._lib.tpe_set_kernel_shard(self._h, int(rank), int(world)))

    def sample_and_partial(self, uniforms, n_asks: int = 1) -> tuple[int, int]:
        """Candidates, l(x) and this engine's slice of g(x): (device address of the [n_asks * C] (max, sum) pairs,
        their padded count)."""
        u = None
        if uniforms is not None:
            u = _f64(uniforms).reshape(-1)
            assert u.size == n_asks * self.uniforms_per_ask()
        ptr, stride = C.c_void_p(), C.c_int64()
        self._check(self._lib.tpe_sample_and_partial(self._h, _ptr(u), int(n_asks), C.byref(ptr), C.byref(stride)))
        self._last_asks = n_asks
        return int(ptr.value), int(stride.value)

    def finish_from_partials(self, gathered_ptr: int, world: int):
        n_asks = self._last_asks
        x = np.empty((n_asks, self._pc), dtype=np.float64)
        acq = np.empty(n_asks, dtype=np.float64)
        best = np.empty(n_asks, dtype=np.int64)
        self._check(self._lib.tpe_finish_from_partials(self._h, C.c_void_p(int(gathered_ptr)), int(world), _ptr(x), _ptr(acq),
                                                       _ptr(best)))
        return x, acq, best

    def sample_and_select_device(self, n_asks: int = 1) -> int:
        """Like ``sample_and_select(None, n_asks)`` but the results stay on the device; returns the device
        address of out_x [n_asks, n_cols] fp64 (valid until the next call on this engine)."""
        self._check(self._lib.tpe_sample_and_select(self._h, None, int(n_asks), None, None, None))
        self._last_asks = n_asks
        px = C.c_void_p()
        self._check(self._lib.tpe_result_device_ptrs(self._h, C.byref(px), None, None))
        return int(px.value)

    def rng_state_device(self) -> int:
        """Device address of the generator state (625 uint32) kept by ``stage_rng``; see tpe_rng_state_device."""
        p = C.c_void_p()
        self._check(self._lib.tpe_rng_state_device(self._h, C.byref(p)))
        return int(p.value)

    def stage_rng(self, rng: np.random.RandomState | None, count: int, skip: int = 0, state=None) -> None:
        """Generate the next `count` outputs of ``rng.random_sample`` on the device (after dropping
        `skip`); the following ``sample_and_select(None, n_asks)`` consumes them.  ``finish_rng(rng)``
        then moves `rng` to the state after the draws.  ``rng=None`` continues from the state the
        previous staged draw ended in (the host generator is then stale until ``finish_rng``)."""
        if rng is None:
            self._check(self._lib.tpe_stage_uniforms_mt19937(self._h, None, 0, int(skip), int(count)))
            return
        st = rng.get_state() if state is None else state
        key = np.ascontiguousarray(st[1], dtype=np.uint32)
        self._rng_tail = (st[0], st[3], st[4])
        self._check(self._lib.tpe_stage_uniforms_mt19937(self._h, _ptr(key), int(st[2]), int(skip), int(count)))

    def get_uniforms(self, count: int) -> np.ndarray:
        out = np.empty(int(count), dtype=np.float64)
        self._check(self._lib.tpe_get_uniforms(self._h, _ptr(out), int(count)))
        return out

    def finish_rng(self, rng: np.random.RandomState) -> None:
        key = np.empty(624, dtype=np.uint32)
        pos = C.c_int32()
        self._check(self._lib.tpe_rng_state(self._h, _ptr(key), C.byref(pos)))
        name, has_gauss, cached = self._rng_tail
        rng.set_state((name, key, int(pos.value), has_gauss, cached))

    def pinned_empty(self, n: int) -> np.ndarray:
        """float64[n] in page-locked host memory (freed with the engine): copies from it are async DMAs."""
        p = C.c_void_p()
        self._check(self._lib.tpe_host_alloc(self._h, C.c_size_t(int(n) * 8), C.byref(p)))
        if not hasattr(self, "_pinned"):
            self._pinned = []
        self._pinned.append(p.value)
        return np.ctypeslib.as_array((C.c_double * int(n)).from_address(p.value))

    def stage_uniforms(self, uniforms: np.ndarray) -> np.ndarray:
        """Start uploading the uniforms of the next `sample_and_select` now (latency hint); pass the
        returned array (same memory) to `sample_and_select`."""
        u = _f64(uniforms).reshape(-1)
        self._check(self._lib.tpe_stage_uniforms(self._h, _ptr(u), int(u.size)))
        return u

    def suggest(self, cols: Sequence[int], uniforms, n_asks: int = 1, w_below=None, w_above=None, **cfg):
        c = self._make_cfg(**cfg)
        cols_a = self._note_cols(cols, c.n_candidates)
        u = _f64(uniforms).reshape(-1)
        assert u.size == n_asks * self.uniforms_per_ask()
        wb = None if w_below is None else _f64(w_below)
        wa = None if w_above is None else _f64(w_above)
        x = np.empty((n_asks, self._pc), dtype=np.float64)
        acq = np.empty(n_asks, dtype=np.float64)
        best = np.empty(n_asks, dtype=np.int64)
        self._check(self._lib.tpe_suggest(self._h, C.byref(c), _ptr(cols_a), len(cols_a), _ptr(wb), _ptr(wa),
                                          _ptr(u), int(n_asks), _ptr(x), _ptr(acq), _ptr(best)))
        self._last_asks = n_asks
        self._info = self.split_info()
        return x, acq, best

    def suggest_univariate_batch(self, cols: Sequence[int], uniforms, w_below=None, w_above=None, **cfg):
        """The per-parameter suggestions of one univariate trial together (tpe_suggest_univariate_batch);
        uniforms=None consumes the device-generated uniforms of ``stage_rng(.., len(cols) * 2 * C)``.
        Raises RuntimeError("... not batchable ...") when the columns cannot share a split."""
        c = self._make_cfg(**cfg)
        cols_a = np.ascontiguousarray([int(v) for v in cols], dtype=np.int32)
        u = None
        if uniforms is not None:
            u = _f64(uniforms).reshape(-1)
            assert u.size == len(cols_a) * 2 * c.n_candidates
        wb = None if w_below is None else _f64(w_below)
        wa = None if w_above is None else _f64(w_above)
        x = np.empty(len(cols_a), dtype=np.float64)
        acq = np.empty(len(cols_a), dtype=np.float64)
        best = np.empty(len(cols_a), dtype=np.int64)
        self._check(self._lib.tpe_suggest_univariate_batch(self._h, C.byref(c), _ptr(cols_a), len(cols_a), _ptr(wb),
                                                           _ptr(wa), _ptr(u), _ptr(x), _ptr(acq), _ptr(best)))
        return x, acq, best

    def suggest_univariate_batch_async(self, cols: Sequence[int], uniforms, w_below=None, w_above=None, **cfg) -> None:
        """Queue ``suggest_univariate_batch`` and return; ``collect_univariate()`` waits and returns the results."""
        c = self._make_cfg(**cfg)
        cols_a = np.ascontiguousarray([int(v) for v in cols], dtype=np.int32)
        u = None
        if uniforms is not None:
            u = _f64(uniforms).reshape(-1)
            assert u.size == len(cols_a) * 2 * c.n_candidates
        wb = None if w_below is None else _f64(w_below)
        wa = None if w_above is None else _f64(w_above)
        self._check(self._lib.tpe_suggest_univariate_batch_async(self._h, C.byref(c), _ptr(cols_a), len(cols_a), _ptr(wb),
                                                                 _ptr(wa), _ptr(u)))
        self._uni_pending = len(cols_a)

    def collect_univariate(self):
        n = self._uni_pending
        x = np.empty(n, dtype=np.float64)
        acq = np.empty(n, dtype=np.float64)
        best = np.empty(n, dtype=np.int64)
        self._check(self._lib.tpe_collect_univariate(self._h, _ptr(x), _ptr(acq), _ptr(best)))
        return x, acq, best

    def split_info(self) -> tuple[int, int, int]:
        info = _lib.SplitInfo()
        self._check(self._lib.tpe_get_split_info(self._h, C.byref(info)))
        return int(info.n_below_all), int(info.n_below_obs), int(info.n_above_obs)

    # -- importance --------------------------------------------------------------------------------
    def ped_anova(self, cols: Sequence[int], grids, n_grid, *, target_quantile: float, region_quantile: float,
                  evaluate_on_local: bool, loss=None, prior_weight: float = 1.0, min_n_top: int = 2,
                  n_steps: int = 50, counts: bool = False):
        """PED-ANOVA importance of the history columns `cols` (tpe_ped_anova).  grids [n_cols, n_steps]: the host's
        np.linspace grid per numerical column (rows of categorical columns are ignored); n_grid [n_cols]: bins per
        column; loss [history size] or None = the uploaded sort key.  Returns (importances [n_cols], (kept, target,
        region), counts [n_cols, 2, max n_grid] of the target / region bins, or None)."""
        cols_a = np.ascontiguousarray([int(c) for c in cols], dtype=np.int32)
        ng = np.ascontiguousarray(n_grid, dtype=np.int32).reshape(-1)
        g = _f64(grids, (len(cols_a), int(n_steps)))
        lv = None if loss is None else _f64(loss).reshape(-1)
        if lv is not None:
            assert lv.size == self.history_size, (lv.size, self.history_size)
        c = _lib.PedCfg(float(target_quantile), float(region_quantile), float(prior_weight), int(bool(evaluate_on_local)),
                        int(min_n_top), int(n_steps))
        imp = np.empty(len(cols_a), dtype=np.float64)
        sizes = np.empty(3, dtype=np.int64)
        cnt = np.empty((len(cols_a), 2, int(ng.max(initial=1))), dtype=np.int32) if counts else None
        self._check(self._lib.tpe_ped_anova(self._h, C.byref(c), _ptr(cols_a), len(cols_a), _ptr(g), _ptr(ng), _ptr(lv),
                                            _ptr(imp), _ptr(sizes), _ptr(cnt)))
        return imp, tuple(int(v) for v in sizes), cnt

    # -- inspection --------------------------------------------------------------------------------
    def get_split(self) -> tuple[np.ndarray, np.ndarray]:
        below = np.empty(self._info[1], dtype=np.int64)
        above = np.empty(self._info[2], dtype=np.int64)
        self._check(self._lib.tpe_get_split(self._h, _ptr(below), _ptr(above)))
        return below, above

    def get_mixture(self, which: int):
        K = self._info[1 + which] + 1
        w = np.empty(K)
        mu = np.empty((K, self._pc))
        sg = np.empty((K, self._pc))
        self._check(self._lib.tpe_get_mixture(self._h, int(which), _ptr(w), _ptr(mu), _ptr(sg)))
        return w, mu, sg

    def get_mo_weights(self) -> np.ndarray:
        w = np.empty(self._info[0])
        self._check(self._lib.tpe_get_mo_weights(self._h, _ptr(w)))
        return w

    def get_candidates(self):
        ct = self._last_asks * self._C
        s = np.empty((ct, self._pc))
        ll = np.empty(ct)
        lg = np.empty(ct)
        self._check(self._lib.tpe_get_candidates(self._h, _ptr(s), _ptr(ll), _ptr(lg)))
        return s, ll, lg

    def logpdf(self, which: int, x) -> np.ndarray:
        x = _f64(x, (-1, self._pc))
        out = np.empty(x.shape[0])
        self._check(self._lib.tpe_logpdf(self._h, int(which), _ptr(x), x.shape[0], _ptr(out)))
        return out

    def last_timing(self) -> tuple[np.ndarray, int]:
        ms = np.zeros(9, dtype=np.float32)
        n = C.c_int32()
        self._check(self._lib.tpe_last_timing(self._h, _ptr(ms), C.byref(n)))
        return ms, int(n.value)

    def probe_fp64_tflops(self) -> float:
        v = C.c_double()
        self._check(self._lib.tpe_probe_fp64_tflops(self._h, C.byref(v)))
        return float(v.value)

    def last_logpdf_kernel(self) -> str:
        return self._lib.tpe_last_logpdf_kernel(self._h).decode()
