/*
 * optuna_b200_tpe.h -- C ABI of the B200-native TPE suggestion engine (libtpe_b200.so).
 *
 * This is the drop-in boundary for the reference's TPE hot path.  Each entry point names the
 * reference interface it replaces (paths relative to the optuna checkout @ 4df4b72).  The
 * Python host (optuna_b200/sampler.py) binds these with ctypes; INTEGRATION.md shows the stub a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - every function returns 0 on success or a negative TPE_E_* code; the message is
 *     retrievable with tpe_last_error(ctx) (per context, valid until the next call on it);
 *   - the caller owns all host buffers; the library copies and retains no host pointer;
 *   - the library owns all device memory; one context is bound to one CUDA device;
 *   - no callbacks into the host: Python callables of the reference (gamma, weights,
 *     constraints_func, categorical_distance_func) are evaluated by the host and passed as data;
 *   - all entry points take a per-context mutex (ctypes releases the GIL, and the reference
 *     shares one sampler across n_jobs threads: optuna/study/_optimize.py:87-121);
 *   - doubles are IEEE fp64, indices int64, "internal representation" of a parameter is the
 *     reference's (optuna/distributions.py:182,365,509): float value / int as float / choice index.
 */
#ifndef OPTUNA_B200_TPE_H_
#define OPTUNA_B200_TPE_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* 2: + tpe_history_update, tpe_stage_uniforms, tpe_stage_uniforms_mt19937, tpe_rng_state,
 *      tpe_get_uniforms, tpe_host_alloc / tpe_host_free; tpe_sample_and_select accepts uniforms == NULL
 *      after tpe_stage_uniforms_mt19937 */
/* 3: + TPE_CAT_EXCLUDED; tpe_history_update may extend the history; tpe_sample_and_select accepts out_x == NULL
 *      (results stay on the device: tpe_result_device_ptrs); tpe_rng_state_device; tpe_suggest_univariate_batch */
/* 4: + tpe_sample_and_select_async / tpe_collect */
/* 5: + tpe_suggest_univariate_batch_async / tpe_collect_univariate */
/* 6: + tpe_set_kernel_shard / tpe_sample_and_partial / tpe_finish_from_partials */
/* 7: + tpe_ped_anova */
#define TPE_ABI_VERSION 7

enum {
  TPE_OK = 0,
  TPE_E_INVALID = -1,  /* bad argument (mirrors the reference's ValueError) */
  TPE_E_CUDA = -2,     /* CUDA runtime failure */
  TPE_E_STATE = -3,    /* call order violated (e.g. suggest before history/space are set) */
  TPE_E_NOMEM = -4
};

/* optuna/distributions.py: FloatDistribution :109, IntDistribution :310, CategoricalDistribution :470 */
enum { TPE_KIND_FLOAT = 0, TPE_KIND_INT = 1, TPE_KIND_CAT = 2 };

/* Trial groups of TPESampler._split_trials (optuna/samplers/_tpe/sampler.py:686-722). */
enum {
  TPE_CAT_COMPLETE = 0,
  TPE_CAT_PRUNED = 1,
  TPE_CAT_INFEASIBLE = 2,
  TPE_CAT_RUNNING = 3,
  /* A row that takes part in neither set: the placeholder of a trial the sampler must not see yet (WAITING,
   * RUNNING without constant_liar, the trial being sampled itself -- sampler.py:526-535 filters it out) or ever
   * (FAIL).  Keeps row index == position in the study's trial list, so that a trial finishing late is one
   * tpe_history_update in place instead of a re-upload. */
  TPE_CAT_EXCLUDED = 4
};

typedef struct tpe_ctx tpe_ctx;

typedef struct {
  int32_t kind;      /* TPE_KIND_* */
  int32_t log;       /* 1 = log-scaled domain */
  int32_t has_step;  /* 1 = discretised (always 1 for TPE_KIND_INT) */
  int32_t n_choices; /* categorical only */
  double low, high, step;
} tpe_param_desc;

/* TPESampler constructor arguments that reach the numeric path (sampler.py:305-360) plus the
 * per-call values the host evaluates (gamma(n) -> n_below). */
typedef struct {
  double prior_weight;   /* _ParzenEstimatorParameters.prior_weight */
  int32_t magic_clip;    /* consider_magic_clip */
  int32_t endpoints;     /* consider_endpoints */
  int32_t multivariate;  /* multivariate */
  int32_t n_candidates;  /* n_ei_candidates */
  int64_t n_below;       /* gamma(n_finished), evaluated by the host (sampler.py:538-542) */
} tpe_cfg;

/* Shapes of the two estimators after tpe_prepare. */
typedef struct {
  int64_t n_below_all;  /* |below| before dropping trials that lack a selected param */
  int64_t n_below_obs;  /* observations in l(x) (kernels = +1 prior) */
  int64_t n_above_obs;  /* observations in g(x) */
} tpe_split_info;

int tpe_abi_version(void);
int tpe_ctx_create(int device, tpe_ctx** out);
void tpe_ctx_destroy(tpe_ctx* ctx);
const char* tpe_last_error(tpe_ctx* ctx);

/* Search space = every parameter the study has seen, in the host's column order
 * (replaces the dict[str, BaseDistribution] handed to sample_relative, samplers/_base.py:96).
 * cat_dist: optional concatenation of row-major [n_choices, n_choices] distance tables for the
 * categorical params that have a categorical_distance_func (parzen_estimator.py:152-160),
 * cat_dist_offset[p] = offset into cat_dist or -1. */
int tpe_space_set(tpe_ctx* ctx, const tpe_param_desc* params, int32_t n_params,
                  const double* cat_dist, const int64_t* cat_dist_offset);

/* Trial history (replaces the list[FrozenTrial] walk of _get_internal_repr / _split_trials,
 * sampler.py:511-521, :686-722).
 *   X        [n, n_params] row-major internal representation, NaN = parameter absent
 *   category [n] TPE_CAT_*
 *   key      [n, 2] the reference's sort key inside the category (sampler.py:735-742, :782-821):
 *            COMPLETE (signed value, 0); PRUNED (-last_step, signed value); INFEASIBLE (violation, 0)
 * tpe_history_set replaces everything; tpe_history_append adds rows (after_trial hook). */
int tpe_history_set(tpe_ctx* ctx, const double* X, const int8_t* category, const double* key,
                    int64_t n);
int tpe_history_append(tpe_ctx* ctx, const double* X, const int8_t* category, const double* key,
                       int64_t n);
/* Overwrite rows [at_row, at_row + n) in place: a trial that has finished keeps its position (trial-number order)
 * and only changes its category / key / parameters (a TPE_CAT_EXCLUDED placeholder becoming COMPLETE; with
 * constant_liar=True, sampler.py:526-535, a RUNNING row of the above set).  at_row <= current size; a write that
 * runs past the end extends the history, so "the previous trial finished + the next one started" is one call. */
int tpe_history_update(tpe_ctx* ctx, const double* X, const int8_t* category, const double* key, int64_t n,
                       int64_t at_row);
/* Same, with DEVICE pointers on ctx's device (used after an NCCL broadcast of the history). */
int tpe_history_set_device(tpe_ctx* ctx, const double* dX, const int8_t* dcategory,
                           const double* dkey, int64_t n, const uint8_t* col_has_missing);
/* Multi-objective studies: objective values of rows [at_row, at_row + n), sign-normalised so that
 * every objective is minimised (sampler.py:755).  values [n, n_objectives] row-major.  With
 * n_objectives >= 2 the COMPLETE group is split by non-domination rank + greedy hypervolume subset
 * selection (sampler.py:745-779) and l(x) is weighted by hypervolume contributions (:824-863)
 * unless tpe_build is given explicit below-weights.  n_objectives <= 16; any number of below trials (the exact
 * hypervolumes run over the Pareto front of the below set / the selected subset only; their scratch is O(n^2 M) per
 * warp, TPE_E_NOMEM beyond 16 GB). */
int tpe_history_set_values(tpe_ctx* ctx, const double* values, int64_t n, int32_t n_objectives, int64_t at_row);
int64_t tpe_history_size(tpe_ctx* ctx);
/* Device pointers of the resident history (for the NCCL broadcast done by the host plumbing). */
int tpe_history_device_ptrs(tpe_ctx* ctx, double** dX, int8_t** dcategory, double** dkey);

/* Stage 1: split + observation gathering for the selected columns.
 * Replaces _split_trials + _get_internal_repr.  cols[n_cols] index into the space. */
int tpe_prepare(tpe_ctx* ctx, const tpe_cfg* cfg, const int32_t* cols, int32_t n_cols,
                tpe_split_info* info);

/* Stage 2: build l(x) and g(x) (replaces _ParzenEstimator.__init__, parzen_estimator.py:39-78).
 * w_below / w_above: raw per-observation weights (weights_func(n)[:n], or the MOTPE weights,
 * sampler.py:574-576) or NULL for the reference's default_weights (sampler.py:61-69). */
int tpe_build(tpe_ctx* ctx, const double* w_below, const double* w_above);

/* Stage 3+4: draw candidates from l(x) with host-supplied uniforms and pick the best by
 * log l(x) - log g(x) (replaces mpe_below.sample, _compute_acquisition_func, _compare;
 * sampler.py:553-555).  n_asks independent suggestions share the estimators.
 *   uniforms [n_asks, C * (1 + n_cat + n_num)] per ask in the reference's RNG order
 *            (probability_distributions.py:87,100,138-144): C for rng.choice, then C per
 *            categorical param in column order, then an [n_num, C] block.
 *   out_x    [n_asks, n_cols] chosen candidate (internal representation); NULL = leave the results on the device
 *            (tpe_result_device_ptrs): a multi-GPU caller gathers them with NCCL without a host bounce
 *   out_acq  [n_asks] its acquisition value (may be NULL)
 *   out_best [n_asks] its candidate index (may be NULL) */
int tpe_sample_and_select(tpe_ctx* ctx, const double* uniforms, int64_t n_asks, double* out_x,
                          double* out_acq, int64_t* out_best);

/* The same in two halves: tpe_sample_and_select_async queues the work (and the copy of the results into page-locked
 * memory of the context) and returns; tpe_collect waits for it and hands the results out.  A caller that knows the
 * next suggestion's inputs early -- the sampler at `tell` time: the history with the finished trial, the generator
 * where the last ask left it (BaseSampler.after_trial, optuna/samplers/_base.py:178-203, runs before the next
 * Study.ask) -- overlaps the device work with its own host work; results are those of tpe_sample_and_select.
 * `uniforms` is read before tpe_sample_and_select_async returns.  Any tpe_prepare abandons uncollected results. */
int tpe_sample_and_select_async(tpe_ctx* ctx, const double* uniforms, int64_t n_asks);
int tpe_collect(tpe_ctx* ctx, double* out_x, double* out_acq, int64_t* out_best);

/* ONE suggestion over several GPUs (SURVEY section 8e, the alternative for a single ask): every rank holds the whole
 * history and builds both estimators (cheap), but evaluates g(x) -- the C x K x P grid -- only over its slice of the
 * above kernels.  tpe_set_kernel_shard(rank, world) selects the slice for the following calls (world = 1: off).
 * tpe_sample_and_partial replaces tpe_sample_and_select: candidates (every rank draws the same ones from the same
 * uniforms), l(x) in full, g(x) over the slice, reduced to one (max, sum) pair per candidate:
 *   *d_partials  device pointer, [n_asks * C] double2 padded to *stride pairs.
 * The caller gathers the partials of all ranks into one device buffer [world][*stride] double2 (ncclAllGather) and
 * calls tpe_finish_from_partials on every rank: log-sum-exp across ranks in rank order, acquisition, argmax -- the
 * same numbers on every rank.  Multivariate suggestions over continuous parameters only (TPE_E_STATE otherwise). */
int tpe_set_kernel_shard(tpe_ctx* ctx, int32_t rank, int32_t world);
int tpe_sample_and_partial(tpe_ctx* ctx, const double* uniforms, int64_t n_asks, double** d_partials, int64_t* stride);
int tpe_finish_from_partials(tpe_ctx* ctx, const double* d_gathered, int32_t world, double* out_x, double* out_acq,
                             int64_t* out_best);

/* Device pointers of the results of the last tpe_sample_and_select: out_x [n_asks, n_cols], out_acq [n_asks],
 * out_best [n_asks] (valid until the next call on the context; the work has completed when that call returned). */
int tpe_result_device_ptrs(tpe_ctx* ctx, double** out_x, double** out_acq, int64_t** out_best);

/* One-call convenience = prepare + build + sample_and_select (TPESampler._sample, sampler.py:523-560). */
int tpe_suggest(tpe_ctx* ctx, const tpe_cfg* cfg, const int32_t* cols, int32_t n_cols,
                const double* w_below, const double* w_above, const double* uniforms,
                int64_t n_asks, double* out_x, double* out_acq, int64_t* out_best);

/* Univariate TPE (multivariate = 0, the reference's default): the n_cols sample_independent calls of ONE trial
 * (sampler.py:458-491, one TPESampler._sample per parameter) evaluated together.  Column cols[j] gets its own pair
 * of 1-D estimators (the split is shared: it does not depend on the parameter), its own C candidates from
 * uniforms[j * 2C, (j + 1) * 2C) -- C for rng.choice, then C for the value, the order a sequence of per-parameter
 * calls consumes the generator -- and its own argmax; the columns run concurrently on the device.
 * uniforms == NULL: the n_cols * 2C uniforms staged by tpe_stage_uniforms_mt19937.
 * TPE_E_STATE ("not batchable") when the columns cannot share a split (a parameter absent from some trials) or the
 * history is multi-objective: the caller then makes the per-parameter calls.
 *   out_x [n_cols] chosen value per column (internal representation); out_acq, out_best [n_cols] may be NULL. */
int tpe_suggest_univariate_batch(tpe_ctx* ctx, const tpe_cfg* cfg, const int32_t* cols, int32_t n_cols,
                                 const double* w_below, const double* w_above, const double* uniforms,
                                 double* out_x, double* out_acq, int64_t* out_best);

/* The same in two halves (as tpe_sample_and_select_async / tpe_collect): queue the whole batch and return; collect
 * waits and hands the results out.  Only for trials whose selected parameters are all continuous (the path that runs
 * stage by stage over all columns); TPE_E_STATE "not batchable asynchronously" otherwise.  `uniforms`, `w_below` and
 * `w_above` are read before the call returns. */
int tpe_suggest_univariate_batch_async(tpe_ctx* ctx, const tpe_cfg* cfg, const int32_t* cols, int32_t n_cols,
                                       const double* w_below, const double* w_above, const double* uniforms);
int tpe_collect_univariate(tpe_ctx* ctx, double* out_x, double* out_acq, int64_t* out_best);

/* Optional: start the upload of the uniforms of the NEXT tpe_sample_and_select early (e.g. right
 * after tpe_prepare, so that the copy overlaps tpe_build).  `count` doubles are copied from
 * `uniforms` on a side stream; tpe_sample_and_select called with the same pointer and the matching
 * count then skips its own copy.  Purely a latency hint: no effect on results.  The reference has no
 * counterpart (its uniforms never leave the host, probability_distributions.py:86-152). */
int tpe_stage_uniforms(tpe_ctx* ctx, const double* uniforms, int64_t count);

/* Device-side uniforms: generate the next `count` outputs of numpy.random.RandomState.random_sample
 * (MT19937, legacy 53-bit doubles) on the GPU, after discarding `skip` of them, straight into the
 * buffer tpe_sample_and_select reads -- the exact stream the reference draws on the host
 * (probability_distributions.py:87,100,138-144), without the host RNG (0.45 ms per config-2 ask) and
 * without the upload.  key[624] / pos are RandomState.get_state()[1:3].  The following
 * tpe_sample_and_select must be called with uniforms == NULL and count == n_asks * per_ask.
 * tpe_rng_state returns the generator state after the (skip + count) draws, for set_state().
 * key == NULL continues from the state the previous staged draw ended in (it is kept on the device), so a
 * caller that owns the generator exclusively can defer get_state()/set_state() until somebody else needs it. */
int tpe_stage_uniforms_mt19937(tpe_ctx* ctx, const uint32_t* key, int32_t pos, int64_t skip, int64_t count);
int tpe_rng_state(tpe_ctx* ctx, uint32_t* key_out, int32_t* pos_out);
/* The same state where it lives: 625 words (key[624], pos) in device memory.  For multi-GPU plumbing -- the rank that
 * drew the LAST stretch of a batch broadcasts its end state into every rank's buffer (NCCL, device to device), so all
 * ranks continue as one generator that drew everything (optuna_b200/dist.py).  The library forgets its host copy. */
int tpe_rng_state_device(tpe_ctx* ctx, uint32_t** state625);
/* Inspection: the first `count` staged uniforms (device-generated or uploaded). */
int tpe_get_uniforms(tpe_ctx* ctx, double* out, int64_t count);

/* Page-locked host memory for buffers handed to tpe_sample_and_select / tpe_suggest (uniforms): a copy
 * from pinned memory is a true asynchronous DMA, a copy from pageable memory is staged by the host
 * thread first.  Optional; any host pointer is accepted everywhere. */
int tpe_host_alloc(tpe_ctx* ctx, size_t bytes, void** out);
int tpe_host_free(tpe_ctx* ctx, void* p);

/* ---- parity / inspection entry points (used by tests and by custom _parzen_estimator_cls-style
 * consumers, sampler.py:358-359) ------------------------------------------------------------- */
/* Shapes of the last tpe_prepare / tpe_suggest. */
int tpe_get_split_info(tpe_ctx* ctx, tpe_split_info* info);
/* Index lists produced by the last tpe_prepare (ascending trial order). */
int tpe_get_split(tpe_ctx* ctx, int64_t* below_rows, int64_t* above_rows);
/* Estimator parameters of the last tpe_build.  which: 0 = below, 1 = above.
 * weights [K]; mu, sigma [K, n_cols] (categorical columns hold the observed choice index / 0);
 * K = n_obs + 1.  Any pointer may be NULL. */
int tpe_get_mixture(tpe_ctx* ctx, int which, double* weights, double* mu, double* sigma);
/* MOTPE: raw hypervolume weights of ALL below trials (length n_below_all) of the last tpe_build. */
int tpe_get_mo_weights(tpe_ctx* ctx, double* weights);
/* Candidates / log-densities of the last tpe_sample_and_select (all asks).
 * samples [n_asks * C, n_cols]; logl, logg [n_asks * C].  Any pointer may be NULL. */
int tpe_get_candidates(tpe_ctx* ctx, double* samples, double* logl, double* logg);
/* log-density of arbitrary points under the last-built estimator
 * (replaces _ParzenEstimator.log_pdf, parzen_estimator.py:84-86).  x [n, n_cols]. */
int tpe_logpdf(tpe_ctx* ctx, int which, const double* x, int64_t n, double* out);

/* CUDA-event timing (ms, on the context stream) of the stages of the last prepare / build /
 * sample_and_select sequence: [0] split, [1] estimator build, [2] uniforms H2D, [3] sample,
 * [4] log-density under l(x), [5] main log-density kernel under g(x), [6] its fix-up pass,
 * [7] select, [8] first-to-last span.  launches = kernels launched by the sequence. */
int tpe_last_timing(tpe_ctx* ctx, float* ms9, int32_t* launches);
/* Peak-probe: fp64 FMA throughput of this device (TFLOP/s), measured by a dependent-chain-free
 * DFMA kernel; used by bench.py as the compute-roof denominator. */
int tpe_probe_fp64_tflops(tpe_ctx* ctx, double* tflops);
/* Which kernel variant the last log-density pass used (static string). */
const char* tpe_last_logpdf_kernel(tpe_ctx* ctx);

/* ---- PED-ANOVA hyperparameter importance ---------------------------------------------------------------------
 * Replaces PedAnovaImportanceEvaluator.evaluate after its search-space walk (optuna/importance/_ped_anova/
 * evaluator.py:222-266): _get_filtered_trials (importance/_base.py:145-156), _QuantileFilter.filter
 * (evaluator.py:37-55), the binning of scott_parzen_estimator.py:90-135, _ScottParzenEstimator
 * (scott_parzen_estimator.py:16-87) and _compute_pearson_divergence (evaluator.py:196-220), on the resident history.
 * Fields are the evaluator's constructor arguments and its fixed settings (evaluator.py:141-172):
 * prior_weight (> 0; 1.0), min_n_top (2) and n_steps (<= 128; 50). */
typedef struct {
  double target_quantile, region_quantile, prior_weight;
  int32_t evaluate_on_local, min_n_top, n_steps;
} tpe_ped_cfg;

/* A row is kept when its category is TPE_CAT_COMPLETE, none of cols[] is NaN and its loss is finite.  The loss is
 * key[r][0] (the sign-normalised objective) or loss[r] (a host-evaluated target; length = history size).  The target
 * set is the kept rows with loss <= the k-th smallest kept loss, k = max(min_n_top - 1, ceil(q * n) - 1) at
 * q = target_quantile; the region set likewise at region_quantile, or every kept row when it is 1.0.
 *   cols       [n_cols] columns to filter on and evaluate
 *   grids      [n_cols][n_steps] np.linspace grid of each numerical column (log domain for log columns), as the host
 *              computes it (scott_parzen_estimator.py:96-105); ignored for categorical columns; may be NULL when
 *              every column is categorical
 *   n_grid     [n_cols] bins per column: <= n_steps, or n_choices for a categorical column
 *   loss       [history size] or NULL = key[:, 0]
 *   out_importance [n_cols] (n_target / n_region)^2 * Pearson divergence; all 0 when n_kept <= min_n_top
 *   out_n      [3] kept, target, region (target = region = 0 when n_kept <= min_n_top)
 *   out_counts optional [n_cols][2][max n_grid]: target / region histograms (inspection)
 * Runs on the context stream, returns when the results are on the host, and leaves the history, the split and the
 * estimators of the suggestion path untouched. */
int tpe_ped_anova(tpe_ctx* ctx, const tpe_ped_cfg* cfg, const int32_t* cols, int32_t n_cols, const double* grids,
                  const int32_t* n_grid, const double* loss, double* out_importance, int64_t* out_n,
                  int32_t* out_counts);

#ifdef __cplusplus
}
#endif
#endif /* OPTUNA_B200_TPE_H_ */
