// C ABI of libtpe_b200.so (see include/optuna_b200_tpe.h) -- host orchestration of the kernels in
// tpe_kernels.cuh.  No torch types, no Python: plain pointers and sizes.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stddef.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <mutex>
#include <thread>
#include <set>
#include <string>
#include <vector>

#include "../../include/optuna_b200_tpe.h"
#include "tpe_kernels.cuh"
#include "tpe_motpe_kernels.cuh"
#include "tpe_uni.cuh"
#include "tpe_mixed.cuh"
#include "tpe_tcscreen.cuh"
#include "tpe_unib.cuh"
#include "tpe_importance.cuh"
// Lab build (-DTPE_LAB): the experimental grid kernels and the timing-attribution variants measured in
// profiles/r1_variants.md / r2_variants.md, selectable by environment variables.  Some of them switch parts of the
// log-sum-exp off (wrong results by design).  The product library contains none of them.
#ifdef TPE_LAB
#include "tpe_mma2.cuh"
#include "tpe_mma3.cuh"
#include "tpe_screen.cuh"
#endif

using namespace tpe;

namespace {

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  bool owned = true;   // false: a view of another context's buffer (batched univariate sub-contexts)
  void alias(void* q, size_t bytes) {
    if (owned && p) cudaFree(p);
    p = q;
    cap = bytes;
    owned = false;
  }
  cudaError_t ensure(size_t bytes) {
    if (!owned) { p = nullptr; cap = 0; owned = true; }
    if (bytes <= cap) return cudaSuccess;
    // 12 % headroom: a study grows by one trial per suggestion, and a cudaFree + cudaMalloc of a 50 MB table in the
    // middle of an ask costs milliseconds (and synchronises the device)
    size_t want = std::max(bytes + bytes / 8, cap + cap / 2);
    want = (want + 255) & ~(size_t)255;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  // grow while keeping the first `keep` bytes
  cudaError_t grow(size_t bytes, size_t keep, cudaStream_t st) {
    if (bytes <= cap) return cudaSuccess;
    size_t want = std::max(bytes, cap * 2);
    want = (want + 255) & ~(size_t)255;
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, want);
    if (e != cudaSuccess) return e;
    if (p && keep) e = cudaMemcpyAsync(q, p, keep, cudaMemcpyDeviceToDevice, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (p) cudaFree(p);
    p = q;
    cap = want;
    return e;
  }
  template <class T>
  T* as() const { return reinterpret_cast<T*>(p); }
  void release() {
    if (p && owned) cudaFree(p);
    p = nullptr;
    cap = 0;
    owned = true;
  }
};

struct Estimator {
  int64_t n = 0, K = 0;
  DevBuf rows, pos, wstage, wpart, w, logw, cdf, mu, sigma, cst_part, cst, tabp, tabc, colprm, tab, part, fix;
  DevBuf tab32, tab64p, d32;   // fp32-screening copies (tpe_screen.cuh)
  DevBuf cls, dtab, offgrid;   // tabulated discrete columns (multivariate)
  DevBuf tabm, hb, ckk;        // tensor-core kernel: fragment-major table, |mu''|^2 / 2, cst - |mu''|^2 / 2
  DevBuf uord, us32, usmi, usc, umeta;  // univariate 1-D grid (tpe_uni.cuh): sorted order and sorted tables
  DevBuf ucoef, ubox, ubstart, utlist;  // ... and the fast Gauss transform of the floor-bandwidth kernels
  bool fgt = false;
  DevBuf tcs_h, tcs_ak, tcs_ak64;       // bf16 tensor-core screen of the multivariate grid (tpe_tcscreen.cuh)
  bool tcs = false;
  int64_t tcs_kpad = 0;
  DevBuf mxc, mxd;                      // mixed spaces, many candidates (tpe_mixed.cuh): kernel-minor tables
  bool mixed = false;
  int64_t mix_kstride = 0;
  bool uni_ready = false;
  bool mma = false;            // tables above are valid for this build
  bool screen_ready = false;
  int nsplit = 0;
  void release() {
    for (DevBuf* b : {&uord, &us32, &usmi, &usc, &umeta, &ucoef, &ubox, &ubstart, &utlist, &mxc, &mxd, &tcs_h, &tcs_ak, &tcs_ak64, &tabm, &hb, &ckk, &cls, &dtab, &offgrid, &tab32, &tab64p, &d32, &rows, &pos, &wstage, &wpart, &w, &logw, &cdf, &mu, &sigma, &cst_part, &cst, &tabp, &tabc, &colprm, &tab,
                      &part, &fix})
      b->release();
  }
};

}  // namespace

struct tpe_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  // the above-set estimator is built on a second stream while the main stream builds l(x), samples
  // the candidates and evaluates them under l(x); joined before the first consumer of est[1]
  cudaStream_t stream2 = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  bool above_pending = false;
  // tpe_suggest uploads the uniforms on a third stream before the split starts
  cudaStream_t stream3 = nullptr;
  cudaEvent_t ev_u = nullptr;
  const double* u_staged = nullptr;
  int64_t u_staged_count = 0;
  bool u_device_rng = false;     // U was filled by k_mt19937_uniform (tpe_stage_uniforms_mt19937)
  DevBuf mt_state;               // 624 state words + pos: generator state after the staged uniforms
  // Speculation: while an ask is evaluated, the uniforms of the NEXT ask (same count) are generated from
  // the end state into U2 / mt_spec.  The next tpe_stage_uniforms_mt19937 adopts them if the caller's
  // generator is exactly in that state (mt_host, as returned by tpe_rng_state); otherwise they are dropped.
  DevBuf U2, mt_spec;
  DevBuf mt_jump, mt_tmp;        // jump-ahead polynomials (kMtJumpTable) / end state of the multi-CTA generator
  bool mt_jump_ready = false;
  cudaEvent_t ev_spec = nullptr;
  bool spec_pending = false, mt_host_valid = false;
  int64_t spec_count = 0;
  uint32_t* mt_host = nullptr;   // page-locked host copy of mt_state (625 words), read back with the results of the ask
                                 // (page-locked: a copy into pageable memory would make the asynchronous entry points wait)
  cudaEvent_t ev[9] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  std::mutex mu;
  std::string err;
  int sm_count = 148;

  // search space
  std::vector<tpe_param_desc> space;
  std::vector<double> cat_dist_h;
  std::vector<int64_t> cat_dist_off;
  DevBuf cat_dist;

  // history
  DevBuf X, cat, key, vals;
  int32_t M = 1;                 // objectives (>= 2: MOTPE)
  std::vector<int8_t> cat_h;     // host mirror of the categories (MOTPE list building)
  int64_t cat_cnt[5] = {0, 0, 0, 0, 0};  // trials per category incl. TPE_CAT_EXCLUDED (sizes of the split without a read-back)
  // the split depends on the history and n_below only (not on the selected columns, unless rows lack
  // parameters): consecutive tpe_prepare calls on the same history -- the P sample_independent calls of a
  // univariate trial -- reuse it
  uint64_t hist_version = 0, split_version = 0;
  int64_t split_n_below = -1;
  bool split_valid = false;
  int64_t N = 0;
  // MOTPE scratch
  DevBuf mo_list, mo_alive, mo_dom, mo_first, mo_rank, mo_ctr, mo_tie, mo_ntie, mo_lexpos, mo_isdup, mo_sorted,
      mo_uniq, mo_nuniq, mo_ref, mo_removed, mo_contrib, mo_state, mo_arena, mo_chosen, mo_diag, mo_w, mo_table, mo_sample,
      mo_surv, mo_nsurv, mo_fv, mo_ps, mo_map, mo_front, mo_head;
  bool mo_weights_ready = false;
  std::vector<uint8_t> col_missing, col_oor, col_offgrid;   // col_offgrid: a step column holds a value off its grid
  bool history_set = false;

  // current call
  bool prepared = false, built = false, sampled = false;
  tpe_cfg cfg{};
  std::vector<ColMeta> cols_h;
  DevBuf cols;
  int32_t pc = 0, ncont = 0, ndisc = 0, ncat = 0, nnum = 0, pb = 0;
  int64_t tab_doubles = 0;
  int64_t dtab_doubles = 0;  // cell-mass tables of tabulated discrete columns
  bool fast = false;
  bool uni_fast = false;   // one continuous column, univariate: the sorted 1-D grid kernel (tpe_uni.cuh)
  bool cands_sorted = false;
  DevBuf uxs, ucidx;
  int fast_mode = 0;  // 0 generic, 1 PAIR (sigma per kernel), 2 CONST (sigma per column)
  tpe_split_info info{};
  DevBuf row_ok, member, counts, split_work, below_all;
  Estimator est[2];
  DevBuf sort_val, sort_idx, sort_work;

  // candidates
  int64_t n_asks = 0, Ct = 0, ct_stride = 0;
  DevBuf U, S, xT, oob, logl, logg, out_x, out_acq, out_best, x64s, x32s, e32s, gmax, lse_gmax;
  bool screen_attr_set = false;
  float ms[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  int32_t launches = 0;
  const char* last_kernel = "none";
  int32_t launch_counter = 0;
  std::set<const void*> prepared_cfgs;
  // batched univariate suggestions (tpe_suggest_univariate_batch): one light sub-context per column -- own streams,
  // own estimator / candidate buffers, views of this context's history and split
  std::vector<tpe_ctx*> uni_sub;
  cudaEvent_t ev_uni = nullptr;
  bool is_sub = false;
  // staged univariate batch (tpe_unib.cuh): one arena carved per call + the sorted orders kept between calls
  DevBuf ub_arena, ub_ord_a, ub_ord_b, ub_wstage;
  int ub_ord_cur = 0;                  // which of ub_ord_a / ub_ord_b holds the latest above orders
  uint64_t ub_ord_seq = 0, ub_ord_lineage = 0;
  int64_t ub_ord_K = -1, ub_ord_ks = 0;
  std::vector<int32_t> ub_ord_cols;
  int ub_sort_g = 0;
  bool mixed_ok = false;         // the selected columns suit k_logpdf_mixed (setup_columns)
  std::vector<MixCol> mixcols_h;
  DevBuf mixcols;
  int mix_ncont = 0, mix_nd = 0, mix_tabd = 0;
  bool user_points = false;      // the resident candidates came through tpe_logpdf, not from k_sample
  static constexpr size_t kUpSlot = 8192;     // page-locked staging of small history uploads (upload_history)
  static constexpr int kUpSlots = 16;
  void* up_host = nullptr;
  cudaEvent_t up_ev[kUpSlots] = {};
  bool up_used[kUpSlots] = {};
  int up_next = 0;
  // one suggestion over several GPUs: this context evaluates g(x) over its slice of the above kernels only
  // (tpe_set_kernel_shard, tpe_sample_and_partial, tpe_finish_from_partials)
  int32_t kshard_rank = 0, kshard_world = 1;
  DevBuf kpart;
  bool partial_ready = false;
  bool deferred = false;         // tpe_sample_and_select_async issued, tpe_collect not yet called
  int64_t deferred_uni = 0;      // tpe_suggest_univariate_batch_async issued (columns), not yet collected
  bool deferred_uni_rng = false;
  bool issued_dev_rng = false;
  void* res_host = nullptr;      // page-locked staging of deferred results
  size_t res_host_cap = 0;
  int sort_cta_cap = 0;          // sub-contexts: CTAs of a cooperative sort (several sorts share the GPU)
  // incremental sorted orders (univariate batch): the parent compares the above rows of this call with the previous
  // call's; every column context then updates its order instead of sorting (k_rows_delta / k_order_update)
  uint64_t hist_lineage = 0;     // changes whenever rows the estimators can see are replaced (not on appends)
  DevBuf uni_prev_rows, uni_mode, uni_work;
  int64_t uni_prev_n = -1;
  uint64_t uni_prev_lineage = 0;
  const int* uni_mode_ptr = nullptr;   // sub-contexts: the parent's mode word, or nullptr (always sort)
  uint64_t uni_seq = 0;                // batch calls so far (sub-contexts: the running call's number)
  uint64_t uni_ord_seq = 0;            // sub-contexts: the call that left the cached order of est[1] ...
  uint64_t uni_ord_lineage = 0;        // ... and what else it belongs to
  int32_t uni_ord_col = -1;
  int64_t uni_ord_K = -1;
  // PED-ANOVA importance (tpe_ped_anova): scratch of its own, nothing a suggestion reads
  DevBuf ped_member, ped_okey, ped_work, ped_cols, ped_grid, ped_counts, ped_pdf, ped_imp, ped_loss;
};

namespace {

int fail(tpe_ctx* c, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (c) c->err = buf;
  return code;
}

#define CU(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess)                                                                         \
      return fail(ctx, e_ == cudaErrorMemoryAllocation ? TPE_E_NOMEM : TPE_E_CUDA, "%s failed: %s (%s:%d)", \
                  #call, cudaGetErrorString(e_), __FILE__, __LINE__);                              \
  } while (0)

// slot of a history category in cat_cnt: anything outside 0..3 is TPE_CAT_EXCLUDED
inline int cat_slot(int8_t c) { return (c >= 0 && c <= 3) ? c : 4; }

inline int grid_for(int64_t work, int threads, int cap) {
  int64_t g = (work + threads - 1) / threads;
  if (g < 1) g = 1;
  if (g > cap) g = cap;
  return (int)g;
}

template <class T>
constexpr T round_up(T v, T m) { return (v + m - 1) / m * m; }

// ---- fast-kernel configuration table ------------------------------------------------------------
struct FastCfg {
  int pb, cands_per_cta, nt, tk, st, minb;
  size_t smem;
  void (*launch)(dim3, size_t, cudaStream_t, const void*, const double*, int64_t, const double2*, const double*,
                 int64_t, int64_t, double, double2*, unsigned long long*);
  cudaError_t (*prepare)();
};

template <int PB, int PS, int RC, int NT, int TK, int ST, bool PAIR, int MINB>
struct FastInst {
  static constexpr size_t smem = (size_t)ST * TK * PB * (PAIR ? 16 : 8) + (size_t)ST * TK * 8 + (size_t)ST * 8;
  static void launch(dim3 grid, size_t sm, cudaStream_t st, const void* tab, const double* cst, int64_t Kf,
                     const double2* colprm, const double* xT, int64_t ct_stride, int64_t kps, double skip,
                     double2* part, unsigned long long*) {
    k_logpdf_fast<PB, PS, RC, NT, TK, ST, PAIR, MINB>
        <<<grid, NT, sm, st>>>(tab, cst, Kf, colprm, xT, ct_stride, kps, skip, part);
  }
  static cudaError_t prepare() {
    return cudaFuncSetAttribute(k_logpdf_fast<PB, PS, RC, NT, TK, ST, PAIR, MINB>,
                                cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  }
  static FastCfg cfg() { return FastCfg{PB, (NT / 32) * (32 / PS) * RC, NT, TK, ST, MINB, smem, &launch, &prepare}; }
};

// Tensor-core (DMMA) instances of the CONST kernel: same launch signature (tab = fragment-major table,
// cst = ckk, Kf = kernels rounded up to 8).
constexpr int kMmaKPad = 32;  // kernels are padded to 8 * KG (KG <= 4)
template <int PB, int M, int KG, int NT, int TK, int ST, int MINB, int DBG = 0>
struct MmaInst {
  static constexpr size_t smem = (size_t)ST * TK * PB * 8 + (size_t)ST * TK * 8 + (size_t)ST * 16;
  static void launch(dim3 grid, size_t sm, cudaStream_t st, const void* tab, const double* cst, int64_t Kf,
                     const double2* colprm, const double* xT, int64_t ct_stride, int64_t kps, double skip,
                     double2* part, unsigned long long* gmax) {
    // near tier: within ln K + 17.5 of the reference max (see LseTier); TPE_TNEAR_DELTA shrinks it for
    // timing experiments only (the accuracy bound no longer holds)
#ifdef TPE_LAB
    static const double delta = [] { const char* v = getenv("TPE_TNEAR_DELTA"); return v ? atof(v) : 0.0; }();
#else
    constexpr double delta = 0.0;
#endif
    k_logpdf_mma<PB, M, KG, NT, TK, ST, MINB, DBG><<<grid, NT, sm, st>>>(static_cast<const double*>(tab), cst, Kf, colprm,
                                                                        xT, ct_stride, kps, skip, part, gmax,
                                                                        skip - 12.5 - delta);
  }
  static cudaError_t prepare() {
    return cudaFuncSetAttribute(k_logpdf_mma<PB, M, KG, NT, TK, ST, MINB, DBG>,
                                cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  }
  static FastCfg cfg() { return FastCfg{PB, (NT / 32) * 8 * M, NT, TK, ST, MINB, smem, &launch, &prepare}; }
};
#ifdef TPE_LAB
// round-2 kernel (tpe_mma2.cuh): OPT bit 0 = seeded base, bit 1 = pipelined classification
template <int PB, int M, int KG, int NT, int TK, int ST, int MINB, int OPT>
struct MmaInst2 {
  static constexpr size_t smem = (size_t)ST * TK * PB * 8 + (size_t)ST * TK * 8 + (size_t)ST * 16;
  static void launch(dim3 grid, size_t sm, cudaStream_t st, const void* tab, const double* cst, int64_t Kf,
                     const double2* colprm, const double* xT, int64_t ct_stride, int64_t kps, double skip,
                     double2* part, unsigned long long* gmax) {
    // OPT bit 2 (budgeted log-sum-exp): the last argument is the fp32-tier budget of one lane, 2e-7 / (4 * k-splits)
    const double last = (OPT & 4) ? 2e-7 / (4.0 * grid.y) : skip - 12.5;
    k_logpdf_mma2<PB, M, KG, NT, TK, ST, MINB, OPT><<<grid, NT, sm, st>>>(static_cast<const double*>(tab), cst, Kf, colprm,
                                                                         xT, ct_stride, kps, skip, part, gmax, last);
  }
  static cudaError_t prepare() {
    return cudaFuncSetAttribute(k_logpdf_mma2<PB, M, KG, NT, TK, ST, MINB, OPT>,
                                cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  }
  static FastCfg cfg() { return FastCfg{PB, (NT / 32) * 8 * M, NT, TK, ST, MINB, smem, &launch, &prepare}; }
};
// warp-compacted exact tier (tpe_mma3.cuh)
template <int PB, int KG, int NT, int TK, int ST, int MINB>
struct MmaInst3 {
  static constexpr size_t smem = (size_t)ST * TK * PB * 8 + (size_t)ST * TK * 8 + (size_t)ST * 16 + (size_t)(NT / 32) * kQWarpBytes;
  static void launch(dim3 grid, size_t sm, cudaStream_t st, const void* tab, const double* cst, int64_t Kf,
                     const double2* colprm, const double* xT, int64_t ct_stride, int64_t kps, double skip,
                     double2* part, unsigned long long* gmax) {
    k_logpdf_mma3<PB, KG, NT, TK, ST, MINB><<<grid, NT, sm, st>>>(static_cast<const double*>(tab), cst, Kf, colprm, xT,
                                                                 ct_stride, kps, skip, part, gmax, skip - 12.5);
  }
  static cudaError_t prepare() {
    return cudaFuncSetAttribute(k_logpdf_mma3<PB, KG, NT, TK, ST, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)smem);
  }
  static FastCfg cfg() { return FastCfg{PB, (NT / 32) * 8, NT, TK, ST, MINB, smem, &launch, &prepare}; }
};
const FastCfg kMma32V3[] = {
    MmaInst3<32, 2, 512, 128, 3, 2>::cfg(),  // i
    MmaInst3<32, 4, 256, 128, 3, 2>::cfg(),  // j: 4 kernel groups in flight, 16 warps / SM
    MmaInst3<32, 2, 256, 128, 3, 3>::cfg(),  // k: 3 CTAs x 8 warps
};
const FastCfg kMma32V2[] = {
    MmaInst2<32, 1, 2, 512, 128, 3, 2, 1>::cfg(),  // 8: seed
    MmaInst2<32, 1, 2, 512, 128, 3, 2, 3>::cfg(),  // 9: seed + pipe
    MmaInst2<32, 1, 2, 512, 128, 3, 2, 2>::cfg(),  // a: pipe
    MmaInst2<32, 1, 4, 256, 128, 3, 2, 3>::cfg(),  // b: seed + pipe, 4 kernel groups in flight, 16 warps / SM
    MmaInst2<32, 1, 2, 256, 128, 3, 3, 3>::cfg(),  // c: seed + pipe, 3 CTAs x 8 warps
    MmaInst2<32, 1, 2, 512, 128, 3, 2, 4>::cfg(),  // d: budgeted log-sum-exp
    MmaInst2<32, 1, 2, 512, 128, 3, 2, 5>::cfg(),  // e: budgeted + seed
    MmaInst2<32, 1, 4, 256, 128, 3, 2, 5>::cfg(),  // f: budgeted + seed, KG = 4, 16 warps / SM
    MmaInst2<32, 1, 2, 512, 128, 3, 2, 8>::cfg(),  // g: near terms parked in a lane-private local-memory buffer
    MmaInst2<32, 1, 2, 512, 128, 3, 2, 9>::cfg(),  // h: g + seed
};
#endif  // TPE_LAB
// Measured at config 2 (profiles/r1_variants.md): 32 warps/SM with two kernel groups in flight per
// warp is the best of the tilings tried (1.17 ms); two candidate groups per warp (M = 2) halve the
// CTA count and lose.
//                                   PB M KG  NT   TK ST MINB
const FastCfg kMmaBig[] = {
    MmaInst<8, 1, 4, 256, 512, 3, 2>::cfg(), MmaInst<16, 1, 4, 256, 256, 3, 2>::cfg(),
    MmaInst<32, 1, 2, 512, 128, 3, 2>::cfg(), MmaInst<64, 1, 2, 256, 64, 3, 1>::cfg(),
};
const FastCfg kMmaSmall[] = {
    MmaInst<8, 1, 4, 64, 512, 3, 4>::cfg(), MmaInst<16, 1, 4, 64, 256, 3, 4>::cfg(),
    MmaInst<32, 1, 4, 64, 128, 3, 4>::cfg(), MmaInst<64, 1, 2, 64, 64, 3, 3>::cfg(),
};
#ifdef TPE_LAB
const FastCfg kMma32Variants[] = {
    MmaInst<32, 1, 4, 256, 128, 3, 2>::cfg(), MmaInst<32, 1, 2, 256, 128, 3, 2>::cfg(),
    MmaInst<32, 1, 1, 512, 128, 3, 2>::cfg(), MmaInst<32, 1, 2, 256, 128, 2, 3>::cfg(),
    MmaInst<32, 1, 2, 512, 128, 3, 2>::cfg(), MmaInst<32, 1, 2, 512, 128, 3, 2, 1>::cfg(),
    MmaInst<32, 1, 2, 512, 128, 3, 2, 2>::cfg(), MmaInst<32, 1, 4, 256, 128, 3, 2, 1>::cfg(),
};
#endif  // TPE_LAB

const FastCfg* pick_mma(int pb, int64_t Ct) {
  const bool small = Ct <= 64;
#ifdef TPE_LAB
  if (pb == 32 && !small) {
    const char* v = getenv("TPE_MMA_VARIANT");
    if (v && v[0] >= '0' && v[0] <= '7') return &kMma32Variants[v[0] - '0'];
    if (v && v[0] == '8') return &kMma32V2[0];
    if (v && v[0] == '9') return &kMma32V2[1];
    if (v && v[0] >= 'a' && v[0] <= 'h') return &kMma32V2[2 + (v[0] - 'a')];
    if (v && v[0] >= 'i' && v[0] <= 'k') return &kMma32V3[v[0] - 'i'];
  }
#endif
  const FastCfg* tabs = small ? kMmaSmall : kMmaBig;
  for (int i = 0; i < 4; ++i)
    if (tabs[i].pb == pb) return &tabs[i];
  return nullptr;
}

// "big": many candidates (c-tiles of `cands_per_cta`, kernels split over blockIdx.y);
// "small": a single ask with few candidates -- one warp per CTA, the grid splits the kernel axis.
// CONST = one sigma per column (multivariate TPE), PAIR = sigma per kernel (univariate TPE).
//                 PB PS RC  NT    TK ST  PAIR MINB
// Measured at config 2 (profiles/r1_variants.md): one candidate per lane with 16 warps/SM beats the
// lane-split tilings (shuffles cost ~6 clk each on the shared pipe) and the 2-candidate tiling
// (8 warps/SM cannot hide the DADD->DFMA latency).
const FastCfg kConstBig[] = {
    FastInst<1, 1, 4, 256, 2048, 3, false, 2>::cfg(), FastInst<2, 1, 4, 256, 1024, 3, false, 2>::cfg(),
    FastInst<4, 1, 4, 256, 1024, 3, false, 2>::cfg(), FastInst<8, 1, 4, 256, 512, 3, false, 1>::cfg(),
    FastInst<16, 1, 2, 256, 256, 3, false, 2>::cfg(), FastInst<32, 1, 1, 512, 128, 3, false, 1>::cfg(),
    FastInst<64, 1, 1, 256, 64, 3, false, 1>::cfg(),
};
const FastCfg kPairBig[] = {
    FastInst<1, 1, 4, 256, 1024, 3, true, 2>::cfg(), FastInst<2, 1, 4, 256, 1024, 3, true, 1>::cfg(),
    FastInst<4, 1, 4, 256, 512, 3, true, 1>::cfg(),  FastInst<8, 1, 4, 256, 256, 3, true, 1>::cfg(),
    FastInst<16, 1, 4, 256, 128, 3, true, 1>::cfg(), FastInst<32, 1, 2, 256, 64, 3, true, 1>::cfg(),
    FastInst<64, 1, 1, 256, 32, 3, true, 1>::cfg(),
};
const FastCfg kConstSmall[] = {
    FastInst<1, 1, 1, 32, 1024, 2, false, 1>::cfg(), FastInst<2, 1, 1, 32, 512, 2, false, 1>::cfg(),
    FastInst<4, 1, 1, 32, 256, 2, false, 1>::cfg(),  FastInst<8, 1, 1, 32, 128, 2, false, 1>::cfg(),
    FastInst<16, 1, 1, 32, 64, 2, false, 1>::cfg(),  FastInst<32, 1, 1, 32, 32, 2, false, 1>::cfg(),
    FastInst<64, 1, 1, 32, 16, 2, false, 1>::cfg(),
};
const FastCfg kPairSmall[] = {
    FastInst<1, 1, 1, 32, 512, 2, true, 1>::cfg(), FastInst<2, 1, 1, 32, 256, 2, true, 1>::cfg(),
    FastInst<4, 1, 1, 32, 128, 2, true, 1>::cfg(), FastInst<8, 1, 1, 32, 64, 2, true, 1>::cfg(),
    FastInst<16, 1, 1, 32, 32, 2, true, 1>::cfg(), FastInst<32, 1, 1, 32, 16, 2, true, 1>::cfg(),
    FastInst<64, 1, 1, 32, 8, 2, true, 1>::cfg(),
};
#ifdef TPE_LAB
// tuning variants of the P = 32 CONST kernel, selectable with TPE_FAST_VARIANT=0..3 (experiments)
const FastCfg kConst32Variants[] = {
    FastInst<32, 1, 1, 256, 128, 3, false, 2>::cfg(),  // 0: 1 candidate / lane, 16 warps / SM
    FastInst<32, 1, 2, 256, 128, 3, false, 1>::cfg(),  // 1: 2 candidates / lane, 8 warps / SM
    FastInst<32, 2, 4, 256, 128, 3, false, 1>::cfg(),  // 2: params split over 2 lanes, 4 candidates
    FastInst<32, 4, 4, 256, 128, 3, false, 2>::cfg(),  // 3: params split over 4 lanes, 4 candidates
    FastInst<32, 1, 2, 320, 128, 3, false, 1>::cfg(),  // 4: 2 candidates / lane, 10 warps / SM
    FastInst<32, 1, 2, 384, 128, 3, false, 1>::cfg(),  // 5: 2 candidates / lane, 12 warps / SM
    FastInst<32, 1, 2, 128, 64, 3, false, 2>::cfg(),   // 6: 2 candidates / lane, 2 CTAs x 4 warps
    FastInst<32, 1, 1, 128, 64, 3, false, 4>::cfg(),   // 7: 4 CTAs x 4 warps
    FastInst<32, 1, 1, 256, 128, 2, false, 2>::cfg(),  // 8: 2 stages
    FastInst<32, 1, 1, 512, 128, 3, false, 1>::cfg(),  // 9: 1 CTA x 16 warps
};
#endif  // TPE_LAB
constexpr int kMaxFastP = 64;

int pick_pb(int ncont) {
  for (int pb : {1, 2, 4, 8, 16, 32, 64})
    if (ncont <= pb) return pb;
  return 0;
}
const FastCfg* pick_fast(int mode, int pb, int64_t Ct) {
  const bool small = Ct <= 128;
#ifdef TPE_LAB
  if (mode == 2 && pb == 32 && !small) {
    const char* v = getenv("TPE_FAST_VARIANT");
    if (v && v[0] >= '0' && v[0] <= '9') return &kConst32Variants[v[0] - '0'];
  }
#endif
  const FastCfg* tabs = (mode == 2) ? (small ? kConstSmall : kConstBig) : (small ? kPairSmall : kPairBig);
  for (int i = 0; i < 7; ++i)
    if (tabs[i].pb == pb) return &tabs[i];
  return nullptr;
}

// `count` outputs of the MT19937 stream after dropping `skip`, from the 625-word device state `state` (updated in
// place to the state after the draws).  Short stretches: one CTA walks the recurrence (k_mt19937_uniform).  Long
// ones (a batch of asks, or a rank's slice far into the batch): every CTA jumps to its own chunk
// (k_mt19937_uniform_mc) -- no serial prefix walk.
int launch_mt(tpe_ctx* ctx, cudaStream_t st, uint32_t* state, int64_t skip, int64_t count, double* out) {
  static const int64_t mc_min = [] { const char* v = getenv("TPE_MT_MC_MIN"); return v ? atoll(v) : (int64_t)400000; }();
  if (skip + count < mc_min) {
    k_mt19937_uniform<<<1, kMtThreads, 0, st>>>(state, reinterpret_cast<int*>(state + 624), skip, count, out);
    ctx->launch_counter++;
    CU(cudaGetLastError());
    return TPE_OK;
  }
  if (!ctx->mt_jump_ready) {
    CU(ctx->mt_jump.ensure(sizeof(kMtJumpTable)));
    CU(ctx->mt_tmp.ensure(625 * 4));
    CU(cudaMemcpyAsync(ctx->mt_jump.p, kMtJumpTable, sizeof(kMtJumpTable), cudaMemcpyHostToDevice, st));
    CU(cudaFuncSetAttribute(k_mt19937_uniform_mc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMtJumpSmem));
    ctx->mt_jump_ready = true;
  }
  const int64_t G = std::max<int64_t>(1, std::min<int64_t>(ctx->sm_count, (count + 16383) / 16384));
  const int64_t chunk = round_up<int64_t>((count + G - 1) / G, 256);
  const int64_t grid = (count + chunk - 1) / chunk;
  k_mt19937_uniform_mc<<<(unsigned)grid, kMtThreads, kMtJumpSmem, st>>>(state, skip, count, chunk, ctx->mt_jump.as<uint32_t>(),
                                                                       kMtJumpKMin, kMtJumpKMax, out,
                                                                       ctx->mt_tmp.as<uint32_t>());
  ctx->launch_counter++;
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(state, ctx->mt_tmp.p, 625 * 4, cudaMemcpyDeviceToDevice, st));
  return TPE_OK;
}

int join_above(tpe_ctx* ctx) {
  if (ctx->above_pending) {
    CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));
    ctx->above_pending = false;
  }
  return TPE_OK;
}
int set_device(tpe_ctx* ctx, bool join = true) {
  CU(cudaSetDevice(ctx->device));
  if (join) return join_above(ctx);
  return TPE_OK;
}

// A few rows from the host (the per-trial case) go through a slot of page-locked staging memory, without waiting: a
// copy from pageable memory would first wait for everything queued on the stream, i.e. for a suggestion that was
// queued ahead of time (tpe_sample_and_select_async) and must keep running while the caller goes on.
bool rows_fit_staging(const tpe_ctx* ctx, int64_t n) {
  return (size_t)n * ((size_t)ctx->space.size() * 8 + 16 + 1) + 64 <= tpe_ctx::kUpSlot;
}
int stage_rows(tpe_ctx* ctx, const double* X, const int8_t* category, const double* key, int64_t n, int64_t at) {
  const int64_t P = (int64_t)ctx->space.size();
  if (!ctx->up_host) {
    CU(cudaHostAlloc(&ctx->up_host, tpe_ctx::kUpSlot * tpe_ctx::kUpSlots, cudaHostAllocDefault));
    for (auto& e : ctx->up_ev) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  }
  const int slot = ctx->up_next;
  ctx->up_next = (slot + 1) % tpe_ctx::kUpSlots;
  if (ctx->up_used[slot]) CU(cudaEventSynchronize(ctx->up_ev[slot]));   // (its copies of kUpSlots uploads ago)
  char* h = static_cast<char*>(ctx->up_host) + (size_t)slot * tpe_ctx::kUpSlot;
  const size_t xb = (size_t)n * P * 8, kb = (size_t)n * 16;
  memcpy(h, X, xb);
  memcpy(h + xb, key, kb);
  memcpy(h + xb + kb, category, (size_t)n);
  CU(cudaMemcpyAsync(ctx->X.as<double>() + at * P, h, xb, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(ctx->key.as<double>() + at * 2, h + xb, kb, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(ctx->cat.as<int8_t>() + at, h + xb + kb, (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaEventRecord(ctx->up_ev[slot], ctx->stream));
  ctx->up_used[slot] = true;
  return TPE_OK;
}

int upload_history(tpe_ctx* ctx, const double* X, const int8_t* category, const double* key, int64_t n,
                   int64_t at, bool device_src) {
  const int64_t P = (int64_t)ctx->space.size();
  const int64_t total = at + n;
  CU(ctx->X.grow((size_t)std::max<int64_t>(total, 1) * P * 8, (size_t)at * P * 8, ctx->stream));
  CU(ctx->cat.grow((size_t)std::max<int64_t>(total, 1), (size_t)at, ctx->stream));
  CU(ctx->key.grow((size_t)std::max<int64_t>(total, 1) * 16, (size_t)at * 16, ctx->stream));
  const cudaMemcpyKind kind = device_src ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  if (n > 0 && !device_src && rows_fit_staging(ctx, n)) {
    if (int rc = stage_rows(ctx, X, category, key, n, at)) return rc;
  } else if (n > 0) {
    CU(cudaMemcpyAsync(ctx->X.as<double>() + at * P, X, (size_t)n * P * 8, kind, ctx->stream));
    CU(cudaMemcpyAsync(ctx->cat.as<int8_t>() + at, category, (size_t)n, kind, ctx->stream));
    CU(cudaMemcpyAsync(ctx->key.as<double>() + at * 2, key, (size_t)n * 16, kind, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
  }
  ctx->cat_h.resize((size_t)total);
  if (n > 0) {
    if (device_src) CU(cudaMemcpy(ctx->cat_h.data() + at, category, (size_t)n, cudaMemcpyDeviceToHost));
    else memcpy(ctx->cat_h.data() + at, category, (size_t)n);
  }
  if (at == 0) ctx->cat_cnt[0] = ctx->cat_cnt[1] = ctx->cat_cnt[2] = ctx->cat_cnt[3] = ctx->cat_cnt[4] = 0;
  for (int64_t i = at; i < total; ++i) ctx->cat_cnt[cat_slot(ctx->cat_h[(size_t)i])]++;
  if (at == 0) ctx->M = 1;  // a fresh history is single-objective until values are supplied
  ctx->N = total;
  ctx->history_set = true;
  ctx->prepared = ctx->built = ctx->sampled = false;
  ctx->hist_version++;
  return TPE_OK;
}

// ---- MOTPE: selection of the below part of the COMPLETE group (sampler.py:745-779) ----------------
// Fills ctx->member (u8 per history row) and returns how many COMPLETE trials went below.
// Per-thread scratch (doubles, odd so that the threads spread over the banks) of an M <= 3
// hypervolume of up to n points held in shared memory: caller's point list + hypervolume()'s copy,
// tmp row and order / mask words.  0 = does not fit (or M > 3, where hv_nd needs the O(n^2) arena).
int mo_smem_stride(int n, int M) {
  if (M > 3) return 0;
  const int stride = (2 * n * M + M + n + 9) | 1;
  return ((size_t)kMoMaxSet * stride * 8 <= 160 * 1024) ? stride : 0;
}

int mo_select_complete(tpe_ctx* ctx, int64_t n_below, int64_t* taken) {
  cudaStream_t st = ctx->stream;
  const int M = ctx->M;
  const int64_t N = ctx->N;
  std::vector<int64_t> list;
  for (int64_t i = 0; i < N; ++i)
    if (ctx->cat_h[i] == TPE_CAT_COMPLETE) list.push_back(i);
  const int nc = (int)list.size();
  const int64_t m = std::min<int64_t>(std::max<int64_t>(n_below, 0), nc);
  *taken = m;
  CU(ctx->member.ensure((size_t)std::max<int64_t>(N, 1)));
  CU(cudaMemsetAsync(ctx->member.p, 0, (size_t)std::max<int64_t>(N, 1), st));
  if (m == 0) return TPE_OK;
  if (m == nc) {
    std::vector<uint8_t> mem((size_t)N, 0);
    for (int64_t r : list) mem[(size_t)r] = 1;
    CU(cudaMemcpyAsync(ctx->member.p, mem.data(), (size_t)N, cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));
    return TPE_OK;
  }
  CU(ctx->mo_list.ensure((size_t)nc * 8));
  CU(cudaMemcpyAsync(ctx->mo_list.p, list.data(), (size_t)nc * 8, cudaMemcpyHostToDevice, st));
  for (DevBuf* b : {&ctx->mo_alive, &ctx->mo_dom, &ctx->mo_first, &ctx->mo_isdup, &ctx->mo_removed})
    CU(b->ensure((size_t)nc));
  for (DevBuf* b : {&ctx->mo_rank, &ctx->mo_tie, &ctx->mo_lexpos, &ctx->mo_sorted, &ctx->mo_uniq, &ctx->mo_chosen})
    CU(b->ensure((size_t)nc * 4));
  CU(ctx->mo_ctr.ensure(sizeof(MoCounters)));
  CU(ctx->mo_ntie.ensure(16));
  CU(ctx->mo_nuniq.ensure(16));
  CU(ctx->mo_ref.ensure(kMoMaxM * 8));
  CU(ctx->mo_contrib.ensure((size_t)nc * 8));
  CU(ctx->mo_diag.ensure((size_t)nc * 16));
  CU(ctx->mo_sample.ensure(256 * 4));
  CU(ctx->mo_surv.ensure((size_t)nc * 4));
  CU(ctx->mo_nsurv.ensure(16));
  CU(cudaMemsetAsync(ctx->mo_alive.p, 1, (size_t)nc, st));
  CU(cudaMemsetAsync(ctx->mo_rank.p, 0, (size_t)nc * 4, st));
  CU(cudaMemsetAsync(ctx->mo_ctr.p, 0, sizeof(MoCounters), st));
  const double* vals = ctx->vals.as<double>();
  const int64_t* dlist = ctx->mo_list.as<int64_t>();
  const int gb = (nc + 255) / 256;
  // peel Pareto fronts until n_below unique vectors are ranked
  std::vector<int64_t> rank_count;
  MoCounters ctr{};
  int r = 0;
  int64_t prev_all = 0;
  for (;;) {
    if (r == 0) {  // duplicates of the whole complete set, once
      uint32_t tsize = 1024;
      while (tsize < 2u * (uint32_t)nc) tsize <<= 1;
      CU(ctx->mo_table.ensure((size_t)tsize * 4));
      CU(cudaMemsetAsync(ctx->mo_table.p, 0x7f, (size_t)tsize * 4, st));
      k_mo_first_insert<<<gb, 256, 0, st>>>(vals, M, dlist, nc, ctx->mo_table.as<int>(), tsize - 1);
      k_mo_first_lookup<<<gb, 256, 0, st>>>(vals, M, dlist, nc, ctx->mo_table.as<int>(), tsize - 1,
                                            ctx->mo_first.as<uint8_t>(), ctx->mo_ctr.as<MoCounters>());
      ctx->launch_counter += 2;
    }
    k_mo_sample<<<1, 1024, 0, st>>>(nc, ctx->mo_alive.as<uint8_t>(), ctx->mo_sample.as<int32_t>(),
                                    ctx->mo_nsurv.as<int>(), ctx->mo_nsurv.as<int>() + 1);
    k_mo_peel_a<<<gb, 256, 256 * M * 8, st>>>(vals, M, dlist, nc, ctx->mo_alive.as<uint8_t>(),
                                               ctx->mo_sample.as<int32_t>(), ctx->mo_nsurv.as<int>(),
                                               ctx->mo_dom.as<uint8_t>(), ctx->mo_surv.as<int32_t>(),
                                               ctx->mo_nsurv.as<int>() + 1);
    k_mo_peel_b<<<std::min(nc, ctx->sm_count * 8), 256, 0, st>>>(vals, M, dlist, nc, ctx->mo_alive.as<uint8_t>(),
                                                                  ctx->mo_surv.as<int32_t>(), ctx->mo_nsurv.as<int>() + 1,
                                                                  ctx->mo_dom.as<uint8_t>());
    ctx->launch_counter += 1;
    k_mo_commit<<<gb, 256, 0, st>>>(nc, ctx->mo_alive.as<uint8_t>(), ctx->mo_dom.as<uint8_t>(),
                                     ctx->mo_first.as<uint8_t>(), ctx->mo_rank.as<int32_t>(), r,
                                     ctx->mo_ctr.as<MoCounters>());
    ctx->launch_counter += 2;
    CU(cudaMemcpyAsync(&ctr, ctx->mo_ctr.p, sizeof(ctr), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    rank_count.push_back(ctr.covered_all - prev_all);
    prev_all = ctr.covered_all;
    ++r;
    const int64_t goal = std::min<int64_t>(m, ctr.n_unique);
    if (ctr.covered_unique >= goal || ctr.covered_all >= nc) break;
    if (rank_count.back() == 0) return fail(ctx, TPE_E_INVALID, "MOTPE rank peeling made no progress (NaN objective values?)");
  }
  if (ctr.covered_all < nc) {
    k_mo_fill_rank<<<gb, 256, 0, st>>>(nc, ctx->mo_alive.as<uint8_t>(), ctx->mo_rank.as<int32_t>(), r);
    ctx->launch_counter++;
    rank_count.push_back(nc - ctr.covered_all);
  }
  // whole ranks that fit
  int64_t cum = 0;
  int last = -1;
  for (size_t q = 0; q < rank_count.size(); ++q) {
    if (cum + rank_count[q] > m) break;
    cum += rank_count[q];
    last = (int)q;
  }
  k_mo_gather_rank<<<1, 1024, 0, st>>>(nc, ctx->mo_rank.as<int32_t>(), last, dlist, ctx->member.as<uint8_t>(),
                                       ctx->mo_tie.as<int32_t>(), ctx->mo_ntie.as<int>());
  ctx->launch_counter++;
  const int subset = (int)(m - cum);
  if (subset > 0) {
    int n_tie = 0;
    CU(cudaMemcpyAsync(&n_tie, ctx->mo_ntie.p, 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    k_mo_refpoint<<<1, 256, 0, st>>>(vals, M, dlist, ctx->mo_tie.as<int32_t>(), n_tie, ctx->mo_ref.as<double>());
    double ref[kMoMaxM];
    CU(cudaMemcpyAsync(ref, ctx->mo_ref.p, (size_t)M * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    ctx->launch_counter += 1;
    bool finite = true;
    for (int j = 0; j < M; ++j) finite = finite && std::isfinite(ref[j]);
    std::vector<int32_t> chosen;
    int n_chosen = subset;
    bool chosen_on_device = false;
    if (!finite) {
      for (int i = 0; i < subset; ++i) chosen.push_back(i);  // rank_i_indices[:subset_size] (hssp.py:106-107)
    } else {
      k_mo_lexrank<<<(n_tie + 127) / 128, 128, 0, st>>>(vals, M, dlist, ctx->mo_tie.as<int32_t>(), n_tie,
                                                         ctx->mo_lexpos.as<int32_t>(), ctx->mo_isdup.as<uint8_t>());
      k_mo_unique<<<1, 1024, 0, st>>>(n_tie, ctx->mo_lexpos.as<int32_t>(), ctx->mo_isdup.as<uint8_t>(),
                                      ctx->mo_sorted.as<int32_t>(), ctx->mo_uniq.as<int32_t>(), ctx->mo_nuniq.as<int>());
      ctx->launch_counter += 2;
      int nu = 0;
      CU(cudaMemcpyAsync(&nu, ctx->mo_nuniq.p, 4, cudaMemcpyDeviceToHost, st));
      CU(cudaStreamSynchronize(st));
      chosen_on_device = true;
      if (nu <= subset) {
        // every unique vector, then the first duplicates in trial order (hssp.py:162-171)
        CU(cudaMemcpyAsync(ctx->mo_chosen.p, ctx->mo_uniq.p, (size_t)nu * 4, cudaMemcpyDeviceToDevice, st));
        if (nu < subset) {
          k_mo_fill_dups<<<1, 1024, 0, st>>>(n_tie, ctx->mo_isdup.as<uint8_t>(), subset - nu,
                                             ctx->mo_chosen.as<int32_t>(), nu);
          ctx->launch_counter++;
        }
      } else {
        CU(ctx->mo_state.ensure(hssp_bytes(subset, M)));
        CU(cudaMemsetAsync(ctx->mo_state.p, 0, hssp_bytes(subset, M), st));
        {
          HsspState head{0.0, 0, subset};
          CU(cudaMemcpyAsync(ctx->mo_state.p, &head, sizeof(head), cudaMemcpyHostToDevice, st));
          CU(cudaStreamSynchronize(st));  // `head` is a stack object
        }
        CU(cudaMemsetAsync(ctx->mo_removed.p, 0, (size_t)nc, st));
        if (M == 2) {
          k_hssp_2d<<<1, 256, 0, st>>>(vals, dlist, ctx->mo_tie.as<int32_t>(), ctx->mo_uniq.as<int32_t>(), nu, subset,
                                       ctx->mo_ref.as<double>(), ctx->mo_diag.as<double>(),
                                       ctx->mo_removed.as<uint8_t>(), ctx->mo_state.as<HsspState>());
          ctx->launch_counter++;
        } else {
          const size_t stride = (size_t)(subset + 2) * M + hv_arena_doubles(subset + 1, M);
          const int sstride = mo_smem_stride(subset + 1, M);
          const int cthreads = sstride ? 32 : 64;
          const size_t csmem = sstride ? (size_t)cthreads * sstride * 8 : 0;
          // more than three objectives: one warp per candidate, a private WFG arena per lane (global memory);
          // falls back to one thread per candidate when that would need more than 2 GB
          const size_t nd_lane_stride = hv_lane_doubles(subset, M);
          const size_t nd_warp_stride = hv_warp_scratch_doubles(subset, M) + 32 * nd_lane_stride;
          const bool nd_warp = M > 3 && (size_t)nu * nd_warp_stride * 8 <= ((size_t)8 << 30);
          const size_t stride3 = (size_t)(subset + 1) * 8 + 16;  // hv3_warp scratch per candidate beyond the shared-memory size
          const bool big3 = M == 3 && subset + 1 > kMoMaxSet + 1;
          if (!nd_warp && M > 3 && (size_t)nu * stride * 8 > ((size_t)32 << 30))
            return fail(ctx, TPE_E_NOMEM, "MOTPE subset selection: %d candidates x %d picks in %d objectives need %zu GB of "
                        "hypervolume scratch", nu, subset, M, ((size_t)nu * stride * 8) >> 30);
          if (nd_warp) CU(ctx->mo_arena.ensure((size_t)nu * nd_warp_stride * 8));
          else if (big3) CU(ctx->mo_arena.ensure((size_t)nu * stride3 * 8));
          else if (!sstride && M != 3) CU(ctx->mo_arena.ensure((size_t)nu * stride * 8));
          if (csmem > 48 * 1024)
            CU(cudaFuncSetAttribute(k_hssp_contrib, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)csmem));
          for (int t = 0; t < subset; ++t) {
            if (M == 3) {
              k_hssp_contrib3<<<(nu + 3) / 4, 128, 0, st>>>(vals, dlist, ctx->mo_tie.as<int32_t>(),
                                                            ctx->mo_uniq.as<int32_t>(), nu,
                                                            ctx->mo_removed.as<uint8_t>(), ctx->mo_ref.as<double>(),
                                                            ctx->mo_state.as<HsspState>(), ctx->mo_contrib.as<double>(),
                                                            ctx->mo_arena.as<double>(), stride3);
            } else if (nd_warp) {
              k_hssp_contrib_nd<<<(nu + 3) / 4, 128, 0, st>>>(
                  vals, M, dlist, ctx->mo_tie.as<int32_t>(), ctx->mo_uniq.as<int32_t>(), nu,
                  ctx->mo_removed.as<uint8_t>(), ctx->mo_ref.as<double>(), ctx->mo_state.as<HsspState>(),
                  ctx->mo_contrib.as<double>(), ctx->mo_arena.as<double>(), nd_warp_stride, nd_lane_stride);
            } else {
              k_hssp_contrib<<<(nu + cthreads - 1) / cthreads, cthreads, csmem, st>>>(
                  vals, M, dlist, ctx->mo_tie.as<int32_t>(), ctx->mo_uniq.as<int32_t>(), nu,
                  ctx->mo_removed.as<uint8_t>(), ctx->mo_ref.as<double>(), ctx->mo_state.as<HsspState>(),
                  ctx->mo_contrib.as<double>(), ctx->mo_arena.as<double>(), stride, sstride);
            }
            k_hssp_pick<<<1, 256, 0, st>>>(vals, M, dlist, ctx->mo_tie.as<int32_t>(), ctx->mo_uniq.as<int32_t>(), nu,
                                           ctx->mo_removed.as<uint8_t>(), ctx->mo_contrib.as<double>(),
                                           ctx->mo_state.as<HsspState>());
            ctx->launch_counter += 2;
          }
        }
        CU(cudaMemcpyAsync(ctx->mo_chosen.p, (char*)ctx->mo_state.p + sizeof(HsspState) + (size_t)subset * M * 8,
                           (size_t)subset * 4, cudaMemcpyDeviceToDevice, st));
      }
    }
    if (!chosen_on_device)
      CU(cudaMemcpyAsync(ctx->mo_chosen.p, chosen.data(), (size_t)n_chosen * 4, cudaMemcpyHostToDevice, st));
    k_mo_mark<<<(n_chosen + 127) / 128, 128, 0, st>>>(dlist, ctx->mo_tie.as<int32_t>(), ctx->mo_chosen.as<int32_t>(),
                                                      n_chosen, ctx->member.as<uint8_t>());
    ctx->launch_counter++;
    CU(cudaStreamSynchronize(st));
  }
  CU(cudaGetLastError());
  return TPE_OK;
}

// Host scan of uploaded rows: which columns have absent values (the split then needs the row filter) and which
// hold observations outside the column's current [low, high] (legal: optuna lets a range change between trials;
// the a-priori rounding bound of the tensor-core grid kernel assumes |mu''| <= range / (2 sigma), so such columns
// take the elementwise kernel).  TPE_CAT_EXCLUDED placeholders are in no estimator and do not count.
void scan_missing(tpe_ctx* ctx, const double* X, const int8_t* category, int64_t n) {
  const int64_t P = (int64_t)ctx->space.size();
  for (int64_t i = 0; i < n; ++i) {
    if (category && cat_slot(category[i]) == 4) continue;
    for (int64_t j = 0; j < P; ++j) {
      const double v = X[i * P + j];
      if (v != v) { ctx->col_missing[j] = 1; continue; }
      const tpe_param_desc& d = ctx->space[j];
      if (d.kind != TPE_KIND_CAT && (v < d.low || v > d.high)) ctx->col_oor[j] = 1;
      if (d.kind != TPE_KIND_CAT && d.has_step) {   // the test k_build_mv applies to tabulated columns
        const double gsz = floor((d.high - d.low) / d.step + 0.5) + 1.0;
        const double g = rint((v - d.low) / d.step);
        if (!(g >= 0.0 && g < gsz && d.low + g * d.step == v)) ctx->col_offgrid[j] = 1;
      }
    }
  }
}

bool mma_enabled() {
  static const bool on = [] { const char* v = getenv("TPE_MMA"); return !(v && v[0] == '0'); }();
  return on;
}

int build_estimator(tpe_ctx* ctx, int which, const double* w_host, cudaStream_t st) {
  Estimator& e = ctx->est[which];
  e.screen_ready = false;
  const int64_t n = e.n, K = n + 1;
  const int32_t pc = ctx->pc;
  const int cap = ctx->sm_count * 8;
  e.K = K;
  const int64_t k_alloc = round_up<int64_t>(K + 32, 32);  // >= round_up(K - 1, kMmaKPad), bulk-copy padding
  CU(e.mu.ensure((size_t)K * pc * 8));
  CU(e.sigma.ensure((size_t)K * pc * 8));
  CU(e.cst_part.ensure((size_t)K * 8));
  CU(e.cst.ensure((size_t)(k_alloc + kTcsTile) * 8));   // (+ one tile: k_tcs copies whole tiles)
  CU(e.w.ensure((size_t)K * 8));
  CU(e.logw.ensure((size_t)K * 8));
  CU(e.cdf.ensure((size_t)K * 8));
  if (ctx->fast_mode == 1) CU(e.tabp.ensure((size_t)K * ctx->pb * 16 + 16));
  if (ctx->fast_mode == 2) CU(e.tabc.ensure((size_t)(K + kTcsTile) * ctx->pb * 8 + 16));
  if (ctx->fast) CU(e.colprm.ensure((size_t)ctx->pb * 16));
  bool in_range = true;  // every selected column's observations lie inside its current [low, high]
  for (const ColMeta& cm : ctx->cols_h) in_range = in_range && !ctx->col_oor[cm.src];
  e.mma = ctx->fast_mode == 2 && ctx->pb >= 8 && in_range && mma_enabled();
  if (e.mma) {
    CU(e.tabm.ensure((size_t)k_alloc * ctx->pb * 8));
    CU(e.hb.ensure((size_t)k_alloc * 8));
    CU(e.ckk.ensure((size_t)k_alloc * 8));
    CU(cudaMemsetAsync(e.tabm.p, 0, (size_t)k_alloc * ctx->pb * 8, st));  // padded slots, last group, prior row
  }
  if (ctx->tab_doubles) CU(e.tab.ensure((size_t)ctx->tab_doubles * 8));
  if (ctx->dtab_doubles) {
    CU(e.dtab.ensure((size_t)ctx->dtab_doubles * 8));
    CU(e.cls.ensure((size_t)K * pc * 4));
    CU(e.offgrid.ensure(16));
    CU(cudaMemsetAsync(e.offgrid.p, 0, 16, st));
  }

  if (ctx->fast && ctx->pb > ctx->ncont) {
    k_tab_pad<<<grid_for(K * (ctx->pb - ctx->ncont), 256, cap), 256, 0, st>>>(
        ctx->fast_mode == 1 ? e.tabp.as<double2>() : nullptr, ctx->fast_mode == 2 ? e.tabc.as<double>() : nullptr,
        e.colprm.as<double2>(), ctx->fast_mode == 2 ? K - 1 : K, ctx->pb, ctx->ncont);
    ctx->launch_counter++;
  }
  if (ctx->cfg.multivariate) {
    k_build_mv<<<grid_for(K * 32, 256, cap), 256, 0, st>>>(
        ctx->X.as<double>(), (int32_t)ctx->space.size(), e.rows.as<int64_t>(), n, ctx->cols.as<ColMeta>(), pc,
        ctx->cfg.magic_clip, ctx->pb, ctx->fast_mode, e.mu.as<double>(), e.sigma.as<double>(), e.tabp.as<double2>(),
        e.tabc.as<double>(), e.colprm.as<double2>(), e.cst_part.as<double>(),
        ctx->dtab_doubles ? e.cls.as<int32_t>() : nullptr, ctx->dtab_doubles ? e.offgrid.as<int>() : nullptr,
        e.mma ? e.tabm.as<double>() : nullptr, e.mma ? e.hb.as<double>() : nullptr);
    ctx->launch_counter++;
    e.mixed = ctx->mixed_ok && K - 1 >= 2048;
    if (e.mixed) {
      const int ncp = (ctx->mix_ncont + 1) / 2, nd4 = (ctx->mix_nd + 3) / 4;
      e.mix_kstride = round_up<int64_t>(K - 1, 32);
      CU(e.mxc.ensure((size_t)std::max(ncp, 1) * e.mix_kstride * 16));
      CU(e.mxd.ensure((size_t)std::max(nd4, 1) * e.mix_kstride * 8));
      k_mixed_tables<<<grid_for(e.mix_kstride, 256, 1 << 20), 256, 0, st>>>(
          ctx->mixcols.as<MixCol>(), ctx->mix_ncont, ctx->mix_nd, ctx->cols.as<ColMeta>(), pc, e.mu.as<double>(),
          e.sigma.as<double>(), ctx->dtab_doubles ? e.cls.as<int32_t>() : nullptr, K - 1, e.mix_kstride,
          e.mxc.as<double2>(), e.mxd.as<ushort4>());
      ctx->launch_counter++;
    }
  } else {
    k_mu<<<grid_for(K * pc, 256, cap), 256, 0, st>>>(ctx->X.as<double>(), (int32_t)ctx->space.size(),
                                                     e.rows.as<int64_t>(), n, ctx->cols.as<ColMeta>(), pc,
                                                     e.mu.as<double>());
    ctx->launch_counter++;
    // categorical columns: sigma unused; numeric columns: sort-based neighbour gaps
    CU(cudaMemsetAsync(e.sigma.p, 0, (size_t)K * pc * 8, st));
    int64_t m2 = 1;
    while (m2 < K) m2 <<= 1;
    CU(ctx->sort_idx.ensure((size_t)std::max<int64_t>(m2, K * 3) * 4));
    for (int j = 0; j < pc; ++j) {
      if (ctx->cols_h[j].cls == COL_CAT) continue;
      if (m2 <= 4096) {
        k_sort_small<<<1, 1024, 0, st>>>(e.mu.as<double>(), pc, j, (int)K, (int)m2, ctx->sort_idx.as<int32_t>());
        ctx->launch_counter++;
      } else {
        // cooperative stable radix sort (one launch instead of ~150 bitonic steps)
        CU(ctx->sort_val.ensure((size_t)K * 8 * 2));
        CU(ctx->sort_idx.ensure((size_t)K * 4 * 3));
        CU(ctx->sort_work.ensure(sizeof(SortWork)));
        const double* d_mu = e.mu.as<double>();
        int32_t pc_i = pc;
        int j_i = j, n_i = (int)K;
        uint64_t* ka = ctx->sort_val.as<uint64_t>();
        uint64_t* kb = ka + K;
        int32_t* order = ctx->sort_idx.as<int32_t>();
        int32_t* ia = order + K;
        int32_t* ib = ia + K;
        SortWork* wk = ctx->sort_work.as<SortWork>();
        // column contexts of a univariate batch: the previous trial's order, if it belongs to this column of this
        // history and the set has the same size or one observation more, is updated instead (the sort then returns
        // at once unless the parent found the rows changed otherwise)
        const int* run_flag = nullptr;
        if (which == 1 && ctx->uni_fast && ctx->uni_mode_ptr != nullptr && ctx->uni_ord_seq + 1 == ctx->uni_seq &&
            ctx->uni_ord_lineage == ctx->hist_lineage &&
            ctx->uni_ord_col == ctx->cols_h[0].src && (ctx->uni_ord_K == K || ctx->uni_ord_K == K - 1) &&
            e.uord.cap >= (size_t)ctx->uni_ord_K * 4) {
          run_flag = ctx->uni_mode_ptr;
          CU(ctx->uni_work.ensure(16));
          CU(cudaMemsetAsync(ctx->uni_work.p, 0, 16, st));
          k_order_update<<<grid_for(ctx->uni_ord_K, 256, ctx->sm_count), 256, 0, st>>>(
              run_flag, e.uord.as<int32_t>(), (int)ctx->uni_ord_K, (int)K, e.mu.as<double>(), order, ctx->uni_work.as<int>());
          ctx->launch_counter++;
        }
        void* args[] = {&d_mu, &pc_i, &j_i, &n_i, &ka, &kb, &ia, &ib, &wk, &order, &run_flag};
        int G = (int)std::max<int64_t>(1, std::min<int64_t>(std::min(ctx->sm_count, 160), (K + 1023) / 1024));
        if (ctx->sort_cta_cap > 0) G = std::min(G, ctx->sort_cta_cap);
        CU(cudaLaunchCooperativeKernel((const void*)k_radix_sort_coop, dim3(G), dim3(512), args, 0, st));
        ctx->launch_counter++;
      }
      k_sigma_uni<<<grid_for(K, 256, cap), 256, 0, st>>>(e.mu.as<double>(), ctx->sort_idx.as<int32_t>(),
                                                         ctx->cols.as<ColMeta>(), pc, j, n, ctx->cfg.magic_clip,
                                                         ctx->cfg.endpoints, e.sigma.as<double>());
      ctx->launch_counter++;
      if (ctx->uni_fast) {   // the 1-D grid walks the kernels in this order
        CU(e.uord.ensure((size_t)(K + 1024) * 4));   // room to grow without a reallocation (the old order is read above)
        CU(cudaMemcpyAsync(e.uord.p, ctx->sort_idx.p, (size_t)K * 4, cudaMemcpyDeviceToDevice, st));
        if (which == 1) {
          ctx->uni_ord_seq = ctx->uni_seq;
          ctx->uni_ord_lineage = ctx->hist_lineage;
          ctx->uni_ord_col = ctx->cols_h[0].src;
          ctx->uni_ord_K = K;
        }
      }
    }
    k_const<<<grid_for(K * 32, 256, cap), 256, 0, st>>>(e.mu.as<double>(), e.sigma.as<double>(),
                                                        ctx->cols.as<ColMeta>(), pc, K, ctx->pb, ctx->fast_mode,
                                                        e.tabp.as<double2>(), e.tabc.as<double>(),
                                                        e.colprm.as<double2>(), e.cst_part.as<double>());
    ctx->launch_counter++;
  }
  const double* w_dev = nullptr;
  const int64_t* w_pos = nullptr;
  if (w_host != nullptr && n > 0) {
    CU(e.wstage.ensure((size_t)n * 8));
    CU(cudaMemcpyAsync(e.wstage.p, w_host, (size_t)n * 8, cudaMemcpyHostToDevice, st));
    w_dev = e.wstage.as<double>();
  } else if (which == 0 && ctx->M >= 2 && n > 0) {
    // MOTPE: hypervolume weights of ALL below trials, then the rows holding every selected param
    // pick theirs through `pos` (weights_below[param_mask_below], sampler.py:570-576)
    const int nba = (int)ctx->info.n_below_all;
    const int M = ctx->M;
    const int64_t* brows = ctx->below_all.as<int64_t>();   // every below trial, trial order (k_split_coop)
    CU(ctx->mo_w.ensure((size_t)std::max(nba, 1) * 8));
    if (nba <= kMoMaxSet) {
      // small below set (the default gamma caps it at 25): one CTA, everything staged in shared memory
      const size_t stride = (size_t)(nba + 2) * M + hv_arena_doubles(nba + 1, M);
      const int sstride = mo_smem_stride(nba + 1, M);
      const size_t wsmem = sstride ? (size_t)kMoMaxSet * sstride * 8 : 0;
      if (!sstride) CU(ctx->mo_arena.ensure((size_t)(nba + 1) * stride * 8));
      if (wsmem > 32 * 1024)
        CU(cudaFuncSetAttribute(k_mo_weights, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsmem));
      if (M == 3) {
        static const size_t w3smem = (size_t)32 * kHv3Scratch * 8;
        CU(cudaFuncSetAttribute(k_mo_weights3, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)w3smem));
        k_mo_weights3<<<1, 1024, w3smem, st>>>(ctx->vals.as<double>(), brows, nba, ctx->cat.as<int8_t>(),
                                               ctx->mo_w.as<double>());
      } else if (M > 3) {
        const size_t lane_stride = hv_lane_doubles(nba + 1, M);
        const size_t warp_stride = hv_warp_scratch_doubles(nba + 1, M) + 32 * lane_stride;
        CU(ctx->mo_arena.ensure((size_t)32 * warp_stride * 8));
        k_mo_weights_nd<<<1, 1024, 0, st>>>(ctx->vals.as<double>(), M, brows, nba, ctx->cat.as<int8_t>(),
                                            ctx->mo_w.as<double>(), ctx->mo_arena.as<double>(), warp_stride, lane_stride);
      } else {
        k_mo_weights<<<1, kMoMaxSet, wsmem, st>>>(ctx->vals.as<double>(), M, brows, nba, ctx->cat.as<int8_t>(),
                                                  ctx->mo_w.as<double>(), ctx->mo_arena.as<double>(), stride, sstride);
      }
    } else {
      // any size: global-memory kernels; the exact hypervolumes run over the Pareto front of the below set only
      CU(ctx->mo_fv.ensure((size_t)nba * M * 8));
      CU(ctx->mo_ps.ensure((size_t)nba * M * 8));
      CU(ctx->mo_map.ensure((size_t)nba * 4));
      CU(ctx->mo_front.ensure((size_t)nba * 4));
      CU(ctx->mo_contrib.ensure((size_t)nba * 8));
      CU(ctx->mo_head.ensure(sizeof(MowHead)));
      k_mow_prep<<<1, 1024, 0, st>>>(ctx->vals.as<double>(), M, brows, nba, ctx->cat.as<int8_t>(), ctx->mo_w.as<double>(),
                                     ctx->mo_fv.as<double>(), ctx->mo_map.as<int32_t>(), ctx->mo_ps.as<double>(),
                                     ctx->mo_front.as<int32_t>(), ctx->mo_contrib.as<double>(), ctx->mo_head.as<MowHead>());
      MowHead head{};
      CU(cudaMemcpyAsync(&head, ctx->mo_head.p, sizeof(head), cudaMemcpyDeviceToHost, st));
      CU(cudaStreamSynchronize(st));
      ctx->launch_counter++;
      const int np = head.np;
      if (head.nf > 1 && np > 0) {
        size_t lane_stride = 0, warp_stride;
        if (M > 3) {
          lane_stride = hv_lane_doubles(np, M);
          warp_stride = (size_t)np * M + hv_warp_scratch_doubles(np, M) + 32 * lane_stride;
        } else {
          warp_stride = (size_t)np * M + hv_arena_doubles(np, M) + (size_t)np * 8 + 64;
        }
        const size_t budget = (size_t)16 << 30;
        int64_t warps = std::min<int64_t>(np, (int64_t)ctx->sm_count * 16);
        warps = std::min<int64_t>(warps, (int64_t)(budget / (warp_stride * 8)));
        if (warps < 1)
          return fail(ctx, TPE_E_NOMEM, "MOTPE weights: a Pareto front of %d points in %d objectives needs %zu GB of exact-"
                      "hypervolume scratch per warp", np, M, (warp_stride * 8) >> 30);
        const int blocks = (int)((warps + 3) / 4);
        CU(ctx->mo_arena.ensure((size_t)blocks * 4 * warp_stride * 8));
        k_mow_hv<<<1, 128, 0, st>>>(ctx->mo_ps.as<double>(), ctx->mo_front.as<int32_t>(), M, ctx->mo_head.as<MowHead>(), np,
                                    np, ctx->mo_contrib.as<double>(), ctx->mo_arena.as<double>(), warp_stride, lane_stride);
        k_mow_hv<<<blocks, 128, 0, st>>>(ctx->mo_ps.as<double>(), ctx->mo_front.as<int32_t>(), M,
                                         ctx->mo_head.as<MowHead>(), 0, np - 1, ctx->mo_contrib.as<double>(),
                                         ctx->mo_arena.as<double>(), warp_stride, lane_stride);
        k_mow_norm<<<1, 1024, 0, st>>>(ctx->mo_head.as<MowHead>(), ctx->mo_contrib.as<double>(), ctx->mo_map.as<int32_t>(),
                                       ctx->mo_w.as<double>());
        ctx->launch_counter += 3;
      }
    }
    w_pos = e.pos.as<int64_t>();   // an observation row picks the weight of its position among ALL below trials
                                   // (weights_below[param_mask_below], sampler.py:570-576)
    ctx->launch_counter++;
    ctx->mo_weights_ready = true;
    w_dev = ctx->mo_w.as<double>();
  }
  {
    const int nparts = grid_for(K, 2048, ctx->sm_count * 2);
    if (nparts == 1) {
      k_weights_one<<<1, 256, 0, st>>>(w_dev, w_pos, n, ctx->cfg.prior_weight, e.w.as<double>(), e.logw.as<double>(),
                                       e.cst_part.as<double>(), e.cst.as<double>(),
                                       which == 0 ? e.cdf.as<double>() : nullptr, k_alloc,
                                       e.mma ? e.hb.as<double>() : nullptr, e.mma ? e.ckk.as<double>() : nullptr);
      ctx->launch_counter += 1;
    } else {
      CU(e.wpart.ensure((size_t)nparts * 8));
      k_wraw<<<nparts, 256, 0, st>>>(w_dev, w_pos, n, ctx->cfg.prior_weight, e.w.as<double>(), e.wpart.as<double>());
      k_wfinal<<<grid_for(k_alloc, 256, ctx->sm_count * 4), 256, 0, st>>>(
          e.wpart.as<double>(), nparts, n, e.w.as<double>(), e.logw.as<double>(), e.cst_part.as<double>(),
          e.cst.as<double>(), which == 0 ? e.cdf.as<double>() : nullptr, k_alloc,
          e.mma ? e.hb.as<double>() : nullptr, e.mma ? e.ckk.as<double>() : nullptr);
      k_wnorm<<<grid_for(K, 256, ctx->sm_count * 4), 256, 0, st>>>(e.wpart.as<double>(), nparts, K, e.w.as<double>());
      ctx->launch_counter += 3;
    }
  }
  if (ctx->ncat) {
    k_cat_tables<<<pc, 64, 0, st>>>(ctx->cols.as<ColMeta>(), pc, n, ctx->cfg.prior_weight,
                                    ctx->cat_dist.as<double>(), e.tab.as<double>());
    ctx->launch_counter++;
  }
  // Experimental and OFF by default (TPE_TCS=1): correct (same parity tests) but 1.9 ms against 1.17 ms for
  // k_logpdf_mma at config 2 -- the bf16 screen itself takes 0.13 ms, the exact evaluation of the 8.9 % survivors on
  // the CUDA cores the rest (profiles/r2_variants.md, section 4)
  static const bool tcs_on = [] { const char* v = getenv("TPE_TCS"); return v && v[0] == '1'; }();
  e.tcs = tcs_on && e.mma && K - 1 >= 1024 && (ctx->pb == 16 || ctx->pb == 32 || ctx->pb == 64);
  if (e.tcs) {
    e.tcs_kpad = round_up<int64_t>(K - 1, kTcsTile);
    CU(e.tcs_h.ensure((size_t)e.tcs_kpad * (ctx->pb + 8) * 2));
    CU(e.tcs_ak.ensure((size_t)e.tcs_kpad * 4));
    CU(e.tcs_ak64.ensure((size_t)e.tcs_kpad * 8));
    k_tcs_tables<<<grid_for(e.tcs_kpad, 256, 1 << 20), 256, 0, st>>>(
        e.tabc.as<double>(), e.cst.as<double>(), K - 1, e.tcs_kpad, ctx->pb,
        reinterpret_cast<__nv_bfloat16*>(e.tcs_h.p), e.tcs_ak.as<float>(), e.tcs_ak64.as<double>());
    ctx->launch_counter++;
  }
  e.uni_ready = false;
  if (ctx->uni_fast) {
    const int64_t ntiles = (K + kUniTile - 1) / kUniTile;
    CU(e.us32.ensure((size_t)ntiles * kUniTile * 16));
    CU(e.usmi.ensure((size_t)ntiles * kUniTile * 16));
    CU(e.usc.ensure((size_t)ntiles * kUniTile * 8));
    CU(e.umeta.ensure((size_t)ntiles * sizeof(UniTileMeta)));
    // large estimators: the kernels at the bandwidth floor go through the fast Gauss transform (k_fgt_*)
    static const int64_t fgt_min = [] { const char* v = getenv("TPE_FGT_MIN_K"); return v ? atoll(v) : 1024ll; }();
    e.fgt = ctx->cfg.magic_clip && K >= fgt_min;
    if (e.fgt) {
      CU(e.ucoef.ensure((size_t)kFgtMaxBoxes * kFgtRow * 8));
      CU(e.ubox.ensure((size_t)kFgtMaxBoxes * sizeof(FgtBox)));
      CU(e.ubstart.ensure((size_t)(kFgtMaxBoxes + 1) * 4));
    }
    k_uni_tables<<<(unsigned)ntiles, kUniTile, 0, st>>>(e.uord.as<int32_t>(), e.mu.as<double>(), e.sigma.as<double>(),
                                                        e.cst.as<double>(), ctx->cols.as<ColMeta>(), K, e.us32.as<float4>(),
                                                        e.usmi.as<double2>(), e.usc.as<double>(), e.umeta.as<UniTileMeta>(),
                                                        e.fgt ? 1 : 0, ctx->cfg.magic_clip, e.ubstart.as<int32_t>());
    ctx->launch_counter++;
    if (e.fgt) {
      k_fgt_coeff<<<kFgtMaxBoxes, 128, 0, st>>>(e.uord.as<int32_t>(), e.mu.as<double>(), e.sigma.as<double>(),
                                                e.cst.as<double>(), ctx->cols.as<ColMeta>(), K, ctx->cfg.magic_clip,
                                                e.ubstart.as<int32_t>(), e.ucoef.as<double>(), e.ubox.as<FgtBox>());
      CU(e.utlist.ensure((size_t)(ntiles + 1) * 4));
      k_uni_tile_list<<<1, 256, 0, st>>>(e.umeta.as<UniTileMeta>(), (int)ntiles, e.utlist.as<int32_t>());
      ctx->launch_counter += 2;
    }
    e.uni_ready = true;
  }
  CU(cudaGetLastError());
  return TPE_OK;
}

// k_logpdf_mixed: candidates per CTA that fit the shared memory (0: none do), and the bytes they take
size_t mixed_smem(const tpe_ctx* ctx, int CB) {
  const int ncp = (ctx->mix_ncont + 1) / 2, nd4 = (ctx->mix_nd + 3) / 4;
  return (size_t)CB * (2 * ncp + ctx->mix_tabd + 1) * 8 + (size_t)nd4 * 16 + 16;
}
int mixed_cb(const tpe_ctx* ctx) {
  for (int CB : {8, 4, 2})
    if (mixed_smem(ctx, CB) <= 200 * 1024) return CB;
  return 0;
}

// log-density of the Ct resident candidates under estimator `which`: fills e.part (k-split
// partials) and, for out-of-support candidates, e.fix.
int run_logpdf(tpe_ctx* ctx, int which, int64_t Ct, cudaEvent_t after_main = nullptr) {
  Estimator& e = ctx->est[which];
  cudaStream_t st = ctx->stream;
  if (which == 1 && join_above(ctx)) return TPE_E_CUDA;
  const int64_t K = e.K;
  if (which == 1 && ctx->kshard_world > 1 && !(ctx->fast && ctx->fast_mode == 2))
    return fail(ctx, TPE_E_STATE, "kernel sharding is for multivariate all-continuous suggestions");
  if (ctx->uni_fast && e.uni_ready && Ct <= 4096) {
    // one continuous column, univariate: sorted candidates x sorted kernels (tpe_uni.cuh)
    const int C = (int)Ct;
    if (!ctx->cands_sorted) {
      CU(ctx->uxs.ensure((size_t)round_up<int64_t>(C, 32) * 8));
      CU(ctx->ucidx.ensure((size_t)round_up<int64_t>(C, 32) * 4));
      k_uni_sort_cands<<<1, 1024, 0, st>>>(ctx->xT.as<double>(), C, ctx->cols.as<ColMeta>(), ctx->uxs.as<double>(),
                                           ctx->ucidx.as<int32_t>());
      ctx->launch_counter++;
      ctx->cands_sorted = true;
    }
    CU(e.part.ensure((size_t)2 * ctx->ct_stride * 16));
    const double skip = std::min(46.0, log((double)std::max<int64_t>(K, 1)) + 30.0);
    k_uni_grid<<<(unsigned)((C + 31) / 32), kUniWarps * 32, 0, st>>>(e.us32.as<float4>(), e.usmi.as<double2>(),
                                                                     e.usc.as<double>(), e.umeta.as<UniTileMeta>(), K,
                                                                     ctx->uxs.as<double>(), ctx->ucidx.as<int32_t>(), C, skip,
                                                                     e.part.as<double2>(), e.fgt ? e.utlist.as<int32_t>() : nullptr);
    ctx->launch_counter++;
    if (e.fgt) {
      static bool fgt_attr = false;
      if (!fgt_attr) {
        CU(cudaFuncSetAttribute(k_fgt_eval, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFgtEvalSmem));
        fgt_attr = true;
      }
      k_fgt_eval<<<(unsigned)((C + kFgtCands - 1) / kFgtCands), 256, kFgtEvalSmem, st>>>(
          e.ucoef.as<double>(), e.ubox.as<FgtBox>(), e.ubstart.as<int32_t>(), e.us32.as<float4>(), e.usmi.as<double2>(),
          e.usc.as<double>(), e.mu.as<double>(), e.sigma.as<double>(), e.cst.as<double>(), ctx->cols.as<ColMeta>(), K,
          ctx->cfg.magic_clip, ctx->xT.as<double>(), C, e.part.as<double2>() + ctx->ct_stride);
      ctx->launch_counter++;
    }
    ctx->last_kernel = e.fgt ? "k_uni_grid<sorted 1-D> + k_fgt_eval" : "k_uni_grid<sorted 1-D>";
    if (after_main) CU(cudaEventRecord(after_main, st));
    CU(e.fix.ensure((size_t)ctx->ct_stride * 16));
    k_logpdf_prior_fix<<<(unsigned)((Ct * 32 + 255) / 256), 256, 0, st>>>(
        ctx->S.as<double>(), Ct, ctx->cols.as<ColMeta>(), ctx->pc, e.mu.as<double>(), e.sigma.as<double>(),
        e.cst.as<double>(), K, e.tab.as<double>(), nullptr, ctx->oob.as<uint8_t>(), e.fix.as<double2>());
    ctx->launch_counter++;
    e.nsplit = e.fgt ? 2 : 1;
    CU(cudaGetLastError());
    return TPE_OK;
  }
  if (ctx->fast) {
    const bool cst_mode = ctx->fast_mode == 2;
    // tensor-core kernel unless the expanded square would lose more than 5e-13 (see k_logpdf_mma)
    bool use_mma = false;
    if (e.mma && K > 1) {
      const double nobs = (double)std::max<int64_t>(e.n, 1);
      double fac = 0.2 * pow(nobs, -1.0 / (ctx->pc + 4));
      if (ctx->cfg.magic_clip) fac = std::max(fac, 1.0 / std::min(100.0, 1.0 + (double)K));
      fac = std::min(std::max(fac, 1e-9), 1.0);
      const double rho = 0.5 / fac;
      use_mma = ctx->pb * rho * rho * 2.3e-16 <= 5e-13 && pick_mma(ctx->pb, Ct) != nullptr;
    }
    const FastCfg* fc = use_mma ? pick_mma(ctx->pb, Ct) : pick_fast(ctx->fast_mode, ctx->pb, Ct);
    // CONST tables exclude the prior kernel (its sigma differs); the mma table is padded to groups of 8
    int64_t Kf = use_mma ? round_up<int64_t>(K - 1, kMmaKPad) : (cst_mode ? K - 1 : K);
    // kernel sharding (g(x) only): this context takes the tiles [k_lo, k_hi) of the table; the prior kernel's slice
    // belongs to rank 0
    int64_t k_lo = 0;
    const bool sharded = which == 1 && ctx->kshard_world > 1;
    if (sharded) {
      if (!cst_mode) return fail(ctx, TPE_E_STATE, "kernel sharding is for multivariate all-continuous suggestions");
      const int64_t chunk = round_up<int64_t>((Kf + ctx->kshard_world - 1) / ctx->kshard_world, fc->tk);
      k_lo = std::min(Kf, chunk * ctx->kshard_rank);
      Kf = std::min(Kf, k_lo + chunk) - k_lo;
    }
    const int tc = fc->cands_per_cta;
    const int64_t ctiles = (Ct + tc - 1) / tc;
    // k-splits: two full waves of resident CTAs for the big configurations
    const int64_t ktiles = (Kf + fc->tk - 1) / fc->tk;
    const int64_t target = (fc->nt >= 256) ? (int64_t)ctx->sm_count * fc->minb * 2 : (int64_t)ctx->sm_count * 8;
    int64_t nsplit = 0, kps = fc->tk;
    if (ktiles > 0) {
      nsplit = std::max<int64_t>(1, std::min<int64_t>(ktiles, target / ctiles));
      const int64_t tiles_per = (ktiles + nsplit - 1) / nsplit;
      nsplit = (ktiles + tiles_per - 1) / tiles_per;
      kps = tiles_per * fc->tk;
    }
    // bf16 tensor-core screen + exact survivors (tpe_tcscreen.cuh): many candidates, rounding bound small enough
    bool use_tcs = false;
    if (e.tcs && cst_mode && Ct >= 256 && !sharded) {
      const double nobs = (double)std::max<int64_t>(e.n, 1);
      double fac = 0.2 * pow(nobs, -1.0 / (ctx->pc + 4));
      if (ctx->cfg.magic_clip) fac = std::max(fac, 1.0 / std::min(100.0, 1.0 + (double)K));
      fac = std::min(std::max(fac, 1e-9), 1.0);
      const double rho = 0.5 / fac, pr2 = ctx->pb * rho * rho;
      const double delta = pr2 * (1.0 / 256 + 1.0 / 65536 + (ctx->pb + 2) * 5.97e-8) * 1.02 + 2e-3;
      if (delta <= 6.0 && pr2 * 2.3e-16 <= 5e-13) {   // (the second: conditioning of the expanded square, as for k_logpdf_mma)
        use_tcs = true;
        const int pb = ctx->pb;
        const size_t smem_sum = pb == 16 ? sizeof(TcsSmem<16>) : pb == 32 ? sizeof(TcsSmem<32>) : sizeof(TcsSmem<64>);
        const size_t smem_max = pb == 16 ? offsetof(TcsSmem<16>, b64) : pb == 32 ? offsetof(TcsSmem<32>, b64) : offsetof(TcsSmem<64>, b64);
        const int64_t tctiles = (Ct + kTcsRows - 1) / kTcsRows, tktiles = e.tcs_kpad / kTcsTile;
        const int64_t slots = (int64_t)ctx->sm_count * (smem_sum <= 113 * 1024 ? 2 : 1);
        int64_t tns = std::max<int64_t>(1, std::min<int64_t>(tktiles, slots / tctiles));
        const int64_t tiles_per = (tktiles + tns - 1) / tns;
        tns = (tktiles + tiles_per - 1) / tiles_per;
        const int64_t tkps = tiles_per * kTcsTile;
        CU(e.part.ensure((size_t)(tns + 1) * ctx->ct_stride * 16));
        CU(ctx->x64s.ensure((size_t)ctx->ct_stride * pb * 8));
        CU(ctx->e32s.ensure((size_t)ctx->ct_stride * 4));
        CU(ctx->x32s.ensure((size_t)ctx->ct_stride * 8));   // (-|x''|^2 / 2 in fp64)
        CU(ctx->gmax.ensure((size_t)ctx->ct_stride * 4));
        k_tcs_xprep<<<grid_for(ctx->ct_stride, 256, 1 << 20), 256, 0, st>>>(
            ctx->xT.as<double>(), e.colprm.as<double2>(), ctx->ct_stride, pb, ctx->x64s.as<double>(),
            ctx->e32s.as<float>(), ctx->x32s.as<double>(), ctx->gmax.as<int>());
        const double skip_t = std::min(46.0, log((double)std::max<int64_t>(K, 1)) + 30.0);
        const float window = (float)(skip_t + 2.0 * delta);
        // TPE_TCS_STATS=1 (diagnostics): count the survivors of every launch and print them
        static const bool tcs_stats_on = [] { const char* v = getenv("TPE_TCS_STATS"); return v && v[0] == '1'; }();
        unsigned long long* tcs_stats = nullptr;
        if (tcs_stats_on) {
          CU(ctx->lse_gmax.ensure(64));
          CU(cudaMemsetAsync(ctx->lse_gmax.p, 0, 8, st));
          tcs_stats = ctx->lse_gmax.as<unsigned long long>();
        }
#define TPE_TCS_LAUNCH(PBV)                                                                                            \
        do {                                                                                                           \
          static bool attr_done = false;                                                                               \
          if (!attr_done) {                                                                                            \
            CU(cudaFuncSetAttribute(k_tcs<PBV, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));   \
            CU(cudaFuncSetAttribute(k_tcs<PBV, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_sum));    \
            attr_done = true;                                                                                          \
          }                                                                                                            \
          k_tcs<PBV, false><<<dim3((unsigned)tctiles, (unsigned)tns), kTcsNT, smem_max, st>>>(                         \
              reinterpret_cast<const __nv_bfloat16*>(e.tcs_h.p), e.tcs_ak.as<float>(), e.tabc.as<double>(),            \
              e.tcs_ak64.as<double>(), e.tcs_kpad, tkps, ctx->x64s.as<double>(), ctx->e32s.as<float>(),               \
              ctx->x32s.as<double>(), ctx->gmax.as<int>(), Ct, ctx->ct_stride, window, e.part.as<double2>(), tcs_stats);                                                       \
          k_tcs<PBV, true><<<dim3((unsigned)tctiles, (unsigned)tns), kTcsNT, smem_sum, st>>>(                          \
              reinterpret_cast<const __nv_bfloat16*>(e.tcs_h.p), e.tcs_ak.as<float>(), e.tabc.as<double>(),            \
              e.tcs_ak64.as<double>(), e.tcs_kpad, tkps, ctx->x64s.as<double>(), ctx->e32s.as<float>(),               \
              ctx->x32s.as<double>(), ctx->gmax.as<int>(), Ct, ctx->ct_stride, window, e.part.as<double2>(), tcs_stats);                                                       \
        } while (0)
        if (pb == 16) TPE_TCS_LAUNCH(16);
        else if (pb == 32) TPE_TCS_LAUNCH(32);
        else TPE_TCS_LAUNCH(64);
#undef TPE_TCS_LAUNCH
        ctx->launch_counter += 3;
        if (tcs_stats_on) {
          unsigned long long hs = 0;
          CU(cudaMemcpyAsync(&hs, tcs_stats, 8, cudaMemcpyDeviceToHost, st));
          CU(cudaStreamSynchronize(st));
          fprintf(stderr, "[tpe] k_tcs: %llu survivors of %lld x %lld cells (%.2f %%), window %.2f\n", hs, (long long)Ct,
                  (long long)(K - 1), 100.0 * (double)hs / ((double)Ct * (double)(K - 1)), (double)window);
        }
        nsplit = tns;
        ctx->last_kernel = "k_tcs<bf16 screen + exact survivors>";
      }
    }
#ifdef TPE_LAB
    // fp32-screened variant (tpe_screen.cuh): multivariate, 17..32 continuous columns, many candidates
    // Experimental and OFF by default: correct (same parity tests) but 2.62 ms vs 2.40 ms for the exact
    // kernel at config 2 -- see profiles/r1_variants.md.  TPE_SCREEN=1 enables it.
    static const bool screen_on = [] { const char* v = getenv("TPE_SCREEN"); return v && v[0] == '1'; }();
    const bool use_screen = !use_tcs && cst_mode && !use_mma && ctx->pb == kScrP && Ct > 128 && Kf > 0 && screen_on;
    if (use_screen) {
      const int64_t sctiles = (Ct + kScrCands - 1) / kScrCands;
      const int64_t sktiles = (Kf + kScrTK - 1) / kScrTK;
      int64_t sns = std::max<int64_t>(1, std::min<int64_t>(sktiles, (int64_t)ctx->sm_count * 2 / sctiles));
      const int64_t tiles_per = (sktiles + sns - 1) / sns;
      sns = (sktiles + tiles_per - 1) / tiles_per;
      const int64_t skps = tiles_per * kScrTK;
      CU(e.part.ensure((size_t)(sns + 1) * ctx->ct_stride * 16));
      if (!e.screen_ready) {
        CU(e.tab32.ensure((size_t)Kf * kScrP * 4 + 64));
        CU(e.tab64p.ensure((size_t)Kf * kScrStride * 8 + 64));
        CU(e.d32.ensure((size_t)Kf * 4 + 64));
        k_screen_tabprep<<<grid_for(Kf * 32, 256, ctx->sm_count * 8), 256, 0, st>>>(
            e.tabc.as<double>(), e.cst.as<double>(), Kf, e.tab32.as<float>(), e.tab64p.as<double>(), e.d32.as<float>());
        ctx->launch_counter++;
        e.screen_ready = true;
      }
      CU(ctx->x64s.ensure((size_t)ctx->ct_stride * kScrP * 8));
      CU(ctx->x32s.ensure((size_t)ctx->ct_stride * kScrP * 4));
      CU(ctx->e32s.ensure((size_t)ctx->ct_stride * 4));
      CU(ctx->gmax.ensure((size_t)ctx->ct_stride * 4));
      k_screen_xprep<<<grid_for(ctx->ct_stride, 256, 1 << 20), 256, 0, st>>>(
          ctx->xT.as<double>(), e.colprm.as<double2>(), ctx->ct_stride, ctx->x64s.as<double>(), ctx->x32s.as<float>(),
          ctx->e32s.as<float>(), ctx->gmax.as<float>());
      ctx->launch_counter++;
      if (!ctx->screen_attr_set) {
        CU(cudaFuncSetAttribute(k_logpdf_screen, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ScreenSmem)));
        ctx->screen_attr_set = true;
      }
      // fp32 error bound of the screening value: dot product of P terms + input rounding, over
      // |x''|, |mu''| <= rho = (range / 2) / sigma (identical for every column of a multivariate estimator)
      const double nobs = (double)std::max<int64_t>(e.n, 1);
      double fac = 0.2 * pow(nobs, -1.0 / (ctx->pc + 4));
      if (ctx->cfg.magic_clip) fac = std::max(fac, 1.0 / std::min(100.0, 1.0 + (double)K));
      fac = std::min(std::max(fac, 1e-9), 1.0);
      const double rho = 0.5 / fac;
      const float margin = (float)(0.5 + 8e-6 * kScrP * rho * rho);
      k_logpdf_screen<<<dim3((unsigned)sctiles, (unsigned)sns), kScrNT, sizeof(ScreenSmem), st>>>(
          e.tab32.as<float>(), e.tab64p.as<double>(), e.cst.as<double>(), e.d32.as<float>(), Kf,
          ctx->x64s.as<double>(), ctx->x32s.as<float>(), ctx->e32s.as<float>(), ctx->gmax.as<float>(),
          ctx->ct_stride, skps,
          std::min(46.0, log((double)std::max<int64_t>(K, 1)) + 30.0), margin, e.part.as<double2>());
      ctx->launch_counter++;
      nsplit = sns;
      ctx->last_kernel = "k_logpdf_screen<fp32 screen + fp64 exact>";
    }
#else
    constexpr bool use_screen = false;
#endif
    if (!use_screen && !use_tcs) CU(e.part.ensure((size_t)(nsplit + 1) * ctx->ct_stride * 16));
    if (nsplit > 0 && !use_screen && !use_tcs) {
      if (!ctx->prepared_cfgs.count(fc)) {
        CU(fc->prepare());
        ctx->prepared_cfgs.insert(fc);
      }
      if (use_mma) {
        CU(ctx->lse_gmax.ensure((size_t)ctx->ct_stride * 8));
        CU(cudaMemsetAsync(ctx->lse_gmax.p, 0, (size_t)ctx->ct_stride * 8, st));
      }
      // (both CONST tables are blocked by whole kernels -- the fragment-major one in groups of 8 -- so a slice that
      // starts at a multiple of the tile is a plain offset)
      fc->launch(dim3((unsigned)ctiles, (unsigned)nsplit), fc->smem, st,
                 use_mma ? (const void*)(e.tabm.as<double>() + k_lo * ctx->pb)
                         : (cst_mode ? (const void*)(e.tabc.as<double>() + k_lo * ctx->pb) : (const void*)e.tabp.p),
                 (use_mma ? e.ckk.as<double>() : e.cst.as<double>()) + k_lo, Kf,
                 e.colprm.as<double2>(), ctx->xT.as<double>(), ctx->ct_stride, kps,
                 std::min(46.0, log((double)std::max<int64_t>(K, 1)) + 30.0), e.part.as<double2>(),
                 use_mma ? ctx->lse_gmax.as<unsigned long long>() : nullptr);
      ctx->launch_counter++;
    }
    if (use_tcs) {
    } else if (use_mma && !use_screen)
      ctx->last_kernel = (fc->nt >= 256) ? "k_logpdf_mma<big>" : "k_logpdf_mma<small>";
    else if (!use_screen)
      ctx->last_kernel = cst_mode ? ((fc->nt >= 256) ? "k_logpdf_fast<const,big>" : "k_logpdf_fast<const,small>")
                                  : ((fc->nt >= 256) ? "k_logpdf_fast<pair,big>" : "k_logpdf_fast<pair,small>");
    if (after_main) CU(cudaEventRecord(after_main, st));
    // the prior kernel of CONST tables (one more partial row) and the exact fix-up of the candidates
    // outside [low, high], one launch
    CU(e.fix.ensure((size_t)ctx->ct_stride * 16));
    k_logpdf_prior_fix<<<(unsigned)((Ct * 32 + 255) / 256), 256, 0, st>>>(
        ctx->S.as<double>(), Ct, ctx->cols.as<ColMeta>(), ctx->pc, e.mu.as<double>(), e.sigma.as<double>(),
        e.cst.as<double>(), K, e.tab.as<double>(),
        (cst_mode && !(sharded && ctx->kshard_rank != 0)) ? e.part.as<double2>() + nsplit * ctx->ct_stride : nullptr,
        ctx->oob.as<uint8_t>(), e.fix.as<double2>());
    ctx->launch_counter++;
    if (cst_mode && !(sharded && ctx->kshard_rank != 0)) nsplit += 1;
    e.nsplit = (int)nsplit;
  } else if (e.mixed && !ctx->user_points && Ct >= 64 && mixed_cb(ctx) > 0) {
    // mixed space, many candidates: kernel-minor tables, the candidates' table rows in shared memory (tpe_mixed.cuh)
    if (ctx->dtab_doubles) {
      int64_t rows_max = 1;
      for (const ColMeta& cm : ctx->cols_h)
        if (cm.grid > 0) rows_max = std::max<int64_t>(rows_max, (int64_t)std::min<int64_t>(Ct, cm.grid) * (cm.grid + 1));
      const unsigned gx = (unsigned)std::min<int64_t>((rows_max + 255) / 256, ctx->sm_count * 4);
      k_disc_tables<<<dim3(gx, (unsigned)ctx->pc), 256, 0, st>>>(ctx->cols.as<ColMeta>(), ctx->pc, e.mu.as<double>(),
                                                                 e.sigma.as<double>(), K, ctx->S.as<double>(), Ct,
                                                                 e.dtab.as<double>());
      ctx->launch_counter++;
    }
    const int CB = mixed_cb(ctx);
    const int64_t nx = (Ct + CB - 1) / CB;
    int64_t nsplit = std::max<int64_t>(1, std::min<int64_t>(32, (2ll * ctx->sm_count + nx - 1) / nx));
    const int64_t kps = round_up<int64_t>((K - 1 + nsplit - 1) / nsplit, 512);
    nsplit = (K - 1 + kps - 1) / kps;
    CU(e.part.ensure((size_t)(nsplit + 1) * ctx->ct_stride * 16));
    CU(e.fix.ensure((size_t)ctx->ct_stride * 16));
    const size_t smem = mixed_smem(ctx, CB);
    const double skip = std::min(46.0, log((double)std::max<int64_t>(K, 1)) + 30.0);
#define TPE_MIXED_LAUNCH(CBV)                                                                                          \
    do {                                                                                                               \
      static bool attr_done = false;                                                                                   \
      if (!attr_done) {                                                                                                \
        CU(cudaFuncSetAttribute(k_logpdf_mixed<CBV>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));        \
        attr_done = true;                                                                                              \
      }                                                                                                                \
      k_logpdf_mixed<CBV><<<dim3((unsigned)nx, (unsigned)nsplit), 512, smem, st>>>(                                    \
          ctx->S.as<double>(), Ct, ctx->cols.as<ColMeta>(), ctx->pc, ctx->mixcols.as<MixCol>(), ctx->mix_ncont,        \
          ctx->mix_nd, ctx->mix_tabd, e.sigma.as<double>(), e.cst.as<double>(), K - 1, e.mix_kstride, kps,             \
          e.mxc.as<double2>(), e.mxd.as<ushort4>(), e.tab.as<double>(), e.dtab.as<double>(), ctx->oob.as<uint8_t>(),   \
          skip, e.part.as<double2>(), ctx->ct_stride);                                                                 \
    } while (0)
    if (CB == 8) TPE_MIXED_LAUNCH(8);
    else if (CB == 4) TPE_MIXED_LAUNCH(4);
    else TPE_MIXED_LAUNCH(2);
#undef TPE_MIXED_LAUNCH
    ctx->launch_counter++;
    ctx->last_kernel = "k_logpdf_mixed";
    if (after_main) CU(cudaEventRecord(after_main, st));
    k_logpdf_prior_fix<<<(unsigned)((Ct * 32 + 255) / 256), 256, 0, st>>>(
        ctx->S.as<double>(), Ct, ctx->cols.as<ColMeta>(), ctx->pc, e.mu.as<double>(), e.sigma.as<double>(),
        e.cst.as<double>(), K, e.tab.as<double>(), e.part.as<double2>() + nsplit * ctx->ct_stride, ctx->oob.as<uint8_t>(),
        e.fix.as<double2>(), 0);
    ctx->launch_counter++;
    e.nsplit = (int)nsplit + 1;
  } else {
    // pair-parallel generic kernel: grid = (candidates, kernel chunks of 256 * kpt)
    int kpt = 1;
    while ((K + 256ll * kpt - 1) / (256ll * kpt) > 65535 ||
           ((K + 256ll * kpt - 1) / (256ll * kpt)) * Ct > (1ll << 22) * 4)
      kpt *= 2;  // keep the partial table (nsplit x Ct) and the grid within bounds
    const int64_t nsplit = (K + 256ll * kpt - 1) / (256ll * kpt);
    CU(e.part.ensure((size_t)nsplit * ctx->ct_stride * 16));
    e.nsplit = (int)nsplit;
    if (ctx->dtab_doubles) {
      int64_t rows_max = 1;
      for (const ColMeta& cm : ctx->cols_h)
        if (cm.grid > 0) rows_max = std::max<int64_t>(rows_max, (int64_t)std::min<int64_t>(Ct, cm.grid) * (cm.grid + 1));
      const unsigned gx = (unsigned)std::min<int64_t>((rows_max + 255) / 256, ctx->sm_count * 4);
      k_disc_tables<<<dim3(gx, (unsigned)ctx->pc), 256, 0, st>>>(ctx->cols.as<ColMeta>(), ctx->pc, e.mu.as<double>(),
                                                                 e.sigma.as<double>(), K, ctx->S.as<double>(), Ct,
                                                                 e.dtab.as<double>());
      ctx->launch_counter++;
    }
    if (K >= 4096) {
      constexpr int CB = 8;
      k_logpdf_pairs<CB><<<dim3((unsigned)((Ct + CB - 1) / CB), (unsigned)nsplit), 256,
                           (size_t)CB * ctx->pc * sizeof(PairCol) + (((size_t)ctx->pc + 7) & ~(size_t)7), st>>>(
          ctx->S.as<double>(), Ct, ctx->cols.as<ColMeta>(), ctx->pc, e.mu.as<double>(), e.sigma.as<double>(),
          e.cst.as<double>(), K, kpt, e.tab.as<double>(), ctx->dtab_doubles ? e.cls.as<int32_t>() : nullptr,
          ctx->dtab_doubles ? e.dtab.as<double>() : nullptr, ctx->dtab_doubles ? e.offgrid.as<int>() : nullptr,
          ctx->oob.as<uint8_t>(), e.part.as<double2>(), ctx->ct_stride);
    } else {
      constexpr int CB = 1;
      k_logpdf_pairs<CB><<<dim3((unsigned)((Ct + CB - 1) / CB), (unsigned)nsplit), 256,
                           (size_t)CB * ctx->pc * sizeof(PairCol) + (((size_t)ctx->pc + 7) & ~(size_t)7), st>>>(
          ctx->S.as<double>(), Ct, ctx->cols.as<ColMeta>(), ctx->pc, e.mu.as<double>(), e.sigma.as<double>(),
          e.cst.as<double>(), K, kpt, e.tab.as<double>(), ctx->dtab_doubles ? e.cls.as<int32_t>() : nullptr,
          ctx->dtab_doubles ? e.dtab.as<double>() : nullptr, ctx->dtab_doubles ? e.offgrid.as<int>() : nullptr,
          ctx->oob.as<uint8_t>(), e.part.as<double2>(), ctx->ct_stride);
    }
    ctx->launch_counter++;
    ctx->last_kernel = "k_logpdf_pairs";
    if (after_main) CU(cudaEventRecord(after_main, st));
  }
  CU(cudaGetLastError());
  return TPE_OK;
}

int ensure_candidate_buffers(tpe_ctx* ctx, int64_t Ct) {
  ctx->Ct = Ct;
  ctx->cands_sorted = false;
  ctx->ct_stride = round_up<int64_t>(Ct, 1024);
  CU(ctx->S.ensure((size_t)ctx->ct_stride * ctx->pc * 8));
  CU(ctx->oob.ensure((size_t)ctx->ct_stride));
  CU(ctx->logl.ensure((size_t)ctx->ct_stride * 8));
  CU(ctx->logg.ensure((size_t)ctx->ct_stride * 8));
  CU(cudaMemsetAsync(ctx->oob.p, 0, (size_t)ctx->ct_stride, ctx->stream));
  if (ctx->fast) {
    CU(ctx->xT.ensure((size_t)ctx->ct_stride * ctx->pb * 8));
    CU(cudaMemsetAsync(ctx->xT.p, 0, (size_t)ctx->ct_stride * ctx->pb * 8, ctx->stream));
  }
  return TPE_OK;
}

}  // namespace


// ---- univariate batch, stage by stage over all columns (tpe_unib.cuh) ---------------------------------------------------
struct Carver {
  char* base = nullptr;
  size_t off = 0;
  template <class T>
  T* take(size_t count) {
    off = (off + 255) & ~(size_t)255;
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += count * sizeof(T);
    return p;
  }
};
struct UbPtrs {
  double *mu[2], *sigma[2], *cstp[2], *cst[2], *w[2], *logw[2], *cdf, *wpart, *zero, *cstscr, *sc[2], *coef;
  int32_t *ord0, *bstart, *cidx, *sidx, *tlist;
  float4* s32[2];
  double2 *smi[2], *part[2], *fix[2];
  UniTileMeta* meta[2];
  FgtBox* box;
  double *S, *xT, *xs, *logl, *logg;
  uint8_t* oob;
  uint64_t* skeys;
  SortWork* swk;
  int* work;
  ColMeta* cols;
};
static void ub_carve(Carver& c, UbPtrs& p, int P, const int64_t ks[2], int64_t cs, bool big_sort) {
  for (int w = 0; w < 2; ++w) {
    p.mu[w] = c.take<double>((size_t)P * ks[w]);
    p.sigma[w] = c.take<double>((size_t)P * ks[w]);
    p.cstp[w] = c.take<double>((size_t)P * ks[w]);
    p.cst[w] = c.take<double>((size_t)P * ks[w]);
    p.w[w] = c.take<double>((size_t)ks[w]);
    p.logw[w] = c.take<double>((size_t)ks[w]);
    p.s32[w] = c.take<float4>((size_t)P * ks[w]);
    p.smi[w] = c.take<double2>((size_t)P * ks[w]);
    p.sc[w] = c.take<double>((size_t)P * ks[w]);
    p.meta[w] = c.take<UniTileMeta>((size_t)P * (ks[w] / kUniTile));
    p.part[w] = c.take<double2>((size_t)P * 2 * cs);
    p.fix[w] = c.take<double2>((size_t)P * cs);
  }
  p.cdf = c.take<double>((size_t)ks[0]);
  p.wpart = c.take<double>(1024);
  p.zero = c.take<double>((size_t)ks[1]);
  p.cstscr = c.take<double>((size_t)ks[1]);
  p.ord0 = c.take<int32_t>((size_t)P * ks[0]);
  p.bstart = c.take<int32_t>((size_t)P * (kFgtMaxBoxes + 1));
  p.tlist = c.take<int32_t>((size_t)P * (ks[1] / kUniTile + 1));
  p.coef = c.take<double>((size_t)P * kFgtMaxBoxes * kFgtRow);
  p.box = c.take<FgtBox>((size_t)P * kFgtMaxBoxes);
  p.S = c.take<double>((size_t)P * cs);
  p.xT = c.take<double>((size_t)P * cs);
  p.xs = c.take<double>((size_t)P * cs);
  p.cidx = c.take<int32_t>((size_t)P * cs);
  p.logl = c.take<double>((size_t)P * cs);
  p.logg = c.take<double>((size_t)P * cs);
  p.oob = c.take<uint8_t>((size_t)P * cs);
  p.work = c.take<int>((size_t)P * 4);
  p.cols = c.take<ColMeta>((size_t)P);
  if (big_sort) {
    p.skeys = c.take<uint64_t>((size_t)P * 2 * ks[1]);
    p.sidx = c.take<int32_t>((size_t)P * 2 * ks[1]);
    p.swk = c.take<SortWork>((size_t)P);
  } else {
    p.skeys = nullptr;
    p.sidx = nullptr;
    p.swk = nullptr;
  }
}

// The caller (tpe_suggest_univariate_batch) has run the split, checked the weights and compared the above rows with
// the previous call's (ctx->uni_mode); U holds the uniforms [n_cols][2 C] (ctx->ev_u).  Results into ctx->out_*.
static int uni_batch_staged(tpe_ctx* ctx, const tpe_cfg* cfg, const int32_t* cols, int32_t P, const double* w_below,
                            const double* w_above) {
  cudaStream_t st = ctx->stream;
  const int32_t C = cfg->n_candidates;
  const int64_t n[2] = {ctx->est[0].n, ctx->est[1].n};
  const int64_t K[2] = {n[0] + 1, n[1] + 1};
  const int64_t ks[2] = {round_up<int64_t>(K[0] + 160, 1024), round_up<int64_t>(K[1] + 160, 1024)};
  const int64_t cs = round_up<int64_t>(C, 1024);
  const bool big_sort = K[1] > 4096 || K[0] > 4096;
  Carver c0;
  UbPtrs p{};
  ub_carve(c0, p, P, ks, cs, big_sort);
  CU(ctx->ub_arena.ensure(c0.off + 4096));
  Carver c;
  c.base = static_cast<char*>(ctx->ub_arena.p);
  ub_carve(c, p, P, ks, cs, big_sort);
  UbDims d[2];
  for (int w = 0; w < 2; ++w) {
    d[w].ks = ks[w];
    d[w].cs = cs;
    d[w].pall = (int32_t)ctx->space.size();
  }
  kb_cols<<<(P + 63) / 64, 64, 0, st>>>(ctx->cols.as<ColMeta>(), P, p.cols);   // (on the device: a copy from pageable
                                                                               // host memory would wait for the split)
  const ColMeta* dcols = p.cols;
  const int cap = ctx->sm_count * 8;
  const unsigned Pu = (unsigned)P;
  CU(cudaMemsetAsync(p.zero, 0, (size_t)ks[1] * 8, st));
  CU(cudaMemsetAsync(p.oob, 0, (size_t)P * cs, st));
  CU(cudaMemsetAsync(p.work, 0, (size_t)P * 16, st));
  // the above orders of the previous call, if they belong to this one
  DevBuf& ord_new_buf = ctx->ub_ord_cur == 0 ? ctx->ub_ord_b : ctx->ub_ord_a;
  DevBuf& ord_old_buf = ctx->ub_ord_cur == 0 ? ctx->ub_ord_a : ctx->ub_ord_b;
  CU(ord_new_buf.ensure((size_t)P * ks[1] * 4));
  const bool inc = K[1] > 4096 && ctx->ub_ord_seq + 1 == ctx->uni_seq && ctx->ub_ord_lineage == ctx->hist_lineage &&
                   (ctx->ub_ord_K == K[1] || ctx->ub_ord_K == K[1] - 1) && ctx->ub_ord_ks == ks[1] &&
                   ord_old_buf.cap >= (size_t)P * ks[1] * 4 && ctx->ub_ord_cols.size() == (size_t)P &&
                   std::equal(cols, cols + P, ctx->ub_ord_cols.begin());
  int32_t* ord[2] = {p.ord0, ord_new_buf.as<int32_t>()};
  for (int w = 0; w < 2; ++w) {
    const double* wh = w == 0 ? w_below : w_above;
    kb_mu<<<dim3((unsigned)grid_for(K[w], 256, cap), Pu), 256, 0, st>>>(ctx->X.as<double>(), d[w],
                                                                        ctx->est[w].rows.as<int64_t>(), n[w], dcols, p.mu[w]);
    int64_t m2 = 1;
    while (m2 < K[w]) m2 <<= 1;
    if (m2 <= 4096) {
      kb_sort_small<<<dim3(1, Pu), 1024, 0, st>>>(p.mu[w], d[w], (int)K[w], (int)m2, ord[w]);
    } else {
      const int* run_flag = nullptr;
      if (w == 1 && inc) {
        run_flag = ctx->uni_mode.as<int>();
        kb_order_update<<<dim3((unsigned)grid_for(ctx->ub_ord_K, 256, ctx->sm_count), Pu), 256, 0, st>>>(
            run_flag, ord_old_buf.as<int32_t>(), d[1], (int)ctx->ub_ord_K, (int)K[1], p.mu[1], ord[1], p.work);
        ctx->launch_counter++;
      }
      if (ctx->ub_sort_g == 0) {
        int occ = 0;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kb_radix_sort, 512, 0));
        ctx->ub_sort_g = std::max(1, occ) * ctx->sm_count;
      }
      const int G = (int)std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>(160, ctx->ub_sort_g / P), (K[w] + 1023) / 1024));
      if (G * P > ctx->ub_sort_g) return fail(ctx, TPE_E_STATE, "not batchable: %d columns exceed the cooperative sort", P);
      const double* a_mu = p.mu[w];
      UbDims a_d = d[w];
      int a_n = (int)K[w];
      uint64_t* a_keys = p.skeys;
      int32_t* a_idx = p.sidx;
      SortWork* a_wk = p.swk;
      int32_t* a_order = ord[w];
      void* args[] = {&a_mu, &a_d, &a_n, &a_keys, &a_idx, &a_wk, &a_order, &run_flag};
      CU(cudaLaunchCooperativeKernel((const void*)kb_radix_sort, dim3((unsigned)G, Pu), dim3(512), args, 0, st));
    }
    kb_sigma_uni<<<dim3((unsigned)grid_for(K[w], 256, cap), Pu), 256, 0, st>>>(
        p.mu[w], ord[w], d[w], dcols, n[w], cfg->magic_clip, cfg->endpoints, p.sigma[w]);
    kb_const<<<dim3((unsigned)grid_for(K[w], 256, cap), Pu), 256, 0, st>>>(p.mu[w], p.sigma[w], d[w], dcols, K[w], p.cstp[w]);
    // mixture weights: the same for every column
    const double* w_dev = nullptr;
    if (wh != nullptr && n[w] > 0) {
      CU(ctx->ub_wstage.ensure((size_t)(n[0] + n[1] + 2) * 8));
      double* dst = ctx->ub_wstage.as<double>() + (w == 0 ? 0 : n[0] + 1);
      CU(cudaMemcpyAsync(dst, wh, (size_t)n[w] * 8, cudaMemcpyHostToDevice, st));
      w_dev = dst;
    }
    const int64_t k_alloc = round_up<int64_t>(K[w] + 32, 32);
    const int nparts = grid_for(K[w], 2048, ctx->sm_count * 2);
    if (nparts == 1) {
      k_weights_one<<<1, 256, 0, st>>>(w_dev, nullptr, n[w], cfg->prior_weight, p.w[w], p.logw[w], p.zero, p.cstscr,
                                       w == 0 ? p.cdf : nullptr, k_alloc, nullptr, nullptr);
      ctx->launch_counter += 1;
    } else {
      k_wraw<<<nparts, 256, 0, st>>>(w_dev, nullptr, n[w], cfg->prior_weight, p.w[w], p.wpart);
      k_wfinal<<<grid_for(k_alloc, 256, ctx->sm_count * 4), 256, 0, st>>>(p.wpart, nparts, n[w], p.w[w], p.logw[w], p.zero,
                                                                          p.cstscr, w == 0 ? p.cdf : nullptr, k_alloc,
                                                                          nullptr, nullptr);
      k_wnorm<<<grid_for(K[w], 256, ctx->sm_count * 4), 256, 0, st>>>(p.wpart, nparts, K[w], p.w[w]);
      ctx->launch_counter += 3;
    }
    kb_cst<<<dim3((unsigned)grid_for(ks[w], 256, cap), Pu), 256, 0, st>>>(p.cstp[w], p.logw[w], d[w], K[w], p.cst[w]);
    static const int64_t fgt_min = [] { const char* v = getenv("TPE_FGT_MIN_K"); return v ? atoll(v) : 1024ll; }();
    const bool fgt = cfg->magic_clip && K[w] >= fgt_min;
    const unsigned ntiles = (unsigned)((K[w] + kUniTile - 1) / kUniTile);
    kb_uni_tables<<<dim3(ntiles, Pu), kUniTile, 0, st>>>(ord[w], p.mu[w], p.sigma[w], p.cst[w], d[w], dcols, K[w], p.s32[w],
                                                         p.smi[w], p.sc[w], p.meta[w], fgt ? 1 : 0, cfg->magic_clip, p.bstart);
    if (fgt) {
      if (w == 0) return fail(ctx, TPE_E_STATE, "not batchable: a below set of %lld trials", (long long)n[0]);
      kb_fgt_coeff<<<dim3(kFgtMaxBoxes, Pu), 128, 0, st>>>(ord[w], p.mu[w], p.sigma[w], p.cst[w], d[w], dcols, K[w],
                                                           cfg->magic_clip, p.bstart, p.coef, p.box);
      kb_uni_tile_list<<<dim3(1, Pu), 256, 0, st>>>(p.meta[w], d[w], (int)ntiles, p.tlist);
      ctx->launch_counter += 2;
    }
    ctx->launch_counter += 6;
  }
  // candidates of every column from its l(x), both log-densities, the argmax
  CU(cudaStreamWaitEvent(st, ctx->ev_u, 0));
  kb_sample<<<dim3((unsigned)grid_for((int64_t)C, 128, ctx->sm_count * 16), Pu), 128, 0, st>>>(
      ctx->U.as<double>(), C, d[0], dcols, p.cdf, K[0], p.mu[0], p.sigma[0], p.S, p.xT, p.oob);
  kb_uni_sort_cands<<<dim3(1, Pu), 1024, 0, st>>>(p.xT, C, d[0], dcols, p.xs, p.cidx);
  const unsigned ngrp = (unsigned)((C + 31) / 32);
  static const int64_t fgt_min2 = [] { const char* v = getenv("TPE_FGT_MIN_K"); return v ? atoll(v) : 1024ll; }();
  int nsl[2] = {1, 1};
  for (int w = 0; w < 2; ++w) {
    const double skip = std::min(46.0, log((double)std::max<int64_t>(K[w], 1)) + 30.0);
    const bool fgt_w = cfg->magic_clip && K[w] >= fgt_min2;
    kb_uni_grid<<<dim3(ngrp, Pu), kUniWarps * 32, 0, st>>>(p.s32[w], p.smi[w], p.sc[w], p.meta[w], d[w], K[w], p.xs, p.cidx, C,
                                                           skip, p.part[w], fgt_w ? p.tlist : nullptr);
    if (fgt_w) {
      static bool fgt_attr = false;
      if (!fgt_attr) {
        CU(cudaFuncSetAttribute(kb_fgt_eval, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFgtEvalSmem));
        fgt_attr = true;
      }
      kb_fgt_eval<<<dim3((unsigned)((C + kFgtCands - 1) / kFgtCands), Pu), 256, kFgtEvalSmem, st>>>(
          p.coef, p.box, p.bstart, p.s32[w], p.smi[w], p.sc[w], p.mu[w], p.sigma[w], p.cst[w], d[w], dcols, K[w],
          cfg->magic_clip, p.xT, C, p.part[w]);
      nsl[w] = 2;
      ctx->launch_counter++;
    }
    kb_prior_fix<<<dim3((unsigned)(((int64_t)C * 32 + 255) / 256), Pu), 256, 0, st>>>(p.S, C, d[w], dcols, p.mu[w], p.sigma[w],
                                                                                     p.cst[w], K[w], p.oob, p.fix[w]);
    ctx->launch_counter += 2;
  }
  kb_acq2<<<dim3((unsigned)((C + 255) / 256), Pu), 256, 0, st>>>(
      p.part[0], nsl[0], p.part[1], nsl[1], d[0], p.oob, p.fix[0], p.fix[1], C, p.logl, p.logg);
  kb_select<<<dim3(1, Pu), 256, 0, st>>>(p.logl, p.logg, C, d[0], p.S, ctx->out_x.as<double>(), ctx->out_acq.as<double>(),
                                         ctx->out_best.as<int64_t>());
  ctx->launch_counter += 4;
  CU(cudaGetLastError());
  // what the next call may start from
  ctx->ub_ord_cur ^= 1;
  ctx->ub_ord_seq = ctx->uni_seq;
  ctx->ub_ord_lineage = ctx->hist_lineage;
  ctx->ub_ord_K = K[1];
  ctx->ub_ord_ks = ks[1];
  ctx->ub_ord_cols.assign(cols, cols + P);
  ctx->last_kernel = (cfg->magic_clip && K[1] >= fgt_min2) ? "k_uni_grid<sorted 1-D> + k_fgt_eval (staged)"
                                                           : "k_uni_grid<sorted 1-D> (staged)";
  return TPE_OK;
}


// =================================================================================================
extern "C" {

int tpe_abi_version(void) { return TPE_ABI_VERSION; }

int tpe_ctx_create(int device, tpe_ctx** out) {
  if (!out) return TPE_E_INVALID;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) return TPE_E_CUDA;
  tpe_ctx* ctx = new tpe_ctx();
  ctx->device = device;
  if (cudaSetDevice(device) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->stream3, cudaStreamNonBlocking) != cudaSuccess) {
    delete ctx;
    return TPE_E_CUDA;
  }
  for (auto& e : ctx->ev) cudaEventCreate(&e);
  cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&ctx->ev_u, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&ctx->ev_spec, cudaEventDisableTiming);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->sm_count = prop.multiProcessorCount;
  void* mh = nullptr;
  if (cudaHostAlloc(&mh, 625 * 4, cudaHostAllocDefault) != cudaSuccess) {
    tpe_ctx_destroy(ctx);
    return TPE_E_NOMEM;
  }
  memset(mh, 0, 625 * 4);
  ctx->mt_host = static_cast<uint32_t*>(mh);
  *out = ctx;
  return TPE_OK;
}

void tpe_ctx_destroy(tpe_ctx* ctx) {
  if (!ctx) return;
  for (tpe_ctx* c : ctx->uni_sub) tpe_ctx_destroy(c);
  ctx->uni_sub.clear();
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (ctx->stream2) cudaStreamSynchronize(ctx->stream2);
  if (ctx->stream3) cudaStreamSynchronize(ctx->stream3);
  for (DevBuf* b : {&ctx->cat_dist, &ctx->X, &ctx->cat, &ctx->key, &ctx->vals, &ctx->mo_list, &ctx->mo_alive, &ctx->mo_dom,
                    &ctx->mo_first, &ctx->mo_rank, &ctx->mo_ctr, &ctx->mo_tie, &ctx->mo_ntie, &ctx->mo_lexpos,
                    &ctx->mo_isdup, &ctx->mo_sorted, &ctx->mo_uniq, &ctx->mo_nuniq, &ctx->mo_ref, &ctx->mo_removed, &ctx->mo_table,
                    &ctx->mo_sample, &ctx->mo_surv, &ctx->mo_nsurv, &ctx->mo_fv, &ctx->mo_ps, &ctx->mo_map, &ctx->mo_front, &ctx->mo_head,
                    &ctx->mo_contrib, &ctx->mo_state, &ctx->mo_arena, &ctx->mo_chosen, &ctx->mo_diag, &ctx->mo_w, &ctx->cols, &ctx->row_ok, &ctx->member,
                    &ctx->counts, &ctx->split_work, &ctx->below_all, &ctx->kpart, &ctx->mixcols, &ctx->ub_arena, &ctx->ub_ord_a, &ctx->ub_ord_b, &ctx->ub_wstage, &ctx->uxs, &ctx->ucidx, &ctx->uni_prev_rows, &ctx->uni_mode, &ctx->uni_work, &ctx->sort_val, &ctx->sort_idx, &ctx->sort_work, &ctx->U, &ctx->S,
                    &ctx->xT, &ctx->x64s, &ctx->x32s, &ctx->e32s, &ctx->gmax, &ctx->lse_gmax, &ctx->mt_state, &ctx->U2, &ctx->mt_spec, &ctx->mt_jump, &ctx->mt_tmp, &ctx->oob, &ctx->logl, &ctx->logg, &ctx->out_x, &ctx->out_acq, &ctx->out_best,
                    &ctx->ped_member, &ctx->ped_okey, &ctx->ped_work, &ctx->ped_cols, &ctx->ped_grid, &ctx->ped_counts,
                    &ctx->ped_pdf, &ctx->ped_imp, &ctx->ped_loss})
    b->release();
  ctx->est[0].release();
  ctx->est[1].release();
  if (ctx->res_host) cudaFreeHost(ctx->res_host);
  if (ctx->mt_host) cudaFreeHost(ctx->mt_host);
  if (ctx->up_host) cudaFreeHost(ctx->up_host);
  for (auto& e : ctx->up_ev)
    if (e) cudaEventDestroy(e);
  for (auto& e : ctx->ev)
    if (e) cudaEventDestroy(e);
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
  if (ctx->ev_u) cudaEventDestroy(ctx->ev_u);
  if (ctx->ev_spec) cudaEventDestroy(ctx->ev_spec);
  if (ctx->ev_uni) cudaEventDestroy(ctx->ev_uni);
  if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
  if (ctx->stream3) cudaStreamDestroy(ctx->stream3);
  cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char* tpe_last_error(tpe_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int tpe_space_set(tpe_ctx* ctx, const tpe_param_desc* params, int32_t n_params, const double* cat_dist,
                  const int64_t* cat_dist_offset) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (!params || n_params <= 0) return fail(ctx, TPE_E_INVALID, "space must hold at least one parameter");
  if (set_device(ctx)) return TPE_E_CUDA;
  for (int i = 0; i < n_params; ++i) {
    const tpe_param_desc& d = params[i];
    if (d.kind == TPE_KIND_CAT) {
      if (d.n_choices < 1) return fail(ctx, TPE_E_INVALID, "param %d: categorical needs n_choices >= 1", i);
    } else if (d.kind == TPE_KIND_FLOAT || d.kind == TPE_KIND_INT) {
      if (!(d.low <= d.high)) return fail(ctx, TPE_E_INVALID, "param %d: low <= high must hold", i);
      if (d.kind == TPE_KIND_INT && !d.has_step) return fail(ctx, TPE_E_INVALID, "param %d: int needs a step", i);
      if (d.has_step && !(d.step > 0)) return fail(ctx, TPE_E_INVALID, "param %d: step > 0 must hold", i);
      if (d.log && d.kind == TPE_KIND_FLOAT && d.has_step)
        return fail(ctx, TPE_E_INVALID, "param %d: step is not supported when log is true", i);
      if (d.log && !(d.low - (d.has_step ? d.step / 2 : 0.0) > 0))
        return fail(ctx, TPE_E_INVALID, "param %d: low > 0 must hold for log", i);
    } else {
      return fail(ctx, TPE_E_INVALID, "param %d: unknown kind %d", i, d.kind);
    }
  }
  ctx->space.assign(params, params + n_params);
  ctx->cat_dist_off.assign(n_params, -1);
  ctx->cat_dist_h.clear();
  if (cat_dist && cat_dist_offset) {
    int64_t end = 0;
    for (int i = 0; i < n_params; ++i) {
      ctx->cat_dist_off[i] = cat_dist_offset[i];
      if (cat_dist_offset[i] >= 0)
        end = std::max<int64_t>(end, cat_dist_offset[i] + (int64_t)params[i].n_choices * params[i].n_choices);
    }
    ctx->cat_dist_h.assign(cat_dist, cat_dist + end);
    CU(ctx->cat_dist.ensure((size_t)std::max<int64_t>(end, 1) * 8));
    if (end) CU(cudaMemcpy(ctx->cat_dist.p, cat_dist, (size_t)end * 8, cudaMemcpyHostToDevice));
  }
  ctx->col_missing.assign(n_params, 0);
  ctx->col_oor.assign(n_params, 0);
  ctx->col_offgrid.assign(n_params, 0);
  ctx->hist_lineage++;
  ctx->N = 0;
  ctx->history_set = false;
  ctx->prepared = ctx->built = ctx->sampled = false;
  ctx->hist_version++;
  return TPE_OK;
}

int tpe_history_set(tpe_ctx* ctx, const double* X, const int8_t* category, const double* key, int64_t n) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (ctx->space.empty()) return fail(ctx, TPE_E_STATE, "tpe_space_set must precede tpe_history_set");
  if (n < 0 || (n > 0 && (!X || !category || !key))) return fail(ctx, TPE_E_INVALID, "bad history arguments");
  if (n >= (1ll << 31) - 4096) return fail(ctx, TPE_E_INVALID, "history too long");
  if (set_device(ctx)) return TPE_E_CUDA;
  std::fill(ctx->col_missing.begin(), ctx->col_missing.end(), 0);
  std::fill(ctx->col_oor.begin(), ctx->col_oor.end(), 0);
  std::fill(ctx->col_offgrid.begin(), ctx->col_offgrid.end(), 0);
  ctx->hist_lineage++;
  scan_missing(ctx, X, category, n);
  return upload_history(ctx, X, category, key, n, 0, false);
}

int tpe_history_append(tpe_ctx* ctx, const double* X, const int8_t* category, const double* key, int64_t n) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (ctx->space.empty()) return fail(ctx, TPE_E_STATE, "tpe_space_set must precede tpe_history_append");
  if (n < 0 || (n > 0 && (!X || !category || !key))) return fail(ctx, TPE_E_INVALID, "bad history arguments");
  if (ctx->N + n >= (1ll << 31) - 4096) return fail(ctx, TPE_E_INVALID, "history too long");
  if (set_device(ctx)) return TPE_E_CUDA;
  scan_missing(ctx, X, category, n);
  return upload_history(ctx, X, category, key, n, ctx->N, false);
}

int tpe_history_update(tpe_ctx* ctx, const double* X, const int8_t* category, const double* key, int64_t n,
                       int64_t at_row) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (!ctx->history_set) return fail(ctx, TPE_E_STATE, "tpe_history_set must precede tpe_history_update");
  if (n < 0 || at_row < 0 || at_row > ctx->N || (n > 0 && (!X || !category || !key)))
    return fail(ctx, TPE_E_INVALID, "tpe_history_update: rows [%lld, %lld) do not continue the history of %lld rows",
                (long long)at_row, (long long)(at_row + n), (long long)ctx->N);
  if (n == 0) return TPE_OK;
  if (at_row + n >= (1ll << 31) - 4096) return fail(ctx, TPE_E_INVALID, "history too long");
  if (set_device(ctx)) return TPE_E_CUDA;
  if ((int64_t)ctx->cat_h.size() != ctx->N)
    return fail(ctx, TPE_E_STATE, "tpe_history_update needs a host-uploaded history");
  scan_missing(ctx, X, category, n);
  const int64_t P = (int64_t)ctx->space.size();
  const int64_t total = std::max(ctx->N, at_row + n);
  if (total > ctx->N) {  // the write runs past the end: the history grows (rows [at_row, N) are overwritten)
    CU(ctx->X.grow((size_t)total * P * 8, (size_t)ctx->N * P * 8, ctx->stream));
    CU(ctx->cat.grow((size_t)total, (size_t)ctx->N, ctx->stream));
    CU(ctx->key.grow((size_t)total * 16, (size_t)ctx->N * 16, ctx->stream));
    if (ctx->M >= 2)
      CU(ctx->vals.grow((size_t)total * ctx->M * 8, (size_t)ctx->N * ctx->M * 8, ctx->stream));
  }
  if (rows_fit_staging(ctx, n)) {
    if (int rc = stage_rows(ctx, X, category, key, n, at_row)) return rc;
  } else {
    CU(cudaMemcpyAsync(ctx->X.as<double>() + at_row * P, X, (size_t)n * P * 8, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(ctx->cat.as<int8_t>() + at_row, category, (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(ctx->key.as<double>() + at_row * 2, key, (size_t)n * 16, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
  }
  ctx->cat_h.resize((size_t)total, (int8_t)TPE_CAT_EXCLUDED);
  for (int64_t i = 0; i < n; ++i) {
    const int64_t r = at_row + i;
    if (r < ctx->N) {
      if (cat_slot(ctx->cat_h[(size_t)r]) != 4) ctx->hist_lineage++;   // a row the estimators could see is replaced
      ctx->cat_cnt[cat_slot(ctx->cat_h[(size_t)r])]--;
    }
    ctx->cat_h[(size_t)r] = category[i];
    ctx->cat_cnt[cat_slot(category[i])]++;
  }
  ctx->N = total;
  ctx->prepared = ctx->built = ctx->sampled = false;
  ctx->hist_version++;
  return TPE_OK;
}

int tpe_history_set_device(tpe_ctx* ctx, const double* dX, const int8_t* dcategory, const double* dkey, int64_t n,
                           const uint8_t* col_has_missing) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (ctx->space.empty()) return fail(ctx, TPE_E_STATE, "tpe_space_set must precede tpe_history_set_device");
  if (n < 0 || (n > 0 && (!dX || !dcategory || !dkey))) return fail(ctx, TPE_E_INVALID, "bad history arguments");
  if (set_device(ctx)) return TPE_E_CUDA;
  ctx->hist_lineage++;
  for (size_t j = 0; j < ctx->col_missing.size(); ++j) ctx->col_missing[j] = col_has_missing ? col_has_missing[j] : 1;
  // a history adopted from device memory is not scanned on the host: treat every column as possibly out of range
  // unless the caller vouches for it through col_has_missing (the broadcast path of optuna_b200/dist.py does)
  std::fill(ctx->col_oor.begin(), ctx->col_oor.end(), col_has_missing ? 0 : 1);
  std::fill(ctx->col_offgrid.begin(), ctx->col_offgrid.end(), col_has_missing ? 0 : 1);
  return upload_history(ctx, dX, dcategory, dkey, n, 0, true);
}

int tpe_history_set_values(tpe_ctx* ctx, const double* values, int64_t n, int32_t n_objectives, int64_t at_row) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (!ctx->history_set) return fail(ctx, TPE_E_STATE, "tpe_history_set must precede tpe_history_set_values");
  if (n_objectives < 1 || n_objectives > kMoMaxM)
    return fail(ctx, TPE_E_INVALID, "n_objectives must be in [1, %d]", kMoMaxM);
  if (n < 0 || at_row < 0 || at_row + n > ctx->N || (n > 0 && !values))
    return fail(ctx, TPE_E_INVALID, "bad values range");
  if (at_row > 0 && n_objectives != ctx->M) return fail(ctx, TPE_E_INVALID, "n_objectives changed");
  ctx->hist_lineage++;
  if (set_device(ctx)) return TPE_E_CUDA;
  // a partial write keeps every row already there (rows after the written range included)
  const size_t keep = (n_objectives == ctx->M && at_row > 0)
                          ? std::min(ctx->vals.cap, (size_t)ctx->N * n_objectives * 8) : 0;
  CU(ctx->vals.grow((size_t)std::max<int64_t>(ctx->N, 1) * n_objectives * 8, keep, ctx->stream));
  if (n > 0)
    CU(cudaMemcpyAsync(ctx->vals.as<double>() + at_row * n_objectives, values, (size_t)n * n_objectives * 8,
                       cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->M = n_objectives;
  ctx->prepared = ctx->built = ctx->sampled = false;
  ctx->hist_version++;
  return TPE_OK;
}

int tpe_get_mo_weights(tpe_ctx* ctx, double* weights) {
  if (!ctx || !weights) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (!ctx->built || !ctx->mo_weights_ready) return fail(ctx, TPE_E_STATE, "no MOTPE weights available");
  if (set_device(ctx)) return TPE_E_CUDA;
  CU(cudaMemcpyAsync(weights, ctx->mo_w.p, (size_t)ctx->info.n_below_all * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return TPE_OK;
}

int64_t tpe_history_size(tpe_ctx* ctx) { return ctx ? ctx->N : -1; }

int tpe_history_device_ptrs(tpe_ctx* ctx, double** dX, int8_t** dcategory, double** dkey) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (!ctx->history_set) return fail(ctx, TPE_E_STATE, "no history");
  if (dX) *dX = ctx->X.as<double>();
  if (dcategory) *dcategory = ctx->cat.as<int8_t>();
  if (dkey) *dkey = ctx->key.as<double>();
  return TPE_OK;
}

// The selected columns of a call: kinds, kernel-space bounds, table offsets, which grid kernel family applies;
// uploads the ColMeta array.  Returns (through need_rowok) whether any selected column has absent values.
static int setup_columns(tpe_ctx* ctx, const tpe_cfg* cfg, const int32_t* cols, int32_t n_cols, bool* need_rowok_out) {
  const int P = (int)ctx->space.size();
  ctx->cols_h.clear();
  ctx->ncont = ctx->ndisc = ctx->ncat = ctx->nnum = 0;
  int64_t tab = 0, dtab = 0;
  bool need_rowok = false;
  for (int j = 0; j < n_cols; ++j) {
    const int src = cols[j];
    if (src < 0 || src >= P) return fail(ctx, TPE_E_INVALID, "column %d out of range", src);
    const tpe_param_desc& d = ctx->space[src];
    ColMeta cm{};
    cm.src = src;
    cm.log = d.log;
    cm.nch = d.n_choices;
    cm.low = d.low;
    cm.high = d.high;
    cm.step = d.has_step ? d.step : 0.0;
    cm.num_rank = cm.cat_rank = -1;
    cm.dist_off = -1;
    if (d.kind == TPE_KIND_CAT) {
      cm.cls = COL_CAT;
      cm.cat_rank = ctx->ncat++;
      cm.slot = cm.cat_rank;
      cm.tab_off = (int32_t)tab;
      tab += 2ll * (d.n_choices + 1) * d.n_choices;
      cm.dist_off = (int32_t)ctx->cat_dist_off[src];
    } else {
      cm.num_rank = ctx->nnum++;
      double lo = d.low, hi = d.high;
      if (d.has_step) {
        lo -= d.step / 2;
        hi += d.step / 2;
      }
      if (d.log) {
        lo = log(lo);
        hi = log(hi);
      }
      cm.klow = lo;
      cm.khigh = hi;
      if (d.has_step) {
        cm.cls = COL_DISC;
        cm.slot = ctx->ndisc++;
        const double gsz = floor((d.high - d.low) / d.step + 0.5) + 1.0;
        if (cfg->multivariate && gsz >= 1.0 && gsz <= 4096.0 && dtab + (int64_t)(gsz + 1) * (int64_t)gsz <= (1ll << 24)) {
          cm.grid = (int32_t)gsz;
          cm.dtab_off = dtab;
          dtab += (int64_t)(gsz + 1) * (int64_t)gsz;
        }
      } else {
        cm.cls = COL_CONT;
        cm.slot = ctx->ncont++;
      }
    }
    need_rowok = need_rowok || ctx->col_missing[src];
    ctx->cols_h.push_back(cm);
  }
  ctx->pc = n_cols;
  ctx->tab_doubles = tab;
  ctx->dtab_doubles = dtab;
  ctx->fast = (ctx->ndisc == 0 && ctx->ncat == 0 && ctx->ncont <= kMaxFastP);
  ctx->pb = ctx->fast ? pick_pb(ctx->ncont) : 0;
  ctx->fast_mode = ctx->fast ? (cfg->multivariate ? 2 : 1) : 0;
  static const bool uni_on = [] { const char* v = getenv("TPE_UNI_FAST"); return !(v && v[0] == '0'); }();
  ctx->uni_fast = uni_on && !cfg->multivariate && n_cols == 1 && ctx->ncont == 1;
  // mixed spaces with many candidates: kernel-minor tables + per-candidate table rows in shared memory
  static const bool mixed_on = [] { const char* v = getenv("TPE_MIXED"); return !(v && v[0] == '0'); }();
  ctx->mixed_ok = mixed_on && cfg->multivariate && !ctx->fast && ctx->ndisc + ctx->ncat > 0 && ctx->ncont <= 128 &&
                  ctx->ndisc + ctx->ncat <= 128;
  ctx->mixcols_h.clear();
  if (ctx->mixed_ok) {
    int off = 0;
    std::vector<MixCol> tail;
    for (int j = 0; j < n_cols && ctx->mixed_ok; ++j) {
      const ColMeta& cm = ctx->cols_h[j];
      if (cm.cls == COL_CONT) {
        ctx->mixcols_h.push_back(MixCol{j, 0, 0, 0});
      } else if (cm.cls == COL_DISC) {
        if (cm.grid <= 0 || cm.grid > 65535 || ctx->col_offgrid[cm.src]) ctx->mixed_ok = false;
        tail.push_back(MixCol{j, 1, cm.grid, off});
        off += cm.grid;
      } else {
        tail.push_back(MixCol{j, 2, cm.nch, off});
        off += cm.nch;
      }
    }
    ctx->mix_ncont = (int)ctx->mixcols_h.size();
    ctx->mix_nd = (int)tail.size();
    ctx->mix_tabd = off;
    ctx->mixcols_h.insert(ctx->mixcols_h.end(), tail.begin(), tail.end());
    if (ctx->mixed_ok) {
      CU(ctx->mixcols.ensure(sizeof(MixCol) * ctx->mixcols_h.size()));
      CU(cudaMemcpyAsync(ctx->mixcols.p, ctx->mixcols_h.data(), sizeof(MixCol) * ctx->mixcols_h.size(),
                         cudaMemcpyHostToDevice, ctx->stream));
    }
  }
  CU(ctx->cols.ensure(sizeof(ColMeta) * n_cols));
  CU(cudaMemcpyAsync(ctx->cols.p, ctx->cols_h.data(), sizeof(ColMeta) * n_cols, cudaMemcpyHostToDevice, ctx->stream));

  *need_rowok_out = need_rowok;
  return TPE_OK;
}

static int prepare_locked(tpe_ctx* ctx, const tpe_cfg* cfg, const int32_t* cols, int32_t n_cols,
                          tpe_split_info* info) {
  if (!ctx->history_set) return fail(ctx, TPE_E_STATE, "tpe_history_set must precede tpe_prepare");
  if (!cfg || !cols || n_cols <= 0) return fail(ctx, TPE_E_INVALID, "bad prepare arguments");
  if (cfg->prior_weight < 0)
    return fail(ctx, TPE_E_INVALID, "A non-negative value must be specified for prior_weight, but got %g.",
                cfg->prior_weight);
  if (cfg->n_candidates <= 0) return fail(ctx, TPE_E_INVALID, "n_candidates must be positive");
  if (set_device(ctx)) return TPE_E_CUDA;
  ctx->cfg = *cfg;
  ctx->launch_counter = 0;
  ctx->deferred = false;   // a new sequence abandons results nobody collected
  ctx->deferred_uni = 0;
  CU(cudaEventRecord(ctx->ev[0], ctx->stream));
  bool need_rowok = false;
  if (int rc0 = setup_columns(ctx, cfg, cols, n_cols, &need_rowok)) return rc0;
  const int P = (int)ctx->space.size();
  const int64_t N = ctx->N;
  const int64_t nal = std::max<int64_t>(N, 1);
  CU(ctx->counts.ensure(64));
  for (int w = 0; w < 2; ++w) {
    CU(ctx->est[w].rows.ensure((size_t)nal * 8));
  }
  CU(ctx->est[0].pos.ensure((size_t)nal * 8));
  const uint8_t* rowok = nullptr;
  if (need_rowok && N > 0) {
    CU(ctx->row_ok.ensure((size_t)nal));
    k_rowok<<<grid_for(N, 256, ctx->sm_count * 8), 256, 0, ctx->stream>>>(
        ctx->X.as<double>(), N, P, ctx->cols.as<ColMeta>(), n_cols, ctx->row_ok.as<uint8_t>());
    ctx->launch_counter++;
    rowok = ctx->row_ok.as<uint8_t>();
  }
  const uint8_t* pre_member = nullptr;
  int64_t nb_rest = cfg->n_below;
  ctx->mo_weights_ready = false;
  if (ctx->M >= 2) {
    int64_t taken = 0;
    int rc = mo_select_complete(ctx, cfg->n_below, &taken);
    if (rc) return rc;
    pre_member = ctx->member.as<uint8_t>();
    nb_rest = std::max<int64_t>(0, cfg->n_below - taken);
  }
  const bool plain = !need_rowok && ctx->M < 2;
  // univariate only: a multivariate suggestion prepares once per trial anyway, and a benchmark that asks
  // repeatedly against a frozen history must pay for its split every time
  const bool reuse_split = plain && !cfg->multivariate && ctx->split_valid &&
                           ctx->split_version == ctx->hist_version && ctx->split_n_below == (int64_t)cfg->n_below;
  if (!reuse_split) {
    CU(ctx->split_work.ensure(sizeof(SplitWork)));
    CU(cudaMemsetAsync(ctx->split_work.p, 0, sizeof(SplitWork), ctx->stream));
    int n_i = (int)N;
    int64_t nb = nb_rest;
    const int8_t* d_cat = ctx->cat.as<int8_t>();
    const double* d_key = ctx->key.as<double>();
    SplitWork* d_wk = ctx->split_work.as<SplitWork>();
    int64_t* d_b = ctx->est[0].rows.as<int64_t>();
    int64_t* d_p = ctx->est[0].pos.as<int64_t>();
    int64_t* d_a = ctx->est[1].rows.as<int64_t>();
    int64_t* d_c = ctx->counts.as<int64_t>();
    int64_t* d_ball = nullptr;
    if (ctx->M >= 2) {
      CU(ctx->below_all.ensure((size_t)nal * 8));
      d_ball = ctx->below_all.as<int64_t>();
    }
    void* args[] = {&n_i, &d_cat, &d_key, &nb, &rowok, &pre_member, &d_wk, &d_b, &d_p, &d_a, &d_c, &d_ball};
    const int G = (int)std::max<int64_t>(1, std::min<int64_t>(ctx->sm_count, (N + 1023) / 1024));
    CU(cudaLaunchCooperativeKernel((const void*)k_split_coop, dim3(G), dim3(512), args, 0, ctx->stream));
    ctx->launch_counter++;
    ctx->split_valid = plain;
    ctx->split_version = ctx->hist_version;
    ctx->split_n_below = cfg->n_below;
  }
  CU(cudaGetLastError());
  CU(cudaEventRecord(ctx->ev[1], ctx->stream));
  int64_t counts[3];
  // Without missing parameters the sizes of the two sets follow from the category counts alone
  // (sampler.py:686-722: whole categories in order, the cut inside one of them), which the host
  // mirror knows: no read-back, the builds are queued while the split still runs.
  // TPE_VERIFY_COUNTS=1 reads the device counts back as well and compares.
  static const bool verify_counts = [] { const char* v = getenv("TPE_VERIFY_COUNTS"); return v && v[0] == '1'; }();
  const bool predict = !need_rowok && ctx->M < 2 && (int64_t)ctx->cat_h.size() == N;
  if (predict) {
    const int64_t* cnt = ctx->cat_cnt;
    int64_t remaining = std::max<int64_t>(cfg->n_below, 0), below = 0;
    for (int c = 0; c < 3; ++c) {
      const int64_t take = std::min(remaining, cnt[c]);
      below += take;
      remaining -= take;
      if (take < cnt[c]) break;
    }
    counts[0] = counts[1] = below;
    counts[2] = N - cnt[4] - below;  // TPE_CAT_EXCLUDED rows are in neither set
  }
  if (!predict || verify_counts) {
    int64_t dev[3];
    CU(cudaMemcpyAsync(dev, ctx->counts.p, sizeof(dev), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    if (predict && (dev[0] != counts[0] || dev[1] != counts[1] || dev[2] != counts[2]))
      return fail(ctx, TPE_E_STATE, "split sizes: host prediction (%lld, %lld, %lld) != device (%lld, %lld, %lld)",
                  (long long)counts[0], (long long)counts[1], (long long)counts[2], (long long)dev[0],
                  (long long)dev[1], (long long)dev[2]);
    counts[0] = dev[0]; counts[1] = dev[1]; counts[2] = dev[2];
  }
  ctx->info.n_below_all = counts[0];
  ctx->info.n_below_obs = counts[1];
  ctx->info.n_above_obs = counts[2];
  ctx->est[0].n = counts[1];
  ctx->est[1].n = counts[2];
  if (info) *info = ctx->info;
  ctx->prepared = true;
  ctx->built = ctx->sampled = false;
  return TPE_OK;
}

int tpe_prepare(tpe_ctx* ctx, const tpe_cfg* cfg, const int32_t* cols, int32_t n_cols, tpe_split_info* info) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  return prepare_locked(ctx, cfg, cols, n_cols, info);
}

static int build_locked(tpe_ctx* ctx, const double* w_below, const double* w_above) {
  if (!ctx->prepared) return fail(ctx, TPE_E_STATE, "tpe_prepare must precede tpe_build");
  if (set_device(ctx)) return TPE_E_CUDA;
  for (int which = 0; which < 2; ++which) {
    const double* w = which == 0 ? w_below : w_above;
    const int64_t n = ctx->est[which].n;
    if (w) {  // the reference's _call_weights_func checks (parzen_estimator.py:88-109)
      double tot = 0;
      for (int64_t i = 0; i < n; ++i) {
        if (w[i] < 0) return fail(ctx, TPE_E_INVALID, "The `weights` function is not allowed to return negative values.");
        if (!isfinite(w[i]))
          return fail(ctx, TPE_E_INVALID, "The `weights`function is not allowed to return infinite or NaN values.");
        tot += w[i];
      }
      if (n > 0 && tot <= 0)
        return fail(ctx, TPE_E_INVALID, "The `weight` function is not allowed to return all-zero values.");
    }
  }
  // multivariate builds share no scratch: g(x)'s estimator (the big one) goes to the second stream
  const bool fork = ctx->cfg.multivariate != 0;
  if (fork) {
    CU(cudaEventRecord(ctx->ev_fork, ctx->stream));
    CU(cudaStreamWaitEvent(ctx->stream2, ctx->ev_fork, 0));
    int rc = build_estimator(ctx, 1, w_above, ctx->stream2);
    if (rc) return rc;
    CU(cudaEventRecord(ctx->ev_join, ctx->stream2));
    ctx->above_pending = true;
    rc = build_estimator(ctx, 0, w_below, ctx->stream);
    if (rc) return rc;
  } else {
    for (int which = 0; which < 2; ++which) {
      int rc = build_estimator(ctx, which, which == 0 ? w_below : w_above, ctx->stream);
      if (rc) return rc;
    }
  }
  CU(cudaEventRecord(ctx->ev[2], ctx->stream));
  ctx->built = true;
  ctx->sampled = false;
  return TPE_OK;
}

int tpe_build(tpe_ctx* ctx, const double* w_below, const double* w_above) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  return build_locked(ctx, w_below, w_above);
}

// Candidates, both log-density grids and the argmax of n_asks asks whose uniforms are resident in ctx->U: launches
// only (ctx->stream); results in ctx->out_x / out_acq / out_best.
static int launch_sample_select(tpe_ctx* ctx, int64_t n_asks, bool used_dev_rng, bool timed) {
  cudaStream_t st = ctx->stream;
  const int32_t C = ctx->cfg.n_candidates;
  const int64_t Ct = n_asks * C;
  const int64_t per_ask = (int64_t)C * (1 + ctx->ncat + ctx->nnum);
  int rc = TPE_OK;
  (void)per_ask;
  if (timed) CU(cudaEventRecord(ctx->ev[3], st));
  ctx->user_points = false;
  Estimator& eb = ctx->est[0];
  k_sample<<<grid_for(Ct * ctx->pc, 128, ctx->sm_count * 16), 128, 0, st>>>(
      ctx->U.as<double>(), n_asks, C, ctx->cols.as<ColMeta>(), ctx->pc, ctx->ncat, ctx->nnum, eb.cdf.as<double>(),
      eb.K, eb.mu.as<double>(), eb.sigma.as<double>(), eb.tab.as<double>(), ctx->S.as<double>(),
      ctx->fast ? ctx->xT.as<double>() : nullptr, ctx->ct_stride, ctx->oob.as<uint8_t>());
  ctx->launch_counter++;
  if (timed) CU(cudaEventRecord(ctx->ev[4], st));
  if (used_dev_rng) {
    // speculative draw for the next ask (same count) from the state this ask's draw ended in; runs on
    // the side stream while the grid kernels of this ask run
    static const bool spec_on = [] { const char* v = getenv("TPE_RNG_SPECULATE"); return !(v && v[0] == '0'); }();
    const int64_t count = n_asks * per_ask;
    if (spec_on) {
      CU(ctx->U2.ensure((size_t)count * 8));
      CU(ctx->mt_spec.ensure(625 * 4));
      CU(cudaMemcpyAsync(ctx->mt_spec.p, ctx->mt_state.p, 625 * 4, cudaMemcpyDeviceToDevice, ctx->stream3));
      if (int rc2 = launch_mt(ctx, ctx->stream3, ctx->mt_spec.as<uint32_t>(), 0, count, ctx->U2.as<double>())) return rc2;
      CU(cudaEventRecord(ctx->ev_spec, ctx->stream3));
      ctx->spec_pending = true;
      ctx->spec_count = count;
    }
    // the generator's end state comes back with the results (tpe_rng_state then needs no device access)
    CU(cudaMemcpyAsync(ctx->mt_host, ctx->mt_state.p, (size_t)625 * 4, cudaMemcpyDeviceToHost, st));
  }
  rc = run_logpdf(ctx, 0, Ct);
  if (rc) return rc;
  if (timed) CU(cudaEventRecord(ctx->ev[5], st));
  rc = run_logpdf(ctx, 1, Ct, timed ? ctx->ev[6] : nullptr);
  if (rc) return rc;
  if (timed) CU(cudaEventRecord(ctx->ev[7], st));
  if (ctx->kshard_world > 1) {
    // one (max, sum) per candidate over this context's slice of g(x); the caller gathers them from all ranks and
    // finishes with tpe_finish_from_partials
    CU(ctx->kpart.ensure((size_t)ctx->ct_stride * 16));
    k_reduce_parts<<<grid_for(Ct, 256, ctx->sm_count * 8), 256, 0, st>>>(ctx->est[1].part.as<double2>(), ctx->est[1].nsplit,
                                                                         ctx->ct_stride, Ct, ctx->kpart.as<double2>());
    ctx->launch_counter++;
    ctx->partial_ready = true;
    return TPE_OK;
  }
  k_acq<<<grid_for(Ct * 32, 256, ctx->sm_count * 8), 256, 0, st>>>(
      ctx->est[0].part.as<double2>(), ctx->est[0].nsplit, ctx->est[1].part.as<double2>(), ctx->est[1].nsplit,
      ctx->ct_stride, ctx->fast ? ctx->oob.as<uint8_t>() : nullptr, ctx->est[0].fix.as<double2>(),
      ctx->est[1].fix.as<double2>(), Ct, ctx->logl.as<double>(), ctx->logg.as<double>());
  k_select<<<(unsigned)n_asks, 256, 0, st>>>(ctx->logl.as<double>(), ctx->logg.as<double>(), C, ctx->S.as<double>(),
                                             ctx->pc, ctx->out_x.as<double>(), ctx->out_acq.as<double>(),
                                             ctx->out_best.as<int64_t>());
  ctx->launch_counter += 2;
  return TPE_OK;
}

// Everything of tpe_sample_and_select up to the last kernel.  defer: the results are also copied into the
// context's page-locked staging area and nothing is waited for (tpe_sample_and_select_async).
static int sample_select_issue(tpe_ctx* ctx, const double* uniforms, int64_t n_asks, bool defer) {
  if (!ctx->built) return fail(ctx, TPE_E_STATE, "tpe_build must precede tpe_sample_and_select");
  if ((!uniforms && !ctx->u_device_rng) || n_asks <= 0)
    return fail(ctx, TPE_E_INVALID, "bad sample arguments");
  if (set_device(ctx, /*join=*/false)) return TPE_E_CUDA;  // est[1] is joined by run_logpdf(ctx, 1)
  cudaStream_t st = ctx->stream;
  const int32_t C = ctx->cfg.n_candidates;
  const int64_t Ct = n_asks * C;
  const int64_t per_ask = (int64_t)C * (1 + ctx->ncat + ctx->nnum);
  ctx->n_asks = n_asks;
  ctx->deferred = false;
  int rc = ensure_candidate_buffers(ctx, Ct);
  if (rc) return rc;
  CU(ctx->U.ensure((size_t)n_asks * per_ask * 8));
  CU(ctx->out_x.ensure((size_t)n_asks * ctx->pc * 8));
  CU(ctx->out_acq.ensure((size_t)n_asks * 8));
  CU(ctx->out_best.ensure((size_t)n_asks * 8));
  const bool used_dev_rng = !uniforms;
  if (!uniforms) {
    if (ctx->u_staged_count != n_asks * per_ask)
      return fail(ctx, TPE_E_INVALID, "device-generated uniforms: %lld staged, %lld needed",
                  (long long)ctx->u_staged_count, (long long)(n_asks * per_ask));
    CU(cudaStreamWaitEvent(st, ctx->ev_u, 0));  // generated by tpe_stage_uniforms_mt19937
    ctx->u_device_rng = false;
  } else if (ctx->u_staged == uniforms && ctx->u_staged_count == n_asks * per_ask) {
    CU(cudaStreamWaitEvent(st, ctx->ev_u, 0));  // uploaded by tpe_suggest while the split ran
  } else {
    if (ctx->u_device_rng) {  // a device draw nobody consumed is still writing U on the side stream
      CU(cudaStreamWaitEvent(st, ctx->ev_u, 0));
      ctx->u_device_rng = false;
    }
    CU(cudaMemcpyAsync(ctx->U.p, uniforms, (size_t)n_asks * per_ask * 8, cudaMemcpyHostToDevice, st));
  }
  ctx->u_staged = nullptr;
  rc = launch_sample_select(ctx, n_asks, used_dev_rng, true);
  if (rc) return rc;
  CU(cudaEventRecord(ctx->ev[8], st));
  CU(cudaGetLastError());
  ctx->issued_dev_rng = used_dev_rng;
  if (defer) {
    const size_t need = (size_t)n_asks * (ctx->pc + 2) * 8;
    if (ctx->res_host_cap < need) {
      if (ctx->res_host) cudaFreeHost(ctx->res_host);
      ctx->res_host = nullptr;
      ctx->res_host_cap = 0;
      CU(cudaHostAlloc(&ctx->res_host, need + 4096, cudaHostAllocDefault));
      ctx->res_host_cap = need + 4096;
    }
    char* h = static_cast<char*>(ctx->res_host);
    CU(cudaMemcpyAsync(h, ctx->out_x.p, (size_t)n_asks * ctx->pc * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(h + (size_t)n_asks * ctx->pc * 8, ctx->out_acq.p, (size_t)n_asks * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(h + (size_t)n_asks * (ctx->pc + 1) * 8, ctx->out_best.p, (size_t)n_asks * 8,
                       cudaMemcpyDeviceToHost, st));
    ctx->deferred = true;
  }
  return TPE_OK;
}

static int sample_select_finish(tpe_ctx* ctx) {
  CU(cudaStreamSynchronize(ctx->stream));
  if (ctx->issued_dev_rng) ctx->mt_host_valid = true;
  for (int i = 0; i < 8; ++i) cudaEventElapsedTime(&ctx->ms[i], ctx->ev[i], ctx->ev[i + 1]);
  cudaEventElapsedTime(&ctx->ms[8], ctx->ev[0], ctx->ev[8]);
  ctx->launches = ctx->launch_counter;
  ctx->sampled = true;
  ctx->deferred = false;
  return TPE_OK;
}

static int sample_select_locked(tpe_ctx* ctx, const double* uniforms, int64_t n_asks, double* out_x, double* out_acq,
                                int64_t* out_best) {
  int rc = sample_select_issue(ctx, uniforms, n_asks, false);
  if (rc) return rc;
  cudaStream_t st = ctx->stream;
  if (out_x) CU(cudaMemcpyAsync(out_x, ctx->out_x.p, (size_t)n_asks * ctx->pc * 8, cudaMemcpyDeviceToHost, st));
  if (out_acq) CU(cudaMemcpyAsync(out_acq, ctx->out_acq.p, (size_t)n_asks * 8, cudaMemcpyDeviceToHost, st));
  if (out_best) CU(cudaMemcpyAsync(out_best, ctx->out_best.p, (size_t)n_asks * 8, cudaMemcpyDeviceToHost, st));
  return sample_select_finish(ctx);
}

int tpe_sample_and_select(tpe_ctx* ctx, const double* uniforms, int64_t n_asks, double* out_x, double* out_acq,
                          int64_t* out_best) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  return sample_select_locked(ctx, uniforms, n_asks, out_x, out_acq, out_best);
}

int tpe_sample_and_select_async(tpe_ctx* ctx, const double* uniforms, int64_t n_asks) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  return sample_select_issue(ctx, uniforms, n_asks, true);
}

int tpe_collect(tpe_ctx* ctx, double* out_x, double* out_acq, int64_t* out_best) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (!ctx->deferred) return fail(ctx, TPE_E_STATE, "tpe_collect needs a pending tpe_sample_and_select_async");
  if (set_device(ctx, /*join=*/false)) return TPE_E_CUDA;
  const int64_t n_asks = ctx->n_asks;
  int rc = sample_select_finish(ctx);
  if (rc) return rc;
  const char* h = static_cast<const char*>(ctx->res_host);
  if (out_x) memcpy(out_x, h, (size_t)n_asks * ctx->pc * 8);
  if (out_acq) memcpy(out_acq, h + (size_t)n_asks * ctx->pc * 8, (size_t)n_asks * 8);
  if (out_best) memcpy(out_best, h + (size_t)n_asks * (ctx->pc + 1) * 8, (size_t)n_asks * 8);
  return TPE_OK;
}

int tpe_set_kernel_shard(tpe_ctx* ctx, int32_t rank, int32_t world) {
  if (!ctx || world < 1 || rank < 0 || rank >= world) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  ctx->kshard_rank = rank;
  ctx->kshard_world = world;
  ctx->partial_ready = false;
  return TPE_OK;
}

int tpe_sample_and_partial(tpe_ctx* ctx, const double* uniforms, int64_t n_asks, double** d_partials, int64_t* stride) {
  if (!ctx || !d_partials) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (ctx->kshard_world < 2) return fail(ctx, TPE_E_STATE, "tpe_set_kernel_shard(rank, world >= 2) must precede tpe_sample_and_partial");
  int rc = sample_select_issue(ctx, uniforms, n_asks, false);
  if (rc) return rc;
  CU(cudaStreamSynchronize(ctx->stream));
  if (ctx->issued_dev_rng) ctx->mt_host_valid = true;
  *d_partials = ctx->kpart.as<double>();
  if (stride) *stride = ctx->ct_stride;
  return TPE_OK;
}

int tpe_finish_from_partials(tpe_ctx* ctx, const double* d_gathered, int32_t world, double* out_x, double* out_acq,
                             int64_t* out_best) {
  if (!ctx || !d_gathered || world < 1) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (!ctx->partial_ready) return fail(ctx, TPE_E_STATE, "tpe_sample_and_partial must precede tpe_finish_from_partials");
  if (set_device(ctx, /*join=*/false)) return TPE_E_CUDA;
  cudaStream_t st = ctx->stream;
  const int64_t n_asks = ctx->n_asks, Ct = n_asks * ctx->cfg.n_candidates;
  k_acq<<<grid_for(Ct * 32, 256, ctx->sm_count * 8), 256, 0, st>>>(
      ctx->est[0].part.as<double2>(), ctx->est[0].nsplit, reinterpret_cast<const double2*>(d_gathered), world,
      ctx->ct_stride, ctx->fast ? ctx->oob.as<uint8_t>() : nullptr, ctx->est[0].fix.as<double2>(),
      ctx->est[1].fix.as<double2>(), Ct, ctx->logl.as<double>(), ctx->logg.as<double>());
  k_select<<<(unsigned)n_asks, 256, 0, st>>>(ctx->logl.as<double>(), ctx->logg.as<double>(), ctx->cfg.n_candidates,
                                             ctx->S.as<double>(), ctx->pc, ctx->out_x.as<double>(),
                                             ctx->out_acq.as<double>(), ctx->out_best.as<int64_t>());
  ctx->launch_counter += 2;
  CU(cudaEventRecord(ctx->ev[8], st));
  CU(cudaGetLastError());
  if (out_x) CU(cudaMemcpyAsync(out_x, ctx->out_x.p, (size_t)n_asks * ctx->pc * 8, cudaMemcpyDeviceToHost, st));
  if (out_acq) CU(cudaMemcpyAsync(out_acq, ctx->out_acq.p, (size_t)n_asks * 8, cudaMemcpyDeviceToHost, st));
  if (out_best) CU(cudaMemcpyAsync(out_best, ctx->out_best.p, (size_t)n_asks * 8, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  for (int i = 0; i < 8; ++i) cudaEventElapsedTime(&ctx->ms[i], ctx->ev[i], ctx->ev[i + 1]);
  cudaEventElapsedTime(&ctx->ms[8], ctx->ev[0], ctx->ev[8]);
  ctx->launches = ctx->launch_counter;
  ctx->partial_ready = false;
  ctx->sampled = true;
  return TPE_OK;
}

int tpe_stage_uniforms_mt19937(tpe_ctx* ctx, const uint32_t* key, int32_t pos, int64_t skip, int64_t count) {
  // key == NULL: continue from the state the previous staged draw ended in (kept on the device)
  if (!ctx || (key && (pos < 0 || pos > 624)) || skip < 0 || count <= 0) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (set_device(ctx, /*join=*/false)) return TPE_E_CUDA;
  if (!key && !ctx->mt_state.p)
    return fail(ctx, TPE_E_STATE, "tpe_stage_uniforms_mt19937(key = NULL) needs a previous staged draw to continue");
  ctx->u_staged = nullptr;
  ctx->u_device_rng = false;
  const bool same_state = !key || (ctx->mt_host_valid && (uint32_t)pos == ctx->mt_host[624] &&
                                   memcmp(key, ctx->mt_host, 624 * 4) == 0);
  if (ctx->spec_pending && skip == 0 && count == ctx->spec_count && same_state) {
    // the caller's generator is where the previous ask left it: the speculative draw is this ask's
    std::swap(ctx->U, ctx->U2);
    std::swap(ctx->mt_state, ctx->mt_spec);
    std::swap(ctx->ev_u, ctx->ev_spec);
    ctx->spec_pending = false;
    ctx->mt_host_valid = false;
    ctx->u_staged_count = count;
    ctx->u_device_rng = true;
    return TPE_OK;
  }
  ctx->spec_pending = false;
  ctx->mt_host_valid = false;
  CU(cudaStreamSynchronize(ctx->stream3));
  CU(ctx->U.ensure((size_t)count * 8));
  CU(ctx->mt_state.ensure(625 * 4));
  if (key) {
    uint32_t h[625];
    memcpy(h, key, 624 * 4);
    h[624] = (uint32_t)pos;
    CU(cudaMemcpyAsync(ctx->mt_state.p, h, sizeof(h), cudaMemcpyHostToDevice, ctx->stream3));
  }
  if (int rc = launch_mt(ctx, ctx->stream3, ctx->mt_state.as<uint32_t>(), skip, count, ctx->U.as<double>())) return rc;
  CU(cudaEventRecord(ctx->ev_u, ctx->stream3));
  ctx->u_staged_count = count;
  ctx->u_device_rng = true;
  return TPE_OK;
}
int tpe_rng_state(tpe_ctx* ctx, uint32_t* key_out, int32_t* pos_out) {
  if (!ctx || !key_out || !pos_out) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (set_device(ctx, /*join=*/false)) return TPE_E_CUDA;
  if (!ctx->mt_state.p) return fail(ctx, TPE_E_STATE, "tpe_stage_uniforms_mt19937 must precede tpe_rng_state");
  if (!ctx->mt_host_valid) {  // not yet read back with the results of an ask
    CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_u, 0));
    CU(cudaMemcpyAsync(ctx->mt_host, ctx->mt_state.p, (size_t)625 * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->mt_host_valid = true;
  }
  memcpy(key_out, ctx->mt_host, 624 * 4);
  *pos_out = (int32_t)ctx->mt_host[624];
  return TPE_OK;
}
int tpe_result_device_ptrs(tpe_ctx* ctx, double** out_x, double** out_acq, int64_t** out_best) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (!ctx->sampled) return fail(ctx, TPE_E_STATE, "tpe_sample_and_select must precede tpe_result_device_ptrs");
  if (out_x) *out_x = ctx->out_x.as<double>();
  if (out_acq) *out_acq = ctx->out_acq.as<double>();
  if (out_best) *out_best = ctx->out_best.as<int64_t>();
  return TPE_OK;
}
int tpe_rng_state_device(tpe_ctx* ctx, uint32_t** state625) {
  if (!ctx || !state625) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (set_device(ctx, /*join=*/false)) return TPE_E_CUDA;
  if (!ctx->mt_state.p) return fail(ctx, TPE_E_STATE, "tpe_stage_uniforms_mt19937 must precede tpe_rng_state_device");
  CU(cudaStreamSynchronize(ctx->stream3));  // the generator that last wrote the state
  // the caller may overwrite the state (a broadcast from the rank that drew last): forget what the host knows
  ctx->mt_host_valid = false;
  ctx->spec_pending = false;
  *state625 = ctx->mt_state.as<uint32_t>();
  return TPE_OK;
}
int tpe_get_uniforms(tpe_ctx* ctx, double* out, int64_t count) {
  if (!ctx || !out || count <= 0) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (set_device(ctx, /*join=*/false)) return TPE_E_CUDA;
  if ((size_t)count * 8 > ctx->U.cap) return fail(ctx, TPE_E_INVALID, "only %zu uniforms are staged", ctx->U.cap / 8);
  CU(cudaStreamSynchronize(ctx->stream3));
  CU(cudaMemcpyAsync(out, ctx->U.p, (size_t)count * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return TPE_OK;
}

int tpe_host_alloc(tpe_ctx* ctx, size_t bytes, void** out) {
  if (!ctx || !out || bytes == 0) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (set_device(ctx, /*join=*/false)) return TPE_E_CUDA;
  *out = nullptr;
  CU(cudaHostAlloc(out, bytes, cudaHostAllocDefault));
  return TPE_OK;
}
int tpe_host_free(tpe_ctx* ctx, void* p) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (!p) return TPE_OK;
  if (set_device(ctx, /*join=*/false)) return TPE_E_CUDA;
  CU(cudaFreeHost(p));
  return TPE_OK;
}

int tpe_stage_uniforms(tpe_ctx* ctx, const double* uniforms, int64_t count) {
  if (!ctx || !uniforms || count <= 0) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (set_device(ctx, /*join=*/false)) return TPE_E_CUDA;
  ctx->u_staged = nullptr;
  CU(cudaStreamSynchronize(ctx->stream3));  // a previous, unconsumed staging
  CU(ctx->U.ensure((size_t)count * 8));
  CU(cudaMemcpyAsync(ctx->U.p, uniforms, (size_t)count * 8, cudaMemcpyHostToDevice, ctx->stream3));
  CU(cudaEventRecord(ctx->ev_u, ctx->stream3));
  ctx->u_staged = uniforms;
  ctx->u_staged_count = count;
  return TPE_OK;
}

int tpe_suggest(tpe_ctx* ctx, const tpe_cfg* cfg, const int32_t* cols, int32_t n_cols, const double* w_below,
                const double* w_above, const double* uniforms, int64_t n_asks, double* out_x, double* out_acq,
                int64_t* out_best) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  ctx->u_staged = nullptr;
  if (cfg && uniforms && n_asks > 0 && n_cols > 0 && cfg->n_candidates > 0) {
    // every selected column consumes C uniforms, plus C for the kernel choice: the count is known
    // before the split, so the upload overlaps it
    const int64_t count = n_asks * (int64_t)cfg->n_candidates * (1 + n_cols);
    if (set_device(ctx)) return TPE_E_CUDA;
    CU(ctx->U.ensure((size_t)count * 8));
    CU(cudaMemcpyAsync(ctx->U.p, uniforms, (size_t)count * 8, cudaMemcpyHostToDevice, ctx->stream3));
    CU(cudaEventRecord(ctx->ev_u, ctx->stream3));
    ctx->u_staged = uniforms;
    ctx->u_staged_count = count;
  }
  int rc = prepare_locked(ctx, cfg, cols, n_cols, nullptr);
  if (!rc) rc = build_locked(ctx, w_below, w_above);
  if (!rc) rc = sample_select_locked(ctx, uniforms, n_asks, out_x, out_acq, out_best);
  if (ctx->u_staged) {  // an early error left the upload in flight: the caller's buffer must be free on return
    cudaStreamSynchronize(ctx->stream3);
    ctx->u_staged = nullptr;
  }
  return rc;
}

// ---- the P sample_independent calls of one univariate trial, in one go -------------------------------------------

static tpe_ctx* make_sub(tpe_ctx* parent) {
  tpe_ctx* c = new tpe_ctx();
  c->device = parent->device;
  c->is_sub = true;
  c->sm_count = parent->sm_count;
  c->sort_cta_cap = std::max(8, parent->sm_count / 8);   // ~8 column sorts share the GPU at a time
  if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&c->stream3, cudaStreamNonBlocking) != cudaSuccess) {
    delete c;
    return nullptr;
  }
  for (auto& e : c->ev) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&c->ev_u, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&c->ev_spec, cudaEventDisableTiming);
  return c;
}

static int uni_batch_locked(tpe_ctx* ctx, const tpe_cfg* cfg, const int32_t* cols, int32_t n_cols,
                            const double* w_below, const double* w_above, const double* uniforms, double* out_x,
                            double* out_acq, int64_t* out_best, bool defer) {
  if (!cfg || !cols || n_cols <= 0 || (!out_x && !defer)) return fail(ctx, TPE_E_INVALID, "bad arguments");
  ctx->deferred_uni = 0;
  if (cfg->multivariate) return fail(ctx, TPE_E_INVALID, "tpe_suggest_univariate_batch is for multivariate = 0");
  if (ctx->M >= 2) return fail(ctx, TPE_E_STATE, "not batchable: multi-objective history (use the per-parameter calls)");
  if (set_device(ctx)) return TPE_E_CUDA;
  const int32_t C = cfg->n_candidates;
  const int64_t per_col = 2ll * C, count = per_col * n_cols;
  // uniforms: uploaded on the side stream now, or already generated there by tpe_stage_uniforms_mt19937
  const bool dev_rng = uniforms == nullptr;
  if (dev_rng) {
    if (!ctx->u_device_rng || ctx->u_staged_count != count)
      return fail(ctx, TPE_E_INVALID, "device-generated uniforms: %lld staged, %lld needed", (long long)ctx->u_staged_count,
                  (long long)count);
  } else {
    if (ctx->u_device_rng) CU(cudaStreamSynchronize(ctx->stream3));
    CU(ctx->U.ensure((size_t)count * 8));
    CU(cudaMemcpyAsync(ctx->U.p, uniforms, (size_t)count * 8, cudaMemcpyHostToDevice, ctx->stream3));
    CU(cudaEventRecord(ctx->ev_u, ctx->stream3));
  }
  ctx->u_device_rng = false;
  ctx->u_staged = nullptr;
  // one split for every column (sampler.py:686-722 does not look at the parameters)
  int rc = prepare_locked(ctx, cfg, cols, n_cols, nullptr);
  if (rc) return rc;
  for (const ColMeta& cm : ctx->cols_h)
    if (ctx->col_missing[cm.src])
      return fail(ctx, TPE_E_STATE, "not batchable: a selected parameter is absent from some trials (their estimators use "
                  "different trials; use the per-parameter calls)");
  for (int which = 0; which < 2; ++which) {   // _call_weights_func checks (parzen_estimator.py:88-109), once
    const double* w = which == 0 ? w_below : w_above;
    const int64_t n = ctx->est[which].n;
    if (!w) continue;
    double tot = 0;
    for (int64_t i = 0; i < n; ++i) {
      if (w[i] < 0) return fail(ctx, TPE_E_INVALID, "The `weights` function is not allowed to return negative values.");
      if (!isfinite(w[i])) return fail(ctx, TPE_E_INVALID, "The `weights`function is not allowed to return infinite or NaN values.");
      tot += w[i];
    }
    if (n > 0 && tot <= 0) return fail(ctx, TPE_E_INVALID, "The `weight` function is not allowed to return all-zero values.");
  }
  {
    // how the above set differs from the previous call's (the column contexts then update their sorted orders
    // instead of sorting: k_order_update); the answer stays on the device
    const int64_t n_new = ctx->est[1].n;
    int cand = 2;
    if (ctx->uni_prev_n >= 0 && ctx->uni_prev_lineage == ctx->hist_lineage)
      cand = n_new == ctx->uni_prev_n ? 0 : n_new == ctx->uni_prev_n + 1 ? 1 : 2;
    CU(ctx->uni_mode.ensure(16));
    CU(cudaMemsetAsync(ctx->uni_mode.p, 0, 4, ctx->stream));
    k_rows_delta<<<cand == 2 ? 1 : grid_for(std::max<int64_t>(ctx->uni_prev_n, 1), 256, ctx->sm_count), 256, 0, ctx->stream>>>(
        ctx->est[1].rows.as<int64_t>(), ctx->uni_prev_rows.as<int64_t>(), cand == 2 ? 0 : ctx->uni_prev_n, cand,
        ctx->uni_mode.as<int>());
    ctx->launch_counter++;
    CU(ctx->uni_prev_rows.ensure((size_t)(n_new + 1) * 8));
    CU(cudaMemcpyAsync(ctx->uni_prev_rows.p, ctx->est[1].rows.p, (size_t)n_new * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    ctx->uni_prev_n = n_new;
    ctx->uni_prev_lineage = ctx->hist_lineage;
    ctx->uni_seq++;
  }
  if (!ctx->ev_uni) CU(cudaEventCreateWithFlags(&ctx->ev_uni, cudaEventDisableTiming));
  CU(cudaEventRecord(ctx->ev_uni, ctx->stream));
  CU(ctx->out_x.ensure((size_t)n_cols * 8));
  CU(ctx->out_acq.ensure((size_t)n_cols * 8));
  CU(ctx->out_best.ensure((size_t)n_cols * 8));
  // all columns continuous: stage by stage over all of them (one launch per stage)
  static const bool staged_on = [] { const char* v = getenv("TPE_UNI_STAGED"); return !(v && v[0] == '0'); }();
  bool staged = staged_on && C <= 4096 && n_cols >= 2;
  for (const ColMeta& cm : ctx->cols_h) staged = staged && cm.cls == COL_CONT;
  if (staged) {
    ctx->launch_counter = 0;
    rc = uni_batch_staged(ctx, cfg, cols, n_cols, w_below, w_above);
    if (rc) return rc;
    if (dev_rng) CU(cudaMemcpyAsync(ctx->mt_host, ctx->mt_state.p, (size_t)625 * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaEventRecord(ctx->ev[8], ctx->stream));
    if (defer) {   // results into the page-locked staging area; tpe_collect_univariate waits and hands them out
      const size_t need = (size_t)n_cols * 3 * 8;
      if (ctx->res_host_cap < need) {
        if (ctx->res_host) cudaFreeHost(ctx->res_host);
        ctx->res_host = nullptr;
        ctx->res_host_cap = 0;
        CU(cudaHostAlloc(&ctx->res_host, need + 4096, cudaHostAllocDefault));
        ctx->res_host_cap = need + 4096;
      }
      char* h = static_cast<char*>(ctx->res_host);
      CU(cudaMemcpyAsync(h, ctx->out_x.p, (size_t)n_cols * 8, cudaMemcpyDeviceToHost, ctx->stream));
      CU(cudaMemcpyAsync(h + (size_t)n_cols * 8, ctx->out_acq.p, (size_t)n_cols * 8, cudaMemcpyDeviceToHost, ctx->stream));
      CU(cudaMemcpyAsync(h + (size_t)n_cols * 16, ctx->out_best.p, (size_t)n_cols * 8, cudaMemcpyDeviceToHost, ctx->stream));
      ctx->deferred_uni = n_cols;
      ctx->deferred_uni_rng = dev_rng;
      ctx->spec_pending = false;
      ctx->launches = ctx->launch_counter;
      ctx->prepared = ctx->built = ctx->sampled = false;
      return TPE_OK;
    }
    CU(cudaMemcpyAsync(out_x, ctx->out_x.p, (size_t)n_cols * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (out_acq) CU(cudaMemcpyAsync(out_acq, ctx->out_acq.p, (size_t)n_cols * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (out_best) CU(cudaMemcpyAsync(out_best, ctx->out_best.p, (size_t)n_cols * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    if (dev_rng) ctx->mt_host_valid = true;
    ctx->spec_pending = false;
    for (int i = 0; i < 9; ++i) ctx->ms[i] = 0.0f;
    cudaEventElapsedTime(&ctx->ms[8], ctx->ev[0], ctx->ev[8]);
    ctx->launches = ctx->launch_counter;
    ctx->prepared = ctx->built = ctx->sampled = false;
    return TPE_OK;
  }
  if (defer)
    return fail(ctx, TPE_E_STATE, "not batchable asynchronously: only trials whose parameters are all continuous are "
                "evaluated stage by stage");
  while ((int)ctx->uni_sub.size() < n_cols) {
    tpe_ctx* c = make_sub(ctx);
    if (!c) return fail(ctx, TPE_E_CUDA, "could not create the streams of a column context");
    ctx->uni_sub.push_back(c);
  }
  int launches = ctx->launch_counter;
  // Issuing ~20 launches per column is host work (~10 us each through 32 streams): the columns are independent,
  // so a few host threads issue them side by side.  Each column context is touched by exactly one thread.
  auto issue_column = [&](int j) -> int {
    tpe_ctx* sub = ctx->uni_sub[j];
    int rc = TPE_OK;
    sub->err.clear();
#define CUS(call)                                                                                            \
    do {                                                                                                       \
      cudaError_t e_ = (call);                                                                                 \
      if (e_ != cudaSuccess)                                                                                   \
        return fail(sub, e_ == cudaErrorMemoryAllocation ? TPE_E_NOMEM : TPE_E_CUDA, "%s failed: %s (%s:%d)", \
                    #call, cudaGetErrorString(e_), __FILE__, __LINE__);                                        \
    } while (0)
    CUS(cudaSetDevice(ctx->device));
    sub->space = ctx->space;
    sub->cat_dist_off = ctx->cat_dist_off;
    sub->cat_dist.alias(ctx->cat_dist.p, ctx->cat_dist.cap);
    sub->col_missing = ctx->col_missing;
    sub->col_oor = ctx->col_oor;
    sub->col_offgrid = ctx->col_offgrid;
    sub->X.alias(ctx->X.p, ctx->X.cap);
    sub->cat.alias(ctx->cat.p, ctx->cat.cap);
    sub->key.alias(ctx->key.p, ctx->key.cap);
    sub->N = ctx->N;
    sub->hist_lineage = ctx->hist_lineage;
    sub->uni_seq = ctx->uni_seq;
    sub->uni_mode_ptr = ctx->uni_mode.as<int>();
    sub->M = 1;
    sub->history_set = true;
    sub->cfg = *cfg;
    sub->launch_counter = 0;
    bool rowok_unused = false;
    rc = setup_columns(sub, cfg, cols + j, 1, &rowok_unused);
    if (rc) return rc;
    for (int which = 0; which < 2; ++which) {
      sub->est[which].rows.alias(ctx->est[which].rows.p, ctx->est[which].rows.cap);
      sub->est[which].n = ctx->est[which].n;
    }
    sub->est[0].pos.alias(ctx->est[0].pos.p, ctx->est[0].pos.cap);
    sub->info = ctx->info;
    sub->prepared = true;
    CUS(cudaStreamWaitEvent(sub->stream, ctx->ev_uni, 0));
    for (int which = 0; which < 2; ++which) {
      rc = build_estimator(sub, which, which == 0 ? w_below : w_above, sub->stream);
      if (rc) return rc;
    }
    sub->built = true;
    sub->U.alias(ctx->U.as<double>() + (size_t)j * per_col, (size_t)per_col * 8);
    CUS(cudaStreamWaitEvent(sub->stream, ctx->ev_u, 0));
    sub->n_asks = 1;
    rc = ensure_candidate_buffers(sub, C);
    if (rc) return rc;
    CUS(sub->out_x.ensure(8));
    CUS(sub->out_acq.ensure(8));
    CUS(sub->out_best.ensure(8));
    rc = launch_sample_select(sub, 1, false, false);
    if (rc) return rc;
    CUS(cudaMemcpyAsync(ctx->out_x.as<double>() + j, sub->out_x.p, 8, cudaMemcpyDeviceToDevice, sub->stream));
    CUS(cudaMemcpyAsync(ctx->out_acq.as<double>() + j, sub->out_acq.p, 8, cudaMemcpyDeviceToDevice, sub->stream));
    CUS(cudaMemcpyAsync(ctx->out_best.as<int64_t>() + j, sub->out_best.p, 8, cudaMemcpyDeviceToDevice, sub->stream));
    CUS(cudaEventRecord(sub->ev_join, sub->stream));
#undef CUS
    return TPE_OK;
  };
  static const int n_threads_env = [] { const char* v = getenv("TPE_UNI_THREADS"); return v ? atoi(v) : 6; }();
  const int T = std::max(1, std::min(n_threads_env, (int)n_cols));
  std::vector<int> rcs((size_t)n_cols, TPE_OK);
  if (T == 1) {
    for (int j = 0; j < n_cols; ++j) rcs[(size_t)j] = issue_column(j);
  } else {
    std::vector<std::thread> pool;
    for (int w = 0; w < T; ++w)
      pool.emplace_back([&, w] { for (int j = w; j < n_cols; j += T) rcs[(size_t)j] = issue_column(j); });
    for (auto& th : pool) th.join();
  }
  for (int j = 0; j < n_cols; ++j) {
    if (rcs[(size_t)j]) {
      ctx->err = ctx->uni_sub[(size_t)j]->err;
      for (int q = 0; q < n_cols; ++q) cudaStreamSynchronize(ctx->uni_sub[(size_t)q]->stream);
      return rcs[(size_t)j];
    }
    CU(cudaStreamWaitEvent(ctx->stream, ctx->uni_sub[(size_t)j]->ev_join, 0));
    launches += ctx->uni_sub[(size_t)j]->launch_counter;
  }
  if (dev_rng) CU(cudaMemcpyAsync(ctx->mt_host, ctx->mt_state.p, (size_t)625 * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaEventRecord(ctx->ev[8], ctx->stream));
  CU(cudaMemcpyAsync(out_x, ctx->out_x.p, (size_t)n_cols * 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (out_acq) CU(cudaMemcpyAsync(out_acq, ctx->out_acq.p, (size_t)n_cols * 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (out_best) CU(cudaMemcpyAsync(out_best, ctx->out_best.p, (size_t)n_cols * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  if (dev_rng) ctx->mt_host_valid = true;
  ctx->spec_pending = false;
  for (int i = 0; i < 9; ++i) ctx->ms[i] = 0.0f;
  cudaEventElapsedTime(&ctx->ms[8], ctx->ev[0], ctx->ev[8]);
  ctx->launches = launches;
  ctx->last_kernel = ctx->uni_sub[0]->last_kernel;
  ctx->prepared = ctx->built = ctx->sampled = false;   // the per-column state lives in the column contexts
  return TPE_OK;
}

int tpe_suggest_univariate_batch(tpe_ctx* ctx, const tpe_cfg* cfg, const int32_t* cols, int32_t n_cols,
                                 const double* w_below, const double* w_above, const double* uniforms, double* out_x,
                                 double* out_acq, int64_t* out_best) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  return uni_batch_locked(ctx, cfg, cols, n_cols, w_below, w_above, uniforms, out_x, out_acq, out_best, false);
}

int tpe_suggest_univariate_batch_async(tpe_ctx* ctx, const tpe_cfg* cfg, const int32_t* cols, int32_t n_cols,
                                       const double* w_below, const double* w_above, const double* uniforms) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  return uni_batch_locked(ctx, cfg, cols, n_cols, w_below, w_above, uniforms, nullptr, nullptr, nullptr, true);
}

int tpe_collect_univariate(tpe_ctx* ctx, double* out_x, double* out_acq, int64_t* out_best) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (ctx->deferred_uni <= 0)
    return fail(ctx, TPE_E_STATE, "tpe_collect_univariate needs a pending tpe_suggest_univariate_batch_async");
  if (set_device(ctx, /*join=*/false)) return TPE_E_CUDA;
  const int64_t n = ctx->deferred_uni;
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->deferred_uni = 0;
  if (ctx->deferred_uni_rng) ctx->mt_host_valid = true;
  for (int i = 0; i < 9; ++i) ctx->ms[i] = 0.0f;
  cudaEventElapsedTime(&ctx->ms[8], ctx->ev[0], ctx->ev[8]);
  const char* h = static_cast<const char*>(ctx->res_host);
  if (out_x) memcpy(out_x, h, (size_t)n * 8);
  if (out_acq) memcpy(out_acq, h + (size_t)n * 8, (size_t)n * 8);
  if (out_best) memcpy(out_best, h + (size_t)n * 16, (size_t)n * 8);
  return TPE_OK;
}

int tpe_get_split_info(tpe_ctx* ctx, tpe_split_info* info) {
  if (!ctx || !info) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (!ctx->prepared) return fail(ctx, TPE_E_STATE, "tpe_prepare must precede tpe_get_split_info");
  *info = ctx->info;
  return TPE_OK;
}

int tpe_get_split(tpe_ctx* ctx, int64_t* below_rows, int64_t* above_rows) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (!ctx->prepared) return fail(ctx, TPE_E_STATE, "tpe_prepare must precede tpe_get_split");
  if (set_device(ctx)) return TPE_E_CUDA;
  if (below_rows && ctx->est[0].n)
    CU(cudaMemcpyAsync(below_rows, ctx->est[0].rows.p, (size_t)ctx->est[0].n * 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (above_rows && ctx->est[1].n)
    CU(cudaMemcpyAsync(above_rows, ctx->est[1].rows.p, (size_t)ctx->est[1].n * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return TPE_OK;
}

int tpe_get_mixture(tpe_ctx* ctx, int which, double* weights, double* mu, double* sigma) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (!ctx->built) return fail(ctx, TPE_E_STATE, "tpe_build must precede tpe_get_mixture");
  if (which < 0 || which > 1) return fail(ctx, TPE_E_INVALID, "which must be 0 or 1");
  if (set_device(ctx)) return TPE_E_CUDA;
  Estimator& e = ctx->est[which];
  if (weights) CU(cudaMemcpyAsync(weights, e.w.p, (size_t)e.K * 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (mu) CU(cudaMemcpyAsync(mu, e.mu.p, (size_t)e.K * ctx->pc * 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (sigma) CU(cudaMemcpyAsync(sigma, e.sigma.p, (size_t)e.K * ctx->pc * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return TPE_OK;
}

int tpe_get_candidates(tpe_ctx* ctx, double* samples, double* logl, double* logg) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (!ctx->sampled) return fail(ctx, TPE_E_STATE, "tpe_sample_and_select must precede tpe_get_candidates");
  if (set_device(ctx)) return TPE_E_CUDA;
  if (samples) CU(cudaMemcpyAsync(samples, ctx->S.p, (size_t)ctx->Ct * ctx->pc * 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (logl) CU(cudaMemcpyAsync(logl, ctx->logl.p, (size_t)ctx->Ct * 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (logg) CU(cudaMemcpyAsync(logg, ctx->logg.p, (size_t)ctx->Ct * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return TPE_OK;
}

int tpe_logpdf(tpe_ctx* ctx, int which, const double* x, int64_t n, double* out) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (!ctx->built) return fail(ctx, TPE_E_STATE, "tpe_build must precede tpe_logpdf");
  if (which < 0 || which > 1 || !x || !out || n <= 0) return fail(ctx, TPE_E_INVALID, "bad logpdf arguments");
  if (set_device(ctx)) return TPE_E_CUDA;
  cudaStream_t st = ctx->stream;
  int rc = ensure_candidate_buffers(ctx, n);
  if (rc) return rc;
  ctx->sampled = false;
  ctx->user_points = true;
  CU(cudaMemcpyAsync(ctx->S.p, x, (size_t)n * ctx->pc * 8, cudaMemcpyHostToDevice, st));
  k_prep_points<<<grid_for(n * ctx->pc, 256, ctx->sm_count * 8), 256, 0, st>>>(
      ctx->S.as<double>(), n, ctx->cols.as<ColMeta>(), ctx->pc, ctx->fast ? ctx->xT.as<double>() : nullptr,
      ctx->ct_stride, ctx->oob.as<uint8_t>());
  ctx->launch_counter++;
  rc = run_logpdf(ctx, which, n);
  if (rc) return rc;
  Estimator& e = ctx->est[which];
  k_finish_logpdf<<<grid_for(n, 256, ctx->sm_count * 8), 256, 0, st>>>(
      e.part.as<double2>(), e.nsplit, ctx->ct_stride, ctx->fast ? ctx->oob.as<uint8_t>() : nullptr,
      e.fix.as<double2>(), n, ctx->logl.as<double>());
  ctx->launch_counter++;
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(out, ctx->logl.p, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return TPE_OK;
}

int tpe_last_timing(tpe_ctx* ctx, float* ms9, int32_t* launches) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (ms9)
    for (int i = 0; i < 9; ++i) ms9[i] = ctx->ms[i];
  if (launches) *launches = ctx->launches;
  return TPE_OK;
}

int tpe_probe_fp64_tflops(tpe_ctx* ctx, double* tflops) {
  if (!ctx || !tflops) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (set_device(ctx)) return TPE_E_CUDA;
  const int blocks = ctx->sm_count * 4, threads = 512, iters = 20000;
  DevBuf out;
  CU(out.ensure((size_t)blocks * threads * 8));
  float best = 1e30f;
  for (int rep = 0; rep < 4; ++rep) {
    CU(cudaEventRecord(ctx->ev[0], ctx->stream));
    k_fp64_probe<<<blocks, threads, 0, ctx->stream>>>(out.as<double>(), iters);
    CU(cudaEventRecord(ctx->ev[1], ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
    if (rep > 0 && ms < best) best = ms;
  }
  out.release();
  const double flops = 2.0 * 8.0 * (double)iters * blocks * threads;
  *tflops = flops / (best * 1e-3) / 1e12;
  return TPE_OK;
}

const char* tpe_last_logpdf_kernel(tpe_ctx* ctx) { return ctx ? ctx->last_kernel : "none"; }

int tpe_ped_anova(tpe_ctx* ctx, const tpe_ped_cfg* cfg, const int32_t* cols, int32_t n_cols, const double* grids,
                  const int32_t* n_grid, const double* loss, double* out_importance, int64_t* out_n,
                  int32_t* out_counts) {
  if (!ctx) return TPE_E_INVALID;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (!ctx->history_set) return fail(ctx, TPE_E_STATE, "tpe_history_set must precede tpe_ped_anova");
  if (!cfg || !cols || n_cols <= 0 || !n_grid || !out_importance || !out_n)
    return fail(ctx, TPE_E_INVALID, "bad tpe_ped_anova arguments");
  if (!(0.0 < cfg->target_quantile && cfg->target_quantile < cfg->region_quantile && cfg->region_quantile <= 1.0))
    return fail(ctx, TPE_E_INVALID, "condition 0.0 < `target_quantile` < `region_quantile` <= 1.0 must be satisfied");
  if (!(cfg->prior_weight > 0.0)) return fail(ctx, TPE_E_INVALID, "prior_weight must be positive");
  if (cfg->min_n_top < 1) return fail(ctx, TPE_E_INVALID, "min_n_top must be positive");
  if (cfg->n_steps < 1 || cfg->n_steps > kPedMaxSteps)
    return fail(ctx, TPE_E_INVALID, "n_steps must be in [1, %d]", kPedMaxSteps);
  const int P = (int)ctx->space.size();
  std::vector<PedCol> meta((size_t)n_cols);
  int width = 1;
  bool numeric = false;
  for (int j = 0; j < n_cols; ++j) {
    const int src = cols[j];
    if (src < 0 || src >= P) return fail(ctx, TPE_E_INVALID, "column %d out of range", src);
    const tpe_param_desc& d = ctx->space[src];
    const bool is_cat = d.kind == TPE_KIND_CAT;
    if (is_cat ? n_grid[j] != d.n_choices : (n_grid[j] < 1 || n_grid[j] > cfg->n_steps))
      return fail(ctx, TPE_E_INVALID, "column %d: %d bins (n_choices of a categorical column, 1..n_steps otherwise)",
                  src, n_grid[j]);
    meta[j] = PedCol{src, is_cat ? 1 : 0, d.log ? 1 : 0, n_grid[j]};
    width = std::max(width, (int)n_grid[j]);
    numeric = numeric || !is_cat;
  }
  if (numeric && !grids) return fail(ctx, TPE_E_INVALID, "numerical columns need their grids");
  if (set_device(ctx)) return TPE_E_CUDA;
  const int64_t N = ctx->N;
  const int64_t nal = std::max<int64_t>(N, 1);
  const size_t ncnt = (size_t)n_cols * 2 * width;
  CU(ctx->ped_member.ensure((size_t)nal));
  CU(ctx->ped_okey.ensure((size_t)nal * 8));
  CU(ctx->ped_work.ensure(sizeof(PedWork)));
  CU(ctx->ped_cols.ensure(sizeof(PedCol) * n_cols));
  CU(ctx->ped_grid.ensure((size_t)n_cols * cfg->n_steps * 8));
  CU(ctx->ped_counts.ensure(ncnt * 4));
  CU(ctx->ped_pdf.ensure(ncnt * 8));
  CU(ctx->ped_imp.ensure((size_t)n_cols * 8));
  cudaStream_t st = ctx->stream;
  CU(cudaMemsetAsync(ctx->ped_work.p, 0, sizeof(PedWork), st));
  CU(cudaMemsetAsync(ctx->ped_counts.p, 0, ncnt * 4, st));
  CU(cudaMemcpyAsync(ctx->ped_cols.p, meta.data(), sizeof(PedCol) * n_cols, cudaMemcpyHostToDevice, st));
  if (numeric)
    CU(cudaMemcpyAsync(ctx->ped_grid.p, grids, (size_t)n_cols * cfg->n_steps * 8, cudaMemcpyHostToDevice, st));
  const double* d_loss = nullptr;
  if (loss) {
    CU(ctx->ped_loss.ensure((size_t)nal * 8));
    if (N) CU(cudaMemcpyAsync(ctx->ped_loss.p, loss, (size_t)N * 8, cudaMemcpyHostToDevice, st));
    d_loss = ctx->ped_loss.as<double>();
  }
  int n_i = (int)N, pall = P, nc = n_cols, mnt = cfg->min_n_top;
  double qt = cfg->target_quantile, qr = cfg->region_quantile;
  const double* d_X = ctx->X.as<double>();
  const int8_t* d_cat = ctx->cat.as<int8_t>();
  const double* d_key = ctx->key.as<double>();
  const PedCol* d_cols = ctx->ped_cols.as<PedCol>();
  uint8_t* d_member = ctx->ped_member.as<uint8_t>();
  uint64_t* d_okey = ctx->ped_okey.as<uint64_t>();
  PedWork* d_wk = ctx->ped_work.as<PedWork>();
  void* args[] = {&n_i, &pall, &d_X, &d_cat, &d_key, &d_loss, &d_cols, &nc, &qt, &qr, &mnt, &d_member, &d_okey, &d_wk};
  const int G = (int)std::max<int64_t>(1, std::min<int64_t>(ctx->sm_count, (N + 1023) / 1024));
  CU(cudaLaunchCooperativeKernel((const void*)k_ped_select_coop, dim3(G), dim3(kPedThreads), args, 0, st));
  // histograms: shared memory unless a categorical column is too wide for it (global integer atomics then)
  const bool use_smem = (size_t)2 * width * 4 <= 32768;
  const size_t smem = (size_t)cfg->n_steps * 8 + (use_smem ? (size_t)2 * width * 4 : 0);
  const int bx = (int)std::max<int64_t>(1, std::min<int64_t>((N + 4095) / 4096,
                                                                  std::max(1, ctx->sm_count * 8 / n_cols)));
  if (N > 0)
    k_ped_bin<<<dim3(bx, n_cols), 256, smem, st>>>(n_i, pall, d_X, d_member, d_cols, ctx->ped_grid.as<double>(),
                                                   cfg->n_steps, width, use_smem ? 1 : 0, ctx->ped_counts.as<int>());
  k_ped_estimate<<<dim3(n_cols, cfg->evaluate_on_local ? 2 : 1), 128, 0, st>>>(
      d_cols, ctx->ped_counts.as<int>(), width, d_wk, mnt, cfg->prior_weight, ctx->ped_pdf.as<double>());
  k_ped_divergence<<<(n_cols + 127) / 128, 128, 0, st>>>(d_cols, n_cols, width, d_wk, mnt, cfg->evaluate_on_local ? 1 : 0,
                                                         ctx->ped_pdf.as<double>(), ctx->ped_imp.as<double>());
  CU(cudaGetLastError());
  unsigned long long n3[3];
  CU(cudaMemcpyAsync(n3, ctx->ped_work.p, sizeof(n3), cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(out_importance, ctx->ped_imp.p, (size_t)n_cols * 8, cudaMemcpyDeviceToHost, st));
  if (out_counts) CU(cudaMemcpyAsync(out_counts, ctx->ped_counts.p, ncnt * 4, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  const bool none = (int64_t)n3[0] <= cfg->min_n_top;
  out_n[0] = (int64_t)n3[0];
  out_n[1] = none ? 0 : (int64_t)n3[1];
  out_n[2] = none ? 0 : (int64_t)n3[2];
  return TPE_OK;
}

}  // extern "C"
