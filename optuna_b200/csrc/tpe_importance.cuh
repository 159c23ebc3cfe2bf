// PED-ANOVA hyperparameter importance on the resident history (sm_100a).  Host orchestration: tpe_ped_anova in
// tpe_capi.cu.
//
// Stage map (reference file:line each kernel replaces; optuna/importance/...):
//   k_ped_select_coop  _base.py:145-156 (_get_filtered_trials), _ped_anova/evaluator.py:37-55 (_QuantileFilter)
//   k_ped_bin          _ped_anova/scott_parzen_estimator.py:90-135 (grid indices and counts)
//   k_ped_estimate     _ped_anova/scott_parzen_estimator.py:16-87 (_ScottParzenEstimator), on top of
//                      samplers/_tpe/parzen_estimator.py:39-78, :132-166 and probability_distributions.py:154-223
//   k_ped_divergence   _ped_anova/evaluator.py:196-220, :258-263 (Pearson divergence, (n_target/n_region)^2)
#pragma once
#include <cooperative_groups.h>

#include "tpe_common.cuh"
#include "tpe_math.cuh"

namespace tpe {

constexpr int kPedMaxSteps = 128;   // bound on tpe_ped_cfg.n_steps (the reference uses 50)
constexpr int kPedThreads = 512;    // k_ped_select_coop block size

// One selected column.  n_grid: bins (numerical: <= n_steps points of the host's np.linspace; categorical: choices).
struct PedCol {
  int32_t src, is_cat, log, n_grid;
};

struct PedWork {                       // zeroed by the host before each call
  unsigned long long n_keep;           // rows that pass the filter
  unsigned long long n_member[2];      // target, region
  int hist[2][8][256];                 // per quantile, one histogram per radix pass (MSB first)
};

// member[r] bits: 1 kept, 2 in the target set, 4 in the region set
enum { kPedKept = 1, kPedTarget = 2, kPedRegion = 4 };

__device__ __forceinline__ unsigned long long ped_block_sum(unsigned long long v, unsigned long long* s_red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
  __syncthreads();
  unsigned long long t = 0;
  if (threadIdx.x == 0)
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += s_red[w];
  return t;  // valid in thread 0
}

// Row filter, the order statistics of both quantiles and set membership (cooperative launch, blockDim 512).
// The cut-off of quantile q is the k-th smallest kept loss, k = max(min_n_top - 1, ceil(q n) - 1): what the two
// np.partition calls of _QuantileFilter.filter select.  It is found by an MSB-first radix select over the
// order-preserving integer image of the loss (the byte-wise histogram passes of k_split_coop on a 64-bit key):
// eight passes, each histogramming the next byte of the rows that still match the chosen prefix; no sort.
// Membership is key <= cut-off key, i.e. loss <= cut-off in fp64 with -0.0 == 0.0 (order_bits folds them).
__global__ void __launch_bounds__(kPedThreads, 1)
k_ped_select_coop(int n, int32_t pall, const double* __restrict__ X, const int8_t* __restrict__ cat,
                  const double* __restrict__ key, const double* __restrict__ loss, const PedCol* __restrict__ cols,
                  int n_cols, double q_target, double q_region, int min_n_top, uint8_t* __restrict__ member,
                  uint64_t* __restrict__ okey, PedWork* __restrict__ wk) {
  cooperative_groups::grid_group grid = cooperative_groups::this_grid();
  __shared__ int s_hist[2][256];
  __shared__ unsigned long long s_red[32];
  __shared__ uint64_t s_prefix[2];
  __shared__ long long s_need[2];
  const int tid = threadIdx.x;
  const int G = gridDim.x, b = blockIdx.x;
  const int chunk = (n + G - 1) / G;
  const int lo_i = min(n, b * chunk), hi_i = min(n, lo_i + chunk);

  // ---- filter ---------------------------------------------------------------------------------------
  unsigned long long mine = 0;
  for (int i = lo_i + tid; i < hi_i; i += blockDim.x) {
    const double lv = loss != nullptr ? loss[i] : key[2 * (int64_t)i];
    bool ok = cat[i] == TPE_CAT_COMPLETE && isfinite(lv);
    for (int j = 0; j < n_cols && ok; ++j) {
      const double v = X[(int64_t)i * pall + cols[j].src];
      ok = v == v;
    }
    member[i] = ok ? kPedKept : 0;
    okey[i] = ok ? order_bits(lv) : ~0ull;
    mine += ok;
  }
  const unsigned long long kept_here = ped_block_sum(mine, s_red);
  if (tid == 0 && kept_here) atomicAdd(&wk->n_keep, kept_here);
  grid.sync();
  const long long nk = (long long)wk->n_keep;
  if (nk <= min_n_top) return;  // the reference returns zeros (evaluator.py:244-245); uniform over the grid

  // ---- radix select -----------------------------------------------------------------------------------
  const int nq = q_region < 1.0 ? 2 : 1;
  if (tid < 2) {
    const double q = tid == 0 ? q_target : q_region;
    const long long kq = (long long)ceil(q * (double)nk) - 1;
    s_need[tid] = kq > min_n_top - 1 ? kq : (long long)(min_n_top - 1);
    s_prefix[tid] = 0;
  }
  __syncthreads();
  for (int d = 7; d >= 0; --d) {
    for (int t = tid; t < 512; t += blockDim.x) (&s_hist[0][0])[t] = 0;
    __syncthreads();
    const uint64_t p0 = s_prefix[0], p1 = s_prefix[1];
    const int sh = 8 * (d + 1);
    for (int i = lo_i + tid; i < hi_i; i += blockDim.x) {
      if (!member[i]) continue;
      const uint64_t kb = okey[i];
      const int dg = (int)((kb >> (8 * d)) & 0xffull);
      if (sh == 64 || (kb >> sh) == (p0 >> sh)) atomicAdd(&s_hist[0][dg], 1);
      if (nq == 2 && (sh == 64 || (kb >> sh) == (p1 >> sh))) atomicAdd(&s_hist[1][dg], 1);
    }
    __syncthreads();
    for (int t = tid; t < 256 * nq; t += blockDim.x) {
      const int h = s_hist[t >> 8][t & 255];
      if (h) atomicAdd(&wk->hist[t >> 8][d][t & 255], h);
    }
    grid.sync();
    if (tid < nq) {
      const int* h = wk->hist[tid][d];
      long long cum = 0, need = s_need[tid];
      int q = 0;
      for (; q < 255; ++q) {
        if (cum + h[q] > need) break;
        cum += h[q];
      }
      s_need[tid] = need - cum;
      s_prefix[tid] |= (uint64_t)q << (8 * d);
    }
    __syncthreads();
  }

  // ---- membership -------------------------------------------------------------------------------------
  const uint64_t cut_t = s_prefix[0], cut_r = s_prefix[1];
  unsigned long long nt = 0, nr = 0;
  for (int i = lo_i + tid; i < hi_i; i += blockDim.x) {
    if (!member[i]) continue;
    const uint64_t kb = okey[i];
    const bool t = kb <= cut_t, r = nq == 1 || kb <= cut_r;
    member[i] = (uint8_t)(kPedKept | (t ? kPedTarget : 0) | (r ? kPedRegion : 0));
    nt += t;
    nr += r;
  }
  const unsigned long long st = ped_block_sum(nt, s_red);
  if (tid == 0 && st) atomicAdd(&wk->n_member[0], st);
  const unsigned long long sr = ped_block_sum(nr, s_red);
  if (tid == 0 && sr) atomicAdd(&wk->n_member[1], sr);
}

// Bin index of every member value and the target / region histograms of one column (blockIdx.y) over one row chunk
// (blockIdx.x).  Numerical: searchsorted(grid, v' - step_size / 2, side="left"), v' = ln v for log columns, over
// the host's np.linspace grid; categorical: the choice index.  Counts go into shared-memory integer histograms
// (use_smem; [2][n_grid] ints) or straight to global memory for very wide categorical columns, always by integer
// atomics: the counts do not depend on the order of the additions.  counts: [n_cols][2][width], zeroed by the host.
__global__ void __launch_bounds__(256)
k_ped_bin(int n, int32_t pall, const double* __restrict__ X, const uint8_t* __restrict__ member,
          const PedCol* __restrict__ cols, const double* __restrict__ grids, int n_steps, int width, int use_smem,
          int* __restrict__ counts) {
  extern __shared__ double ped_smem[];
  double* s_grid = ped_smem;                           // [n_steps]
  int* s_cnt = reinterpret_cast<int*>(ped_smem + n_steps);  // [2][n_grid]
  const PedCol c = cols[blockIdx.y];
  const int ng = c.n_grid;
  if (!c.is_cat)
    for (int t = threadIdx.x; t < ng; t += blockDim.x) s_grid[t] = grids[(int64_t)blockIdx.y * n_steps + t];
  if (use_smem)
    for (int t = threadIdx.x; t < 2 * ng; t += blockDim.x) s_cnt[t] = 0;
  __syncthreads();
  int* gcnt = counts + (int64_t)blockIdx.y * 2 * width;
  int* hist = use_smem ? s_cnt : gcnt;
  const int stride = use_smem ? ng : width;
  const double half = (!c.is_cat && ng >= 2) ? TPE_SUB(s_grid[1], s_grid[0]) / 2 : 0.0;
  const int chunk = (n + gridDim.x - 1) / gridDim.x;
  const int lo_i = min(n, (int)blockIdx.x * chunk), hi_i = min(n, lo_i + chunk);
  for (int i = lo_i + threadIdx.x; i < hi_i; i += blockDim.x) {
    const int m = member[i];
    if (!(m & (kPedTarget | kPedRegion))) continue;
    const double v = X[(int64_t)i * pall + c.src];
    int bin;
    if (c.is_cat) {
      bin = (int)v;
    } else {
      const double x = TPE_SUB(c.log ? log(v) : v, half);
      int lo = 0, hi = ng;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (s_grid[mid] < x) lo = mid + 1;
        else hi = mid;
      }
      bin = lo;
    }
    bin = min(max(bin, 0), ng - 1);
    if (m & kPedTarget) atomicAdd(&hist[bin], 1);
    if (m & kPedRegion) atomicAdd(&hist[stride + bin], 1);
  }
  if (use_smem) {
    __syncthreads();
    for (int t = threadIdx.x; t < 2 * ng; t += blockDim.x) {
      const int h = s_cnt[t];
      if (h) atomicAdd(&gcnt[(t / ng) * width + t % ng], h);
    }
  }
}

// _ScottParzenEstimator._calculate_numerical_distributions (scott_parzen_estimator.py:48-80) for the counts of one
// set: kernels at the occupied bins with one Scott bandwidth, then the prior kernel (mu = (n_steps - 1) / 2,
// sigma = n_steps); mixture weights (counts > 0 ++ prior_weight) / sum (parzen_estimator.py:56-67).
// One thread; returns the number of kernels.
__device__ __forceinline__ int ped_numeric_kernels(const int* __restrict__ cnt, int ng, double prior_weight, double* mu,
                                   double* sigma, double* logw) {
  double n_trials = 0.0;
  for (int i = 0; i < ng; ++i) n_trials += (double)cnt[i];
  double mean = 0.0;
  for (int i = 0; i < ng; ++i)
    if (cnt[i] > 0) mean = TPE_ADD(mean, TPE_MUL((double)i, TPE_DIV((double)cnt[i], n_trials)));
  double ss = 0.0;
  for (int i = 0; i < ng; ++i)
    if (cnt[i] > 0) {
      const double dv = TPE_SUB((double)i, mean);
      ss = TPE_ADD(ss, TPE_MUL(TPE_MUL(dv, dv), (double)cnt[i]));
    }
  const double sd = sqrt(TPE_DIV(ss, fmax(1.0, n_trials - 1.0)));
  // interquartile range from the cumulative counts: searchsorted(cum, n // 4, "left"), (n * 3 // 4, "right")
  const double q25 = floor(n_trials / 4.0), q75 = floor(n_trials * 3.0 / 4.0);
  int k = 0, i25 = -1, i75 = -1, last = 0;
  double cum = 0.0;
  for (int i = 0; i < ng; ++i) {
    if (cnt[i] <= 0) continue;
    cum += (double)cnt[i];
    if (i25 < 0 && cum >= q25) i25 = i;
    if (i75 < 0 && cum > q75) i75 = i;
    last = i;
    mu[k++] = (double)i;
  }
  if (i25 < 0) i25 = last;  // searchsorted past the end indexes mus[-1] only through min(size - 1, .)
  if (i75 < 0) i75 = last;
  const double iqr = (double)(i75 - i25);
  const double est = TPE_MUL(TPE_MUL(1.059, fmin(TPE_DIV(iqr, 1.34), sd)), pow(n_trials, -0.2));
  const double s = fmax(est, 0.5 / 1.64);
  const double tot = n_trials + prior_weight;
  k = 0;
  for (int i = 0; i < ng; ++i) {
    if (cnt[i] <= 0) continue;
    sigma[k] = s;
    logw[k] = log(TPE_DIV((double)cnt[i], tot));
    ++k;
  }
  mu[k] = TPE_MUL(0.5, (double)(ng - 1));
  sigma[k] = (double)ng;
  logw[k] = log(TPE_DIV(prior_weight, tot));
  return k + 1;
}

// One CTA per (column, set): the Scott estimator of the target (blockIdx.y = 0) or region (1) counts evaluated on the
// grid 0..n_grid-1, pdf + 1e-12 (evaluator.py:205-216).  pdf: [n_cols][2][width].  evaluate_on_local = 0 launches
// the target set only.
__global__ void __launch_bounds__(128)
k_ped_estimate(const PedCol* __restrict__ cols, const int* __restrict__ counts, int width,
               const PedWork* __restrict__ wk, int min_n_top, double prior_weight, double* __restrict__ pdf) {
  __shared__ double s_mu[kPedMaxSteps + 1], s_sg[kPedMaxSteps + 1], s_lw[kPedMaxSteps + 1], s_nm[kPedMaxSteps + 1];
  __shared__ int s_k;
  if ((long long)wk->n_keep <= min_n_top) return;
  const int j = blockIdx.x, set = blockIdx.y;
  const PedCol c = cols[j];
  const int ng = c.n_grid;
  const int* cnt = counts + ((int64_t)j * 2 + set) * width;
  double* out = pdf + ((int64_t)j * 2 + set) * width;
  const double n_set = (double)wk->n_member[set];
  const double tot = n_set + prior_weight;
  if (c.is_cat) {
    // Aitchison-Aitken rows (parzen_estimator.py:145-166): K = (#occupied choices) + 1 kernels; an observation row
    // holds prior_weight / K everywhere and + 1 at its choice, the prior row prior_weight / K; rows normalised.
    // Every observed choice is one kernel, so the mixture at choice i is a base shared by all choices plus the
    // extra mass of the kernel sitting at i.
    if (threadIdx.x == 0) {
      int k = 0;
      for (int i = 0; i < ng; ++i) k += cnt[i] > 0;
      s_k = k + 1;
    }
    __syncthreads();
    const double base_w = TPE_DIV(prior_weight, (double)s_k);
    const double rs_obs = TPE_ADD(TPE_MUL(base_w, (double)ng), 1.0);
    const double rs_pri = TPE_MUL(base_w, (double)ng);
    const double base = TPE_ADD(TPE_MUL(TPE_DIV(n_set, tot), TPE_DIV(base_w, rs_obs)),
                                TPE_MUL(TPE_DIV(prior_weight, tot), TPE_DIV(base_w, rs_pri)));
    for (int i = threadIdx.x; i < ng; i += blockDim.x) {
      double p = base;
      if (cnt[i] > 0) p = TPE_ADD(p, TPE_MUL(TPE_DIV((double)cnt[i], tot), TPE_DIV(1.0, rs_obs)));
      out[i] = p + 1e-12;
    }
    return;
  }
  if (threadIdx.x == 0) s_k = ped_numeric_kernels(cnt, ng, prior_weight, s_mu, s_sg, s_lw);
  __syncthreads();
  const int K = s_k;
  // normaliser of each discrete truncated normal over 0..ng-1 (probability_distributions.py:188-191)
  const double dlo = -0.5, dhi = TPE_ADD((double)(ng - 1), 0.5);
  for (int k = threadIdx.x; k < K; k += blockDim.x)
    s_nm[k] = log_gauss_mass(TPE_DIV(TPE_SUB(dlo, s_mu[k]), s_sg[k]), TPE_DIV(TPE_SUB(dhi, s_mu[k]), s_sg[k]));
  __syncthreads();
  for (int i = threadIdx.x; i < ng; i += blockDim.x) {
    const double xl = TPE_SUB((double)i, 0.5), xh = TPE_ADD((double)i, 0.5);
    double m = -INFINITY, s = 0.0;
    for (int k = 0; k < K; ++k) {
      const double lm = log_gauss_mass(TPE_DIV(TPE_SUB(xl, s_mu[k]), s_sg[k]), TPE_DIV(TPE_SUB(xh, s_mu[k]), s_sg[k]));
      lse_push(TPE_ADD(TPE_SUB(lm, s_nm[k]), s_lw[k]), m, s);
    }
    out[i] = exp(m + log(s)) + 1e-12;
  }
}

// One thread per column: sum_i pdf_local[i] * (pdf_top[i] / pdf_local[i] - 1)^2 in index order
// (evaluator.py:220), times (n_target / n_region)^2; evaluate_on_local = 0: pdf_local = 1 / n_grid.
__global__ void k_ped_divergence(const PedCol* __restrict__ cols, int n_cols, int width, const PedWork* __restrict__ wk,
                                 int min_n_top, int local, const double* __restrict__ pdf, double* __restrict__ imp) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_cols) return;
  if ((long long)wk->n_keep <= min_n_top) {
    imp[j] = 0.0;
    return;
  }
  const int ng = cols[j].n_grid;
  const double* pt = pdf + (int64_t)j * 2 * width;
  const double* pl = pt + width;
  const double uni = 1.0 / (double)ng;
  double div = 0.0;
  for (int i = 0; i < ng; ++i) {
    const double l = local ? pl[i] : uni;
    const double r = TPE_SUB(TPE_DIV(pt[i], l), 1.0);
    div = TPE_ADD(div, TPE_MUL(l, TPE_MUL(r, r)));
  }
  const double q = (double)wk->n_member[0] / (double)wk->n_member[1];
  imp[j] = TPE_MUL(TPE_MUL(q, q), div);
}

}  // namespace tpe
