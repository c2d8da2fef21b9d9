// loo.cuh -- PSIS-LOO over S posterior draws (Vehtari, Simpson, Gelman, Yao & Gabry 2024; the
// `psis()` of R's loo package with r_eff = 1) and the pointwise log-likelihood matrix.
//
// Stage 1, loglik_kernel<T, P>: l_is = log p(y_i | beta_s) for a chunk of rows x all S draws into
// a float64 matrix L[i][s] (rows contiguous), with the tiling and the link function of
// predictive_kernel: a 64-row X tile transposed in shared memory, the draws k-major in the mode's
// dtype, a 4 x 4 register tile of explicit FMAs, predictive_terms.  The 16 threads of a row (a
// half-warp) store its 64 draws of a tile contiguously.
//
// Stage 2, psis_kernel: one CTA per row of the chunk (grid-striding), the row staged in shared
// memory when it fits, else read from L (L2 for a chunk sized to stay there).  With r_s = -l_s:
//   1. max / min of l and the log-sum-exp for lppd;
//   2. an exact radix select (order-preserving 64-bit keys of l, 8-bit digits, shared-memory
//      histogram) of the M + 1 smallest l = the M + 1 largest r: the tail and the cutoff;
//   3. the candidates compacted and rank-sorted in shared memory;
//   4. the generalized Pareto fit of Zhang & Stephens (2009) with loo's weak prior and wip
//      adjustment: theta-grid points across warps, each a fixed-order sum over the tail;
//   5. the smoothed, truncated tail, and one more pass for the non-tail denominator (never
//      total - tail: the tail dominates exactly when k-hat is large).
// Outside the tail lw_s + l_s = -max r, so the numerator's non-tail part is (S - M) exp(-max r).
// Ties at the cutoff do not matter: tied draws have equal l, so every sum sees the same multiset.
//
// Every per-row result is computed in a fixed order by one CTA: independent of the grid, the chunk
// size and timing.  The totals are per-64-row-tile partials merged in tile order.
#pragma once
#include <math_constants.h>

#include <cmath>

#include "predictive.cuh"

namespace lrb {

constexpr long long kLooMaxDraws = 1ll << 21;   // S cap: 64 rows of L are 1 GB
constexpr int kLooRowSmem = 12288;              // rows of up to this many draws are staged in shared memory
constexpr int kLoglikGroup = 4;                 // draw tiles (of 64) per work item of loglik_kernel
constexpr int kGpdMaxGrid = 128;                // theta-grid points: 30 + floor(sqrt(M)) <= 95 for S <= 2^21
constexpr int kLooPartial = 9;                  // per tile: n, sum elpd, mean elpd, M2 elpd, sum p_loo, mean p_loo, M2 p_loo, k max, # k > threshold

// ---- the PSIS formulas, shared by psis_kernel and the host path of lrb_debug_psis
__host__ __device__ inline long long psis_tail_len(long long S) {        // M = ceil(min(0.2 S, 3 sqrt(S)))
  const double s = (double)S;
  return (long long)ceil(fmin(0.2 * s, 3.0 * sqrt(s)));
}
__host__ __device__ inline int gpd_grid_len(long long N) { return 30 + (int)floor(sqrt((double)N)); }
__host__ __device__ inline double gpd_theta(int j, int m, double xmax, double xstar) {   // j = 1..m
  return 1.0 / xmax + (1.0 - sqrt((double)m / ((double)j - 0.5))) / 3.0 / xstar;       // prior = 3
}
__host__ __device__ inline double gpd_ltheta(double theta, double k, long long N) {
  return (double)N * (log(-theta / k) - k - 1.0);
}
__host__ __device__ inline double gpd_wip(double k, long long N) {          // loo's adjust_k_wip
  const double n = (double)N;
  const double kw = k * n / (n + 10.0) + 10.0 * 0.5 / (n + 10.0);
  return kw != kw ? (double)INFINITY : kw;
}
__host__ __device__ inline double psis_quantile(long long j, long long M) { // j = 1..M
  return ((double)j - 0.5) / (double)M;
}
__host__ __device__ inline double psis_smoothed(double k, double sigma, double p, double exp_cutoff) {
  return log(sigma * expm1(-k * log1p(-p)) / k + exp_cutoff);
}
__host__ __device__ inline double loo_k_threshold(long long S) {           // min(1 - 1/log10 S, 0.7)
  return fmin(1.0 - 1.0 / log10((double)S), 0.7);
}
// max that propagates NaN (as NumPy's max does)
__host__ __device__ inline double nan_max(double a, double b) { return (a != a || b != b) ? a + b : fmax(a, b); }

struct LoglikArgs {
  const void* X;            // rows of the chunk, nrows x P, mode dtype
  const uint8_t* y;
  long long n;              // rows of the chunk
  const void* B;            // draws, P x Spad (k-major), mode dtype, zero beyond p and S
  long long S, Spad;
  double* L;                // [n][ld]
  long long ld;
};

template <typename T, int P>
__global__ void __launch_bounds__(kBlock, sizeof(T) == 4 ? 2 : 1) loglik_kernel(const LoglikArgs a) {
  extern __shared__ __align__(16) unsigned char ll_smem[];
  T* Xs = reinterpret_cast<T*>(ll_smem);     // [P][kPredLd]: X tile, (coefficient, row)
  T* Bs = Xs + P * kPredLd;                  // [min(P, 64)][kPredLd]: draw chunk, (coefficient, draw)

  const int tid = threadIdx.x, tr = tid >> 4, td = tid & 15;
  const long long n = a.n, S = a.S;
  const long long ntiles = (n + kPredRows - 1) / kPredRows;
  const int ndt = (int)(a.Spad / kPredDraws);
  const T* __restrict__ Bg = reinterpret_cast<const T*>(a.B);

  // work item = (row tile, group of kLoglikGroup draw tiles): the outputs are independent, so a
  // chunk of few rows still spreads over the whole GPU when S is large
  const int ngroups = (ndt + kLoglikGroup - 1) / kLoglikGroup;
  for (long long w = blockIdx.x; w < ntiles * ngroups; w += gridDim.x) {
    const long long tile = w / ngroups;
    const int dt0 = (int)(w % ngroups) * kLoglikGroup, dt1 = min(dt0 + kLoglikGroup, ndt);
    const long long row0 = tile * kPredRows;
    const unsigned ybits = stage_x_tile<T, P>(Xs, a.X, a.y, n, row0, tid, tr);

    for (int dt = dt0; dt < dt1; ++dt) {
      T eta[4][4];
      draw_tile_eta<T, P>(eta, Xs, Bs, Bg, a.Spad, dt, tid, tr, td);
      const long long d0 = (long long)dt * kPredDraws + td * 4;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const long long row = row0 + tr * 4 + i;
        if (row >= n) continue;
        double* dst = a.L + row * a.ld + d0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          T sig;
          const T l = predictive_terms(eta[i][j], (ybits >> i) & 1u, sig);
          if (d0 + j < S) dst[j] = (double)l;
        }
      }
    }
  }
}

struct PsisArgs {
  const double* L;          // [rows][S]
  long long rows, S, M;     // M: tail length (psis_tail_len)
  int stage;                // 1: the row fits kLooRowSmem and is copied to shared memory
  double* elpd;             // [rows] each
  double* p_loo;
  double* pareto_k;
};

inline size_t psis_smem(long long S, long long M, int stage) {
  return ((stage ? (size_t)S : 0) + 2 * (size_t)(M + 1)) * sizeof(double);
}

// order-preserving key of a double (+0 for -0): key(a) < key(b) <=> a < b
__device__ __forceinline__ unsigned long long order_key(double v) {
  const unsigned long long u = (unsigned long long)__double_as_longlong(v == 0.0 ? 0.0 : v);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double key_value(unsigned long long k) {
  return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k));
}

// NaN-propagating max over the CTA (fixed order; every thread receives it)
__device__ inline double block_max(double v, double* scratch) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = nan_max(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  double m = scratch[0];
#pragma unroll
  for (int w = 1; w < kWarps; ++w) m = nan_max(m, scratch[w]);
  return m;
}

__global__ void __launch_bounds__(kBlock) psis_kernel(const PsisArgs a) {
  static_assert(kBlock == 256, "one histogram bin per thread, 32 lanes x 8 bins in the scan");
  extern __shared__ __align__(16) unsigned char psis_dyn[];
  __shared__ unsigned int hist[256];
  __shared__ double scratch[kWarps];
  __shared__ double s_theta[kGpdMaxGrid], s_kj[kGpdMaxGrid];
  __shared__ unsigned int s_sel[3];
  __shared__ unsigned int s_cnt;
  __shared__ double s_fit[2];             // k-hat, sigma

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long S = a.S, M = a.M;
  const bool tail = M >= 5;
  double* cand = reinterpret_cast<double*>(psis_dyn);   // [M + 1]: r of the candidates, then the x of the fit
  double* srt = cand + (M + 1);                         // [M + 1]: r sorted ascending: cutoff, tail
  double* row_s = srt + (M + 1);                        // [S] when staged

  for (long long row = blockIdx.x; row < a.rows; row += gridDim.x) {
    const double* src = a.L + row * S;
    if (a.stage) {
      __syncthreads();
      for (long long s = tid; s < S; s += kBlock) row_s[s] = src[s];
      src = row_s;
    }
    // ---- 1. max / min of l, log-sum-exp of l
    double lmax = -CUDART_INF, lmin = CUDART_INF;
    for (long long s = tid; s < S; s += kBlock) {
      const double l = src[s];
      lmax = nan_max(lmax, l);
      lmin = -nan_max(-lmin, -l);
    }
    lmax = block_max(lmax, scratch);
    lmin = -block_max(-lmin, scratch);
    double se = 0.0;
    for (long long s = tid; s < S; s += kBlock) se += exp(src[s] - lmax);
    se = block_sum(se, scratch);
    const double lppd = lmax + log(se) - log((double)S);
    const double rmax = 0.0 - lmin;

    // ---- 2. radix select of the (M + 1)-th smallest l: key K, c_lt keys below it, c_eq equal to it
    unsigned long long K = 0, mask = 0;
    unsigned int c_lt = 0, c_eq = 0;
    double khat = CUDART_INF, lw_cut = 0.0;
    const long long T = tail ? M : 0;     // tail draws handled apart (none without a tail)
    if (tail) {
      unsigned int need = (unsigned int)M + 1;
      const long long rounds = (S + kBlock - 1) / kBlock;
      for (int shift = 56; shift >= 0; shift -= 8) {
        __syncthreads();
        hist[tid] = 0;
        __syncthreads();
        for (long long rd = 0; rd < rounds; ++rd) {
          const long long s = rd * kBlock + tid;
          int bin = 256;
          if (s < S) {
            const unsigned long long key = order_key(src[s]);
            if ((key & mask) == K) bin = (int)((key >> shift) & 255);
          }
          const unsigned peers = __match_any_sync(0xffffffffu, bin);
          if (bin < 256 && lane == __ffs(peers) - 1) atomicAdd(&hist[bin], (unsigned)__popc(peers));
        }
        __syncthreads();
        if (warp == 0) {
          unsigned int c[8], loc = 0;
#pragma unroll
          for (int b = 0; b < 8; ++b) { c[b] = hist[lane * 8 + b]; loc += c[b]; }
          unsigned int inc = loc;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const unsigned int t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
          }
          unsigned int before = inc - loc;
          if (before < need && need <= inc) {
#pragma unroll
            for (int b = 0; b < 8; ++b) {
              if (before < need && need <= before + c[b]) { s_sel[0] = lane * 8 + b; s_sel[1] = before; s_sel[2] = c[b]; }
              before += c[b];
            }
          }
        }
        __syncthreads();
        K |= (unsigned long long)s_sel[0] << shift;
        mask |= 255ull << shift;
        c_lt += s_sel[1];
        need -= s_sel[1];
        c_eq = s_sel[2];
      }

      // ---- 3. candidates (r = -l) and their ascending order; srt[0] is the cutoff, srt[1..M] the tail
      const double r_cut = 0.0 - key_value(K);
      if (tid == 0) s_cnt = 0;
      __syncthreads();
      for (long long s = tid; s < S; s += kBlock) {
        const double l = src[s];
        if (order_key(l) < K) cand[atomicAdd(&s_cnt, 1u)] = 0.0 - l;
      }
      for (long long j = c_lt + tid; j <= M; j += kBlock) cand[j] = r_cut;
      __syncthreads();
      for (long long i = tid; i <= M; i += kBlock) {
        const double v = cand[i];
        long long rank = 0;
        for (long long j = 0; j <= M; ++j) {
          const double u = cand[j];
          rank += (u > v || (u == v && j < i)) ? 1 : 0;   // descending r first ...
        }
        srt[M - rank] = v;                                   // ... stored ascending
      }
      __syncthreads();

      // ---- 4. generalized Pareto fit to x = exp(tail lw) - exp(cutoff lw), lw = r - max r
      lw_cut = srt[0] - rmax;
      const double tmin = srt[1] - rmax, tmax = srt[M] - rmax;
      double* x = cand;
      double sigma = 0.0;
      const double ec = exp(lw_cut);
      if (fabs(tmax - tmin) >= 2.220446049250313e-16 / 100.0) {
        for (long long j = tid; j < M; j += kBlock) x[j] = exp(srt[1 + j] - rmax) - ec;
        __syncthreads();
        const int mg = gpd_grid_len(M);
        const double xmax = x[M - 1], xstar = x[(long long)floor((double)M / 4.0 + 0.5) - 1];
        for (int j = warp; j < mg; j += kWarps) {
          const double th = gpd_theta(j + 1, mg, xmax, xstar);
          double sk = 0.0;
          for (long long t = lane; t < M; t += 32) sk += log1p(-th * x[t]);
          sk = warp_sum(sk);
          if (lane == 0) { s_theta[j] = th; s_kj[j] = sk / (double)M; }
        }
        __syncthreads();
        if (tid == 0) {   // theta-hat: the posterior mean over the grid
          double lmx = -CUDART_INF;
          for (int j = 0; j < mg; ++j) { s_kj[j] = gpd_ltheta(s_theta[j], s_kj[j], M); lmx = nan_max(lmx, s_kj[j]); }
          double sw = 0.0;
          for (int j = 0; j < mg; ++j) sw += exp(s_kj[j] - lmx);
          const double lse = lmx + log(sw);
          double th = 0.0;
          for (int j = 0; j < mg; ++j) th += s_theta[j] * exp(s_kj[j] - lse);
          s_fit[0] = th;
        }
        __syncthreads();
        const double th = s_fit[0];
        double sk = 0.0;
        for (long long t = tid; t < M; t += kBlock) sk += log1p(-th * x[t]);
        sk = block_sum(sk, scratch);                     // every thread is done with x
        const double kraw = sk / (double)M;
        sigma = -kraw / th;
        khat = gpd_wip(kraw, M);
      }
      // the tail's final log weights (smoothed when k-hat is finite, truncated at 0) replace x
      const bool smooth = isfinite(khat);
      for (long long j = tid; j < M; j += kBlock) {
        double lw = smooth ? psis_smoothed(khat, sigma, psis_quantile(j + 1, M), ec) : srt[1 + j] - rmax;
        cand[j] = lw > 0.0 ? 0.0 : lw;
      }
      __syncthreads();
    }

    // ---- 5. elpd_loo = log sum exp(lw + l) - log sum exp(lw), in the frame lw = r - max r.
    // Numerator: (S - T) non-tail terms equal to -max r, tail terms lw_j - r_j.  Denominator: the
    // non-tail draws (keys above K, and the cutoff-valued draws left out of the tail), the tail's lw_j.
    double tmx = -CUDART_INF, nmx = -CUDART_INF;
    for (long long j = tid; j < T; j += kBlock) {
      tmx = nan_max(tmx, cand[j]);
      nmx = nan_max(nmx, cand[j] - srt[1 + j]);
    }
    tmx = block_max(tmx, scratch);
    nmx = block_max(nmx, scratch);
    const double dref = tail ? nan_max(tmx, lw_cut) : 0.0;
    const double nref = nan_max(nmx, -rmax);
    double dn = 0.0;
    for (long long s = tid; s < S; s += kBlock) {
      const double l = src[s];
      if (!tail || order_key(l) > K) dn += exp(((0.0 - l) - rmax) - dref);
    }
    dn = block_sum(dn, scratch);
    double dt = 0.0, nt = 0.0;
    for (long long j = tid; j < T; j += kBlock) {
      dt += exp(cand[j] - dref);
      nt += exp((cand[j] - srt[1 + j]) - nref);
    }
    dt = block_sum(dt, scratch);
    nt = block_sum(nt, scratch);
    if (tid == 0) {
      const double n_cut_out = tail ? (double)(c_eq - ((unsigned int)M - c_lt)) : 0.0;
      const double den = dref + log((dn + n_cut_out * exp(lw_cut - dref)) + dt);
      const double num = nref + log((double)(S - T) * exp(-rmax - nref) + nt);
      const double elpd = num - den;
      a.elpd[row] = elpd;
      a.p_loo[row] = lppd - elpd;
      a.pareto_k[row] = khat;
    }
  }
}

// Per 64-row tile of the chunk: kLooPartial doubles, rows in order.
__global__ void __launch_bounds__(kBlock) loo_tile_kernel(const double* elpd, const double* p_loo, const double* pareto_k,
                                                          long long rows, double k_threshold, double* partials) {
  const long long tile = (long long)blockIdx.x * kBlock + threadIdx.x;
  if (tile * kPredRows >= rows) return;
  double q[kLooPartial] = {};
  const long long end = rows < (tile + 1) * kPredRows ? rows : (tile + 1) * kPredRows;
  for (long long i = tile * kPredRows; i < end; ++i) {
    const double e = elpd[i], pl = p_loo[i], k = pareto_k[i];
    q[0] += 1.0;
    q[1] += e;
    const double d = e - q[2];
    q[2] += d / q[0];
    q[3] = fma(d, e - q[2], q[3]);
    q[4] += pl;
    const double dp = pl - q[5];
    q[5] += dp / q[0];
    q[6] = fma(dp, pl - q[5], q[6]);
    q[7] = i == tile * kPredRows ? k : nan_max(q[7], k);
    q[8] += k > k_threshold ? 1.0 : 0.0;
  }
  double* dst = partials + tile * kLooPartial;
#pragma unroll
  for (int j = 0; j < kLooPartial; ++j) dst[j] = q[j];
}

__device__ __forceinline__ void merge_loo(double* a, const double* b) {
  if (b[0] == 0.0) return;   // an empty partial (a thread with no tiles) has no k max
  const double n = a[0];
  merge_moments(a[0], a[2], a[3], b[0], b[2], b[3]);
  double n2 = n;
  merge_moments(n2, a[5], a[6], b[0], b[5], b[6]);
  a[1] += b[1];
  a[4] += b[4];
  a[7] = n == 0.0 ? b[7] : nan_max(a[7], b[7]);
  a[8] += b[8];
}

// One CTA: thread t merges a contiguous run of tiles, thread 0 the threads' results in order.
// totals: n, elpd_loo, se_elpd_loo, p_loo, se_p_loo, k_max, n_k_high
__global__ void __launch_bounds__(kBlock) loo_totals_kernel(const double* partials, long long ntiles, double* totals) {
  __shared__ double part[kBlock][kLooPartial];
  const int tid = threadIdx.x;
  const long long per = (ntiles + kBlock - 1) / kBlock;
  double q[kLooPartial] = {};
  for (long long t = tid * per; t < ntiles && t < (tid + 1) * per; ++t) merge_loo(q, partials + t * kLooPartial);
#pragma unroll
  for (int j = 0; j < kLooPartial; ++j) part[tid][j] = q[j];
  __syncthreads();
  if (tid != 0) return;
  for (int t = 1; t < kBlock; ++t) merge_loo(q, part[t]);
  const double n = q[0];
  totals[0] = n;
  totals[1] = q[1];
  totals[2] = sqrt(n * (q[3] / (n - 1.0)));
  totals[3] = q[4];
  totals[4] = sqrt(n * (q[6] / (n - 1.0)));
  totals[5] = q[7];
  totals[6] = q[8];
}

}  // namespace lrb
