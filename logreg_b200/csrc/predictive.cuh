// predictive.cuh -- posterior predictive summaries over S draws in one pass over X:
// for every row i, with eta_is = x_i . beta_s and l_is = log p(y_i | beta_s),
//   prob_mean[i] = mean_s sigma(eta_is)        prob_sd[i] = sd_s sigma(eta_is)   (ddof 1)
//   lppd[i]      = log mean_s exp(l_is)        p_waic[i]  = var_s l_is            (ddof 1)
// and the totals lppd, p_waic, elpd_waic = lppd - p_waic, se_elpd_waic = sqrt(n var_i(elpd_i)).
//
// Tiling (an SGEMM micro-kernel with a statistics epilogue): a CTA owns a tile of 64 rows,
// stored transposed in shared memory (read from HBM once per call), and loops over all draws
// in tiles of 64; the draws (k-major, mode dtype, prepared by the host) come from L2 in chunks
// of <= 64 coefficients.  Thread (tr, td) of the 16 x 16 thread grid computes the 4 x 4 block
// eta[rows tr*4..+3][draws td*4..+3] with explicit FMAs (float32 in FP32 mode, float64 in FP64
// mode), then runs the link function once per element.
//
// Accumulation: per element in the mode's type over the thread's 4 draws of a tile, flushed into
// float64 per-row accumulators once per tile:
//   sigma, l   shifted sums sum(v - K), sum((v - K)^2) with K the thread's first value of the row
//              (no cancellation in the variance while K lies within the spread of the values);
//   exp(l)     sum expm1(l - c) around a per-row reference c, the largest l seen when it was set:
//              exp never overflows (c is re-based when a tile's max exceeds it by 30) and never
//              underflows to a wrong result (the term at c contributes exactly 1 to the sum), so
//              lppd = c + log1p(sum / S) stays finite and accurate when every l_is < -745, and
//              keeps its relative accuracy when lppd is close to 0.
// The 16 threads sharing a row (one half-warp) merge their partial moments (Chan et al.) and
// log-sum-exp states with a butterfly that always puts the lower lane first: fixed order, so every
// per-row result is independent of the grid and of timing.  The totals follow eval_mc_kernel's
// pattern: one partial per CTA, summed in CTA order by the last CTA to take a ticket.
#pragma once
#include <math_constants.h>

#include "eval_kernel.cuh"

namespace lrb {

constexpr int kPredRows = 64;              // rows per CTA tile: 16 row groups x 4
constexpr int kPredDraws = 64;             // draws per tile: 16 draw groups x 4
constexpr int kPredLd = 64 + 4;            // shared-memory row length (padding keeps 16-byte alignment)
constexpr int kPredPartial = 5;            // doubles per CTA partial: sum lppd, sum p_waic, n, mean, M2 of elpd_i
constexpr int kPredTotals = 4;             // lppd, p_waic, elpd_waic, se_elpd_waic

struct PredictiveArgs {
  const void* X;            // bound rows, n x P, mode dtype
  const uint8_t* y;
  long long n;
  const void* B;            // draws, P x Spad (k-major), mode dtype, zero beyond p and S
  long long S, Spad;
  double* prob_mean;        // [n] each; nullptr = not computed into HBM
  double* prob_sd;
  double* lppd;
  double* p_waic;
  double* partials;         // [grid][kPredPartial]
  unsigned int* ticket;     // zero on entry
  double* totals;           // [kPredTotals]
};

template <typename T, int P>
constexpr size_t predictive_smem() {
  return (size_t)(P + (P < 64 ? P : 64)) * kPredLd * sizeof(T);
}

// row_terms of eval_kernel.cuh with sigma(eta) in place of the residual y - sigma(eta) (which
// would have to be turned back into sigma with a cancellation for y = 1): the same
// e = exp(-|eta|) feeds sigma and the overflow-free log-likelihood term.
__device__ __forceinline__ float predictive_terms(float eta, bool y1, float& sig) {
  const float e = expf(-fabsf(eta));
  const float inv = 1.0f / (1.0f + e);
  sig = eta >= 0.0f ? inv : e * inv;
  const float z = y1 ? eta : -eta;
  return fminf(z, 0.0f) - log1pf(e);
}
__device__ __forceinline__ double predictive_terms(double eta, bool y1, double& sig) {
  const double e = exp(-fabs(eta));
  const double inv = 1.0 / (1.0 + e);
  sig = eta >= 0.0 ? inv : e * inv;
  const double z = y1 ? eta : -eta;
  return fmin(z, 0.0) - log1p(e);
}

__device__ __forceinline__ void lds4(const float* p, float (&v)[4]) {
  const float4 t = *reinterpret_cast<const float4*>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
__device__ __forceinline__ void lds4(const double* p, double (&v)[4]) {
  const double2 a = reinterpret_cast<const double2*>(p)[0], b = reinterpret_cast<const double2*>(p)[1];
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}

// Rows row0..+63 into Xs, transposed ([coefficient][row], zero past n), after a barrier that
// frees Xs of the previous tile.  Returns the labels of row group tr's 4 rows as bits.
template <typename T, int P>
__device__ __forceinline__ unsigned stage_x_tile(T* Xs, const void* X, const uint8_t* y, long long n, long long row0,
                                                 int tid, int tr) {
  using vec = typename Chunk<T>::vec;
  constexpr int V = Chunk<T>::V;
  constexpr int CPR = P / V;                 // 16-byte chunks per row of X
  const vec* __restrict__ Xv = reinterpret_cast<const vec*>(X);
  __syncthreads();   // every thread is done with the previous tile's X
  for (int idx = tid; idx < kPredRows * CPR; idx += kBlock) {
    const int r = idx / CPR, c = idx % CPR;
    const long long row = row0 + r;
    const vec v = row < n ? ldg_stream(Xv + row * CPR + c) : zero_vec((vec*)nullptr);
#pragma unroll
    for (int i = 0; i < V; ++i) Xs[(c * V + i) * kPredLd + r] = elem(v, i);
  }
  unsigned ybits = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long row = row0 + tr * 4 + i;
    if (row < n && y[row] != 0) ybits |= 1u << i;
  }
  return ybits;
}

// eta[i][j] = x(row tr*4 + i of the tile in Xs) . beta(draw dt*64 + td*4 + j), the draws (P x Spad,
// k-major in Bg) staged through Bs in chunks of KC coefficients.
template <typename T, int P>
__device__ __forceinline__ void draw_tile_eta(T (&eta)[4][4], const T* Xs, T* Bs, const T* Bg, long long Spad, int dt,
                                              int tid, int tr, int td) {
  using vec = typename Chunk<T>::vec;
  constexpr int V = Chunk<T>::V;
  constexpr int KC = P < 64 ? P : 64;        // coefficients per chunk of draws in shared memory
  constexpr int DV = kPredDraws / V;         // 16-byte chunks per 64 draws
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) eta[i][j] = (T)0;
  for (int k0 = 0; k0 < P; k0 += KC) {
    __syncthreads();   // the previous chunk is consumed (and, the first time, Xs is complete)
    for (int idx = tid; idx < KC * DV; idx += kBlock) {
      const int k = idx / DV, dv = idx % DV;
      *reinterpret_cast<vec*>(Bs + k * kPredLd + dv * V) =
          *reinterpret_cast<const vec*>(Bg + (long long)(k0 + k) * Spad + (long long)dt * kPredDraws + dv * V);
    }
    __syncthreads();
#pragma unroll 4
    for (int k = 0; k < KC; ++k) {
      T xv[4], bv[4];
      lds4(Xs + (k0 + k) * kPredLd + tr * 4, xv);
      lds4(Bs + k * kPredLd + td * 4, bv);
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) eta[i][j] = fma(xv[i], bv[j], eta[i][j]);
    }
  }
}

// (n, mean, M2) of a into which b is merged (Chan, Golub & LeVeque).
__device__ __forceinline__ void merge_moments(double& n, double& mean, double& m2, double nb, double meanb,
                                              double m2b) {
  if (nb == 0.0) return;
  if (n == 0.0) { n = nb; mean = meanb; m2 = m2b; return; }
  const double t = n + nb, d = meanb - mean;
  mean = fma(d, nb / t, mean);
  m2 = m2 + m2b + d * d * (n * nb / t);
  n = t;
}

// Log-sum-exp state: sum_j exp(l_j - c) = m + s over m terms.  Re-base a onto max(c, cb), merge b.
__device__ __forceinline__ void merge_lse(double& c, double& s, double m, double cb, double sb, double mb) {
  if (mb == 0.0) return;
  if (m == 0.0) { c = cb; s = sb; return; }
  const double C = fmax(c, cb), da = c - C, db = cb - C;
  s = (s * exp(da) + m * expm1(da)) + (sb * exp(db) + mb * expm1(db));
  c = C;
}

template <typename T, int P>
__global__ void __launch_bounds__(kBlock, sizeof(T) == 4 ? 2 : 1) predictive_kernel(const PredictiveArgs a) {
  extern __shared__ __align__(16) unsigned char pred_smem[];
  T* Xs = reinterpret_cast<T*>(pred_smem);   // [P][kPredLd]: X tile, (coefficient, row)
  T* Bs = Xs + P * kPredLd;                  // [min(P, 64)][kPredLd]: draw chunk, (coefficient, draw)
  __shared__ double s_own[16][kPredPartial];
  __shared__ T s_ref[3][4][kBlock];          // per thread and row: shifts of sigma and l, log-sum-exp reference c
  __shared__ double s_lse[4][kBlock];        // per thread and row: sum expm1(l - c)
  __shared__ unsigned int s_ticket;

  const int tid = threadIdx.x, tr = tid >> 4, td = tid & 15;
  const long long n = a.n, S = a.S;
  const long long ntiles = (n + kPredRows - 1) / kPredRows;
  const int ndt = (int)(a.Spad / kPredDraws);
  const T* __restrict__ Bg = reinterpret_cast<const T*>(a.B);
  const double Sd = (double)S;

  // s_own[tr]: running sums over the rows of row group tr, updated only by its owner (td == 0);
  // kept in shared memory, not registers, which the 4 x 4 tile's statistics need
  if (tid < 16)
#pragma unroll
    for (int k = 0; k < kPredPartial; ++k) s_own[tid][k] = 0.0;

  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long long row0 = tile * kPredRows;
    const unsigned ybits = stage_x_tile<T, P>(Xs, a.X, a.y, n, row0, tid, tr);   // labels of this thread's 4 rows

    // s_ref and s_lse are touched once per tile: registers are kept for the tile
    double s1s[4], s2s[4], s1l[4], s2l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      s_ref[0][i][tid] = s_ref[1][i][tid] = (T)0;
      s_ref[2][i][tid] = -(T)CUDART_INF;
      s1s[i] = s2s[i] = s1l[i] = s2l[i] = s_lse[i][tid] = 0.0;
    }
    int m = 0;                               // draws this thread has accumulated

    for (int dt = 0; dt < ndt; ++dt) {
      T eta[4][4];
      draw_tile_eta<T, P>(eta, Xs, Bs, Bg, a.Spad, dt, tid, tr, td);

      // link functions and statistics: valid draws of this thread in this tile (< 4 only in the last)
      const long long d0 = (long long)dt * kPredDraws + td * 4;
      const int nv = (int)(S - d0 < 0 ? 0 : (S - d0 > 4 ? 4 : S - d0));
      if (nv > 0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          T &ks = s_ref[0][i][tid], &kl = s_ref[1][i][tid], &c = s_ref[2][i][tid];
          T sig[4], l[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) l[j] = predictive_terms(eta[i][j], (ybits >> i) & 1u, sig[j]);
          if (dt == 0) { ks = sig[0]; kl = l[0]; }
          T mt = l[0];
#pragma unroll
          for (int j = 1; j < 4; ++j)
            if (j < nv) mt = fmax(mt, l[j]);
          if (mt > c + (T)30) {              // re-base: keeps every exp(l - c) below e^30
            const double dl = (double)c - (double)mt;
            s_lse[i][tid] = s_lse[i][tid] * exp(dl) + (double)m * expm1(dl);
            c = mt;
          }
          const T ksv = ks, klv = kl, cv = c;
          T t1s = 0, t2s = 0, t1l = 0, t2l = 0, te = 0;
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (j < nv) {
              const T ds = sig[j] - ksv, dl = l[j] - klv;
              t1s += ds; t2s = fma(ds, ds, t2s);
              t1l += dl; t2l = fma(dl, dl, t2l);
              te += expm1(l[j] - cv);
            }
          s1s[i] += (double)t1s; s2s[i] += (double)t2s;
          s1l[i] += (double)t1l; s2l[i] += (double)t2l;
          s_lse[i][tid] += (double)te;
        }
        m += nv;
      }
    }

    // merge the 16 threads of each row (one half-warp), lower lane first
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      double cnt = (double)m, ms = 0.0, m2s = 0.0, ml = 0.0, m2l = 0.0, cc = (double)s_ref[2][i][tid], ss = s_lse[i][tid];
      if (m > 0) {
        ms = (double)s_ref[0][i][tid] + s1s[i] / cnt;
        m2s = fmax(0.0, s2s[i] - s1s[i] * (s1s[i] / cnt));
        ml = (double)s_ref[1][i][tid] + s1l[i] / cnt;
        m2l = fmax(0.0, s2l[i] - s1l[i] * (s1l[i] / cnt));
      }
#pragma unroll
      for (int o = 1; o < 16; o <<= 1) {
        const double p_cnt = __shfl_xor_sync(0xffffffffu, cnt, o);
        const double p_ms = __shfl_xor_sync(0xffffffffu, ms, o), p_m2s = __shfl_xor_sync(0xffffffffu, m2s, o);
        const double p_ml = __shfl_xor_sync(0xffffffffu, ml, o), p_m2l = __shfl_xor_sync(0xffffffffu, m2l, o);
        const double p_cc = __shfl_xor_sync(0xffffffffu, cc, o), p_ss = __shfl_xor_sync(0xffffffffu, ss, o);
        const bool upper = (td & o) != 0;
        double na = upper ? p_cnt : cnt, a_ms = upper ? p_ms : ms, a_m2s = upper ? p_m2s : m2s;
        double a_ml = upper ? p_ml : ml, a_m2l = upper ? p_m2l : m2l, a_cc = upper ? p_cc : cc, a_ss = upper ? p_ss : ss;
        const double nb = upper ? cnt : p_cnt, b_ms = upper ? ms : p_ms, b_m2s = upper ? m2s : p_m2s;
        const double b_ml = upper ? ml : p_ml, b_m2l = upper ? m2l : p_m2l, b_cc = upper ? cc : p_cc, b_ss = upper ? ss : p_ss;
        merge_lse(a_cc, a_ss, na, b_cc, b_ss, nb);
        double na2 = na;
        merge_moments(na2, a_ml, a_m2l, nb, b_ml, b_m2l);
        merge_moments(na, a_ms, a_m2s, nb, b_ms, b_m2s);
        cnt = na; ms = a_ms; m2s = a_m2s; ml = a_ml; m2l = a_m2l; cc = a_cc; ss = a_ss;
      }
      const long long row = row0 + tr * 4 + i;
      if (td == 0 && row < n) {
        const double lp = cc + log1p(ss / Sd);
        const double pw = m2l / (Sd - 1.0);          // NaN for S = 1
        if (a.prob_mean) a.prob_mean[row] = ms;
        if (a.prob_sd) a.prob_sd[row] = sqrt(m2s / (Sd - 1.0));
        if (a.lppd) a.lppd[row] = lp;
        if (a.p_waic) a.p_waic[row] = pw;
        double* own = s_own[tr];
        own[0] += lp;
        own[1] += pw;
        const double e = lp - pw;                    // Welford over the group's rows
        own[2] += 1.0;
        const double d = e - own[3];
        own[3] += d / own[2];
        own[4] = fma(d, e - own[3], own[4]);
      }
    }
  }

  // ---- CTA partial: the 16 row groups in order
  __syncthreads();
  if (tid == 0) {
    double sl = 0.0, sp = 0.0, cn = 0.0, cm = 0.0, c2 = 0.0;
    for (int w = 0; w < 16; ++w) {
      sl += s_own[w][0];
      sp += s_own[w][1];
      merge_moments(cn, cm, c2, s_own[w][2], s_own[w][3], s_own[w][4]);
    }
    double* mine = a.partials + (size_t)blockIdx.x * kPredPartial;
    mine[0] = sl; mine[1] = sp; mine[2] = cn; mine[3] = cm; mine[4] = c2;
  }

  // ---- last CTA: CTA partials in CTA order
  __threadfence();
  __syncthreads();
  if (tid == 0) s_ticket = atomicAdd(a.ticket, 1u);
  __syncthreads();
  if (s_ticket != gridDim.x - 1) return;
  __threadfence();
  if (tid == 0) {
    double sl = 0.0, sp = 0.0, cn = 0.0, cm = 0.0, c2 = 0.0;
    for (int b = 0; b < (int)gridDim.x; ++b) {
      const double* q = a.partials + (size_t)b * kPredPartial;
      sl += __ldcg(q);
      sp += __ldcg(q + 1);
      merge_moments(cn, cm, c2, __ldcg(q + 2), __ldcg(q + 3), __ldcg(q + 4));
    }
    a.totals[0] = sl;
    a.totals[1] = sp;
    a.totals[2] = sl - sp;
    a.totals[3] = sqrt(cn * (c2 / (cn - 1.0)));   // sqrt(n var_i(elpd_i)), ddof 1
  }
}

}  // namespace lrb
