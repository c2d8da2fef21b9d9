// eval_kernel.cuh -- the fused single-pass log-likelihood + gradient kernel.
//
// Replaces, in ONE pass over X (paths relative to the reference root):
//   ll   Python/fit-numpy.py:23-24     sum(-log(1+exp(-(2y-1)*(X.dot(beta)))))
//   glp  Python/fit-np-ul.py:45-48     X.T.dot(y - 1/(1+exp(-X.dot(beta)))) - beta/pscale^2
// (the reference makes one pass for ll and two for glp, with 4 length-n temporaries).
//
// Data layout in HBM: X row-major, n x P (P = p zero-padded to 8/16/../256),
// element type T (float in FP32 mode, double in FP64 mode); y one byte per row.
// Rows are contiguous, so a warp streams the matrix as consecutive 512-byte
// "slabs": lane l of slab s reads the 16-byte chunk (s*32 + l) with one
// ld.global.nc.L1::no_allocate.v4 -- perfectly coalesced, each byte of X read
// exactly once.  A warp handles a batch of S=16 slabs (8 KB) at a time; with
// >= 16 warps per SM that is >= 128 KB in flight per SM, several times the
// latency-bandwidth product (~35 KB/SM), without a shared-memory stage.
//
// Per batch:
//   1. every lane forms the partial dot product of its chunk with its slice of beta;
//   2. the partials of a row (spread over L = min(32, chunks per row) lanes) are
//      combined with a recursive-halving exchange: log2(L) shuffle rounds after
//      which every lane owns the COMPLETE eta of distinct rows (no redundancy);
//   3. the owning lane evaluates softplus / sigmoid once per row (overflow-free:
//      e = exp(-|eta|) is shared by log1p(e) and by the sigmoid), adds the row's
//      log-likelihood term to its fp64 accumulator and forms the residual
//      r = y - p without cancellation (y=1: sigma(-eta); y=0: -sigma(eta));
//   4. r is shuffled back to the lanes holding the row's chunks, which do the
//      rank-1 update g[cols of this lane] += r * x -- each lane keeps only V
//      (4 or 2) gradient accumulators per slab-column group.
// FP32 mode: eta and the per-batch gradient partial (<= 32 rows) are float32 FMAs,
// flushed into float64 accumulators once per batch; beta is carried as hi+lo
// floats so its rounding does not enter eta.  FP64 mode: everything float64.
//
// Reduction: warp shuffles -> shared memory -> one (P+1)-vector per CTA in global
// memory -> the LAST CTA to finish (atomic ticket) sums the CTA partials in a
// fixed order (deterministic for a fixed grid), then runs finish_eval(): optional
// fused peer-memory allreduce, prior, and the sampler update -- so a sampler
// iteration costs one kernel launch per evaluation and no host round trip.
#pragma once
#include "common.cuh"
#include "sampler.cuh"

namespace lrb {

struct EvalArgs {
  const void* X;
  const uint8_t* y;
  long long n;
  double* partials;   // [grid][P+1]
  unsigned int* ticket;
  double* sums;       // [P+1] un-fused output: [ll, gll]
  int fuse_finish;    // 1: run finish_eval in the last CTA; 0: only write `sums`
  FinishArgs fin;
  long long* timeline;  // development aid (lrb_debug_timeline): %globaltimer stamps, [grid][4] + [8]; else nullptr
};

__device__ __forceinline__ long long global_ns() {
  long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
#define EV_STAMP(slot) do { if (a.timeline != nullptr && tid == 0) a.timeline[(size_t)blockIdx.x * 4 + (slot)] = global_ns(); } while (0)
#define EV_STAMP_LAST(slot) do { if (a.timeline != nullptr && tid == 0) a.timeline[(size_t)gridDim.x * 4 + (slot)] = global_ns(); } while (0)

template <typename T> struct Chunk;
template <> struct Chunk<float> {
  static constexpr int V = 4;
  using vec = float4;
  using acc_t = float;
};
template <> struct Chunk<double> {
  static constexpr int V = 2;
  using vec = double2;
  using acc_t = double;
};

__device__ __forceinline__ float4 ldg_stream(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ double2 ldg_stream(const double2* p) {
  double2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0,%1}, [%2];"
               : "=d"(r.x), "=d"(r.y) : "l"(p));
  return r;
}
__device__ __forceinline__ float4 zero_vec(float4*) { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ double2 zero_vec(double2*) { return make_double2(0.0, 0.0); }

__device__ __forceinline__ float elem(const float4& v, int i) {
  return i == 0 ? v.x : i == 1 ? v.y : i == 2 ? v.z : v.w;
}
__device__ __forceinline__ double elem(const double2& v, int i) { return i == 0 ? v.x : v.y; }

__host__ __device__ constexpr int ilog2(int v) { return v <= 1 ? 0 : 1 + ilog2(v >> 1); }

// Recursive halving over lane bits [B, LOG_L): on entry the lane holds CNT row
// partials; a lane whose bit B is set keeps the upper half and sends the lower
// half to its partner (and vice versa).  Once one value is left the remaining
// bits are plain butterflies.
template <int CNT, int B, int LOG_L, typename A, int N>
__device__ __forceinline__ void reduce_rows(A (&q)[N], int lane) {
  if constexpr (B < LOG_L) {
    if constexpr (CNT > 1) {
      constexpr int H = CNT / 2;
      const bool up = (lane >> B) & 1;
#pragma unroll
      for (int i = 0; i < H; ++i) {
        const A send = up ? q[i] : q[i + H];
        const A keep = up ? q[i + H] : q[i];
        q[i] = keep + __shfl_xor_sync(0xffffffffu, send, 1 << B);
      }
      reduce_rows<H, B + 1, LOG_L>(q, lane);
    } else {
      q[0] += __shfl_xor_sync(0xffffffffu, q[0], 1 << B);
      reduce_rows<1, B + 1, LOG_L>(q, lane);
    }
  }
}

// Per-row link functions. Returns the log-likelihood term; r = y - sigmoid(eta).
__device__ __forceinline__ float row_terms(float eta, bool y1, float& r) {
  const float e = expf(-fabsf(eta));
  const float inv = 1.0f / (1.0f + e);
  const float big = inv, small = e * inv;            // sigma(|eta|), sigma(-|eta|)
  const bool pos = eta >= 0.0f;
  r = y1 ? (pos ? small : big) : -(pos ? big : small);
  const float z = y1 ? eta : -eta;
  return fminf(z, 0.0f) - log1pf(e);
}
__device__ __forceinline__ double row_terms(double eta, bool y1, double& r) {
  const double e = exp(-fabs(eta));
  const double inv = 1.0 / (1.0 + e);
  const double big = inv, small = e * inv;
  const bool pos = eta >= 0.0;
  r = y1 ? (pos ? small : big) : -(pos ? big : small);
  const double z = y1 ? eta : -eta;
  return fmin(z, 0.0) - log1p(e);
}

// One warp's row batch in the SIMT evaluation kernels (eval_kernel, eval_persist_kernel,
// eval_mc_kernel): the tiling, this lane's place in it, and the per-batch arithmetic (steps 1-4
// above).  The kernels own only which batches a warp takes and where the sums go.
template <typename T, int P>
struct BatchTile {
  using C = Chunk<T>;
  using vec = typename C::vec;
  using A = typename C::acc_t;
  static constexpr int V = C::V;
  static constexpr int CPR = P / V;                // 16-byte chunks per row
  static constexpr int L = CPR < 32 ? CPR : 32;    // lanes sharing a row inside one slab
  static constexpr int SPR = CPR / L;              // slabs per row (>1 when a row exceeds 512 B)
  static constexpr int G = 32 / L;                 // rows per slab (SPR == 1)
  static constexpr int S = 16;                     // slabs per batch
  static constexpr int SG = S / SPR;               // row groups per batch
  static constexpr int RB = SG * G;                // rows per batch
  static constexpr int LOG_L = ilog2(L), LOG_SG = ilog2(SG);
  static constexpr int NH = LOG_L < LOG_SG ? LOG_L : LOG_SG;  // halving rounds
  static constexpr int M = SG >> NH;               // etas a lane owns per batch
  static_assert(S % SPR == 0 && SG >= 1, "row too wide for the batch");
  static_assert((1 << LOG_L) == L && (1 << LOG_SG) == SG, "power-of-two tiling");

  // this lane's slice of a coefficient vector, columns (sl*L + t_in_row)*V .. +V, as hi + lo
  // (lo is exactly 0 in FP64 mode)
  struct Coef {
    A hi[SPR][V];
    float lo[SPR][V];
  };
  // labels and validity of the M rows this lane owns in a batch
  struct Rows {
    bool y1[M], valid[M];
  };

  long long n;              // rows of X
  long long total_chunks;   // 16-byte chunks of X; formed here, once: formed in load, it changed how the
                            // compiler unrolls the drive kernel's finish step
  long long nbatch;         // batches of X, the last one possibly partial
  int lane;
  int t_in_row;    // which chunk of the row segment
  int g_in_slab;   // which row of the slab
  int khigh;       // rows this lane owns after the exchange: k = j + khigh, row = row0 + k*G + g_in_slab
  bool owner;

  __device__ __forceinline__ BatchTile(long long n_, int lane_)
      : n(n_), total_chunks(n_ * CPR), nbatch((n_ + RB - 1) / RB), lane(lane_), t_in_row(lane_ & (L - 1)),
        g_in_slab(lane_ >> LOG_L), khigh(0) {
#pragma unroll
    for (int b = 0; b < NH; ++b) khigh += ((t_in_row >> b) & 1) * (SG >> (b + 1));
    owner = (t_in_row >> NH) == 0;
  }

  // The S slabs of batch bt; chunks past the end of X read as zero.
  __device__ __forceinline__ void load(vec (&v)[S], const vec* __restrict__ Xv, long long bt) const {
    const long long chunk0 = bt * (S * 32) + lane;
    if (bt * RB + RB <= n) {
#pragma unroll
      for (int s = 0; s < S; ++s) v[s] = ldg_stream(Xv + chunk0 + s * 32);
    } else {
#pragma unroll
      for (int s = 0; s < S; ++s) {
        const long long c = chunk0 + s * 32;
        v[s] = c < total_chunks ? ldg_stream(Xv + c) : zero_vec((vec*)nullptr);
      }
    }
  }

  // Read through L2: in the fused kernels the previous evaluation's last CTA wrote beta.
  __device__ __forceinline__ void load_coef(Coef& cf, const double* beta, int p) const {
#pragma unroll
    for (int sl = 0; sl < SPR; ++sl)
#pragma unroll
      for (int i = 0; i < V; ++i) {
        const int col = (sl * L + t_in_row) * V + i;
        const double x = col < p ? __ldcg(beta + col) : 0.0;
        cf.hi[sl][i] = (A)x;
        cf.lo[sl][i] = (float)(x - (double)cf.hi[sl][i]);
      }
  }

  __device__ __forceinline__ void load_rows(Rows& rw, const uint8_t* y, long long bt) const {
    const long long row0 = bt * RB;
#pragma unroll
    for (int j = 0; j < M; ++j) {
      const long long row = row0 + (long long)(j + khigh) * G + g_in_slab;
      rw.valid[j] = owner && row < n;
      rw.y1[j] = rw.valid[j] ? (y[row] != 0) : false;
    }
  }

  // One batch at one coefficient vector: the rows' log-likelihood terms into ll, and with GRAD
  // this lane's gradient columns into acc.
  template <bool GRAD>
  __device__ __forceinline__ void accumulate(const vec (&v)[S], const Rows& rw, const Coef& cf, double& ll,
                                             double (&acc)[SPR][V]) const {
    // 1. partial dot products, combined over the slabs of a row
    A q[SG];
#pragma unroll
    for (int k = 0; k < SG; ++k) {
      A s_hi = (A)0;
#pragma unroll
      for (int sl = 0; sl < SPR; ++sl)
#pragma unroll
        for (int i = 0; i < V; ++i) s_hi = fma(elem(v[k * SPR + sl], i), cf.hi[sl][i], s_hi);
      if constexpr (sizeof(T) == 4) {
        float s_lo = 0.f;
#pragma unroll
        for (int sl = 0; sl < SPR; ++sl)
#pragma unroll
          for (int i = 0; i < V; ++i) s_lo = fmaf((float)elem(v[k * SPR + sl], i), cf.lo[sl][i], s_lo);
        s_hi += (A)s_lo;
      }
      q[k] = s_hi;
    }
    // 2. row sums: afterwards q[0..M) are complete etas of distinct rows
    reduce_rows<SG, 0, LOG_L>(q, lane);

    // 3. link functions, once per row
    A r[M];
#pragma unroll
    for (int j = 0; j < M; ++j) {
      A rr;
      const A lt = row_terms(q[j], rw.y1[j], rr);
      r[j] = rr;
      if (rw.valid[j]) ll += (double)lt;
    }

    // 4. gradient: g[cols of this lane] += r(row) * x
    if constexpr (GRAD) {
      A gb[SPR][V];
#pragma unroll
      for (int sl = 0; sl < SPR; ++sl)
#pragma unroll
        for (int i = 0; i < V; ++i) gb[sl][i] = (A)0;
#pragma unroll
      for (int k = 0; k < SG; ++k) {
        const int j = k & (M - 1);
        int tsrc = 0;
#pragma unroll
        for (int b = 0; b < NH; ++b) tsrc |= ((k >> (LOG_SG - 1 - b)) & 1) << b;
        const A rr = __shfl_sync(0xffffffffu, r[j], (lane & ~(L - 1)) | tsrc);
#pragma unroll
        for (int sl = 0; sl < SPR; ++sl)
#pragma unroll
          for (int i = 0; i < V; ++i) gb[sl][i] = fma(rr, (A)elem(v[k * SPR + sl], i), gb[sl][i]);
      }
#pragma unroll
      for (int sl = 0; sl < SPR; ++sl)
#pragma unroll
        for (int i = 0; i < V; ++i) acc[sl][i] += (double)gb[sl][i];
    }
  }

  // The warp's gradient sums: acc over the lanes of equal t_in_row, column c to dst[c].
  __device__ __forceinline__ void store_grad(const double (&acc)[SPR][V], double* dst) const {
#pragma unroll
    for (int sl = 0; sl < SPR; ++sl)
#pragma unroll
      for (int i = 0; i < V; ++i) {
        double x = acc[sl][i];
#pragma unroll
        for (int o = L; o < 32; o <<= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        if (lane < L) dst[(sl * L + lane) * V + i] = x;
      }
  }
};

template <typename T, int P, bool GRAD>
__global__ void __launch_bounds__(kBlock, 2) eval_kernel(const EvalArgs a) {
  using Tile = BatchTile<T, P>;
  using vec = typename Tile::vec;

  __shared__ double red[kWarps][P + 1];
  __shared__ double redll[kWarps];
  __shared__ double tot[P + 1];
  __shared__ double scratch[kWarps];
  __shared__ unsigned int s_ticket;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const Tile tl(a.n, lane);
  const vec* __restrict__ Xv = reinterpret_cast<const vec*>(a.X);
  const long long nbatch = tl.nbatch;
  const long long nwarps = (long long)gridDim.x * kWarps;
  const long long bt0 = (long long)blockIdx.x * kWarps + warp;

  // Programmatic dependent launch: this grid may start while the previous evaluation's last
  // CTA is still reducing / running the sampler update.  X never changes, so the first batch
  // is fetched BEFORE waiting for the previous grid (hides launch latency and the DRAM ramp);
  // everything that depends on it (beta, the pause flag, the partials buffer) comes after.
  EV_STAMP(0);
  vec v[Tile::S];
  if (bt0 < nbatch) tl.load(v, Xv, bt0);
  asm volatile("griddepcontrol.wait;" ::: "memory");
  EV_STAMP(1);

  // A paused sampler makes surplus graph nodes no-ops (every CTA sees the same phase:
  // the last CTA only changes it after all CTAs have taken their ticket).
  if (a.fin.state != nullptr && __ldcg(&a.fin.state->phase) == PH_PAUSED) return;

  typename Tile::Coef cf;
  tl.load_coef(cf, a.fin.beta, a.fin.p);
  double acc[Tile::SPR][Tile::V] = {};
  double ll_acc = 0.0;

  for (long long bt = bt0; bt < nbatch; bt += nwarps) {
    if (bt != bt0) tl.load(v, Xv, bt);
    typename Tile::Rows rw;
    tl.load_rows(rw, a.y, bt);
    tl.template accumulate<GRAD>(v, rw, cf, ll_acc, acc);
  }

  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // streaming done: let the next grid in
  EV_STAMP(2);

  // ---- CTA reduction
  if constexpr (GRAD) tl.store_grad(acc, red[warp]);
  ll_acc = warp_sum(ll_acc);
  if (lane == 0) redll[warp] = ll_acc;
  __syncthreads();
  double* mypart = a.partials + (size_t)blockIdx.x * (P + 1);
  if (tid == 0) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) s += redll[w];
    mypart[0] = s;
  }
  if constexpr (GRAD) {
    for (int c = tid; c < P; c += kBlock) {
      double s = 0.0;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) s += red[w][c];
      mypart[1 + c] = s;
    }
  }

  // ---- last CTA: sum the CTA partials in a fixed order, then finish
  __threadfence();
  __syncthreads();
  if (tid == 0) s_ticket = atomicAdd(a.ticket, 1u);
  __syncthreads();
  EV_STAMP(3);
  if (s_ticket != gridDim.x - 1) return;
  __threadfence();
  if (a.timeline != nullptr && tid == 0) a.timeline[(size_t)gridDim.x * 4 + 4] = a.timeline[(size_t)gridDim.x * 4 + 2];  // previous evaluation's finish
  EV_STAMP_LAST(0);
  if (tid == 0) *a.ticket = 0u;  // re-arm for the next launch (stream-ordered)
  if (a.fuse_finish) prefetch_finish_inputs(a.fin);

  // warp w sums the partial vectors of CTAs w, w+8, ... (4 independent accumulators keep
  // 4 L2 loads in flight per lane), lanes stride over the columns; then the 8 warp sums are
  // added in warp order.  Fixed order => bit-reproducible for a fixed grid.
  constexpr int NC = GRAD ? P + 1 : 1;
  const int G_ = (int)gridDim.x;
  for (int c = lane; c < NC; c += 32) {
    const double* src = a.partials + c;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    int bb = warp;
    for (; bb + 3 * kWarps < G_; bb += 4 * kWarps) {
      const double v0 = __ldcg(src + (size_t)bb * (P + 1));
      const double v1 = __ldcg(src + (size_t)(bb + kWarps) * (P + 1));
      const double v2 = __ldcg(src + (size_t)(bb + 2 * kWarps) * (P + 1));
      const double v3 = __ldcg(src + (size_t)(bb + 3 * kWarps) * (P + 1));
      s0 += v0; s1 += v1; s2 += v2; s3 += v3;
    }
    for (; bb < G_; bb += kWarps) s0 += __ldcg(src + (size_t)bb * (P + 1));
    red[warp][c] = (s0 + s1) + (s2 + s3);
  }
  __syncthreads();
  for (int c = tid; c <= P; c += kBlock) {
    double s = 0.0;
    if (c < NC) {
#pragma unroll
      for (int w = 0; w < kWarps; ++w) s += red[w][c];
    }
    tot[c] = s;
  }
  __syncthreads();
  EV_STAMP_LAST(1);
  if (a.fuse_finish) {
    finish_eval(a.fin, tot, scratch);
    EV_STAMP_LAST(2);
  } else {
    for (int c = tid; c <= a.fin.p; c += kBlock) a.sums[c] = tot[c];
  }
}

}  // namespace lrb
