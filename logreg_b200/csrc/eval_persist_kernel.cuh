// eval_persist_kernel.cuh -- the fused lpost+glp kernel in "drive mode": ONE cooperative
// launch runs a whole sequence of evaluations (BASELINE.json north_star (c): "CUDA Graphs or a
// persistent kernel so no per-iteration host round-trip remains").
//
// Each row batch goes through BatchTile of eval_kernel.cuh (see there for the lane mapping and
// the reference lines: ll Python/fit-numpy.py:23-24, glp Python/fit-np-ul.py:45-48), as in the
// static kernel; what changes is how the work is handed out and how one evaluation hands over
// to the next:
//
//   * Dynamic row-batch scheduling.  Per-SM streaming rates differ (measured: the slowest 48
//     CTAs of a 296-CTA grid finish 15-22 % after the median on one box, 4 % on another), so
//     with a static split the pass lasts as long as the slowest SM.  Here each warp owns a static
//     prefix of its share (no atomics, first batch prefetchable before beta is known) and takes
//     the remaining batches one at a time from a per-CTA pool in shared memory; the pool is
//     refilled in chunks of 8 batches from one global counter, two chunks ahead of use.  (Claiming
//     every batch straight from the global counter was measured at 4.7 TB/s: ~850 M same-address
//     atomics per second is more than L2 delivers.)  Every SM streams until X is exhausted.
//   * The CTA sums go into a (p+1)-vector with fire-and-forget red.global.add.f64; the last CTA
//     (atomic ticket) reads-and-zeroes it, runs finish_eval (fused peer-memory allreduce, prior,
//     sampler update -> the next evaluation point) and publishes an epoch flag with
//     st.release.gpu.  The order of the floating-point additions therefore depends on timing:
//     results agree with the static kernel to rounding (tests: 1e-10 / 1e-5), not bit for bit.
//     LRB_DETERMINISTIC=1 selects the static, fixed-order kernel of eval_kernel.cuh instead.
//   * No kernel boundary between evaluations: CTAs that finish streaming loop straight into the
//     next evaluation, fetch their first X batch (X is immutable) and only then spin on the
//     epoch flag, so HBM stays busy while the last CTA is in its serial tail.
//
// All CTAs must be co-resident (they wait for each other): the host launches
// min(SMs x occupancy, needed) CTAs with cudaLaunchCooperativeKernel.  Every wait is bounded
// (%globaltimer) and raises an abort flag instead of hanging the GPU.
#pragma once
#include "eval_kernel.cuh"

namespace lrb {

struct PersistArgs {
  unsigned long long* epoch;   // evaluations completed by drive-mode launches on this handle (monotone)
  unsigned int* work;          // [2] dynamic batch counters by evaluation parity; zero at rest
  double* acc;                 // [kMaxP+1] running sums [ll, gll]; zero at rest
  int* abort;                  // raised when a wait exceeded spin_limit_ns
  int n_evals;                 // evaluations this launch performs
  int static_eighths;          // share of each warp's batches that is assigned statically, in 1/8 (0..8)
  long long spin_limit_ns;
};

constexpr int kPoolChunk = 8;    // batches per global claim (one per warp of a CTA)
constexpr int kPoolSlots = 16;   // chunk descriptors per CTA: the producer runs at most 4 chunks ahead of the draws, so a
                                 // slot is recycled only 12 chunks (96 draws of this CTA) after its last draw was handed out

__device__ __forceinline__ unsigned long long ld_acquire_gpu(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// Spin until *epoch >= want.  false: the wait was abandoned (abort raised by this or another warp).
__device__ __forceinline__ bool wait_epoch(const unsigned long long* epoch, unsigned long long want, int* abort,
                                           long long limit_ns) {
  unsigned int spins = 0;
  long long t_start = 0;
  for (;;) {
    if (ld_acquire_gpu(epoch) >= want) return true;
    if ((++spins & 0x3ffu) == 0) {
      if (__ldcg(abort) != 0) return false;
      const long long now = global_ns();
      if (t_start == 0) t_start = now;
      else if (now - t_start > limit_ns) { *abort = 1; __threadfence(); return false; }
    }
  }
}

template <typename T, int P, bool GRAD>
__global__ void __launch_bounds__(kBlock, 2) eval_persist_kernel(const EvalArgs a, const PersistArgs pa) {
  using Tile = BatchTile<T, P>;
  using vec = typename Tile::vec;

  __shared__ double red[kWarps][P + 1];   // [.][0] = log-likelihood, [.][1+c] = gradient column c
  __shared__ double tot[P + 1];
  __shared__ double scratch[kWarps];
  __shared__ unsigned int s_ticket;
  // per-CTA batch pool: draw c (shared counter) is slot c%8 of chunk c/8; chunk k's first batch
  // (relative to dyn0) is published in s_base[k%16] with tag k+1
  __shared__ unsigned int s_claims;
  __shared__ volatile unsigned int s_base[kPoolSlots], s_tag[kPoolSlots];
  __shared__ volatile unsigned int s_last;   // first exhausted chunk of this CTA's pool (0xffffffff: none yet)
  // Every CTA keeps a working copy of the chain state (and of the prior scales): whichever CTA
  // turns out to be the last of an evaluation runs the sampler update out of shared memory, with
  // the random draws already computed while X was streaming.
  __shared__ SamplerState s_st;
  __shared__ double s_ps[kMaxP], s_lps[kMaxP];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) { s_claims = 0u; s_last = 0xffffffffu; s_st.cache_has = 0; s_st.cache_t = -1; }
  if (tid < kPoolSlots) s_tag[tid] = 0u;
  for (int j = tid; j < a.fin.p; j += kBlock) { s_ps[j] = a.fin.pscale[j]; s_lps[j] = a.fin.log_pscale[j]; }
  __syncthreads();
  const Tile tl(a.n, lane);
  const vec* __restrict__ Xv = reinterpret_cast<const vec*>(a.X);
  const long long nbatch = tl.nbatch;
  const long long nwarps = (long long)gridDim.x * kWarps;
  const long long bt0 = (long long)blockIdx.x * kWarps + warp;
  // static prefix: KS batches per warp (strided), the rest is claimed dynamically from dyn0 on
  const long long KS = (nbatch / nwarps) * pa.static_eighths / 8;
  const long long dyn0 = KS * nwarps;

  // stable at launch: nobody can complete evaluation 0 before every warp has passed this read
  const unsigned long long e0 = ld_acquire_gpu(pa.epoch);

  vec v[Tile::S];

  for (int e = 0; e < pa.n_evals; ++e) {
    unsigned int* work = pa.work + ((e0 + (unsigned long long)e) & 1ull);
    EV_STAMP(0);
    long long cur = bt0;
    bool loaded = false;
    if (KS > 0) { tl.load(v, Xv, cur); loaded = true; }   // X is immutable: fetch before beta is known

    if (e > 0 && !wait_epoch(pa.epoch, e0 + (unsigned long long)e, pa.abort, pa.spin_limit_ns)) return;
    EV_STAMP(1);
    if (a.fin.state != nullptr && __ldcg(&a.fin.state->phase) == PH_PAUSED) return;   // same answer in every CTA
    // Pool refill, single producer: lane 0 of warp 0 issues every global claim of this CTA (so the
    // chunk bases are monotone: the first exhausted chunk ends the pool) and publishes a claim on
    // its next visit, by which time the atomic has long returned.  It keeps the pool up to four
    // chunks ahead of the draws.  The first visit comes after the last possible exit above, so
    // the global counter is never left dirty.
    unsigned int issued = 0u, npend = 0u, pc0 = 0u, pb0 = 0u, pc1 = 0u, pb1 = 0u;
    const unsigned int span = (unsigned int)(nbatch - dyn0);
    auto publish = [&](unsigned int chunk, unsigned int base) {
      s_base[chunk % kPoolSlots] = base;
      __threadfence_block();
      s_tag[chunk % kPoolSlots] = chunk + 1u;
      if (base >= span && s_last == 0xffffffffu) s_last = chunk;
    };
    auto producer_visit = [&]() {   // warp 0, lane 0 only
      if (npend >= 1u) publish(pc0, pb0);
      if (npend == 2u) publish(pc1, pb1);
      npend = 0u;
      const unsigned int target = (s_last != 0xffffffffu) ? 0u : *reinterpret_cast<volatile unsigned int*>(&s_claims) / kPoolChunk + 4u;
      if (issued < target) { pb0 = atomicAdd(work, (unsigned int)kPoolChunk); pc0 = issued++; npend = 1u; }
      if (issued < target) { pb1 = atomicAdd(work, (unsigned int)kPoolChunk); pc1 = issued++; npend = 2u; }
    };
    auto next_dynamic = [&]() -> long long {
      unsigned int c = 0u;
      if (lane == 0) c = atomicAdd(&s_claims, 1u);
      c = __shfl_sync(0xffffffffu, c, 0);
      const unsigned int chunk = c / kPoolChunk, slot = c % kPoolChunk;
      unsigned int base = 0xffffffffu;   // exhausted unless a published chunk says otherwise
      if (lane == 0) {
        for (unsigned int spins = 0;; ++spins) {
          if (s_tag[chunk % kPoolSlots] == chunk + 1u) { __threadfence_block(); base = s_base[chunk % kPoolSlots]; break; }
          if (chunk >= s_last) break;
          if (warp == 0) producer_visit();   // the producer must not wait for itself
          if (spins > (1u << 28)) { *pa.abort = 1; break; }   // never seen; a bug here must not hang the GPU
        }
      }
      base = __shfl_sync(0xffffffffu, base, 0);
      return base >= span ? nbatch : dyn0 + (long long)base + (long long)slot;
    };
    if (tid == 0) producer_visit();
    if (a.fin.state != nullptr) {   // working copy + draws; visible to the tail through the reduction's barrier
      state_load(&s_st, a.fin.state);
      sampler_precompute_draws(&s_st, a.fin.state);
    }

    typename Tile::Coef cf;
    tl.load_coef(cf, a.fin.beta, a.fin.p);
    double acc[Tile::SPR][Tile::V] = {};
    double ll_acc = 0.0;

    long long ks = 0;
    if (KS == 0) cur = next_dynamic();
    while (cur < nbatch) {
      if (!loaded) tl.load(v, Xv, cur);
      loaded = false;
      // the index of the batch after this one, while the loads are in flight: static stride as
      // long as the prefix lasts, then a draw from the pool
      ++ks;
      if (tid == 0) producer_visit();
      const long long nxt = ks < KS ? bt0 + ks * nwarps : next_dynamic();
      typename Tile::Rows rw;
      tl.load_rows(rw, a.y, cur);
      tl.template accumulate<GRAD>(v, rw, cf, ll_acc, acc);
      cur = nxt;
    }
    // The producer may leave the loop only once the END of the pool is published.  It normally gets
    // here by drawing from a chunk that is already marked exhausted, but when the dynamic region is
    // not a multiple of 8 batches one chunk straddles the end of X, and an out-of-range slot of THAT
    // chunk ends the loop with the next (exhausted) chunk possibly still unpublished -- the other warps
    // of this CTA would wait for it forever (found with tests/test_pool_model.py).  A few more visits
    // publish it: every claim made from here on lies beyond the end.
    if (tid == 0) {
      for (int i = 0; i < 64 && s_last == 0xffffffffu; ++i) producer_visit();
    }
    EV_STAMP(2);

    // ---- CTA reduction -> running sums
    if constexpr (GRAD) tl.store_grad(acc, red[warp] + 1);
    ll_acc = warp_sum(ll_acc);
    if (lane == 0) red[warp][0] = ll_acc;
    __syncthreads();
    constexpr int NC = GRAD ? P + 1 : 1;
    for (int c = tid; c < NC; c += kBlock) {
      double s = 0.0;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) s += red[w][c];
      atomicAdd(pa.acc + c, s);   // result unused: red.global.add.f64
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) { s_ticket = atomicAdd(a.ticket, 1u); s_claims = 0u; s_last = 0xffffffffu; }   // every warp is past its last claim
    if (tid < kPoolSlots) s_tag[tid] = 0u;
    __syncthreads();
    EV_STAMP(3);
    if (s_ticket != gridDim.x - 1) continue;   // on to the next evaluation: prefetch, then wait for its beta

    // ---- last CTA of this evaluation
    __threadfence();
    if (a.timeline != nullptr && tid == 0) a.timeline[(size_t)gridDim.x * 4 + 4] = a.timeline[(size_t)gridDim.x * 4 + 2];
    EV_STAMP_LAST(0);
    for (int c = tid; c <= P; c += kBlock) {
      double s = 0.0;
      if (c < NC)
        s = __longlong_as_double((long long)atomicExch(reinterpret_cast<unsigned long long*>(pa.acc + c), 0ull));
      tot[c] = s;
    }
    if (tid == 0) { *a.ticket = 0u; *work = 0u; }   // every warp of every CTA is past its last claim
    __syncthreads();
    EV_STAMP_LAST(1);
    if (a.fuse_finish) {
      if (a.fin.state != nullptr) finish_eval(a.fin, tot, scratch, &s_st, s_st.beta_in, s_ps, s_lps);
      else finish_eval(a.fin, tot, scratch, nullptr, a.fin.beta, s_ps, s_lps);
      if (a.fin.state != nullptr) {
        __syncthreads();
        state_store(a.fin.state, &s_st);   // the next evaluation point and the chain state go home
      }
    } else {
      for (int c = tid; c <= a.fin.p; c += kBlock) a.sums[c] = tot[c];
    }
    __syncthreads();
    if (tid == 0) {
      __threadfence();
      st_release_gpu(pa.epoch, e0 + (unsigned long long)e + 1ull);   // beta of evaluation e+1 is published
    }
    EV_STAMP_LAST(2);
  }
}

}  // namespace lrb
