// eval_mc_kernel.cuh -- SIMT many-chain variant of the fused kernel: each 8 KB batch
// of X is loaded ONCE into registers and reused for NC chains (coefficient vectors),
// so X traffic per chain drops NC-fold.  This is the path for small chain counts;
// above the chain-count threshold the tcgen05 kernel (eval_tc_kernel.cuh) takes
// over, where eta = X B' and G = R' X become tensor-core contractions.
//
// Each chain's batch goes through BatchTile (eval_kernel.cuh), as in the single-chain kernels;
// the finish step runs in a separate launch with one CTA per chain.  Chain c uses row c of the
// handle's per-chain sums, result and state arrays; the single-chain kernels use row 0.
#pragma once
#include "eval_kernel.cuh"

namespace lrb {

constexpr int kSumStride = kMaxP + 1;   // doubles per chain in the sums array
constexpr int kResStride = kMaxP + 3;   // doubles per chain in the result array

struct EvalMcArgs {
  const void* X;
  const uint8_t* y;
  long long n;
  double* partials;          // [grid][NC][P+1]
  unsigned int* ticket;
  const double* beta_base;   // chain c's coefficients at beta_base + c*beta_stride
  long long beta_stride;     // in doubles
  int chain0, nc_active, p;
  double* sums;              // [C][kSumStride]: [ll, gll] per chain
  const SamplerState* states;  // nullptr for a bare evaluation (else: pause check)
};

template <typename T, int P, int NC>
__global__ void __launch_bounds__(kBlock, 1) eval_mc_kernel(const EvalMcArgs a) {
  using Tile = BatchTile<T, P>;
  using vec = typename Tile::vec;

  __shared__ double red[kWarps][P];
  __shared__ double redll[kWarps];
  __shared__ unsigned int s_ticket;

  if (a.states != nullptr && a.states[a.chain0].phase == PH_PAUSED) return;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const Tile tl(a.n, lane);
  const vec* __restrict__ Xv = reinterpret_cast<const vec*>(a.X);
  const long long nbatch = tl.nbatch;

  typename Tile::Coef cf[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    const int cc = c < a.nc_active ? c : 0;   // surplus slots recompute chain0's first chain (discarded)
    tl.load_coef(cf[c], a.beta_base + (long long)(a.chain0 + cc) * a.beta_stride, a.p);
  }
  double acc[NC][Tile::SPR][Tile::V] = {};
  double ll_acc[NC] = {};

  const long long nwarps = (long long)gridDim.x * kWarps;
  for (long long bt = (long long)blockIdx.x * kWarps + warp; bt < nbatch; bt += nwarps) {
    vec v[Tile::S];
    tl.load(v, Xv, bt);
    typename Tile::Rows rw;
    tl.load_rows(rw, a.y, bt);
#pragma unroll
    for (int c = 0; c < NC; ++c) tl.template accumulate<true>(v, rw, cf[c], ll_acc[c], acc[c]);
  }

  // ---- CTA reduction, one chain at a time through the same scratch
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    tl.store_grad(acc[c], red[warp]);
    const double lw = warp_sum(ll_acc[c]);
    if (lane == 0) redll[warp] = lw;
    __syncthreads();
    double* mypart = a.partials + ((size_t)blockIdx.x * NC + c) * (P + 1);
    if (tid == 0) {
      double s = 0.0;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) s += redll[w];
      mypart[0] = s;
    }
    for (int col = tid; col < P; col += kBlock) {
      double s = 0.0;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) s += red[w][col];
      mypart[1 + col] = s;
    }
    __syncthreads();
  }

  __threadfence();
  __syncthreads();
  if (tid == 0) s_ticket = atomicAdd(a.ticket, 1u);
  __syncthreads();
  if (s_ticket != gridDim.x - 1) return;
  __threadfence();
  if (tid == 0) *a.ticket = 0u;

  // last CTA: fixed-order sum of the CTA partials for each active chain
  for (int idx = tid; idx < a.nc_active * (P + 1); idx += kBlock) {
    const int c = idx / (P + 1), col = idx % (P + 1);
    const double* src = a.partials + (size_t)c * (P + 1) + col;
    const size_t stride = (size_t)NC * (P + 1);
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    int b = 0;
    for (; b + 3 < (int)gridDim.x; b += 4) {
      const double v0 = __ldcg(src + (size_t)b * stride), v1 = __ldcg(src + (size_t)(b + 1) * stride);
      const double v2 = __ldcg(src + (size_t)(b + 2) * stride), v3 = __ldcg(src + (size_t)(b + 3) * stride);
      s0 += v0; s1 += v1; s2 += v2; s3 += v3;
    }
    for (; b < (int)gridDim.x; ++b) s0 += __ldcg(src + (size_t)b * stride);
    if (col <= a.p) a.sums[(size_t)(a.chain0 + c) * kSumStride + col] = (s0 + s1) + (s2 + s3);
  }
}

// Chain c's finish arguments in a finish launch of its own (one CTA per chain): its state,
// coefficients and result row.  Its sums are complete by then (an NCCL allreduce runs between the
// launches), so there is no peer exchange.  false: the chain is paused and its CTA has nothing to do.
__device__ inline bool chain_finish_args(FinishArgs& f, int c, SamplerState* states, const double* beta_base,
                                         long long beta_stride, double* res) {
  f.state = states ? states + c : nullptr;
  if (f.state && f.state->phase == PH_PAUSED) return false;
  f.beta = beta_base + (long long)c * beta_stride;
  f.res = res + (size_t)c * kResStride;
  f.p2p = 0;
  return true;
}

// One CTA per chain: prior + result + sampler update from the reduced sums.  Also the finish of
// a single-chain evaluation whose kernel left it out (row-sharded with NCCL).
__global__ void finish_mc_kernel(FinishArgs base, const double* sums, SamplerState* states,
                                 const double* beta_base, long long beta_stride, double* res) {
  __shared__ double s_sums[kMaxP + 1];
  __shared__ double scratch[kWarps];
  const int c = blockIdx.x;
  FinishArgs f = base;
  if (!chain_finish_args(f, c, states, beta_base, beta_stride, res)) return;
  for (int i = threadIdx.x; i <= f.p; i += kBlock) s_sums[i] = sums[(size_t)c * kSumStride + i];
  __syncthreads();
  finish_eval(f, s_sums, scratch);
}

}  // namespace lrb
