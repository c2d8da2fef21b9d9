// eval_tc_kernel.cuh -- many-chain fused lpost+glp on the 5th-generation tensor
// cores (tcgen05 + TMEM + TMA), FP32-storage mode, "3xTF32" arithmetic.
//
// For C chains the two passes over X become dense contractions (BASELINE.json
// north_star (b), config 4):
//     Eta' [chains x rows] = B [chains x p] . X' [p x rows]          (MMA1)
//     G    [chains x p]    = R [chains x rows] . X [rows x p]        (MMA2)
// with the link functions (softplus / sigmoid residual) applied element-wise in
// between, per (chain, row).  Reference arithmetic replaced: ll fit-numpy.py:23-24,
// glp fit-np-ul.py:45-48, evaluated for 128 chains x 128 rows per tile.
//
// One CTA (768 threads, 1 per SM) owns one group of 128 chains and a strided set of
// 64-row tiles:
//   warp 0      TMA producer: the X tile TWICE (P/32 boxes of 64 rows x 32 floats each):
//               once with the plain 128-byte swizzle (K-major operand of MMA1) and once
//               with the 128B/32B-atom swizzle (the only layout tcgen05 accepts for an
//               MN-major TF32 operand, needed by MMA2), + the 64 y bytes; 3-stage ring.
//   warp 1      MMA issuer (one elected lane issues every tcgen05.mma / commit).
//   warp 2      TMEM allocator (512 columns: eta/R x2, gradient x2, beta hi, beta lo).
//   warps 4-19  epilogue: thread = (chain = TMEM lane, 16-row slice of the tile); four
//               warps per scheduler keep the MUFU pipe (3 ops per element) busy.
//               tcgen05.ld eta, link functions, log-likelihood into a per-thread
//               accumulator (no cross-thread reduction: a thread owns its chain),
//               residual r rounded to TF32 and written back IN PLACE with tcgen05.st,
//               so MMA2 takes R straight from TMEM as its A operand.  beta itself is
//               the TMEM A operand of MMA1 (written once per launch), which leaves
//               shared memory for a 3-stage X ring.
//   warps 20-23 converters: Xl = X - trunc_tf32(X) into the lo buffers; y -> float.
// Precision (SURVEY.md section 7, hard part 4): single-pass TF32 cannot meet 1e-5, so
//   eta = Xh.Bh + Xl.Bh + Xh.Bl   (3 MMAs; the tensor core ignores the 13 low mantissa
//                                   bits of an fp32 operand, so raw X serves as Xh)
//   G   = Rh.Xh + Rh.Xl + Rl.Xh   (the residual is split the same way by the epilogue)
// and the TMEM (fp32) gradient accumulator is flushed into float64 partial sums in
// global memory every kFlush tiles (1024 rows).
//
// X is the K-major B operand of MMA1 (N = rows, K = p) and the MN-major B operand of
// MMA2 (N = p, K = rows): no transpose is ever materialised, TMA delivers both swizzles.
#pragma once
#include <cuda.h>

#include "eval_mc_kernel.cuh"

namespace lrb {

constexpr int kTcThreads = 768;   // 4 control warps + 16 epilogue warps + 4 converter warps
constexpr int kTcSub = 4;         // epilogue warps per TMEM lane quarter (16 rows of a tile each)
constexpr int kTcRows = 64;      // rows per tile (MMA1 N, MMA2 K)
constexpr int kTcChains = 128;   // chains per CTA (MMA M)
constexpr int kFlush = 16;       // tiles (1024 rows) between float64 flushes of the TMEM gradient

struct EvalTcArgs {
  const uint8_t* y;            // n bytes, allocation padded to a multiple of 128
  long long n;
  int ntiles;                  // ceil(n / kTcRows)
  const double* beta_base;     // chain c at beta_base + c*beta_stride (doubles)
  long long beta_stride;
  int C;                       // chains
  int p;
  double* partials;            // [gridDim.x][gridDim.y][P+kTcSub][128]: ll slices, then gll_j
  const SamplerState* states;  // pause check (nullptr for a bare evaluation)
  float* dbg_eta;              // optional: eta of tile 0, [gridDim.y*128][kTcRows]
  long long* dbg_time;         // optional: clock64 stamps of CTA (0,0), [64 tiles][16 events] (development)
};

namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(bar), "r"(parity) : "memory");
  } while (!done);
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// true in exactly one lane of a converged warp (the others fall through)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// D[tmem] (+)= A[smem] . B[smem]
__device__ __forceinline__ void mma_ss(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}"
      ::"r"(d), "l"(a), "l"(b), "r"(idesc), "r"(acc), "r"(0u) : "memory");
}
// D[tmem] (+)= A[tmem] . B[smem]
__device__ __forceinline__ void mma_ts(uint32_t d, uint32_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, {%5, %5, %5, %5}, p;\n\t}"
      ::"r"(d), "r"(a), "l"(b), "r"(idesc), "r"(acc), "r"(0u) : "memory");
}

// Shared-memory matrix descriptor (cute::UMMA::SmemDescriptor), version 1.
// layout_type: 2 = SWIZZLE_128B (K-major operands), 1 = SWIZZLE_128B_BASE32B (MN-major TF32).
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                              uint32_t layout_type = 2u) {
  return (uint64_t)((addr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46) | ((uint64_t)layout_type << 61);
}
// Instruction descriptor (cute::UMMA::InstrDescriptor): TF32 x TF32 -> F32.
__host__ __device__ constexpr uint32_t instr_desc(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
        "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]),
        "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]),
        "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
        "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ float ex2_approx(float x) { float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float lg2_approx(float x) { float r; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float rcp_approx(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float trunc_tf32(float x) { return __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); }

}  // namespace tc

template <int P>
struct TcLayout {
  static constexpr int kStages = 3;
  static constexpr int kBoxes = P / 32;                        // 32-float (128-byte) column boxes per tile
  static constexpr uint32_t kXBoxBytes = kTcRows * 128;        // X box: 64 rows x 128 bytes
  static constexpr uint32_t kXTileBytes = kBoxes * kXBoxBytes;
  // stage: [Xk | Xlk | Xm | Xlm]  (k = SW128 copy for MMA1, m = SW128/32B-atom copy for MMA2)
  static constexpr uint32_t kOffXk = 0, kOffXlk = kXTileBytes, kOffXm = 2 * kXTileBytes, kOffXlm = 3 * kXTileBytes;
  static constexpr uint32_t kStageBytes = 4 * kXTileBytes;
  static constexpr uint32_t kOffY = kStages * kStageBytes;      // raw y bytes, one 128-byte slot per stage
  static constexpr uint32_t kOffYf = kOffY + kStages * 128;     // y as float, 256 bytes per stage
  static constexpr uint32_t kOffBar = kOffYf + kStages * 256;
  static constexpr uint32_t kNumBar = 3 * kStages + 8;
  static constexpr uint32_t kOffTmemPtr = kOffBar + kNumBar * 8;
  static constexpr uint32_t kBytes = kOffTmemPtr + 16;
  static constexpr uint32_t kDynSmem = kBytes + 1024;           // manual 1024-byte alignment slack
  // TMEM columns: eta / R-hi double buffer, R-lo double buffer, gradient double buffer,
  // beta hi / lo (A operand of MMA1)
  static constexpr uint32_t kColD1 = 0, kColRl = 2 * kTcRows, kColG = 4 * kTcRows, kColBh = kColG + 2 * P,
                            kColBl = kColBh + P;
  static constexpr uint32_t kTmemCols = 512;
  static_assert(kColBl + P <= kTmemCols, "TMEM budget");
};

// Link functions for 16 rows of one chain: v holds eta on entry, the TF32 hi part of the
// residual r = y - sigmoid(eta) on exit; w receives the remainder r - hi. Returns the
// log-likelihood contribution sum_i [y*eta - max(eta,0) - log1p(exp(-|eta|))].
template <bool TAIL>
__device__ __forceinline__ float tc_link_chunk(uint32_t (&v)[16], uint32_t (&w)[16], const float4* yf, int valid) {
  using namespace tc;
  const float LOG2E = 1.4426950408889634f, LN2 = 0.6931471805599453f;
  float acc = 0.f;
#pragma unroll
  for (int k4 = 0; k4 < 4; ++k4) {
    const float4 y4 = yf[k4];
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      const int k = k4 * 4 + kk;
      const float eta = __uint_as_float(v[k]);
      const float yv = kk == 0 ? y4.x : kk == 1 ? y4.y : kk == 2 ? y4.z : y4.w;
      const float e = ex2_approx(-fabsf(eta) * LOG2E);
      const float t = 1.0f + e;
      const float inv = rcp_approx(t);                   // sigmoid(|eta|)
      const float lg = lg2_approx(t);
      float term = fmaf(yv, eta, -fmaxf(eta, 0.0f));
      term = fmaf(-LN2, lg, term);
      if (TAIL) term = (k < valid) ? term : 0.0f;
      acc += term;
      const float sig = eta >= 0.0f ? inv : 1.0f - inv;  // e/(1+e) = 1 - 1/(1+e)
      const float r = yv - sig;
      const float rh = trunc_tf32(r);
      v[k] = __float_as_uint(rh);
      w[k] = __float_as_uint(r - rh);
    }
  }
  return acc;
}

#define TC_STAMP(i, ev) do { if (a.dbg_time != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && (i) < 64) a.dbg_time[(i) * 16 + (ev)] = clock64(); } while (0)

template <int P>
__global__ void __launch_bounds__(kTcThreads, 1)
eval_tc_kernel(const __grid_constant__ CUtensorMap xmap_k, const __grid_constant__ CUtensorMap xmap_mn,
               const EvalTcArgs a) {
  using namespace tc;
  using Lay = TcLayout<P>;
  static_assert(P == 64, "tensor-core path: P = 64");
  constexpr int NS = Lay::kStages;
  constexpr int KQ = P / 8;            // MMA1 k-chunks (TF32 UMMA_K = 8)
  constexpr int RQ = kTcRows / 8;      // MMA2 k-chunks

  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));   // generic pointer to the aligned base

  if (a.states != nullptr && a.states[0].phase == PH_PAUSED) return;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int cg = blockIdx.y;                       // chain group
  const int ntiles_mine = (a.ntiles > (int)blockIdx.x) ? (a.ntiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;

  auto bar = [&](int i) { return base + Lay::kOffBar + 8u * i; };
  constexpr int X_FULL = 0, XL_FULL = NS, X_EMPTY = 2 * NS, D1_FULL = 3 * NS, R_FULL = 3 * NS + 2,
                G_FULL = 3 * NS + 4, G_FREE = 3 * NS + 6;

  if (tid == 0) {
    for (int s = 0; s < NS; ++s) {
      mbar_init(bar(X_FULL + s), 1);
      mbar_init(bar(XL_FULL + s), 128);
      mbar_init(bar(X_EMPTY + s), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(bar(D1_FULL + b), 1);
      mbar_init(bar(R_FULL + b), 128 * kTcSub);
      mbar_init(bar(G_FULL + b), 1);
      mbar_init(bar(G_FREE + b), 128 * kTcSub);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(base + Lay::kOffTmemPtr), "r"(Lay::kTmemCols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(gen + Lay::kOffTmemPtr);

  const bool is_epi = warp >= 4 && warp < 4 + 4 * kTcSub;
  const int quarter = warp & 3;                     // TMEM lane quarter this warp may access
  const int sub = (warp - 4) >> 2;                  // epilogue: which 16 rows of a tile / which 16 G columns
  const int ci = quarter * 32 + lane;               // chain within the group == TMEM lane
  const uint32_t lane_addr = ((uint32_t)(quarter * 32)) << 16;

  // beta of this chain group -> TMEM (A operand of MMA1): epilogue warps sub 0,1 write the
  // TF32 hi part (32 columns each), sub 2,3 the remainder beta - hi
  if (is_epi) {
    const int chain = cg * kTcChains + ci;
    const double* bsrc = a.beta_base + (long long)chain * a.beta_stride;
    const bool hi = sub < 2;
    const int c0 = (sub & 1) * 32;
    uint32_t v[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) {
      const int col = c0 + k;
      const double b = (chain < a.C && col < a.p) ? bsrc[col] : 0.0;
      const float bh = trunc_tf32((float)b);
      v[k] = __float_as_uint(hi ? bh : (float)(b - (double)bh));
    }
    tmem_st32(tmem + lane_addr + (hi ? Lay::kColBh : Lay::kColBl) + c0, v);
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  if (warp == 0) {
    // ===================== TMA producer
    if (lane == 0) {
      for (int i = 0; i < ntiles_mine; ++i) {
        const int s = i % NS;
        const int tile = blockIdx.x + i * gridDim.x;
        mbar_wait(bar(X_EMPTY + s), ((i / NS) & 1) ^ 1);
        TC_STAMP(i, 0);
        mbar_expect_tx(bar(X_FULL + s), 2u * Lay::kXTileBytes + (uint32_t)kTcRows);
        const uint32_t dst = base + s * Lay::kStageBytes;
#pragma unroll
        for (int b = 0; b < Lay::kBoxes; ++b) {
          tma_load_2d(dst + Lay::kOffXk + b * Lay::kXBoxBytes, &xmap_k, bar(X_FULL + s), 32 * b, tile * kTcRows);
          tma_load_2d(dst + Lay::kOffXm + b * Lay::kXBoxBytes, &xmap_mn, bar(X_FULL + s), 32 * b, tile * kTcRows);
        }
        bulk_load(base + Lay::kOffY + s * 128, a.y + (long long)tile * kTcRows, (uint32_t)kTcRows, bar(X_FULL + s));
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer.  The whole warp stays converged (so descriptors live in
    // uniform registers); one elected lane issues the tcgen05.mma / commit instructions.
    constexpr uint32_t idesc1 = instr_desc(kTcChains, kTcRows, 0, 0);   // A = beta (TMEM), B = X rows (K-major)
    constexpr uint32_t idesc2 = instr_desc(kTcChains, P, 0, 1);         // A = R (TMEM), B = X (MN-major)
    auto issue_mma2 = [&](int j) {
      const int s = j % NS, b = j & 1, g = j / kFlush, gb = g & 1;
      mbar_wait(bar(R_FULL + b), (j >> 1) & 1);
      const bool first_of_group = (j % kFlush) == 0;
      if (first_of_group && g >= 2) mbar_wait(bar(G_FREE + gb), ((g >> 1) - 1) & 1);
      tc_fence_after();
      if (lane == 0) TC_STAMP(j, 9);
      const uint32_t xs = base + s * Lay::kStageBytes;
      // MN-major, 128B swizzle with 32-byte atoms: 8 rows (K) of 128 bytes per k-chunk;
      // LBO = stride between 32-column (MN) groups, SBO = stride between 4-row (K) groups
      const uint64_t dm = smem_desc(xs + Lay::kOffXm, Lay::kXBoxBytes, 512u, 1u);
      const uint64_t dlm = smem_desc(xs + Lay::kOffXlm, Lay::kXBoxBytes, 512u, 1u);
      const uint32_t rh = tmem + Lay::kColD1 + b * kTcRows, rl = tmem + Lay::kColRl + b * kTcRows;
      const uint32_t d_t = tmem + Lay::kColG + gb * P;
      const uint32_t acc0 = first_of_group ? 0u : 1u;
      if (elect_one()) {
#pragma unroll
        for (int q = 0; q < RQ; ++q) mma_ts(d_t, rh + q * 8, dm + (uint64_t)(q * 64), idesc2, q == 0 ? acc0 : 1u);
#pragma unroll
        for (int q = 0; q < RQ; ++q) mma_ts(d_t, rh + q * 8, dlm + (uint64_t)(q * 64), idesc2, 1u);
#pragma unroll
        for (int q = 0; q < RQ; ++q) mma_ts(d_t, rl + q * 8, dm + (uint64_t)(q * 64), idesc2, 1u);
        tc_commit(bar(X_EMPTY + s));                 // stage s and eta/R buffer b are free again
        if ((j % kFlush) == kFlush - 1 || j == ntiles_mine - 1) tc_commit(bar(G_FULL + gb));
      }
      __syncwarp();
      if (lane == 0) TC_STAMP(j, 10);
    };
    for (int i = 0; i < ntiles_mine; ++i) {
      const int s = i % NS, b = i & 1;
      mbar_wait(bar(X_FULL + s), (i / NS) & 1);
      mbar_wait(bar(XL_FULL + s), (i / NS) & 1);
      tc_fence_after();
      if (lane == 0) TC_STAMP(i, 3);
      const uint32_t xs = base + s * Lay::kStageBytes;
      const uint64_t dk = smem_desc(xs + Lay::kOffXk, 16u, 1024u);
      const uint64_t dlk = smem_desc(xs + Lay::kOffXlk, 16u, 1024u);
      const uint32_t d1 = tmem + Lay::kColD1 + b * kTcRows;
      const uint32_t bh = tmem + Lay::kColBh, bl = tmem + Lay::kColBl;
      if (elect_one()) {
        // eta' = Bh.Xh' + Bh.Xl' + Bl.Xh'; k-chunk q lives in box q/4 at byte (q%4)*32 of the 128B row
#pragma unroll
        for (int q = 0; q < KQ; ++q)
          mma_ts(d1, bh + q * 8, dk + (uint64_t)(((q >> 2) * Lay::kXBoxBytes + (q & 3) * 32u) >> 4), idesc1, q == 0 ? 0u : 1u);
#pragma unroll
        for (int q = 0; q < KQ; ++q)
          mma_ts(d1, bh + q * 8, dlk + (uint64_t)(((q >> 2) * Lay::kXBoxBytes + (q & 3) * 32u) >> 4), idesc1, 1u);
#pragma unroll
        for (int q = 0; q < KQ; ++q)
          mma_ts(d1, bl + q * 8, dk + (uint64_t)(((q >> 2) * Lay::kXBoxBytes + (q & 3) * 32u) >> 4), idesc1, 1u);
        tc_commit(bar(D1_FULL + b));
      }
      __syncwarp();
      if (lane == 0) TC_STAMP(i, 4);
      if (i > 0) issue_mma2(i - 1);
    }
    if (ntiles_mine > 0) issue_mma2(ntiles_mine - 1);
  } else if (warp >= 4 + 4 * kTcSub) {
    // ===================== converters: Xl = X - trunc_tf32(X) (same swizzled offsets), y -> float
    const int ct = tid - 32 * (4 + 4 * kTcSub);
    for (int i = 0; i < ntiles_mine; ++i) {
      const int s = i % NS;
      mbar_wait(bar(X_FULL + s), (i / NS) & 1);
      if (ct == 0) TC_STAMP(i, 1);
      if (ct < kTcRows)
        reinterpret_cast<float*>(gen + Lay::kOffYf + s * 256)[ct] = (float)(gen + Lay::kOffY + s * 128)[ct];
      // both swizzled copies (the offsets are swizzle-agnostic); 8 independent 16-byte loads in
      // flight per thread: this conversion sits on the stage's critical path
#pragma unroll
      for (int set = 0; set < 2; ++set) {
        const float4* src = reinterpret_cast<const float4*>(gen + s * Lay::kStageBytes + (set ? Lay::kOffXm : Lay::kOffXk));
        float4* dst = reinterpret_cast<float4*>(gen + s * Lay::kStageBytes + (set ? Lay::kOffXlm : Lay::kOffXlk));
        constexpr int kPer = (int)(Lay::kXTileBytes / 16) / 128;   // chunks per thread per copy (8 at P = 64)
        float4 x[kPer];
#pragma unroll
        for (int u = 0; u < kPer; ++u) x[u] = src[ct + u * 128];
#pragma unroll
        for (int u = 0; u < kPer; ++u) {
          float4 l;
          l.x = x[u].x - trunc_tf32(x[u].x); l.y = x[u].y - trunc_tf32(x[u].y);
          l.z = x[u].z - trunc_tf32(x[u].z); l.w = x[u].w - trunc_tf32(x[u].w);
          dst[ct + u * 128] = l;
        }
      }
      fence_async_smem();
      mbar_arrive(bar(XL_FULL + s));
      if (ct == 0) TC_STAMP(i, 2);
    }
  } else if (is_epi) {
    // ===================== epilogue: thread = (chain, 16-row slice of the tile)
    double ll_acc = 0.0;
    constexpr int PR = P + kTcSub;   // partial rows: kTcSub log-likelihood slots, then the gradient
    double* part = a.partials + ((size_t)blockIdx.x * gridDim.y + cg) * (size_t)PR * kTcChains;
    // flush gradient group g (TMEM fp32 accumulator) into the float64 partial sums;
    // this thread owns 16 of the P columns of its chain
    auto flush = [&](int g) {
      const int gb = g & 1;
      mbar_wait(bar(G_FULL + gb), (g >> 1) & 1);
      tc_fence_after();
      uint32_t gv[16];
      tmem_ld16(tmem + lane_addr + Lay::kColG + gb * P + sub * 16, gv);
      tc_fence_before();
      mbar_arrive(bar(G_FREE + gb));
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        double* dst = part + (size_t)(kTcSub + sub * 16 + k) * kTcChains + ci;
        const double add = (double)__uint_as_float(gv[k]);
        *dst = (g == 0) ? add : (*dst + add);
      }
    };
    for (int i = 0; i < ntiles_mine; ++i) {
      const int s = i % NS, b = i & 1;
      const long long row0 = (long long)(blockIdx.x + (long long)i * gridDim.x) * kTcRows + sub * 16;
      mbar_wait(bar(D1_FULL + b), (i >> 1) & 1);
      tc_fence_after();
      if (tid == 128) TC_STAMP(i, 5);
      const float4* yf = reinterpret_cast<const float4*>(gen + Lay::kOffYf + s * 256 + sub * 64);
      uint32_t v[16], w[16];
      const uint32_t taddr = tmem + lane_addr + Lay::kColD1 + b * kTcRows + sub * 16;
      tmem_ld16(taddr, v);
      if (tid == 128) TC_STAMP(i, 6);
      if (a.dbg_eta != nullptr && blockIdx.x == 0 && i == 0) {
#pragma unroll
        for (int k = 0; k < 16; ++k) a.dbg_eta[(size_t)(cg * kTcChains + ci) * kTcRows + sub * 16 + k] = __uint_as_float(v[k]);
      }
      float ll_tile;
      if (row0 + 16 <= a.n) ll_tile = tc_link_chunk<false>(v, w, yf, 16);
      else ll_tile = tc_link_chunk<true>(v, w, yf, (int)max(0ll, a.n - row0));
      if (tid == 128) TC_STAMP(i, 7);
      tmem_st16(taddr, v);
      tmem_st16(tmem + lane_addr + Lay::kColRl + b * kTcRows + sub * 16, w);
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(bar(R_FULL + b));
      if (tid == 128) TC_STAMP(i, 8);
      ll_acc += (double)ll_tile;
      if ((i % kFlush) == 0 && i > 0) flush(i / kFlush - 1);   // deferred: the group's MMA2s are long done
    }
    if (ntiles_mine > 0) flush((ntiles_mine - 1) / kFlush);
    part[(size_t)sub * kTcChains + ci] = ll_acc;
    if (ntiles_mine == 0) {
      for (int k = 0; k < 16; ++k) part[(size_t)(kTcSub + sub * 16 + k) * kTcChains + ci] = 0.0;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(Lay::kTmemCols));
  }
}

// One CTA per chain: sum the per-CTA float64 partials over row CTAs in a fixed order,
// then the common finish (prior, result, sampler update).
// partials: [row_ctas][groups][P+kTcSub][128]; rows 0..kTcSub-1 = log-likelihood slices, then gll_j
__global__ void finish_tc_kernel(FinishArgs base, const double* partials, int row_ctas, int groups, int P,
                                 SamplerState* states, const double* beta_base, long long beta_stride,
                                 double* res) {
  __shared__ double s_sums[kMaxP + 1];
  __shared__ double scratch[kWarps];
  const int c = blockIdx.x;
  FinishArgs f = base;
  if (!chain_finish_args(f, c, states, beta_base, beta_stride, res)) return;
  const int cg = c / kTcChains, ci = c % kTcChains;
  for (int j = threadIdx.x; j <= f.p; j += kBlock) {
    double s = 0.0;
    for (int bx = 0; bx < row_ctas; ++bx) {
      const double* pb = partials + ((size_t)bx * groups + cg) * (size_t)(P + kTcSub) * kTcChains;
      if (j == 0) {
        for (int q = 0; q < kTcSub; ++q) s += pb[(size_t)q * kTcChains + ci];
      } else {
        s += pb[(size_t)(kTcSub - 1 + j) * kTcChains + ci];
      }
    }
    s_sums[j] = s;
  }
  __syncthreads();
  finish_eval(f, s_sums, scratch);
}

}  // namespace lrb
