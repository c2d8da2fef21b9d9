// lrb_api.cu -- the C ABI of include/logreg_b200.h: handle, data binding,
// evaluation, on-device sampler runs (CUDA-graph driven) and the row-sharded
// communicators.  Host C++ only orchestrates; all arithmetic is in the kernels of
// eval_kernel.cuh / sampler.cuh / data.cuh.  There is no CPU fallback anywhere.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/logreg_b200.h"
#include "data.cuh"
#include "eval_kernel.cuh"
#include "eval_mc_kernel.cuh"
#include "eval_persist_kernel.cuh"
#include "eval_tc_kernel.cuh"
#include "loo.cuh"
#include "newton.cuh"
#include "predictive.cuh"
#include "sampler.cuh"

using namespace lrb;

namespace {

thread_local std::string g_err;  // errors raised without a handle

// ---- NCCL through dlopen: the library must load (and every single-GPU path must
// work) on a box where libnccl is not on the loader path.
struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t,
                            cudaStream_t) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
NcclApi g_nccl;

bool load_nccl(const char* path, std::string& err) {
  if (g_nccl.lib) return true;
  const char* cands[] = {path, "libnccl.so.2", "libnccl.so"};
  void* lib = nullptr;
  for (const char* c : cands) {
    if (!c || !*c) continue;
    lib = dlopen(c, RTLD_NOW | RTLD_GLOBAL);
    if (lib) break;
  }
  if (!lib) { err = std::string("cannot dlopen libnccl: ") + dlerror(); return false; }
  g_nccl.GetUniqueId = (decltype(g_nccl.GetUniqueId))dlsym(lib, "ncclGetUniqueId");
  g_nccl.CommInitRank = (decltype(g_nccl.CommInitRank))dlsym(lib, "ncclCommInitRank");
  g_nccl.AllReduce = (decltype(g_nccl.AllReduce))dlsym(lib, "ncclAllReduce");
  g_nccl.CommDestroy = (decltype(g_nccl.CommDestroy))dlsym(lib, "ncclCommDestroy");
  g_nccl.GetErrorString = (decltype(g_nccl.GetErrorString))dlsym(lib, "ncclGetErrorString");
  if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllReduce || !g_nccl.CommDestroy) {
    err = "libnccl is missing required symbols";
    return false;
  }
  g_nccl.lib = lib;
  return true;
}

using EvalFn = void (*)(const EvalArgs);
using EvalMcFn = void (*)(const EvalMcArgs);
using EvalPersistFn = void (*)(const EvalArgs, const PersistArgs);
constexpr int kMcChains = 4;   // chains sharing one X batch in the SIMT many-chain kernel

struct KernelChoice {
  EvalFn grad = nullptr, nograd = nullptr;
  EvalMcFn mc = nullptr;
  EvalPersistFn drive = nullptr, drive_nograd = nullptr;   // drive mode: dynamic scheduling, many evaluations per launch
  int rows_per_batch = 0;
};

template <typename T, int P>
KernelChoice choice() {
  KernelChoice k;
  k.grad = eval_kernel<T, P, true>;
  k.nograd = eval_kernel<T, P, false>;
  k.mc = eval_mc_kernel<T, P, kMcChains>;
  k.drive = eval_persist_kernel<T, P, true>;
  k.drive_nograd = eval_persist_kernel<T, P, false>;
  k.rows_per_batch = 512 * Chunk<T>::V / P;
  return k;
}

// f(std::integral_constant<int, P>()) for a padded width P the kernels are instantiated for;
// false for any other width.
template <typename F>
bool with_width(int P, F&& f) {
  switch (P) {
    case 8: f(std::integral_constant<int, 8>()); return true;
    case 16: f(std::integral_constant<int, 16>()); return true;
    case 32: f(std::integral_constant<int, 32>()); return true;
    case 64: f(std::integral_constant<int, 64>()); return true;
    case 128: f(std::integral_constant<int, 128>()); return true;
    case 256: f(std::integral_constant<int, 256>()); return true;
  }
  return false;
}

int pad_p(int p) {
  int P = 8;
  while (P < p) P <<= 1;
  return P;
}

}  // namespace

struct lrb_handle {
  int device = 0;
  int sms = 0;
  cudaStream_t own_stream = nullptr, stream = nullptr;
  std::string err;

  // data
  void* X = nullptr;
  uint8_t* y = nullptr;
  long long n = 0;
  int p = 0, P = 0, mode = 0;
  double* d_pscale = nullptr;     // [kMaxP]
  double* d_logps = nullptr;      // [kMaxP]
  bool bound = false;

  // evaluation scratch
  KernelChoice kern;
  int grid = 0, grid_nograd = 0;
  double* partials = nullptr;
  unsigned int* ticket = nullptr;
  double* pinned = nullptr; // host staging [2*kMaxP+8]
  // drive mode (eval_persist_kernel.cuh): one block of device words [epoch u64][work u32 x2][abort i32][pad][acc f64 x (kMaxP+1)]
  void* drive_mem = nullptr;
  unsigned long long* epoch = nullptr;
  unsigned int* work = nullptr;
  int* drive_abort = nullptr;
  double* drive_acc = nullptr;
  bool capturing = false;     // inside build_graph's stream capture: static kernels only
  bool chain_live_partial = false;    // launch_run: at least one drive chunk of the current run is enqueued
  bool drive_launch_failed = false;   // a cooperative launch was refused: static kernel from then on
  bool drive_multi = false;   // experimental: drive mode on row-sharded handles (LRB_DRIVE_MULTI=1)
  bool drive = true;          // LRB_DRIVE=0 / LRB_DETERMINISTIC=1: static fixed-order kernel, one launch per evaluation
  int grid_drive = 0, grid_drive_nograd = 0;
  long long drive_spin_ns = 20ll * 1000 * 1000 * 1000;
  int drive_static_eighths = -1;  // -1: chosen per shape in configure(); LRB_DRIVE_STATIC overrides

  // sampler
  double* d_scale = nullptr;  // [kMaxP]
  double* d_out = nullptr; size_t out_cap = 0;
  double* d_z = nullptr; size_t z_cap = 0;
  double* d_u = nullptr; size_t u_cap = 0;
  double* d_mom_mean = nullptr; size_t mom_mean_cap = 0;   // [C][p] running means (LRB_RUN_MOMENTS)
  double* d_mom_m2 = nullptr; size_t mom_m2_cap = 0;       // [C][p][p] running cross-moments
  bool run_moments = false, run_no_samples = false;
  bool chain_moments = false;                              // the live chain carries moments
  bool chain_live = false;    // a paused chain exists that a run may continue
  int chain_kind = -1;
  bool run_armed = false;
  int run_kind = 0, run_l = 1;
  bool run_want_grad = true;
  bool pending_init_eval = false;
  bool run_consumed = false;
  const double* run_dz = nullptr;
  const double* run_du = nullptr;
  long long run_thin = 0, run_iters = 0;
  lrb_sampler_params run_params{};
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t gexec = nullptr;
  int graph_nodes = 0;
  bool graph_grad = true;

  // communicator
  int world = 1, rank = 0, comm = 0;
  ncclComm_t nccl = nullptr;
  double* mailbox = nullptr;               // [2][kMaxRanks][kMailStride]
  unsigned long long* flags = nullptr;     // [2][kMaxRanks], directly after the mailbox
  unsigned long long* seq = nullptr;
  int* comm_error = nullptr;
  void* peer_base[kMaxRanks] = {};
  bool peer_open[kMaxRanks] = {};
  long long p2p_timeout_ns = 60ll * 1000 * 1000 * 1000;

  // per-chain arrays of chain_cap rows; a single chain or evaluation uses row 0
  SamplerState* states = nullptr;
  double* sums = nullptr;   // [C][kSumStride]
  double* res = nullptr;    // [C][kResStride]
  double* beta = nullptr;   // [C][kMaxP] staging for host coefficient / init matrices
  int chain_cap = 0;
  int run_C = 1, chain_C = 1, graph_C = 1;
  int grid_mc = 0;
  long long graph_kl_per_replay = 0, graph_el_per_replay = 0;
  // tensor-core many-chain path (fp32 mode, P = 32 or 64)
  bool tc_ok = false;
  CUtensorMap xmap_k{}, xmap_mn{};
  double* partials_tc = nullptr; size_t partials_tc_cap = 0;
  float* dbg_eta = nullptr;
  long long* dbg_time = nullptr;
  int tc_min_chains = 12;   // measured crossover, profiles/r1_many_chain_threshold.txt
  bool pdl = true;
  bool l2_persist = true;

  long long* timeline = nullptr;   // lrb_debug_timeline: per-CTA %globaltimer stamps of the latest evaluation

  long long kernel_launches = 0, eval_launches = 0;
};

namespace {

constexpr size_t kMailDoubles = (size_t)2 * kMaxRanks * kMailStride;
constexpr size_t kMailBytes = kMailDoubles * sizeof(double) + (size_t)2 * kMaxRanks * sizeof(unsigned long long);

int fail(lrb_handle* h, int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (h) h->err = buf; else g_err = buf;
  return code;
}

#define CK(h, call)                                                                       \
  do {                                                                                    \
    cudaError_t e_ = (call);                                                              \
    if (e_ != cudaSuccess)                                                                \
      return fail(h, LRB_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_),  \
                  __FILE__, __LINE__);                                                    \
  } while (0)

#define CKN(h, call)                                                                      \
  do {                                                                                    \
    ncclResult_t r_ = (call);                                                             \
    if (r_ != ncclSuccess)                                                                \
      return fail(h, LRB_E_NCCL, "%s failed: %s", #call,                                  \
                  g_nccl.GetErrorString ? g_nccl.GetErrorString(r_) : "nccl error");      \
  } while (0)

// temporary device allocation released on every return path
struct DevTmp {
  void* p = nullptr;
  ~DevTmp() { if (p) cudaFree(p); }
  cudaError_t alloc(size_t bytes) { return cudaMalloc(&p, bytes ? bytes : 1); }
  template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

// After a synchronisation point of a row-sharded (peer-memory) handle: did an exchange time out?
// The flag is cleared so the handle stays usable once the group is healthy again.
int check_comm(lrb_handle* h) {
  if (h->world <= 1 || h->comm != 2) return LRB_OK;
  int err = 0;
  CK(h, cudaMemcpyAsync(&err, h->comm_error, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  if (!err) return LRB_OK;
  CK(h, cudaMemsetAsync(h->comm_error, 0, sizeof(int), h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  return fail(h, LRB_E_NCCL, "peer-memory allreduce timed out: a rank of the row-sharded group did not deliver its sums "
              "(results of this call are NaN)");
}

int use_device(lrb_handle* h) {
  CK(h, cudaSetDevice(h->device));
  return LRB_OK;
}

int free_data(lrb_handle* h) {
  if (h->X) cudaFree(h->X);
  if (h->y) cudaFree(h->y);
  h->X = nullptr; h->y = nullptr; h->bound = false;
  return LRB_OK;
}

void drop_graph(lrb_handle* h) {
  if (h->gexec) cudaGraphExecDestroy(h->gexec);
  if (h->graph) cudaGraphDestroy(h->graph);
  h->gexec = nullptr; h->graph = nullptr; h->graph_nodes = 0;
}

// When X is not much larger than L2 (config 2: 128 MB vs 126 MB) pin as much of it as the device
// allows in the persisting part of L2, so most of each pass is served from L2 instead of HBM.
// For X >> L2 (configs 3, 5) the window is cleared: pure streaming.
void apply_l2_policy(lrb_handle* h) {
  cudaStreamAttrValue attr{};
  const size_t es = h->mode == LRB_MODE_FP32 ? 4 : 8;
  const size_t xbytes = (size_t)h->n * h->P * es;
  cudaDeviceProp prop;
  bool on = false;
  if (h->l2_persist && h->X && cudaGetDeviceProperties(&prop, h->device) == cudaSuccess &&
      prop.persistingL2CacheMaxSize > 0 && xbytes <= (size_t)prop.l2CacheSize * 3) {
    const size_t carve = (size_t)prop.persistingL2CacheMaxSize;
    if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve) == cudaSuccess) {
      const size_t win = std::min<size_t>(xbytes, (size_t)prop.accessPolicyMaxWindowSize);
      attr.accessPolicyWindow.base_ptr = h->X;
      attr.accessPolicyWindow.num_bytes = win;
      attr.accessPolicyWindow.hitRatio = (float)std::min(1.0, (double)carve / (double)win);
      attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
      attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
      on = true;
    }
  }
  if (!on) {
    attr.accessPolicyWindow.base_ptr = nullptr;
    attr.accessPolicyWindow.num_bytes = 0;
    attr.accessPolicyWindow.hitRatio = 0.f;
    attr.accessPolicyWindow.hitProp = cudaAccessPropertyNormal;
    attr.accessPolicyWindow.missProp = cudaAccessPropertyNormal;
  }
  if (cudaStreamSetAttribute(h->stream, cudaStreamAttributeAccessPolicyWindow, &attr) != cudaSuccess) cudaGetLastError();
}

// choose kernels and grid for the bound shape
int configure(lrb_handle* h) {
  const bool fp32 = h->mode == LRB_MODE_FP32;
  const bool ok = with_width(h->P, [&](auto w) {
    h->kern = fp32 ? choice<float, decltype(w)::value>() : choice<double, decltype(w)::value>();
  });
  if (!ok) return fail(h, LRB_E_UNSUPPORTED, "unsupported padded column count %d", h->P);
  int occ = 0, occ2 = 0;
  CK(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, h->kern.grad, kBlock, 0));
  CK(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ2, h->kern.nograd, kBlock, 0));
  if (occ < 1 || occ2 < 1) return fail(h, LRB_E_CUDA, "fused kernel does not fit an SM");
  const long long nbatch = (h->n + h->kern.rows_per_batch - 1) / h->kern.rows_per_batch;
  const long long want = std::max<long long>(1, (nbatch + kWarps - 1) / kWarps);
  h->grid = (int)std::min<long long>((long long)h->sms * occ, want);
  h->grid_nograd = (int)std::min<long long>((long long)h->sms * occ2, want);
  {
    int od = 0, odn = 0, coop = 0;
    CK(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&od, h->kern.drive, kBlock, 0));
    CK(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&odn, h->kern.drive_nograd, kBlock, 0));
    CK(h, cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, h->device));
    h->grid_drive = (int)std::min<long long>((long long)h->sms * od, want);
    h->grid_drive_nograd = (int)std::min<long long>((long long)h->sms * odn, want);
    if (od < 1 || odn < 1 || !coop || nbatch >= (1ll << 31)) h->grid_drive = h->grid_drive_nograd = 0;   // static kernel only
    // Static share of the schedule (measured, tools/drive_sweep.py): 6/8 when a warp has many
    // batches (still absorbs SMs up to 33 % slower than average), 4/8 for short passes.
    if (!getenv("LRB_DRIVE_STATIC"))
      h->drive_static_eighths = nbatch / std::max<long long>(1, (long long)h->grid_drive * kWarps) >= 32 ? 6 : 4;
  }
  int occ3 = 0;
  CK(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ3, h->kern.mc, kBlock, 0));
  if (occ3 < 1) return fail(h, LRB_E_CUDA, "many-chain kernel does not fit an SM");
  h->grid_mc = (int)std::min<long long>((long long)h->sms * occ3, want);
  drop_graph(h);
  h->chain_live = false;
  h->run_armed = false;
  // TMA descriptor of X for the tensor-core many-chain kernel
  h->tc_ok = false;
  if (h->mode == LRB_MODE_FP32 && h->P == 64 && h->n < (1ll << 31)) {
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                 const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                 CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess && fn &&
        qres == cudaDriverEntryPointSuccess) {
      const cuuint64_t dims[2] = {(cuuint64_t)h->P, (cuuint64_t)h->n};
      const cuuint64_t strides[1] = {(cuuint64_t)h->P * 4};
      const cuuint32_t box[2] = {32, (cuuint32_t)kTcRows};
      const cuuint32_t estr[2] = {1, 1};
      CUresult r = ((EncodeFn)fn)(&h->xmap_k, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, h->X, dims, strides, box, estr,
                                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                  CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      CUresult r2 = ((EncodeFn)fn)(&h->xmap_mn, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, h->X, dims, strides, box, estr,
                                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B,
                                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      h->tc_ok = (r == CUDA_SUCCESS && r2 == CUDA_SUCCESS);
    }
    if (h->tc_ok) {
      cudaError_t e = cudaFuncSetAttribute(eval_tc_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)TcLayout<64>::kDynSmem);
      if (e != cudaSuccess) { cudaGetLastError(); h->tc_ok = false; }
    }
  }
  apply_l2_policy(h);
  return LRB_OK;
}

int set_prior(lrb_handle* h, const double* pscale) {
  std::vector<double> ps(kMaxP, 1.0), lps(kMaxP, 0.0);
  for (int j = 0; j < h->p; ++j) {
    ps[j] = pscale ? pscale[j] : 1.0;
    if (!(ps[j] > 0.0)) return fail(h, LRB_E_BAD_ARG, "pscale[%d] must be > 0", j);
    lps[j] = std::log(ps[j]);
  }
  CK(h, cudaMemcpyAsync(h->d_pscale, ps.data(), kMaxP * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  CK(h, cudaMemcpyAsync(h->d_logps, lps.data(), kMaxP * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  return LRB_OK;
}

FinishArgs finish_args(lrb_handle* h, const double* beta, SamplerState* st) {
  FinishArgs f{};
  f.beta = beta;
  f.pscale = h->d_pscale;
  f.log_pscale = h->d_logps;
  f.res = h->res;
  f.state = st;
  f.p = h->p;
  f.world = h->world;
  f.rank = h->rank;
  f.p2p = (h->comm == 2) ? (getenv("LRB_P2P_FENCE") ? 3 : 1) : 0;
  f.mailbox_local = h->mailbox;
  f.flags_local = h->flags;
  f.seq = h->seq;
  f.comm_error = h->comm_error;
  f.timeout_ns = h->p2p_timeout_ns;
  for (int r = 0; r < kMaxRanks; ++r) {
    f.mailbox_peer[r] = nullptr;
    f.flags_peer[r] = nullptr;
    if (h->comm == 2 && r < h->world && h->peer_base[r]) {
      f.mailbox_peer[r] = reinterpret_cast<double*>(h->peer_base[r]);
      f.flags_peer[r] = reinterpret_cast<unsigned long long*>(
          reinterpret_cast<char*>(h->peer_base[r]) + kMailDoubles * sizeof(double));
    }
  }
  return f;
}

// Drive mode is used on single-GPU handles only.  Row-sharded handles (world > 1) keep the static
// kernel, one launch per evaluation in a replayed graph -- the path validated at N = 2, 4, 8 in both
// rounds.  Drive mode with the fused peer-memory exchange measured +2.9 % at N = 2 (four bench runs on
// two boxes, digests agreeing across ranks), but it did not complete at N = 4 / 8 in the one run round
// 2's GPU budget allowed, and the last 2-GPU parity run of the round reported one failure that could
// not be re-run; until that is understood the combination is opt-in: LRB_DRIVE_MULTI=1.
bool drive_ok(const lrb_handle* h, bool want_grad) {
  if (!h->drive || h->capturing) return false;
  if (h->world > 1 && !h->drive_multi) return false;
  return (want_grad ? h->grid_drive : h->grid_drive_nograd) > 0;
}

// The arguments of the static and the drive-mode kernel for one evaluation at `beta` (device).
// Row-sharded with NCCL the kernel only writes its sums, and finish_unfused completes the evaluation.
EvalArgs eval_args(lrb_handle* h, const double* beta, SamplerState* st) {
  EvalArgs a{};
  a.X = h->X; a.y = h->y; a.n = h->n;
  a.partials = h->partials; a.ticket = h->ticket; a.sums = h->sums;
  a.fin = finish_args(h, beta, st);
  a.timeline = h->timeline;
  a.fuse_finish = (h->comm == 1 && h->world > 1) ? 0 : 1;
  return a;
}

// After a kernel that did not run the finish step: NCCL allreduce of the sums, then the finish of
// chain 0 in a launch of its own.
int finish_unfused(lrb_handle* h, const EvalArgs& a) {
  if (a.fuse_finish) return LRB_OK;
  CKN(h, g_nccl.AllReduce(h->sums, h->sums, (size_t)h->p + 1, ncclDouble, ncclSum, h->nccl, h->stream));
  finish_mc_kernel<<<1, kBlock, 0, h->stream>>>(a.fin, h->sums, a.fin.state, a.fin.beta, 0, h->res);
  CK(h, cudaGetLastError());
  h->kernel_launches++;
  return LRB_OK;
}

// Drive mode: ONE cooperative launch performs `n_evals` consecutive evaluations (dynamic batch
// scheduling; with a sampler state the last CTA of each evaluation produces the next point).
int enqueue_drive(lrb_handle* h, const double* beta, SamplerState* st, bool want_grad, int n_evals) {
  EvalArgs a = eval_args(h, beta, st);
  if (!a.fuse_finish && n_evals != 1) return fail(h, LRB_E_STATE, "drive mode with NCCL takes one evaluation per launch (internal error)");
  PersistArgs pa{};
  pa.epoch = h->epoch; pa.work = h->work; pa.acc = h->drive_acc; pa.abort = h->drive_abort;
  pa.n_evals = n_evals; pa.spin_limit_ns = h->drive_spin_ns;
  pa.static_eighths = h->drive_static_eighths;
  void* fn = (void*)(want_grad ? h->kern.drive : h->kern.drive_nograd);
  const int grid = want_grad ? h->grid_drive : h->grid_drive_nograd;
  void* args[2] = {&a, &pa};
  cudaError_t le = cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(kBlock), args, 0, h->stream);
  if (le != cudaSuccess) {
    // e.g. the device is shared and the grid cannot be co-resident: nothing was enqueued; the
    // callers fall back to the static kernel (one launch per evaluation) for the rest of this handle
    cudaGetLastError();
    h->drive = false;
    h->drive_launch_failed = true;
    return fail(h, LRB_E_CUDA, "cooperative launch of the drive-mode kernel failed: %s", cudaGetErrorString(le));
  }
  h->kernel_launches++;
  h->eval_launches += n_evals;
  return finish_unfused(h, a);
}

// After a synchronisation: did a drive-mode launch abandon a wait?  Leaves the counters clean.
int check_drive(lrb_handle* h) {
  int ab = 0;
  CK(h, cudaMemcpyAsync(&ab, h->drive_abort, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  if (!ab) return LRB_OK;
  CK(h, cudaMemset(h->work, 0, 2 * sizeof(unsigned int)));
  CK(h, cudaMemset(h->drive_abort, 0, sizeof(int)));
  CK(h, cudaMemset(h->drive_acc, 0, (kMaxP + 1) * sizeof(double)));
  CK(h, cudaMemset(h->ticket, 0, sizeof(unsigned int)));
  h->chain_live = false;
  return fail(h, LRB_E_STATE, "drive-mode kernel abandoned a wait (a CTA or a peer rank did not arrive); the run is void");
}

// Enqueue one fused evaluation at `beta` (device) on h->stream.
int enqueue_eval(lrb_handle* h, const double* beta, SamplerState* st, bool want_grad) {
  if (drive_ok(h, want_grad)) {
    const int rc = enqueue_drive(h, beta, st, want_grad, 1);
    if (rc == LRB_OK || !h->drive_launch_failed) return rc;
    // the cooperative launch was refused before anything ran: use the static kernel instead
  }
  const EvalArgs a = eval_args(h, beta, st);
  EvalFn fn = want_grad ? h->kern.grad : h->kern.nograd;
  const int grid = want_grad ? h->grid : h->grid_nograd;
  if (h->pdl && h->world == 1) {   // measured: helps single-GPU small-n loops, neutral-to-negative with the peer exchange
    // programmatic dependent launch: the grid may start while the previous evaluation's last CTA
    // is still in its reduction / sampler update (see the prologue of eval_kernel)
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kBlock); cfg.dynamicSmemBytes = 0; cfg.stream = h->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    CK(h, cudaLaunchKernelEx(&cfg, fn, a));
  } else {
    fn<<<grid, kBlock, 0, h->stream>>>(a);
  }
  CK(h, cudaGetLastError());
  h->kernel_launches++;
  h->eval_launches++;
  return finish_unfused(h, a);
}

template <typename ST, typename T>
int ingest_launch(lrb_handle* h, const ST* src, bool colmajor, long long ld, long long nr, T* dst) {
  dim3 block(32, 8);
  dim3 grid((unsigned)((nr + 31) / 32), (unsigned)((h->P + 31) / 32));
  if (colmajor)
    ingest_kernel<ST, T, true><<<grid, block, 0, h->stream>>>(src, ld, nr, h->p, dst, h->P);
  else
    ingest_kernel<ST, T, false><<<grid, block, 0, h->stream>>>(src, ld, nr, h->p, dst, h->P);
  CK(h, cudaGetLastError());
  h->kernel_launches++;
  return LRB_OK;
}

template <typename ST>
int ingest_any(lrb_handle* h, const ST* src, bool colmajor, long long ld, long long nr, long long r0) {
  if (h->mode == LRB_MODE_FP32)
    return ingest_launch<ST, float>(h, src, colmajor, ld, nr, reinterpret_cast<float*>(h->X) + r0 * h->P);
  return ingest_launch<ST, double>(h, src, colmajor, ld, nr, reinterpret_cast<double*>(h->X) + r0 * h->P);
}

int alloc_data(lrb_handle* h, long long n, int p, int mode) {
  if (n <= 0 || p <= 0) return fail(h, LRB_E_BAD_ARG, "n and p must be positive (n=%lld p=%d)", n, p);
  if (p > kMaxP) return fail(h, LRB_E_UNSUPPORTED, "p=%d exceeds the supported maximum %d", p, kMaxP);
  if (mode != LRB_MODE_FP32 && mode != LRB_MODE_FP64) return fail(h, LRB_E_BAD_ARG, "bad mode %d", mode);
  free_data(h);
  h->n = n; h->p = p; h->P = pad_p(p); h->mode = mode;
  const size_t es = mode == LRB_MODE_FP32 ? 4 : 8;
  CK(h, cudaMalloc(&h->X, (size_t)n * h->P * es));
  const size_t ybytes = ((size_t)n + 127) / 128 * 128 + 128;   // the tensor-core path copies y in whole row tiles
  CK(h, cudaMalloc(&h->y, ybytes));
  CK(h, cudaMemset(h->y, 0, ybytes));
  return LRB_OK;
}

// states / results / sums / coefficients for C chains
int ensure_chains(lrb_handle* h, int C) {
  if (C <= h->chain_cap) return LRB_OK;
  // The launch graph bakes these pointers into its kernel arguments: it dies with the reallocation.
  // So does a paused many-chain run; a paused or armed single chain carries on from row 0.
  CK(h, cudaStreamSynchronize(h->stream));
  drop_graph(h);
  if (h->chain_C > 1) { h->chain_live = false; h->run_armed = false; }
  // The old rows are copied before the old array is freed.  SamplerState holds no pointer into its
  // own array (z, u, out and mom_* point into d_z, d_u, d_out and d_mom_*): a byte copy moves a row.
  auto regrow = [&](auto*& buf, size_t row_bytes, bool zero) {
    void* fresh = nullptr;
    cudaError_t e = cudaMalloc(&fresh, (size_t)C * row_bytes);
    if (e == cudaSuccess && zero) e = cudaMemsetAsync(fresh, 0, (size_t)C * row_bytes, h->stream);
    if (e == cudaSuccess && buf)
      e = cudaMemcpyAsync(fresh, buf, (size_t)h->chain_cap * row_bytes, cudaMemcpyDeviceToDevice, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) { cudaFree(fresh); return e; }
    cudaFree(buf);
    buf = static_cast<std::remove_reference_t<decltype(buf)>>(fresh);
    return cudaSuccess;
  };
  // states last, so that lrb_create places the single-chain state right before the drive-mode words
  // it allocates next: config 2 (drive mode) measured 0.6-0.8 % slower on a B200 (1000 W) with the
  // state allocated first.
  CK(h, regrow(h->sums, kSumStride * sizeof(double), false));
  CK(h, regrow(h->res, kResStride * sizeof(double), false));
  CK(h, regrow(h->beta, kMaxP * sizeof(double), false));
  CK(h, regrow(h->states, sizeof(SamplerState), true));
  h->chain_cap = C;
  return LRB_OK;
}

}  // namespace

// ============================================================ lifetime
extern "C" int lrb_abi_version(void) { return LRB_ABI_VERSION; }

extern "C" int lrb_device_count(int* count) {
  int c = 0;
  cudaError_t e = cudaGetDeviceCount(&c);
  if (e != cudaSuccess || c == 0) {
    if (count) *count = 0;
    return fail(nullptr, LRB_E_NO_DEVICE, "no CUDA device available (%s); logreg_b200 has no CPU fallback",
                e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
  }
  if (count) *count = c;
  return LRB_OK;
}

extern "C" int lrb_create(int device, lrb_handle** out) {
  if (!out) return fail(nullptr, LRB_E_BAD_ARG, "out is NULL");
  *out = nullptr;
  int c = 0;
  int rc = lrb_device_count(&c);
  if (rc != LRB_OK) return rc;
  if (device < 0 || device >= c) return fail(nullptr, LRB_E_BAD_ARG, "device %d out of range (%d devices)", device, c);
  lrb_handle* h = new lrb_handle();
  h->device = device;
  auto bail = [&](int code) { g_err = h->err; lrb_destroy(h); return code; };
#define CKC(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { fail(h, LRB_E_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); return bail(LRB_E_CUDA); } } while (0)
  CKC(cudaSetDevice(device));
  cudaDeviceProp prop;
  CKC(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) {
    fail(h, LRB_E_UNSUPPORTED, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
    return bail(LRB_E_UNSUPPORTED);
  }
  h->sms = prop.multiProcessorCount;
  CKC(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
  h->stream = h->own_stream;
  CKC(cudaMalloc(&h->d_pscale, kMaxP * sizeof(double)));
  CKC(cudaMalloc(&h->d_logps, kMaxP * sizeof(double)));
  CKC(cudaMalloc(&h->partials, (size_t)h->sms * 8 * kMcChains * (kMaxP + 1) * sizeof(double)));
  CKC(cudaMalloc(&h->ticket, sizeof(unsigned int)));
  CKC(cudaMemset(h->ticket, 0, sizeof(unsigned int)));
  CKC(cudaMalloc(&h->d_scale, kMaxP * sizeof(double)));
  if (ensure_chains(h, 1)) return bail(LRB_E_CUDA);
  CKC(cudaMalloc(&h->seq, sizeof(unsigned long long)));
  CKC(cudaMemset(h->seq, 0, sizeof(unsigned long long)));
  CKC(cudaMalloc(&h->comm_error, sizeof(int)));
  CKC(cudaMemset(h->comm_error, 0, sizeof(int)));
  CKC(cudaMallocHost(&h->pinned, (2 * kMaxP + 8) * sizeof(double)));
  {
    const size_t bytes = 32 + (kMaxP + 1) * sizeof(double);
    CKC(cudaMalloc(&h->drive_mem, bytes));
    CKC(cudaMemset(h->drive_mem, 0, bytes));
    char* b = reinterpret_cast<char*>(h->drive_mem);
    h->epoch = reinterpret_cast<unsigned long long*>(b);
    h->work = reinterpret_cast<unsigned int*>(b + 8);
    h->drive_abort = reinterpret_cast<int*>(b + 16);
    h->drive_acc = reinterpret_cast<double*>(b + 32);
  }
  // development / A-B knobs (the supported interface is lrb_set_option)
  if (const char* env = getenv("LRB_TC_MIN_CHAINS")) h->tc_min_chains = atoi(env);
  if (const char* env = getenv("LRB_PDL")) h->pdl = atoi(env) != 0;
  if (const char* env = getenv("LRB_P2P_TIMEOUT_MS")) h->p2p_timeout_ns = std::max(1ll, atoll(env)) * 1000000ll;
  if (const char* env = getenv("LRB_L2_PERSIST")) h->l2_persist = atoi(env) != 0;
  if (const char* env = getenv("LRB_DRIVE")) h->drive = atoi(env) != 0;
  if (const char* env = getenv("LRB_DRIVE_MULTI")) h->drive_multi = atoi(env) != 0;
  if (const char* env = getenv("LRB_DRIVE_STATIC")) h->drive_static_eighths = std::min(8, std::max(0, atoi(env)));
  if (const char* env = getenv("LRB_DETERMINISTIC")) { if (atoi(env) != 0) h->drive = false; }
#undef CKC
  *out = h;
  return LRB_OK;
}

extern "C" int lrb_destroy(lrb_handle* h) {
  if (!h) return LRB_OK;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  drop_graph(h);
  if (h->nccl && g_nccl.CommDestroy) g_nccl.CommDestroy(h->nccl);
  for (int r = 0; r < kMaxRanks; ++r)
    if (h->peer_open[r]) cudaIpcCloseMemHandle(h->peer_base[r]);
  free_data(h);
  void* bufs[] = {h->d_pscale, h->d_logps, h->partials, h->ticket, h->d_scale, h->seq, h->comm_error,
                  h->d_out, h->d_z, h->d_u, h->mailbox, h->states, h->sums, h->res, h->beta, h->partials_tc,
                  h->timeline, h->drive_mem, h->d_mom_mean, h->d_mom_m2};
  for (void* b : bufs) if (b) cudaFree(b);
  if (h->pinned) cudaFreeHost(h->pinned);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h;
  return LRB_OK;
}

extern "C" const char* lrb_last_error(const lrb_handle* h) { return h ? h->err.c_str() : g_err.c_str(); }

extern "C" int lrb_set_stream(lrb_handle* h, void* cuda_stream) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  if (use_device(h)) return LRB_E_CUDA;
  CK(h, cudaStreamSynchronize(h->stream));
  h->stream = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
  drop_graph(h);  // graphs are captured per stream
  if (h->bound) apply_l2_policy(h);
  return LRB_OK;
}

extern "C" int lrb_set_option(lrb_handle* h, int option, int64_t value) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  if (use_device(h)) return LRB_E_CUDA;
  CK(h, cudaStreamSynchronize(h->stream));
  switch (option) {
    case LRB_OPT_DETERMINISTIC: h->drive = value == 0; break;
    case LRB_OPT_TC_MIN_CHAINS: h->tc_min_chains = (int)std::max<int64_t>(1, value); break;
    case LRB_OPT_P2P_TIMEOUT_MS:
      h->p2p_timeout_ns = std::max<int64_t>(1, value) * 1000000ll;
      h->drive_spin_ns = h->p2p_timeout_ns;
      break;
    case LRB_OPT_PDL: h->pdl = value != 0; break;
    case LRB_OPT_L2_PERSIST: h->l2_persist = value != 0; if (h->bound) apply_l2_policy(h); break;
    default: return fail(h, LRB_E_BAD_ARG, "unknown option %d", option);
  }
  drop_graph(h);
  return LRB_OK;
}

extern "C" int lrb_synchronize(lrb_handle* h) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  if (use_device(h)) return LRB_E_CUDA;
  CK(h, cudaStreamSynchronize(h->stream));
  return check_comm(h);   // the synchronisation point of lrb_eval_device on a row-sharded handle
}

extern "C" int lrb_get_info(const lrb_handle* h, lrb_info* info) {
  if (!h || !info) return fail(nullptr, LRB_E_BAD_ARG, "NULL argument");
  info->n = h->n; info->p = h->p; info->p_pad = h->P; info->mode = h->mode;
  info->grid = h->grid; info->block = kBlock; info->world = h->world; info->rank = h->rank;
  info->comm = h->comm;
  info->bytes_per_eval = h->n * h->p * (h->mode == LRB_MODE_FP32 ? 4 : 8) + h->n;
  info->kernel_launches = h->kernel_launches;
  info->eval_launches = h->eval_launches;
  return LRB_OK;
}

// ============================================================ data
extern "C" int lrb_bind_data(lrb_handle* h, const void* X, int x_dtype, int layout, int64_t ld,
                             const void* y, int y_dtype, int64_t n, int p, const double* pscale,
                             int mode, int location) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  if (!X || !y) return fail(h, LRB_E_BAD_ARG, "X and y must not be NULL");
  if (x_dtype != LRB_F32 && x_dtype != LRB_F64) return fail(h, LRB_E_BAD_ARG, "X dtype must be F32 or F64");
  if (layout != LRB_ROW_MAJOR && layout != LRB_COL_MAJOR) return fail(h, LRB_E_BAD_ARG, "bad layout %d", layout);
  if (location != LRB_HOST && location != LRB_DEVICE) return fail(h, LRB_E_BAD_ARG, "bad location %d", location);
  const bool colmajor = layout == LRB_COL_MAJOR;
  if (ld < (colmajor ? n : (int64_t)p)) return fail(h, LRB_E_BAD_ARG, "leading dimension %lld too small", (long long)ld);
  if (use_device(h)) return LRB_E_CUDA;
  CK(h, cudaStreamSynchronize(h->stream));
  int rc = alloc_data(h, n, p, mode);
  if (rc) return rc;
  rc = set_prior(h, pscale);
  if (rc) return rc;
  const size_t es = x_dtype == LRB_F32 ? 4 : 8;

  if (location == LRB_DEVICE) {
    rc = x_dtype == LRB_F32 ? ingest_any<float>(h, (const float*)X, colmajor, ld, n, 0)
                            : ingest_any<double>(h, (const double*)X, colmajor, ld, n, 0);
    if (rc) return rc;
  } else {
    // stage row blocks (<= 256 MB) through device memory, re-laying each out
    long long chunk = std::max<long long>(1, (256ll << 20) / ((long long)p * (long long)es));
    chunk = std::min<long long>(chunk, n);
    DevTmp stage_buf;
    CK(h, stage_buf.alloc((size_t)chunk * p * es));
    void* stage = stage_buf.p;
    for (long long r0 = 0; r0 < n; r0 += chunk) {
      const long long nr = std::min<long long>(chunk, n - r0);
      if (colmajor)
        CK(h, cudaMemcpy2DAsync(stage, (size_t)nr * es, (const char*)X + (size_t)r0 * es, (size_t)ld * es,
                                (size_t)nr * es, (size_t)p, cudaMemcpyHostToDevice, h->stream));
      else
        CK(h, cudaMemcpy2DAsync(stage, (size_t)p * es, (const char*)X + (size_t)r0 * ld * es, (size_t)ld * es,
                                (size_t)p * es, (size_t)nr, cudaMemcpyHostToDevice, h->stream));
      const long long sld = colmajor ? nr : p;
      rc = x_dtype == LRB_F32 ? ingest_any<float>(h, (const float*)stage, colmajor, sld, nr, r0)
                              : ingest_any<double>(h, (const double*)stage, colmajor, sld, nr, r0);
      if (rc) return rc;
      CK(h, cudaStreamSynchronize(h->stream));
    }
  }

  // y -> u8 with validation
  if (y_dtype != LRB_F32 && y_dtype != LRB_F64 && y_dtype != LRB_U8) return fail(h, LRB_E_BAD_ARG, "bad y dtype");
  DevTmp bad_buf, ystage;
  CK(h, bad_buf.alloc(sizeof(int)));
  int* d_bad = bad_buf.as<int>();
  CK(h, cudaMemsetAsync(d_bad, 0, sizeof(int), h->stream));
  const size_t ys = y_dtype == LRB_F32 ? 4 : y_dtype == LRB_F64 ? 8 : 1;
  const void* ysrc = y;
  if (location == LRB_HOST) {
    CK(h, ystage.alloc((size_t)n * ys));
    CK(h, cudaMemcpyAsync(ystage.p, y, (size_t)n * ys, cudaMemcpyHostToDevice, h->stream));
    ysrc = ystage.p;
  }
  const unsigned gy = (unsigned)((n + 255) / 256);
  if (y_dtype == LRB_F32) ingest_y_kernel<float><<<gy, 256, 0, h->stream>>>((const float*)ysrc, n, h->y, d_bad);
  else if (y_dtype == LRB_F64) ingest_y_kernel<double><<<gy, 256, 0, h->stream>>>((const double*)ysrc, n, h->y, d_bad);
  else ingest_y_kernel<uint8_t><<<gy, 256, 0, h->stream>>>((const uint8_t*)ysrc, n, h->y, d_bad);
  CK(h, cudaGetLastError());
  h->kernel_launches++;
  int bad = 0;
  CK(h, cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  if (bad) {
    free_data(h);
    h->n = 0; h->p = 0; h->P = 0; h->kern = KernelChoice{};
    return fail(h, LRB_E_BAD_ARG, "y must contain only 0 and 1");
  }
  rc = configure(h);
  if (rc) return rc;
  h->bound = true;
  return LRB_OK;
}

extern "C" int lrb_gen_synthetic(lrb_handle* h, int64_t n_local, int p, int mode, uint64_t seed,
                                 const double* beta_true, const double* pscale, int64_t row_offset) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  if (!beta_true) return fail(h, LRB_E_BAD_ARG, "beta_true is NULL");
  if (use_device(h)) return LRB_E_CUDA;
  CK(h, cudaStreamSynchronize(h->stream));
  int rc = alloc_data(h, n_local, p, mode);
  if (rc) return rc;
  rc = set_prior(h, pscale);
  if (rc) return rc;
  DevTmp bt_buf;
  CK(h, bt_buf.alloc(kMaxP * sizeof(double)));
  double* d_bt = bt_buf.as<double>();
  CK(h, cudaMemcpyAsync(d_bt, beta_true, p * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  const long long nthreads = n_local * (h->P / 4);
  const unsigned gx = (unsigned)((nthreads + 255) / 256), gy = (unsigned)((n_local + 255) / 256);
  if (mode == LRB_MODE_FP32) {
    synth_x_kernel<float><<<gx, 256, 0, h->stream>>>((float*)h->X, n_local, p, h->P, seed, row_offset);
    synth_y_kernel<float><<<gy, 256, 0, h->stream>>>((const float*)h->X, n_local, p, h->P, d_bt, seed, row_offset, h->y);
  } else {
    synth_x_kernel<double><<<gx, 256, 0, h->stream>>>((double*)h->X, n_local, p, h->P, seed, row_offset);
    synth_y_kernel<double><<<gy, 256, 0, h->stream>>>((const double*)h->X, n_local, p, h->P, d_bt, seed, row_offset, h->y);
  }
  h->kernel_launches += 2;
  CK(h, cudaGetLastError());
  CK(h, cudaStreamSynchronize(h->stream));
  rc = configure(h);
  if (rc) return rc;
  h->bound = true;
  return LRB_OK;
}

extern "C" int lrb_copy_rows(lrb_handle* h, int64_t row0, int64_t nrows, double* X_out, float* y_out) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  if (!h->bound) return fail(h, LRB_E_STATE, "no data bound");
  if (row0 < 0 || nrows < 0 || row0 + nrows > h->n) return fail(h, LRB_E_BAD_ARG, "row range out of bounds");
  if (nrows == 0) return LRB_OK;
  if (use_device(h)) return LRB_E_CUDA;
  DevTmp bx, by;
  CK(h, bx.alloc((size_t)nrows * h->p * sizeof(double)));
  CK(h, by.alloc((size_t)nrows * sizeof(float)));
  double* dX = bx.as<double>(); float* dy = by.as<float>();
  const unsigned g = (unsigned)((nrows * h->P + 255) / 256);
  if (h->mode == LRB_MODE_FP32)
    export_rows_kernel<float><<<g, 256, 0, h->stream>>>((const float*)h->X, h->y, row0, nrows, h->p, h->P, dX, dy);
  else
    export_rows_kernel<double><<<g, 256, 0, h->stream>>>((const double*)h->X, h->y, row0, nrows, h->p, h->P, dX, dy);
  h->kernel_launches++;
  CK(h, cudaGetLastError());
  CK(h, cudaMemcpyAsync(X_out, dX, (size_t)nrows * h->p * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaMemcpyAsync(y_out, dy, (size_t)nrows * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  return LRB_OK;
}

// ============================================================ evaluation
namespace {

bool use_tc(const lrb_handle* h, int C) {
  return h->tc_ok && h->world == 1 && C >= h->tc_min_chains && (C + kTcChains - 1) / kTcChains <= h->sms;
}

// Scratch for the tensor-core path; must be reserved outside stream capture.
int reserve_tc(lrb_handle* h, int C) {
  if (!use_tc(h, C)) return LRB_OK;
  const int groups = (C + kTcChains - 1) / kTcChains;
  const int ntiles = (int)((h->n + kTcRows - 1) / kTcRows);
  const int gx = std::max(1, std::min(h->sms / groups, ntiles));
  const size_t need = (size_t)gx * groups * (h->P + kTcSub) * kTcChains;
  if (need <= h->partials_tc_cap) return LRB_OK;
  CK(h, cudaStreamSynchronize(h->stream));
  drop_graph(h);   // captured tensor-core launches hold the old scratch pointer
  if (h->partials_tc) cudaFree(h->partials_tc);
  h->partials_tc = nullptr; h->partials_tc_cap = 0;
  CK(h, cudaMalloc(&h->partials_tc, need * sizeof(double)));
  h->partials_tc_cap = need;
  return LRB_OK;
}

// Tensor-core many-chain evaluation: one launch of eval_tc_kernel (CTA = 128 chains x a
// strided set of 128-row tiles) + one finish launch with a CTA per chain.
int enqueue_eval_tc(lrb_handle* h, const double* beta_base, long long beta_stride, int C, SamplerState* states) {
  const int groups = (C + kTcChains - 1) / kTcChains;
  const int ntiles = (int)((h->n + kTcRows - 1) / kTcRows);
  const int gx = std::max(1, std::min(h->sms / groups, ntiles));
  const size_t need = (size_t)gx * groups * (h->P + kTcSub) * kTcChains;
  if (need > h->partials_tc_cap) return fail(h, LRB_E_STATE, "tensor-core scratch not reserved (internal error)");
  EvalTcArgs a{};
  a.y = h->y; a.n = h->n; a.ntiles = ntiles;
  a.beta_base = beta_base; a.beta_stride = beta_stride; a.C = C; a.p = h->p;
  a.partials = h->partials_tc; a.states = states; a.dbg_eta = h->dbg_eta;
  a.dbg_time = h->dbg_time;
  dim3 grid(gx, groups);
  eval_tc_kernel<64><<<grid, kTcThreads, TcLayout<64>::kDynSmem, h->stream>>>(h->xmap_k, h->xmap_mn, a);
  CK(h, cudaGetLastError());
  h->kernel_launches++;
  h->eval_launches++;
  FinishArgs f = finish_args(h, nullptr, nullptr);
  finish_tc_kernel<<<C, kBlock, 0, h->stream>>>(f, h->partials_tc, gx, groups, h->P, states, beta_base, beta_stride, h->res);
  CK(h, cudaGetLastError());
  h->kernel_launches++;
  return LRB_OK;
}

// Enqueue one fused evaluation of C >= 2 chains: ceil(C/4) passes of the SIMT many-chain
// kernel (each X batch reused for 4 chains) + one finish launch with a CTA per chain.
int enqueue_eval_mc(lrb_handle* h, const double* beta_base, long long beta_stride, int C,
                    SamplerState* states) {
  if (use_tc(h, C)) return enqueue_eval_tc(h, beta_base, beta_stride, C, states);
  constexpr int NC = kMcChains;
  for (int c0 = 0; c0 < C; c0 += NC) {
    EvalMcArgs a{};
    a.X = h->X; a.y = h->y; a.n = h->n;
    a.partials = h->partials; a.ticket = h->ticket;
    a.beta_base = beta_base; a.beta_stride = beta_stride;
    a.chain0 = c0; a.nc_active = std::min(NC, C - c0); a.p = h->p;
    a.sums = h->sums; a.states = states;
    h->kern.mc<<<h->grid_mc, kBlock, 0, h->stream>>>(a);
    CK(h, cudaGetLastError());
    h->kernel_launches++;
    h->eval_launches++;
  }
  if (h->comm == 1 && h->world > 1)
    CKN(h, g_nccl.AllReduce(h->sums, h->sums, (size_t)C * kSumStride, ncclDouble, ncclSum, h->nccl, h->stream));
  FinishArgs f = finish_args(h, nullptr, nullptr);
  finish_mc_kernel<<<C, kBlock, 0, h->stream>>>(f, h->sums, states, beta_base, beta_stride, h->res);
  CK(h, cudaGetLastError());
  h->kernel_launches++;
  return LRB_OK;
}

bool mc_capable(const lrb_handle* h) { return h->world == 1 || h->comm == 1; }

}  // namespace

extern "C" int lrb_eval_device(lrb_handle* h, const double* d_beta, double* d_out, int want_grad) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  if (!h->bound) return fail(h, LRB_E_STATE, "lrb_eval before lrb_bind_data / lrb_gen_synthetic");
  if (!d_beta) return fail(h, LRB_E_BAD_ARG, "d_beta is NULL");
  if (use_device(h)) return LRB_E_CUDA;
  int rc = enqueue_eval(h, d_beta, nullptr, want_grad != 0);
  if (rc) return rc;
  if (d_out && d_out != h->res)
    CK(h, cudaMemcpyAsync(d_out, h->res, (size_t)(h->p + 3) * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  return LRB_OK;
}

extern "C" int lrb_eval(lrb_handle* h, const double* beta, int C, int want_grad, double* lpost,
                        double* ll, double* glp) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  if (!h->bound) return fail(h, LRB_E_STATE, "lrb_eval before lrb_bind_data / lrb_gen_synthetic");
  if (!beta || C < 1) return fail(h, LRB_E_BAD_ARG, "beta is NULL or C < 1");
  if (use_device(h)) return LRB_E_CUDA;
  const int p = h->p;
  if (C >= 2 && mc_capable(h)) {
    // many-chain path: X is streamed once per 4 chains
    int rc = ensure_chains(h, C);
    if (rc) return rc;
    if ((rc = reserve_tc(h, C))) return rc;
    CK(h, cudaMemcpyAsync(h->beta, beta, (size_t)C * p * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    if ((rc = enqueue_eval_mc(h, h->beta, p, C, nullptr))) return rc;
    std::vector<double> back((size_t)C * kResStride);
    CK(h, cudaMemcpyAsync(back.data(), h->res, back.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    for (int c = 0; c < C; ++c) {
      const double* r = back.data() + (size_t)c * kResStride;
      if (lpost) lpost[c] = r[0];
      if (ll) ll[c] = r[1];
      if (glp && want_grad) std::memcpy(glp + (size_t)c * p, r + 3, p * sizeof(double));
    }
    return LRB_OK;
  }
  for (int c = 0; c < C; ++c) {
    std::memcpy(h->pinned, beta + (size_t)c * p, p * sizeof(double));
    CK(h, cudaMemcpyAsync(h->beta, h->pinned, p * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    int rc = enqueue_eval(h, h->beta, nullptr, want_grad != 0);
    if (rc) return rc;
    double* back = h->pinned + kMaxP;
    CK(h, cudaMemcpyAsync(back, h->res, (size_t)(p + 3) * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    if ((rc = check_comm(h))) return rc;
    if ((rc = check_drive(h))) return rc;
    if (lpost) lpost[c] = back[0];
    if (ll) ll[c] = back[1];
    if (glp && want_grad) std::memcpy(glp + (size_t)c * p, back + 3, p * sizeof(double));
  }
  return LRB_OK;
}

extern "C" int lrb_tc_tile_rows(void) { return kTcRows; }

extern "C" int lrb_debug_tc_eta(lrb_handle* h, const double* beta, int C, float* eta_out) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  if (!h->bound) return fail(h, LRB_E_STATE, "no data bound");
  if (!h->tc_ok) return fail(h, LRB_E_UNSUPPORTED, "tensor-core path unavailable for this shape/mode");
  if (!beta || !eta_out || C < 1) return fail(h, LRB_E_BAD_ARG, "bad arguments");
  if (use_device(h)) return LRB_E_CUDA;
  int rc = ensure_chains(h, C);
  if (rc) return rc;
  if ((rc = reserve_tc(h, C))) return rc;
  if (!use_tc(h, C)) return fail(h, LRB_E_UNSUPPORTED, "C below the tensor-core threshold");
  const int groups = (C + kTcChains - 1) / kTcChains;
  const size_t cnt = (size_t)groups * kTcChains * kTcRows;
  CK(h, cudaMalloc(&h->dbg_eta, cnt * sizeof(float)));
  CK(h, cudaMemsetAsync(h->dbg_eta, 0, cnt * sizeof(float), h->stream));
  cudaError_t e = cudaMemcpyAsync(h->beta, beta, (size_t)C * h->p * sizeof(double), cudaMemcpyHostToDevice, h->stream);
  if (e == cudaSuccess) rc = enqueue_eval_tc(h, h->beta, h->p, C, nullptr);
  if (e == cudaSuccess && rc == LRB_OK) e = cudaMemcpyAsync(eta_out, h->dbg_eta, cnt * sizeof(float), cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess && rc == LRB_OK) e = cudaStreamSynchronize(h->stream);
  cudaFree(h->dbg_eta);
  h->dbg_eta = nullptr;
  if (getenv("LRB_TC_TIMELINE") && rc == LRB_OK) {
    // development aid: per-tile clock64 stamps of CTA (0,0) for a second, instrumented launch
    std::vector<long long> tl(64 * 16, 0);
    cudaMalloc(&h->dbg_time, tl.size() * sizeof(long long));
    cudaMemset(h->dbg_time, 0, tl.size() * sizeof(long long));
    enqueue_eval_tc(h, h->beta, h->p, C, nullptr);
    cudaStreamSynchronize(h->stream);
    cudaMemcpy(tl.data(), h->dbg_time, tl.size() * sizeof(long long), cudaMemcpyDeviceToHost);
    cudaFree(h->dbg_time);
    h->dbg_time = nullptr;
    const char* names[11] = {"tma_issue", "x_full", "xl_done", "mma1_go", "mma1_issued", "d1_full", "ldtm_done",
                             "math_done", "r_full", "mma2_go", "mma2_issued"};
    printf("tile");
    for (int e = 0; e < 11; ++e) printf(" %11s", names[e]);
    printf("\n");
    for (int i = 8; i < 40; ++i) {
      printf("%4d", i);
      for (int e = 0; e < 11; ++e) printf(" %11lld", tl[i * 16 + e] ? tl[i * 16 + e] - tl[8 * 16] : -1);
      printf("\n");
    }
  }
  if (rc) return rc;
  if (e != cudaSuccess) return fail(h, LRB_E_CUDA, "debug_tc_eta failed: %s", cudaGetErrorString(e));
  return LRB_OK;
}

// Development aid: record %globaltimer stamps of every CTA of the fused kernel (entry, after the
// grid dependency, end of streaming, after the ticket) and of the last CTA's tail.  The stamps of
// the LATEST evaluation are kept.
extern "C" int lrb_debug_timeline(lrb_handle* h, int enable) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  if (use_device(h)) return LRB_E_CUDA;
  CK(h, cudaStreamSynchronize(h->stream));
  drop_graph(h);
  if (h->timeline) { cudaFree(h->timeline); h->timeline = nullptr; }
  if (enable) {
    const size_t cnt = (size_t)h->sms * 8 * 4 + 8;
    CK(h, cudaMalloc(&h->timeline, cnt * sizeof(long long)));
    CK(h, cudaMemset(h->timeline, 0, cnt * sizeof(long long)));
  }
  return LRB_OK;
}

extern "C" int lrb_debug_timeline_read(lrb_handle* h, int64_t* out, int64_t cap, int64_t* grid) {
  if (!h || !out || !grid) return fail(h, LRB_E_BAD_ARG, "NULL argument");
  if (!h->timeline) return fail(h, LRB_E_STATE, "timeline not enabled");
  if (use_device(h)) return LRB_E_CUDA;
  const int64_t cnt = (int64_t)h->grid * 4 + 8;
  if (cap < cnt) return fail(h, LRB_E_BAD_ARG, "out too small: need %lld", (long long)cnt);
  CK(h, cudaStreamSynchronize(h->stream));
  CK(h, cudaMemcpy(out, h->timeline, cnt * sizeof(long long), cudaMemcpyDeviceToHost));
  *grid = h->grid;
  return LRB_OK;
}

extern "C" int lrb_lprior(lrb_handle* h, const double* beta, int C, double* out) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  if (!h->bound) return fail(h, LRB_E_STATE, "lrb_lprior before lrb_bind_data / lrb_gen_synthetic");
  if (!beta || !out || C < 1) return fail(h, LRB_E_BAD_ARG, "bad arguments");
  if (use_device(h)) return LRB_E_CUDA;
  DevTmp bb, bo;
  CK(h, bb.alloc((size_t)C * h->p * sizeof(double)));
  CK(h, bo.alloc((size_t)C * sizeof(double)));
  double *db = bb.as<double>(), *dout = bo.as<double>();
  CK(h, cudaMemcpyAsync(db, beta, (size_t)C * h->p * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  prior_kernel<<<C, kBlock, 0, h->stream>>>(db, h->d_pscale, h->d_logps, h->p, dout);
  CK(h, cudaGetLastError());
  h->kernel_launches++;
  CK(h, cudaMemcpyAsync(out, dout, (size_t)C * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  return LRB_OK;
}

// ============================================================ posterior predictive / WAIC
namespace {

using PredFn = void (*)(const PredictiveArgs);
using LoglikFn = void (*)(const LoglikArgs);
const auto predictive_pick = [](auto t, auto w) -> PredFn { return predictive_kernel<decltype(t), decltype(w)::value>; };
const auto loglik_pick = [](auto t, auto w) -> LoglikFn { return loglik_kernel<decltype(t), decltype(w)::value>; };

// draws (S x p, float64, row-major, host) -> dst: P x Spad in the mode's dtype, k-major, zero padded
template <typename T>
int upload_draws(lrb_handle* h, void* dst, const double* draws, long long S, long long Spad) {
  std::vector<T> bt((size_t)h->P * Spad, (T)0);
  for (long long s = 0; s < S; ++s)
    for (int k = 0; k < h->p; ++k) bt[(size_t)k * Spad + s] = (T)draws[(size_t)s * h->p + k];
  CK(h, cudaMemcpyAsync(dst, bt.data(), bt.size() * sizeof(T), cudaMemcpyHostToDevice, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));   // bt is pageable host memory and dies here
  return LRB_OK;
}

// The draws of one call, uploaded for predictive_kernel or loglik_kernel (both read the same
// layout and dynamic shared memory), and the launch shape of the kernel Fn.
template <typename Fn>
struct Draws {
  DevTmp dB;
  Fn fn = nullptr;
  size_t smem = 0;
  int occ = 0;
  long long S = 0, Spad = 0;
};

// pick(T(), std::integral_constant<int, P>()) is the kernel for dtype T and padded width P.
template <typename Fn, typename Pick>
int draws_prepare(lrb_handle* h, const char* what, Pick pick, const double* draws, long long S, Draws<Fn>& g) {
  const bool fp32 = h->mode == LRB_MODE_FP32;
  const bool ok = with_width(h->P, [&](auto w) {
    g.fn = fp32 ? pick(float(), w) : pick(double(), w);
    g.smem = fp32 ? predictive_smem<float, decltype(w)::value>() : predictive_smem<double, decltype(w)::value>();
  });
  if (!ok) return fail(h, LRB_E_UNSUPPORTED, "unsupported padded column count %d", h->P);
  CK(h, cudaFuncSetAttribute((const void*)g.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem));
  CK(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&g.occ, g.fn, kBlock, g.smem));
  if (g.occ < 1) return fail(h, LRB_E_CUDA, "%s kernel does not fit an SM", what);
  g.S = S;
  g.Spad = (S + kPredDraws - 1) / kPredDraws * kPredDraws;
  CK(h, g.dB.alloc((size_t)h->P * g.Spad * (fp32 ? 4 : 8)));
  return fp32 ? upload_draws<float>(h, g.dB.p, draws, S, g.Spad) : upload_draws<double>(h, g.dB.p, draws, S, g.Spad);
}

int check_single_gpu(lrb_handle* h, const char* what) {
  if (h->world > 1)
    return fail(h, LRB_E_UNSUPPORTED, "%s works on single-GPU handles only: this handle is rank %d of a row-sharded "
                "group of %d, and its per-shard totals would need a collective", what, h->rank, h->world);
  return LRB_OK;
}

}  // namespace

extern "C" int lrb_predictive(lrb_handle* h, const double* draws, int64_t S, int location, double* prob_mean,
                              double* prob_sd, double* lppd, double* p_waic, lrb_predictive_totals* totals) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  if (!h->bound) return fail(h, LRB_E_STATE, "lrb_predictive before lrb_bind_data / lrb_gen_synthetic");
  if (!draws || S < 1) return fail(h, LRB_E_BAD_ARG, "draws is NULL or S < 1 (S=%lld)", (long long)S);
  if (S > (1ll << 30)) return fail(h, LRB_E_BAD_ARG, "S=%lld draws exceeds 2^30", (long long)S);
  if (location != LRB_HOST && location != LRB_DEVICE) return fail(h, LRB_E_BAD_ARG, "bad location %d", location);
  if (int rc = check_single_gpu(h, "lrb_predictive")) return rc;
  if (use_device(h)) return LRB_E_CUDA;
  Draws<PredFn> g;
  if (int rc = draws_prepare(h, "predictive", predictive_pick, draws, S, g)) return rc;
  const long long ntiles = (h->n + kPredRows - 1) / kPredRows;
  const int grid = (int)std::min<long long>((long long)h->sms * g.occ, ntiles);

  // scratch: CTA partials, totals, ticket; per-row outputs on the device when the caller's are on the host
  DevTmp work, out[4];
  const size_t wdoubles = (size_t)grid * kPredPartial + kPredTotals;
  CK(h, work.alloc(wdoubles * sizeof(double) + sizeof(unsigned int)));
  unsigned int* ticket = reinterpret_cast<unsigned int*>(work.as<double>() + wdoubles);
  CK(h, cudaMemsetAsync(ticket, 0, sizeof(unsigned int), h->stream));
  double* user[4] = {prob_mean, prob_sd, lppd, p_waic};
  double* dev[4] = {};
  for (int k = 0; k < 4; ++k) {
    if (!user[k]) continue;
    if (location == LRB_DEVICE) { dev[k] = user[k]; continue; }
    CK(h, out[k].alloc((size_t)h->n * sizeof(double)));
    dev[k] = out[k].as<double>();
  }

  PredictiveArgs a{};
  a.X = h->X; a.y = h->y; a.n = h->n;
  a.B = g.dB.p; a.S = S; a.Spad = g.Spad;
  a.prob_mean = dev[0]; a.prob_sd = dev[1]; a.lppd = dev[2]; a.p_waic = dev[3];
  a.partials = work.as<double>();
  a.ticket = ticket;
  a.totals = work.as<double>() + (size_t)grid * kPredPartial;
  g.fn<<<grid, kBlock, g.smem, h->stream>>>(a);
  CK(h, cudaGetLastError());
  h->kernel_launches++;

  double tot[kPredTotals];
  CK(h, cudaMemcpyAsync(tot, a.totals, sizeof tot, cudaMemcpyDeviceToHost, h->stream));
  if (location == LRB_HOST)
    for (int k = 0; k < 4; ++k)
      if (user[k]) CK(h, cudaMemcpyAsync(user[k], dev[k], (size_t)h->n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));   // the temporaries die with this scope
  if (totals) {
    totals->n = h->n;
    totals->draws = S;
    totals->lppd = tot[0];
    totals->p_waic = tot[1];
    totals->elpd_waic = tot[2];
    totals->se_elpd_waic = tot[3];
  }
  return LRB_OK;
}

// ============================================================ PSIS-LOO / pointwise log-likelihood
namespace {

// L[i][s] (row stride S) for the bound rows [row0, row0 + rows)
int loglik_launch(lrb_handle* h, const Draws<LoglikFn>& g, long long row0, long long rows, double* L) {
  const size_t es = h->mode == LRB_MODE_FP32 ? 4 : 8;
  LoglikArgs a{};
  a.X = static_cast<const char*>(h->X) + (size_t)row0 * h->P * es;
  a.y = h->y + row0;
  a.n = rows;
  a.B = g.dB.p; a.S = g.S; a.Spad = g.Spad;
  a.L = L; a.ld = g.S;
  const long long ntiles = (rows + kPredRows - 1) / kPredRows;
  const long long ngroups = (g.Spad / kPredDraws + kLoglikGroup - 1) / kLoglikGroup;
  const int grid = (int)std::min<long long>((long long)h->sms * g.occ, ntiles * ngroups);
  g.fn<<<grid, kBlock, g.smem, h->stream>>>(a);
  CK(h, cudaGetLastError());
  h->kernel_launches++;
  return LRB_OK;
}

// Rows of L per chunk: a multiple of 64 whose L fits the scratch budget (at least 64 rows).
// LRB_LOO_CHUNK_MB overrides the budget, to measure what keeping a chunk in L2 is worth.
long long loo_chunk_rows(long long n, long long S) {
  long long budget = 64ll << 20;
  if (const char* e = getenv("LRB_LOO_CHUNK_MB")) budget = std::max(1ll, atoll(e)) << 20;
  long long R = budget / (S * (long long)sizeof(double)) / kPredRows * kPredRows;
  R = std::max<long long>(R, kPredRows);
  return std::min<long long>(R, (n + kPredRows - 1) / kPredRows * kPredRows);
}

}  // namespace

extern "C" int lrb_loglik(lrb_handle* h, const double* draws, int64_t S, int64_t row0, int64_t nrows, int location,
                          double* out) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  if (!h->bound) return fail(h, LRB_E_STATE, "lrb_loglik before lrb_bind_data / lrb_gen_synthetic");
  if (!draws || !out || S < 1) return fail(h, LRB_E_BAD_ARG, "draws or out is NULL, or S < 1 (S=%lld)", (long long)S);
  if (S > kLooMaxDraws) return fail(h, LRB_E_BAD_ARG, "S=%lld draws exceeds 2^21", (long long)S);
  if (row0 < 0 || nrows < 1 || row0 + nrows > h->n)
    return fail(h, LRB_E_BAD_ARG, "rows [%lld, %lld) outside the %lld bound rows", (long long)row0,
                (long long)(row0 + nrows), h->n);
  if (location != LRB_HOST && location != LRB_DEVICE) return fail(h, LRB_E_BAD_ARG, "bad location %d", location);
  if (int rc = check_single_gpu(h, "lrb_loglik")) return rc;
  if (use_device(h)) return LRB_E_CUDA;
  Draws<LoglikFn> g;
  if (int rc = draws_prepare(h, "log-likelihood", loglik_pick, draws, S, g)) return rc;
  if (location == LRB_DEVICE) {
    if (int rc = loglik_launch(h, g, row0, nrows, out)) return rc;
  } else {   // chunk by chunk through a bounded device buffer
    const long long R = loo_chunk_rows(nrows, S);
    DevTmp L;
    CK(h, L.alloc((size_t)R * S * sizeof(double)));
    for (long long c0 = 0; c0 < nrows; c0 += R) {
      const long long rows = std::min(R, (long long)nrows - c0);
      if (int rc = loglik_launch(h, g, row0 + c0, rows, L.as<double>())) return rc;
      CK(h, cudaMemcpyAsync(out + (size_t)c0 * S, L.p, (size_t)rows * S * sizeof(double), cudaMemcpyDeviceToHost,
                            h->stream));
    }
  }
  CK(h, cudaStreamSynchronize(h->stream));   // the temporaries die with this scope
  return LRB_OK;
}

extern "C" int lrb_loo(lrb_handle* h, const double* draws, int64_t S, int location, double* elpd_loo, double* p_loo,
                       double* pareto_k, lrb_loo_totals* totals) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  if (!h->bound) return fail(h, LRB_E_STATE, "lrb_loo before lrb_bind_data / lrb_gen_synthetic");
  if (!draws || S < 1) return fail(h, LRB_E_BAD_ARG, "draws is NULL or S < 1 (S=%lld)", (long long)S);
  if (S > kLooMaxDraws)
    return fail(h, LRB_E_BAD_ARG, "S=%lld draws exceeds 2^21: PSIS needs a row's S log-likelihoods at once, and 64 "
                "rows of them (the smallest chunk) would exceed 1 GB of scratch", (long long)S);
  if (location != LRB_HOST && location != LRB_DEVICE) return fail(h, LRB_E_BAD_ARG, "bad location %d", location);
  if (int rc = check_single_gpu(h, "lrb_loo")) return rc;
  if (use_device(h)) return LRB_E_CUDA;
  const bool stage2 = !getenv("LRB_LOO_STAGE1_ONLY");   // timing of stage 1 alone (header, tools/loo_bench.py)
  Draws<LoglikFn> g;
  if (int rc = draws_prepare(h, "log-likelihood", loglik_pick, draws, S, g)) return rc;
  const long long n = h->n, M = psis_tail_len(S);
  const int stage = S <= kLooRowSmem ? 1 : 0;
  const size_t smem = psis_smem(S, M, stage);
  CK(h, cudaFuncSetAttribute((const void*)psis_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 0;
  CK(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, psis_kernel, kBlock, smem));
  if (occ < 1) return fail(h, LRB_E_CUDA, "PSIS kernel does not fit an SM");

  const long long R = loo_chunk_rows(n, S);
  const long long ntiles = (n + kPredRows - 1) / kPredRows;
  DevTmp L, rowbuf, work;
  CK(h, L.alloc((size_t)R * S * sizeof(double)));
  CK(h, rowbuf.alloc((size_t)3 * R * sizeof(double)));
  CK(h, work.alloc(((size_t)ntiles * kLooPartial + 8) * sizeof(double)));
  double* re = rowbuf.as<double>();
  double *rp = re + R, *rk = rp + R;
  double* partials = work.as<double>();
  double* dtot = partials + (size_t)ntiles * kLooPartial;
  double* user[3] = {elpd_loo, p_loo, pareto_k};
  double* chunk[3] = {re, rp, rk};
  const cudaMemcpyKind kind = location == LRB_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
  const double kthr = loo_k_threshold(S);
  for (long long c0 = 0; c0 < n; c0 += R) {
    const long long rows = std::min(R, n - c0);
    if (int rc = loglik_launch(h, g, c0, rows, L.as<double>())) return rc;
    if (!stage2) continue;
    PsisArgs a{};
    a.L = L.as<double>(); a.rows = rows; a.S = S; a.M = M; a.stage = stage;
    a.elpd = re; a.p_loo = rp; a.pareto_k = rk;
    psis_kernel<<<(int)std::min<long long>((long long)h->sms * occ, rows), kBlock, smem, h->stream>>>(a);
    CK(h, cudaGetLastError());
    const long long ct = (rows + kPredRows - 1) / kPredRows;
    loo_tile_kernel<<<(int)((ct + kBlock - 1) / kBlock), kBlock, 0, h->stream>>>(re, rp, rk, rows, kthr,
                                                                               partials + (c0 / kPredRows) * kLooPartial);
    CK(h, cudaGetLastError());
    h->kernel_launches += 2;
    for (int k = 0; k < 3; ++k)
      if (user[k]) CK(h, cudaMemcpyAsync(user[k] + c0, chunk[k], (size_t)rows * sizeof(double), kind, h->stream));
  }
  double tot[7];
  for (double& t : tot) t = NAN;
  if (!stage2)   // stage 1 was timed alone: no result exists, so every output reads NaN
    for (int k = 0; k < 3; ++k) {
      if (!user[k]) continue;
      if (location == LRB_DEVICE) CK(h, cudaMemsetAsync(user[k], 0xff, (size_t)n * sizeof(double), h->stream));
      else std::fill(user[k], user[k] + n, (double)NAN);
    }
  if (stage2) {
    loo_totals_kernel<<<1, kBlock, 0, h->stream>>>(partials, ntiles, dtot);
    CK(h, cudaGetLastError());
    h->kernel_launches++;
    CK(h, cudaMemcpyAsync(tot, dtot, sizeof tot, cudaMemcpyDeviceToHost, h->stream));
  }
  CK(h, cudaStreamSynchronize(h->stream));   // the temporaries die with this scope
  if (totals) {
    totals->n = n;
    totals->draws = S;
    totals->elpd_loo = tot[1];
    totals->se_elpd_loo = tot[2];
    totals->p_loo = tot[3];
    totals->se_p_loo = tot[4];
    totals->looic = -2.0 * tot[1];
    totals->k_threshold = kthr;
    totals->k_max = tot[5];
    totals->n_k_high = stage2 ? (int64_t)tot[6] : -1;
  }
  return LRB_OK;
}

extern "C" int lrb_debug_psis(const double* log_ratios, int64_t S, double* log_weights, double* khat) {
  if (!log_ratios || !log_weights || !khat || S < 1) return fail(nullptr, LRB_E_BAD_ARG, "bad arguments");
  const double* r = log_ratios;
  double rmax = r[0];
  for (int64_t s = 1; s < S; ++s) rmax = nan_max(rmax, r[s]);
  std::vector<double> lw(S);
  for (int64_t s = 0; s < S; ++s) lw[s] = r[s] - rmax;
  double k = INFINITY;
  const int64_t M = psis_tail_len(S);
  if (M >= 5) {
    std::vector<int64_t> order(S);
    for (int64_t s = 0; s < S; ++s) order[s] = s;
    std::stable_sort(order.begin(), order.end(), [&](int64_t a, int64_t b) { return lw[a] < lw[b]; });
    const double tmin = lw[order[S - M]], tmax = lw[order[S - 1]];
    if (std::fabs(tmax - tmin) >= 2.220446049250313e-16 / 100.0) {
      const double cutoff = lw[order[S - M - 1]], ec = std::exp(cutoff);
      std::vector<double> x(M);
      for (int64_t j = 0; j < M; ++j) x[j] = std::exp(lw[order[S - M + j]]) - ec;
      const int mg = gpd_grid_len(M);
      const double xmax = x[M - 1], xstar = x[(int64_t)std::floor(M / 4.0 + 0.5) - 1];
      std::vector<double> th(mg), lt(mg);
      double lmx = -INFINITY;
      for (int j = 0; j < mg; ++j) {
        th[j] = gpd_theta(j + 1, mg, xmax, xstar);
        double sk = 0.0;
        for (int64_t t = 0; t < M; ++t) sk += std::log1p(-th[j] * x[t]);
        lt[j] = gpd_ltheta(th[j], sk / (double)M, M);
        lmx = nan_max(lmx, lt[j]);
      }
      double sw = 0.0;
      for (int j = 0; j < mg; ++j) sw += std::exp(lt[j] - lmx);
      const double lse = lmx + std::log(sw);
      double theta = 0.0;
      for (int j = 0; j < mg; ++j) theta += th[j] * std::exp(lt[j] - lse);
      double sk = 0.0;
      for (int64_t t = 0; t < M; ++t) sk += std::log1p(-theta * x[t]);
      const double kraw = sk / (double)M, sigma = -kraw / theta;
      k = gpd_wip(kraw, M);
      if (std::isfinite(k))
        for (int64_t j = 0; j < M; ++j) lw[order[S - M + j]] = psis_smoothed(k, sigma, psis_quantile(j + 1, M), ec);
    }
  }
  for (int64_t s = 0; s < S; ++s) log_weights[s] = (lw[s] > 0.0 ? 0.0 : lw[s]) + rmax;
  *khat = k;
  return LRB_OK;
}

// ============================================================ MAP optimiser (f1)
namespace {

// d_H (p x p, leading dimension ld, device) = X' W X at d_beta over the rows of this handle, summed
// over the ranks of a row-sharded group (NCCL communicator only).
int compute_hessian(lrb_handle* h, const double* d_beta, double* d_H, int ld) {
  const int p = h->p, P = h->P;
  const int PW = std::min(P, kHessPanel);
  const int npanels = (p + kHessPanel - 1) / kHessPanel;
  const long long ntiles = (h->n + kHessRows - 1) / kHessRows;
  const int gridh = (int)std::max<long long>(1, std::min<long long>((long long)h->sms * 2, ntiles));
  const int gridw = (int)std::max<long long>(1, std::min<long long>((long long)h->sms * 8, (h->n + kBlock - 1) / kBlock));
  if (h->world > 1 && h->comm != 1)
    return fail(h, LRB_E_UNSUPPORTED, "the Hessian of a row-sharded problem needs the NCCL communicator (p x p allreduce)");
  DevTmp wbuf, part;
  CK(h, wbuf.alloc((size_t)h->n * sizeof(double)));
  CK(h, part.alloc((size_t)gridh * kHessPanel * kHessPanel * sizeof(double)));
  CK(h, cudaMemsetAsync(d_H, 0, (size_t)ld * p * sizeof(double), h->stream));
  if (h->mode == LRB_MODE_FP32)
    newton_weights_kernel<float><<<gridw, kBlock, 0, h->stream>>>((const float*)h->X, h->n, P, p, d_beta, wbuf.as<double>());
  else
    newton_weights_kernel<double><<<gridw, kBlock, 0, h->stream>>>((const double*)h->X, h->n, P, p, d_beta, wbuf.as<double>());
  CK(h, cudaGetLastError());
  h->kernel_launches++;
  for (int bi = 0; bi < npanels; ++bi)
    for (int bj = 0; bj <= bi; ++bj) {
      if (h->mode == LRB_MODE_FP32)
        newton_hess_block_kernel<float><<<gridh, kBlock, 0, h->stream>>>((const float*)h->X, wbuf.as<double>(), h->n, P,
                                                                         bi * kHessPanel, bj * kHessPanel, PW, part.as<double>());
      else
        newton_hess_block_kernel<double><<<gridh, kBlock, 0, h->stream>>>((const double*)h->X, wbuf.as<double>(), h->n, P,
                                                                          bi * kHessPanel, bj * kHessPanel, PW, part.as<double>());
      CK(h, cudaGetLastError());
      newton_hess_reduce_kernel<<<(PW * PW + kBlock - 1) / kBlock, kBlock, 0, h->stream>>>(
          part.as<double>(), gridh, PW, bi * kHessPanel, bj * kHessPanel, p, d_H, ld);
      CK(h, cudaGetLastError());
      h->kernel_launches += 2;
    }
  if (h->world > 1) CKN(h, g_nccl.AllReduce(d_H, d_H, (size_t)ld * p, ncclDouble, ncclSum, h->nccl, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));   // the temporaries die with this scope
  return LRB_OK;
}

}  // namespace

extern "C" int lrb_hessian(lrb_handle* h, const double* beta, double* H_out) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  if (!h->bound) return fail(h, LRB_E_STATE, "lrb_hessian before lrb_bind_data / lrb_gen_synthetic");
  if (!beta || !H_out) return fail(h, LRB_E_BAD_ARG, "NULL argument");
  if (use_device(h)) return LRB_E_CUDA;
  const int p = h->p;
  DevTmp db, dH;
  CK(h, db.alloc(kMaxP * sizeof(double)));
  CK(h, dH.alloc((size_t)p * p * sizeof(double)));
  CK(h, cudaMemcpyAsync(db.p, beta, p * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  int rc = compute_hessian(h, db.as<double>(), dH.as<double>(), p);
  if (rc) return rc;
  CK(h, cudaMemcpyAsync(H_out, dH.p, (size_t)p * p * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  std::vector<double> ps(p);
  CK(h, cudaMemcpyAsync(ps.data(), h->d_pscale, p * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  for (int j = 0; j < p; ++j) H_out[(size_t)j * p + j] += 1.0 / (ps[j] * ps[j]);
  return LRB_OK;
}

extern "C" int lrb_map(lrb_handle* h, const double* init, double tol, int maxit, double* beta_out, lrb_map_info* info) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  if (!h->bound) return fail(h, LRB_E_STATE, "lrb_map before lrb_bind_data / lrb_gen_synthetic");
  if (!init || !beta_out) return fail(h, LRB_E_BAD_ARG, "NULL argument");
  if (!(tol > 0.0) || maxit < 1) return fail(h, LRB_E_BAD_ARG, "tol must be > 0 and maxit >= 1");
  if (use_device(h)) return LRB_E_CUDA;
  const int p = h->p;
  DevTmp stbuf, dH;
  CK(h, stbuf.alloc(sizeof(NewtonState)));
  CK(h, dH.alloc((size_t)p * p * sizeof(double)));
  NewtonState* st = stbuf.as<NewtonState>();
  CK(h, cudaMemsetAsync(st, 0, sizeof(NewtonState), h->stream));
  CK(h, cudaMemcpyAsync(st->beta, init, p * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  lrb_map_info out{};
  int rc = LRB_OK;
  struct { double lp_cur, grad_norm; int32_t chol_fail, accepted, halvings, pad; } back{};
  static_assert(sizeof(back) == sizeof(NewtonState) - offsetof(NewtonState, lp_cur), "NewtonState tail layout");
  for (int it = 0; it < maxit; ++it) {
    if ((rc = enqueue_eval(h, st->beta, nullptr, true))) return rc;            // lpost, glp at beta
    out.evals++;
    if ((rc = compute_hessian(h, st->beta, dH.as<double>(), p))) return rc;    // X'WX at beta
    newton_step_kernel<<<1, 32, 0, h->stream>>>(st, dH.as<double>(), p, p, h->d_pscale, h->res);
    CK(h, cudaGetLastError());
    h->kernel_launches++;
    bool accepted = false;
    for (int j = 0; j < 15 && !accepted; ++j) {                                // fit-jax.py:70-74
      if ((rc = enqueue_eval(h, st->beta_try, nullptr, false))) return rc;
      out.evals++;
      newton_decide_kernel<<<1, 32, 0, h->stream>>>(st, p, h->res, 0);
      CK(h, cudaGetLastError());
      h->kernel_launches++;
      CK(h, cudaMemcpyAsync(&back, &st->lp_cur, sizeof(back), cudaMemcpyDeviceToHost, h->stream));
      CK(h, cudaStreamSynchronize(h->stream));
      if ((rc = check_comm(h))) return rc;
      if ((rc = check_drive(h))) return rc;
      if (back.chol_fail)
        return fail(h, LRB_E_STATE, "Newton: X'WX + diag(pscale^-2) is not positive definite at column %d", back.chol_fail - 1);
      accepted = back.accepted != 0;
      if (!accepted) out.halvings++;
    }
    if (!accepted) {   // 15 halvings used up: take the (tiny) step anyway, as the reference does (:75)
      newton_decide_kernel<<<1, 32, 0, h->stream>>>(st, p, h->res, 1);
      CK(h, cudaGetLastError());
      h->kernel_launches++;
      CK(h, cudaStreamSynchronize(h->stream));
    }
    out.iterations = it + 1;
    out.grad_norm = back.grad_norm;
    if (back.grad_norm < tol) { out.converged = 1; break; }                    // :76-77, the gradient of the OLD iterate
  }
  if ((rc = enqueue_eval(h, st->beta, nullptr, false))) return rc;             // report lpost at the result
  out.evals++;
  double lp = 0.0;
  CK(h, cudaMemcpyAsync(&lp, h->res, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaMemcpyAsync(beta_out, st->beta, p * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  if ((rc = check_comm(h))) return rc;
  if ((rc = check_drive(h))) return rc;
  out.lpost = lp;
  if (info) *info = out;
  return LRB_OK;
}

extern "C" int lrb_debug_chol_solve(double* A, int ld, int p, const double* pscale, const double* g, double* step) {
  return newton_chol_solve(A, ld, p, pscale, g, step);
}

// ============================================================ samplers
namespace {

long long evals_per_step(int kind, int l) { return kind == LRB_HMC ? (long long)l : 1; }

int grow(lrb_handle* h, double** buf, size_t* cap, size_t need) {
  if (need <= *cap) return LRB_OK;
  if (*buf) cudaFree(*buf);
  *buf = nullptr; *cap = 0;
  CK(h, cudaMalloc(buf, need * sizeof(double)));
  *cap = need;
  return LRB_OK;
}

// one evaluation of every chain of the armed run at its state's beta_in
int enqueue_run_eval(lrb_handle* h) {
  if (h->run_C > 1)
    return enqueue_eval_mc(h, h->states->beta_in, (long long)(sizeof(SamplerState) / sizeof(double)),
                           h->run_C, h->states);
  return enqueue_eval(h, h->states->beta_in, h->states, h->run_want_grad);
}

// capture `nodes` consecutive evaluations into an executable graph
int build_graph(lrb_handle* h, int nodes, bool want_grad) {
  if (h->gexec && h->graph_nodes == nodes && h->graph_grad == want_grad && h->graph_C == h->run_C) return LRB_OK;
  drop_graph(h);
  const long long kl = h->kernel_launches, el = h->eval_launches;
  CK(h, cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
  int rc = LRB_OK;
  h->capturing = true;     // graphs hold the static kernel (one launch per evaluation)
  for (int i = 0; i < nodes && rc == LRB_OK; ++i) rc = enqueue_run_eval(h);
  h->capturing = false;
  cudaGraph_t g = nullptr;
  cudaError_t e = cudaStreamEndCapture(h->stream, &g);
  h->graph_kl_per_replay = h->kernel_launches - kl;
  h->graph_el_per_replay = h->eval_launches - el;
  h->kernel_launches = kl; h->eval_launches = el;  // capture does not execute
  if (rc) { if (g) cudaGraphDestroy(g); return rc; }
  if (e != cudaSuccess) return fail(h, LRB_E_CUDA, "graph capture failed: %s", cudaGetErrorString(e));
  h->graph = g;
  CK(h, cudaGraphInstantiate(&h->gexec, h->graph, 0));
  h->graph_nodes = nodes;
  h->graph_grad = want_grad;
  h->graph_C = h->run_C;
  return LRB_OK;
}

int arm_run(lrb_handle* h, const lrb_sampler_params* params, const double* init, int C, int64_t thin,
            int64_t iters, const double* replay_z, const double* replay_u) {
  if (!h->bound) return fail(h, LRB_E_STATE, "lrb_run before lrb_bind_data / lrb_gen_synthetic");
  if (!params || !params->scale) return fail(h, LRB_E_BAD_ARG, "params / params->scale is NULL");
  const int kind = params->sampler;
  if (kind < LRB_RWMH || kind > LRB_HMC) return fail(h, LRB_E_BAD_ARG, "unknown sampler %d", kind);
  if (thin < 1 || iters < 0) return fail(h, LRB_E_BAD_ARG, "thin must be >= 1 and iters >= 0");
  if (kind == LRB_HMC && params->l < 1) return fail(h, LRB_E_BAD_ARG, "HMC needs l >= 1");
  if (kind != LRB_RWMH && !(params->step > 0.0)) return fail(h, LRB_E_BAD_ARG, "step (dt / eps) must be > 0");
  if (params->rng != LRB_RNG_PHILOX && params->rng != LRB_RNG_REPLAY && params->rng != LRB_RNG_KEYED)
    return fail(h, LRB_E_BAD_ARG, "bad rng %d", params->rng);
  if ((params->flags & LRB_RUN_SET_T0) && params->t0 < 0) return fail(h, LRB_E_BAD_ARG, "t0 must be >= 0");
  if (params->rng == LRB_RNG_REPLAY && (!replay_z || (kind != LRB_UL && !replay_u)))
    return fail(h, LRB_E_BAD_ARG, "replay rng needs replay_z (and replay_u unless UL)");
  if (!init && (!h->chain_live || h->chain_kind != kind || h->chain_C != C))
    return fail(h, LRB_E_STATE, "init is NULL but there is no paused chain of this sampler to continue");
  for (int j = 0; j < h->p; ++j)
    if (!(params->scale[j] > 0.0)) return fail(h, LRB_E_BAD_ARG, "scale[%d] must be > 0", j);
  if (use_device(h)) return LRB_E_CUDA;

  const int p = h->p;
  const long long steps = thin * iters;
  int rc;
  if ((rc = ensure_chains(h, C))) return rc;
  if (C > 1 && (rc = reserve_tc(h, C))) return rc;
  const bool want_moments = (params->flags & LRB_RUN_MOMENTS) != 0;
  const bool no_samples = (params->flags & LRB_RUN_NO_SAMPLES) != 0;
  if (!no_samples && (rc = grow(h, &h->d_out, &h->out_cap, std::max<size_t>(1, (size_t)C * iters * p)))) return rc;
  if (want_moments) {
    if (init) {
      if ((rc = grow(h, &h->d_mom_mean, &h->mom_mean_cap, (size_t)C * p))) return rc;
      if ((rc = grow(h, &h->d_mom_m2, &h->mom_m2_cap, (size_t)C * p * p))) return rc;
    } else if (!h->chain_moments) {
      return fail(h, LRB_E_STATE, "LRB_RUN_MOMENTS on a continued run needs a chain that was started with it");
    }
  }
  const double *dz = nullptr, *du = nullptr;
  if (params->rng == LRB_RNG_REPLAY && steps > 0) {
    if ((rc = grow(h, &h->d_z, &h->z_cap, (size_t)C * steps * p))) return rc;
    CK(h, cudaMemcpyAsync(h->d_z, replay_z, (size_t)C * steps * p * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    dz = h->d_z;
    if (kind != LRB_UL) {
      if ((rc = grow(h, &h->d_u, &h->u_cap, (size_t)C * steps))) return rc;
      CK(h, cudaMemcpyAsync(h->d_u, replay_u, (size_t)C * steps * sizeof(double), cudaMemcpyHostToDevice, h->stream));
      du = h->d_u;
    }
  }
  h->run_params = *params;
  h->run_params.scale = nullptr;
  std::memcpy(h->pinned, params->scale, p * sizeof(double));
  CK(h, cudaMemcpyAsync(h->d_scale, h->pinned, p * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  if (init) CK(h, cudaMemcpyAsync(h->beta, init, (size_t)C * p * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  // reuse the cached gradient / lpost of the paused chain when the caller vouches that init is its state
  const int reuse = (init && (params->flags & LRB_RUN_REUSE_CACHE) && h->chain_live && h->chain_kind == kind &&
                     h->chain_C == C && (kind == LRB_MALA || kind == LRB_HMC)) ? 1 : 0;
  h->run_C = C;
  sampler_begin_kernel<<<C, kBlock, 0, h->stream>>>(h->states, init ? h->beta : nullptr, h->d_scale, kind, params->l, p,
                                                    params->rng, params->step, params->seed,
                                                    params->init_lpost, steps, thin, dz, du,
                                                    no_samples ? nullptr : h->d_out, reuse,
                                                    (params->flags & LRB_RUN_SET_T0) ? (long long)params->t0 : 0ll,
                                                    want_moments ? h->d_mom_mean : nullptr,
                                                    want_moments ? h->d_mom_m2 : nullptr);
  CK(h, cudaGetLastError());
  h->kernel_launches++;
  CK(h, cudaStreamSynchronize(h->stream));  // staging buffers are reused by the caller's next call

  h->run_kind = kind;
  h->run_l = kind == LRB_HMC ? params->l : 1;
  h->run_want_grad = kind != LRB_RWMH;
  h->run_thin = thin;
  h->run_iters = iters;
  h->run_moments = want_moments;
  h->run_no_samples = no_samples;
  if (init) h->chain_moments = want_moments;
  h->pending_init_eval = init != nullptr && !reuse && (kind == LRB_MALA || kind == LRB_HMC) && steps > 0;
  h->run_dz = dz;
  h->run_du = du;
  h->run_consumed = false;
  h->run_armed = true;
  if (init) h->chain_live = false;   // the old chain is overwritten; the new one exists once it has been launched
  h->chain_kind = kind;
  h->chain_C = C;
  return LRB_OK;
}

int launch_run(lrb_handle* h) {
  if (!h->run_armed) return fail(h, LRB_E_STATE, "lrb_run_launch before lrb_run_begin");
  if (use_device(h)) return LRB_E_CUDA;
  const long long steps = h->run_thin * h->run_iters;
  if (steps == 0) return LRB_OK;
  if (h->run_consumed) {
    // A repeated launch continues the chain: re-arm the window [t, t+steps) and
    // propose from the paused state (replayed draws, if any, start over).
    sampler_begin_kernel<<<h->run_C, kBlock, 0, h->stream>>>(h->states, nullptr, h->d_scale, h->run_kind,
                                                             h->run_params.l, h->p, h->run_params.rng,
                                                             h->run_params.step, h->run_params.seed, 0.0, steps,
                                                             h->run_thin, h->run_dz, h->run_du,
                                                             h->run_no_samples ? nullptr : h->d_out, 0, 0ll,
                                                             h->run_moments ? h->d_mom_mean : nullptr,
                                                             h->run_moments ? h->d_mom_m2 : nullptr);
    CK(h, cudaGetLastError());
    h->kernel_launches++;
  }
  h->run_consumed = true;
  long long needed = steps * evals_per_step(h->run_kind, h->run_l) + (h->pending_init_eval ? 1 : 0);
  h->pending_init_eval = false;
  const bool nccl_mode = (h->comm == 1 && h->world > 1);
  if (h->run_C == 1 && !nccl_mode && drive_ok(h, h->run_want_grad)) {
    // drive mode: the whole run is one launch (chunked only to keep the counter in an int)
    bool refused = false;
    while (needed > 0) {
      const int chunk = (int)std::min<long long>(needed, 1ll << 24);
      int rc = enqueue_drive(h, h->states->beta_in, h->states, h->run_want_grad, chunk);
      if (rc && h->drive_launch_failed && !h->chain_live_partial) { refused = true; break; }   // nothing ran yet: static path below
      if (rc) return rc;
      h->chain_live_partial = true;
      needed -= chunk;
    }
    h->chain_live_partial = false;
    if (!refused) {
      h->chain_live = true;
      return LRB_OK;
    }
  }
  // graph of up to 64 evaluations, replayed; the remainder goes out as plain launches
  const int nodes = (int)std::min<long long>(64, needed);
  int rc = build_graph(h, nodes, h->run_want_grad);
  if (rc) return rc;
  while (needed >= nodes) {
    CK(h, cudaGraphLaunch(h->gexec, h->stream));
    h->kernel_launches += h->graph_kl_per_replay;
    h->eval_launches += h->graph_el_per_replay;
    needed -= nodes;
  }
  for (; needed > 0; --needed)
    if ((rc = enqueue_run_eval(h))) return rc;
  h->chain_live = true;
  return LRB_OK;
}

int finish_run(lrb_handle* h, double* out, int64_t* accepted) {
  if (!h->run_armed) return fail(h, LRB_E_STATE, "lrb_run_finish before lrb_run_begin");
  if (use_device(h)) return LRB_E_CUDA;
  const int C = h->run_C;
  const size_t cnt = (size_t)C * h->run_iters * h->p;
  if (out && cnt && !h->run_no_samples)
    CK(h, cudaMemcpyAsync(out, h->d_out, cnt * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  std::vector<long long> acc(C, 0);
  std::vector<int> phase(C, -1);
  SamplerState* st = h->states;
  CK(h, cudaMemcpy2DAsync(acc.data(), sizeof(long long), &st->accepted, sizeof(SamplerState), sizeof(long long), C,
                          cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaMemcpy2DAsync(phase.data(), sizeof(int), &st->phase, sizeof(SamplerState), sizeof(int), C,
                          cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  if (int rcc = check_comm(h)) return rcc;
  if (int rcd = check_drive(h)) return rcd;
  for (int c = 0; c < C; ++c) {
    if (accepted) accepted[c] = acc[c];
    if (phase[c] != PH_PAUSED)
      return fail(h, LRB_E_STATE, "chain %d did not reach the end of the run (phase %d): launch count mismatch", c, phase[c]);
  }
  return LRB_OK;
}

}  // namespace

extern "C" int lrb_run_begin(lrb_handle* h, const lrb_sampler_params* params, const double* init,
                             int64_t thin, int64_t iters, const double* replay_z, const double* replay_u) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  return arm_run(h, params, init, 1, thin, iters, replay_z, replay_u);
}

extern "C" int lrb_run_evals_per_launch(const lrb_handle* h, int64_t* evals) {
  if (!h || !evals) return fail(nullptr, LRB_E_BAD_ARG, "NULL argument");
  if (!h->run_armed) return fail(nullptr, LRB_E_STATE, "no run armed");
  *evals = h->run_thin * h->run_iters * evals_per_step(h->run_kind, h->run_l);
  return LRB_OK;
}

extern "C" int lrb_run_launch(lrb_handle* h) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  return launch_run(h);
}

extern "C" int lrb_run_finish(lrb_handle* h, double* out, int64_t* accepted) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  return finish_run(h, out, accepted);
}

extern "C" int lrb_chain_state(lrb_handle* h, double* x, double* lpost, int64_t* steps) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  if (!h->chain_live) return fail(h, LRB_E_STATE, "no chain has been run on this handle");
  if (use_device(h)) return LRB_E_CUDA;
  long long t = 0; double lp = 0.0;
  SamplerState* st = h->states;   // chain 0 of a many-chain run
  if (x) CK(h, cudaMemcpyAsync(x, st->x, h->p * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaMemcpyAsync(&lp, &st->lp_x, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaMemcpyAsync(&t, &st->t, sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  if (lpost) *lpost = lp;
  if (steps) *steps = t;
  return LRB_OK;
}

extern "C" int lrb_run(lrb_handle* h, const lrb_sampler_params* params, const double* init, int C,
                       int64_t thin, int64_t iters, const double* replay_z, const double* replay_u,
                       double* out, int64_t* accepted) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  if (C < 1) return fail(h, LRB_E_BAD_ARG, "C must be >= 1");
  if (C == 1 || mc_capable(h)) {
    // all chains advance in lock-step on the device (many-chain kernel for C >= 2)
    int rc = arm_run(h, params, init, C, thin, iters, replay_z, replay_u);
    if (rc) return rc;
    if ((rc = launch_run(h))) return rc;
    return finish_run(h, out, accepted);
  }
  // row-sharded with the fused peer-memory allreduce: chains one after the other
  if (!init) return fail(h, LRB_E_BAD_ARG, "continuing (init == NULL) needs C == 1 in this configuration");
  if (params && (params->flags & LRB_RUN_MOMENTS))
    return fail(h, LRB_E_UNSUPPORTED, "LRB_RUN_MOMENTS with several chains on a fused-P2P row-sharded handle is not supported "
                                      "(the chains run one after the other through one state); use the NCCL communicator");
  const int p = h->p;
  const size_t steps = (size_t)(thin * iters);
  for (int c = 0; c < C; ++c) {
    lrb_sampler_params pc = *params;
    pc.seed = params->seed + (uint64_t)c * 0x9E3779B97F4A7C15ull;  // the key chain c gets in the lock-step path
    int rc = arm_run(h, &pc, init + (size_t)c * p, 1, thin, iters,
                     replay_z ? replay_z + (size_t)c * steps * p : nullptr,
                     replay_u ? replay_u + (size_t)c * steps : nullptr);
    if (rc) return rc;
    if ((rc = launch_run(h))) return rc;
    int64_t acc0 = 0;
    if ((rc = finish_run(h, out ? out + (size_t)c * iters * p : nullptr, &acc0))) return rc;
    if (accepted) accepted[c] = acc0;
  }
  return LRB_OK;
}

extern "C" int lrb_run_moments(lrb_handle* h, int pooled, int64_t* count, double* mean, double* cov) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  if (!count || !mean) return fail(h, LRB_E_BAD_ARG, "count / mean is NULL");
  if (!h->chain_live || !h->chain_moments) return fail(h, LRB_E_STATE, "no run with LRB_RUN_MOMENTS on this handle");
  if (use_device(h)) return LRB_E_CUDA;
  const int C = h->chain_C, p = h->p;
  const int rows = pooled ? 1 : C;
  DevTmp bc, bm, bv;
  CK(h, bc.alloc((size_t)rows * sizeof(long long)));
  CK(h, bm.alloc((size_t)rows * p * sizeof(double)));
  if (cov) CK(h, bv.alloc((size_t)rows * p * p * sizeof(double)));
  moments_out_kernel<<<rows, kBlock, 0, h->stream>>>(h->states, C, p, pooled ? 1 : 0, bc.as<long long>(), bm.as<double>(),
                                                     cov ? bv.as<double>() : nullptr);
  CK(h, cudaGetLastError());
  h->kernel_launches++;
  static_assert(sizeof(long long) == sizeof(int64_t), "count layout");
  CK(h, cudaMemcpyAsync(count, bc.p, (size_t)rows * sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaMemcpyAsync(mean, bm.p, (size_t)rows * p * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (cov) CK(h, cudaMemcpyAsync(cov, bv.p, (size_t)rows * p * p * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  return LRB_OK;
}

extern "C" uint64_t lrb_key_child(uint64_t key, uint64_t i) { return philox_child(key, i); }

extern "C" int lrb_rng_dump(lrb_handle* h, uint64_t seed, int64_t t0, int64_t count, int p,
                            double* z_out, double* u_out) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  if (count < 1 || p < 1 || !z_out || !u_out) return fail(h, LRB_E_BAD_ARG, "bad arguments");
  if (use_device(h)) return LRB_E_CUDA;
  DevTmp bz, bu;
  CK(h, bz.alloc((size_t)count * p * sizeof(double)));
  CK(h, bu.alloc((size_t)count * sizeof(double)));
  double *dz = bz.as<double>(), *du = bu.as<double>();
  rng_dump_kernel<<<(unsigned)((count * p + 255) / 256), 256, 0, h->stream>>>(seed, t0, count, p, dz, du);
  h->kernel_launches++;
  CK(h, cudaGetLastError());
  CK(h, cudaMemcpyAsync(z_out, dz, (size_t)count * p * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaMemcpyAsync(u_out, du, (size_t)count * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  return LRB_OK;
}

// ============================================================ communicators
extern "C" int lrb_nccl_unique_id(void* id_out, const char* libnccl_path) {
  if (!id_out) return fail(nullptr, LRB_E_BAD_ARG, "id_out is NULL");
  std::string err;
  if (!load_nccl(libnccl_path, err)) return fail(nullptr, LRB_E_NCCL, "%s", err.c_str());
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  ncclUniqueId id;
  CKN(nullptr, g_nccl.GetUniqueId(&id));
  std::memcpy(id_out, &id, sizeof id);
  return LRB_OK;
}

extern "C" int lrb_comm_init_nccl(lrb_handle* h, int rank, int world, const void* unique_id,
                                  const char* libnccl_path) {
  if (!h) return fail(nullptr, LRB_E_BAD_ARG, "handle is NULL");
  if (world < 1 || world > kMaxRanks || rank < 0 || rank >= world) return fail(h, LRB_E_BAD_ARG, "bad rank/world %d/%d", rank, world);
  if (!unique_id) return fail(h, LRB_E_BAD_ARG, "unique_id is NULL");
  std::string err;
  if (!load_nccl(libnccl_path, err)) return fail(h, LRB_E_NCCL, "%s", err.c_str());
  if (use_device(h)) return LRB_E_CUDA;
  ncclUniqueId id;
  std::memcpy(&id, unique_id, sizeof id);
  CKN(h, g_nccl.CommInitRank(&h->nccl, world, id, rank));
  h->world = world; h->rank = rank; h->comm = 1;
  drop_graph(h);
  return LRB_OK;
}

extern "C" int lrb_comm_p2p_export(lrb_handle* h, void* ipc_out) {
  if (!h || !ipc_out) return fail(h, LRB_E_BAD_ARG, "NULL argument");
  if (use_device(h)) return LRB_E_CUDA;
  if (!h->mailbox) {
    CK(h, cudaMalloc(&h->mailbox, kMailBytes));
    CK(h, cudaMemset(h->mailbox, 0, kMailBytes));
    h->flags = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(h->mailbox) + kMailDoubles * sizeof(double));
  }
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  cudaIpcMemHandle_t mh;
  CK(h, cudaIpcGetMemHandle(&mh, h->mailbox));
  std::memcpy(ipc_out, &mh, sizeof mh);
  return LRB_OK;
}

extern "C" int lrb_comm_p2p_connect(lrb_handle* h, int rank, int world, const void* all_handles) {
  if (!h || !all_handles) return fail(h, LRB_E_BAD_ARG, "NULL argument");
  if (world < 1 || world > kMaxRanks || rank < 0 || rank >= world) return fail(h, LRB_E_BAD_ARG, "bad rank/world %d/%d", rank, world);
  if (!h->mailbox) return fail(h, LRB_E_STATE, "call lrb_comm_p2p_export first");
  if (use_device(h)) return LRB_E_CUDA;
  CK(h, cudaStreamSynchronize(h->stream));
  for (int r = 0; r < kMaxRanks; ++r) {   // a reconnect: drop the previous mappings
    if (h->peer_open[r]) cudaIpcCloseMemHandle(h->peer_base[r]);
    h->peer_open[r] = false; h->peer_base[r] = nullptr;
  }
  // Stale sums / flags of a previous connection would satisfy the first acquire waits: start clean.
  // The caller must barrier between connect and the first evaluation (dist.init_comm does), so no
  // peer has written yet.
  CK(h, cudaMemset(h->mailbox, 0, kMailBytes));
  CK(h, cudaMemset(h->comm_error, 0, sizeof(int)));
  for (int r = 0; r < world; ++r) {
    if (r == rank) { h->peer_base[r] = h->mailbox; continue; }
    cudaIpcMemHandle_t mh;
    std::memcpy(&mh, (const char*)all_handles + (size_t)r * sizeof mh, sizeof mh);
    void* base = nullptr;
    CK(h, cudaIpcOpenMemHandle(&base, mh, cudaIpcMemLazyEnablePeerAccess));
    h->peer_base[r] = base;
    h->peer_open[r] = true;
  }
  CK(h, cudaMemset(h->seq, 0, sizeof(unsigned long long)));
  h->world = world; h->rank = rank; h->comm = 2;
  drop_graph(h);
  return LRB_OK;
}
