/* logreg_b200.h -- C ABI of the B200-native logistic log-posterior / gradient /
 * sampler library (liblogreg_b200.so).
 *
 * The reference (darrenjw/logreg) has NO plugin / FFI interface for this path:
 * its boundary is a set of Python callables that close over module globals
 * (SURVEY.md section 8b).  Each entry point below therefore cites the reference
 * callable(s) it stands behind; paths are relative to the reference root.
 * The Python shim `logreg_b200` binds these with ctypes and re-exports the
 * reference's names; INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - every function returns an int status: 0 = LRB_OK, otherwise an LRB_E_* code;
 *     the message is available from lrb_last_error(h) (h may be NULL for errors
 *     raised before a handle exists).  There is no CPU fallback: without a CUDA
 *     device lrb_create fails with LRB_E_NO_DEVICE.
 *   - plain pointers and sizes only; all host arrays are caller-owned; the handle
 *     owns every device allocation, stream, graph and communicator and frees them
 *     in lrb_destroy.
 *   - a handle is bound to ONE device and is not thread-safe (one caller thread).
 *   - all results (lpost, ll, glp, samples) are float64, as in the reference.
 */
#ifndef LOGREG_B200_H
#define LOGREG_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LRB_ABI_VERSION 2

enum lrb_status {
  LRB_OK = 0,
  LRB_E_NO_DEVICE = 1,   /* no CUDA device / driver: the product path refuses to run */
  LRB_E_BAD_ARG = 2,
  LRB_E_CUDA = 3,
  LRB_E_NCCL = 4,
  LRB_E_STATE = 5,       /* call out of order (e.g. eval before bind_data) */
  LRB_E_UNSUPPORTED = 6
};

enum lrb_dtype { LRB_F32 = 0, LRB_F64 = 1, LRB_U8 = 2 };
enum lrb_layout { LRB_ROW_MAJOR = 0, LRB_COL_MAJOR = 1 };
enum lrb_location { LRB_HOST = 0, LRB_DEVICE = 1 };

/* Arithmetic mode of the fused kernel (BASELINE.json north_star):
 *   FP64: X stored and streamed as float64, every operation in float64
 *         (parity target 1e-10 relative against the reference);
 *   FP32: X stored and streamed as float32; eta = x.beta and the per-row
 *         softplus / sigmoid in float32 (beta carried as a hi+lo float pair),
 *         log-likelihood and gradient accumulated in float64
 *         (parity target 1e-5 relative). */
enum lrb_mode { LRB_MODE_FP64 = 0, LRB_MODE_FP32 = 1 };

enum lrb_sampler {
  LRB_RWMH = 0, /* Python/fit-numpy.py:53-62 (mhKernel) + :81-84 (rprop)          */
  LRB_UL = 1,   /* Python/fit-np-ul.py:61-68 (ulKernel)                            */
  LRB_MALA = 2, /* Python/fit-np-mala.py:61-78 (mhKernel + malaKernel)             */
  LRB_HMC = 3   /* Python/fit-np-hmc.py:56-87 (mhKernel + hmcKernel)               */
};

enum lrb_rng {
  LRB_RNG_PHILOX = 0, /* on-device Philox4x32-10, counter = (iteration, coordinate) */
  LRB_RNG_REPLAY = 1, /* host-supplied N(0,1) rows Z and uniforms U, consumed in the
                         reference's order: randn(p) then rand() per kernel call
                         (fit-numpy.py:84,58; fit-np-hmc.py:85,60; UL: no U)         */
  LRB_RNG_KEYED = 2   /* JAX-style split keys (Python/fit-jax2.py:98-116): `seed` is the root key;
                         kernel application t of the run uses
                         split(split(root, iters)[t / thin], thin)[t % thin], split once more
                         inside the kernel exactly as the reference kernels do (mhKernel
                         fit-jax2.py:90, hmcKernel fit-jax-hmc.py:126-129, ulKernel
                         fit-jax-ul.py:86-88); split(k, n)[i] = lrb_key_child(k, i)           */
};

/* lrb_sampler_params.flags: `init` is bit-for-bit the state the previous run of the SAME sampler
 * (MALA or HMC) on this handle ended in, so its cached gradient (and, for HMC, lpost) are reused
 * instead of re-evaluated. The result is identical to a run without the flag; one pass over X is
 * saved. Ignored when there is no such paused chain. */
#define LRB_RUN_REUSE_CACHE 1
/* Start the chain's kernel-application counter (the Philox counter of LRB_RNG_PHILOX) at
 * params->t0 instead of 0: a chain checkpointed with lrb_chain_state after `steps` applications
 * resumes in a NEW process / handle with init = x, init_lpost = lpost, t0 = steps and the same seed
 * and continues the same random stream.  Ignored when init is NULL. */
#define LRB_RUN_SET_T0 2
/* Accumulate running mean and cross-moments of the thinned states on the device (Welford), per
 * chain; read them with lrb_run_moments.  They restart with a new chain (init != NULL) and keep
 * accumulating over continued runs (Dex/djwutils.dx:97-103 meanAndCovariance, analyse.R:16). */
#define LRB_RUN_MOMENTS 4
/* Do not store the thinned states at all (use with LRB_RUN_MOMENTS for many chains): lrb_run's
 * `out` is ignored and nothing but the moments ever leaves the device. */
#define LRB_RUN_NO_SAMPLES 8

typedef struct lrb_handle lrb_handle;

typedef struct lrb_sampler_params {
  int32_t sampler;     /* enum lrb_sampler */
  int32_t l;           /* HMC: number of leap-frog position updates (fit-np-hmc.py:65 `l`) */
  double step;         /* UL/MALA: dt (fit-np-ul.py:61, fit-np-mala.py:72); HMC: eps; RWMH: unused */
  const double* scale; /* host, length p.  RWMH: proposal sd per coordinate (0.02*pre,
                          fit-numpy.py:84); UL/MALA: `pre`; HMC: `dmm` (mass diagonal) */
  uint64_t seed;       /* Philox key */
  int32_t rng;         /* enum lrb_rng */
  int32_t flags;       /* LRB_RUN_* bits */
  double init_lpost;   /* log-density carried in with `init` for the samplers that thread it
                          (RWMH, MALA: the `ll` argument of kernel(x, ll), fit-numpy.py:54).
                          mcmc() passes -inf, which makes the first proposal always accepted
                          (fit-numpy.py:66).  Ignored when init is NULL, by UL and by HMC. */
  int64_t t0;          /* with LRB_RUN_SET_T0: kernel applications already done by the resumed chain */
} lrb_sampler_params;

typedef struct lrb_info {
  int64_t n;            /* rows bound on THIS handle (the local shard) */
  int32_t p;            /* columns (coefficients) */
  int32_t p_pad;        /* columns as laid out in HBM (zero-padded to 8/16/32/.../256) */
  int32_t mode;         /* enum lrb_mode */
  int32_t grid;         /* CTAs of the fused kernel */
  int32_t block;        /* threads per CTA */
  int32_t world;        /* ranks in the row-sharded group (1 = single GPU) */
  int32_t rank;
  int32_t comm;         /* 0 none, 1 NCCL allreduce, 2 fused peer-memory allreduce */
  int64_t bytes_per_eval;   /* ALGORITHMIC bytes one fused evaluation streams: n*p*sizeof(X)+n*sizeof(y) */
  int64_t kernel_launches;  /* kernels launched by this handle so far (all kinds) */
  int64_t eval_launches;    /* fused-evaluation kernel launches so far */
} lrb_info;

/* ---- lifetime ----------------------------------------------------------- */
int lrb_abi_version(void);
int lrb_device_count(int* count);
int lrb_create(int device, lrb_handle** out);
int lrb_destroy(lrb_handle* h);
const char* lrb_last_error(const lrb_handle* h);
/* Launch everything on `cuda_stream` (a cudaStream_t) instead of the handle's own
 * stream, so a caller can time with events on its own stream. NULL restores the
 * handle's stream. */
int lrb_set_stream(lrb_handle* h, void* cuda_stream);
int lrb_synchronize(lrb_handle* h);

/* Per-handle options.
 *   DETERMINISTIC  0 (default): single-chain evaluations on a single-GPU handle run in "drive
 *                  mode" -- a persistent cooperative kernel (one launch per run) with dynamic
 *                  row-batch scheduling and atomic (timing-ordered) accumulation of the CTA sums;
 *                  results are reproducible to rounding (~1e-15 relative), not bit for bit.
 *                  1: the static kernel, one launch per evaluation (replayed CUDA graph), CTA sums
 *                  added in a fixed order => bit-identical results for a fixed shape.  Row-sharded
 *                  handles (world > 1) and many-chain runs always use the static kernels.
 *   TC_MIN_CHAINS  chain count from which the tensor-core many-chain kernel is used (default 12).
 *   P2P_TIMEOUT_MS bound of every in-kernel wait for a peer rank / another CTA (default 60000).
 *   PDL            programmatic dependent launch between evaluations of the static kernel.
 *   L2_PERSIST     pin X in the persisting part of L2 when it is at most 3x the L2 size. */
enum lrb_option {
  LRB_OPT_DETERMINISTIC = 1,
  LRB_OPT_TC_MIN_CHAINS = 2,
  LRB_OPT_P2P_TIMEOUT_MS = 3,
  LRB_OPT_PDL = 4,
  LRB_OPT_L2_PERSIST = 5
};
int lrb_set_option(lrb_handle* h, int option, int64_t value);
int lrb_get_info(const lrb_handle* h, lrb_info* info);

/* ---- data: the script globals X, y, pscale --------------------------------
 * Replaces the closure over `X`, `y` (fit-numpy.py:12-19) and `pscale`
 * (fit-np-ul.py:31).  X is n x p in `x_dtype` (F32/F64), `layout` row- or
 * column-major with leading dimension `ld` (elements; the reference's X is
 * column-major float64, SURVEY.md A8); y is n responses in {0,1} (F32/F64/U8).
 * The library copies and re-lays the data out row-major in the mode's dtype
 * (the ingest kernels), so the caller's arrays may be freed afterwards.
 * `location` says whether X and y are host or device pointers. */
int lrb_bind_data(lrb_handle* h, const void* X, int x_dtype, int layout, int64_t ld,
                  const void* y, int y_dtype, int64_t n, int p,
                  const double* pscale, int mode, int location);

/* Synthetic problem generated in HBM (SURVEY.md 8d): X[:,0]=1, X[:,1:]~N(0,1),
 * y~Bernoulli(expit(X beta_true)), Philox counters keyed on the GLOBAL row index
 * `row_offset + i`, so each row shard regenerates exactly its rows. */
int lrb_gen_synthetic(lrb_handle* h, int64_t n_local, int p, int mode, uint64_t seed,
                      const double* beta_true, const double* pscale, int64_t row_offset);

/* Copy rows [row0, row0+nrows) of the bound data back to the host as float64
 * row-major X (nrows x p) and float32 y: lets a checker evaluate the same rows. */
int lrb_copy_rows(lrb_handle* h, int64_t row0, int64_t nrows, double* X_out, float* y_out);

/* ---- evaluation: lpost / ll / glp ------------------------------------------
 * ONE fused pass over X per coefficient vector: replaces `ll` (fit-numpy.py:23-24),
 * `lprior` (fit-np-ul.py:33-34), `lpost` (fit-numpy.py:43-44) and `glp`
 * (fit-np-ul.py:45-48).  beta: C x p row-major (host).  Outputs (host, any may
 * be NULL): lpost[C], ll[C], glp[C x p].  want_grad=0 skips the gradient.
 * With a row-sharded communicator every rank must call it with the same beta;
 * all ranks receive the global result. */
int lrb_eval(lrb_handle* h, const double* beta, int C, int want_grad,
             double* lpost, double* ll, double* glp);

/* Same, device-resident and asynchronous on the handle's stream:
 * d_beta: p doubles; d_out: [lpost, ll, lprior, glp[0..p)] = p+3 doubles. */
int lrb_eval_device(lrb_handle* h, const double* d_beta, double* d_out, int want_grad);

/* Diagnostic for the tensor-core many-chain kernel: runs it on C coefficient vectors and
 * returns eta = x.beta of the FIRST row tile, eta_out[ceil(C/128)*128][lrb_tc_tile_rows()]
 * (chain-major), as the tensor cores produced it (3xTF32).  Test instrumentation; not part of the
 * drop-in path. */
int lrb_debug_tc_eta(lrb_handle* h, const double* beta, int C, float* eta_out);
int lrb_tc_tile_rows(void);

/* Development instrumentation of the fused streaming kernel: when enabled every CTA records
 * %globaltimer (ns) at entry, after the grid dependency, at the end of streaming and after its
 * ticket; the last CTA adds the end of its reduction and of the finish/sampler step.
 * lrb_debug_timeline_read returns [grid][4] + [8] stamps of the latest evaluation. */
int lrb_debug_timeline(lrb_handle* h, int enable);
int lrb_debug_timeline_read(lrb_handle* h, int64_t* out, int64_t cap, int64_t* grid);

/* ---- MAP optimiser: the step before the samplers (provides `init`) ---------------------
 * Newton's method with the exact Hessian and step halving, Python/fit-jax.py:62-79 (same loop
 * in fit-jax2.py and fit-jax-ul.py): step = solve(X'WX + diag(pscale^-2), glp(beta)), halved up
 * to 15 times until lpost improves, stop when ||glp|| < tol at the iterate the step came from
 * (the reference uses tol = 0.01, maxit = 500).  lpost/glp come from the fused kernel (one pass
 * each), X'WX from a float64 block kernel, the Cholesky solve and the accept/halve decision run
 * on the device; the host sequences launches and reads one flag per trial.  init, beta_out: p
 * doubles (host).  Row-sharded handles need the NCCL communicator (p x p allreduce). */
typedef struct lrb_map_info {
  int32_t iterations;  /* Newton iterations performed */
  int32_t converged;   /* 1 if ||glp|| < tol was reached within maxit */
  int32_t halvings;    /* step halvings over the whole run */
  int32_t evals;       /* fused evaluations (passes over X for lpost / glp) */
  double lpost;        /* lpost at beta_out */
  double grad_norm;    /* ||glp||_2 at the last iterate a step was computed from */
} lrb_map_info;
int lrb_map(lrb_handle* h, const double* init, double tol, int maxit, double* beta_out, lrb_map_info* info);
/* H_out (p x p, row-major, host) = X'WX + diag(pscale^-2) = -Hessian of lpost at beta
 * (jacfwd(jacrev(lpost)) in fit-jax.py:58-61, up to the sign). */
int lrb_hessian(lrb_handle* h, const double* beta, double* H_out);
/* The Cholesky solve lrb_map runs on the device, callable on the host (it is the same
 * __host__ __device__ code): A (p x p, lower triangle used, overwritten) += diag(pscale^-2),
 * step = A^-1 g.  Returns 0 or k+1 if A is not positive definite at column k.  No GPU needed. */
int lrb_debug_chol_solve(double* A, int ld, int p, const double* pscale, const double* g, double* step);

/* lprior alone (fit-np-ul.py:33-34; no pass over X). beta: C x p host; out: C. */
int lrb_lprior(lrb_handle* h, const double* beta, int C, double* out);

/* ---- posterior predictive summaries and WAIC over posterior draws ------------------------
 * One pass over the bound rows for all S draws (draws: S x p float64, host, row-major).  With
 * eta_is = x_i . beta_s and l_is = log p(y_i | beta_s), per row i (each output n doubles, may be
 * NULL: a NULL output is neither computed into HBM nor copied):
 *   prob_mean[i] = mean_s sigmoid(eta_is)     prob_sd[i] = sd_s sigmoid(eta_is)   (ddof 1)
 *   lppd[i]      = log mean_s exp(l_is)       p_waic[i]  = var_s l_is             (ddof 1)
 * (prob_sd and p_waic are NaN for S = 1.)  `location` (LRB_HOST / LRB_DEVICE) says where the four
 * output pointers live.  totals (may be NULL): lppd = sum lppd[i], p_waic = sum p_waic[i],
 * elpd_waic = lppd - p_waic, se_elpd_waic = sqrt(n var_i(lppd[i] - p_waic[i])) (ddof 1).
 * Arithmetic of the mode: eta in float32 (FP32, beta rounded to float) or float64 (FP64); the
 * statistics are accumulated in float64.  Results are bit-reproducible for a fixed shape.  The
 * sampler state and a paused chain are untouched.  Row-sharded handles: LRB_E_UNSUPPORTED. */
typedef struct lrb_predictive_totals {
  int64_t n;            /* rows scored (this handle's rows) */
  int64_t draws;        /* S */
  double lppd, p_waic, elpd_waic, se_elpd_waic;
} lrb_predictive_totals;   /* 48 bytes */
int lrb_predictive(lrb_handle* h, const double* draws, int64_t S, int location,
                   double* prob_mean, double* prob_sd, double* lppd, double* p_waic,
                   lrb_predictive_totals* totals);

/* ---- PSIS-LOO cross-validation and the pointwise log-likelihood over posterior draws ---------
 * Pareto-smoothed importance-sampling leave-one-out (Vehtari, Simpson, Gelman, Yao & Gabry 2024),
 * exactly R's loo package: psis() with r_eff = 1 (generalized Pareto fit of Zhang & Stephens 2009
 * with loo's weak prior and wip adjustment; tail length M = ceil(min(0.2 S, 3 sqrt(S))); no
 * smoothing and k-hat = +inf when M < 5, i.e. S < 21, or the tail is constant).  Per row i, with
 * l_is = log p(y_i | beta_s) and lw_i the log weights of the log ratios -l_i:
 *   elpd_loo[i] = log sum_s exp(lw_is + l_is) - log sum_s exp(lw_is)
 *   p_loo[i]    = lppd_i - elpd_loo[i]       (lppd_i = log mean_s exp(l_is))
 *   pareto_k[i] = k-hat of the row (the reliability diagnostic of elpd_loo[i])
 * draws: S x p float64, host, row-major; 1 <= S <= 2^21.  Each per-row output (n doubles) may be
 * NULL; `location` (LRB_HOST / LRB_DEVICE) says where they live.  totals (may be NULL):
 * elpd_loo and p_loo summed over the rows, se_* = sqrt(n var_i(.)) (ddof 1), looic = -2 elpd_loo,
 * k_threshold = min(1 - 1/log10 S, 0.7) (loo >= 2.7), k_max and n_k_high = #{i : pareto_k[i] >
 * k_threshold}.  Rows are scored in chunks through a bounded scratch matrix; results are
 * bit-reproducible for a fixed shape.  The sampler state and a paused chain are untouched.
 * Row-sharded handles: LRB_E_UNSUPPORTED.
 * Benchmark switch: with the environment variable LRB_LOO_STAGE1_ONLY set, only the
 * log-likelihood stage runs (to time it alone); every per-row output and every floating-point
 * total is then NaN and n_k_high is -1.  LRB_LOO_CHUNK_MB overrides the 64 MB scratch budget. */
typedef struct lrb_loo_totals {
  int64_t n, draws;
  double elpd_loo, se_elpd_loo, p_loo, se_p_loo, looic;
  double k_threshold, k_max;
  int64_t n_k_high;
} lrb_loo_totals;                                   /* 80 bytes */
int lrb_loo(lrb_handle* h, const double* draws, int64_t S, int location,
            double* elpd_loo, double* p_loo, double* pareto_k, lrb_loo_totals* totals);
/* l_is = log p(y_i | beta_s) for the bound rows [row0, row0 + nrows) and all S draws (1 <= S <=
 * 2^21): out is nrows x S, row-major, float64, on the host or the device (`location`); the matrix
 * loo::loo() and ArviZ take, transposed.  Host output is copied chunk by chunk (bounded device
 * memory).  Arithmetic of the mode, as lrb_predictive.  Row-sharded handles: LRB_E_UNSUPPORTED. */
int lrb_loglik(lrb_handle* h, const double* draws, int64_t S, int64_t row0, int64_t nrows,
               int location, double* out);          /* out: nrows x S, row-major, float64 */
/* loo's psis() of one row on the host, the same formulas psis_kernel runs (no GPU needed):
 * log_ratios[S] -> log_weights[S] (smoothed, truncated at the largest raw weight) and k-hat. */
int lrb_debug_psis(const double* log_ratios, int64_t S, double* log_weights, double* khat);

/* ---- samplers: mcmc(init, kernel, thin, iters) -------------------------------
 * Runs the whole chain on the device (no per-iteration host round trip):
 * replaces `mcmc` (fit-numpy.py:64-79, fit-np-ul.py:70-84) driving `mhKernel` /
 * `ulKernel` / `malaKernel` / `hmcKernel`.  init: C x p (host) or NULL to
 * continue the chain(s) from the previous lrb_run on this handle.  out: C x iters x p
 * (row i of chain c = state after (i+1)*thin kernel applications; init is never
 * stored, fit-numpy.py:71-76).  accepted: C counters (may be NULL).
 * replay_z: C x (thin*iters) x p and replay_u: C x (thin*iters) (host) when
 * params->rng == LRB_RNG_REPLAY (replay_u unused for UL). */
int lrb_run(lrb_handle* h, const lrb_sampler_params* params, const double* init, int C,
            int64_t thin, int64_t iters, const double* replay_z, const double* replay_u,
            double* out, int64_t* accepted);

/* The same run split in three so the device part can be timed alone:
 * begin (upload init/params, build the launch graph), launch (enqueue the whole
 * chain asynchronously; repeatable: each call continues the chain and overwrites
 * the same sample buffer), finish (synchronise, copy samples out). Single chain. */
int lrb_run_begin(lrb_handle* h, const lrb_sampler_params* params, const double* init,
                  int64_t thin, int64_t iters, const double* replay_z, const double* replay_u);
int lrb_run_launch(lrb_handle* h);
int lrb_run_finish(lrb_handle* h, double* out, int64_t* accepted);
/* Current state of the (paused) chain: x[p], the cached log-density carried with it
 * (what kernel(x, ll) returns as ll) and the number of kernel applications so far. */
int lrb_chain_state(lrb_handle* h, double* x, double* lpost, int64_t* steps);
/* fused evaluations one lrb_run_launch enqueues (e.g. thin*iters*l for HMC) */
int lrb_run_evals_per_launch(const lrb_handle* h, int64_t* evals);

/* Running moments of the thinned states of the latest LRB_RUN_MOMENTS run.
 * pooled == 0: count[C], mean[C x p], cov[C x p x p] per chain (C = chains of that run);
 * pooled != 0: all chains combined into count[1], mean[p], cov[p x p].
 * cov = sum (x - mean)(x - mean)' / (count - 1) (Dex/djwutils.dx:100-102); cov may be NULL. */
int lrb_run_moments(lrb_handle* h, int pooled, int64_t* count, double* mean, double* cov);

/* split(key, n)[i] of the keyed front-end: words (x, y) of Philox4x32-10 at counter
 * (i_lo, i_hi, 0, 4) under `key`.  Pure host arithmetic (no GPU needed). */
uint64_t lrb_key_child(uint64_t key, uint64_t i);

/* Dump the device RNG stream: z_out[count x p] and u_out[count] for iterations
 * t0 .. t0+count-1 under `seed` (what LRB_RNG_PHILOX feeds the samplers). */
int lrb_rng_dump(lrb_handle* h, uint64_t seed, int64_t t0, int64_t count, int p,
                 double* z_out, double* u_out);

/* ---- row-sharded multi-GPU (one process per GPU) ------------------------------
 * Precedent: the Spark map/reduce of ll over row partitions,
 * Scala/spark/src/main/scala/fit-spark.scala:54-58.  Each rank binds its row
 * block; each evaluation's (p+1) partial sums [ll, X'(y-p)] are summed over ranks.
 *   NCCL: ncclAllReduce(sum, float64, p+1) between the fused kernel and the
 *         sampler update (captured in the launch graph);
 *   P2P : the fused kernel's last CTA stores its sums into every peer's mailbox
 *         over NVLink and combines the peers' sums in rank order in the same
 *         kernel (one launch per evaluation, no separate collective). */
int lrb_nccl_unique_id(void* id_out_128_bytes, const char* libnccl_path);
int lrb_comm_init_nccl(lrb_handle* h, int rank, int world, const void* unique_id_128_bytes,
                       const char* libnccl_path);
/* P2P: each rank exports a 64-byte IPC handle of its mailbox, the caller
 * all-gathers them (torch.distributed is the plumbing), every rank connects. */
int lrb_comm_p2p_export(lrb_handle* h, void* ipc_handle_out_64_bytes);
int lrb_comm_p2p_connect(lrb_handle* h, int rank, int world, const void* all_ipc_handles);

#ifdef __cplusplus
}
#endif
#endif /* LOGREG_B200_H */
