// sampler.cuh -- on-device sampler state machine (RWMH / UL / MALA / HMC) and the
// "finish" step that turns the reduced row sums into lpost / glp.
//
// One CTA of kBlock threads executes these functions; thread j owns coefficient j.
// Every reduction over coefficients is a fixed-order block sum, so all ranks of a
// row-sharded run (same inputs after the allreduce, same code) take bit-identical
// decisions without any broadcast (SURVEY.md section 8e).
//
// Reference semantics followed (paths relative to the reference root):
//   RWMH  Python/fit-numpy.py:53-62 (mhKernel), :81-84 (rprop), :64-79 (mcmc)
//   UL    Python/fit-np-ul.py:61-68 (ulKernel), :70-84 (mcmc)
//   MALA  Python/fit-np-mala.py:61-70 (mhKernel), :72-78 (malaKernel), :80-95 (mcmc)
//   HMC   Python/fit-np-hmc.py:56-63 (mhKernel), :65-87 (hmcKernel), :89-103 (mcmc)
// What differs, by design: the reference re-evaluates glp/lpost at the current
// state on every step (7 passes over X per MALA step, 2l+4 per HMC step); here
// (lpost, glp) of the current state are cached, so MALA costs ONE fused pass and
// HMC costs l (BASELINE.md section 2).  The MALA acceptance ratio uses the closed
// form in which the Gaussian normalisers cancel (Dex/fit-mala.dx:65-68).
#pragma once
#include "common.cuh"

namespace lrb {

enum { PH_PAUSED = 0, PH_INIT = 1, PH_STEP = 2 };
enum { S_RWMH = 0, S_UL = 1, S_MALA = 2, S_HMC = 3 };
enum { RNG_PHILOX = 0, RNG_REPLAY = 1, RNG_KEYED = 2 };

struct SamplerState {
  int32_t kind, l, p, rng;
  double step, sqrt_step;
  uint64_t seed;
  long long t;          // kernel applications completed since the chain began
  long long t_run0;     // t when the current run began (thinning rows count from here)
  long long t_replay0;  // t at which the replay arrays start
  long long t_end;      // pause when t reaches this
  long long thin;
  long long accepted;   // accepted proposals since the chain began
  int32_t phase, leap;
  double lp_x;          // cached lpost(x); -inf until first known (fit-numpy.py:66)
  double k0;            // HMC: kinetic energy at the start of the trajectory
  const double* z;      // replay normals [steps][p]
  const double* u;      // replay uniforms [steps]
  double* out;          // thinned samples [iters][p]; nullptr = do not store (moments only)
  // running moments of the thinned states (Dex/djwutils.dx:97-103 meanAndCovariance), or nullptr
  double* mom_mean;     // [p]
  double* mom_m2;       // [p][p] sum of (x - mean_before)(x - mean_after)'
  long long mom_count;
  double x[kMaxP], gx[kMaxP], q[kMaxP], mom[kMaxP];
  double scale[kMaxP], sqrt_scale[kMaxP];
  double beta_in[kMaxP];  // where the next fused evaluation happens
  double d1[kMaxP], d2[kMaxP];  // scratch of the moment update
  // Draws computed ahead of the evaluation that needs them (drive mode keeps a shared-memory copy
  // of the state in every CTA and fills these while X streams, so Philox / Box-Muller / log are off
  // the serial tail).  Never set in the global copy (cache_has == 0 there).
  int32_t cache_has, cache_pad;   // bit 0: cache_z0 = z(cache_t, .), bit 1: cache_z1 = z(cache_t+1, .), bit 2: cache_logu = log u(cache_t)
  long long cache_t;
  double cache_logu;
  double cache_z0[kMaxP], cache_z1[kMaxP];
};
// everything before x[] is the scalar header, copied as 8-byte words
constexpr size_t kStateHeaderWords = offsetof(SamplerState, x) / 8;
static_assert(offsetof(SamplerState, x) % 8 == 0, "header is copied as 8-byte words");

struct FinishArgs {
  const double* beta;        // the evaluated point (device, p doubles)
  const double* pscale;      // prior sd, p doubles
  const double* log_pscale;  // log(pscale)
  double* res;               // [lpost, ll, lprior, glp[0..p)]
  SamplerState* state;       // nullptr for a bare evaluation
  int32_t p, world, rank, p2p;
  // fused peer-memory allreduce (comm.cuh)
  double* mailbox_local;
  unsigned long long* flags_local;
  double* mailbox_peer[kMaxRanks];
  unsigned long long* flags_peer[kMaxRanks];
  unsigned long long* seq;
  int* comm_error;           // set to 1 if a peer's sums did not arrive within timeout_ns (a rank died)
  long long timeout_ns;      // bound of the peer wait (%globaltimer); LRB_P2P_TIMEOUT_MS, default 60 s
};

__device__ __forceinline__ long long globaltimer_ns() {
  long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

constexpr int kMailStride = kMaxP + 1;  // doubles per (slot, rank) mailbox entry

// Where a chain's draws come from (a register-sized view of the state header).
struct DrawSrc {
  int32_t rng, kind, p;
  uint64_t seed;
  long long t_run0, thin, t_replay0;
  const double* z;
  const double* u;
};
__device__ inline DrawSrc draw_src(const SamplerState* st) {
  return DrawSrc{st->rng, st->kind, st->p, st->seed, st->t_run0, st->thin, st->t_replay0, st->z, st->u};
}

// Keyed mode (the JAX-style front-end, Python/fit-jax2.py:98-116): the key of kernel application
// t of a run is split(split(root, iters)[t / thin], thin)[t % thin]; the kernels then split it as
// the reference kernels do (mhKernel fit-jax2.py:90: key0 -> proposal noise, key1 -> uniform;
// hmcKernel fit-jax-hmc.py:126-129: key0 -> momentum, key1 -> mhKernel -> its key1 -> uniform;
// ulKernel fit-jax-ul.py:86-88: the step key itself -> noise).
__device__ inline uint64_t step_key(const DrawSrc& d, long long t) {
  const long long rel = t - d.t_run0;
  return philox_child(philox_child(d.seed, (uint64_t)(rel / d.thin)), (uint64_t)(rel % d.thin));
}
__device__ inline double draw_z_raw(const DrawSrc& d, long long t, int j) {
  if (d.rng == RNG_REPLAY) return d.z[(t - d.t_replay0) * d.p + j];
  if (d.rng == RNG_KEYED) {
    const uint64_t k = step_key(d, t);
    return philox_normal(d.kind == S_UL ? k : philox_child(k, 0), 0ull, (uint32_t)j);
  }
  return philox_normal(d.seed, (uint64_t)t, (uint32_t)j);
}
__device__ inline double draw_u_raw(const DrawSrc& d, long long t) {
  if (d.rng == RNG_REPLAY) return d.u[t - d.t_replay0];
  if (d.rng == RNG_KEYED) {
    uint64_t k = philox_child(step_key(d, t), 1);
    if (d.kind == S_HMC) k = philox_child(k, 1);
    return philox_uniform(k, 0ull);
  }
  return philox_uniform(d.seed, (uint64_t)t);
}
__device__ inline double draw_z(const SamplerState* st, long long t, int j) {
  if ((st->cache_has & 1) && t == st->cache_t) return st->cache_z0[j];
  if ((st->cache_has & 2) && t == st->cache_t + 1) return st->cache_z1[j];
  return draw_z_raw(draw_src(st), t, j);
}
__device__ inline double draw_u(const SamplerState* st, long long t) { return draw_u_raw(draw_src(st), t); }
__device__ inline double draw_logu(const SamplerState* st, long long t) {
  if ((st->cache_has & 4) && t == st->cache_t) return st->cache_logu;
  return log(draw_u(st, t));
}

// Drive mode, while X streams: compute the draws the evaluation now under way will need if it
// completes a kernel application, into the CTA's shared-memory copy `dst` of the state whose home
// is `src` (global; read with ld.cg: another SM wrote it).  Threads j < p and thread 0 take part;
// no barrier inside -- the results are consumed after the CTA-wide barrier of the reduction.
__device__ inline void sampler_precompute_draws(SamplerState* dst, const SamplerState* src) {
  const int j = threadIdx.x;
  const int p = __ldcg(&src->p);
  if (j >= p) return;
  DrawSrc d;
  d.rng = __ldcg(&src->rng); d.kind = __ldcg(&src->kind); d.p = p;
  d.seed = __ldcg(&src->seed);
  d.t_run0 = __ldcg(&src->t_run0); d.thin = __ldcg(&src->thin); d.t_replay0 = __ldcg(&src->t_replay0);
  d.z = reinterpret_cast<const double*>(__ldcg(reinterpret_cast<const unsigned long long*>(&src->z)));
  d.u = reinterpret_cast<const double*>(__ldcg(reinterpret_cast<const unsigned long long*>(&src->u)));
  const int phase = __ldcg(&src->phase), leap = __ldcg(&src->leap), l = __ldcg(&src->l);
  const long long t = __ldcg(&src->t), t_end = __ldcg(&src->t_end);
  const bool completes = phase == PH_STEP && (d.kind != S_HMC || leap == l - 1);
  int has = 0;
  if (phase == PH_INIT || (completes && d.kind == S_UL)) {
    dst->cache_z0[j] = draw_z_raw(d, t, j);   // proposal from the initial state / the UL noise
    has |= 1;
  }
  if (completes && d.kind != S_UL) {
    if (t + 1 < t_end) {                       // the proposal of the next application
      dst->cache_z1[j] = draw_z_raw(d, t + 1, j);
      has |= 2;
    }
    if (j == 0) dst->cache_logu = log(draw_u_raw(d, t));
    has |= 4;
  }
  if (j == 0) { dst->cache_t = t; dst->cache_has = has; }
}

// Shared-memory working copy of a chain's state <-> its home in global memory (whole CTA).
__device__ inline void state_load(SamplerState* dst, const SamplerState* src) {
  const int tid = threadIdx.x;
  const unsigned long long* s8 = reinterpret_cast<const unsigned long long*>(src);
  unsigned long long* d8 = reinterpret_cast<unsigned long long*>(dst);
  for (int i = tid; i < (int)kStateHeaderWords; i += kBlock) d8[i] = __ldcg(s8 + i);
  const int p = __ldcg(&src->p);
  for (int j = tid; j < p; j += kBlock) {
    dst->x[j] = __ldcg(src->x + j); dst->gx[j] = __ldcg(src->gx + j);
    dst->q[j] = __ldcg(src->q + j); dst->mom[j] = __ldcg(src->mom + j);
    dst->scale[j] = __ldcg(src->scale + j); dst->sqrt_scale[j] = __ldcg(src->sqrt_scale + j);
    dst->beta_in[j] = __ldcg(src->beta_in + j);
  }
}
__device__ inline void state_store(SamplerState* dst, const SamplerState* src) {
  const int tid = threadIdx.x;
  const unsigned long long* s8 = reinterpret_cast<const unsigned long long*>(src);
  unsigned long long* d8 = reinterpret_cast<unsigned long long*>(dst);
  for (int i = tid; i < (int)kStateHeaderWords; i += kBlock) d8[i] = s8[i];
  const int p = src->p;
  for (int j = tid; j < p; j += kBlock) {
    dst->x[j] = src->x[j]; dst->gx[j] = src->gx[j]; dst->q[j] = src->q[j]; dst->mom[j] = src->mom[j];
    dst->beta_in[j] = src->beta_in[j];
  }
}

// Generate the next evaluation point from the current state (x, gx) with the
// draws of iteration st->t.  Called by the whole CTA.
__device__ inline void sampler_propose(SamplerState* st, double* scratch) {
  const int j = threadIdx.x;
  const bool act = j < st->p;
  const long long t = st->t;
  const int kind = st->kind;
  double ksum = 0.0;
  if (act) {
    const double x = st->x[j];
    if (kind == S_RWMH) {
      // fit-numpy.py:84: beta + 0.02*pre*randn(p), scale = 0.02*pre
      st->beta_in[j] = x + st->scale[j] * draw_z(st, t, j);
    } else if (kind == S_UL) {
      st->beta_in[j] = x;  // the evaluation at x IS the step (fit-np-ul.py:65)
    } else if (kind == S_MALA) {
      // fit-np-mala.py:76-77: advance(x) + randn(p)*spre*sdt
      const double adv = x + 0.5 * st->scale[j] * st->gx[j] * st->step;
      const double prop = adv + draw_z(st, t, j) * st->sqrt_scale[j] * st->sqrt_step;
      st->q[j] = prop;
      st->beta_in[j] = prop;
    } else {
      // fit-np-hmc.py:85 p = randn(d)*sdmm; :68 half kick with the cached gradient; :70 drift
      const double dmm = st->scale[j];
      double m = draw_z(st, t, j) * st->sqrt_scale[j];
      ksum = (m * m) / dmm;
      m = m + 0.5 * st->step * st->gx[j];
      const double q = x + st->step * m / dmm;
      st->mom[j] = m;
      st->q[j] = q;
      st->beta_in[j] = q;
    }
  }
  if (kind == S_HMC) {
    const double k0 = 0.5 * block_sum(ksum, scratch);
    if (j == 0) { st->k0 = k0; st->leap = 0; }
  }
}

// Consume one fused evaluation (lp = lpost, g = this thread's glp component at
// st->beta_in) and advance the chain until the next evaluation point is known.
__device__ inline void sampler_on_eval(SamplerState* st, double lp, double g, double* scratch) {
  const int j = threadIdx.x;
  const int p = st->p;
  const bool act = j < p;
  const int kind = st->kind;
  const int phase = st->phase;
  const double lp_x = st->lp_x;
  const long long t = st->t;
  const int leap_now = st->leap;
  __syncthreads();  // everyone has read the scalars thread 0 is about to change
  if (phase == PH_PAUSED) return;

  if (phase == PH_INIT) {
    // evaluation at the initial state: cache its gradient (and, for HMC, lpost).
    // MALA/RWMH keep lp_x = -inf: the reference never evaluates lpost(init) and
    // always accepts the first proposal (fit-np-mala.py:82).
    if (act) st->gx[j] = g;
    if (j == 0) {
      if (kind == S_HMC) st->lp_x = lp;
      st->phase = PH_STEP;
    }
    __syncthreads();
    sampler_propose(st, scratch);
    return;
  }

  bool stepped = true;  // did this evaluation complete a kernel application?
  bool acc = false;

  if (kind == S_RWMH) {
    // fit-numpy.py:57-60 (dprop cancels): a = lp - ll; accept iff log(u) < a
    const double a = lp - lp_x;
    acc = draw_logu(st, t) < a;
    __syncthreads();
    if (acc && act) st->x[j] = st->beta_in[j];
  } else if (kind == S_UL) {
    // fit-np-ul.py:65-67
    if (act) {
      const double adv = st->x[j] + 0.5 * st->scale[j] * g * st->step;
      st->x[j] = adv + draw_z(st, t, j) * st->sqrt_scale[j] * st->sqrt_step;
    }
    acc = true;
  } else if (kind == S_MALA) {
    // fit-np-mala.py:65 with dprop(new, old) = sum logpdf(new; advance(old), spre*sdt):
    // a = lp - ll - 1/2 sum((x - adv(prop))/s)^2 + 1/2 sum((prop - adv(x))/s)^2
    double fwd = 0.0, bwd = 0.0;
    if (act) {
      const double pre = st->scale[j], s = st->sqrt_scale[j] * st->sqrt_step;
      const double x = st->x[j], prop = st->q[j];
      const double adv_x = x + 0.5 * pre * st->gx[j] * st->step;
      const double adv_p = prop + 0.5 * pre * g * st->step;
      const double zf = (prop - adv_x) / s, zb = (x - adv_p) / s;
      fwd = zf * zf;
      bwd = zb * zb;
    }
    fwd = block_sum(fwd, scratch);
    bwd = block_sum(bwd, scratch);
    const double a = lp - lp_x + (-0.5 * bwd) - (-0.5 * fwd);
    acc = draw_logu(st, t) < a;
    __syncthreads();
    if (acc && act) { st->x[j] = st->q[j]; st->gx[j] = g; }
  } else {
    const int leap = leap_now;
    if (leap < st->l - 1) {
      // fit-np-hmc.py:70-72: full kick then drift
      if (act) {
        const double m = st->mom[j] + st->step * g;
        const double q = st->q[j] + st->step * m / st->scale[j];
        st->mom[j] = m;
        st->q[j] = q;
        st->beta_in[j] = q;
      }
      __syncthreads();
      if (j == 0) st->leap = leap + 1;
      stepped = false;
    } else {
      // fit-np-hmc.py:74 last half kick; :59,:76-78 a = alpi(prop) - alpi(x)
      double ksum = 0.0;
      if (act) {
        const double m = st->mom[j] + 0.5 * st->step * g;
        st->mom[j] = m;
        ksum = (m * m) / st->scale[j];
      }
      const double k1 = 0.5 * block_sum(ksum, scratch);
      const double a = (lp - k1) - (lp_x - st->k0);
      acc = draw_logu(st, t) < a;
      __syncthreads();
      if (acc && act) { st->x[j] = st->q[j]; st->gx[j] = g; }
    }
  }
  if (!stepped) return;

  __syncthreads();
  const long long t1 = t + 1;
  const long long done_in_run = t1 - st->t_run0;
  const bool emit = (done_in_run % st->thin) == 0;
  const bool last = (t1 == st->t_end);
  if (emit && act && st->out != nullptr) st->out[(done_in_run / st->thin - 1) * p + j] = st->x[j];
  if (emit && st->mom_mean != nullptr) {
    // Welford update of mean and cross-moments with the thinned state
    const double k = (double)(st->mom_count + 1);
    if (act) {
      const double xj = st->x[j], m0 = st->mom_mean[j];
      const double da = xj - m0;
      const double m1 = m0 + da / k;
      st->mom_mean[j] = m1;
      st->d1[j] = da;
      st->d2[j] = xj - m1;
    }
    __syncthreads();
    for (int idx = j; idx < p * p; idx += kBlock) st->mom_m2[idx] += st->d1[idx / p] * st->d2[idx % p];
  }
  __syncthreads();
  if (j == 0) {
    st->t = t1;
    if (acc) {
      if (kind != S_UL) st->lp_x = lp;
      st->accepted += 1;
    }
    if (emit && st->mom_mean != nullptr) st->mom_count += 1;
    if (last) st->phase = PH_PAUSED;
  }
  __syncthreads();
  if (!last) sampler_propose(st, scratch);
}

// Arm the state(s) for a run of `steps` kernel applications. init == nullptr
// continues from the paused chain.  Launched as <<<C, kBlock>>>: block c arms chain c
// (states[c], init + c*p, Philox key seed + c*golden, replay rows c*steps.., samples
// out + c*iters*p).
__global__ void sampler_begin_kernel(SamplerState* states, const double* init, const double* scale,
                                     int kind, int l, int p, int rng, double step, uint64_t seed,
                                     double init_lpost, long long steps, long long thin, const double* z,
                                     const double* u, double* out, int reuse_cache, long long t0,
                                     double* mom_mean, double* mom_m2) {
  __shared__ double scratch[kWarps];
  const int j = threadIdx.x;
  const long long c = blockIdx.x;
  SamplerState* st = states + c;
  if (init) init += c * p;
  if (j < p) {
    st->scale[j] = scale[j];
    st->sqrt_scale[j] = sqrt(scale[j]);
    if (init) st->x[j] = init[j];
  }
  if (j == 0) {
    st->kind = kind; st->l = l; st->p = p; st->rng = rng;
    st->step = step; st->sqrt_step = sqrt(step);
    st->seed = seed + (uint64_t)c * 0x9E3779B97F4A7C15ull;
    if (init) {
      st->t = t0; st->accepted = 0; st->k0 = 0.0;   // t0 != 0: a chain resumed at Philox counter t0
      if (!(reuse_cache && kind == S_HMC)) st->lp_x = init_lpost;   // HMC keeps the cached lpost(x)
    }
    st->t_run0 = st->t;
    st->t_replay0 = st->t;
    st->t_end = st->t + steps;
    st->thin = thin;
    st->z = z ? z + c * steps * p : nullptr;
    st->u = u ? u + c * steps : nullptr;
    st->out = out ? out + c * (steps / thin) * p : nullptr;
    st->leap = 0;
    st->cache_has = 0; st->cache_t = -1;
    st->mom_mean = mom_mean ? mom_mean + c * p : nullptr;
    st->mom_m2 = mom_m2 ? mom_m2 + c * (long long)p * p : nullptr;
    if (init || mom_mean == nullptr) st->mom_count = 0;
  }
  if (init && mom_mean != nullptr) {   // a new chain starts with empty moments
    if (j < p) mom_mean[c * p + j] = 0.0;
    for (int idx = j; idx < p * p; idx += kBlock) mom_m2[c * (long long)p * p + idx] = 0.0;
  }
  __syncthreads();
  if (steps <= 0) { if (j == 0) st->phase = PH_PAUSED; return; }
  // Which samplers need the gradient (and lpost) of the starting state first?
  // A continued MALA/HMC chain still has them cached.
  const bool need_init = init != nullptr && !reuse_cache && (kind == S_MALA || kind == S_HMC);
  if (need_init) {
    if (j < p) st->beta_in[j] = st->x[j];
    if (j == 0) st->phase = PH_INIT;
  } else {
    if (j == 0) st->phase = PH_STEP;
    __syncthreads();
    sampler_propose(st, scratch);
  }
}

// Warm L1 with everything finish_eval / sampler_on_eval will read, so those (dependent) loads
// overlap the reduction of the CTA partials instead of following it.  Call only after the
// gpu-scope fence that follows the ticket (it invalidates this SM's L1).
__device__ inline void prefetch_finish_inputs(const FinishArgs& f) {
  const int j = threadIdx.x;
  auto pf = [](const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); };
  if (j < f.p) {
    pf(f.beta + j); pf(f.pscale + j); pf(f.log_pscale + j);
    if (f.state) {
      const SamplerState* st = f.state;
      pf(st->x + j); pf(st->gx + j); pf(st->q + j); pf(st->mom + j); pf(st->scale + j); pf(st->sqrt_scale + j);
    }
  }
  if (j == 0 && f.state) pf(f.state);
}

// ---------------------------------------------------------------- finish
// sums (shared memory, p+1 doubles): [ll, X'(y-p)] summed over all rows of this
// rank.  Combines across ranks (fused peer-memory mode), adds the prior
// (fit-np-ul.py:33-34,46), publishes [lpost, ll, glp] and feeds the sampler.
// `st`, `beta`, `pscale`, `log_pscale` default to f's; drive mode passes its shared-memory copies.
__device__ inline void finish_eval(const FinishArgs& f, double* sums, double* scratch, SamplerState* st,
                                   const double* beta, const double* pscale, const double* log_pscale) {
  const int j = threadIdx.x;
  const int p = f.p;
  const bool act = j < p;

  if (f.p2p && f.world > 1) {
    __shared__ int s_timed_out;
    if (j == 0) s_timed_out = 0;
    // One-shot allreduce over NVLink peer memory: store my sums into slot
    // (seq&1, my rank) of every peer's mailbox, publish a flag, wait for every
    // peer's flag, add in rank order.  Two slots suffice: a peer cannot run two
    // evaluations ahead because it needs my sums of evaluation k to finish k.
    const unsigned long long seq = *f.seq;
    const int slot = (int)(seq & 1ull);
    for (int r = 0; r < f.world; ++r) {
      if (r == f.rank) continue;
      double* dst = f.mailbox_peer[r] + ((size_t)slot * kMaxRanks + f.rank) * kMailStride;
      for (int c = j; c <= p; c += kBlock) dst[c] = sums[c];
    }
    // No system fence per thread: the CTA barrier orders every thread's remote stores before the
    // st.release.sys of the flag (release is cumulative over what happens-before it), which is
    // the single system-scope fence of the exchange.
    if (f.p2p & 2) __threadfence_system();   // A/B knob (LRB_P2P_FENCE=1): the conservative variant
    __syncthreads();
    if (j < f.world && j != f.rank) {
      unsigned long long* fl = f.flags_peer[j] + (size_t)slot * kMaxRanks + f.rank;
      asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(fl), "l"(seq + 1) : "memory");
      const unsigned long long* mine = f.flags_local + (size_t)slot * kMaxRanks + j;
      unsigned long long got;
      const long long t_start = globaltimer_ns();
      unsigned int spins = 0;
      do {
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(got) : "l"(mine) : "memory");
        if (got < seq + 1 && (++spins & 0x3ffu) == 0 && globaltimer_ns() - t_start > f.timeout_ns) {
          // a peer is gone (or hopelessly late): do not hang the GPU; the host turns this into LRB_E_NCCL
          if (f.comm_error) *f.comm_error = 1;
          s_timed_out = 1;
          break;
        }
      } while (got < seq + 1);
    }
    __syncthreads();
    const bool poisoned = s_timed_out != 0;
    for (int c = j; c <= p; c += kBlock) {
      double tot = 0.0;
      for (int r = 0; r < f.world; ++r) {
        const double* src = f.mailbox_local + ((size_t)slot * kMaxRanks + r) * kMailStride;
        tot += (r == f.rank) ? sums[c] : __ldcg(src + c);
      }
      // a timed-out exchange must not produce a usable number
      sums[c] = poisoned ? __longlong_as_double(0x7ff8000000000000ll) : tot;  // each thread reads and writes only its own c
    }
    __syncthreads();
    if (j == 0) *f.seq = seq + 1;
  }

  const double LOG_SQRT_2PI = 0.91893853320467274178;
  double lpr = 0.0, g = 0.0;
  if (act) {
    const double b = beta[j], ps = pscale[j];
    const double zz = b / ps;
    lpr = -(zz * zz) / 2.0 - LOG_SQRT_2PI - log_pscale[j];
    g = -b / (ps * ps) + sums[1 + j];
  }
  const double lprior = block_sum(lpr, scratch);
  const double ll = sums[0];
  const double lpost = ll + lprior;
  if (j == 0) { f.res[0] = lpost; f.res[1] = ll; f.res[2] = lprior; }
  if (act) f.res[3 + j] = g;
  if (st) {
    __syncthreads();
    sampler_on_eval(st, lpost, g, scratch);
  }
}
__device__ inline void finish_eval(const FinishArgs& f, double* sums, double* scratch) {
  finish_eval(f, sums, scratch, f.state, f.beta, f.pscale, f.log_pscale);
}

// lprior only (no data pass): out[c] = sum_j logpdf(beta[c][j]; 0, pscale[j])
__global__ void prior_kernel(const double* beta, const double* pscale, const double* log_pscale,
                             int p, double* out) {
  __shared__ double scratch[kWarps];
  const double LOG_SQRT_2PI = 0.91893853320467274178;
  const int j = threadIdx.x;
  double lpr = 0.0;
  if (j < p) {
    const double zz = beta[(size_t)blockIdx.x * p + j] / pscale[j];
    lpr = -(zz * zz) / 2.0 - LOG_SQRT_2PI - log_pscale[j];
  }
  const double s = block_sum(lpr, scratch);
  if (j == 0) out[blockIdx.x] = s;
}

// Moments out: per chain (pooled == 0: count[c], mean[c][p], cov[c][p][p]) or all chains pooled into
// one (count[0], mean[p], cov[p][p]) with the pairwise-combination formula.  cov = M2 / (count - 1)
// (Dex/djwutils.dx:100-102; numpy.cov default).  <<<pooled ? 1 : C, kBlock>>>
__global__ void moments_out_kernel(const SamplerState* states, int C, int p, int pooled, long long* count,
                                   double* mean, double* cov) {
  const int j = threadIdx.x;
  if (!pooled) {
    const SamplerState* st = states + blockIdx.x;
    const long long k = st->mom_count;
    if (j == 0) count[blockIdx.x] = k;
    if (j < p) mean[(size_t)blockIdx.x * p + j] = st->mom_mean[j];
    if (cov)
      for (int idx = j; idx < p * p; idx += kBlock)
        cov[(size_t)blockIdx.x * p * p + idx] = k > 1 ? st->mom_m2[idx] / (double)(k - 1) : 0.0;
    return;
  }
  __shared__ double s_mean[kMaxP];
  long long N = 0;
  for (int c = 0; c < C; ++c) N += states[c].mom_count;
  if (j < p) {
    double m = 0.0;
    for (int c = 0; c < C; ++c) m += (double)states[c].mom_count * states[c].mom_mean[j];
    s_mean[j] = N > 0 ? m / (double)N : 0.0;
    mean[j] = s_mean[j];
  }
  if (j == 0) count[0] = N;
  __syncthreads();
  if (cov)
    for (int idx = j; idx < p * p; idx += kBlock) {
      const int a = idx / p, b = idx % p;
      double m2 = 0.0;
      for (int c = 0; c < C; ++c) {
        const SamplerState* st = states + c;
        m2 += st->mom_m2[idx] + (double)st->mom_count * (st->mom_mean[a] - s_mean[a]) * (st->mom_mean[b] - s_mean[b]);
      }
      cov[idx] = N > 1 ? m2 / (double)(N - 1) : 0.0;
    }
}

}  // namespace lrb
