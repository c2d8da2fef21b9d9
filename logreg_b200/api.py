"""The reference-facing Python API: same names and call signatures as the
reference's NumPy scripts, backed by the CUDA library.

Reference definitions mirrored (paths relative to the reference root):
    ll        Python/fit-numpy.py:23-24        lprior   Python/fit-np-ul.py:33-34
    lpost     Python/fit-numpy.py:43-44        glp      Python/fit-np-ul.py:45-48
    mhKernel  Python/fit-numpy.py:53-62 and Python/fit-np-hmc.py:56-63
    ulKernel  Python/fit-np-ul.py:61-68        malaKernel  Python/fit-np-mala.py:72-78
    hmcKernel Python/fit-np-hmc.py:65-87       mcmc  Python/fit-numpy.py:64-79, fit-np-ul.py:70-84

The scripts close over module globals (X, y, pscale, init); a script switches to
this backend with

    from logreg_b200 import *          # instead of defining ll/lprior/lpost/glp/...Kernel/mcmc
    bind_data(X, y, pscale)            # the one extra line: closures cannot be imported

Beyond the reference, a Problem scores its bound rows under posterior draws on the device:
`predictive` (posterior predictive probabilities, lppd, WAIC), `loo` (PSIS-LOO: elpd_loo, p_loo and
the Pareto k-hat of every row, as R's loo package computes them) and `loglik` (the pointwise
log-likelihood matrix).

Everything numeric runs on the GPU; without a CUDA device every call raises
`LogregB200Error` (there is no CPU fallback).
"""
from __future__ import annotations

import ctypes as C
import inspect

import numpy as np

from . import _native as N
from ._native import LogregB200Error

_MODES = {"fp64": N.MODE_FP64, "fp32": N.MODE_FP32, N.MODE_FP64: N.MODE_FP64, N.MODE_FP32: N.MODE_FP32}
_REPLAY_CHUNK_BYTES = 64 << 20
_PREDICTIVE_OUTPUTS = ("prob_mean", "prob_sd", "lppd", "p_waic")   # argument order of lrb_predictive
_LOO_OUTPUTS = ("elpd_loo", "p_loo", "pareto_k")                    # argument order of lrb_loo


def _vec(v, p, name):
    """scalar or length-p -> float64 vector of length p (the reference's `pre=1`, `dmm=1` defaults)."""
    a = np.asarray(v, dtype=np.float64)
    if a.ndim == 0:
        a = np.full(p, float(a))
    if a.shape != (p,):
        raise ValueError(f"{name} must be a scalar or have length {p}, got shape {a.shape}")
    return np.ascontiguousarray(a)


class Problem:
    """Owns one library handle: the data (the scripts' globals X, y, pscale) on one GPU."""

    def __init__(self, device: int = 0, deterministic: bool = False):
        self._lib = N.load()
        h = C.c_void_p()
        N.check(self._lib.lrb_create(int(device), C.byref(h)))
        self._h = h
        if deterministic:
            self.set_option(N.OPT_DETERMINISTIC, 1)
        self.device = int(device)
        self.n = 0
        self.p = 0
        self._cache_key = None
        self._cache = None
        self.last_accept_rate = None
        self._last_x = None          # bytes of the state the last single-chain run ended in
        self._last_sampler = None
        self.last_accepted = None
        self.world, self.rank, self.n_global = 1, 0, 0

    # ------------------------------------------------------------ lifetime
    def close(self):
        if getattr(self, "_h", None):
            self._lib.lrb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        N.check(rc, self._h)

    def set_stream(self, cuda_stream_ptr):
        self._ck(self._lib.lrb_set_stream(self._h, C.c_void_p(cuda_stream_ptr or 0)))

    def set_option(self, option: int, value: int):
        """lrb_set_option: N.OPT_DETERMINISTIC (fixed-order static kernel: bit-identical results),
        N.OPT_TC_MIN_CHAINS, N.OPT_P2P_TIMEOUT_MS, N.OPT_PDL, N.OPT_L2_PERSIST."""
        self._ck(self._lib.lrb_set_option(self._h, int(option), int(value)))

    def synchronize(self):
        self._ck(self._lib.lrb_synchronize(self._h))

    def info(self) -> dict:
        inf = N.Info()
        self._ck(self._lib.lrb_get_info(self._h, C.byref(inf)))
        return {k: getattr(inf, k) for k, _ in N.Info._fields_}

    # ------------------------------------------------------------ data
    def bind_data(self, X, y, pscale=None, mode="fp64"):
        """X: (n, p) NumPy array, float32/float64, any strides (the reference's is
        column-major float64); y: (n,) of 0/1; pscale: prior sd per coefficient."""
        X = np.asarray(X)
        if X.ndim != 2:
            raise ValueError("X must be 2-D")
        if X.dtype not in (np.float32, np.float64):
            X = X.astype(np.float64)
        n, p = X.shape
        es = X.dtype.itemsize
        if X.flags["C_CONTIGUOUS"]:
            layout, ld = N.ROW_MAJOR, p
        elif X.flags["F_CONTIGUOUS"]:
            layout, ld = N.COL_MAJOR, n
        elif X.strides[1] == es and X.strides[0] % es == 0 and X.strides[0] >= p * es:
            layout, ld = N.ROW_MAJOR, X.strides[0] // es
        elif X.strides[0] == es and X.strides[1] % es == 0 and X.strides[1] >= n * es:
            layout, ld = N.COL_MAJOR, X.strides[1] // es
        else:
            X = np.ascontiguousarray(X)
            layout, ld = N.ROW_MAJOR, p
        y = np.ascontiguousarray(y)
        if y.shape != (n,):
            raise ValueError(f"y must have shape ({n},), got {y.shape}")
        if y.dtype == np.float32:
            yd = N.F32
        elif y.dtype == np.uint8 or y.dtype == np.bool_:
            y = y.view(np.uint8)
            yd = N.U8
        else:
            y = y.astype(np.float64)
            yd = N.F64
        ps = _vec(1.0 if pscale is None else pscale, p, "pscale")
        self._ck(self._lib.lrb_bind_data(
            self._h, C.c_void_p(X.ctypes.data), N.F32 if X.dtype == np.float32 else N.F64, layout, ld,
            C.c_void_p(y.ctypes.data), yd, n, p, N.as_dp(ps), _MODES[mode], N.HOST))
        self.n, self.p, self.pscale = n, p, ps
        self.n_global = self.n_global or n
        self._cache_key = None
        self._last_x = None
        return self

    def bind_torch(self, X, y, pscale=None, mode="fp32"):
        """Bind data that already lives on this GPU as torch tensors (float32/float64 X of shape
        (n, p) with unit stride along one axis; y float32/float64/uint8). torch is only the owner
        of the buffers: the library re-lays the data out into its own storage."""
        import torch
        if not (X.is_cuda and y.is_cuda and X.dim() == 2):
            raise ValueError("bind_torch needs 2-D CUDA tensors")
        n, p = X.shape
        xd = {torch.float32: N.F32, torch.float64: N.F64}[X.dtype]
        yd = {torch.float32: N.F32, torch.float64: N.F64, torch.uint8: N.U8}[y.dtype]
        if X.stride(1) == 1:
            layout, ld = N.ROW_MAJOR, X.stride(0)
        elif X.stride(0) == 1:
            layout, ld = N.COL_MAJOR, X.stride(1)
        else:
            X = X.contiguous()
            layout, ld = N.ROW_MAJOR, p
        y = y.contiguous()
        ps = _vec(1.0 if pscale is None else pscale, p, "pscale")
        torch.cuda.current_stream(X.device).synchronize()
        self._ck(self._lib.lrb_bind_data(self._h, C.c_void_p(X.data_ptr()), xd, layout, int(ld),
                                         C.c_void_p(y.data_ptr()), yd, int(n), int(p), N.as_dp(ps),
                                         _MODES[mode], N.DEVICE))
        self.n, self.p, self.pscale = int(n), int(p), ps
        self.n_global = self.n_global or int(n)
        self._cache_key = None
        return self

    def gen_synthetic(self, n, p, mode="fp32", seed=42, beta_true=None, pscale=None, row_offset=0):
        """On-device synthetic problem (SURVEY.md 8d). Returns beta_true."""
        if beta_true is None:
            beta_true = np.random.RandomState(41).randn(p) / np.sqrt(p)
        bt = np.ascontiguousarray(beta_true, dtype=np.float64)
        if pscale is None:
            pscale = np.ones(p)
            pscale[0] = 10.0
        ps = _vec(pscale, p, "pscale")
        self._ck(self._lib.lrb_gen_synthetic(self._h, int(n), int(p), _MODES[mode], int(seed),
                                             N.as_dp(bt), N.as_dp(ps), int(row_offset)))
        self.n, self.p, self.pscale = int(n), int(p), ps
        self.n_global = self.n_global or int(n)
        self._cache_key = None
        self._last_x = None
        return bt

    def copy_rows(self, row0, nrows):
        Xo = np.empty((nrows, self.p))
        yo = np.empty(nrows, dtype=np.float32)
        self._ck(self._lib.lrb_copy_rows(self._h, int(row0), int(nrows), N.as_dp(Xo),
                                         yo.ctypes.data_as(C.POINTER(C.c_float))))
        return Xo, yo

    # ------------------------------------------------------------ evaluation
    def _beta(self, beta):
        b = np.ascontiguousarray(beta, dtype=np.float64)
        if b.shape != (self.p,):
            raise ValueError(f"beta must have shape ({self.p},), got {b.shape}")
        return b

    def eval(self, beta, want_grad=True):
        """One fused pass: returns (lpost, ll, glp or None)."""
        b = self._beta(beta)
        key = (b.tobytes(), bool(want_grad))
        if self._cache_key is not None and self._cache_key[0] == key[0] and (self._cache_key[1] or not want_grad):
            return self._cache
        lp, l = C.c_double(), C.c_double()
        g = np.empty(self.p)
        self._ck(self._lib.lrb_eval(self._h, N.as_dp(b), 1, 1 if want_grad else 0,
                                    C.byref(lp), C.byref(l), N.as_dp(g)))
        self._cache_key = key
        self._cache = (lp.value, l.value, g if want_grad else None)
        return self._cache

    def eval_many(self, B, want_grad=True):
        B = np.ascontiguousarray(B, dtype=np.float64)
        c = B.shape[0]
        lp, l, g = np.empty(c), np.empty(c), np.empty((c, self.p))
        self._ck(self._lib.lrb_eval(self._h, N.as_dp(B), c, 1 if want_grad else 0,
                                    N.as_dp(lp), N.as_dp(l), N.as_dp(g)))
        return lp, l, (g if want_grad else None)

    # the four reference callables (bound methods, so kernels can recognise them)
    def ll(self, beta):
        return self.eval(beta, want_grad=False)[1]

    def lprior(self, beta):
        b = self._beta(beta)
        out = C.c_double()
        self._ck(self._lib.lrb_lprior(self._h, N.as_dp(b), 1, C.byref(out)))
        return out.value

    def lpost(self, beta):
        return self.eval(beta, want_grad=False)[0]

    def glp(self, beta):
        return self.eval(beta, want_grad=True)[2].copy()

    # ------------------------------------------------------------ MAP (the step before the samplers)
    def map(self, init, tol=0.01, maxit=500):
        """Newton's method with the exact Hessian and step halving on the device (lrb_map;
        Python/fit-jax.py:62-79, whose tol = 0.01 and maxit = 500 are the defaults).
        Returns (beta, info dict)."""
        b0 = self._beta(init)
        out = np.empty(self.p)
        inf = N.MapInfo()
        self._ck(self._lib.lrb_map(self._h, N.as_dp(b0), float(tol), int(maxit), N.as_dp(out), C.byref(inf)))
        self._cache_key = None
        return out, {k: getattr(inf, k) for k, _ in N.MapInfo._fields_}

    def hessian(self, beta):
        """X'WX + diag(pscale^-2) = -Hessian of lpost at beta, (p, p) float64 (lrb_hessian)."""
        b = self._beta(beta)
        H = np.empty((self.p, self.p))
        self._ck(self._lib.lrb_hessian(self._h, N.as_dp(b), N.as_dp(H)))
        return H

    # ------------------------------------------------------------ posterior predictive / WAIC
    def predictive(self, draws, pointwise=True, device_out=False):
        """Posterior predictive summaries of the bound rows over posterior draws, one pass over X
        on the device (lrb_predictive). draws: (S, p), or (C, iters, p) from run_chains (flattened).

        Returns a dict with the totals lppd, p_waic, elpd_waic, se_elpd_waic, n and draws (= S), and
        with pointwise=True also out["pointwise"] = {prob_mean, prob_sd, lppd, p_waic}: per-row
        arrays of length n (the mean and sd of sigmoid(x.beta) over the draws, log of the mean
        predictive density of y, variance of the log density; sd and variance have ddof 1 and are
        NaN for S = 1). They are NumPy arrays, or float64 torch CUDA tensors with device_out=True.
        The sampler state, a paused chain and the cached evaluation are left as they were."""
        return self._predictive(draws, _PREDICTIVE_OUTPUTS if pointwise else (), device_out)

    def _predictive(self, draws, outputs, device_out):
        B = self._draws(draws)
        bufs, ptr, loc = self._row_outputs(outputs, (self.n,), device_out)
        ptrs = [C.c_void_p(ptr(bufs[k])) if k in bufs else None for k in _PREDICTIVE_OUTPUTS]
        tot = N.PredictiveTotals()
        self._ck(self._lib.lrb_predictive(self._h, N.as_dp(B), B.shape[0], loc, *ptrs, C.byref(tot)))
        out = {k: getattr(tot, k) for k, _ in N.PredictiveTotals._fields_}
        if outputs:
            out["pointwise"] = bufs
        return out

    # ------------------------------------------------------------ PSIS-LOO / pointwise log-likelihood
    def _draws(self, draws):
        B = np.asarray(draws, dtype=np.float64)
        if B.ndim == 3:
            B = B.reshape(-1, B.shape[-1])
        if B.ndim != 2 or (self.p and B.shape[1] != self.p):
            raise LogregB200Error(N.E_BAD_ARG, f"draws must have shape (S, {self.p}) or (C, iters, {self.p}), "
                                               f"got {np.shape(draws)}")
        return np.ascontiguousarray(B)

    def loo(self, draws, pointwise=True, device_out=False):
        """Pareto-smoothed importance-sampling leave-one-out cross-validation of the bound rows over
        posterior draws (lrb_loo; R's loo::loo() with r_eff = 1). draws: (S, p), or (C, iters, p)
        from run_chains (flattened); 1 <= S <= 2^21.

        Returns a dict with the totals elpd_loo, se_elpd_loo, p_loo, se_p_loo, looic, se_looic
        (= 2 se_elpd_loo), k_threshold (= min(1 - 1/log10 S, 0.7)), k_max, n_k_high (rows whose
        pareto_k exceeds k_threshold: their elpd_loo is unreliable), n and draws, and with
        pointwise=True also out["pointwise"] = {elpd_loo, p_loo, pareto_k}: per-row arrays of length
        n, NumPy arrays or float64 torch CUDA tensors with device_out=True. The sampler state, a paused
        chain and the cached evaluation are left as they were."""
        B = self._draws(draws)
        bufs, ptr, loc = self._row_outputs(_LOO_OUTPUTS if pointwise else (), (self.n,), device_out)
        ptrs = [C.c_void_p(ptr(bufs[k])) if k in bufs else None for k in _LOO_OUTPUTS]
        tot = N.LooTotals()
        self._ck(self._lib.lrb_loo(self._h, N.as_dp(B), B.shape[0], loc, *ptrs, C.byref(tot)))
        out = {k: getattr(tot, k) for k, _ in N.LooTotals._fields_}
        out["se_looic"] = 2.0 * out["se_elpd_loo"]
        if pointwise:
            out["pointwise"] = bufs
        return out

    def loglik(self, draws, row0=0, nrows=None, device_out=False):
        """log p(y_i | beta_s) for the bound rows row0 .. row0 + nrows - 1 and every draw (lrb_loglik):
        an (nrows, S) float64 array (a torch CUDA tensor with device_out=True). Its transpose is the
        S x n matrix R's loo::loo() and ArviZ take. 1 <= S <= 2^21."""
        B = self._draws(draws)
        nrows = self.n - int(row0) if nrows is None else int(nrows)
        bufs, ptr, loc = self._row_outputs(("L",), (max(nrows, 0), B.shape[0]), device_out)
        self._ck(self._lib.lrb_loglik(self._h, N.as_dp(B), B.shape[0], int(row0), nrows, loc,
                                      C.c_void_p(ptr(bufs["L"]))))
        return bufs["L"]

    def _row_outputs(self, names, shape, device_out):
        """float64 output buffers on the host or this Problem's GPU, and how to pass them."""
        if device_out:
            import torch
            dev = torch.device("cuda", self.device)
            bufs = {k: torch.empty(shape, dtype=torch.float64, device=dev) for k in names}
            torch.cuda.current_stream(dev).synchronize()
            return bufs, (lambda t: t.data_ptr()), N.DEVICE
        return {k: np.empty(shape) for k in names}, (lambda a: a.ctypes.data), N.HOST

    # ------------------------------------------------------------ sampler runs
    def _params(self, k, seed, rng, init_lpost, flags=0, t0=0):
        sp = N.SamplerParams()
        sp.sampler, sp.l, sp.step = k.sampler, int(k.l), float(k.step)
        sp.scale = N.as_dp(k.scale)
        sp.seed, sp.rng, sp.flags, sp.init_lpost = int(seed) & (2 ** 64 - 1), rng, int(flags), float(init_lpost)
        sp.t0 = int(t0)
        return sp

    def run(self, kernel, init, thin, iters, Z=None, U=None, seed=0, init_lpost=-np.inf, t0=None,
            moments=False, keep_samples=True, keyed=False):
        """One lrb_run call. init=None continues the paused chain. Returns (mat, accepted).

        t0: resume a checkpointed chain (x, lpost, steps = chain_state()) in a new handle: pass
            init=x, init_lpost=lpost, t0=steps and the same seed -- the Philox stream continues.
        moments: accumulate running mean / cross-moments of the thinned states on the device
            (read with .moments()); keep_samples=False then returns mat=None and copies nothing.
        keyed: `seed` is a JAX-style root key (logreg_b200.jaxlike); draws follow its split tree."""
        rng = N.RNG_REPLAY if Z is not None else (N.RNG_KEYED if keyed else N.RNG_PHILOX)
        ini = None if init is None else self._beta(init)
        # init is exactly where the last run of this sampler stopped: its cached gradient / lpost
        # are still valid, so the evaluation at init is skipped (same result, one pass less)
        flags = 0
        if (ini is not None and self._last_x is not None and self._last_sampler == kernel.sampler
                and kernel.sampler in (N.MALA, N.HMC) and ini.tobytes() == self._last_x):
            flags = N.RUN_REUSE_CACHE
        if t0 is not None:
            flags |= N.RUN_SET_T0
        if moments:
            flags |= N.RUN_MOMENTS
        if not keep_samples:
            flags |= N.RUN_NO_SAMPLES
        sp = self._params(kernel, seed, rng, init_lpost, flags, t0 or 0)
        if moments:
            self._moment_chains = 1
        out = np.empty((int(iters), self.p)) if keep_samples else None
        acc = C.c_int64(0)
        if Z is not None:
            Z = np.ascontiguousarray(Z, dtype=np.float64)
            if Z.shape != (thin * iters, self.p):
                raise ValueError(f"Z must have shape ({thin * iters}, {self.p})")
        if U is not None:
            U = np.ascontiguousarray(U, dtype=np.float64)
        self._ck(self._lib.lrb_run(
            self._h, C.byref(sp), None if ini is None else N.as_dp(ini), 1, int(thin), int(iters),
            None if Z is None else N.as_dp(Z), None if U is None else N.as_dp(U),
            None if out is None else N.as_dp(out), C.byref(acc)))
        self._cache_key = None
        if int(iters) > 0 and out is not None:
            self._last_x, self._last_sampler = out[-1].tobytes(), kernel.sampler
        elif ini is not None or out is None:
            self._last_x = None
        return out, acc.value

    def moments(self, pooled=False, cov=True):
        """Device-side running moments of the latest run(s) with moments=True
        (Dex/djwutils.dx:97-103 meanAndCovariance; what analyse.R's mcmcSummary starts from).
        Returns (count, mean, cov): per chain (C,), (C, p), (C, p, p), or pooled over the chains
        int, (p,), (p, p). cov uses the n-1 denominator."""
        c = 1 if pooled else max(1, getattr(self, "_moment_chains", 1))
        cnt = np.zeros(c, dtype=np.int64)
        mean = np.empty((c, self.p))
        cv = np.empty((c, self.p, self.p)) if cov else None
        self._ck(self._lib.lrb_run_moments(self._h, 1 if pooled else 0, cnt.ctypes.data_as(C.POINTER(C.c_int64)),
                                           N.as_dp(mean), None if cv is None else N.as_dp(cv)))
        if pooled or getattr(self, "_moment_chains", 1) == 1:
            return int(cnt[0]), mean[0], (None if cv is None else cv[0])
        return cnt, mean, cv

    def run_chains(self, kernel, inits, thin, iters, Z=None, U=None, seed=0, init_lpost=-np.inf,
                   moments=False, keep_samples=True):
        """C chains in lock-step on the device (lrb_run with C > 1): inits (C, p) -> samples
        (C, iters, p) and accepted counts (C,). Chain c uses Philox key seed + c*0x9E3779B97F4A7C15
        (mod 2^64), or rows of Z (C, thin*iters, p) / U (C, thin*iters) in replay mode."""
        inits = np.ascontiguousarray(inits, dtype=np.float64)
        if inits.ndim != 2 or inits.shape[1] != self.p:
            raise ValueError(f"inits must have shape (C, {self.p})")
        c = inits.shape[0]
        rng = N.RNG_REPLAY if Z is not None else N.RNG_PHILOX
        flags = (N.RUN_MOMENTS if moments else 0) | (0 if keep_samples else N.RUN_NO_SAMPLES)
        sp = self._params(kernel, seed, rng, init_lpost, flags)
        out = np.empty((c, int(iters), self.p)) if keep_samples else None
        acc = np.zeros(c, dtype=np.int64)
        if moments:
            self._moment_chains = c
        if Z is not None:
            Z = np.ascontiguousarray(Z, dtype=np.float64)
            if Z.shape != (c, thin * iters, self.p):
                raise ValueError(f"Z must have shape ({c}, {thin * iters}, {self.p})")
        if U is not None:
            U = np.ascontiguousarray(U, dtype=np.float64)
        self._ck(self._lib.lrb_run(
            self._h, C.byref(sp), N.as_dp(inits), c, int(thin), int(iters),
            None if Z is None else N.as_dp(Z), None if U is None else N.as_dp(U),
            None if out is None else N.as_dp(out), acc.ctypes.data_as(C.POINTER(C.c_int64))))
        self._cache_key = None
        self._last_x = None
        return out, acc

    def chain_state(self):
        x = np.empty(self.p)
        lp, t = C.c_double(), C.c_int64()
        self._ck(self._lib.lrb_chain_state(self._h, N.as_dp(x), C.byref(lp), C.byref(t)))
        return x, lp.value, t.value

    def rng_dump(self, seed, t0, count):
        return self.rng_dump_p(seed, t0, count, self.p)

    def rng_dump_p(self, seed, t0, count, p):
        """The device RNG stream under Philox key `seed`: normals (count, p) and uniforms (count,)
        for iterations t0 .. t0+count-1 (lrb_rng_dump)."""
        z = np.empty((count, p))
        u = np.empty(count)
        self._ck(self._lib.lrb_rng_dump(self._h, int(seed) & (2 ** 64 - 1), int(t0), int(count), int(p),
                                        N.as_dp(z), N.as_dp(u)))
        return z, u


# ---------------------------------------------------------------- kernels

class RandomWalk:
    """rprop of fit-numpy.py:83-84 as a descriptor: beta + scale*randn(p) (scale =
    0.02*pre there). Callable like the reference's rprop (host RNG) and recognised
    by mhKernel so the chain can run on the device."""

    def __init__(self, scale):
        self.scale = np.asarray(scale, dtype=np.float64)

    def __call__(self, beta):
        beta = np.asarray(beta, dtype=np.float64)
        return beta + self.scale * np.random.randn(len(beta))


def _unit_dprop(new, old):
    return 1.


class DeviceKernel:
    """A transition kernel whose whole loop can run on the GPU. Still callable one
    step at a time with the reference's signature: kernel(x, ll) -> (x, ll) for
    the samplers that thread the log-density (RWMH, MALA), kernel(x) -> x for UL
    and HMC. A single call draws from the global NumPy RNG exactly as the
    reference kernel would (randn(p) then rand()) and replays those draws on the
    device."""

    def __init__(self, problem, sampler, scale, step=0.0, l=1):
        self.problem = problem
        self.sampler = sampler
        self.scale = _vec(scale, problem.p, "scale")
        self.step = float(step)
        self.l = int(l)
        self.threaded = sampler in (N.RWMH, N.MALA)

    @property
    def evals_per_step(self):
        return self.l if self.sampler == N.HMC else 1

    def __call__(self, x, ll=None):
        p = self.problem.p
        Z = np.random.randn(p)[None, :]
        U = None if self.sampler == N.UL else np.array([np.random.rand()])
        if self.threaded and ll is None:
            raise TypeError("this kernel threads the log-density: call kernel(x, ll)")
        mat, _ = self.problem.run(self, x, 1, 1, Z=Z, U=U,
                                  init_lpost=(ll if self.threaded else -np.inf))
        if self.threaded:
            _, lp, _ = self.problem.chain_state()
            return mat[0], lp
        return mat[0]


_current: Problem | None = None


def current() -> Problem:
    if _current is None:
        raise LogregB200Error(N.E_STATE, "no data bound: call logreg_b200.bind_data(X, y, pscale) first")
    return _current


def bind_data(X, y, pscale=None, mode="fp64", device=0):
    """Bind the script globals X, y (fit-numpy.py:12-19) and pscale (fit-np-ul.py:31)
    to the GPU; makes the module-level ll/lprior/lpost/glp refer to them."""
    global _current
    prob = Problem(device)
    prob.bind_data(X, y, pscale, mode)
    _current = prob
    return prob


def use(problem: Problem):
    global _current
    _current = problem
    return problem


def ll(beta):
    return current().ll(beta)


def lprior(beta):
    return current().lprior(beta)


def lpost(beta):
    return current().lpost(beta)


def glp(beta):
    return current().glp(beta)


def _owner(fn, name):
    """The Problem whose bound method `name` fn is (also accepts the module-level wrappers)."""
    self = getattr(fn, "__self__", None)
    if isinstance(self, Problem) and getattr(fn, "__name__", "") == name:
        return self
    if fn is globals().get(name):
        return current()
    return None


def mhKernel(lpost, rprop, dprop=_unit_dprop, threaded=True):
    """fit-numpy.py:53-62 (threaded=True, the default: kernel(x, ll) -> (x, ll) carries the old
    log-density along) or fit-np-hmc.py:56-63 (threaded=False: kernel(x) -> x re-evaluates
    lpost(x) every step; `logreg_b200.np_hmc.mhKernel` is this form, so that script's
    two-argument call keeps its meaning).  With lpost = this module's lpost and rprop a
    RandomWalk the threaded kernel runs on the device; any other callables give the reference's
    host-side closure (with the device lpost inside it if that is what was passed)."""
    if not threaded:
        def kernel1(x):
            prop = rprop(x)
            a = lpost(prop) - lpost(x)
            if np.log(np.random.rand()) < a:
                x = prop
            return x
        return kernel1
    prob = _owner(lpost, "lpost")
    if prob is not None and isinstance(rprop, RandomWalk) and dprop is _unit_dprop:
        return DeviceKernel(prob, N.RWMH, rprop.scale)
    def kernel(x, ll):
        prop = rprop(x)
        lp = lpost(prop)
        a = lp - ll + dprop(x, prop) - dprop(prop, x)
        if np.log(np.random.rand()) < a:
            x = prop
            ll = lp
        return x, ll
    return kernel


def ulKernel(glpi, dt=1e-4, pre=1):
    """fit-np-ul.py:61-68 (p comes from the bound data, not from a global `init`)."""
    prob = _owner(glpi, "glp")
    if prob is not None:
        return DeviceKernel(prob, N.UL, pre, step=dt)
    sdt, spre = np.sqrt(dt), np.sqrt(pre)
    def kernel(x):
        return x + 0.5 * pre * glpi(x) * dt + np.random.randn(len(x)) * spre * sdt
    return kernel


def malaKernel(lpi, glpi, dt=1e-4, pre=1):
    """fit-np-mala.py:72-78."""
    prob = _owner(lpi, "lpost")
    if prob is not None and _owner(glpi, "glp") is prob:
        return DeviceKernel(prob, N.MALA, pre, step=dt)
    sdt, spre = np.sqrt(dt), np.sqrt(pre)
    advance = lambda x: x + 0.5 * pre * glpi(x) * dt
    logpdf = lambda x, loc, scale: -((x - loc) / scale) ** 2 / 2.0 - np.log(np.sqrt(2 * np.pi)) - np.log(scale)
    return mhKernel(lpi, lambda x: advance(x) + np.random.randn(len(x)) * spre * sdt,
                    lambda new, old: np.sum(logpdf(new, advance(old), spre * sdt)))


def hmcKernel(lpi, glpi, eps=1e-4, l=10, dmm=1):
    """fit-np-hmc.py:65-87."""
    prob = _owner(lpi, "lpost")
    if prob is not None and _owner(glpi, "glp") is prob:
        return DeviceKernel(prob, N.HMC, dmm, step=eps, l=l)
    sdmm = np.sqrt(dmm)
    def leapf(q, p):
        p = p + 0.5 * eps * glpi(q)
        for i in range(l):
            q = q + eps * p / dmm
            p = p + (eps if i < l - 1 else 0.5 * eps) * glpi(q)
        return (q, -p)
    def alpi(x):
        return lpi(x[0]) - 0.5 * np.sum((x[1] ** 2) / dmm)
    def kern(q):
        x = (q, np.random.randn(len(q)) * sdmm)
        prop = leapf(*x)
        a = alpi(prop) - alpi(x)
        return prop[0] if np.log(np.random.rand()) < a else q
    return kern


def mcmc(init, kernel, thin=10, iters=10000, verb=True, rng="philox", seed=None):
    """fit-numpy.py:64-79 / fit-np-ul.py:70-84: returns the (iters, p) matrix of
    thinned states. A DeviceKernel runs entirely on the GPU.

    rng="philox" (default): on-device Philox draws; the key comes from the global
        NumPy RNG unless `seed` is given, so np.random.seed() still pins a run.
    rng="numpy": the draws are taken from the global NumPy RNG in exactly the order
        the reference consumes them and replayed on the device, so a seeded run
        reproduces the reference chain (up to floating-point ties in accept/reject).
    """
    init = np.asarray(init, dtype=np.float64)
    p = len(init)
    if not isinstance(kernel, DeviceKernel):
        # a user-supplied Python kernel: the reference's loop, stepping the callable
        threaded = len(inspect.signature(kernel).parameters) >= 2
        ll = -np.inf
        mat = np.zeros((iters, p))
        x = init
        if verb:
            print(str(iters) + " iterations")
        for i in range(iters):
            if verb:
                print(str(i), end=" ", flush=True)
            for _ in range(thin):
                if threaded:
                    x, ll = kernel(x, ll)
                else:
                    x = kernel(x)
            mat[i, :] = x
        if verb:
            print("\nDone.", flush=True)
        return mat

    prob = kernel.problem
    if p != prob.p:
        raise ValueError(f"init has length {p} but the bound data have p={prob.p}")
    if rng not in ("philox", "numpy"):
        raise ValueError("rng must be 'philox' or 'numpy'")
    if seed is None and rng == "philox":
        seed = int(np.random.randint(0, 2 ** 63 - 1, dtype=np.int64))
    mat = np.empty((iters, p))
    if verb:
        print(str(iters) + " iterations")
    # progress granularity / replay upload size: run the chain in blocks of outer iterations
    if rng == "numpy":
        per_iter = thin * (p + 1) * 8
        block = max(1, min(iters, _REPLAY_CHUNK_BYTES // max(1, per_iter)))
    else:
        block = max(1, -(-iters // 50)) if verb else max(1, iters)
    done, accepted, first = 0, 0, True
    while done < iters:
        nb = min(block, iters - done)
        if verb:
            print(" ".join(str(i) for i in range(done, done + nb)), end=" ", flush=True)
        Z = U = None
        if rng == "numpy":
            steps = nb * thin
            Z = np.empty((steps, p))
            U = None if kernel.sampler == N.UL else np.empty(steps)
            for s in range(steps):
                Z[s] = np.random.randn(p)
                if U is not None:
                    U[s] = np.random.rand()
        out, accepted = prob.run(kernel, init if first else None, thin, nb, Z=Z, U=U, seed=seed or 0)
        mat[done:done + nb] = out
        done += nb
        first = False
    prob.last_accepted = accepted
    prob.last_accept_rate = accepted / max(1, thin * iters)
    if verb:
        print("\nDone.", flush=True)
    return mat
