#!/usr/bin/env python3
"""bench.py -- the driver's measurement contract for logreg_b200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload c3|c2|c5]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[2], the one `metric` is quoted on; 25.6 GB fits one
B200): HMC with a diagonal mass matrix, L=20 leap-frog steps, synthetic n=1e8, p=64,
float32 X, row-sharded over the N GPUs (strong scaling: n is the TOTAL row count).
A "step" is one HMC iteration = L fused lpost+glp evaluations over all n rows.

metric  "lpost+grad evals/s" = L * (HMC iterations / s): leap-frog gradient
        evaluations completed per second.  The same definition is used for the
        reference arm (which spends 2L+4 passes over X per iteration to deliver the
        same L leap-frog evaluations, fit-np-hmc.py:56-87), so the ratio of the two
        arms is the ratio of HMC iterations/s.
value   device-resident: data and chain state in HBM, CUDA-event timed, max over ranks.
digest  after the timed run every rank hashes its sample matrix and final (lpost, x); the hashes
        are all-gathered and the run FAILS (rc 1) if ranks disagree; final_lpost / final_x_l2 /
        accepted are printed so the N=1 and N=8 lines of a scaling sweep can be compared
        (same seed => the same chain up to the summation order of the row shards).
secondary  (N=1, and c4 at every N) configs 2 and 4 run in-process after the headline
        measurement: MALA n=1e6 p=32 (latency-bound streaming) and 4096 MALA chains n=1e6 p=64
        (tcgen05 many-chain kernel, chains sharded over the ranks, moments-only output).
e2e     the same K iterations through the public Python API, one
        mcmc(x, hmcKernel(lpost, glp, ...), thin=1, iters=1) call per step with HOST
        state in and HOST samples out (pinned staging inside the library).  X itself is
        bound once (bind_data / gen_synthetic), exactly as the reference keeps X in a
        module global; its one-off H2D cost is not part of a sampler step.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: sampler, n, p, mode, L, step(n) -> tuned so that acceptance is healthy
    "c3": dict(sampler="hmc", n=100_000_000, p=64, mode="fp32", L=20, desc="HMC L=20 diag mass, n=1e8 p=64 fp32 X"),
    "c2": dict(sampler="mala", n=1_000_000, p=32, mode="fp32", L=1, desc="MALA diag precond, n=1e6 p=32 fp32 X"),
    "c5": dict(sampler="ul", n=400_000_000, p=128, mode="fp64", L=1, desc="UL, n=4e8 p=128 fp64 X (needs >= 3 GPUs)"),
    # config 4: many chains, X replicated, chains sharded over the GPUs, no collective
    "c4": dict(sampler="mala", n=1_000_000, p=64, mode="fp32", L=1, chains=4096,
               desc="4096 MALA chains, n=1e6 p=64 fp32 X (tcgen05 3xTF32 many-chain kernel)"),
}
SAMPLE_ROWS = 1_000_000     # rows of the same workload the CPU arm is timed on
DUMP_BYTES = 64 << 20       # what --dump-outputs may write in all


def dump_outputs(d, **arrays):
    """--dump-outputs: each array as d/<name>.npy in float64, so that two builds run with the same
    arguments (hence the same inputs) can be compared output for output."""
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), np.asarray(a, dtype=np.float64))


def step_size(w, n):
    # posterior sd ~ 2.2/sqrt(n) per coefficient (unit-variance covariates): scale steps with it
    sd = 2.2 / np.sqrt(n)
    if w["sampler"] == "hmc":
        return 5.0 * sd / w["L"]          # 0.25 sd per leap-frog step, trajectory ~ 5 sd
    if w["sampler"] == "mala":
        return (0.6 * sd) ** 2            # dt = sd_prop^2
    return (0.3 * sd) ** 2


# ---------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons, power = [], None, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9 or not (t0 - 0.05 <= ts <= t1 + 0.15):
                continue
            try:
                sm.append(float(f[1])); smax = float(f[2]); power.append(float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------- CPU arm (oracle port of the reference)
def synth_host(n, p, seed=42):
    """Same distribution as the device generator: X[:,0]=1, X[:,1:]~N(0,1), y~Bernoulli(expit(X bt))."""
    rs = np.random.RandomState(seed)
    bt = np.random.RandomState(41).randn(p) / np.sqrt(p)
    X = np.empty((n, p), order="F")        # the reference's X is column-major float64 (SURVEY.md A8)
    X[:, 0] = 1.0
    for j in range(1, p):
        X[:, j] = rs.randn(n)
    y = (rs.rand(n) < 1 / (1 + np.exp(-X.dot(bt)))).astype(np.float32)
    ps = np.ones(p); ps[0] = 10.0
    return X, y, ps, bt


def cpu_kernel(w, ns, order="F", xdtype=np.float64):
    """The reference's sampler kernel (oracle port) on an ns-row sample of the workload.
    order / xdtype select the variants SURVEY.md 8(d) lists: the reference builds X float64
    column-major ("F"); row-major ("C") and float32 X are reported beside it."""
    from oracle import logreg_oracle as O
    X, y, ps, bt = synth_host(ns, w["p"])
    if order == "C":
        X = np.ascontiguousarray(X)
    if xdtype != np.float64:
        X = X.astype(xdtype, order=order)
    tgt = O.Target(X, y, ps)
    h = step_size(w, ns)      # tuned for the sample it runs on (same acceptance regime)
    if w["sampler"] == "hmc":
        k = O.hmc_kernel(tgt.lpost, tgt.glp, eps=h, l=w["L"], dmm=1.0)
        step = lambda st: (k(st[0]), None)
    elif w["sampler"] == "mala":
        k = O.mala_kernel(tgt.lpost, tgt.glp, w["p"], dt=h, pre=1.0)
        step = lambda st: k(st[0], st[1])
    else:
        k = O.ul_kernel(tgt.glp, w["p"], dt=h, pre=1.0)
        step = lambda st: (k(st[0]), None)
    return step, (bt.copy(), -np.inf)


def _time_steps(step, st, steps, warmup, budget_s):
    """(min, mean) seconds per step over `steps` steps (at least one), after `warmup`."""
    for _ in range(warmup):
        st = step(st)
    ts = []
    t_all = time.perf_counter()
    for _ in range(max(1, steps)):
        t0 = time.perf_counter()
        st = step(st)
        ts.append(time.perf_counter() - t0)
        if budget_s and time.perf_counter() - t_all > budget_s:
            break
    return min(ts), float(np.mean(ts)), len(ts)


def time_cpu(w, n_full, steps, warmup, budget_s=None, variants=True):
    """The CPU arm.  The port is timed at TWO sample sizes (1e6 and 4e6 rows) with every host
    thread; a line T(n) = a + b*n through the two points gives the time at the full n (the path
    is a stream over rows).  Beside it: one thread, row-major X and float32 X at the small size."""
    from threadpoolctl import threadpool_info, threadpool_limits
    ncpu = os.cpu_count() or 1
    # torchrun exports OMP_NUM_THREADS=1 to its workers, which would silently make the reference
    # arm single-threaded: ask for every core explicitly
    threadpool_limits(limits=ncpu)
    sizes = [min(SAMPLE_ROWS, n_full), min(4 * SAMPLE_ROWS, n_full)]
    if sizes[1] == sizes[0]:
        sizes = sizes[:1]
    pts, done0 = [], 0
    for i, ns in enumerate(sizes):
        step, st = cpu_kernel(w, ns)
        np.random.seed(7)
        k = steps if i == 0 else max(1, steps // 4)
        tmin, tmean, done = _time_steps(step, st, k, max(1, warmup if i == 0 else min(warmup, 1)), budget_s)   # never time a cold first step
        pts.append((ns, tmean, tmin))
        if i == 0:
            done0 = done
        del step, st
    if len(pts) == 2:
        b = (pts[1][1] - pts[0][1]) / (pts[1][0] - pts[0][0])
        a = pts[0][1] - b * pts[0][0]
        t_full = a + b * n_full
    else:
        a, b, t_full = 0.0, pts[0][1] / pts[0][0], pts[0][1] * n_full / pts[0][0]
    blas = max([i.get("num_threads", 1) for i in threadpool_info()] + [1])
    out = {"ms_per_step": t_full * 1e3, "iters_per_s": 1.0 / t_full, "steps": done0,
           "sample_ms_per_step": pts[0][1] * 1e3, "sample_rows": pts[0][0],
           "cores": int(blas), "host_cpus": ncpu,
           "sizes": [p[0] for p in pts], "ms_at_size": [p[1] * 1e3 for p in pts],
           "min_ms_at_size": [p[2] * 1e3 for p in pts],
           "fit": {"intercept_ms": a * 1e3, "ms_per_1e6_rows": b * 1e9, "model": "T(n) = a + b*n through the measured sizes"},
           "threads": [1, int(blas)]}
    if variants:
        ns = sizes[0]
        var = {}
        with threadpool_limits(limits=1):
            step, st = cpu_kernel(w, ns)
            np.random.seed(7)
            var["one_thread_F_f64"] = _time_steps(step, st, 2, 0, budget_s)[1] * 1e3
        for name, order, dt in (("all_threads_C_f64", "C", np.float64), ("all_threads_F_f32", "F", np.float32)):
            step, st = cpu_kernel(w, ns, order=order, xdtype=dt)
            np.random.seed(7)
            var[name] = _time_steps(step, st, 2, 0, budget_s)[1] * 1e3
        var["all_threads_F_f64"] = pts[0][1] * 1e3
        out["variants_ms_per_step_at_%d_rows" % ns] = var
    out["sample"] = (f"{w['desc'].split(',')[0]} reference kernel (oracle port, NumPy/OpenBLAS, X float64 column-major as "
                     f"the reference builds it), {int(blas)} threads, measured at {' and '.join(str(p[0]) for p in pts)} rows "
                     f"({done0} iterations at the first size); T(n)=a+b*n through the measured sizes gives n={n_full} "
                     f"(a={a * 1e3:.1f} ms, b={b * 1e9:.1f} ms per 1e6 rows)")
    return out


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def measure_c4(lr, prob, bt, w, rank, world, K, W, barrier, maxr, dump=None):
    """Config 4: C chains in lock-step per GPU (tcgen05 3xTF32 many-chain kernel), chains sharded
    over the ranks with no collective.  A step = one MALA iteration of every chain.  Only the
    running moments leave the device (f3): no per-step D2H of the C x p states.
    dump: directory for this rank's outputs of the timed run (pooled moments, accepted counts)."""
    n, p, C = w["n"], w["p"], w["chains"]
    c_lo, c_hi = (rank * C) // world, ((rank + 1) * C) // world
    Cl = c_hi - c_lo
    sd = 2.2 / np.sqrt(n)
    kern = lr.malaKernel(prob.lpost, prob.glp, dt=step_size(w, n), pre=1.0)
    inits = bt + 0.5 * sd * np.random.RandomState(100 + rank).randn(Cl, p)
    prob.run_chains(kern, inits, 1, W, seed=7 + rank, moments=True, keep_samples=False)
    inf0 = prob.info()
    barrier()
    t0 = time.perf_counter()
    _, acc = prob.run_chains(kern, inits, 1, K, seed=7 + rank, moments=True, keep_samples=False)   # host inits in
    cnt, mean, cov = prob.moments(pooled=True)                                                     # O(p^2) out, once
    dt = maxr(time.perf_counter() - t0)
    inf1 = prob.info()
    if dump:
        dump_outputs(dump, moments_count=[cnt], moments_mean=mean, moments_cov=cov, accepted=acc)
    peaks = load_peaks()
    value = C * K / dt
    flops = 4.0 * n * p * Cl * (K + 1)             # algorithmic (1-pass) flops on this rank, incl. the init evaluation
    peak_tf32 = float(peaks.get("bf16_tflops", 1590.0)) / 2
    return {"chain_iters_per_s": value, "ms_per_step": dt / K * 1e3, "steps": K, "warmup": W, "chains": C,
            "chains_per_gpu": Cl, "accept_rate": float(acc.mean() / K), "tflops_1pass": flops / dt / 1e12,
            "frac": flops / dt / 1e12 / peak_tf32, "peak_tflops": peak_tf32,
            "peak_source": "MEASURED_PEAKS.json bf16_tflops / 2 (TF32 dense runs at half the bf16 rate)" if peaks else "fallback 1590/2",
            "h2d_bytes_per_step": Cl * p * 8 / K, "d2h_bytes_per_step": (p * p + p + 1 + Cl) * 8 / K,
            "pooled_posterior_mean_l2": float(np.linalg.norm(mean)), "moment_count": int(cnt),
            "gpu_launches": int(inf1["kernel_launches"] - inf0["kernel_launches"]),
            "note": "timed through Problem.run_chains(moments=True, keep_samples=False) + Problem.moments(pooled=True): "
                    "host inits in, pooled mean/covariance out; algorithmic 4*n*p*C flops per all-chain evaluation "
                    "(the 3xTF32 kernel executes 3x that on the tensor pipe)"}


def measure_c2(lr, local, K=4000, W=400):
    """Config 2: MALA, one chain, n=1e6 p=32 fp32 X (129 MB, about the size of L2): latency-bound."""
    import torch
    w = WORKLOADS["c2"]
    prob = lr.Problem(local)
    bt = prob.gen_synthetic(w["n"], w["p"], mode=w["mode"], seed=42)
    kern = lr.malaKernel(prob.lpost, prob.glp, dt=step_size(w, w["n"]), pre=1.0)
    prob.run(kern, bt, 1, W, seed=3)
    t0 = time.perf_counter()
    mat, acc = prob.run(kern, None, 1, K, seed=3)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    byt = prob.info()["bytes_per_eval"]
    prob.close()
    peak = float(load_peaks().get("hbm_gbs", 6650.0))
    us = dt / K * 1e6
    return {"iters_per_s": K / dt, "us_per_iter": us, "accept_rate": acc / K, "GBps": byt / us / 1e3,
            "frac": byt / us / 1e3 / peak, "bytes_per_iter": byt, "steps": K,
            "l2": "X is 128 MB, about the L2 size (126 MB): partly L2-resident by design (persisting window), not flushed",
            "note": "host-timed Problem.run of K MALA iterations (one fused evaluation each), whole loop on the device"}


# ---------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--comm", default="auto", choices=["auto", "p2p", "nccl"])
    ap.add_argument("--n", type=int, default=0, help="override total rows (development only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--deterministic", action="store_true", help="static fixed-order kernel instead of drive mode")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what they computed as DIR/<name>.npy (float64, rank 0): "
                         "the sample matrix (its last rows if above 32 MB), final state and lpost, and the number of "
                         "timed steps accepted; for c4 the pooled moments and each chain's accepted timed steps")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; the reference arm has none to write")
    w = dict(WORKLOADS[args.workload])
    if args.n:
        w["n"] = args.n
    K, W, L = args.steps, max(args.warmup, 0), w["L"]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    metric = "lpost+grad evals/s"
    xb = w["n"] / world * w["p"] * (4 if w["mode"] == "fp32" else 8)
    config = {"workload": f"{w['desc']}, {w['sampler'].upper()} on-device loop", "n": w["n"], "p": w["p"],
              "L": L, "x_dtype": w["mode"], "parallelism": f"row-sharded x{world}" if world > 1 else "single GPU",
              "l2": ("inputs exceed L2 (X is %.1f GB per GPU vs 126 MB L2)" % (xb / 1e9)) if xb > 3 * 126e6 else
                    ("X is %.0f MB per GPU, about the L2 size (126 MB): partly L2-resident by design, not flushed" % (xb / 1e6))}

    if args.impl == "reference":
        if rank != 0:
            return 0
        r = time_cpu(w, w["n"], K, W, variants=False)
        val = L * r["iters_per_s"]
        cb = {"value": val, "unit": "evals/s", "cores": r["cores"], "kind": "port", "sample": r["sample"],
              "sizes": r["sizes"], "ms_at_size": r["ms_at_size"], "fit": r["fit"], "threads": [r["cores"]],
              "host_cpus": r["host_cpus"]}
        line = {"impl": "reference", "metric": metric, "value": val, "unit": "evals/s", "n_gpus": args.gpus,
                "steps": r["steps"], "warmup": W,
                # the time one step of the bounded SAMPLE took (so steps x ms_per_step is this run's wall time);
                # `value` is the same metric at the full n through the fitted line
                "ms_per_step": r["sample_ms_per_step"], "ms_per_step_at_full_n": r["ms_per_step"],
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config, "iters_per_s": r["iters_per_s"], "cpu_baseline": cb,
                "e2e": {"value": val, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist
    import logreg_b200 as lr
    from logreg_b200 import dist as lrd

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; logreg_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def maxr(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def finish(rc=0):
        if world > 1:
            dist.destroy_process_group()
        return rc

    n, p = w["n"], w["p"]
    if "chains" in w:
        # --workload c4 as the headline line (development / profiles); the driver's line is c3
        prob = lr.Problem(local, deterministic=args.deterministic)
        bt = prob.gen_synthetic(n, p, mode=w["mode"], seed=42)
        r = measure_c4(lr, prob, bt, w, rank, world, K, max(W, 10), barrier, maxr,
                       dump=args.dump_outputs if rank == 0 else None)
        if rank == 0:
            line = {"metric": metric, "value": r["chain_iters_per_s"], "unit": "evals/s", "n_gpus": world, "steps": r["steps"],
                    "warmup": r["warmup"], "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                    "scaling": "weak" if world > 1 else "strong", "vs_baseline": None, "dtype": "tf32x3", "data": "synthetic",
                    "config": dict(config, chains=r["chains"], chains_per_gpu=r["chains_per_gpu"], parallelism=f"chain-sharded x{world}",
                                   l2="X (256 MB) exceeds L2 (126 MB)"),
                    "chain_iters_per_s": r["chain_iters_per_s"], "accept_rate": r["accept_rate"],
                    "roofline": {"bound": "tensor", "achieved": r["tflops_1pass"], "peak": r["peak_tflops"], "unit": "TFLOP/s",
                                 "frac": r["frac"], "traffic": None, "peak_source": r["peak_source"], "note": r["note"]},
                    "cpu_baseline": None,
                    "e2e": {"value": r["chain_iters_per_s"], "unit": "evals/s", "h2d_bytes_per_step": r["h2d_bytes_per_step"],
                            "d2h_bytes_per_step": r["d2h_bytes_per_step"], "note": r["note"]},
                    "gpu_launches": r["gpu_launches"], "clocks": None}
            print(json.dumps(line))
        return finish()

    lo, hi = lrd.shard_rows(n, rank, world)
    prob = lr.Problem(local, deterministic=args.deterministic)
    prob.n_global = n
    bt = prob.gen_synthetic(hi - lo, p, mode=w["mode"], seed=42, row_offset=lo)
    if world > 1:
        lrd.init_comm(prob, args.comm)
    h = step_size(w, n)
    if w["sampler"] == "hmc":
        kern = lr.hmcKernel(prob.lpost, prob.glp, eps=h, l=L, dmm=1.0)
    elif w["sampler"] == "mala":
        kern = lr.malaKernel(prob.lpost, prob.glp, dt=h, pre=1.0)
    else:
        kern = lr.ulKernel(prob.glp, dt=h, pre=1.0)

    lib, hd = prob._lib, prob._h
    import ctypes as C
    import hashlib
    from logreg_b200 import _native as N
    stream = torch.cuda.Stream()
    prob.set_stream(stream.cuda_stream)
    sp = prob._params(kern, seed=2026, rng=N.RNG_PHILOX, init_lpost=-np.inf)

    # ---- device-resident timing: warm-up run (W iterations), then K iterations in one launch call
    def begin(iters):
        N.check(lib.lrb_run_begin(hd, C.byref(sp), N.as_dp(np.ascontiguousarray(bt)), 1, iters, None, None), hd)
    with torch.cuda.stream(stream):
        begin(max(W, 1))
        N.check(lib.lrb_run_launch(hd), hd)       # includes the one-off evaluation at init
        acc = C.c_int64()
        N.check(lib.lrb_run_finish(hd, None, C.byref(acc)), hd)
        # continue the same chain for K timed iterations
        sp2 = prob._params(kern, seed=2026, rng=N.RNG_PHILOX, init_lpost=-np.inf)
        N.check(lib.lrb_run_begin(hd, C.byref(sp2), None, 1, K, None, None), hd)
        inf0 = prob.info()
        clocks = ClockSampler(local)
        if rank == 0:
            clocks.start()
            time.sleep(0.3)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tw0 = time.time()
        e0.record(stream)
        N.check(lib.lrb_run_launch(hd), hd)
        e1.record(stream)
        stream.synchronize()
        barrier()
        tw1 = time.time()
        ms_total = maxr(e0.elapsed_time(e1))
        clk = clocks.stop(tw0, tw1) if rank == 0 else None
        inf1 = prob.info()
        out = np.empty((K, p))
        acc1 = C.c_int64()
        N.check(lib.lrb_run_finish(hd, N.as_dp(out), C.byref(acc1)), hd)
    accept_rate = (acc1.value - acc.value) / K
    launches = inf1["kernel_launches"] - inf0["kernel_launches"]
    evals = inf1["eval_launches"] - inf0["eval_launches"]
    assert evals == K * L, (evals, K, L)
    ms_step = ms_total / K
    value = K * L / (ms_total / 1e3)
    prob.set_stream(None)

    # ---- state digest: every rank must have walked the same chain (replicated sampler state)
    x_fin, lp_fin, t_fin = prob.chain_state()
    dig = hashlib.sha256(out.tobytes() + x_fin.tobytes() + np.float64(lp_fin).tobytes() + np.int64(acc1.value).tobytes()).digest()
    ranks_agree = True
    if world > 1:
        mine = torch.frombuffer(bytearray(dig), dtype=torch.uint8).cuda()
        alld = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(alld, mine)
        ranks_agree = all(bool(torch.equal(alld[0], d)) for d in alld)
    digest = {"final_lpost": lp_fin, "final_x_l2": float(np.linalg.norm(x_fin)), "final_x0": float(x_fin[0]),
              "accepted": int(acc1.value), "kernel_applications": int(t_fin), "samples_sha16": dig.hex()[:16],
              "ranks_agree": ranks_agree,
              "note": "chain from beta_true, seed 2026, W warm-up + K timed HMC iterations; lines of a scaling sweep "
                      "agree to the summation order of the row shards (sha differs across N, the values agree)"}
    if not ranks_agree:
        if rank == 0:
            print(json.dumps({"error": "ranks disagree on the sample matrix / final state", "digest": digest}))
        finish()
        return 1
    if args.dump_outputs and rank == 0:
        keep = DUMP_BYTES // 2 // (8 * p)
        dump_outputs(args.dump_outputs, samples=out[-keep:], final_x=x_fin, final_lpost=[lp_fin],
                     accepted=[acc1.value - acc.value])

    # ---- e2e through the public API: host state in, host sample out, every step
    x = out[-1].copy()
    for _ in range(min(W, 2)):
        x = lr.mcmc(x, kern, thin=1, iters=1, verb=False, seed=11)[0]
    barrier()
    t0 = time.perf_counter()
    for i in range(K):
        x = lr.mcmc(x, kern, thin=1, iters=1, verb=False, seed=100 + i)[0]
    torch.cuda.synchronize()
    e2e_s = maxr(time.perf_counter() - t0)
    e2e_val = K * L / e2e_s
    # one call for all K iterations (how a script calls it)
    barrier()
    t0 = time.perf_counter()
    lr.mcmc(x, kern, thin=1, iters=K, verb=False, seed=5)
    e2e_single = K * L / maxr(time.perf_counter() - t0)

    # ---- roofline of the fused kernel (it is the only kernel in the timed region)
    peaks = load_peaks()
    peak = float(peaks.get("hbm_gbs", 6650.0))
    bytes_eval_rank = inf1["bytes_per_eval"]            # this rank's shard
    kern_ms = ms_total / evals                           # per evaluation: includes the in-kernel allreduce + sampler update
    achieved = bytes_eval_rank / (kern_ms * 1e-3) / 1e9
    is_drive = launches < evals     # drive mode: one launch for the whole timed region (single-GPU handles)
    traffic, traffic_src = None, None
    try:
        if world == 1 and not args.n:   # the committed ncu capture is of the single-GPU kernel
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            key = args.workload + ("" if is_drive else "_static")
            traffic = tj.get(key, {}).get("bytes_per_eval") * evals / max(1, launches)
            traffic_src = tj.get(key, {}).get("source")
    except Exception:
        pass
    tname = "float" if w["mode"] == "fp32" else "double"
    kname = ("lrb::eval_persist_kernel<%s,%d,grad>" if is_drive else "lrb::eval_kernel<%s,%d,grad>") % (tname, inf1["p_pad"])
    roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "traffic_source": traffic_src,
            "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
            "frac_of_nominal_8TBs": achieved / 8000.0, "kernel": kname,
            "evals_per_launch": evals / max(1, launches), "algorithmic_bytes_per_eval": bytes_eval_rank,
            "algorithmic_bytes_per_launch": bytes_eval_rank * evals / max(1, launches),
            "avg_launch_ms": ms_total / max(1, launches), "avg_eval_ms": kern_ms,
            "note": "drive mode: ONE cooperative launch performs all K*L evaluations of the timed region; "
                    "achieved = algorithmic bytes of the launch / its duration (CUDA events on the launching stream)"
                    if is_drive else "static kernel: one launch per evaluation (replayed CUDA graph); row-sharded handles "
                                     "always run this kernel, the fused peer-memory exchange is inside it"}

    # ---- secondary workloads (configs 2 and 4), after the headline measurement
    secondary = None
    if not args.no_secondary and not args.n and args.workload == "c3":
        secondary = {}
        try:
            w4 = dict(WORKLOADS["c4"])
            p4 = lr.Problem(local)
            bt4 = p4.gen_synthetic(w4["n"], w4["p"], mode=w4["mode"], seed=42)
            r4 = measure_c4(lr, p4, bt4, w4, rank, world, 40, 10, barrier, maxr)
            p4.close()
            secondary["c4"] = dict(r4, config=w4["desc"], parallelism=f"chain-sharded x{world}, no collective")
        except Exception as e:   # never let a secondary figure break the contract line
            secondary["c4"] = {"error": str(e)}
        if world == 1:
            try:
                secondary["c2"] = dict(measure_c2(lr, local), config=WORKLOADS["c2"]["desc"])
            except Exception as e:
                secondary["c2"] = {"error": str(e)}

    if rank != 0:
        return finish()
    # one-off ingest (bind_data) of a host-resident X in the reference's own layout (float64,
    # column-major), on a 2e6-row sample: reported beside e2e, not part of a sampler step
    ingest = None
    if world == 1:
        try:
            ns_i = 2_000_000
            Xh = np.asfortranarray(np.random.RandomState(1).randn(ns_i, p))
            yh = (np.random.RandomState(2).rand(ns_i) < 0.5).astype(np.float32)
            pi = lr.Problem(local)
            t0 = time.perf_counter()
            pi.bind_data(Xh, yh, np.ones(p), mode=w["mode"])
            dt_i = time.perf_counter() - t0
            pi.close()
            ingest = {"rows": ns_i, "host_layout": "float64 column-major (reference)", "seconds": dt_i,
                      "host_GB_per_s": Xh.nbytes / dt_i / 1e9,
                      "extrapolated_seconds_full_n": dt_i * n / ns_i}
            del Xh, yh
        except Exception as e:  # never let the optional figure break the contract line
            ingest = {"error": str(e)}
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        r = time_cpu(w, n, steps=6, warmup=1, budget_s=12.0)
        cpu = {"value": L * r["iters_per_s"], "unit": "evals/s", "cores": r["cores"], "kind": "port",
               "sample": r["sample"], "iters_per_s": r["iters_per_s"], "host_cpus": r["host_cpus"],
               "sizes": r["sizes"], "ms_at_size": r["ms_at_size"], "fit": r["fit"], "threads": r["threads"]}
        for k_ in r:
            if k_.startswith("variants_"):
                cpu[k_] = r[k_]
    line = {"metric": metric, "value": value, "unit": "evals/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32" if w["mode"] == "fp32" else "f64", "data": "synthetic", "config": config,
            "iters_per_s": 1e3 / ms_step, "accept_rate": accept_rate, "step_size": h,
            "roofline": roof, "cpu_baseline": cpu,
            "e2e": {"value": e2e_val, "unit": "evals/s", "h2d_bytes_per_step": 2 * p * 8, "d2h_bytes_per_step": p * 8 + 8 + 4,
                    "single_call_value": e2e_single, "one_off_ingest": ingest,
                    "note": "K mcmc(x, kernel, thin=1, iters=1) calls, host state in/out each step (a call that starts "
                            "where the previous one stopped reuses the cached gradient: L passes per step); "
                            "single_call_value = one mcmc(iters=K) call"},
            "digest": digest, "secondary": secondary,
            "gpu_launches": int(launches), "gpu_evals": int(evals),
            "mode": "drive" if is_drive else "static",
            "comm": (getattr(prob, "comm_kind", args.comm) if world > 1 else None), "clocks": clk}
    print(json.dumps(line))
    return finish()


if __name__ == "__main__":
    sys.exit(main())
