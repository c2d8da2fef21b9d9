"""Time lrb_predictive (posterior predictive summaries / WAIC over S draws) on one B200.

    python tools/predictive_bench.py [--device 0] [--calls 7] [--out FILE]

One JSON line per shape: the C3 data shape (gen_synthetic(1e8, 64, fp32), S = 64 and 1000) and a
held-out shape (n = 1e6, p = 64, S = 4000) in both modes.  Draws are beta_true + (2.2/sqrt(n)) N(0, I)
with a fixed seed (no sampler run).  Time per call = median of CUDA events on a caller stream around
each call (totals only: no per-row output is written), after one warm-up call.  The FMA-pipe bound
is the data-sheet rate at the card's maximum SM clock (FP32: 128 lanes per SM, FP64: 64), not a
measurement.  `numpy_float64_1e5_rows_s` is NumPy on a 1e5-row sample of the same rows, for scale.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = [(100_000_000, 64, "fp32", 64), (100_000_000, 64, "fp32", 1000),
          (1_000_000, 64, "fp32", 4000), (1_000_000, 64, "fp64", 4000)]


def gpu_card(device):
    r = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader,nounits"], capture_output=True, text=True, check=True)
    name, power, clock = [s.strip() for s in r.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit_w": float(power), "max_sm_clock_mhz": float(clock)}


def numpy_reference_time(X, y, B):
    from scipy.special import expit, logsumexp
    t0 = time.perf_counter()
    eta = X @ B.T
    ll = -np.logaddexp(0.0, -np.where(y[:, None] > 0, eta, -eta))
    sig = expit(eta)
    lppd = logsumexp(ll, axis=1) - np.log(B.shape[0])
    pw = ll.var(axis=1, ddof=1)
    _ = (sig.mean(axis=1), sig.std(axis=1, ddof=1), lppd.sum(), pw.sum())
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--calls", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import logreg_b200 as lr
    card = gpu_card(args.device)
    sms = torch.cuda.get_device_properties(args.device).multi_processor_count
    stream = torch.cuda.Stream(device=args.device)
    lines = []
    for n, p, mode, S in SHAPES:
        q = lr.Problem(args.device)
        bt = q.gen_synthetic(n, p, mode=mode, seed=42)
        B = bt + (2.2 / np.sqrt(n)) * np.random.RandomState(0).randn(S, p)
        q.set_stream(stream.cuda_stream)
        first = q.predictive(B, pointwise=False)                    # warm-up
        ms = []
        for _ in range(args.calls):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            out = q.predictive(B, pointwise=False)
            e1.record(stream)
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
            assert out["lppd"] == first["lppd"]
        t = float(np.median(ms)) / 1e3
        P = q.info()["p_pad"]
        es = 4 if mode == "fp32" else 8
        fma = n * S * p
        lanes = 128 if mode == "fp32" else 64
        bound = sms * lanes * card["max_sm_clock_mhz"] * 1e6          # FMA/s
        Xs, ys = q.copy_rows(0, 100_000)
        line = {"kernel": "predictive_kernel", "n": n, "p": p, "p_pad": P, "mode": mode, "draws": S,
                "outputs": "totals only", "calls": args.calls, "median_s": t, "min_s": min(ms) / 1e3,
                "max_s": max(ms) / 1e3, "fma": fma, "fma_per_s": fma / t,
                "fma_pipe_bound_per_s": bound, "fma_pipe_bound_source": f"data sheet: {sms} SMs x {lanes} lanes x max SM clock",
                "fraction_of_fma_bound": fma / t / bound,
                "hbm_bytes_read": n * P * es + n + P * (-(-S // 64) * 64) * es,
                "lppd": out["lppd"], "p_waic": out["p_waic"], "elpd_waic": out["elpd_waic"],
                "numpy_float64_1e5_rows_s": numpy_reference_time(Xs, ys, B), **card}
        q.close()
        print(json.dumps(line), flush=True)
        lines.append(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write("".join(json.dumps(l) + "\n" for l in lines))


if __name__ == "__main__":
    main()
