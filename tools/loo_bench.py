"""Time lrb_loo (PSIS-LOO over S draws) on one B200, stage by stage, beside lrb_predictive.

    python tools/loo_bench.py [--device 0] [--calls 5] [--out FILE]

One JSON line per shape: n = 1e6, p = 64, S = 4000 in FP32 and FP64; n = 1e8, p = 64, S = 64 in
FP32; n = 1e4, p = 64, S = 2^21 (the draw cap) in FP32.  Draws are beta_true + (2.2/sqrt(n)) N(0, I)
with a fixed seed (no sampler run).  Each time is the median of CUDA events on a caller stream
around each call (totals only: no per-row output is copied), after one warm-up call.  Stage 1 is
timed as lrb_loo with LRB_LOO_STAGE1_ONLY set (the log-likelihood chunks alone); stage 2 is the
difference from the full call.  For n = 1e6 the full call is also timed with a 1 GB chunk budget
(LRB_LOO_CHUNK_MB=1024), whose chunks of L do not stay in L2.  lrb_predictive is timed at the same
shape in the same process, and the card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = [(1_000_000, 64, "fp32", 4000), (1_000_000, 64, "fp64", 4000),
          (100_000_000, 64, "fp32", 64), (10_000, 64, "fp32", 1 << 21)]


def gpu_card(device):
    r = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader,nounits"], capture_output=True, text=True, check=True)
    name, power, clock = [s.strip() for s in r.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit_w": float(power), "max_sm_clock_mhz": float(clock)}


def timed(stream, fn, calls):
    import torch
    first = fn()                                         # warm-up
    ms = []
    for _ in range(calls):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        out = fn()
        e1.record(stream)
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return float(np.median(ms)) / 1e3, min(ms) / 1e3, max(ms) / 1e3, first, out


def with_env(key, value, fn):
    old = os.environ.get(key)
    os.environ[key] = value
    try:
        return fn()
    finally:
        if old is None:
            del os.environ[key]
        else:
            os.environ[key] = old


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import logreg_b200 as lr
    card = gpu_card(args.device)
    stream = torch.cuda.Stream(device=args.device)
    lines = []
    for n, p, mode, S in SHAPES:
        q = lr.Problem(args.device)
        bt = q.gen_synthetic(n, p, mode=mode, seed=42)
        B = bt + (2.2 / np.sqrt(n)) * np.random.RandomState(0).randn(S, p)
        q.set_stream(stream.cuda_stream)
        calls = 2 if S > 100_000 else args.calls
        loo = lambda: q.loo(B, pointwise=False)
        t, tmin, tmax, first, out = timed(stream, loo, calls)
        assert out["elpd_loo"] == first["elpd_loo"] and out["k_max"] == first["k_max"]
        t1 = with_env("LRB_LOO_STAGE1_ONLY", "1", lambda: timed(stream, loo, calls))[0]
        line = {"kernel": "loglik_kernel + psis_kernel", "n": n, "p": p, "mode": mode, "draws": S,
                "tail_len": int(np.ceil(min(0.2 * S, 3 * np.sqrt(S)))), "outputs": "totals only",
                "calls": calls, "loo_median_s": t, "loo_min_s": tmin, "loo_max_s": tmax,
                "stage1_median_s": t1, "stage2_s": t - t1,
                "L_bytes_written": n * S * 8}
        if n == 1_000_000:
            line["loo_1gb_chunks_median_s"] = with_env("LRB_LOO_CHUNK_MB", "1024", lambda: timed(stream, loo, calls))[0]
        if S <= 1 << 16:
            line["predictive_median_s"] = timed(stream, lambda: q.predictive(B, pointwise=False), calls)[0]
            line["loo_over_predictive"] = t / line["predictive_median_s"]
        line.update({k: out[k] for k in ("elpd_loo", "p_loo", "k_max", "n_k_high")})
        line.update(card)
        q.close()
        print(json.dumps(line), flush=True)
        lines.append(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write("".join(json.dumps(l) + "\n" for l in lines))


if __name__ == "__main__":
    main()
