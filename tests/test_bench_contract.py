"""bench.py contract checks.  Without a GPU: the reference arm prints one JSON line with the
contract's keys; under a multi-rank launch only rank 0 prints.  On a GPU (marked): --steps sets the
number of timed steps, and --dump-outputs writes what those steps computed."""
import json
import os
import subprocess

import pytest
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra, *args):
    env = dict(os.environ, **env_extra)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          timeout=600, env=env, cwd=ROOT)


def test_reference_arm_line():
    r = _run({}, "--impl", "reference", "--steps", "1", "--warmup", "0")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "lpost+grad evals/s" and d["unit"] == "evals/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1
    assert d["config"]["n"] == 100_000_000 and d["config"]["p"] == 64 and "HMC" in d["config"]["workload"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and "rows" in cb["sample"] and cb["value"] == d["value"]
    # measured at two sample sizes, a line through them gives the figure at the full n (VERDICT r1, weak 4)
    assert cb["sizes"] == [1_000_000, 4_000_000] and len(cb["ms_at_size"]) == 2 and cb["ms_at_size"][1] > cb["ms_at_size"][0]
    fit = cb["fit"]
    t_full = fit["intercept_ms"] + fit["ms_per_1e6_rows"] * 100.0
    assert d["ms_per_step_at_full_n"] == pytest.approx(t_full, rel=1e-9)
    assert d["value"] == pytest.approx(20 * 1e3 / t_full, rel=1e-9)            # L = 20 evaluations per HMC iteration
    # ms_per_step is the measured time of a step of the bounded sample (so steps x ms_per_step is this run's work)
    assert d["ms_per_step"] == pytest.approx(cb["ms_at_size"][0], rel=1e-9)
    assert d["e2e"] == {"value": d["value"], "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_are_silent():
    r = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, "--impl", "reference", "--gpus", "2", "--steps", "1")
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_holds_the_timed_steps(tmp_path):
    """--steps sets the number of timed HMC iterations, and --dump-outputs writes what they computed."""
    import numpy as np
    K = 7
    r = _run({}, "--steps", str(K), "--warmup", "2", "--n", "1000000", "--no-cpu-baseline", "--no-secondary",
             "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.strip().splitlines() if l.startswith("{")][-1])
    assert d["steps"] == K and d["gpu_evals"] == K * 20
    out = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert sorted(out) == ["accepted", "final_lpost", "final_x", "samples"]
    assert all(a.dtype == np.float64 for a in out.values())
    assert out["samples"].shape == (K, 64) and np.all(np.isfinite(out["samples"]))
    np.testing.assert_array_equal(out["final_x"], out["samples"][-1])      # thin = 1: the last step's state
    assert out["final_lpost"][0] == d["digest"]["final_lpost"]
    assert out["accepted"][0] == round(d["accept_rate"] * K)                # the timed steps only, not the warm-up


@pytest.mark.gpu
def test_dump_outputs_of_the_many_chain_workload(tmp_path):
    """c4: --steps below the old floor of 40 is honoured, and the dump holds the pooled moments of the
    timed run (every chain's every timed state) and each chain's accepted timed steps."""
    import numpy as np
    K, C, p = 5, 4096, 64
    r = _run({}, "--workload", "c4", "--steps", str(K), "--warmup", "2", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.strip().splitlines() if l.startswith("{")][-1])
    assert d["steps"] == K
    out = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert sorted(out) == ["accepted", "moments_count", "moments_cov", "moments_mean"]
    assert all(a.dtype == np.float64 for a in out.values())
    assert out["moments_count"].tolist() == [C * K]
    assert out["moments_mean"].shape == (p,) and np.all(np.isfinite(out["moments_mean"]))
    cov = out["moments_cov"]
    assert cov.shape == (p, p) and np.all(np.isfinite(cov)) and np.all(np.diag(cov) > 0)
    np.testing.assert_allclose(cov, cov.T, rtol=1e-9, atol=1e-9 * np.max(np.diag(cov)))
    acc = out["accepted"]
    assert acc.shape == (C,) and np.all((acc >= 0) & (acc <= K)) and np.all(acc == np.round(acc))
    assert acc.sum() / (C * K) == pytest.approx(d["accept_rate"], rel=1e-12)
