"""The steps either side of the hot path (SURVEY.md 8f): ingest, MAP, output/summaries."""
import os
import subprocess
import sys

import numpy as np
import pytest

from logreg_b200.workflow import describe, effective_sample_size, load_pima, save_samples

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_load_pima_formats(pima, tmp_path):
    X, y = load_pima(os.path.join(ROOT, "tests", "golden", "pima.npz"))
    assert X.flags["F_CONTIGUOUS"] and X.shape == (200, 8) and y.dtype == np.float32
    np.testing.assert_array_equal(X, pima["X"])
    # the text format of C/fit-bayes.c:46-68 (pima.data): write one, read it back
    path = tmp_path / "pima.data"
    with open(path, "w") as fh:
        for i in range(200):
            fh.write(" ".join(repr(float(v)) for v in pima["X"][i, 1:]) + (' "Yes"\n' if pima["y"][i] else ' "No"\n'))
    X2, y2 = load_pima(path)
    np.testing.assert_array_equal(X2, pima["X"])
    np.testing.assert_array_equal(y2, pima["y"])
    # the reference's pima.parquet (R/create-dataset.R writes MASS::Pima.tr) in the schema recorded in
    # SURVEY.md (data files): five int32 and two float64 covariates, then `type`, a Yes/No category
    import pandas as pd
    schema = {"npreg": "int32", "glu": "int32", "bp": "int32", "skin": "int32", "bmi": "float64", "ped": "float64",
              "age": "int32"}
    cov = pima["X"][:, 1:]
    ints = [j for j, t in enumerate(schema.values()) if t == "int32"]
    np.testing.assert_array_equal(cov[:, ints], np.round(cov[:, ints]))     # the int32 columns hold integers
    df = pd.DataFrame({name: cov[:, j].astype(t) for j, (name, t) in enumerate(schema.items())})
    df["type"] = pd.Categorical(np.where(pima["y"] == 1, "Yes", "No"), categories=["No", "Yes"])
    df.to_parquet(tmp_path / "pima.parquet")
    back = pd.read_parquet(tmp_path / "pima.parquet")
    assert {c: str(t) for c, t in back.dtypes.items()} == dict(schema, type="category")
    X3, y3 = load_pima(tmp_path / "pima.parquet")
    assert X3.flags["F_CONTIGUOUS"] and y3.dtype == np.float32
    np.testing.assert_array_equal(X3, pima["X"])
    np.testing.assert_array_equal(y3, pima["y"])


def test_describe_matches_scipy_and_save_roundtrip(tmp_path):
    import scipy.stats
    m = np.random.RandomState(1).randn(500, 4) * np.array([1., 2., 3., 4.]) + 1.0
    d, s = describe(m), scipy.stats.describe(m)
    np.testing.assert_allclose(d["mean"], s.mean, rtol=1e-13)
    np.testing.assert_allclose(d["variance"], s.variance, rtol=1e-13)
    ess = effective_sample_size(m)
    assert np.all(ess > 300) and np.all(ess <= 500 * 1.5)
    ar = np.cumsum(m, axis=0)            # strongly autocorrelated: tiny ESS
    assert np.all(effective_sample_size(ar) < 30)
    p = save_samples(m, str(tmp_path / "out.parquet"))
    import pandas as pd
    df = pd.read_parquet(p)
    assert list(df.columns) == ["b0", "b1", "b2", "b3"]
    np.testing.assert_array_equal(df.to_numpy(), m)


@pytest.mark.gpu
def test_map_estimate_matches_reference_map(pima):
    """fit-np-ul.py:54 (BFGS with the hand-coded gradient): same optimum as the reference run."""
    import logreg_b200 as lr
    from logreg_b200.workflow import map_estimate
    prob = lr.bind_data(np.asfortranarray(pima["X"]), pima["y"], pima["pscale"])
    b0 = np.array([-9.8, 0.1, 0.03, -0.005, 0.0, 0.08, 1.8, 0.04])
    before = prob.info()["eval_launches"]
    res = map_estimate(prob, b0, method="BFGS")
    used = prob.info()["eval_launches"] - before
    np.testing.assert_allclose(res.x, pima["map"], rtol=1e-5, atol=1e-6)
    assert -res.fun == pytest.approx(-100.44943693563214, rel=1e-10)
    assert np.max(np.abs(prob.glp(res.x))) < 1e-3
    assert used <= res.nfev + 1          # ONE fused pass per (lpost, glp) pair


@pytest.mark.gpu
def test_example_script_runs_all_samplers(tmp_path):
    for sampler, iters, thin in (("rwmh", 200, 50), ("ul", 100, 100), ("mala", 200, 50), ("hmc", 200, 2)):
        out = tmp_path / f"{sampler}.parquet"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "fit_pima.py"), "--sampler", sampler,
                            "--iters", str(iters), "--thin", str(thin), "--out", str(out)],
                           capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        import pandas as pd
        df = pd.read_parquet(out)
        assert df.shape == (iters, 8)
        m = df.to_numpy().mean(axis=0)
        # posterior mean of the intercept is about -9.2 +- 1.2, of b6 about 1.3 +- 0.7
        assert -14 < m[0] < -5 and -1.5 < m[6] < 4.5, (sampler, m)


@pytest.mark.gpu
def test_zero_length_runs_and_empty_inputs(pima):
    import logreg_b200 as lr
    prob = lr.Problem().bind_data(pima["X"], pima["y"], pima["pscale"])
    k = lr.malaKernel(prob.lpost, prob.glp, dt=1e-5, pre=pima["pre"])
    mat, acc = prob.run(k, pima["chain_init"], 10, 0)
    assert mat.shape == (0, 8) and acc == 0
    out = lr.mcmc(pima["chain_init"], k, thin=3, iters=0, verb=False)
    assert out.shape == (0, 8)
    with pytest.raises(lr.LogregB200Error, match="positive"):
        lr.Problem().bind_data(np.zeros((0, 8)), np.zeros(0, dtype=np.float32))
