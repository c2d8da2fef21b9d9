"""The steps either side of the hot path (SURVEY.md 8f), as thin host helpers around the
device kernels: data ingest (f2), MAP initialisation (f1), output + summaries (f3), and what a
fitted model is for: predictions and WAIC / held-out lppd over the posterior draws.

Reference lines mirrored (paths relative to the reference root):
    load_pima       Python/fit-numpy.py:12-19 (parquet -> X with a ones column, y float32)
                    C/fit-bayes.c:46-68 reads the same table from the text file pima.data
    map_estimate    method="newton": Python/fit-jax.py:62-79, Newton with the exact Hessian and step
                    halving, on the device (lrb_map: X'WX block kernel, Cholesky solve, decisions);
                    method="BFGS": Python/fit-np-ul.py:54  minimize(-lpost, init, jac=-glp, method='BFGS'),
                    SciPy on the host around the fused evaluation (one pass per iteration)
    describe_device running mean / covariance accumulated on the device during the run (lrb_run_moments;
                    Dex/djwutils.dx:97-103 meanAndCovariance)
    save_samples    Python/fit-numpy.py:89-90  DataFrame(out, columns=b0..).to_parquet(...)
    describe        Python/fit-numpy.py:92-96  scipy.stats.describe(out): mean / variance

Beyond the reference (which stops at the samples), over S posterior draws on the device
(lrb_predictive, one pass over the bound rows for all draws):
    waic            elpd_waic, p_waic, lppd, se_elpd_waic of the rows bound to a Problem: WAIC on the
                    training rows, or the held-out lppd on a Problem bound to test rows
    waic_from_pointwise  the same totals from per-row lppd / p_waic arrays, e.g. of several Problems
    predict_proba   posterior mean and sd of P(y = 1 | x) for unlabelled rows
and PSIS-LOO (lrb_loo: Pareto-smoothed importance-sampling leave-one-out, R's loo::loo()):
    loo             elpd_loo, p_loo, looic and their SEs, with the Pareto k-hat diagnostic (k_max,
                    n_k_high) of the rows bound to a Problem
    loo_from_pointwise  the same totals from per-row elpd_loo / p_loo / pareto_k, e.g. of several Problems
    loo_compare     elpd difference of two models on the same rows and its SE (loo::loo_compare)
"""
from __future__ import annotations

import numpy as np


def load_pima(path):
    """Pima.tr as the scripts build it: X (n x 8, float64, column-major, leading ones), y float32.
    Accepts pima.parquet (pandas/pyarrow), the space-separated pima.data, or an .npz with X, y."""
    path = str(path)
    if path.endswith(".npz"):
        g = np.load(path)
        return np.asfortranarray(g["X"]), g["y"].astype(np.float32)
    if path.endswith(".parquet"):
        import pandas as pd
        df = pd.read_parquet(path)
        n = df.shape[0]
        y = pd.get_dummies(df["type"])["Yes"].to_numpy(dtype="float32")
        X = df.drop(columns="type").to_numpy()
        return np.asfortranarray(np.hstack((np.ones((n, 1)), X))), y
    rows = [line.split() for line in open(path) if line.strip()]
    y = np.array([1.0 if r[-1].strip('"') == "Yes" else 0.0 for r in rows], dtype=np.float32)
    X = np.array([[float(v) for v in r[:-1]] for r in rows])
    return np.asfortranarray(np.hstack((np.ones((len(rows), 1)), X))), y


class MapResult(dict):
    """Result of map_estimate: attribute access like scipy's OptimizeResult (x, fun, nit, success)."""
    __getattr__ = dict.__getitem__


def map_estimate(problem, init, method="newton", tol=None, maxit=None, **kw):
    """MAP estimate, the `init` of the samplers.

    method="newton" (default): the reference's Newton loop (fit-jax.py:62-79) entirely on the
        device -- gradient and lpost from the fused kernel, the Hessian X'WX + diag(pscale^-2) from
        a float64 block kernel, Cholesky solve and step halving in device kernels (lrb_map).
        tol (default 0.01, the reference's) bounds ||glp||; maxit defaults to 500.
    method="BFGS" (or any scipy.optimize.minimize method): quasi-Newton with the hand-coded gradient
        as fit-np-ul.py:54; lpost and glp at the same point come from ONE fused pass over X (the
        reference spends three per iteration), the iteration itself runs in SciPy on the host."""
    init = np.asarray(init, dtype=np.float64)
    if method.lower() == "newton":
        x, info = problem.map(init, tol=0.01 if tol is None else tol, maxit=500 if maxit is None else maxit)
        return MapResult(x=x, fun=-info["lpost"], nit=info["iterations"], success=bool(info["converged"]),
                         nfev=info["evals"], halvings=info["halvings"], grad_norm=info["grad_norm"], method="newton")
    from scipy.optimize import minimize
    if tol is not None:
        kw.setdefault("tol", tol)
    if maxit is not None:
        kw.setdefault("options", {}).setdefault("maxiter", maxit)

    def fun(b):
        lp, _, g = problem.eval(b, want_grad=True)
        return -lp, -g

    res = minimize(fun, init, jac=True, method=method, **kw)
    return res


def describe_device(problem, pooled=True):
    """The same summary from the moments the device accumulated during run(..., moments=True):
    nothing but O(p^2) numbers crosses the bus (what config 4's 4096 chains need)."""
    n, mean, cov = problem.moments(pooled=pooled, cov=True)
    var = np.diagonal(cov, axis1=-2, axis2=-1)
    return {"nobs": n, "mean": mean, "variance": var, "covariance": cov}


def describe(mat):
    """mean / variance per coefficient (ddof=1), the numbers fit-numpy.py:95-96 prints."""
    mat = np.asarray(mat, dtype=np.float64)
    return {"nobs": mat.shape[0], "mean": mat.mean(axis=0), "variance": mat.var(axis=0, ddof=1),
            "min": mat.min(axis=0), "max": mat.max(axis=0)}


def effective_sample_size(mat, max_lag=200):
    """Per-coefficient ESS from the initial positive sequence of autocorrelations (what
    smfsb::mcmcSummary reports in Python/analyse.R:16)."""
    mat = np.asarray(mat, dtype=np.float64)
    n, p = mat.shape
    out = np.empty(p)
    for j in range(p):
        x = mat[:, j] - mat[:, j].mean()
        v = x.dot(x) / n
        if v == 0:
            out[j] = n
            continue
        s = 0.0
        for k in range(1, min(max_lag, n - 1)):
            r = x[:-k].dot(x[k:]) / (n * v)
            if r <= 0:
                break
            s += r
        out[j] = n / (1 + 2 * s)
    return out


_WAIC_KEYS = ("elpd_waic", "p_waic", "lppd", "se_elpd_waic", "n", "draws")


def waic(problem, draws):
    """WAIC of the rows bound to `problem` over posterior draws (S, p) or (C, iters, p):
    {elpd_waic, p_waic, lppd, se_elpd_waic, n, draws}, with lppd = sum_i log mean_s p(y_i | beta_s),
    p_waic = sum_i var_s log p(y_i | beta_s), elpd_waic = lppd - p_waic and
    se_elpd_waic = sqrt(n var_i(elpd_i)) as R's loo package reports them. Bound to held-out rows,
    `lppd` is the held-out log pointwise predictive density. Nothing per row leaves the device."""
    t = problem.predictive(draws, pointwise=False)
    return {k: t[k] for k in _WAIC_KEYS}


def waic_from_pointwise(lppd, p_waic, draws):
    """The totals of `waic` from per-row arrays (predictive(...)["pointwise"]["lppd"] / ["p_waic"]),
    e.g. concatenated over Problems holding parts of one data set; `draws` is S."""
    lppd = np.asarray(lppd, dtype=np.float64)
    p_waic = np.asarray(p_waic, dtype=np.float64)
    elpd = lppd - p_waic
    n = elpd.shape[0]
    return {"elpd_waic": float(elpd.sum()), "p_waic": float(p_waic.sum()), "lppd": float(lppd.sum()),
            "se_elpd_waic": float(np.sqrt(n * elpd.var(ddof=1))) if n > 1 else float("nan"),
            "n": n, "draws": int(draws)}


_LOO_KEYS = ("elpd_loo", "se_elpd_loo", "p_loo", "se_p_loo", "looic", "se_looic", "k_threshold", "k_max",
             "n_k_high", "n", "draws")


def loo(problem, draws):
    """PSIS-LOO of the rows bound to `problem` over posterior draws (S, p) or (C, iters, p), as
    R's loo package reports it (r_eff = 1): {elpd_loo, se_elpd_loo, p_loo, se_p_loo, looic,
    se_looic, k_threshold, k_max, n_k_high, n, draws}. Rows with pareto_k > k_threshold (n_k_high of
    them) have unreliable elpd_loo terms. Nothing per row leaves the device."""
    t = problem.loo(draws, pointwise=False)
    return {k: t[k] for k in _LOO_KEYS}


def _se(v):
    n = v.shape[0]
    return float(np.sqrt(n * v.var(ddof=1))) if n > 1 else float("nan")


def loo_from_pointwise(elpd_loo, p_loo, pareto_k, draws):
    """The totals of `loo` from per-row arrays (loo(...)["pointwise"]), e.g. concatenated over
    Problems holding parts of one data set; `draws` is S."""
    e = np.asarray(elpd_loo, dtype=np.float64)
    p = np.asarray(p_loo, dtype=np.float64)
    k = np.asarray(pareto_k, dtype=np.float64)
    thr = min(1.0 - 1.0 / np.log10(draws), 0.7) if draws > 1 else -np.inf
    return {"elpd_loo": float(e.sum()), "se_elpd_loo": _se(e), "p_loo": float(p.sum()), "se_p_loo": _se(p),
            "looic": -2.0 * float(e.sum()), "se_looic": 2.0 * _se(e), "k_threshold": float(thr),
            "k_max": float(k.max()), "n_k_high": int(np.sum(k > thr)), "n": e.shape[0], "draws": int(draws)}


def loo_compare(elpd_a, elpd_b):
    """Model comparison on the same rows from pointwise elpd_loo (loo::loo_compare for two models):
    elpd_diff = sum(elpd_a - elpd_b) (positive: model a predicts better) and
    se_diff = sqrt(n var(elpd_a - elpd_b)) (ddof 1)."""
    a = np.asarray(elpd_a, dtype=np.float64)
    b = np.asarray(elpd_b, dtype=np.float64)
    if a.shape != b.shape or a.ndim != 1:
        raise ValueError(f"pointwise elpd of both models must be 1-D over the same rows, got {a.shape} and {b.shape}")
    d = a - b
    return {"elpd_diff": float(d.sum()), "se_diff": _se(d)}


def predict_proba(X_new, draws, mode="fp64", device=0):
    """Posterior mean and sd (ddof 1) of P(y = 1 | x) = sigmoid(x.beta) over the draws for the
    rows of X_new (n_new, p): returns (prob_mean, prob_sd) as NumPy arrays. X_new is bound to a
    fresh Problem with all-zero labels; the labels are unused (only the two probability outputs
    are requested)."""
    from .api import Problem
    X_new = np.asarray(X_new)
    prob = Problem(device)
    try:
        prob.bind_data(X_new, np.zeros(X_new.shape[0], dtype=np.float32), mode=mode)
        pw = prob._predictive(draws, ("prob_mean", "prob_sd"), device_out=False)["pointwise"]
    finally:
        prob.close()
    return pw["prob_mean"], pw["prob_sd"]


def save_samples(mat, path):
    """Samples -> parquet (columns b0..b{p-1}, fit-numpy.py:89-90) or .npy / .tsv by extension."""
    path = str(path)
    cols = [f"b{j}" for j in range(mat.shape[1])]
    if path.endswith(".parquet"):
        import pandas as pd
        pd.DataFrame(mat, columns=cols).to_parquet(path)
    elif path.endswith(".tsv"):
        np.savetxt(path, mat, delimiter="\t", header="\t".join(cols), comments="")
    else:
        np.save(path, mat)
    return path
