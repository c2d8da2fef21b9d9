"""PSIS-LOO restated in NumPy: R's loo package, psis() with r_eff = 1 (Vehtari, Simpson, Gelman,
Yao & Gabry 2024; generalized Pareto fit of Zhang & Stephens 2009 with loo's weak prior and wip
adjustment). `psis` and `gpdfit` are the specification, one row at a time; `psis_rows` is the same
statement vectorized over rows, and `loo_pointwise` turns a log-likelihood matrix into the per-row
elpd_loo, p_loo and pareto_k. Ties are ordered stably, so the log weights of tied draws are
well-defined (any order gives the same elpd_loo)."""
import numpy as np

EPS = np.finfo(float).eps


def lse(a, axis=None):
    """log sum exp with a NaN-propagating max as the reference point."""
    a = np.asarray(a, dtype=np.float64)
    m = np.max(a, axis=axis, keepdims=True)
    out = m + np.log(np.sum(np.exp(a - m), axis=axis, keepdims=True))
    return out.reshape(()) if axis is None else np.squeeze(out, axis=axis)


def tail_len(S):
    return int(np.ceil(min(0.2 * S, 3 * np.sqrt(S))))


def gpdfit(x):
    N = len(x)
    prior = 3.0
    M = 30 + int(np.floor(np.sqrt(N)))
    j = np.arange(1, M + 1)
    xstar = x[int(np.floor(N / 4 + 0.5)) - 1]
    with np.errstate(all="ignore"):
        theta = 1 / x[-1] + (1 - np.sqrt(M / (j - 0.5))) / prior / xstar
        k = np.mean(np.log1p(-theta[:, None] * x[None, :]), axis=1)
        l_theta = N * (np.log(-theta / k) - k - 1)
        theta_hat = np.sum(theta * np.exp(l_theta - lse(l_theta)))
        k = np.mean(np.log1p(-theta_hat * x))
        sigma = -k / theta_hat
        k = k * N / (N + 10) + 10 * 0.5 / (N + 10)
    return (np.inf if np.isnan(k) else k), sigma


def psis(r):
    r = np.asarray(r, dtype=np.float64)
    S = len(r)
    lw = r - r.max()
    khat = np.inf
    M = tail_len(S)
    if M >= 5:
        order = np.argsort(lw, kind="stable")
        xs = lw[order]
        tail = xs[S - M:]
        if abs(tail.max() - tail.min()) >= EPS / 100:
            cutoff = xs[S - M - 1]
            k, sigma = gpdfit(np.exp(tail) - np.exp(cutoff))
            if np.isfinite(k):
                p = (np.arange(1, M + 1) - 0.5) / M
                with np.errstate(all="ignore"):
                    lw[order[S - M:]] = np.log(sigma * np.expm1(-k * np.log1p(-p)) / k + np.exp(cutoff))
            khat = k
    lw[lw > 0] = 0
    return lw + r.max(), khat


def psis_rows(R, chunk=256):
    """psis of every row of R (rows x S): (log weights, k-hat per row)."""
    R = np.asarray(R, dtype=np.float64)
    n, S = R.shape
    LW = np.empty_like(R)
    K = np.full(n, np.inf)
    M = tail_len(S)
    for c0 in range(0, n, chunk):
        r = R[c0:c0 + chunk]
        rmax = r.max(axis=1, keepdims=True)
        lw = r - rmax
        if M >= 5:
            order = np.argsort(lw, axis=1, kind="stable")
            xs = np.take_along_axis(lw, order, axis=1)
            tail, cutoff = xs[:, S - M:], xs[:, S - M - 1:S - M]
            fit = np.abs(tail.max(axis=1) - tail.min(axis=1)) >= EPS / 100
            if fit.any():
                x = np.exp(tail[fit]) - np.exp(cutoff[fit])
                N = M
                Mg = 30 + int(np.floor(np.sqrt(N)))
                j = np.arange(1, Mg + 1)
                xstar = x[:, int(np.floor(N / 4 + 0.5)) - 1]
                with np.errstate(all="ignore"):
                    theta = 1 / x[:, -1:] + (1 - np.sqrt(Mg / (j - 0.5)))[None, :] / 3.0 / xstar[:, None]
                    k = np.mean(np.log1p(-theta[:, :, None] * x[:, None, :]), axis=2)
                    l_theta = N * (np.log(-theta / k) - k - 1)
                    theta_hat = np.sum(theta * np.exp(l_theta - lse(l_theta, axis=1)[:, None]), axis=1)
                    k = np.mean(np.log1p(-theta_hat[:, None] * x), axis=1)
                    sigma = -k / theta_hat
                    k = k * N / (N + 10) + 10 * 0.5 / (N + 10)
                k = np.where(np.isnan(k), np.inf, k)
                rows = np.flatnonzero(fit)
                K[c0 + rows] = k
                ok = np.isfinite(k)
                p = (np.arange(1, M + 1) - 0.5) / M
                with np.errstate(all="ignore"):
                    sm = np.log(sigma[ok, None] * np.expm1(-k[ok, None] * np.log1p(-p)[None, :]) / k[ok, None]
                                + np.exp(cutoff[fit][ok]))
                sub = lw[rows[ok]]
                np.put_along_axis(sub, order[rows[ok], S - M:], sm, axis=1)
                lw[rows[ok]] = sub
        lw[lw > 0] = 0
        LW[c0:c0 + chunk] = lw + rmax
    return LW, K


def loo_pointwise(L):
    """elpd_loo, p_loo, pareto_k per row of the log-likelihood matrix L (rows x S draws)."""
    L = np.asarray(L, dtype=np.float64)
    S = L.shape[1]
    LW, K = psis_rows(-L)
    elpd = lse(LW + L, axis=1) - lse(LW, axis=1)
    lppd = lse(L, axis=1) - np.log(S)
    return elpd, lppd - elpd, K


def loo_totals(elpd, p_loo, k, S):
    n = len(elpd)
    thr = min(1 - 1 / np.log10(S), 0.7) if S > 1 else -np.inf
    se = (lambda v: np.sqrt(n * v.var(ddof=1))) if n > 1 else (lambda v: np.nan)
    return {"elpd_loo": elpd.sum(), "se_elpd_loo": se(elpd), "p_loo": p_loo.sum(), "se_p_loo": se(p_loo),
            "looic": -2 * elpd.sum(), "k_threshold": thr, "k_max": k.max(), "n_k_high": int(np.sum(k > thr))}


def log_lik(X, y, B):
    """log p(y_i | beta_s) in float64, rows x draws, as the device computes it."""
    eta = np.asarray(X, dtype=np.float64) @ np.asarray(B, dtype=np.float64).T
    z = np.where(np.asarray(y)[:, None] > 0, eta, -eta)
    return np.minimum(z, 0.0) - np.log1p(np.exp(-np.abs(eta)))
