"""Host side of PSIS-LOO: lrb_debug_psis (the PSIS formulas psis_kernel runs, on the host) against
the NumPy statement of loo's psis(), the shape recovery of that statement, the vectorized
reference the GPU tests use, the lrb_loo_totals layout and the host arithmetic of
loo_from_pointwise / loo_compare (no GPU needed)."""
import ctypes as C

import numpy as np
import pytest

from tests import loo_reference as R


def debug_psis(r):
    from logreg_b200 import _native as N
    r = np.ascontiguousarray(r, dtype=np.float64)
    lw = np.empty_like(r)
    k = C.c_double()
    N.check(N.load().lrb_debug_psis(N.as_dp(r), len(r), N.as_dp(lw), C.byref(k)))
    return lw, k.value


def gpd_log_ratios(rs, S, k):
    """log of S draws from a generalized Pareto distribution with shape k, scale 1."""
    return np.log(np.expm1(-k * np.log(rs.rand(S))) / k)


def tied_tail(rs):
    """S = 1000, tail M = 95: 60 distinct largest ratios, then 120 ties, so the cutoff and 35 tail
    values are tied and the first quartile of the exceedances is 0."""
    return rs.permutation(np.concatenate([np.linspace(0.5, 1.5, 60), np.zeros(120), -rs.rand(820) - 0.1]))


def cases():
    rs = np.random.RandomState(5)
    for S in (1, 5, 20, 21, 24, 25, 100, 1000, 4000, 10001):
        yield f"normal-S{S}", rs.randn(S) * 1.5
    for k in (0.3, 0.7, 1.2):
        yield f"gpd-k{k}", gpd_log_ratios(rs, 4000, k)
    yield "constant", np.full(500, -0.6931471805599453)
    r = rs.randn(1000)
    rep = rs.rand(1000) < 0.4                       # 40 % of the draws repeat their predecessor
    for i in np.flatnonzero(rep)[1:] if rep[0] else np.flatnonzero(rep):
        r[i] = r[i - 1]
    yield "duplicates", r
    yield "tail-tied-with-cutoff", tied_tail(rs)           # xstar = 0: k-hat is NaN -> inf
    yield "span-1e3", rs.rand(3000) * 1e3 - 700.0


@pytest.mark.parametrize("name,r", list(cases()), ids=[c[0] for c in cases()])
def test_debug_psis_matches_the_numpy_statement(name, r):
    lw_ref, k_ref = R.psis(r)
    lw, k = debug_psis(r)
    if np.isinf(k_ref):
        assert k == k_ref, (name, k, k_ref)
    else:
        assert abs(k - k_ref) <= 1e-12, (name, k, k_ref)
    np.testing.assert_array_equal(np.isnan(lw), np.isnan(lw_ref))
    err = np.max(np.abs(lw - lw_ref) / np.maximum(1.0, np.abs(lw_ref)))
    assert err <= 1e-12, (name, err)


def test_debug_psis_edge_cases_follow_loo():
    assert np.isinf(debug_psis(np.zeros(20))[1])                       # S < 21: tail shorter than 5
    assert np.isinf(debug_psis(np.random.RandomState(1).randn(20))[1])
    assert np.isfinite(debug_psis(np.random.RandomState(1).randn(21))[1])
    lw, k = debug_psis(np.full(64, 3.0))                               # constant row: no smoothing
    assert np.isinf(k) and np.all(lw == 3.0)
    r = tied_tail(np.random.RandomState(2))
    assert np.isinf(R.psis(r)[1]) and np.isinf(debug_psis(r)[1])       # xstar = 0 -> NaN -> inf


@pytest.mark.parametrize("k", [0.3, 0.7, 1.0])
def test_the_statement_recovers_the_pareto_shape(k):
    """Median k-hat over 200 seeds of GPD(k) log ratios at S = 4000, in the NumPy statement and in
    lrb_debug_psis."""
    ks, kd = [], []
    for seed in range(200):
        r = gpd_log_ratios(np.random.RandomState(1000 + seed), 4000, k)
        ks.append(R.psis(r)[1])
        kd.append(debug_psis(r)[1])
    assert abs(np.median(ks) - k) <= 0.05, np.median(ks)
    assert abs(np.median(kd) - k) <= 0.05, np.median(kd)


def test_vectorized_reference_equals_the_statement():
    rs = np.random.RandomState(8)
    for S in (7, 21, 64, 1000):
        L = -np.abs(rs.randn(37, S)) * rs.rand(37, 1) * 3
        L[3] = -0.6931471805599453                                      # x = 0
        L[5, : S // 2] = L[5, 0]                                       # duplicated draws
        LW, K = R.psis_rows(-L, chunk=10)
        for i in range(L.shape[0]):
            lw, k = R.psis(-L[i])
            np.testing.assert_allclose(LW[i], lw, rtol=1e-13, atol=1e-13)
            assert (k == K[i]) or abs(k - K[i]) <= 1e-12
        elpd, p_loo, k = R.loo_pointwise(L)
        assert abs(elpd[3] + np.log(2)) <= 1e-15 and np.isinf(k[3])


def test_loo_totals_layout_matches_header():
    from logreg_b200 import _native as N
    assert C.sizeof(N.LooTotals) == 80
    offsets = {name: getattr(N.LooTotals, name).offset for name, _ in N.LooTotals._fields_}
    assert offsets == {"n": 0, "draws": 8, "elpd_loo": 16, "se_elpd_loo": 24, "p_loo": 32, "se_p_loo": 40,
                       "looic": 48, "k_threshold": 56, "k_max": 64, "n_k_high": 72}


def test_loo_from_pointwise_and_loo_compare_arithmetic():
    from logreg_b200 import workflow as W
    rs = np.random.RandomState(3)
    n, S = 301, 4000
    e = -np.abs(rs.randn(n))
    p = np.abs(rs.randn(n)) * 0.1
    k = rs.rand(n) * 0.9
    k[7] = np.inf
    got = W.loo_from_pointwise(e, p, k, S)
    thr = min(1 - 1 / np.log10(S), 0.7)
    assert got["k_threshold"] == thr == 0.7
    assert got["n_k_high"] == int(np.sum(k > 0.7)) and got["k_max"] == np.inf
    np.testing.assert_allclose(got["elpd_loo"], e.sum(), rtol=1e-14)
    np.testing.assert_allclose(got["p_loo"], p.sum(), rtol=1e-14)
    np.testing.assert_allclose(got["looic"], -2 * e.sum(), rtol=1e-14)
    se = np.sqrt(n * np.sum((e - e.mean()) ** 2) / (n - 1))
    np.testing.assert_allclose(got["se_elpd_loo"], se, rtol=1e-13)
    np.testing.assert_allclose(got["se_looic"], 2 * se, rtol=1e-13)
    np.testing.assert_allclose(got["se_p_loo"], np.sqrt(n * np.sum((p - p.mean()) ** 2) / (n - 1)), rtol=1e-13)
    assert got["n"] == n and got["draws"] == S
    assert W.loo_from_pointwise(e, p, k, 100)["k_threshold"] == 0.5
    assert np.isnan(W.loo_from_pointwise(e[:1], p[:1], k[:1], S)["se_elpd_loo"])
    b = e + rs.randn(n) * 0.01 - 0.003
    cmp = W.loo_compare(e, b)
    d = e - b
    np.testing.assert_allclose(cmp["elpd_diff"], d.sum(), rtol=1e-13)
    np.testing.assert_allclose(cmp["se_diff"], np.sqrt(n * np.sum((d - d.mean()) ** 2) / (n - 1)), rtol=1e-13)
    assert W.loo_compare(e, e) == {"elpd_diff": 0.0, "se_diff": 0.0}
    with pytest.raises(ValueError):
        W.loo_compare(e, e[:-1])
