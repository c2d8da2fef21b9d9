"""Host side of the posterior predictive / WAIC feature: the ABI struct and the WAIC arithmetic
on per-row arrays (no GPU needed)."""
import ctypes as C

import numpy as np


def test_predictive_totals_layout_matches_header():
    from logreg_b200 import _native as N
    # lrb_predictive_totals: int64 n, int64 draws, 4 x double = 48 bytes
    assert C.sizeof(N.PredictiveTotals) == 48
    offsets = {name: getattr(N.PredictiveTotals, name).offset for name, _ in N.PredictiveTotals._fields_}
    assert offsets == {"n": 0, "draws": 8, "lppd": 16, "p_waic": 24, "elpd_waic": 32, "se_elpd_waic": 40}


def test_waic_from_pointwise_equals_numpy_restatement():
    from scipy.special import logsumexp
    from logreg_b200 import workflow as W
    rs = np.random.RandomState(3)
    n, S = 257, 40
    ll = -np.logaddexp(0.0, -rs.randn(n, S) * 2.0 - 1.0)      # log p(y_i | beta_s), i rows, s draws
    lppd_i = logsumexp(ll, axis=1) - np.log(S)
    pw_i = ll.var(axis=1, ddof=1)
    got = W.waic_from_pointwise(lppd_i, pw_i, S)
    elpd_i = lppd_i - pw_i
    assert got["n"] == n and got["draws"] == S
    np.testing.assert_allclose(got["lppd"], lppd_i.sum(), rtol=1e-14)
    np.testing.assert_allclose(got["p_waic"], pw_i.sum(), rtol=1e-14)
    np.testing.assert_allclose(got["elpd_waic"], lppd_i.sum() - pw_i.sum(), rtol=1e-13)
    # loo's se: sqrt(n * var(elpd_i)) with R's var (ddof 1)
    se = np.sqrt(n * np.sum((elpd_i - elpd_i.mean()) ** 2) / (n - 1))
    np.testing.assert_allclose(got["se_elpd_waic"], se, rtol=1e-13)
    assert np.isnan(W.waic_from_pointwise(lppd_i[:1], pw_i[:1], S)["se_elpd_waic"])
