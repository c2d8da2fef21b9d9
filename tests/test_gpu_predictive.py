"""Posterior predictive probabilities, lppd and WAIC over posterior draws on the device
(lrb_predictive / Problem.predictive / workflow.waic, predict_proba) against a float64
NumPy/SciPy restatement on the same rows (read back with copy_rows)."""
import numpy as np
import pytest
from scipy.special import expit, logsumexp

pytestmark = pytest.mark.gpu

# FP32 mode: worst relative difference of p_waic[i] from FP64 mode on identical rows, 2.4e-6 as
# measured over the synthetic grid below on a B200 (DESIGN.md 3.6), times 3
PWAIC_FP32_BOUND = 3 * 2.4e-6


@pytest.fixture(scope="module")
def lr():
    import logreg_b200
    assert logreg_b200.device_count() >= 1
    return logreg_b200


def reference(X, y, B):
    """The per-row outputs and totals in float64 NumPy/SciPy."""
    eta = X @ B.T                                    # n x S
    z = np.where(np.asarray(y)[:, None] > 0, eta, -eta)
    ll = -np.logaddexp(0.0, -z)                      # log p(y_i | beta_s)
    sig = expit(eta)
    S = B.shape[0]
    lppd = logsumexp(ll, axis=1) - np.log(S)
    if S > 1:
        psd, pw = sig.std(axis=1, ddof=1), ll.var(axis=1, ddof=1)
    else:
        psd = pw = np.full(X.shape[0], np.nan)
    e = lppd - pw
    tot = {"lppd": lppd.sum(), "p_waic": pw.sum(), "elpd_waic": e.sum(),
           "se_elpd_waic": np.sqrt(len(e) * e.var(ddof=1)) if len(e) > 1 else np.nan}
    return {"prob_mean": sig.mean(axis=1), "prob_sd": psd, "lppd": lppd, "p_waic": pw}, tot


def rel_err(got, ref):
    """max |got - ref| / max(1, |ref|), NaN where (and only where) ref is NaN."""
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    np.testing.assert_array_equal(np.isnan(got), np.isnan(ref))
    ok = ~np.isnan(ref)
    if not ok.any():
        return 0.0
    return float(np.max(np.abs(got[ok] - ref[ok]) / np.maximum(1.0, np.abs(ref[ok]))))


def pima_draws(lr, pima, S, seed=11):
    prob = lr.Problem().bind_data(np.asfortranarray(pima["X"]), pima["y"], pima["pscale"], mode="fp64")
    k = lr.hmcKernel(prob.lpost, prob.glp, eps=2e-3, l=7, dmm=1 / pima["pre"])
    mat, acc = prob.run(k, pima["chain_init"], 2, S, seed=seed)
    assert acc > S // 4
    return prob, mat


def test_pima_fp64_matches_numpy(lr, pima):
    prob, B = pima_draws(lr, pima, 500)
    out = prob.predictive(B)
    ref, tot = reference(np.asarray(pima["X"]), pima["y"], B)
    for k in ("prob_mean", "prob_sd", "lppd", "p_waic"):
        assert rel_err(out["pointwise"][k], ref[k]) <= 1e-12, k
    for k in ("lppd", "p_waic", "elpd_waic", "se_elpd_waic"):
        assert abs(out[k] - tot[k]) <= 1e-12 * max(1.0, abs(tot[k])), (k, out[k], tot[k])
    assert out["n"] == 200 and out["draws"] == 500


def test_single_draw_lppd_is_the_log_likelihood(lr, pima):
    prob, B = pima_draws(lr, pima, 3)
    b = B[-1]
    out = prob.predictive(b[None, :])
    assert abs(out["lppd"] - prob.ll(b)) <= 1e-12 * abs(prob.ll(b))
    assert np.all(np.isnan(out["pointwise"]["prob_sd"])) and np.all(np.isnan(out["pointwise"]["p_waic"]))
    assert np.isnan(out["p_waic"]) and np.isnan(out["elpd_waic"])
    q = lr.Problem()
    bt = q.gen_synthetic(100_003, 64, mode="fp32", seed=4)
    o32 = q.predictive(bt[None, :], pointwise=False)
    assert abs(o32["lppd"] - q.ll(bt)) <= 1e-5 * abs(q.ll(bt))


def test_synthetic_grid_fp32_against_numpy_and_fp64_mode(lr):
    """Every padded width (p = 3 .. 256 -> P = 8 .. 256), S below, at and above the 64-draw tile,
    n not a multiple of the 64-row tile; both modes on identical rows."""
    n = 3001
    rs = np.random.RandomState(0)
    worst_pw = 0.0
    for p in (3, 8, 33, 64, 130, 256):
        a, b = lr.Problem(), lr.Problem()
        bt = a.gen_synthetic(n, p, mode="fp32", seed=p)
        b.gen_synthetic(n, p, mode="fp64", seed=p, beta_true=bt)
        X, y = a.copy_rows(0, n)
        np.testing.assert_array_equal(X, b.copy_rows(0, n)[0])
        for S in (1, 7, 64, 1000):
            B = bt + 0.1 * rs.randn(S, p)
            o32, o64 = a.predictive(B), b.predictive(B)
            ref, tot = reference(X, y, B)
            w32, w64 = o32["pointwise"], o64["pointwise"]
            tag = (p, S)
            assert np.max(np.abs(w32["prob_mean"] - ref["prob_mean"])) <= 1e-6, tag
            np.testing.assert_allclose(w32["lppd"], ref["lppd"], rtol=1e-5, atol=0, err_msg=str(tag))
            assert abs(o32["lppd"] - tot["lppd"]) <= 1e-5 * abs(tot["lppd"]), tag
            for k in ("prob_mean", "prob_sd", "lppd", "p_waic"):          # FP64 mode: float64 throughout
                assert rel_err(w64[k], ref[k]) <= 1e-12, (tag, k)
            if S > 1:
                for k in ("p_waic", "elpd_waic"):
                    assert abs(o32[k] - tot[k]) <= 1e-5 * abs(tot[k]), (tag, k)
                assert abs(o32["se_elpd_waic"] - tot["se_elpd_waic"]) <= 1e-5 * abs(tot["se_elpd_waic"]), tag
                assert np.max(np.abs(w32["prob_sd"] - ref["prob_sd"])) <= 1e-6, tag
                worst_pw = max(worst_pw, float(np.max(np.abs(w32["p_waic"] - w64["p_waic"]) / w64["p_waic"])))
    print(f"\nFP32-mode p_waic[i] vs FP64 mode: worst relative difference {worst_pw:.3e}")
    assert worst_pw <= PWAIC_FP32_BOUND


def test_extreme_rows_lppd_is_finite_and_exact(lr):
    """|eta| up to ~700; on the rows whose label disagrees every draw gives p(y | beta) < 1e-300,
    where exp(l) underflows: lppd must still be log-mean-exp of l to 1e-12."""
    rs = np.random.RandomState(7)
    n, p, S = 999, 5, 300
    b0 = np.array([0.5, -1.0, 0.7, 0.2, -0.4])
    V = rs.randn(n, p)
    V += ((1.0 - V @ b0) / (b0 @ b0))[:, None] * b0      # V @ b0 == 1, |V| ~ sqrt(p)
    a = np.linspace(-700.0, 700.0, n)
    X = V * a[:, None]
    y = (rs.rand(n) < 0.5).astype(np.float32)
    far = np.abs(a) > 695
    y[far] = a[far] < 0                                  # label against the sign: l ~ -|eta|
    B = b0 + 1e-4 * rs.randn(S, p)
    prob = lr.Problem().bind_data(X, y, mode="fp64")
    out = prob.predictive(B)
    ref, tot = reference(prob.copy_rows(0, n)[0], y, B)
    eta = X @ B.T
    assert np.max(np.abs(eta)) > 690
    lpy = np.where(y[:, None] > 0, -np.logaddexp(0, -eta), -np.logaddexp(0, eta))
    assert np.sum(np.all(lpy < np.log(1e-300), axis=1)) >= 5
    lp = out["pointwise"]["lppd"]
    assert np.all(np.isfinite(lp))
    # (on the rows the model predicts right lppd ~ -1e-301, which NumPy's logsumexp - log S rounds to 0)
    for k in ("lppd", "prob_mean", "prob_sd", "p_waic"):
        assert rel_err(out["pointwise"][k], ref[k]) <= 1e-12, k
    assert abs(out["lppd"] - tot["lppd"]) <= 1e-12 * abs(tot["lppd"])


def test_held_out_rows_predict_proba_and_waic(lr, pima):
    from logreg_b200 import workflow as W
    X = np.asarray(pima["X"])
    y = pima["y"]
    train = lr.Problem().bind_data(np.asfortranarray(X[:150]), y[:150], pima["pscale"], mode="fp64")
    k = lr.hmcKernel(train.lpost, train.glp, eps=2e-3, l=7, dmm=1 / pima["pre"])
    B, _ = train.run(k, pima["chain_init"], 2, 400, seed=3)
    pm, psd = W.predict_proba(X[150:], B)
    ref, _ = reference(X[150:], y[150:], B)
    assert rel_err(pm, ref["prob_mean"]) <= 1e-12 and rel_err(psd, ref["prob_sd"]) <= 1e-12
    test = lr.Problem().bind_data(np.asfortranarray(X[150:]), y[150:], pima["pscale"], mode="fp64")
    w = W.waic(test, B)
    assert set(w) == {"elpd_waic", "p_waic", "lppd", "se_elpd_waic", "n", "draws"}
    assert w["n"] == 50 and w["draws"] == 400
    assert abs(w["lppd"] - ref["lppd"].sum()) <= 1e-12 * abs(ref["lppd"].sum())
    wt = W.waic(train, B)                                 # WAIC on the training rows
    rt, tt = reference(X[:150], y[:150], B)
    assert abs(wt["elpd_waic"] - tt["elpd_waic"]) <= 1e-12 * abs(tt["elpd_waic"])
    assert abs(wt["se_elpd_waic"] - tt["se_elpd_waic"]) <= 1e-12 * abs(tt["se_elpd_waic"])


def test_bit_reproducible_and_device_out(lr):
    import torch
    n, p, S = 200_001, 64, 300
    a = lr.Problem()
    bt = a.gen_synthetic(n, p, mode="fp32", seed=9)
    B = (bt + 0.02 * np.random.RandomState(1).randn(S, p)).reshape(3, 100, p)    # (C, iters, p)
    o1, o2 = a.predictive(B), a.predictive(B)
    d = lr.Problem(deterministic=True)
    d.gen_synthetic(n, p, mode="fp32", seed=9, beta_true=bt)
    o3 = d.predictive(B)
    dv = a.predictive(B, device_out=True)
    for k in ("prob_mean", "prob_sd", "lppd", "p_waic"):
        np.testing.assert_array_equal(o1["pointwise"][k], o2["pointwise"][k])
        np.testing.assert_array_equal(o1["pointwise"][k], o3["pointwise"][k])
        t = dv["pointwise"][k]
        assert t.is_cuda and t.dtype == torch.float64
        np.testing.assert_array_equal(t.cpu().numpy(), o1["pointwise"][k])
    for k in ("lppd", "p_waic", "elpd_waic", "se_elpd_waic"):
        assert o1[k] == o2[k] == o3[k] == dv[k], k
    assert o1["draws"] == S


def test_a_paused_chain_continues_as_if_nothing_happened(lr, pima):
    X = np.asfortranarray(pima["X"])
    full = lr.Problem(deterministic=True).bind_data(X, pima["y"], pima["pscale"])
    kf = lr.hmcKernel(full.lpost, full.glp, eps=2e-3, l=7, dmm=1 / pima["pre"])
    m_full, acc_full = full.run(kf, pima["chain_init"], 1, 40, seed=21)
    q = lr.Problem(deterministic=True).bind_data(X, pima["y"], pima["pscale"])
    k = lr.hmcKernel(q.lpost, q.glp, eps=2e-3, l=7, dmm=1 / pima["pre"])
    m1, acc1 = q.run(k, pima["chain_init"], 1, 20, seed=21)
    last_x, launches = q._last_x, q.info()["kernel_launches"]
    q.predictive(m1)
    assert q._last_x == last_x
    assert q.info()["kernel_launches"] == launches + 1
    m2, acc2 = q.run(k, None, 1, 20, seed=21)
    np.testing.assert_array_equal(np.vstack([m1, m2]), m_full)
    assert acc1 <= acc2 == acc_full          # the counter of a continued chain is cumulative


def test_headline_shape_windows_and_totals(lr):
    from logreg_b200 import workflow as W
    n, p, S = 100_000_000, 64, 64
    q = lr.Problem()
    bt = q.gen_synthetic(n, p, mode="fp32", seed=42)
    B = bt + 0.1 * np.random.RandomState(2).randn(S, p)
    out = q.predictive(B)
    pw = out["pointwise"]
    for r0 in (0, n // 2 - 50_000, n - 100_000):
        X, y = q.copy_rows(r0, 100_000)
        ref, _ = reference(X, y, B)
        sl = slice(r0, r0 + 100_000)
        assert np.max(np.abs(pw["prob_mean"][sl] - ref["prob_mean"])) <= 1e-6, r0
        assert np.max(np.abs(pw["prob_sd"][sl] - ref["prob_sd"])) <= 1e-6, r0
        np.testing.assert_allclose(pw["lppd"][sl], ref["lppd"], rtol=1e-5, atol=0, err_msg=str(r0))
        err = float(np.max(np.abs(pw["p_waic"][sl] - ref["p_waic"]) / ref["p_waic"]))
        print(f"\nrows {r0}..: FP32-mode p_waic[i] vs NumPy float64: worst relative difference {err:.3e}")
        assert err <= PWAIC_FP32_BOUND, r0
    host = W.waic_from_pointwise(pw["lppd"], pw["p_waic"], S)
    for k in ("lppd", "p_waic", "elpd_waic", "se_elpd_waic"):
        assert abs(out[k] - host[k]) <= 1e-12 * abs(host[k]), (k, out[k], host[k])
    assert out["n"] == n


def test_errors(lr, pima):
    from logreg_b200 import _native as N
    prob = lr.Problem().bind_data(np.asfortranarray(pima["X"]), pima["y"], pima["pscale"])
    with pytest.raises(lr.LogregB200Error) as e:
        prob.predictive(np.zeros((5, 9)))
    assert e.value.code == N.E_BAD_ARG
    with pytest.raises(lr.LogregB200Error) as e:
        prob.predictive(np.zeros((0, 8)))
    assert e.value.code == N.E_BAD_ARG
    with pytest.raises(lr.LogregB200Error) as e:
        lr.Problem().predictive(np.zeros((5, 8)))
    assert e.value.code == N.E_STATE
