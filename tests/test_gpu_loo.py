"""PSIS-LOO and the pointwise log-likelihood on the device (lrb_loo / lrb_loglik, Problem.loo /
Problem.loglik, workflow.loo) against the NumPy statement of loo's psis() in tests/loo_reference.py,
on log-likelihoods computed in float64 NumPy from the rows read back with copy_rows."""
import numpy as np
import pytest

from tests import loo_reference as R

pytestmark = pytest.mark.gpu

# FP32 mode against FP64 mode on identical rows over the synthetic grid below: worst relative
# difference of elpd_loo[i] and worst absolute difference of pareto_k[i], as measured on a B200
# (DESIGN.md 3.7), times 3
ELPD_FP32_BOUND = 3 * 3.4e-6
K_FP32_BOUND = 3 * 1.8e-2
# The fit sees x = exp(tail lw) - exp(cutoff lw) as the statement forms it: when the tail's log
# ratios span less than ~1e-6, exp(lw) is within that of 1 and x is quantized at the spacing of doubles below 1 (1.1e-16),
# so a one-ulp difference between the device's exp and NumPy's moves k-hat by up to 0.1 (a spread
# of 1e-14 leaves ~30 distinct x). pareto_k is held to 1e-9 on the rows whose tail is wider.
K_WELL_CONDITIONED_SPREAD = 1e-6
POINTWISE = ("elpd_loo", "p_loo", "pareto_k")


@pytest.fixture(scope="module")
def lr():
    import logreg_b200
    assert logreg_b200.device_count() >= 1
    return logreg_b200


def rel_err(got, ref):
    """max |got - ref| / max(1, |ref|); NaN and inf where (and only where) ref has them."""
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    np.testing.assert_array_equal(np.isfinite(got), np.isfinite(ref))
    np.testing.assert_array_equal(got[~np.isfinite(ref)], ref[~np.isfinite(ref)])
    ok = np.isfinite(ref)
    if not ok.any():
        return 0.0
    return float(np.max(np.abs(got[ok] - ref[ok]) / np.maximum(1.0, np.abs(ref[ok]))))


def k_err(got, ref):
    got, ref = np.asarray(got), np.asarray(ref)
    np.testing.assert_array_equal(np.isinf(got), np.isinf(ref))
    ok = np.isfinite(ref)
    return float(np.max(np.abs(got[ok] - ref[ok]))) if ok.any() else 0.0


def reference(X, y, B):
    L = R.log_lik(X, y, B)
    e, p, k = R.loo_pointwise(L)
    S, M = B.shape[0], R.tail_len(B.shape[0])
    r = np.sort(-L, axis=1)
    spread = r[:, -1] - r[:, S - M] if M >= 5 else np.full(len(e), np.inf)
    return ({"elpd_loo": e, "p_loo": p, "pareto_k": k, "tail_spread": spread},
            R.loo_totals(e, p, k, S))


def check_fp64(out, ref, tot, tag):
    pw = out["pointwise"]
    assert rel_err(pw["elpd_loo"], ref["elpd_loo"]) <= 1e-12, tag
    assert rel_err(pw["p_loo"], ref["p_loo"]) <= 1e-12, tag
    wide = ref["tail_spread"] >= K_WELL_CONDITIONED_SPREAD
    np.testing.assert_array_equal(np.isinf(pw["pareto_k"]), np.isinf(ref["pareto_k"]))
    assert k_err(pw["pareto_k"][wide], ref["pareto_k"][wide]) <= 1e-9, tag
    for k in ("elpd_loo", "se_elpd_loo", "p_loo", "se_p_loo", "looic"):
        assert abs(out[k] - tot[k]) <= 1e-12 * max(1.0, abs(tot[k])), (tag, k, out[k], tot[k])
    assert out["k_threshold"] == tot["k_threshold"] and out["n_k_high"] == tot["n_k_high"], tag
    assert out["k_max"] == tot["k_max"] or abs(out["k_max"] - tot["k_max"]) <= 1e-9, tag


def test_loglik_matches_numpy(lr, monkeypatch):
    """Every padded width in both modes, ragged n, windows at row0 > 0 and across chunk
    boundaries (a 1 MB chunk budget: 128 rows at S = 1000), host and device output."""
    import torch
    monkeypatch.setenv("LRB_LOO_CHUNK_MB", "1")
    n, S = 3001, 1000
    rs = np.random.RandomState(0)
    for p in (3, 8, 33, 64, 130, 256):
        for mode, tol in (("fp64", 1e-12), ("fp32", 1e-5)):
            q = lr.Problem()
            bt = q.gen_synthetic(n, p, mode=mode, seed=p)
            B = bt + 0.1 * rs.randn(S, p)
            X, y = q.copy_rows(0, n)
            ref = R.log_lik(X, y, B)
            for r0, nr in ((0, n), (1, 127), (127, 3), (255, 514), (2937, 64)):
                got = q.loglik(B, r0, nr)
                assert got.shape == (nr, S)
                assert rel_err(got, ref[r0:r0 + nr]) <= tol, (p, mode, r0, nr)
            dv = q.loglik(B, 63, 2938, device_out=True)
            assert dv.is_cuda and dv.dtype == torch.float64 and dv.shape == (2938, S)
            np.testing.assert_array_equal(dv.cpu().numpy(), q.loglik(B, 63))
            q.close()


def pima_draws(lr, pima, S, seed=11):
    prob = lr.Problem().bind_data(np.asfortranarray(pima["X"]), pima["y"], pima["pscale"], mode="fp64")
    k = lr.hmcKernel(prob.lpost, prob.glp, eps=2e-3, l=7, dmm=1 / pima["pre"])
    mat, acc = prob.run(k, pima["chain_init"], 2, S, seed=seed)
    assert acc > S // 4
    return prob, mat


def test_pima_fp64_matches_numpy(lr, pima):
    prob, B = pima_draws(lr, pima, 500)
    assert len(np.unique(B, axis=0)) < len(B)            # rejected proposals: duplicated draws
    out = prob.loo(B)
    ref, tot = reference(np.asarray(pima["X"]), pima["y"], B)
    check_fp64(out, ref, tot, "pima")
    assert out["n"] == 200 and out["draws"] == 500 and out["se_looic"] == 2 * out["se_elpd_loo"]
    from logreg_b200 import workflow as W
    w = W.loo(prob, B)
    assert all(w[k] == out[k] for k in w)


def test_synthetic_grid_both_modes(lr):
    """Widths p = 3 .. 256 x S below, at and above the 21-draw smoothing threshold and the 64-draw
    tile; FP64 against NumPy, FP32 against FP64 mode on identical rows."""
    n = 1001
    rs = np.random.RandomState(1)
    worst_e = worst_k = 0.0
    for p in (3, 8, 33, 64, 130, 256):
        a, b = lr.Problem(), lr.Problem()
        bt = a.gen_synthetic(n, p, mode="fp32", seed=p)
        b.gen_synthetic(n, p, mode="fp64", seed=p, beta_true=bt)
        X, y = a.copy_rows(0, n)
        for S in (1, 20, 21, 64, 1000, 4000):
            B = bt + 0.3 / np.sqrt(p) * rs.randn(S, p)
            o32, o64 = a.loo(B), b.loo(B)
            ref, tot = reference(X, y, B)
            check_fp64(o64, ref, tot, (p, S))
            w32, w64 = o32["pointwise"], o64["pointwise"]
            worst_e = max(worst_e, rel_err(w32["elpd_loo"], w64["elpd_loo"]))
            worst_k = max(worst_k, k_err(w32["pareto_k"], w64["pareto_k"]))
            if S < 21:
                assert np.all(np.isinf(w64["pareto_k"])) and o64["n_k_high"] == n
        a.close()
        b.close()
    print(f"\nFP32 mode vs FP64 mode: elpd_loo[i] worst relative difference {worst_e:.3e}, "
          f"pareto_k[i] worst absolute difference {worst_k:.3e}")
    assert worst_e <= ELPD_FP32_BOUND and worst_k <= K_FP32_BOUND


def test_draw_cap_and_rows_across_chunks(lr):
    """S = 2^21 (the cap): 64 rows per chunk, each row read from global memory (not staged)."""
    from logreg_b200 import _native as N
    n, p, S = 130, 8, 1 << 21
    q = lr.Problem()
    bt = q.gen_synthetic(n, p, mode="fp64", seed=3)
    B = bt + 0.2 * np.random.RandomState(4).randn(S, p)
    out = q.loo(B)
    X, y = q.copy_rows(0, n)
    pw = out["pointwise"]
    for i in (0, 63, 64, 65, 127, 128, 129):
        lw, k = R.psis(-R.log_lik(X[i:i + 1], y[i:i + 1], B)[0])
        l = R.log_lik(X[i:i + 1], y[i:i + 1], B)[0]
        e = R.lse(lw + l) - R.lse(lw)
        assert abs(pw["elpd_loo"][i] - e) <= 1e-12 * max(1.0, abs(e)), i
        assert abs(pw["pareto_k"][i] - k) <= 1e-9, i
        pl = R.lse(l) - np.log(S) - e
        assert abs(pw["p_loo"][i] - pl) <= 1e-12 * max(1.0, abs(pl)), i
    with pytest.raises(lr.LogregB200Error) as e:
        q.loo(np.vstack([B, B[:1]]))
    assert e.value.code == N.E_BAD_ARG and "2^21" in str(e.value)


def influential_problem(lr):
    """Three mislabelled rows that alone inform one coefficient each: draws from the Laplace
    approximation of the posterior give them k-hat well above 0.7."""
    rs = np.random.RandomState(4)
    n, p = 200, 5
    X = np.column_stack([np.ones(n), rs.randn(n, 1), np.zeros((n, 3))])
    y = (rs.rand(n) < 1 / (1 + np.exp(-(0.3 + X[:, 1])))).astype(np.float32)
    bad = [5, 77, 151]
    for j, i in enumerate(bad):
        X[i, 1] = 4.0 if j == 1 else -4.0
        X[i, 2 + j] = 3.0
        y[i] = float(not X[i, 1] > 0)
    ps = np.array([10.0, 1.0, 3.0, 3.0, 3.0])
    prob = lr.Problem().bind_data(X, y, ps, mode="fp64")
    beta, info = prob.map(np.zeros(p))
    assert info["converged"]
    C = np.linalg.cholesky(np.linalg.inv(prob.hessian(beta)))
    B = beta + rs.randn(2000, p) @ C.T
    return prob, X, y, B, bad


def test_influential_rows_get_high_k(lr):
    prob, X, y, B, bad = influential_problem(lr)
    out = prob.loo(B)
    ref, tot = reference(X, y, B)
    check_fp64(out, ref, tot, "influential")
    k = out["pointwise"]["pareto_k"]
    assert np.all(ref["pareto_k"][bad] > tot["k_threshold"]) and np.all(k[bad] > out["k_threshold"])
    assert out["n_k_high"] == tot["n_k_high"] >= 3
    assert out["k_max"] == np.max(k) and abs(out["k_max"] - tot["k_max"]) <= 1e-9


def test_extreme_rows_and_a_zero_row(lr):
    """|eta| up to ~700, where p(y | beta) < 1e-300 for every draw on the mislabelled rows, and a
    row x = 0 (constant log ratios: k-hat = inf, elpd_loo = -log 2, counted in n_k_high)."""
    rs = np.random.RandomState(7)
    n, p, S = 999, 5, 1000
    b0 = np.array([0.5, -1.0, 0.7, 0.2, -0.4])
    V = rs.randn(n, p)
    V += ((1.0 - V @ b0) / (b0 @ b0))[:, None] * b0
    a = np.linspace(-700.0, 700.0, n)
    X = V * a[:, None]
    X[500] = 0.0
    y = (rs.rand(n) < 0.5).astype(np.float32)
    far = np.abs(a) > 695
    y[far] = a[far] < 0
    B = b0 + 1e-4 * rs.randn(S, p)
    prob = lr.Problem().bind_data(X, y, mode="fp64")
    out = prob.loo(B)
    L = R.log_lik(prob.copy_rows(0, n)[0], y, B)
    assert np.sum(np.all(L < np.log(1e-300), axis=1)) >= 5
    ref, tot = reference(prob.copy_rows(0, n)[0], y, B)
    pw = out["pointwise"]
    assert np.all(np.isfinite(pw["elpd_loo"])) and np.all(np.isfinite(pw["p_loo"]))
    check_fp64(out, ref, tot, "extreme")
    assert np.isinf(pw["pareto_k"][500]) and pw["elpd_loo"][500] == pytest.approx(-np.log(2), abs=1e-15)
    assert out["n_k_high"] >= 1 and np.isinf(out["k_max"])


def test_bit_reproducible_and_device_out(lr):
    import torch
    n, p, S = 20_001, 64, 1000
    a = lr.Problem()
    bt = a.gen_synthetic(n, p, mode="fp32", seed=9)
    B = (bt + 0.05 * np.random.RandomState(1).randn(S, p)).reshape(4, 250, p)     # (C, iters, p)
    o1, o2 = a.loo(B), a.loo(B)
    d = lr.Problem(deterministic=True)
    d.gen_synthetic(n, p, mode="fp32", seed=9, beta_true=bt)
    o3 = d.loo(B)
    dv = a.loo(B, device_out=True)
    for k in POINTWISE:
        np.testing.assert_array_equal(o1["pointwise"][k], o2["pointwise"][k])
        np.testing.assert_array_equal(o1["pointwise"][k], o3["pointwise"][k])
        t = dv["pointwise"][k]
        assert t.is_cuda and t.dtype == torch.float64
        np.testing.assert_array_equal(t.cpu().numpy(), o1["pointwise"][k])
    for k in ("elpd_loo", "se_elpd_loo", "p_loo", "se_p_loo", "k_max", "n_k_high"):
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
    last_x = q._last_x
    q.loo(m1)
    q.loglik(m1, 3, 50)
    assert q._last_x == last_x
    m2, acc2 = q.run(k, None, 1, 20, seed=21)
    np.testing.assert_array_equal(np.vstack([m1, m2]), m_full)
    assert acc1 <= acc2 == acc_full


def test_headline_shape_windows_and_totals(lr):
    from logreg_b200 import workflow as W
    n, p, S = 100_000_000, 64, 64
    q = lr.Problem()
    bt = q.gen_synthetic(n, p, mode="fp32", seed=42)
    B = bt + 0.1 * np.random.RandomState(2).randn(S, p)
    out = q.loo(B)
    pw = out["pointwise"]
    for r0 in (0, n // 2 - 50_000, n - 100_000):
        X, y = q.copy_rows(r0, 100_000)
        ref, _ = reference(X, y, B)
        sl = slice(r0, r0 + 100_000)
        e = rel_err(pw["elpd_loo"][sl], ref["elpd_loo"])
        kd = k_err(pw["pareto_k"][sl], ref["pareto_k"])
        print(f"\nrows {r0}..: FP32 mode vs NumPy float64: elpd_loo[i] {e:.3e} relative, pareto_k[i] {kd:.3e}")
        assert e <= ELPD_FP32_BOUND and kd <= K_FP32_BOUND, r0
    host = W.loo_from_pointwise(pw["elpd_loo"], pw["p_loo"], pw["pareto_k"], S)
    for k in ("elpd_loo", "se_elpd_loo", "p_loo", "se_p_loo", "looic"):
        assert abs(out[k] - host[k]) <= 1e-12 * abs(host[k]), (k, out[k], host[k])
    assert out["n_k_high"] == host["n_k_high"] and out["k_max"] == host["k_max"] and out["n"] == n


def test_errors(lr, pima):
    from logreg_b200 import _native as N
    prob = lr.Problem().bind_data(np.asfortranarray(pima["X"]), pima["y"], pima["pscale"])
    for call in (lambda B: prob.loo(B), lambda B: prob.loglik(B)):
        with pytest.raises(lr.LogregB200Error) as e:
            call(np.zeros((5, 9)))
        assert e.value.code == N.E_BAD_ARG
        with pytest.raises(lr.LogregB200Error) as e:
            call(np.zeros((0, 8)))
        assert e.value.code == N.E_BAD_ARG
    with pytest.raises(lr.LogregB200Error) as e:
        prob.loglik(np.zeros((5, 8)), 190, 11)
    assert e.value.code == N.E_BAD_ARG
    for call in (lambda q: q.loo(np.zeros((5, 8))), lambda q: q.loglik(np.zeros((5, 8)), 0, 1)):
        with pytest.raises(lr.LogregB200Error) as e:
            call(lr.Problem())
        assert e.value.code == N.E_STATE


def test_k_max_when_every_k_hat_is_negative(lr):
    """Draws concentrated around one point on 10 rows: every k-hat is negative, and k_max is the
    largest of them (the tile partials of empty threads carry no k)."""
    rs = np.random.RandomState(10)
    X = np.column_stack([np.ones(10), rs.randn(10, 2)])
    y = (rs.rand(10) < 0.5).astype(np.float32)
    B = np.array([0.2, -0.5, 0.8]) + 0.05 * rs.randn(4000, 3)
    prob = lr.Problem().bind_data(X, y, mode="fp64")
    out = prob.loo(B)
    ref, tot = reference(X, y, B)
    assert np.all(ref["pareto_k"] < 0)
    check_fp64(out, ref, tot, "negative k")
    assert out["k_max"] == np.max(out["pointwise"]["pareto_k"]) < 0 and out["n_k_high"] == 0


def smoothing_problem():
    """Rows whose result depends on every step of the smoothing: rows 0-5 have log ratios from a
    GPD with k = 1 (the fitted tail overshoots the largest raw weight on most of them, so the
    truncation at 0 matters), row 6 has one draw with a ratio e^50 times the others (the tail
    outweighs the rest of the row by ~e^50, so a non-tail denominator formed as total - tail would
    cancel to nothing), row 7 is x = 0, and 12 ordinary rows."""
    rs = np.random.RandomState(12)
    S, p = 1000, 8
    B = 0.01 * rs.randn(S, p)
    for j in range(6):
        r = np.log(np.expm1(-1.0 * np.log(rs.rand(S))))        # log GPD(k = 1) ratios
        B[:, j] = np.log(np.expm1(r + 20.0))                   # -l = softplus(eta) = r + 20
    t = 1e-3 + 1e-5 * rs.randn(S)
    t[417] = 50.0
    B[:, 6] = np.log(np.expm1(t))
    X = np.vstack([np.eye(p)[:7], np.zeros(p), rs.randn(12, p) * 0.1])
    y = np.zeros(len(X), dtype=np.float32)
    y[8:] = rs.rand(12) < 0.5
    return X, y, B


def test_rows_that_depend_on_truncation_and_the_denominator(lr):
    X, y, B = smoothing_problem()
    prob = lr.Problem().bind_data(X, y, mode="fp64")
    out = prob.loo(B)
    ref, tot = reference(X, y, B)
    check_fp64(out, ref, tot, "smoothing")
    assert np.all(out["pointwise"]["pareto_k"][:7] > 0.7) and np.isinf(out["pointwise"]["pareto_k"][7])


def test_stage1_only_switch_leaves_nan_outputs(lr, monkeypatch):
    X, y, B = smoothing_problem()
    prob = lr.Problem().bind_data(X, y, mode="fp64")
    monkeypatch.setenv("LRB_LOO_STAGE1_ONLY", "1")
    out = prob.loo(B)
    dv = prob.loo(B, device_out=True)
    for o in (out, dv):
        assert np.isnan(o["elpd_loo"]) and np.isnan(o["k_max"]) and o["n_k_high"] == -1
    for k in POINTWISE:
        assert np.all(np.isnan(out["pointwise"][k])) and bool(dv["pointwise"][k].isnan().all())
