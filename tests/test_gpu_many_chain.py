"""The many-chain kernels (C >= 2 coefficient vectors per pass over X) against a float64
NumPy restatement of the same operation, at the widths, tile counts, chain counts and data
regimes where they can go wrong.

  * eval_mc_kernel (SIMT, 4 chains per X batch): every padded width in both modes, row
    counts around one batch (RB = 8192 / (P * itemsize) rows) and past the largest grid,
    chain counts with full and partial 4-chain passes; each chain also equals single-chain
    evaluation of the same coefficients.
  * eval_tc_kernel (tcgen05, FP32 mode, padded P = 64, C >= 12): zero-padded widths, tile
    counts per CTA across the 3-stage ring and the 16-tile gradient flush, chain counts at the
    128-chain group edges and at the SIMT fall-back, bit-exact independence of the chains,
    separable / extreme / one-class / badly scaled data, and the lock-step samplers.
  * eval_kernel (static, deterministic=True) at every width.

Conventions as in test_gpu_eval.py: lpost and ll relative to max(1, |ref|), glp against the
un-cancelled magnitude |X|'|y - p| + |beta / pscale^2| of each chain. The likelihood part is
also bounded on its own (ll relative to |ll|, X'(y - p) against |X|'|y - p|): with large
coefficients, as on separable data, the prior term would hide errors in it. The reference is
computed a few chains at a time, so X . B' is never n x C in memory; large chain counts are
checked chain by chain against the SIMT path on the same handle and on a sample of chains
(always 0, 127, 128 and C - 1) against float64.
"""
import ctypes
import time

import numpy as np
import pytest
from scipy.special import expit

from oracle import logreg_oracle as O

pytestmark = pytest.mark.gpu

TOL = {"fp64": 1e-10, "fp32": 1e-5}
# The tensor-core contraction (3xTF32, float32 accumulation in the MMA) computes eta to
# ~1e-6 relative, where the SIMT kernel's float32 FMAs get ~1e-7: below this floor the
# tensor-core path is not expected to track the SIMT kernel's error.
TC_ETA_FLOOR = 4e-6
TC_MIN_CHAINS = 12          # the library's default crossover to the tensor-core kernel


@pytest.fixture(scope="module")
def lr():
    import logreg_b200
    assert logreg_b200.device_count() >= 1
    t0 = time.perf_counter()
    yield logreg_b200
    print(f"\ntest_gpu_many_chain.py: {time.perf_counter() - t0:.1f} s")


@pytest.fixture(scope="module")
def N():
    from logreg_b200 import _native
    return _native


@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---------------------------------------------------------------- float64 reference
def ref_like(X, y, B, chunk=16):
    """Likelihood part for each row of B: ll, X'(y - p) and |X|'|y - p|, a few chains at a time."""
    B = np.atleast_2d(B)
    C, p = B.shape
    s = 2.0 * np.asarray(y, dtype=np.float64) - 1.0
    Xa = np.abs(X)
    ll, g, mag = np.empty(C), np.empty((C, p)), np.empty((C, p))
    for c0 in range(0, C, chunk):
        z = s[:, None] * (X @ B[c0:c0 + chunk].T)
        ll[c0:c0 + chunk] = np.sum(np.minimum(z, 0.0) - np.log1p(np.exp(-np.abs(z))), axis=0)
        r = s[:, None] * expit(-z)          # y - sigmoid(eta) without cancellation
        g[c0:c0 + chunk] = (X.T @ r).T
        mag[c0:c0 + chunk] = (Xa.T @ np.abs(r)).T
    return ll, g, mag


def lprior(B, ps):
    return np.sum(-0.5 * (B / ps) ** 2 - np.log(ps) - 0.5 * np.log(2 * np.pi), axis=-1)


def errors(X, y, ps, B, res, idx):
    """Errors of the device results res = (lpost, ll, glp) for the chains idx, each a max over them."""
    lp, l, g = res
    idx = np.asarray(idx)
    Bi = B[idx]
    ll_r, gl_r, mag = ref_like(X, y, Bi)
    gpr = -Bi / ps ** 2
    lp_r = ll_r + lprior(Bi, ps)
    ge = np.abs(g[idx] - (gl_r + gpr))
    return dict(
        lpost=float(np.max(np.abs(lp[idx] - lp_r) / np.maximum(1.0, np.abs(lp_r)))),
        ll=float(np.max(np.abs(l[idx] - ll_r) / np.maximum(1.0, np.abs(ll_r)))),
        glp=float(np.max(np.max(ge, axis=1) / np.max(mag + np.abs(gpr), axis=1))),
        ll_like=float(np.max(np.abs(l[idx] - ll_r) / np.maximum(np.abs(ll_r), 1e-300))),
        g_like=float(np.max(np.max(np.abs((g[idx] - gpr) - gl_r), axis=1) / np.maximum(np.max(mag, axis=1), 1e-300))),
    )


def assert_errors(e, tol, what):
    for k in ("lpost", "ll", "glp", "ll_like", "g_like"):
        assert e[k] <= tol, (what, k, e)


def rows(rs, n, p):
    """N(0, 1) rows with an intercept column, float32-representable (both modes store them exactly)."""
    X = rs.randn(n, p).astype(np.float32).astype(np.float64)
    X[:, 0] = 1.0
    return X


def sample(C, rs, extra=3):
    idx = {0, 127, 128, C - 1} | set(rs.randint(0, C, extra).tolist())
    return sorted(i for i in idx if 0 <= i < C)


def pad(p):
    P = 8
    while P < p:
        P *= 2
    return P


def eval_launches(prob):
    return prob.info()["eval_launches"]


def eval_tc(prob, B):
    """eval_many that must have gone through the tensor-core kernel (one evaluation launch)."""
    e0 = eval_launches(prob)
    res = prob.eval_many(B)
    assert eval_launches(prob) - e0 == 1, "expected the tensor-core path"
    return res


def eval_simt(prob, N, B):
    """The same evaluation forced onto the SIMT many-chain kernel (ceil(C/4) launches)."""
    prob.set_option(N.OPT_TC_MIN_CHAINS, 1 << 30)
    try:
        e0 = eval_launches(prob)
        res = prob.eval_many(B)
        assert eval_launches(prob) - e0 == -(-len(B) // 4)
        return res
    finally:
        prob.set_option(N.OPT_TC_MIN_CHAINS, TC_MIN_CHAINS)


def assert_close_to_simt(tc, simt, B, ps, colsum, tol=1e-6):
    """Every chain: tensor-core result within tol of the SIMT FP32 result (lpost / ll relative to
    max(1, |.|); glp against max_j sum_i |x_ij| + |beta_j / pscale_j^2|, a bound of the un-cancelled
    magnitude). On these rows both kernels are ~1e-8 from float64, so tol = 1e-6 has a wide margin."""
    for k in (0, 1):
        d = np.abs(tc[k] - simt[k]) / np.maximum(1.0, np.abs(simt[k]))
        assert np.max(d) <= tol, (k, int(np.argmax(d)), float(np.max(d)))
    scale = np.max(colsum) + np.max(np.abs(B / ps ** 2), axis=1)
    d = np.max(np.abs(tc[2] - simt[2]), axis=1) / scale
    assert np.max(d) <= tol, ("glp", int(np.argmax(d)), float(np.max(d)))


def assert_same_bits(a, b, what=""):
    for u, v in zip(a, b):
        np.testing.assert_array_equal(u, v, err_msg=what)


# ---------------------------------------------------------------- 1. SIMT eval_mc_kernel
WIDTHS = [1, 8, 13, 16, 32, 33, 64, 100, 128, 200, 256]


@pytest.mark.parametrize("mode", ["fp64", "fp32"])
@pytest.mark.parametrize("p", WIDTHS)
def test_simt_many_chain_kernel_at_every_width(lr, sms, mode, p):
    """Row counts 1, RB - 1, RB, RB + 1 and one past the largest possible grid (every warp loops);
    C = 2..11 (one pass, partial last pass, full passes) and C = 13 wherever it stays SIMT."""
    P = pad(p)
    RB = 8192 // (P * (4 if mode == "fp32" else 8))
    n_big = RB * (sms * 64 + 3) + 5          # > RB * (SMs * 8 CTAs * 8 warps): more batches than warps
    rs = np.random.RandomState(7000 + p + (0 if mode == "fp64" else 500))
    Xall = rows(rs, n_big, p)
    bt = rs.randn(p) / np.sqrt(p)
    yall = (rs.rand(n_big) < expit(Xall @ bt)).astype(np.float32)
    ps = 0.5 + 3 * rs.rand(p)
    counts = [2, 3, 4, 5, 8, 11] + ([13] if (mode == "fp64" or P != 64) else [])
    B = bt + 0.3 * rs.randn(max(counts), p) / np.sqrt(p)
    B[1] = 0.0
    prob = lr.Problem()
    worst = {}
    for n in sorted({1, RB - 1, RB, RB + 1, n_big} - {0}):
        X, y = Xall[:n], yall[:n]
        prob.bind_data(X, y, ps, mode=mode)
        single = [prob.eval(b) for b in B]
        ll_r, gl_r, mag = ref_like(X, y, B)
        gscale = np.max(mag + np.abs(B / ps ** 2), axis=1)
        for C in counts:
            res = prob.eval_many(B[:C])
            e = errors(X, y, ps, B, res, range(C))
            assert_errors(e, TOL[mode], (n, C))
            for k, v in e.items():
                worst[k] = max(worst.get(k, 0.0), v)
            for c in range(C):
                lp1, l1, g1 = single[c]
                assert abs(res[0][c] - lp1) <= 1e-12 * max(1.0, abs(lp1)), (n, C, c)
                assert abs(res[1][c] - l1) <= 1e-12 * max(1.0, abs(l1)), (n, C, c)
                assert np.max(np.abs(res[2][c] - g1)) <= 1e-12 * gscale[c], (n, C, c)
    prob.close()
    print(f"simt mc p={p} {mode}: " + ", ".join(f"{k} {v:.1e}" for k, v in worst.items()))


# ---------------------------------------------------------------- 4. static eval_kernel
@pytest.mark.parametrize("mode", ["fp64", "fp32"])
@pytest.mark.parametrize("p", [1, 3, 8, 13, 32, 64, 100, 128, 200, 256])
def test_static_kernel_at_every_width(lr, mode, p):
    """The fixed-order static kernel (deterministic=True, also the row-sharded path) on the grid of
    test_gpu_eval.py::test_shapes_against_oracle, which runs the default (drive-mode) handles."""
    rs = np.random.RandomState(1000 + p)
    for n in (1, 7, 200, 1031, 4099, 20011):
        X = rows(rs, n, p)
        beta = rs.randn(p) / np.sqrt(p)
        y = (rs.rand(n) < expit(X @ beta)).astype(np.float32)
        ps = 0.5 + rs.rand(p) * 3
        prob = lr.Problem(deterministic=True).bind_data(X, y, ps, mode=mode)
        for b in (beta, np.zeros(p), beta + 0.3 * rs.randn(p)):
            lp, l, g = prob.eval(b)
            e = errors(X, y, ps, b[None, :], (np.array([lp]), np.array([l]), g[None, :]), [0])
            assert_errors(e, TOL[mode], (n, p))
            assert prob.eval(b.copy() + 0.0)[0] == lp
        again = lr.Problem(deterministic=True).bind_data(X, y, ps, mode=mode)
        assert_same_bits(again.eval(beta), prob.eval(beta), "static kernel is not bit-reproducible")
        prob.close()
        again.close()


# ---------------------------------------------------------------- 2. eval_tc_kernel
@pytest.mark.parametrize("p", [33, 40, 63, 64])
def test_tensor_core_padded_widths(lr, N, p):
    """p = 33..63 leaves zero-padded columns of beta and G in tensor memory."""
    rs = np.random.RandomState(300 + p)
    n, C = 40_009, 130
    X = rows(rs, n, p)
    bt = rs.randn(p) / np.sqrt(p)
    y = (rs.rand(n) < expit(X @ bt)).astype(np.float32)
    ps = 0.5 + 3 * rs.rand(p)
    B = bt + 0.3 * rs.randn(C, p) / np.sqrt(p)
    prob = lr.Problem().bind_data(X, y, ps, mode="fp32")
    tc = eval_tc(prob, B)
    assert_close_to_simt(tc, eval_simt(prob, N, B), B, ps, np.abs(X).sum(0))
    e = errors(X, y, ps, B, tc, sample(C, rs))
    assert_errors(e, TOL["fp32"], p)
    print(f"tc p={p}: " + ", ".join(f"{k} {v:.1e}" for k, v in e.items()))


def test_tensor_core_width_40_equals_64_with_zero_columns(lr):
    rs = np.random.RandomState(40)
    n, C, p = 20_011, 140, 40
    X = rows(rs, n, p)
    bt = rs.randn(p) / np.sqrt(p)
    y = (rs.rand(n) < expit(X @ bt)).astype(np.float32)
    B = bt + 0.3 * rs.randn(C, p) / np.sqrt(p)
    ps = 0.5 + 3 * rs.rand(p)
    a = lr.Problem().bind_data(X, y, ps, mode="fp32")
    b = lr.Problem().bind_data(np.hstack([X, np.zeros((n, 24))]), y, np.concatenate([ps, np.ones(24)]), mode="fp32")
    ra = eval_tc(a, B)
    rb = eval_tc(b, np.hstack([B, np.zeros((C, 24))]))
    np.testing.assert_array_equal(ra[1], rb[1])
    np.testing.assert_array_equal(ra[2], rb[2][:, :40])
    np.testing.assert_array_equal(rb[2][:, 40:], 0.0)


K_SWEEP = list(range(1, 21)) + [31, 32, 33, 47, 48, 49, 64, 65]


@pytest.fixture(scope="module")
def sweep_rows(lr, sms):
    """Rows of the largest sweep case, read back once: gen_synthetic is prefix-stable."""
    n_max = 64 * (sms * (max(K_SWEEP) - 1) + 1)
    prob = lr.Problem()
    bt = prob.gen_synthetic(n_max, 64, mode="fp32", seed=42)
    X, y = prob.copy_rows(0, n_max)
    prob.close()
    return bt, X, y, np.cumsum(np.abs(X), axis=0)


@pytest.mark.parametrize("groups,C", [(1, 128), (3, 300)])
def test_tensor_core_tile_count_sweep(lr, N, sms, sweep_rows, groups, C):
    """CTA bx streams ceil((ntiles - bx) / gx) tiles, gx = min(SMs // groups, ntiles). With
    ntiles = gx (k - 1) + 1, CTA 0 gets k tiles and the others k - 1: k sweeps the 3-stage X ring
    and the double-buffered 16-tile gradient flush through all their phases; r trims a ragged tail."""
    bt, Xall, yall, cum = sweep_rows
    rs = np.random.RandomState(groups)
    B = bt + 0.3 * rs.randn(C, 64) / 8
    prob = lr.Problem()
    gx = sms // groups
    for k in K_SWEEP:
        ntiles = gx * (k - 1) + 1
        for r in (0, 1, 63):
            n = 64 * ntiles - r
            prob.gen_synthetic(n, 64, mode="fp32", seed=42, beta_true=bt)
            X, y = Xall[:n], yall[:n]
            tc = eval_tc(prob, B)
            assert_close_to_simt(tc, eval_simt(prob, N, B), B, prob.pscale, cum[n - 1])
            e = errors(X, y, prob.pscale, B, tc, sample(C, rs, extra=1))
            assert_errors(e, TOL["fp32"], (k, r))
    prob.close()


def test_tensor_core_chain_count_edges(lr, N, sms):
    rs = np.random.RandomState(11)
    n = 64 * 300 + 37
    prob = lr.Problem()
    bt = prob.gen_synthetic(n, 64, mode="fp32", seed=7)
    X, y = prob.copy_rows(0, n)
    colsum = np.abs(X).sum(0)
    for C in (11, 12, 127, 128, 129, 255, 256, 257):
        B = bt + 0.3 * rs.randn(C, 64) / 8
        res = eval_tc(prob, B) if C >= TC_MIN_CHAINS else prob.eval_many(B)
        assert_close_to_simt(res, eval_simt(prob, N, B), B, prob.pscale, colsum)
        assert_errors(errors(X, y, prob.pscale, B, res, sample(C, rs)), TOL["fp32"], C)
    # C = 128 * SMs: one CTA per chain group, each streaming every tile; one more chain and the
    # groups no longer fit the SMs: the SIMT kernel takes over
    n = 200
    prob.gen_synthetic(n, 64, mode="fp32", seed=7, beta_true=bt)
    X, y = prob.copy_rows(0, n)
    C = 128 * sms
    B = bt + 0.3 * rs.randn(C + 1, 64) / 8
    tc = eval_tc(prob, B[:C])
    assert_close_to_simt(tc, eval_simt(prob, N, B[:C]), B[:C], prob.pscale, np.abs(X).sum(0))
    assert_errors(errors(X, y, prob.pscale, B, tc, sample(C, rs)), TOL["fp32"], C)
    e0 = eval_launches(prob)
    fall = prob.eval_many(B)
    assert eval_launches(prob) - e0 == -(-(C + 1) // 4)
    assert_same_bits(fall, eval_simt(prob, N, B), "SIMT fall-back differs from forced SIMT")
    assert_errors(errors(X, y, prob.pscale, B, fall, sample(C + 1, rs)), TOL["fp32"], C + 1)
    prob.close()


def test_tensor_core_chains_are_independent_bit_for_bit(lr):
    """A chain's result depends on its own coefficients only: not on the other chains' values, not
    on its position (TMEM lane, chain group, beta stride) at a fixed group count, not on the call."""
    rs = np.random.RandomState(12)
    prob = lr.Problem()
    bt = prob.gen_synthetic(64 * 500 + 19, 64, mode="fp32", seed=3)
    C = 300
    B = bt + 0.3 * rs.randn(C, 64) / 8
    ref = eval_tc(prob, B)
    assert_same_bits(eval_tc(prob, B), ref, "repeated call")
    keep = [0, 1, 31, 32, 127, 128, 129, 255, 256, 299]
    B2 = B + 0.5 * rs.randn(C, 64) / 8
    B2[keep] = B[keep]
    other = eval_tc(prob, B2)
    for k in range(3):
        np.testing.assert_array_equal(other[k][keep], ref[k][keep])
    perm = rs.permutation(C)
    moved = eval_tc(prob, B[perm])
    for k in range(3):
        np.testing.assert_array_equal(moved[k], ref[k][perm])
    prob.close()


# ---------------------------------------------------------------- 2. data regimes
def regime_case(lr, N, X, y, B, ps, what, like_tol=True):
    """Tensor-core vs SIMT (both FP32 storage) vs float64 on the same handle. Returns the errors.
    The tensor-core error is bounded by 4x the SIMT kernel's on the same rows (plus a float32-level
    floor) and, where like_tol, by the FP32-mode tolerance for the likelihood part too."""
    prob = lr.Problem().bind_data(X, y, ps, mode="fp32")
    tc = eval_tc(prob, B)
    simt = eval_simt(prob, N, B)
    prob.close()
    for r in (tc, simt):
        assert np.all(np.isfinite(r[0])) and np.all(np.isfinite(r[1])) and np.all(np.isfinite(r[2])), what
    rows_tc = [errors(X, y, ps, B, tc, [c]) for c in range(len(B))]
    rows_simt = [errors(X, y, ps, B, simt, [c]) for c in range(len(B))]
    for k in rows_tc[0]:
        print(f"{what} {k}: tc {max(e[k] for e in rows_tc):.1e} simt {max(e[k] for e in rows_simt):.1e}")
    for c in range(len(B)):
        et, es = rows_tc[c], rows_simt[c]
        for k in ("lpost", "ll", "glp"):
            assert et[k] <= TOL["fp32"], (what, c, k, et)
        keys = ("ll_like", "g_like") if like_tol else ()
        for k in keys:
            assert et[k] <= TOL["fp32"], (what, c, k, et)
        for k in et:
            assert et[k] <= 4 * es[k] + TC_ETA_FLOOR, (what, c, k, et[k], es[k])
    return rows_tc, rows_simt


def separable_data(rs, n, p, margin=0.05, flip=0.0):
    X = rows(rs, n + n // 2, p)
    bstar = rs.randn(p) / np.sqrt(p)
    eta = X @ bstar
    X, eta = X[np.abs(eta) >= margin][:n], eta[np.abs(eta) >= margin][:n]
    y = (eta > 0).astype(np.float32)
    if flip:
        bad = rs.rand(n) < flip
        y[bad] = 1.0 - y[bad]
    return X, y, bstar


@pytest.mark.parametrize("flip", [
    pytest.param(0.0, marks=pytest.mark.xfail(strict=True, reason=(
        "tc_link_chunk: lg2.approx(1 + e) and y - (1 - inv) lose the relative accuracy of the tiny "
        "terms of separable data (DESIGN.md 3.3); the measured repairs cost 6-9 % of c4 throughput"))),
    1e-3])
def test_tensor_core_separable_data(lr, N, flip):
    """y = [x.beta* > 0] (|x.beta*| >= 0.05), optionally with 0.1 % of the labels flipped, at
    c * beta*: for large c the likelihood is a sum of tiny exp(-|eta|) terms (|eta| >= 20 at
    c = 400, where 1 + exp(-|eta|) rounds to 1 in float32) and glp is dominated by the prior."""
    rs = np.random.RandomState(20 + int(flip * 1e4))
    n, p = 100_000, 64
    X, y, bstar = separable_data(rs, n, p, flip=flip)
    cs = np.array([1, 5, 20, 100, 400, 1, 5, 20, 100, 400, 1, 5, 20, 100, 400, 2], dtype=np.float64)
    B = cs[:, None] * bstar * (1 + 1e-3 * rs.randn(len(cs), p) * (np.arange(len(cs)) >= 5)[:, None])
    tc, simt = regime_case(lr, N, X, y, B, np.full(p, 1000.0), f"separable flip={flip}",
                           like_tol=False)
    for c in range(5):
        e, s = tc[c], simt[c]
        print(f"separable flip={flip} c={cs[c]:g}: ll rel tc {e['ll_like']:.1e} simt {s['ll_like']:.1e}; "
              f"X'(y-p) err / |X|'|y-p| tc {e['g_like']:.1e} simt {s['g_like']:.1e}")
    # the likelihood part itself to the FP32-mode tolerance wherever eta's float32 rounding allows it
    for c in range(len(cs)):
        if cs[c] <= 20:
            assert tc[c]["ll_like"] <= TOL["fp32"] and tc[c]["g_like"] <= TOL["fp32"], (cs[c], tc[c])


def test_tensor_core_extreme_eta_with_mislabelled_rows(lr, N):
    """|eta| from 100 to ~1e4 (beyond 88, where exp(-|eta|) flushes to zero in float32) with 10 % of
    the labels wrong: every value finite and ll = -sum |eta| over the mislabelled rows."""
    rs = np.random.RandomState(30)
    n, p = 50_000, 64
    X, y, bstar = separable_data(rs, n, p, margin=0.05, flip=0.1)
    cs = np.linspace(2000.0, 2600.0, 16)
    B = cs[:, None] * bstar
    eta = X @ B.T
    assert np.min(np.abs(eta)) > 88 and np.max(np.abs(eta)) < 2e4
    tc, simt = regime_case(lr, N, X, y, B, np.full(p, 1e4), "extreme eta")
    prob = lr.Problem().bind_data(X, y, np.full(p, 1e4), mode="fp32")
    _, l, _ = eval_tc(prob, B)
    prob.close()
    wrong = (eta > 0) != (y[:, None] > 0)
    want = -np.sum(np.abs(eta) * wrong, axis=0)
    np.testing.assert_allclose(l, want, rtol=TOL["fp32"])


@pytest.mark.parametrize("label", [0.0, 1.0])
def test_tensor_core_one_class(lr, N, label):
    rs = np.random.RandomState(40 + int(label))
    n, p = 30_011, 64
    X = rows(rs, n, p)
    B = rs.randn(16, p) / np.sqrt(p) * np.linspace(0.1, 4, 16)[:, None]
    regime_case(lr, N, X, np.full(n, label, dtype=np.float32), B, np.ones(p), f"y all {label:g}")


def test_tensor_core_mixed_column_magnitudes(lr, N):
    """Columns scaled by 1e-3 .. 1e3 with coefficients scaled inversely (eta stays O(1))."""
    rs = np.random.RandomState(50)
    n, p = 50_021, 64
    sc = 10.0 ** rs.uniform(-3, 3, p)
    sc[0] = 1.0
    X = (rows(rs, n, p) * sc).astype(np.float32).astype(np.float64)
    bt = rs.randn(p) / np.sqrt(p) / sc
    y = (rs.rand(n) < expit(X @ bt)).astype(np.float32)
    B = bt * (1 + 0.3 * rs.randn(16, p))
    regime_case(lr, N, X, y, B, 1e3 / sc, "mixed magnitudes")


# ---------------------------------------------------------------- 3. lock-step samplers
SAMPLER_ITERS = {"rwmh": 70, "ul": 70, "mala": 70, "hmc": 12}   # HMC: 12 x 7 + 1 evaluations > one 64-node graph


@pytest.fixture(scope="module")
def sampler_problem(lr):
    n = 50_000
    prob = lr.Problem()
    bt = prob.gen_synthetic(n, 64, mode="fp32", seed=42)
    X, y = prob.copy_rows(0, n)
    return prob, bt, O.Target(X, y, prob.pscale), 2.2 / np.sqrt(n)


def tuning(sd):
    return dict(rw=0.3 * sd, dt=(0.5 * sd) ** 2, eps=0.25 * sd, l=7)


def device_kernel(lr, prob, kind, sd):
    t = tuning(sd)
    if kind == "rwmh":
        return lr.mhKernel(prob.lpost, lr.RandomWalk(np.full(prob.p, t["rw"])))
    if kind == "ul":
        return lr.ulKernel(prob.glp, dt=t["dt"])
    if kind == "mala":
        return lr.malaKernel(prob.lpost, prob.glp, dt=t["dt"])
    return lr.hmcKernel(prob.lpost, prob.glp, eps=t["eps"], l=t["l"], dmm=1.0)


def oracle_step(kind, tgt, sd, x, z, u, first=False):
    """One step of the reference kernel over the float64 density with draws z, u.
    Returns (next state, |log alpha - log u| or None for UL). RWMH and MALA thread the
    log-density, which a new chain starts at -inf (the first proposal is accepted)."""
    t, trace = tuning(sd), []
    ll = -np.inf if first else tgt.lpost(x)
    rng = O.ReplayRNG(z[None, :], None if u is None else np.array([u]))
    if kind == "rwmh":
        k = O.mh_kernel(tgt.lpost, O.rw_proposal(np.full(tgt.p, t["rw"]), rng), rng=rng, trace=trace)
        x_new = k(x, ll)[0]
    elif kind == "ul":
        return O.ul_kernel(tgt.glp, tgt.p, dt=t["dt"], rng=rng)(x), None
    elif kind == "mala":
        k = O.mala_kernel(tgt.lpost, tgt.glp, tgt.p, dt=t["dt"], rng=rng, trace=trace)
        x_new = k(x, ll)[0]
    else:
        x_new = O.hmc_kernel(tgt.lpost, tgt.glp, eps=t["eps"], l=t["l"], dmm=1.0, rng=rng, trace=trace)(x)
    return x_new, abs(trace[-1][0] - trace[-1][1])


def continue_chains(prob, N, k, C, iters, seed):
    """lrb_run with init = NULL: continue the paused C-chain run."""
    sp = prob._params(k, seed, N.RNG_PHILOX, -np.inf)
    out = np.empty((C, iters, prob.p))
    acc = np.zeros(C, dtype=np.int64)
    prob._ck(prob._lib.lrb_run(prob._h, ctypes.byref(sp), None, C, 1, iters, None, None, N.as_dp(out),
                               acc.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))))
    return out, acc


def chain_key(seed, c):
    return (seed + c * 0x9E3779B97F4A7C15) % 2 ** 64


@pytest.mark.parametrize("C", [16, 300])
@pytest.mark.parametrize("kind", ["rwmh", "ul", "mala", "hmc"])
def test_tensor_core_lockstep_philox_matches_simt(lr, N, sampler_problem, kind, C):
    """Same Philox keys on the tensor-core and the forced-SIMT path, each run as a first part plus
    a continuation: the decisions agree and the states agree to float32 level until the first
    decision that the float64 oracle shows to be a near-tie (|log alpha - log u| < 5e-3). On the
    tensor-core path the split run equals one uninterrupted run bit for bit."""
    prob, bt, tgt, sd = sampler_problem
    k = device_kernel(lr, prob, kind, sd)
    iters, seed = SAMPLER_ITERS[kind], 1234
    m = iters // 3
    inits = bt + 0.5 * sd * np.random.RandomState(C).randn(C, 64)
    full, acc_full = prob.run_chains(k, inits, 1, iters, seed=seed)
    a, _ = prob.run_chains(k, inits, 1, m, seed=seed)
    b, acc_b = continue_chains(prob, N, k, C, iters - m, seed)
    tc = np.concatenate([a, b], axis=1)
    np.testing.assert_array_equal(tc, full)
    np.testing.assert_array_equal(acc_b, acc_full)
    prob.set_option(N.OPT_TC_MIN_CHAINS, 1 << 30)
    try:
        e0 = eval_launches(prob)
        a, _ = prob.run_chains(k, inits, 1, m, seed=seed)
        b, _ = continue_chains(prob, N, k, C, iters - m, seed)
        assert eval_launches(prob) - e0 >= -(-C // 4) * iters
    finally:
        prob.set_option(N.OPT_TC_MIN_CHAINS, TC_MIN_CHAINS)
    simt = np.concatenate([a, b], axis=1)
    if kind != "ul":
        assert 0.05 < acc_full.mean() / iters < 1.0, acc_full.mean() / iters
    ties = 0
    for c in range(C):
        same = np.all(np.abs(tc[c] - simt[c]) <= 5e-3 * sd, axis=1)
        if same.all():
            continue
        i = int(np.argmin(same))
        assert kind != "ul", (c, i)
        x = inits[c] if i == 0 else tc[c, i - 1]
        Z, U = prob.rng_dump(chain_key(seed, c), i, 1)
        _, margin = oracle_step(kind, tgt, sd, x, Z[0], U[0], first=i == 0)
        assert margin < 5e-3, (c, i, margin)
        ties += 1
    assert ties <= max(1, C // 20), ties


@pytest.mark.parametrize("kind", ["rwmh", "ul", "mala", "hmc"])
def test_tensor_core_lockstep_replay_matches_oracle(lr, sampler_problem, kind):
    """Replayed per-chain draws on the tensor-core path: from every device state x_t of a subset of
    chains, the reference kernel over the float64 density with the same draws gives the device's
    x_{t+1}; a decision may differ only on a near-tie of the accept test."""
    prob, bt, tgt, sd = sampler_problem
    k = device_kernel(lr, prob, kind, sd)
    C, iters = 16, SAMPLER_ITERS[kind]
    rs = np.random.RandomState(99)
    inits = bt + 0.5 * sd * rs.randn(C, 64)
    Z = rs.randn(C, iters, 64)
    U = rs.rand(C, iters)
    e0 = eval_launches(prob)
    mats, accs = prob.run_chains(k, inits, 1, iters, Z=Z, U=None if kind == "ul" else U)
    assert eval_launches(prob) - e0 == iters * (tuning(sd)["l"] if kind == "hmc" else 1) + (kind in ("mala", "hmc"))
    compared = 0
    for c in (0, 5, 15):
        x = inits[c]
        for i in range(iters):
            x_ref, margin = oracle_step(kind, tgt, sd, x, Z[c, i], U[c, i], first=i == 0)
            acc_dev = bool(np.any(mats[c, i] != x))
            acc_ref = bool(np.any(x_ref != x))
            if margin is not None and acc_dev != acc_ref:
                assert margin < 5e-3, (c, i, margin)
            else:
                assert np.max(np.abs(mats[c, i] - x_ref)) <= 1e-2 * sd, (c, i, np.max(np.abs(mats[c, i] - x_ref)) / sd)
                compared += 1
            x = mats[c, i]
    assert compared >= 3 * iters - 3


def test_tensor_core_hmc_moments(lr, sampler_problem):
    """Device running moments of an HMC run on the tensor-core path equal NumPy's on the returned
    samples, per chain and pooled."""
    prob, bt, tgt, sd = sampler_problem
    k = device_kernel(lr, prob, "hmc", sd)
    C = 24
    inits = bt + 0.5 * sd * np.random.RandomState(5).randn(C, 64)
    e0 = eval_launches(prob)
    mats, _ = prob.run_chains(k, inits, 2, 6, seed=77, moments=True)
    assert eval_launches(prob) - e0 == 2 * 6 * 7 + 1   # one launch per evaluation: the tensor-core path
    cnt, mean, cov = prob.moments()
    np.testing.assert_array_equal(cnt, 6)
    for c in range(C):
        np.testing.assert_allclose(mean[c], mats[c].mean(0), rtol=1e-12, atol=1e-12 * sd)
        np.testing.assert_allclose(cov[c], np.cov(mats[c].T), rtol=1e-6, atol=1e-9 * sd ** 2)
    n_all, m_all, c_all = prob.moments(pooled=True)
    flat = mats.reshape(-1, 64)
    assert n_all == C * 6
    np.testing.assert_allclose(m_all, flat.mean(0), rtol=1e-12, atol=1e-12 * sd)
    np.testing.assert_allclose(c_all, np.cov(flat.T), rtol=1e-6, atol=1e-9 * sd ** 2)
