"""Pin the CPU oracle (oracle/logreg_oracle.py) to the reference.

Two anchors: (1) the committed golden fixtures, which are outputs of the
reference's own functions (tests/golden/make_golden.py); (2) when
LOGREG_REFERENCE names a checkout of the reference project, the live
AST-lifted reference functions.
"""
import os

import numpy as np
import pytest

from oracle import logreg_oracle as O

REFERENCE = os.environ.get("LOGREG_REFERENCE", "")

CHAINS_THREADED = {
    # tag: (kind, kwargs)
    "rwmh_t1": "rwmh", "rwmh_t50": "rwmh",
    "mala_t1": "mala", "mala_t25": "mala", "mala_scalar_t1": "mala_scalar",
}
CHAINS_PLAIN = {
    "ul_t1": "ul", "ul_t40": "ul",
    "hmc_t1": "hmc", "hmc_t5": "hmc", "hmc_l7_t1": "hmc_l7",
}


def _target(g):
    # the reference builds X column-major (pandas to_numpy + hstack, SURVEY.md A8);
    # using the same layout keeps OpenBLAS on the same dgemv path => identical bits
    return O.Target(np.asfortranarray(g["X"]), g["y"], g["pscale"])


def test_known_answers_appendix_b(pima):
    """SURVEY.md appendix B values, recomputed by the oracle."""
    t = _target(pima)
    z = np.zeros(8)
    assert t.ll(z) == pytest.approx(-200 * np.log(2), rel=1e-14)
    assert t.lprior(z) == pytest.approx(-9.654093358631428, rel=1e-14)
    assert t.lpost(z) == pytest.approx(-148.28352947062046, rel=1e-14)
    np.testing.assert_allclose(
        t.glp(z), [-32.0, -28.0, -2533.0, -2054.0, -669.5, -870.8, -8.7675, -648.0], rtol=1e-12)
    b0 = np.array([-9.8, 0.1, 0.03, -0.005, 0.0, 0.08, 1.8, 0.04])
    assert t.lpost(b0) == pytest.approx(-103.86338162923353, rel=1e-13)


def test_point_values_match_reference_outputs(pima):
    t = _target(pima)
    for i, b in enumerate(pima["B"]):
        assert t.ll(b) == pytest.approx(pima["ll"][i], rel=1e-13)
        assert t.lprior(b) == pytest.approx(pima["lprior"][i], rel=1e-13)
        assert t.lprior(b) == pytest.approx(pima["lprior_fitnumpy"][i], rel=1e-13)
        assert t.lpost(b) == pytest.approx(pima["lpost"][i], rel=1e-13)
        np.testing.assert_allclose(t.glp(b), pima["glp"][i], rtol=1e-11, atol=1e-9)


def test_synthetic_point_values(synth):
    X = synth["X32"].astype(np.float64)
    t = O.Target(X, synth["y"], synth["pscale"])
    for i, b in enumerate(synth["B"]):
        assert t.lpost(b) == pytest.approx(synth["lpost"][i], rel=1e-13)
        np.testing.assert_allclose(t.glp(b), synth["glp"][i], rtol=1e-10, atol=1e-9)
        lp, g = t.lpost_glp_chunked(b, chunk=300)
        assert lp == pytest.approx(synth["lpost"][i], rel=1e-12)
        np.testing.assert_allclose(g, synth["glp"][i], rtol=1e-9, atol=1e-9)
        assert O.stable_ll(X, synth["y"], b) == pytest.approx(synth["ll"][i], rel=1e-12)


def test_mala_closed_form_log_alpha(pima):
    t = _target(pima)
    b0 = pima["B"][1]
    a = O.mala_log_alpha(t, b0, pima["mala_prop"], 1e-5, pima["pre"])
    assert a == pytest.approx(float(pima["mala_log_alpha"]), rel=1e-9)
    assert float(pima["mala_log_alpha"]) == pytest.approx(-29.492981396187382, rel=1e-9)


def _run_oracle_chain(pima, tag, kind):
    t = _target(pima)
    seed, thin, iters = (int(v) for v in pima[tag + "_cfg"])
    U = pima[tag + "_U"]
    rng = O.ReplayRNG(pima[tag + "_Z"], U if U.size else None)
    init = pima["chain_init"]
    pre = pima["pre"]
    if kind == "rwmh":
        k = O.mh_kernel(t.lpost, O.rw_proposal(0.02 * pima["pre_rw"], rng), rng=rng)
        return O.mcmc_threaded(init, k, thin, iters)
    if kind == "mala":
        return O.mcmc_threaded(init, O.mala_kernel(t.lpost, t.glp, 8, dt=1e-5, pre=pre, rng=rng), thin, iters)
    if kind == "mala_scalar":
        return O.mcmc_threaded(init, O.mala_kernel(t.lpost, t.glp, 8, dt=1e-6, rng=rng), thin, iters)
    if kind == "ul":
        return O.mcmc_plain(init, O.ul_kernel(t.glp, 8, dt=1e-6, pre=pre, rng=rng), thin, iters)
    if kind == "hmc":
        return O.mcmc_plain(init, O.hmc_kernel(t.lpost, t.glp, eps=1e-3, l=50, dmm=1 / pre, rng=rng), thin, iters)
    if kind == "hmc_l7":
        return O.mcmc_plain(init, O.hmc_kernel(t.lpost, t.glp, eps=2e-3, l=7, dmm=1 / pre, rng=rng), thin, iters)
    raise AssertionError(kind)


@pytest.mark.parametrize("tag,kind", list(CHAINS_THREADED.items()) + list(CHAINS_PLAIN.items()))
def test_replayed_chains_bit_identical_to_reference(pima, tag, kind):
    """The reference's chain under np.random.seed(s) == the oracle's chain fed
    the pre-drawn (Z, U) stream: proves both the arithmetic and the RNG
    consumption order (SURVEY.md 8a15)."""
    mat = _run_oracle_chain(pima, tag, kind)
    ref = pima[tag + "_mat"]
    assert mat.shape == ref.shape
    # same arithmetic, same BLAS path => the difference is exactly 0 in the build
    # container; 1e-9 leaves room for a different BLAS build on another host
    np.testing.assert_allclose(mat, ref, rtol=1e-9, atol=1e-9)


def test_first_proposal_always_accepted(pima):
    """ll starts at -inf (fit-numpy.py:66) so step 1 always moves."""
    t = _target(pima)
    # a move to a far worse point, with u ~ 1: still accepted on step 1, rejected on step 2
    rng = O.ReplayRNG(np.ones((2, 8)), np.array([1.0 - 1e-16, 1.0 - 1e-16]))
    k = O.mh_kernel(t.lpost, O.rw_proposal(np.ones(8), rng), rng=rng)
    out = O.mcmc_threaded(np.zeros(8), k, 1, 2)
    np.testing.assert_array_equal(out[0], np.ones(8))
    np.testing.assert_array_equal(out[1], np.ones(8))
    # and lp = -inf (naive overflow) on step 1 gives a = nan => rejected (SURVEY.md 7, hard part 8)
    rng = O.ReplayRNG(np.ones((1, 8)) * 50.0, np.array([0.5]))
    k = O.mh_kernel(t.lpost, O.rw_proposal(np.ones(8), rng), rng=rng)
    with np.errstate(over="ignore", invalid="ignore"):
        out = O.mcmc_threaded(np.zeros(8), k, 1, 1)
    np.testing.assert_array_equal(out[0], np.zeros(8))


def test_naive_ll_overflows_like_reference(pima):
    t = _target(pima)
    with np.errstate(over="ignore"):
        assert t.ll(50 * np.ones(8)) == -np.inf
    with np.errstate(over="ignore"):
        assert np.all(np.isfinite(t.glp(50 * np.ones(8))))
    assert np.isfinite(O.stable_ll(pima["X"], pima["y"], 50 * np.ones(8)))


@pytest.mark.skipif(not (REFERENCE and os.path.isdir(os.path.join(REFERENCE, "Python"))),
                    reason="set LOGREG_REFERENCE to a checkout of the reference project (Python/, pima.parquet)")
def test_against_live_reference(pima):
    """What this adds to the fixtures: fit-np-hmc.py's own lpost / glp at 20 seeded points near the MAP,
    the load of the real pima.parquet, and a fresh HMC chain (seed 99, l=10, thin 2).  The reference
    project is not part of this repository and its outputs for these checks are not stored, so the
    test runs only where LOGREG_REFERENCE names a checkout of it."""
    import importlib.util
    spec = importlib.util.spec_from_file_location(
        "make_golden", os.path.join(os.path.dirname(__file__), "golden", "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    X, y, n, p = mg.load_pima()
    np.testing.assert_array_equal(X, pima["X"])
    np.testing.assert_array_equal(y, pima["y"])
    ns = mg.namespace("fit-np-hmc.py", {"ll", "pscale", "lprior", "lpost", "glp", "mhKernel", "hmcKernel", "mcmc"},
                      X=X, y=y, n=n, p=p, init=np.zeros(p))
    t = O.Target(X, y, ns["pscale"])
    rs = np.random.RandomState(5)
    for _ in range(20):
        b = pima["map"] + rs.randn(8) * 0.05
        assert t.lpost(b) == pytest.approx(ns["lpost"](b), rel=1e-14)
        np.testing.assert_allclose(t.glp(b), ns["glp"](b), rtol=1e-12, atol=1e-10)
    # a fresh chain, not in the fixtures
    np.random.seed(99)
    ref = ns["mcmc"](pima["map"], ns["hmcKernel"](ns["lpost"], ns["glp"], eps=1e-3, l=10, dmm=1 / pima["pre"]),
                     thin=2, iters=15, verb=False)
    np.random.seed(99)
    Z, U = O.predraw(np.random, 30, 8)
    rng = O.ReplayRNG(Z, U)
    mine = O.mcmc_plain(pima["map"], O.hmc_kernel(t.lpost, t.glp, eps=1e-3, l=10, dmm=1 / pima["pre"], rng=rng), 2, 15)
    np.testing.assert_allclose(mine, ref, rtol=1e-12, atol=1e-12)


def test_oracle_gradient_is_the_derivative_of_lpost(pima, synth):
    """glp (fit-np-ul.py:45-48) is hand-coded in the reference; check it against central finite
    differences of lpost (fit-numpy.py:43-44) -- the check the reference does by eye
    (fit-np-ul.py:50-51,57)."""
    for X, y, ps, b in ((pima["X"], pima["y"], pima["pscale"], pima["B"][1]),
                        (synth["X32"].astype(np.float64), synth["y"], synth["pscale"], synth["B"][2])):
        t = O.Target(X, y, ps)
        g = t.glp(b)
        scale = np.abs(X).T.dot(np.ones(len(y))) + 1.0
        for j in range(len(b)):
            h = 1e-5 / np.sqrt(scale[j])
            e = np.zeros(len(b)); e[j] = h
            fd = (t.lpost(b + e) - t.lpost(b - e)) / (2 * h)
            assert abs(fd - g[j]) <= 1e-4 * scale[j] * 1e-2 + 1e-6 * abs(g[j]), (j, fd, g[j])


def test_oracle_row_additivity_hypothesis(synth):
    """ll and X'(y-p) are row sums (the property the row-sharded GPU path relies on)."""
    from hypothesis import given, settings, strategies as st
    X = synth["X32"].astype(np.float64)
    t = O.Target(X, synth["y"], synth["pscale"])
    b = synth["B"][1]
    full_ll, full_g = t.ll_gll_rows(b, 0, t.n)

    @settings(max_examples=25, deadline=None)
    @given(st.lists(st.integers(min_value=1, max_value=t.n - 1), min_size=1, max_size=6, unique=True))
    def check(cuts):
        edges = [0] + sorted(cuts) + [t.n]
        ll = 0.0
        g = np.zeros(t.p)
        for lo, hi in zip(edges, edges[1:]):
            a, c = t.ll_gll_rows(b, lo, hi)
            ll += a
            g += c
        assert ll == pytest.approx(full_ll, rel=1e-12)
        np.testing.assert_allclose(g, full_g, rtol=1e-9, atol=1e-9)

    check()


def test_pima_mala_tuning_is_chaotic_even_for_the_oracle(pima):
    """Why whole-chain parity for the reference's Pima MALA tuning (dt=1e-5, pre=[100,1,..,25,1],
    fit-np-mala.py:97-99) is stated on a prefix plus one-step-ahead: the map amplifies rounding.
    The oracle itself, fed the reference's own draws, reproduces the reference chain bit for bit
    with the reference's column-major X, but with the SAME numbers stored row-major (a different
    BLAS summation order in X.dot / X.T.dot, ~1e-16 relative) it leaves the reference trajectory
    after a few dozen steps.  A GPU kernel has yet another summation order, so the same happens."""
    Z, U, ref = pima["mala_t1_Z"], pima["mala_t1_U"], pima["mala_t1_mat"]
    out = {}
    for name, X in (("F", np.asfortranarray(pima["X"])), ("C", np.ascontiguousarray(pima["X"]))):
        tgt = O.Target(X, pima["y"], pima["pscale"])
        rng = O.ReplayRNG(Z, U)
        k = O.mala_kernel(tgt.lpost, tgt.glp, 8, dt=1e-5, pre=pima["pre"], rng=rng)
        out[name] = O.mcmc_threaded(pima["chain_init"], k, 1, len(ref))
    np.testing.assert_array_equal(out["F"], ref)                       # same layout: identical
    d = np.max(np.abs(out["C"] - ref), axis=1)
    assert d[:25].max() < 1e-9                                         # the prefix the GPU test compares
    assert d.max() > 1e-3                                              # ... and then it is a different chain
    first = int(np.argmax(d > 1e-6))
    assert 25 < first < len(ref)
    # both layouts evaluate the same function: one step from any reference state agrees to rounding
    tf = O.Target(np.asfortranarray(pima["X"]), pima["y"], pima["pscale"])
    tc = O.Target(np.ascontiguousarray(pima["X"]), pima["y"], pima["pscale"])
    for i in (0, first, len(ref) - 1):
        assert tc.lpost(ref[i]) == pytest.approx(tf.lpost(ref[i]), rel=1e-13)
        np.testing.assert_allclose(tc.glp(ref[i]), tf.glp(ref[i]), rtol=1e-9, atol=1e-9)
