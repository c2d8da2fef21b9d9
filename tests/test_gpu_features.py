"""Round-2 rows (SURVEY.md 8f and the checkpoint row of section 5): restartable Philox stream,
device-side running moments (f3), the keyed JAX-style front-end (f4), the one-argument mhKernel
of fit-np-hmc.py (a7), and the buffer-lifetime hazards found in review."""
import numpy as np
import pytest

from oracle import logreg_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lr():
    import logreg_b200
    assert logreg_b200.device_count() >= 1
    return logreg_b200


def kernels(lr, prob, pima):
    pre = pima["pre"]
    return {"rwmh": lr.mhKernel(prob.lpost, lr.RandomWalk(0.02 * pima["pre_rw"])),
            "ul": lr.ulKernel(prob.glp, dt=1e-6, pre=pre),
            "mala": lr.malaKernel(prob.lpost, prob.glp, dt=1e-5, pre=pre),
            "hmc": lr.hmcKernel(prob.lpost, prob.glp, eps=2e-3, l=7, dmm=1 / pre)}


@pytest.mark.parametrize("kind", ["rwmh", "ul", "mala", "hmc"])
def test_chain_resumes_in_a_new_handle_at_counter_t0(lr, pima, kind):
    """100 steps == 40 steps + (new handle, same seed, t0 = 40) 60 steps: the Philox counter is
    part of the checkpoint (lrb_chain_state -> LRB_RUN_SET_T0)."""
    X = np.asfortranarray(pima["X"])
    a = lr.Problem(deterministic=True).bind_data(X, pima["y"], pima["pscale"])
    full, acc_full = a.run(kernels(lr, a, pima)[kind], pima["chain_init"], 2, 50, seed=2024)
    b = lr.Problem(deterministic=True).bind_data(X, pima["y"], pima["pscale"])
    first, acc1 = b.run(kernels(lr, b, pima)[kind], pima["chain_init"], 2, 20, seed=2024)
    x, lp, t = b.chain_state()
    assert t == 40
    b.close()
    c = lr.Problem(deterministic=True).bind_data(X, pima["y"], pima["pscale"])     # "a new process"
    rest, acc2 = c.run(kernels(lr, c, pima)[kind], x, 2, 30, seed=2024, init_lpost=lp, t0=t)
    np.testing.assert_array_equal(np.vstack([first, rest]), full)
    assert acc1 + acc2 == acc_full
    assert c.chain_state()[2] == 100
    # without t0 the stream restarts at counter 0: a different chain
    d = lr.Problem(deterministic=True).bind_data(X, pima["y"], pima["pscale"])
    other, acc_o = d.run(kernels(lr, d, pima)[kind], x, 2, 30, seed=2024, init_lpost=lp)
    if acc2 > 0 or acc_o > 0:     # (the Pima MALA tuning can sit still for 60 steps)
        assert np.max(np.abs(other - rest)) > 0


@pytest.mark.parametrize("kind", ["rwmh", "hmc"])
def test_device_moments_equal_numpy_on_the_samples(lr, pima, kind):
    prob = lr.Problem().bind_data(np.asfortranarray(pima["X"]), pima["y"], pima["pscale"])
    k = kernels(lr, prob, pima)[kind]
    mat, _ = prob.run(k, pima["chain_init"], 3, 400, seed=5, moments=True)
    n, mean, cov = prob.moments()
    assert n == 400
    np.testing.assert_allclose(mean, mat.mean(axis=0), rtol=1e-12, atol=1e-13)
    ref_cov = np.cov(mat, rowvar=False)
    np.testing.assert_allclose(cov, ref_cov, rtol=1e-9, atol=1e-12 * np.abs(ref_cov).max())
    # a continued run keeps accumulating; keep_samples=False copies nothing back
    more, _ = prob.run(k, None, 3, 100, seed=5, moments=True)
    none, _ = prob.run(k, None, 3, 50, seed=5, moments=True, keep_samples=False)
    assert none is None
    n2, mean2, _ = prob.moments(cov=False)
    assert n2 == 550
    m3, _ = lr.Problem().bind_data(np.asfortranarray(pima["X"]), pima["y"], pima["pscale"]).run(
        k.__class__(prob, k.sampler, k.scale, k.step, k.l), pima["chain_init"], 3, 550, seed=5)
    np.testing.assert_allclose(mean2, m3.mean(axis=0), rtol=1e-9, atol=1e-12)
    # a new chain starts with empty moments
    prob.run(k, pima["chain_init"], 1, 7, seed=6, moments=True)
    assert prob.moments()[0] == 7


def test_device_moments_many_chains_pooled_and_per_chain(lr):
    """Config-4 shape in small: lock-step chains on the tensor-core path, nothing but moments
    leaves the device."""
    q = lr.Problem()
    bt = q.gen_synthetic(20_000, 64, mode="fp32", seed=8)
    C, iters = 40, 25
    sd = 2.2 / np.sqrt(20_000)
    inits = bt + 0.5 * sd * np.random.RandomState(0).randn(C, 64)
    k = lr.malaKernel(q.lpost, q.glp, dt=(0.6 * sd) ** 2, pre=1.0)
    mats, acc = q.run_chains(k, inits, 2, iters, seed=3, moments=True)
    cnt, mean, cov = q.moments()
    assert cnt.shape == (C,) and np.all(cnt == iters)
    np.testing.assert_allclose(mean, mats.mean(axis=1), rtol=1e-11, atol=1e-13)
    for c in (0, 17, C - 1):
        np.testing.assert_allclose(cov[c], np.cov(mats[c], rowvar=False), rtol=1e-8, atol=1e-16)
    n, pm, pc = q.moments(pooled=True)
    allm = mats.reshape(C * iters, 64)
    assert n == C * iters
    np.testing.assert_allclose(pm, allm.mean(axis=0), rtol=1e-11, atol=1e-13)
    np.testing.assert_allclose(pc, np.cov(allm, rowvar=False), rtol=1e-8, atol=1e-16)
    # same chains again, samples never stored: identical moments
    none, acc2 = q.run_chains(k, inits, 2, iters, seed=3, moments=True, keep_samples=False)
    assert none is None
    np.testing.assert_array_equal(acc2, acc)
    n_b, pm_b, pc_b = q.moments(pooled=True)
    assert n_b == n
    np.testing.assert_allclose(pm_b, pm, rtol=1e-12)
    np.testing.assert_allclose(pc_b, pc, rtol=1e-9, atol=1e-18)


@pytest.mark.parametrize("kind", ["rwmh", "ul", "mala", "hmc"])
def test_keyed_chain_equals_replay_with_the_derived_keys(lr, pima, kind):
    """jaxlike.mcmc (device loop in LRB_RNG_KEYED mode) == the counter-free replay whose draws are
    produced on the host side of the same key tree: split(split(root, iters)[i], thin)[s], then
    the kernel's own split (fit-jax2.py:90,100,109; fit-jax-hmc.py:126-129; fit-jax-ul.py:86-88)."""
    import logreg_b200.jaxlike as J
    from logreg_b200 import _native as N
    X = np.asfortranarray(pima["X"])
    prob = lr.Problem(deterministic=True).bind_data(X, pima["y"], pima["pscale"], mode="fp64")
    lr.use(prob)
    pre = pima["pre"].astype(np.float32)
    kk = {"rwmh": lambda: J.mhKernel(J.lpost, J.RandomWalk(0.02 * pima["pre_rw"])),
          "ul": lambda: J.ulKernel(J.lpost, dt=1e-6, pre=pre),
          "mala": lambda: J.malaKernel(J.lpost, dt=1e-6, pre=pre),
          "hmc": lambda: J.hmcKernel(J.lpost, J.glp, eps=2e-3, l=7, dmm=1 / pre)}[kind]()
    assert isinstance(kk, J.KeyedKernel)
    thin, iters = 3, 12
    mat = J.mcmc(pima["chain_init"], kk, thin=thin, iters=iters)         # root key PRNGKey(42)
    assert mat.dtype == np.float32 and mat.shape == (iters, 8)
    # host side of the tree
    Z = np.empty((thin * iters, 8)); U = np.empty(thin * iters)
    for i, ki in enumerate(J.split(J.PRNGKey(42), iters)):
        for s, ks in enumerate(J.split(ki, thin)):
            if kind == "ul":
                kz, ku = ks, None
            else:
                kz, ku = J.split(ks)
                if kind == "hmc":
                    ku = J.split(ku)[1]
            Z[i * thin + s] = prob.rng_dump_p(kz, 0, 1, 8)[0][0]
            if ku is not None:
                U[i * thin + s] = prob.rng_dump_p(ku, 0, 1, 1)[1][0]
    rep, _ = prob.run(kk.dev, pima["chain_init"], thin, iters, Z=Z, U=None if kind == "ul" else U)
    np.testing.assert_array_equal(mat, rep.astype(np.float32))
    # and the oracle's reference kernels driven by the same draws walk the same chain
    tgt = O.Target(X, pima["y"], pima["pscale"])
    rng = O.ReplayRNG(Z, U)
    pre64 = pre.astype(np.float64)
    ok = {"rwmh": lambda: O.mcmc_threaded(pima["chain_init"], O.mh_kernel(tgt.lpost, O.rw_proposal(0.02 * pima["pre_rw"], rng), rng=rng), thin, iters),
          "ul": lambda: O.mcmc_plain(pima["chain_init"], O.ul_kernel(tgt.glp, 8, dt=1e-6, pre=pre64, rng=rng), thin, iters),
          "mala": lambda: O.mcmc_threaded(pima["chain_init"], O.mala_kernel(tgt.lpost, tgt.glp, 8, dt=1e-6, pre=pre64, rng=rng), thin, iters),
          "hmc": lambda: O.mcmc_plain(pima["chain_init"], O.hmc_kernel(tgt.lpost, tgt.glp, eps=2e-3, l=7, dmm=1 / pre64, rng=rng), thin, iters)}[kind]()
    np.testing.assert_allclose(rep, ok, rtol=1e-7, atol=1e-7)
    # one keyed step through the callable == the first step of the chain with thin=1
    k0 = J.split(J.split(J.PRNGKey(42), iters)[0], thin)[0]
    if kk.threaded:
        x1, l1 = kk(k0, pima["chain_init"], -np.inf)
    else:
        x1 = kk(k0, pima["chain_init"])
    one = J.mcmc(pima["chain_init"], kk, thin=1, iters=1, key=None)
    first_key_thin1 = J.split(J.split(J.PRNGKey(42), 1)[0], 1)[0]
    x1b = kk(first_key_thin1, pima["chain_init"], -np.inf)[0] if kk.threaded else kk(first_key_thin1, pima["chain_init"])
    np.testing.assert_array_equal(one[0], x1b)
    assert x1.shape == (8,) and x1.dtype == np.float32


def test_jaxlike_user_kernel_path_and_host_split(lr, pima):
    """A user-written rprop(key, x) goes through the reference's host closure around the device
    lpost; split/normal/uniform are reproducible functions of the key."""
    import logreg_b200.jaxlike as J
    J.bind_data(np.asfortranarray(pima["X"]), pima["y"], pima["pscale"], mode="fp64")
    assert J.split(7, 3) == J.split(7, 3) and len(set(J.split(7, 50))) == 50
    z1, z2 = J.normal(11, [8]), J.normal(11, [8])
    np.testing.assert_array_equal(z1, z2)
    assert 0.0 < J.uniform(5) < 1.0
    scale = (0.02 * pima["pre_rw"]).astype(np.float32)
    user = J.mhKernel(J.lpost, lambda key, x: x + scale * J.normal(key, [8]))
    dev = J.mhKernel(J.lpost, J.RandomWalk(scale))
    a = J.mcmc(pima["chain_init"], user, thin=2, iters=6)
    b = J.mcmc(pima["chain_init"], dev, thin=2, iters=6)
    np.testing.assert_allclose(a, b, rtol=2e-6, atol=2e-6)      # host closure works in float32 states


def test_mhkernel_one_argument_form_of_the_hmc_script(lr, pima):
    """fit-np-hmc.py:56-63: mhKernel(lpost, rprop) -> kernel(x) -> x (lpost re-evaluated at x)."""
    from logreg_b200 import np_hmc as H
    H.bind_data(np.asfortranarray(pima["X"]), pima["y"], pima["pscale"])
    tgt = O.Target(np.asfortranarray(pima["X"]), pima["y"], pima["pscale"])
    rw = lambda x: x + 0.02 * pima["pre_rw"] * np.random.randn(8)
    np.random.seed(3)
    mine = H.mcmc(pima["chain_init"], H.mhKernel(H.lpost, rw), thin=2, iters=20, verb=False)
    np.random.seed(3)
    ref = O.mcmc_plain(pima["chain_init"], O.mh_kernel_recompute(tgt.lpost, rw), 2, 20)
    np.testing.assert_allclose(mine, ref, rtol=1e-9, atol=1e-9)
    assert len(np.unique(mine[:, 0])) > 1


def test_many_chain_buffers_may_grow_between_runs(lr):
    """ADVICE r1 (high): growing the many-chain buffers must invalidate the cached launch graph
    and any paused many-chain run instead of replaying against freed memory."""
    q = lr.Problem(deterministic=True)
    bt = q.gen_synthetic(30_000, 64, mode="fp32", seed=2)
    sd = 2.2 / np.sqrt(30_000)
    k = lr.malaKernel(q.lpost, q.glp, dt=(0.6 * sd) ** 2, pre=1.0)
    inits = bt + 0.5 * sd * np.random.RandomState(1).randn(8, 64)
    m1, a1 = q.run_chains(k, inits, 1, 70, seed=9)          # > 64 evaluations: a replayed graph exists
    q.eval_many(np.tile(bt, (40, 1)))                       # grows every per-chain buffer
    with pytest.raises(lr.LogregB200Error):                 # the paused 8-chain run died with the buffers
        q._ck(q._lib.lrb_run(q._h, __import__("ctypes").byref(q._params(k, 9, 0, -np.inf)), None, 8, 1, 5, None, None,
                             m1[:, :5].copy().ctypes.data_as(__import__("ctypes").POINTER(__import__("ctypes").c_double)), None))
    m2, a2 = q.run_chains(k, inits, 1, 70, seed=9)
    np.testing.assert_array_equal(m2, m1)
    np.testing.assert_array_equal(a2, a1)


@pytest.mark.parametrize("deterministic", [False, True], ids=["drive", "static"])
def test_single_chain_survives_many_chain_buffer_growth(lr, deterministic):
    """A single chain lives in row 0 of the per-chain buffers: growing them (eval_many with more
    chains than ever before) must carry a paused chain, and a run armed with lrb_run_begin, over.
    200 rows are one row batch, so drive mode's sums are exact too and the runs compare bit for bit."""
    import ctypes as C
    from logreg_b200 import _native as N

    def chain(grow):
        q = lr.Problem(deterministic=deterministic)
        bt = q.gen_synthetic(200, 8, mode="fp32", seed=4)
        sd = 2.2 / np.sqrt(200)
        k = lr.malaKernel(q.lpost, q.glp, dt=(0.6 * sd) ** 2, pre=1.0)
        kl = q.info()["kernel_launches"]
        m1, a1 = q.run(k, bt, 1, 30, seed=7)
        drive = q.info()["kernel_launches"] - kl == 2            # sampler_begin + one drive-mode launch
        if grow:
            q.eval_many(np.tile(bt, (16, 1)))
        m2, a2 = q.run(k, None, 1, 30, seed=7)                     # continues the paused chain
        sp = q._params(k, 7, N.RNG_PHILOX, -np.inf)
        q._ck(q._lib.lrb_run_begin(q._h, C.byref(sp), None, 1, 30, None, None))
        if grow:
            q.eval_many(np.tile(bt, (40, 1)))
        q._ck(q._lib.lrb_run_launch(q._h))
        m3, a3 = np.empty((30, 8)), C.c_int64()
        q._ck(q._lib.lrb_run_finish(q._h, N.as_dp(m3), C.byref(a3)))
        return drive, [m1, m2, m3], [a1, a2, a3.value], q.chain_state()

    (d_ref, m_ref, a_ref, st_ref), (d, m, a, st) = chain(False), chain(True)
    assert d_ref == d == (not deterministic)
    for got, ref in zip(m, m_ref):
        np.testing.assert_array_equal(got, ref)
    assert a == a_ref and sum(a) > 0
    np.testing.assert_array_equal(st[0], st_ref[0])
    assert st[1:] == st_ref[1:] and st[2] == 90
