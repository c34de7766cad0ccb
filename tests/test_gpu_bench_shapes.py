"""Oracle parity AT THE BENCHMARKED SHAPES (BASELINE.json configs): the kernel instantiations bench.py times are the ones
compared with the CPU oracle here, through the C ABI.

  C2  1024 x 2000   one full lock-step sweep of the public call against the oracle's gpirtMCMC restatement
  C3  4096 x 10000  the oracle needs hours per sweep, but given theta and L every item is independent (draw-f.cpp:69-71,
                    draw-fstar.cpp:23-29, draw-beta.cpp:16-38) and every respondent's grid draw is independent given f*
                    (draw-theta.cpp:12-34): each step runs on the FULL GPU state and >= 32 random items / >= 16 random
                    respondents are checked against the oracle with the same addressed variates (stream maps), with the
                    fixed-point (int8 tensor-core) products on and off, with and without 5 % missing cells
  C5  16384 x 20000 the same steps on the full C5 state (fixed-point products on, 0 % / 5 % missing): K* solves by blocked
                    substitution, streaming per-item kernels, the rebuilt factor checked on sampled rows
  n > 4096          the streaming launch shape of the per-item kernels (C5's shape) on small-m problems

Every test asserts WHICH code path ran (gpirt_b200_sampler_uses).  Tolerances as in test_gpu_parity.py: discrete decisions
(ESS proposal counts, theta grid indices) identical, values to 1e-9 / 1e-8 (solves: cond(S) ~ 1e7)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ITEM_CTA, ITEM_PERSISTENT, ITEM_STREAM = 0, 1, 2


@pytest.fixture(scope="module")
def G():
    import gpirt_b200.sampler as g
    from gpirt_b200 import _lib
    assert _lib.load().gpirt_b200_device_count() > 0, "no CUDA device"
    return g


def test_c2_one_full_lockstep_sweep(G, O):
    """BASELINE configs[1]: 1024 x 2000, synthetic data of bench.py, initial draws + one sweep, draw by draw"""
    from gpirt_b200 import ResponseMatrix, synthetic
    c = synthetic.WORKLOADS["c2"]
    d = synthetic.make(c["n"], c["m"])
    seed = synthetic.SEED
    got = G.gpirtMCMC(ResponseMatrix(d["y"]), 1, 0, beta_prior_means=d["pm"], beta_prior_sds=d["psd"],
                      beta_proposal_sds=d["pstep"], theta_init=d["theta_init"], seed=seed)
    want = O.mcmc(d["y"], d["theta_init"], 1, 0, d["pm"], d["psd"], d["pstep"], O.Rng.keyed(seed), theta_cdf_mode=1)
    assert np.array_equal(got["theta"], want["theta"]), "theta draws (grid points) must be identical"
    assert np.max(np.abs(got["beta"] - want["beta"])) <= 1e-9
    assert np.max(np.abs(got["f"] - want["f"])) <= 1e-7
    assert np.max(np.abs(got["IRFs"] - want["IRFs"])) <= 1e-7
    # the paths the bench times at this shape: fixed-point products, int8 theta contraction, persistent ESS
    s = G.Sampler(d["y"], d["theta_init"], seed=seed)
    s.init_draws(); s.sweep(1)
    assert (s.uses(0), s.uses(1), s.uses(2)) == (1, 1, ITEM_PERSISTENT)
    s.close()


def _c3_state(G, missing, monkeypatch, int8, workload="c3"):
    from gpirt_b200 import synthetic, _lib
    monkeypatch.setenv("GPIRT_GEMM_INT8", "1" if int8 else "0")
    c = synthetic.WORKLOADS[workload]
    d = synthetic.make(c["n"], c["m"], missing=missing)
    s = G.Sampler(d["y"], d["theta_init"], d["pm"], d["psd"], d["pstep"], seed=synthetic.SEED)
    s.set_pipeline(False)          # steps are run one at a time below
    s.init_draws()
    s.sweep(2)                     # theta now lives on the 0.01 grid with thousands of duplicated rows (SURVEY F2)
    assert s.uses(1) == (1 if int8 else 0) and s.uses(0) == 1
    return d, s, _lib


@pytest.mark.parametrize("workload,missing,int8", [
    pytest.param("c3", 0.0, True, id="0.0-True"), pytest.param("c3", 0.0, False, id="0.0-False"),
    pytest.param("c3", 0.05, True, id="0.05-True"), pytest.param("c3", 0.05, False, id="0.05-False"),
    pytest.param("c5", 0.0, True, id="c5-0.0-True"), pytest.param("c5", 0.05, True, id="c5-0.05-True")])
def test_c3_sampled_items_and_respondents_against_the_oracle(G, O, monkeypatch, workload, missing, int8):
    """BASELINE configs[2] (the bench workload): one step at a time on the full 4096 x 10000 state.  The same at C5
    (BASELINE configs[4], 16384 x 20000): L Z with K = 16384, the f* solves by blocked substitution (route 1), the theta
    contraction over 20000 items for 16384 rows and the streaming item kernels."""
    from gpirt_b200 import synthetic
    d, s, _lib = _c3_state(G, missing, monkeypatch, int8, workload)
    n, m = d["y"].shape
    big = n > 4096                 # C5: per-item kernels in the streaming shape, K* solves by substitution
    item_shape = ITEM_STREAM if big else ITEM_PERSISTENT
    assert s.uses(4) == (1 if big else 0)
    seed = synthetic.SEED
    rs = np.random.RandomState(42 + int(100 * missing) + int(int8))
    J = np.sort(rs.choice(m, 32, replace=False))
    I = np.sort(rs.choice(n, 16, replace=False))
    theta = s.get(_lib.THETA); beta = s.get(_lib.BETA); L = s.get(_lib.CHOL)
    assert len(np.unique(theta)) <= 1001 < n, "theta on the grid: duplicated rows, PD only through the jitter"
    yJ = np.asfortranarray(d["y"][:, J])
    ts, prior = O.grid()

    # ---- draw_f (draw-f.cpp:21-60): proposals nu = L z, shrink counts, new f ----
    f0 = s.get(_lib.F)
    sweep = 11
    s.step(_lib.STEP_DRAW_F, sweep)
    assert s.uses(2) == item_shape
    nu = s.get(_lib.NU); f1 = s.get(_lib.F); nprop = s.get(_lib.ESS_NPROP).astype(int)
    rng = O.Rng.keyed(seed); rng.set_sweep(sweep); rng.set_item_map(J)
    mu = O.linear_mean(theta, beta[:, J])
    fo, npo = O.draw_f(f0[:, J], yJ, L, mu, rng)
    for jj, j in enumerate(J[:4]):   # the proposal itself for a few items: nu_j = L z_j
        z = np.array([O.keyed_normal(seed, sweep, O.P_ESS_Z, int(j), i) for i in range(n)])
        # C5: the fixed-point bound K 2^-51 max|L_i| max|z| with L sliced at the fixed scale |L| < 2^L_FIXED_EXP = 2
        tol = n * 2.0 ** -51 * 2.0 * np.abs(z).max() if big else 1e-11
        assert np.max(np.abs(nu[:, j] - L @ z)) <= tol
    assert np.array_equal(nprop[J], npo), "ESS proposal counts must match the oracle"
    assert np.max(np.abs(f1[:, J] - fo)) <= 1e-9

    # ---- draw_fstar (draw-fstar.cpp:10-31) ----
    sweep = 12
    s.step(_lib.STEP_DRAW_FSTAR, sweep)
    fs = s.get(_lib.FSTAR); sd = s.get(_lib.FSTAR_S)
    rng = O.Rng.keyed(seed); rng.set_sweep(sweep); rng.set_item_map(J)
    fso, so, _ = O.draw_fstar(f1[:, J], theta, ts, L, O.linear_mean(ts, beta[:, J]), rng)
    assert np.max(np.abs(sd - so)) <= 1e-8
    assert np.max(np.abs(fs[:, J] - fso)) <= 1e-7 * max(1.0, np.abs(fso).max())

    # ---- draw_theta (draw-theta.cpp:12-34): log-posterior rows and grid index of sampled respondents ----
    sweep = 13
    s.step(_lib.STEP_DRAW_THETA, sweep)
    idx = s.get(_lib.THETA_IDX).astype(int); logp = s.get(_lib.LOGP); theta_new = s.get(_lib.THETA)
    rng = O.Rng.keyed(seed); rng.set_sweep(sweep); rng.set_respondent_map(I)
    tho, idxo, logpo = O.draw_theta(ts, d["y"][I, :], prior, fs, rng, mode=1)
    want_ll = logpo - prior[None, :]
    assert np.max(np.abs(logp[I, :] - want_ll) / np.maximum(1.0, np.abs(want_ll))) <= 1e-12
    assert np.array_equal(idx[I], idxo), "grid indices must match the oracle (stabilised CDF)"
    assert np.array_equal(theta_new[I], tho)

    # ---- draw_beta (draw-beta.cpp:16-38) with the NEW theta and the current f ----
    sweep = 14
    s.step(_lib.STEP_DRAW_BETA, sweep)
    assert s.uses(3) == item_shape
    b1 = s.get(_lib.BETA)
    rng = O.Rng.keyed(seed); rng.set_sweep(sweep); rng.set_item_map(J)
    bo, _ = O.draw_beta(beta[:, J], theta_new, yJ, f1[:, J], d["pm"][:, J], d["psd"][:, J], d["pstep"][:, J], rng)
    assert np.max(np.abs(b1[:, J] - bo)) <= 1e-12

    # ---- rebuild (gpirtMCMC.cpp:76-78): the Cholesky chain kernels against the definition ----
    del nu, f0, f1, L
    s.step(_lib.STEP_REBUILD, 0)
    L2 = s.get(_lib.CHOL)
    s.close()
    S = O.K(theta_new, theta_new) + 1e-3 * np.eye(n)
    assert np.array_equal(np.triu(L2, 1), np.zeros_like(L2)), "strict upper triangle must be exactly zero"
    if not big:
        assert np.max(np.abs(L2 @ L2.T - S)) <= 1e-12 * 12
    else:   # 64 sampled rows (and the first and last) against 2 n u max|S|, as test_gpu_large_n.py::_check_factor
        R = np.unique(np.r_[0, n - 1, rs.choice(n, 64, replace=False)])
        assert np.max(np.abs(L2[R, :] @ L2.T - S[R, :])) <= 2 * n * 2.0 ** -53 * np.abs(S).max()


@pytest.mark.parametrize("n,m,missing", [(4097, 8, 0.0), (6000, 6, 0.1), (8192, 4, 0.0)])
def test_streaming_item_kernels_beyond_4096_respondents(G, O, n, m, missing):
    """n > 4096: an item no longer fits the register file of one CTA; ESS and beta run in the streaming launch shape
    (the shape of BASELINE configs[4], n = 16384).  Same body, same oracle."""
    from gpirt_b200 import _lib
    from conftest import make_problem
    prob = make_problem(n, m, seed=n, missing=missing, grid_theta=True)
    seed = 9000 + n
    s = G.Sampler(prob["y"], prob["theta"], prob["pm"], prob["psd"], prob["pstep"], seed=seed)
    rs = np.random.RandomState(n)
    L = s.get(_lib.CHOL)
    f = np.asfortranarray(L @ rs.randn(n, m)); beta = rs.randn(2, m)
    s.set(_lib.F, f); s.set(_lib.BETA, beta)
    sweep = 5
    s.step(_lib.STEP_DRAW_F, sweep)
    assert s.uses(2) == ITEM_STREAM
    f1 = s.get(_lib.F); nprop = s.get(_lib.ESS_NPROP).astype(int)
    rng = O.Rng.keyed(seed); rng.set_sweep(sweep)
    fo, npo = O.draw_f(f, prob["y"], L, O.linear_mean(prob["theta"], beta), rng)
    assert np.array_equal(nprop, npo), "ESS proposal counts must match the oracle"
    assert np.max(np.abs(f1 - fo)) <= 1e-9
    sweep = 6
    s.step(_lib.STEP_DRAW_BETA, sweep)
    assert s.uses(3) == ITEM_STREAM
    b1 = s.get(_lib.BETA)
    rng = O.Rng.keyed(seed); rng.set_sweep(sweep)
    bo, _ = O.draw_beta(beta, prob["theta"], prob["y"], f1, prob["pm"], prob["psd"], prob["pstep"], rng)
    assert np.max(np.abs(b1 - bo)) <= 1e-12
    s.close()


def test_thinned_and_summarised_draw_storage(G):
    """opts.thin / f_mean_out / f_sd_out (the draw-storage options beside gpirtMCMC.cpp:99-103): the thinned slots are
    exactly every k-th slot of the un-thinned chain, and the on-device mean / sd of f equal the host's over all slots"""
    from gpirt_b200 import ResponseMatrix
    from conftest import make_problem
    prob = make_problem(300, 70, seed=8, missing=0.05)
    kw = dict(beta_prior_means=prob["pm"], beta_prior_sds=prob["psd"], beta_proposal_sds=prob["pstep"],
              theta_init=prob["theta"], seed=5)
    S, B, k = 12, 3, 4
    full = G.gpirtMCMC(ResponseMatrix(prob["y"]), S, B, f_summary=True, **kw)
    thin = G.gpirtMCMC(ResponseMatrix(prob["y"]), S, B, thin=k, f_summary=True, **kw)
    assert thin["theta"].shape == (S // k + 1, 300) and thin["f"].shape == (300, 70, S // k + 1)
    assert np.array_equal(thin["theta"], full["theta"][::k])
    assert np.array_equal(thin["beta"], full["beta"][:, :, ::k])
    assert np.array_equal(thin["f"], full["f"][:, :, ::k])
    assert np.array_equal(thin["IRFs"], full["IRFs"]), "IRFs average over ALL sampling iterations"
    fm, fsd = full["f"][:, :, 1:].mean(axis=2), full["f"][:, :, 1:].std(axis=2, ddof=1)
    for r in (full, thin):
        assert np.max(np.abs(r["f_mean"] - fm)) <= 1e-12
        assert np.max(np.abs(r["f_sd"] - fsd)) <= 1e-11
    only = G.gpirtMCMC(ResponseMatrix(prob["y"]), S, B, thin=k, store_f=False, f_summary=True, **kw)
    assert "f" not in only and np.array_equal(only["f_mean"], thin["f_mean"])
