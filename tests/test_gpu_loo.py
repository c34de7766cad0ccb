"""PSIS-LOO cross-validation (gpirtMCMC(..., loo=True), opts.loo): every output against the numpy port of the definitions
(tests/psis_loo_numpy.py) on the log-likelihoods rebuilt from the chain's own stored draws; psis_loo() on adversarial
columns; consistency with predictive=True in the same call; no side effects, thinning invariance, determinism; refusals,
the memory check and the release of the state; and what the Pareto k is for."""
import ctypes as C

import numpy as np
import pytest

import psis_loo_numpy as P

pytestmark = pytest.mark.gpu

N_GRID = 1001
CELL_TOL = 1e-10      # |delta| <= CELL_TOL max(1, |value|) for elpd_loo_cell and p_loo_cell
K_TOL = 1e-9
TOTAL_RTOL = 1e-11


@pytest.fixture(scope="module")
def G():
    import gpirt_b200.sampler as g
    from gpirt_b200 import _lib
    assert _lib.load().gpirt_b200_device_count() > 0, "no CUDA device"
    return g


def _problem(n, m, missing, seed):
    from gpirt_b200 import synthetic
    return synthetic.make(n, m, seed=seed, missing=missing)


def _run(G, prob, S, B, seed=11, **kw):
    from gpirt_b200 import ResponseMatrix
    return G.gpirtMCMC(ResponseMatrix(prob["y"]), S, B, beta_prior_means=prob["pm"], beta_prior_sds=prob["psd"],
                       beta_proposal_sds=prob["pstep"], theta_init=prob["theta_init"], seed=seed, **kw)


def _close_cells(got, want, tol):
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan)
    inf = np.isinf(want)
    assert np.array_equal(got[inf], want[inf])
    ok = ~nan & ~inf
    err = np.abs(got[ok] - want[ok])
    bound = tol * np.maximum(1.0, np.abs(want[ok]))
    assert np.all(err <= bound), (err.max(), np.argmax(err / bound))


def _check_cells(got_e, got_p, got_k, ref, k_cond=None):
    """k_cond (optional, per cell): how far k of the reference moves when its inputs move by the rounding that separates
    them from the device's inputs; the device's k may differ by that much on top of K_TOL"""
    _close_cells(got_e, ref["elpd"], CELL_TOL)
    _close_cells(got_p, ref["p_loo"], CELL_TOL)
    nan = np.isnan(ref["k"])
    assert np.array_equal(np.isnan(got_k), nan)
    assert np.array_equal(np.isinf(got_k), np.isinf(ref["k"]))
    fin = np.isfinite(ref["k"])
    tol = K_TOL + (0.0 if k_cond is None else 2.0 * k_cond[fin])
    err = np.abs(got_k[fin] - ref["k"][fin])
    assert np.all(err <= tol), (err.max(), np.max(err - tol))


def _check_against_draws(out, y):
    ll, sg = P.loglik_from_draws(out, y)
    n, m, S = ll.shape
    ref = P.psis_loo(ll.reshape(n * m, S, order="F"), sg.reshape(n * m, S, order="F"))
    # The device forms g with one fma and its own exp / log1p, so its ll differ from these by a few ulps.  k depends on
    # the tail exceedances exp(lw) - exp(cutoff), which lose relative accuracy when tail draws lie close to the cutoff:
    # the reference is only defined to within how far its k moves under such a perturbation.
    llp, sgp = P.loglik_from_draws(out, y, np.random.default_rng(0))
    k_cond = np.abs(P.psis_loo(llp.reshape(n * m, S, order="F"), sgp.reshape(n * m, S, order="F"))["k"] - ref["k"])
    obs = ~np.isnan(y).ravel(order="F")
    for k in ("elpd", "p_loo", "k"):
        ref[k] = np.where(obs, ref[k], np.nan)
    got = out["loo"]
    thr = P.k_threshold(S)
    _check_cells(got["elpd_loo_cell"].ravel(order="F"), got["p_loo_cell"].ravel(order="F"), got["pareto_k"].ravel(order="F"),
                 ref, np.where(np.isfinite(k_cond), k_cond, 0.0))
    agg = P.aggregate(y, ref)
    for k in ("elpd_loo_item", "elpd_loo_resp"):
        assert np.allclose(got[k], agg[k], rtol=TOTAL_RTOL, atol=1e-12), k
    for k in ("elpd_loo", "p_loo", "looic", "se_elpd_loo"):
        assert abs(got[k] - agg[k]) <= TOTAL_RTOL * abs(agg[k]), (k, got[k], agg[k])
    assert got["n_obs"] == agg["n_obs"]
    k_ref = ref["k"][obs]
    near = int(np.sum(np.abs(k_ref - thr) <= K_TOL + 2.0 * np.nan_to_num(k_cond[obs], posinf=0.0)))
    assert abs(got["n_k_high"] - int(np.sum(k_ref > thr))) <= near
    assert got["k_threshold"] == thr
    M = P.tail_len(S)
    assert got["tail_len"] == M and got["tail_bytes"] == 8 * (M + 4) * n * m
    return ref


# (n, m): one CTA per item and the small-n sweep, the graph-replayed fixed-point sweep, the n > 4096 streaming shape
SHAPES = [(257, 37), (640, 300), (4097, 64)]


@pytest.mark.parametrize("missing", [0.0, 0.05])
@pytest.mark.parametrize("n,m", SHAPES)
def test_loo_against_numpy_on_the_stored_draws(G, n, m, missing):
    prob = _problem(n, m, missing, seed=n + m)
    if n == 640:
        s = G.Sampler(prob["y"], prob["theta_init"], prob["pm"], prob["psd"], prob["pstep"], seed=5)
        s.set_timing(False)
        s.init_draws()
        s.sweep(3)
        assert s.uses(1) == 1 and s.uses(5) > 0, "this shape must run the fixed-point products as graph-replayed sweeps"
        s.close()
    S = 23                                                  # M = 5: the smoothing runs
    out = _run(G, prob, S, 2, loo=True, predictive=True)
    ref = _check_against_draws(out, prob["y"])
    assert np.sum(np.isfinite(ref["k"])) > 0
    # consistency with predictive=True in the same call: lpd is bit-equal to lpd_cell, so the sum differs by the
    # roundings of p_loo = lpd - elpd and of the sum
    lo, pr = out["loo"], out["predictive"]
    obs = ~np.isnan(prob["y"])
    back = lo["p_loo_cell"][obs] + lo["elpd_loo_cell"][obs]
    lpd = pr["lpd_cell"][obs]
    scale = np.maximum(np.abs(lpd), np.abs(lo["elpd_loo_cell"][obs]))
    assert np.all(np.abs(back - lpd) <= 2 * np.spacing(scale)), np.abs(back - lpd).max()
    assert lo["n_obs"] == pr["n_obs"]


# ---- psis_loo() on adversarial columns -------------------------------------------------------------------------------
@pytest.mark.parametrize("S", [0, 1, 4, 20, 21, 22, 5000])
def test_psis_loo_adversarial_columns(G, S):
    rs = np.random.default_rng(S + 1)
    ll = P.adversarial(S, rs)
    e, p, k = G.psis_loo(ll)
    ref = P.psis_loo(ll)
    if S == 0:
        assert np.all(np.isnan(e)) and np.all(np.isnan(p)) and np.all(np.isnan(k))
        return
    _check_cells(e, p, k, ref)
    if S == 1:
        assert np.array_equal(e, ll[:, 0]) and np.all(k == np.inf)
    if S >= 21:
        assert np.any(np.isfinite(k)) and np.any(np.isinf(k))
    if S == 5000:
        assert np.any(k > 1.0)


def test_psis_loo_times_its_kernels(G):
    rs = np.random.default_rng(0)
    ll = P.adversarial(200, rs)
    e, p, k, (ms_update, ms_finish) = G.psis_loo(ll, reps=2)
    assert ms_update > 0.0 and ms_finish > 0.0
    assert np.array_equal(e, G.psis_loo(ll)[0])


# ---- side effects, thinning, determinism, S = 0 / 1 ------------------------------------------------------------------
LOO_KEYS = ("elpd_loo_cell", "p_loo_cell", "pareto_k", "elpd_loo_item", "elpd_loo_resp", "elpd_loo", "p_loo", "looic",
            "se_elpd_loo", "k_threshold", "n_obs", "n_k_high", "tail_len", "tail_bytes")


def test_no_side_effects_thinning_and_determinism(G):
    prob = _problem(300, 40, 0.05, seed=7)
    base = _run(G, prob, 30, 2, irf_band=0.9)
    a = _run(G, prob, 30, 2, irf_band=0.9, loo=True)
    b = _run(G, prob, 30, 2, irf_band=0.9, loo=True)
    t = _run(G, prob, 30, 2, thin=7, loo=True)
    for k in ("theta", "beta", "f", "IRFs"):
        assert np.array_equal(base[k], a[k]), k
    for k in ("mean", "sd", "lower", "upper"):
        assert np.array_equal(base["IRF_summary"][k], a["IRF_summary"][k]), k
    for k in LOO_KEYS:
        assert np.array_equal(a["loo"][k], b["loo"][k], equal_nan=True), k
        assert np.array_equal(a["loo"][k], t["loo"][k], equal_nan=True), k


def test_zero_and_one_sampling_iterations(G):
    prob = _problem(200, 30, 0.05, seed=8)
    out = _run(G, prob, 0, 3, loo=True)["loo"]
    for k in ("elpd_loo_cell", "p_loo_cell", "pareto_k", "elpd_loo_item", "elpd_loo_resp"):
        assert np.all(np.isnan(out[k])), k
    for k in ("elpd_loo", "p_loo", "looic", "se_elpd_loo", "k_threshold"):
        assert np.isnan(out[k]), k
    assert out["tail_len"] == 0 and out["n_k_high"] == 0 and out["n_obs"] == int(np.sum(~np.isnan(prob["y"])))
    one = _run(G, prob, 1, 3, loo=True, predictive=True)
    obs = ~np.isnan(prob["y"])
    ll, _ = P.loglik_from_draws(one, prob["y"])
    lo = one["loo"]
    assert np.allclose(lo["elpd_loo_cell"][obs], ll[:, :, 0][obs], rtol=1e-14, atol=1e-15)
    assert np.all(lo["pareto_k"][obs] == np.inf) and lo["n_k_high"] == lo["n_obs"]
    assert np.allclose(lo["p_loo_cell"][obs], 0.0, atol=1e-14)


# ---- refusals and memory --------------------------------------------------------------------------------------------
def _raw_call(G, y, S, opts):
    """gpirt_b200_mcmc without the Python argument checks; returns (status, last error)"""
    from gpirt_b200 import _lib
    L = _lib.load()
    n, m = y.shape
    C_ = opts.chains.contents.chains if opts.chains else 1
    slots = S // max(1, opts.thin) + 1
    theta_init = np.zeros((n, C_), order="F")
    pm, psd, pstep = np.zeros((2, m), order="F"), np.full((2, m), 3.0, order="F"), np.full((2, m), 0.1, order="F")
    theta = np.empty((slots, n, C_), order="F"); beta = np.empty((2, m, slots, C_), order="F")
    irf = np.empty((N_GRID, m, C_), order="F")
    opts.skip_f_draws = 1
    cb = _lib.PROGRESS_CB(lambda p, c: 0)
    rc = L.gpirt_b200_mcmc(_lib.ptr(np.asfortranarray(y)), n, m, _lib.ptr(theta_init), S, 0, _lib.ptr(pm), _lib.ptr(psd),
                           _lib.ptr(pstep), C.byref(opts), _lib.ptr(theta), _lib.ptr(beta), None, _lib.ptr(irf), cb, None)
    return rc, L.gpirt_b200_last_error().decode()


def test_loo_with_chains_or_shard_is_refused_by_the_library(G):
    from gpirt_b200 import _lib
    y = _problem(64, 8, 0.0, seed=3)["y"]
    lo = _lib.Loo()
    opts = G.make_opts(seed=1)
    ch = _lib.Chains(); ch.chains = 2
    opts.chains = C.pointer(ch)
    opts.loo = C.pointer(lo)
    rc, msg = _raw_call(G, y, 2, opts)
    assert rc == _lib.ERR_ARG and "PSIS-LOO" in msg
    opts = G.make_opts(seed=1, rank=0, world_size=2, m_global=16, item_offset=0)
    opts.loo = C.pointer(lo)
    rc, msg = _raw_call(G, y, 2, opts)
    assert rc == _lib.ERR_ARG and "sharded" in msg


def test_state_beyond_free_memory_is_refused_before_the_first_sweep(G):
    import time
    from gpirt_b200 import _lib
    n, m, S = 100, 4000, 10 ** 9
    M = P.tail_len(S)
    want = 8 * (M + 4) * n * m
    assert want > 200e9
    y = _problem(n, m, 0.0, seed=1)["y"]
    lo = _lib.Loo()
    opts = G.make_opts(seed=1, thin=S)
    opts.loo = C.pointer(lo)
    t0 = time.perf_counter()
    rc, msg = _raw_call(G, y, S, opts)
    assert rc == _lib.ERR_NOMEM, msg
    assert time.perf_counter() - t0 < 60.0            # 10^9 sweeps would take days
    assert lo.tail_bytes == want and lo.tail_len == M
    assert ("%d bytes" % want) in msg


def test_state_is_returned_after_the_call(G):
    import torch
    prob = _problem(100, 20000, 0.0, seed=8)
    S = 500
    assert 8 * (P.tail_len(S) + 4) * 100 * 20000 >= 1 << 30
    _run(G, prob, S, 0, store_f=False, thin=S)
    torch.cuda.synchronize()
    free_without = torch.cuda.mem_get_info()[0]
    out = _run(G, prob, S, 0, store_f=False, thin=S, loo=True)
    assert out["loo"]["tail_bytes"] >= 1 << 30
    torch.cuda.synchronize()
    free_with = torch.cuda.mem_get_info()[0]
    assert abs(free_with - free_without) <= 64 << 20, (free_without, free_with)


# ---- usefulness ------------------------------------------------------------------------------------------------------
def test_loo_predicts_held_out_cells_and_flags_surprising_ones(G):
    """n = 600, m = 40, S = 1000 with 10 % of the observed cells held out.  The mean elpd_loo per observed cell estimates
    the mean held-out log predictive density per cell, and elpd_loo lies close to elpd_waic.  Expected before the first
    run: 30 responses flipped against a confident prediction get a Pareto k above k_threshold clearly more often than the
    other cells.  Measured on a B200 (DESIGN 8.5): 0 % of the flipped cells against 0.08 % of the others, mean Pareto k
    0.322 against 0.157, mean elpd_loo_cell -3.37 against -0.49.  The test pins what holds: the flipped responses have
    the larger Pareto k on average, and elpd_loo_cell calls them badly predicted."""
    n, m, S, B = 600, 40, 1000, 300
    prob = _problem(n, m, 0.0, seed=31)
    rs = np.random.default_rng(32)
    y = prob["y"].copy()
    held = rs.random((n, m)) < 0.10
    y_hold = np.where(held, y, np.nan)
    y[held] = np.nan
    out = _run(G, dict(prob, y=y), S, B, store_f=False, thin=50, loo=True, predictive=True, y_holdout=y_hold)
    lo, pr = out["loo"], out["predictive"]
    per_cell = lo["elpd_loo"] / lo["n_obs"]
    hold = pr["lpd_cell"][held]
    se = np.sqrt((lo["se_elpd_loo"] / lo["n_obs"]) ** 2 + np.var(hold, ddof=1) / hold.size)
    waic_gap = abs(lo["elpd_loo"] - pr["elpd_waic"])
    # flip 30 responses the model predicts with probability > 0.95
    obs = ~np.isnan(y)
    p_obs = np.where(y > 0, pr["pred"], 1.0 - pr["pred"])
    cand = np.flatnonzero((obs & (p_obs > 0.95)).ravel(order="F"))
    flip = rs.choice(cand, 30, replace=False)
    y2 = y.copy().ravel(order="F")
    y2[flip] = -y2[flip]
    y2 = y2.reshape(n, m, order="F")
    lo2 = _run(G, dict(prob, y=y2), S, B, store_f=False, thin=50, loo=True)["loo"]
    kf = lo2["pareto_k"].ravel(order="F")
    mask = np.zeros(n * m, bool); mask[flip] = True
    rest = obs.ravel(order="F") & ~mask
    share_flip, share_rest = np.mean(kf[mask] > lo2["k_threshold"]), np.mean(kf[rest] > lo2["k_threshold"])
    ef = lo2["elpd_loo_cell"].ravel(order="F")
    print("elpd_loo per cell %.4f, held-out lpd per cell %.4f (se %.4f); |elpd_loo - elpd_waic| = %.3f, se_elpd_loo = %.3f; "
          "n_k_high %d of %d; k > %.3f for %.1f %% of flipped and %.2f %% of other cells; mean k %.3f flipped, %.3f others; "
          "mean elpd_loo_cell %.3f flipped, %.3f others"
          % (per_cell, hold.mean(), se, waic_gap, lo["se_elpd_loo"], lo["n_k_high"], lo["n_obs"], lo2["k_threshold"],
             100 * share_flip, 100 * share_rest, kf[mask].mean(), kf[rest].mean(), ef[mask].mean(), ef[rest].mean()))
    assert abs(per_cell - hold.mean()) <= 3.0 * se
    assert waic_gap <= lo["se_elpd_loo"]
    assert ef[mask].mean() < ef[rest].mean() + np.log(0.1)     # the flipped responses are at least 10 times less likely
    assert kf[mask].mean() > 1.5 * kf[rest].mean()
