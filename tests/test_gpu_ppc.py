"""Posterior predictive model checks (gpirtMCMC(..., ppc=True, ppc_pairs=True), opts.ppc): the chi-square PPP-values per
item, per respondent and in all, and the pairwise odds-ratio PPP-values, against numpy rebuilding every replicate from the
chain's own stored draws and the Philox uniforms of purpose 8; the odds-ratio kernels alone (ppc_pairs) against integer
products on adversarial data; no side effects, thinning invariance, determinism, edge cases, refusals, and the checks
finding a planted second dimension."""
import ctypes as C
import mmap

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N_GRID = 1001
MAP_NORESERVE = 0x4000   # Linux: no swap reservation for a mapping that is never written


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


def _counts(Y, M):
    """n11, n10, n01, n00 of every item pair from Y (+1 / -1, 0 where missing) and M = observed mask, exact in float64"""
    Y = Y.astype(np.float64); M = M.astype(np.float64)
    P1, P2, P3, P4 = Y.T @ Y, Y.T @ M, M.T @ Y, M.T @ M
    q = [np.rint(v).astype(np.int64) for v in (P4 + P1 + P2 + P3, P4 - P1 + P2 - P3, P4 - P1 - P2 + P3, P4 + P1 - P2 - P3)]
    assert all(np.all(v % 4 == 0) for v in q)
    return [v // 4 for v in q]


def _or_at_least(rep, obs):
    """OR(rep) >= OR(obs) with the +1/2 correction, compared exactly in Python integers"""
    f = lambda v: (2 * v.astype(object) + 1)
    a, b, c, d = rep
    ao, bo, co, do = obs
    return (f(a) * f(d) * f(bo) * f(co) >= f(ao) * f(do) * f(b) * f(c)).astype(bool)


def _log_or(obs):
    a, b, c, d = (v.astype(np.float64) for v in obs)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.log(((a + 0.5) * (d + 0.5)) / ((b + 0.5) * (c + 0.5)))


def _pair_nan(obs):
    nan = (obs[0] + obs[1] + obs[2] + obs[3]) == 0
    np.fill_diagonal(nan, True)
    return nan


def _reference(G, out, y, seed, B):
    """every output of out["ppc"] rebuilt in numpy from the stored draws (thin = 1: slot s = sampling iteration s)"""
    f, th, be = out["f"], out["theta"], out["beta"]
    n, m, S = f.shape[0], f.shape[1], f.shape[2] - 1
    obs = ~np.isnan(y)
    yo = np.where(obs, y, 0.0)
    o_counts = _counts(yo, obs)
    cnt = dict(item=np.zeros(m, int), resp=np.zeros(n, int), glob=0, pair=np.zeros((m, m), int))
    amb = dict(item=np.zeros(m, int), resp=np.zeros(n, int), glob=0)
    for s in range(1, S + 1):
        g = f[:, :, s] + (th[s, :][:, None] * be[1, :, s][None, :] + be[0, :, s][None, :])
        p = 1.0 / (1.0 + np.exp(-g))
        u = np.stack([G.rng_probe(seed, B + s, 8, j, 0, n)[0] for j in range(m)], axis=1)
        assert np.all(np.abs(u - p)[obs] >= 1e-12), "the chosen seed puts a uniform within 1e-12 of p"
        yr = np.where(obs, np.where(u < p, 1.0, -1.0), 0.0)
        to = np.where(obs, np.exp(-yo * g), 0.0)
        tr = np.where(obs, np.exp(-yr * g), 0.0)
        for key, ax in (("item", 0), ("resp", 1), ("glob", None)):
            do, dr = to.sum(axis=ax), tr.sum(axis=ax)
            same = np.all(yr == yo, axis=ax)
            cnt[key] = cnt[key] + (dr >= do)
            amb[key] = amb[key] + ((np.abs(dr - do) <= 1e-12 * do) & ~same)
        cnt["pair"] += _or_at_least(_counts(yr, obs), o_counts)
    return S, obs, o_counts, cnt, amb


def _check(G, out, y, seed, B, pairs=True):
    S, obs, o_counts, cnt, amb = _reference(G, out, y, seed, B)
    got = out["ppc"]
    for key, name in (("item", "item_ppp"), ("resp", "resp_ppp")):
        dev = np.rint(got[name] * S).astype(int)
        assert np.allclose(got[name] * S, dev, rtol=0, atol=1e-9)
        assert np.all(np.abs(dev - cnt[key]) <= amb[key]), name
    assert abs(int(round(got["ppp"] * S)) - int(cnt["glob"])) <= int(amb["glob"])
    if pairs:
        nan = _pair_nan(o_counts)
        want = np.where(nan, np.nan, cnt["pair"] * (1.0 / S))
        assert np.array_equal(got["pair_ppp"], want, equal_nan=True)
        ref = np.where(nan, np.nan, _log_or(o_counts))
        assert np.array_equal(np.isnan(got["pair_log_or"]), np.isnan(ref))
        ok = ~np.isnan(ref)
        assert np.all(np.abs(got["pair_log_or"][ok] - ref[ok]) <= 2 * np.spacing(np.abs(ref[ok])))
        assert np.array_equal(got["pair_ppp"], got["pair_ppp"].T, equal_nan=True)
        assert np.array_equal(got["pair_log_or"], got["pair_log_or"].T, equal_nan=True)
        assert got["pair_bytes"] > 20 * (m := y.shape[1]) * (m + 1) // 2


# (n, m, S, B): the per-item ESS / beta launch shapes, the graph-replayed pipelined sweep and the n > 4096 streaming shape
SHAPES = [(257, 37, 6, 3), (640, 300, 5, 4), (4097, 64, 3, 2)]


@pytest.mark.parametrize("missing", [0.0, 0.05])
@pytest.mark.parametrize("n,m,S,B", SHAPES)
def test_ppc_against_numpy_on_the_stored_draws(G, n, m, S, B, missing):
    prob = _problem(n, m, missing, seed=n + m)
    seed = 1234 + n
    out = _run(G, prob, S, B, seed=seed, ppc=True, ppc_pairs=True)
    _check(G, out, prob["y"], seed, B)


def test_no_side_effects_thinning_and_determinism(G):
    prob = _problem(300, 40, 0.05, seed=7)
    base = _run(G, prob, 6, 2, irf_band=0.9)
    a = _run(G, prob, 6, 2, irf_band=0.9, ppc=True, ppc_pairs=True)
    b = _run(G, prob, 6, 2, irf_band=0.9, ppc=True, ppc_pairs=True)
    t = _run(G, prob, 6, 2, thin=4, ppc=True, ppc_pairs=True)
    for k in ("theta", "beta", "f", "IRFs"):
        assert np.array_equal(base[k], a[k]), k
    for k in ("mean", "sd", "lower", "upper"):
        assert np.array_equal(base["IRF_summary"][k], a["IRF_summary"][k]), k
    for k in ("item_ppp", "resp_ppp", "ppp", "pair_ppp", "pair_log_or", "pair_bytes"):
        assert np.array_equal(a["ppc"][k], b["ppc"][k], equal_nan=True), k
        assert np.array_equal(a["ppc"][k], t["ppc"][k], equal_nan=True), k
    # the chi-square outputs alone are the same as with the pair outputs
    c = _run(G, prob, 6, 2, ppc=True)
    for k in ("item_ppp", "resp_ppp", "ppp"):
        assert np.array_equal(a["ppc"][k], c["ppc"][k], equal_nan=True), k
    assert "pair_ppp" not in c["ppc"]


def test_zero_and_one_sampling_iterations(G):
    prob = _problem(200, 30, 0.05, seed=8)
    out = _run(G, prob, 0, 3, ppc=True, ppc_pairs=True)
    for k in ("item_ppp", "resp_ppp", "pair_ppp"):
        assert np.all(np.isnan(out["ppc"][k])), k
    assert np.isnan(out["ppc"]["ppp"])
    assert np.all(np.isnan(out["ppc"]["pair_log_or"]))
    seed = 99
    one = _run(G, prob, 1, 3, seed=seed, store_f=True, ppc=True, ppc_pairs=True)
    _check(G, one, prob["y"], seed, 3)
    for k in ("item_ppp", "resp_ppp"):
        assert np.all(np.isin(one["ppc"][k], (0.0, 1.0))), k


def _raw_call(G, y, S, opts):
    """gpirt_b200_mcmc without the Python argument checks; returns (status, last error)"""
    from gpirt_b200 import _lib
    L = _lib.load()
    n, m = y.shape
    C_ = opts.chains.contents.chains if opts.chains else 1
    slots = S + 1
    theta_init = np.zeros((n, C_), order="F")
    pm, psd, pstep = np.zeros((2, m), order="F"), np.full((2, m), 3.0, order="F"), np.full((2, m), 0.1, order="F")
    theta = np.empty((slots, n, C_), order="F"); beta = np.empty((2, m, slots, C_), order="F")
    irf = np.empty((N_GRID, m, C_), order="F")
    opts.skip_f_draws = 1
    cb = _lib.PROGRESS_CB(lambda p, c: 0)
    rc = L.gpirt_b200_mcmc(_lib.ptr(np.asfortranarray(y)), n, m, _lib.ptr(theta_init), S, 0, _lib.ptr(pm), _lib.ptr(psd),
                           _lib.ptr(pstep), C.byref(opts), _lib.ptr(theta), _lib.ptr(beta), None, _lib.ptr(irf), cb, None)
    return rc, L.gpirt_b200_last_error().decode()


def test_ppc_with_chains_is_refused_by_the_library(G):
    from gpirt_b200 import _lib
    y = _problem(64, 8, 0.0, seed=3)["y"]
    opts = G.make_opts(seed=1)
    ch = _lib.Chains(); ch.chains = 2
    pp = _lib.Ppc()
    item = np.empty(8); pp.item_ppp = _lib.ptr(item)
    opts.chains = C.pointer(ch)
    opts.ppc = C.pointer(pp)
    rc, msg = _raw_call(G, y, 2, opts)
    assert rc == _lib.ERR_ARG and "ppc" in msg


def test_pair_state_beyond_free_memory_is_refused(G):
    """large m, small n: the pair state (about 20 bytes per pair) cannot fit in the device's memory; the call refuses
    before its first sweep and reports the bytes it needed.  The m x m output is an unreserved mapping (never written)."""
    from gpirt_b200 import _lib
    n, m = 8, 160000
    rs = np.random.default_rng(4)
    y = np.where(rs.random((n, m)) < 0.5, 1.0, -1.0)
    y[0, :], y[1, :] = 1.0, -1.0
    buf = mmap.mmap(-1, 8 * m * m, flags=mmap.MAP_PRIVATE | mmap.MAP_ANONYMOUS | MAP_NORESERVE)
    out = np.frombuffer(buf, dtype=np.float64)
    pp = _lib.Ppc()
    pp.pair_ppp = out.ctypes.data_as(C.POINTER(C.c_double))
    opts = G.make_opts(seed=1)
    opts.ppc = C.pointer(pp)
    rc, msg = _raw_call(G, y, 1, opts)
    assert rc == _lib.ERR_NOMEM, msg
    assert "bytes" in msg
    assert pp.pair_bytes >= 20 * m * (m + 1) // 2 > 180e9
    del out
    buf.close()


# ---- the odds-ratio kernels alone ------------------------------------------------------------------------------------
def _pm1(rs, shape):
    return np.where(rs.random(shape) < 0.5, 1.0, -1.0)


def _pairs_reference(y, reps):
    obs = ~np.isnan(y)
    o = _counts(np.where(obs, y, 0.0), obs)
    nan = _pair_nan(o)
    ex = np.zeros(nan.shape, int)
    for r in range(reps.shape[2]):
        ex += _or_at_least(_counts(np.where(obs, reps[:, :, r], 0.0), obs), o)
    return np.where(nan, np.nan, _log_or(o)), np.where(nan, np.nan, ex.astype(np.float64))


@pytest.mark.parametrize("n,m,missing", [(100, 418, 0.0), (257, 301, 0.0), (257, 301, 0.05), (4097, 1000, 0.0),
                                         (4097, 1000, 0.05), (1024, 2000, 0.05)])
def test_ppc_pairs_against_integer_products(G, n, m, missing):
    rs = np.random.default_rng(n * 7 + m)
    y = _pm1(rs, (n, m))
    y[rs.random((n, m)) < missing] = np.nan
    reps = _pm1(rs, (n, m, 3))
    reps[np.isnan(y)] = 7.0                      # read where y is observed only
    lor, ex = G.ppc_pairs(y, reps)
    ref_lor, ref_ex = _pairs_reference(y, reps)
    assert np.array_equal(ex, ref_ex, equal_nan=True)
    ok = ~np.isnan(ref_lor)
    assert np.array_equal(np.isnan(lor), ~ok)
    assert np.all(np.abs(lor[ok] - ref_lor[ok]) <= 2 * np.spacing(np.abs(ref_lor[ok])))
    # replicates equal to y: every pair ties, so every replicate counts
    _, ex = G.ppc_pairs(y, np.repeat(np.where(np.isnan(y), 7.0, y)[:, :, None], 3, axis=2))
    assert np.array_equal(ex, np.where(np.isnan(ref_ex), np.nan, 3.0), equal_nan=True)


def test_ppc_pairs_empty_cells_and_pairs_nobody_answered(G):
    rs = np.random.default_rng(5)
    n, m = 300, 6
    y = _pm1(rs, (n, m))
    y[:, 1] = y[:, 0]                     # n10 = n01 = 0
    y[:, 2] = -y[:, 0]                    # n11 = n00 = 0
    y[:, 3] = 1.0; y[0, 3] = -1.0         # almost constant
    y[: n // 2, 4] = np.nan               # items 4 and 5 share no respondent
    y[n // 2:, 5] = np.nan
    reps = _pm1(rs, (n, m, 4))
    lor, ex = G.ppc_pairs(y, reps)
    ref_lor, ref_ex = _pairs_reference(y, reps)
    assert np.array_equal(ex, ref_ex, equal_nan=True)
    assert np.isnan(lor[4, 5]) and np.isnan(lor[5, 4]) and np.isnan(ex[4, 5])
    assert np.all(np.isnan(np.diag(lor))) and np.all(np.isnan(np.diag(ex)))
    ok = ~np.isnan(ref_lor)
    assert np.all(np.abs(lor[ok] - ref_lor[ok]) <= 2 * np.spacing(np.abs(ref_lor[ok])))


def _column_pair(counts):
    a, b, c, d = counts
    col_j = np.r_[np.ones(a + b), -np.ones(c + d)]
    col_k = np.r_[np.ones(a), -np.ones(b), np.ones(c), -np.ones(d)]
    return np.stack([col_j, col_k], axis=1)


# observed and replicated counts over n = 200000 respondents where both sides of the comparison exceed 2^64 and their
# low 64 bits order them the wrong way round (found by a seeded search)
OVERFLOW_CASES = [((52675, 48219, 54922, 44184), (45439, 43537, 49993, 61031), 1.0),
                  ((50870, 42150, 57387, 49593), (56438, 48245, 53247, 42070), 0.0)]


@pytest.mark.parametrize("obs,rep,want", OVERFLOW_CASES)
def test_ppc_pairs_comparison_needs_128_bits(G, obs, rep, want):
    f = lambda v: 2 * v + 1
    (a, b, c, d), (ar, br, cr, dr) = obs, rep
    lhs, rhs = f(ar) * f(dr) * f(b) * f(c), f(a) * f(d) * f(br) * f(cr)
    assert lhs >= 2 ** 64 and rhs >= 2 ** 64
    assert (lhs >= rhs) == bool(want) and ((lhs % 2 ** 64) >= (rhs % 2 ** 64)) != bool(want)
    y = _column_pair(obs)
    lor, ex = G.ppc_pairs(y, _column_pair(rep)[:, :, None])
    assert ex[0, 1] == ex[1, 0] == want


def test_ppc_pairs_more_respondents_than_a_grid_column_holds(G):
    """n beyond 65535 x 256 respondents: the plane conversion keeps respondents on grid.x"""
    n = (1 << 24) + 1000
    rs = np.random.default_rng(6)
    y = _pm1(rs, (n, 2))
    y[rs.random(n) < 0.05, 1] = np.nan
    reps = _pm1(rs, (n, 2, 1))
    lor, ex = G.ppc_pairs(y, reps)
    ref_lor, ref_ex = _pairs_reference(y, reps)
    assert np.array_equal(ex, ref_ex, equal_nan=True)
    assert abs(lor[0, 1] - ref_lor[0, 1]) <= 2 * np.spacing(abs(ref_lor[0, 1]))


def test_ppc_pairs_rejects_other_values(G):
    from gpirt_b200 import _lib
    y = np.ones((20, 3)); y[0, 0] = -1.0
    bad = np.ones((20, 3, 1)); bad[3, 1, 0] = 0.0
    with pytest.raises(_lib.GpirtError) as e:
        G.ppc_pairs(y, bad)
    assert e.value.status == _lib.ERR_Y_VALUE
    y2 = y.copy(); y2[2, 2] = 0.5
    with pytest.raises(_lib.GpirtError) as e:
        G.ppc_pairs(y2, np.ones((20, 3, 1)))
    assert e.value.status == _lib.ERR_Y_VALUE


# ---- usefulness ------------------------------------------------------------------------------------------------------
def _two_dimensional(n, m, seed):
    """2PL responses where items 0 .. m/2 - 1 load on one trait and the rest on a second, independent one"""
    rs = np.random.Generator(np.random.Philox(seed))
    t1, t2 = rs.standard_normal(n), rs.standard_normal(n)
    a, b = rs.standard_normal(m), rs.uniform(0.5, 3.0, m)
    th = np.where(np.arange(m)[None, :] < m // 2, t1[:, None], t2[:, None])
    p = 1.0 / (1.0 + np.exp(-(a[None, :] + b[None, :] * th)))
    y = np.asfortranarray(np.where(rs.random((n, m)) < p, 1.0, -1.0))
    return dict(y=y, theta_init=rs.standard_normal(n), pm=np.zeros((2, m)), psd=np.full((2, m), 3.0),
                pstep=np.full((2, m), 0.1))


def test_pair_checks_find_a_planted_second_dimension(G):
    """Expected before the first run: a median within-cluster pair_ppp below 0.05 on the planted data.  Measured on a B200
    (n = 600, m = 40, S = 300): 0.173 (cluster medians 0.31 and 0.05, between clusters 0.59): the one-dimensional fit
    absorbs part of each cluster.  What the test pins instead is what the check is for: within-cluster pairs are flagged
    (pair_ppp < 0.05) many times as often as pairs across clusters, and unidimensional data is rarely flagged."""
    n, m, S, B = 600, 40, 300, 200
    uni = _run(G, _problem(n, m, 0.0, seed=21), S, B, store_f=False, thin=10, ppc=True, ppc_pairs=True)["ppc"]
    two = _run(G, _two_dimensional(n, m, seed=22), S, B, store_f=False, thin=10, ppc=True, ppc_pairs=True)["ppc"]
    iu = np.triu_indices(m, 1)
    h = m // 2
    within = np.array([(j < h) == (k < h) for j, k in zip(*iu)])
    p_two = two["pair_ppp"][iu]
    p_uni = uni["pair_ppp"][iu]
    extreme = np.mean((p_uni < 0.01) | (p_uni > 0.99))
    flagged_within, flagged_between = np.mean(p_two[within] < 0.05), np.mean(p_two[~within] < 0.05)
    print("planted: median within-cluster pair_ppp %.4f, between %.4f, pair_ppp < 0.05 for %.1f %% of within-cluster and "
          "%.1f %% of between-cluster pairs; unidimensional: %.1f %% of pairs outside [0.01, 0.99]"
          % (np.median(p_two[within]), np.median(p_two[~within]), 100 * flagged_within, 100 * flagged_between, 100 * extreme))
    assert np.median(p_two[within]) < 0.5 * np.median(p_two[~within])
    assert flagged_within > 0.15 and flagged_within > 5 * flagged_between
    assert extreme < 0.10
