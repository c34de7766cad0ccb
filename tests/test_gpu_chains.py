"""Several chains in one gpirtMCMC call (chains=C, opts.chains): every chain bit for bit equal to a call of its own with
the same seed and theta_init, on every sweep route; the split-R-hat and ESS of theta and beta computed on the device against
gpirt_b200_theta_diagnostics on the returned draws; the IRF split-R-hat against numpy on the f* draws of the solo chains;
thinning invariance, determinism, no side effects of the diagnostics; refusals, interrupts and the memory left behind."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N_GRID = 1001


@pytest.fixture(scope="module")
def G():
    import gpirt_b200.sampler as g
    from gpirt_b200 import _lib
    assert _lib.load().gpirt_b200_device_count() > 0, "no CUDA device"
    return g


def _senate116():
    import warnings
    import gpirt_b200
    from conftest import make_problem
    codes, _, _ = gpirt_b200.senate116()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        y = np.asfortranarray(np.asarray(gpirt_b200.response_matrix(codes), dtype=np.float64))
    prob = make_problem(4, y.shape[1])
    prob["y"] = y
    return prob


def _problem(n, m):
    from conftest import make_problem
    return _senate116() if (n, m) == (100, 418) else make_problem(n, m, seed=n + m, missing=0.05)


def _run(G, prob, S, B, **kw):
    from gpirt_b200 import ResponseMatrix
    return G.gpirtMCMC(ResponseMatrix(prob["y"]), S, B, beta_prior_means=prob["pm"], beta_prior_sds=prob["psd"],
                       beta_proposal_sds=prob["pstep"], **kw)


def _thetas(prob, C_):
    n = prob["y"].shape[0]
    return np.asfortranarray(np.random.RandomState(n + C_).randn(n, C_))


def _assert_chain_equals_solo(got, solo, c, store_f):
    assert np.array_equal(got["theta"][..., c], solo["theta"]), "theta of chain %d" % c
    assert np.array_equal(got["beta"][..., c], solo["beta"]), "beta of chain %d" % c
    assert np.array_equal(got["IRFs"][..., c], solo["IRFs"]), "IRFs of chain %d" % c
    if store_f:
        assert np.array_equal(got["f"][..., c], solo["f"]), "f of chain %d" % c


# (n, m, C, environment, path): 100 x 418 = senate116 (small-n sweep), 257 x 37 (odd n, DMMA products), 640 x 300
# (pipelined, graph-replayed, fixed-point products), 1152 x 260 on the substitution route, 1024 x 2000 = C2
CASES = [(100, 418, 4, None, None), (257, 37, 3, None, None), (640, 300, 2, None, (5, 1)),
         (1152, 260, 2, "1", (4, 1)), (1024, 2000, 2, None, (1, 1))]


@pytest.mark.parametrize("store_f", [True, False])
@pytest.mark.parametrize("thin", [1, 7])
@pytest.mark.parametrize("n,m,C_,solve_mode,path", CASES)
def test_every_chain_equals_its_solo_call(G, n, m, C_, solve_mode, path, thin, store_f, monkeypatch):
    if solve_mode is not None:
        monkeypatch.setenv("GPIRT_SOLVE_MODE", solve_mode)   # read in create(): every chain takes this route
    prob = _problem(n, m)
    if path is not None:   # the route this shape takes, on a resident sampler of the same shape
        s = G.Sampler(prob["y"], prob["theta"] if prob["theta"].size == n else np.zeros(n), prob["pm"], prob["psd"],
                      prob["pstep"], seed=5)
        s.set_timing(False)
        s.init_draws()
        s.sweep(3)
        assert s.uses(path[0]) >= path[1], "this shape must run feature %d" % path[0]
        s.close()
    S, B = 10, 3
    th = _thetas(prob, C_)
    got = _run(G, prob, S, B, theta_init=th, seed=77, chains=C_, thin=thin, store_f=store_f)
    slots = S // thin + 1
    assert got["theta"].shape == (slots, n, C_) and got["beta"].shape == (2, m, slots, C_)
    assert got["IRFs"].shape == (N_GRID, m, C_)
    if store_f:
        assert got["f"].shape == (n, m, slots, C_)
    for c in range(C_):
        solo = _run(G, prob, S, B, theta_init=th[:, c].copy(), seed=77 + c, thin=thin, store_f=store_f)
        _assert_chain_equals_solo(got, solo, c, store_f)


def test_one_chain_equals_the_call_without_chains(G):
    prob = _problem(257, 37)
    th = _thetas(prob, 1)
    got = _run(G, prob, 9, 2, theta_init=th, seed=[123], chains=1)
    solo = _run(G, prob, 9, 2, theta_init=th[:, 0].copy(), seed=123)
    _assert_chain_equals_solo(got, solo, 0, True)


def test_seed_sequence_is_used_as_given(G):
    prob = _problem(257, 37)
    th = _thetas(prob, 2)
    got = _run(G, prob, 5, 1, theta_init=th, seed=[9, 4], chains=2, store_f=False)
    for c, sd in enumerate([9, 4]):
        _assert_chain_equals_solo(got, _run(G, prob, 5, 1, theta_init=th[:, c].copy(), seed=sd, store_f=False), c, False)


def _beta_draws(beta_c):
    """2 x m x slots of one chain without slot 0 -> draws x 2m (column p = i + 2 j)"""
    two, m, slots = beta_c.shape
    return beta_c[:, :, 1:].reshape(two * m, slots - 1, order="F").T


def _host_diag(G, draws_per_chain):
    if draws_per_chain[0].shape[0] < 4:
        p = draws_per_chain[0].shape[1]
        return np.full(p, np.nan), np.full(p, np.nan)
    return G.theta_diagnostics(draws_per_chain)


def _check_diagnostics(G, out, C_, m, beta_keep=None):
    """beta_keep: the beta parameters (index i + 2 j) to compare; a constant chain is left out, because the host's
    mean of S equal values need not give the value back, so its spread there is rounding noise instead of exactly zero"""
    d = out["diagnostics"]
    keep = np.arange(2 * m) if beta_keep is None else beta_keep
    rt, et = _host_diag(G, [out["theta"][1:, :, c] for c in range(C_)])
    rb, eb = _host_diag(G, [_beta_draws(out["beta"][..., c]) for c in range(C_)])
    for got, want, tol in ((d["theta_rhat"], rt, 1e-12), (d["theta_ess"], et, 1e-9),
                           (d["beta_rhat"].ravel(order="F")[keep], rb[keep], 1e-12),
                           (d["beta_ess"].ravel(order="F")[keep], eb[keep], 1e-9)):
        assert np.array_equal(np.isnan(got), np.isnan(want))
        assert np.allclose(got, want, rtol=tol, atol=0.0, equal_nan=True)
    assert d["beta_rhat"].shape == (2, m) and d["irf_rhat"].shape == (N_GRID, m)


@pytest.mark.parametrize("n,m,C_,S", [(100, 418, 3, 40), (257, 37, 2, 41), (640, 300, 2, 25), (257, 37, 2, 3),
                                      (257, 37, 2, 0)])
def test_theta_and_beta_diagnostics_equal_the_host_formulas(G, n, m, C_, S):
    prob = _problem(n, m)
    out = _run(G, prob, S, 2, theta_init=_thetas(prob, C_), seed=3, chains=C_, chain_diagnostics=True, store_f=False)
    _check_diagnostics(G, out, C_, m)
    d = out["diagnostics"]
    if S < 4:
        for k in ("theta_rhat", "theta_ess", "beta_rhat", "beta_ess", "irf_rhat"):
            assert np.all(np.isnan(d[k])), k
        assert d["diag_bytes"] == 0
    else:
        assert d["diag_bytes"] == 8 * S * (n + 2 * m) * C_ + 32 * N_GRID * m * C_
        assert np.all(np.isfinite(d["theta_rhat"])) and np.all(d["theta_ess"] > 0)


def test_constant_beta_chain_gives_nan(G):
    prob = dict(_problem(257, 37))
    pstep = prob["pstep"].copy()
    pstep[:, 5] = 0.0   # item 5's beta never moves
    prob["pstep"] = pstep
    out = _run(G, prob, 30, 2, theta_init=_thetas(prob, 2), seed=8, chains=2, chain_diagnostics=True, store_f=False)
    assert np.all(out["beta"][:, 5, :, :] == out["beta"][:, 5, :1, :])
    _check_diagnostics(G, out, 2, 37, beta_keep=np.setdiff1d(np.arange(74), [10, 11]))
    d = out["diagnostics"]
    assert np.all(np.isnan(d["beta_rhat"][:, 5])) and np.all(np.isnan(d["beta_ess"][:, 5]))
    assert np.all(np.isfinite(np.delete(d["beta_rhat"], 5, axis=1)))


def _split_rhat(chains_x):
    """numpy split-R-hat over the last axis of each chain's (cols x S) draws"""
    S = chains_x[0].shape[1]
    half = S // 2
    halves = []
    for x in chains_x:
        halves += [x[:, :half], x[:, S - half:]]
    means = np.stack([h.mean(axis=1) for h in halves])
    W = np.stack([h.var(axis=1, ddof=1) for h in halves]).mean(axis=0)
    Bv = half * means.var(axis=0, ddof=1)
    var_plus = (half - 1) / half * W + Bv / half
    return np.sqrt(var_plus / W)


@pytest.mark.parametrize("n,m,C_,S", [(257, 37, 3, 40), (640, 300, 2, 33)])
def test_irf_rhat_equals_numpy_on_the_solo_fstar_draws(G, n, m, C_, S):
    prob = _problem(n, m)
    th = _thetas(prob, C_)
    out = _run(G, prob, S, 2, theta_init=th, seed=11, chains=C_, chain_diagnostics=True, store_f=False)
    xs = []
    for c in range(C_):
        solo = _run(G, prob, S, 2, theta_init=th[:, c].copy(), seed=11 + c, store_f=False, store_fstar=True)
        assert np.array_equal(solo["IRFs"], out["IRFs"][..., c])
        xs.append(1.0 / (1.0 + np.exp(-solo["fstar"][:, :, 1:].reshape(-1, S, order="F"))))
    want = _split_rhat(xs).reshape(N_GRID, m, order="F")
    got = out["diagnostics"]["irf_rhat"]
    # where P saturates at 0 or 1 its spread is a few ulps, and any two summation orders disagree in the leading digits of
    # W: compare the cells whose within-half sd is at least 1e-4 (relative rounding of W well below 1e-10 there)
    sd = np.sqrt(np.mean([np.concatenate([x[:, :S // 2], x[:, S - S // 2:]], axis=1).var(axis=1) for x in xs], axis=0))
    ok = (sd >= 1e-4).reshape(N_GRID, m, order="F")
    assert ok.mean() > 0.5
    assert np.allclose(got[ok], want[ok], rtol=1e-10, atol=0.0)


def test_thinning_determinism_and_no_side_effects(G):
    prob = _problem(257, 37)
    th = _thetas(prob, 3)
    kw = dict(theta_init=th, seed=21, chains=3, store_f=False)
    a = _run(G, prob, 30, 3, chain_diagnostics=True, **kw)
    b = _run(G, prob, 30, 3, chain_diagnostics=True, **kw)
    t5 = _run(G, prob, 30, 3, chain_diagnostics=True, thin=5, **kw)
    plain = _run(G, prob, 30, 3, **kw)
    for k in ("theta_rhat", "theta_ess", "beta_rhat", "beta_ess", "irf_rhat", "diag_bytes"):
        assert np.array_equal(a["diagnostics"][k], b["diagnostics"][k], equal_nan=True), k
        assert np.array_equal(a["diagnostics"][k], t5["diagnostics"][k], equal_nan=True), k
    for k in ("theta", "beta", "IRFs"):
        assert np.array_equal(a[k], b[k]) and np.array_equal(a[k], plain[k]), k
    assert np.array_equal(t5["theta"], a["theta"][::5]) and np.array_equal(t5["beta"], a["beta"][:, :, ::5])
    assert "diagnostics" not in plain


def _direct(G, prob, S, chains, cb=None, thin=1):
    """gpirt_b200_mcmc through ctypes, so that the Chains struct (diag_bytes) survives a refused call"""
    from gpirt_b200 import _lib
    L = _lib.load()
    y = prob["y"]
    n, m = y.shape
    C_ = chains.chains
    th = _thetas(prob, C_)
    opts = G.make_opts(seed=1, skip_f_draws=True, thin=thin)
    opts.chains = C.pointer(chains)
    slots = S // thin + 1
    theta = np.empty((slots, n, C_), order="F"); beta = np.empty((2, m, slots, C_), order="F")
    irf = np.empty((N_GRID, m, C_), order="F")
    cbf = _lib.PROGRESS_CB(cb or (lambda pct, ctx: 0))
    pm, psd, pstep = (np.asfortranarray(prob[k]) for k in ("pm", "psd", "pstep"))
    rc = L.gpirt_b200_mcmc(_lib.ptr(y), n, m, _lib.ptr(th), S, 0, _lib.ptr(pm), _lib.ptr(psd), _lib.ptr(pstep), C.byref(opts), _lib.ptr(theta), _lib.ptr(beta), None, _lib.ptr(irf),
                           cbf, None)
    return rc, L.gpirt_b200_last_error().decode()


def test_diagnostics_beyond_free_memory_are_refused_before_the_first_sweep(G):
    from gpirt_b200 import _lib
    prob = _problem(100, 418)
    n, m = prob["y"].shape
    rt = np.empty(n)
    ch = _lib.Chains(chains=2)
    ch.theta_rhat = _lib.ptr(rt)
    S = 400_000_000                     # 8 S (n + 2m) C = 6 TB of traces
    calls = []

    def cb(pct, ctx):                   # a sweep that started would be interrupted at once
        calls.append(pct)
        return 1
    rc, msg = _direct(G, prob, S, ch, cb=cb, thin=S)
    assert rc == _lib.ERR_NOMEM, msg
    assert calls == []
    assert ch.diag_bytes == 8 * S * (n + 2 * m) * 2
    assert "need" in msg


def test_interrupt_stops_every_chain_and_the_next_call_succeeds(G):
    from gpirt_b200 import _lib
    prob = _problem(257, 37)
    calls = []

    def cb(pct, ctx):
        calls.append(pct)
        return 1 if len(calls) > 5 else 0
    ch = _lib.Chains(chains=3)
    rc, msg = _direct(G, prob, 200, ch, cb=cb)
    assert rc == _lib.ERR_INTERRUPT
    assert "chain" in msg and "interrupted" in msg
    assert len(calls) == 6 and calls[:2] == [0.0, 100.0 / 200]
    ch2 = _lib.Chains(chains=3)
    rc, msg = _direct(G, prob, 20, ch2)
    assert rc == _lib.OK, msg


def test_device_memory_is_returned_after_four_chains_at_c2(G):
    import torch
    from gpirt_b200 import _lib
    prob = _problem(1024, 2000)
    torch.cuda.init()
    torch.cuda.mem_get_info()
    _run(G, prob, 2, 1, theta_init=_thetas(prob, 1)[:, 0].copy(), seed=2, store_f=False)   # warm one-time state
    _lib.check(_lib.load().gpirt_b200_release_memory())
    before = torch.cuda.mem_get_info()[0]
    out = _run(G, prob, 9, 2, theta_init=_thetas(prob, 4), seed=2, chains=4, store_f=False, chain_diagnostics=True)
    after = torch.cuda.mem_get_info()[0]
    assert out["theta"].shape[2] == 4
    assert abs(before - after) <= 256 << 20, (before, after)
