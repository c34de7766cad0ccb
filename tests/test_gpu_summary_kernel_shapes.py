"""Every launch shape of the PSIS-LOO finish and of the chain diagnostics, up to the largest sizes they are built for,
against the numpy port of the definitions (tests/psis_loo_numpy.py) and the host formulas of gpirt_b200_theta_diagnostics.

k_loo_finish (loo.cu, loo_finish_shape) runs one warp per cell, and its shape follows from the number of draws S:

  M = ceil(min(0.2 S, 3 sqrt S))     tail draws
  P = the power of two >= M + 1      the cell's heap of K = M + 1 values, padded for the bitonic sort
  G = 30 + floor(sqrt M)             profile grid points, ceil(G / 32) per lane
  W = min(8, 6144 // (P + M + G + 3)) warps (cells) per CTA, in 48 KiB of shared memory (at least 1)

The cooperative load indexes shared memory by e / W and e - k W, so W that is not a power of two and a ragged last CTA
matter.  K is built up to 8192 (M = 8191, S = 7 454 720); larger S is refused.  The cases run the first S of every
(P, W, ceil(G / 32)) the build has, and S = 7225 on the other side of W = 8 -> 7.

k_chain_diag (kernels.cu) stages each chain in dynamic shared memory when 8 S + 1024 bytes fit under the device's opt-in
limit per block (chain_diag_smem_bytes), and otherwise reads it from global memory: S_max = (optin - 1024) // 8 is the
last staged S.  The cases run S_max, S_max + 1 and S_max + 3 (odd: the middle draw is in neither half), with walks of
Geyer's initial sequence longer than one block of 8 lag pairs, and C = 32 chains, the most opts.chains takes."""
import time

import numpy as np
import pytest

import psis_loo_numpy as P
from test_gpu_chains import _assert_chain_equals_solo, _check_diagnostics, _split_rhat, _thetas
from test_gpu_chains import _run as _run_chains
from test_gpu_loo import _check_against_draws, _check_cells
from test_gpu_loo import _problem as _loo_problem
from test_gpu_loo import _run as _run_loo

pytestmark = pytest.mark.gpu

N_GRID = 1001
LOO_S_MAX = 7454720          # loo.cuh: LOO_MAX_HEAP = 8192 = M + 1
DIAG_PAIRS_PER_BLOCK = 8     # kernels.cu: DIAG_WARPS lag pairs per block of the Geyer walk


@pytest.fixture(scope="module")
def G():
    import gpirt_b200.sampler as g
    from gpirt_b200 import _lib
    assert _lib.load().gpirt_b200_device_count() > 0, "no CUDA device"
    return g


# ---- A. the PSIS-LOO finish through psis_loo() ----------------------------------------------------------------------
def finish_shape(S):
    """(M, P, G, W) of k_loo_finish at S draws, restating loo_finish_shape() in loo.cu (S may be a numpy array)"""
    S = np.asarray(S, dtype=np.int64)
    M = np.ceil(np.minimum(0.2 * S, 3.0 * np.sqrt(S))).astype(np.int64)
    Pw = np.ones_like(M)
    while np.any(Pw < M + 1):
        Pw = np.where(Pw < M + 1, 2 * Pw, Pw)
    Gp = 30 + np.floor(np.sqrt(M)).astype(np.int64)
    W = np.clip(6144 // (Pw + M + Gp + 3), 1, 8)
    return M, Pw, Gp, W


def _first_s_of_every_shape():
    """the first S of every (P, W, ceil(G / 32)) from S = 1 up to the largest built S"""
    S = np.arange(1, LOO_S_MAX + 1, dtype=np.int64)
    _, Pw, Gp, W = finish_shape(S)
    key = (Pw * 16 + W) * 8 + (Gp + 31) // 32
    return [int(s) for s in S[np.r_[0, np.flatnonzero(np.diff(key)) + 1]]]


# the first S of each shape from S = 6 (S = 1 is run by test_gpu_loo), and 7225, the last S with W = 8 before 7226
LOO_CASES = [6, 16, 36, 41, 76, 156, 442, 1793, 7225, 7226, 11026, 23308, 29014, 102401, 116282, 166465, 465579,
             1863226, 2238017, LOO_S_MAX]
WIDE_COLS = 31              # 4 x 8 adversarial columns less one: 31 is no multiple of W = 7, 6, 5, 3 or 2


def _loo_id(S):
    _, Pw, Gp, W = (int(v) for v in finish_shape(S))
    return "S%d-P%d-W%d-grid%d" % (S, Pw, W, -(-Gp // 32))


def test_cases_cover_every_finish_shape():
    assert _first_s_of_every_shape()[1:] == sorted(set(LOO_CASES) - {7225, LOO_S_MAX})
    M, Pw, Gp, W = (int(v) for v in finish_shape(LOO_S_MAX))
    assert (M, Pw, Gp, W) == (8191, 8192, 120, 1)
    assert int(finish_shape(LOO_S_MAX + 1)[0]) == 8192
    assert [int(finish_shape(S)[3]) for S in (7225, 7226)] == [8, 7]
    for S in LOO_CASES:        # the columns leave the last CTA ragged wherever W is 2 ... 7
        W = int(finish_shape(S)[3])
        if 1 < W < 8:
            assert WIDE_COLS % W != 0


def _reference(ll):
    """P.psis_loo in blocks of rows, so that its temporaries stay near 128 MB at any S"""
    rows = max(1, (16 << 20) // max(1, ll.shape[1]))
    parts = [P.psis_loo(ll[r:r + rows]) for r in range(0, ll.shape[0], rows)]
    return {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}


@pytest.mark.parametrize("S", LOO_CASES, ids=_loo_id)
def test_psis_loo_finish_shape_against_numpy(G, S):
    M, Pw, Gp, W = (int(v) for v in finish_shape(S))
    rs = np.random.default_rng(S)
    # 31 columns (a ragged last CTA wherever W < 8) up to S = 116 282, beyond it one column of each kind (8 S doubles:
    # 477 MB at the largest S)
    ll = P.adversarial(S, rs)[:WIDE_COLS] if S <= 116282 else P.adversarial(S, rs, reps=1)
    e, p, k = G.psis_loo(ll)
    ref = _reference(ll)
    _check_cells(e, p, k, ref)
    kinds = np.array([P.ADVERSARIAL_KINDS[i % 8] for i in range(ll.shape[0])])
    print("S = %d: M %d, P %d, G %d, W %d, %d columns; k of the Pareto 1.5 columns %s"
          % (S, M, Pw, Gp, W, ll.shape[0], np.array2string(k[kinds == "Pareto 1.5"], precision=3)))
    if M >= 5:                 # the tail fit ran: some cells are smoothed, the constant ones are not
        assert np.any(np.isfinite(k)) and np.any(np.isinf(k))
    if S >= 1793:
        assert np.any(k[kinds == "Pareto 1.5"] > 1.0)


def test_psis_loo_beyond_the_largest_heap_is_refused(G):
    from gpirt_b200 import _lib
    with pytest.raises(_lib.GpirtError) as exc:
        G.psis_loo(np.full((1, LOO_S_MAX + 1), -0.5))
    assert exc.value.status == _lib.ERR_ARG
    assert "8191" in str(exc.value)


# ---- B. PSIS-LOO in gpirtMCMC(loo=True) at W < 8 with missing cells ---------------------------------------------------
N_B, M_B = 37, 11            # 407 cells: neither W = 7 nor W = 3 divides them


@pytest.mark.parametrize("S", [7226, 29014], ids=_loo_id)
def test_sampler_loo_at_fewer_than_eight_cells_per_cta(G, S):
    W = int(finish_shape(S)[3])
    assert W < 8 and (N_B * M_B) % W != 0
    prob = _loo_problem(N_B, M_B, 0.1, seed=S)
    y = prob["y"]
    miss = np.isnan(y).ravel(order="F")
    assert miss.any() and (~miss).any()
    # missing cells at several positions within their CTA, so that the per-warp obs[] flags are exercised
    assert len(set(np.flatnonzero(miss) % W)) > 1
    out = _run_loo(G, prob, S, 2, loo=True, predictive=True)
    ref = _check_against_draws(out, y)
    assert np.any(np.isfinite(ref["k"])) and np.any(np.isfinite(out["loo"]["pareto_k"]))
    lo, pr = out["loo"], out["predictive"]
    obs = ~np.isnan(y)
    back = lo["p_loo_cell"][obs] + lo["elpd_loo_cell"][obs]
    lpd = pr["lpd_cell"][obs]
    scale = np.maximum(np.abs(lpd), np.abs(lo["elpd_loo_cell"][obs]))
    assert np.all(np.abs(back - lpd) <= 2 * np.spacing(scale)), np.abs(back - lpd).max()
    assert lo["n_obs"] == pr["n_obs"] == int(obs.sum())


def test_sampler_loo_beyond_the_largest_heap_is_refused_before_the_first_sweep(G):
    from gpirt_b200 import _lib
    prob = _loo_problem(N_B, M_B, 0.1, seed=1)
    S = LOO_S_MAX + 1
    calls = []

    def progress(pct):          # a sweep that started would be interrupted at once
        calls.append(pct)
        return True
    t0 = time.perf_counter()
    with pytest.raises(_lib.GpirtError) as exc:
        _run_loo(G, prob, S, 2, loo=True, thin=S, store_f=False, progress=progress)
    assert time.perf_counter() - t0 < 30.0
    assert exc.value.status == _lib.ERR_ARG
    assert "8191" in str(exc.value)
    assert calls == []


# ---- C. chain diagnostics on both sides of the staging switch --------------------------------------------------------
def _staged_s_max():
    """the largest S whose chain k_chain_diag stages in shared memory: 8 S + 1024 bytes within the opt-in limit"""
    import torch
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    return (optin - 1024) // 8


def geyer_pairs(x):
    """lag pairs Geyer's initial positive sequence adds before it stops (the walk of k_chain_diag and chain_ess)"""
    T = x.size
    y = x - x.mean()
    f = np.fft.rfft(y, 2 * T)
    ac = np.fft.irfft(f * np.conj(f), 2 * T)[:T] / T
    if not ac[0] > 0.0:
        return 0
    h = T // 2                                       # pairs k with 2 k + 1 < T
    pairs = (ac[0:2 * h:2] + ac[1:2 * h:2]) / ac[0]
    stop = np.flatnonzero(pairs <= 0.0)
    return int(stop[0]) if stop.size else h


N_C, M_C = 40, 12
CONST_ITEM, SLOW_ITEMS = 3, (4, 5)


def _diag_problem():
    from conftest import make_problem
    prob = make_problem(N_C, M_C, seed=N_C + M_C, missing=0.05)
    pstep = prob["pstep"].copy()
    pstep[:, CONST_ITEM] = 0.0                       # this beta never moves: NaN R-hat and ESS
    pstep[:, list(SLOW_ITEMS)] = 1e-3                # strongly autocorrelated: Geyer walks of many blocks
    prob["pstep"] = pstep
    return prob


BETA_KEEP = np.setdiff1d(np.arange(2 * M_C), [2 * CONST_ITEM, 2 * CONST_ITEM + 1])


@pytest.mark.parametrize("offset", [0, 1, 3], ids=["staged-S_max", "global-S_max+1", "global-odd-S_max+3"])
def test_chain_diagnostics_on_both_sides_of_the_staging_switch(G, offset):
    s_max = _staged_s_max()
    assert s_max < 100000, "S_max = %d: the cases would no longer be cheap" % s_max
    S = s_max + offset
    prob = _diag_problem()
    out = _run_chains(G, prob, S, 2, theta_init=_thetas(prob, 2), seed=5, chains=2, chain_diagnostics=True,
                      store_f=False)
    assert np.all(out["beta"][:, CONST_ITEM] == out["beta"][:, CONST_ITEM, :1])
    d = out["diagnostics"]
    assert np.all(np.isnan(d["beta_rhat"][:, CONST_ITEM])) and np.all(np.isnan(d["beta_ess"][:, CONST_ITEM]))
    walks = [geyer_pairs(out["beta"][i, j, 1:, c]) for i in range(2) for j in SLOW_ITEMS for c in range(2)]
    print("S = %d (S_max = %d): longest beta walk %d lag pairs, theta walks up to %d"
          % (S, s_max, max(walks), max(geyer_pairs(out["theta"][1:, i, c]) for i in range(N_C) for c in range(2))))
    assert max(walks) > 8 * DIAG_PAIRS_PER_BLOCK, walks
    _check_diagnostics(G, out, 2, M_C, beta_keep=BETA_KEEP)


def test_chain_diagnostics_of_thirty_two_chains(G):
    C_, S = 32, 41
    prob = _diag_problem()
    th = _thetas(prob, C_)
    out = _run_chains(G, prob, S, 2, theta_init=th, seed=11, chains=C_, chain_diagnostics=True, store_f=False)
    _check_diagnostics(G, out, C_, M_C, beta_keep=BETA_KEEP)
    d = out["diagnostics"]
    assert np.all(np.isnan(d["beta_rhat"][:, CONST_ITEM])) and np.all(np.isnan(d["beta_ess"][:, CONST_ITEM]))
    xs = []
    for c in range(C_):
        solo = _run_chains(G, prob, S, 2, theta_init=th[:, c].copy(), seed=11 + c, store_f=False, store_fstar=True)
        _assert_chain_equals_solo(out, solo, c, False)
        xs.append(1.0 / (1.0 + np.exp(-solo["fstar"][:, :, 1:].reshape(-1, S, order="F"))))
    want = _split_rhat(xs).reshape(N_GRID, M_C, order="F")
    got = d["irf_rhat"]
    # as test_gpu_chains: compare the cells whose within-half sd is at least 1e-4
    sd = np.sqrt(np.mean([np.concatenate([x[:, :S // 2], x[:, S - S // 2:]], axis=1).var(axis=1) for x in xs], axis=0))
    ok = (sd >= 1e-4).reshape(N_GRID, M_C, order="F")
    assert ok.mean() > 0.5
    assert np.allclose(got[ok], want[ok], rtol=1e-10, atol=0.0)
