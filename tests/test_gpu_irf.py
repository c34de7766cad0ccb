"""Posterior summaries of the item response functions on the grid (gpirtMCMC(..., irf_band=b, store_fstar=True),
opts.irf): the mean, sd and exact pointwise credible bands of P(y = +1 | theta*) against numpy on the f* draws of the very
same chain, the f* draws against the resident sampler, the absence of side effects, thinning invariance, determinism,
edge cases, the band computation alone on adversarial columns (irf_bands), memory release and item sharding."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

N_GRID = 1001
MOMENTS = dict(rtol=1e-12, atol=1e-13)


@pytest.fixture(scope="module")
def G():
    import gpirt_b200.sampler as g
    from gpirt_b200 import _lib
    assert _lib.load().gpirt_b200_device_count() > 0, "no CUDA device"
    return g


def plogis(x):
    return 1.0 / (1.0 + np.exp(-x))


def plan(S, band):
    """the order statistics a band needs: (r, t) for q_lo and q_hi and the tail sizes K_lo, K_hi (include/gpirt_b200.h)"""
    out = []
    for q in ((1.0 - band) / 2.0, (1.0 + band) / 2.0):
        h = (S - 1) * q
        r = min(S - 1, int(np.floor(h)))
        out.append((r, h - r))
    (r_lo, _), (r_hi, _) = out
    return out, min(S, r_lo + 2), S - r_hi


def type7(x, band):
    """x: cols x S -> (Q(q_lo), Q(q_hi)) by the definition, written out: x_(r) + t (x_(r+1) - x_(r)), no contraction"""
    S = x.shape[1]
    xs = np.sort(x, axis=1)
    res = []
    for r, t in plan(S, band)[0]:
        if r == S - 1:
            res.append(xs[:, S - 1].copy())
        else:
            x0, x1 = xs[:, r], xs[:, r + 1]
            res.append(x0 + t * (x1 - x0))
    return res


def _run(G, prob, S, B, seed=5, **kw):
    from gpirt_b200 import ResponseMatrix
    return G.gpirtMCMC(ResponseMatrix(prob["y"]), S, B, beta_prior_means=prob["pm"], beta_prior_sds=prob["psd"],
                       beta_proposal_sds=prob["pstep"], theta_init=prob["theta"], seed=seed, **kw)


def _check_against_draws(G, out, band, items=None):
    """every output of IRF_summary against numpy on the stored f* draws (thin = 1: slot s = sampling iteration s)"""
    fs = out["fstar"][:, :, 1:]
    S = fs.shape[2]
    m = fs.shape[1]
    items = np.arange(m) if items is None else items
    got = out["IRF_summary"]
    x = fs[:, items, :].reshape(-1, S, order="F")           # cols x S, cell k + 1001 j
    P = plogis(x)
    shape = (N_GRID, len(items))
    assert np.allclose(got["mean"][:, items], P.mean(axis=1).reshape(shape, order="F"), **MOMENTS)
    assert np.allclose(got["sd"][:, items], P.std(axis=1, ddof=1).reshape(shape, order="F"), **MOMENTS)
    q_lo, q_hi = type7(x, band)
    assert np.allclose(got["lower"][:, items], plogis(q_lo).reshape(shape, order="F"), rtol=1e-14, atol=0.0)
    assert np.allclose(got["upper"][:, items], plogis(q_hi).reshape(shape, order="F"), rtol=1e-14, atol=0.0)
    assert np.all(got["lower"][:, items] <= got["upper"][:, items])
    # the band computation alone on the same draws: bit for bit the written-out formula, and numpy's own quantile
    lo, hi = G.irf_bands(x, band)
    assert np.array_equal(lo, q_lo) and np.array_equal(hi, q_hi)
    for g, q in ((lo, (1.0 - band) / 2.0), (hi, (1.0 + band) / 2.0)):
        ref = np.quantile(x, q, axis=1, method="linear")
        assert np.all(np.abs(g - ref) <= 4 * np.spacing(np.abs(x).max(axis=1)))
    # the stored slots are the f* the sweeps drew: their sequential sum reproduces the IRFs
    acc = np.zeros(x.shape[0])
    for s in range(S):
        acc = acc + x[:, s]
    assert np.allclose(out["IRFs"][:, items], plogis(acc * (1.0 / S)).reshape(shape, order="F"), rtol=1e-14, atol=0.0)
    klo, khi = plan(S, band)[1:]
    assert got["band_bytes"] == 8 * N_GRID * m * (klo + khi)
    assert got["band"] == band


@pytest.mark.parametrize("n,m,S", [(257, 37, 41), (257, 37, 40), (640, 300, 41), (640, 300, 40)])
def test_against_the_chains_own_draws(G, n, m, S):
    """257 x 37: DMMA products, small-n sweep; 640 x 300: fixed-point products, graph-replayed sweeps.  Band 0.5 at
    S = 41 puts both quantiles on order statistics (t = 0), at S = 40 between two (t != 0)"""
    from conftest import make_problem
    prob = make_problem(n, m, seed=n, missing=0.05)
    if n > 512:
        s = G.Sampler(prob["y"], prob["theta"], prob["pm"], prob["psd"], prob["pstep"], seed=5)
        s.set_timing(False)
        s.init_draws()
        s.sweep(3)
        assert s.uses(1) == 1 and s.uses(5) > 0, "this shape must run the fixed-point products as graph-replayed sweeps"
        s.close()
    band = 0.5
    out = _run(G, prob, S, 2, irf_band=band, store_fstar=True, store_f=False)
    assert out["fstar"].shape == (N_GRID, m, S + 1)
    t = [t for _, t in plan(S, band)[0]]
    assert (S == 41) == (t == [0.0, 0.0])
    _check_against_draws(G, out, band)


def test_fstar_slots_equal_the_resident_sampler(G):
    from conftest import make_problem
    from gpirt_b200 import _lib
    prob = make_problem(640, 300, seed=3, missing=0.05)
    S, B = 4, 2
    out = _run(G, prob, S, B, irf_band=0.9, store_fstar=True, store_f=False)
    s = G.Sampler(prob["y"], prob["theta"], prob["pm"], prob["psd"], prob["pstep"], seed=5)
    s.set_timing(False)
    s.init_draws()
    assert np.array_equal(s.get(_lib.FSTAR), out["fstar"][:, :, 0])
    s.sweep(B)
    for k in range(1, S + 1):
        s.sweep(1, accumulate_irf=True)
        assert np.array_equal(s.get(_lib.FSTAR), out["fstar"][:, :, k]), k
    s.close()


def test_no_side_effects_on_the_chain(G):
    from conftest import make_problem
    prob = make_problem(200, 40, seed=4, missing=0.1)
    plain = _run(G, prob, 5, 1, f_summary=True, predictive=True)
    irf = _run(G, prob, 5, 1, f_summary=True, predictive=True, irf_band=0.95, store_fstar=True)
    for k in ("theta", "beta", "f", "IRFs", "f_mean", "f_sd"):
        assert np.array_equal(plain[k], irf[k], equal_nan=True), k
    for k in plain["predictive"]:
        assert np.array_equal(plain["predictive"][k], irf["predictive"][k], equal_nan=True), k


def test_thinning_invariance_and_determinism(G):
    from conftest import make_problem
    prob = make_problem(257, 50, seed=6, missing=0.1)
    a = _run(G, prob, 8, 1, irf_band=0.8, store_fstar=True, store_f=False)
    b = _run(G, prob, 8, 1, irf_band=0.8, store_fstar=True, store_f=False, thin=4)
    c = _run(G, prob, 8, 1, irf_band=0.8, store_fstar=True, store_f=False)
    for other in (b, c):
        for k in a["IRF_summary"]:
            assert np.array_equal(a["IRF_summary"][k], other["IRF_summary"][k]), k
    assert np.array_equal(a["fstar"], c["fstar"])
    assert b["fstar"].shape == (N_GRID, 50, 3)
    assert np.array_equal(b["fstar"], a["fstar"][:, :, ::4])


def test_edge_cases(G):
    from conftest import make_problem
    prob = make_problem(100, 20, seed=2, missing=0.1)
    s0 = _run(G, prob, 0, 2, irf_band=0.95, store_fstar=True)
    for k in ("mean", "sd", "lower", "upper"):
        assert s0["IRF_summary"][k].shape == (N_GRID, 20) and np.all(np.isnan(s0["IRF_summary"][k])), k
    assert s0["IRF_summary"]["band_bytes"] == 0 and s0["fstar"].shape == (N_GRID, 20, 1)
    s1 = _run(G, prob, 1, 2, irf_band=0.95, store_fstar=True)
    g = s1["IRF_summary"]
    assert np.all(np.isnan(g["sd"]))
    assert np.all(np.isfinite(g["mean"]))
    assert np.array_equal(g["lower"], g["mean"]) and np.array_equal(g["upper"], g["mean"])
    assert np.allclose(g["mean"], plogis(s1["fstar"][:, :, 1]), rtol=1e-15, atol=0.0)
    assert g["band_bytes"] == 8 * N_GRID * 20 * (1 + 1)


def _mcmc_direct(prob, S, irf, thin=1):
    """gpirt_b200_mcmc through ctypes with a hand-built gpirt_b200_irf (no host-side checks in between)"""
    from gpirt_b200 import _lib
    from gpirt_b200.sampler import make_opts
    L = _lib.load()
    y = np.asfortranarray(prob["y"])
    n, m = y.shape
    opts = make_opts(seed=1, skip_f_draws=True, thin=thin)
    opts.irf = C.pointer(irf)
    slots = S // thin + 1
    theta = np.empty((slots, n), order="F"); beta = np.empty((2, m, slots), order="F"); irfs = np.empty((N_GRID, m), order="F")
    th = np.ascontiguousarray(prob["theta"])
    pm, psd, pstep = (np.asfortranarray(prob[k]) for k in ("pm", "psd", "pstep"))
    return L.gpirt_b200_mcmc(_lib.ptr(y), n, m, _lib.ptr(th), S, 0, _lib.ptr(pm), _lib.ptr(psd), _lib.ptr(pstep), C.byref(opts),
                             _lib.ptr(theta), _lib.ptr(beta), None, _lib.ptr(irfs), _lib.PROGRESS_CB(lambda p, c: 0), None)


@pytest.mark.parametrize("band", [0.0, 1.0, 1.5, -0.5, float("nan"), float("inf")])
def test_band_outside_the_unit_interval_is_refused_by_the_library(G, band):
    from conftest import make_problem
    from gpirt_b200 import _lib
    prob = make_problem(50, 10, seed=1)
    upper = np.empty((N_GRID, 10), order="F")
    irf = _lib.Irf()
    irf.band = band
    irf.upper = _lib.ptr(upper)
    assert _mcmc_direct(prob, 2, irf) == _lib.ERR_ARG


def test_tail_buffers_that_cannot_fit_are_refused_before_the_first_sweep(G):
    import time
    from conftest import make_problem
    from gpirt_b200 import _lib
    prob = make_problem(50, 2000, seed=1)
    S, band = 10 ** 7, 0.95
    klo, khi = plan(S, band)[1:]
    want = 8 * N_GRID * 2000 * (klo + khi)
    lower = np.empty((N_GRID, 2000), order="F")
    irf = _lib.Irf()
    irf.band = band
    irf.lower = _lib.ptr(lower)
    t0 = time.perf_counter()
    rc = _mcmc_direct(prob, S, irf, thin=S)
    assert rc == _lib.ERR_NOMEM
    assert time.perf_counter() - t0 < 60.0            # 10^7 sweeps would take hours
    assert ("%d bytes" % want) in L_last_error()
    with pytest.raises(_lib.GpirtError) as e:
        _run(G, prob, S, 0, irf_band=band, store_f=False, thin=S)
    assert e.value.status == _lib.ERR_NOMEM


def L_last_error():
    from gpirt_b200 import _lib
    return _lib.load().gpirt_b200_last_error().decode()


def _adversarial_columns(S, rs):
    cols = []
    for rep in range(5):
        cols.append(rs.standard_normal(S))                                      # generic
        cols.append(rs.integers(0, 3, S).astype(np.float64) - 1.0)              # heavy ties
        cols.append(np.full(S, 0.75 * (rep - 2)))                               # all equal
        cols.append(rs.choice(np.array([-0.0, 0.0, 1.0, -1.0]), S))             # signed zeros
        cols.append(np.arange(S, dtype=np.float64) - S / 2)                     # increasing: every draw enters the upper heap
        cols.append((np.arange(S, dtype=np.float64) - S / 2)[::-1].copy())      # decreasing: every draw enters the lower heap
        cols.append(rs.choice([-1.0, 1.0], S) * 10.0 ** rs.uniform(-300, 300, S))   # 1e-300 .. 1e300
    return np.asfortranarray(np.stack(cols))                                    # 35 columns: not a multiple of 32


@pytest.mark.parametrize("S", [1, 2, 3, 31, 32, 33, 1000, 4097, 70000])
def test_irf_bands_adversarial_columns(G, S):
    rs = np.random.default_rng(S)
    x = _adversarial_columns(S, rs)
    xs = np.sort(x, axis=1)
    for band in (1e-9, 0.5, 0.95, 1.0 - 1e-9):
        lo, hi = G.irf_bands(x, band)
        want_lo, want_hi = type7(x, band)
        assert np.array_equal(lo, want_lo), (band, np.flatnonzero(lo != want_lo))   # values: -0.0 == +0.0
        assert np.array_equal(hi, want_hi), (band, np.flatnonzero(hi != want_hi))
        scale = np.maximum(np.abs(xs[:, 0]), np.abs(xs[:, -1]))
        for g, q in ((lo, (1.0 - band) / 2.0), (hi, (1.0 + band) / 2.0)):
            ref = np.quantile(x, q, axis=1, method="linear")
            assert np.all(np.abs(g - ref) <= 4 * np.spacing(scale)), (band, q)


def test_irf_bands_times_its_kernels(G):
    x = _adversarial_columns(100, np.random.default_rng(0))
    lo, hi, (ms_update, ms_finish) = G.irf_bands(x, 0.9, reps=2)
    assert ms_update > 0.0 and ms_finish > 0.0
    assert np.array_equal(lo, type7(x, 0.9)[0])


def test_tail_buffers_are_returned_after_the_call(G):
    import torch
    from conftest import make_problem
    prob = make_problem(100, 2000, seed=8, missing=0.0)
    S = 1500
    klo, khi = plan(S, 0.95)[1:]
    assert 8 * N_GRID * 2000 * (klo + khi) >= 1 << 30
    _run(G, prob, S, 0, store_f=False, thin=S)
    torch.cuda.synchronize()
    free_without = torch.cuda.mem_get_info()[0]
    out = _run(G, prob, S, 0, store_f=False, thin=S, irf_band=0.95)
    assert out["IRF_summary"]["band_bytes"] >= 1 << 30
    torch.cuda.synchronize()
    free_with = torch.cuda.mem_get_info()[0]
    assert abs(free_with - free_without) <= 64 << 20, (free_without, free_with)


def test_bench_shape_sampled_items(G):
    """C3 (4096 x 10000): the check against the chain's own draws on 64 random items"""
    from gpirt_b200 import synthetic
    c = synthetic.WORKLOADS["c3"]
    d = synthetic.make(c["n"], c["m"])
    prob = dict(y=d["y"], theta=d["theta_init"], pm=d["pm"], psd=d["psd"], pstep=d["pstep"])
    out = _run(G, prob, 3, 1, seed=synthetic.SEED, irf_band=0.95, store_fstar=True, store_f=False)
    items = np.sort(np.random.RandomState(0).choice(c["m"], 64, replace=False))
    _check_against_draws(G, out, 0.95, items)


def _shard_worker(rank, world, tmpdir):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import time
    os.environ["GPIRT_SOLVE_MODE"] = "1"
    import gpirt_b200.sampler as G
    from conftest import make_problem
    from gpirt_b200 import ResponseMatrix
    from gpirt_b200.sharding import item_block
    uid_path = os.path.join(tmpdir, "uid")
    if rank == 0:
        with open(uid_path + ".tmp", "wb") as fh:
            fh.write(G.nccl_unique_id())
        os.replace(uid_path + ".tmp", uid_path)
    while not os.path.exists(uid_path):
        time.sleep(0.05)
    uid = open(uid_path, "rb").read()
    prob = make_problem(300, 90, seed=5, missing=0.05)
    m = prob["y"].shape[1]
    j0, j1 = item_block(m, rank, world)
    out = G.gpirtMCMC(ResponseMatrix(prob["y"][:, j0:j1]), 6, 2, beta_prior_means=prob["pm"][:, j0:j1],
                      beta_prior_sds=prob["psd"][:, j0:j1], beta_proposal_sds=prob["pstep"][:, j0:j1], theta_init=prob["theta"],
                      seed=99, device=rank, shard=(rank, world, m, j0, uid), irf_band=0.9, store_fstar=True, store_f=False)
    res = {k: v for k, v in out["IRF_summary"].items() if isinstance(v, np.ndarray)}
    np.savez(os.path.join(tmpdir, "rank%d.npz" % rank), fstar=out["fstar"], IRFs=out["IRFs"], **res)


def test_two_gpus_item_sharded(G, tmp_path, monkeypatch):
    """GPIRT_SOLVE_MODE=1 on both sides: the sharded chain is bit-identical to the single-GPU one, so every output of
    each rank must be its item block of the single-GPU run, bit for bit"""
    from gpirt_b200 import _lib
    from gpirt_b200.sharding import item_block
    from gpirt_b200 import ResponseMatrix
    from conftest import make_problem
    if _lib.load().gpirt_b200_device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    mp.spawn(_shard_worker, args=(2, str(tmp_path)), nprocs=2, join=True)
    monkeypatch.setenv("GPIRT_SOLVE_MODE", "1")
    prob = make_problem(300, 90, seed=5, missing=0.05)
    full = G.gpirtMCMC(ResponseMatrix(prob["y"]), 6, 2, beta_prior_means=prob["pm"], beta_prior_sds=prob["psd"],
                       beta_proposal_sds=prob["pstep"], theta_init=prob["theta"], seed=99, device=0, irf_band=0.9,
                       store_fstar=True, store_f=False)
    want = dict(full["IRF_summary"], fstar=full["fstar"], IRFs=full["IRFs"])
    for rank in range(2):
        got = dict(np.load(tmp_path / ("rank%d.npz" % rank)))
        j0, j1 = item_block(prob["y"].shape[1], rank, 2)
        for k in ("mean", "sd", "lower", "upper", "fstar", "IRFs"):
            assert np.array_equal(got[k], want[k][:, j0:j1]), (rank, k)
