"""Posterior predictive summaries accumulated on the device (gpirtMCMC(..., predictive=True), opts.fit) against the same
quantities computed in numpy from the stored draws of the very same chain, plus their edge cases, held-out cells, the
absence of side effects on the chain, thinning invariance, determinism and item sharding."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

CELL = dict(rtol=1e-12, atol=1e-13, equal_nan=True)
SCALARS = ("lppd", "p_waic", "elpd_waic", "waic", "se_elpd_waic", "lpd_holdout")


@pytest.fixture(scope="module")
def G():
    import gpirt_b200.sampler as g
    from gpirt_b200 import _lib
    assert _lib.load().gpirt_b200_device_count() > 0, "no CUDA device"
    return g


def _sigmoid_and_log(a):
    e = np.exp(-np.abs(a))
    return np.where(a >= 0, 1.0, e) / (1.0 + e), -(np.maximum(-a, 0.0) + np.log1p(e))


def reference(y, y_holdout, out, items=None):
    """every output from the stored draws (thin = 1: slot s = sampling iteration s), by the definitions of gpirt_b200_fit"""
    items = np.arange(y.shape[1]) if items is None else items
    y = y[:, items]
    theta = out["theta"][1:]                       # S x n
    beta = out["beta"][:, items, 1:]               # 2 x m x S
    f = out["f"][:, items, 1:]                     # n x m x S
    S = theta.shape[0]
    g = f + beta[0][None] + beta[1][None] * theta.T[:, None, :]
    obs = ~np.isnan(y)
    yh = np.full(y.shape, np.nan) if y_holdout is None else y_holdout[:, items]
    hold = ~obs & ~np.isnan(yh)
    yt = np.where(obs, y, np.where(hold, yh, 1.0))
    sig, ls = _sigmoid_and_log(yt[..., None] * g)
    sig_g, _ = _sigmoid_and_log(g)
    lpd = np.where(obs | hold, np.log(sig.mean(axis=2)), np.nan)
    pw = np.where(obs, ls.var(axis=2, ddof=1) if S > 1 else np.nan, np.nan)
    e = np.where(obs, lpd - pw, 0.0)
    lppd, p_waic = lpd[obs].sum(), pw[obs].sum()
    return dict(pred=sig_g.mean(axis=2), lpd_cell=lpd, pwaic_cell=pw, elpd_item=e.sum(axis=0), elpd_resp=e.sum(axis=1),
                lppd=lppd, p_waic=p_waic, elpd_waic=lppd - p_waic, waic=-2 * (lppd - p_waic),
                se_elpd_waic=np.sqrt(obs.sum() * np.var(e[obs], ddof=1)), lpd_holdout=lpd[hold].sum(),
                n_obs=int(obs.sum()), n_holdout=int(hold.sum()))


def _run(G, prob, S, B, seed=5, **kw):
    from gpirt_b200 import ResponseMatrix
    return G.gpirtMCMC(ResponseMatrix(prob["y"]), S, B, beta_prior_means=prob["pm"], beta_prior_sds=prob["psd"],
                       beta_proposal_sds=prob["pstep"], theta_init=prob["theta"], seed=seed, **kw)


def _check(got, want, cells=("pred", "lpd_cell", "pwaic_cell", "elpd_item", "elpd_resp")):
    for k in cells:
        assert got[k].shape == want[k].shape, k
        assert np.allclose(got[k], want[k], **CELL), (k, np.nanmax(np.abs(got[k] - want[k])))
    for k in SCALARS:
        assert np.isclose(got[k], want[k], rtol=1e-11, atol=0.0), (k, got[k], want[k])
    assert got["n_obs"] == want["n_obs"] and got["n_holdout"] == want["n_holdout"]


@pytest.mark.parametrize("n,m,missing", [(257, 37, 0.10), (640, 300, 0.05)])
def test_against_the_stored_draws(G, n, m, missing):
    """257 x 37: DMMA products, small-n sweep; 640 x 300: fixed-point products and the pipelined, graph-replayed sweep"""
    from conftest import make_problem
    prob = make_problem(n, m, seed=n, missing=missing)
    if n > 512:
        s = G.Sampler(prob["y"], prob["theta"], prob["pm"], prob["psd"], prob["pstep"], seed=5)
        s.set_timing(False)        # as gpirtMCMC runs it
        s.init_draws()
        s.sweep(3)
        assert s.uses(1) == 1 and s.uses(5) > 0, "this shape must run the fixed-point products as graph-replayed sweeps"
        s.close()
    out = _run(G, prob, 6, 2, predictive=True)
    _check(out["predictive"], reference(prob["y"], None, out))


def test_held_out_cells(G):
    from conftest import make_problem
    prob = make_problem(300, 60, seed=11, missing=0.05)
    y = prob["y"].copy(order="F")
    rs = np.random.RandomState(3)
    held = ~np.isnan(y) & (rs.rand(*y.shape) < 0.05)
    y_holdout = np.where(held, y, np.nan)
    y[held] = np.nan
    prob = dict(prob, y=np.asfortranarray(y))
    out = _run(G, prob, 5, 2, predictive=True, y_holdout=y_holdout)
    got, want = out["predictive"], reference(y, y_holdout, out)
    assert got["n_holdout"] == held.sum() > 0
    assert np.isclose(got["lpd_holdout"], want["lpd_holdout"], rtol=1e-11, atol=0.0)
    assert np.allclose(got["pred"][held], want["pred"][held], **CELL)
    _check(got, want)


def test_no_side_effects_on_the_chain(G):
    from conftest import make_problem
    prob = make_problem(200, 40, seed=4, missing=0.1)
    plain = _run(G, prob, 4, 1, f_summary=True)
    pred = _run(G, prob, 4, 1, f_summary=True, predictive=True)
    for k in ("theta", "beta", "f", "IRFs", "f_mean", "f_sd"):
        assert np.array_equal(plain[k], pred[k], equal_nan=True), k


def test_thinning_invariance_and_determinism(G):
    from conftest import make_problem
    prob = make_problem(257, 50, seed=6, missing=0.1)
    a = _run(G, prob, 8, 1, predictive=True)["predictive"]
    b = _run(G, prob, 8, 1, predictive=True, thin=4, store_f=False)["predictive"]
    c = _run(G, prob, 8, 1, predictive=True)["predictive"]
    for other in (b, c):
        for k in a:
            assert np.array_equal(a[k], other[k], equal_nan=True), k


def test_edge_cases(G):
    from conftest import make_problem
    from gpirt_b200 import _lib
    prob = make_problem(100, 20, seed=2, missing=0.1)
    p0 = _run(G, prob, 0, 2, predictive=True)["predictive"]
    for k in ("pred", "lpd_cell", "pwaic_cell", "elpd_item", "elpd_resp") + SCALARS:
        assert np.all(np.isnan(p0[k])), k
    p1 = _run(G, prob, 1, 2, predictive=True)["predictive"]
    for k in ("pwaic_cell", "elpd_item", "elpd_resp", "p_waic", "elpd_waic", "waic", "se_elpd_waic"):
        assert np.all(np.isnan(p1[k])), k
    assert np.isfinite(p1["lppd"]) and np.all(np.isfinite(p1["pred"]))
    obs = ~np.isnan(prob["y"])
    assert np.all(np.isfinite(p1["lpd_cell"][obs])) and np.all(np.isnan(p1["lpd_cell"][~obs]))
    bad = np.where(np.isnan(prob["y"]), 0.5, np.nan)
    with pytest.raises(_lib.GpirtError) as e:
        _run(G, prob, 2, 1, predictive=True, y_holdout=bad)
    assert e.value.status == _lib.ERR_Y_VALUE


def test_bench_shape_sampled_items(G):
    """C3 (4096 x 10000), every draw stored: the full numpy check on 64 random items"""
    from gpirt_b200 import synthetic
    c = synthetic.WORKLOADS["c3"]
    d = synthetic.make(c["n"], c["m"])
    prob = dict(y=d["y"], theta=d["theta_init"], pm=d["pm"], psd=d["psd"], pstep=d["pstep"])
    out = _run(G, prob, 3, 1, seed=synthetic.SEED, predictive=True)
    got = out["predictive"]
    items = np.sort(np.random.RandomState(0).choice(c["m"], 64, replace=False))
    want = reference(d["y"], None, out, items)
    for k in ("pred", "lpd_cell", "pwaic_cell"):
        assert np.allclose(got[k][:, items], want[k], **CELL), k
    assert np.allclose(got["elpd_item"][items], want["elpd_item"], **CELL)
    # per-respondent sums and totals over all items, from the device's own per-cell outputs
    obs = ~np.isnan(d["y"])
    assert got["n_obs"] == obs.sum() and got["n_holdout"] == 0
    assert np.isclose(got["lppd"], np.nansum(np.where(obs, got["lpd_cell"], np.nan)), rtol=1e-11, atol=0.0)
    assert np.isclose(got["p_waic"], np.nansum(np.where(obs, got["pwaic_cell"], np.nan)), rtol=1e-11, atol=0.0)
    assert np.allclose(got["elpd_resp"], np.where(obs, got["lpd_cell"] - got["pwaic_cell"], 0.0).sum(axis=1), rtol=1e-11, atol=1e-11)


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
    out = G.gpirtMCMC(ResponseMatrix(prob["y"][:, j0:j1]), 4, 2, beta_prior_means=prob["pm"][:, j0:j1], beta_prior_sds=prob["psd"][:, j0:j1],
                      beta_proposal_sds=prob["pstep"][:, j0:j1], theta_init=prob["theta"], seed=99, device=rank,
                      shard=(rank, world, m, j0, uid), predictive=True, store_f=False)
    np.savez(os.path.join(tmpdir, "rank%d.npz" % rank), **out["predictive"])


def test_two_gpus_item_sharded(G, tmp_path, monkeypatch):
    """GPIRT_SOLVE_MODE=1 on both sides: the sharded chain is bit-identical to the single-GPU one, so the global
    per-respondent sums and totals must agree to rounding and each rank's cells must be its item block"""
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
    full = G.gpirtMCMC(ResponseMatrix(prob["y"]), 4, 2, beta_prior_means=prob["pm"], beta_prior_sds=prob["psd"], beta_proposal_sds=prob["pstep"],
                       theta_init=prob["theta"], seed=99, device=0, predictive=True, store_f=False)["predictive"]
    for rank in range(2):
        got = dict(np.load(tmp_path / ("rank%d.npz" % rank)))
        j0, j1 = item_block(prob["y"].shape[1], rank, 2)
        assert np.allclose(got["elpd_resp"], full["elpd_resp"], rtol=1e-12, atol=1e-12)
        for k in SCALARS:
            assert np.isclose(got[k], full[k], rtol=1e-12, atol=0.0), k
        assert got["n_obs"] == full["n_obs"] and got["n_holdout"] == full["n_holdout"]
        assert np.array_equal(got["pred"], full["pred"][:, j0:j1])
        assert np.array_equal(got["elpd_item"], full["elpd_item"][j0:j1], equal_nan=True)
