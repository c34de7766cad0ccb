"""The sweep bench.py times, compared with the oracle step by step at the benchmark shapes: C3 (4096 x 10000) with 0 %
and 5 % missing cells and C5 (16384 x 20000) with 5 %.

The timed sweep differs from the one-step-at-a-time sweep of test_gpu_bench_shapes.py: it is replayed as one CUDA graph;
its ESS uses the proposals nu that the previous sweep accumulated slice by slice behind its Cholesky panels (fixed-point
launches over L sliced at the fixed scale |L| < 2, every slice after the first added onto nu: 2 slices at C3, 3 at C5 on
the substitution route); its K* solves were left by the previous sweep and run beside its ESS (C3 through L^-1, C5 as a
backward pass on the 1024-block inverses built behind the panels); and its beta step runs on a side stream.  Given
theta_t, beta_t, f_t and L_t every item is independent and every respondent's grid draw is independent given f*, so the
tile strata of tests/bench_strata.py are checked against the oracle with the same addressed variates (stream maps).

Tolerances: those of test_c3_sampled_items_and_respondents_against_the_oracle (ESS counts and theta indices identical,
f 1e-9, f* sd 1e-8, f* 1e-7 relative, logP 1e-12 relative, beta 1e-12); nu within the fixed-point bound summed over the
slices; the factor bit for bit equal to the stand-alone factorisation and within test_gpu_large_n.py's residual bound."""
import time

import numpy as np
import pytest

import bench_strata as B

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
ITEM_CTA, ITEM_PERSISTENT, ITEM_STREAM = 0, 1, 2
# (K* solve route, slices of the pipelined nu = L Z, ESS launch shape, beta launch shape) per workload, as
# rebuild_pipelined / ess_only in sampler.cu choose them.  Slices: 16 panels each through L^-1 (32 panels at C3); on the
# substitution route they end at half the panels, at all but an eighth and at the last.  Beyond 4096 rows both item
# kernels stream; at C3 the ESS runs in persistent CTAs and beta on its side stream with one CTA per item.
PATHS = {"c3": (0, 2, ITEM_PERSISTENT, ITEM_CTA), "c5": (1, 3, ITEM_STREAM, ITEM_STREAM)}


@pytest.fixture(scope="module")
def G():
    import gpirt_b200.sampler as g
    from gpirt_b200 import _lib
    assert _lib.load().gpirt_b200_device_count() > 0, "no CUDA device"
    return g


def _cols(s, field, J):
    return np.asfortranarray(s.get(field)[:, J])


def _check_nu(O, L, nu, J, seed, sweep, slices):
    """nu_j = L z_j with z drawn with purpose P_ESS_Z at `sweep`: each slice of the fixed-point product is within
    K_slice 2^-51 max|L| max|z_j| (|L| < 2), the slices sum to K = n, and every addition of a slice onto nu rounds once
    in FP64.  Returns (L Z in FP64, worst error / bound)."""
    n = L.shape[0]
    Z = B.keyed_normals(O, seed, sweep, O.P_ESS_Z, J, n)
    ref = L @ Z                                    # one BLAS-3 product: L is read once, not once per item
    bound = n * 2.0 ** -51 * 2.0 * np.abs(Z).max(axis=0) + slices * U * np.abs(ref).max(axis=0)
    ratio = np.max(np.abs(nu - ref).max(axis=0) / bound)
    assert ratio <= 1.0, "nu = L z beyond the fixed-point bound: %.3g x" % ratio
    return ref, ratio


def _check_factor(G, O, L, theta, rows):
    """L as the sweep left it for theta: bit for bit the stand-alone factorisation of the same device-built
    S = K(theta, theta) + 1e-3 I (the pipelined factorisation runs the same kernels with the panel hook, whose nu slices,
    forward steps and block-inverse steps only read L), and the residual |L L^T - S| on `rows` (None: all rows) within
    2 n u max|S| (test_gpu_large_n.py::_check_factor).  Returns residual / bound."""
    n = L.shape[0]
    assert not np.triu(L, 1).any(), "strict upper triangle must be exactly zero"
    assert np.all(np.diag(L) > 0)
    assert max(L.max(), -L.min()) < 2.0, "|L| < 2^L_FIXED_EXP is what the fixed-scale slicing of L relies on"
    alone = G.chol_lower(G.se_cov(theta, theta, jitter=1e-3))
    assert np.array_equal(alone, L), "max |stand-alone - sweep| = %.3g" % np.abs(alone - L).max()
    del alone
    if rows is None:
        S = O.K(theta, theta) + 1e-3 * np.eye(n)
        resid = np.abs(L @ L.T - S).max()
    else:
        S = O.K(theta[rows], theta)
        S[np.arange(rows.size), rows] += 1e-3
        resid = np.abs(L[rows, :] @ L.T - S).max()
    ratio = resid / (2 * n * U * np.abs(S).max())
    assert ratio <= 1.0, "residual %.3g x the bound" % ratio
    return ratio


@pytest.mark.parametrize("workload,missing", [("c3", 0.0), ("c3", 0.05), ("c5", 0.05)])
def test_graph_replayed_pipelined_sweep_against_the_oracle(G, O, workload, missing):
    """bench.py's sampler (synthetic data and seed, default options: pipelined) after init_draws() and two sweeps, in
    steady state with theta on the grid; then one more sweep, t + 1 = 3, as one graph replay, checked step by step"""
    from gpirt_b200 import synthetic, _lib
    t_start = time.time()
    c = synthetic.WORKLOADS[workload]
    n, m = c["n"], c["m"]
    big = n > 4096
    route, slices, ess_shape, beta_shape = PATHS[workload]
    d = synthetic.make(n, m, missing=missing)
    seed = synthetic.SEED
    s = G.Sampler(d["y"], d["theta_init"], d["pm"], d["psd"], d["pstep"], seed=seed)
    s.set_timing(False)     # as bench.py times it: without per-step timers every sweep after the first is a graph replay
    s.init_draws()
    s.sweep(2)
    t = 2
    J, I = B.items(m, big), B.respondents(n, big)
    rows = B.panel_rows(n) if big else None        # C5: first and last row of every panel; C3: all rows
    ts, prior = O.grid()
    yJ = np.asfortranarray(d["y"][:, J])
    worst = {}

    # ---- the state sweep t left: theta_t, beta_t, f_t, L_t and nu = L_t z(t + 1) ----
    theta0 = s.get(_lib.THETA); beta0 = s.get(_lib.BETA); L0 = s.get(_lib.CHOL)
    assert len(np.unique(theta0)) <= 1001 < n, "theta on the grid: duplicated rows, PD only through the jitter"
    f0 = _cols(s, _lib.F, J); nu = _cols(s, _lib.NU, J)
    nu_ref, worst["nu"] = _check_nu(O, L0, nu, J, seed, t + 1, slices)
    worst["L L^T"] = _check_factor(G, O, L0, theta0, rows)
    del nu

    # ---- sweep t + 1: one graph replay, on the paths bench.py times ----
    replays = s.uses(5)
    assert replays >= 1, "sweep t was captured and launched as a graph"
    s.sweep(1)
    assert s.uses(5) == replays + 1, "the checked sweep ran as one graph replay"
    assert (s.uses(0), s.uses(1)) == (1, 1), "int8 theta contraction and fixed-point products"
    assert s.uses(4) == route, "K* solve route"
    assert (s.uses(2), s.uses(3)) == (ess_shape, beta_shape), "ESS and beta launch shapes"
    f1 = _cols(s, _lib.F, J); nprop = s.get(_lib.ESS_NPROP).astype(int)
    fs = s.get(_lib.FSTAR); sd = s.get(_lib.FSTAR_S); Dm = _cols(s, _lib.FSTAR_MEAN, J)
    logp = s.get(_lib.LOGP)[I, :]; idx = s.get(_lib.THETA_IDX).astype(int); theta1 = s.get(_lib.THETA)
    beta1 = s.get(_lib.BETA); L1 = s.get(_lib.CHOL); nu2 = _cols(s, _lib.NU, J)
    s.close()
    sweep = t + 1

    # ---- ESS (draw-f.cpp:21-60) from f_t, L_t and mu(theta_t, beta_t), with the proposals nu = L_t z ----
    mu = O.linear_mean(theta0, beta0[:, J])
    rng = O.Rng.keyed(seed); rng.set_sweep(sweep)     # items addressed by their global index, no map
    fo = np.empty_like(f1); npo = np.empty(len(J), dtype=int)
    for jj, j in enumerate(J):
        fo[:, jj], _, npo[jj] = O.ess(f0[:, jj], yJ[:, jj], L0, mu[:, jj], int(j), rng, nu=nu_ref[:, jj])
    assert np.array_equal(nprop[J], npo), "ESS proposal counts must match the oracle"
    worst["f"] = np.max(np.abs(f1 - fo)) / 1e-9
    assert worst["f"] <= 1.0
    del mu, nu_ref, f0, fo

    # ---- f* (draw-fstar.cpp:10-31) on f_{t+1}, theta_t, L_t and mu*(beta_t), all 1001 grid points ----
    rng = O.Rng.keyed(seed); rng.set_sweep(sweep); rng.set_item_map(J)
    fso, so, _ = O.draw_fstar(f1, theta0, ts, L0, O.linear_mean(ts, beta0[:, J]), rng)
    del L0
    worst["sd"] = np.max(np.abs(sd - so)) / 1e-8
    worst["f*"] = np.max(np.abs(fs[:, J] - fso)) / (1e-7 * max(1.0, np.abs(fso).max()))
    assert worst["sd"] <= 1.0 and worst["f*"] <= 1.0
    # FSTAR_MEAN holds the f* means until the theta step of the sweep overwrites it with D = log(2 cosh(f*/2)), the
    # per-(grid point, item) term of its contraction (k_theta_prep).  D is 1/2-Lipschitz in f*: within half of f*'s
    # tolerance from the oracle's draws, the other half left for the evaluation of D
    Do = 0.5 * np.abs(fso) + np.log1p(np.exp(-np.abs(fso)))
    worst["D(f*)"] = np.max(np.abs(Dm - Do)) / (1e-7 * max(1.0, np.abs(fso).max()))
    assert worst["D(f*)"] <= 1.0
    del fso, Do, Dm

    # ---- theta (draw-theta.cpp:12-34) on the stratum respondents with the device's f* ----
    tho, idxo, logpo = B.draw_theta_rows(O, ts, d["y"], prior, fs, seed, sweep, I)
    want_ll = logpo - prior[None, :]
    worst["logP"] = np.max(np.abs(logp - want_ll) / np.maximum(1.0, np.abs(want_ll))) / 1e-12
    assert worst["logP"] <= 1.0
    assert np.array_equal(idx[I], idxo), "grid indices must match the oracle (stabilised CDF)"
    assert np.array_equal(theta1[I], tho)
    del fs, logp, logpo, want_ll

    # ---- beta (draw-beta.cpp:16-38) from beta_t with theta_{t+1} and f_{t+1} ----
    rng = O.Rng.keyed(seed); rng.set_sweep(sweep); rng.set_item_map(J)
    bo, _ = O.draw_beta(beta0[:, J], theta1, yJ, f1, d["pm"][:, J], d["psd"][:, J], d["pstep"][:, J], rng)
    worst["beta"] = np.max(np.abs(beta1[:, J] - bo)) / 1e-12
    assert worst["beta"] <= 1.0

    # ---- rebuild: L_{t+1} and the proposals nu = L_{t+1} z(t + 2) it left for sweep t + 2 ----
    worst["L L^T next"] = _check_factor(G, O, L1, theta1, rows)
    _, worst["nu next"] = _check_nu(O, L1, nu2, J, seed, t + 2, slices)
    print("%s %g%% missing, pipelined graph sweep: %d items, %d respondents, %s rows of L; worst error / bound: %s; %.0f s" % (
        workload, 100 * missing, len(J), len(I), "all" if rows is None else str(rows.size),
        ", ".join("%s %.2e" % kv for kv in worst.items()), time.time() - t_start))
