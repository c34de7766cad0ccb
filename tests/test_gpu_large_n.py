"""Oracle parity beyond n = 4096 respondents, where the sampler switches to its large-n code paths: the look-ahead
Cholesky with a ragged last panel, the K*-solve route by blocked substitution (the default for n > 6144, with the
1024-block inverses of the backward pass and their ragged merges), and the fixed-point products at long contraction
lengths.  Sizes are chosen for their edges: 6144 / 6145 straddle the route switch and 6145 ends in a one-row panel;
9000 = 8 x 1024 + 808 leaves a ragged pair in the block-inverse levels 256 and 512; 16384 is C5's n.

Tolerances (each with its reason at the assertion):
  Cholesky factor   residual |L L^T - S| on sampled rows <= 2 n u max|S| (Higham's gamma_{n+1} |L||L^T| backward error,
                    |L||L^T|_ij <= sqrt(S_ii S_jj) = 1.001, plus as much again for numpy's FP64 evaluation of L L^T);
                    |L - LAPACK| <= 1e-9 as in test_gpu_parity.py::test_chol_lower
  f* step           as at C3 (test_gpu_bench_shapes.py): sd 1e-8, mean and f* 1e-7 relative
  sweeps            as test_gpu_full_size.py (pipelined vs not) and test_c2_one_full_lockstep_sweep (lock-step)
  fixed point       K 2^-51 max|a_i| max|b_j| (include/gpirt_b200.h)"""
import numpy as np
import pytest
import scipy.linalg as sla

from conftest import make_problem

pytestmark = pytest.mark.gpu

U = 2.0 ** -53


@pytest.fixture(scope="module")
def G():
    import gpirt_b200.sampler as g
    from gpirt_b200 import _lib
    assert _lib.load().gpirt_b200_device_count() > 0, "no CUDA device"
    return g


def _grid_theta(n, seed):
    return np.round(np.clip(np.random.RandomState(seed).randn(n), -5, 5), 2)


def _check_factor(L, S, Lref, rows, label):
    """the checks every factor of S = K(theta, theta) + 1e-3 I must pass; returns the measured / allowed ratios"""
    n = S.shape[0]
    assert not np.triu(L, 1).any(), "%s: strict upper triangle must be exactly zero" % label
    assert np.all(np.diag(L) > 0), label
    assert max(L.max(), -L.min()) < 2.0, "%s: |L| < 2^L_FIXED_EXP is what the fixed-scale slicing of L relies on" % label
    resid = np.abs(L[rows, :] @ L.T - S[rows, :]).max()
    bound = 2 * n * U * np.abs(S).max()
    assert resid <= bound, "%s: residual %.3g > %.3g" % (label, resid, bound)
    err = np.abs(L - Lref).max()
    assert err <= 1e-9, "%s: |L - LAPACK| = %.3g" % (label, err)
    return resid / bound, err / 1e-9


@pytest.mark.parametrize("n", [4097, 6144, 6145, 9000, 16384])
def test_sampler_factor_beyond_4096_respondents(G, O, n):
    """The factor the sampler itself builds (step_rebuild: look-ahead stream, panel hook), then a second factorisation of
    a different theta in the same sampler: panel counters, the 128-block inverses and the look-ahead events carried over
    from the first must not leak into the second.  The stand-alone gpirt_b200_chol_lower is checked the same way on the
    same S.  It runs the same panel, update and bulk kernels on the same block partition, only without the look-ahead
    stream, so given the S the sampler builds on the device (whose exp() may differ from the host's by an ulp) it returns
    the sampler's factor bit for bit."""
    from gpirt_b200 import _lib
    prob = make_problem(n, 256, seed=n, grid_theta=True)   # theta on the 0.01 grid: duplicated rows, PD only by jitter
    s = G.Sampler(prob["y"], prob["theta"], seed=n)
    assert s.uses(1) == 1, "m >= 256: the fixed-point products (and with them the |L| < 2 scale) are selected"
    rs = np.random.RandomState(n)
    for label, theta in (("first", prob["theta"]), ("rebuilt", _grid_theta(n, n + 1))):
        if label == "rebuilt":
            s.set(_lib.THETA, theta)
            s.step(_lib.STEP_REBUILD, 0)
        L = s.get(_lib.CHOL)
        S = O.K(theta, theta) + 1e-3 * np.eye(n)
        Lref = sla.cholesky(S, lower=True, check_finite=False)
        rows = np.unique(np.r_[0, n - 1, rs.choice(n, 64, replace=False)])
        for path, F in (("sampler", L), ("stand-alone", G.chol_lower(S))):
            ratios = _check_factor(F, S, Lref, rows, "%s %s" % (label, path))
            print("n = %d %s %s: residual / bound = %.2e, |L - LAPACK| / 1e-9 = %.2e" % ((n, label, path) + ratios))
        del Lref, S, F
        alone = G.chol_lower(G.se_cov(theta, theta, jitter=1e-3))
        assert np.array_equal(alone, L), "max |stand-alone - sampler| = %.3g" % np.abs(alone - L).max()
        del L, alone
    s.close()


@pytest.mark.parametrize("n,route", [(6144, 0), (6145, 1), (9000, 1)])
def test_fstar_step_across_the_solve_route_switch(G, O, n, route, monkeypatch):
    """STEP_DRAW_FSTAR on every item against draw_fstar of the oracle, on the default route of each size and, beyond
    the switch, on the other route as well: 6145 ends in a one-row panel, 9000 has ragged pairs at the block-inverse
    levels 256 and 512 (trtri_lower, the backward pass on 1024-blocks)"""
    from gpirt_b200 import _lib
    m, seed, sweep = 256, n + 77, 2
    prob = make_problem(n, m, seed=n + 1, grid_theta=True)
    rs = np.random.RandomState(n + 2)
    ts, _ = O.grid()
    want = None
    L0 = None
    for forced in ([None, "0"] if route == 1 else [None]):
        if forced is None:
            monkeypatch.delenv("GPIRT_SOLVE_MODE", raising=False)
        else:
            monkeypatch.setenv("GPIRT_SOLVE_MODE", forced)
        s = G.Sampler(prob["y"], prob["theta"], prob["pm"], prob["psd"], prob["pstep"], seed=seed)
        assert s.uses(1) == 1
        assert s.uses(4) == (route if forced is None else int(forced)), "K* solve route"
        L = s.get(_lib.CHOL)
        if L0 is None:   # same state for every route: f = L z, random beta (as test_gpu_parity.py::_state)
            L0 = L
            f = L @ rs.randn(n, m)
            beta = rs.randn(2, m)
            mu_star = O.linear_mean(ts, beta)
            rng = O.Rng.keyed(seed); rng.set_sweep(sweep)
            want = O.draw_fstar(f, prob["theta"], ts, L, mu_star, rng)
        else:
            assert np.array_equal(L, L0), "the route does not change the factor"
        s.set(_lib.F, f); s.set(_lib.BETA, beta)
        s.step(_lib.STEP_DRAW_FSTAR, sweep)
        fs = s.get(_lib.FSTAR); sd = s.get(_lib.FSTAR_S); mean = s.get(_lib.FSTAR_MEAN)
        s.close()
        fso, so, meano = want
        tag = "route %d" % (route if forced is None else int(forced))
        # C3's tolerances (test_c3_sampled_items_and_respondents_against_the_oracle); the mean carries f*'s error
        err = (np.abs(sd - so).max(),
               np.abs(mean + mu_star - meano).max() / max(1.0, np.abs(meano).max()),
               np.abs(fs - fso).max() / max(1.0, np.abs(fso).max()))
        print("n = %d %s: |sd| %.2e / 1e-8, |mean| %.2e / 1e-7, |f*| %.2e / 1e-7" % ((n, tag) + err))
        assert err[0] <= 1e-8, tag
        assert err[1] <= 1e-7, tag
        assert err[2] <= 1e-7, tag


def test_route1_sweeps_pipelined_and_unpipelined_agree(G):
    """n = 9000 on the substitution route: the pipelined sweep builds the 1024-block inverses step by step behind the
    panels (trtri_lower_step, incl. the ragged pairs the last panel completes), lets the forward steps trail the panels
    on their own stream and shrinks the L Z slices towards the end of the factorisation; the sequential sweep does none
    of that.  Tolerances of test_gpu_full_size.py::test_full_size_sweeps_pipelined_and_unpipelined_agree."""
    from gpirt_b200 import _lib
    n, m = 9000, 300
    prob = make_problem(n, m, seed=19, missing=0.03)
    out = {}
    for pipe in (True, False):
        s = G.Sampler(prob["y"], prob["theta"], prob["pm"], prob["psd"], prob["pstep"], seed=11)
        assert s.uses(1) == 1 and s.uses(4) == 1
        s.set_pipeline(pipe)
        s.init_draws()
        s.sweep(3)
        out[pipe] = {k: s.get(f) for k, f in (("theta", _lib.THETA), ("beta", _lib.BETA), ("f", _lib.F), ("nprop", _lib.ESS_NPROP))}
        s.close()
    a, b = out[True], out[False]
    print("n = 9000: |beta| %.2e / 1e-10, |f| %.2e / 1e-9" % (np.abs(a["beta"] - b["beta"]).max(), np.abs(a["f"] - b["f"]).max()))
    assert np.array_equal(a["theta"], b["theta"])
    assert np.max(np.abs(a["beta"] - b["beta"])) <= 1e-10
    assert np.max(np.abs(a["f"] - b["f"])) <= 1e-9
    assert np.array_equal(a["nprop"], b["nprop"])


def test_lockstep_sweep_beyond_the_route_switch(G, O):
    """initial draws + one full sweep of the public call at n = 6145 (route 1, one-row last panel, streaming item
    kernels, fixed-point products) draw by draw against the oracle's gpirtMCMC restatement; tolerances of
    test_gpu_bench_shapes.py::test_c2_one_full_lockstep_sweep"""
    from gpirt_b200 import ResponseMatrix
    n, m, seed = 6145, 256, 6145
    prob = make_problem(n, m, seed=21, missing=0.05)
    s = G.Sampler(prob["y"], prob["theta"], seed=seed)
    assert (s.uses(1), s.uses(4)) == (1, 1)
    s.close()
    got = G.gpirtMCMC(ResponseMatrix(prob["y"]), 1, 0, beta_prior_means=prob["pm"], beta_prior_sds=prob["psd"],
                      beta_proposal_sds=prob["pstep"], theta_init=prob["theta"], seed=seed)
    want = O.mcmc(prob["y"], prob["theta"], 1, 0, prob["pm"], prob["psd"], prob["pstep"], O.Rng.keyed(seed), theta_cdf_mode=1)
    print("n = 6145: |beta| %.2e / 1e-9, |f| %.2e / 1e-7, |IRFs| %.2e / 1e-7" % (
        np.abs(got["beta"] - want["beta"]).max(), np.abs(got["f"] - want["f"]).max(), np.abs(got["IRFs"] - want["IRFs"]).max()))
    assert np.array_equal(got["theta"], want["theta"]), "theta draws (grid points) must be identical"
    assert np.max(np.abs(got["beta"] - want["beta"])) <= 1e-9
    assert np.max(np.abs(got["f"] - want["f"])) <= 1e-7
    assert np.max(np.abs(got["IRFs"] - want["IRFs"])) <= 1e-7


def _digits_of(X):
    """balanced base-128 digits of the 56-bit integer X, most significant first (digits_of in dgemm_i8.cu)"""
    d = [0] * 8
    for s in range(7, 0, -1):
        d[s] = ((X + 64) & 127) - 64
        X = (X - d[s]) >> 7
    d[0] = X
    return d


def test_dgemm_i8_level_accumulators_at_the_largest_contraction_length(G):
    """K = 65535, the largest contraction the fixed-point product accepts: a level accumulator sums up to 8 digit-pair
    products of |.| <= 64 x 64 over K, i.e. < 8 64^2 65536 = 2^31.  Operands whose every digit sits at the end of the
    range, with the same sign in every pair of one level, bring level 7 within 0.4 % of 2^31; a wrapped int32 would move
    the result by 2^32 128^-7 2^(ea + eb - 12) = 2^-27, a thousand times the tolerance.  K = 65536 is refused."""
    from gpirt_b200._lib import GpirtError, ERR_ARG
    K, M, N = 65535, 128, 64
    # v = X 2^-54 with X = -(63 128^7 + 64 sum_{s<7} 128^s): |v| in [1, 2) -> row scale 2^(55 - 1), digits (-63, -64 x 7)
    X = -(63 * 128 ** 7 + 64 * sum(128 ** s for s in range(7)))
    v = X * 2.0 ** -54
    assert int(v * 2.0 ** 54) == X, "v is exact in FP64"
    d = _digits_of(X)
    assert d == [-63] + [-64] * 7
    levels = [K * sum(d[s] * d[l - s] for s in range(l + 1)) for l in range(8)]
    assert max(levels) == levels[7] == 32640 * K
    assert 0.996 * 2 ** 31 < levels[7] < 2 ** 31, levels[7]
    rs = np.random.RandomState(65535)
    A = rs.randn(M, K)
    B = rs.randn(K, N)
    A[:M // 2, :] = v                  # against B's v columns every level-7 digit product is +63 x 64 or +64 x 64
    B[:, :N // 2] = v                  # (the other rows and columns: random operands in the same launch)
    got = G.dgemm_i8(A, B)
    want = A.astype(np.longdouble) @ B.astype(np.longdouble)
    bound = K * 2.0 ** -51 * np.abs(A).max(axis=1)[:, None] * np.abs(B).max(axis=0)[None, :]
    err = np.abs(got - want)
    print("K = 65535: max err / bound = %.2e (v block %.2e)" % (np.max(err / bound), np.max(err[:M // 2, :N // 2] / bound[:M // 2, :N // 2])))
    assert np.all(err <= bound)
    with pytest.raises(GpirtError) as e:
        G.dgemm_i8(rs.randn(8, 65536), rs.randn(65536, 4))
    assert e.value.status == ERR_ARG
