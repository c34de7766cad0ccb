"""CPU tests of the oracle (no GPU): hand-computed values, the reference's compiled sources (oracle/_ref, only where
that library is built or oracle/Makefile finds a checkout of duckmayr/gpirt, see GPIRT_REFERENCE there), and the
committed golden vectors that those sources produced."""
import os

import numpy as np
import pytest

from conftest import make_problem
from oracle import oracle as _oracle

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
HAVE_REF = _oracle.have_ref()


def test_philox_known_answer(O):
    # Random123 known-answer vectors for Philox4x32-10
    import ctypes as C
    L = O.lib()
    def ph(c, k):
        arr = (C.c_uint32 * 4)(*c)
        L.gpo_philox(arr, C.c_uint32(k[0]), C.c_uint32(k[1]))
        return [int(x) for x in arr]
    assert ph([0, 0, 0, 0], [0, 0]) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert ph([0xffffffff] * 4, [0xffffffff] * 2) == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert ph([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0]) == [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_addressed_variates_are_sane(O):
    u = np.array([O.keyed_uniform(9, 1, O.P_ESS_U, 3, i) for i in range(4000)])
    z = np.array([O.keyed_normal(9, 1, O.P_ESS_Z, 3, i) for i in range(4000)])
    assert 0 < u.min() and u.max() < 1 and abs(u.mean() - 0.5) < 0.02
    assert abs(z.mean()) < 0.06 and abs(z.std() - 1) < 0.05
    assert O.keyed_uniform(9, 1, O.P_ESS_U, 3, 0) != O.keyed_uniform(9, 2, O.P_ESS_U, 3, 0)   # sweep is part of the address


def test_K_and_ll_hand_values(O):
    K = O.K([0.0, 1.0], [0.0, 2.0, -1.0])
    want = np.exp(-0.5 * np.array([[0, 4, 1], [1, 1, 4]], dtype=float))
    assert np.allclose(K, want, rtol=0, atol=1e-16)
    f = np.array([0.3, -1.2, 2.0]); y = np.array([1.0, np.nan, -1.0])
    assert O.ll(f, y) == pytest.approx(-(np.log(1 + np.exp(-0.3)) + np.log(1 + np.exp(2.0))), abs=1e-15)
    mu = np.array([0.1, 0.2, -0.5])
    assert O.ll_bar(f, y, mu) == pytest.approx(-(np.log(1 + np.exp(-0.4)) + np.log(1 + np.exp(1.5))), abs=1e-15)
    assert O.ll(np.array([800.0]), np.array([-1.0])) == -np.inf     # log(1+exp(800)) overflows like the reference (F1 quirks)


def test_grid_matches_reference_doc(O):
    ts, prior = O.grid()
    assert ts.size == 1001 and ts[0] == -5.0 and ts[500] == pytest.approx(0.0, abs=1e-15) and ts[-1] == pytest.approx(5.0, abs=1e-12)
    assert ts[1] == -5.0 + 1 * 0.01 and ts[777] == -5.0 + 777 * 0.01                 # start + i*delta, two roundings
    assert prior[500] == pytest.approx(-0.9189385332046727, abs=1e-15)


def test_chol_matches_numpy_and_rejects_non_pd(O):
    p = make_problem(60, 2, seed=1, grid_theta=True)
    S = O.K(p["theta"], p["theta"]) + 1e-3 * np.eye(60)
    L = O.chol_lower(S)
    assert np.allclose(L, np.linalg.cholesky(S), atol=1e-10) and np.array_equal(np.triu(L, 1), np.zeros((60, 60)))
    with pytest.raises(np.linalg.LinAlgError):
        O.chol_lower(np.ones((5, 5)))


def test_ess_bracket_quirk_and_invariance(O):
    """initial bracket is [eps-2pi, 2pi] (draw-f.cpp:33-36); the step leaves the likelihood above the slice level"""
    p = make_problem(50, 1, seed=4, missing=0.0)
    L = O.build_cholS(p["theta"])
    f = L @ np.random.RandomState(0).randn(50)
    mu = np.zeros(50)
    rng = O.Rng.keyed(5); rng.set_sweep(1)
    fnew, nu, nprop = O.ess(f, p["y"][:, 0], L, mu, 0, rng)
    u = O.keyed_uniform(5, 1, O.P_ESS_U, 0, 0)
    assert O.ll_bar(fnew, p["y"][:, 0], mu) > O.ll_bar(f, p["y"][:, 0], mu) + np.log(u)
    assert nprop >= 1
    # f' lies on the ellipse through f and nu
    A = np.stack([f, nu], axis=1)
    coef, res, *_ = np.linalg.lstsq(A, fnew, rcond=None)
    assert np.allclose(A @ coef, fnew, atol=1e-12) and coef[0] ** 2 + coef[1] ** 2 == pytest.approx(1.0, abs=1e-12)


def test_theta_cdf_modes_agree_where_reference_is_finite(O):
    p = make_problem(30, 40, seed=6, missing=0.1)
    ts, prior = O.grid()
    fstar = np.asfortranarray(np.random.RandomState(1).randn(1001, 40) * 0.5)
    a = O.draw_theta(ts, p["y"], prior, fstar, O.Rng.keyed(3), mode=0)
    b = O.draw_theta(ts, p["y"], prior, fstar, O.Rng.keyed(3), mode=1)
    assert np.array_equal(a[1], b[1]) and np.array_equal(a[0], b[0])
    assert (a[1] > 0).all(), "grid point 0 carries zero mass (min-subtraction, draw-theta.cpp:24-25)"


def test_theta_reference_underflow_is_reproduced(O):
    """SURVEY F3: with ~1000+ items every exp(logP) underflows, the CDF is 0/0 and the reference reads theta_star[N]."""
    p = make_problem(5, 2500, seed=7, missing=0.0)
    ts, prior = O.grid()
    fstar = np.asfortranarray(np.random.RandomState(2).randn(1001, 2500))
    strict = O.draw_theta(ts, p["y"], prior, fstar, O.Rng.keyed(3), mode=0)
    stab = O.draw_theta(ts, p["y"], prior, fstar, O.Rng.keyed(3), mode=1)
    assert np.isnan(strict[0]).all() and (strict[1] == 1001).all()
    assert np.isfinite(stab[0]).all()


@pytest.mark.parametrize("name", ["tiny_8x5", "small_100x37", "odd_257x12"])
def test_oracle_reproduces_reference_goldens(O, name):
    g = np.load(os.path.join(GOLD, name + ".npz"))
    m = g["y"].shape[1]
    rng = O.Rng.keyed(int(g["seed"]), record=True)
    r = O.mcmc(g["y"], g["theta_init"], int(g["S"]), int(g["B"]), np.zeros((2, m)), np.full((2, m), 3.0), np.full((2, m), 0.1), rng)
    assert rng.recorded()[0].size == int(g["tape_len"]), "same number of variates consumed as the reference"
    assert np.array_equal(r["theta"], g["theta"])
    for k in ("beta", "f", "IRFs"):   # BLAS kernels differ between CPU models: last-bit tolerance, not bitwise
        assert np.max(np.abs(r[k] - g[k])) <= 1e-9, k


def test_oracle_reproduces_senate116_golden(O):
    g = np.load(os.path.join(GOLD, "senate116_100x418.npz"))
    y = g["y_int8"].astype(np.float64); y[y == 0] = np.nan
    assert y.shape == (100, 418)
    m = 418
    r = O.mcmc(y, g["theta_init"], int(g["S"]), int(g["B"]), np.zeros((2, m)), np.full((2, m), 3.0), np.full((2, m), 0.1),
               O.Rng.keyed(int(g["seed"])), theta_cdf_mode=0)
    assert np.array_equal(r["theta"], g["theta"])
    assert np.max(np.abs(r["beta"] - g["beta"])) <= 1e-9
    assert np.max(np.abs(r["f"][:, :, -1] - g["f_last"])) <= 1e-8
    assert np.max(np.abs(r["IRFs"][::10] - g["IRFs_every10"])) <= 1e-9


@pytest.mark.skipif(not HAVE_REF, reason="needs the reference package's own sources (GPIRT_REFERENCE: a checkout of "
                                         "duckmayr/gpirt); without them only the whole-chain goldens above compare with it")
class TestAgainstCompiledReference:
    """The restatement against the reference's own sources (oracle/_ref) on replayed tapes: bit-exact."""

    def test_full_chain_bit_exact(self, O):
        p = make_problem(60, 17, seed=3, missing=0.07)
        rng = O.Rng.keyed(99, record=True)
        port = O.mcmc(p["y"], p["theta"], 3, 2, p["pm"], p["psd"], p["pstep"], rng)
        vals, kinds = rng.recorded()
        with O.RefTape(vals, kinds) as t:
            ref = O.ref_mcmc(p["y"], p["theta"], 3, 2, p["pm"], p["psd"], p["pstep"])
        assert t.error == 0 and t.consumed == vals.size
        for k in ("theta", "beta", "f", "IRFs"):
            assert np.array_equal(port[k], ref[k]), k

    def test_each_function_bit_exact(self, O):
        p = make_problem(45, 9, seed=8, missing=0.1, grid_theta=True)
        rs = np.random.RandomState(0)
        ts, prior = O.grid()
        assert np.array_equal(O.K(p["theta"], ts), O.ref_K(p["theta"], ts))
        S = O.K(p["theta"], p["theta"]) + 1e-3 * np.eye(45)
        L = O.chol_lower(S)
        assert np.array_equal(L, O.ref_chol_lower(S))
        f = np.asfortranarray(L @ rs.randn(45, 9)); beta = np.asfortranarray(rs.randn(2, 9))
        mu, mus = O.linear_mean(p["theta"], beta), O.linear_mean(ts, beta)
        assert O.ll(f[:, 0], p["y"][:, 0]) == O.ref_ll(f[:, 0], p["y"][:, 0])
        assert O.ll_bar(f[:, 1], p["y"][:, 1], mu[:, 1]) == O.ref_ll_bar(f[:, 1], p["y"][:, 1], mu[:, 1])
        for fn_port, fn_ref in [
            (lambda r: O.draw_f(f, p["y"], L, mu, r)[0], lambda: O.ref_draw_f(f, p["y"], L, mu)),
            (lambda r: O.draw_fstar(f, p["theta"], ts, L, mus, r)[0], lambda: O.ref_draw_fstar(f, p["theta"], ts, L, mus)),
            (lambda r: O.draw_beta(beta, p["theta"], p["y"], f, p["pm"], p["psd"], p["pstep"], r)[0],
             lambda: O.ref_draw_beta(beta, p["theta"], p["y"], f, p["pm"], p["psd"], p["pstep"])),
        ]:
            rng = O.Rng.keyed(5, record=True); rng.set_sweep(2)
            a = fn_port(rng)
            with O.RefTape(*rng.recorded()) as t:
                b = fn_ref()
            assert t.error == 0 and np.array_equal(a, b)
        fstar = np.asfortranarray(rs.randn(1001, 9))
        rng = O.Rng.keyed(6, record=True)
        a = O.draw_theta(ts, p["y"], prior, fstar, rng, mode=0)[0]
        with O.RefTape(*rng.recorded()) as t:
            b = O.ref_draw_theta(ts, p["y"], prior, fstar, mus)
        assert np.array_equal(a, b)

    def test_reference_theta_bug_needs_the_stabilised_cdf(self, O):
        """the unmodified reference returns theta_star[N] (NaN sentinel here) for every respondent at m = 2500"""
        p = make_problem(4, 2500, seed=7, missing=0.0)
        ts, prior = O.grid()
        fstar = np.asfortranarray(np.random.RandomState(2).randn(1001, 2500))
        rng = O.Rng.keyed(3, record=True)
        O.draw_theta(ts, p["y"], prior, fstar, rng, mode=0)
        with O.RefTape(*rng.recorded()):
            th = O.ref_draw_theta(ts, p["y"], prior, fstar, np.zeros((1001, 2500)))
        assert np.isnan(th).all()
