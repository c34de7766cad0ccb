"""GPU parity tests (-m gpu): every CUDA step against the CPU oracle on the same seeded inputs and the same addressed
Philox variates, called through the C ABI (gpirt_b200/_lib.py -> libgpirt_b200.so).

Stated FP64 tolerances (north_star: "within a stated FP64 tolerance given identical injected random draws"):
  K                      |dK| <= 4e-16 (exp() implementations differ by <= 1-2 ulp of values <= 1)
  Cholesky factor        |L L^T - S| <= 1e-12 |S|max ; |L - L_oracle| <= 1e-9 (cond(S) up to ~1e7)
  L z, triangular solves relative 1e-12 / 1e-9 (solves, conditioning)
  log-likelihoods, logP  relative 1e-12
  ESS / beta / theta     discrete decisions (accept, shrink count, grid index) identical; values to 1e-9
"""
import numpy as np
import pytest
import scipy.linalg as sla

from conftest import make_problem

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def G():
    import gpirt_b200.sampler as g
    from gpirt_b200 import _lib
    assert _lib.load().gpirt_b200_device_count() > 0, "no CUDA device"
    return g


def test_rng_matches_oracle(G, O):
    seed = 0x1234ABCD9876
    for purpose, stream, sweep in [(2, 0, 1), (3, 17, 5), (4, 999, 1000), (5, 4095, 7)]:
        u, z = G.rng_probe(seed, sweep, purpose, stream, 0, 64)
        uo = np.array([O.keyed_uniform(seed, sweep, purpose, stream, i) for i in range(64)])
        zo = np.array([O.keyed_normal(seed, sweep, purpose, stream, i) for i in range(64)])
        assert np.array_equal(u, uo), "Philox uniforms must be bit-exact"
        assert np.max(np.abs(z - zo)) <= 2e-15
    assert (u > 0).all() and (u < 1).all()


@pytest.mark.parametrize("n1,n2", [(1, 1), (7, 5), (100, 1001), (257, 257), (1024, 130)])
def test_se_cov(G, O, n1, n2):
    rs = np.random.RandomState(n1 + n2)
    x1, x2 = rs.randn(n1) * 2, rs.randn(n2) * 2
    got, want = G.se_cov(x1, x2), O.K(x1, x2)
    assert np.max(np.abs(got - want)) <= 4e-16
    if n1 == n2:
        got = G.se_cov(x1, x1, jitter=1e-3)
        want = O.K(x1, x1) + 1e-3 * np.eye(n1)
        assert np.max(np.abs(got - want)) <= 4e-16


@pytest.mark.parametrize("ta,tb", [(False, False), (True, False), (False, True)])
@pytest.mark.parametrize("M,N,K", [(1, 1, 1), (8, 8, 4), (130, 67, 33), (64, 200, 64), (300, 257, 100), (1001, 700, 513),
                                   (1500, 1400, 260)])
def test_dgemm(G, ta, tb, M, N, K):
    rs = np.random.RandomState(M * 7 + N * 3 + K)
    A = rs.randn(*((K, M) if ta else (M, K)))
    B = rs.randn(*((N, K) if tb else (K, N)))
    C0 = rs.randn(M, N)
    want = 1.5 * (A.T if ta else A) @ (B.T if tb else B) - 0.5 * C0
    got = G.dgemm(A, B, C0, alpha=1.5, beta=-0.5, ta=ta, tb=tb)
    scale = np.abs(A).max() * np.abs(B).max() * K + 1
    assert np.max(np.abs(got - want)) <= 1e-13 * scale
    got0 = G.dgemm(A, B, None, ta=ta, tb=tb)
    assert np.max(np.abs(got0 - (A.T if ta else A) @ (B.T if tb else B))) <= 1e-13 * scale


@pytest.mark.parametrize("ta,lower,M,N,K", [(0, 0, 1, 1, 1), (0, 0, 128, 64, 64), (1, 0, 100, 37, 50), (1, 0, 300, 200, 257),
                                             (0, 1, 257, 130, 257), (0, 1, 1000, 333, 1000), (1, 0, 1001, 500, 1100),
                                             (0, 0, 129, 65, 4097), (0, 1, 16384, 70, 16384), (1, 2, 16384, 70, 16384)])
def test_dgemm_i8_fixed_point_tensor_core_product(G, ta, lower, M, N, K):
    """op(A) B in 56-bit fixed point on the int8 tensor cores (tcgen05): the kernel behind nu = L Z (draw-f.cpp:20) and the
    f* product.  The plane products are exact integers, so the only error is the dropped digit levels:
    |err_ij| <= K 2^-51 max|A[i,:]| max|B[:,j]|  (the tolerance stated in include/gpirt_b200.h).  lower = 1: op(A) lower
    triangular (L Z); lower = 2: op(A) = A^T upper triangular (the L^-T product); K = 16384 is C5's n.  The reference is
    summed in long double, its own rounding far below K 2^-51; at K = 16384 on 64 sampled rows and the first and last 32."""
    rs = np.random.RandomState(M * 11 + N * 5 + K)
    tri = {0: lambda X: X, 1: np.tril, 2: np.triu}[lower]
    A = tri(rs.randn(M, K) * np.exp(2.0 * rs.randn(M, 1)))     # rows of very different magnitude
    B = rs.randn(K, N) * np.exp(2.0 * rs.randn(1, N))
    if M > 2:
        A[1, :] = 0.0                                            # an all-zero row
    if K > 3:
        A[0, 3] = 0.0
    rows = np.arange(M) if M <= 4096 else np.unique(np.r_[0:32, M - 32:M, rs.choice(M, 64, replace=False)])
    got = G.dgemm_i8(np.asfortranarray(A.T) if ta else A, B, ta=bool(ta), a_lower=lower)[rows]
    want = A[rows].astype(np.longdouble) @ B.astype(np.longdouble)
    bound = K * 2.0 ** -51 * np.abs(A[rows]).max(axis=1)[:, None] * np.abs(B).max(axis=0)[None, :]
    assert np.all(np.abs(got - want) <= bound + 1e-300)
    del A
    # against an FP64 product's own error scale: within a few units of K u sum|a||b| when rows are evenly scaled
    A2 = tri(rs.randn(M, K))
    B2 = rs.randn(K, N)
    got2 = G.dgemm_i8(np.asfortranarray(A2.T) if ta else A2, B2, ta=bool(ta), a_lower=lower)[rows]
    A2 = A2[rows]
    assert np.max(np.abs(got2 - A2 @ B2)) <= 64 * 2.0 ** -53 * max(1.0, np.max(np.abs(A2) @ np.abs(B2)))


@pytest.mark.parametrize("n,N", [(64, 3), (300, 70), (1000, 1001)])
def test_dgemm_i8_upper_triangular_transposed_operand(G, n, N):
    """op(A) = A^T with A stored lower triangular (the L^-T product of draw-fstar.cpp:24): row tiles start at the diagonal"""
    rs = np.random.RandomState(n)
    A = np.tril(rs.randn(n, n)) * np.exp(rs.randn(1, n))
    B = rs.randn(n, N)
    got = G.dgemm_i8(A, B, ta=True, a_lower=2)
    want = A.T @ B
    bound = n * 2.0 ** -51 * np.abs(A).max(axis=0)[:, None] * np.abs(B).max(axis=0)[None, :]
    assert np.all(np.abs(got - want) <= bound + 1e-300)


def test_dgemm_i8_is_deterministic_and_matches_dmma(G):
    rs = np.random.RandomState(3)
    L = np.tril(rs.randn(700, 700)) / 30.0
    Z = rs.randn(700, 900)
    a = G.dgemm_i8(L, Z, a_lower=True)
    b = G.dgemm_i8(L, Z, a_lower=True)
    assert np.array_equal(a, b), "integer accumulation: bit-identical from run to run"
    assert np.array_equal(G.dgemm_i8(L, Z[:, 100:300], a_lower=True), a[:, 100:300]), "columns are independent (item sharding)"
    assert np.max(np.abs(a - G.dgemm(L, Z, None, tri=1))) <= 1e-13


@pytest.mark.parametrize("n,m", [(100, 37), (300, 300), (1100, 1300)])
def test_dgemm_triangular_modes(G, n, m):
    rs = np.random.RandomState(n)
    L = np.tril(rs.randn(n, n))
    Z = rs.randn(n, m)
    got = G.dgemm(L, Z, None, tri=1)                       # A lower triangular: skipped k-tiles must be exactly the zeros
    assert np.max(np.abs(got - L @ Z)) <= 1e-12 * n
    got = G.dgemm(L, Z, None, ta=True, tri=3)              # op(A) = L^T upper triangular
    assert np.max(np.abs(got - L.T @ Z)) <= 1e-12 * n
    A = rs.randn(n, 70)
    C0 = rs.randn(n, n)
    got = G.dgemm(A, A, C0, alpha=-1.0, beta=1.0, tb=True, tri=2)   # symmetric update, lower triangle only
    want = C0 - A @ A.T
    lower = np.tril_indices(n)
    upper = np.triu_indices(n, 1)
    assert np.max(np.abs(got[lower] - want[lower])) <= 1e-12 * 70
    assert np.array_equal(got[upper], C0[upper]), "strict upper triangle must be untouched"


@pytest.mark.parametrize("n", [1, 8, 63, 64, 65, 100, 257, 1000, 2048])
def test_chol_lower(G, O, n):
    prob = make_problem(n, 2, seed=n, grid_theta=True)     # theta on the 0.01 grid => duplicated rows, PD only by jitter
    S = O.K(prob["theta"], prob["theta"]) + 1e-3 * np.eye(n)
    L = G.chol_lower(S)
    Lo = O.chol_lower(S)
    assert np.array_equal(np.triu(L, 1), np.zeros_like(L)), "strict upper must be exactly zero"
    assert np.max(np.abs(L @ L.T - S)) <= 1e-12 * np.abs(S).max() * max(1, np.log2(n + 1))
    assert np.max(np.abs(L - Lo)) <= 1e-9


def test_chol_repeatable_under_load(G, O):
    """the single-CTA diagonal-block kernel is barrier-heavy: repeat it many times and demand bitwise-identical factors"""
    prob = make_problem(384, 2, seed=5, grid_theta=True)
    S = O.K(prob["theta"], prob["theta"]) + 1e-3 * np.eye(384)
    ref = G.chol_lower(S)
    assert np.isfinite(ref).all()
    for _ in range(150):
        assert np.array_equal(G.chol_lower(S), ref)


def test_chol_not_pd(G):
    from gpirt_b200._lib import GpirtError, ERR_NOT_PD
    S = np.ones((70, 70))                                  # rank one, no jitter -> chol(): decomposition failed
    with pytest.raises(GpirtError) as e:
        G.chol_lower(S)
    assert e.value.status == ERR_NOT_PD


@pytest.mark.parametrize("trans", [False, True])
@pytest.mark.parametrize("n,r", [(5, 3), (64, 10), (100, 1001), (257, 40), (1000, 300)])
def test_trsm_lower(G, O, n, r, trans):
    prob = make_problem(n, 2, seed=n + r, grid_theta=True)
    L = O.build_cholS(prob["theta"])
    B = np.random.RandomState(r).randn(n, r)
    got = G.trsm_lower(L, B, trans=trans)
    want = sla.solve_triangular(L, B, lower=True, trans="T" if trans else "N")
    assert np.max(np.abs(got - want)) <= 1e-9 * max(1.0, np.abs(want).max())
    resid = (L.T if trans else L) @ got - B
    assert np.max(np.abs(resid)) <= 1e-11 * max(1.0, np.abs(got).max())


def test_ll_bar_extremes(G, O):
    """the table-driven log(1+exp(-a)) against the literal formula over the whole range, incl. the overflow quirk"""
    a = np.concatenate([np.linspace(-60, 60, 4001), [-745.0, -709.0, -708.0, -40.0, -39.999, 39.999, 40.0, 700.0, 0.0, 1e-300, -1e-300]])
    f = a.reshape(-1, 1); y = np.ones_like(f); mu = np.zeros_like(f)
    for chunk in (slice(0, 4001), slice(4001, None)):
        got = np.array([G.ll_bar(f[i:i + 1], y[i:i + 1], mu[i:i + 1])[0] for i in range(*chunk.indices(len(a)))][:400]) if False else None
    # one column per value: n = 1
    got = G.ll_bar(f.T.copy(), y.T.copy(), mu.T.copy())
    with np.errstate(over="ignore"):
        want = -np.log(1 + np.exp(-a))
    finite = np.isfinite(want)
    assert np.array_equal(np.isfinite(got), finite)          # -inf exactly where the reference overflows (a < -709.78)
    assert np.max(np.abs(got[finite] - want[finite]) / np.maximum(1.0, np.abs(want[finite]))) <= 1e-15


def test_ll_bar(G, O):
    prob = make_problem(300, 20, seed=3)
    rs = np.random.RandomState(1)
    f = rs.randn(300, 20) * 2; mu = rs.randn(300, 20)
    got = G.ll_bar(f, prob["y"], mu)
    want = np.array([O.ll_bar(f[:, j], prob["y"][:, j], mu[:, j]) for j in range(20)])
    assert np.max(np.abs(got - want) / np.abs(want)) <= 1e-12


# ---------------------------------------------------------------------------------------------------------------------
# step-level parity through the resident sampler: same state, same addressed variates, one step
# ---------------------------------------------------------------------------------------------------------------------
def _state(G, O, n, m, seed, missing, fstar_mode=0):
    from gpirt_b200 import _lib
    prob = make_problem(n, m, seed=seed, missing=missing, grid_theta=True)
    s = G.Sampler(prob["y"], prob["theta"], prob["pm"], prob["psd"], prob["pstep"], seed=seed + 77, fstar_mode=fstar_mode)
    rs = np.random.RandomState(seed + 1)
    L = s.get(_lib.CHOL)
    f = L @ rs.randn(n, m)
    beta = rs.randn(2, m)
    s.set(_lib.F, f); s.set(_lib.BETA, beta)
    return prob, s, L, f, beta


@pytest.mark.parametrize("n,m,missing", [(40, 12, 0.1), (100, 50, 0.05), (300, 64, 0.0), (1100, 20, 0.1), (2500, 6, 0.0)])
def test_step_draw_f(G, O, n, m, missing):
    from gpirt_b200 import _lib
    prob, s, L, f, beta = _state(G, O, n, m, seed=n + m, missing=missing)
    sweep = 3
    s.step(_lib.STEP_DRAW_F, sweep)
    nu = s.get(_lib.NU); f_new = s.get(_lib.F); nprop = s.get(_lib.ESS_NPROP).astype(int)
    rng = O.Rng.keyed(n + m + 77); rng.set_sweep(sweep)
    mu = O.linear_mean(prob["theta"], beta)
    fo, npo = O.draw_f(f, prob["y"], L, mu, rng)
    # proposals nu = L z
    z = np.array([[O.keyed_normal(n + m + 77, sweep, O.P_ESS_Z, j, i) for j in range(m)] for i in range(n)])
    assert np.max(np.abs(nu - L @ z)) <= 1e-12 * max(1.0, np.abs(nu).max())
    assert np.array_equal(nprop, npo), "ESS shrink counts must match the oracle"
    assert np.max(np.abs(f_new - fo)) <= 1e-9
    s.close()


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("n,m,missing", [(40, 12, 0.1), (100, 50, 0.05), (300, 33, 0.0)])
def test_step_draw_fstar(G, O, n, m, missing, mode):
    from gpirt_b200 import _lib
    prob, s, L, f, beta = _state(G, O, n, m, seed=n * 3 + m, missing=missing, fstar_mode=mode)
    sweep = 2
    s.step(_lib.STEP_DRAW_FSTAR, sweep)
    fs = s.get(_lib.FSTAR); sd = s.get(_lib.FSTAR_S); mean = s.get(_lib.FSTAR_MEAN)
    ts, _ = O.grid()
    rng = O.Rng.keyed(n * 3 + m + 77); rng.set_sweep(sweep)
    fso, so, meano = O.draw_fstar(f, prob["theta"], ts, L, O.linear_mean(ts, beta), rng)
    mu_star = O.linear_mean(ts, beta)
    assert np.max(np.abs(sd - so)) <= 1e-9
    assert np.max(np.abs((mean + mu_star) - meano)) <= 1e-8 * max(1.0, np.abs(meano).max())
    assert np.max(np.abs(fs - fso)) <= 1e-8 * max(1.0, np.abs(fso).max())
    s.close()


@pytest.mark.parametrize("n,m,missing", [(40, 12, 0.1), (100, 50, 0.05), (300, 64, 0.0), (700, 150, 0.3)])
def test_step_draw_theta(G, O, n, m, missing):
    from gpirt_b200 import _lib
    prob, s, L, f, beta = _state(G, O, n, m, seed=n * 5 + m, missing=missing)
    rs = np.random.RandomState(5)
    ts, prior = O.grid()
    fstar = np.asfortranarray(0.8 * rs.randn(1001, m).cumsum(axis=0) * 0.05 + rs.randn(1, m))
    s.set(_lib.FSTAR, fstar)
    sweep = 9
    s.step(_lib.STEP_DRAW_THETA, sweep)
    th = s.get(_lib.THETA); idx = s.get(_lib.THETA_IDX).astype(int); logp = s.get(_lib.LOGP)
    rng = O.Rng.keyed(n * 5 + m + 77); rng.set_sweep(sweep)
    tho, idxo, logpo = O.draw_theta(ts, prob["y"], prior, fstar, rng, mode=1)
    want_ll = logpo - prior[None, :]
    assert np.max(np.abs(logp - want_ll) / np.maximum(1.0, np.abs(want_ll))) <= 1e-12
    assert np.array_equal(idx, idxo), "grid indices must match the oracle (stabilised CDF)"
    assert np.array_equal(th, tho), "theta values are grid points: bit-exact"
    s.close()


@pytest.mark.parametrize("n,m,missing", [(130, 129, 0.0), (1100, 700, 0.0), (4096, 300, 0.0),
                                         (130, 129, 0.1), (1100, 700, 0.03), (257, 1000, 0.3)])
def test_theta_int8_tensor_core_path_matches_fp64_path(G, O, n, m, missing, monkeypatch):
    """tcgen05 int8 (exact integer) contraction vs the FP64 DMMA contraction vs the oracle; with missing cells the
    int8 path adds a second product of the observed mask |y| with the digit planes of D = log 2cosh(f*/2)"""
    from gpirt_b200 import _lib
    prob = make_problem(n, m, seed=n + m, missing=missing, grid_theta=True)
    rs = np.random.RandomState(7)
    fstar = np.asfortranarray(rs.randn(1001, m).cumsum(axis=0) * 0.04 + 3.0 * rs.randn(1, m))
    fstar[17, 3] = 0.0; fstar[500, :] *= 1e-6; fstar[900, 0] = 37.5        # zeros, tiny row, large entry
    out = {}
    for flag in ("1", "0"):
        monkeypatch.setenv("GPIRT_THETA_INT8", flag)
        s = G.Sampler(prob["y"], prob["theta"], seed=5)
        s.set(_lib.FSTAR, fstar)
        s.step(_lib.STEP_DRAW_THETA, 3)
        out[flag] = (s.get(_lib.LOGP), s.get(_lib.THETA_IDX).astype(int))
        s.close()
    ts, prior = O.grid()
    rng = O.Rng.keyed(5); rng.set_sweep(3)
    _, idxo, logpo = O.draw_theta(ts, prob["y"], prior, fstar, rng, mode=1)
    want = logpo - prior[None, :]
    for flag in ("1", "0"):
        assert np.max(np.abs(out[flag][0] - want) / np.maximum(1.0, np.abs(want))) <= 1e-12, flag
        assert np.array_equal(out[flag][1], idxo), flag
    assert np.max(np.abs(out["1"][0] - out["0"][0]) / np.maximum(1.0, np.abs(want))) <= 2e-13


@pytest.mark.parametrize("n,m,missing", [(40, 12, 0.1), (100, 50, 0.05), (1100, 20, 0.0), (2500, 6, 0.1)])
def test_step_draw_beta(G, O, n, m, missing):
    from gpirt_b200 import _lib
    prob, s, L, f, beta = _state(G, O, n, m, seed=n * 7 + m, missing=missing)
    sweep = 4
    s.step(_lib.STEP_DRAW_BETA, sweep)
    b = s.get(_lib.BETA)
    rng = O.Rng.keyed(n * 7 + m + 77); rng.set_sweep(sweep)
    bo, acc = O.draw_beta(beta, prob["theta"], prob["y"], f, prob["pm"], prob["psd"], prob["pstep"], rng)
    assert np.max(np.abs(b - bo)) <= 1e-13
    assert 0 < acc.sum() < acc.size or m < 8
    s.close()


# ---------------------------------------------------------------------------------------------------------------------
# lock-step chains: the whole sampler against the oracle's gpirtMCMC restatement, same seed
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,m,S,B,mode", [(2, 1, 1, 1, 0), (5, 3, 2, 0, 0), (30, 10, 3, 2, 0), (30, 10, 3, 2, 1), (100, 40, 2, 1, 0),
                                          (257, 33, 2, 0, 0), (400, 150, 3, 1, 0), (400, 150, 2, 1, 1), (640, 300, 2, 1, 0)])
def test_lockstep_chain(G, O, n, m, S, B, mode):
    # n = 400: pipelined sweep + int8 theta path;  n = 640: also the fixed-point tensor-core products for L Z and f*
    prob = make_problem(n, m, seed=n + 11, missing=0.08 if n not in (400, 640) else 0.0)
    seed = 4242 + n
    from gpirt_b200 import ResponseMatrix
    got = G.gpirtMCMC(ResponseMatrix(prob["y"]), S, B, beta_prior_means=prob["pm"], beta_prior_sds=prob["psd"],
                      beta_proposal_sds=prob["pstep"], theta_init=prob["theta"], seed=seed, fstar_mode=mode)
    rng = O.Rng.keyed(seed)
    want = O.mcmc(prob["y"], prob["theta"], S, B, prob["pm"], prob["psd"], prob["pstep"], rng, theta_cdf_mode=1)
    assert got["theta"].shape == (S + 1, n) and got["beta"].shape == (2, m, S + 1)
    assert got["f"].shape == (n, m, S + 1) and got["IRFs"].shape == (1001, m)
    assert np.array_equal(got["theta"][0], prob["theta"]), "row 0 holds the initial values (gpirtMCMC.cpp:53)"
    assert np.array_equal(got["theta"], want["theta"]), "theta draws (grid points) must be identical"
    assert np.max(np.abs(got["beta"] - want["beta"])) <= 1e-9
    assert np.max(np.abs(got["f"] - want["f"])) <= 1e-7
    assert np.max(np.abs(got["IRFs"] - want["IRFs"])) <= 1e-7


def test_chain_fixed_point_products_match_dmma_products(G, monkeypatch):
    """the same chain with nu = L Z and the f* product on the int8 tensor cores (dgemm_i8.cu) and on FP64 DMMA"""
    from gpirt_b200 import ResponseMatrix
    prob = make_problem(700, 320, seed=99, missing=0.05)
    out = {}
    for flag in ("1", "0"):
        monkeypatch.setenv("GPIRT_GEMM_INT8", flag)
        out[flag] = G.gpirtMCMC(ResponseMatrix(prob["y"]), 4, 2, beta_prior_means=prob["pm"], beta_prior_sds=prob["psd"],
                                beta_proposal_sds=prob["pstep"], theta_init=prob["theta"], seed=77)
    a, b = out["1"], out["0"]
    assert np.array_equal(a["theta"], b["theta"])
    assert np.max(np.abs(a["beta"] - b["beta"])) <= 1e-10
    assert np.max(np.abs(a["f"] - b["f"])) <= 1e-9
    assert np.max(np.abs(a["IRFs"] - b["IRFs"])) <= 1e-9


@pytest.mark.parametrize("n,m", [(100, 40), (400, 150), (700, 320), (1100, 260), (2304, 260), (6145, 260), (9000, 260)])
def test_chain_blocked_substitution_solves_match_inverse_route(G, O, n, m, monkeypatch):
    """GPIRT_SOLVE_MODE=1 (the default when items are sharded over GPUs, and for n > 6144): L^-1 K* and L^-T(.) by blocked
    substitution with the 128-block inverses, forward steps trailing the Cholesky panels, instead of L^-1 + triangular
    products (draw-fstar.cpp:19,24).  Same chain as the inverse route, and in lock-step with the oracle.  n >= 1024: the
    backward pass runs on 512 / 1024-wide diagonal-block inverses (n = 2304: two full 1024-blocks and a ragged one;
    n = 6145: a one-row last panel; n = 9000: ragged pairs at the levels 256 and 512)."""
    from gpirt_b200 import ResponseMatrix
    prob = make_problem(n, m, seed=n + 5, missing=0.04)
    out = {}
    for flag in ("1", "0"):
        monkeypatch.setenv("GPIRT_SOLVE_MODE", flag)
        out[flag] = G.gpirtMCMC(ResponseMatrix(prob["y"]), 3, 1, beta_prior_means=prob["pm"], beta_prior_sds=prob["psd"],
                                beta_proposal_sds=prob["pstep"], theta_init=prob["theta"], seed=31)
    a, b = out["1"], out["0"]
    assert np.array_equal(a["theta"], b["theta"])
    assert np.max(np.abs(a["beta"] - b["beta"])) <= 1e-10
    assert np.max(np.abs(a["f"] - b["f"])) <= 1e-8
    assert np.max(np.abs(a["IRFs"] - b["IRFs"])) <= 1e-8
    if n <= 400:
        rng = O.Rng.keyed(31)
        want = O.mcmc(prob["y"], prob["theta"], 3, 1, prob["pm"], prob["psd"], prob["pstep"], rng, theta_cdf_mode=1)
        assert np.array_equal(a["theta"], want["theta"])
        assert np.max(np.abs(a["f"] - want["f"])) <= 1e-7
        assert np.max(np.abs(a["IRFs"] - want["IRFs"])) <= 1e-7


# calls that change or re-time the sampler's state between sweeps: each drops what a pipelined sweep leaves for the next
_INTERRUPTS = {
    "set": lambda s, lib: s.set(lib.BETA, s.get(lib.BETA)),
    "step": lambda s, lib: s.step(lib.STEP_REBUILD, 0),
    "set_pipeline": lambda s, lib: s.set_pipeline(True),
    "time_factorisation": lambda s, lib: s.time_factorisation(1),
}


@pytest.mark.parametrize("n,m,route,interrupt",
                         [pytest.param(100, 60, "0", None, id="100-60-0"), pytest.param(640, 300, "0", None, id="640-300-0")]
                         + [pytest.param(640, 300, "0", i, id="640-300-0-" + i) for i in _INTERRUPTS]
                         + [pytest.param(640, 300, "1", None, id="640-300-1"), pytest.param(1152, 260, "1", None, id="1152-260-1")]
                         + [pytest.param(1152, 260, "1", i, id="1152-260-1-" + i) for i in _INTERRUPTS]
                         + [pytest.param(9000, 300, None, None, id="9000-300-default")])
def test_graph_replayed_sweeps_equal_eager_sweeps(G, n, m, route, interrupt, monkeypatch):
    """With the per-step timers off every sweep after the first is ONE CUDA-graph launch — captured from the very launch
    sequence of the eager sweep, for n > 256 the pipelined one with its five streams forked and joined inside the graph
    (stream priorities carried as per-node launch attributes).  Same kernels, same addressed RNG: the state after 6 sweeps
    must be bit-identical to 6 eager sweeps, on both K*-solve routes (route None: the default, substitution for n > 6144).
    With `interrupt`, both samplers make that call after the 4th sweep: the chain must resume — as a graph replay on the
    graph sampler — and agree with a chain that had no call (nu is then formed in one product instead of in slices)."""
    from gpirt_b200 import _lib
    if route is None:
        monkeypatch.delenv("GPIRT_SOLVE_MODE", raising=False)
    else:
        monkeypatch.setenv("GPIRT_SOLVE_MODE", route)
    prob = make_problem(n, m, seed=n + 3, missing=0.03)

    def run(use_graph, call):
        s = G.Sampler(prob["y"], prob["theta"], prob["pm"], prob["psd"], prob["pstep"], seed=77, use_graph=use_graph)
        s.set_timing(False)
        s.init_draws()
        s.sweep(4)
        if call is not None:
            _INTERRUPTS[call](s, _lib)
        at_call = s.uses(5)
        s.sweep(2, accumulate_irf=True)
        assert s.uses(4) == (1 if route is None else int(route))
        replays = s.uses(5)
        assert (replays >= 4) if use_graph == 0 else (replays == 0), "graph replay must be the path that ran (or not)"
        if use_graph == 0 and call is not None:
            assert replays > at_call, "graph replay must resume after the call"
        out = {k: s.get(f) for k, f in (("theta", _lib.THETA), ("beta", _lib.BETA), ("f", _lib.F), ("fstar", _lib.FSTAR),
                                        ("irf", _lib.IRF_SUM), ("L", _lib.CHOL))}
        s.close()
        return out

    state = {use_graph: run(use_graph, interrupt) for use_graph in (0, -1)}
    for k in state[0]:
        assert np.array_equal(state[0][k], state[-1][k]), k
    if interrupt is not None:
        plain = run(0, None)
        assert np.array_equal(state[0]["theta"], plain["theta"])
        assert np.max(np.abs(state[0]["beta"] - plain["beta"])) <= 1e-10
        assert np.max(np.abs(state[0]["f"] - plain["f"])) <= 1e-9


def test_senate116_short_chain(G, O):
    import warnings
    import gpirt_b200
    codes, _, _ = gpirt_b200.senate116()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        y = gpirt_b200.response_matrix(codes)
    assert y.shape == (100, 418)
    theta0 = np.random.RandomState(116).randn(100)
    got = G.gpirtMCMC(y, 2, 1, theta_init=theta0, seed=116)
    rng = O.Rng.keyed(116)
    m = y.shape[1]
    want = O.mcmc(np.asarray(y), theta0, 2, 1, np.zeros((2, m)), np.full((2, m), 3.0), np.full((2, m), 0.1), rng,
                  theta_cdf_mode=0)   # strict reference mode is finite on senate116 (SURVEY F3)
    assert np.array_equal(got["theta"], want["theta"])
    assert np.max(np.abs(got["beta"] - want["beta"])) <= 1e-9
    assert np.max(np.abs(got["f"] - want["f"])) <= 1e-7
    assert np.max(np.abs(got["IRFs"] - want["IRFs"])) <= 1e-7


@pytest.mark.parametrize("name", ["tiny_8x5", "small_100x37", "odd_257x12"])
def test_golden_chains_from_the_compiled_reference(G, name):
    """CUDA sampler vs the committed outputs of the reference's OWN sources (tests/golden/make_golden.py), same seed"""
    import os
    from gpirt_b200 import ResponseMatrix
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name + ".npz"))
    got = G.gpirtMCMC(ResponseMatrix(g["y"]), int(g["S"]), int(g["B"]), theta_init=g["theta_init"], seed=int(g["seed"]))
    assert np.array_equal(got["theta"], g["theta"]), "theta draws (grid points) identical to the reference"
    assert np.max(np.abs(got["beta"] - g["beta"])) <= 1e-9
    assert np.max(np.abs(got["f"] - g["f"])) <= 1e-7
    assert np.max(np.abs(got["IRFs"] - g["IRFs"])) <= 1e-7


def test_golden_senate116_from_the_compiled_reference(G):
    import os
    from gpirt_b200 import ResponseMatrix
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "senate116_100x418.npz"))
    y = g["y_int8"].astype(np.float64); y[y == 0] = np.nan
    got = G.gpirtMCMC(ResponseMatrix(y), int(g["S"]), int(g["B"]), theta_init=g["theta_init"], seed=int(g["seed"]))
    assert np.array_equal(got["theta"], g["theta"])
    assert np.max(np.abs(got["beta"] - g["beta"])) <= 1e-9
    assert np.max(np.abs(got["f"][:, :, -1] - g["f_last"])) <= 1e-7
    assert np.max(np.abs(got["IRFs"][::10] - g["IRFs_every10"])) <= 1e-7


def test_senate116_posterior_summaries_agree_within_monte_carlo_error(G, O):
    """north-star check 3: theta posterior means and item response curves on senate116 agree between independent
    chains of the CUDA sampler (different seeds) and an independent chain of the CPU oracle, up to Monte Carlo error
    (the model is identified up to reflection, so chains are sign-aligned first)"""
    import warnings
    import gpirt_b200
    codes, _, _ = gpirt_b200.senate116()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        y = gpirt_b200.response_matrix(codes)
    n, m = y.shape
    theta0 = np.random.RandomState(3).randn(n)
    runs = [G.gpirtMCMC(y, 400, 200, theta_init=theta0, seed=sd, store_f=False) for sd in (101, 202)]
    means = [r["theta"][1:].mean(axis=0) for r in runs]
    sds = [r["theta"][1:].std(axis=0) for r in runs]
    def fitted(run, mean):   # P(yea) of respondent i on item j at the chain's own theta estimate: location/reflection-free
        idx = np.clip(np.rint((mean + 5.0) * 100).astype(int), 0, 1000)
        return run["IRFs"][idx, :]

    def z(v):                # the latent scale is only weakly identified (N(0,1) prior): compare standardised positions
        return (v - v.mean()) / v.std()

    c01 = np.corrcoef(means[0], means[1])[0, 1]
    assert abs(c01) > 0.98
    assert np.median(np.abs(z(means[0]) - np.sign(c01) * z(means[1]))) < 0.1
    assert np.mean(np.abs(fitted(runs[0], means[0]) - fitted(runs[1], means[1]))) < 0.05
    # an independent (short) oracle chain in strict reference mode lands in the same place
    orc = O.mcmc(np.asarray(y), theta0, 25, 15, np.zeros((2, m)), np.full((2, m), 3.0), np.full((2, m), 0.1), O.Rng.keyed(909),
                 theta_cdf_mode=0)
    om = orc["theta"][1:].mean(axis=0)
    c = np.corrcoef(means[0], om)[0, 1]
    assert abs(c) > 0.95
    assert np.median(np.abs(z(means[0]) - np.sign(c) * z(om))) < 0.4    # 40 CPU sweeps only: the short chain is still spreading out
    # (fitted probabilities of a 40-sweep CPU chain are not sharp enough to compare; draw-by-draw agreement with the
    #  reference is what the lock-step and golden tests establish)
    assert sds[0].mean() > 0.0


def test_interrupt_and_bad_y(G):
    from gpirt_b200._lib import GpirtError, ERR_INTERRUPT, ERR_Y_VALUE
    prob = make_problem(20, 6, seed=1)
    from gpirt_b200 import ResponseMatrix
    with pytest.raises(GpirtError) as e:
        G.gpirtMCMC(ResponseMatrix(prob["y"]), 5, 5, theta_init=prob["theta"], seed=1, progress=lambda pct: pct >= 30.0)
    assert e.value.status == ERR_INTERRUPT
    bad_raw = np.array(prob["y"]); bad_raw[0, 0] = 6.0
    s_err = None
    try:
        G.Sampler(bad_raw, prob["theta"])
    except GpirtError as ex:
        s_err = ex.status
    assert s_err == ERR_Y_VALUE
