"""Every launch shape of the per-item kernels against the CPU oracle, at the edges of their instantiations.

The elliptical slice sampler (ess_item) and the beta Metropolis step (beta_item) each run in one of three launch shapes
(kernels.cu): one CTA per item (k_ess<EPT>, k_beta<EPT>), persistent CTAs that claim items from an atomic queue and
prefetch the next item's columns with cp.async (k_ess_persist<EPT>, k_beta_persist<EPT>), and, beyond 4096
respondents, the streaming kernels.  EPT, the values each thread holds in registers, is 1, 2, 4 or 8 by n, and the
persistent kernels run once m exceeds the CTAs the device holds at once: 2 x (4 x 2 + 1) = 18 instantiations.

  thresholds   g = the largest m that still runs one CTA per item, per family and n, found by doubling and bisection
               (device-dependent: printed, never asserted)
  oracle       n on both sides of every EPT seam, m = g, g + 1 and 2g + 1: draw_f, draw_beta, draw_f again in one
               sampler (the second ESS launch must find its queue reset), on the items around g, the last item,
               adversarial columns in the first wave and among the queued items, and random items
  bits         one CTA per item and the persistent kernels give the same bits for the same columns
  ERR_ESS      a NaN column hits the 10 000-proposal cap in each shape without stalling the other items

Tolerances as in test_gpu_bench_shapes.py: ESS proposal counts identical, f to 1e-9 (relative above 1), beta to 1e-12."""
import numpy as np
import pytest

from conftest import make_problem

pytestmark = pytest.mark.gpu

ITEM_CTA, ITEM_PERSISTENT, ITEM_STREAM = 0, 1, 2
ESS, BETA = 0, 1                        # families; gpirt_b200_sampler_uses(s, 2 + family) is the shape of the last launch
FAMILY = ("ess", "beta")
ESS_ITER_CAP = 10000                    # kernels.cu: proposals before the sampler gives up with GPIRT_B200_ERR_ESS
SEAMS = [2, 32, 33, 255, 256, 257, 1023, 1024, 1025, 2047, 2048, 2049, 4095, 4096, 4097]
EMPTY, LAST, TAIL, EDGE40, BIG700 = range(5)   # adversarial column kinds, see _adversarial_y / _adversarial_state

_shapes = {}     # (n, m) -> (ESS shape, beta shape) of one probe
_g = {}          # n -> (g of the ESS, g of the beta step)
_covered = set()  # (family, EPT, shape) compared with the oracle


@pytest.fixture(scope="module")
def G():
    import gpirt_b200.sampler as g
    from gpirt_b200 import _lib
    assert _lib.load().gpirt_b200_device_count() > 0, "no CUDA device"
    return g


def _ept(n):
    """Values per thread of the register-resident kernels, restating item_cta_shape() in kernels.cu: 1 up to 256
    respondents, 2 up to 1024, 4 up to 2048, 8 up to 4096; 0 above 4096, where the streaming kernels run."""
    return 1 if n <= 256 else 2 if n <= 1024 else 4 if n <= 2048 else 8 if n <= 4096 else 0


# ---- 1. the persistent threshold ------------------------------------------------------------------------------------
def _probe(G, n, m):
    """the launch shapes one ESS step and one beta step pick at n x m"""
    if (n, m) not in _shapes:
        from gpirt_b200 import _lib
        rs = np.random.RandomState(n + m)
        y = np.asfortranarray(np.where(rs.rand(n, m) < 0.5, 1.0, -1.0))
        s = G.Sampler(y, rs.randn(n), seed=1)
        s.set(_lib.BETA, np.zeros((2, m)))   # f starts at 0
        s.step(_lib.STEP_DRAW_F, 1)
        s.step(_lib.STEP_DRAW_BETA, 2)
        _shapes[(n, m)] = (s.uses(2), s.uses(3))
        s.close()
    return _shapes[(n, m)]


def _threshold(G, n):
    """(g_ess, g_beta) at n <= 4096: m <= g runs one CTA per item, m > g the persistent kernel"""
    if n not in _g:
        assert _probe(G, n, 1) == (ITEM_CTA, ITEM_CTA)
        lo, hi, m = [1, 1], [None, None], 1
        while None in hi:
            m *= 2
            assert m <= 1 << 20, "no persistent launch up to m = %d at n = %d" % (m, n)
            for fam, shape in enumerate(_probe(G, n, m)):
                if hi[fam] is None:
                    assert shape in (ITEM_CTA, ITEM_PERSISTENT)
                    if shape == ITEM_CTA:
                        lo[fam] = m
                    else:
                        hi[fam] = m
        for fam in (ESS, BETA):
            while hi[fam] - lo[fam] > 1:
                mid = (lo[fam] + hi[fam]) // 2
                if _probe(G, n, mid)[fam] == ITEM_CTA:
                    lo[fam] = mid
                else:
                    hi[fam] = mid
        _g[n] = tuple(lo)
    return _g[n]


@pytest.mark.parametrize("n", [n for n in SEAMS if n <= 4096])
def test_persistent_threshold(G, n):
    g = _threshold(G, n)
    for fam in (ESS, BETA):
        assert _probe(G, n, g[fam])[fam] == ITEM_CTA, "m = g runs one CTA per item"
        assert _probe(G, n, g[fam] + 1)[fam] == ITEM_PERSISTENT, "m = g + 1 runs the persistent kernel"


@pytest.mark.parametrize("m", [1, 4801])   # 4801 > 148 SMs x 32 CTAs: more items than any B200 grid holds at once
def test_streaming_shape_at_any_m(G, m):
    assert _probe(G, 4097, m) == (ITEM_STREAM, ITEM_STREAM)


# ---- adversarial item content ---------------------------------------------------------------------------------------
def _place(m, starts):
    """column -> kind: the five kinds laid out from each start (a later start wins where two overlap)"""
    cols = {}
    for s in starts:
        for k in range(5):
            if 0 <= s + k < m:
                cols[s + k] = k
    return cols


def _adversarial_y(y, cols, rs):
    """y of the adversarial columns, and respondent n // 3 with every item missing"""
    n = y.shape[0]
    y[n // 3, :] = np.nan
    for j, kind in cols.items():
        if kind == EMPTY:
            y[:, j] = np.nan
        elif kind == LAST:       # respondent n - 1: the last register slot in use, of the last thread in use
            y[:, j] = np.nan
            y[n - 1, j] = rs.choice([-1.0, 1.0])
        elif kind == TAIL:       # observed only in the last 16-byte chunk of the int8 column (ragged when n % 16 > 0)
            y[:16 * ((n - 1) // 16), j] = np.nan
            y[n - 1, j] = -1.0
        elif kind == BIG700:     # respondent n - 1 answers -1: the term y g = -709.7 is 0.08 from the overflow branch
            y[n - 1, j] = -1.0


def _adversarial_state(f, beta, cols):
    for j, kind in cols.items():
        if kind == EDGE40:       # |y g| = |40 + f| spans [39.9, 40.1], the end of the softplus table
            beta[:, j] = (40.0, 0.0)
            f[:, j] = np.linspace(-0.1, 0.1, f.shape[0])
        elif kind == BIG700:     # |y g| near 700: large finite terms, and proposals that overflow exp(-y g)
            beta[:, j] = (700.0, 0.0)
            f[-1, j] = 9.7


# ---- 2. every shape and seam against the oracle -------------------------------------------------------------------------
def _check_f(O, s, f, beta, y, theta, L, J, seed, sweep, nu_items):
    """one ESS step on the device against the oracle's draw_f of items J from the same f, beta; returns (f, shape)"""
    from gpirt_b200 import _lib
    s.step(_lib.STEP_DRAW_F, sweep)
    shape = s.uses(2)
    f1 = s.get(_lib.F); nprop = s.get(_lib.ESS_NPROP).astype(int)
    rng = O.Rng.keyed(seed); rng.set_sweep(sweep); rng.set_item_map(J)
    fo, npo = O.draw_f(f[:, J], y[:, J], L, O.linear_mean(theta, beta[:, J]), rng)
    bad = J[nprop[J] != npo]
    assert bad.size == 0, "sweep %d: ESS proposal counts differ from the oracle on items %s" % (sweep, bad)
    err = np.abs(f1[:, J] - fo) / np.maximum(1.0, np.abs(fo))
    assert np.max(err) <= 1e-9, "sweep %d: f differs on items %s" % (sweep, J[np.max(err, axis=0) > 1e-9])
    if nu_items:
        nu = s.get(_lib.NU)
        n = L.shape[0]
        for j in nu_items:      # the proposal itself: nu_j = L z_j (bound of test_gpu_bench_shapes.py)
            z = np.array([O.keyed_normal(seed, sweep, O.P_ESS_Z, int(j), i) for i in range(n)])
            tol = n * 2.0 ** -51 * 2.0 * np.abs(z).max() if n > 4096 else 1e-11
            assert np.max(np.abs(nu[:, j] - L @ z)) <= tol, "sweep %d: nu = L z on item %d" % (sweep, j)
    return f1, shape


def _check_beta(O, s, f, beta, prob, y, J, seed, sweep):
    """one beta step on the device against the oracle's draw_beta of items J; returns (beta, shape)"""
    from gpirt_b200 import _lib
    s.step(_lib.STEP_DRAW_BETA, sweep)
    shape = s.uses(3)
    b1 = s.get(_lib.BETA)
    rng = O.Rng.keyed(seed); rng.set_sweep(sweep); rng.set_item_map(J)
    bo, _ = O.draw_beta(beta[:, J], prob["theta"], y[:, J], f[:, J], prob["pm"][:, J], prob["psd"][:, J],
                        prob["pstep"][:, J], rng)
    err = np.max(np.abs(b1[:, J] - bo), axis=0)
    assert np.max(err) <= 1e-12, "sweep %d: beta differs on items %s" % (sweep, J[err > 1e-12])
    return b1, shape


def _oracle_case(G, O, n, m, g):
    """draw_f (s1), draw_beta (s2), draw_f (s3) in one sampler at n x m; g = (g_ess, g_beta), None beyond 4096"""
    from gpirt_b200 import _lib
    seed = 7919 * n + m
    rs = np.random.RandomState(seed)
    prob = make_problem(n, m, seed=seed, missing=0.05, grid_theta=True)
    y, theta = prob["y"], prob["theta"]
    # the adversarial columns in the first wave, at the first items taken from each queue, and at the end
    cols = _place(m, [2] + ([g[ESS], g[BETA]] if g else []) + [m - 5])
    _adversarial_y(y, cols, rs)
    s = G.Sampler(y, theta, prob["pm"], prob["psd"], prob["pstep"], seed=seed)
    L = s.get(_lib.CHOL)
    f = np.asfortranarray(L @ rs.randn(n, m)); beta = rs.randn(2, m)
    _adversarial_state(f, beta, cols)
    s.set(_lib.F, f); s.set(_lib.BETA, beta)

    edges = {0, 1, m - 1} | ({g[ESS] - 1, g[ESS], g[ESS] + 1, g[BETA] - 1, g[BETA], g[BETA] + 1} if g else set())
    J = np.array(sorted(({j for j in edges if 0 <= j < m} | set(cols) | set(rs.choice(m, min(m, 24), replace=False)))))
    nu_items = sorted({0, m - 1, min(g[ESS], m - 1) if g else m // 2, max(cols)})
    expect = [ITEM_STREAM if g is None else ITEM_CTA if m <= g[fam] else ITEM_PERSISTENT for fam in (ESS, BETA)]
    where = "n = %d, m = %d, g = %s" % (n, m, g)

    f1, shape = _check_f(O, s, f, beta, y, theta, L, J, seed, 1, nu_items)
    assert shape == expect[ESS], where
    b2, shape = _check_beta(O, s, f1, beta, prob, y, J, seed, 2)
    assert shape == expect[BETA], where
    _, shape = _check_f(O, s, f1, b2, y, theta, L, J, seed, 3, nu_items[:2])
    assert shape == expect[ESS], where
    s.close()
    _covered.add((ESS, _ept(n), expect[ESS]))
    _covered.add((BETA, _ept(n), expect[BETA]))


@pytest.mark.parametrize("n", SEAMS)
def test_item_kernels_against_the_oracle(G, O, n):
    if n > 4096:
        _oracle_case(G, O, n, 48, None)
        return
    g = _threshold(G, n)
    for m in sorted({g[ESS], g[ESS] + 1, 2 * g[ESS] + 1, g[BETA], g[BETA] + 1, 2 * g[BETA] + 1}):
        _oracle_case(G, O, n, m, g)


# ---- 4. the same columns give the same bits in either shape ------------------------------------------------------------
@pytest.mark.parametrize("n", [200, 700, 1500, 2049, 3000])
def test_bits_identical_across_launch_shapes(G, monkeypatch, n):
    """m_a = min g: one CTA per item in both families; m_b = 2 max g + 1: persistent in both.  The fixed-point L Z is
    forced on (its default depends on m) so that the proposals nu of the shared columns are the same bits too."""
    from gpirt_b200 import _lib
    g = _threshold(G, n)
    monkeypatch.setenv("GPIRT_GEMM_INT8", "1")
    ma, mb = min(g), 2 * max(g) + 1
    seed = 31 + n
    rs = np.random.RandomState(n)
    prob = make_problem(n, mb, seed=n, missing=0.05, grid_theta=True)
    cols = _place(mb, [2, ma - 5])
    _adversarial_y(prob["y"], cols, rs)

    def sampler(m):
        return G.Sampler(prob["y"][:, :m], prob["theta"], prob["pm"][:, :m], prob["psd"][:, :m], prob["pstep"][:, :m],
                         seed=seed)

    s = sampler(ma)
    f = np.asfortranarray(s.get(_lib.CHOL) @ rs.randn(n, mb)); beta = rs.randn(2, mb)
    s.close()
    _adversarial_state(f, beta, cols)
    runs = []
    for m in (ma, mb, mb):
        s = sampler(m)
        assert s.uses(1) == 1
        s.set(_lib.F, f[:, :m]); s.set(_lib.BETA, beta[:, :m])
        s.step(_lib.STEP_DRAW_F, 1)
        r = dict(nu=s.get(_lib.NU), f=s.get(_lib.F), nprop=s.get(_lib.ESS_NPROP), ess=s.uses(2))
        s.step(_lib.STEP_DRAW_BETA, 2)
        r.update(beta=s.get(_lib.BETA), beta_shape=s.uses(3))
        s.close()
        runs.append(r)
    a = runs[0]
    assert (a["ess"], a["beta_shape"]) == (ITEM_CTA, ITEM_CTA)
    for b in runs[1:]:
        assert (b["ess"], b["beta_shape"]) == (ITEM_PERSISTENT, ITEM_PERSISTENT)
        assert np.array_equal(b["nu"][:, :ma], a["nu"]), "precondition: the proposals of the shared columns"
        assert np.array_equal(b["f"][:, :ma], a["f"]) and np.array_equal(b["nprop"][:ma], a["nprop"])
        assert np.array_equal(b["beta"][:, :ma], a["beta"])
    for k in ("f", "nprop", "beta"):   # the queue hands out items in another order on every run
        assert np.array_equal(runs[1][k], runs[2][k])


# ---- 5. the proposal cap, in each shape --------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [ITEM_CTA, ITEM_PERSISTENT, ITEM_STREAM])
def test_ess_cap_in_each_shape(G, O, shape):
    """A NaN f column makes every log-likelihood NaN: its ESS stops at the cap and the step returns ERR_ESS.  The other
    items are still drawn as the oracle draws them (in the persistent shape the capped item is the first one taken
    from the queue), and a fresh sampler on the same finite state runs clean."""
    from gpirt_b200 import _lib
    if shape == ITEM_STREAM:
        n, m, bad = 4097, 12, 5
    else:
        n = 257
        g = _threshold(G, n)[ESS]
        m, bad = (min(g, 40), 5) if shape == ITEM_CTA else (g + 16, g)
    seed = 555 + shape
    rs = np.random.RandomState(seed)
    prob = make_problem(n, m, seed=seed, missing=0.05, grid_theta=True)
    y, theta = prob["y"], prob["theta"]
    s = G.Sampler(y, theta, prob["pm"], prob["psd"], prob["pstep"], seed=seed)
    L = s.get(_lib.CHOL)
    f = np.asfortranarray(L @ rs.randn(n, m)); beta = rs.randn(2, m)
    f_nan = f.copy(); f_nan[:, bad] = np.nan
    s.set(_lib.F, f_nan); s.set(_lib.BETA, beta)
    with pytest.raises(_lib.GpirtError) as e:
        s.step(_lib.STEP_DRAW_F, 1)
    assert e.value.status == _lib.ERR_ESS
    assert s.uses(2) == shape
    f1 = s.get(_lib.F); nprop = s.get(_lib.ESS_NPROP).astype(int)
    s.close()
    assert nprop[bad] == ESS_ITER_CAP
    J = np.array(sorted(({0, 1, bad - 1, bad + 1, m - 1} | set(rs.choice(m, min(m, 12), replace=False))) - {bad}))
    rng = O.Rng.keyed(seed); rng.set_sweep(1); rng.set_item_map(J)
    fo, npo = O.draw_f(f[:, J], y[:, J], L, O.linear_mean(theta, beta[:, J]), rng)
    assert np.array_equal(nprop[J], npo), "the capped item must not change the other items' draws"
    assert np.max(np.abs(f1[:, J] - fo)) <= 1e-9

    s = G.Sampler(y, theta, prob["pm"], prob["psd"], prob["pstep"], seed=seed)
    s.set(_lib.F, f); s.set(_lib.BETA, beta)
    s.step(_lib.STEP_DRAW_F, 1)
    assert s.uses(2) == shape
    J = np.append(J, bad)
    f1 = s.get(_lib.F); nprop = s.get(_lib.ESS_NPROP).astype(int)
    s.close()
    rng = O.Rng.keyed(seed); rng.set_sweep(1); rng.set_item_map(J)
    fo, npo = O.draw_f(f[:, J], y[:, J], L, O.linear_mean(theta, beta[:, J]), rng)
    assert np.array_equal(nprop[J], npo)
    assert np.max(np.abs(f1[:, J] - fo)) <= 1e-9
    _covered.add((ESS, _ept(n), shape))


# ---- every instantiation was compared with the oracle ----------------------------------------------------------------
def test_every_instantiation_met_the_oracle(capsys):
    with capsys.disabled():
        print("\n  largest m with one CTA per item (g), per family and n:")
        print("  %6s %8s %8s" % ("n", "ess", "beta"))
        for n in sorted(_g):
            print("  %6d %8d %8d" % (n, _g[n][ESS], _g[n][BETA]))
    want = {(fam, e, shape) for fam in (ESS, BETA) for e in (1, 2, 4, 8) for shape in (ITEM_CTA, ITEM_PERSISTENT)}
    want |= {(ESS, 0, ITEM_STREAM), (BETA, 0, ITEM_STREAM)}
    missing = sorted(want - _covered)
    assert not missing, "never compared with the oracle: %s" % [
        "%s EPT %d shape %d" % (FAMILY[fam], e, shape) for fam, e, shape in missing]
    assert len(want) == 18
