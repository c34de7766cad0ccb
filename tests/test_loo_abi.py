"""The ctypes mirror of gpirt_b200_loo (opts.loo, PSIS-LOO) against the real header, the argument checks gpirtMCMC(loo=...)
makes before anything reaches the device, and the numpy port of the definitions (tests/psis_loo_numpy.py) on columns
with known answers — no GPU needed."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import psis_loo_numpy as P

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# offsets of gpirt_b200_opts before the loo field was appended (every one must stay where it was, LP64)
OPTS_BEFORE = dict(seed=0, device=8, fstar_mode=12, skip_f_draws=16, use_graph=20, rank=24, world_size=28, m_global=32,
                   item_offset=40, nccl_unique_id=48, thin=56, reserved0=60, f_mean_out=64, f_sd_out=72, fit=80, irf=88,
                   chains=96, ppc=104)


def test_loo_struct_layout_matches_header(tmp_path):
    from gpirt_b200._lib import Loo, Opts
    fields = [name for name, _ in Loo._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "gpirt_b200.h"\nint main(void) {\n'
                   + "".join('  printf("%s %%zu\\n", offsetof(gpirt_b200_loo, %s));\n' % (f, f) for f in fields)
                   + '  printf("sizeof %zu\\n", sizeof(gpirt_b200_loo));\n'
                   + "".join('  printf("opts.%s %%zu\\n", offsetof(gpirt_b200_opts, %s));\n' % (f, f)
                             for f in list(OPTS_BEFORE) + ["loo"])
                   + '  printf("opts.sizeof %zu\\n", sizeof(gpirt_b200_opts));\n  return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = dict(line.split() for line in subprocess.check_output([str(exe)], text=True).splitlines())
    for f in fields:
        assert int(got[f]) == getattr(Loo, f).offset, f
    assert int(got["sizeof"]) == C.sizeof(Loo) == 112
    for f, off in OPTS_BEFORE.items():
        assert int(got["opts." + f]) == getattr(Opts, f).offset == off, f
    assert int(got["opts.loo"]) == Opts.loo.offset == 112   # right after ppc
    assert int(got["opts.sizeof"]) == C.sizeof(Opts) == 120


def test_default_opts_request_no_loo():
    from gpirt_b200.sampler import make_opts
    assert not make_opts(seed=1).loo


def test_psis_loo_is_exported():
    from gpirt_b200 import _lib
    assert "gpirt_b200_psis_loo" in _lib.EXPORTS


def _no_device(monkeypatch):
    from gpirt_b200 import _lib

    def no_device(*a, **k):
        raise AssertionError("the library was reached")
    monkeypatch.setattr(_lib, "load", no_device)


def _y():
    from gpirt_b200 import ResponseMatrix
    return ResponseMatrix(np.array([[1.0, -1.0, np.nan], [-1.0, 1.0, 1.0], [1.0, 1.0, -1.0]]))


def test_loo_with_chains_is_refused(monkeypatch):
    import gpirt_b200.sampler as G
    _no_device(monkeypatch)
    with pytest.raises(ValueError, match="chains cannot be combined with loo"):
        G.gpirtMCMC(_y(), 4, 0, theta_init=np.zeros((3, 2)), chains=2, loo=True)


def test_loo_with_shard_is_refused(monkeypatch):
    import gpirt_b200.sampler as G
    _no_device(monkeypatch)
    with pytest.raises(ValueError, match="loo cannot be combined with shard"):
        G.gpirtMCMC(_y(), 4, 0, theta_init=np.zeros(3), loo=True, shard=(0, 2, 6, 0, b"\0" * 128))


def test_psis_loo_needs_a_matrix(monkeypatch):
    import gpirt_b200.sampler as G
    _no_device(monkeypatch)
    with pytest.raises(ValueError, match="cols x S"):
        G.psis_loo(np.zeros(5))


# ---- the numpy port on columns with known answers ----------------------------------------------------------------
def _raw_is_loo(ll):
    """importance sampling LOO with the raw ratios 1 / sigma: -log mean_s exp(-ll_s)"""
    return -np.log(np.mean(np.exp(-ll), axis=1))


@pytest.mark.parametrize("S,M", [(1, 1), (4, 1), (5, 1), (6, 2), (20, 4), (21, 5), (22, 5), (100, 20), (225, 45),
                                 (226, 46), (1000, 95), (5000, 213)])
def test_tail_length(S, M):
    assert P.tail_len(S) == M


def test_threshold():
    assert P.k_threshold(1) == -np.inf
    assert P.k_threshold(10) == 0.0
    assert P.k_threshold(1000) == pytest.approx(2.0 / 3.0)
    assert P.k_threshold(10 ** 6) == 0.7
    assert np.isnan(P.k_threshold(0))


def test_draw_order_sum_equals_the_loop_over_draws():
    """lpd needs the sum of sigma in draw order, bit for bit as the device adds it; cumsum must give the loop's bits"""
    ll = P.adversarial(5000, np.random.default_rng(5))
    sig = np.exp(ll)
    acc = sig[:, 0].copy()
    for s in range(1, sig.shape[1]):
        acc = acc + sig[:, s]
    assert np.array_equal(P.draw_order_sum(sig), acc)
    assert not np.array_equal(np.sum(sig, axis=1), acc)   # the pairwise sum differs: the test can tell the orders apart


def test_constant_column():
    ll = np.full((3, 50), -0.3)
    ll[1] = -2.0
    ll[2] = -1e-9
    r = P.psis_loo(ll)
    assert np.all(np.isinf(r["k"]))
    assert np.allclose(r["elpd"], ll[:, 0], rtol=0.0, atol=1e-14)   # log S - log S cancels: absolute error only
    assert np.allclose(r["p_loo"], 0.0, atol=1e-14)


@pytest.mark.parametrize("S", [1, 2, 4, 19, 20])
def test_fewer_than_five_tail_draws_are_not_smoothed(S):
    rs = np.random.default_rng(S)
    ll = -rs.exponential(1.0, (7, S))
    r = P.psis_loo(ll)
    assert P.tail_len(S) < 5
    assert np.all(r["k"] == np.inf)
    assert np.allclose(r["elpd"], _raw_is_loo(ll), rtol=1e-13, atol=1e-14)
    if S == 1:
        assert np.array_equal(r["elpd"], ll[:, 0]) and np.allclose(r["p_loo"], 0.0, atol=1e-15)


def test_tail_tied_with_the_cutoff():
    """the M + 1 largest ratios are equal: the tail has no range, stays raw and k = inf"""
    S = 100
    M = P.tail_len(S)
    rs = np.random.default_rng(1)
    ll = -rs.uniform(0.0, 1.0, (4, S))
    ll[:, :M + 1] = -3.0
    r = P.psis_loo(ll)
    assert np.all(r["k"] == np.inf)
    assert np.allclose(r["elpd"], _raw_is_loo(ll), rtol=1e-13)


def test_tail_partly_tied_with_the_cutoff_has_x_star_zero():
    """a quarter of the tail equal to the cutoff: x* = 0, the grid is -inf and k = inf (raw tail)"""
    S = 100
    M = P.tail_len(S)
    rs = np.random.default_rng(2)
    ll = -rs.uniform(0.0, 1.0, (3, S))
    ll[:, :M // 2] = -3.0 - rs.uniform(0.0, 1.0, (3, M // 2))
    ll[:, M // 2:M + 1] = -3.0
    r = P.psis_loo(ll)
    assert np.all(r["k"] == np.inf)
    assert np.allclose(r["elpd"], _raw_is_loo(ll), rtol=1e-13)


@pytest.mark.parametrize("k_true", [0.0, 0.5, 1.2])
def test_pareto_shape_is_recovered(k_true):
    """ratios whose tail is generalized Pareto with shape k_true, S = 4000 (M = 190): the mean k over 40 columns lies
    within sampling error (sd of one estimate about (1 + k) / sqrt(M)) plus the pull of the prior toward 0.5"""
    S, cols = 4000, 40
    rs = np.random.default_rng(3)
    u = rs.uniform(size=(S, cols))
    w = -np.log(u) if k_true == 0.0 else (u ** -k_true - 1.0) / k_true + 1.0
    k = P.psis_loo(-np.log(w).T)["k"]
    M = P.tail_len(S)
    sd = (1.0 + k_true) / np.sqrt(M)
    prior = abs(0.5 - k_true) * 10.0 / (M + 10.0)
    assert abs(k.mean() - k_true) <= 4.0 * sd / np.sqrt(cols) + prior, k.mean()
    assert np.all(np.abs(k - k_true) <= 4.0 * sd + prior)
    thr = P.k_threshold(S)
    if k_true != 0.5:   # 0.5 lies within two sd of the threshold 2/3
        assert np.mean(k > thr) == (k_true > thr)

