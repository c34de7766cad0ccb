"""The ctypes mirror of gpirt_b200_chains (opts.chains, several chains in one call) against the real header, and the
argument checks gpirtMCMC(chains=...) makes before anything reaches the device — no GPU needed."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# offsets of gpirt_b200_opts before the chains field was appended (every one must stay where it was)
OPTS_BEFORE = ["seed", "device", "fstar_mode", "skip_f_draws", "use_graph", "rank", "world_size", "m_global", "item_offset",
               "nccl_unique_id", "thin", "reserved0", "f_mean_out", "f_sd_out", "fit", "irf"]


def test_chains_struct_layout_matches_header(tmp_path):
    from gpirt_b200._lib import Chains, Opts
    fields = [name for name, _ in Chains._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "gpirt_b200.h"\nint main(void) {\n'
                   + "".join('  printf("%s %%zu\\n", offsetof(gpirt_b200_chains, %s));\n' % (f, f) for f in fields)
                   + '  printf("sizeof %zu\\n", sizeof(gpirt_b200_chains));\n'
                   + "".join('  printf("opts.%s %%zu\\n", offsetof(gpirt_b200_opts, %s));\n' % (f, f)
                             for f in OPTS_BEFORE + ["chains"])
                   + '  printf("opts.sizeof %zu\\n", sizeof(gpirt_b200_opts));\n  return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = dict(line.split() for line in subprocess.check_output([str(exe)], text=True).splitlines())
    for f in fields:
        assert int(got[f]) == getattr(Chains, f).offset, f
    assert int(got["sizeof"]) == C.sizeof(Chains)
    for f in OPTS_BEFORE:
        assert int(got["opts." + f]) == getattr(Opts, f).offset, f
    assert int(got["opts.chains"]) == Opts.chains.offset == Opts.irf.offset + C.sizeof(C.c_void_p)   # right after irf
    assert int(got["opts.sizeof"]) == C.sizeof(Opts)


def test_previous_opts_offsets_are_unchanged():
    """the offsets of the fields before chains, as the previous release of the header laid them out (LP64)"""
    from gpirt_b200._lib import Opts
    want = dict(seed=0, device=8, fstar_mode=12, skip_f_draws=16, use_graph=20, rank=24, world_size=28, m_global=32,
                item_offset=40, nccl_unique_id=48, thin=56, reserved0=60, f_mean_out=64, f_sd_out=72, fit=80, irf=88)
    assert {f: getattr(Opts, f).offset for f in OPTS_BEFORE} == want
    assert Opts.chains.offset == 96


def test_default_opts_request_one_chain():
    from gpirt_b200.sampler import make_opts
    assert not make_opts(seed=1).chains


def _no_device(monkeypatch):
    from gpirt_b200 import _lib

    def no_device(*a, **k):
        raise AssertionError("the library was reached")
    monkeypatch.setattr(_lib, "load", no_device)


def _y():
    from gpirt_b200 import ResponseMatrix
    return ResponseMatrix(np.array([[1.0, -1.0, np.nan], [-1.0, 1.0, 1.0], [1.0, 1.0, -1.0]]))


@pytest.mark.parametrize("chains", [0, 33, -1, 2.0, "2", True, [2]])
def test_bad_chains_value_is_refused_on_the_host(chains, monkeypatch):
    import gpirt_b200.sampler as G
    _no_device(monkeypatch)
    with pytest.raises(ValueError, match="chains"):
        G.gpirtMCMC(_y(), 4, 0, theta_init=np.zeros((3, 2)), chains=chains)


@pytest.mark.parametrize("theta_init", [np.zeros(3), np.zeros((3, 3)), np.zeros((2, 2)), np.zeros((3, 2, 1))])
def test_theta_init_of_the_wrong_shape_is_refused(theta_init, monkeypatch):
    import gpirt_b200.sampler as G
    _no_device(monkeypatch)
    with pytest.raises(ValueError, match="theta_init"):
        G.gpirtMCMC(_y(), 4, 0, theta_init=theta_init, chains=2)


@pytest.mark.parametrize("seed", [[1], [1, 2, 3], ()])
def test_seed_sequence_of_the_wrong_length_is_refused(seed, monkeypatch):
    import gpirt_b200.sampler as G
    _no_device(monkeypatch)
    with pytest.raises(ValueError, match="seed"):
        G.gpirtMCMC(_y(), 4, 0, theta_init=np.zeros((3, 2)), chains=2, seed=seed)


@pytest.mark.parametrize("kw", [dict(shard=(0, 2, 6, 0, b"\0" * 128)), dict(predictive=True), dict(irf_band=0.9),
                                dict(store_fstar=True), dict(f_summary=True)])
def test_chains_with_features_not_built_for_them_are_refused(kw, monkeypatch):
    import gpirt_b200.sampler as G
    _no_device(monkeypatch)
    with pytest.raises(ValueError, match="chains cannot be combined with %s" % next(iter(kw))):
        G.gpirtMCMC(_y(), 4, 0, theta_init=np.zeros((3, 2)), chains=2, **kw)


def test_chain_diagnostics_without_chains_is_refused(monkeypatch):
    import gpirt_b200.sampler as G
    _no_device(monkeypatch)
    with pytest.raises(ValueError, match="chain_diagnostics"):
        G.gpirtMCMC(_y(), 4, 0, theta_init=np.zeros(3), chain_diagnostics=True)
