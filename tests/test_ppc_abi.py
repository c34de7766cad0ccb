"""The ctypes mirror of gpirt_b200_ppc (opts.ppc, posterior predictive checks) against the real header, and the argument
checks gpirtMCMC(ppc=...) and ppc_pairs() make before anything reaches the device — no GPU needed."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# offsets of gpirt_b200_opts before the ppc field was appended (every one must stay where it was, LP64)
OPTS_BEFORE = dict(seed=0, device=8, fstar_mode=12, skip_f_draws=16, use_graph=20, rank=24, world_size=28, m_global=32,
                   item_offset=40, nccl_unique_id=48, thin=56, reserved0=60, f_mean_out=64, f_sd_out=72, fit=80, irf=88,
                   chains=96)


def test_ppc_struct_layout_matches_header(tmp_path):
    from gpirt_b200._lib import Opts, Ppc
    fields = [name for name, _ in Ppc._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "gpirt_b200.h"\nint main(void) {\n'
                   + "".join('  printf("%s %%zu\\n", offsetof(gpirt_b200_ppc, %s));\n' % (f, f) for f in fields)
                   + '  printf("sizeof %zu\\n", sizeof(gpirt_b200_ppc));\n'
                   + "".join('  printf("opts.%s %%zu\\n", offsetof(gpirt_b200_opts, %s));\n' % (f, f)
                             for f in list(OPTS_BEFORE) + ["ppc"])
                   + '  printf("opts.sizeof %zu\\n", sizeof(gpirt_b200_opts));\n  return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = dict(line.split() for line in subprocess.check_output([str(exe)], text=True).splitlines())
    for f in fields:
        assert int(got[f]) == getattr(Ppc, f).offset, f
    assert int(got["sizeof"]) == C.sizeof(Ppc) == 48
    for f, off in OPTS_BEFORE.items():
        assert int(got["opts." + f]) == getattr(Opts, f).offset == off, f
    assert int(got["opts.ppc"]) == Opts.ppc.offset == Opts.chains.offset + C.sizeof(C.c_void_p) == 104   # right after chains
    assert int(got["opts.sizeof"]) == C.sizeof(Opts)


def test_default_opts_request_no_checks():
    from gpirt_b200.sampler import make_opts
    assert not make_opts(seed=1).ppc


def test_ppc_pairs_is_exported():
    from gpirt_b200 import _lib
    assert "gpirt_b200_ppc_pairs" in _lib.EXPORTS


def _no_device(monkeypatch):
    from gpirt_b200 import _lib

    def no_device(*a, **k):
        raise AssertionError("the library was reached")
    monkeypatch.setattr(_lib, "load", no_device)


def _y():
    from gpirt_b200 import ResponseMatrix
    return ResponseMatrix(np.array([[1.0, -1.0, np.nan], [-1.0, 1.0, 1.0], [1.0, 1.0, -1.0]]))


def test_ppc_pairs_without_ppc_is_refused(monkeypatch):
    import gpirt_b200.sampler as G
    _no_device(monkeypatch)
    with pytest.raises(ValueError, match="ppc_pairs needs ppc"):
        G.gpirtMCMC(_y(), 4, 0, theta_init=np.zeros(3), ppc_pairs=True)


@pytest.mark.parametrize("pairs", [False, True])
def test_ppc_with_chains_is_refused(pairs, monkeypatch):
    import gpirt_b200.sampler as G
    _no_device(monkeypatch)
    with pytest.raises(ValueError, match="chains cannot be combined with ppc"):
        G.gpirtMCMC(_y(), 4, 0, theta_init=np.zeros((3, 2)), chains=2, ppc=True, ppc_pairs=pairs)


def test_ppc_with_shard_is_refused(monkeypatch):
    import gpirt_b200.sampler as G
    _no_device(monkeypatch)
    with pytest.raises(ValueError, match="ppc cannot be combined with shard"):
        G.gpirtMCMC(_y(), 4, 0, theta_init=np.zeros(3), ppc=True, shard=(0, 2, 6, 0, b"\0" * 128))


@pytest.mark.parametrize("reps", [np.zeros((3, 2, 1)), np.zeros((2, 3, 1)), np.zeros((3, 3, 1, 1))])
def test_ppc_pairs_replicates_of_the_wrong_shape_are_refused(reps, monkeypatch):
    import gpirt_b200.sampler as G
    _no_device(monkeypatch)
    with pytest.raises(ValueError, match="y_reps"):
        G.ppc_pairs(np.ones((3, 3)), reps)
