"""The ctypes mirror of gpirt_b200_irf (opts.irf, the posterior summaries of the IRFs on the grid) against the real header,
and the argument checks gpirtMCMC(irf_band=...) makes before anything reaches the device — no GPU needed."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_irf_struct_layout_matches_header(tmp_path):
    from gpirt_b200._lib import Irf, Opts
    fields = [name for name, _ in Irf._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "gpirt_b200.h"\nint main(void) {\n'
                   + "".join('  printf("%s %%zu\\n", offsetof(gpirt_b200_irf, %s));\n' % (f, f) for f in fields)
                   + '  printf("sizeof %zu\\n", sizeof(gpirt_b200_irf));\n'
                   + '  printf("opts.irf %zu\\n", offsetof(gpirt_b200_opts, irf));\n'
                   + '  printf("opts.sizeof %zu\\n", sizeof(gpirt_b200_opts));\n  return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = dict(line.split() for line in subprocess.check_output([str(exe)], text=True).splitlines())
    for f in fields:
        assert int(got[f]) == getattr(Irf, f).offset, f
    assert int(got["sizeof"]) == C.sizeof(Irf)
    assert int(got["opts.irf"]) == Opts.irf.offset == Opts.fit.offset + C.sizeof(C.c_void_p)   # right after fit
    assert int(got["opts.sizeof"]) == C.sizeof(Opts)


def test_default_opts_request_no_irf_summaries():
    from gpirt_b200.sampler import make_opts
    assert not make_opts(seed=1).irf


def test_irf_bands_is_exported():
    from gpirt_b200 import _lib
    assert "gpirt_b200_irf_bands" in _lib.EXPORTS


@pytest.mark.parametrize("band", [0.0, 1.0, -0.5, float("nan")])
def test_bad_irf_band_is_refused_on_the_host(band, monkeypatch):
    import gpirt_b200.sampler as G
    from gpirt_b200 import ResponseMatrix, _lib

    def no_device(*a, **k):
        raise AssertionError("the library was reached")
    monkeypatch.setattr(_lib, "load", no_device)
    y = ResponseMatrix(np.array([[1.0, -1.0, np.nan], [-1.0, 1.0, 1.0]]))
    with pytest.raises(ValueError, match="irf_band"):
        G.gpirtMCMC(y, 1, 0, theta_init=np.zeros(2), irf_band=band)
