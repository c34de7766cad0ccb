"""The ctypes mirror of gpirt_b200_fit (opts.fit, the posterior predictive summaries) against the real header, and the
argument checks gpirtMCMC(predictive=True) makes before anything reaches the device — no GPU needed."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_fit_struct_layout_matches_header(tmp_path):
    from gpirt_b200._lib import Fit, Opts
    fields = [name for name, _ in Fit._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "gpirt_b200.h"\nint main(void) {\n'
                   + "".join('  printf("%s %%zu\\n", offsetof(gpirt_b200_fit, %s));\n' % (f, f) for f in fields)
                   + '  printf("sizeof %zu\\n", sizeof(gpirt_b200_fit));\n'
                   + '  printf("opts.fit %zu\\n", offsetof(gpirt_b200_opts, fit));\n  return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = dict(line.split() for line in subprocess.check_output([str(exe)], text=True).splitlines())
    for f in fields:
        assert int(got[f]) == getattr(Fit, f).offset, f
    assert int(got["sizeof"]) == C.sizeof(Fit)
    assert int(got["opts.fit"]) == Opts.fit.offset == Opts.f_sd_out.offset + C.sizeof(C.c_void_p)   # appended last


def test_default_opts_request_no_predictive_summaries():
    from gpirt_b200.sampler import make_opts
    assert not make_opts(seed=1).fit


def test_y_holdout_is_checked_on_the_host():
    import gpirt_b200.sampler as G
    from gpirt_b200 import ResponseMatrix
    y = ResponseMatrix(np.array([[1.0, -1.0, np.nan], [-1.0, 1.0, 1.0]]))
    with pytest.raises(ValueError, match="shape"):
        G.gpirtMCMC(y, 1, 0, theta_init=np.zeros(2), predictive=True, y_holdout=np.full((3, 2), np.nan))
    with pytest.raises(ValueError, match="predictive"):
        G.gpirtMCMC(y, 1, 0, theta_init=np.zeros(2), y_holdout=np.full((2, 3), np.nan))
