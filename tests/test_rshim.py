"""The R-facing shim (gpirt_b200/csrc/rshim/gpirt_rshim.c) built against stand-in R headers (tests/fake_r):
registration exactly as the reference's generated glue (src/RcppExports.cpp:32-40), error path without a GPU,
and — on the GPU box — a real .Call-style invocation compared with the direct C-ABI result."""
import os
import struct
import subprocess

import numpy as np
import pytest

from conftest import make_problem

HERE = os.path.dirname(os.path.abspath(__file__))
FAKE = os.path.join(HERE, "fake_r")


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    """the harness is built outside the source tree, which may be read-only"""
    from gpirt_b200 import _lib
    _lib.load()   # makes sure libgpirt_b200.so exists
    out = str(tmp_path_factory.mktemp("fake_r") / "fake_r_harness")
    subprocess.check_call(["make", "-s", "-C", FAKE, "OUT=" + out])
    return out


def write_input(path, p, S, B, rng_state):
    n, m = p["y"].shape
    with open(path, "wb") as fh:
        fh.write(struct.pack("<4iQ", n, m, S, B, rng_state))
        for a in (p["y"], p["theta"], p["pm"], p["psd"], p["pstep"]):
            fh.write(np.asfortranarray(a, dtype=np.float64).tobytes(order="F"))


def test_shim_registers_the_reference_routine_with_arity_7(harness):
    """R_init_gpirt registers _gpirt_gpirtMCMC with 7 arguments exactly as src/RcppExports.cpp:32-40 does (dynamic symbols
    off); the only other routine is the same call with the draw-storage options as three trailing arguments"""
    out = subprocess.run([harness], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert out.stdout.split("\n")[:2] == ["registered _gpirt_gpirtMCMC arity 7", "registered _gpirt_gpirtMCMC_b200 arity 10"]


def test_shim_raises_r_error_without_gpu(harness, tmp_path):
    from gpirt_b200 import _lib
    if _lib.load().gpirt_b200_device_count() > 0:
        pytest.skip("GPU present")
    p = make_problem(12, 5, seed=1)
    write_input(tmp_path / "in.bin", p, 2, 1, 42)
    out = subprocess.run([harness, str(tmp_path / "in.bin"), str(tmp_path / "out.bin")], capture_output=True, text=True)
    assert out.returncode == 3 and "no CUDA device" in out.stderr      # Rf_error(), i.e. an R-level stop()


@pytest.mark.gpu
def test_shim_call_matches_c_abi(harness, tmp_path):
    import gpirt_b200
    import gpirt_b200.sampler as G
    n, m, S, B = 60, 21, 3, 2
    p = make_problem(n, m, seed=9, missing=0.1)
    write_input(tmp_path / "in.bin", p, S, B, 20261018)
    out = subprocess.run([harness, str(tmp_path / "in.bin"), str(tmp_path / "out.bin")], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    raw = open(tmp_path / "out.bin", "rb").read()
    seed = struct.unpack("<Q", raw[:8])[0]
    vals = np.frombuffer(raw[8:], dtype=np.float64)
    sizes = [(S + 1) * n, 2 * m * (S + 1), n * m * (S + 1), 1001 * m]
    assert vals.size == sum(sizes)
    th, be, f, irf = np.split(vals, np.cumsum(sizes)[:-1])
    got = G.gpirtMCMC(gpirt_b200.ResponseMatrix(p["y"]), S, B, beta_prior_means=p["pm"], beta_prior_sds=p["psd"],
                      beta_proposal_sds=p["pstep"], theta_init=p["theta"], seed=seed)
    assert np.array_equal(th.reshape((S + 1, n), order="F"), got["theta"])
    assert np.array_equal(be.reshape((2, m, S + 1), order="F"), got["beta"])
    assert np.array_equal(f.reshape((n, m, S + 1), order="F"), got["f"])
    assert np.array_equal(irf.reshape((1001, m), order="F"), got["IRFs"])


@pytest.mark.gpu
def test_shim_extended_call_thins_and_summarises(harness, tmp_path):
    """.Call(`_gpirt_gpirtMCMC_b200`, ..., thin, store_f, f_summary): list of 6 with 1 + S %/% thin slots"""
    import gpirt_b200
    import gpirt_b200.sampler as G
    n, m, S, B, thin = 40, 13, 9, 2, 3
    p = make_problem(n, m, seed=4, missing=0.05)
    write_input(tmp_path / "in.bin", p, S, B, 777)
    out = subprocess.run([harness, str(tmp_path / "in.bin"), str(tmp_path / "out.bin"), str(thin)], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    raw = open(tmp_path / "out.bin", "rb").read()
    seed = struct.unpack("<Q", raw[:8])[0]
    vals = np.frombuffer(raw[8:], dtype=np.float64)
    slots = S // thin + 1
    sizes = [slots * n, 2 * m * slots, n * m * slots, 1001 * m, n * m, n * m]
    assert vals.size == sum(sizes)
    th, be, f, irf, fm, fsd = np.split(vals, np.cumsum(sizes)[:-1])
    got = G.gpirtMCMC(gpirt_b200.ResponseMatrix(p["y"]), S, B, beta_prior_means=p["pm"], beta_prior_sds=p["psd"],
                      beta_proposal_sds=p["pstep"], theta_init=p["theta"], seed=seed, thin=thin, f_summary=True)
    assert np.array_equal(th.reshape((slots, n), order="F"), got["theta"])
    assert np.array_equal(f.reshape((n, m, slots), order="F"), got["f"])
    assert np.array_equal(irf.reshape((1001, m), order="F"), got["IRFs"])
    assert np.array_equal(fm.reshape((n, m), order="F"), got["f_mean"])
    assert np.array_equal(fsd.reshape((n, m), order="F"), got["f_sd"])
