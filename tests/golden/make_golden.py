"""Generates tests/golden/*.npz.  Needs the reference package's sources (a checkout of duckmayr/gpirt where
oracle/Makefile looks for it, or named by GPIRT_REFERENCE) to compile oracle/_ref.

Every golden output comes from the reference's OWN sampler sources (src/gpirtMCMC.cpp etc. compiled unmodified against
the stand-in headers in oracle/refshim, = oracle/_ref/libgpirt_ref.so), driven by the tape of variates that the addressed
Philox generator (oracle/gpo_rng.h) hands out for the recorded seed.  The oracle restatement and the CUDA sampler are
both checked against these files (tests/test_oracle.py, tests/test_gpu_parity.py::test_golden_*).

    GPIRT_REFERENCE=<checkout of duckmayr/gpirt> python tests/golden/make_golden.py
"""
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from conftest import make_problem  # noqa: E402
from oracle import oracle as O  # noqa: E402
import gpirt_b200  # noqa: E402

CASES = [dict(name="tiny_8x5", n=8, m=5, S=3, B=1, seed=11, missing=0.15, mode=0),
         dict(name="small_100x37", n=100, m=37, S=2, B=1, seed=22, missing=0.05, mode=0),
         dict(name="odd_257x12", n=257, m=12, S=1, B=1, seed=33, missing=0.0, mode=0)]


def run_ref(y, theta0, S, B, pm, psd, pstep, seed, mode):
    rng = O.Rng.keyed(seed, record=True)
    port = O.mcmc(y, theta0, S, B, pm, psd, pstep, rng, theta_cdf_mode=mode)   # records the tape in consumption order
    vals, kinds = rng.recorded()
    with O.RefTape(vals, kinds) as t:
        ref = O.ref_mcmc(y, theta0, S, B, pm, psd, pstep)
    assert t.error == 0 and t.consumed == vals.size, "reference consumed the tape differently from the restatement"
    return ref, port, vals.size


def main():
    O.build("ref")
    for c in CASES:
        p = make_problem(c["n"], c["m"], seed=c["seed"], missing=c["missing"])
        ref, port, ntape = run_ref(p["y"], p["theta"], c["S"], c["B"], p["pm"], p["psd"], p["pstep"], c["seed"], c["mode"])
        np.savez_compressed(os.path.join(HERE, c["name"] + ".npz"), y=p["y"], theta_init=p["theta"], S=c["S"], B=c["B"],
                            seed=c["seed"], theta=ref["theta"], beta=ref["beta"], f=ref["f"], IRFs=ref["IRFs"], tape_len=ntape)
        print(c["name"], "tape", ntape, "port==ref:", all(np.array_equal(ref[k], port[k]) for k in ("theta", "beta", "f", "IRFs")))
    # senate116 (BASELINE config 1): 100 x 418 after response_matrix(); strict reference theta-CDF
    codes, _, _ = gpirt_b200.senate116()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        y = np.asarray(gpirt_b200.response_matrix(codes))
    m = y.shape[1]
    theta0 = np.random.RandomState(116).randn(100)
    S, B, seed = 2, 1, 116
    ref, port, ntape = run_ref(y, theta0, S, B, np.zeros((2, m)), np.full((2, m), 3.0), np.full((2, m), 0.1), seed, 0)
    np.savez_compressed(os.path.join(HERE, "senate116_100x418.npz"), y_int8=np.where(np.isnan(y), 0, y).astype(np.int8),
                        theta_init=theta0, S=S, B=B, seed=seed, theta=ref["theta"], beta=ref["beta"],
                        f_last=ref["f"][:, :, -1], IRFs_every10=ref["IRFs"][::10], tape_len=ntape)
    print("senate116", y.shape, "tape", ntape, "port==ref:", all(np.array_equal(ref[k], port[k]) for k in ("theta", "beta", "f", "IRFs")))


if __name__ == "__main__":
    main()
