"""Cost of the IRF posterior summaries (gpirtMCMC(..., irf_band=0.95), opts.irf) at the senate116 shape (C1, 100 x 418,
S = 2000), C2 (1024 x 2000, S = 500) and C3 (4096 x 10000, S = 200).

  python tools/irf_cost.py [--repeats 3] [--band 0.95] [--out profiles/r04_irf_cost.json]

Prints one JSON line:
  e2e      gpirtMCMC(S, 0, thin=10, store_f=False) without and with irf_band, alternated in one process after an un-timed
           warm call of each; ms per sampling iteration (host clock around the whole call, which ends in a device
           synchronise, so it includes the finish kernel and the copies of the four 1001 x m outputs)
  bands    irf_bands() on synthetic draws of the same shape (1001 m cells x S draws, uploaded once): mean time of one update
           launch over the S launches of a pass and the time of the finish (CUDA events), the tail-buffer bytes and the
           update's nominal traffic (8 B f*, 32 B Welford read + write, 16 B heap roots per cell) over its time
  device   card name and power limit, read in the same run"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gpirt_b200.sampler as G  # noqa: E402
from gpirt_b200 import ResponseMatrix, synthetic  # noqa: E402

SHAPES = (("c1", 2000), ("c2", 500), ("c3", 200))   # (workload, sampling iterations); c1 is the senate116 shape


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    if q.returncode:
        raise RuntimeError("nvidia-smi failed: %s" % q.stderr)
    name, power, clock = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def tails(S, band):
    r = [int(np.floor((S - 1) * q)) for q in ((1.0 - band) / 2.0, (1.0 + band) / 2.0)]
    return min(S, r[0] + 2), S - r[1]


def e2e(name, S, band, repeats):
    c = synthetic.WORKLOADS[name]
    d = synthetic.make(c["n"], c["m"])
    y = ResponseMatrix(d["y"])

    def call(b, iters):
        t0 = time.perf_counter()
        G.gpirtMCMC(y, iters, 0, beta_prior_means=d["pm"], beta_prior_sds=d["psd"], beta_proposal_sds=d["pstep"],
                    theta_init=d["theta_init"], seed=synthetic.SEED, thin=10, store_f=False, irf_band=b)
        return (time.perf_counter() - t0) * 1e3 / iters

    call(None, 20), call(band, 20)   # warm-up: module loads, pinned buffers, the pool's memory
    runs = {"without": [], "with": []}
    for _ in range(repeats):
        runs["without"].append(call(None, S))
        runs["with"].append(call(band, S))
    base, irf = float(np.median(runs["without"])), float(np.median(runs["with"]))
    return dict(call="gpirtMCMC(S=%d, B=0, thin=10, store_f=False)" % S, n=c["n"], m=c["m"], S=S, repeats=repeats,
                ms_per_iter_without=[round(x, 4) for x in runs["without"]], ms_per_iter_with=[round(x, 4) for x in runs["with"]],
                median_without=round(base, 4), median_with=round(irf, 4), slowdown=round(irf / base - 1.0, 4))


def bands(name, S, band):
    m = synthetic.WORKLOADS[name]["m"]
    cols = 1001 * m
    rs = np.random.default_rng(1)
    base = rs.standard_normal((cols, 16))
    a, b = rs.uniform(0.5, 2.0, S), rs.standard_normal(S)
    draws = np.empty((cols, S), order="F")
    for s in range(S):   # distinct draws per cell without S full random fills
        np.multiply(base[:, s % 16], a[s], out=draws[:, s])
        draws[:, s] += b[s]
    del base
    _, _, (ms_upd, ms_fin) = G.irf_bands(draws, band, reps=1)
    klo, khi = tails(S, band)
    upd_bytes = 56.0 * cols
    return dict(cells=cols, S=S, K_lo=klo, K_hi=khi, band_bytes=8 * cols * (klo + khi),
                ms_per_update=round(ms_upd, 5), ms_finish=round(ms_fin, 4),
                update_nominal_TBps=round(upd_bytes / (ms_upd * 1e-3) / 1e12, 3))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--band", type=float, default=0.95)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = dict(band=a.band, device=device_info(), shapes={})
    for name, S in SHAPES:
        r = dict(e2e=e2e(name, S, a.band, a.repeats), bands=bands(name, S, a.band))
        r["finish_share_of_run"] = round(r["bands"]["ms_finish"] / (r["e2e"]["median_with"] * S), 5)
        res["shapes"][name] = r
        print(name, json.dumps(r), file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
