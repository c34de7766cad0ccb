"""Cost of the posterior predictive checks (gpirtMCMC(..., ppc=True[, ppc_pairs=True]), opts.ppc) at the senate116 shape
(C1, 100 x 418, S = 2000), C2 (1024 x 2000, S = 500) and C3 (4096 x 10000, S = 100) with 0 % and 5 % missing cells.

  python tools/ppc_cost.py [--repeats 3] [--out profiles/r06_ppc_cost.json]

Prints one JSON line:
  e2e      gpirtMCMC(S, 0, thin=10, store_f=False) without checks, with ppc and with ppc + ppc_pairs, alternated in one
           process after an un-timed warm call of each; ms per sampling iteration (host clock around the whole call, which
           ends in a device synchronise: it includes the observed-count pass and the copies of the m x m outputs)
  pairs    ppc_pairs() on the same response matrix with one replicate: CUDA-event time of one per-draw launch (k_ppc_pairs,
           plus the replicate's column sums without missing cells) and of the observed pass; the int8 operations of the
           products it runs (2 x 128^2 x K per upper-triangle tile and product; 1 product without missing cells, 3 with)
           over that time, against int8_peak_tops() and int8_peak_tops(random_operands=True) of the same run; and its
           bytes per launch (operand tiles read by TMA + 24 B per pair entry of the epilogue: observed counts read,
           counter read and written)
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

SHAPES = (("c1", 0.0, 2000), ("c2", 0.0, 500), ("c3", 0.0, 100), ("c3", 0.05, 100))   # (workload, missing, S)


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    if q.returncode:
        raise RuntimeError("nvidia-smi failed: %s" % q.stderr)
    name, power, clock = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def e2e(d, S, repeats):
    y = ResponseMatrix(d["y"])
    modes = {"without": {}, "ppc": dict(ppc=True), "ppc_pairs": dict(ppc=True, ppc_pairs=True)}

    def call(kw, iters):
        t0 = time.perf_counter()
        G.gpirtMCMC(y, iters, 0, beta_prior_means=d["pm"], beta_prior_sds=d["psd"], beta_proposal_sds=d["pstep"],
                    theta_init=d["theta_init"], seed=synthetic.SEED, thin=10, store_f=False, **kw)
        return (time.perf_counter() - t0) * 1e3 / iters

    for kw in modes.values():   # warm-up: module loads, pinned buffers, the pool's memory
        call(kw, 20)
    runs = {k: [] for k in modes}
    for _ in range(repeats):
        for k, kw in modes.items():
            runs[k].append(call(kw, S))
    med = {k: float(np.median(v)) for k, v in runs.items()}
    return dict(call="gpirtMCMC(S=%d, B=0, thin=10, store_f=False)" % S, S=S, repeats=repeats,
                ms_per_iter={k: [round(x, 4) for x in v] for k, v in runs.items()},
                median={k: round(v, 4) for k, v in med.items()},
                slowdown_ppc=round(med["ppc"] / med["without"] - 1.0, 4),
                slowdown_ppc_pairs=round(med["ppc_pairs"] / med["without"] - 1.0, 4))


def pairs(d, peak, peak_random, reps=20):
    y = d["y"]
    n, m = y.shape
    rs = np.random.default_rng(2)
    rep = np.where(rs.random((n, m)) < 0.5, 1.0, -1.0)[:, :, None]
    _, _, (ms_draw, ms_obs) = G.ppc_pairs(y, rep, reps=reps)
    missing = bool(np.isnan(y).any())
    mt = -(-m // 128)
    tiles = mt * (mt + 1) // 2
    kpad = -(-n // 128) * 128
    products = 3 if missing else 1
    ops = 2.0 * 128 * 128 * kpad * tiles * products
    operand_bytes = tiles * (4 if missing else 2) * 128 * kpad
    epilogue_bytes = 24 * tiles * 128 * 128
    tops = ops / (ms_draw * 1e-3) / 1e12
    return dict(missing=missing, tiles=tiles, ms_per_draw_launch=round(ms_draw, 4), ms_observed_pass=round(ms_obs, 4),
                int8_ops_per_launch=ops, achieved_TOPs=round(tops, 1), share_of_int8_peak=round(tops / peak, 4),
                share_of_int8_peak_random=round(tops / peak_random, 4), bytes_per_launch=operand_bytes + epilogue_bytes,
                achieved_TBps=round((operand_bytes + epilogue_bytes) / (ms_draw * 1e-3) / 1e12, 3))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    peak, peak_random = G.int8_peak_tops(), G.int8_peak_tops(random_operands=True)
    res = dict(device=device_info(), int8_peak_TOPs=round(peak, 1), int8_peak_random_TOPs=round(peak_random, 1), shapes={})
    for name, missing, S in SHAPES:
        c = synthetic.WORKLOADS[name]
        d = synthetic.make(c["n"], c["m"], missing=missing)
        key = "%s_%dpct_missing" % (name, round(100 * missing))
        r = dict(n=c["n"], m=c["m"], missing=missing, e2e=e2e(d, S, a.repeats), pairs=pairs(d, peak, peak_random))
        res["shapes"][key] = r
        print(key, json.dumps(r), file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
