"""Throughput of several chains in one call (gpirtMCMC(..., chains=C), opts.chains) and the cost of their diagnostics, at
the senate116 shape (C1, 100 x 418), C2 (1024 x 2000) and C3 (4096 x 10000).

  python tools/chains_cost.py [--repeats 3] [--out profiles/r05_chains_cost.json]

Prints one JSON line.  For each shape and C (1, 2, 4, 8 at C1 and C2; 1, 2 at C3) gpirtMCMC(S, B, thin=10, store_f=False)
runs without and with chain_diagnostics, alternated, after one un-timed warm call of each; the host clock around the whole
call (which ends in a device synchronise) gives the summed sweeps per second over the chains, S + B sweeps per chain.
The medians of the repeats are reported, with the speed-up of C chains over one and the slowdown the diagnostics add.
The card's name and power limit are read in the same run."""
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

SHAPES = (("c1", 2000, 200, (1, 2, 4, 8)), ("c2", 300, 30, (1, 2, 4, 8)), ("c3", 60, 6, (1, 2)))   # (workload, S, B, C)


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    if q.returncode:
        raise RuntimeError("nvidia-smi failed: %s" % q.stderr)
    name, power, clock = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def measure(name, S, B, C_, repeats):
    c = synthetic.WORKLOADS[name]
    d = synthetic.make(c["n"], c["m"])
    y = ResponseMatrix(d["y"])
    th = np.asfortranarray(np.repeat(np.asarray(d["theta_init"], dtype=np.float64)[:, None], C_, axis=1))

    def call(diag, iters, burn):
        t0 = time.perf_counter()
        G.gpirtMCMC(y, iters, burn, beta_prior_means=d["pm"], beta_prior_sds=d["psd"], beta_proposal_sds=d["pstep"],
                    theta_init=th, seed=synthetic.SEED, thin=10, store_f=False, chains=C_, chain_diagnostics=diag)
        return C_ * (iters + burn) / (time.perf_counter() - t0)

    call(False, 10, 2), call(True, 10, 2)   # warm-up: module loads, pinned buffers, the pool's memory
    runs = {"without": [], "with": []}
    for _ in range(repeats):
        runs["without"].append(call(False, S, B))
        runs["with"].append(call(True, S, B))
    base, diag = float(np.median(runs["without"])), float(np.median(runs["with"]))
    return dict(C=C_, sweeps_per_s_without=[round(x, 2) for x in runs["without"]],
                sweeps_per_s_with=[round(x, 2) for x in runs["with"]], median_without=round(base, 2),
                median_with=round(diag, 2), diagnostics_slowdown=round(base / diag - 1.0, 4))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = dict(device=device_info(), shapes={})
    for name, S, B, Cs in SHAPES:
        c = synthetic.WORKLOADS[name]
        rows = [measure(name, S, B, C_, a.repeats) for C_ in Cs]
        one = rows[0]["median_without"]
        for r in rows:
            r["speedup_over_one_chain"] = round(r["median_without"] / one, 3)
        res["shapes"][name] = dict(call="gpirtMCMC(S=%d, B=%d, thin=10, store_f=False, chains=C)" % (S, B), n=c["n"],
                                   m=c["m"], S=S, B=B, repeats=a.repeats, runs=rows)
        print(name, json.dumps(res["shapes"][name]), file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
