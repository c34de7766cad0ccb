"""Cost of the posterior predictive summaries (gpirtMCMC(..., predictive=True)) at the bench shape C3 (4096 x 10000).

  python tools/predictive_cost.py [--iters 500] [--pairs 2] [--reps 200] [--out FILE]

Prints one JSON line:
  accumulate   mean time of one k_predictive_accumulate launch over `reps` launches (CUDA events), the bytes it must move
               (57 per cell: f, cell code, three FP64 accumulators read and written) over that time, and the same run's
               device-to-device copy rate (read + write bytes / time) it is compared with
  e2e          gpirtMCMC(S, 0, thin=10, store_f=False) without and with predictive=True, alternated in one process after an
               un-timed warm call of each; ms per sampling iteration (host clock around the whole call, which ends in a
               device synchronise, so it includes the finish kernels and the copies of the three n x m outputs)
  device       card name and power limit, read in the same run"""
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


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    if q.returncode:
        raise RuntimeError("nvidia-smi failed: %s" % q.stderr)
    name, power, clock = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=500)
    ap.add_argument("--pairs", type=int, default=2)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    c = synthetic.WORKLOADS["c3"]
    n, m = c["n"], c["m"]
    cells = n * m
    ms_acc, ms_copy = G.predictive_accumulate_time(n, m, a.reps)
    acc_bytes = 57.0 * cells
    copy_bytes = 2 * 3 * 8.0 * (-(-n // 8) * 8) * m
    acc_rate, copy_rate = acc_bytes / (ms_acc * 1e-3), copy_bytes / (ms_copy * 1e-3)

    d = synthetic.make(n, m)
    y = ResponseMatrix(d["y"])

    def call(predictive, S):
        t0 = time.perf_counter()
        G.gpirtMCMC(y, S, 0, beta_prior_means=d["pm"], beta_prior_sds=d["psd"], beta_proposal_sds=d["pstep"],
                    theta_init=d["theta_init"], seed=synthetic.SEED, thin=10, store_f=False, predictive=predictive)
        return (time.perf_counter() - t0) * 1e3 / S

    call(False, 20), call(True, 20)   # warm-up: module loads, pinned buffers, the pool's memory
    runs = {False: [], True: []}
    for _ in range(a.pairs):
        for p in (False, True):
            runs[p].append(call(p, a.iters))
    base, pred = float(np.median(runs[False])), float(np.median(runs[True]))
    res = dict(
        workload="c3", n=n, m=m, device=device_info(),
        accumulate=dict(ms_per_launch=round(ms_acc, 4), bytes_per_launch=acc_bytes, achieved_TBps=round(acc_rate / 1e12, 3),
                        copy_TBps_same_run=round(copy_rate / 1e12, 3), frac_of_copy_rate=round(acc_rate / copy_rate, 3),
                        launches=a.reps),
        e2e=dict(call="gpirtMCMC(S=%d, B=0, thin=10, store_f=False)" % a.iters, pairs=a.pairs,
                 ms_per_iter_without=[round(x, 3) for x in runs[False]], ms_per_iter_with=[round(x, 3) for x in runs[True]],
                 median_without=round(base, 3), median_with=round(pred, 3), slowdown=round(pred / base - 1.0, 4)))
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
