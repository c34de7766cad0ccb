"""Cost of PSIS-LOO (gpirtMCMC(..., loo=True), opts.loo) at the senate116 shape (C1, 100 x 418, S = 2000), C2 (1024 x 2000,
S = 500) and C3 (4096 x 10000, S = 200).

  python tools/loo_cost.py [--repeats 3] [--out profiles/r07_loo_cost.json]

Prints one JSON line:
  e2e      gpirtMCMC(S, 0, thin=10, store_f=False) without and with loo, alternated in one process after an un-timed warm
           call of each; ms per sampling iteration (host clock around the whole call, which ends in a device synchronise:
           it includes the state's allocation, the finish, the reductions and the copies of the per-cell outputs)
  kernels  psis_loo() on log-likelihood draws shaped like the workload's cells (logistic log-likelihoods of g ~ N(mu_c, 1)
           per cell, draws in random order) at the workload's S: CUDA-event time of one update launch and of the finish.
           The draws of every cell are uploaded at once, so at C2 and C3 the run covers the first `cols` cells only
           (cols_run); `scaled_ms` multiplies by cells / cols_run (both kernels are one thread / one warp per cell).
           Bytes per update launch: at least 49 per cell (f or ll read, state root, running max, outside sum and sum of
           sigma read, sum of sigma written); per finish: the 8 (M + 4) bytes of state read plus 24 written per cell.
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

SHAPES = (("c1", 2000), ("c2", 500), ("c3", 200))   # (workload, S)
MAX_COLS = 1 << 20                                  # cells of the psis_loo() run (8 cols S bytes of draws on the device)


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    if q.returncode:
        raise RuntimeError("nvidia-smi failed: %s" % q.stderr)
    name, power, clock = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def tail_len(S):
    return int(np.ceil(min(0.2 * S, 3.0 * np.sqrt(S))))


def e2e(d, S, repeats):
    y = ResponseMatrix(d["y"])
    modes = {"without": {}, "loo": dict(loo=True)}

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
                slowdown_loo=round(med["loo"] / med["without"] - 1.0, 4))


def kernels(cells, S, reps=2):
    cols = min(cells, MAX_COLS)
    rs = np.random.default_rng(5)
    g = rs.standard_normal((cols, 1)) * 2.0 + rs.standard_normal((cols, S))
    ll = -(np.maximum(-g, 0.0) + np.log1p(np.exp(-np.abs(g))))
    del g
    _, _, _, (ms_upd, ms_fin) = G.psis_loo(ll, reps=reps)
    M = tail_len(S)
    scale = cells / cols
    upd_bytes, fin_bytes = 49.0 * cols, (8.0 * (M + 4) + 24.0) * cols
    return dict(cols_run=cols, M=M, ms_update=round(ms_upd, 5), ms_finish=round(ms_fin, 4),
                scaled_ms_update=round(ms_upd * scale, 4), scaled_ms_finish=round(ms_fin * scale, 3),
                update_min_bytes=upd_bytes, update_TBps=round(upd_bytes / (ms_upd * 1e-3) / 1e12, 3),
                finish_bytes=fin_bytes, finish_TBps=round(fin_bytes / (ms_fin * 1e-3) / 1e12, 3),
                finish_log1p_per_cell=(30 + int(np.floor(np.sqrt(M))) + 1) * M)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = dict(device=device_info(), shapes={})
    for name, S in SHAPES:
        c = synthetic.WORKLOADS[name]
        d = synthetic.make(c["n"], c["m"])
        r = dict(n=c["n"], m=c["m"], e2e=e2e(d, S, a.repeats), kernels=kernels(c["n"] * c["m"], S))
        run_ms = r["e2e"]["median"]["without"] * S
        r["finish_share_of_run"] = round(r["kernels"]["scaled_ms_finish"] / run_ms, 4)
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
