#!/usr/bin/env python
"""bench.py — Gibbs sweeps/sec of the GP-IRT sampler (BASELINE.json metric) on synthetic data of a named n x m shape.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3] [--impl reference] [--dump-outputs DIR]

A "step" is one Gibbs sweep (reference loop body, src/gpirtMCMC.cpp:68-78) over the whole response matrix.
  value : sweeps/s with everything resident in HBM, timed by CUDA events on the sampler's own stream inside the C library
          (gpirt_b200_sampler_sweep), max over ranks.
  e2e   : sweeps/s through the public drop-in call gpirtMCMC() -> C-ABI gpirt_b200_mcmc() with HOST buffers: the H2D
          copy of the response matrix and the per-sweep D2H of the theta / beta / f draws are inside the timed region.
  N > 1 : launched under torchrun, one rank per GPU; items are sharded across ranks (strong scaling of the named
          workload) and the per-respondent log-posterior partial sums are all-reduced over NCCL once per sweep.
  --impl reference : the reference's own CPU sampler (its sources compiled against stand-in Armadillo headers,
          oracle/_ref; else the oracle port) on a bounded item sample, extrapolated linearly in m (stated in `sample`).
  --dump-outputs DIR : after the timed sweeps, the sampler state they left (what gpirt_b200_sampler_get returns) goes to
          DIR/<name>.npy, float64: theta and beta whole, f and f* on a fixed seeded sample of items (dump_outputs()).
          Inputs and seeds depend on the arguments only, so two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from gpirt_b200 import synthetic  # noqa: E402

N_GRID = 1001


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            return json.load(fh), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.stop_flag = False
        self.proc = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc:
            try:
                self.proc.terminate()
            except Exception:
                pass
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        busy = [s for s in sm if s > 0.5 * max(sm)] or sm
        return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's loop body (its own sources, oracle/_ref; else the oracle port) on host cores
# ---------------------------------------------------------------------------------------------------------------------
def cpu_reference_sweeps(n, m, data, steps, warmup, m_s, threads, n_sub=None, seed=12345):
    """Times `steps` sweeps of the reference CPU path on the first m_s items and, for the theta step only, on n_sub evenly
    spaced respondents (all n respondents everywhere else: K, chol, the ESS, the solves and the beta step need the full
    n x n factor).  m_s == m and n_sub == n is a MEASURED full sweep.  Otherwise the full-size sweep is EXTRAPOLATED:
        T(m) = T_fixed + T_item m / m_s,   T_item = draw_f + per-item part of draw_fstar + draw_theta n / n_sub + draw_beta
    Every step but K / Cholesky and the K* solve (T_fixed, measured at full size) is exactly linear in m, and draw_theta is
    exactly linear in the number of respondents (src/draw-theta.cpp:12-34 loops over them independently)."""
    from oracle import oracle as O
    n_sub = n if n_sub is None else min(n, n_sub)
    m_s = min(m, m_s)
    use_ref = os.path.exists(O.REF_SO)
    O.set_blas_threads(threads)
    y = np.asfortranarray(data["y"][:, :m_s])
    I = np.unique(np.linspace(0, n - 1, n_sub).astype(int))
    y_sub = np.asfortranarray(y[I, :])
    pm, psd, pstep = data["pm"][:, :m_s], data["psd"][:, :m_s], data["pstep"][:, :m_s]
    theta = data["theta_init"].copy()
    ts, prior = O.grid()
    if use_ref:
        O.ref().gpref_seed(seed)
        def chol(th):
            S = O.ref_K(th, th)                                # K(theta, theta), gpirtMCMC.cpp:76
            S[np.diag_indices(n)] += 0.001                     # :77
            return O.ref_chol_lower(S)                         # :78
        draw_f = lambda f, L, mu: O.ref_draw_f(f, y, L, mu)                      # noqa: E731
        draw_fstar = lambda f, th, L, mus: O.ref_draw_fstar(f, th, ts, L, mus)   # noqa: E731
        draw_theta = lambda fs, mus: O.ref_draw_theta(ts, y_sub, prior, fs, mus)     # noqa: E731
        draw_beta = lambda b, th, f: O.ref_draw_beta(b, th, y, f, pm, psd, pstep)  # noqa: E731
        kind = "reference"
    else:
        rng = O.Rng.keyed(seed)
        chol = lambda th: O.build_cholS(th)                                      # noqa: E731
        draw_f = lambda f, L, mu: O.draw_f(f, y, L, mu, rng)[0]                  # noqa: E731
        draw_fstar = lambda f, th, L, mus: O.draw_fstar(f, th, ts, L, mus, rng)[0]  # noqa: E731
        draw_theta = lambda fs, mus: O.draw_theta(ts, y_sub, prior, fs, rng, mode=0)[0]  # noqa: E731
        draw_beta = lambda b, th, f: O.draw_beta(b, th, y, f, pm, psd, pstep, rng)[0]  # noqa: E731
        kind = "port"
    rs = np.random.RandomState(7)
    L = chol(theta)
    f = np.asfortranarray(L @ rs.randn(n, m_s))
    beta = np.asfortranarray(rs.randn(2, m_s) * 3.0)
    parts = {k: [] for k in ("draw_f", "draw_fstar", "draw_theta", "draw_beta", "rebuild", "step")}
    for it in range(warmup + steps):
        if kind == "port":
            rng.set_sweep(it + 1)
        mu, mus = O.linear_mean(theta, beta), O.linear_mean(ts, beta)
        t0 = time.perf_counter()
        f = draw_f(f, L, mu)                                   # gpirtMCMC.cpp:68
        t1 = time.perf_counter()
        fs = draw_fstar(f, theta, L, mus)                      # :69
        t2 = time.perf_counter()
        th_new = draw_theta(fs, mus)                           # :70
        t3 = time.perf_counter()
        ok = np.isfinite(th_new)                               # the reference's theta_star[N] read (SURVEY F3) cannot happen
        theta[I[ok]] = th_new[ok]                              # at m_s <= 128; the guard keeps a full-size run alive
        beta = draw_beta(beta, theta, f)                       # :72
        mu, mus = O.linear_mean(theta, beta), O.linear_mean(ts, beta)   # :74-75
        t4 = time.perf_counter()
        L = chol(theta)                                        # :76-78
        t5 = time.perf_counter()
        if it >= warmup:
            for k, v in zip(("draw_f", "draw_fstar", "draw_theta", "draw_beta", "rebuild", "step"),
                            (t1 - t0, t2 - t1, t3 - t2, t4 - t3, t5 - t4, t5 - t0)):
                parts[k].append(v)
    # fixed part of draw_fstar (K*, L^-1 K*): time it with a single item
    t0 = time.perf_counter()
    if use_ref:
        O.ref_draw_fstar(f[:, :1], theta, ts, L, O.linear_mean(ts, beta[:, :1]))
    else:
        O.draw_fstar(f[:, :1], theta, ts, L, O.linear_mean(ts, beta[:, :1]), rng)
    t_fs1 = time.perf_counter() - t0
    mean = {k: float(np.mean(v)) for k, v in parts.items()}
    T_fix = mean["rebuild"] + t_fs1
    T_item = mean["draw_f"] + max(0.0, mean["draw_fstar"] - t_fs1) + mean["draw_theta"] * (n / len(I)) + mean["draw_beta"]
    full = m_s == m and len(I) == n
    T_full = mean["step"] if full else T_fix + T_item * (m / m_s)
    src = "reference sources (oracle/_ref)" if use_ref else "oracle port"
    if full:
        sample = "%d MEASURED full sweep(s) of the %s at %d x %d, %.2f s/sweep" % (steps, src, n, m, T_full)
    else:
        sample = ("%d sweep(s) of the %s on the first %d of %d items (theta step on %d of %d respondents), %.2f s per sampled "
                  "sweep measured; EXTRAPOLATED linearly in m (and in n for the theta step) to %.1f s/sweep (fixed part "
                  "K+chol+L^-1K* %.2f s)" % (steps, src, m_s, m, len(I), n, mean["step"], T_full, T_fix))
    return dict(value=1.0 / T_full, unit="sweeps/s", cores=threads if threads > 1 else 1, kind=kind, sample=sample,
                blas_threads=threads, sampler_threads=1, s_per_sweep=T_full, extrapolated=not full,
                sample_s_per_step=mean["step"], measured_s=float(np.sum(parts["step"])), items=m_s, respondents_theta=len(I),
                per_step_s={k: mean[k] for k in ("draw_f", "draw_fstar", "draw_theta", "draw_beta", "rebuild")},
                fixed_s=T_fix)


def cpu_fixed_part_by_blas_threads(n, theta, thread_counts):
    """K + Cholesky and the K* solve of one sweep (the BLAS/LAPACK-bound part, gpirtMCMC.cpp:76-78, draw-fstar.cpp:17-19) at
    each BLAS thread count; the sampler code around it is single-threaded like the reference."""
    from oracle import oracle as O
    ts, _ = O.grid()
    out = {}
    use_ref = os.path.exists(O.REF_SO)
    for t in thread_counts:
        O.set_blas_threads(t)
        t0 = time.perf_counter()
        if use_ref:
            S = O.ref_K(theta, theta); S[np.diag_indices(n)] += 0.001
            L = O.ref_chol_lower(S)
        else:
            L = O.build_cholS(theta)
        t1 = time.perf_counter()
        f1 = np.zeros((n, 1), order="F")
        if use_ref:
            O.ref_draw_fstar(f1, theta, ts, L, np.zeros((1001, 1), order="F"))
        else:
            O.draw_fstar(f1, theta, ts, L, np.zeros((1001, 1), order="F"), O.Rng.keyed(1))
        t2 = time.perf_counter()
        out[str(t)] = {"k_chol_s": t1 - t0, "kstar_solve_s": t2 - t1}
    return out


def cpu_reference_chain_ess(y, theta_init, S, B):
    """theta ESS/s of the reference's own gpirtMCMC() (oracle/_ref) on a small problem: the second half of BASELINE's metric"""
    from oracle import oracle as O
    from gpirt_b200.diagnostics import ess_geyer
    if not os.path.exists(O.REF_SO):
        return None
    m = y.shape[1]
    O.ref().gpref_seed(2026)
    t0 = time.perf_counter()
    r = O.ref_mcmc(np.asarray(y), theta_init, S, B, np.zeros((2, m)), np.full((2, m), 3.0), np.full((2, m), 0.1))
    el = time.perf_counter() - t0
    ess = ess_geyer(r["theta"][1:])
    ess = ess[np.isfinite(ess)]
    return {"samples": S, "burn": B, "seconds": el, "s_per_sweep_measured": el / (S + B), "sweeps_per_s": (S + B) / el,
            "ess_median": float(np.median(ess)), "ess_per_sec_median": float(np.median(ess) / el),
            "ess_per_sec_min": float(ess.min() / el), "note": "MEASURED full chain of the reference's own gpirtMCMC()"}


DUMP_BYTES = 48 << 20    # f and f* samples of one dump, summed over ranks; theta and beta add n per rank + 2 m doubles
DUMP_MAX_ITEMS = 256     # items sampled in all


def dump_outputs(s, out_dir, rank=0, world=1):
    """Writes the resident sampler's state after the last timed sweep as out_dir/<name>.npy (float64): theta (n),
    beta (2 x m), and f (n x k) / fstar (1001 x k) of k items drawn without replacement by a fixed seed, whose indices
    (0-based, local to this sampler's item block) go to `items`.  With world > 1 every rank writes its own item block as
    rank<r>_<name>.npy and samples 1 / world of the items and of the byte budget.  Returns the names written."""
    from gpirt_b200 import _lib
    n, m = s.n, s.m
    prefix = "rank%d_" % rank if world > 1 else ""
    k = int(min(m, max(1, DUMP_MAX_ITEMS // world), max(1, DUMP_BYTES // world // ((n + N_GRID) * 8))))
    items = np.sort(np.random.default_rng(synthetic.SEED + rank).choice(m, size=k, replace=False))
    # one whole field on the host at a time: the sampled columns are copied out before the next field is read
    arrays = {"theta": s.get(_lib.THETA), "beta": s.get(_lib.BETA), "items": items.astype(np.float64),
              "f": s.get(_lib.F)[:, items], "fstar": s.get(_lib.FSTAR)[:, items]}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))
    return sorted(prefix + name for name in arrays)


def shard_check(G, dist, rank, world, local_rank, fresh_uid):
    """N > 1: before anything is timed, the item-sharded sampler (CUDA path, NCCL exchanges) must reproduce the single-GPU
    chain on a small problem that takes the same code paths (fixed-point products, pipelined sweep, blocked-substitution
    solves).  Every rank compares its own item block with an unsharded run on its own GPU; the worst difference over ranks
    is returned.  Same solve route: bit-identical (addressed RNG, integer accumulation); default single-GPU route (through
    L^-1): theta identical, values to rounding."""
    import torch
    from gpirt_b200 import ResponseMatrix
    from gpirt_b200.sharding import item_block
    n, m, S, B = 640, 600, 2, 1
    d = synthetic.make(n, m, seed=77, missing=0.05)
    j0, j1 = item_block(m, rank, world)
    kw = dict(theta_init=d["theta_init"], seed=99, device=local_rank)
    got = G.gpirtMCMC(ResponseMatrix(d["y"][:, j0:j1]), S, B, beta_prior_means=d["pm"][:, j0:j1], beta_prior_sds=d["psd"][:, j0:j1],
                      beta_proposal_sds=d["pstep"][:, j0:j1], shard=(rank, world, m, j0, fresh_uid()), **kw)
    diffs = {}
    for route in ("1", None):
        old = os.environ.get("GPIRT_SOLVE_MODE")
        if route is not None:
            os.environ["GPIRT_SOLVE_MODE"] = route
        try:
            full = G.gpirtMCMC(ResponseMatrix(d["y"]), S, B, beta_prior_means=d["pm"], beta_prior_sds=d["psd"],
                               beta_proposal_sds=d["pstep"], **kw)
        finally:
            if route is not None:
                if old is None:
                    os.environ.pop("GPIRT_SOLVE_MODE", None)
                else:
                    os.environ["GPIRT_SOLVE_MODE"] = old
        v = [float(not np.array_equal(got["theta"], full["theta"])), float(np.max(np.abs(got["beta"] - full["beta"][:, j0:j1]))),
             float(np.max(np.abs(got["f"] - full["f"][:, j0:j1]))), float(np.max(np.abs(got["IRFs"] - full["IRFs"][:, j0:j1])))]
        t = torch.tensor(v, dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        diffs["same_route" if route else "default_route"] = dict(zip(("theta_differs", "max_dbeta", "max_df", "max_dirf"), t.tolist()))
    a, b = diffs["same_route"], diffs["default_route"]
    ok = (a["theta_differs"] == 0 and a["max_dbeta"] == 0 and a["max_df"] == 0 and a["max_dirf"] == 0 and
          b["theta_differs"] == 0 and b["max_dbeta"] <= 1e-9 and b["max_df"] <= 1e-7 and b["max_dirf"] <= 1e-7)
    return {"status": "ok" if ok else "FAILED", "shape": "%d x %d, %d sweeps, 5%% missing, world %d" % (n, m, S + B, world), **diffs}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="c3", choices=sorted(synthetic.WORKLOADS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--ess-samples", type=int, default=300)
    ap.add_argument("--fstar-mode", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the sampler state after the last timed sweep to DIR/<name>.npy (B200 arm)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the state of the B200 sampler; --impl reference has none")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    K, W = max(1, args.steps), max(0, args.warmup)
    cfg = synthetic.WORKLOADS[args.workload]
    n, m = cfg["n"], cfg["m"]
    config = {"workload": "%s (%s), synthetic 2PL responses, seed %d, priors pm=0 psd=3 step=0.1" % (args.workload, cfg["desc"], synthetic.SEED),
              "n": n, "m": m, "n_grid": N_GRID, "cache": "inputs larger than L2 (f, Z, nu are 3 x %.0f MB)" % (n * m * 8 / 1e6),
              "parallelism": "items sharded over %d GPU(s), logP all-reduce per sweep" % world if world > 1 else "single GPU"}
    host_threads = os.cpu_count() or 1

    # ------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        data = synthetic.make(n, m)
        # every step is one sampled sweep: all respondents, an item sample sized so that K + W steps end within a few
        # minutes (the same 64-item sample as the cpu_baseline leg of the B200 arm whenever that fits), the theta step on a
        # respondent sample.  Small workloads (c1, c2 with few steps) run whole.
        per_item = 2.2e-8 * n * N_GRID * min(1.0, 256.0 / n) + 1.4e-8 * n * n    # rough seconds per item of a sampled sweep
        fixed = 8e-11 * n ** 3 / max(1, min(host_threads, 8)) + 2e-8 * n * n
        budget = 240.0 / max(1, K + W)
        m_s = int(max(8, min(m, 64, (budget - fixed) / per_item)))
        whole = n * float(N_GRID) * m * 2.2e-8 * (K + W) < 240.0
        res = cpu_reference_sweeps(n, m, data, K, W, m if whole else m_s, host_threads, n_sub=None if whole else 256)
        line = {"impl": "reference", "metric": "gibbs_sweeps_per_sec", "value": res["value"], "unit": "sweeps/s", "n_gpus": args.gpus,
                "steps": K, "warmup": W, "ms_per_step": 1000.0 * res["sample_s_per_step"], "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
                "note": "ms_per_step is the MEASURED time of one sampled step (see cpu_baseline.sample); value is the full-size "
                        "throughput, 1 / ms_per_full_sweep%s" % ("" if not res["extrapolated"] else
                                                                 ", EXTRAPOLATED from the sample (exactly linear parts only)"),
                "ms_per_full_sweep": 1000.0 * res["s_per_sweep"], "extrapolated": res["extrapolated"],
                "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample", "blas_threads", "sampler_threads",
                                                       "items", "respondents_theta", "per_step_s", "fixed_s")},
                "e2e": {"value": res["value"], "unit": "sweeps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ B200 arm
    import gpirt_b200.sampler as G
    from gpirt_b200 import _lib
    dist = None
    uid = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        from gpirt_b200.sharding import share_unique_id

        def fresh_uid():   # one ncclUniqueId per communicator
            return share_unique_id(dist, rank, G.nccl_unique_id, device="cuda")
        uid = fresh_uid()
    shard_ok = shard_check(G, dist, rank, world, local_rank, fresh_uid) if world > 1 else None
    if shard_ok is not None and shard_ok["status"] != "ok":
        if rank == 0:
            print(json.dumps({"metric": "gibbs_sweeps_per_sec", "value": None, "n_gpus": world, "shard_check": shard_ok,
                              "error": "the sharded sampler does not reproduce the single-GPU chain; nothing was timed"}))
        dist.destroy_process_group()
        return 1
    data = synthetic.make(n, m)
    # contiguous item block of this rank
    from gpirt_b200.sharding import item_block
    j0, j1 = item_block(m, rank, world)
    y_loc = np.asfortranarray(data["y"][:, j0:j1])
    kw = dict(seed=synthetic.SEED, device=local_rank, fstar_mode=args.fstar_mode)
    if world > 1:
        kw.update(rank=rank, world_size=world, m_global=m, item_offset=j0, nccl_unique_id=uid)
    s = G.Sampler(y_loc, data["theta_init"], data["pm"][:, j0:j1], data["psd"][:, j0:j1], data["pstep"][:, j0:j1], **kw)
    s.init_draws()
    # The timed region runs the sampler the way gpirt_b200_mcmc() runs it: per-step timers off, every sweep after the first
    # replayed as one CUDA graph launch (the pipelined sweep is launch-bound on the host otherwise: ~15 API calls per
    # Cholesky panel).  The per-step breakdown is taken afterwards from a second, eager pass with the timers on.
    s.set_timing(False)
    s.sweep(max(3, W) + 1)                   # >= 3 untimed warm-up sweeps (+ the eager one that precedes the graph capture)
    launches0 = s.launches()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
        time.sleep(0.3)
    if dist is not None:
        dist.barrier()
    ms = s.sweep(K)                          # CUDA events on the sampler's stream, sync on both sides inside the call
    if dist is not None:
        import torch
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        dist.barrier()
    clk = clocks.finish() if rank == 0 else None
    launches = s.launches() - launches0
    dumped = None
    if args.dump_outputs:                    # read-only copies of the state the timed sweeps left
        dumped = dump_outputs(s, args.dump_outputs, rank, world)
    s.set_timing(True)                       # eager pass with CUDA-event timers around every step
    s.sweep(2)
    s.timings(reset=True)
    ms_eager = s.sweep(K)
    timers = s.timings()
    value = 1000.0 * K / ms

    # roofline of the dominant KERNEL: timer segments are grouped by the kernel that runs them (the fixed-point tensor-core
    # GEMM serves three segments), the group with the largest summed CUDA-event time in the timed region is reported
    m_loc = j1 - j0
    work = {"lz_gemm": ("tensor", float(n) * n * m_loc), "fstar_gemm": ("tensor", 2.0 * n * N_GRID * m_loc),
            "chol": ("tensor", n ** 3 / 3.0), "trtri": ("tensor", n ** 3 / 3.0),
            "trsm": ("tensor", 2.0 * n * n * N_GRID if args.fstar_mode == 0 else n * n * N_GRID + 2.0 * n * n * m_loc),
            "ess": ("hbm", 25.0 * n * m_loc), "beta": ("hbm", 17.0 * n * m_loc), "kbuild": ("hbm", 4.0 * n * n)}
    fixed_point = s.uses(1) == 1
    groups = {k: [k] for k in work}
    names = {"chol": "potrf_lower_rl (k_diag128 + gemm_f64_kernel updates)", "trtri": "trtri_lower (gemm_f64_kernel)",
             "lz_gemm": "gemm_f64_kernel (nu = L Z)", "fstar_gemm": "gemm_f64_kernel (f* product)", "trsm": "gemm_f64_kernel (K* solves)",
             "ess": "k_ess_persist", "beta": "k_beta", "kbuild": "k_se_cov"}
    if fixed_point:
        # 36 exact int8 plane-pair products on tcgen05 (dgemm_i8.cu): the tensor pipe executes 36 x the FP64 product's work
        i8_segs = ["lz_gemm", "fstar_gemm"] + (["trsm"] if args.fstar_mode == 0 and world == 1 else [])
        for k in i8_segs:
            del groups[k]
        groups["k_dgemm_i8"] = i8_segs
        names["k_dgemm_i8"] = "k_dgemm_i8 (%s)" % " + ".join(i8_segs)
    seg_ms = {k: timers[k][0] / K for k in work}              # per sweep, pipelined (a segment may be several launches)
    dom = max(groups, key=lambda g: sum(seg_ms[k] for k in groups[g]))
    segs = groups[dom]
    dom_ms = sum(seg_ms[k] for k in segs)
    fp64_work = sum(work[k][1] for k in segs)
    bound = work[segs[0]][0]
    peaks, peak_src = _peaks()
    dmma, dfma = G.fp64_peak_tflops()
    fp64_src = ("FP64 tensor pipe (DMMA.8x8x4) issue-rate microbenchmark measured in this run; "
                "MEASURED_PEAKS.json has no FP64 figure")
    # the same segments timed WITHOUT sweep pipelining (no co-running kernels): kernel quality, not schedule
    s.set_pipeline(False)
    s.sweep(1)
    s.timings(reset=True)
    Ki = 3
    ms_iso = s.sweep(Ki)
    t_iso = s.timings()
    s.set_pipeline(True)
    iso_ms = sum(t_iso[k][0] for k in segs) / Ki
    i8_note = None
    if dom == "k_dgemm_i8":
        # the int8 ceiling is MEASURED in this run: tcgen05.mma.kind::i8 (M128 N256 K32, operands in shared memory) issued
        # back to back on every SM (gpirt_b200_int8_peak_tops); MEASURED_PEAKS.json has no int8 figure
        i8_peak = G.int8_peak_tops()
        i8_peak_rand = G.int8_peak_tops(random_operands=True)
        alg = 36.0 * fp64_work
        peak = iso_peak = i8_peak
        achieved, iso, unit = alg / dom_ms * 1e-9, alg / iso_ms * 1e-9, "TOP/s"
        peak_src = ("tcgen05.mma.kind::i8 issue-rate microbenchmark measured in this run (%.0f TOP/s; nominal dense int8 4500; "
                    "2 x the dense bf16 figure of MEASURED_PEAKS.json would be %.0f)" % (i8_peak, 2.0 * peaks["bf16_tflops"]))
        i8_note = {"plane_pair_products": 36, "fp64_tensor_peak_tflops": dmma,
                   "power_limited_peak": {"value": i8_peak_rand, "unit": "TOP/s",
                                          "frac": alg / dom_ms * 1e-9 / i8_peak_rand, "frac_isolated": alg / iso_ms * 1e-9 / i8_peak_rand,
                                          "note": "the same issue-rate microbenchmark with pseudo-random digit planes as operands: "
                                                  "identical cycles per MMA, but the switching power pulls the SM clock down "
                                                  "(profiles/r02_umma_i8_shapes.txt); `peak` / `frac` above stay on the "
                                                  "near-constant-operand figure, the stricter denominator"},
                   "fp64_equivalent_tflops": fp64_work / dom_ms * 1e-9, "fp64_equivalent_tflops_isolated": fp64_work / iso_ms * 1e-9,
                   "segments_ms": {k: seg_ms[k] for k in segs}, "segments_ms_isolated": {k: t_iso[k][0] / Ki for k in segs},
                   "note": "`achieved` counts the 36 exact int8 plane-pair products the scheme EXECUTES per FP64 product; the "
                           "algorithmic work of SURVEY 8(d) is the FP64 product itself: see fp64_equivalent_frac (FP64 flop / "
                           "measured FP64 tensor peak; > 1 means faster than any FP64-pipe GEMM could be).  Segment times include "
                           "the operand slicing kernels of each product"}
        bound = "tensor"
    elif bound == "tensor":
        alg = fp64_work
        achieved, iso, peak, iso_peak, unit, peak_src = alg / dom_ms * 1e-9, alg / iso_ms * 1e-9, dmma, dmma, "TFLOP/s", fp64_src
    else:
        alg = fp64_work
        achieved, iso, peak, iso_peak, unit = alg / dom_ms * 1e-6, alg / iso_ms * 1e-6, peaks["hbm_gbs"], peaks["hbm_gbs"], "GB/s"
    traffic = None
    tp = os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")
    if os.path.exists(tp):
        try:
            with open(tp) as fh:
                traffic = json.load(fh).get(args.workload, {}).get(dom)
        except Exception:
            traffic = None
    roofline = {"kernel": names.get(dom, dom), "bound": bound, "achieved": achieved, "peak": peak, "unit": unit, "frac": achieved / peak,
                "traffic": traffic, "peak_source": peak_src, "algorithmic_work_per_sweep": alg,
                "ms_per_sweep": dom_ms, "share_of_step": dom_ms / (ms_eager / K),
                "ms_per_step_eager_with_timers": ms_eager / K,
                "note": "timed region runs pipelined: the L Z product and the beta step execute UNDER the Cholesky chain and the K* "
                        "solves beside the ESS, so their event durations include co-running kernels (shares can sum to > 1); "
                        "`isolated` repeats the measurement with pipelining off",
                "isolated": {"achieved": iso, "peak": iso_peak, "frac": iso / iso_peak, "ms_per_sweep": iso_ms,
                             "sweep_ms_unpipelined": ms_iso / Ki},
                "fixed_point": i8_note,
                "fp64_equivalent_frac": (fp64_work / dom_ms * 1e-9) / dmma if bound == "tensor" else None,
                "fp64_equivalent_frac_isolated": (fp64_work / iso_ms * 1e-9) / dmma if bound == "tensor" else None,
                "cholesky": {"ms_isolated": t_iso["chol"][0] / Ki, "ms_pipelined": timers["chol"][0] / K,
                             "tflops_isolated": n ** 3 / 3.0 / (t_iso["chol"][0] / Ki) * 1e-9,
                             "frac_of_fp64_tensor_peak_isolated": n ** 3 / 3.0 / (t_iso["chol"][0] / Ki) * 1e-9 / dmma,
                             "note": "potrf_lower_rl: k_diag128 + k_panel_update chain with look-ahead bulk updates on gemm_f64_kernel"},
                "per_step_ms": {k: v[0] / K for k, v in timers.items() if v[1]},
                "per_step_ms_isolated": {k: v[0] / Ki for k, v in t_iso.items() if v[1]}}
    try:   # the factorisation alone, eager and as the product runs it (replayed as a CUDA graph): K build + chain
        chol_eager, chol_graph = s.time_factorisation(10, False), s.time_factorisation(10, True)
        roofline["cholesky"].update({"ms_alone_eager_incl_k_build": chol_eager, "ms_alone_graph_replay_incl_k_build": chol_graph,
                                     "frac_of_fp64_tensor_peak_graph_replay": n ** 3 / 3.0 / chol_graph * 1e-9 / dmma})
    except Exception as exc:   # measurement extra only
        roofline["cholesky"]["graph_replay_error"] = str(exc)
    s.close()

    line = {"metric": "gibbs_sweeps_per_sec", "value": value, "unit": "sweeps/s", "n_gpus": world, "steps": K, "warmup": max(3, W),
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": config, "gpu_launches": int(launches), "clocks": clk, "roofline": roofline}
    if shard_ok is not None:
        line["shard_check"] = shard_ok
    if dumped is not None:
        line["outputs"] = {"dir": args.dump_outputs, "arrays": dumped}

    # ------------------------------------------------------------------ chain-parallel mode (BASELINE config 4), N > 1 only
    # every rank runs an INDEPENDENT chain of the whole workload (own seed, no communication): aggregate sweeps/s
    if world > 1 and not args.no_extras:
        sc = G.Sampler(data["y"], data["theta_init"], data["pm"], data["psd"], data["pstep"], seed=synthetic.SEED + 1000 + rank,
                       device=local_rank, fstar_mode=args.fstar_mode)
        sc.set_timing(False)
        sc.init_draws()
        sc.sweep(max(3, W))
        dist.barrier()
        ms_c = sc.sweep(K)
        import torch
        t = torch.tensor([ms_c], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sc.close()
        line["chain_parallel"] = {"value": 1000.0 * K * world / float(t.item()), "unit": "sweeps/s (sum over %d independent chains)" % world,
                                  "ms_per_step_per_chain": float(t.item()) / K, "scaling": "weak",
                                  "note": "one full-size chain per GPU, no collective (BASELINE config 4); `value` above is the item-sharded single chain (config 3)"}

    # ------------------------------------------------------------------ end-to-end through the public call (host buffers)
    if not args.no_e2e:
        from gpirt_b200 import ResponseMatrix
        # f draws are n*m*8 bytes per stored sweep on the host: 30 sampling iterations of the local item block (10 GB at C3 on
        # one GPU) amortise the fixed cost of a call (create 35 ms, first eager sweeps) the way a real run does; bounded
        # by the host allocation, independent of --steps
        per_slot = n * m_loc * 8
        Ke = int(max(4, min(30, (12 << 30) // max(per_slot, 1))))
        yrm = ResponseMatrix(y_loc)
        common = dict(beta_prior_means=data["pm"][:, j0:j1], beta_prior_sds=data["psd"][:, j0:j1],
                      beta_proposal_sds=data["pstep"][:, j0:j1], theta_init=data["theta_init"], seed=synthetic.SEED,
                      device=local_rank, fstar_mode=args.fstar_mode)
        shard = (rank, world, m, j0, fresh_uid()) if world > 1 else None
        G.gpirtMCMC(yrm, 1, 0, shard=shard, **common)     # warm the call path (allocator, pinning, communicator)
        shard = (rank, world, m, j0, None) if world > 1 else None   # re-use the communicator of the previous call
        if dist is not None:
            dist.barrier()
        t0 = time.perf_counter()
        out = G.gpirtMCMC(yrm, Ke, 0, shard=shard, **common)
        el = time.perf_counter() - t0
        if dist is not None:
            import torch
            t = torch.tensor([el], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            el = float(t.item())
        assert np.isfinite(out["theta"]).all()
        h2d = (n * m_loc + n + 6 * m_loc) * 8 / Ke
        d2h = (n * m_loc + 2 * m_loc + n) * 8 * (Ke + 1) / Ke + N_GRID * m_loc * 8 / Ke
        line["e2e"] = {"value": Ke / el, "unit": "sweeps/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                       "note": "gpirtMCMC(sample_iterations=%d, burn_iterations=0) wall time incl. setup, initial draws, H2D of y "
                               "and D2H of every theta/beta/f draw (reference output contract)" % Ke}
        del out
        if world == 1 and not args.no_extras:
            # the same public call keeping every 10th sampling iteration (opts.thin) and the posterior mean / sd of f
            # accumulated on the device: the n x m x (S+1) array of f draws is what bounds `e2e`
            St = 100
            t0 = time.perf_counter()
            out = G.gpirtMCMC(yrm, St, 0, thin=10, f_summary=True, **common)
            el_t = time.perf_counter() - t0
            assert out["f"].shape[2] == St // 10 + 1 and np.isfinite(out["f_mean"]).all()
            line["e2e"]["thin10"] = {"value": St / el_t, "unit": "sweeps/s", "frac_of_value": (St / el_t) / value,
                                     "d2h_bytes_per_step": int((n * m_loc + 2 * m_loc + n) * 8 * (St // 10 + 1) / St + (N_GRID + 2 * n) * m_loc * 8 / St),
                                     "note": "gpirtMCMC(%d, 0, thin=10, f_summary=True): every 10th draw of theta / beta / f stored, "
                                             "f mean and sd over all %d iterations returned" % (St, St)}
            del out

    # ------------------------------------------------------------------ theta ESS/sec (second half of BASELINE's metric), N = 1 only
    if rank == 0 and world == 1 and not args.no_extras:
        try:
            from gpirt_b200 import ResponseMatrix
            from gpirt_b200.diagnostics import ess_geyer
            S_ess, B_ess = args.ess_samples, 50
            t0 = time.perf_counter()
            ch = G.gpirtMCMC(ResponseMatrix(y_loc), S_ess, B_ess, beta_prior_means=data["pm"], beta_prior_sds=data["psd"],
                             beta_proposal_sds=data["pstep"], theta_init=data["theta_init"], seed=synthetic.SEED, device=local_rank,
                             store_f=False, fstar_mode=args.fstar_mode)
            el_ess = time.perf_counter() - t0
            ess = ess_geyer(ch["theta"][1:])
            ess = ess[np.isfinite(ess)]
            line["theta_ess"] = {"samples": S_ess, "burn": B_ess, "seconds": el_ess, "ess_median": float(np.median(ess)),
                                 "ess_min": float(ess.min()), "ess_per_sec_median": float(np.median(ess) / el_ess),
                                 "ess_per_sec_min": float(ess.min() / el_ess),
                                 "estimator": "Geyer initial positive sequence per respondent; seconds = wall time of the "
                                              "gpirtMCMC(S, B, store_f=False) call incl. burn-in",
                                 "corr_with_generating_theta": float(abs(np.corrcoef(ch["theta"][1:].mean(axis=0), data["theta_true"])[0, 1]))}
            if "e2e" in line:   # the same public call without the n x m x (S+1) f array: what bounds `e2e` is storing f
                line["e2e"]["without_f_draws"] = {"value": (S_ess + B_ess) / el_ess, "unit": "sweeps/s",
                                                  "note": "gpirtMCMC(%d, %d, store_f=False) wall time: theta, beta and IRFs "
                                                          "still come back to the host every sweep" % (S_ess, B_ess)}
        except Exception as ex:
            line["theta_ess"] = {"error": repr(ex)}

    # ------------------------------------------------------------------ the other single-GPU configs, briefly (N = 1 only)
    if rank == 0 and world == 1 and args.workload == "c3" and not args.no_extras:
        extras = {}
        for wl, miss, k2 in (("c1", 0.0, 200), ("c2", 0.0, 50), ("c3", 0.05, 10), ("c5", 0.0, 5)):
            key = wl if miss == 0.0 else "%s_missing%d" % (wl, int(100 * miss))
            try:
                c = synthetic.WORKLOADS[wl]
                d2 = synthetic.make(c["n"], c["m"], missing=miss)
                s2 = G.Sampler(d2["y"], d2["theta_init"], d2["pm"], d2["psd"], d2["pstep"], seed=synthetic.SEED, device=local_rank)
                s2.init_draws()
                s2.sweep(3)
                s2.set_timing(False)                 # the per-step events cost as much as the kernels at the small shapes
                ms2 = s2.sweep(k2)
                s2.set_timing(True)
                s2.timings(reset=True)
                s2.sweep(min(k2, 20))
                t2 = {k: (v[0] * k2 / min(k2, 20), v[1]) for k, v in s2.timings().items()}
                extras[key] = {"n": c["n"], "m": c["m"], "missing": miss, "value": 1000.0 * k2 / ms2, "unit": "sweeps/s",
                               "ms_per_step": ms2 / k2, "steps": k2, "per_step_ms": {k: v[0] / k2 for k, v in t2.items() if v[1]}}
                if wl == "c5":   # the large-n configuration: Cholesky roofline and footprint
                    s2.set_pipeline(False)
                    s2.sweep(1); s2.timings(reset=True); s2.sweep(2)
                    ti = s2.timings()
                    nn = c["n"]
                    extras[key]["cholesky"] = {"ms_isolated": ti["chol"][0] / 2, "tflops_isolated": nn ** 3 / 3.0 / (ti["chol"][0] / 2) * 1e-9,
                                               "frac_of_fp64_tensor_peak_isolated": nn ** 3 / 3.0 / (ti["chol"][0] / 2) * 1e-9 / dmma}
                    extras[key]["hbm_footprint_gb"] = (6 * nn * nn * 8 + 3 * nn * c["m"] * 8 + 11 * nn * c["m"] + 3 * 1008 * c["m"] * 8 + 16 * nn * nn) / 1e9
                s2.close()
                del d2, s2
            except Exception as ex:
                extras[key] = {"error": repr(ex)}
        line["other_workloads"] = extras

    # ------------------------------------------------------------------ CPU baseline beside it (rank 0, N = 1 only)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            # the bench workload: one sampled sweep (64 items, theta step on 256 respondents), extrapolated as stated in `sample`
            res = cpu_reference_sweeps(n, m, data, 1, 0, 64, host_threads, n_sub=256)
            cb = {k: res[k] for k in ("value", "unit", "cores", "kind", "sample", "blas_threads", "sampler_threads", "items",
                                      "respondents_theta", "per_step_s", "fixed_s", "extrapolated")}
            if not args.no_extras:
                cb["fixed_part_by_blas_threads"] = cpu_fixed_part_by_blas_threads(n, data["theta_init"], sorted({1, min(8, host_threads), host_threads}))
                # MEASURED full sweeps of the reference at the small configurations, and its theta ESS/s on the real data set
                c2 = synthetic.WORKLOADS["c2"]
                r2 = cpu_reference_sweeps(c2["n"], c2["m"], synthetic.make(c2["n"], c2["m"]), 1, 0, c2["m"], host_threads)
                cb["c2_full_sweep"] = {k: r2[k] for k in ("value", "unit", "sample", "per_step_s", "extrapolated")}
                import warnings
                import gpirt_b200
                codes, _, _ = gpirt_b200.senate116()
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    y1 = gpirt_b200.response_matrix(codes)
                th1 = np.random.RandomState(116).randn(y1.shape[0])
                cb["c1_senate116_chain"] = cpu_reference_chain_ess(y1, th1, 30, 10)
                t0 = time.perf_counter()
                g1 = G.gpirtMCMC(y1, 300, 100, theta_init=th1, seed=116, device=local_rank, store_f=False)
                el1 = time.perf_counter() - t0
                from gpirt_b200.diagnostics import ess_geyer
                e1 = ess_geyer(g1["theta"][1:]); e1 = e1[np.isfinite(e1)]
                cb["c1_senate116_chain_b200"] = {"samples": 300, "burn": 100, "seconds": el1, "sweeps_per_s": 400 / el1,
                                                 "ess_median": float(np.median(e1)), "ess_per_sec_median": float(np.median(e1) / el1)}
            line["cpu_baseline"] = cb
        except Exception as ex:  # the baseline is informative; never lose the GPU line over it
            line["cpu_baseline"] = {"value": None, "unit": "sweeps/s", "cores": host_threads, "kind": "port", "sample": "failed: %r" % (ex,)}
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(line))
    return 0


if __name__ == "__main__":
    sys.exit(main())
