"""Host-side mirror of the reference's R entry point over the C ABI.

gpirtMCMC() has the reference's signature and return value (R/gpirtMCMC.R:85-105 -> src/gpirtMCMC.cpp:5-117):
    gpirtMCMC(data, sample_iterations, burn_iterations, vote_codes=..., beta_prior_means=None, beta_prior_sds=None,
              beta_proposal_sds=None, theta_init=None)  ->  dict(theta, beta, f, IRFs)
with theta (S+1, n), beta (2, m, S+1), f (n, m, S+1), IRFs (1001, m), slot 0 holding the initial values.
Everything numerical happens in libgpirt_b200.so (CUDA); this file only marshals arrays."""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import Chains, Fit, GpirtError, Irf, Loo, Opts, Ppc, N_GRID
from .response_matrix import DEFAULT_CODES, as_response_matrix


def _F(a, shape=None):
    a = np.asfortranarray(np.asarray(a, dtype=np.float64))
    if shape is not None and a.shape != shape:
        raise ValueError("expected shape %r, got %r" % (shape, a.shape))
    return a


def make_opts(seed=0, device=-1, fstar_mode=0, skip_f_draws=False, rank=0, world_size=1, m_global=0, item_offset=0,
              nccl_unique_id=None, thin=1, use_graph=0):
    o = Opts()
    o.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    o.device = device
    o.fstar_mode = fstar_mode
    o.skip_f_draws = int(bool(skip_f_draws))
    o.rank, o.world_size, o.m_global, o.item_offset = rank, world_size, m_global, item_offset
    o.thin = int(thin)
    o.use_graph = int(use_graph)
    o._uid_keepalive = None
    if nccl_unique_id is not None:
        buf = C.create_string_buffer(bytes(nccl_unique_id), 128)
        o._uid_keepalive = buf
        o.nccl_unique_id = C.cast(buf, C.c_void_p)
    return o


def nccl_unique_id():
    buf = C.create_string_buffer(128)
    _lib.check(_lib.load().gpirt_b200_nccl_unique_id(buf))
    return buf.raw


def gpirtMCMC(data, sample_iterations, burn_iterations, vote_codes=None, beta_prior_means=None, beta_prior_sds=None,
              beta_proposal_sds=None, theta_init=None, *, seed=None, progress=None, store_f=True, fstar_mode=0,
              device=-1, shard=None, thin=1, f_summary=False, use_graph=0, predictive=False, y_holdout=None,
              irf_band=None, store_fstar=False, chains=None, chain_diagnostics=False, ppc=False, ppc_pairs=False,
              loo=False):
    """Drop-in for the reference's gpirtMCMC().  Keyword-only extras (not in the reference): seed (Philox key; default
    drawn from numpy's global RNG, as the R shim draws it from R's), progress(percent) -> truthy to interrupt,
    store_f=False to skip the n*m*(S+1) f draws, shard=(rank, world, m_global, item_offset, unique_id) for item
    sharding across GPUs, thin=k to keep every k-th sampling iteration only (outputs then hold 1 + S // k slots; IRFs
    still average over all S), f_summary=True to also return the posterior mean / sd of f over all sampling iterations
    (accumulated on the device: "f_mean", "f_sd", n x m), predictive=True to also return posterior predictive
    probabilities, WAIC and held-out scores over all sampling iterations ("predictive": dict with pred, lpd_cell, pwaic_cell
    (n x m), elpd_item (m), elpd_resp (n) and the scalars lppd, p_waic, elpd_waic, waic, se_elpd_waic, lpd_holdout, n_obs,
    n_holdout; accumulated on the device, definitions in include/gpirt_b200.h), y_holdout = n x m array of the coded
    response matrix's shape holding +1 / -1 where a missing response was held out (NaN elsewhere; read where y is NA).
    With shard, per-cell and per-item outputs cover the local items, elpd_resp and the scalars all items.
    irf_band=b (0 < b < 1) to also return "IRF_summary": dict(mean, sd, lower, upper) of P(y = +1 | theta*) on the grid
    (1001 x m, over all sampling iterations; lower / upper are the exact pointwise type-7 quantiles at (1 -+ b) / 2 of f*
    mapped through plogis), band = b and band_bytes = the device memory of its tail buffers; store_fstar=True to also return
    the f* draws "fstar" (1001 x m x slots, the slots of theta / beta).  With shard both cover the local items.
    chains=C (1..32) runs C chains concurrently on one GPU in this call: theta_init may be n x C (None: each chain's drawn
    from numpy's global RNG), an integer seed gives chain c the seed seed + c (chain 0 equals a call with that seed), a
    sequence of C seeds is used as given, and theta, beta, f and IRFs gain a trailing chain axis.  chain_diagnostics=True
    also returns "diagnostics": dict(theta_rhat, theta_ess (n), beta_rhat, beta_ess (2 x m), irf_rhat (1001 x m),
    diag_bytes), split-R-hat and summed Geyer ESS over all S sampling iterations (any thin), computed on the device
    (definitions in include/gpirt_b200.h).  chains cannot be combined with shard, predictive, irf_band, store_fstar,
    f_summary or ppc.
    ppc=True also returns "ppc": posterior predictive checks over all S sampling iterations (any thin), computed on the
    device (definitions in include/gpirt_b200.h): dict(item_ppp (m), resp_ppp (n), ppp), the PPP-values of the Pearson
    chi-square per item, per respondent and in all; ppc_pairs=True adds pair_ppp and pair_log_or (m x m, symmetric), the
    PPP-values and observed values of the pairwise log odds ratios (local dependence), and pair_bytes, the device memory
    of their state.  ppc cannot be combined with shard.
    loo=True also returns "loo": leave-one-out cross-validation by Pareto-smoothed importance sampling over all S sampling
    iterations (any thin), computed on the device with every observed cell one left-out unit (definitions in
    include/gpirt_b200.h): dict(elpd_loo_cell, p_loo_cell, pareto_k (n x m, NaN on unobserved cells), elpd_loo_item (m),
    elpd_loo_resp (n), elpd_loo, p_loo, looic, se_elpd_loo, k_threshold, n_obs, n_k_high (cells whose Pareto k exceeds
    k_threshold: their elpd_loo_cell is unreliable), tail_len, tail_bytes (the device memory of its state, 8 (tail_len + 4)
    bytes per cell)).  loo cannot be combined with chains or shard."""
    C_ = None
    if chains is not None:
        if isinstance(chains, (bool, np.bool_)) or not isinstance(chains, (int, np.integer)) or not 1 <= int(chains) <= 32:
            raise ValueError("chains must be an integer in [1, 32], got %r" % (chains,))
        C_ = int(chains)
        for name, v in (("shard", shard is not None), ("predictive", predictive), ("irf_band", irf_band is not None),
                        ("store_fstar", store_fstar), ("f_summary", f_summary), ("ppc", ppc), ("loo", loo)):
            if v:
                raise ValueError("chains cannot be combined with %s" % name)
    elif chain_diagnostics:
        raise ValueError("chain_diagnostics needs chains")
    if ppc_pairs and not ppc:
        raise ValueError("ppc_pairs needs ppc")
    if ppc and shard is not None:
        raise ValueError("ppc cannot be combined with shard")
    if loo and shard is not None:
        raise ValueError("loo cannot be combined with shard")
    if irf_band is not None:
        irf_band = float(irf_band)
        if not 0.0 < irf_band < 1.0:   # NaN fails too
            raise ValueError("irf_band must lie in (0, 1), got %r" % irf_band)
    y = as_response_matrix(data, vote_codes or DEFAULT_CODES)                        # R/gpirtMCMC.R:93
    y = np.asfortranarray(np.asarray(y, dtype=np.float64))
    n, m = y.shape
    if C_ is not None:
        if theta_init is None:
            theta_init = np.stack([np.random.standard_normal(n) for _ in range(C_)], axis=1)
        theta_init = np.asfortranarray(theta_init, dtype=np.float64)
        if theta_init.shape != (n, C_):
            raise ValueError("theta_init must be nrow(data) x chains = %r, got %r" % ((n, C_), theta_init.shape))
        if seed is not None and not isinstance(seed, (int, np.integer)):
            seed = [int(v) for v in seed]
            if len(seed) != C_:
                raise ValueError("seed must be an integer or a sequence of %d seeds, got %d" % (C_, len(seed)))
    else:
        if theta_init is None:
            theta_init = np.random.standard_normal(n)                               # R/gpirtMCMC.R:95-97
        theta_init = np.ascontiguousarray(theta_init, dtype=np.float64)
        if theta_init.shape != (n,):
            raise ValueError("theta_init must have length nrow(data)")
    pm = _F(np.zeros((2, m)) if beta_prior_means is None else beta_prior_means, (2, m))   # R/gpirtMCMC.R:88
    psd = _F(np.full((2, m), 3.0) if beta_prior_sds is None else beta_prior_sds, (2, m))  # :89
    pstep = _F(np.full((2, m), 0.1) if beta_proposal_sds is None else beta_proposal_sds, (2, m))  # :90
    S, B = int(sample_iterations), int(burn_iterations)                             # RcppExports.cpp:22-23 coerce to int
    if seed is None:
        seed = int(np.random.randint(0, 2 ** 31 - 1)) | (int(np.random.randint(0, 2 ** 31 - 1)) << 32)
    seeds = None
    if C_ is not None:
        given = [int(seed) + c for c in range(C_)] if isinstance(seed, (int, np.integer)) else seed
        seeds = np.array([v & 0xFFFFFFFFFFFFFFFF for v in given], dtype=np.uint64)
        seed = int(seeds[0])
    kw = {}
    if shard is not None:
        kw = dict(rank=shard[0], world_size=shard[1], m_global=shard[2], item_offset=shard[3], nccl_unique_id=shard[4])
    thin = int(thin)
    if thin < 1:
        raise ValueError("thin must be >= 1")
    opts = make_opts(seed=seed, device=device, fstar_mode=fstar_mode, skip_f_draws=not store_f, thin=thin, use_graph=use_graph, **kw)
    slots = S // thin + 1
    ch = () if C_ is None else (C_,)
    theta = np.empty((slots, n) + ch, order="F")
    beta = np.empty((2, m, slots) + ch, order="F")
    f = np.empty((n, m, slots) + ch, order="F") if store_f else None
    irf = np.empty((N_GRID, m) + ch, order="F")
    chains_s = diag = None
    if C_ is not None:
        chains_s = Chains()
        chains_s.chains = C_
        chains_s.seeds = seeds.ctypes.data_as(C.POINTER(C.c_uint64))
        if chain_diagnostics:
            diag = dict(theta_rhat=np.empty(n), theta_ess=np.empty(n), beta_rhat=np.empty((2, m), order="F"),
                        beta_ess=np.empty((2, m), order="F"), irf_rhat=np.empty((N_GRID, m), order="F"))
            for k, a in diag.items():
                setattr(chains_s, k, _lib.ptr(a))
        opts.chains = C.pointer(chains_s)
    f_mean = f_sd = None
    fit = None
    if y_holdout is not None and not predictive:
        raise ValueError("y_holdout is only read with predictive=True")
    if predictive:
        fit = Fit()
        if y_holdout is not None:
            y_holdout = _F(y_holdout)
            if y_holdout.shape != (n, m):
                raise ValueError("y_holdout must have the shape of the coded response matrix %r, got %r" % ((n, m), y_holdout.shape))
            fit.y_holdout = _lib.ptr(y_holdout)
        pred = dict(pred=np.empty((n, m), order="F"), lpd_cell=np.empty((n, m), order="F"),
                    pwaic_cell=np.empty((n, m), order="F"), elpd_item=np.empty(m), elpd_resp=np.empty(n))
        for k, a in pred.items():
            setattr(fit, k, _lib.ptr(a))
        opts.fit = C.pointer(fit)
    if f_summary:
        f_mean = np.empty((n, m), order="F"); f_sd = np.empty((n, m), order="F")
        opts.f_mean_out = _lib.ptr(f_mean); opts.f_sd_out = _lib.ptr(f_sd)
    irf_s = None
    fstar = np.empty((N_GRID, m, slots), order="F") if store_fstar else None
    if irf_band is not None or store_fstar:
        irf_s = Irf()
        irf_s.fstar_draws = _lib.ptr(fstar)
        if irf_band is not None:
            summ = {k: np.empty((N_GRID, m), order="F") for k in ("mean", "sd", "lower", "upper")}
            irf_s.band = irf_band
            irf_s.prob_mean, irf_s.prob_sd = _lib.ptr(summ["mean"]), _lib.ptr(summ["sd"])
            irf_s.lower, irf_s.upper = _lib.ptr(summ["lower"]), _lib.ptr(summ["upper"])
        opts.irf = C.pointer(irf_s)
    ppc_s = None
    if ppc:
        ppc_s = Ppc()
        checks = dict(item_ppp=np.empty(m), resp_ppp=np.empty(n))
        if ppc_pairs:
            checks.update(pair_ppp=np.empty((m, m), order="F"), pair_log_or=np.empty((m, m), order="F"))
        for k, a in checks.items():
            setattr(ppc_s, k, _lib.ptr(a))
        opts.ppc = C.pointer(ppc_s)
    loo_s = None
    if loo:
        loo_s = Loo()
        loo_out = dict(elpd_loo_cell=np.empty((n, m), order="F"), p_loo_cell=np.empty((n, m), order="F"),
                       pareto_k=np.empty((n, m), order="F"), elpd_loo_item=np.empty(m), elpd_loo_resp=np.empty(n))
        for k, a in loo_out.items():
            setattr(loo_s, k, _lib.ptr(a))
        opts.loo = C.pointer(loo_s)

    def _cb(pct, _ctx):
        try:
            return 1 if (progress is not None and progress(pct)) else 0
        except KeyboardInterrupt:
            return 1
    cb = _lib.PROGRESS_CB(_cb)
    L = _lib.load()
    rc = L.gpirt_b200_mcmc(_lib.ptr(y), n, m, _lib.ptr(theta_init), S, B, _lib.ptr(pm), _lib.ptr(psd), _lib.ptr(pstep),
                           C.byref(opts), _lib.ptr(theta), _lib.ptr(beta), _lib.ptr(f), _lib.ptr(irf), cb, None)
    _lib.check(rc)
    out = dict(theta=theta, beta=beta, IRFs=irf)
    if store_f:
        out["f"] = f
    if f_summary:
        out["f_mean"], out["f_sd"] = f_mean, f_sd
    if predictive:
        for k in ("lppd", "p_waic", "elpd_waic", "waic", "se_elpd_waic", "lpd_holdout", "n_obs", "n_holdout"):
            pred[k] = getattr(fit, k)
        out["predictive"] = pred
    if irf_band is not None:
        out["IRF_summary"] = dict(summ, band=irf_band, band_bytes=int(irf_s.band_bytes))
    if store_fstar:
        out["fstar"] = fstar
    if ppc:
        out["ppc"] = dict(checks, ppp=float(ppc_s.ppp))
        if ppc_pairs:
            out["ppc"]["pair_bytes"] = int(ppc_s.pair_bytes)
    if loo:
        for k in ("elpd_loo", "p_loo", "looic", "se_elpd_loo", "k_threshold"):
            loo_out[k] = float(getattr(loo_s, k))
        for k in ("n_obs", "n_k_high", "tail_len", "tail_bytes"):
            loo_out[k] = int(getattr(loo_s, k))
        out["loo"] = loo_out
    if diag is not None:
        out["diagnostics"] = dict(diag, diag_bytes=int(chains_s.diag_bytes))
    return out


class Sampler:
    """Resident sampler (state stays in HBM between calls): bench `value`, step-level parity tests."""

    def __init__(self, y, theta_init, beta_prior_means=None, beta_prior_sds=None, beta_proposal_sds=None, **opt_kw):
        L = _lib.load()
        y = np.asfortranarray(np.asarray(y, dtype=np.float64))
        self.n, self.m = y.shape
        n, m = self.n, self.m
        pm = _F(np.zeros((2, m)) if beta_prior_means is None else beta_prior_means, (2, m))
        psd = _F(np.full((2, m), 3.0) if beta_prior_sds is None else beta_prior_sds, (2, m))
        pstep = _F(np.full((2, m), 0.1) if beta_proposal_sds is None else beta_proposal_sds, (2, m))
        th = np.ascontiguousarray(theta_init, dtype=np.float64)
        self._opts = make_opts(**opt_kw)
        self.h = C.c_void_p()
        _lib.check(L.gpirt_b200_sampler_create(C.byref(self.h), _lib.ptr(y), n, m, _lib.ptr(th), _lib.ptr(pm),
                                               _lib.ptr(psd), _lib.ptr(pstep), C.byref(self._opts)))

    def init_draws(self):
        _lib.check(_lib.load().gpirt_b200_sampler_init_draws(self.h))

    def sweep(self, n_sweeps=1, accumulate_irf=False):
        ms = C.c_float(0)
        _lib.check(_lib.load().gpirt_b200_sampler_sweep(self.h, n_sweeps, int(accumulate_irf), C.byref(ms)))
        return ms.value

    def step(self, step, sweep):
        _lib.check(_lib.load().gpirt_b200_sampler_step(self.h, step, sweep))

    def _shape(self, field):
        n, m, N = self.n, self.m, N_GRID
        return {_lib.THETA: (n,), _lib.BETA: (2, m), _lib.F: (n, m), _lib.FSTAR: (N, m), _lib.CHOL: (n, n),
                _lib.LOGP: (n, N), _lib.NU: (n, m), _lib.FSTAR_S: (N,), _lib.FSTAR_MEAN: (N, m), _lib.IRF_SUM: (N, m),
                _lib.THETA_IDX: (n,), _lib.ESS_NPROP: (m,)}[field]

    def get(self, field):
        out = np.empty(self._shape(field), order="F")
        _lib.check(_lib.load().gpirt_b200_sampler_get(self.h, field, _lib.ptr(out)))
        return out

    def set(self, field, value):
        v = _F(value, self._shape(field))
        _lib.check(_lib.load().gpirt_b200_sampler_set(self.h, field, _lib.ptr(v)))

    def set_timing(self, on):
        _lib.check(_lib.load().gpirt_b200_sampler_set_timing(self.h, int(on)))

    def set_pipeline(self, on):
        _lib.check(_lib.load().gpirt_b200_sampler_set_pipeline(self.h, int(on)))

    def time_factorisation(self, reps=10, as_graph=False):
        """ms per K(theta) build + Cholesky alone on the GPU, eager or replayed as a CUDA graph"""
        ms = C.c_float(0)
        _lib.check(_lib.load().gpirt_b200_sampler_time_factorisation(self.h, int(reps), int(as_graph), C.byref(ms)))
        return ms.value

    def timings(self, reset=False):
        ms = np.zeros(len(_lib.TIMER_NAMES))
        calls = np.zeros(len(_lib.TIMER_NAMES), dtype=np.int64)
        _lib.check(_lib.load().gpirt_b200_sampler_timings(self.h, _lib.ptr(ms), calls.ctypes.data_as(C.POINTER(C.c_int64)), int(reset)))
        return {k: (float(a), int(b)) for k, a, b in zip(_lib.TIMER_NAMES, ms, calls)}

    def launches(self):
        return int(_lib.load().gpirt_b200_sampler_launches(self.h))

    def uses(self, feature):
        """1 if this sampler runs feature 0 (int8 theta contraction) / 1 (fixed-point tensor-core products)"""
        return int(_lib.load().gpirt_b200_sampler_uses(self.h, int(feature)))

    def close(self):
        if self.h:
            _lib.load().gpirt_b200_sampler_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---- single operations (each replaces one reference function) ----
def se_cov(x1, x2, jitter=0.0):
    """K(x1, x2) — src/covariance-function.cpp:3-14"""
    x1 = np.ascontiguousarray(x1, dtype=np.float64); x2 = np.ascontiguousarray(x2, dtype=np.float64)
    out = np.empty((x1.size, x2.size), order="F")
    _lib.check(_lib.load().gpirt_b200_se_cov(_lib.ptr(x1), x1.size, _lib.ptr(x2), x2.size, jitter, _lib.ptr(out)))
    return out


def chol_lower(S):
    """arma::chol(S, "lower") — src/gpirtMCMC.cpp:17"""
    S = np.array(S, dtype=np.float64, order="F", copy=True)
    _lib.check(_lib.load().gpirt_b200_chol_lower(_lib.ptr(S), S.shape[0]))
    return S


def dgemm(A, B, C_=None, alpha=1.0, beta=0.0, ta=False, tb=False, tri=0):
    A = _F(A); B = _F(B)
    M = A.shape[1] if ta else A.shape[0]
    K = A.shape[0] if ta else A.shape[1]
    N = B.shape[0] if tb else B.shape[1]
    Cm = np.zeros((M, N), order="F") if C_ is None else np.array(C_, dtype=np.float64, order="F", copy=True)
    _lib.check(_lib.load().gpirt_b200_dgemm(int(ta), int(tb), M, N, K, alpha, _lib.ptr(A), max(1, A.shape[0]), _lib.ptr(B),
                                            max(1, B.shape[0]), beta, _lib.ptr(Cm), max(1, M), tri))
    return Cm


def dgemm_i8(A, B, ta=False, a_lower=0, reps=0):
    """op(A) @ B in 56-bit fixed point on the int8 tensor cores (the sampler's L·Z / f* product kernel).
    a_lower: 1 = A lower triangular (ta False), 2 = A^T upper triangular (ta True).  reps > 0: also returns
    (kernel ms, slicing ms)"""
    A = _F(A); B = _F(B)
    M = A.shape[1] if ta else A.shape[0]
    K = A.shape[0] if ta else A.shape[1]
    N = B.shape[1]
    Cm = np.zeros((M, N), order="F")
    ms = np.zeros(2)
    _lib.check(_lib.load().gpirt_b200_dgemm_i8(int(ta), int(a_lower), M, N, K, _lib.ptr(A), max(1, A.shape[0]), _lib.ptr(B),
                                               max(1, B.shape[0]), _lib.ptr(Cm), max(1, M), int(reps), _lib.ptr(ms)))
    return (Cm, ms) if reps > 0 else Cm


def trsm_lower(L, B, trans=False):
    """solve(trimatl(L), B) / solve(trimatu(L.t()), B) — src/draw-fstar.cpp:7,19"""
    L = _F(L); B = np.array(B, dtype=np.float64, order="F", copy=True)
    if B.ndim == 1:
        B = B.reshape(-1, 1, order="F")
    _lib.check(_lib.load().gpirt_b200_trsm_lower(int(trans), L.shape[0], B.shape[1], _lib.ptr(L), _lib.ptr(B)))
    return B


def ll_bar(f, y, mu):
    """ll_bar for every column — src/log-likelihood.cpp:25-37"""
    f = _F(f); y = _F(y); mu = _F(mu)
    if f.ndim == 1:
        f = f.reshape(-1, 1, order="F"); y = y.reshape(-1, 1, order="F"); mu = mu.reshape(-1, 1, order="F")
    out = np.empty(f.shape[1])
    _lib.check(_lib.load().gpirt_b200_ll_bar(_lib.ptr(f), _lib.ptr(y), _lib.ptr(mu), f.shape[0], f.shape[1], _lib.ptr(out)))
    return out


def fp64_peak_tflops():
    a = C.c_double(0); b = C.c_double(0)
    _lib.check(_lib.load().gpirt_b200_fp64_peak_tflops(C.byref(a), C.byref(b)))
    return a.value, b.value


def response_matrix_native(codes, yea=(1, 2, 3), nay=(4, 5, 6), missing=(0, 7, 8, 9)):
    """Numeric response codes -> (y n x m_kept in {+1,-1,NaN}, kept column indices, number of uncoded cells), coded and
    filtered on the device (the numeric case of R/response_matrix.R:79-98; NaN in `codes` is NA)."""
    codes = _F(codes)
    n, m = codes.shape
    lists = [np.ascontiguousarray(v, dtype=np.float64) for v in (yea, nay, missing)]
    y = np.empty((n, m), order="F")
    kept = np.zeros(m, dtype=np.int64)
    mk, unc = C.c_int64(0), C.c_int64(0)
    _lib.check(_lib.load().gpirt_b200_response_matrix(
        _lib.ptr(codes), n, m, _lib.ptr(lists[0]), lists[0].size, _lib.ptr(lists[1]), lists[1].size, _lib.ptr(lists[2]), lists[2].size,
        _lib.ptr(y), kept.ctypes.data_as(C.POINTER(C.c_int64)), C.byref(mk), C.byref(unc)))
    return np.asfortranarray(y[:, :mk.value]), kept[:mk.value].copy(), unc.value


def theta_diagnostics(theta_chains):
    """theta_chains: list of (draws, n) arrays (one per chain, initial row removed) -> (split-R-hat, ESS) per respondent"""
    chains = [np.asfortranarray(np.asarray(c, dtype=np.float64)) for c in theta_chains]
    draws, n = chains[0].shape
    buf = np.concatenate([c.ravel(order="F") for c in chains])
    rhat = np.empty(n); ess = np.empty(n)
    _lib.check(_lib.load().gpirt_b200_theta_diagnostics(_lib.ptr(buf), draws, n, len(chains), _lib.ptr(rhat), _lib.ptr(ess)))
    return rhat, ess


def int8_peak_tops(random_operands=False):
    """measured tcgen05.mma.kind::i8 issue-rate peak of the device, 10^12 int8 operations per second (random_operands:
    with pseudo-random digit planes instead of near-constant ones — lower, the SM clock drops under the switching power)"""
    a = C.c_double(0)
    L = _lib.load()
    _lib.check((L.gpirt_b200_int8_peak_tops_random if random_operands else L.gpirt_b200_int8_peak_tops)(C.byref(a)))
    return a.value


def predictive_accumulate_time(n, m, reps=100):
    """(ms per launch of the posterior predictive accumulation over an n x m state, ms per device-to-device copy of its
    accumulator planes), CUDA events in one run"""
    a = C.c_double(0); b = C.c_double(0)
    _lib.check(_lib.load().gpirt_b200_predictive_accumulate_time(int(n), int(m), int(reps), C.byref(a), C.byref(b)))
    return a.value, b.value


def irf_bands(draws, band, reps=0):
    """The IRF band ends of gpirtMCMC(irf_band=band) in f* space, computed on the device by the same update and finish
    kernels: draws is cols x S (one column per draw, e.g. out["fstar"][:, :, 1:].reshape(-1, S, order="F")); returns
    (Q(q_lo), Q(q_hi)), each of length cols, and with reps > 0 also (ms per update launch, ms per finish) over reps passes"""
    d = _F(draws)
    if d.ndim != 2:
        raise ValueError("draws must be a cols x S matrix")
    cols, S = d.shape
    lo = np.empty(cols); hi = np.empty(cols); ms = np.zeros(2)
    _lib.check(_lib.load().gpirt_b200_irf_bands(_lib.ptr(d), cols, S, float(band), _lib.ptr(lo), _lib.ptr(hi), int(reps),
                                                _lib.ptr(ms)))
    return (lo, hi, (float(ms[0]), float(ms[1]))) if reps > 0 else (lo, hi)


def ppc_pairs(y, y_reps, reps=0):
    """The odds-ratio check of gpirtMCMC(ppc=True, ppc_pairs=True) on given data, through the same device kernels: y is
    n x m in {+1, -1, NaN}, y_reps n x m x R replicates (+1 / -1 where y is observed, read there only).  Returns
    (log_or, exceed): the observed pairwise log odds ratios and the number of replicates whose odds ratio is at least the
    observed one (m x m each, NaN on the diagonal and for pairs nobody answered both of); with reps > 0 also
    (ms per per-draw launch, ms per observed pass), CUDA events over reps repetitions"""
    y = _F(y)
    if y.ndim != 2:
        raise ValueError("y must be an n x m matrix")
    n, m = y.shape
    r = np.asarray(y_reps, dtype=np.float64)
    if r.ndim == 2:
        r = r[:, :, None]
    if r.ndim != 3 or r.shape[:2] != (n, m):
        raise ValueError("y_reps must be n x m x R with n x m = %r, got %r" % ((n, m), r.shape))
    r = np.asfortranarray(r)
    R = r.shape[2]
    log_or = np.empty((m, m), order="F"); exceed = np.empty((m, m), order="F"); ms = np.zeros(2)
    _lib.check(_lib.load().gpirt_b200_ppc_pairs(_lib.ptr(y), _lib.ptr(r) if R else None, n, m, R, _lib.ptr(log_or),
                                                _lib.ptr(exceed), int(reps), _lib.ptr(ms)))
    return (log_or, exceed, (float(ms[0]), float(ms[1]))) if reps > 0 else (log_or, exceed)


def psis_loo(loglik, reps=0):
    """PSIS-LOO of gpirtMCMC(loo=True) on given log-likelihood draws, through the same device update and finish: loglik is
    cols x S (row = left-out unit, column = draw; sigma = exp(loglik)), for example per-respondent sums of the per-cell
    log-likelihoods for leave-one-respondent-out.  Returns (elpd_loo, p_loo, pareto_k), each of length cols, and with
    reps > 0 also (ms per update launch, ms per finish) over reps passes, CUDA events"""
    ll = _F(loglik)
    if ll.ndim != 2:
        raise ValueError("loglik must be a cols x S matrix")
    cols, S = ll.shape
    elpd = np.empty(cols); p = np.empty(cols); k = np.empty(cols); ms = np.zeros(2)
    _lib.check(_lib.load().gpirt_b200_psis_loo(_lib.ptr(ll) if S else None, cols, S, _lib.ptr(elpd), _lib.ptr(p),
                                               _lib.ptr(k), int(reps), _lib.ptr(ms)))
    return (elpd, p, k, (float(ms[0]), float(ms[1]))) if reps > 0 else (elpd, p, k)


def rng_probe(seed, sweep, purpose, stream, idx0, count):
    u = np.empty(count); z = np.empty(count)
    _lib.check(_lib.load().gpirt_b200_rng_probe(seed, sweep, purpose, stream, idx0, count, _lib.ptr(u), _lib.ptr(z)))
    return u, z
