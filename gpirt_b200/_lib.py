"""ctypes loader for libgpirt_b200.so (the C-ABI CUDA library declared in include/gpirt_b200.h).

There is no CPU fallback: if the library is missing the import of anything that computes fails loudly; if it loads but
no CUDA device is usable every entry point returns GPIRT_B200_ERR_CUDA, surfaced here as GpirtError."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GPIRT_B200_LIB") or os.path.join(HERE, "libgpirt_b200.so")   # override: development A/B builds
N_GRID = 1001

# every symbol include/gpirt_b200.h declares (tests check the .so exports exactly these)
EXPORTS = [
    "gpirt_b200_mcmc", "gpirt_b200_strerror", "gpirt_b200_last_error", "gpirt_b200_last_degenerate_theta", "gpirt_b200_device_count",
    "gpirt_b200_release_memory",
    "gpirt_b200_nccl_unique_id", "gpirt_b200_sampler_create", "gpirt_b200_sampler_init_draws",
    "gpirt_b200_sampler_sweep", "gpirt_b200_sampler_step", "gpirt_b200_sampler_get", "gpirt_b200_sampler_set",
    "gpirt_b200_sampler_timings", "gpirt_b200_sampler_set_timing", "gpirt_b200_sampler_set_pipeline", "gpirt_b200_sampler_time_factorisation",
    "gpirt_b200_sampler_launches", "gpirt_b200_sampler_uses",
    "gpirt_b200_sampler_destroy", "gpirt_b200_se_cov", "gpirt_b200_chol_lower", "gpirt_b200_dgemm", "gpirt_b200_dgemm_i8",
    "gpirt_b200_trsm_lower", "gpirt_b200_ll_bar", "gpirt_b200_fp64_peak_tflops", "gpirt_b200_int8_peak_tops", "gpirt_b200_int8_peak_tops_random", "gpirt_b200_rng_probe", "gpirt_b200_response_matrix", "gpirt_b200_theta_diagnostics",
    "gpirt_b200_predictive_accumulate_time", "gpirt_b200_irf_bands", "gpirt_b200_ppc_pairs",
]

# enums of include/gpirt_b200.h
OK, ERR_ARG, ERR_CUDA, ERR_NOT_PD, ERR_INTERRUPT, ERR_Y_VALUE, ERR_ESS, ERR_NCCL, ERR_NOMEM = 0, -1, -2, -3, -4, -5, -6, -7, -8
(THETA, BETA, F, FSTAR, CHOL, LOGP, NU, FSTAR_S, FSTAR_MEAN, IRF_SUM, THETA_IDX, ESS_NPROP) = range(12)
STEP_DRAW_F, STEP_DRAW_FSTAR, STEP_DRAW_THETA, STEP_DRAW_BETA, STEP_REBUILD = 1, 2, 3, 4, 5
TIMER_NAMES = ["fill_z", "lz_gemm", "ess", "kstar", "trsm", "fstar_gemm", "fstar_draw", "theta_prep", "theta_gemm",
               "allreduce", "theta_draw", "beta", "kbuild", "chol", "trtri"]


class GpirtError(RuntimeError):
    def __init__(self, status, message):
        super().__init__("gpirt_b200: %s (status %d)" % (message, status))
        self.status = status


class Fit(C.Structure):
    """gpirt_b200_fit: posterior predictive summaries accumulated on the device (include/gpirt_b200.h)"""
    _fields_ = [("y_holdout", C.POINTER(C.c_double)), ("pred", C.POINTER(C.c_double)), ("lpd_cell", C.POINTER(C.c_double)),
                ("pwaic_cell", C.POINTER(C.c_double)), ("elpd_item", C.POINTER(C.c_double)),
                ("elpd_resp", C.POINTER(C.c_double)), ("lppd", C.c_double), ("p_waic", C.c_double),
                ("elpd_waic", C.c_double), ("waic", C.c_double), ("se_elpd_waic", C.c_double), ("lpd_holdout", C.c_double),
                ("n_obs", C.c_int64), ("n_holdout", C.c_int64)]


class Irf(C.Structure):
    """gpirt_b200_irf: posterior mean, sd, pointwise credible bands and draws of the IRFs on the grid (include/gpirt_b200.h)"""
    _fields_ = [("band", C.c_double), ("prob_mean", C.POINTER(C.c_double)), ("prob_sd", C.POINTER(C.c_double)),
                ("lower", C.POINTER(C.c_double)), ("upper", C.POINTER(C.c_double)),
                ("fstar_draws", C.POINTER(C.c_double)), ("band_bytes", C.c_int64)]


class Chains(C.Structure):
    """gpirt_b200_chains: several chains in one call and their convergence diagnostics (include/gpirt_b200.h)"""
    _fields_ = [("chains", C.c_int32), ("reserved0", C.c_int32), ("seeds", C.POINTER(C.c_uint64)),
                ("theta_rhat", C.POINTER(C.c_double)), ("theta_ess", C.POINTER(C.c_double)),
                ("beta_rhat", C.POINTER(C.c_double)), ("beta_ess", C.POINTER(C.c_double)),
                ("irf_rhat", C.POINTER(C.c_double)), ("diag_bytes", C.c_int64)]


class Ppc(C.Structure):
    """gpirt_b200_ppc: posterior predictive checks of item, person and pair fit (include/gpirt_b200.h)"""
    _fields_ = [("item_ppp", C.POINTER(C.c_double)), ("resp_ppp", C.POINTER(C.c_double)), ("pair_ppp", C.POINTER(C.c_double)),
                ("pair_log_or", C.POINTER(C.c_double)), ("ppp", C.c_double), ("pair_bytes", C.c_int64)]


class Opts(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("device", C.c_int32), ("fstar_mode", C.c_int32), ("skip_f_draws", C.c_int32),
                ("use_graph", C.c_int32), ("rank", C.c_int32), ("world_size", C.c_int32), ("m_global", C.c_int64),
                ("item_offset", C.c_int64), ("nccl_unique_id", C.c_void_p), ("thin", C.c_int32), ("reserved0", C.c_int32),
                ("f_mean_out", C.POINTER(C.c_double)), ("f_sd_out", C.POINTER(C.c_double)), ("fit", C.POINTER(Fit)),
                ("irf", C.POINTER(Irf)), ("chains", C.POINTER(Chains)), ("ppc", C.POINTER(Ppc))]


PROGRESS_CB = C.CFUNCTYPE(C.c_int, C.c_double, C.c_void_p)
_dp = C.POINTER(C.c_double)
_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        try:   # a source-only checkout: compile the CUDA library now (nvcc cross-compiles, no GPU needed)
            from .build import build
            build()
        except Exception as ex:
            raise ImportError("gpirt_b200: %s is missing and could not be built (%s) — run `python -m gpirt_b200.build` "
                              "(there is no CPU fallback)" % (LIB_PATH, ex))
    L = C.CDLL(LIB_PATH)
    L.gpirt_b200_strerror.restype = C.c_char_p
    L.gpirt_b200_last_error.restype = C.c_char_p
    L.gpirt_b200_last_degenerate_theta.restype = C.c_int64
    L.gpirt_b200_mcmc.argtypes = [_dp, C.c_int64, C.c_int64, _dp, C.c_int, C.c_int, _dp, _dp, _dp, C.POINTER(Opts), _dp,
                                  _dp, _dp, _dp, PROGRESS_CB, C.c_void_p]
    L.gpirt_b200_nccl_unique_id.argtypes = [C.c_void_p]
    L.gpirt_b200_sampler_create.argtypes = [C.POINTER(C.c_void_p), _dp, C.c_int64, C.c_int64, _dp, _dp, _dp, _dp, C.POINTER(Opts)]
    L.gpirt_b200_sampler_init_draws.argtypes = [C.c_void_p]
    L.gpirt_b200_sampler_sweep.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_float)]
    L.gpirt_b200_sampler_step.argtypes = [C.c_void_p, C.c_int, C.c_uint32]
    L.gpirt_b200_sampler_get.argtypes = [C.c_void_p, C.c_int, _dp]
    L.gpirt_b200_sampler_set.argtypes = [C.c_void_p, C.c_int, _dp]
    L.gpirt_b200_sampler_timings.argtypes = [C.c_void_p, _dp, C.POINTER(C.c_int64), C.c_int]
    L.gpirt_b200_sampler_set_timing.argtypes = [C.c_void_p, C.c_int]
    L.gpirt_b200_sampler_set_pipeline.argtypes = [C.c_void_p, C.c_int]
    L.gpirt_b200_sampler_time_factorisation.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_float)]
    L.gpirt_b200_sampler_launches.argtypes = [C.c_void_p]
    L.gpirt_b200_sampler_launches.restype = C.c_int64
    L.gpirt_b200_sampler_uses.argtypes = [C.c_void_p, C.c_int]
    L.gpirt_b200_sampler_destroy.argtypes = [C.c_void_p]
    L.gpirt_b200_sampler_destroy.restype = None
    L.gpirt_b200_se_cov.argtypes = [_dp, C.c_int64, _dp, C.c_int64, C.c_double, _dp]
    L.gpirt_b200_chol_lower.argtypes = [_dp, C.c_int64]
    L.gpirt_b200_dgemm.argtypes = [C.c_int, C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_double, _dp, C.c_int64, _dp,
                                   C.c_int64, C.c_double, _dp, C.c_int64, C.c_int]
    L.gpirt_b200_dgemm_i8.argtypes = [C.c_int, C.c_int, C.c_int64, C.c_int64, C.c_int64, _dp, C.c_int64, _dp, C.c_int64, _dp,
                                      C.c_int64, C.c_int, _dp]
    L.gpirt_b200_trsm_lower.argtypes = [C.c_int, C.c_int64, C.c_int64, _dp, _dp]
    L.gpirt_b200_ll_bar.argtypes = [_dp, _dp, _dp, C.c_int64, C.c_int64, _dp]
    L.gpirt_b200_fp64_peak_tflops.argtypes = [_dp, _dp]
    L.gpirt_b200_int8_peak_tops.argtypes = [_dp]
    L.gpirt_b200_int8_peak_tops_random.argtypes = [_dp]
    _ip64 = C.POINTER(C.c_int64)
    L.gpirt_b200_response_matrix.argtypes = [_dp, C.c_int64, C.c_int64, _dp, C.c_int, _dp, C.c_int, _dp, C.c_int, _dp, _ip64, _ip64, _ip64]
    L.gpirt_b200_theta_diagnostics.argtypes = [_dp, C.c_int64, C.c_int64, C.c_int, _dp, _dp]
    L.gpirt_b200_predictive_accumulate_time.argtypes = [C.c_int64, C.c_int64, C.c_int, _dp, _dp]
    L.gpirt_b200_irf_bands.argtypes = [_dp, C.c_int64, C.c_int64, C.c_double, _dp, _dp, C.c_int, _dp]
    L.gpirt_b200_ppc_pairs.argtypes = [_dp, _dp, C.c_int64, C.c_int64, C.c_int, _dp, _dp, C.c_int, _dp]
    L.gpirt_b200_rng_probe.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, _dp, _dp]
    _lib = L
    return L


def check(status):
    if status != OK:
        L = load()
        detail = L.gpirt_b200_last_error().decode() or L.gpirt_b200_strerror(status).decode()
        raise GpirtError(status, detail)


def ptr(a):
    return a.ctypes.data_as(_dp) if a is not None else None
