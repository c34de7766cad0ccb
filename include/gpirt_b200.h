/* gpirt_b200 — C ABI of the B200-native GP-IRT Gibbs sampler.
 *
 * This is the drop-in boundary for the one hot path of duckmayr/gpirt: the native sampler behind
 *   .Call(`_gpirt_gpirtMCMC`, y, theta, sample_iterations, burn_iterations, beta_prior_means, beta_prior_sds,
 *         beta_step_sizes)                       (reference R/RcppExports.R:4-6, src/RcppExports.cpp:16-30)
 * i.e. Rcpp::List gpirtMCMC(...)                  (reference src/gpirtMCMC.cpp:5-117).
 * Plain pointers and sizes only; all matrices are column-major FP64 exactly as R / Armadillo hand them over.
 * The R-facing shim (gpirt_b200/csrc/rshim/gpirt_rshim.c) and the Python host mirror (gpirt_b200/) both call
 * gpirt_b200_mcmc(); tests and bench additionally use the resident-sampler entry points below.
 * There is no CPU fallback: every entry point returns GPIRT_B200_ERR_CUDA when no CUDA device can be used.
 */
#ifndef GPIRT_B200_H
#define GPIRT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GPIRT_B200_N_GRID 1001 /* theta* = -5.00, -4.99, ..., 5.00  (src/gpirtMCMC.cpp:35) */

enum gpirt_b200_status {
    GPIRT_B200_OK = 0,
    GPIRT_B200_ERR_ARG = -1,      /* bad argument */
    GPIRT_B200_ERR_CUDA = -2,     /* CUDA runtime error / no device (see gpirt_b200_last_error) */
    GPIRT_B200_ERR_NOT_PD = -3,   /* chol(): decomposition failed (src/gpirtMCMC.cpp:17,78,97 -> R error) */
    GPIRT_B200_ERR_INTERRUPT = -4,/* progress callback asked to stop (Rcpp::checkUserInterrupt, gpirtMCMC.cpp:66,85) */
    GPIRT_B200_ERR_Y_VALUE = -5,  /* y holds something other than +1, -1, NA(NaN) (R/response_matrix.R:108-114) */
    GPIRT_B200_ERR_ESS = -6,      /* elliptical slice sampler did not terminate (NaN likelihood) */
    GPIRT_B200_ERR_NCCL = -7,     /* NCCL not loadable / collective failed */
    GPIRT_B200_ERR_NOMEM = -8
};

/* Posterior predictive summaries accumulated on the device over all S sampling iterations (burn-in excluded, thin has no
 * effect), each iteration's end-of-sweep state (f, theta, beta).  Per cell g = f_ij + beta0_j + beta1_j theta_i; the
 * scoring orientation yt_ij is y_ij where observed, y_holdout_ij where y is NA and y_holdout gives +1 / -1, else +1.
 * Zero-initialise, set the pointers you want; the library fills the scalars.  With items sharded, per-cell and per-item
 * outputs cover the local item block, elpd_resp and every scalar are global (all-reduced); every rank must set fit.
 * S = 0: every output is NaN.  S = 1: pwaic_cell, p_waic, elpd_*, waic and se_elpd_waic are NaN. */
typedef struct gpirt_b200_fit {
    const double* y_holdout; /* optional n x m {+1, -1, NaN}: held-out responses, read only where y is NA
                                (any other value: GPIRT_B200_ERR_Y_VALUE) */
    double* pred;         /* optional n x m: mean_s sigma(g), the posterior predictive P(y_ij = +1), every cell */
    double* lpd_cell;     /* optional n x m: log(mean_s sigma(yt g)) on observed and held-out cells, NaN elsewhere */
    double* pwaic_cell;   /* optional n x m: sample variance (denominator S - 1) over s of log sigma(yt g), observed cells
                             only, NaN elsewhere */
    double* elpd_item;    /* optional m: sum of lpd_cell - pwaic_cell over the observed cells of the item */
    double* elpd_resp;    /* optional n: the same sum over the observed cells of the respondent */
    double lppd;          /* out: sum of lpd_cell over the observed cells */
    double p_waic;        /* out: sum of pwaic_cell over the observed cells */
    double elpd_waic;     /* out: lppd - p_waic */
    double waic;          /* out: -2 elpd_waic */
    double se_elpd_waic;  /* out: sqrt(n_obs var(lpd_cell - pwaic_cell)) over the observed cells (sample variance) */
    double lpd_holdout;   /* out: sum of lpd_cell over the held-out cells */
    int64_t n_obs;        /* out: number of observed cells */
    int64_t n_holdout;    /* out: number of held-out cells */
} gpirt_b200_fit;

/* Posterior summaries of the item response functions on the grid theta* (1001 points), accumulated on the device.
 * S = sample_iterations.  For grid point k and local item j, x_s is the f*_kj that sampling iteration s (s = 1..S) draws
 * (the value the IRF sum accumulates) and P_s = 1 / (1 + exp(-x_s)), as in irf_out.
 *   prob_mean = mean_s P_s, prob_sd = sd_s P_s (denominator S - 1): FP64 Welford over ALL S iterations (thin has no effect).
 *   Bands at level b (0 < b < 1): q_lo = (1 - b) / 2, q_hi = (1 + b) / 2 (FP64, on the host); for each q
 *     h = (S - 1) q, r = floor(h), t = h - r,
 *     Q = x_(r) + t (x_(r+1) - x_(r))  (0-based ascending order statistics of x_1..x_S: R's type 7, numpy's "linear";
 *         computed as __dadd_rn(x_(r), __dmul_rn(t, __dsub_rn(x_(r+1), x_(r)))), no contraction), Q = x_(S-1) if r = S - 1;
 *     lower = plogis(Q(q_lo)), upper = plogis(Q(q_hi)): the band is taken in f* space and mapped to P.
 *   The order statistics are exact: per grid cell the device keeps the K_lo = r_lo + 2 smallest and the K_hi = S - r_hi
 *   largest f* seen (two heaps, 8 (K_lo + K_hi) bytes per cell, reported in band_bytes) instead of every draw.
 *   fstar_draws: 1001 x m x (1 + S / thin), slot 0 = the initial f*, slot k = f* after sampling iteration k * thin.
 *   S = 0: prob_mean, prob_sd, lower, upper are NaN.  S = 1: prob_sd is NaN, lower = upper = prob_mean = P_1.
 * Zero-initialise and set the pointers you want (each 1001 x m over the local items; with items sharded each rank's
 * outputs cover its own item block and no collective is involved).  lower / upper need 0 < band < 1 (else
 * GPIRT_B200_ERR_ARG); a run whose tail buffers do not fit in free device memory is refused with GPIRT_B200_ERR_NOMEM
 * before its first sweep.  The buffers are allocated for the call and returned to the device when it ends. */
typedef struct gpirt_b200_irf {
    double band;          /* level b of the pointwise credible band (lower / upper only) */
    double* prob_mean;    /* optional 1001 x m */
    double* prob_sd;      /* optional 1001 x m */
    double* lower;        /* optional 1001 x m */
    double* upper;        /* optional 1001 x m */
    double* fstar_draws;  /* optional 1001 x m x (1 + S / thin) */
    int64_t band_bytes;   /* out: device bytes of the tail buffers, 8 * 1001 * m * (K_lo + K_hi) (0 without bands) */
} gpirt_b200_irf;

/* Several chains in one gpirt_b200_mcmc call, run concurrently on one device (one host thread enqueues them round-robin),
 * with convergence diagnostics computed on the device.  With opts.chains set, C = chains and every array takes a trailing
 * chain dimension; chain c's block is exactly what a call without opts.chains, with seed seeds[c] (NULL: opts.seed + c)
 * and theta_init[:, c], writes:
 *   theta_init n x C,  theta_out slots x n x C,  beta_out 2 x m x slots x C,  f_out n x m x slots x C (or NULL with
 *   skip_f_draws),  irf_out 1001 x m x C.
 * thin, skip_f_draws, use_graph, device and fstar_mode apply to every chain.  Not built (GPIRT_B200_ERR_ARG): world_size
 * > 1, opts.fit, opts.irf, f_mean_out or f_sd_out set, chains outside [1, 32].
 * Diagnostics use all S sampling iterations whatever thin is, with the formulas of gpirt_b200_theta_diagnostics:
 *   half = floor(S / 2); each chain contributes its first and its last `half` iterations (the middle one of an odd S is
 *   dropped).  split-R-hat = sqrt(var+ / W) over the 2C half-chains, NaN when W = 0.  ESS: per chain, autocovariances with
 *   denominator S and Geyer's initial monotone sequence over lag pairs (NaN for a constant chain), summed over chains.
 *   irf_rhat is the split-R-hat of P = plogis(f*) per grid cell.  S < 4: every diagnostic output is NaN.
 * Before the first sweep the call checks that C - 1 more samplers of chain 0's footprint and the diagnostics buffers fit
 * in free device memory (else GPIRT_B200_ERR_NOMEM, the bytes needed in the message).  If any chain fails or the progress
 * callback interrupts, every chain stops and gpirt_b200_last_error names the chain.  The callback is called on the calling
 * thread only, once per iteration of all chains.  gpirt_b200_last_degenerate_theta() returns the sum over chains. */
typedef struct gpirt_b200_chains {
    int32_t chains;          /* C, 1 <= C <= 32 */
    int32_t reserved0;
    const uint64_t* seeds;   /* optional C Philox keys; NULL: chain c uses opts.seed + c */
    double* theta_rhat;      /* optional n        split-R-hat over the 2C half-chains, all S sampling iterations */
    double* theta_ess;       /* optional n        sum over chains of Geyer's initial-monotone ESS per chain */
    double* beta_rhat;       /* optional 2 x m */
    double* beta_ess;        /* optional 2 x m */
    double* irf_rhat;        /* optional 1001 x m split-R-hat of P = plogis(f*) per grid cell */
    int64_t diag_bytes;      /* out: device bytes of the traces (8 S (n + 2m) C with theta / beta diagnostics) and
                                half-chain accumulators (32 x 1001 m C with irf_rhat) */
} gpirt_b200_chains;

/* Posterior predictive model checks, accumulated on the device over all S sampling iterations (burn-in excluded, thin has
 * no effect).  Sampling iteration s (s = 1..S) uses the end-of-sweep state opts.fit uses: g_ij = f_ij + beta0_j +
 * beta1_j theta_i, p_ij = 1 / (1 + exp(-g_ij)).  Only observed cells are replicated (missing cells stay missing):
 *   y^rep_ij = +1 if u_ij < p_ij, else -1,  u_ij = the Philox uniform of purpose 8 (gpirt_b200_rng_probe(seed, B + s, 8,
 *   j, i, 1)), stream = global item index j, idx = respondent i, sweep = B + s (the counter of the sweep that produced
 *   the state; the chain's own draws do not change).
 * Pearson chi-square: the term of an observed cell is (y01 - p)^2 / (p (1 - p)) = exp(-y g) for y in {+1, -1}.
 *   D_j(y; s) sums the terms of the observed cells of item j, D_i(y; s) those of respondent i, D(y; s) all of them, and
 *   D(y^rep; s) the same with y^rep for y.  Observed and replicated sums run in the same fixed order (a replicate equal to
 *   y gives bit-equal sums, which counts as ">=").
 *   item_ppp[j] = (1/S) #{s : D_j(y^rep; s) >= D_j(y; s)}; resp_ppp and ppp likewise.  NaN where the item / respondent has
 *   no observed cell.
 * Pairs of items j != k, over the respondents who answered both: a = n11, b = n10, c = n01, d = n00.
 *   pair_log_or = log(((a + 1/2)(d + 1/2)) / ((b + 1/2)(c + 1/2))) of the observed y (FP64).
 *   pair_ppp = (1/S) #{s : OR(y^rep; s) >= OR(y)}, compared exactly in integers:
 *     (2a_r+1)(2d_r+1)(2b_o+1)(2c_o+1) >= (2a_o+1)(2d_o+1)(2b_r+1)(2c_r+1)   (128-bit products).
 *   Both m x m and symmetric; NaN on the diagonal and for pairs with no jointly observed respondent.
 * S = 0: every output is NaN.  Not built (GPIRT_B200_ERR_ARG): world_size > 1, opts.chains.  The pair state (observed
 * counts and exceedance counters of every pair, about 20 bytes per pair of the upper triangle, plus the replicate plane)
 * is one device allocation for the call, checked against free device memory before the first sweep
 * (GPIRT_B200_ERR_NOMEM, the bytes needed in the message). */
typedef struct gpirt_b200_ppc {
    double* item_ppp;     /* optional m */
    double* resp_ppp;     /* optional n */
    double* pair_ppp;     /* optional m x m, symmetric */
    double* pair_log_or;  /* optional m x m, symmetric: observed log odds ratio */
    double  ppp;          /* out: global PPP of the total chi-square */
    int64_t pair_bytes;   /* out: device bytes of the pair state (0 without pair outputs) */
} gpirt_b200_ppc;

/* Options beyond the reference's seven arguments.  Zero-initialise, then set what you need. */
typedef struct gpirt_b200_opts {
    uint64_t seed;        /* Philox4x32-10 key; the R shim derives it from R's RNG so set.seed() reproduces runs */
    int32_t device;       /* CUDA device ordinal; -1 = leave the current device alone */
    int32_t fstar_mode;   /* 0: mean_j = (S^-1 K*)^T f_j (two n x 1001 triangular solves per sweep);
                             1: literal per-item alpha_j = L^-T L^-1 f_j (draw-fstar.cpp:3-8,24) */
    int32_t skip_f_draws; /* 1: do not store f draws (f_out may be NULL); reference behaviour is 0 */
    int32_t use_graph;    /* 0 (default): with the per-step timers off (always in gpirt_b200_mcmc) every sweep after the first is
                             replayed as ONE CUDA graph launch — for n > 256 the pipelined sweep with its side streams
                             forked and joined inside the graph, NCCL exchanges included; -1: never (every kernel
                             launched individually); draws are bit-identical either way */
    /* item sharding across GPUs (one process per GPU).  world_size <= 1: single GPU, fields ignored. */
    int32_t rank, world_size;
    int64_t m_global;     /* total items over all ranks */
    int64_t item_offset;  /* global index of this rank's first item (y, priors and outputs are the LOCAL block) */
    const void* nccl_unique_id; /* 128-byte ncclUniqueId shared by all ranks (rank 0: gpirt_b200_nccl_unique_id);
                                   NULL on a later call re-uses the communicator the previous call created */
    /* draw storage (src/gpirtMCMC.cpp:49-55,99-103 stores every sampling iteration: n*m*8 bytes of f each) */
    int32_t thin;         /* > 1: keep the draws of every thin-th sampling iteration only; theta_out / beta_out / f_out then
                             hold 1 + sample_iterations / thin slots (slot 0 = initial values, slot k = sampling iteration
                             k * thin).  IRFs still average over ALL sampling iterations.  0 or 1: the reference's contract */
    int32_t reserved0;
    double* f_mean_out;   /* optional n x m: posterior mean of f over all sampling iterations, accumulated on the device */
    double* f_sd_out;     /* optional n x m: posterior standard deviation of f (denominator S - 1, as R's sd()) */
    gpirt_b200_fit* fit;  /* optional: posterior predictive probabilities, WAIC and held-out scores (gpirt_b200_fit);
                             NULL = none.  Costs 25 bytes of device memory per cell for the run */
    gpirt_b200_irf* irf;  /* optional: posterior mean, sd, pointwise credible bands and draws of f* on the grid
                             (gpirt_b200_irf); NULL = none */
    gpirt_b200_chains* chains; /* optional: several chains in this call and their diagnostics (gpirt_b200_chains);
                             NULL = one chain */
    gpirt_b200_ppc* ppc;  /* optional: posterior predictive checks of item, person and pair fit (gpirt_b200_ppc);
                             NULL = none */
} gpirt_b200_opts;

/* Progress / interrupt callback: called once per iteration with percent complete (as the reference's Rprintf,
 * src/gpirtMCMC.cpp:64,83); return non-zero to abort the run with GPIRT_B200_ERR_INTERRUPT. */
typedef int (*gpirt_b200_progress_cb)(double percent_complete, void* ctx);

/* The sampler.  Replaces gpirtMCMC() (src/gpirtMCMC.cpp:5).  HOST pointers, column-major:
 *   y            n x m   values exactly {+1, -1, NaN}          (borrowed, read-only; RcppExports.cpp:20)
 *   theta_init   n                                              (copied; RcppExports.cpp:21)
 *   beta_prior_means / beta_prior_sds / beta_step_sizes  2 x m  (RcppExports.cpp:24-26)
 *   theta_out    (S+1) x n        row 0 = initial values       (gpirtMCMC.cpp:49,53,99)
 *   beta_out     2 x m x (S+1)    slice 0 = initial draw       (gpirtMCMC.cpp:50,54,100)
 *   f_out        n x m x (S+1)    slice 0 = initial draw       (gpirtMCMC.cpp:51,55,101)
 *   irf_out      1001 x m         plogis(mean f*)              (gpirtMCMC.cpp:42,103,106-111)
 * with S = sample_iterations.  Returns 0 or a negative gpirt_b200_status. */
int gpirt_b200_mcmc(const double* y, int64_t n, int64_t m, const double* theta_init, int sample_iterations,
                    int burn_iterations, const double* beta_prior_means, const double* beta_prior_sds,
                    const double* beta_step_sizes, const gpirt_b200_opts* opts, double* theta_out,
                    double* beta_out, double* f_out, double* irf_out, gpirt_b200_progress_cb cb, void* cb_ctx);

const char* gpirt_b200_strerror(int status);
const char* gpirt_b200_last_error(void); /* detail of the last failure on this thread (CUDA / NCCL message) */
/* number of theta draws of the last gpirt_b200_mcmc() call on this thread whose grid CDF was degenerate (all mass on grid
 * point 0 after max-subtraction): the sampler takes grid point 0 there, the reference reads theta_star[1001] out of bounds
 * (src/draw-theta.cpp:28-33).  0 in every healthy run; the R shim turns a non-zero count into a warning. */
int64_t gpirt_b200_last_degenerate_theta(void);
int gpirt_b200_device_count(void);
/* device memory and the NCCL communicator are kept across calls (a second gpirtMCMC() re-uses them); this releases them */
int gpirt_b200_release_memory(void);
int gpirt_b200_nccl_unique_id(void* out128); /* rank 0 creates, the host distributes (any transport) */

/* ---- resident sampler: state lives in HBM between calls (bench "value", step-level parity tests) ---- */
typedef struct gpirt_b200_sampler gpirt_b200_sampler;

enum gpirt_b200_field { /* what gpirt_b200_sampler_get/_set move; shapes column-major, HOST side */
    GPIRT_B200_THETA = 0,   /* n */
    GPIRT_B200_BETA = 1,    /* 2 x m */
    GPIRT_B200_F = 2,       /* n x m */
    GPIRT_B200_FSTAR = 3,   /* 1001 x m */
    GPIRT_B200_CHOL = 4,    /* n x n lower Cholesky factor of K(theta,theta)+1e-3 I, strict upper = 0 */
    GPIRT_B200_LOGP = 5,    /* n x 1001 log-likelihood part of the theta log-posterior (prior not included) */
    GPIRT_B200_NU = 6,      /* n x m  ESS proposals nu = L z of the last draw_f */
    GPIRT_B200_FSTAR_S = 7, /* 1001   predictive "sd" s = 1 - sqrt(colsum(tmp^2)) */
    GPIRT_B200_FSTAR_MEAN = 8, /* 1001 x m predictive means K*^T alpha (without mu*) of the last draw_fstar */
    GPIRT_B200_IRF_SUM = 9, /* 1001 x m running sum of f* over sampling iterations */
    GPIRT_B200_THETA_IDX = 10, /* n grid indices of the last draw_theta (as doubles) */
    GPIRT_B200_ESS_NPROP = 11  /* m number of ESS proposals evaluated per item in the last draw_f (as doubles) */
};

enum gpirt_b200_step { /* one Gibbs sweep = steps 1..6 in this order (src/gpirtMCMC.cpp:68-78) */
    GPIRT_B200_STEP_DRAW_F = 1,     /* draw-f.cpp:64-73 (ESS for every item) */
    GPIRT_B200_STEP_DRAW_FSTAR = 2, /* draw-fstar.cpp:10-31 */
    GPIRT_B200_STEP_DRAW_THETA = 3, /* draw-theta.cpp:3-37 (stabilised CDF) */
    GPIRT_B200_STEP_DRAW_BETA = 4,  /* draw-beta.cpp:3-41 */
    GPIRT_B200_STEP_REBUILD = 5,    /* K(theta,theta)+1e-3 I and its Cholesky, gpirtMCMC.cpp:76-78 (mu, mu* are implicit) */
    GPIRT_B200_STEP_COUNT = 6
};

/* create: uploads y (ingested to int8 {+1,-1,0=NA}), priors, theta_init; builds K + Cholesky. No draws yet. */
int gpirt_b200_sampler_create(gpirt_b200_sampler** out, const double* y, int64_t n, int64_t m,
                              const double* theta_init, const double* beta_prior_means,
                              const double* beta_prior_sds, const double* beta_step_sizes,
                              const gpirt_b200_opts* opts);
/* the reference's initialisation draws: f_j = L z_j, beta ~ prior, f* (gpirtMCMC.cpp:18-41); sweep counter = 0 */
int gpirt_b200_sampler_init_draws(gpirt_b200_sampler* s);
/* run n_sweeps full sweeps; accumulate_irf != 0 adds f* into the IRF sum after each (sampling phase).
 * elapsed_ms (optional): CUDA-event time of the whole batch on the sampler's stream. */
int gpirt_b200_sampler_sweep(gpirt_b200_sampler* s, int n_sweeps, int accumulate_irf, float* elapsed_ms);
/* run one step of the sweep in isolation under sweep counter `sweep` (step-level parity tests) */
int gpirt_b200_sampler_step(gpirt_b200_sampler* s, int step, uint32_t sweep);
int gpirt_b200_sampler_get(gpirt_b200_sampler* s, int field, double* host_out);
int gpirt_b200_sampler_set(gpirt_b200_sampler* s, int field, const double* host_in);
/* per-step CUDA-event timings accumulated since the last reset: ms[GPIRT_B200_TIMER_COUNT], calls[...] */
enum gpirt_b200_timer {
    GPIRT_B200_T_FILL_Z = 0, GPIRT_B200_T_LZ_GEMM = 1, GPIRT_B200_T_ESS = 2, GPIRT_B200_T_KSTAR = 3,
    GPIRT_B200_T_TRSM = 4, GPIRT_B200_T_FSTAR_GEMM = 5, GPIRT_B200_T_FSTAR_DRAW = 6, GPIRT_B200_T_THETA_PREP = 7,
    GPIRT_B200_T_THETA_GEMM = 8, GPIRT_B200_T_ALLREDUCE = 9, GPIRT_B200_T_THETA_DRAW = 10, GPIRT_B200_T_BETA = 11,
    GPIRT_B200_T_KBUILD = 12, GPIRT_B200_T_CHOL = 13, GPIRT_B200_T_TRTRI = 14, GPIRT_B200_TIMER_COUNT = 15
};
int gpirt_b200_sampler_timings(gpirt_b200_sampler* s, double* ms, int64_t* calls, int reset);
int gpirt_b200_sampler_set_timing(gpirt_b200_sampler* s, int enabled); /* per-step events on (default) / off */
/* sweep pipelining on (default) / off: on, the Cholesky chain of a sweep overlaps its beta step and the next sweep's
 * Z fill and L Z product (identical draws either way; off gives un-overlapped per-kernel timings) */
int gpirt_b200_sampler_set_pipeline(gpirt_b200_sampler* s, int enabled);
/* measurement: milliseconds per repetition of K(theta,theta) + 0.001 I and its Cholesky factorisation alone on the GPU
 * (gpirtMCMC.cpp:76-78), as the eager launch sequence (as_graph = 0) or replayed as a CUDA graph of it (as_graph = 1) */
int gpirt_b200_sampler_time_factorisation(gpirt_b200_sampler* s, int reps, int as_graph, float* ms_per_rep);
int64_t gpirt_b200_sampler_launches(gpirt_b200_sampler* s); /* kernels launched by this sampler so far */
/* which code path this sampler selected (bench.py picks the roofline denominator by it, the parity tests assert it):
 * feature 0 = int8 theta contraction (1/0), 1 = fixed-point (int8) L Z / f* / K*-solve products (1/0),
 * 2 / 3 = launch shape of the last ESS / beta step (0 one CTA per item, 1 persistent CTAs, 2 streaming shape for
 * n > 4096; -1 before the first launch), 4 = K*-solve route (0 through L^-1, 1 blocked substitution), 5 = number of
 * sweeps so far that ran as ONE CUDA-graph launch; -1 for an unknown feature */
int gpirt_b200_sampler_uses(gpirt_b200_sampler* s, int feature);
void gpirt_b200_sampler_destroy(gpirt_b200_sampler* s);

/* ---- single operations on HOST buffers (each replaces one reference function; used by the parity tests) ---- */
/* K(x1,x2), src/covariance-function.cpp:3-14; jitter is added where i == j (0 for a plain K) -> out n1 x n2 */
int gpirt_b200_se_cov(const double* x1, int64_t n1, const double* x2, int64_t n2, double jitter, double* out);
/* arma::chol(S,"lower") (src/gpirtMCMC.cpp:17): in place, strict upper zeroed; GPIRT_B200_ERR_NOT_PD if it fails */
int gpirt_b200_chol_lower(double* S, int64_t n);
/* C = alpha op(A) op(B) + beta C on the DMMA GEMM (column-major; ta/tb: 0 = N, 1 = T). tri: 0 none,
 * 1 = A lower-triangular (skip structurally-zero k blocks), 2 = only the lower triangle of C is written */
int gpirt_b200_dgemm(int ta, int tb, int64_t M, int64_t N, int64_t K, double alpha, const double* A, int64_t lda,
                     const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int tri);
/* C = op(A) B in 56-bit fixed point on the int8 tensor cores (tcgen05; the path the sampler uses for L Z and for the f*
 * product): ta = 0: A is M x K, ta = 1: A is K x M; B is K x N; a_lower = 1 (ta = 0 only): op(A) is lower triangular,
 * a_lower = 2 (ta = 1 only): op(A) = A^T is upper triangular and the strict upper triangle of the stored A holds zeros.
 * reps > 0 and ms != NULL: the product is repeated and the mean kernel time (CUDA events) is returned in ms[0],
 * operand slicing in ms[1].  |error| <= K 2^-51 max|A[i,:]| max|B[:,j]| */
int gpirt_b200_dgemm_i8(int ta, int a_lower, int64_t M, int64_t N, int64_t K, const double* A, int64_t lda,
                        const double* B, int64_t ldb, double* C, int64_t ldc, int reps, double* ms);
/* solve L X = B (trans = 0) or L^T X = B (trans = 1) in place, L n x n lower, B n x nrhs (arma::solve(trimatl/u)) */
int gpirt_b200_trsm_lower(int trans, int64_t n, int64_t nrhs, const double* L, double* B);
/* ll_bar for every column: out[j] = -sum_i log(1+exp(-y_ij (f_ij + mu_ij))), src/log-likelihood.cpp:25-37 */
int gpirt_b200_ll_bar(const double* f, const double* y, const double* mu, int64_t n, int64_t m, double* out);
/* FP64 tensor-pipe peak of the current device, TFLOP/s (DMMA.8x8x4 issue-rate microbenchmark; roofline denominator) */
int gpirt_b200_fp64_peak_tflops(double* dmma_tflops, double* dfma_tflops);
/* int8 tensor-pipe peak of the current device in 10^12 operations/s: tcgen05.mma.kind::i8 (M128 N256 K32, operands in
 * shared memory) issued back to back on every SM with no loads (roofline denominator of the int8 kernels) */
int gpirt_b200_int8_peak_tops(double* tops);
/* the same microbenchmark with pseudo-random digits in [-64, 63] as operands: the MMAs issue at the same rate in cycles
 * (tools/umma_i8_shapes.cu), but the switching power pulls the SM clock down, so the sustained operations/s are lower —
 * the practical ceiling of a kernel that multiplies real operand planes */
int gpirt_b200_int8_peak_tops_random(double* tops);
/* measurement: mean milliseconds of one launch of the posterior predictive accumulation (opts.fit) over an n x m state
 * (f, theta, beta standard normal, every cell observed; 57 bytes of HBM traffic per cell), CUDA events over `reps`
 * launches, and of a device-to-device copy of its 3 accumulator planes (24 (n rounded up to 8) m bytes read and as many
 * written) in the same run: the copy rate the accumulation is compared with */
int gpirt_b200_predictive_accumulate_time(int64_t n, int64_t m, int reps, double* ms_accumulate, double* ms_copy);
/* The band computation of gpirt_b200_irf on arbitrary draws (tests, measurement): draws is cols x S, column-major, on the
 * host (for example fstar_draws without slot 0, reshaped to (1001 m) x S).  The draws are uploaded once (8 cols S bytes of
 * device memory), streamed one at a time through the update kernel gpirt_b200_mcmc uses, then finished as there.
 * Returns the f*-space Q(q_lo) in lower and Q(q_hi) in upper (cols each, no plogis).  reps > 0: the whole pass is repeated
 * reps times, timed with CUDA events: ms[0] = mean time of one update launch, ms[1] = mean time of the finish. */
int gpirt_b200_irf_bands(const double* draws, int64_t cols, int64_t S, double band, double* lower, double* upper, int reps,
                         double* ms);
/* The odds-ratio check of gpirt_b200_ppc on caller data (tests, measurement), through the observed-count and per-draw
 * kernels gpirt_b200_mcmc uses: y is n x m {+1, -1, NaN}, y_reps n x m x R replicates read where y is observed (+1 / -1
 * there; any other value, or one in y: GPIRT_B200_ERR_Y_VALUE).  log_or (optional, m x m) = pair_log_or of y;
 * exceed (optional, m x m) = the number of replicates r with OR(y_reps[:, :, r]) >= OR(y), NaN where pair_ppp is NaN.
 * reps > 0: ms[0] = mean CUDA-event time of one per-draw launch, ms[1] = of the observed pass, over reps repetitions. */
int gpirt_b200_ppc_pairs(const double* y, const double* y_reps, int64_t n, int64_t m, int R, double* log_or, double* exceed,
                         int reps, double* ms);
/* ---- the host steps either side of the sampler (SURVEY 8 f4) ---- */
/* Response coding, the producer of y (reference R/response_matrix.R:79-98) for numeric code matrices, on the device:
 * codes n x m (column-major doubles, NaN = NA); yea / nay / missing code lists; cells with a code in none of the lists are
 * treated as missing and counted in n_uncoded (the reference warns about them).  y_out (n x m, the first *m_kept columns
 * are written) receives exactly {+1, -1, NaN}; unanimous items (one distinct non-missing value) are discarded; kept[c]
 * is the original column of output column c. */
int gpirt_b200_response_matrix(const double* codes, int64_t n, int64_t m, const double* yea, int n_yea, const double* nay,
                               int n_nay, const double* missing, int n_missing, double* y_out, int64_t* kept, int64_t* m_kept,
                               int64_t* n_uncoded);
/* Multi-chain diagnostics of theta draws: theta_draws holds `chains` blocks of draws x n (column-major, as the theta
 * output without its first row); per respondent the split-R-hat over the 2 x chains half-chains (rhat, optional) and the
 * summed effective sample size, Geyer's initial monotone sequence estimator per chain (ess, optional). */
int gpirt_b200_theta_diagnostics(const double* theta_draws, int64_t draws, int64_t n, int chains, double* rhat, double* ess);
/* device-side Philox variates by address (tests: must equal the oracle's gpo_keyed_* bit-for-bit / to 1 ulp) */
int gpirt_b200_rng_probe(uint64_t seed, uint32_t sweep, uint32_t purpose, uint32_t stream, uint32_t idx0, int count,
                         double* uniforms, double* normals);

#ifdef __cplusplus
}
#endif
#endif /* GPIRT_B200_H */
