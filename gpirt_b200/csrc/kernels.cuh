// Host-callable launchers for the non-GEMM kernels of the sweep (kernels.cu).
#pragma once
#include "common.cuh"
#include "philox.cuh"

namespace gpirt {

// K(x1,x2)[i,j] = exp(-0.5 (x1_i-x2_j)^2) (+ jitter where i == j); lower_only: entries above the diagonal are
// written as exact zeros (the Cholesky factor's strict upper triangle) and their exp() skipped.
int launch_se_cov(cudaStream_t st, const double* x1, int n1, const double* x2, int n2, double jitter, bool lower_only,
                  double* out, int64_t ld);
// theta*_k = -5 + k*0.01 and log N(theta*_k; 0, 1)
int launch_grid_init(cudaStream_t st, double* theta_star, double* prior);
// y (double, {+1,-1,NaN}) -> int8 {+1,-1,0} and a double copy {+1,-1,0}; counts NaN cells and illegal values
int launch_ingest_y(cudaStream_t st, const double* y, int n, int m, int8_t* y8, int64_t ldy8, double* yd, int64_t ldyd,
                    unsigned long long* n_missing, unsigned long long* n_bad);
// Z[i,j] = standard normal addressed (sweep, purpose, item_offset + j, i)
int launch_fill_normal(cudaStream_t st, double* Z, int n, int m, int64_t ld, RngKey key, uint32_t purpose,
                       uint32_t item_offset);
// the same normals as int8 digit planes (operand of the fixed-point L Z product) with the fixed column scale 2^-2;
// Z_or_null: also store them as doubles
int launch_fill_normal_planes(cudaStream_t st, int8_t* planes, double* scale, int64_t rows_pad, int64_t k_pad, int n, int m,
                              RngKey key, uint32_t purpose, uint32_t item_offset, double* Z_or_null, int64_t ld);
// beta[p,j] = pm + psd * z  (gpirtMCMC.cpp:23-27)
int launch_init_beta(cudaStream_t st, double* beta, const double* pm, const double* psd, int m, RngKey key,
                     uint32_t item_offset);
// launch shape the per-item kernels (ESS, beta) picked: one CTA per item with the item in registers, one persistent CTA
// per SM with prefetch, or the n > 4096 streaming shape (reported through gpirt_b200_sampler_uses for the parity tests)
enum ItemShape : int { ITEM_SHAPE_CTA = 0, ITEM_SHAPE_PERSISTENT = 1, ITEM_SHAPE_STREAM = 2 };
// elliptical slice sampler for all items (draw-f.cpp); f updated in place
int launch_ess(cudaStream_t st, double* f, const double* nu, int64_t ld, const int8_t* y8, int64_t ldy,
               const double* theta, const double* beta, int n, int m, RngKey key, uint32_t item_offset, int* nprop,
               int* status, int* work = nullptr, int* shape = nullptr);   // work: one zeroable int (item counter of the persistent shape)
// s_k = 1 - sqrt(sum_i tmp_ik^2)
int launch_fstar_sd(cudaStream_t st, const double* tmp, int64_t ld, int n, int N, double* s);
// f*_kj = (mean_kj + beta0_j + beta1_j theta*_k) + s_k z_kj, in place over mean; optional IRF accumulation
int launch_fstar_finish(cudaStream_t st, double* fstar, int64_t ld, int N, int m, const double* s, const double* beta,
                        const double* theta_star, RngKey key, uint32_t item_offset, double* irf_sum, int accumulate);
// D_kj = log(2 cosh(f*_kj / 2)); rowsum[k] = sum_j D_kj (two-pass, fixed order)
int launch_theta_prep(cudaStream_t st, const double* fstar, double* D, int64_t ld, int N, int m, double* partial,
                      int n_chunks, double* rowsum);
// inverse-CDF draw on the grid for every respondent (draw-theta.cpp:20-34, max-subtracted)
int launch_theta_draw(cudaStream_t st, const double* logPt, int64_t ld, const double* rowsum_or_null,
                      const double* prior, const double* theta_star, int n, int N, RngKey key, double* theta,
                      int* idx, int* n_degenerate);
// Metropolis step for the two mean coefficients of every item (draw-beta.cpp)
int launch_beta(cudaStream_t st, double* beta, const double* f, int64_t ld, const int8_t* y8, int64_t ldy,
                const double* theta, const double* pm, const double* psd, const double* pstep, int n, int m,
                RngKey key, uint32_t item_offset, int* status, int* work = nullptr, int* shape = nullptr);
// out[j] = ll_bar(f_j, y_j, mu_j) for explicit mu (host-API helper)
int launch_ll_bar(cudaStream_t st, const double* f, const double* y, const double* mu, int n, int m, double* out);
// IRF = plogis(sum / S)
int launch_irf_finish(cudaStream_t st, const double* irf_sum, int64_t ld, int N, int m, double inv_samples, double* out);
// response coding (R/response_matrix.R:79-98, numeric codes) and compaction of the kept items
int launch_response_code(cudaStream_t st, const double* codes, int n, int m, const double* yea, int n_yea, const double* nay,
                         int n_nay, const double* mis, int n_mis, double* y, int* unanimous, unsigned long long* n_uncoded);
int launch_gather_columns(cudaStream_t st, const double* y, int n, const int64_t* kept, int m_kept, double* out);
int launch_rng_probe(cudaStream_t st, RngKey key, uint32_t purpose, uint32_t stream, uint32_t idx0, int count,
                     double* uniforms, double* normals);

// ---- posterior predictive summaries (opts.fit) ----
// cell code (int8, pitch ldy8): +-1 observed y, +-PRED_HOLDOUT held-out value, 0 neither (scored as +1); sign = orientation
constexpr int8_t PRED_HOLDOUT = 2;
enum PredOut : int { PRED_OUT_PRED = 0, PRED_OUT_LPD = 1, PRED_OUT_PWAIC = 2 };
// per-item statistics / totals: lppd, p_waic, elpd, elpd^2, lpd_holdout, n_obs, n_holdout (sums over the item's cells)
constexpr int PRED_STATS = 7;
// code from y8 and the optional held-out values (n x m, NaN = none; read where y is NA); counts values not in {+1,-1,NaN}
int launch_predictive_code(cudaStream_t st, const int8_t* y8, int64_t ldy8, const double* y_holdout, int n, int m,
                           int8_t* code, unsigned long long* n_bad);
// one sampling iteration (count = 1, 2, ...) into acc = 3 planes of ld x m: sum sigma, Welford mean / M2 of log sigma
int launch_predictive_accumulate(cudaStream_t st, const double* f, int64_t ld, const int8_t* code, int64_t ldc,
                                 const double* theta, const double* beta, int n, int m, double count, double* acc);
// one per-cell output (PredOut) of S accumulated iterations -> out, n x m tightly packed
int launch_predictive_cells(cudaStream_t st, const double* acc, int64_t ld, const int8_t* code, int64_t ldc, int n, int m,
                            double S, int which, double* out);
// stats (PRED_STATS x m, per item), resp_totals = elpd per respondent (n) then the PRED_STATS totals; partial: n_chunks x n
// scratch.  Every sum runs in a fixed order (bit-identical run to run, no floating-point atomics).
int launch_predictive_reduce(cudaStream_t st, const double* acc, int64_t ld, const int8_t* code, int64_t ldc, int n, int m,
                             double S, double* stats, double* partial, int n_chunks, double* resp_totals);
// the two fixed-order steps of that reduction on their own: out[k] = sum over c < n_chunks of partial[c * N + k], in order
// of c; totals[k] = sum over j < m of stats[k * m + j] for k < n_stats (one CTA per statistic)
int launch_reduce_partials(cudaStream_t st, const double* partial, int N, int n_chunks, double* out);
int launch_stat_totals(cudaStream_t st, const double* stats, int n_stats, int m, double* totals);

// ---- IRF posterior summaries (opts.irf, definitions in include/gpirt_b200.h) ----
// Which order statistics a band at level `band` over S draws needs (type 7 quantiles at q_lo = (1 - b)/2, q_hi = (1 + b)/2)
// and how many values per cell the two tail heaps keep: K_lo = r_lo + 2 (at most S) smallest, K_hi = S - r_hi largest.
struct IrfBandPlan {
    int klo = 0, khi = 0;
    bool lo_last = false, hi_last = false;   // r = S - 1: Q = x_(S-1)
    double tlo = 0.0, thi = 0.0;
};
IrfBandPlan irf_band_plan(int S, double band);
// draw s (1-based) of `cells` grid cells, cell c = k + j rows read from x[k + j ld]: Welford mean / M2 of plogis(x) and,
// with klo > 0, the tail heaps (slot-major: heap[slot * cells + c]; lo a max-heap of the klo smallest, hi a min-heap of
// the khi largest)
int launch_irf_accumulate(cudaStream_t st, const double* x, int64_t ld, int rows, int64_t cells, int s, double* mean,
                          double* m2, double* lo, int klo, double* hi, int khi);
// after S >= 1 draws: sd_out = sqrt(m2 / (S - 1)) (sd_out may be m2; NULL: skipped) and, with lo != NULL, the band ends
// Q(q_lo) -> lower, Q(q_hi) -> upper (plogis applied if asked; lower may alias heap slot 0 of lo, upper of hi)
int launch_irf_finish_bands(cudaStream_t st, int64_t cells, int S, const double* m2, double* sd_out, const double* lo,
                            const double* hi, const IrfBandPlan& plan, bool plogis, double* lower, double* upper);

// ---- convergence diagnostics of several chains (opts.chains, definitions in include/gpirt_b200.h) ----
// sampling iteration s (1-based) of S of one chain: with halves != NULL the Welford mean / M2 of plogis(x) of the half the
// iteration belongs to (planes mean_0, m2_0, mean_1, m2_1 of `cells`; the middle iteration of an odd S is skipped); with
// trace != NULL trace[p S + s - 1] = theta[p] (p < n) or beta[p - n] (n <= p < n + nbeta)
int launch_chain_halves(cudaStream_t st, const double* x, int64_t ld, int rows, int64_t cells, int s, int S, double* halves,
                        const double* theta, int n, const double* beta, int nbeta, double* trace);
// after S >= 4 iterations of C chains (trace: C blocks of P x S, parameter-major): split-R-hat and summed Geyer ESS per
// parameter (rhat / ess: P, either may be NULL); fixed-order reductions, no atomics
int launch_chain_diag(cudaStream_t st, const double* trace, int P, int S, int C, double* rhat, double* ess);
// dynamic shared memory k_chain_diag stages one chain in (0: the chain is read from global memory)
int chain_diag_smem_bytes(int S);
// split-R-hat of P per cell over the 2C half-chain states (chain c's four planes at halves + 4 c cells), S >= 4
int launch_chain_irf_rhat(cudaStream_t st, const double* halves, int64_t cells, int S, int C, double* rhat);


}  // namespace gpirt
