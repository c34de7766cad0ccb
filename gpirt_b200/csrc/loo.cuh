// Leave-one-out cross-validation by Pareto-smoothed importance sampling (opts.loo, definitions in include/gpirt_b200.h):
// a per-cell update over the draws (loo.cu: k_loo_accumulate from the sampler's state, k_loo_update_ll from given
// log-likelihoods), the per-cell finish (k_loo_finish: sort, generalized Pareto fit, smoothed log-sum-exps) and the
// fixed-order reductions per item, per respondent and in all.
#pragma once
#include "common.cuh"

namespace gpirt {

// State of one cell, planes of `cells` doubles (slot-major, cell c of plane p at p * cells + c), K = M + 1:
//   planes [0, K)  a max-heap of the K smallest log-likelihoods seen (root = the cutoff candidate)
//   plane K        the running max of the log ratios r = -ll
//   plane K + 1    sum of exp(r - running max) over the draws outside the heap
//   plane K + 2    sum of sigma, in draw order
constexpr int LOO_STATE_EXTRA = 3;
constexpr int LOO_MAX_HEAP = 8192;   // largest K the finish sorts in shared memory (M <= 8191, S <= 7 454 720)
constexpr int LOO_STATS = 5;         // per item / totals: sum elpd, sum elpd^2, sum p_loo, n_obs, n_k_high
constexpr int LOO_CHUNKS = 64;       // item chunks of the per-respondent sums

// M = ceil(min(0.2 S, 3 sqrt(S))) in FP64 (loo's n_pareto_tail with r_eff = 1); 0 for S <= 0
int64_t loo_tail_len(int64_t S);
// device bytes of the state of `cells` cells: 8 (M + 4) per cell
double loo_state_bytes(int64_t S, int64_t cells);
// k_threshold = min(1 - 1 / log10 S, 0.7) (NaN for S = 0)
double loo_k_threshold(int64_t S);

// sampling iteration s (1-based) of the sampler's end-of-sweep state: g = f + beta0 + beta1 theta on the observed cells of
// y8 (n x m, pitch ldy8), cell c = i + j n of the state (K = M + 1)
int launch_loo_accumulate(cudaStream_t st, const double* f, int64_t ld, const int8_t* y8, int64_t ldy8, const double* theta,
                          const double* beta, int n, int m, int s, int K, double* state);
// draw s (1-based) of given log-likelihoods ll[c], c < cells, every cell a left-out unit, sigma = exp(ll)
int launch_loo_update_ll(cudaStream_t st, const double* ll, int64_t cells, int s, int K, double* state);
// after S draws: elpd_loo_cell, p_loo_cell and pareto_k into planes 0, 1, 2 of the state (in place), NaN where y8 is 0
// (y8 NULL: every cell observed; cell c = i + j n) and everywhere for S = 0
int launch_loo_finish(cudaStream_t st, double* state, int64_t cells, int64_t S, const int8_t* y8, int64_t ldy8, int n);
// from the finished planes: stats (LOO_STATS x m, per item), resp_totals = elpd per respondent (n) then the LOO_STATS
// totals; partial: LOO_CHUNKS x n scratch.  Fixed order, no atomics.
int launch_loo_reduce(cudaStream_t st, const double* state, const int8_t* y8, int64_t ldy8, int n, int m, double k_threshold,
                      double* stats, double* partial, double* resp_totals);

}  // namespace gpirt
