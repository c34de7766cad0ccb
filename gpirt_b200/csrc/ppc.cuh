// Posterior predictive model checks (opts.ppc, definitions in include/gpirt_b200.h): the replication of y and the
// Pearson chi-square exceedances (ppc.cu: k_ppc_replicate and its fixed-order reductions), and the pairwise odds-ratio
// exceedances on the int8 tensor cores (k_ppc_pairs).
#pragma once
#include <functional>

#include "common.cuh"
#include "philox.cuh"

namespace gpirt {

constexpr int PPC_CHUNKS = 64;   // item chunks of the replication grid (the per-respondent sums run over these in order)
constexpr int PPC_STAGE_COLS = 512;   // columns of the m x m outputs staged on the device per copy to the host

// Chi-square state of one chain: exceedance counters and the scratch of the fixed-order reductions.  One pool
// allocation; layout in ppc.cu.
struct PpcChi2 {
    int n = 0, m = 0;
    void* buf = nullptr;
    uint32_t *item_cnt = nullptr, *resp_cnt = nullptr, *glob_cnt = nullptr;
    int *item_nobs = nullptr, *resp_nobs = nullptr;
    double2 *wpart = nullptr, *rpart = nullptr, *item_d = nullptr;
    cudaStream_t stream_for_free = nullptr;

    int init(cudaStream_t st, const int8_t* y8, int64_t ldy8, int n, int m);
    // one sampling iteration: y^rep drawn from the state (f, theta, beta) with key (the counter of the sweep that produced
    // it), written to yrep (pitch ldy8; NULL: not kept), the discrepancies of y and y^rep compared, the counters bumped
    int iterate(cudaStream_t st, const double* f, int64_t ld, const int8_t* y8, int64_t ldy8, const double* theta,
                const double* beta, RngKey key, uint32_t item_offset, int8_t* yrep);
    // the PPP-values after S iterations (NaN with S = 0 and where an item / respondent has no observed cell); outputs
    // may be NULL
    int finish(cudaStream_t st, int S, double* item_ppp, double* resp_ppp, double* ppp);
    void destroy();
};

// Odds-ratio state: the observed counts of every item pair of the upper tile triangle, the exceedance counters, the
// replicate plane the caller fills, the observed-cell mask (with missing cells) and the output staging.  One cudaMalloc
// (not the pool: it can be GBs and must not stay reserved after the call).
struct PpcPairs {
    struct Maps;
    int n = 0, m = 0, mt = 0;
    int64_t ldy = 0, tiles = 0;
    bool missing = false;
    char* buf = nullptr;
    size_t bytes = 0;
    int8_t *yrep = nullptr, *mask = nullptr;
    int *colsum_obs = nullptr, *colsum_rep = nullptr;
    int4* obs = nullptr;
    uint32_t* cnt = nullptr;
    double* stage = nullptr;
    Maps* maps = nullptr;

    static size_t bytes_needed(int64_t n, int64_t m, bool missing);
    // y8: n x m {+1, -1, 0 = missing}, pitch ldy (a multiple of 16): counts the observed pairs (one tensor-core pass)
    int init(cudaStream_t st, const int8_t* y8, int64_t ldy, int n, int m, bool missing);
    // one replicate (yrep filled, 0 where y is missing): counters += [OR(rep) >= OR(obs)] for every pair
    int iterate(cudaStream_t st);
    // scale = 1 / S (pair_ppp) or 1 (counts); all_nan: every output NaN.  Host outputs m x m, either may be NULL, written
    // through copy(host, device, count), which must return when the copy has landed.
    using CopyOut = std::function<int(double*, const double*, size_t)>;
    int finish(cudaStream_t st, double scale, bool all_nan, double* log_or, double* ppp, const CopyOut& copy);
    void destroy();
    // the observed counts from y8 (init runs it; idempotent) and the exceedance counters back to zero (measurement)
    int observed_pass(cudaStream_t st, const int8_t* y8);
    int clear_counters(cudaStream_t st);
};

// n x m doubles (column-major, tight) -> int8 plane of pitch ldy (padding rows are left alone).  mask NULL: +1 / -1 / NaN
// -> +1 / -1 / 0, counts[0] += NaN cells; mask set: +1 / -1 read where mask != 0, 0 elsewhere.  counts[1] += other values.
int launch_ppc_plane(cudaStream_t st, const double* src, int n, int m, const int8_t* mask, int8_t* dst, int64_t ldy,
                     unsigned long long* counts);

}  // namespace gpirt
