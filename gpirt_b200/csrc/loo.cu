// PSIS-LOO (opts.loo, gpirt_b200_psis_loo): definitions in include/gpirt_b200.h, state layout in loo.cuh.
#include <algorithm>
#include <cmath>

#include "kernels.cuh"
#include "loo.cuh"
#include "tails.cuh"

namespace gpirt {

int64_t loo_tail_len(int64_t S) {
    if (S <= 0) return 0;
    const double Sd = (double)S;
    return (int64_t)std::ceil(std::min(0.2 * Sd, 3.0 * std::sqrt(Sd)));
}
double loo_state_bytes(int64_t S, int64_t cells) {
    return 8.0 * ((double)loo_tail_len(S) + 4.0) * (double)cells;
}
double loo_k_threshold(int64_t S) {
    if (S <= 0) return NAN;
    return std::min(1.0 - 1.0 / std::log10((double)S), 0.7);
}

// ---- update: one draw of one cell ----
// Rejected and evicted draws go into the outside sum directly; it is never formed as "all minus tail", which cancels
// exactly when the tail is heavy.
__device__ __forceinline__ void loo_update(double* __restrict__ st, int64_t cells, int64_t c, int K, int s, double ll,
                                           double sig) {
    double* mxp = st + (int64_t)K * cells + c;
    double* outp = mxp + cells;
    double* sump = outp + cells;
    const double r = -ll;
    if (s == 1) {   // first draw: no memset of the state
        st[c] = ll;
        *mxp = r;
        *outp = 0.0;
        *sump = sig;
        return;
    }
    *sump += sig;   // in draw order, as k_predictive_accumulate sums sigma
    double mx = *mxp, out = *outp, left;
    bool dirty = false;
    if (r > mx) {   // the new draw enters the heap: rescale the outside sum to the new max
        out *= exp(mx - r);
        mx = r;
        *mxp = mx;
        dirty = true;
    }
    if (heap_add<true>(st, cells, c, K, min(s - 1, K), ll, &left)) {
        out += exp(-left - mx);
        dirty = true;
    }
    if (dirty) *outp = out;
}

__global__ void __launch_bounds__(256) k_loo_accumulate(const double* __restrict__ f, int64_t ld,
                                                        const int8_t* __restrict__ y8, int64_t ldy8,
                                                        const double* __restrict__ theta, const double* __restrict__ beta,
                                                        int n, int s, int K, double* __restrict__ state, int64_t cells) {
    const int i = blockIdx.y * blockDim.x + threadIdx.x, j = blockIdx.x;
    if (i >= n) return;
    const int8_t y = y8[i + (int64_t)j * ldy8];
    if (y == 0) return;
    const double b0 = __ldg(beta + 2 * j), b1 = __ldg(beta + 2 * j + 1);
    const double g = f[i + (int64_t)j * ld] + fma(__ldg(theta + i), b1, b0);   // as k_predictive_accumulate
    double sig, ls;
    log_sigmoid(y < 0 ? -g : g, sig, ls);
    loo_update(state, cells, i + (int64_t)j * n, K, s, ls, sig);
}
int launch_loo_accumulate(cudaStream_t st, const double* f, int64_t ld, const int8_t* y8, int64_t ldy8, const double* theta,
                          const double* beta, int n, int m, int s, int K, double* state) {
    dim3 grid((unsigned)m, (unsigned)ceil_div(n, 256));
    GP_LAUNCH(k_loo_accumulate, grid, 256, 0, st, f, ld, y8, ldy8, theta, beta, n, s, K, state, (int64_t)n * m);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

__global__ void __launch_bounds__(256) k_loo_update_ll(const double* __restrict__ ll, int64_t cells, int s, int K,
                                                       double* __restrict__ state) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cells) return;
    const double v = ll[c];
    loo_update(state, cells, c, K, s, v, exp(v));
}
int launch_loo_update_ll(cudaStream_t st, const double* ll, int64_t cells, int s, int K, double* state) {
    if (cells <= 0) return GPIRT_B200_OK;
    GP_LAUNCH(k_loo_update_ll, (unsigned)ceil_div(cells, 256), 256, 0, st, ll, cells, s, K, state);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

// ---- finish: one warp per cell ----
// Shared memory per warp: the heap padded to P (a power of two) with +inf and sorted ascending, the M tail exceedances
// x, the G profile log-likelihoods of the grid and the three scalars of the cell.
struct LooFinishShape {
    int K = 0, M = 0, P = 1, G = 0, per_warp = 0, warps = 1;
};
static LooFinishShape loo_finish_shape(int64_t S) {
    LooFinishShape f;
    f.M = (int)loo_tail_len(S);
    f.K = f.M + 1;
    while (f.P < f.K) f.P <<= 1;
    f.G = 30 + (int)std::floor(std::sqrt((double)f.M));
    f.per_warp = f.P + f.M + f.G + LOO_STATE_EXTRA;
    f.warps = (int)std::max<int64_t>(1, std::min<int64_t>(8, (48 << 10) / (8 * (int64_t)f.per_warp)));
    return f;
}
static constexpr int LOO_SMEM_MAX = 8 * (LOO_MAX_HEAP + (LOO_MAX_HEAP - 1) + 30 + 90 + LOO_STATE_EXTRA);

__device__ __forceinline__ bool loo_observed(const int8_t* y8, int64_t ldy8, int n, int64_t c) {
    if (!y8) return true;
    const int64_t j = c / n, i = c - j * n;
    return y8[i + j * ldy8] != 0;
}

__global__ void k_loo_finish(double* __restrict__ state, int64_t cells, int S, int M, int P, int G, int per_warp,
                             const int8_t* __restrict__ y8, int64_t ldy8, int n) {
    extern __shared__ double sm[];
    __shared__ int obs[8];
    const int W = blockDim.x >> 5, w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t c0 = (int64_t)blockIdx.x * W;
    const int K = M + 1, Kreal = min(S, K);
    if (threadIdx.x < W) obs[threadIdx.x] = c0 + threadIdx.x < cells && loo_observed(y8, ldy8, n, c0 + threadIdx.x);
    __syncthreads();
    // cooperative load: consecutive threads read consecutive cells of one plane
    for (int64_t e = threadIdx.x; e < (int64_t)(P + LOO_STATE_EXTRA) * W; e += blockDim.x) {
        const int k = (int)(e / W), ww = (int)(e - (int64_t)k * W);
        if (!obs[ww]) continue;
        double* base = sm + (size_t)ww * per_warp;
        if (k < P) base[k] = k < Kreal ? state[(int64_t)k * cells + c0 + ww] : INFINITY;
        else base[P + M + G + (k - P)] = state[(int64_t)(K + k - P) * cells + c0 + ww];
    }
    __syncthreads();
    const int64_t c = c0 + w;
    if (c >= cells) return;
    double* out_e = state + c;
    double* out_p = state + cells + c;
    double* out_k = state + 2 * cells + c;
    if (!obs[w]) {
        if (lane == 0) *out_e = *out_p = *out_k = NAN;
        return;
    }
    double* v = sm + (size_t)w * per_warp;
    double* x = v + P;
    double* lg = x + M;
    const double outside = lg[G + 1], sumsig = lg[G + 2];
    // bitonic sort, ascending in ll (descending in the log ratio r = -ll)
    for (int k = 2; k <= P; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = lane; i < P; i += 32) {
                const int l = i ^ j;
                if (l > i) {
                    const double a = v[i], b = v[l];
                    if ((a > b) == ((i & k) == 0)) { v[i] = b; v[l] = a; }
                }
            }
            __syncwarp();
        }
    }
    // the tail: the T = min(M, S) smallest ll; tail rank i (0-based, ascending in lw) is v[T - 1 - i]
    const int T = min(M, S);
    const double Td = (double)T;
    const double mx = -v[0];
    const bool has_cut = S > M;
    const double cut = has_cut ? -v[M] - mx : -INFINITY;
    const double ec = exp(cut);
    bool smooth = false;
    if (T >= 5) smooth = (-v[0] - mx) - (-v[T - 1] - mx) >= 2.220446049250313e-16 / 100.0;
    double khat = INFINITY, sigma = 0.0;
    if (smooth) {
        for (int i = lane; i < T; i += 32) x[i] = exp(-v[T - 1 - i] - mx) - ec;
        __syncwarp();
        // generalized Pareto fit (Zhang & Stephens 2009, loo's gpdfit).  The profile likelihood: lanes over the grid
        // points, each summing over x in order (independent log1p per iteration, no shuffle chain per grid point)
        const double xstar = x[(int)floor(Td / 4.0 + 0.5) - 1], xN = x[T - 1];
        auto grid_theta = [&](int j) { return 1.0 / xN + (1.0 - sqrt((double)G / ((double)j - 0.5))) / (3.0 * xstar); };
        for (int j = lane + 1; j <= G; j += 32) {
            const double th = grid_theta(j);
            double part = 0.0;
            for (int i = 0; i < T; ++i) part += log1p(-th * x[i]);
            const double kap = part / Td;
            lg[j - 1] = Td * (log(-th / kap) - kap - 1.0);
        }
        __syncwarp();
        double lmax = -INFINITY;
        for (int j = 0; j < G; ++j) lmax = fmax(lmax, lg[j]);
        double se = 0.0;
        for (int j = 0; j < G; ++j) se += exp(lg[j] - lmax);
        const double lse = lmax + log(se);
        double th_hat = 0.0;
        for (int j = 1; j <= G; ++j) th_hat += grid_theta(j) * exp(lg[j - 1] - lse);
        double part = 0.0;
        for (int i = lane; i < T; i += 32) part += log1p(-th_hat * x[i]);
        const double k = warp_sum(part) / Td;
        sigma = -k / th_hat;
        khat = k * Td / (Td + 10.0) + 5.0 / (Td + 10.0);
        if (isnan(khat)) khat = INFINITY;
    }
    const bool smoothed = smooth && isfinite(khat);
    // the two log-sum-exps: the tail draws one per lane, the draws outside the tail in closed form (a non-tail draw has
    // lw + ll = -mx; its weights sum to the outside sum plus the cutoff's term)
    double mxd = -INFINITY, mxn = -INFINITY;
    for (int i = lane; i < T; i += 32) {
        const double ll = v[T - 1 - i];
        double lw = smoothed ? log(sigma * expm1(-khat * log1p(-((double)i + 0.5) / Td)) / khat + ec) : -ll - mx;
        lw = lw > 0.0 ? 0.0 : lw;
        x[i] = lw;   // x is no longer needed
        mxd = fmax(mxd, lw);
        mxn = fmax(mxn, lw + ll);
    }
    const int64_t rest = (int64_t)S - T;
    mxd = fmax(warp_max(mxd), cut);
    mxn = warp_max(mxn);
    if (rest > 0) mxn = fmax(mxn, -mx);
    __syncwarp();
    double den = 0.0, num = 0.0;
    for (int i = lane; i < T; i += 32) {
        den += exp(x[i] - mxd);
        num += exp(x[i] + v[T - 1 - i] - mxn);
    }
    den = warp_sum(den);
    num = warp_sum(num);
    if (has_cut) den += exp(cut - mxd) + exp(log(outside) - mxd);
    if (rest > 0) num += (double)rest * exp(-mx - mxn);
    const double elpd = (mxn + log(num)) - (mxd + log(den));
    const double lpd = log(sumsig / (double)S);   // bit-equal to lpd_cell of opts.fit
    if (lane == 0) {
        *out_e = elpd;
        *out_p = lpd - elpd;
        *out_k = khat;
    }
}
__global__ void __launch_bounds__(256) k_loo_nan(double* __restrict__ out, int64_t count) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c < count) out[c] = NAN;
}
int launch_loo_finish(cudaStream_t st, double* state, int64_t cells, int64_t S, const int8_t* y8, int64_t ldy8, int n) {
    if (cells <= 0) return GPIRT_B200_OK;
    if (S <= 0) {
        GP_LAUNCH(k_loo_nan, (unsigned)ceil_div(3 * cells, 256), 256, 0, st, state, 3 * cells);
        GP_CUDA(cudaGetLastError());
        return GPIRT_B200_OK;
    }
    const LooFinishShape f = loo_finish_shape(S);
    if (f.K > LOO_MAX_HEAP) {
        set_last_error("PSIS-LOO over %lld draws keeps a tail of %d draws per cell; at most %d are built",
                       (long long)S, f.M, LOO_MAX_HEAP - 1);
        return GPIRT_B200_ERR_ARG;
    }
    static bool flags[64];
    {
        DeviceOnce once(flags);
        if (once.first) GP_CUDA(cudaFuncSetAttribute(k_loo_finish, cudaFuncAttributeMaxDynamicSharedMemorySize, LOO_SMEM_MAX));
    }
    const size_t smem = (size_t)f.warps * f.per_warp * sizeof(double);
    GP_LAUNCH(k_loo_finish, (unsigned)ceil_div(cells, f.warps), 32 * f.warps, smem, st, state, cells, (int)S, f.M, f.P, f.G,
              f.per_warp, y8, ldy8, n);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

// ---- reductions over the finished planes ----
// per item, one CTA, fixed order: stats[k * m + j], k = sum elpd, sum elpd^2, sum p_loo, n_obs, n_k_high
__global__ void __launch_bounds__(256) k_loo_items(const double* __restrict__ state, int64_t cells,
                                                   const int8_t* __restrict__ y8, int64_t ldy8, int n, int m, double kthr,
                                                   double* __restrict__ stats) {
    __shared__ double red[2][32];
    const int j = blockIdx.x;
    double v[LOO_STATS] = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        if (y8[i + (int64_t)j * ldy8] == 0) continue;
        const int64_t c = i + (int64_t)j * n;
        const double e = state[c];
        v[0] += e; v[1] += e * e; v[2] += state[cells + c]; v[3] += 1.0;
        v[4] += state[2 * cells + c] > kthr ? 1.0 : 0.0;
    }
#pragma unroll
    for (int k = 0; k < LOO_STATS; ++k) {
        const double t = block_sum(v[k], red[k & 1]);
        if (threadIdx.x == 0) stats[(int64_t)k * m + j] = t;
    }
}
// per respondent: partial[chunk * n + i] = sum of elpd over the observed cells of item chunk `chunk`
__global__ void __launch_bounds__(128) k_loo_resp(const double* __restrict__ state, const int8_t* __restrict__ y8,
                                                  int64_t ldy8, int n, int m, double* __restrict__ partial, int n_chunks) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, chunk = blockIdx.y;
    if (i >= n) return;
    const int per = (int)ceil_div(m, n_chunks), j0 = chunk * per, j1 = min(m, j0 + per);
    double t = 0.0;
    for (int j = j0; j < j1; ++j)
        if (y8[i + (int64_t)j * ldy8] != 0) t += state[i + (int64_t)j * n];
    partial[(int64_t)chunk * n + i] = t;
}
int launch_loo_reduce(cudaStream_t st, const double* state, const int8_t* y8, int64_t ldy8, int n, int m, double k_threshold,
                      double* stats, double* partial, double* resp_totals) {
    const int64_t cells = (int64_t)n * m;
    GP_LAUNCH(k_loo_items, (unsigned)m, 256, 0, st, state, cells, y8, ldy8, n, m, k_threshold, stats);
    dim3 grid((unsigned)ceil_div(n, 128), (unsigned)LOO_CHUNKS);
    GP_LAUNCH(k_loo_resp, grid, 128, 0, st, state, y8, ldy8, n, m, partial, LOO_CHUNKS);
    GP_CUDA(cudaGetLastError());
    GP_TRY(launch_reduce_partials(st, partial, n, LOO_CHUNKS, resp_totals));
    return launch_stat_totals(st, stats, LOO_STATS, m, resp_totals + n);
}

}  // namespace gpirt
