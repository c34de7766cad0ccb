// Non-GEMM kernels of the Gibbs sweep: covariance builder, response ingest, Philox fills, the batched elliptical
// slice sampler with the fused logistic log-likelihood, f* finishing draw, theta grid sampler, beta Metropolis step.
#include <algorithm>
#include <cmath>
#include <map>
#include <mutex>
#include <tuple>

#include "kernels.cuh"
#include "softplus_table.cuh"

namespace gpirt {

// ------------------------------------------------------------------------------------------------------------------
// Squared-exponential covariance, reference src/covariance-function.cpp:3-14 (+ S.diag() += 0.001, gpirtMCMC.cpp:16).
// HBM-write-bound: each thread owns two consecutive rows (one 16-byte store) and walks 8 columns re-using x1.
// ------------------------------------------------------------------------------------------------------------------
constexpr int SE_COLS = 8;
__global__ void __launch_bounds__(128) k_se_cov(const double* __restrict__ x1, int n1, const double* __restrict__ x2,
                                                int n2, double jitter, int lower_only, double* __restrict__ out,
                                                int64_t ld) {
    const int i0 = 2 * (blockIdx.x * blockDim.x + threadIdx.x);
    if (i0 >= n1) return;
    const bool two = (i0 + 1 < n1);
    const double a0 = x1[i0], a1 = two ? x1[i0 + 1] : 0.0;
    const int j0 = blockIdx.y * SE_COLS;
#pragma unroll
    for (int jj = 0; jj < SE_COLS; ++jj) {
        const int j = j0 + jj;
        if (j >= n2) break;
        const double b = x2[j];
        double v0 = 0.0, v1 = 0.0;
        if (!lower_only || i0 >= j) { const double d = a0 - b; v0 = exp(-0.5 * d * d); if (i0 == j) v0 += jitter; }
        if (two && (!lower_only || i0 + 1 >= j)) { const double d = a1 - b; v1 = exp(-0.5 * d * d); if (i0 + 1 == j) v1 += jitter; }
        double* dst = out + i0 + (int64_t)j * ld;
        if (two) *reinterpret_cast<double2*>(dst) = make_double2(v0, v1);  // ld even, i0 even => 16-byte aligned
        else *dst = v0;
    }
}

int launch_se_cov(cudaStream_t st, const double* x1, int n1, const double* x2, int n2, double jitter, bool lower_only,
                  double* out, int64_t ld) {
    if (n1 <= 0 || n2 <= 0) return GPIRT_B200_OK;
    if (ld % 2) { set_last_error("se_cov: leading dimension must be even"); return GPIRT_B200_ERR_ARG; }
    dim3 grid((unsigned)ceil_div(ceil_div(n1, 2), 128), (unsigned)ceil_div(n2, SE_COLS));
    GP_LAUNCH(k_se_cov, grid, 128, 0, st, x1, n1, x2, n2, jitter, lower_only ? 1 : 0, out, ld);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

// theta*_k = start + (k * delta) with two roundings, exactly arma::regspace (gpirtMCMC.cpp:35); prior = dnorm(.,0,1,log)
__global__ void k_grid_init(double* theta_star, double* prior) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= N_GRID) return;
    const double t = __dadd_rn(-5.0, __dmul_rn((double)k, 0.01));
    theta_star[k] = t;
    const double a = fabs(t);
    prior[k] = -(0.918938533204672741780329736406 + __dmul_rn(__dmul_rn(0.5, a), a) + log(1.0));
}
int launch_grid_init(cudaStream_t st, double* theta_star, double* prior) {
    GP_LAUNCH(k_grid_init, (unsigned)ceil_div(N_GRID, 256), 256, 0, st, theta_star, prior);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

// Response ingest (contract: R/response_matrix.R:79-98 produces REALSXP {1,-1,NA_real_}; log-likelihood.cpp:16,30 tests isnan)
__global__ void k_ingest_y(const double* __restrict__ y, int n, int m, int8_t* __restrict__ y8, int64_t ldy8,
                           double* __restrict__ yd, int64_t ldyd, unsigned long long* n_missing,
                           unsigned long long* n_bad) {
    const int i = blockIdx.y * blockDim.x + threadIdx.x, j = blockIdx.x;   // items on grid.x (2^31-1), rows on grid.y
    if (i >= n) return;
    const double v = y[i + (int64_t)j * n];
    int8_t c = 0;
    if (v == 1.0) c = 1;
    else if (v == -1.0) c = -1;
    else if (isnan(v)) atomicAdd(n_missing, 1ull);
    else atomicAdd(n_bad, 1ull);
    y8[i + (int64_t)j * ldy8] = c;
    if (yd) yd[i + (int64_t)j * ldyd] = (double)c;
}
int launch_ingest_y(cudaStream_t st, const double* y, int n, int m, int8_t* y8, int64_t ldy8, double* yd, int64_t ldyd,
                    unsigned long long* n_missing, unsigned long long* n_bad) {
    dim3 grid((unsigned)m, (unsigned)ceil_div(n, 256));
    GP_LAUNCH(k_ingest_y, grid, 256, 0, st, y, n, m, y8, ldy8, yd, ldyd, n_missing, n_bad);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// Philox fills
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_fill_normal(double* __restrict__ Z, int n, int64_t ld, RngKey key,
                                                     uint32_t purpose, uint32_t item_offset) {
    const int pair = blockIdx.y * blockDim.x + threadIdx.x, j = blockIdx.x;
    const int i0 = 2 * pair;
    if (i0 >= n) return;
    double za, zb;
    rng_normal_pair(key, purpose, item_offset + (uint32_t)j, (uint32_t)pair, za, zb);
    double* dst = Z + i0 + (int64_t)j * ld;
    if (i0 + 1 < n) *reinterpret_cast<double2*>(dst) = make_double2(za, zb);
    else *dst = za;
}
int launch_fill_normal(cudaStream_t st, double* Z, int n, int m, int64_t ld, RngKey key, uint32_t purpose,
                       uint32_t item_offset) {
    if (n <= 0 || m <= 0) return GPIRT_B200_OK;
    dim3 grid((unsigned)m, (unsigned)ceil_div(ceil_div(n, 2), 256));
    GP_LAUNCH(k_fill_normal, grid, 256, 0, st, Z, n, ld, key, purpose, item_offset);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

// The same normals written straight as the 8 balanced base-128 digit planes of the fixed-point product nu = L Z
// (dgemm_i8.cu): |z| < 8.7 for every 53-bit Box-Muller draw, so all columns share the scale 2^4 and no column-maximum
// pass (and no FP64 copy of Z) is needed.  One thread = 4 consecutive respondents = one 32-bit store per plane.
constexpr int Z_FIXED_EXP = 4;
__global__ void __launch_bounds__(256) k_fill_normal_planes(int8_t* __restrict__ planes, double* __restrict__ scale,
                                                            int64_t rows_pad, int64_t k_pad, int n, RngKey key,
                                                            uint32_t purpose, uint32_t item_offset,
                                                            double* __restrict__ Z, int64_t ld) {
    const int quad = blockIdx.y * blockDim.x + threadIdx.x, j = blockIdx.x;
    const int i0 = 4 * quad;
    if (quad == 0) scale[j] = 0.25;                 // 2^(Z_FIXED_EXP - 6)
    if (i0 >= n) return;
    double z[4];
    rng_normal_pair(key, purpose, item_offset + (uint32_t)j, (uint32_t)(2 * quad), z[0], z[1]);
    if (i0 + 2 < n) rng_normal_pair(key, purpose, item_offset + (uint32_t)j, (uint32_t)(2 * quad + 1), z[2], z[3]);
    else z[2] = z[3] = 0.0;
    unsigned packed[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        const double v = (i0 + b < n) ? z[b] : 0.0;
        if (Z && i0 + b < n) Z[i0 + b + (int64_t)j * ld] = v;
        long long X = __double2ll_rn(v * 2251799813685248.0);   // 2^(55 - Z_FIXED_EXP) = 2^51
#pragma unroll
        for (int s = 7; s >= 1; --s) {
            const int d = (int)((X + 64) & 127) - 64;
            packed[s] |= (unsigned)(d & 0xFF) << (8 * b);
            X = (X - d) >> 7;
        }
        packed[0] |= (unsigned)((int)X & 0xFF) << (8 * b);
    }
#pragma unroll
    for (int s = 0; s < 8; ++s)
        *reinterpret_cast<unsigned*>(planes + ((int64_t)s * rows_pad + j) * k_pad + i0) = packed[s];
}
int launch_fill_normal_planes(cudaStream_t st, int8_t* planes, double* scale, int64_t rows_pad, int64_t k_pad, int n, int m,
                              RngKey key, uint32_t purpose, uint32_t item_offset, double* Z_or_null, int64_t ld) {
    if (n <= 0 || m <= 0) return GPIRT_B200_OK;
    dim3 grid((unsigned)m, (unsigned)ceil_div(ceil_div(n, 4), 256));
    GP_LAUNCH(k_fill_normal_planes, grid, 256, 0, st, planes, scale, rows_pad, k_pad, n, key, purpose, item_offset, Z_or_null, ld);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

__global__ void k_init_beta(double* beta, const double* pm, const double* psd, int m, RngKey key, uint32_t item_offset) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    double z0, z1;
    rng_normal_pair(key, P_INIT_BETA, item_offset + (uint32_t)j, 0u, z0, z1);
    beta[2 * j] = __dadd_rn(pm[2 * j], __dmul_rn(psd[2 * j], z0));          // R::rnorm(mu, sigma) = mu + sigma * z
    beta[2 * j + 1] = __dadd_rn(pm[2 * j + 1], __dmul_rn(psd[2 * j + 1], z1));
}
int launch_init_beta(cudaStream_t st, double* beta, const double* pm, const double* psd, int m, RngKey key,
                     uint32_t item_offset) {
    GP_LAUNCH(k_init_beta, (unsigned)ceil_div(m, 128), 128, 0, st, beta, pm, psd, m, key, item_offset);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

__global__ void k_rng_probe(RngKey key, uint32_t purpose, uint32_t stream, uint32_t idx0, int count, double* u, double* z) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    u[t] = rng_uniform(key, purpose, stream, idx0 + t);
    z[t] = rng_normal(key, purpose, stream, idx0 + t);
}
int launch_rng_probe(cudaStream_t st, RngKey key, uint32_t purpose, uint32_t stream, uint32_t idx0, int count,
                     double* uniforms, double* normals) {
    GP_LAUNCH(k_rng_probe, (unsigned)ceil_div(count, 128), 128, 0, st, key, purpose, stream, idx0, count, uniforms, normals);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// Elliptical slice sampler (reference src/draw-f.cpp:21-60, likelihood src/log-likelihood.cpp:25-37) and beta Metropolis
// step (src/draw-beta.cpp:16-38): ONE __device__ body each (ess_item, beta_item), shared by three launch shapes
//   k_*          one CTA per item, the item's columns in registers (EPT values per thread)
//   k_*_persist  one CTA per SM claims items from an atomic counter and cp.async-prefetches the next item's columns
//   k_*_stream   n > 4096: the item no longer fits the register file of a CTA; every evaluation re-streams it from L2
// The shapes differ only in where a thread's cells come from (the Cur / Prop / Eval functors below).
// The block-wide log-likelihood sum is a fixed-order shuffle + shared-memory reduction (every thread ends with the same
// bits, so the accept test needs no broadcast); the uniforms come from Philox by address, recomputed by every thread.
// ------------------------------------------------------------------------------------------------------------------
constexpr int ESS_ITER_CAP = 10000;

// log-likelihood term of one cell, 0 for a missing cell (y = 0; the reference skips NA, log-likelihood.cpp:18,32).
// Branch-free on purpose: with `if (y != 0)` around every term the compiler cannot interleave the independent
// evaluations of a thread's values and the FP64 dependency chains run one after the other.
__device__ __forceinline__ double obs_term(const double* __restrict__ sp, double y, double a) {
    const double t = ll_term_fast(sp, a);
    return (y != 0.0) ? t : 0.0;
}

// One item's slice step.  cur() -> this thread's partial of ll_bar(f, y, mu);  prop(c, s) -> its partial of
// ll_bar(f c + nu s, y, mu).  Returns the number of proposals; (c_out, s_out) = cosine / sine of the accepted angle.
// The angle of proposal t+1 does not depend on the likelihood of proposal t, only on its being rejected: the shrunk
// bracket, the next Philox uniform, the next angle and its sine / cosine are computed by warp 0 WHILE proposal t is
// evaluated and published through shared memory ahead of the barrier of the block sum, so the serial part of a round
// is the reduction alone.  Same formulas, same bits as the sequential loop.
template <class Cur, class Prop>
__device__ __forceinline__ int ess_item(const RngKey& key, uint32_t item, double (*red)[32], double (*nxt)[4], int* status,
                                        Cur&& cur, Prop&& prop, double& c_out, double& s_out) {
    const int tid = threadIdx.x;
    const double ll_cur = block_sum(cur(), red[0]);
    const double log_y = ll_cur + log(rng_uniform(key, P_ESS_U, item, 0u));             // draw-f.cpp:28-29
    const double TWO_PI = 6.283185307179586476925286766559;
    double eps_min = 0.0, eps_max = TWO_PI;                                             // :33-34
    double eps = eps_min + (eps_max - eps_min) * rng_uniform(key, P_ESS_U, item, 1u);   // :35 R::runif(a,b) = a + (b-a) u
    eps_min = eps - TWO_PI;                                                             // :36 (eps_max stays 2 pi)
    int iter = 0;
    double s, c;
    sincos(eps, &s, &c);
    const bool leader = tid < 32;
    for (;;) {
        iter += 1;
        const double emin_n = (eps < 0.0) ? eps : eps_min, emax_n = (eps < 0.0) ? eps_max : eps;   // :50-55 if rejected
        if (leader) {
            const double eps_n = emin_n + (emax_n - emin_n) * rng_uniform(key, P_ESS_U, item, 1u + (uint32_t)iter);  // :56
            double sn, cn;
            sincos(eps_n, &sn, &cn);
            if (tid == 0) { nxt[iter & 1][0] = eps_n; nxt[iter & 1][1] = sn; nxt[iter & 1][2] = cn; }
        }
        const double ll_new = block_sum(prop(c, s), red[iter & 1]);
        if (ll_new > log_y) break;                                                      // :45 strict
        eps_min = emin_n; eps_max = emax_n;
        eps = nxt[iter & 1][0]; s = nxt[iter & 1][1]; c = nxt[iter & 1][2];
        if (iter >= ESS_ITER_CAP) { if (tid == 0) atomicExch(status, 1); break; }       // NaN likelihood: reference would spin
    }
    c_out = c; s_out = s;
    return iter;
}

// an item's cells held in registers: value e of thread tid is respondent tid + e * blockDim.x
template <int EPT> struct ItemRegs {
    double fv[EPT], nv[EPT], gm[EPT], yv[EPT];
    __device__ __forceinline__ double cur(const double* __restrict__ sp) const {
        double part = 0.0;
#pragma unroll
        for (int e = 0; e < EPT; ++e) part -= obs_term(sp, yv[e], yv[e] * (fv[e] + gm[e]));
        return part;
    }
    __device__ __forceinline__ double prop(const double* __restrict__ sp, double c, double s) const {
        double part = 0.0;
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            const double fp = __dadd_rn(__dmul_rn(fv[e], c), __dmul_rn(nv[e], s));      // :43, no FMA contraction
            part -= obs_term(sp, yv[e], yv[e] * (fp + gm[e]));
        }
        return part;
    }
    __device__ __forceinline__ void store(double* __restrict__ fj, int n, double c, double s) const {
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            const int i = threadIdx.x + e * blockDim.x;
            if (i < n) fj[i] = __dadd_rn(__dmul_rn(fv[e], c), __dmul_rn(nv[e], s));
        }
    }
};

template <int EPT>
__global__ void __launch_bounds__(512) k_ess(double* __restrict__ f, const double* __restrict__ nu, int64_t ld, const int8_t* __restrict__ y8,
                      int64_t ldy, const double* __restrict__ theta, const double* __restrict__ beta, int n, RngKey key,
                      uint32_t item_offset, int* __restrict__ nprop, int* __restrict__ status,
                      const double* __restrict__ sp) {
    __shared__ double red[2][32];
    __shared__ double nxt[2][4];   // speculative next proposal: angle, sine, cosine (double-buffered like red)
    const int j = blockIdx.x, tid = threadIdx.x, T = blockDim.x;
    const double b0 = beta[2 * j], b1 = beta[2 * j + 1];
    ItemRegs<EPT> it;
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
        const int i = tid + e * T;
        if (i < n) {
            it.fv[e] = f[i + (int64_t)j * ld];
            it.nv[e] = nu[i + (int64_t)j * ld];
            it.yv[e] = (double)y8[i + (int64_t)j * ldy];
            it.gm[e] = fma(theta[i], b1, b0);
        } else { it.fv[e] = it.nv[e] = it.gm[e] = it.yv[e] = 0.0; }
    }
    double c, s;
    const int iter = ess_item(key, item_offset + (uint32_t)j, red, nxt, status, [&] { return it.cur(sp); },
                              [&](double cc, double ss) { return it.prop(sp, cc, ss); }, c, s);
    it.store(f + (int64_t)j * ld, n, c, s);
    if (tid == 0 && nprop) nprop[j] = iter;
}

// Large-n shape (n > 4096): same body, but every evaluation re-streams f, nu, y, theta from L2 (the 17n bytes of an item
// stay L2-resident across its shrink loop).
__global__ void __launch_bounds__(1024) k_ess_stream(double* __restrict__ f, const double* __restrict__ nu, int64_t ld,
                                                     const int8_t* __restrict__ y8, int64_t ldy,
                                                     const double* __restrict__ theta, const double* __restrict__ beta,
                                                     int n, RngKey key, uint32_t item_offset, int* __restrict__ nprop,
                                                     int* __restrict__ status, const double* __restrict__ sp) {
    __shared__ double red[2][32];
    __shared__ double nxt[2][4];
    const int j = blockIdx.x, tid = threadIdx.x, T = blockDim.x;
    const double b0 = beta[2 * j], b1 = beta[2 * j + 1];
    double* fj = f + (int64_t)j * ld;
    const double* nj = nu + (int64_t)j * ld;
    const int8_t* yj = y8 + (int64_t)j * ldy;
    auto cur = [&] {
        double part = 0.0;
#pragma unroll 4
        for (int i = tid; i < n; i += T) {
            const double yv = (double)yj[i];
            part -= obs_term(sp, yv, yv * (fj[i] + fma(theta[i], b1, b0)));
        }
        return part;
    };
    auto prop = [&](double c, double s) {
        double part = 0.0;
#pragma unroll 4
        for (int i = tid; i < n; i += T) {
            const double yv = (double)yj[i];
            const double fp = __dadd_rn(__dmul_rn(fj[i], c), __dmul_rn(nj[i], s));
            part -= obs_term(sp, yv, yv * (fp + fma(theta[i], b1, b0)));
        }
        return part;
    };
    double c, s;
    const int iter = ess_item(key, item_offset + (uint32_t)j, red, nxt, status, cur, prop, c, s);
    for (int i = tid; i < n; i += T) fj[i] = __dadd_rn(__dmul_rn(fj[i], c), __dmul_rn(nj[i], s));
    if (tid == 0 && nprop) nprop[j] = iter;
}

// ---- persistent shape -----------------------------------------------------------------------------------------------
// One CTA per SM walks the item list (next item claimed with an atomic counter, so the data-dependent proposal counts
// balance themselves) and the NEXT item's f, nu and y columns are fetched into shared memory with cp.async while the
// current item's shrink loop runs: with one register-heavy CTA per SM the HBM latency of every item's loads was fully
// exposed (ncu: a quarter of all stall samples sat on the first use of the loaded columns).  theta is read once per CTA.
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int EPT>
__global__ void __launch_bounds__(512) k_ess_persist(double* __restrict__ f, const double* __restrict__ nu, int64_t ld,
                                                      const int8_t* __restrict__ y8, int64_t ldy, const double* __restrict__ theta,
                                                      const double* __restrict__ beta, int n, int m, RngKey key,
                                                      uint32_t item_offset, int* __restrict__ nprop, int* __restrict__ status,
                                                      const double* __restrict__ sp, int* __restrict__ work) {
    extern __shared__ __align__(16) unsigned char dsm[];
    __shared__ double red[2][32];
    __shared__ double nxt[2][4];
    __shared__ int s_next;
    const int tid = threadIdx.x, T = blockDim.x, NP = EPT * T;
    double* fbuf = reinterpret_cast<double*>(dsm);
    double* nbuf = fbuf + 2 * NP;
    int8_t* ybuf = reinterpret_cast<int8_t*>(nbuf + 2 * NP);
    double th[EPT];
#pragma unroll
    for (int e = 0; e < EPT; ++e) { const int i = tid + e * T; th[e] = (i < n) ? theta[i] : 0.0; }
    auto prefetch = [&](int j, int b) {
        const double* fs = f + (int64_t)j * ld;
        const double* ns = nu + (int64_t)j * ld;
        const int8_t* ys = y8 + (int64_t)j * ldy;
        for (int c = tid; c < (n + 1) / 2; c += T) {
            cp_async16(fbuf + b * NP + 2 * c, fs + 2 * c);
            cp_async16(nbuf + b * NP + 2 * c, ns + 2 * c);
        }
        for (int c = tid; c < (n + 15) / 16; c += T) cp_async16(ybuf + b * NP + 16 * c, ys + 16 * c);
        cp_async_commit();
    };
    int j = blockIdx.x, b = 0;
    if (j < m) prefetch(j, 0);
    while (j < m) {
        if (tid == 0) s_next = (int)gridDim.x + atomicAdd(work, 1);
        __syncthreads();
        const int jn = s_next;
        if (jn < m) { prefetch(jn, b ^ 1); cp_async_wait<1>(); } else cp_async_wait<0>();
        __syncthreads();
        const double b0 = beta[2 * j], b1 = beta[2 * j + 1];
        ItemRegs<EPT> it;
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            const int i = tid + e * T;
            if (i < n) {
                it.fv[e] = fbuf[b * NP + i];
                it.nv[e] = nbuf[b * NP + i];
                it.yv[e] = (double)ybuf[b * NP + i];
                it.gm[e] = fma(th[e], b1, b0);
            } else { it.fv[e] = it.nv[e] = it.gm[e] = it.yv[e] = 0.0; }
        }
        double c, s;
        const int iter = ess_item(key, item_offset + (uint32_t)j, red, nxt, status, [&] { return it.cur(sp); },
                                  [&](double cc, double ss) { return it.prop(sp, cc, ss); }, c, s);
        it.store(f + (int64_t)j * ld, n, c, s);
        if (tid == 0 && nprop) nprop[j] = iter;
        j = jn;
        b ^= 1;
    }
}

// persistent grid: as many CTAs as fit the device at once; 0 when every item gets its own CTA anyway (then the plain
// one-CTA-per-item kernel is used).  The occupancy query is cached per (kernel, block size, shared memory, device).
template <typename K>
static int persistent_grid(K kernel, int threads, size_t smem, int m, int* grid) {
    struct Key { const void* k; int threads; size_t smem; int dev; bool operator<(const Key& o) const {
        return std::tie(k, threads, smem, dev) < std::tie(o.k, o.threads, o.smem, o.dev); } };
    static std::mutex mu;
    static std::map<Key, int> cache;
    // the shared-memory limit is an attribute of the kernel, not of a launch shape: it only ever grows, so that a smaller
    // shape prepared later (another n) cannot take it below what a shape already in the cache launches with
    static std::map<std::pair<const void*, int>, size_t> smem_limit;
    int dev = 0;
    GP_CUDA(cudaGetDevice(&dev));
    const Key key{(const void*)kernel, threads, smem, dev};
    std::lock_guard<std::mutex> lock(mu);
    auto it = cache.find(key);
    if (it == cache.end()) {
        int sms = 0, per_sm = 0;
        GP_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        size_t& limit = smem_limit[{(const void*)kernel, dev}];
        if (smem > limit) {
            GP_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            limit = smem;
        }
        GP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
        if (per_sm < 1) { set_last_error("per-item kernel does not fit on an SM"); return GPIRT_B200_ERR_CUDA; }
        it = cache.emplace(key, sms * per_sm).first;
    }
    *grid = m > it->second ? it->second : 0;
    return GPIRT_B200_OK;
}
// block size / elements-per-thread for a per-item CTA holding n <= 4096 respondents in registers (ept = 0: stream)
static void item_cta_shape(int n, int& ept, int& threads) {
    // 2048 < n <= 4096: 512 threads x 8 values.  1024 x 4 (32 warps per SM instead of 16) was measured 10% SLOWER at
    // n = 4096 — the kernels are bound by the L1 gather of table rows, not by latency.
    if (n <= 256) ept = 1; else if (n <= 1024) ept = 2; else if (n <= 2048) ept = 4; else if (n <= 4096) ept = 8; else ept = 0;
    threads = ept ? (int)round_up(ceil_div(n, ept), 32) : 1024;
    if (threads < 32) threads = 32;
}

#define ESS_PERSIST_CASE(E)                                                                                                  \
    {                                                                                                                            \
        const size_t smem = (size_t)2 * (E) * threads * 17;                                                                      \
        int grid = 0;                                                                                                            \
        GP_TRY(persistent_grid(k_ess_persist<E>, threads, smem, m, &grid));                                                  \
        if (grid > 0) {                                                                                                          \
            GP_CUDA(cudaMemsetAsync(work, 0, sizeof(int), st));                                                                  \
            GP_LAUNCH((k_ess_persist<E>), grid, threads, smem, st, f, nu, ld, y8, ldy, theta, beta, n, m, key, item_offset,  \
                      nprop, status, sp, work);                                                                                  \
            launched = true;                                                                                                     \
        }                                                                                                                        \
    }

int launch_ess(cudaStream_t st, double* f, const double* nu, int64_t ld, const int8_t* y8, int64_t ldy,
               const double* theta, const double* beta, int n, int m, RngKey key, uint32_t item_offset, int* nprop,
               int* status, int* work, int* shape) {
    if (m <= 0) return GPIRT_B200_OK;
    int ept, threads;
    item_cta_shape(n, ept, threads);
    const double* sp = nullptr;
    GP_TRY(softplus_table(&sp));
    if (work && ept) {
        bool launched = false;
        switch (ept) {
            case 1: ESS_PERSIST_CASE(1) break;
            case 2: ESS_PERSIST_CASE(2) break;
            case 4: ESS_PERSIST_CASE(4) break;
            default: ESS_PERSIST_CASE(8) break;
        }
        GP_CUDA(cudaGetLastError());
        if (launched) { if (shape) *shape = ITEM_SHAPE_PERSISTENT; return GPIRT_B200_OK; }
    }
    if (shape) *shape = ept ? ITEM_SHAPE_CTA : ITEM_SHAPE_STREAM;
    switch (ept) {
        case 1: GP_LAUNCH(k_ess<1>, m, threads, 0, st, f, nu, ld, y8, ldy, theta, beta, n, key, item_offset, nprop, status, sp); break;
        case 2: GP_LAUNCH(k_ess<2>, m, threads, 0, st, f, nu, ld, y8, ldy, theta, beta, n, key, item_offset, nprop, status, sp); break;
        case 4: GP_LAUNCH(k_ess<4>, m, threads, 0, st, f, nu, ld, y8, ldy, theta, beta, n, key, item_offset, nprop, status, sp); break;
        case 8: GP_LAUNCH(k_ess<8>, m, threads, 0, st, f, nu, ld, y8, ldy, theta, beta, n, key, item_offset, nprop, status, sp); break;
        default: GP_LAUNCH(k_ess_stream, m, threads, 0, st, f, nu, ld, y8, ldy, theta, beta, n, key, item_offset, nprop, status, sp); break;
    }
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// f* pieces (reference src/draw-fstar.cpp:19-28)
// ------------------------------------------------------------------------------------------------------------------
// s_k = 1 - sqrt(sum_i tmp_ik^2)   (:20 — note 1 - sqrt(.), not sqrt(1 - .)); one warp per grid point
__global__ void __launch_bounds__(256) k_fstar_sd(const double* __restrict__ tmp, int64_t ld, int n, int N, double* s) {
    const int k = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (k >= N) return;
    const double* col = tmp + (int64_t)k * ld;
    double acc = 0.0;
    for (int i = lane; i < n; i += 32) { const double t = col[i]; acc += t * t; }
    acc = warp_sum(acc);
    if (lane == 0) s[k] = 1.0 - sqrt(acc);
}
int launch_fstar_sd(cudaStream_t st, const double* tmp, int64_t ld, int n, int N, double* s) {
    GP_LAUNCH(k_fstar_sd, (unsigned)ceil_div(N, 8), 256, 0, st, tmp, ld, n, N, s);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

// f*_kj = rnorm(mean_kj + mu*_kj, s_k), k ascending within item j (:25-28); mu*_kj = beta0_j + beta1_j theta*_k
__global__ void __launch_bounds__(256) k_fstar_finish(double* __restrict__ fstar, int64_t ld, int N, const double* __restrict__ s,
                                                      const double* __restrict__ beta, const double* __restrict__ theta_star,
                                                      RngKey key, uint32_t item_offset, double* __restrict__ irf_sum,
                                                      int accumulate) {
    const int pair = blockIdx.y * blockDim.x + threadIdx.x, j = blockIdx.x;
    const int k0 = 2 * pair;
    if (k0 >= N) return;
    double za, zb;
    rng_normal_pair(key, P_FSTAR_Z, item_offset + (uint32_t)j, (uint32_t)pair, za, zb);
    const double b0 = beta[2 * j], b1 = beta[2 * j + 1];
    const int64_t off = k0 + (int64_t)j * ld;
    {
        const double mean = fstar[off] + fma(theta_star[k0], b1, b0);
        const double v = __dadd_rn(mean, __dmul_rn(s[k0], za));
        fstar[off] = v;
        if (accumulate) irf_sum[off] += v;
    }
    if (k0 + 1 < N) {
        const double mean = fstar[off + 1] + fma(theta_star[k0 + 1], b1, b0);
        const double v = __dadd_rn(mean, __dmul_rn(s[k0 + 1], zb));
        fstar[off + 1] = v;
        if (accumulate) irf_sum[off + 1] += v;
    }
}
int launch_fstar_finish(cudaStream_t st, double* fstar, int64_t ld, int N, int m, const double* s, const double* beta,
                        const double* theta_star, RngKey key, uint32_t item_offset, double* irf_sum, int accumulate) {
    if (m <= 0) return GPIRT_B200_OK;
    dim3 grid((unsigned)m, (unsigned)ceil_div(ceil_div(N, 2), 256));
    GP_LAUNCH(k_fstar_finish, grid, 256, 0, st, fstar, ld, N, s, beta, theta_star, key, item_offset, irf_sum, accumulate);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

__global__ void k_irf_finish(const double* __restrict__ irf_sum, int64_t ld, int N, double inv_samples, double* __restrict__ out) {
    const int k = blockIdx.y * blockDim.x + threadIdx.x, j = blockIdx.x;
    if (k >= N) return;
    const double x = irf_sum[k + (int64_t)j * ld] * inv_samples;                   // gpirtMCMC.cpp:106
    out[k + (int64_t)j * N] = 1.0 / (1.0 + exp(-x));                               // R::plogis, :109
}
int launch_irf_finish(cudaStream_t st, const double* irf_sum, int64_t ld, int N, int m, double inv_samples, double* out) {
    if (m <= 0) return GPIRT_B200_OK;
    dim3 grid((unsigned)m, (unsigned)ceil_div(N, 256));
    GP_LAUNCH(k_irf_finish, grid, 256, 0, st, irf_sum, ld, N, inv_samples, out);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// theta step (reference src/draw-theta.cpp).  The O(n N m) loop of exp+log pairs becomes a contraction:
//   -log(1+exp(-y f)) = y f / 2 - D(f),  D(f) = log(2 cosh(f/2))   for y = +-1
//   logP_ik = prior_k + 1/2 sum_j y_ij f*_kj - sum_j obs_ij D_kj
// k_theta_prep evaluates D once per (k, j) (N m transcendentals instead of n N m) and its row sums.
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_theta_prep(const double* __restrict__ fstar, double* __restrict__ D, int64_t ld,
                                                    int N, int m, double* __restrict__ partial, int n_chunks,
                                                    const double* __restrict__ sp) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x, chunk = blockIdx.y;
    if (k >= N) return;
    const int per = (int)ceil_div(m, n_chunks), j0 = chunk * per, j1 = min(m, j0 + per);
    double acc = 0.0;
#pragma unroll 4   // four independent evaluations in flight; the sum keeps its order
    for (int j = j0; j < j1; ++j) {
        const double v = fstar[k + (int64_t)j * ld];
        const double a = fabs(v);
        const double d = 0.5 * a + sp_h(sp, a);   // log(2 cosh(v/2)) = |v|/2 + log(1 + exp(-|v|))
        D[k + (int64_t)j * ld] = d;
        acc += d;
    }
    partial[(int64_t)chunk * N + k] = acc;
}
__global__ void k_reduce_partials(const double* __restrict__ partial, int N, int n_chunks, double* __restrict__ rowsum) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= N) return;
    double acc = 0.0;
    for (int c = 0; c < n_chunks; ++c) acc += partial[(int64_t)c * N + k];
    rowsum[k] = acc;
}
int launch_theta_prep(cudaStream_t st, const double* fstar, double* D, int64_t ld, int N, int m, double* partial,
                      int n_chunks, double* rowsum) {
    dim3 grid((unsigned)ceil_div(N, 128), (unsigned)n_chunks);
    const double* sp = nullptr;
    GP_TRY(softplus_table(&sp));
    GP_LAUNCH(k_theta_prep, grid, 128, 0, st, fstar, D, ld, N, m, partial, n_chunks, sp);
    GP_LAUNCH(k_reduce_partials, (unsigned)ceil_div(N, 128), 128, 0, st, partial, N, n_chunks, rowsum);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

// One CTA (256 threads x 4 consecutive grid points) per respondent: P = exp(logP - max), inclusive scan,
// (P - P_0) / (P_last - P_0) > u  -> first such grid index  (draw-theta.cpp:21-34).
constexpr int TH_THREADS = 256, TH_EPT = 4;
static_assert(TH_THREADS * TH_EPT >= N_GRID, "theta draw CTA must cover the grid");
__global__ void __launch_bounds__(TH_THREADS) k_theta_draw(const double* __restrict__ logPt, int64_t ld,
                                                           const double* __restrict__ rowsum, const double* __restrict__ prior,
                                                           const double* __restrict__ theta_star, int N, RngKey key,
                                                           double* __restrict__ theta, int* __restrict__ idx_out,
                                                           int* __restrict__ n_degenerate) {
    __shared__ double red[32];
    __shared__ double s_first;
    __shared__ int s_idx[32];
    const int i = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const double* col = logPt + (int64_t)i * ld;
    double v[TH_EPT];
    double mx = -INFINITY;
#pragma unroll
    for (int e = 0; e < TH_EPT; ++e) {
        const int k = tid * TH_EPT + e;
        v[e] = (k < N) ? prior[k] + (col[k] - (rowsum ? rowsum[k] : 0.0)) : -INFINITY;
        mx = fmax(mx, v[e]);
    }
    mx = warp_max(mx);
    if (lane == 0) red[w] = mx;
    __syncthreads();
    mx = red[0];
    for (int q = 1; q < TH_THREADS / 32; ++q) mx = fmax(mx, red[q]);
    __syncthreads();
    // local inclusive cumsum
    double run = 0.0;
#pragma unroll
    for (int e = 0; e < TH_EPT; ++e) {
        const int k = tid * TH_EPT + e;
        const double p = (k < N) ? exp(v[e] - mx) : 0.0;
        run += p;
        v[e] = run;
    }
    // exclusive scan of thread totals: warp scan then warp totals
    double incl = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) red[w] = incl;
    if (tid == 0) s_first = v[0];
    __syncthreads();
    double woff = 0.0, total = 0.0;
    for (int q = 0; q < TH_THREADS / 32; ++q) { if (q < w) woff += red[q]; total += red[q]; }
    const double offset = woff + (incl - run);
    const double p_min = s_first, denom = total - p_min;                              // cumsum is monotone: min = first, max = last
    const double u = rng_uniform(key, P_THETA_U, (uint32_t)i, 0u);
    int best = 0x7fffffff;
#pragma unroll
    for (int e = TH_EPT - 1; e >= 0; --e) {
        const int k = tid * TH_EPT + e;
        const double cdf = ((offset + v[e]) - p_min) / denom;
        if (k < N && cdf > u) best = k;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) best = min(best, __shfl_xor_sync(0xffffffffu, best, o));
    if (lane == 0) s_idx[w] = best;
    __syncthreads();
    if (tid == 0) {
        for (int q = 1; q < TH_THREADS / 32; ++q) best = min(best, s_idx[q]);
        if (best == 0x7fffffff) {  // degenerate CDF (all mass on grid point 0 => 0/0): the reference reads out of bounds here
            best = 0;
            atomicAdd(n_degenerate, 1);
        }
        theta[i] = theta_star[best];
        if (idx_out) idx_out[i] = best;
    }
}
int launch_theta_draw(cudaStream_t st, const double* logPt, int64_t ld, const double* rowsum_or_null,
                      const double* prior, const double* theta_star, int n, int N, RngKey key, double* theta,
                      int* idx, int* n_degenerate) {
    GP_LAUNCH(k_theta_draw, (unsigned)n, TH_THREADS, 0, st, logPt, ld, rowsum_or_null, prior, theta_star, N, key, theta,
              idx, n_degenerate);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// beta Metropolis step, one CTA per item (reference src/draw-beta.cpp:16-38)
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double dnorm_log(double x, double mu, double sd) {  // R::dnorm(x, mu, sd, log = 1)
    const double t = fabs((x - mu) / sd);
    return -(0.918938533204672741780329736406 + 0.5 * t * t + log(sd));
}

// One item's Metropolis step for the two mean coefficients (draw-beta.cpp:16-38).
//   eval(p0, p1, c0, c1, with_c, part_p, part_c): this thread's partials of ll_bar(f, y, X (p0,p1)^T) and, if with_c,
//   of ll_bar(f, y, X (c0,c1)^T), evaluated in one pass over its cells.
// The reference recomputes ll_bar(f, y, X cv) for k = 1 (:28); it is the value kept from k = 0 (same inputs, same bits).
template <class Eval>
__device__ __forceinline__ void beta_item(const RngKey& key, uint32_t item, int j, double* __restrict__ beta,
                                          const double* __restrict__ pm, const double* __restrict__ psd,
                                          const double* __restrict__ pstep, double (*red)[32], Eval&& eval) {
    double cv[2] = {beta[2 * j], beta[2 * j + 1]};
    double pv[2] = {cv[0], cv[1]};
    double cv_ll = 0.0;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const double z = rng_normal(key, P_BETA_Z, item, (uint32_t)k);
        pv[k] = __dadd_rn(cv[k], __dmul_rn(pstep[2 * j + k], z));                   // :22
        const double pv_prior = dnorm_log(pv[k], pm[2 * j + k], psd[2 * j + k]);    // :25
        const double cv_prior = dnorm_log(cv[k], pm[2 * j + k], psd[2 * j + k]);    // :26
        double part_p = 0.0, part_c = 0.0;
        eval(pv[0], pv[1], cv[0], cv[1], k == 0, part_p, part_c);                   // :27 (and :28 for k = 0)
        const double pv_ll = block_sum(part_p, red[2 * k]);
        if (k == 0) cv_ll = block_sum(part_c, red[2 * k + 1]);
        const double r = pv_prior + pv_ll - cv_prior - cv_ll;                       // :29
        const double u = rng_uniform(key, P_BETA_U, item, (uint32_t)k);
        if (log(u) < r) { cv[k] = pv[k]; cv_ll = pv_ll; } else pv[k] = cv[k];       // :30-35
    }
    if (threadIdx.x == 0) { beta[2 * j] = cv[0]; beta[2 * j + 1] = cv[1]; }
}

// an item's f, y and the respondents' theta held in registers
template <int EPT> struct BetaRegs {
    double fv[EPT], th[EPT], yv[EPT];
    __device__ __forceinline__ void eval(const double* __restrict__ sp, double p0, double p1, double c0, double c1, bool with_c,
                                         double& part_p, double& part_c) const {
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            part_p -= obs_term(sp, yv[e], yv[e] * (fv[e] + fma(th[e], p1, p0)));
            if (with_c) part_c -= obs_term(sp, yv[e], yv[e] * (fv[e] + fma(th[e], c1, c0)));
        }
    }
};

template <int EPT>
__global__ void __launch_bounds__(512) k_beta(double* __restrict__ beta, const double* __restrict__ f, int64_t ld, const int8_t* __restrict__ y8,
                       int64_t ldy, const double* __restrict__ theta, const double* __restrict__ pm,
                       const double* __restrict__ psd, const double* __restrict__ pstep, int n, RngKey key,
                       uint32_t item_offset, const double* __restrict__ sp) {
    __shared__ double red[4][32];
    const int j = blockIdx.x, tid = threadIdx.x, T = blockDim.x;
    BetaRegs<EPT> it;
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
        const int i = tid + e * T;
        if (i < n) { it.fv[e] = f[i + (int64_t)j * ld]; it.th[e] = theta[i]; it.yv[e] = (double)y8[i + (int64_t)j * ldy]; }
        else { it.fv[e] = it.th[e] = it.yv[e] = 0.0; }
    }
    beta_item(key, item_offset + (uint32_t)j, j, beta, pm, psd, pstep, red,
              [&](double p0, double p1, double c0, double c1, bool wc, double& pp, double& pc) { it.eval(sp, p0, p1, c0, c1, wc, pp, pc); });
}

// persistent shape of the beta step (see k_ess_persist): next item's f and y columns prefetched, theta read once
template <int EPT>
__global__ void __launch_bounds__(512) k_beta_persist(double* __restrict__ beta, const double* __restrict__ f, int64_t ld,
                                                       const int8_t* __restrict__ y8, int64_t ldy, const double* __restrict__ theta,
                                                       const double* __restrict__ pm, const double* __restrict__ psd,
                                                       const double* __restrict__ pstep, int n, int m, RngKey key,
                                                       uint32_t item_offset, const double* __restrict__ sp, int* __restrict__ work) {
    extern __shared__ __align__(16) unsigned char dsm[];
    __shared__ double red[4][32];
    __shared__ int s_next;
    const int tid = threadIdx.x, T = blockDim.x, NP = EPT * T;
    double* fbuf = reinterpret_cast<double*>(dsm);
    int8_t* ybuf = reinterpret_cast<int8_t*>(fbuf + 2 * NP);
    BetaRegs<EPT> it;
#pragma unroll
    for (int e = 0; e < EPT; ++e) { const int i = tid + e * T; it.th[e] = (i < n) ? theta[i] : 0.0; }
    auto prefetch = [&](int j, int b) {
        const double* fs = f + (int64_t)j * ld;
        const int8_t* ys = y8 + (int64_t)j * ldy;
        for (int c = tid; c < (n + 1) / 2; c += T) cp_async16(fbuf + b * NP + 2 * c, fs + 2 * c);
        for (int c = tid; c < (n + 15) / 16; c += T) cp_async16(ybuf + b * NP + 16 * c, ys + 16 * c);
        cp_async_commit();
    };
    int j = blockIdx.x, b = 0;
    if (j < m) prefetch(j, 0);
    while (j < m) {
        if (tid == 0) s_next = (int)gridDim.x + atomicAdd(work, 1);
        __syncthreads();
        const int jn = s_next;
        if (jn < m) { prefetch(jn, b ^ 1); cp_async_wait<1>(); } else cp_async_wait<0>();
        __syncthreads();
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            const int i = tid + e * T;
            if (i < n) { it.fv[e] = fbuf[b * NP + i]; it.yv[e] = (double)ybuf[b * NP + i]; }
            else { it.fv[e] = it.yv[e] = 0.0; }
        }
        beta_item(key, item_offset + (uint32_t)j, j, beta, pm, psd, pstep, red,
                  [&](double p0, double p1, double c0, double c1, bool wc, double& pp, double& pc) { it.eval(sp, p0, p1, c0, c1, wc, pp, pc); });
        j = jn;
        b ^= 1;
    }
}

__global__ void __launch_bounds__(1024) k_beta_stream(double* __restrict__ beta, const double* __restrict__ f, int64_t ld,
                                                      const int8_t* __restrict__ y8, int64_t ldy,
                                                      const double* __restrict__ theta, const double* __restrict__ pm,
                                                      const double* __restrict__ psd, const double* __restrict__ pstep,
                                                      int n, RngKey key, uint32_t item_offset,
                                                      const double* __restrict__ sp) {
    __shared__ double red[4][32];
    const int j = blockIdx.x, tid = threadIdx.x, T = blockDim.x;
    const double* fj = f + (int64_t)j * ld;
    const int8_t* yj = y8 + (int64_t)j * ldy;
    beta_item(key, item_offset + (uint32_t)j, j, beta, pm, psd, pstep, red,
              [&](double p0, double p1, double c0, double c1, bool wc, double& pp, double& pc) {
#pragma unroll 4
                  for (int i = tid; i < n; i += T) {
                      const double yv = (double)yj[i], fi = fj[i], ti = theta[i];
                      pp -= obs_term(sp, yv, yv * (fi + fma(ti, p1, p0)));
                      if (wc) pc -= obs_term(sp, yv, yv * (fi + fma(ti, c1, c0)));
                  }
              });
}

#define BETA_PERSIST_CASE(E)                                                                                                 \
    {                                                                                                                            \
        const size_t smem = (size_t)2 * (E) * threads * 9;                                                                       \
        int grid = 0;                                                                                                            \
        GP_TRY(persistent_grid(k_beta_persist<E>, threads, smem, m, &grid));                                                 \
        if (grid > 0) {                                                                                                          \
            GP_CUDA(cudaMemsetAsync(work, 0, sizeof(int), st));                                                                  \
            GP_LAUNCH((k_beta_persist<E>), grid, threads, smem, st, beta, f, ld, y8, ldy, theta, pm, psd, pstep, n, m, key,  \
                      item_offset, sp, work);                                                                                    \
            launched = true;                                                                                                     \
        }                                                                                                                        \
    }

int launch_beta(cudaStream_t st, double* beta, const double* f, int64_t ld, const int8_t* y8, int64_t ldy,
                const double* theta, const double* pm, const double* psd, const double* pstep, int n, int m,
                RngKey key, uint32_t item_offset, int* status, int* work, int* shape) {
    (void)status;
    if (m <= 0) return GPIRT_B200_OK;
    int ept, threads;
    item_cta_shape(n, ept, threads);
    const double* sp = nullptr;
    GP_TRY(softplus_table(&sp));
    if (work && ept) {
        bool launched = false;
        switch (ept) {
            case 1: BETA_PERSIST_CASE(1) break;
            case 2: BETA_PERSIST_CASE(2) break;
            case 4: BETA_PERSIST_CASE(4) break;
            default: BETA_PERSIST_CASE(8) break;
        }
        GP_CUDA(cudaGetLastError());
        if (launched) { if (shape) *shape = ITEM_SHAPE_PERSISTENT; return GPIRT_B200_OK; }
    }
    if (shape) *shape = ept ? ITEM_SHAPE_CTA : ITEM_SHAPE_STREAM;
    switch (ept) {
        case 1: GP_LAUNCH(k_beta<1>, m, threads, 0, st, beta, f, ld, y8, ldy, theta, pm, psd, pstep, n, key, item_offset, sp); break;
        case 2: GP_LAUNCH(k_beta<2>, m, threads, 0, st, beta, f, ld, y8, ldy, theta, pm, psd, pstep, n, key, item_offset, sp); break;
        case 4: GP_LAUNCH(k_beta<4>, m, threads, 0, st, beta, f, ld, y8, ldy, theta, pm, psd, pstep, n, key, item_offset, sp); break;
        case 8: GP_LAUNCH(k_beta<8>, m, threads, 0, st, beta, f, ld, y8, ldy, theta, pm, psd, pstep, n, key, item_offset, sp); break;
        default: GP_LAUNCH(k_beta_stream, m, threads, 0, st, beta, f, ld, y8, ldy, theta, pm, psd, pstep, n, key, item_offset, sp); break;
    }
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

// ll_bar per column with explicit mu and double y (host-API helper mirroring log-likelihood.cpp:25-37)
__global__ void __launch_bounds__(256) k_ll_bar(const double* __restrict__ f, const double* __restrict__ y,
                                                const double* __restrict__ mu, int n, double* __restrict__ out,
                                                const double* __restrict__ sp) {
    __shared__ double red[32];
    const int j = blockIdx.x;
    double part = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double yi = y[i + (int64_t)j * n];
        if (isnan(yi)) continue;
        const double g = f[i + (int64_t)j * n] + mu[i + (int64_t)j * n];
        part -= ll_term_fast(sp, yi * g);
    }
    const double tot = block_sum(part, red);
    if (threadIdx.x == 0) out[j] = tot;
}
int launch_ll_bar(cudaStream_t st, const double* f, const double* y, const double* mu, int n, int m, double* out) {
    if (m <= 0) return GPIRT_B200_OK;
    const double* sp = nullptr;
    GP_TRY(softplus_table(&sp));
    GP_LAUNCH(k_ll_bar, (unsigned)m, 256, 0, st, f, y, mu, n, out, sp);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

}  // namespace gpirt

// ------------------------------------------------------------------------------------------------------------------
// Response coding on the device (reference R/response_matrix.R:79-98, numeric codes): yea -> +1, nay -> -1, everything
// else (missing codes, NA, codes nobody listed) -> NA, later rules winning on overlapping codes (yea, then nay, then
// missing, as the reference assigns them).  One CTA per item; it also reports whether the item is unanimous
// (length(unique(na.omit(x))) == 1: exactly one of {+1, -1} occurs) and how many cells had no code at all.
// ------------------------------------------------------------------------------------------------------------------
namespace gpirt {

__global__ void __launch_bounds__(256) k_response_code(const double* __restrict__ codes, int n, const double* __restrict__ yea,
                                                       int n_yea, const double* __restrict__ nay, int n_nay,
                                                       const double* __restrict__ mis, int n_mis, double* __restrict__ y,
                                                       int* __restrict__ unanimous, unsigned long long* __restrict__ n_uncoded) {
    __shared__ int s_flags;
    const int j = blockIdx.x;
    if (threadIdx.x == 0) s_flags = 0;
    __syncthreads();
    int flags = 0;
    unsigned long long uncoded = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double v = codes[i + (int64_t)j * n];
        double out = nan("");
        bool known = isnan(v);                         // NA is always missing
        for (int k = 0; k < n_yea; ++k) if (v == yea[k]) { out = 1.0; known = true; }
        for (int k = 0; k < n_nay; ++k) if (v == nay[k]) { out = -1.0; known = true; }
        for (int k = 0; k < n_mis; ++k) if (v == mis[k]) { out = nan(""); known = true; }
        if (!known) ++uncoded;
        if (out == 1.0) flags |= 1; else if (out == -1.0) flags |= 2;
        y[i + (int64_t)j * n] = out;
    }
    if (flags) atomicOr(&s_flags, flags);
    if (uncoded) atomicAdd(n_uncoded, uncoded);
    __syncthreads();
    if (threadIdx.x == 0) unanimous[j] = (s_flags == 1 || s_flags == 2) ? 1 : 0;
}
// compaction of the kept items: out[:, c] = y[:, kept[c]]
__global__ void __launch_bounds__(256) k_gather_columns(const double* __restrict__ y, int n, const int64_t* __restrict__ kept,
                                                        double* __restrict__ out) {
    const int i = blockIdx.y * blockDim.x + threadIdx.x, c = blockIdx.x;
    if (i < n) out[i + (int64_t)c * n] = y[i + kept[c] * (int64_t)n];
}

int launch_response_code(cudaStream_t st, const double* codes, int n, int m, const double* yea, int n_yea, const double* nay,
                         int n_nay, const double* mis, int n_mis, double* y, int* unanimous, unsigned long long* n_uncoded) {
    if (n <= 0 || m <= 0) return GPIRT_B200_OK;
    GP_LAUNCH(k_response_code, (unsigned)m, 256, 0, st, codes, n, yea, n_yea, nay, n_nay, mis, n_mis, y, unanimous, n_uncoded);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}
int launch_gather_columns(cudaStream_t st, const double* y, int n, const int64_t* kept, int m_kept, double* out) {
    if (n <= 0 || m_kept <= 0) return GPIRT_B200_OK;
    dim3 grid((unsigned)m_kept, (unsigned)ceil_div(n, 256));
    GP_LAUNCH(k_gather_columns, grid, 256, 0, st, y, n, kept, out);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// Posterior predictive summaries (opts.fit).  Per cell and sampling iteration, with g = f + beta0 + beta1 theta and the
// scoring orientation yt (y where observed, the held-out value where given, +1 otherwise):
//   acc[0] += sigma(yt g)      acc[1], acc[2] = Welford mean / M2 of l = log sigma(yt g)
// Orienting the sum by yt keeps log(mean sigma) accurate in badly predicted cells (tiny mean likelihood); pred for a
// yt = -1 cell is then 1 - mean sigma(-g), accurate in absolute terms.  HBM-bound: 57 bytes per cell and iteration.
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_predictive_code(const int8_t* __restrict__ y8, int64_t ldy8,
                                                         const double* __restrict__ y_holdout, int n,
                                                         int8_t* __restrict__ code, unsigned long long* n_bad) {
    const int i = blockIdx.y * blockDim.x + threadIdx.x, j = blockIdx.x;
    if (i >= n) return;
    int8_t c = y8[i + (int64_t)j * ldy8];
    if (c == 0 && y_holdout) {                                   // held-out values are read where y is NA only
        const double v = y_holdout[i + (int64_t)j * n];
        if (v == 1.0) c = PRED_HOLDOUT;
        else if (v == -1.0) c = -PRED_HOLDOUT;
        else if (!isnan(v)) atomicAdd(n_bad, 1ull);
    }
    code[i + (int64_t)j * ldy8] = c;
}
int launch_predictive_code(cudaStream_t st, const int8_t* y8, int64_t ldy8, const double* y_holdout, int n, int m,
                           int8_t* code, unsigned long long* n_bad) {
    dim3 grid((unsigned)m, (unsigned)ceil_div(n, 256));
    GP_LAUNCH(k_predictive_code, grid, 256, 0, st, y8, ldy8, y_holdout, n, code, n_bad);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

// sigma(a) and log sigma(a) from one exp and one log1p, both stable for either sign of a
__device__ __forceinline__ void log_sigmoid(double a, double& sig, double& ls) {
    const double e = exp(-fabs(a));
    sig = (a >= 0.0 ? 1.0 : e) / (1.0 + e);
    ls = -(fmax(-a, 0.0) + log1p(e));
}
__device__ __forceinline__ void predictive_update(double g, int8_t c, double count, double& s, double& mu, double& q) {
    double sig, ls;
    log_sigmoid(c < 0 ? -g : g, sig, ls);
    if (count == 1.0) { s = sig; mu = ls; q = 0.0; return; }   // first sampling iteration: no memset of the accumulators
    s += sig;
    const double d = ls - mu;
    mu += d / count;
    q = fma(d, ls - mu, q);
}
// one thread = two consecutive respondents of one item (16-byte loads and stores; ld even, code pitch a multiple of 16)
__global__ void __launch_bounds__(256) k_predictive_accumulate(const double* __restrict__ f, int64_t ld,
                                                               const int8_t* __restrict__ code, int64_t ldc,
                                                               const double* __restrict__ theta,
                                                               const double* __restrict__ beta, int n, double count,
                                                               double* __restrict__ acc, size_t plane) {
    const int i0 = 2 * (blockIdx.y * blockDim.x + threadIdx.x), j = blockIdx.x;
    if (i0 >= n) return;
    const double b0 = __ldg(beta + 2 * j), b1 = __ldg(beta + 2 * j + 1);
    const int64_t o = i0 + (int64_t)j * ld;
    double* s = acc + o;
    double* mu = acc + plane + o;
    double* q = acc + 2 * plane + o;
    if (i0 + 1 < n) {
        const double2 fv = *reinterpret_cast<const double2*>(f + o);
        const double2 th = __ldg(reinterpret_cast<const double2*>(theta + i0));
        const char2 cv = *reinterpret_cast<const char2*>(code + i0 + (int64_t)j * ldc);
        double2 sv = make_double2(0.0, 0.0), mv = sv, qv = sv;
        if (count != 1.0) {
            sv = *reinterpret_cast<const double2*>(s);
            mv = *reinterpret_cast<const double2*>(mu);
            qv = *reinterpret_cast<const double2*>(q);
        }
        predictive_update(fv.x + fma(th.x, b1, b0), cv.x, count, sv.x, mv.x, qv.x);
        predictive_update(fv.y + fma(th.y, b1, b0), cv.y, count, sv.y, mv.y, qv.y);
        *reinterpret_cast<double2*>(s) = sv;
        *reinterpret_cast<double2*>(mu) = mv;
        *reinterpret_cast<double2*>(q) = qv;
    } else {
        double sv = 0.0, mv = 0.0, qv = 0.0;
        if (count != 1.0) { sv = *s; mv = *mu; qv = *q; }
        predictive_update(f[o] + fma(theta[i0], b1, b0), code[i0 + (int64_t)j * ldc], count, sv, mv, qv);
        *s = sv; *mu = mv; *q = qv;
    }
}
int launch_predictive_accumulate(cudaStream_t st, const double* f, int64_t ld, const int8_t* code, int64_t ldc,
                                 const double* theta, const double* beta, int n, int m, double count, double* acc) {
    if (ld % 2) { set_last_error("predictive accumulation: leading dimension must be even"); return GPIRT_B200_ERR_ARG; }
    dim3 grid((unsigned)m, (unsigned)ceil_div(ceil_div(n, 2), 256));
    GP_LAUNCH(k_predictive_accumulate, grid, 256, 0, st, f, ld, code, ldc, theta, beta, n, count, acc, (size_t)ld * m);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

// the per-cell outputs of one finished cell: lpd = log(mean sigma(yt g)), pwaic = var_s(l) with denominator S - 1
__device__ __forceinline__ void predictive_cell(const double* acc, size_t plane, int64_t o, double S, double& lpd, double& pw) {
    lpd = log(acc[o] / S);
    pw = acc[2 * plane + o] / (S - 1.0);   // S = 1: 0 / 0 = NaN
}
__global__ void __launch_bounds__(256) k_predictive_cells(const double* __restrict__ acc, int64_t ld, size_t plane,
                                                          const int8_t* __restrict__ code, int64_t ldc, int n, double S,
                                                          int which, double* __restrict__ out) {
    const int i = blockIdx.y * blockDim.x + threadIdx.x, j = blockIdx.x;
    if (i >= n) return;
    const int64_t o = i + (int64_t)j * ld;
    const int c = code[i + (int64_t)j * ldc];
    double lpd, pw, v;
    predictive_cell(acc, plane, o, S, lpd, pw);
    if (which == PRED_OUT_PRED) {
        const double p = acc[o] / S;
        v = c < 0 ? 1.0 - p : p;
    } else if (which == PRED_OUT_LPD) {
        v = c != 0 ? lpd : nan("");
    } else {
        v = (c == 1 || c == -1) ? pw : nan("");
    }
    out[i + (int64_t)j * n] = v;
}
int launch_predictive_cells(cudaStream_t st, const double* acc, int64_t ld, const int8_t* code, int64_t ldc, int n, int m,
                            double S, int which, double* out) {
    dim3 grid((unsigned)m, (unsigned)ceil_div(n, 256));
    GP_LAUNCH(k_predictive_cells, grid, 256, 0, st, acc, ld, (size_t)ld * m, code, ldc, n, S, which, out);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

// per item, one CTA, fixed order: stats[k * m + j] for k = lppd, p_waic, elpd, elpd^2, lpd_holdout, n_obs, n_holdout
__global__ void __launch_bounds__(256) k_predictive_items(const double* __restrict__ acc, int64_t ld, size_t plane,
                                                          const int8_t* __restrict__ code, int64_t ldc, int n, int m,
                                                          double S, double* __restrict__ stats) {
    __shared__ double red[2][32];
    const int j = blockIdx.x;
    double v[PRED_STATS] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int c = code[i + (int64_t)j * ldc];
        if (c == 0) continue;
        double lpd, pw;
        predictive_cell(acc, plane, i + (int64_t)j * ld, S, lpd, pw);
        if (c == 1 || c == -1) {
            const double e = lpd - pw;
            v[0] += lpd; v[1] += pw; v[2] += e; v[3] += e * e; v[5] += 1.0;
        } else {
            v[4] += lpd; v[6] += 1.0;
        }
    }
#pragma unroll
    for (int k = 0; k < PRED_STATS; ++k) {
        const double t = block_sum(v[k], red[k & 1]);
        if (threadIdx.x == 0) stats[(int64_t)k * m + j] = t;
    }
}
// per respondent: partial[c * n + i] = sum of the elpd of the observed cells of item chunk c (then k_reduce_partials)
__global__ void __launch_bounds__(128) k_predictive_resp(const double* __restrict__ acc, int64_t ld, size_t plane,
                                                         const int8_t* __restrict__ code, int64_t ldc, int n, int m,
                                                         double S, double* __restrict__ partial, int n_chunks) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, chunk = blockIdx.y;
    if (i >= n) return;
    const int per = (int)ceil_div(m, n_chunks), j0 = chunk * per, j1 = min(m, j0 + per);
    double t = 0.0;
    for (int j = j0; j < j1; ++j) {
        const int c = code[i + (int64_t)j * ldc];
        if (c != 1 && c != -1) continue;
        double lpd, pw;
        predictive_cell(acc, plane, i + (int64_t)j * ld, S, lpd, pw);
        t += lpd - pw;
    }
    partial[(int64_t)chunk * n + i] = t;
}
// totals[k] = sum over items of stats[k * m + j], one CTA per statistic, fixed order
__global__ void __launch_bounds__(256) k_predictive_totals(const double* __restrict__ stats, int m, double* __restrict__ totals) {
    __shared__ double red[32];
    const int k = blockIdx.x;
    double t = 0.0;
    for (int j = threadIdx.x; j < m; j += blockDim.x) t += stats[(int64_t)k * m + j];
    t = block_sum(t, red);
    if (threadIdx.x == 0) totals[k] = t;
}
int launch_predictive_reduce(cudaStream_t st, const double* acc, int64_t ld, const int8_t* code, int64_t ldc, int n, int m,
                             double S, double* stats, double* partial, int n_chunks, double* resp_totals) {
    const size_t plane = (size_t)ld * m;
    GP_LAUNCH(k_predictive_items, (unsigned)m, 256, 0, st, acc, ld, plane, code, ldc, n, m, S, stats);
    dim3 grid((unsigned)ceil_div(n, 128), (unsigned)n_chunks);
    GP_LAUNCH(k_predictive_resp, grid, 128, 0, st, acc, ld, plane, code, ldc, n, m, S, partial, n_chunks);
    GP_LAUNCH(k_reduce_partials, (unsigned)ceil_div(n, 128), 128, 0, st, partial, n, n_chunks, resp_totals);
    GP_LAUNCH(k_predictive_totals, (unsigned)PRED_STATS, 256, 0, st, stats, m, resp_totals + n);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// IRF posterior summaries (opts.irf).  One thread per grid cell, cells contiguous in k.  Per draw: the Welford mean / M2
// of P = plogis(f*) and two bounded heaps per cell that end up holding exactly the order statistics the bands need — a
// max-heap of the K_lo smallest f* and a min-heap of the K_hi largest, stored slot-major so that a warp's root reads are
// one coalesced load.  Once a heap is full most draws only compare against its root; the rare insertion sifts down.
// ------------------------------------------------------------------------------------------------------------------
IrfBandPlan irf_band_plan(int S, double band) {
    IrfBandPlan p;
    if (S <= 0) return p;
    const double q_lo = (1.0 - band) / 2.0, q_hi = (1.0 + band) / 2.0;
    const double h_lo = (double)(S - 1) * q_lo, h_hi = (double)(S - 1) * q_hi;
    const int r_lo = std::min(S - 1, (int)std::floor(h_lo)), r_hi = std::min(S - 1, (int)std::floor(h_hi));
    p.tlo = h_lo - (double)r_lo;
    p.thi = h_hi - (double)r_hi;
    p.lo_last = r_lo == S - 1;
    p.hi_last = r_hi == S - 1;
    p.klo = std::min(S, r_lo + 2);
    p.khi = S - r_hi;
    return p;
}

// MAXH: max-heap (root = largest kept value); `above(a, b)`: a belongs nearer the root than b
template <bool MAXH>
__device__ __forceinline__ bool heap_above(double a, double b) { return MAXH ? a > b : a < b; }
// adds v to the heap of cell c, which holds `size` values (capacity K): while not full every value goes in (sift up);
// once full v replaces the root only if it belongs strictly below it in the kept tail (sift down)
template <bool MAXH>
__device__ __forceinline__ void heap_add(double* h, int64_t cells, int64_t c, int K, int size, double v) {
    auto at = [&](int i) -> double& { return h[(int64_t)i * cells + c]; };
    if (size < K) {
        int i = size;
        while (i > 0) {
            const int p = (i - 1) >> 1;
            const double pv = at(p);
            if (!heap_above<MAXH>(v, pv)) break;
            at(i) = pv;
            i = p;
        }
        at(i) = v;
        return;
    }
    if (!heap_above<MAXH>(at(0), v)) return;   // v is not inside the kept tail (ties keep the value already there)
    int i = 0;
    for (;;) {
        const int l = 2 * i + 1;
        if (l >= K) break;
        int ci = l;
        double cv = at(l);
        if (l + 1 < K) {
            const double rv = at(l + 1);
            if (heap_above<MAXH>(rv, cv)) { ci = l + 1; cv = rv; }
        }
        if (!heap_above<MAXH>(cv, v)) break;
        at(i) = cv;
        i = ci;
    }
    at(i) = v;
}

__global__ void __launch_bounds__(256) k_irf_accumulate(const double* __restrict__ x, int64_t ld, int rows, int64_t cells,
                                                        int s, double* __restrict__ mean, double* __restrict__ m2,
                                                        double* __restrict__ lo, int klo, double* __restrict__ hi, int khi) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cells) return;
    const int64_t j = c / rows, k = c - j * rows;
    const double v = x[k + j * ld];
    const double p = 1.0 / (1.0 + exp(-v));                    // as k_irf_finish
    if (s == 1) {                                              // first draw: no memset of the accumulators
        mean[c] = p;
        m2[c] = 0.0;
    } else {
        const double mu = mean[c], d = p - mu, mu2 = mu + d / (double)s;
        mean[c] = mu2;
        m2[c] = fma(d, p - mu2, m2[c]);
    }
    if (klo > 0) {
        heap_add<true>(lo, cells, c, klo, min(s - 1, klo), v);
        heap_add<false>(hi, cells, c, khi, min(s - 1, khi), v);
    }
}
int launch_irf_accumulate(cudaStream_t st, const double* x, int64_t ld, int rows, int64_t cells, int s, double* mean,
                          double* m2, double* lo, int klo, double* hi, int khi) {
    if (cells <= 0) return GPIRT_B200_OK;
    GP_LAUNCH(k_irf_accumulate, (unsigned)ceil_div(cells, 256), 256, 0, st, x, ld, rows, cells, s, mean, m2, lo, klo, hi, khi);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

// type-7 quantile from the two order statistics next to it, without contraction (a numpy reference matches it bit for bit)
__device__ __forceinline__ double irf_lerp(double x0, double x1, double t) { return __dadd_rn(x0, __dmul_rn(t, __dsub_rn(x1, x0))); }
// lower, upper and sd_out may alias the inputs of their own cell (each thread reads its cell before it writes it)
__global__ void __launch_bounds__(256) k_irf_finish_bands(int64_t cells, double S, const double* m2, double* sd_out,
                                                          const double* lo, const double* hi, int klo, int khi, int lo_last,
                                                          int hi_last, double tlo, double thi, int plogis, double* lower,
                                                          double* upper) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cells) return;
    if (sd_out) sd_out[c] = sqrt(m2[c] / (S - 1.0));          // S = 1: 0 / 0 = NaN, as R's sd() of one value
    if (!lo) return;
    // lo: max-heap of x_(0..r_lo+1): root = x_(r_lo+1), the larger child = x_(r_lo); hi: min-heap of x_(r_hi..S-1)
    const double l0 = lo[c], h0 = hi[c];
    double ql = l0, qh = h0;
    if (!lo_last) {
        const double l1 = lo[cells + c];
        const double below = klo > 2 ? fmax(l1, lo[2 * cells + c]) : l1;
        ql = irf_lerp(below, l0, tlo);
    }
    if (!hi_last) {
        const double h1 = hi[cells + c];
        const double above = khi > 2 ? fmin(h1, hi[2 * cells + c]) : h1;
        qh = irf_lerp(h0, above, thi);
    }
    if (plogis) {
        ql = 1.0 / (1.0 + exp(-ql));
        qh = 1.0 / (1.0 + exp(-qh));
    }
    lower[c] = ql;
    upper[c] = qh;
}
int launch_irf_finish_bands(cudaStream_t st, int64_t cells, int S, const double* m2, double* sd_out, const double* lo,
                            const double* hi, const IrfBandPlan& p, bool plogis, double* lower, double* upper) {
    if (cells <= 0 || S <= 0) return GPIRT_B200_OK;
    GP_LAUNCH(k_irf_finish_bands, (unsigned)ceil_div(cells, 256), 256, 0, st, cells, (double)S, m2, sd_out, lo, hi, p.klo,
              p.khi, (int)p.lo_last, (int)p.hi_last, p.tlo, p.thi, (int)plogis, lower, upper);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

// ---- convergence diagnostics of several chains (opts.chains) ----
// Sampling iteration t = s - 1 of S belongs to the first half (t < half), the second (t >= S - half) or, for odd S, to
// neither (the middle one); half = S / 2.  Returns the half (-1: none) and the 1-based count within it.
__device__ __forceinline__ int chain_half(int s, int S, int* count) {
    const int t = s - 1, half = S / 2;
    if (t < half) { *count = t + 1; return 0; }
    if (t >= S - half) { *count = t - (S - half) + 1; return 1; }
    return -1;
}
// One thread per grid cell (halves != NULL) and per traced parameter (trace != NULL).  Cells: the Welford mean / M2 of
// P = plogis(f*) of the half this iteration belongs to, planes [mean_0, m2_0, mean_1, m2_1] of `cells`.  Parameters:
// trace[p S + s - 1] = (theta | beta)[p], parameter-major so that the diagnostics read each chain contiguously.
__global__ void __launch_bounds__(256) k_chain_irf_halves(const double* __restrict__ x, int64_t ld, int rows, int64_t cells,
                                                          int s, int S, double* __restrict__ halves,
                                                          const double* __restrict__ theta, int n,
                                                          const double* __restrict__ beta, int nbeta,
                                                          double* __restrict__ trace) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (trace && c < n + nbeta) trace[c * S + (s - 1)] = c < n ? theta[c] : beta[c - n];
    if (!halves || c >= cells) return;
    int cnt = 0;
    const int h = chain_half(s, S, &cnt);
    if (h < 0) return;
    double* mean = halves + (int64_t)(2 * h) * cells;
    double* m2 = mean + cells;
    const int64_t j = c / rows, k = c - j * rows;
    const double p = 1.0 / (1.0 + exp(-x[k + j * ld]));        // as k_irf_accumulate
    if (cnt == 1) {
        mean[c] = p;
        m2[c] = 0.0;
    } else {
        const double mu = mean[c], d = p - mu, mu2 = mu + d / (double)cnt;
        mean[c] = mu2;
        m2[c] = fma(d, p - mu2, m2[c]);
    }
}
int launch_chain_halves(cudaStream_t st, const double* x, int64_t ld, int rows, int64_t cells, int s, int S, double* halves,
                        const double* theta, int n, const double* beta, int nbeta, double* trace) {
    const int64_t work = std::max(halves ? cells : 0, trace ? (int64_t)n + nbeta : 0);
    if (work <= 0) return GPIRT_B200_OK;
    GP_LAUNCH(k_chain_irf_halves, (unsigned)ceil_div(work, 256), 256, 0, st, x, ld, rows, cells, s, S, halves, theta, n, beta,
              nbeta, trace);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

constexpr int DIAG_THREADS = 256, DIAG_WARPS = DIAG_THREADS / 32;
// sum over the CTA of one value per thread, in a fixed order (thread-strided partial sums, shuffle tree, warp partials in
// warp order): bit-identical run to run.  Every thread gets the total.
__device__ __forceinline__ double diag_block_sum(double v, double* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int warp = threadIdx.x >> 5;
    __syncthreads();                                           // red[] free (previous sum read by every thread)
    if ((threadIdx.x & 31) == 0) red[warp] = v;
    __syncthreads();
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < DIAG_WARPS; ++w) t += red[w];
    return t;
}
// One CTA per parameter p, chains in order.  Per chain (S draws at trace + (c P + p) S): the means and sums of squared
// deviations of its two halves, and Geyer's initial monotone sequence ESS over all S draws with autocovariances of
// denominator S.  Warp w computes lag pair k = base + w (lags 2k, 2k + 1), eight pairs per block of lags; thread 0 walks
// them in order and stops at the first non-positive pair.  The formulas of gpirt_b200_theta_diagnostics.
// use_smem: the chain is staged (centred) in S doubles of dynamic shared memory; else it is read from global memory.
__global__ void __launch_bounds__(DIAG_THREADS) k_chain_diag(const double* __restrict__ trace, int P, int S, int C,
                                                             int use_smem, double* __restrict__ rhat, double* __restrict__ ess) {
    extern __shared__ double xs[];
    __shared__ double red[DIAG_WARPS], acv[2 * DIAG_WARPS], means[64];
    __shared__ int done;
    const int p = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int half = S / 2;
    const double T = (double)S;
    double W = 0.0, grand = 0.0, ess_sum = 0.0;               // thread 0's running values
    for (int c = 0; c < C; ++c) {
        const double* x = trace + ((int64_t)c * P + p) * S;
        if (use_smem) {
            __syncthreads();                                   // previous chain's readers are done with xs
            for (int t = tid; t < S; t += DIAG_THREADS) xs[t] = x[t];
            __syncthreads();
        }
        const double* src = use_smem ? xs : x;
        // Every sum runs over values shifted by the first value of their segment: the same statistics as the host's, and
        // exactly zero spread for a constant segment (a sum of S equal values over S need not give the value back).
        for (int h = 0; h < 2; ++h) {
            const double* seg = src + (h ? S - half : 0);
            const double x0 = seg[0];
            double a = 0.0;
            for (int t = tid; t < half; t += DIAG_THREADS) a += seg[t] - x0;
            const double dmu = diag_block_sum(a, red) / (double)half;
            double q = 0.0;
            for (int t = tid; t < half; t += DIAG_THREADS) { const double d = (seg[t] - x0) - dmu; q += d * d; }
            const double v = diag_block_sum(q, red);
            if (tid == 0) {
                const double mu = x0 + dmu;
                W += v / (double)(half - 1);
                means[2 * c + h] = mu;
                grand += mu;
            }
        }
        const double x0 = src[0];
        double a = 0.0;
        for (int t = tid; t < S; t += DIAG_THREADS) a += src[t] - x0;
        const double dmean = diag_block_sum(a, red) / T;
        double sub1 = x0, sub2 = dmean;                        // y_t = (x_t - x0) - dmean
        if (use_smem) {                                        // centre in place
            for (int t = tid; t < S; t += DIAG_THREADS) xs[t] = (xs[t] - x0) - dmean;
            __syncthreads();
            sub1 = sub2 = 0.0;
        }
        double c0 = 0.0, sum = 0.0, prev = INFINITY;
        if (tid == 0) done = 0;
        for (int base = 0;; base += DIAG_WARPS) {
            const int k = base + warp;
            double s0 = 0.0, s1 = 0.0;                         // lags 2k and 2k + 1
            if (2 * k + 1 < S) {
                const int lag = 2 * k;
                for (int t = lane; t + lag < S; t += 32) {
                    const double yt = (src[t] - sub1) - sub2;
                    s0 += yt * ((src[t + lag] - sub1) - sub2);
                    if (t + lag + 1 < S) s1 += yt * ((src[t + lag + 1] - sub1) - sub2);
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    s0 += __shfl_xor_sync(0xffffffffu, s0, o);
                    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
                }
            }
            __syncthreads();                                   // acv[] of the previous block has been read
            if (lane == 0) { acv[2 * warp] = s0 / T; acv[2 * warp + 1] = s1 / T; }
            __syncthreads();
            if (tid == 0) {
                for (int w = 0; w < DIAG_WARPS && !done; ++w) {
                    const int kk = base + w;
                    if (kk == 0) {
                        c0 = acv[0];
                        if (!(c0 > 0.0)) { done = 2; break; }  // constant chain
                    }
                    if (!(2 * kk + 1 < S)) { done = 1; break; }
                    double pair = (acv[2 * w] + acv[2 * w + 1]) / c0;
                    if (pair <= 0.0) { done = 1; break; }
                    pair = fmin(pair, prev);                   // initial monotone sequence
                    prev = pair;
                    sum += pair;
                }
            }
            __syncthreads();
            if (done) break;
        }
        if (tid == 0) {
            const double tau = -1.0 + 2.0 * sum;
            ess_sum += done == 2 ? NAN : T / fmax(tau, 1e-12);
        }
    }
    if (tid == 0) {
        const double M = 2.0 * C;
        W /= M; grand /= M;
        double Bv = 0.0;
        for (int i = 0; i < 2 * C; ++i) Bv += (means[i] - grand) * (means[i] - grand);
        Bv *= (double)half / (M - 1.0);
        const double var_plus = ((double)(half - 1) / (double)half) * W + Bv / (double)half;
        if (rhat) rhat[p] = W > 0.0 ? sqrt(var_plus / W) : NAN;
        if (ess) ess[p] = ess_sum;
    }
}
int chain_diag_smem_bytes(int S) {
    int dev = 0, optin = 0;
    GP_CUDA(cudaGetDevice(&dev));
    GP_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    const size_t fixed = 1024;                                 // the kernel's static shared memory, rounded up
    const size_t want = (size_t)S * sizeof(double);
    return want + fixed <= (size_t)optin ? (int)want : 0;
}
int launch_chain_diag(cudaStream_t st, const double* trace, int P, int S, int C, double* rhat, double* ess) {
    if (P <= 0) return GPIRT_B200_OK;
    if (S < 4 || C < 1 || C > 32) return GPIRT_B200_ERR_ARG;
    const int smem = chain_diag_smem_bytes(S);
    if (smem > 0) GP_CUDA(cudaFuncSetAttribute(k_chain_diag, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    GP_LAUNCH(k_chain_diag, (unsigned)P, DIAG_THREADS, (size_t)smem, st, trace, P, S, C, smem > 0 ? 1 : 0, rhat, ess);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}
// one thread per cell: split-R-hat of P over the 2C half-chain Welford states (chain c's planes at halves + 4 c cells)
__global__ void __launch_bounds__(256) k_chain_irf_rhat(const double* __restrict__ halves, int64_t cells, int S, int C,
                                                        double* __restrict__ rhat) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cells) return;
    const int half = S / 2;
    double W = 0.0, grand = 0.0;
    for (int ch = 0; ch < C; ++ch)
        for (int h = 0; h < 2; ++h) {
            const double* mean = halves + (int64_t)(4 * ch + 2 * h) * cells;
            W += mean[cells + c] / (double)(half - 1);
            grand += mean[c];
        }
    const double M = 2.0 * C;
    W /= M; grand /= M;
    double Bv = 0.0;
    for (int ch = 0; ch < C; ++ch)
        for (int h = 0; h < 2; ++h) {
            const double mu = halves[(int64_t)(4 * ch + 2 * h) * cells + c];
            Bv += (mu - grand) * (mu - grand);
        }
    Bv *= (double)half / (M - 1.0);
    const double var_plus = ((double)(half - 1) / (double)half) * W + Bv / (double)half;
    rhat[c] = W > 0.0 ? sqrt(var_plus / W) : NAN;
}
int launch_chain_irf_rhat(cudaStream_t st, const double* halves, int64_t cells, int S, int C, double* rhat) {
    if (cells <= 0) return GPIRT_B200_OK;
    if (S < 4) return GPIRT_B200_ERR_ARG;
    GP_LAUNCH(k_chain_irf_rhat, (unsigned)ceil_div(cells, 256), 256, 0, st, halves, cells, S, C, rhat);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

}  // namespace gpirt
