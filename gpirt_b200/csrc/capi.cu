// Single-operation entry points on HOST buffers (each replaces one reference function; the parity tests call these)
// and the FP64 peak microbenchmark used as the tensor-roofline denominator.
#include <vector>
#include <algorithm>
#include <cmath>

#include <climits>

#include "gemm_f64.cuh"
#include "dgemm_i8.cuh"
#include "kernels.cuh"
#include "linalg.cuh"
#include "theta_int8.cuh"

using namespace gpirt;

namespace {

struct DevBuf {
    double* p = nullptr;
    int alloc(size_t count) {
        cudaError_t e = cudaMalloc((void**)&p, (count ? count : 1) * sizeof(double));
        if (e != cudaSuccess) { set_last_error("cudaMalloc: %s", cudaGetErrorString(e)); return GPIRT_B200_ERR_NOMEM; }
        return GPIRT_B200_OK;
    }
    ~DevBuf() { if (p) cudaFree(p); }
};

int have_device() {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
        set_last_error("no CUDA device available (this library has no CPU fallback)");
        return GPIRT_B200_ERR_CUDA;
    }
    return GPIRT_B200_OK;
}

int h2d(double* dst, int64_t ld, const double* src, int64_t lds, int64_t rows, int64_t cols) {
    if (rows == 0 || cols == 0) return GPIRT_B200_OK;
    GP_CUDA(cudaMemcpy2D(dst, ld * sizeof(double), src, lds * sizeof(double), rows * sizeof(double), cols, cudaMemcpyHostToDevice));
    return GPIRT_B200_OK;
}
int d2h(double* dst, int64_t ldd, const double* src, int64_t ld, int64_t rows, int64_t cols) {
    if (rows == 0 || cols == 0) return GPIRT_B200_OK;
    GP_CUDA(cudaMemcpy2D(dst, ldd * sizeof(double), src, ld * sizeof(double), rows * sizeof(double), cols, cudaMemcpyDeviceToHost));
    return GPIRT_B200_OK;
}

__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
__global__ void k_peak_dmma(double* out, int iters, double seed) {
    double c[8][2];
    const double a = seed + threadIdx.x * 1e-9, b = seed * 0.5;
#pragma unroll
    for (int i = 0; i < 8; ++i) { c[i][0] = i; c[i][1] = -i; }
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 8; ++i) dmma(c[i][0], c[i][1], a, b);
    }
    double s = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += c[i][0] + c[i][1];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
__global__ void k_peak_dfma(double* out, int iters, double seed) {
    double c[8];
    const double a = 1.0 + seed * 1e-9, b = seed * 1e-3;
#pragma unroll
    for (int i = 0; i < 8; ++i) c[i] = i + threadIdx.x;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 8; ++i) c[i] = fma(c[i], a, b);
    }
    double s = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += c[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

}  // namespace

extern "C" {

int gpirt_b200_se_cov(const double* x1, int64_t n1, const double* x2, int64_t n2, double jitter, double* out) {
    if (!x1 || !x2 || !out || n1 < 0 || n2 < 0) return GPIRT_B200_ERR_ARG;
    GP_TRY(have_device());
    if (n1 == 0 || n2 == 0) return GPIRT_B200_OK;
    const int64_t ld = round_up(n1, 8);
    DevBuf a, b, o;
    GP_TRY(a.alloc(n1)); GP_TRY(b.alloc(n2)); GP_TRY(o.alloc(ld * n2));
    GP_CUDA(cudaMemcpy(a.p, x1, n1 * sizeof(double), cudaMemcpyHostToDevice));
    GP_CUDA(cudaMemcpy(b.p, x2, n2 * sizeof(double), cudaMemcpyHostToDevice));
    GP_TRY(launch_se_cov(0, a.p, (int)n1, b.p, (int)n2, jitter, false, o.p, ld));
    GP_CUDA(cudaDeviceSynchronize());
    return d2h(out, n1, o.p, ld, n1, n2);
}

int gpirt_b200_chol_lower(double* S, int64_t n) {
    if (!S || n < 0) return GPIRT_B200_ERR_ARG;
    GP_TRY(have_device());
    if (n == 0) return GPIRT_B200_OK;
    const int64_t ld = round_up(n, 8);
    DevBuf a, dinv, flag;   // flag: one double-sized slot used as the int status word
    GP_TRY(a.alloc(ld * n)); GP_TRY(dinv.alloc(ld * CHOL_NB)); GP_TRY(flag.alloc(1));
    int* st = reinterpret_cast<int*>(flag.p);
    GP_CUDA(cudaMemset(st, 0, sizeof(double)));
    GP_CUDA(cudaMemset(dinv.p, 0, (size_t)ld * CHOL_NB * sizeof(double)));   // potrf_lower_rl writes the lower triangles only
    GP_TRY(h2d(a.p, ld, S, n, n, n));
    DevBuf flags;   // one counter per panel step (ints; the buffer is sized in doubles)
    GP_TRY(flags.alloc((size_t)ceil_div(n, CHOL_NB) / 2 + 2));
    int rc = potrf_lower_rl(0, a.p, ld, (int)n, dinv.p, ld, st, reinterpret_cast<int*>(flags.p));
    int h = 0;
    if (rc == GPIRT_B200_OK && cudaMemcpy(&h, st, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) rc = GPIRT_B200_ERR_CUDA;
    if (rc) return rc;
    if (h) { set_last_error("chol(): decomposition failed"); return GPIRT_B200_ERR_NOT_PD; }
    GP_TRY(d2h(S, n, a.p, ld, n, n));
    for (int64_t j = 1; j < n; ++j)      // strict upper := 0, as arma::chol(.,"lower")
        for (int64_t i = 0; i < j; ++i) S[i + j * n] = 0.0;
    return GPIRT_B200_OK;
}

int gpirt_b200_dgemm(int ta, int tb, int64_t M, int64_t N, int64_t K, double alpha, const double* A, int64_t lda,
                     const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int tri) {
    if (!A || !B || !C || M < 0 || N < 0 || K < 0) return GPIRT_B200_ERR_ARG;
    GP_TRY(have_device());
    const int64_t ar = ta ? K : M, ac = ta ? M : K, br = tb ? N : K, bc = tb ? K : N;
    DevBuf a, b, c;
    GP_TRY(a.alloc(lda * ac)); GP_TRY(b.alloc(ldb * bc)); GP_TRY(c.alloc(ldc * N));
    GP_TRY(h2d(a.p, lda, A, lda, ar, ac)); GP_TRY(h2d(b.p, ldb, B, ldb, br, bc)); GP_TRY(h2d(c.p, ldc, C, ldc, M, N));
    GemmArgs g;
    g.M = (int)M; g.N = (int)N; g.K = (int)K; g.A = a.p; g.lda = lda; g.B = b.p; g.ldb = ldb; g.C = c.p; g.ldc = ldc;
    g.alpha = alpha; g.beta = beta; g.tri = tri;
    GP_TRY(gemm_f64(0, ta != 0, tb != 0, g));
    GP_CUDA(cudaDeviceSynchronize());
    return d2h(C, ldc, c.p, ldc, M, N);
}

int gpirt_b200_dgemm_i8(int ta, int a_lower, int64_t M, int64_t N, int64_t K, const double* A, int64_t lda, const double* B,
                        int64_t ldb, double* C, int64_t ldc, int reps, double* ms) {
    if (!A || !B || !C || M < 0 || N < 0 || K < 0 || (ta && a_lower == 1) || (!ta && a_lower == 2) || a_lower < 0 || a_lower > 2)
        return GPIRT_B200_ERR_ARG;
    GP_TRY(have_device());
    if (M == 0 || N == 0) return GPIRT_B200_OK;
    const int64_t ar = ta ? K : M, ac = ta ? M : K;
    DevBuf a, b, c;
    GP_TRY(a.alloc(lda * ac)); GP_TRY(b.alloc(ldb * N)); GP_TRY(c.alloc(ldc * N));
    GP_TRY(h2d(a.p, lda, A, lda, ar, ac)); GP_TRY(h2d(b.p, ldb, B, ldb, K, N));
    GP_CUDA(cudaMemset(c.p, 0, (size_t)ldc * N * sizeof(double)));
    DigitPlanes pa, pb;
    int rc = pa.init(0, (int)M, (int)K, 128);
    if (rc == GPIRT_B200_OK) rc = pb.init(0, (int)N, (int)K, 64);
    cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
    for (auto& e : ev) if (rc == GPIRT_B200_OK && cudaEventCreate(&e) != cudaSuccess) rc = GPIRT_B200_ERR_CUDA;
    const int R = (reps > 0 && ms) ? reps : 1;
    float t_slice = 0.f, t_mm = 0.f;
    if (rc == GPIRT_B200_OK) {
        cudaEventRecord(ev[0], 0);
        for (int it = 0; it < R && rc == GPIRT_B200_OK; ++it) {
            rc = ta ? pa.slice_kcontig(0, a.p, lda) : pa.slice_mcontig(0, a.p, lda, a_lower == 1, 0, (int)K, INT_MIN);
            if (rc == GPIRT_B200_OK) rc = pb.slice_kcontig(0, b.p, ldb);
        }
        cudaEventRecord(ev[1], 0);
        for (int it = 0; it < R && rc == GPIRT_B200_OK; ++it)
            rc = dgemm_i8(0, pa, pb, c.p, ldc, a_lower, 0, (int)K, false, a_lower ? 24 : 18);
        cudaEventRecord(ev[2], 0);
        if (rc == GPIRT_B200_OK && cudaDeviceSynchronize() != cudaSuccess) {
            set_last_error("dgemm_i8 failed: %s", cudaGetErrorString(cudaGetLastError()));
            rc = GPIRT_B200_ERR_CUDA;
        }
        if (rc == GPIRT_B200_OK) { cudaEventElapsedTime(&t_slice, ev[0], ev[1]); cudaEventElapsedTime(&t_mm, ev[1], ev[2]); }
    }
    for (auto& e : ev) if (e) cudaEventDestroy(e);
    pa.destroy(); pb.destroy();
    if (rc) return rc;
    if (ms) { ms[0] = t_mm / R; ms[1] = t_slice / R; }
    return d2h(C, ldc, c.p, ldc, M, N);
}

int gpirt_b200_trsm_lower(int trans, int64_t n, int64_t nrhs, const double* L, double* B) {
    if (!L || !B || n < 0 || nrhs < 0) return GPIRT_B200_ERR_ARG;
    GP_TRY(have_device());
    if (n == 0 || nrhs == 0) return GPIRT_B200_OK;
    const int64_t ld = round_up(n, 8);
    DevBuf l, dinv, b;
    GP_TRY(l.alloc(ld * n)); GP_TRY(dinv.alloc(ld * DIAG_NB)); GP_TRY(b.alloc(ld * nrhs));
    GP_TRY(h2d(l.p, ld, L, n, n, n)); GP_TRY(h2d(b.p, ld, B, n, n, nrhs));
    GP_TRY(trtri_diag_blocks(0, l.p, ld, (int)n, dinv.p, ld));   // inverses of L's 64 x 64 diagonal blocks
    GP_TRY(trsm_left_lower(0, trans != 0, (int)n, (int)nrhs, l.p, ld, dinv.p, ld, b.p, ld));
    GP_CUDA(cudaDeviceSynchronize());
    return d2h(B, n, b.p, ld, n, nrhs);
}

int gpirt_b200_ll_bar(const double* f, const double* y, const double* mu, int64_t n, int64_t m, double* out) {
    if (!f || !y || !mu || !out || n < 0 || m < 0) return GPIRT_B200_ERR_ARG;
    GP_TRY(have_device());
    if (m == 0) return GPIRT_B200_OK;
    DevBuf df, dy, dm, o;
    GP_TRY(df.alloc(n * m)); GP_TRY(dy.alloc(n * m)); GP_TRY(dm.alloc(n * m)); GP_TRY(o.alloc(m));
    GP_CUDA(cudaMemcpy(df.p, f, n * m * sizeof(double), cudaMemcpyHostToDevice));
    GP_CUDA(cudaMemcpy(dy.p, y, n * m * sizeof(double), cudaMemcpyHostToDevice));
    GP_CUDA(cudaMemcpy(dm.p, mu, n * m * sizeof(double), cudaMemcpyHostToDevice));
    GP_TRY(launch_ll_bar(0, df.p, dy.p, dm.p, (int)n, (int)m, o.p));
    GP_CUDA(cudaMemcpy(out, o.p, m * sizeof(double), cudaMemcpyDeviceToHost));
    return GPIRT_B200_OK;
}

int gpirt_b200_fp64_peak_tflops(double* dmma_tflops, double* dfma_tflops) {
    GP_TRY(have_device());
    cudaDeviceProp p;
    GP_CUDA(cudaGetDeviceProperties(&p, 0));
    int dev = 0;
    GP_CUDA(cudaGetDevice(&dev));
    GP_CUDA(cudaGetDeviceProperties(&p, dev));
    const int sms = p.multiProcessorCount, threads = 256, blocks = sms * 2, iters = 20000;
    DevBuf o;
    GP_TRY(o.alloc((size_t)blocks * threads));
    cudaEvent_t e0, e1;
    GP_CUDA(cudaEventCreate(&e0)); GP_CUDA(cudaEventCreate(&e1));
    float best_m = 1e30f, best_f = 1e30f, t;
    for (int r = 0; r < 4; ++r) {
        GP_CUDA(cudaEventRecord(e0)); GP_LAUNCH(k_peak_dmma, blocks, threads, 0, 0, o.p, iters, 1.0); GP_CUDA(cudaEventRecord(e1));
        GP_CUDA(cudaEventSynchronize(e1)); GP_CUDA(cudaEventElapsedTime(&t, e0, e1)); if (r && t < best_m) best_m = t;
        GP_CUDA(cudaEventRecord(e0)); GP_LAUNCH(k_peak_dfma, blocks, threads, 0, 0, o.p, iters, 1.0); GP_CUDA(cudaEventRecord(e1));
        GP_CUDA(cudaEventSynchronize(e1)); GP_CUDA(cudaEventElapsedTime(&t, e0, e1)); if (r && t < best_f) best_f = t;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (dmma_tflops) *dmma_tflops = (double)blocks * (threads / 32) * iters * 8 * 512.0 / best_m * 1e-9;
    if (dfma_tflops) *dfma_tflops = (double)blocks * threads * (double)iters * 8 * 2.0 / best_f * 1e-9;
    return GPIRT_B200_OK;
}

int gpirt_b200_response_matrix(const double* codes, int64_t n, int64_t m, const double* yea, int n_yea, const double* nay,
                               int n_nay, const double* missing, int n_missing, double* y_out, int64_t* kept, int64_t* m_kept,
                               int64_t* n_uncoded) {
    if (!codes || !y_out || !kept || !m_kept || n < 0 || m < 0 || n_yea < 0 || n_nay < 0 || n_missing < 0 ||
        (n_yea && !yea) || (n_nay && !nay) || (n_missing && !missing) || n > INT_MAX || m > INT_MAX)
        return GPIRT_B200_ERR_ARG;
    GP_TRY(have_device());
    *m_kept = 0;
    if (n_uncoded) *n_uncoded = 0;
    if (n == 0 || m == 0) return GPIRT_B200_OK;
    DevBuf dc, dy, dout, dlists, dflags, dkept, dcount;
    GP_TRY(dc.alloc((size_t)n * m)); GP_TRY(dy.alloc((size_t)n * m)); GP_TRY(dlists.alloc((size_t)n_yea + n_nay + n_missing + 1));
    GP_TRY(dflags.alloc((size_t)m / 2 + 1)); GP_TRY(dkept.alloc((size_t)m)); GP_TRY(dcount.alloc(1));
    GP_CUDA(cudaMemcpy(dc.p, codes, (size_t)n * m * sizeof(double), cudaMemcpyHostToDevice));
    if (n_yea) GP_CUDA(cudaMemcpy(dlists.p, yea, n_yea * sizeof(double), cudaMemcpyHostToDevice));
    if (n_nay) GP_CUDA(cudaMemcpy(dlists.p + n_yea, nay, n_nay * sizeof(double), cudaMemcpyHostToDevice));
    if (n_missing) GP_CUDA(cudaMemcpy(dlists.p + n_yea + n_nay, missing, n_missing * sizeof(double), cudaMemcpyHostToDevice));
    GP_CUDA(cudaMemset(dcount.p, 0, sizeof(double)));
    int* flags = reinterpret_cast<int*>(dflags.p);
    GP_TRY(launch_response_code(0, dc.p, (int)n, (int)m, dlists.p, n_yea, dlists.p + n_yea, n_nay, dlists.p + n_yea + n_nay, n_missing,
                                dy.p, flags, reinterpret_cast<unsigned long long*>(dcount.p)));
    std::vector<int> h((size_t)m);
    unsigned long long unc = 0;
    GP_CUDA(cudaMemcpy(h.data(), flags, (size_t)m * sizeof(int), cudaMemcpyDeviceToHost));
    GP_CUDA(cudaMemcpy(&unc, dcount.p, sizeof(unc), cudaMemcpyDeviceToHost));
    if (n_uncoded) *n_uncoded = (int64_t)unc;
    int64_t mk = 0;
    for (int64_t j = 0; j < m; ++j) if (!h[(size_t)j]) kept[mk++] = j;       // unanimous items are discarded (:80-88)
    *m_kept = mk;
    if (mk == 0) return GPIRT_B200_OK;
    GP_TRY(dout.alloc((size_t)n * mk));
    GP_CUDA(cudaMemcpy(dkept.p, kept, (size_t)mk * sizeof(int64_t), cudaMemcpyHostToDevice));
    GP_TRY(launch_gather_columns(0, dy.p, (int)n, reinterpret_cast<const int64_t*>(dkept.p), (int)mk, dout.p));
    GP_CUDA(cudaMemcpy(y_out, dout.p, (size_t)n * mk * sizeof(double), cudaMemcpyDeviceToHost));
    return GPIRT_B200_OK;
}

// Geyer initial-monotone-sequence ESS of one chain (draws x) and the pieces split-R-hat needs
static double chain_ess(const double* x, int64_t T) {
    double mean = 0.0;
    for (int64_t t = 0; t < T; ++t) mean += x[t];
    mean /= (double)T;
    auto acov = [&](int64_t lag) { double a = 0.0; for (int64_t t = 0; t + lag < T; ++t) a += (x[t] - mean) * (x[t + lag] - mean); return a / (double)T; };
    const double c0 = acov(0);
    if (!(c0 > 0.0)) return NAN;                      // constant chain
    double sum = 0.0, prev = INFINITY;
    for (int64_t k = 0; 2 * k + 1 < T; ++k) {
        double pair = (acov(2 * k) + acov(2 * k + 1)) / c0;
        if (pair <= 0.0) break;
        pair = std::min(pair, prev);                  // initial monotone sequence
        prev = pair;
        sum += pair;
    }
    const double tau = -1.0 + 2.0 * sum;
    return (double)T / std::max(tau, 1e-12);
}

int gpirt_b200_theta_diagnostics(const double* theta_draws, int64_t draws, int64_t n, int chains, double* rhat, double* ess) {
    if (!theta_draws || draws < 4 || n < 0 || chains < 1 || (!rhat && !ess)) return GPIRT_B200_ERR_ARG;
    const int64_t half = draws / 2;                   // split-R-hat: every chain contributes its two halves
    std::vector<double> col((size_t)draws);
    for (int64_t i = 0; i < n; ++i) {
        double W = 0.0, grand = 0.0, ess_sum = 0.0;
        std::vector<double> means;
        for (int c = 0; c < chains; ++c) {
            const double* x = theta_draws + (size_t)c * draws * n + (size_t)i * draws;   // chain c: draws x n, column-major
            for (int h = 0; h < 2; ++h) {
                const double* seg = x + (h ? draws - half : 0);
                double mu = 0.0, v = 0.0;
                for (int64_t t = 0; t < half; ++t) mu += seg[t];
                mu /= (double)half;
                for (int64_t t = 0; t < half; ++t) v += (seg[t] - mu) * (seg[t] - mu);
                W += v / (double)(half - 1);
                means.push_back(mu);
                grand += mu;
            }
            if (ess) ess_sum += chain_ess(x, draws);
        }
        const double M = (double)means.size();
        W /= M; grand /= M;
        double Bv = 0.0;
        for (double mu : means) Bv += (mu - grand) * (mu - grand);
        Bv *= (double)half / (M - 1.0);
        const double var_plus = ((double)(half - 1) / (double)half) * W + Bv / (double)half;
        if (rhat) rhat[i] = W > 0.0 ? std::sqrt(var_plus / W) : NAN;
        if (ess) ess[i] = ess_sum;
    }
    return GPIRT_B200_OK;
}

int gpirt_b200_int8_peak_tops(double* tops) {
    GP_TRY(have_device());
    return int8_peak_tops(tops);
}
int gpirt_b200_int8_peak_tops_random(double* tops) {
    GP_TRY(have_device());
    return int8_peak_tops(tops, 1);
}

int gpirt_b200_predictive_accumulate_time(int64_t n, int64_t m, int reps, double* ms_accumulate, double* ms_copy) {
    if (n <= 0 || m <= 0 || n > INT_MAX || m > INT_MAX || reps <= 0 || !ms_accumulate || !ms_copy) return GPIRT_B200_ERR_ARG;
    GP_TRY(have_device());
    const int64_t ld = round_up(n, 8), ldc = round_up(n, 16);
    const size_t acc_doubles = 3 * (size_t)ld * m;
    DevBuf f, acc, copy, theta, beta, code;
    GP_TRY(f.alloc((size_t)ld * m)); GP_TRY(acc.alloc(acc_doubles)); GP_TRY(copy.alloc(acc_doubles));
    GP_TRY(theta.alloc((size_t)ld)); GP_TRY(beta.alloc(2 * (size_t)m)); GP_TRY(code.alloc((size_t)ldc * m / 8 + 1));
    // a sampler-like state: f, theta, beta standard normal, every cell observed (+1)
    const RngKey key{12345u, 678u, 1u, nullptr};
    GP_TRY(launch_fill_normal(0, f.p, (int)n, (int)m, ld, key, 0, 0));
    GP_TRY(launch_fill_normal(0, theta.p, (int)n, 1, ld, key, 1, 0));
    GP_TRY(launch_fill_normal(0, beta.p, 2, (int)m, 2, key, 2, 0));
    int8_t* c8 = reinterpret_cast<int8_t*>(code.p);
    GP_CUDA(cudaMemset(c8, 1, (size_t)ldc * m));
    GP_TRY(launch_predictive_accumulate(0, f.p, ld, c8, ldc, theta.p, beta.p, (int)n, (int)m, 1.0, acc.p));   // count 1 initialises
    GP_CUDA(cudaMemcpyAsync(copy.p, acc.p, acc_doubles * sizeof(double), cudaMemcpyDeviceToDevice, 0));
    cudaEvent_t e[3];
    for (auto& x : e) GP_CUDA(cudaEventCreate(&x));
    int rc = GPIRT_B200_OK;
    cudaEventRecord(e[0], 0);
    for (int r = 0; r < reps && rc == GPIRT_B200_OK; ++r)
        rc = launch_predictive_accumulate(0, f.p, ld, c8, ldc, theta.p, beta.p, (int)n, (int)m, 2.0 + r, acc.p);
    cudaEventRecord(e[1], 0);
    for (int r = 0; r < reps && rc == GPIRT_B200_OK; ++r)   // the same bytes read and written as the accumulator planes
        if (cudaMemcpyAsync(r & 1 ? acc.p : copy.p, r & 1 ? copy.p : acc.p, acc_doubles * sizeof(double), cudaMemcpyDeviceToDevice, 0) != cudaSuccess)
            rc = GPIRT_B200_ERR_CUDA;
    cudaEventRecord(e[2], 0);
    float t_acc = 0.f, t_copy = 0.f;
    if (rc == GPIRT_B200_OK && cudaEventSynchronize(e[2]) != cudaSuccess) {
        set_last_error("predictive accumulation timing failed: %s", cudaGetErrorString(cudaGetLastError()));
        rc = GPIRT_B200_ERR_CUDA;
    }
    if (rc == GPIRT_B200_OK) { cudaEventElapsedTime(&t_acc, e[0], e[1]); cudaEventElapsedTime(&t_copy, e[1], e[2]); }
    for (auto& x : e) cudaEventDestroy(x);
    if (rc) return rc;
    *ms_accumulate = t_acc / reps;
    *ms_copy = t_copy / reps;
    return GPIRT_B200_OK;
}

int gpirt_b200_rng_probe(uint64_t seed, uint32_t sweep, uint32_t purpose, uint32_t stream, uint32_t idx0, int count,
                         double* uniforms, double* normals) {
    if (count < 0 || !uniforms || !normals) return GPIRT_B200_ERR_ARG;
    GP_TRY(have_device());
    if (count == 0) return GPIRT_B200_OK;
    DevBuf u, z;
    GP_TRY(u.alloc(count)); GP_TRY(z.alloc(count));
    RngKey key{(uint32_t)seed, (uint32_t)(seed >> 32), sweep, nullptr};
    GP_TRY(launch_rng_probe(0, key, purpose, stream, idx0, count, u.p, z.p));
    GP_CUDA(cudaMemcpy(uniforms, u.p, count * sizeof(double), cudaMemcpyDeviceToHost));
    GP_CUDA(cudaMemcpy(normals, z.p, count * sizeof(double), cudaMemcpyDeviceToHost));
    return GPIRT_B200_OK;
}

}  // extern "C"
