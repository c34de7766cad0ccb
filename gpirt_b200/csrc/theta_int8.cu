// theta-step contraction on the 5th-generation tensor cores (tcgen05 / TMEM / TMA), exact integer arithmetic.
//
// The theta step needs  G[k,i] = sum_j f*[k,j] y[i,j]  for 1001 grid points x n respondents over m items
// (reference src/draw-theta.cpp:15-19 in contraction form, see kernels.cu::k_theta_prep).  y is EXACTLY {+1,-1,0}, so it
// is an int8 operand with no error at all.  f* (FP64) is written per grid row k as a 56-bit fixed-point number
//     f*[k,j] = 2^(e_k - 55) X[k,j],   X = sum_{s=0..7} d_s 128^(7-s),  d_s in [-64, 64]  (balanced base-128 digits)
// and each digit plane is an int8 matrix.  Then
//     G[k,i] = 2^(e_k - 6) sum_s 128^(-s) ( sum_j d_s[k,j] y[i,j] )
// where the inner sums are int8 x int8 -> int32 tensor-core products, EXACT (|sum| <= 64 m < 2^31).  The only error is
// the 2^-56 relative truncation of f* — smaller than one FP64 rounding of the result — so the step keeps FP64 accuracy
// while running on tcgen05.mma.kind::i8 instead of the 36.9 TFLOP/s FP64 pipe.
//
// GEMM shape: D[i, c] = sum_j Yt[i, j] Q[c, j],  i < n (M), c = 8 k + s < 8008 (N, padded to 8192), j < m (K, padded
// to 128).  Both operands K-major int8, SWIZZLE_128B tiles staged by TMA; 128 x 256 x 128 CTA tile, 4-stage mbarrier
// ring; one elected thread issues tcgen05.mma (M = 128, N = 256, K = 32), the int32 accumulator lives in TMEM
// (256 columns).  The epilogue warps read TMEM with tcgen05.ld, combine the 8 digit planes of each grid point in
// registers and write the FP64 result straight into logP^T — the int32 products never touch HBM.
#include <mutex>

#include "tcgen05_i8.cuh"
#include "theta_int8.cuh"

namespace gpirt {

namespace {

constexpr int TI_BM = 128, TI_BN = 256, TI_BK = 128, TI_STAGES = 4, TI_UMMA_K = 32;
constexpr int TI_A_BYTES = TI_BM * TI_BK, TI_B_BYTES = TI_BN * TI_BK, TI_STAGE_BYTES = TI_A_BYTES + TI_B_BYTES;
constexpr int TI_SMEM = TI_STAGES * TI_STAGE_BYTES + 1024 /* alignment slack */ + 256 /* barriers */;
constexpr int TI_TMEM_COLS = 256;

using namespace i8tc;
constexpr uint32_t TI_IDESC = idesc_i8(TI_BM, TI_BN);

__global__ void __launch_bounds__(256, 1)
k_igemm_theta(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, int num_kblocks,
              int mtiles, int n_rows, int n_grid, const double* __restrict__ scale, double* __restrict__ logPt,
              int64_t ldP, int accumulate) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);   // SWIZZLE_128B tiles need 1024-byte alignment
    uint64_t* bars = (uint64_t*)(smem + TI_STAGES * TI_STAGE_BYTES);
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + TI_STAGES), tfull = smem_u32(bars + 2 * TI_STAGES);
    uint32_t* tmem_slot = (uint32_t*)(bars + 2 * TI_STAGES + 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int m_tile = blockIdx.x % mtiles, n_tile = blockIdx.x / mtiles;   // CTAs of a wave share few B tiles

    if (warp == 1 && lane == 0) {
        for (int s = 0; s < TI_STAGES; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        mbar_init(tfull, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {   // one warp allocates the accumulator columns in tensor memory
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TI_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ---- TMA producer ----
        if (elect_one())
        for (int kb = 0; kb < num_kblocks; ++kb) {
            const int s = kb % TI_STAGES;
            const uint32_t ph = (uint32_t)(kb / TI_STAGES) & 1u;
            mbar_wait(empty0 + 8 * s, ph ^ 1u);
            mbar_expect_tx(full0 + 8 * s, TI_STAGE_BYTES);
            const uint32_t sa = smem_u32(smem + s * TI_STAGE_BYTES), sb = sa + TI_A_BYTES;
            tma_load_2d(sa, &tmA, kb * TI_BK, m_tile * TI_BM, full0 + 8 * s);
            tma_load_2d(sb, &tmB, kb * TI_BK, n_tile * TI_BN, full0 + 8 * s);
        }
    } else if (warp == 1) {
        if (elect_one()) {
        // ---- MMA issuer: one thread drives the tensor core for the whole CTA ----
        for (int kb = 0; kb < num_kblocks; ++kb) {
            const int s = kb % TI_STAGES;
            const uint32_t ph = (uint32_t)(kb / TI_STAGES) & 1u;
            mbar_wait(full0 + 8 * s, ph);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t sa = smem_u32(smem + s * TI_STAGE_BYTES), sb = sa + TI_A_BYTES;
#pragma unroll
            for (int k4 = 0; k4 < TI_BK / TI_UMMA_K; ++k4)
                umma_i8<TI_IDESC>(tmem_base, umma_desc_sw128(sa + k4 * TI_UMMA_K), umma_desc_sw128(sb + k4 * TI_UMMA_K),
                        (uint32_t)((kb | k4) != 0));
            umma_commit(empty0 + 8 * s);   // frees the shared-memory slot once these MMAs have read it
        }
        umma_commit(tfull);                // accumulator complete
        }
    } else if (warp >= 4) {
        // ---- epilogue: TMEM -> registers, combine the 8 digit planes of each grid point, FP64 store ----
        mbar_wait(tfull, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int q = warp - 4;                                  // TMEM lane quarter this warp may touch (warp % 4)
        const int i = m_tile * TI_BM + q * 32 + lane;            // respondent
        const int kbase = n_tile * (TI_BN / 8);                  // first grid point of this column tile
        const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
        for (int c = 0; c < TI_BN / 16; ++c) {                   // 16 columns = 2 grid points x 8 digits
            uint32_t r[16];
            asm volatile(
                "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                  "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                : "r"(trow + (uint32_t)(c * 16)) : "memory");
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int k = kbase + 2 * c + h;
                double v = (double)(int)r[8 * h + 7];
#pragma unroll
                for (int s = 6; s >= 0; --s) v = fma(v, 0.0078125, (double)(int)r[8 * h + s]);
                if (i < n_rows && k < n_grid) {
                    double* dst = logPt + (int64_t)k + (int64_t)i * ldP;
                    *dst = accumulate ? fma(scale[k], v, *dst) : scale[k] * v;
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 2) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TI_TMEM_COLS) : "memory");
    }
}

// ---- int8 tensor-pipe peak (roofline denominator of the int8 kernels) ---------------------------------------------------
// One CTA per SM; one elected thread issues `iters` x 4 tcgen05.mma.kind::i8 (M128 N256 K32, both operands from shared
// memory in the SWIZZLE_128B layout of the real kernels) back to back into two alternating TMEM accumulators, with no
// loads at all: what the tensor pipe sustains when nothing else limits it.  2 x 128 x 256 x 32 int8 operations per MMA.
__global__ void __launch_bounds__(128, 1) k_peak_umma_i8(int iters, unsigned* sink, int random_operands) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = (uint64_t*)(smem + TI_STAGE_BYTES);
    const uint32_t done = smem_u32(bars);
    uint32_t* tmem_slot = (uint32_t*)(bars + 1);
    const int tid = threadIdx.x, warp = tid >> 5;
    for (int i = tid; i < TI_STAGE_BYTES / 4; i += 128) {
        uint32_t w = 0x01010101u * (uint32_t)(i & 3);   // near-constant operands: the pipe's issue rate at low switching power
        if (random_operands) {                          // digits spread over [-64, 63] like real operand planes
            uint32_t x = (uint32_t)i * 2654435761u + blockIdx.x * 40503u;
            x ^= x >> 15; x *= 2246822519u; x ^= x >> 13; x *= 3266489917u; x ^= x >> 16;
            w = (x & 0x3f3f3f3fu) | (((x >> 6) & 0x01010101u) * 0xc0u);
        }
        ((uint32_t*)smem)[i] = w;
    }
    if (tid == 0) {
        mbar_init(done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy fill above -> async-proxy reads of the MMA
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    if (warp == 0) {
        if (elect_one()) {
            const uint32_t sa = smem_u32(smem), sb = sa + TI_A_BYTES;
            for (int it = 0; it < iters; ++it) {
#pragma unroll
                for (int k4 = 0; k4 < TI_BK / TI_UMMA_K; ++k4)
                    umma_i8<TI_IDESC>(tmem_base + (uint32_t)((it & 1) * TI_TMEM_COLS), umma_desc_sw128(sa + k4 * TI_UMMA_K),
                            umma_desc_sw128(sb + k4 * TI_UMMA_K), (uint32_t)(it > 1 || k4 != 0));
            }
            umma_commit(done);
        }
    }
    mbar_wait(done, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if (warp == 0) {   // read one accumulator word so the products are observable
        uint32_t r;
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r) : "r"(tmem_base) : "memory");
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        if (r == 0xdeadbeefu) sink[blockIdx.x] = r;
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512) : "memory");
}

// ---- operand preparation ----------------------------------------------------------------------------------------------
// Yt[i][j] (int8, row stride m_pad) from y8[i + j ldy] : 64 x 64 byte tiles through shared memory
__global__ void __launch_bounds__(256) k_build_yt(const int8_t* __restrict__ y8, int64_t ldy, int n, int m,
                                                  int8_t* __restrict__ yt, int64_t m_pad, int take_abs) {
    __shared__ int8_t tile[64][65];
    const int i0 = blockIdx.x * 64, j0 = blockIdx.y * 64;
    for (int e = threadIdx.x; e < 64 * 64; e += 256) {
        const int ii = e % 64, jj = e / 64;
        int8_t v = (i0 + ii < n && j0 + jj < m) ? y8[(i0 + ii) + (int64_t)(j0 + jj) * ldy] : (int8_t)0;
        tile[jj][ii] = (take_abs && v < 0) ? (int8_t)(-v) : v;
    }
    __syncthreads();
    for (int e = threadIdx.x; e < 64 * 64; e += 256) {
        const int jj = e % 64, ii = e / 64;
        if (i0 + ii < n && j0 + jj < m) yt[(int64_t)(i0 + ii) * m_pad + j0 + jj] = tile[jj][ii];
    }
}

// per grid row k: partial max_j |f*[k,j]| over a chunk of items
__global__ void __launch_bounds__(128) k_rowabsmax_partial(const double* __restrict__ fstar, int64_t ld, int n_grid, int m,
                                                           double* __restrict__ partial, int n_chunks) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x, chunk = blockIdx.y;
    if (k >= n_grid) return;
    const int per = (int)ceil_div(m, n_chunks), j0 = chunk * per, j1 = min(m, j0 + per);
    double mx = 0.0;
    for (int j = j0; j < j1; ++j) mx = fmax(mx, fabs(fstar[k + (int64_t)j * ld]));
    partial[(int64_t)chunk * n_grid + k] = mx;
}
// e_k = ilogb(max) + 1 ;  qscale[k] = 2^(55 - e_k) (quantiser) ;  oscale[k] = out_factor 2^(e_k - 6) (epilogue)
__global__ void k_rowabsmax_final(const double* __restrict__ partial, int n_grid, int n_chunks, double out_factor,
                                  double* __restrict__ qscale, double* __restrict__ oscale) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_grid) return;
    double mx = 0.0;
    for (int c = 0; c < n_chunks; ++c) mx = fmax(mx, partial[(int64_t)c * n_grid + k]);
    const int e = (mx > 0.0 && isfinite(mx)) ? ilogb(mx) + 1 : 0;
    qscale[k] = scalbn(1.0, 55 - e);
    oscale[k] = out_factor * scalbn(1.0, e - 6);
}

// Q[(8 k + s)][j] = digit s of round(f*[k,j] 2^(55-e_k)) : tile of 32 grid rows x 128 items staged through shared
// memory so that every digit row is written as 128 contiguous bytes
__global__ void __launch_bounds__(256) k_slice_digits(const double* __restrict__ fstar, int64_t ld, int n_grid, int m,
                                                      const double* __restrict__ qscale, int8_t* __restrict__ Q,
                                                      int64_t m_pad) {
    __shared__ __align__(16) int8_t dig[32 * 8][128 + 16];
    const int k0 = blockIdx.x * 32, j0 = blockIdx.y * 128;
    // thread -> grid row kk (fastest: coalesced reads of f*) and a group of 4 consecutive items
    for (int e = threadIdx.x; e < 32 * 32; e += 256) {
        const int kk = e % 32, jq = e / 32;
        const int k = k0 + kk;
        const double qs = (k < n_grid) ? qscale[k] : 0.0;
        unsigned packed[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const int j = j0 + 4 * jq + b;
            long long X = 0;
            if (k < n_grid && j < m) X = __double2ll_rn(fstar[k + (int64_t)j * ld] * qs);
#pragma unroll
            for (int s = 7; s >= 1; --s) {
                const int d = (int)((X + 64) & 127) - 64;   // balanced base-128 digit
                packed[s] |= (unsigned)(d & 0xFF) << (8 * b);
                X = (X - d) >> 7;
            }
            packed[0] |= (unsigned)((int)X & 0xFF) << (8 * b);   // |X| <= 64 here
        }
#pragma unroll
        for (int s = 0; s < 8; ++s) *reinterpret_cast<unsigned*>(&dig[kk * 8 + s][4 * jq]) = packed[s];
    }
    __syncthreads();
    for (int e = threadIdx.x; e < 256 * 32; e += 256) {  // 256 digit rows x 32 words of 4 bytes
        const int w = e % 32, row = e / 32;
        const int k = k0 + row / 8;
        if (k < n_grid && j0 + 4 * w < m_pad)
            *reinterpret_cast<unsigned*>(Q + (int64_t)(k0 * 8 + row) * m_pad + j0 + 4 * w) = *reinterpret_cast<const unsigned*>(&dig[row][4 * w]);
    }
}

}  // namespace

typedef CUresult (*encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                              const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                              CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int i8tc::make_map_k_major(CUtensorMap* map, void* base, uint64_t rows, uint64_t cols, uint64_t row_stride, uint32_t box_rows) {
    static encode_fn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        GP_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres));
        if (!p || qres != cudaDriverEntryPointSuccess) { set_last_error("cuTensorMapEncodeTiled is not available"); return GPIRT_B200_ERR_CUDA; }
        fn = (encode_fn)p;
    }
    const cuuint64_t dims[2] = {cols, rows};
    const cuuint64_t strides[1] = {row_stride};
    const cuuint32_t box[2] = {128u, box_rows};   // 128 bytes: one swizzle span
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_last_error("cuTensorMapEncodeTiled failed (%d)", (int)r); return GPIRT_B200_ERR_CUDA; }
    return GPIRT_B200_OK;
}

struct ThetaInt8::Maps { CUtensorMap a, a_abs, b; };

int ThetaInt8::init(cudaStream_t st, const int8_t* y8, int64_t ldy, int n_, int m_, bool with_observed_mask) {
    n = n_; m = m_;
    m_pad = round_up(m, TI_BK);
    n_pad = round_up(n, TI_BM);
    c_pad = round_up((int64_t)8 * N_GRID, TI_BN);
    GP_TRY(pool_alloc((void**)&yt, (size_t)n_pad * m_pad, st));
    GP_TRY(pool_alloc((void**)&Q, (size_t)c_pad * m_pad, st));
    GP_TRY(pool_alloc((void**)&partial, (size_t)N_CHUNKS * N_GRID * sizeof(double), st));
    GP_TRY(pool_alloc((void**)&qscale, (size_t)N_GRID * sizeof(double), st));
    GP_TRY(pool_alloc((void**)&oscale, (size_t)N_GRID * sizeof(double), st));
    stream_for_free = st;
    GP_CUDA(cudaMemsetAsync(yt, 0, (size_t)n_pad * m_pad, st));
    GP_CUDA(cudaMemsetAsync(Q, 0, (size_t)c_pad * m_pad, st));
    dim3 grid((unsigned)ceil_div(n, 64), (unsigned)ceil_div(m, 64));
    GP_LAUNCH(k_build_yt, grid, 256, 0, st, y8, ldy, n, m, yt, m_pad, 0);
    GP_CUDA(cudaGetLastError());
    maps = new Maps();
    GP_TRY(make_map_k_major(&maps->a, yt, (uint64_t)n_pad, (uint64_t)m_pad, (uint64_t)m_pad, TI_BM));
    if (with_observed_mask) {   // |y| in {0,1}: the observed-cell operand of the second product (missing data)
        GP_TRY(pool_alloc((void**)&yt_abs, (size_t)n_pad * m_pad, st));
        GP_CUDA(cudaMemsetAsync(yt_abs, 0, (size_t)n_pad * m_pad, st));
        GP_LAUNCH(k_build_yt, grid, 256, 0, st, y8, ldy, n, m, yt_abs, m_pad, 1);
        GP_CUDA(cudaGetLastError());
        GP_TRY(make_map_k_major(&maps->a_abs, yt_abs, (uint64_t)n_pad, (uint64_t)m_pad, (uint64_t)m_pad, TI_BM));
    }
    GP_TRY(make_map_k_major(&maps->b, Q, (uint64_t)c_pad, (uint64_t)m_pad, (uint64_t)m_pad, TI_BN));
    GP_CUDA(cudaFuncSetAttribute(k_igemm_theta, cudaFuncAttributeMaxDynamicSharedMemorySize, TI_SMEM));
    ready = true;
    return GPIRT_B200_OK;
}

// logPt[k + i ldP] (+)= out_factor * sum_j src[k,j] y[i,j]     (observed_mask: |y| instead of y)
int ThetaInt8::run(cudaStream_t st, const double* fstar, int64_t ld, double out_factor, double* logPt, int64_t ldP,
                   bool observed_mask, bool accumulate) {
    if (!ready) { set_last_error("ThetaInt8 not initialised"); return GPIRT_B200_ERR_ARG; }
    if (observed_mask && !yt_abs) { set_last_error("ThetaInt8: observed-mask operand was not built"); return GPIRT_B200_ERR_ARG; }
    {
        dim3 grid((unsigned)ceil_div(N_GRID, 128), (unsigned)N_CHUNKS);
        GP_LAUNCH(k_rowabsmax_partial, grid, 128, 0, st, fstar, ld, N_GRID, m, partial, N_CHUNKS);
        GP_LAUNCH(k_rowabsmax_final, (unsigned)ceil_div(N_GRID, 128), 128, 0, st, partial, N_GRID, N_CHUNKS, out_factor, qscale, oscale);
    }
    {
        dim3 grid((unsigned)ceil_div(N_GRID, 32), (unsigned)ceil_div(m, 128));
        GP_LAUNCH(k_slice_digits, grid, 256, 0, st, fstar, ld, N_GRID, m, qscale, Q, m_pad);
    }
    const int mtiles = (int)(n_pad / TI_BM), ntiles = (int)(c_pad / TI_BN);
    GP_LAUNCH(k_igemm_theta, (unsigned)(mtiles * ntiles), 256, TI_SMEM, st, observed_mask ? maps->a_abs : maps->a, maps->b,
              (int)(m_pad / TI_BK), mtiles, n, N_GRID, oscale, logPt, ldP, accumulate ? 1 : 0);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

void ThetaInt8::destroy() {
    for (void* p : {(void*)yt, (void*)yt_abs, (void*)Q, (void*)partial, (void*)qscale, (void*)oscale}) pool_free(p, stream_for_free);
    yt = nullptr; yt_abs = nullptr; Q = nullptr; partial = nullptr; qscale = oscale = nullptr;
    delete maps; maps = nullptr;
    ready = false;
}

int int8_peak_tops(double* tops, int random_operands) {
    int dev = 0, sms = 0;
    GP_CUDA(cudaGetDevice(&dev));
    GP_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int smem = TI_STAGE_BYTES + 1024 + 256, iters = random_operands ? 60000 : 20000;   // long enough for the clocks to settle
    GP_CUDA(cudaFuncSetAttribute(k_peak_umma_i8, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    unsigned* sink = nullptr;
    GP_CUDA(cudaMalloc((void**)&sink, (size_t)sms * sizeof(unsigned)));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    float best = 1e30f;
    cudaError_t err = cudaSuccess;
    for (int r = 0; r < 4 && err == cudaSuccess; ++r) {
        cudaEventRecord(e0);
        GP_LAUNCH(k_peak_umma_i8, (unsigned)sms, 128, smem, 0, iters, sink, random_operands);
        cudaEventRecord(e1);
        err = cudaEventSynchronize(e1);
        float t = 0.f;
        if (err == cudaSuccess && cudaEventElapsedTime(&t, e0, e1) == cudaSuccess && r > 0 && t < best) best = t;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(sink);
    if (err != cudaSuccess) { set_last_error("int8 peak microbenchmark failed: %s", cudaGetErrorString(err)); return GPIRT_B200_ERR_CUDA; }
    // iters x 4 MMAs of 2 x 128 x 256 x 32 operations per SM
    if (tops) *tops = (double)sms * iters * 4.0 * 2.0 * TI_BM * TI_BN * TI_UMMA_K / best * 1e-9;
    return GPIRT_B200_OK;
}

}  // namespace gpirt
