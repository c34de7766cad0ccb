// Posterior predictive model checks (opts.ppc, definitions in include/gpirt_b200.h).
//
// Per sampling iteration, outside the captured sweep, on the sampler's stream:
//   k_ppc_replicate   y^rep from the end-of-sweep state, the Pearson terms exp(-y g) of y and y^rep per observed cell,
//                     summed per respondent (over PPC_CHUNKS item chunks) and per item (per warp of 64 respondents)
//   k_ppc_items       per item: the warp partials in a fixed order, D_j(y) / D_j(y^rep), item counter
//   k_ppc_resp_glob   per respondent: the chunk partials in a fixed order, respondent counter; one more CTA: the item sums
//                     in a fixed order, global counter
//   k_ppc_pairs       (pair outputs only) the item x item products of y^rep over respondents on the int8 tensor cores;
//                     the epilogue forms the 2 x 2 counts of every pair and compares the odds ratios exactly
// The observed and replicated sums of a discrepancy run through the same reduction tree, so a replicate equal to y gives
// bit-equal sums.  No floating-point atomics anywhere: every run is bit-identical.
#include <algorithm>
#include <vector>

#include "ppc.cuh"
#include "tcgen05_i8.cuh"

namespace gpirt {

namespace {

using namespace i8tc;

// ---- chi-square ---------------------------------------------------------------------------------------------------
// one observed cell: y^rep = +1 if u < p = sigma(g) (else -1), and exp(-y g), exp(-y^rep g) from the one e = exp(-|g|)
__device__ __forceinline__ void ppc_cell(double g, int8_t y, double u, int8_t& r, double& to, double& tr) {
    const double e = exp(-fabs(g));
    const bool pos = g >= 0.0;
    r = (u * (1.0 + e) < (pos ? 1.0 : e)) ? (int8_t)1 : (int8_t)-1;   // u < 1 / (1 + e) resp. e / (1 + e)
    const double inv = 1.0 / e;
    to = ((y > 0) == pos) ? e : inv;
    tr = ((r > 0) == pos) ? e : inv;
}

// grid (ceil(n / 256), PPC_CHUNKS) x 128 threads; a thread = two consecutive respondents (16-byte loads of f: ld even),
// a warp = 64 respondents (warp row wr); items j0..j1 of the CTA's chunk in ascending order
__global__ void __launch_bounds__(128) k_ppc_replicate(const double* __restrict__ f, int64_t ld, const int8_t* __restrict__ y8,
                                                       int64_t ldy8, const double* __restrict__ theta,
                                                       const double* __restrict__ beta, int n, int m, RngKey key,
                                                       uint32_t item_offset, int8_t* __restrict__ yrep,
                                                       double2* __restrict__ wpart, int nwr, double2* __restrict__ rpart) {
    const int i0 = 2 * (blockIdx.x * blockDim.x + threadIdx.x), lane = threadIdx.x & 31;
    const int wr = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int per = (int)ceil_div(m, PPC_CHUNKS), j0 = blockIdx.y * per, j1 = min(m, j0 + per);
    const bool live0 = i0 < n, live1 = i0 + 1 < n;
    const double th0 = live0 ? theta[i0] : 0.0, th1 = live1 ? theta[i0 + 1] : 0.0;
    double so0 = 0.0, sr0 = 0.0, so1 = 0.0, sr1 = 0.0;
    for (int j = j0; j < j1; ++j) {
        const int64_t o = i0 + (int64_t)j * ldy8;
        const char2 c = live0 ? *reinterpret_cast<const char2*>(y8 + o) : make_char2(0, 0);
        double to0 = 0.0, tr0 = 0.0, to1 = 0.0, tr1 = 0.0;
        int8_t r0 = 0, r1 = 0;
        if (c.x != 0 || c.y != 0) {
            const double b0 = __ldg(beta + 2 * j), b1 = __ldg(beta + 2 * j + 1);
            const double2 fv = *reinterpret_cast<const double2*>(f + i0 + (int64_t)j * ld);
            if (c.x != 0) ppc_cell(fv.x + fma(th0, b1, b0), c.x, rng_uniform(key, P_PPC_U, item_offset + j, i0), r0, to0, tr0);
            if (live1 && c.y != 0) ppc_cell(fv.y + fma(th1, b1, b0), c.y, rng_uniform(key, P_PPC_U, item_offset + j, i0 + 1), r1, to1, tr1);
        }
        if (yrep && live0) *reinterpret_cast<char2*>(yrep + o) = make_char2(r0, live1 ? r1 : (int8_t)0);
        so0 += to0; sr0 += tr0; so1 += to1; sr1 += tr1;
        const double wo = warp_sum(to0 + to1), wp = warp_sum(tr0 + tr1);
        if (lane == 0) wpart[(int64_t)j * nwr + wr] = make_double2(wo, wp);
    }
    if (live0) rpart[(int64_t)blockIdx.y * n + i0] = make_double2(so0, sr0);
    if (live1) rpart[(int64_t)blockIdx.y * n + i0 + 1] = make_double2(so1, sr1);
}

// one warp per item: the nwr warp partials in a fixed order
__global__ void __launch_bounds__(256) k_ppc_items(const double2* __restrict__ wpart, int nwr, int m,
                                                   double2* __restrict__ item_d, uint32_t* __restrict__ item_cnt) {
    const int j = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (j >= m) return;
    double o = 0.0, r = 0.0;
    for (int w = lane; w < nwr; w += 32) {
        const double2 v = wpart[(int64_t)j * nwr + w];
        o += v.x; r += v.y;
    }
    o = warp_sum(o); r = warp_sum(r);
    if (lane == 0) {
        item_d[j] = make_double2(o, r);
        item_cnt[j] += r >= o ? 1u : 0u;
    }
}

// CTAs 0 .. ceil(n / 256) - 1: one thread per respondent over the PPC_CHUNKS partials in order; the last CTA: the item
// sums in a fixed order (strided per thread, then the block tree)
__global__ void __launch_bounds__(256) k_ppc_resp_glob(const double2* __restrict__ rpart, int n, const double2* __restrict__ item_d,
                                                       int m, uint32_t* __restrict__ resp_cnt, uint32_t* __restrict__ glob_cnt) {
    __shared__ double red[2][32];
    if (blockIdx.x + 1 < gridDim.x) {
        const int i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= n) return;
        double o = 0.0, r = 0.0;
        for (int c = 0; c < PPC_CHUNKS; ++c) {
            const double2 v = rpart[(int64_t)c * n + i];
            o += v.x; r += v.y;
        }
        resp_cnt[i] += r >= o ? 1u : 0u;
        return;
    }
    double o = 0.0, r = 0.0;
    for (int j = threadIdx.x; j < m; j += blockDim.x) { o += item_d[j].x; r += item_d[j].y; }
    o = block_sum(o, red[0]);
    r = block_sum(r, red[1]);
    if (threadIdx.x == 0) *glob_cnt += r >= o ? 1u : 0u;
}

// observed cells per item and per respondent (integer atomics: order-free); grid (ceil(n / 128), PPC_CHUNKS) x 128
__global__ void __launch_bounds__(128) k_ppc_nobs(const int8_t* __restrict__ y8, int64_t ldy8, int n, int m,
                                                  int* __restrict__ item_nobs, int* __restrict__ resp_nobs) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int per = (int)ceil_div(m, PPC_CHUNKS), j0 = blockIdx.y * per, j1 = min(m, j0 + per);
    int ri = 0;
    for (int j = j0; j < j1; ++j) {
        const int o = (i < n && y8[i + (int64_t)j * ldy8] != 0) ? 1 : 0;
        ri += o;
        const int w = __reduce_add_sync(0xffffffffu, o);
        if ((threadIdx.x & 31) == 0 && w) atomicAdd(item_nobs + j, w);
    }
    if (i < n && ri) atomicAdd(resp_nobs + i, ri);
}

// ---- pairs --------------------------------------------------------------------------------------------------------
// Tile = 128 items (rows of A, the j of a pair) x 128 items (rows of B, the k) over K = respondents in blocks of 128.
// Operands K-major as the planes lie (item-major, respondents contiguous, pitch ldy): y^rep (Y) and, with missing
// cells, the observed mask M = |y|.  Accumulators in TMEM (int32, 128 columns each):
//   P1 = Y_j . Y_k; with missing cells P2 = Y_j . M_k, P3 = M_j . Y_k and, in the observed pass, P4 = M_j . M_k
// (without missing cells P2 / P3 are the column sums of Y and P4 = n).  Then, exactly,
//   n11 = (P4 + P1 + P2 + P3) / 4, n10 = (P4 - P1 + P2 - P3) / 4, n01 = (P4 - P1 - P2 + P3) / 4, n00 = (P4 + P1 - P2 - P3) / 4
// The epilogue owns its tile's entries: entry (r, c) of tile t at t 128^2 + c 128 + r (a warp's lanes take consecutive r).
constexpr int PP_T = 128, PP_BK = 128, PP_UMMA_K = 32, PP_TILE_BYTES = PP_T * PP_BK, PP_TILE_ELEMS = PP_T * PP_T;
constexpr uint32_t PP_IDESC = idesc_i8(PP_T, PP_T);
template <bool MISSING> struct PpCfg {
    static constexpr int OPS = MISSING ? 4 : 2;          // staged tiles per k block: Y_j, Y_k (, M_j, M_k)
    static constexpr int STAGES = MISSING ? 3 : 4;
    static constexpr int STAGE_BYTES = OPS * PP_TILE_BYTES;
    static constexpr int SMEM = STAGES * STAGE_BYTES + 1024 /* alignment slack */ + 256 /* barriers */;
    static constexpr int TMEM_COLS = MISSING ? 512 : 128;
};

// OR(rep) >= OR(obs) with the +1/2 correction, in integers: (2a_r+1)(2d_r+1)(2b_o+1)(2c_o+1) >= (2a_o+1)(2d_o+1)(2b_r+1)(2c_r+1).
// Each factor is at most 2n + 1 < 2^32, so each pair product fits 64 bits and the comparison needs 128.
__device__ __forceinline__ bool ppc_or_at_least(int64_t a, int64_t b, int64_t c, int64_t d, int4 o) {
    const uint64_t xr = (uint64_t)(2 * a + 1) * (uint64_t)(2 * d + 1), yr = (uint64_t)(2 * b + 1) * (uint64_t)(2 * c + 1);
    const uint64_t xo = (uint64_t)(2 * (int64_t)o.x + 1) * (uint64_t)(2 * (int64_t)o.w + 1);
    const uint64_t yo = (uint64_t)(2 * (int64_t)o.y + 1) * (uint64_t)(2 * (int64_t)o.z + 1);
    return (unsigned __int128)xr * yo >= (unsigned __int128)xo * yr;
}

template <bool MISSING>
__global__ void __launch_bounds__(256, 1)
k_ppc_pairs(const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmM, int num_kblocks, int mt, int m,
            int n, const int* __restrict__ colsum, int4* __restrict__ obs, uint32_t* __restrict__ cnt, int observed) {
    using Cfg = PpCfg<MISSING>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);   // SWIZZLE_128B tiles need 1024-byte alignment
    uint64_t* bars = (uint64_t*)(smem + Cfg::STAGES * Cfg::STAGE_BYTES);
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + Cfg::STAGES), tfull = smem_u32(bars + 2 * Cfg::STAGES);
    uint32_t* tmem_slot = (uint32_t*)(bars + 2 * Cfg::STAGES + 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    int t = blockIdx.x, tj = 0;                    // tile (tj, tk), tj <= tk: the upper tile triangle, row by row
    while (t >= mt - tj) { t -= mt - tj; ++tj; }
    const int tk = tj + t;

    if (warp == 1 && lane == 0) {
        for (int s = 0; s < Cfg::STAGES; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        mbar_init(tfull, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(Cfg::TMEM_COLS) : "memory");
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
            const int s = kb % Cfg::STAGES;
            const uint32_t ph = (uint32_t)(kb / Cfg::STAGES) & 1u;
            mbar_wait(empty0 + 8 * s, ph ^ 1u);
            mbar_expect_tx(full0 + 8 * s, Cfg::STAGE_BYTES);
            const uint32_t sa = smem_u32(smem + s * Cfg::STAGE_BYTES);
            tma_load_2d(sa, &tmY, kb * PP_BK, tj * PP_T, full0 + 8 * s);
            tma_load_2d(sa + PP_TILE_BYTES, &tmY, kb * PP_BK, tk * PP_T, full0 + 8 * s);
            if (MISSING) {
                tma_load_2d(sa + 2 * PP_TILE_BYTES, &tmM, kb * PP_BK, tj * PP_T, full0 + 8 * s);
                tma_load_2d(sa + 3 * PP_TILE_BYTES, &tmM, kb * PP_BK, tk * PP_T, full0 + 8 * s);
            }
        }
    } else if (warp == 1) {
        if (elect_one()) {
        // ---- MMA issuer ----
        for (int kb = 0; kb < num_kblocks; ++kb) {
            const int s = kb % Cfg::STAGES;
            const uint32_t ph = (uint32_t)(kb / Cfg::STAGES) & 1u;
            mbar_wait(full0 + 8 * s, ph);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t yj = smem_u32(smem + s * Cfg::STAGE_BYTES), yk = yj + PP_TILE_BYTES;
            const uint32_t mj = yj + 2 * PP_TILE_BYTES, mk = yj + 3 * PP_TILE_BYTES;
#pragma unroll
            for (int k4 = 0; k4 < PP_BK / PP_UMMA_K; ++k4) {
                const uint32_t acc = (uint32_t)((kb | k4) != 0), o = k4 * PP_UMMA_K;
                umma_i8<PP_IDESC>(tmem_base, umma_desc_sw128(yj + o), umma_desc_sw128(yk + o), acc);
                if (MISSING) {
                    umma_i8<PP_IDESC>(tmem_base + 128, umma_desc_sw128(yj + o), umma_desc_sw128(mk + o), acc);
                    umma_i8<PP_IDESC>(tmem_base + 256, umma_desc_sw128(mj + o), umma_desc_sw128(yk + o), acc);
                    if (observed) umma_i8<PP_IDESC>(tmem_base + 384, umma_desc_sw128(mj + o), umma_desc_sw128(mk + o), acc);
                }
            }
            umma_commit(empty0 + 8 * s);
        }
        umma_commit(tfull);
        }
    } else if (warp >= 4) {
        // ---- epilogue: TMEM -> counts -> observed counts (observed pass) or exact comparison + counter update ----
        mbar_wait(tfull, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int q = warp - 4, r = q * 32 + lane, j = tj * PP_T + r;
        const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
        const int64_t tile0 = (int64_t)blockIdx.x * PP_TILE_ELEMS;
        const int cj = (!MISSING && j < m) ? colsum[j] : 0;
#pragma unroll 1
        for (int c = 0; c < PP_T / 16; ++c) {
            uint32_t p1[16], p2[16], p3[16], p4[16];
#define PP_LD16(v, col)                                                                                                        \
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"      \
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),             \
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])         \
                 : "r"(trow + (uint32_t)(col)) : "memory")
            PP_LD16(p1, c * 16);
            if (MISSING) {
                PP_LD16(p2, 128 + c * 16);
                PP_LD16(p3, 256 + c * 16);
                if (observed) PP_LD16(p4, 384 + c * 16);
            }
#undef PP_LD16
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int h = 0; h < 16; ++h) {
                const int cc = c * 16 + h, k = tk * PP_T + cc;
                if (j >= m || k >= m) continue;
                const int64_t e = tile0 + (int64_t)cc * PP_T + r;
                const int64_t P1 = (int)p1[h];
                int64_t P2, P3, P4;
                int4 o = make_int4(0, 0, 0, 0);
                if (!observed) o = obs[e];
                if (MISSING) {
                    P2 = (int)p2[h]; P3 = (int)p3[h];
                    P4 = observed ? (int64_t)(int)p4[h] : (int64_t)o.x + o.y + o.z + o.w;
                } else {
                    P2 = cj; P3 = colsum[k]; P4 = n;
                }
                const int64_t a = (P4 + P1 + P2 + P3) >> 2, b = (P4 - P1 + P2 - P3) >> 2;
                const int64_t cn = (P4 - P1 - P2 + P3) >> 2, d = (P4 + P1 - P2 - P3) >> 2;
                if (observed) obs[e] = make_int4((int)a, (int)b, (int)cn, (int)d);
                else cnt[e] += ppc_or_at_least(a, b, cn, d, o) ? 1u : 0u;
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 2) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(Cfg::TMEM_COLS) : "memory");
    }
}

// column sums of an int8 plane (padding rows are zero): one warp per item, 4 bytes per load
__global__ void __launch_bounds__(256) k_ppc_colsum(const int8_t* __restrict__ plane, int64_t ldy, int m, int* __restrict__ colsum) {
    const int j = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (j >= m) return;
    const int* col = reinterpret_cast<const int*>(plane + (int64_t)j * ldy);
    int s = 0;
    for (int64_t w = lane; w < ldy / 4; w += 32) s = __dp4a(col[w], 0x01010101, s);
    s = __reduce_add_sync(0xffffffffu, s);
    if (lane == 0) colsum[j] = s;
}

// |y8| in {0, 1}: the observed-cell operand
__global__ void __launch_bounds__(256) k_ppc_abs(const int8_t* __restrict__ y8, size_t count, int8_t* __restrict__ mask) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) mask[i] = y8[i] != 0 ? (int8_t)1 : (int8_t)0;
}

// pair (j, k) of the m x m outputs for columns k0 .. k0 + gridDim.y - 1, staged column-major (m rows)
__global__ void __launch_bounds__(256) k_ppc_pairs_finish(const int4* __restrict__ obs, const uint32_t* __restrict__ cnt, int mt,
                                                          int m, int k0, double scale, int all_nan, double* __restrict__ lor,
                                                          double* __restrict__ ppp) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x, k = k0 + blockIdx.y;
    if (j >= m) return;
    int tj = j / PP_T, tk = k / PP_T, r = j % PP_T, c = k % PP_T;
    if (tj > tk) { const int x = tj; tj = tk; tk = x; const int y = r; r = c; c = y; }
    const int64_t t = (int64_t)tj * mt - (int64_t)tj * (tj - 1) / 2 + (tk - tj);
    const int64_t e = t * PP_TILE_ELEMS + (int64_t)c * PP_T + r;
    const int4 o = obs[e];
    const bool none = all_nan || j == k || ((int64_t)o.x + o.y + o.z + o.w) == 0;
    const double v = log(((o.x + 0.5) * (o.w + 0.5)) / ((o.y + 0.5) * (o.z + 0.5)));
    const int64_t out = (int64_t)blockIdx.y * m + j;
    lor[out] = none ? nan("") : v;
    ppp[out] = none ? nan("") : (double)cnt[e] * scale;
}

// caller data -> int8 plane (pitch ldy): without mask, +1 / -1 / NaN -> +1 / -1 / 0 (counts[0] += missing); with mask,
// +1 / -1 where mask != 0 and 0 elsewhere.  counts[1] += cells holding anything else.
__global__ void __launch_bounds__(256) k_ppc_plane(const double* __restrict__ src, int n, int m, const int8_t* __restrict__ mask,
                                                   int8_t* __restrict__ dst, int64_t ldy, unsigned long long* counts) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (int j = blockIdx.y; j < m; j += gridDim.y) {   // items beyond the 65535 CTAs of grid.y: strided
        const int64_t o = i + (int64_t)j * ldy;
        int8_t v = 0;
        if (!mask || mask[o] != 0) {
            const double x = src[i + (int64_t)j * n];
            if (x == 1.0) v = 1;
            else if (x == -1.0) v = -1;
            else atomicAdd(counts + ((!mask && isnan(x)) ? 0 : 1), 1ull);
        }
        dst[o] = v;
    }
}

size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

}  // namespace

int launch_ppc_plane(cudaStream_t st, const double* src, int n, int m, const int8_t* mask, int8_t* dst, int64_t ldy,
                     unsigned long long* counts) {
    dim3 grid((unsigned)ceil_div(n, 256), (unsigned)std::min(m, 65535));   // respondents on grid.x: any n the API takes
    GP_LAUNCH(k_ppc_plane, grid, 256, 0, st, src, n, m, mask, dst, ldy, counts);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

// ---- PpcChi2 --------------------------------------------------------------------------------------------------------
// pool block: item_cnt m | resp_cnt n | glob_cnt 1 (uint32), item_nobs m | resp_nobs n (int), wpart nwr x m,
// rpart PPC_CHUNKS x n, item_d m (double2)
static int ppc_nwr(int n) { return (int)ceil_div(n, 256) * 4; }   // warps of the replication grid

int PpcChi2::init(cudaStream_t st, const int8_t* y8, int64_t ldy8, int n_, int m_) {
    n = n_; m = m_;
    const size_t ints = align256(((size_t)2 * m + 2 * n + 1) * 4);
    const size_t d2 = ((size_t)ppc_nwr(n) * m + (size_t)PPC_CHUNKS * n + m) * sizeof(double2);
    GP_TRY(pool_alloc(&buf, ints + d2, st));
    stream_for_free = st;
    item_cnt = (uint32_t*)buf; resp_cnt = item_cnt + m; glob_cnt = resp_cnt + n;
    item_nobs = (int*)(glob_cnt + 1); resp_nobs = item_nobs + m;
    wpart = (double2*)((char*)buf + ints); rpart = wpart + (size_t)ppc_nwr(n) * m; item_d = rpart + (size_t)PPC_CHUNKS * n;
    GP_CUDA(cudaMemsetAsync(buf, 0, ints, st));
    dim3 grid((unsigned)ceil_div(n, 128), (unsigned)PPC_CHUNKS);
    GP_LAUNCH(k_ppc_nobs, grid, 128, 0, st, y8, ldy8, n, m, item_nobs, resp_nobs);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

int PpcChi2::iterate(cudaStream_t st, const double* f, int64_t ld, const int8_t* y8, int64_t ldy8, const double* theta,
                     const double* beta, RngKey key, uint32_t item_offset, int8_t* yrep) {
    if (ld % 2 || ldy8 % 2) { set_last_error("ppc: leading dimensions must be even"); return GPIRT_B200_ERR_ARG; }
    const int nwr = ppc_nwr(n);
    dim3 grid((unsigned)ceil_div(n, 256), (unsigned)PPC_CHUNKS);
    GP_LAUNCH(k_ppc_replicate, grid, 128, 0, st, f, ld, y8, ldy8, theta, beta, n, m, key, item_offset, yrep, wpart, nwr, rpart);
    GP_LAUNCH(k_ppc_items, (unsigned)ceil_div(m, 8), 256, 0, st, wpart, nwr, m, item_d, item_cnt);
    GP_LAUNCH(k_ppc_resp_glob, (unsigned)ceil_div(n, 256) + 1, 256, 0, st, rpart, n, item_d, m, resp_cnt, glob_cnt);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

int PpcChi2::finish(cudaStream_t st, int S, double* item_ppp, double* resp_ppp, double* ppp) {
    std::vector<uint32_t> cnt((size_t)m + n + 1);
    std::vector<int> nobs((size_t)m + n);
    GP_CUDA(cudaMemcpyAsync(cnt.data(), item_cnt, cnt.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    GP_CUDA(cudaMemcpyAsync(nobs.data(), item_nobs, nobs.size() * sizeof(int), cudaMemcpyDeviceToHost, st));
    GP_CUDA(cudaStreamSynchronize(st));
    auto val = [&](uint32_t c, bool any) { return (S > 0 && any) ? (double)c / (double)S : (double)NAN; };
    int64_t total = 0;
    for (int j = 0; j < m; ++j) {
        total += nobs[j];
        if (item_ppp) item_ppp[j] = val(cnt[j], nobs[j] > 0);
    }
    if (resp_ppp) for (int i = 0; i < n; ++i) resp_ppp[i] = val(cnt[(size_t)m + i], nobs[(size_t)m + i] > 0);
    if (ppp) *ppp = val(cnt[(size_t)m + n], total > 0);
    return GPIRT_B200_OK;
}

void PpcChi2::destroy() {
    pool_free(buf, stream_for_free);
    buf = nullptr;
}

// ---- PpcPairs -------------------------------------------------------------------------------------------------------
struct PpcPairs::Maps { CUtensorMap obs_y, rep_y, mask; };

// one cudaMalloc: yrep | mask (missing cells only) | colsum_obs | colsum_rep | obs (int4) | cnt | stage (2 x m x PPC_STAGE_COLS)
size_t PpcPairs::bytes_needed(int64_t n, int64_t m, bool missing) {
    const int64_t ldy = round_up(n, 16), mt = ceil_div(m, PP_T), tiles = mt * (mt + 1) / 2;
    const size_t plane = align256((size_t)ldy * m);
    return plane * (missing ? 2 : 1) + 2 * align256((size_t)m * 4) + align256((size_t)tiles * PP_TILE_ELEMS * 16) +
           align256((size_t)tiles * PP_TILE_ELEMS * 4) + (size_t)2 * PPC_STAGE_COLS * m * sizeof(double);
}

int PpcPairs::init(cudaStream_t st, const int8_t* y8, int64_t ldy_, int n_, int m_, bool missing_) {
    n = n_; m = m_; ldy = ldy_; missing = missing_;
    if (ldy != round_up(n, 16)) { set_last_error("ppc pairs: the response plane must have pitch round_up(n, 16)"); return GPIRT_B200_ERR_ARG; }
    mt = (int)ceil_div(m, PP_T);
    tiles = (int64_t)mt * (mt + 1) / 2;
    bytes = bytes_needed(n, m, missing);
    const cudaError_t e = cudaMalloc((void**)&buf, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        buf = nullptr;
        set_last_error("device allocation of %zu bytes for the pair state of the posterior predictive checks failed: %s", bytes,
                       cudaGetErrorString(e));
        return GPIRT_B200_ERR_NOMEM;
    }
    const size_t plane = align256((size_t)ldy * m);
    char* p = buf;
    yrep = (int8_t*)p; p += plane;
    if (missing) { mask = (int8_t*)p; p += plane; }
    colsum_obs = (int*)p; p += align256((size_t)m * 4);
    colsum_rep = (int*)p; p += align256((size_t)m * 4);
    obs = (int4*)p; p += align256((size_t)tiles * PP_TILE_ELEMS * 16);
    cnt = (uint32_t*)p; p += align256((size_t)tiles * PP_TILE_ELEMS * 4);
    stage = (double*)p;
    GP_CUDA(cudaMemsetAsync(yrep, 0, plane, st));   // padding rows stay zero
    GP_TRY(clear_counters(st));
    if (missing) {
        const size_t count = (size_t)ldy * m;
        GP_LAUNCH(k_ppc_abs, (unsigned)ceil_div((int64_t)count, 256), 256, 0, st, y8, count, mask);
    }
    maps = new Maps();
    GP_TRY(make_map_k_major(&maps->obs_y, (void*)y8, (uint64_t)m, (uint64_t)n, (uint64_t)ldy, PP_T));
    GP_TRY(make_map_k_major(&maps->rep_y, yrep, (uint64_t)m, (uint64_t)n, (uint64_t)ldy, PP_T));
    GP_TRY(make_map_k_major(&maps->mask, missing ? (void*)mask : (void*)yrep, (uint64_t)m, (uint64_t)n, (uint64_t)ldy, PP_T));
    GP_CUDA(cudaFuncSetAttribute(k_ppc_pairs<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, PpCfg<false>::SMEM));
    GP_CUDA(cudaFuncSetAttribute(k_ppc_pairs<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, PpCfg<true>::SMEM));
    return observed_pass(st, y8);
}

int PpcPairs::observed_pass(cudaStream_t st, const int8_t* y8) {
    const int kb = (int)ceil_div(n, PP_BK);
    if (missing) {
        GP_LAUNCH(k_ppc_pairs<true>, (unsigned)tiles, 256, PpCfg<true>::SMEM, st, maps->obs_y, maps->mask, kb, mt, m, n,
                  (const int*)nullptr, obs, cnt, 1);
    } else {
        GP_LAUNCH(k_ppc_colsum, (unsigned)ceil_div(m, 8), 256, 0, st, y8, ldy, m, colsum_obs);
        GP_LAUNCH(k_ppc_pairs<false>, (unsigned)tiles, 256, PpCfg<false>::SMEM, st, maps->obs_y, maps->obs_y, kb, mt, m, n,
                  (const int*)colsum_obs, obs, cnt, 1);
    }
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

int PpcPairs::clear_counters(cudaStream_t st) {
    GP_CUDA(cudaMemsetAsync(cnt, 0, (size_t)tiles * PP_TILE_ELEMS * sizeof(uint32_t), st));
    return GPIRT_B200_OK;
}

int PpcPairs::iterate(cudaStream_t st) {
    const int kb = (int)ceil_div(n, PP_BK);
    if (missing) {
        GP_LAUNCH(k_ppc_pairs<true>, (unsigned)tiles, 256, PpCfg<true>::SMEM, st, maps->rep_y, maps->mask, kb, mt, m, n,
                  (const int*)nullptr, obs, cnt, 0);
    } else {
        GP_LAUNCH(k_ppc_colsum, (unsigned)ceil_div(m, 8), 256, 0, st, yrep, ldy, m, colsum_rep);
        GP_LAUNCH(k_ppc_pairs<false>, (unsigned)tiles, 256, PpCfg<false>::SMEM, st, maps->rep_y, maps->rep_y, kb, mt, m, n,
                  (const int*)colsum_rep, obs, cnt, 0);
    }
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

int PpcPairs::finish(cudaStream_t st, double scale, bool all_nan, double* log_or, double* ppp, const CopyOut& copy) {
    if (!log_or && !ppp) return GPIRT_B200_OK;
    double* lor_s = stage;
    double* ppp_s = stage + (size_t)PPC_STAGE_COLS * m;
    for (int k0 = 0; k0 < m; k0 += PPC_STAGE_COLS) {
        const int kc = std::min(PPC_STAGE_COLS, m - k0);
        dim3 grid((unsigned)ceil_div(m, 256), (unsigned)kc);
        GP_LAUNCH(k_ppc_pairs_finish, grid, 256, 0, st, obs, cnt, mt, m, k0, scale, all_nan ? 1 : 0, lor_s, ppp_s);
        GP_CUDA(cudaGetLastError());
        GP_CUDA(cudaStreamSynchronize(st));   // copy() returns when the block has landed: the staging is then free again
        const size_t count = (size_t)kc * m;
        if (log_or) GP_TRY(copy(log_or + (size_t)k0 * m, lor_s, count));
        if (ppp) GP_TRY(copy(ppp + (size_t)k0 * m, ppp_s, count));
    }
    return GPIRT_B200_OK;
}

void PpcPairs::destroy() {
    if (buf) cudaFree(buf);   // synchronises with the device
    buf = nullptr;
    delete maps;
    maps = nullptr;
}

}  // namespace gpirt
