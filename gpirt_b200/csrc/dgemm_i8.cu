// FP64-accurate GEMM on the 5th-generation tensor cores (tcgen05 / TMEM / TMA) with exact integer arithmetic.
//
// B200 has 36.9 TFLOP/s of FP64 (DMMA) but ~4.5 POP/s of int8 tensor throughput.  The two big products of a sweep,
//     nu = L Z            (reference src/draw-f.cpp:20  "nu = L * randn(n)", all m items at once)
//     f* = (S^-1 K*)^T f  (reference src/draw-fstar.cpp:21-26 in the restructured form, DESIGN.md)
// are therefore computed in fixed point.  Every operand row r (a row of A, a column of B) is written as
//     a[r, k] = 2^(e_r - 55) X[r, k],   X = sum_{s=0..7} d_s 128^(7-s),  d_s in [-64, 64]   (balanced base-128 digits)
// so that
//     sum_k a[i,k] b[j,k] = 2^(ea_i - 6) 2^(eb_j - 6) sum_{l} 128^-l  sum_{s+t=l} ( sum_k da_s[i,k] db_t[j,k] )
// The innermost sums are int8 x int8 -> int32 tensor-core products and are EXACT (|.| <= (l+1) K 64^2 < 2^31 for
// K < 65536).  Levels l = 0..7 are kept (36 plane pairs); the dropped levels l >= 8 contribute less than
// 2^-53 2^(ea+eb) <= 2^-51 amax_i bmax_j per term of the dot product, i.e. the result carries an absolute error of at most
// K 2^-51 amax_i bmax_j — the same order as the K 2^-53 sum|a||b| bound of an FP64 dot product when rows are not badly
// scaled, which is the case for L (rows of unit norm), Z (normal draws), S^-1 K* and f.
//
// Kernel: persistent (one CTA per SM) or one tile per CTA, 128 x 64 output tile, CTAs in clusters of 2 that share the A slab.  A stage of the mbarrier ring holds all 8 digit planes of a
// 128 x KB slab of A and a 64 x KB slab of B (KB = 64 bytes, SWIZZLE_64B, TMA-loaded); from it the elected thread issues
// all 36 plane-pair MMAs (M = 128, N = 64, K = 32), each into the TMEM accumulator of its level l — 8 levels x 64
// columns = the whole 512-column tensor memory.  Operand bytes are therefore read from L2 ONCE per stage, not once per
// plane pair.  Four epilogue warps read the 8 level accumulators with tcgen05.ld, combine them in FP64 by Horner's rule,
// apply the two power-of-two scales and store; the int32 products never touch HBM.
#include <cuda.h>

#include <climits>

#include "dgemm_i8.cuh"

namespace gpirt {

namespace {

constexpr int DG_S = DigitPlanes::S;
#ifndef DG_KB_BYTES
#define DG_KB_BYTES 64
#endif
constexpr int DG_BM = 128, DG_BN = 64, DG_KB = DG_KB_BYTES, DG_UMMA_K = 32;
constexpr int DG_A_PLANE = DG_BM * DG_KB, DG_B_PLANE = DG_BN * DG_KB;
constexpr int DG_A_BYTES = DG_S * DG_A_PLANE, DG_B_BYTES = DG_S * DG_B_PLANE, DG_STAGE_BYTES = DG_A_BYTES + DG_B_BYTES;
constexpr int DG_STAGES = 196608 / DG_STAGE_BYTES;
constexpr int DG_SMEM = DG_STAGES * DG_STAGE_BYTES + 1024 /* alignment slack */ + 256 /* barriers */;
constexpr int DG_TMEM_COLS = 512;
constexpr int DG_THREADS = 192;   // warp 0: TMA producer, warp 1: MMA issuer (+ TMEM alloc), warps 2..5: epilogue
constexpr int CN = 2;             // CTAs per cluster (they share the A slab, see k_dgemm_i8)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// one lane of a converged warp; ptxas recognises the pattern and emits the tensor-core / TMA instructions of the elected
// region back to back (a `lane == 0` branch instead wraps every one of them in a per-thread election loop, which made
// instruction issue — not the tensor pipe — the limit of this kernel)
__device__ __forceinline__ uint32_t elect_one() {
    uint32_t pred = 0;
    asm volatile("{\n\t.reg .pred P1;\n\telect.sync _|P1, 0xffffffff;\n\tselp.u32 %0, 1, 0, P1;\n\t}" : "=r"(pred));
    return pred;
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar) : "memory");
}
// the same load delivered to the same CTA-relative shared-memory offset (and mbarrier) of every CTA in `mask`
__device__ __forceinline__ void tma_load_2d_mc(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar, uint16_t mask) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%2, %3}], [%4], %5;"
                 ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar), "h"(mask) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared-memory matrix descriptor, K-major operand, 64-byte swizzle, tile rows are 64 bytes (one swizzle span):
// start address >> 4 | SBO (8 rows x 64 B = 512 B) >> 4 at bit 32 | version 1 at bit 46 | SWIZZLE_64B (4) at bit 61
__device__ __forceinline__ uint64_t umma_desc_sw64(uint32_t saddr) {
    uint64_t d = (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)((8 * DG_KB) >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)(DG_KB == 64 ? 4 : 6) << 61;
    return d;
}
// instruction descriptor: D = S32 (2 << 4), A = B = signed int8 (1 << 7, 1 << 10), both K-major, N >> 3 at 17, M >> 4 at 24
constexpr uint32_t DG_IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(DG_BN >> 3) << 17) | ((uint32_t)(DG_BM >> 4) << 24);

// collector usage of the A operand: the tensor core keeps the A slab it has just read (fill / use) so that the next MMAs
// on the same slab (use / lastuse) do not read it from shared memory again — with a 128 x 64 tile the operand reads
// (A 4 KB + B 2 KB per MMA) would otherwise exceed the shared-memory bandwidth
enum { COLL_NONE = 0, COLL_FILL = 1, COLL_USE = 2, COLL_LASTUSE = 3 };
template <int COLL>
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t accumulate) {
    if constexpr (COLL == COLL_FILL)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                     "tcgen05.mma.cta_group::1.kind::i8.collector::a::fill [%0], %1, %2, %3, p;\n\t}"
                     ::"r"(tmem_d), "l"(da), "l"(db), "r"(DG_IDESC), "r"(accumulate) : "memory");
    else if constexpr (COLL == COLL_USE)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                     "tcgen05.mma.cta_group::1.kind::i8.collector::a::use [%0], %1, %2, %3, p;\n\t}"
                     ::"r"(tmem_d), "l"(da), "l"(db), "r"(DG_IDESC), "r"(accumulate) : "memory");
    else if constexpr (COLL == COLL_LASTUSE)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                     "tcgen05.mma.cta_group::1.kind::i8.collector::a::lastuse [%0], %1, %2, %3, p;\n\t}"
                     ::"r"(tmem_d), "l"(da), "l"(db), "r"(DG_IDESC), "r"(accumulate) : "memory");
    else
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                     "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
                     ::"r"(tmem_d), "l"(da), "l"(db), "r"(DG_IDESC), "r"(accumulate) : "memory");
}
// all products of A plane P with B planes 0 .. S-1-P (levels P .. S-1), A read from shared memory once
template <int P, int T = 0>
__device__ __forceinline__ void umma_plane_row(uint32_t tmem_base, uint64_t da, uint32_t sb, uint32_t acc_rest, uint32_t acc_p0) {
    constexpr int LAST = DG_S - 1 - P;
    constexpr int COLL = (LAST == 0) ? COLL_NONE : (T == 0 ? COLL_FILL : (T == LAST ? COLL_LASTUSE : COLL_USE));
    umma_i8<COLL>(tmem_base + (uint32_t)((P + T) * DG_BN), da, umma_desc_sw64(sb + T * DG_B_PLANE), P == 0 ? acc_p0 : acc_rest);
    if constexpr (T < LAST) umma_plane_row<P, T + 1>(tmem_base, da, sb, acc_rest, acc_p0);
}
template <int P = 0>
__device__ __forceinline__ void umma_all_planes(uint32_t tmem_base, uint32_t sa, uint32_t sb, uint32_t first) {
    // level l is first written by the pair (A plane 0, B plane l): only those MMAs may overwrite
    umma_plane_row<P>(tmem_base, umma_desc_sw64(sa + P * DG_A_PLANE), sb, 1u, first);
    if constexpr (P + 1 < DG_S) umma_all_planes<P + 1>(tmem_base, sa, sb, first);
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// arrives on the barrier at the same offset in every CTA of `mask`
__device__ __forceinline__ void umma_commit_mc(uint32_t bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"(mask) : "memory");
}

// With clusters of CN CTAs the scheduler's "column tile" is a group of CN adjacent 64-column tiles (one per CTA of the
// cluster, all on the same row tile): ntiles, group_cols and total count those groups.
struct TileSched {
    int mtiles, ntiles, group_cols, total, ascending;   // ascending: row tile 0 is the heaviest (upper-triangular A)
    int mtile0;                                          // first row tile with work (rows above it are skipped entirely)
    // order index -> (row tile, column tile): column tiles in groups whose planes stay in L2, row tiles heaviest first
    __device__ __forceinline__ void at(int o, int& r, int& c) const {
        const int per_group = group_cols * mtiles;
        const int g = o / per_group, o2 = o - g * per_group;
        const int gw = min(group_cols, ntiles - g * group_cols);
        r = mtile0 + (ascending ? o2 / gw : mtiles - 1 - o2 / gw);
        c = g * group_cols + o2 % gw;
    }
};

// Clusters of CN CTAs work on CN adjacent column tiles of the same row tile.  Each CTA loads 128 / CN rows of
// every A plane and MULTICASTS them to the whole cluster, so the A slab crosses the L2 -> SM fabric once per cluster
// instead of once per CTA (the 128 x 64 tile is exactly balanced between the int8 tensor rate and the L2 feed rate:
// 96 KB per 2304 tensor-core cycles per SM = 6.2 KB/clk chip-wide; with CN = 2 it is 64 KB).  A stage may be refilled only
// when every CTA of the cluster has consumed it: the MMA issuer's commit arrives on the stage's empty barrier of ALL CTAs.
__global__ void __launch_bounds__(DG_THREADS, 1)
k_dgemm_i8(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, TileSched sched,
           int a_rows_pad, int b_rows_pad, int kb_lo, int kb_hi, int a_tri, int M, int N,
           const double* __restrict__ ascale, const double* __restrict__ bscale, double* __restrict__ C, int64_t ldc,
           int accumulate) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = (uint64_t*)(smem + DG_STAGES * DG_STAGE_BYTES);
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + DG_STAGES);
    const uint32_t tfull = smem_u32(bars + 2 * DG_STAGES), tempty = smem_u32(bars + 2 * DG_STAGES + 1);
    uint32_t* tmem_slot = (uint32_t*)(bars + 2 * DG_STAGES + 2);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    const uint32_t crank = cluster_ctarank();
    const int cluster_id = blockIdx.x / CN, n_clusters = gridDim.x / CN;
    constexpr uint16_t CMASK = (uint16_t)((1u << CN) - 1u);
    if (warp == 0 && lane == 0) {
        for (int s = 0; s < DG_STAGES; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, CN); }
        mbar_init(tfull, 1);
        mbar_init(tempty, 4);    // one arrival per epilogue warp
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {   // the whole tensor memory: 8 level accumulators x 64 columns
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(DG_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    cluster_sync_all();   // every CTA's barriers are initialised before a peer signals them

    // K-block range of a row tile: a lower-triangular A stops at the diagonal block, an upper-triangular one starts there
    auto kb_end = [&](int r) { return a_tri == 1 ? min(kb_hi, (int)(((int64_t)(r + 1) * DG_BM + DG_KB - 1) / DG_KB)) : kb_hi; };
    auto kb_begin = [&](int r) { return a_tri == 2 ? max(kb_lo, (int)(((int64_t)r * DG_BM) / DG_KB)) : kb_lo; };

    if (warp == 0) {
        if (elect_one()) {
        // ---- TMA producer ----
        uint32_t it = 0;
        constexpr int A_PART_ROWS = DG_BM / CN, A_PART = A_PART_ROWS * DG_KB;   // this CTA's share of every A plane
        for (int o = cluster_id; o < sched.total; o += n_clusters) {
            int r, c;
            sched.at(o, r, c);
            c = c * CN + (int)crank;
            const int ke = kb_end(r);
            for (int kb = kb_begin(r); kb < ke; ++kb, ++it) {
                const uint32_t s = it % DG_STAGES, ph = (it / DG_STAGES) & 1u;
                mbar_wait(empty0 + 8 * s, ph ^ 1u);                 // every CTA of the cluster has consumed the slot
                mbar_expect_tx(full0 + 8 * s, DG_STAGE_BYTES);      // own B slab + the whole A slab (own part + the peers' parts)
                const uint32_t sa = smem_u32(smem + s * DG_STAGE_BYTES), sb = sa + DG_A_BYTES;
#pragma unroll
                for (int p = 0; p < DG_S; ++p) {
                    tma_load_2d_mc(sa + p * DG_A_PLANE + crank * A_PART, &tmA, kb * DG_KB,
                                   p * a_rows_pad + r * DG_BM + (int)crank * A_PART_ROWS, full0 + 8 * s, CMASK);
                    tma_load_2d(sb + p * DG_B_PLANE, &tmB, kb * DG_KB, p * b_rows_pad + c * DG_BN, full0 + 8 * s);
                }
            }
        }
        }
    } else if (warp == 1) {
        if (elect_one()) {
        // ---- MMA issuer ----
        uint32_t it = 0, tile_it = 0;
        for (int o = cluster_id; o < sched.total; o += n_clusters, ++tile_it) {
            int r, c;
            sched.at(o, r, c);
            const int ke = kb_end(r), kb0 = kb_begin(r);
            mbar_wait(tempty, (tile_it & 1u) ^ 1u);          // epilogue has drained the previous tile's accumulators
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            for (int kb = kb0; kb < ke; ++kb, ++it) {
                const uint32_t s = it % DG_STAGES, ph = (it / DG_STAGES) & 1u;
                mbar_wait(full0 + 8 * s, ph);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t sa = smem_u32(smem + s * DG_STAGE_BYTES), sb = sa + DG_A_BYTES;
#pragma unroll
                for (int k2 = 0; k2 < DG_KB / DG_UMMA_K; ++k2)
                    umma_all_planes(tmem_base, sa + k2 * DG_UMMA_K, sb + k2 * DG_UMMA_K, (uint32_t)((kb != kb0) | (k2 != 0)));
                umma_commit_mc(empty0 + 8 * s, CMASK);   // frees the slot in every CTA of the cluster once these MMAs have read it
            }
            umma_commit(tfull);                // all level accumulators of this tile are complete
        }
        }
    } else if (warp >= 2) {
        // ---- epilogue: TMEM -> registers, Horner over the 8 levels in FP64, scale, store ----
        const int q = warp & 3;                                  // TMEM lane quarter this warp may touch (warp % 4)
        const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
        uint32_t tile_it = 0;
        for (int o = cluster_id; o < sched.total; o += n_clusters, ++tile_it) {
            int r, c;
            sched.at(o, r, c);
            c = c * CN + (int)crank;
            const int i = r * DG_BM + q * 32 + lane;
            const double sa_i = (i < M) ? ascale[i] : 0.0;
            mbar_wait(tfull, tile_it & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (kb_end(r) > kb_begin(r)) {
#pragma unroll 1
                for (int cc = 0; cc < DG_BN / 8; ++cc) {
                    uint32_t v[DG_S][8];
#pragma unroll
                    for (int l = 0; l < DG_S; ++l)
                        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                                     : "=r"(v[l][0]), "=r"(v[l][1]), "=r"(v[l][2]), "=r"(v[l][3]), "=r"(v[l][4]), "=r"(v[l][5]),
                                       "=r"(v[l][6]), "=r"(v[l][7])
                                     : "r"(trow + (uint32_t)(l * DG_BN + cc * 8)) : "memory");
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                    for (int h = 0; h < 8; ++h) {
                        const int j = c * DG_BN + cc * 8 + h;
                        double x = (double)(int)v[DG_S - 1][h];
#pragma unroll
                        for (int l = DG_S - 2; l >= 0; --l) x = fma(x, 0.0078125, (double)(int)v[l][h]);
                        if (i < M && j < N) {
                            double* dst = C + (int64_t)i + (int64_t)j * ldc;
                            const double val = x * sa_i * bscale[j];
                            *dst = accumulate ? *dst + val : val;
                        }
                    }
                }
            } else if (!accumulate) {
                for (int h = 0; h < DG_BN; ++h) {
                    const int j = c * DG_BN + h;
                    if (i < M && j < N) C[(int64_t)i + (int64_t)j * ldc] = 0.0;
                }
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty);
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    cluster_sync_all();   // no CTA leaves while a peer may still signal its barriers
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(DG_TMEM_COLS) : "memory");
    }
}

// ---- operand preparation ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void digits_of(double v, double qs, int8_t d[DG_S]) {
    double t = v * qs;
    t = fmin(fmax(t, -36028797018963968.0), 36028797018963968.0);   // |X| <= 2^55 (only a fixed scale can saturate)
    long long X = __double2ll_rn(t);
#pragma unroll
    for (int s = DG_S - 1; s >= 1; --s) {
        const int dd = (int)((X + 64) & 127) - 64;   // balanced base-128 digit
        d[s] = (int8_t)dd;
        X = (X - dd) >> 7;
    }
    d[0] = (int8_t)X;                                // |X| <= 64 here
}
__device__ __forceinline__ void scales_of(double mx, double& qscale, double& oscale) {
    const int e = (mx > 0.0 && isfinite(mx)) ? ilogb(mx) + 1 : 0;
    qscale = scalbn(1.0, 55 - e);
    oscale = scalbn(1.0, e - 6);
}

// one CTA per operand row; the contraction index is contiguous
__global__ void __launch_bounds__(256) k_slice_kcontig(const double* __restrict__ src, int64_t ld, int k,
                                                       int8_t* __restrict__ planes, int64_t rows_pad, int64_t k_pad,
                                                       double* __restrict__ scale) {
    __shared__ double red[8];
    __shared__ double qs_sh;
    const int r = blockIdx.x;
    const double* row = src + (int64_t)r * ld;
    double mx = 0.0;
    for (int kk = threadIdx.x; kk < k; kk += 256) mx = fmax(mx, fabs(row[kk]));
    mx = warp_max(mx);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) mx = fmax(mx, red[w]);
        double qs, os;
        scales_of(mx, qs, os);
        scale[r] = os;
        qs_sh = qs;
    }
    __syncthreads();
    const double qs = qs_sh;
    for (int k4 = threadIdx.x * 4; k4 < k; k4 += 1024) {
        unsigned packed[DG_S];
#pragma unroll
        for (int s = 0; s < DG_S; ++s) packed[s] = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            int8_t d[DG_S];
            digits_of((k4 + b < k) ? row[k4 + b] : 0.0, qs, d);
#pragma unroll
            for (int s = 0; s < DG_S; ++s) packed[s] |= (unsigned)(d[s] & 0xFF) << (8 * b);
        }
#pragma unroll
        for (int s = 0; s < DG_S; ++s)
            *reinterpret_cast<unsigned*>(planes + ((int64_t)s * rows_pad + r) * k_pad + k4) = packed[s];
    }
}

// rows contiguous (column-major source): row maxima by chunks of the contraction index, then a transposing slicer
__global__ void __launch_bounds__(128) k_rowmax_partial(const double* __restrict__ src, int64_t ld, int rows, int k, int lower,
                                                        double* __restrict__ partial, int n_chunks) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x, chunk = blockIdx.y;
    if (r >= rows) return;
    const int per = (int)ceil_div(k, n_chunks), k0 = chunk * per;
    int k1 = min(k, k0 + per);
    if (lower) k1 = min(k1, r + 1);
    double mx = 0.0;
    for (int kk = k0; kk < k1; ++kk) mx = fmax(mx, fabs(src[r + (int64_t)kk * ld]));
    partial[(int64_t)chunk * rows + r] = mx;
}
__global__ void k_rowmax_final(const double* __restrict__ partial, int rows, int n_chunks, int fixed_exp,
                               double* __restrict__ scale) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    if (fixed_exp != INT_MIN) { scale[r] = scalbn(1.0, fixed_exp - 6); return; }
    double mx = 0.0;
    for (int c = 0; c < n_chunks; ++c) mx = fmax(mx, partial[(int64_t)c * rows + r]);
    double qs, os;
    scales_of(mx, qs, os);
    scale[r] = os;
}
// 64 rows x 64 contraction indices per CTA, transposed through shared memory
__global__ void __launch_bounds__(256) k_slice_mcontig(const double* __restrict__ src, int64_t ld, int rows, int k_lo, int k_hi,
                                                       int lower, const double* __restrict__ scale,
                                                       int8_t* __restrict__ planes, int64_t rows_pad, int64_t k_pad) {
    __shared__ __align__(16) int8_t dig[DG_S][64][64 + 16];
    const int r0 = blockIdx.x * 64, k0 = k_lo + blockIdx.y * 64;
    if (lower && k0 > r0 + 63) return;     // entirely above the diagonal: stays zero
    for (int e = threadIdx.x; e < 64 * 64; e += 256) {
        const int rr = e % 64, kk = e / 64;
        const int r = r0 + rr, kx = k0 + kk;
        double v = 0.0, qs = 0.0;
        if (r < rows && kx < k_hi && !(lower && kx > r)) { v = src[r + (int64_t)kx * ld]; qs = 562949953421312.0 / scale[r]; }   // 2^49 / 2^(e-6) = 2^(55-e)
        int8_t d[DG_S];
        digits_of(v, qs, d);
#pragma unroll
        for (int s = 0; s < DG_S; ++s) dig[s][rr][kk] = d[s];
    }
    __syncthreads();
    for (int e = threadIdx.x; e < DG_S * 64 * 16; e += 256) {   // 8 planes x 64 rows x 16 words of 4 bytes
        const int w = e % 16, rr = (e / 16) % 64, s = e / (16 * 64);
        const int r = r0 + rr, kx = k0 + 4 * w;
        if (r < rows && kx < k_pad)
            *reinterpret_cast<unsigned*>(planes + ((int64_t)s * rows_pad + r) * k_pad + kx) = *reinterpret_cast<const unsigned*>(&dig[s][rr][4 * w]);
    }
}

typedef CUresult (*encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                              const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                              CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int make_map_sw64(CUtensorMap* map, void* base, uint64_t rows, uint64_t row_bytes, uint32_t box_rows) {
    static encode_fn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        GP_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres));
        if (!p || qres != cudaDriverEntryPointSuccess) { set_last_error("cuTensorMapEncodeTiled is not available"); return GPIRT_B200_ERR_CUDA; }
        fn = (encode_fn)p;
    }
    const cuuint64_t dims[2] = {row_bytes, rows};
    const cuuint64_t strides[1] = {row_bytes};
    const cuuint32_t box[2] = {(cuuint32_t)DG_KB, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    DG_KB == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_last_error("cuTensorMapEncodeTiled failed (%d)", (int)r); return GPIRT_B200_ERR_CUDA; }
    return GPIRT_B200_OK;
}

constexpr int ROWMAX_CHUNKS = 16;

}  // namespace

struct DigitPlanes::Map { CUtensorMap m, m_part; };   // m_part: box of box_rows / cluster size rows (multicast parts of an A slab)

int DigitPlanes::init(cudaStream_t st, int rows_, int k_, int box_rows_) {
    rows = rows_; k = k_; box_rows = box_rows_;
    rows_pad = round_up(rows, box_rows == DG_BN ? DG_BN * CN : box_rows);   // whole clusters of column tiles
    k_pad = round_up(k, 128);
    const size_t bytes = (size_t)S * rows_pad * k_pad;
    GP_TRY(pool_alloc((void**)&planes, bytes, st));
    GP_TRY(pool_alloc((void**)&scale, (size_t)rows_pad * sizeof(double), st));
    GP_TRY(pool_alloc((void**)&partial, (size_t)ROWMAX_CHUNKS * rows_pad * sizeof(double), st));
    stream_for_free = st;
    GP_CUDA(cudaMemsetAsync(planes, 0, bytes, st));   // padding rows / columns and the strict upper triangle stay zero
    GP_CUDA(cudaMemsetAsync(scale, 0, (size_t)rows_pad * sizeof(double), st));
    map = new Map();
    GP_TRY(make_map_sw64(&map->m, planes, (uint64_t)S * rows_pad, (uint64_t)k_pad, (uint32_t)box_rows));
    GP_TRY(make_map_sw64(&map->m_part, planes, (uint64_t)S * rows_pad, (uint64_t)k_pad, (uint32_t)(box_rows / CN)));
    return GPIRT_B200_OK;
}

int DigitPlanes::slice_kcontig(cudaStream_t st, const double* src, int64_t ld) {
    if (rows <= 0 || k <= 0) return GPIRT_B200_OK;
    GP_LAUNCH(k_slice_kcontig, (unsigned)rows, 256, 0, st, src, ld, k, planes, rows_pad, k_pad, scale);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

int DigitPlanes::slice_mcontig(cudaStream_t st, const double* src, int64_t ld, bool lower, int k_lo, int k_hi, int fixed_exp) {
    if (rows <= 0 || k <= 0 || k_hi <= k_lo) return GPIRT_B200_OK;
    if (fixed_exp == INT_MIN && (k_lo != 0 || k_hi != k)) { set_last_error("slice_mcontig: row scales need the whole row"); return GPIRT_B200_ERR_ARG; }
    if (fixed_exp == INT_MIN) {
        dim3 grid((unsigned)ceil_div(rows, 128), (unsigned)ROWMAX_CHUNKS);
        GP_LAUNCH(k_rowmax_partial, grid, 128, 0, st, src, ld, rows, k, lower ? 1 : 0, partial, ROWMAX_CHUNKS);
    }
    if (fixed_exp == INT_MIN || k_lo == 0)
        GP_LAUNCH(k_rowmax_final, (unsigned)ceil_div(rows, 128), 128, 0, st, partial, rows, ROWMAX_CHUNKS, fixed_exp, scale);
    dim3 grid((unsigned)ceil_div(rows, 64), (unsigned)ceil_div(k_hi - k_lo, 64));
    GP_LAUNCH(k_slice_mcontig, grid, 256, 0, st, src, ld, rows, k_lo, k_hi, lower ? 1 : 0, scale, planes, rows_pad, k_pad);
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

void DigitPlanes::destroy() {
    for (void* p : {(void*)planes, (void*)scale, (void*)partial}) pool_free(p, stream_for_free);
    planes = nullptr; scale = nullptr; partial = nullptr;
    delete map; map = nullptr;
}

int dgemm_i8(cudaStream_t st, const DigitPlanes& A, const DigitPlanes& B, double* C, int64_t ldc, int a_tri, int k_lo,
             int k_hi, bool accumulate, int group_cols, bool persistent) {
    if (A.rows <= 0 || B.rows <= 0) return GPIRT_B200_OK;
    if (!A.map || !B.map || A.k_pad != B.k_pad || A.box_rows != DG_BM || B.box_rows != DG_BN || k_lo % DG_KB != 0 || k_lo < 0 ||
        k_hi > A.k || k_hi > B.k || A.k >= 65536) {
        set_last_error("dgemm_i8: operands do not match");
        return GPIRT_B200_ERR_ARG;
    }
    static int sm_count[64] = {0};
    static bool attr_set[64] = {false};
    int dev = 0;
    GP_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) { set_last_error("dgemm_i8: device ordinal out of range"); return GPIRT_B200_ERR_ARG; }
    {
        DeviceOnce once(attr_set);
        if (once.first) {
            GP_CUDA(cudaDeviceGetAttribute(&sm_count[dev], cudaDevAttrMultiProcessorCount, dev));
            GP_CUDA(cudaFuncSetAttribute(k_dgemm_i8, cudaFuncAttributeMaxDynamicSharedMemorySize, DG_SMEM));
        }
    }
    const int n_sm = sm_count[dev];
    if (B.rows_pad % (DG_BN * CN) != 0) { set_last_error("dgemm_i8: B operand is not padded to whole clusters"); return GPIRT_B200_ERR_ARG; }
    TileSched sched;
    // an accumulating slice of a lower-triangular product adds nothing to the rows above its first column
    sched.mtile0 = (a_tri == DG_TRI_LOWER && accumulate) ? k_lo / DG_BM : 0;
    sched.mtiles = (int)(A.rows_pad / DG_BM) - sched.mtile0;
    if (sched.mtiles <= 0) return GPIRT_B200_OK;
    sched.ntiles = (int)(B.rows_pad / (DG_BN * CN));
    const int gc = group_cols > 0 ? (int)ceil_div(group_cols, CN) : 0;
    sched.group_cols = gc > 0 ? min(gc, sched.ntiles) : sched.ntiles;
    sched.total = sched.mtiles * sched.ntiles;
    sched.ascending = a_tri == DG_TRI_UPPER ? 1 : 0;
    // persistent (one CTA per SM walks the tile list) when the kernel owns the GPU; one tile per CTA when it shares the
    // GPU with a latency-critical chain on a higher-priority stream, so that the chain's CTAs get SMs as tiles retire
    const int clusters = persistent ? min(sched.total, n_sm / CN) : sched.total;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(clusters * CN));
    cfg.blockDim = dim3(DG_THREADS);
    cfg.dynamicSmemBytes = DG_SMEM;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    int prio = 0, na = 0;
    if (st != nullptr && cudaStreamGetPriority(st, &prio) == cudaSuccess) {   // explicit: survives capture into a graph (common.cuh)
        attr[na].id = cudaLaunchAttributePriority;
        attr[na].val.priority = prio;
        ++na;
    }
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = (unsigned)CN; attr[na].val.clusterDim.y = 1; attr[na].val.clusterDim.z = 1;
    ++na;
    cfg.attrs = attr;
    cfg.numAttrs = na;
    const int a_rows_pad = (int)A.rows_pad, b_rows_pad = (int)B.rows_pad, kb_lo = k_lo / DG_KB, kb_hi = (int)ceil_div(k_hi, DG_KB);
    const int acc = accumulate ? 1 : 0;
    GP_CUDA(cudaLaunchKernelEx(&cfg, k_dgemm_i8, A.map->m_part, B.map->m, sched, a_rows_pad, b_rows_pad, kb_lo, kb_hi, a_tri, A.rows, B.rows,
                               (const double*)A.scale, (const double*)B.scale, C, ldc, acc));
    ++g_launch_count;
    GP_CUDA(cudaGetLastError());
    return GPIRT_B200_OK;
}

}  // namespace gpirt
