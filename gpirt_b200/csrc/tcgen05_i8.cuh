// TMA / mbarrier / tcgen05 helpers of the int8 tensor-core kernels that stage K-major SWIZZLE_128B tiles of 128-byte
// rows (theta_int8.cu: k_igemm_theta, k_peak_umma_i8; ppc.cu: k_ppc_pairs).
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace gpirt {
namespace i8tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// one lane of a converged warp (ptxas then emits the TMA / tensor-core instructions of the region back to back)
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
// shared-memory matrix descriptor, K-major operand, 128-byte swizzle, tile rows are 128 bytes (one swizzle span):
// start address >> 4 | SBO (8 rows x 128 B = 1024 B) >> 4 at bit 32 | version 1 at bit 46 | SWIZZLE_128B (2) at bit 61
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
    uint64_t d = (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// instruction descriptor: D = S32 (2 << 4), A = B = signed int8 (1 << 7, 1 << 10), both K-major, N >> 3 at 17, M >> 4 at 24
constexpr uint32_t idesc_i8(int M, int N) {
    return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

template <uint32_t IDESC>
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(da), "l"(db), "r"(IDESC), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// TMA map of an int8 matrix stored K-major: `rows` rows of `cols` bytes, `row_stride` bytes apart (a multiple of 16),
// loaded as boxes of box_rows x 128 bytes with the 128-byte swizzle; boxes reaching past either edge are filled with zeros
int make_map_k_major(CUtensorMap* map, void* base, uint64_t rows, uint64_t cols, uint64_t row_stride, uint32_t box_rows);

}  // namespace i8tc
}  // namespace gpirt
