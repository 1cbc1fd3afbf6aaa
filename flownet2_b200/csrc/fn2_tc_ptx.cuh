// tcgen05 / TMA / mbarrier PTX wrappers shared by the tensor-core kernels (fn2_conv_tc.cu, fn2_conv_tn.cu); sm_100a only.
#pragma once
#include <cuda.h>
#include "fn2_common.cuh"

namespace fn2 {
namespace {

// Mean relative loss of a chain of n tensor-core MMAs accumulating into one FP32 accumulator, which the B200 rounds toward
// zero: RZ_COMP_A + RZ_COMP_B * n (tools/tc_calibrate2.py on a B200, profiles/r01_tc_calibration.txt).
constexpr float RZ_COMP_A = 2.0e-8f, RZ_COMP_B = 1.67e-8f;

// division by a launch constant without the ~40-instruction integer divide (the tile decode is on the critical path of the
// single-thread producer and MMA roles once per tile): q = (umulhi(n, mul) + n) >> shift for n < 2^31
struct FastDiv {
    uint32_t mul, shift, d;
    __host__ void init(int div) {
        d = (uint32_t)div;
        shift = 0;
        while ((1u << shift) < d) shift++;
        mul = (uint32_t)(((1ull << 32) * ((1ull << shift) - d)) / d + 1);
    }
    __device__ __forceinline__ int div(int n) const { return (int)(((uint32_t)__umulhi((uint32_t)n, mul) + (uint32_t)n) >> shift); }
    __device__ __forceinline__ void divmod(int n, int& q, int& r) const { q = div(n); r = n - q * (int)d; }
};

__device__ __forceinline__ uint32_t su32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(su32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(su32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(su32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done = 0, spins = 0;
    while (true) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(su32(bar)), "r"(parity) : "memory");
        if (done) break;
        if (++spins > (1u << 24)) __trap();       // a lost arrival becomes a launch error, never a hang
    }
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
                 ::"r"(su32(dst)), "l"(map), "r"(su32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\telect.sync rx|px, 0xffffffff;\n\tselp.b32 %0, 1, 0, px;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(su32(bar)) : "memory");
}
// D[tmem_c] (+)= A[tmem_a] * B[desc_b]^T, kind::tf32, A from tensor memory
__device__ __forceinline__ void mma_tf32_ts(uint32_t tmem_c, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
                 ::"r"(tmem_c), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t* v) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"
        "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
        ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
          "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]),
          "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]),
          "r"(v[30]), "r"(v[31]) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
          "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
          "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ uint32_t to_tf32(float x) { return (__float_as_uint(x) + 0x1000u) & 0xffffe000u; }
// shared-memory matrix descriptor: K-major, SWIZZLE_128B, 8-row atoms of 1024 B (validated by tools/tc_probe.cu)
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
__host__ __device__ inline uint32_t make_idesc_tf32(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

}  // namespace
}  // namespace fn2
