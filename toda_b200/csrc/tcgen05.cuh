// PTX wrappers shared by the tcgen05 convolution kernels (conv_tc.cu, conv_tma.cu, conv_ts.cu): mbarriers, TMA copies,
// tcgen05.mma issue / commit, shared-memory descriptors and TMEM allocation.  Wrappers only one kernel file uses live in
// that file.
#pragma once
#include <cuda.h>
#include <cstdint>

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
// A lost arrival must not hang the GPU: a wait gives up (trap) after kMaxSpins probes.  The limit is generous (seconds at
// 2^26) because the first NCCL all-reduce of a multi-GPU run can stall every kernel on the device for hundreds of
// milliseconds; each kernel file names its own limit.  (A wall-clock limit read from %globaltimer cost registers in every
// inlined wait and 10 % of conv_ts's speed; -DTODA_TS_VERBOSE_TIMEOUT compiles in the printf that names the barrier and
// lists every stuck waiter before trapping.)
template <uint32_t kMaxSpins>
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0, spins = 0;
    while (!done) {
        // (plain try_wait: the form with a suspend-time hint -- "sleep in hardware until the phase completes or the time
        // is up" -- was used by conv_ts until the end of round 2 and is implicated in its deadlocks: with it the stage-2
        // workload hung in 10 of 12 runs, without it in 0 of 8; profiles/r02_conv_ts.md section 5)
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (!done && ++spins > kMaxSpins) {
#ifdef TODA_TS_VERBOSE_TIMEOUT
            if ((threadIdx.x & 31) == 0)
                printf("mbarrier timeout smem=0x%x parity=%u block=%d warp=%d\n", bar, parity, (int)blockIdx.x, (int)(threadIdx.x >> 5));
            if (spins < kMaxSpins + kMaxSpins / 2) { spins += kMaxSpins / 4; continue; }
#endif
            __trap();
        }
    }
}
// non-blocking probe of a barrier phase (used to look one stage ahead while the current MMAs are being issued)
__device__ __forceinline__ uint32_t mbar_test(uint32_t bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    return done;
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// arrives on `bar` once this thread's outstanding cp.asyncs have landed (no pending-count increment: the barrier's
// expected count includes the arrival)
__device__ __forceinline__ void cp_async_arrive_noinc(uint32_t bar) {
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}

// tiled 2-D TMA copy of the box at (c0 = column, c1 = row) to shared memory; completes transaction bytes on `bar`
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, int c0, int c1, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar)
        : "memory");
}

// arrives on `bar` once every tcgen05.mma this thread has issued so far has completed
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], both operands by shared-memory descriptor
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
//   [0,14) start address >> 4 | [16,30) leading byte offset >> 4 (1 for swizzled K-major) |
//   [32,46) stride byte offset >> 4 (8 rows x 128 B = 1024 B between 8-row groups) | [46,48) version = 1 (sm_100) |
//   [61,64) layout type = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_desc_k_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3fff);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// instruction descriptor (cute::UMMA::InstrDescriptor): D=f32, A=B=bf16, both K-major, M=m, N=n
__host__ __device__ constexpr uint32_t make_idesc_bf16(int m, int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// TMEM allocation of kCols columns by one whole warp (address written to shared memory at `slot`), and its release.  The
// allocating warp also gives up its allocation permit: one allocation per CTA.
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t slot) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot), "n"(kCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t tmem_base) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kCols) : "memory");
}
