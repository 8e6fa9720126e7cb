// Streaming a slice of the neighbour table into shared memory (the indexer warp of the tcgen05 conv kernels).
#pragma once
#include <cstdint>

// One warp copies nbr[k][row_base .. row_base + ROWS) for k = 0..noffs-1 (`nbr_k0` points at offset 0 of the slice,
// rows of the table are `n_out` ints apart) to dst0 as [noffs][ROWS] int32.  Rows >= r_end are written as -1.
// Full tiles take the fast path: a running pointer and ROWS/32 coalesced 128-byte cp.async per offset, ~3 instructions
// per copy.  (The first version recomputed k, r, the bounds test and a 64-bit address per element, ~15 instructions; on
// 16-channel layers the single indexer warp then took longer per tile than the eight producer warps and they stalled
// ~4 k cycles at every tile boundary: the "indexer fix" of profiles/r01_feed_ab.md.)
template <int ROWS>
__device__ __forceinline__ void load_table_slice(uint32_t dst0, const int *__restrict__ nbr_k0, int n_out, int row_base, int r_end,
                                                 int noffs, int lane) {
    const int *src = nbr_k0 + row_base + lane;
    uint32_t dst = dst0 + 4u * lane;
    if (row_base + ROWS <= r_end) {
#pragma unroll 3
        for (int k = 0; k < noffs; ++k, src += n_out, dst += 4u * ROWS) {
#pragma unroll
            for (int j = 0; j < ROWS / 32; ++j)
                asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst + 128u * j), "l"(src + 32 * j) : "memory");
        }
    } else {
        for (int k = 0; k < noffs; ++k, src += n_out, dst += 4u * ROWS) {
#pragma unroll
            for (int j = 0; j < ROWS / 32; ++j) {
                if (row_base + lane + 32 * j < r_end)
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst + 128u * j), "l"(src + 32 * j) : "memory");
                else
                    asm volatile("st.shared.b32 [%0], %1;" ::"r"(dst + 128u * j), "r"(-1) : "memory");
            }
        }
    }
}
