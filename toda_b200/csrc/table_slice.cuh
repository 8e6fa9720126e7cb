// Streaming a slice of the neighbour table into shared memory (the indexer warp of the tcgen05 conv kernels).
#pragma once
#include <cstdint>

#include "tcgen05.cuh"

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

// The indexer warp of the forward kernels (conv_tc.cu, conv_tma.cu): for every tile t of this CTA, the slice of the
// [kvol][n_out] table for the tile's ROWS rows goes into buffer ib = it & 1 (idx_bytes apart from idx_base), one tile ahead of
// the producers.  idx_empty[ib] is waited for before the buffer is reused; idx_full[ib] (expected count 64: the warp's
// cp.async completions and its plain arrivals) completes once the slice has landed.
template <int ROWS, uint32_t kMaxSpins>
__device__ __forceinline__ void index_tiles(uint32_t idx_base, int idx_bytes, uint32_t idx_full, uint32_t idx_empty,
                                            const int *__restrict__ nbr, int n_out, int kvol, int num_tiles, int lane) {
    int it = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
        const int ib = it & 1, use = it >> 1;
        if (use > 0) mbar_wait<kMaxSpins>(idx_empty + 8 * ib, (use - 1) & 1);
        load_table_slice<ROWS>(idx_base + ib * idx_bytes, nbr, n_out, t * ROWS, n_out, kvol, lane);
        cp_async_arrive_noinc(idx_full + 8 * ib);
        mbar_arrive(idx_full + 8 * ib);
    }
}
