// Interface of the row-cache / TMEM-operand convolution kernel (conv_ts.cu) towards conv_tc.cu's dispatcher.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

// Per-tile gather plan of one neighbour table (toda_table_tile_plan): for every 128-row tile and offset group the sorted
// list of distinct input rows (`rows`, `cap` entries reserved per (tile, group), `cnt` used) and the table rewritten as
// 16-bit slots into that list (`lidx` [tile][kvol][128]; 0xFFFF = no neighbour, 0xFFFE = read the row from global memory).
struct TilePlan {
    const uint16_t *lidx;
    const int32_t *rows;
    const int32_t *cnt;
    int ngroups;
    int cap;
};

int conv_ts_slab_capacity(int cin);
bool conv_ts_supported(int cin, int cout, int kvol, const TilePlan *plan);
int conv_ts_fwd(const void *xb, int n_in, int cin, const int32_t *nbr, int n_out, int kvol, const TilePlan &plan, const void *wb,
                int cout, const float *bias, const float *addend, float *y, const int32_t *out_rows, const uint32_t *tile_masks,
                double *bn_sums, cudaStream_t st);
// 2-D bf16 row-major tensor map [rows][cols] with box [box_rows][box_cols], swizzle by box row bytes (conv_tma.cu)
int conv_tma_make_map(CUtensorMap *m, const void *ptr, uint64_t rows, uint64_t cols, uint32_t box_rows, uint32_t box_cols);
