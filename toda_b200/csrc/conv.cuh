// Entry points the convolution files call across one another (conv_simt.cu dispatches by precision to conv_tc.cu and
// conv_x3.cu; conv_tc.cu's forward picks conv_ts.cu or conv_tma.cu by shape).  Not part of the exported C ABI.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

// channels as the tensor-core kernels see them: layers narrower than 16 channels are zero-padded to UMMA K = 16
static inline int pad16(int c) { return c < 16 ? 16 : c; }

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

// 2-D bf16 row-major tensor map [rows][cols] with box [box_rows][box_cols], swizzle by box row bytes (32 / 64 / 128 B)
int make_tensor_map_bf16(CUtensorMap *m, const void *ptr, uint64_t rows, uint64_t cols, uint32_t box_rows, uint32_t box_cols);

// conv_tc.cu: bf16 tensor-core forward / dgrad (dispatching to conv_ts_fwd / conv_tma_fwd) and weight gradient
bool conv_tc_supported(int cin, int cout, int kvol);
size_t conv_tc_fwd_workspace_bytes(int n_in, int cin, int cout, int kvol);
int conv_tc_fwd(const float *x, const void *x_bf16, int n_in, int cin, const int32_t *nbr, int n_out, int kvol, const float *w,
                int cout, const float *bias, float *y, const int32_t *out_rows, const uint32_t *tile_masks, double *bn_sums,
                void *workspace, size_t workspace_bytes,
                cudaStream_t st, const TilePlan *plan, const float *addend, const void *w_bf16);
bool conv_tc_wgrad_supported(int cin, int cout, int kvol);
size_t conv_tc_wgrad_workspace_bytes(int n_in, int n_out, int kvol, int cin, int cout);
int conv_tc_wgrad(const float *x, const void *x_bf16, int n_in, int cin, const int32_t *nbr, int n_out, int kvol,
                  const uint32_t *tile_masks, const float *dy, const void *dy_bf16, int cout, float *dw_param, void *workspace,
                  size_t workspace_bytes, cudaStream_t st);

// conv_tma.cu: TMA-fed forward / dgrad, Cin = Cout = 128 only
int conv_tma_fwd(const void *xb, int n_in, int cin, const int32_t *nbr, int n_out, int kvol, const void *wb, int cout,
                 const float *bias, const float *addend, float *y, const int32_t *out_rows, const uint32_t *tile_masks, double *bn_sums,
                 cudaStream_t st);

// conv_ts.cu: row-cache / TMEM-operand forward / dgrad, taken when a tile plan is given
int conv_ts_slab_capacity(int cin);
bool conv_ts_supported(int cin, int cout, int kvol, const TilePlan *plan);
int conv_ts_fwd(const void *xb, int n_in, int cin, const int32_t *nbr, int n_out, int kvol, const TilePlan &plan, const void *wb,
                int cout, const float *bias, const float *addend, float *y, const int32_t *out_rows, const uint32_t *tile_masks,
                double *bn_sums, cudaStream_t st);

// conv_x3.cu (TODA_CONV_BF16X3): three bf16 tensor-core launches per product, fp32-class accuracy
size_t conv_x3_fwd_workspace_bytes(int n_in, int cin, int cout, int kvol);
int conv_x3_fwd(const float *x, int n_in, int cin, const int32_t *nbr, int n_out, int kvol, const float *w, int cout, const float *bias,
                float *y, const int32_t *out_rows, const uint32_t *tile_masks, double *bn_sums, void *workspace, size_t workspace_bytes,
                cudaStream_t st, const TilePlan *plan, const float *addend);
size_t conv_x3_wgrad_workspace_bytes(int n_in, int n_out, int kvol, int cin, int cout);
int conv_x3_wgrad(const float *x, int n_in, int cin, const int32_t *nbr, int n_out, int kvol, const uint32_t *tile_masks,
                  const float *dy, int cout, float *dw_param, void *workspace, size_t workspace_bytes, cudaStream_t st);
