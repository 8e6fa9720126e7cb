// Shared helpers for libtoda_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/toda_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libtoda_b200 targets sm_100a (B200) only"
#endif

void toda_set_error(const char *fmt, ...);

#define TODA_CHECK_ARG(cond, ...)            \
    do {                                      \
        if (!(cond)) {                        \
            toda_set_error(__VA_ARGS__);      \
            return TODA_ERR_INVALID;          \
        }                                     \
    } while (0)

#define TODA_CUDA_OK(expr)                                                                   \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) {                                                              \
            toda_set_error("%s:%d CUDA error: %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
            return TODA_ERR_CUDA;                                                             \
        }                                                                                     \
    } while (0)

// every kernel launch of the library passes here: the count behind toda_launch_count() (bench.py's gpu_launches)
extern long long g_toda_launches;
#define TODA_LAUNCH_OK() do { ++g_toda_launches; TODA_CUDA_OK(cudaGetLastError()); } while (0)

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs; grids are sized in multiples of this

static inline int ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// grid for a grid-stride kernel over n items: whole waves of 148 SMs, capped at `waves` CTAs/SM
static inline int wave_grid(int64_t n, int block, int waves = 8) {
    int64_t need = (n + block - 1) / block;
    if (need <= 0) need = 1;
    int64_t rounded = (need + kNumSMs - 1) / kNumSMs * kNumSMs;
    int64_t cap = (int64_t)kNumSMs * waves;
    return (int)(rounded < cap ? rounded : cap);
}

// The 2*c doubles that follow the per-CTA partials in a BatchNorm workspace (toda_bn_workspace_bytes): where a one-call
// backward (toda_bn_bwd, toda_layer_bwd) keeps its reduced sums between the reduce and the finish phase.
double *bn_workspace_red(void *workspace, int c);

// ---------------------------------------------------------------------------------------------
// Occupancy index: two-level bitmap + per-word rank.  See include/toda_b200.h.
//   cell id = b * frame_stride + (z*H + y)*W + x      frame_stride = D*H*W rounded up to 4096
//   bits0[w]  : 64 cells per word                      rank0[w] : # marked cells before word w
//   bits1[w1] : which of its 64 bits0 words are != 0   pref1[w1]: # marked cells before L1 word w1
// ---------------------------------------------------------------------------------------------
struct GridIndex {
    unsigned long long *bits0;
    int *rank0;
    unsigned long long *bits1;
    int *pref1;     // words1 + 1 entries (last = total)
    int *tile_sums; // scratch for the scan
    long long frame_stride;
    long long words0;
    int words1;
    int batch, D, H, W;
};

static inline long long index_frame_stride(int D, int H, int W) {
    long long c = (long long)D * H * W;
    return (c + 4095) / 4096 * 4096;
}

static inline size_t index_layout(GridIndex *g, void *base, int batch, int D, int H, int W) {
    long long fs = index_frame_stride(D, H, W);
    long long cells = fs * batch;
    long long words0 = cells / 64;
    long long words1 = words0 / 64;
    size_t off = 0;
    char *p = (char *)base;
    size_t o_bits0 = off; off = align_up(off + (size_t)words0 * 8, 256);
    size_t o_bits1 = off; off = align_up(off + (size_t)words1 * 8, 256);
    size_t zero_bytes = off;  // only the two bitmaps need to be zero
    size_t o_rank0 = off; off = align_up(off + (size_t)words0 * 4, 256);
    size_t o_pref1 = off; off = align_up(off + (size_t)(words1 + 1) * 4, 256);
    size_t o_tiles = off; off = align_up(off + (size_t)(words1 / 1024 + 2) * 4, 256);
    if (g) {
        g->bits0 = (unsigned long long *)(p + o_bits0);
        g->bits1 = (unsigned long long *)(p + o_bits1);
        g->rank0 = (int *)(p + o_rank0);
        g->pref1 = (int *)(p + o_pref1);
        g->tile_sums = (int *)(p + o_tiles);
        g->frame_stride = fs;
        g->words0 = words0;
        g->words1 = (int)words1;
        g->batch = batch; g->D = D; g->H = H; g->W = W;
    }
    (void)zero_bytes;
    return off;
}

__device__ __forceinline__ long long index_cell(const GridIndex &g, int b, int z, int y, int x) {
    return (long long)b * g.frame_stride + ((long long)z * g.H + y) * g.W + x;
}

__device__ __forceinline__ int index_lookup(const GridIndex &g, long long cell) {
    unsigned long long w = __ldg(g.bits0 + (cell >> 6));
    unsigned bit = (unsigned)(cell & 63);
    if (!((w >> bit) & 1ull)) return -1;
    return __ldg(g.rank0 + (cell >> 6)) + __popcll(w & ((1ull << bit) - 1ull));
}

__device__ __forceinline__ void index_mark(const GridIndex &g, long long cell) {
    unsigned long long *wp = g.bits0 + (cell >> 6);
    unsigned long long m = 1ull << (cell & 63);
    if (*wp & m) return;  // already marked (racy read is fine: worst case one extra atomic)
    unsigned long long old = atomicOr(wp, m);
    if (old == 0ull) {
        long long w = cell >> 6;
        atomicOr(g.bits1 + (w >> 6), 1ull << (w & 63));
    }
}

// build steps shared by index.cu and voxelize.cu (defined in index.cu)
int index_build_ranks(const GridIndex &g, int32_t *out_coords, int cap, uint32_t *out_cells, int32_t *n_out,
                      cudaStream_t st);
int scan_exclusive_i32(const int *in, int *out, int n, int *tile_sums, int *total_out, cudaStream_t st);
