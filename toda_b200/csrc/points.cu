// K0 point-stream selection: order-preserving compaction of a collated point cloud under a per-point predicate.
// Restates the point side of the reference's host pre-steps so that raw frames can stay on the GPU:
//   mode 0  range mask     pcdet/utils/common_utils.py L60-63 via data_processor.py L78-91 (x, y inclusive, no z test)
//   mode 1  rectangle      inter_domain_point_cutmix.py L45-55 (strict, thresholds in float64 as numpy promotes them)
//   mode 2  polar sector   inter_domain_point_polarmix.py L76-80 / L103-119 (yaw = -arctan2(y, x) in float32,
//                          strict; optional distance test against dis_th)
//   mode 3  boxes          augmentor_utils.get_points_in_box (pcdet/datasets/augmentor/augmentor_utils.py L474-491) OR-ed over
//                          up to 96 boxes: the point filter of intra_domain_point_mixup.py L50-59 (with `invert`) and the
//                          box side of the mixers.  float32 arithmetic op by op as numpy does it (no FMA), cos / sin of -rz
//                          evaluated in double on the host (math.cos / math.sin) and rounded to float32.
// `invert` keeps the complement (np.delete / ~mask).  Optionally the batch-index column of collate_batch
// (dataset.py L173-178) is written in the same pass (`add_batch_col`), so the host can ship raw (N,F) frames.
// Two launches, no atomics, no inter-CTA waiting: tile = 1024 points; launch 1 writes the ballot words and per-tile
// counts, launch 2 sums the counts of the tiles before it, ranks by popcount and copies rows.  HBM-bound:
// algorithmic bytes = 4*stride*N read + 4*(stride+add)*N' written.
#include "common.cuh"

namespace {

constexpr int kSelThreads = 256;
constexpr int kSelTile = 1024;                 // points per CTA = 4 per thread = 32 ballot words

constexpr int kSelMaxBoxes = 96;
struct SelBox { float cx, cy, cz, hx, hy, hz, ca, sa; };   // centre, half sizes (x, y incl. margin), cos(-rz), sin(-rz)

struct SelParams {
    int mode, invert;
    float lo_x, lo_y, hi_x, hi_y;              // mode 0
    double min_x, min_y, max_x, max_y;         // mode 1
    float start, end, dis_th;                  // mode 2
    int dis_mode;                              // 0 none, 1 keep dis < dis_th, 2 keep dis > dis_th
    int nbox;                                  // mode 3
    SelBox box[kSelMaxBoxes];
};

__device__ __forceinline__ bool sel_keep(const SelParams &p, float x, float y, float z) {
    bool k;
    if (p.mode == 3) {
        k = false;
        for (int b = 0; b < p.nbox; ++b) {
            const SelBox &q = p.box[b];
            const float sx = __fsub_rn(x, q.cx), sy = __fsub_rn(y, q.cy), sz = __fsub_rn(z, q.cz);
            const float lx = __fadd_rn(__fmul_rn(sx, q.ca), __fmul_rn(sy, -q.sa));     // shift_x * cosa + shift_y * (-sina)
            const float ly = __fadd_rn(__fmul_rn(sx, q.sa), __fmul_rn(sy, q.ca));      // shift_x * sina + shift_y * cosa
            k = k || (fabsf(sz) <= q.hz && fabsf(lx) <= q.hx && fabsf(ly) <= q.hy);
        }
    } else if (p.mode == 0) {
        k = x >= p.lo_x && x <= p.hi_x && y >= p.lo_y && y <= p.hi_y;
    } else if (p.mode == 1) {
        const double xd = (double)x, yd = (double)y;
        k = xd < p.max_x && yd < p.max_y && xd > p.min_x && yd > p.min_y;
    } else {
        // float32 result of arctan2 as numpy computes it for float32 inputs; evaluated in double and rounded once
        const float yaw = -(float)atan2((double)y, (double)x);
        k = yaw > p.start && yaw < p.end;
        if (p.dis_mode) {
            const float dis = __fsqrt_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)));   // np.sqrt(x**2 + y**2), float32
            k = k && (p.dis_mode == 1 ? dis < p.dis_th : dis > p.dis_th);
        }
    }
    return k != (p.invert != 0);
}

__global__ void __launch_bounds__(kSelThreads) select_flag_kernel(const float *__restrict__ points, int n, int stride, int x_col,
                                                                  SelParams p, uint32_t *__restrict__ words,
                                                                  int *__restrict__ tile_counts) {
    __shared__ int warp_cnt[kSelThreads / 32];
    const int tile0 = blockIdx.x * kSelTile;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int cnt = 0;
#pragma unroll
    for (int j = 0; j < kSelTile / kSelThreads; ++j) {
        const int i = tile0 + j * kSelThreads + threadIdx.x;      // a warp covers 32 consecutive points = one word
        bool k = false;
        if (i < n) {
            const float *row = points + (size_t)i * stride + x_col;
            k = sel_keep(p, __ldg(row), __ldg(row + 1), p.mode == 3 ? __ldg(row + 2) : 0.f);
        }
        const uint32_t w = __ballot_sync(0xffffffffu, k);
        if (lane == 0) {
            words[(tile0 >> 5) + j * (kSelThreads / 32) + warp] = w;
            cnt += __popc(w);
        }
    }
    if (lane == 0) warp_cnt[warp] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
#pragma unroll
        for (int w = 0; w < kSelThreads / 32; ++w) t += warp_cnt[w];
        tile_counts[blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(kSelThreads) select_copy_kernel(const float *__restrict__ points, int n, int stride,
                                                                  const uint32_t *__restrict__ words,
                                                                  const int *__restrict__ tile_counts,
                                                                  const int32_t *__restrict__ frame_offsets, int batch,
                                                                  int add_batch_col, float *__restrict__ out,
                                                                  int32_t *__restrict__ out_offsets) {
    __shared__ int warp_sums[kSelThreads / 32];
    __shared__ int tile_offset_s;
    __shared__ int word_prefix[kSelTile / 32 + 1];
    __shared__ int frame_lo[65];               // frame_offsets (batch <= 64)
    __shared__ int kept_rows[kSelTile];
    __shared__ uint32_t word_s[kSelTile / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int part = 0;
    for (int j = threadIdx.x; j < (int)blockIdx.x; j += kSelThreads) part += tile_counts[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if (lane == 0) warp_sums[warp] = part;
    if (frame_offsets && (int)threadIdx.x <= batch) frame_lo[threadIdx.x] = frame_offsets[threadIdx.x];
    __syncthreads();
    const int tile0 = blockIdx.x * kSelTile;
    if (warp == 0) {
        // exclusive prefix over this tile's 32 ballot words: one word per lane, warp scan
        const uint32_t w = (tile0 + 32 * lane < n) ? words[(tile0 >> 5) + lane] : 0u;
        word_s[lane] = w;
        const int c = __popc(w);
        int incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        word_prefix[lane] = incl - c;
        if (lane == 31) word_prefix[kSelTile / 32] = incl;
        if (lane == 0) {
            int t = 0;
#pragma unroll
            for (int q = 0; q < kSelThreads / 32; ++q) t += warp_sums[q];
            tile_offset_s = t;
        }
    }
    __syncthreads();
    const int tile_offset = tile_offset_s;
    // new frame boundaries: kept points before frame_offsets[b]
    if (out_offsets) {
        if (frame_offsets) {
            if ((int)threadIdx.x <= batch) {
                const int fo = frame_lo[threadIdx.x];
                const bool mine = (fo >= tile0 && fo < tile0 + kSelTile && fo < n) || (fo >= n && tile0 <= n - 1 && n - 1 < tile0 + kSelTile) ||
                                  (n == 0 && blockIdx.x == 0);
                if (mine) {
                    int v;
                    if (fo >= n) {
                        v = tile_offset + word_prefix[kSelTile / 32];      // total (this is the last tile)
                    } else {
                        const int rel = fo - tile0, w = rel >> 5, b = rel & 31;
                        v = tile_offset + word_prefix[w] + __popc(word_s[w] & ((1u << b) - 1u));
                    }
                    out_offsets[threadIdx.x] = v;
                }
            }
        } else if (threadIdx.x == 0 && (tile0 + kSelTile >= n)) {
            out_offsets[0] = tile_offset + word_prefix[kSelTile / 32];
        }
    }
    // kept rows of this tile, in order, as a list in shared memory; then the tile's output range
    // [tile_offset, tile_offset + count) x out_stride is written element by element: stores are fully coalesced and the
    // loads walk neighbouring rows
    const int out_stride = stride + (add_batch_col ? 1 : 0);
#pragma unroll
    for (int j = 0; j < kSelTile / kSelThreads; ++j) {
        const int i = tile0 + j * kSelThreads + threadIdx.x;
        const int wi = j * (kSelThreads / 32) + warp;
        const uint32_t w = word_s[wi];
        if ((w >> lane) & 1u) kept_rows[word_prefix[wi] + __popc(w & ((1u << lane) - 1u))] = i;
    }
    __syncthreads();
    const int count = word_prefix[kSelTile / 32];
    const int total = count * out_stride;
    const float inv = 1.0f / (float)out_stride;       // e < 1024 * out_stride: (e + 0.5) * inv truncates exactly for stride <= 64
    float *o = out + (size_t)tile_offset * out_stride;
    for (int e = threadIdx.x; e < total; e += kSelThreads) {
        const int r = __float2int_rz(((float)e + 0.5f) * inv);
        const int c = e - r * out_stride;
        const int i = kept_rows[r];
        float v;
        if (add_batch_col) {
            if (c == 0) {
                int b = 0;
                if (frame_offsets)
                    for (int q = 1; q < batch; ++q) b += (i >= frame_lo[q]) ? 1 : 0;   // frame of point i (batch is small)
                v = (float)b;
            } else {
                v = __ldg(points + (size_t)i * stride + c - 1);
            }
        } else {
            v = __ldg(points + (size_t)i * stride + c);
        }
        o[e] = v;
    }
}

}  // namespace

extern "C" size_t toda_points_select_workspace_bytes(int n) {
    if (n < 0) return 0;
    size_t tiles = (size_t)ceil_div(n > 0 ? n : 1, kSelTile);
    return align_up(tiles * (kSelTile / 32) * sizeof(uint32_t), 256) + align_up(tiles * sizeof(int), 256) + 256;
}

extern "C" int toda_points_select(const float *points, int n, int stride, int x_col, const int32_t *frame_offsets, int batch,
                                  int mode, const double *params_host, int invert, int add_batch_col, float *out,
                                  int32_t *out_offsets, void *workspace, size_t workspace_bytes, void *stream) {
    TODA_CHECK_ARG(n >= 0 && stride >= 2 && stride <= 63 && x_col >= 0 && x_col + 1 < stride, "points_select: bad layout n=%d stride=%d x_col=%d", n, stride, x_col);
    TODA_CHECK_ARG(mode >= 0 && mode <= 3 && params_host, "points_select: bad mode %d", mode);
    TODA_CHECK_ARG(mode != 3 || x_col + 2 < stride, "points_select: the box test needs a z column");
    TODA_CHECK_ARG(!frame_offsets || (batch >= 1 && batch <= 64), "points_select: batch %d outside [1, 64]", batch);
    TODA_CHECK_ARG(out_offsets && workspace && (n == 0 || (points && out)), "points_select: null pointer");
    if (workspace_bytes < toda_points_select_workspace_bytes(n)) {
        toda_set_error("points_select: workspace %zu < required %zu bytes", workspace_bytes, toda_points_select_workspace_bytes(n));
        return TODA_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    SelParams p = {};
    p.mode = mode;
    p.invert = invert;
    if (mode == 0) {
        p.lo_x = (float)params_host[0]; p.lo_y = (float)params_host[1]; p.hi_x = (float)params_host[2]; p.hi_y = (float)params_host[3];
    } else if (mode == 1) {
        p.min_x = params_host[0]; p.min_y = params_host[1]; p.max_x = params_host[2]; p.max_y = params_host[3];
    } else if (mode == 3) {
        // params: [number of boxes M, margin, M x (cx, cy, cz, dx, dy, dz, rz)], every value a float32 carried in a double
        p.nbox = (int)params_host[0];
        TODA_CHECK_ARG(p.nbox >= 0 && p.nbox <= kSelMaxBoxes, "points_select: %d boxes (at most %d per call)", p.nbox, kSelMaxBoxes);
        const float margin = (float)params_host[1];
        for (int b = 0; b < p.nbox; ++b) {
            const double *g = params_host + 2 + 7 * b;
            SelBox &q = p.box[b];
            q.cx = (float)g[0]; q.cy = (float)g[1]; q.cz = (float)g[2];
            q.hx = (float)g[3] / 2.0f + margin;        // dx / 2.0 + MARGIN, float32 op by op
            q.hy = (float)g[4] / 2.0f + margin;
            q.hz = (float)g[5] / 2.0f;                 // |z - cz| <= dz / 2.0, no margin
            const double a = (double)(-(float)g[6]);   // math.cos(-rz) / math.sin(-rz) of the float32 heading, in double
            q.ca = (float)cos(a);
            q.sa = (float)sin(a);
        }
    } else {
        p.start = (float)params_host[0]; p.end = (float)params_host[1]; p.dis_th = (float)params_host[2];
        p.dis_mode = (int)params_host[3];
        TODA_CHECK_ARG(p.dis_mode >= 0 && p.dis_mode <= 2, "points_select: bad distance mode");
    }
    const int tiles = ceil_div(n > 0 ? n : 1, kSelTile);
    uint32_t *words = (uint32_t *)workspace;
    int *tile_counts = (int *)((char *)workspace + align_up((size_t)tiles * (kSelTile / 32) * sizeof(uint32_t), 256));
    select_flag_kernel<<<tiles, kSelThreads, 0, st>>>(points, n, stride, x_col, p, words, tile_counts);
    TODA_LAUNCH_OK();
    select_copy_kernel<<<tiles, kSelThreads, 0, st>>>(points, n, stride, words, tile_counts, frame_offsets, batch, add_batch_col,
                                                      out, out_offsets);
    TODA_LAUNCH_OK();
    return TODA_OK;
}

// ------------------------------------------------------------------------------------------------
// World augmentations (DataAugmentor random_world_flip / _rotation / _scaling, augmentor_utils.py L8-82), applied to the
// points of a whole batch in one elementwise pass.  Each step has per-frame parameters drawn on the host.  The float32
// arithmetic is the reference's, op by op:
//   flip x / flip y   points[:, 1] = -points[:, 1] / points[:, 0] = -points[:, 0]: a sign flip
//   scale             points[:, :3] *= noise: x * float32(noise)
//   rotate            common_utils.rotate_points_along_z: torch.matmul(xyz, [[c, s, 0], [-s, c, 0], [0, 0, 1]]) on the CPU,
//                     which for a (1, N, 3) x (1, 3, 3) product takes one of two paths by the frame's row count:
//                       N <= 44  ATen's naive bmm loop (3 * N * 3 < 400): acc = 0; acc += v[k] * R[k][j], every op rounded
//                       N >= 45  the BLAS kernel:                          acc = fma(v[k], R[k][j], acc) from acc = 0
//                     The zero and one entries of R take part, so z' = (x*0 + y*0) + z*1 and x' carries + z*0 (signed zeros,
//                     inf and NaN come out as torch gives them).
// Tile of kTfRows rows staged through shared memory: coalesced loads and stores, one thread per row in between.
namespace {

constexpr int kTfRows = 128;                   // rows per CTA = threads per CTA
constexpr int kTfMaxSteps = 4;
constexpr int kTfMaxBatch = 64;
constexpr int kTfNaiveMaxRows = 44;            // largest frame that torch rotates with the naive loop
constexpr int kTfUnroll = 8;                   // loads in flight per thread

struct TfParams {
    int n_steps;
    int kind[kTfMaxSteps];
    float2 prm[kTfMaxSteps][kTfMaxBatch];      // flip: (enabled, -); rotate: (cos, sin); scale: (noise, -)
    float zero, one;                           // the constant entries of R, passed in so that no product with them is folded
};

__device__ __forceinline__ float neg_bits(float v) { return __int_as_float(__float_as_int(v) ^ 0x80000000); }

// torch.matmul of the row (x, y, z) with column (r0, r1, r2) of the rotation matrix, as one of the two CPU paths rounds it
__device__ __forceinline__ float rot_dot(bool fused, float x, float y, float z, float r0, float r1, float r2, float zero) {
    if (fused) return __fmaf_rn(z, r2, __fmaf_rn(y, r1, __fmaf_rn(x, r0, zero)));
    return __fadd_rn(__fadd_rn(__fadd_rn(zero, __fmul_rn(x, r0)), __fmul_rn(y, r1)), __fmul_rn(z, r2));
}

__global__ void __launch_bounds__(kTfRows) world_transform_kernel(const float *__restrict__ points, int n, int stride, int x_col,
                                                                 const int32_t *__restrict__ frame_offsets, int batch,
                                                                 const TfParams p, float *__restrict__ out) {
    extern __shared__ float tile[];            // [kTfRows][stride]
    __shared__ int off_s[kTfMaxBatch + 1];
    const int row0 = blockIdx.x * kTfRows;
    const int rows = min(kTfRows, n - row0);
    const int total = rows * stride;
    const float *src = points + (size_t)row0 * stride;
    float *dst = out + (size_t)row0 * stride;
    if (frame_offsets) {
        if ((int)threadIdx.x <= batch) off_s[threadIdx.x] = frame_offsets[threadIdx.x];
    } else if (threadIdx.x == 0) {
        off_s[0] = 0;
        off_s[1] = n;
    }
    for (int e0 = 0; e0 < total; e0 += kTfRows * kTfUnroll) {
        float v[kTfUnroll];
#pragma unroll
        for (int u = 0; u < kTfUnroll; ++u) {
            const int e = e0 + u * kTfRows + threadIdx.x;
            if (e < total) v[u] = __ldg(src + e);
        }
#pragma unroll
        for (int u = 0; u < kTfUnroll; ++u) {
            const int e = e0 + u * kTfRows + threadIdx.x;
            if (e < total) tile[e] = v[u];
        }
    }
    __syncthreads();
    if ((int)threadIdx.x < rows) {
        const int i = row0 + threadIdx.x;
        const int nb = frame_offsets ? batch : 1;
        int lo = 0, hi = nb;                   // frame b: off[b] <= i < off[b+1] (the last such b: empty frames are skipped)
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (off_s[mid] <= i) lo = mid; else hi = mid;
        }
        const bool fused = off_s[lo + 1] - off_s[lo] > kTfNaiveMaxRows;
        float *r = tile + threadIdx.x * stride + x_col;
        float x = r[0], y = r[1], z = r[2];
        for (int s = 0; s < p.n_steps; ++s) {
            const float2 q = p.prm[s][lo];
            const int kind = p.kind[s];
            if (kind == TODA_WORLD_FLIP_X) {
                if (q.x != 0.f) y = neg_bits(y);
            } else if (kind == TODA_WORLD_FLIP_Y) {
                if (q.x != 0.f) x = neg_bits(x);
            } else if (kind == TODA_WORLD_ROTATE) {
                const float c = q.x, sn = q.y;
                const float xr = rot_dot(fused, x, y, z, c, neg_bits(sn), p.zero, p.zero);
                const float yr = rot_dot(fused, x, y, z, sn, c, p.zero, p.zero);
                const float zr = rot_dot(fused, x, y, z, p.zero, p.zero, p.one, p.zero);
                x = xr; y = yr; z = zr;
            } else {
                x = __fmul_rn(x, q.x); y = __fmul_rn(y, q.x); z = __fmul_rn(z, q.x);
            }
        }
        r[0] = x; r[1] = y; r[2] = z;
    }
    __syncthreads();
    for (int e = threadIdx.x; e < total; e += kTfRows) dst[e] = tile[e];
}

}  // namespace

extern "C" int toda_points_world_transform(const float *points, int n, int stride, int x_col, const int32_t *frame_offsets,
                                           int batch, int n_steps, const int *kinds_host, const float *params_host, float *out,
                                           void *stream) {
    TODA_CHECK_ARG(n >= 0 && stride >= 3 && stride <= 63 && x_col >= 0 && x_col + 2 < stride,
                   "points_world_transform: bad layout n=%d stride=%d x_col=%d", n, stride, x_col);
    TODA_CHECK_ARG(!frame_offsets || (batch >= 1 && batch <= kTfMaxBatch), "points_world_transform: batch %d outside [1, %d]",
                   batch, kTfMaxBatch);
    TODA_CHECK_ARG(n_steps >= 0 && n_steps <= kTfMaxSteps, "points_world_transform: %d steps (at most %d)", n_steps, kTfMaxSteps);
    TODA_CHECK_ARG(n_steps == 0 || (kinds_host && params_host), "points_world_transform: null step list");
    TODA_CHECK_ARG(n == 0 || (points && out), "points_world_transform: null pointer");
    const int nb = frame_offsets ? batch : 1;
    TfParams p = {};
    p.n_steps = n_steps;
    p.zero = 0.f;
    p.one = 1.f;
    for (int s = 0; s < n_steps; ++s) {
        const int k = kinds_host[s];
        TODA_CHECK_ARG(k >= TODA_WORLD_FLIP_X && k <= TODA_WORLD_SCALE, "points_world_transform: bad step kind %d", k);
        p.kind[s] = k;
        for (int b = 0; b < nb; ++b) p.prm[s][b] = make_float2(params_host[2 * (s * nb + b)], params_host[2 * (s * nb + b) + 1]);
    }
    if (n == 0) return TODA_OK;
    const size_t smem = (size_t)kTfRows * stride * sizeof(float);
    world_transform_kernel<<<ceil_div(n, kTfRows), kTfRows, smem, (cudaStream_t)stream>>>(points, n, stride, x_col, frame_offsets,
                                                                                          batch, p, out);
    TODA_LAUNCH_OK();
    return TODA_OK;
}
