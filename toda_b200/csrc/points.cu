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

// the predicate of toda_points_select: one of the four modes above on the row's x, y (and z)
struct SelKeep {
    const float *points;
    int stride, x_col;
    SelParams p;
    __device__ __forceinline__ bool operator()(int i) const {
        const float *row = points + (size_t)i * stride + x_col;
        return sel_keep(p, __ldg(row), __ldg(row + 1), p.mode == 3 ? __ldg(row + 2) : 0.f);
    }
};

// launch 1 of the compaction: ballot words and per-tile counts of rows i < n for which keep(i) holds
template <class Keep>
__global__ void __launch_bounds__(kSelThreads) select_flag_kernel(int n, const Keep keep, uint32_t *__restrict__ words,
                                                                  int *__restrict__ tile_counts) {
    __shared__ int warp_cnt[kSelThreads / 32];
    const int tile0 = blockIdx.x * kSelTile;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int cnt = 0;
#pragma unroll
    for (int j = 0; j < kSelTile / kSelThreads; ++j) {
        const int i = tile0 + j * kSelThreads + threadIdx.x;      // a warp covers 32 consecutive points = one word
        const bool k = i < n && keep(i);
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
                                                                  int add_batch_col, const int *__restrict__ frame_lead,
                                                                  float *__restrict__ out, int32_t *__restrict__ out_offsets) {
    __shared__ int warp_sums[kSelThreads / 32];
    __shared__ int tile_offset_s;
    __shared__ int word_prefix[kSelTile / 32 + 1];
    __shared__ int frame_lo[65];               // frame_offsets (batch <= 64)
    __shared__ int lead_lo[65];                // rows written in front of the kept rows of the frames before b
    __shared__ int kept_rows[kSelTile];
    __shared__ unsigned char kept_frame[kSelTile];
    __shared__ uint32_t word_s[kSelTile / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int part = 0;
    for (int j = threadIdx.x; j < (int)blockIdx.x; j += kSelThreads) part += tile_counts[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if (lane == 0) warp_sums[warp] = part;
    if (frame_offsets && (int)threadIdx.x <= batch) frame_lo[threadIdx.x] = frame_offsets[threadIdx.x];
    if (frame_lead && threadIdx.x == 0) {
        int t = 0;
        for (int q = 0; q < batch; ++q) {
            lead_lo[q] = t;
            t += frame_lead[q];
        }
        lead_lo[batch] = t;
    }
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
                    out_offsets[threadIdx.x] = v + (frame_lead ? lead_lo[threadIdx.x] : 0);
                }
            }
        } else if (threadIdx.x == 0 && (tile0 + kSelTile >= n)) {
            out_offsets[0] = tile_offset + word_prefix[kSelTile / 32];
        }
    }
    // kept rows of this tile, in order, as a list in shared memory (with their frame where it is needed); then the
    // tile's output range [tile_offset, tile_offset + count) x out_stride is written element by element: stores are
    // fully coalesced and the loads walk neighbouring rows.  With frame_lead, the rows of frame b move down by the
    // frame_lead rows of frames 0..b (a gap in front of each frame's rows, filled by the caller).
    const int out_stride = stride + (add_batch_col ? 1 : 0);
    const bool need_frame = frame_offsets && (add_batch_col || frame_lead);
#pragma unroll
    for (int j = 0; j < kSelTile / kSelThreads; ++j) {
        const int i = tile0 + j * kSelThreads + threadIdx.x;
        const int wi = j * (kSelThreads / 32) + warp;
        const uint32_t w = word_s[wi];
        if ((w >> lane) & 1u) {
            const int r = word_prefix[wi] + __popc(w & ((1u << lane) - 1u));
            kept_rows[r] = i;
            if (need_frame) {
                int b = 0;
                for (int q = 1; q < batch; ++q) b += (i >= frame_lo[q]) ? 1 : 0;   // frame of point i (batch is small)
                kept_frame[r] = (unsigned char)b;
            }
        }
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
                v = frame_offsets ? (float)kept_frame[r] : 0.f;
            } else {
                v = __ldg(points + (size_t)i * stride + c - 1);
            }
        } else {
            v = __ldg(points + (size_t)i * stride + c);
        }
        if (frame_lead) o[e + (size_t)lead_lo[kept_frame[r] + 1] * out_stride] = v;
        else o[e] = v;
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
    select_flag_kernel<<<tiles, kSelThreads, 0, st>>>(n, SelKeep{points, stride, x_col, p}, words, tile_counts);
    TODA_LAUNCH_OK();
    select_copy_kernel<<<tiles, kSelThreads, 0, st>>>(points, n, stride, words, tile_counts, frame_offsets, batch, add_batch_col,
                                                      nullptr, out, out_offsets);
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

// ------------------------------------------------------------------------------------------------
// gt_sampling (DataBaseSampler.__call__ / add_sampled_boxes_to_scene, pcdet/datasets/augmentor/database_sampler.py;
// OpenPCDet v0.5.2) for a whole batch: the sampled database boxes are drawn on the host, the rest runs here in four
// launches on the stream, with no host synchronisation:
//   1 gts_accept_kernel   one CTA per frame.  Classes in SAMPLE_GROUPS order; every sample of a class is tested against
//                         the frame's gt boxes, the boxes accepted for earlier classes (shared memory) and the other
//                         samples of its class, all pairs of a class in parallel.  A sample is accepted iff every iou_bev
//                         is exactly 0 (boxes_bev_iou_cpu, iou1.max + iou2.max == 0).  Writes the accepted flags, the
//                         accepted boxes enlarged by REMOVE_EXTRA_WIDTH, and where each accepted sample's object rows go.
//   2 select_flag_kernel  (K0 compaction, launch 1) scene rows outside every accepted box of their frame
//                         (remove_points_in_boxes3d / points_in_boxes_cpu semantics); the frame by binary search.
//   3 select_copy_kernel  (K0 compaction, launch 2) kept rows, each frame moved down by its object rows.
//   4 gts_paste_kernel    one CTA per sample: the object rows of the accepted samples in front of their frame's rows,
//                         shifted by the database box centre.
// The float32 arithmetic is that of the compiled ops, op by op without FMA (iou3d_cpu.cpp box_overlap, roiaware_pool3d.cpp
// check_pt_in_box3d_cpu); cos / sin of the headings come from the host (toda_gt_sampling_pack_boxes, libm cosf / sinf),
// and point_cmp's atan2f is the fdlibm float algorithm that glibc's libm implements, restated below.
namespace {

constexpr int kGtsThreads = 256;
constexpr int kGtsMaxSamples = 1024;           // sampled boxes per frame (shared memory of gts_accept_kernel)
constexpr int kGtsMaxGroups = 16;
constexpr int kGtsMaxBatch = 64;
constexpr int kGtsBoxFloats = 16;              // packed box: see include/toda_b200.h

struct GtsFrames {
    int n_groups;
    int exist_off[kGtsMaxBatch + 1];           // gt boxes of frame b: [exist_off[b], exist_off[b+1])
    int samp_off[kGtsMaxBatch + 1];            // sampled boxes of frame b, grouped by class in SAMPLE_GROUPS order
    unsigned short group_size[kGtsMaxBatch][kGtsMaxGroups];
};

struct BevBox { float cx, cy, dx, dy, ca, sa, cna, sna; };   // cos / sin of rz and of -rz

__device__ __forceinline__ BevBox load_bev(const float4 *__restrict__ boxes, int i) {
    const float4 u = __ldg(boxes + 4 * i), v = __ldg(boxes + 4 * i + 1), w = __ldg(boxes + 4 * i + 2);
    return BevBox{u.x, u.y, u.w, v.x, v.z, v.w, w.x, w.y};
}

// ---- atan2f as glibc's libm computes it (sysdeps/ieee754/flt-32/e_atan2f.c, s_atanf.c: the fdlibm float algorithm)
__device__ __forceinline__ float ref_atanf(float x) {
    const float atanhi[4] = {4.6364760399e-01f, 7.8539812565e-01f, 9.8279368877e-01f, 1.5707962513e+00f};
    const float atanlo[4] = {5.0121582440e-09f, 3.7748947079e-08f, 3.4473217170e-08f, 7.5497894159e-08f};
    const int hx = __float_as_int(x), ix = hx & 0x7fffffff;
    int id;
    if (ix >= 0x4c000000) {                    // |x| >= 2^25
        if (ix > 0x7f800000) return __fadd_rn(x, x);
        return hx > 0 ? __fadd_rn(atanhi[3], atanlo[3]) : __fsub_rn(-atanhi[3], atanlo[3]);
    }
    if (ix < 0x3ee00000) {                     // |x| < 0.4375
        if (ix < 0x31000000) return x;         // |x| < 2^-29
        id = -1;
    } else {
        x = fabsf(x);
        if (ix < 0x3f980000) {
            if (ix < 0x3f300000) { id = 0; x = __fdiv_rn(__fsub_rn(__fmul_rn(2.0f, x), 1.0f), __fadd_rn(2.0f, x)); }
            else { id = 1; x = __fdiv_rn(__fsub_rn(x, 1.0f), __fadd_rn(x, 1.0f)); }
        } else {
            if (ix < 0x401c0000) { id = 2; x = __fdiv_rn(__fsub_rn(x, 1.5f), __fadd_rn(1.0f, __fmul_rn(1.5f, x))); }
            else { id = 3; x = __fdiv_rn(-1.0f, x); }
        }
    }
    const float z = __fmul_rn(x, x), w = __fmul_rn(z, z);
    const float s1 = __fmul_rn(z, __fadd_rn(3.3333334327e-01f, __fmul_rn(w, __fadd_rn(1.4285714924e-01f, __fmul_rn(w,
                     __fadd_rn(9.0908870101e-02f, __fmul_rn(w, __fadd_rn(6.6610731184e-02f, __fmul_rn(w,
                     __fadd_rn(4.9768779427e-02f, __fmul_rn(w, 1.6285819933e-02f)))))))))));
    const float s2 = __fmul_rn(w, __fadd_rn(-2.0000000298e-01f, __fmul_rn(w, __fadd_rn(-1.1111110449e-01f, __fmul_rn(w,
                     __fadd_rn(-7.6918758452e-02f, __fmul_rn(w, __fadd_rn(-5.8335702866e-02f, __fmul_rn(w, -3.6531571299e-02f)))))))));
    if (id < 0) return __fsub_rn(x, __fmul_rn(x, __fadd_rn(s1, s2)));
    const float r = __fsub_rn(atanhi[id], __fsub_rn(__fsub_rn(__fmul_rn(x, __fadd_rn(s1, s2)), atanlo[id]), x));
    return hx < 0 ? -r : r;
}

__device__ __forceinline__ float ref_atan2f(float y, float x) {
    const float tiny = 1.0e-30f, pi_o_4 = 7.8539818525e-01f, pi_o_2 = 1.5707963705e+00f, pi = 3.1415927410e+00f,
                pi_lo = -8.7422776573e-08f;
    const int hx = __float_as_int(x), ix = hx & 0x7fffffff, hy = __float_as_int(y), iy = hy & 0x7fffffff;
    if (ix > 0x7f800000 || iy > 0x7f800000) return __fadd_rn(x, y);
    if (hx == 0x3f800000) return ref_atanf(y);
    const int m = ((hy >> 31) & 1) | ((hx >> 30) & 2);
    if (iy == 0) {
        if (m < 2) return y;
        return m == 2 ? __fadd_rn(pi, tiny) : __fsub_rn(-pi, tiny);
    }
    if (ix == 0) return hy < 0 ? __fsub_rn(-pi_o_2, tiny) : __fadd_rn(pi_o_2, tiny);
    if (ix == 0x7f800000) {
        if (iy == 0x7f800000) {
            if (m == 0) return __fadd_rn(pi_o_4, tiny);
            if (m == 1) return __fsub_rn(-pi_o_4, tiny);
            if (m == 2) return __fadd_rn(__fmul_rn(3.0f, pi_o_4), tiny);
            return __fsub_rn(__fmul_rn(-3.0f, pi_o_4), tiny);
        }
        if (m == 0) return 0.0f;
        if (m == 1) return -0.0f;
        return m == 2 ? __fadd_rn(pi, tiny) : __fsub_rn(-pi, tiny);
    }
    if (iy == 0x7f800000) return hy < 0 ? __fsub_rn(-pi_o_2, tiny) : __fadd_rn(pi_o_2, tiny);
    const int k = (iy - ix) >> 23;
    float z;
    if (k > 60) z = __fadd_rn(pi_o_2, __fmul_rn(0.5f, pi_lo));
    else if (hx < 0 && k < -60) z = 0.0f;
    else z = ref_atanf(fabsf(__fdiv_rn(y, x)));
    if (m == 0) return z;
    if (m == 1) return __int_as_float(__float_as_int(z) ^ 0x80000000);
    if (m == 2) return __fsub_rn(pi, __fsub_rn(z, pi_lo));
    return __fsub_rn(__fsub_rn(z, pi_lo), pi);
}

// ---- iou3d_cpu.cpp, float32 op by op
__device__ __forceinline__ float ref_min(float a, float b) { return a > b ? b : a; }
__device__ __forceinline__ float ref_max(float a, float b) { return a > b ? a : b; }

__device__ __forceinline__ float cross3(float2 p1, float2 p2, float2 p0) {      // cross(p1, p2, p0)
    return __fsub_rn(__fmul_rn(__fsub_rn(p1.x, p0.x), __fsub_rn(p2.y, p0.y)), __fmul_rn(__fsub_rn(p2.x, p0.x), __fsub_rn(p1.y, p0.y)));
}

__device__ __forceinline__ bool check_rect_cross(float2 p1, float2 p2, float2 q1, float2 q2) {
    return ref_min(p1.x, p2.x) <= ref_max(q1.x, q2.x) && ref_min(q1.x, q2.x) <= ref_max(p1.x, p2.x) &&
           ref_min(p1.y, p2.y) <= ref_max(q1.y, q2.y) && ref_min(q1.y, q2.y) <= ref_max(p1.y, p2.y);
}

__device__ __forceinline__ bool check_in_box2d(const BevBox &b, float2 p) {
    const float sx = __fsub_rn(p.x, b.cx), sy = __fsub_rn(p.y, b.cy);
    const float rx = __fadd_rn(__fmul_rn(sx, b.cna), __fmul_rn(sy, -b.sna));
    const float ry = __fadd_rn(__fmul_rn(sx, b.sna), __fmul_rn(sy, b.cna));
    return fabsf(rx) < __fadd_rn(__fdiv_rn(b.dx, 2.0f), 1e-2f) && fabsf(ry) < __fadd_rn(__fdiv_rn(b.dy, 2.0f), 1e-2f);
}

__device__ __forceinline__ bool intersection(float2 p1, float2 p0, float2 q1, float2 q0, float2 &ans) {
    if (!check_rect_cross(p0, p1, q0, q1)) return false;
    const float s1 = cross3(q0, p1, p0), s2 = cross3(p1, q1, p0), s3 = cross3(p0, q1, q0), s4 = cross3(q1, p1, q0);
    if (!(__fmul_rn(s1, s2) > 0.f && __fmul_rn(s3, s4) > 0.f)) return false;
    const float s5 = cross3(q1, p1, p0);
    const float d = __fsub_rn(s5, s1);
    if (fabsf(d) > 1e-8f) {
        ans.x = __fdiv_rn(__fsub_rn(__fmul_rn(s5, q0.x), __fmul_rn(s1, q1.x)), d);
        ans.y = __fdiv_rn(__fsub_rn(__fmul_rn(s5, q0.y), __fmul_rn(s1, q1.y)), d);
    } else {
        const float a0 = __fsub_rn(p0.y, p1.y), b0 = __fsub_rn(p1.x, p0.x);
        const float c0 = __fsub_rn(__fmul_rn(p0.x, p1.y), __fmul_rn(p1.x, p0.y));
        const float a1 = __fsub_rn(q0.y, q1.y), b1 = __fsub_rn(q1.x, q0.x);
        const float c1 = __fsub_rn(__fmul_rn(q0.x, q1.y), __fmul_rn(q1.x, q0.y));
        const float D = __fsub_rn(__fmul_rn(a0, b1), __fmul_rn(a1, b0));
        ans.x = __fdiv_rn(__fsub_rn(__fmul_rn(b0, c1), __fmul_rn(b1, c0)), D);
        ans.y = __fdiv_rn(__fsub_rn(__fmul_rn(a1, c0), __fmul_rn(a0, c1)), D);
    }
    return true;
}

__device__ __forceinline__ float2 rotate_around_center(float2 c, float cs, float sn, float2 p) {
    const float sx = __fsub_rn(p.x, c.x), sy = __fsub_rn(p.y, c.y);
    return make_float2(__fadd_rn(__fadd_rn(__fmul_rn(sx, cs), __fmul_rn(sy, -sn)), c.x),
                       __fadd_rn(__fadd_rn(__fmul_rn(sx, sn), __fmul_rn(sy, cs)), c.y));
}

__device__ __forceinline__ float box_overlap(const BevBox &a, const BevBox &b) {
    const float adx = __fdiv_rn(a.dx, 2.0f), ady = __fdiv_rn(a.dy, 2.0f), bdx = __fdiv_rn(b.dx, 2.0f), bdy = __fdiv_rn(b.dy, 2.0f);
    const float ax1 = __fsub_rn(a.cx, adx), ay1 = __fsub_rn(a.cy, ady), ax2 = __fadd_rn(a.cx, adx), ay2 = __fadd_rn(a.cy, ady);
    const float bx1 = __fsub_rn(b.cx, bdx), by1 = __fsub_rn(b.cy, bdy), bx2 = __fadd_rn(b.cx, bdx), by2 = __fadd_rn(b.cy, bdy);
    const float2 ca = make_float2(a.cx, a.cy), cb = make_float2(b.cx, b.cy);
    float2 pa[5], pb[5];
    pa[0] = make_float2(ax1, ay1); pa[1] = make_float2(ax2, ay1); pa[2] = make_float2(ax2, ay2); pa[3] = make_float2(ax1, ay2);
    pb[0] = make_float2(bx1, by1); pb[1] = make_float2(bx2, by1); pb[2] = make_float2(bx2, by2); pb[3] = make_float2(bx1, by2);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        pa[k] = rotate_around_center(ca, a.ca, a.sa, pa[k]);
        pb[k] = rotate_around_center(cb, b.ca, b.sa, pb[k]);
    }
    pa[4] = pa[0];
    pb[4] = pb[0];
    float2 pts[16];
    float2 center = make_float2(0.f, 0.f);
    int cnt = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float2 q;
            if (intersection(pa[i + 1], pa[i], pb[j + 1], pb[j], q)) {
                center = make_float2(__fadd_rn(center.x, q.x), __fadd_rn(center.y, q.y));
                pts[cnt++] = q;
            }
        }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (check_in_box2d(a, pb[k])) {
            center = make_float2(__fadd_rn(center.x, pb[k].x), __fadd_rn(center.y, pb[k].y));
            pts[cnt++] = pb[k];
        }
        if (check_in_box2d(b, pa[k])) {
            center = make_float2(__fadd_rn(center.x, pa[k].x), __fadd_rn(center.y, pa[k].y));
            pts[cnt++] = pa[k];
        }
    }
    if (cnt < 2) return 0.f;                   // the reference's area loop does not run: fabs(0) / 2
    center.x = __fdiv_rn(center.x, (float)cnt);
    center.y = __fdiv_rn(center.y, (float)cnt);
    // point_cmp's bubble sort; the angle of a point depends only on the point, so it is computed once per point
    float ang[16];
    for (int k = 0; k < cnt; ++k) ang[k] = ref_atan2f(__fsub_rn(pts[k].y, center.y), __fsub_rn(pts[k].x, center.x));
    for (int j = 0; j < cnt - 1; ++j) {
        for (int i = 0; i < cnt - j - 1; ++i) {
            if (ang[i] > ang[i + 1]) {
                const float2 t = pts[i]; pts[i] = pts[i + 1]; pts[i + 1] = t;
                const float ta = ang[i]; ang[i] = ang[i + 1]; ang[i + 1] = ta;
            }
        }
    }
    float area = 0.f;
    for (int k = 0; k < cnt - 1; ++k) {
        const float d0x = __fsub_rn(pts[k].x, pts[0].x), d0y = __fsub_rn(pts[k].y, pts[0].y);
        const float d1x = __fsub_rn(pts[k + 1].x, pts[0].x), d1y = __fsub_rn(pts[k + 1].y, pts[0].y);
        area = __fadd_rn(area, __fsub_rn(__fmul_rn(d0x, d1y), __fmul_rn(d0y, d1x)));
    }
    return (float)(fabs((double)area) / 2.0);
}

__device__ __forceinline__ float iou_bev(const BevBox &a, const BevBox &b) {
    const float sa = __fmul_rn(a.dx, a.dy), sb = __fmul_rn(b.dx, b.dy);
    const float s = box_overlap(a, b);
    return __fdiv_rn(s, fmaxf(__fsub_rn(__fadd_rn(sa, sb), s), 1e-8f));
}

__global__ void __launch_bounds__(kGtsThreads, 1) gts_accept_kernel(const float4 *__restrict__ exist, const float4 *__restrict__ samp,
                                                                 const long long *__restrict__ samp_rows, const GtsFrames f,
                                                                 int32_t *__restrict__ accepted, float4 *__restrict__ rm_boxes,
                                                                 int *__restrict__ frame_stats, int *__restrict__ obj_dst) {
    extern __shared__ BevBox acc_s[];          // boxes accepted so far in this frame (they join existed_boxes)
    __shared__ int rej_s[kGtsMaxSamples];
    __shared__ int n_acc_s, rows_s;
    const int b = blockIdx.x, batch = gridDim.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int e0 = f.exist_off[b], ne = f.exist_off[b + 1] - e0;
    if (threadIdx.x == 0) {
        n_acc_s = 0;
        rows_s = 0;
    }
    int s_begin = f.samp_off[b];
    for (int g = 0; g < f.n_groups; ++g) {
        const int ns = f.group_size[b][g];
        if (ns == 0) continue;
        for (int t = threadIdx.x; t < ns; t += kGtsThreads) rej_s[t] = 0;
        __syncthreads();
        const int na = n_acc_s;
        const int others = ne + na + ns;       // iou1 columns (gt boxes, then accepted samples), then iou2 columns
        for (int q = threadIdx.x; q < ns * others; q += kGtsThreads) {
            const int i = q / others, j = q - i * others;
            if (j == ne + na + i) continue;    // iou2's diagonal is zeroed
            const BevBox a = load_bev(samp, s_begin + i);
            const BevBox o = j < ne ? load_bev(exist, e0 + j) : j < ne + na ? acc_s[j - ne] : load_bev(samp, s_begin + j - ne - na);
            if (!(iou_bev(a, o) == 0.f)) rej_s[i] = 1;   // a NaN iou rejects too (numpy's max propagates it)
        }
        __syncthreads();
        if (warp == 0) {
            int na2 = na, rows = rows_s;
            for (int c = 0; c < ns; c += 32) {
                const int k = c + lane, s = s_begin + k;
                const bool ok = k < ns && rej_s[k] == 0;
                const uint32_t m = __ballot_sync(0xffffffffu, ok);
                const int cnt = ok ? (int)samp_rows[2 * s + 1] : 0;
                int incl = cnt;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int t = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= o) incl += t;
                }
                if (k < ns) {
                    accepted[s] = ok ? 1 : 0;
                    obj_dst[s] = ok ? rows + incl - cnt : -1;
                }
                if (ok) {
                    const int slot = na2 + __popc(m & ((1u << lane) - 1u));
                    acc_s[slot] = load_bev(samp, s);
                    const float4 u = __ldg(samp + 4 * s), v = __ldg(samp + 4 * s + 1), w = __ldg(samp + 4 * s + 2),
                                 x = __ldg(samp + 4 * s + 3);
                    rm_boxes[2 * (f.samp_off[b] + slot)] = make_float4(u.x, u.y, u.z, w.x);       // cx, cy, cz, cos(-rz)
                    rm_boxes[2 * (f.samp_off[b] + slot) + 1] = make_float4(w.y, w.z, w.w, x.x);   // sin(-rz), enlarged dx, dy, dz
                }
                na2 += __popc(m);
                rows += __shfl_sync(0xffffffffu, incl, 31);
            }
            if (lane == 0) {
                n_acc_s = na2;
                rows_s = rows;
            }
        }
        __syncthreads();
        s_begin += ns;
    }
    if (threadIdx.x == 0) {
        frame_stats[b] = n_acc_s;
        frame_stats[batch + b] = rows_s;
        frame_stats[2 * batch + b] = f.samp_off[b];
    }
}

// roiaware_pool3d.cpp check_pt_in_box3d_cpu: the z test and the half sizes plus margin in double, the local coordinates in
// float32; ca / sa = cosf(-rz) / sinf(-rz) of the box heading rz
__device__ __forceinline__ bool pt_in_box3d(float x, float y, float z, float cx, float cy, float cz, float ca, float sa,
                                            float dx, float dy, float dz) {
    if ((double)fabsf(__fsub_rn(z, cz)) > (double)dz / 2.0) return false;
    const float sx = __fsub_rn(x, cx), sy = __fsub_rn(y, cy);
    const float lx = __fadd_rn(__fmul_rn(sx, ca), __fmul_rn(sy, -sa));
    const float ly = __fadd_rn(__fmul_rn(sx, sa), __fmul_rn(sy, ca));
    return (double)fabsf(lx) < __dadd_rn((double)dx / 2.0, (double)1e-2f) &&
           (double)fabsf(ly) < __dadd_rn((double)dy / 2.0, (double)1e-2f);
}

// the predicate of the scene-point removal: the row lies in none of its frame's accepted boxes
struct GtsOutsideBoxes {
    const float *points;
    int stride, x_col, batch;
    const int32_t *frame_offsets;
    const float4 *rm_boxes;
    const int *frame_stats;
    __device__ __forceinline__ bool operator()(int i) const {
        int lo = 0, hi = batch;                // frame b: off[b] <= i < off[b+1] (the last such b: empty frames are skipped)
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (__ldg(frame_offsets + mid) <= i) lo = mid; else hi = mid;
        }
        const int nb = __ldg(frame_stats + lo), r0 = __ldg(frame_stats + 2 * batch + lo);
        const float *row = points + (size_t)i * stride + x_col;
        const float x = __ldg(row), y = __ldg(row + 1), z = __ldg(row + 2);
        for (int k = 0; k < nb; ++k) {
            const float4 u = __ldg(rm_boxes + 2 * (r0 + k)), v = __ldg(rm_boxes + 2 * (r0 + k) + 1);
            if (pt_in_box3d(x, y, z, u.x, u.y, u.z, u.w, v.x, v.y, v.z, v.w)) return false;
        }
        return true;
    }
};

__global__ void __launch_bounds__(kGtsThreads) gts_paste_kernel(const float *__restrict__ db_points, int feat,
                                                                const long long *__restrict__ samp_rows,
                                                                const double *__restrict__ samp_shift, int shift_f64,
                                                                const int32_t *__restrict__ accepted,
                                                                const int *__restrict__ obj_dst, const GtsFrames f, int batch,
                                                                int x_col, const int32_t *__restrict__ out_offsets,
                                                                float *__restrict__ out) {
    const int s = blockIdx.x;
    if (!accepted[s]) return;
    int b = 0;
    while (b + 1 < batch && f.samp_off[b + 1] <= s) ++b;
    const long long first = samp_rows[2 * s];
    const int cnt = (int)samp_rows[2 * s + 1];
    const int out_stride = x_col + feat;
    const double sh[3] = {samp_shift[3 * s], samp_shift[3 * s + 1], samp_shift[3 * s + 2]};
    float *o = out + ((size_t)out_offsets[b] + obj_dst[s]) * out_stride;
    const float *src = db_points + (size_t)first * feat;
    for (int e = threadIdx.x; e < cnt * out_stride; e += kGtsThreads) {
        const int r = e / out_stride, c = e - r * out_stride - x_col;
        float v;
        if (c < 0) {
            v = (float)b;                      // the batch column of collate_batch
        } else {
            v = __ldg(src + (size_t)r * feat + c);
            if (c < 3)                         // obj_points[:, :3] += box3d_lidar[:3], in the database box's dtype
                v = shift_f64 ? (float)__dadd_rn((double)v, sh[c]) : __fadd_rn(v, (float)sh[c]);
        }
        o[e] = v;
    }
}

}  // namespace

extern "C" int toda_gt_sampling_pack_boxes(const float *boxes_host, int n, const float *extra_width_host, float *packed_host) {
    TODA_CHECK_ARG(n >= 0 && (n == 0 || (boxes_host && packed_host)), "gt_sampling_pack_boxes: bad arguments (n=%d)", n);
    for (int i = 0; i < n; ++i) {
        const float *g = boxes_host + 7 * i;
        float *q = packed_host + kGtsBoxFloats * i;
        for (int k = 0; k < 6; ++k) q[k] = g[k];
        // libm cosf / sinf of the float32 heading, as the compiled ops call cos / sin on a float
        q[6] = cosf(g[6]);
        q[7] = sinf(g[6]);
        q[8] = cosf(-g[6]);
        q[9] = sinf(-g[6]);
        for (int k = 0; k < 3; ++k) q[10 + k] = extra_width_host ? g[3 + k] + extra_width_host[k] : g[3 + k];   // enlarge_box3d
        q[13] = q[14] = q[15] = 0.f;
    }
    return TODA_OK;
}

extern "C" size_t toda_gt_sampling_workspace_bytes(int n, int batch, int n_samples) {
    if (n < 0 || batch < 0 || n_samples < 0) return 0;
    return toda_points_select_workspace_bytes(n) + align_up((size_t)n_samples * 2 * sizeof(float4), 256) +
           align_up((size_t)n_samples * sizeof(int), 256) + align_up((size_t)batch * 3 * sizeof(int), 256);
}

extern "C" int toda_gt_sampling(const float *points, int n, int stride, int x_col, const int32_t *frame_offsets, int batch,
                                const float *exist_boxes, const int *exist_offsets_host, const float *samp_boxes,
                                const int *group_sizes_host, int n_groups, const float *db_points, int db_features,
                                const int64_t *samp_rows, const double *samp_shift, int shift_f64, float *out,
                                int32_t *out_offsets, int32_t *accepted, void *workspace, size_t workspace_bytes, void *stream) {
    TODA_CHECK_ARG(n >= 0 && (x_col == 0 || x_col == 1) && db_features >= 3 && stride == x_col + db_features && stride <= 63,
                   "gt_sampling: bad layout n=%d stride=%d x_col=%d features=%d", n, stride, x_col, db_features);
    TODA_CHECK_ARG(batch >= 1 && batch <= kGtsMaxBatch, "gt_sampling: batch %d outside [1, %d]", batch, kGtsMaxBatch);
    TODA_CHECK_ARG(n_groups >= 1 && n_groups <= kGtsMaxGroups, "gt_sampling: %d sample groups (at most %d)", n_groups, kGtsMaxGroups);
    TODA_CHECK_ARG(exist_offsets_host && group_sizes_host && frame_offsets && out_offsets && accepted && workspace &&
                   (n == 0 || (points && out)), "gt_sampling: null pointer");
    GtsFrames f = {};
    f.n_groups = n_groups;
    int max_frame = 0;
    for (int b = 0; b < batch; ++b) {
        TODA_CHECK_ARG(exist_offsets_host[b] >= 0 && exist_offsets_host[b + 1] >= exist_offsets_host[b],
                       "gt_sampling: gt box offsets are not ascending at frame %d", b);
        f.exist_off[b] = exist_offsets_host[b];
        int frame = 0;
        for (int g = 0; g < n_groups; ++g) {
            const int k = group_sizes_host[b * n_groups + g];
            TODA_CHECK_ARG(k >= 0, "gt_sampling: negative group size");
            frame += k;
            if (frame > kGtsMaxSamples) {
                toda_set_error("gt_sampling: frame %d has more than %d sampled boxes", b, kGtsMaxSamples);
                return TODA_ERR_UNSUPPORTED;
            }
            f.group_size[b][g] = (unsigned short)k;
        }
        f.samp_off[b + 1] = f.samp_off[b] + frame;
        max_frame = frame > max_frame ? frame : max_frame;
    }
    f.exist_off[batch] = exist_offsets_host[batch];
    const int n_samples = f.samp_off[batch];
    TODA_CHECK_ARG(n_samples == 0 || (samp_boxes && db_points && samp_rows && samp_shift), "gt_sampling: null sample table");
    TODA_CHECK_ARG(f.exist_off[batch] == 0 || exist_boxes, "gt_sampling: null gt box table");
    if (workspace_bytes < toda_gt_sampling_workspace_bytes(n, batch, n_samples)) {
        toda_set_error("gt_sampling: workspace %zu < required %zu bytes", workspace_bytes,
                       toda_gt_sampling_workspace_bytes(n, batch, n_samples));
        return TODA_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int tiles = ceil_div(n > 0 ? n : 1, kSelTile);
    char *ws = (char *)workspace;
    uint32_t *words = (uint32_t *)ws;
    int *tile_counts = (int *)(ws + align_up((size_t)tiles * (kSelTile / 32) * sizeof(uint32_t), 256));
    ws += toda_points_select_workspace_bytes(n);
    float4 *rm_boxes = (float4 *)ws;
    ws += align_up((size_t)n_samples * 2 * sizeof(float4), 256);
    int *obj_dst = (int *)ws;
    ws += align_up((size_t)n_samples * sizeof(int), 256);
    int *frame_stats = (int *)ws;              // [3][batch]: accepted boxes, object rows, first removal box

    gts_accept_kernel<<<batch, kGtsThreads, (size_t)max_frame * sizeof(BevBox), st>>>(
        (const float4 *)exist_boxes, (const float4 *)samp_boxes, (const long long *)samp_rows, f, accepted, rm_boxes,
        frame_stats, obj_dst);
    TODA_LAUNCH_OK();
    select_flag_kernel<<<tiles, kSelThreads, 0, st>>>(
        n, GtsOutsideBoxes{points, stride, x_col, batch, frame_offsets, rm_boxes, frame_stats}, words, tile_counts);
    TODA_LAUNCH_OK();
    select_copy_kernel<<<tiles, kSelThreads, 0, st>>>(points, n, stride, words, tile_counts, frame_offsets, batch, 0,
                                                      frame_stats + batch, out, out_offsets);
    TODA_LAUNCH_OK();
    if (n_samples > 0) {
        gts_paste_kernel<<<n_samples, kGtsThreads, 0, st>>>(db_points, db_features, (const long long *)samp_rows, samp_shift,
                                                            shift_f64, accepted, obj_dst, f, batch, x_col, out_offsets, out);
        TODA_LAUNCH_OK();
    }
    return TODA_OK;
}

// ------------------------------------------------------------------------------------------------
// PolarMix rotate-pasting (rotate_copy and the instance paste of Xiao et al., NeurIPS 2022; TODA's
// inter_domain_point_polarmix.py L153-191) for a whole batch, adapted to boxes with gt_sampling's collision rule.  The
// candidate boxes (every instance box rotated by every angle of its frame) are made on the host; five launches and one
// device-to-host copy:
//   1 rp_member_kernel    one CTA per 1024 source rows of a frame (tiles start at frame starts): for every instance box
//                         of the frame, ballot words and per-tile counts of the rows inside the unrotated, unenlarged box
//                         (check_pt_in_box3d_cpu, pt_in_box3d above).  Each row is tested once per box, not per angle.
//   2 rp_box_rows_kernel  one CTA per instance box: its row count, written as the row count of each of its candidates.
//   3 gts_accept_kernel   gt_sampling's collision test with the angles as the sample groups: a candidate is accepted iff
//                         its iou_bev is exactly 0 against the destination boxes, the candidates accepted under earlier
//                         angles and the other candidates of its angle.
//     then the accepted flags and per-frame totals are copied to the host (the call's only synchronisation), which sizes
//     the output through the caller's allocator.
//   4 rp_copy_dst_kernel  the destination rows to their new frame starts; the new frame offsets.
//   5 rp_paste_kernel     one CTA per instance box: its rows (ranked by popcount from launch 1's words) rotated by each
//                         accepted angle, written after the destination rows of the frame in candidate order.
// Rotation: column j of R = [[c, s, 0], [-s, c, 0], [0, 0, 1]] (c, s: cos / sin of the angle in double), each coordinate
// float32((x*R[0][j] + y*R[1][j]) + z*R[2][j]) in double without FMA; every other column is copied bit for bit.
namespace {

constexpr int kRpThreads = 256;
constexpr int kRpTile = 1024;                  // source rows per membership tile = 4 per thread = 32 ballot words

struct RpFrames {
    int inst_off[kGtsMaxBatch + 1];            // instance boxes of frame b: [inst_off[b], inst_off[b+1])
    int cand_off[kGtsMaxBatch + 1];            // candidates of frame b, angle by angle, instance boxes in order
    int ang_off[kGtsMaxBatch + 1];             // angles of frame b: rows [ang_off[b], ang_off[b+1]) of the cos / sin table
};

struct RpBox { float cx, cy, cz, ca, sa, dx, dy, dz; };

// first membership tile of every source frame (a frame of N rows has ceil(N / 1024) tiles); tile_lo[batch] = all tiles
__device__ void rp_tile_starts(const int32_t *__restrict__ off, int batch, int *tile_lo) {
    int t = 0;
    for (int q = 0; q < batch; ++q) {
        tile_lo[q] = t;
        t += (__ldg(off + q + 1) - __ldg(off + q) + kRpTile - 1) / kRpTile;
    }
    tile_lo[batch] = t;
}

// the frame of instance box g (uniform across the CTA)
__device__ __forceinline__ int rp_box_frame(const RpFrames &f, int g) {
    int b = 0;
    while (f.inst_off[b + 1] <= g) ++b;
    return b;
}

__global__ void __launch_bounds__(kRpThreads) rp_member_kernel(const float *__restrict__ src, int stride, int x_col,
                                                               const int32_t *__restrict__ src_off, int batch,
                                                               const float4 *__restrict__ inst, const RpFrames f, int tiles,
                                                               uint32_t *__restrict__ words, int *__restrict__ tile_counts) {
    extern __shared__ RpBox box_s[];           // the frame's instance boxes, then per-warp counts [box][warp] as bytes
    __shared__ int tile_lo[kGtsMaxBatch + 1];
    __shared__ int frame_s;
    const int t = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        rp_tile_starts(src_off, batch, tile_lo);
        int b = 0;
        while (b < batch && tile_lo[b + 1] <= t) ++b;
        frame_s = b;
    }
    __syncthreads();
    const int b = frame_s;
    if (b >= batch) return;                    // the grid is sized for ceil(n / 1024) + batch tiles
    const int i0 = f.inst_off[b], m = f.inst_off[b + 1] - i0;
    if (m == 0) return;
    unsigned char *cnt_s = (unsigned char *)(box_s + m);
    for (int k = threadIdx.x; k < m; k += kRpThreads) {
        const float4 u = __ldg(inst + 4 * (i0 + k)), v = __ldg(inst + 4 * (i0 + k) + 1), w = __ldg(inst + 4 * (i0 + k) + 2);
        box_s[k] = RpBox{u.x, u.y, u.z, w.x, w.y, u.w, v.x, v.y};      // packed: cosf(-rz), sinf(-rz) at 8, 9
    }
    const int row0 = __ldg(src_off + b) + (t - tile_lo[b]) * kRpTile, row_end = __ldg(src_off + b + 1);
    float x[kRpTile / kRpThreads], y[kRpTile / kRpThreads], z[kRpTile / kRpThreads];
    bool valid[kRpTile / kRpThreads];
#pragma unroll
    for (int j = 0; j < kRpTile / kRpThreads; ++j) {
        const int i = row0 + j * kRpThreads + threadIdx.x;   // a warp covers 32 consecutive rows = one word
        valid[j] = i < row_end;
        const float *row = src + (size_t)(valid[j] ? i : row0) * stride + x_col;
        x[j] = __ldg(row);
        y[j] = __ldg(row + 1);
        z[j] = __ldg(row + 2);
    }
    __syncthreads();
    for (int k = 0; k < m; ++k) {
        const RpBox q = box_s[k];
        int cnt = 0;
#pragma unroll
        for (int j = 0; j < kRpTile / kRpThreads; ++j) {
            const bool in = valid[j] && pt_in_box3d(x[j], y[j], z[j], q.cx, q.cy, q.cz, q.ca, q.sa, q.dx, q.dy, q.dz);
            const uint32_t w = __ballot_sync(0xffffffffu, in);
            if (lane == 0) {
                words[((size_t)k * tiles + t) * (kRpTile / 32) + j * (kRpThreads / 32) + warp] = w;
                cnt += __popc(w);
            }
        }
        if (lane == 0) cnt_s[k * (kRpThreads / 32) + warp] = (unsigned char)cnt;     // <= 128
    }
    __syncthreads();
    for (int k = threadIdx.x; k < m; k += kRpThreads) {
        int s = 0;
#pragma unroll
        for (int w = 0; w < kRpThreads / 32; ++w) s += cnt_s[k * (kRpThreads / 32) + w];
        tile_counts[(size_t)k * tiles + t] = s;
    }
}

__global__ void __launch_bounds__(128) rp_box_rows_kernel(const int32_t *__restrict__ src_off, int batch, const RpFrames f,
                                                          int tiles, const int *__restrict__ tile_counts,
                                                          long long *__restrict__ cand_rows) {
    __shared__ int tile_lo[kGtsMaxBatch + 1];
    __shared__ int part[4];
    const int g = blockIdx.x, b = rp_box_frame(f, g);
    const int j = g - f.inst_off[b], m = f.inst_off[b + 1] - f.inst_off[b];
    if (threadIdx.x == 0) rp_tile_starts(src_off, batch, tile_lo);
    __syncthreads();
    int s = 0;
    for (int t = tile_lo[b] + threadIdx.x; t < tile_lo[b + 1]; t += 128) s += tile_counts[(size_t)j * tiles + t];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
    __syncthreads();
    if ((int)threadIdx.x < f.ang_off[b + 1] - f.ang_off[b]) {
        const int c = f.cand_off[b] + threadIdx.x * m + j;
        cand_rows[2 * c] = 0;                  // (first row, row count) as gts_accept_kernel reads its samples' rows
        cand_rows[2 * c + 1] = part[0] + part[1] + part[2] + part[3];
    }
}

__global__ void __launch_bounds__(kRpThreads) rp_copy_dst_kernel(const float *__restrict__ dst, int n, int stride,
                                                                 const int32_t *__restrict__ dst_off, int batch,
                                                                 const int *__restrict__ frame_stats, float *__restrict__ out,
                                                                 int32_t *__restrict__ out_off) {
    __shared__ long long off_e[kGtsMaxBatch + 1];   // frame starts in elements
    __shared__ long long shift_e[kGtsMaxBatch];     // pasted rows of the frames before b, in elements
    if (threadIdx.x == 0) {
        long long p = 0;
        for (int q = 0; q <= batch; ++q) {
            const int o = __ldg(dst_off + q);
            off_e[q] = (long long)o * stride;
            if (q < batch) shift_e[q] = p * stride;
            if (blockIdx.x == 0) out_off[q] = o + (int)p;
            if (q < batch) p += frame_stats[batch + q];
        }
    }
    __syncthreads();
    const long long e0 = (long long)blockIdx.x * kRpTile * stride;
    const long long e1 = min((long long)n * stride, e0 + (long long)kRpTile * stride);
    int b = 0;                                 // frame of element e: the last b with off_e[b] <= e (empty frames skipped)
    for (long long e = e0 + threadIdx.x; e < e1; e += kRpThreads) {
        while (b + 1 < batch && off_e[b + 1] <= e) ++b;
        out[e + shift_e[b]] = __ldg(dst + e);
    }
}

// coordinate k of (x, y, z) times the rotation matrix of (c, s); the 0 and 1 entries are passed in so that no product
// with them is folded
__device__ __forceinline__ float rp_rotate(int k, float x, float y, float z, double c, double s, double zero, double one) {
    double r0, r1, r2;
    if (k == 0) { r0 = c; r1 = -s; r2 = zero; }
    else if (k == 1) { r0 = s; r1 = c; r2 = zero; }
    else { r0 = zero; r1 = zero; r2 = one; }
    return __double2float_rn(__dadd_rn(__dadd_rn(__dmul_rn((double)x, r0), __dmul_rn((double)y, r1)), __dmul_rn((double)z, r2)));
}

__global__ void __launch_bounds__(kRpThreads) rp_paste_kernel(const float *__restrict__ src, int stride, int x_col,
                                                              const int32_t *__restrict__ src_off,
                                                              const int32_t *__restrict__ dst_off, int batch, const RpFrames f,
                                                              int tiles, const uint32_t *__restrict__ words,
                                                              const int *__restrict__ tile_counts,
                                                              const double2 *__restrict__ cos_sin,
                                                              const int *__restrict__ obj_dst, const int32_t *__restrict__ out_off,
                                                              double zero, double one, float *__restrict__ out) {
    __shared__ int tile_lo[kGtsMaxBatch + 1];
    __shared__ int dst_row_s[kGtsMaxGroups];   // first output row of each accepted copy of this box
    __shared__ double2 cs_s[kGtsMaxGroups];    // and its angle's cos / sin
    __shared__ int n_copies_s, n_list_s;
    __shared__ int list_t[32], list_p[32];     // tiles with rows in the box (frame-local index) and the box's rows before each
    __shared__ uint32_t word_s[kRpTile / 32];
    __shared__ int word_prefix[kRpTile / 32 + 1];
    __shared__ int rows_s[kRpTile];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = blockIdx.x, b = rp_box_frame(f, g);
    const int j = g - f.inst_off[b], m = f.inst_off[b + 1] - f.inst_off[b];
    if (threadIdx.x == 0) {
        rp_tile_starts(src_off, batch, tile_lo);
        const int base = out_off[b] + __ldg(dst_off + b + 1) - __ldg(dst_off + b);
        int nc = 0;
        for (int a = 0; a < f.ang_off[b + 1] - f.ang_off[b]; ++a) {
            const int d = obj_dst[f.cand_off[b] + a * m + j];          // -1 when the candidate was rejected
            if (d >= 0) {
                dst_row_s[nc] = base + d;
                cs_s[nc] = cos_sin[f.ang_off[b] + a];
                ++nc;
            }
        }
        n_copies_s = nc;
    }
    __syncthreads();
    const int nc = n_copies_s;
    if (nc == 0) return;
    const int t_lo = tile_lo[b], n_t = tile_lo[b + 1] - t_lo, row_base = __ldg(src_off + b);
    const uint32_t *wbox = words + ((size_t)j * tiles + t_lo) * (kRpTile / 32);
    const int *cbox = tile_counts + (size_t)j * tiles + t_lo;
    int done = 0;                              // rows of the box in the tiles before t0 (warp 0)
    for (int t0 = 0; t0 < n_t; t0 += 32) {
        if (warp == 0) {
            const int c = t0 + lane < n_t ? cbox[t0 + lane] : 0;
            int incl = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += v;
            }
            const uint32_t nz = __ballot_sync(0xffffffffu, c > 0);
            if (c > 0) {
                const int slot = __popc(nz & ((1u << lane) - 1u));
                list_t[slot] = t0 + lane;
                list_p[slot] = done + incl - c;
            }
            if (lane == 0) n_list_s = __popc(nz);
            done += __shfl_sync(0xffffffffu, incl, 31);
        }
        __syncthreads();
        for (int q = 0; q < n_list_s; ++q) {
            const int tl = list_t[q], p = list_p[q];
            if (warp == 0) {
                const uint32_t w = wbox[(size_t)tl * (kRpTile / 32) + lane];
                word_s[lane] = w;
                const int c = __popc(w);
                int incl = c;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int v = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= o) incl += v;
                }
                word_prefix[lane] = incl - c;
                if (lane == 31) word_prefix[kRpTile / 32] = incl;
            }
            __syncthreads();
#pragma unroll
            for (int jj = 0; jj < kRpTile / kRpThreads; ++jj) {
                const int wi = jj * (kRpThreads / 32) + warp;
                const uint32_t w = word_s[wi];
                if ((w >> lane) & 1u) rows_s[word_prefix[wi] + __popc(w & ((1u << lane) - 1u))] = row_base + tl * kRpTile + jj * kRpThreads + threadIdx.x;
            }
            __syncthreads();
            const int total = word_prefix[kRpTile / 32] * stride;
            for (int a = 0; a < nc; ++a) {
                const double2 cs = cs_s[a];
                float *o = out + (size_t)(dst_row_s[a] + p) * stride;
                for (int e = threadIdx.x; e < total; e += kRpThreads) {
                    const int r = e / stride, c = e - r * stride, k = c - x_col;
                    const float *row = src + (size_t)rows_s[r] * stride;
                    float v;
                    if (k < 0) v = (float)b;   // the batch column of collate_batch
                    else if (k < 3) v = rp_rotate(k, __ldg(row + x_col), __ldg(row + x_col + 1), __ldg(row + x_col + 2), cs.x, cs.y, zero, one);
                    else v = __ldg(row + c);
                    o[e] = v;
                }
            }
            __syncthreads();
        }
        __syncthreads();
    }
}

}  // namespace

extern "C" size_t toda_rotate_paste_workspace_bytes(int n_src, int batch, int max_inst, int n_cand) {
    if (n_src < 0 || batch < 0 || max_inst < 0 || n_cand < 0) return 0;
    const size_t slots = (size_t)max_inst * ((size_t)ceil_div(n_src, kRpTile) + batch);   // (box, tile) pairs
    return align_up(slots * (kRpTile / 32) * sizeof(uint32_t), 256) + align_up(slots * sizeof(int), 256) +
           align_up((size_t)n_cand * 2 * sizeof(long long), 256) + align_up((size_t)n_cand * 2 * sizeof(float4), 256) +
           align_up((size_t)n_cand * sizeof(int), 256) + align_up(((size_t)n_cand + 3 * (size_t)batch) * sizeof(int), 256);
}

extern "C" int toda_rotate_paste(const float *src, int n_src, const int32_t *src_offsets, const float *dst, int n_dst,
                                 const int32_t *dst_offsets, int stride, int x_col, int batch, const float *dst_boxes,
                                 const int *dst_box_offsets_host, const float *inst_boxes, const int *inst_offsets_host,
                                 const float *cand_boxes, const double *cos_sin, const int *angle_counts_host,
                                 int32_t *result_host, toda_alloc_fn alloc_out, void *alloc_ctx, int32_t *out_offsets,
                                 void *workspace, size_t workspace_bytes, void *stream) {
    TODA_CHECK_ARG(n_src >= 0 && n_dst >= 0 && (x_col == 0 || x_col == 1) && stride >= x_col + 3 && stride <= 63,
                   "rotate_paste: bad layout n_src=%d n_dst=%d stride=%d x_col=%d", n_src, n_dst, stride, x_col);
    TODA_CHECK_ARG(dst_box_offsets_host && inst_offsets_host && angle_counts_host && inst_offsets_host[0] == 0,
                   "rotate_paste: null box table offsets, or instance box offsets that do not start at 0");
    if (batch < 1 || batch > kGtsMaxBatch) {
        toda_set_error("rotate_paste: batch %d outside [1, %d]", batch, kGtsMaxBatch);
        return batch < 1 ? TODA_ERR_INVALID : TODA_ERR_UNSUPPORTED;
    }
    GtsFrames gf = {};
    RpFrames rf = {};
    int max_inst = 0, max_cand = 0;
    for (int b = 0; b < batch; ++b) {
        const int ne = dst_box_offsets_host[b + 1] - dst_box_offsets_host[b], m = inst_offsets_host[b + 1] - inst_offsets_host[b];
        const int na = angle_counts_host[b];
        TODA_CHECK_ARG(dst_box_offsets_host[b] >= 0 && ne >= 0 && inst_offsets_host[b] >= 0 && m >= 0 && na >= 0,
                       "rotate_paste: box offsets or angle counts of frame %d are not ascending", b);
        if (na > kGtsMaxGroups) {
            toda_set_error("rotate_paste: frame %d has %d angles (at most %d)", b, na, kGtsMaxGroups);
            return TODA_ERR_UNSUPPORTED;
        }
        if (m > kGtsMaxSamples || na * m > kGtsMaxSamples) {
            toda_set_error("rotate_paste: frame %d has %d instance boxes and %d candidates (at most %d each)", b, m, na * m,
                           kGtsMaxSamples);
            return TODA_ERR_UNSUPPORTED;
        }
        gf.exist_off[b] = dst_box_offsets_host[b];
        gf.samp_off[b + 1] = gf.samp_off[b] + na * m;
        for (int a = 0; a < na; ++a) gf.group_size[b][a] = (unsigned short)m;
        gf.n_groups = na > gf.n_groups ? na : gf.n_groups;
        rf.inst_off[b + 1] = rf.inst_off[b] + m;
        rf.ang_off[b + 1] = rf.ang_off[b] + na;
        max_inst = m > max_inst ? m : max_inst;
        max_cand = na * m > max_cand ? na * m : max_cand;
    }
    gf.exist_off[batch] = dst_box_offsets_host[batch];
    for (int b = 0; b <= batch; ++b) rf.cand_off[b] = gf.samp_off[b];
    const int n_inst = rf.inst_off[batch], n_cand = gf.samp_off[batch];
    TODA_CHECK_ARG(src_offsets && dst_offsets && out_offsets && result_host && alloc_out && workspace &&
                   (n_src == 0 || src) && (n_dst == 0 || dst) && (gf.exist_off[batch] == 0 || dst_boxes) &&
                   (n_inst == 0 || inst_boxes) && (n_cand == 0 || (cand_boxes && cos_sin)), "rotate_paste: null pointer");
    const size_t need = toda_rotate_paste_workspace_bytes(n_src, batch, max_inst, n_cand);
    if (workspace_bytes < need) {
        toda_set_error("rotate_paste: workspace %zu < required %zu bytes", workspace_bytes, need);
        return TODA_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int tiles = ceil_div(n_src, kRpTile) + batch;
    const size_t slots = (size_t)max_inst * tiles;
    char *ws = (char *)workspace;
    uint32_t *words = (uint32_t *)ws;
    ws += align_up(slots * (kRpTile / 32) * sizeof(uint32_t), 256);
    int *tile_counts = (int *)ws;
    ws += align_up(slots * sizeof(int), 256);
    long long *cand_rows = (long long *)ws;
    ws += align_up((size_t)n_cand * 2 * sizeof(long long), 256);
    float4 *rm_boxes = (float4 *)ws;           // written by gts_accept_kernel, not used here
    ws += align_up((size_t)n_cand * 2 * sizeof(float4), 256);
    int *obj_dst = (int *)ws;
    ws += align_up((size_t)n_cand * sizeof(int), 256);
    int32_t *accepted = (int32_t *)ws;         // accepted flags, then frame_stats [3][batch]: accepted, pasted rows, first
    int *frame_stats = accepted + n_cand;

    if (n_inst > 0) {
        rp_member_kernel<<<tiles, kRpThreads, (size_t)max_inst * (sizeof(RpBox) + kRpThreads / 32), st>>>(
            src, stride, x_col, src_offsets, batch, (const float4 *)inst_boxes, rf, tiles, words, tile_counts);
        TODA_LAUNCH_OK();
        rp_box_rows_kernel<<<n_inst, 128, 0, st>>>(src_offsets, batch, rf, tiles, tile_counts, cand_rows);
        TODA_LAUNCH_OK();
    }
    gts_accept_kernel<<<batch, kGtsThreads, (size_t)max_cand * sizeof(BevBox), st>>>(
        (const float4 *)dst_boxes, (const float4 *)cand_boxes, cand_rows, gf, accepted, rm_boxes, frame_stats, obj_dst);
    TODA_LAUNCH_OK();
    TODA_CUDA_OK(cudaMemcpyAsync(result_host, accepted, ((size_t)n_cand + 2 * batch) * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    TODA_CUDA_OK(cudaStreamSynchronize(st));
    long long rows = n_dst, pasted = 0;
    for (int b = 0; b < batch; ++b) pasted += result_host[n_cand + batch + b];
    rows += pasted;
    if (rows > 0x7fffffffLL) {
        toda_set_error("rotate_paste: %lld output rows (at most 2^31 - 1)", rows);
        return TODA_ERR_UNSUPPORTED;
    }
    float *out = (float *)alloc_out((size_t)rows, alloc_ctx);
    if (!out && rows > 0) {
        toda_set_error("rotate_paste: the allocator returned no memory for %lld rows", rows);
        return TODA_ERR_INVALID;
    }
    rp_copy_dst_kernel<<<ceil_div(n_dst > 0 ? n_dst : 1, kRpTile), kRpThreads, 0, st>>>(dst, n_dst, stride, dst_offsets, batch,
                                                                                       frame_stats, out, out_offsets);
    TODA_LAUNCH_OK();
    if (pasted > 0) {
        rp_paste_kernel<<<n_inst, kRpThreads, 0, st>>>(src, stride, x_col, src_offsets, dst_offsets, batch, rf, tiles, words,
                                                       tile_counts, (const double2 *)cos_sin, obj_dst, out_offsets, 0.0, 1.0,
                                                       out);
        TODA_LAUNCH_OK();
    }
    return TODA_OK;
}
