// K1 hard voxelizer + K2 MeanVFE, and the uncapped dynamic voxelizer + mean of DynamicMeanVFE (see include/toda_b200.h).
//
// The reference is a sequential loop (SURVEY.md Appendix C.1).  Its parallel-equivalent definition:
//   first[v]  = min{ i : cell(i) = v }                      (per frame)
//   voxel id  = rank of first[v] among the frame's voxels   (first-appearance order)
//   kept      = voxel id < max_voxels                       (points of refused voxels vanish)
//   members   = the max_points smallest point indices of v, ascending
// Pipeline (all frames of the batch in each launch; no host synchronisation):
//   cells   : float4-staged point loads -> cell id per point, mark the occupancy index
//   build   : rank the marked cells (index.cu)               -> dense voxel ids "cid" in (b,z,y,x) order
//   first   : cid per point, atomicMin first[cid]
//   flags   : bit i of pflags set iff point i is the first of its voxel; popcount scan -> appearance rank
//   assign  : cid -> output row (first-appearance or canonical order), applies the max_voxels cap
//   insert  : lock-free sorted insertion of each point index into slots[row][0..K)   (atomicMin chain)
//   write   : slots -> voxels (zero padded), coords, num_points
#include "common.cuh"
#include "scan.cuh"

namespace {

constexpr int kBlock = 256;
constexpr int kEmpty = 0x7fffffff;
constexpr uint32_t kNoCell = 0xffffffffu;

struct VoxGeom {
    float lo[3];     // x,y,z
    float vs[3];     // x,y,z
    int grid[3];     // x,y,z
};

struct VoxWork {
    GridIndex gi;
    uint32_t *pt_cell;   // [n]   cell id, later reused as cid
    uint32_t *cid_cell;  // [vcap] cell id of each cid
    int *first;          // [vcap]
    unsigned *pflags;    // [ceil(n/32)]  (zeroed per call)
    int *pprefix;        // [ceil(n/32)+1]
    unsigned *kflags;    // [ceil(vcap/32)] keep flags per cid
    int *kprefix;        // [ceil(vcap/32)+1]
    int *row_of_cid;     // [vcap]
    int *slots;          // [batch*max_voxels*K]
    int *scan_tmp;       // scratch for scans
    int *counts;         // [0]=Vall, [1..B]=per-frame Vall, then fstart[B+1], voff[B+1]
    size_t bytes;
};

size_t layout(VoxWork *w, void *base, int64_t n, int batch, const int *grid, int K, int max_voxels) {
    size_t off = 0;
    char *p = (char *)base;
    GridIndex *gp = w ? &w->gi : nullptr;
    size_t ib = index_layout(gp, base, batch, grid[2], grid[1], grid[0]);
    off = align_up(ib, 256);
    int64_t vcap = n;  // one voxel per point at most
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    size_t o_ptcell = take((size_t)n * 4);
    size_t o_cidcell = take((size_t)vcap * 4);
    size_t o_first = take((size_t)vcap * 4);
    size_t o_pflags = take((size_t)(n / 32 + 1) * 4);
    size_t o_pprefix = take((size_t)(n / 32 + 2) * 4);
    size_t o_kflags = take((size_t)(vcap / 32 + 1) * 4);
    size_t o_kprefix = take((size_t)(vcap / 32 + 2) * 4);
    size_t o_row = take((size_t)vcap * 4);
    size_t o_slots = take((size_t)batch * max_voxels * K * 4);
    size_t o_tmp = take((size_t)(n / 32 / 1024 + 4) * 4);
    size_t o_counts = take((size_t)(3 * batch + 8) * 4);
    if (w) {
        w->pt_cell = (uint32_t *)(p + o_ptcell);
        w->cid_cell = (uint32_t *)(p + o_cidcell);
        w->first = (int *)(p + o_first);
        w->pflags = (unsigned *)(p + o_pflags);
        w->pprefix = (int *)(p + o_pprefix);
        w->kflags = (unsigned *)(p + o_kflags);
        w->kprefix = (int *)(p + o_kprefix);
        w->row_of_cid = (int *)(p + o_row);
        w->slots = (int *)(p + o_slots);
        w->scan_tmp = (int *)(p + o_tmp);
        w->counts = (int *)(p + o_counts);
        w->bytes = off;
    }
    return off;
}

// --- pass 1: cell id per point ------------------------------------------------------------------
// A CTA owns kBlock consecutive points = kBlock*stride contiguous floats; they are staged into shared
// memory with coalesced 16-byte loads (rows of 5 or 6 floats are not 16-byte aligned individually, but
// the CTA's chunk is), then every thread reads its own x,y,z from shared memory.
__global__ void __launch_bounds__(kBlock) vox_cells_kernel(const float *__restrict__ points, long long n, int stride,
                                                           int xyz_col, const int *__restrict__ frame_off, int batch,
                                                           VoxGeom geo, GridIndex gi, uint32_t *__restrict__ pt_cell) {
    extern __shared__ float4 stage4[];
    float *stage = (float *)stage4;
    long long chunks = (n + kBlock - 1) / kBlock;
    for (long long chunk = blockIdx.x; chunk < chunks; chunk += gridDim.x) {
        long long p0 = chunk * kBlock;
        int cnt = (int)min((long long)kBlock, n - p0);
        const float *src = points + p0 * stride;
        int nfl = cnt * stride;
        if ((((uintptr_t)src) & 15) == 0) {
            int nv = nfl >> 2;
            const float4 *s4 = (const float4 *)src;
            for (int i = threadIdx.x; i < nv; i += kBlock) stage4[i] = __ldg(s4 + i);
            for (int i = (nv << 2) + threadIdx.x; i < nfl; i += kBlock) stage[i] = __ldg(src + i);
        } else {
            for (int i = threadIdx.x; i < nfl; i += kBlock) stage[i] = __ldg(src + i);
        }
        __syncthreads();
        if (threadIdx.x < cnt) {
            long long i = p0 + threadIdx.x;
            const float *pt = stage + threadIdx.x * stride + xyz_col;
            int c[3];
            bool ok = true;
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                // exact fp32 subtract then IEEE divide, as the CPU loop does (no reciprocal, no FMA)
                float q = __fdiv_rn(__fsub_rn(pt[j], geo.lo[j]), geo.vs[j]);
                float fl = floorf(q);
                ok = ok && (fl >= 0.0f) && (fl < (float)geo.grid[j]);
                c[j] = (int)fl;
            }
            uint32_t cell = kNoCell;
            if (ok) {
                int b = 0;
                while (b + 1 < batch && i >= __ldg(frame_off + b + 1)) ++b;
                long long cl = index_cell(gi, b, c[2], c[1], c[0]);
                index_mark(gi, cl);
                cell = (uint32_t)cl;
            }
            pt_cell[i] = cell;
        }
        __syncthreads();
    }
}

__global__ void vox_init_first_kernel(int *__restrict__ first, const int *__restrict__ counts) {
    int vall = counts[0];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < vall; i += gridDim.x * blockDim.x) first[i] = kEmpty;
}

// --- pass 2: cid per point, first point of every voxel ------------------------------------------
__global__ void vox_first_kernel(GridIndex gi, uint32_t *__restrict__ pt_cell, long long n, int *__restrict__ first) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        uint32_t cell = pt_cell[i];
        if (cell == kNoCell) continue;
        int cid = index_lookup(gi, (long long)cell);
        pt_cell[i] = (uint32_t)cid;
        // warp-aggregate: among lanes that hit the same voxel only the smallest point index goes out
        unsigned peers = __match_any_sync(__activemask(), cid);
        int leader = __ffs(peers) - 1;  // lanes are in point order, so the lowest lane has the smallest index
        if ((int)(threadIdx.x & 31) == leader) atomicMin(first + cid, (int)i);
    }
}

__global__ void vox_flag_first_kernel(const int *__restrict__ first, const int *__restrict__ counts,
                                      unsigned *__restrict__ pflags) {
    int vall = counts[0];
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < vall; c += gridDim.x * blockDim.x) {
        int f = first[c];
        atomicOr(pflags + (f >> 5), 1u << (f & 31));
    }
}

// per-frame bookkeeping (one tiny CTA): fstart[b] = first cid of frame b, voff[b] = first output row
__global__ void vox_frames_kernel(int *counts, int batch, int max_voxels, int32_t *voxel_counts) {
    if (threadIdx.x == 0) {
        int *fstart = counts + 1 + batch;       // [batch+1]
        int *voff = counts + 2 + 2 * batch;     // [batch+1]
        int fs = 0, vo = 0;
        for (int b = 0; b < batch; ++b) {
            fstart[b] = fs;
            voff[b] = vo;
            int vb = counts[1 + b];
            fs += vb;
            int kept = vb < max_voxels ? vb : max_voxels;
            voxel_counts[b] = kept;
            vo += kept;
        }
        fstart[batch] = fs;
        voff[batch] = vo;
        voxel_counts[batch] = vo;
    }
}

__device__ __forceinline__ int frame_of_cid(const int *fstart, int batch, int cid) {
    int b = 0;
    while (b + 1 < batch && cid >= fstart[b + 1]) ++b;
    return b;
}

// appearance rank of a voxel within its frame
__device__ __forceinline__ int appearance_rank(const unsigned *pflags, const int *pprefix, int f, int frame_start_cid) {
    int g = pprefix[f >> 5] + __popc(pflags[f >> 5] & ((1u << (f & 31)) - 1u));
    return g - frame_start_cid;  // each earlier-frame voxel has exactly one first-point flag before this frame
}

// order = first appearance: row = voff[b] + rank, dropped when rank >= max_voxels.
// order = canonical: keep flag only; rows follow from the keep-flag scan (vox_rows_canonical_kernel).
__global__ void vox_assign_kernel(const int *__restrict__ first, const int *__restrict__ counts, int batch,
                                  int max_voxels, const unsigned *__restrict__ pflags, const int *__restrict__ pprefix,
                                  int order, int *__restrict__ row_of_cid, unsigned *__restrict__ kflags) {
    int vall = counts[0];
    const int *fstart = counts + 1 + batch;
    const int *voff = counts + 2 + 2 * batch;
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < vall; c += gridDim.x * blockDim.x) {
        int b = frame_of_cid(fstart, batch, c);
        int r = appearance_rank(pflags, pprefix, first[c], fstart[b]);
        bool keep = r < max_voxels;
        if (order == TODA_ORDER_FIRST_APPEARANCE) {
            row_of_cid[c] = keep ? voff[b] + r : -1;
        } else {
            row_of_cid[c] = keep ? 0 : -1;
            if (keep) atomicOr(kflags + (c >> 5), 1u << (c & 31));
        }
    }
}

__global__ void vox_rows_canonical_kernel(const int *__restrict__ counts, const unsigned *__restrict__ kflags,
                                          const int *__restrict__ kprefix, int *__restrict__ row_of_cid) {
    int vall = counts[0];
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < vall; c += gridDim.x * blockDim.x) {
        if (row_of_cid[c] < 0) continue;
        // kept voxels of earlier frames all precede (cid order is frame-major), so the global keep rank is the row
        row_of_cid[c] = kprefix[c >> 5] + __popc(kflags[c >> 5] & ((1u << (c & 31)) - 1u));
    }
}

__global__ void vox_init_slots_kernel(int *__restrict__ slots, const int32_t *__restrict__ voxel_counts, int batch, int K) {
    long long tot = (long long)voxel_counts[batch] * K;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < tot; i += (long long)gridDim.x * blockDim.x)
        slots[i] = kEmpty;
}

// --- pass 3: lock-free sorted insertion -----------------------------------------------------------
// slots[row][0..K) ends up holding the K smallest point indices of the voxel in ascending order:
// slot r sees (via atomicMin) every index that is not among the r smallest, so its final value is
// the (r+1)-th smallest whatever the interleaving.
__global__ void vox_insert_kernel(const uint32_t *__restrict__ pt_cid, long long n, const int *__restrict__ row_of_cid,
                                  int *__restrict__ slots, int K) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        uint32_t cid = pt_cid[i];
        if (cid == kNoCell) continue;
        int row = __ldg(row_of_cid + cid);
        if (row < 0) continue;
        int *s = slots + (long long)row * K;
        int carry = (int)i;
        for (int r = 0; r < K; ++r) {
            int old = atomicMin(s + r, carry);
            if (old == kEmpty) break;         // took a free slot (or displaced nothing)
            if (old > carry) carry = old;     // displaced a larger index: push it down the chain
        }
    }
}

// --- pass 4: write the padded voxel tensor, coords, counts ---------------------------------------
__global__ void vox_write_kernel(const float *__restrict__ points, int stride, int feat_col, int F,
                                 const int *__restrict__ slots, int K, const int32_t *__restrict__ voxel_counts, int batch,
                                 float *__restrict__ voxels) {
    long long tot = (long long)voxel_counts[batch] * K;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < tot; e += (long long)gridDim.x * blockDim.x) {
        int idx = slots[e];
        float *dst = voxels + e * F;
        if (idx != kEmpty) {
            const float *src = points + (long long)idx * stride + feat_col;
            for (int f = 0; f < F; ++f) dst[f] = __ldg(src + f);
        } else {
            for (int f = 0; f < F; ++f) dst[f] = 0.0f;
        }
    }
}

// (b,z,y,x) of an index cell id
__device__ __forceinline__ int4 cell_coords(const GridIndex &gi, long long cell) {
    long long hw = (long long)gi.H * gi.W;
    int b = (int)(cell / gi.frame_stride);
    long long r = cell - (long long)b * gi.frame_stride;
    int z = (int)(r / hw);
    int rem = (int)(r - (long long)z * hw);
    return make_int4(b, z, rem / gi.W, rem % gi.W);
}

__global__ void vox_meta_kernel(GridIndex gi, const uint32_t *__restrict__ cid_cell, const int *__restrict__ counts,
                                const int *__restrict__ row_of_cid, const int *__restrict__ slots, int K,
                                int4 *__restrict__ coords, int *__restrict__ num_points) {
    int vall = counts[0];
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < vall; c += gridDim.x * blockDim.x) {
        int row = row_of_cid[c];
        if (row < 0) continue;
        coords[row] = cell_coords(gi, cid_cell[c]);
        const int *s = slots + (long long)row * K;
        int cnt = 0;
        for (int k = 0; k < K; ++k) cnt += (s[k] != kEmpty);
        num_points[row] = cnt;
    }
}

// clear the index words this call touched (leaves the bitmap region all-zero for the next call)
__global__ void vox_release_kernel(GridIndex gi, const uint32_t *__restrict__ cid_cell, const int *__restrict__ counts) {
    int vall = counts[0];
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < vall; c += gridDim.x * blockDim.x) {
        long long w = (long long)cid_cell[c] >> 6;
        gi.bits0[w] = 0ull;
        gi.bits1[w >> 6] = 0ull;
    }
}

// --- MeanVFE ---------------------------------------------------------------------------------------
template <bool kNumIsFloat>
__global__ void mean_vfe_fwd_kernel(const float *__restrict__ voxels, const void *__restrict__ num, long long total,
                                    int K, int F, float *__restrict__ out) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        long long v = e / F;
        int f = (int)(e - v * F);
        const float *src = voxels + v * K * F + f;
        float s = 0.0f;
        for (int k = 0; k < K; ++k) s += __ldg(src + k * F);
        float nrm = kNumIsFloat ? ((const float *)num)[v] : (float)((const int *)num)[v];
        out[e] = s / fmaxf(nrm, 1.0f);
    }
}

template <bool kNumIsFloat>
__global__ void mean_vfe_bwd_kernel(const float *__restrict__ dout, const void *__restrict__ num, long long total, int K,
                                    int F, float *__restrict__ dvoxels) {
    // total = V*K*F ; every slot (padding included) receives d/nrm, as autograd of sum(dim=1)/nrm does
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        long long v = e / ((long long)K * F);
        int f = (int)(e % F);
        float nrm = kNumIsFloat ? ((const float *)num)[v] : (float)((const int *)num)[v];
        dvoxels[e] = __ldg(dout + v * F + f) / fmaxf(nrm, 1.0f);
    }
}

// --- dynamic voxelization + mean (pcdet DynamicMeanVFE) --------------------------------------------
// No caps: every kept point belongs to its voxel, every voxel is a row, and the rows are the cids (canonical order).
//   cells, build, frames, release : the K1 passes above; coords through cell_coords, as vox_meta_kernel writes them
//   count : cid per point, cnt[cid] += 1                       (warp-aggregated integer atomics)
//   scan  : seg[cid] = exclusive prefix of cnt
//   place : members[seg[cid] + slot] = point index, slot from an atomic cursor: seg[cid] ends as the segment's end
//   short : one thread per voxel: its coords; with <= kShortSeg members, the members in ascending order by selection,
//           ordered fp32 sum, divide; longer voxels are appended to a list
//   long  : one CTA per listed voxel: its members in ascending order through a shared-memory bitmap over its frame's
//           rows, then the ordered sum with the member rows staged in shared memory
// The fp32 sum adds the members in ascending point index from +0.0, so the result does not depend on scheduling.
constexpr int kShortSeg = 32;
constexpr int kShortF = 8;                        // short path: feature columns summed per pass
constexpr int kSegWinWords = 8192;                // long path: 32 KB bitmap window = 2^18 point indices
constexpr int kLongGrid = 2 * kNumSMs;

struct DynWork {
    GridIndex gi;
    uint32_t *pt_cell;   // [n] cell id, then cid; the long path reuses it for its ordered member lists
    uint32_t *cid_cell;  // [n] cell id of each cid
    int *cnt;            // [n] members per cid (zeroed per call)
    int *seg;            // [n+1] segment start per cid, the segment end once the place pass has run
    int *members;        // [n] point indices grouped by cid
    int *long_cids;      // [n/(kShortSeg+1)+1] voxels left to the long path
    int *scan_tmp;
    int *counts;         // as VoxWork::counts, then the length of long_cids
    size_t bytes;
};

size_t layout_dynamic(DynWork *w, void *base, int64_t n, int batch, const int *grid) {
    char *p = (char *)base;
    GridIndex *gp = w ? &w->gi : nullptr;
    size_t off = align_up(index_layout(gp, base, batch, grid[2], grid[1], grid[0]), 256);
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    size_t o_ptcell = take((size_t)n * 4);
    size_t o_cidcell = take((size_t)n * 4);
    size_t o_cnt = take((size_t)n * 4);
    size_t o_seg = take((size_t)(n + 1) * 4);
    size_t o_members = take((size_t)n * 4);
    size_t o_long = take((size_t)(n / (kShortSeg + 1) + 1) * 4);
    size_t o_tmp = take((size_t)(n / kScanTile + 2) * 4);
    size_t o_counts = take((size_t)(3 * batch + 9) * 4);
    if (w) {
        w->pt_cell = (uint32_t *)(p + o_ptcell);
        w->cid_cell = (uint32_t *)(p + o_cidcell);
        w->cnt = (int *)(p + o_cnt);
        w->seg = (int *)(p + o_seg);
        w->members = (int *)(p + o_members);
        w->long_cids = (int *)(p + o_long);
        w->scan_tmp = (int *)(p + o_tmp);
        w->counts = (int *)(p + o_counts);
        w->bytes = off;
    }
    return off;
}

__global__ void dyn_count_kernel(GridIndex gi, uint32_t *__restrict__ pt_cell, long long n, int *__restrict__ cnt) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        uint32_t cell = pt_cell[i];
        if (cell == kNoCell) continue;
        int cid = index_lookup(gi, (long long)cell);
        pt_cell[i] = (uint32_t)cid;
        unsigned peers = __match_any_sync(__activemask(), cid);
        if ((int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(cnt + cid, __popc(peers));
    }
}

__global__ void dyn_place_kernel(const uint32_t *__restrict__ pt_cid, long long n, int *__restrict__ seg,
                                 int *__restrict__ members) {
    int lane = threadIdx.x & 31;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        uint32_t cid = pt_cid[i];
        if (cid == kNoCell) continue;
        unsigned peers = __match_any_sync(__activemask(), cid);
        int leader = __ffs(peers) - 1;
        int base = 0;
        if (lane == leader) base = atomicAdd(seg + cid, __popc(peers));
        base = __shfl_sync(peers, base, leader);
        members[base + __popc(peers & ((1u << lane) - 1u))] = (int)i;
    }
}

__global__ void dyn_mean_short_kernel(const float *__restrict__ points, int stride, int feat_col, int F, GridIndex gi,
                                      const uint32_t *__restrict__ cid_cell, const int *__restrict__ counts,
                                      const int *__restrict__ cnt, const int *__restrict__ seg_end,
                                      const int *__restrict__ members, int *__restrict__ long_cids,
                                      int *__restrict__ n_long, float *__restrict__ features, int4 *__restrict__ coords) {
    int vall = counts[0];
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < vall; c += gridDim.x * blockDim.x) {
        coords[c] = cell_coords(gi, cid_cell[c]);
        int L = cnt[c];
        int e = seg_end[c], s = e - L;
        if (L > kShortSeg) {
            long_cids[atomicAdd(n_long, 1)] = c;
            continue;
        }
        // members in ascending order by repeated selection of the next larger index (read-only, O(L^2) L1 hits),
        // kShortF feature columns per pass in registers
        for (int f0 = 0; f0 < F; f0 += kShortF) {
            float acc[kShortF];
#pragma unroll
            for (int u = 0; u < kShortF; ++u) acc[u] = 0.0f;
            int prev = -1;
            for (int r = 0; r < L; ++r) {
                int m = 0x7fffffff;
                for (int j = s; j < e; ++j) {
                    int x = __ldg(members + j);
                    if (x > prev && x < m) m = x;
                }
                prev = m;
                const float *row = points + (long long)m * stride + feat_col + f0;
#pragma unroll
                for (int u = 0; u < kShortF; ++u)
                    if (f0 + u < F) acc[u] = __fadd_rn(acc[u], __ldg(row + u));
            }
#pragma unroll
            for (int u = 0; u < kShortF; ++u)
                if (f0 + u < F) features[(long long)c * F + f0 + u] = __fdiv_rn(acc[u], (float)L);
        }
    }
}

// exclusive prefix of v over the CTA (blockDim.x == kBlock); *total = the CTA's sum.  Ends with a barrier.
__device__ __forceinline__ int block_exclusive_sum(int v, int *warp_sums, int *total) {
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) warp_sums[warp] = incl;
    __syncthreads();
    int woff = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < kBlock / 32; ++w) {
        int ws = warp_sums[w];
        woff += w < warp ? ws : 0;
        tot += ws;
    }
    *total = tot;
    __syncthreads();
    return woff + incl - v;
}

__global__ void __launch_bounds__(kBlock) dyn_mean_long_kernel(const float *__restrict__ points, int stride, int feat_col,
                                                               int F, GridIndex gi, const uint32_t *__restrict__ cid_cell,
                                                               const int *__restrict__ frame_off, int batch, long long n,
                                                               const int *__restrict__ cnt,
                                                               const int *__restrict__ seg_end,
                                                               const int *__restrict__ members,
                                                               const int *__restrict__ long_cids,
                                                               const int *__restrict__ n_long, int *ordered,
                                                               float *__restrict__ features) {
    __shared__ unsigned win[kSegWinWords];     // member bitmap of one index window, then staged feature rows
    __shared__ int red[kBlock / 32];
    float *stage = (float *)win;
    int nl = *n_long;
    for (int k = blockIdx.x; k < nl; k += gridDim.x) {
        int c = long_cids[k];
        int L = cnt[c];
        int s = seg_end[c] - L;
        // the members lie in their frame's rows [lo, hi], as vox_cells_kernel assigns rows to frames
        int b = (int)((long long)cid_cell[c] / gi.frame_stride);
        int lo = b == 0 ? 0 : __ldg(frame_off + b);
        int hi = b == batch - 1 ? (int)(n - 1) : __ldg(frame_off + b + 1) - 1;
        // ascending member list: one window of 32*kSegWinWords indices at a time, bits extracted in word order
        int done = 0;
        for (long long w0 = lo; w0 <= hi; w0 += 32ll * kSegWinWords) {
            int nw = (int)min((long long)kSegWinWords, ((hi - w0) >> 5) + 1);
            for (int j = threadIdx.x; j < nw; j += kBlock) win[j] = 0u;
            __syncthreads();
            for (int j = threadIdx.x; j < L; j += kBlock) {
                long long d = members[s + j] - w0;
                if (d >= 0 && d < 32ll * nw) atomicOr(win + (d >> 5), 1u << (d & 31));
            }
            __syncthreads();
            int per = (nw + kBlock - 1) / kBlock;
            int wa = min(nw, (int)threadIdx.x * per), wb = min(nw, wa + per);
            int mine = 0;
            for (int w = wa; w < wb; ++w) mine += __popc(win[w]);
            int tot;
            int pos = s + done + block_exclusive_sum(mine, red, &tot);
            for (int w = wa; w < wb; ++w) {
                for (unsigned bits = win[w]; bits; bits &= bits - 1u)
                    ordered[pos++] = (int)(w0 + 32ll * w + (__ffs(bits) - 1));
            }
            done += tot;
            __syncthreads();
        }
        // ordered sum: thread f < F adds column f of the staged rows, in member order
        int rows_per = kSegWinWords / F;
        float acc = 0.0f;
        for (int j0 = 0; j0 < L; j0 += rows_per) {
            int rows = min(rows_per, L - j0);
            for (int t = threadIdx.x; t < rows * F; t += kBlock) {
                int r = t / F;
                stage[t] = __ldg(points + (long long)ordered[s + j0 + r] * stride + feat_col + (t - r * F));
            }
            __syncthreads();
            if ((int)threadIdx.x < F)
                for (int r = 0; r < rows; ++r) acc = __fadd_rn(acc, stage[r * F + threadIdx.x]);
            __syncthreads();
        }
        if ((int)threadIdx.x < F) features[(long long)c * F + threadIdx.x] = __fdiv_rn(acc, (float)L);
    }
}

}  // namespace

extern "C" size_t toda_voxelize_workspace_bytes(int64_t n_points, int batch, const int *grid, int max_points,
                                                int max_voxels) {
    if (n_points < 0 || batch <= 0 || !grid || max_points <= 0 || max_voxels <= 0) return 0;
    return layout(nullptr, nullptr, n_points > 0 ? n_points : 1, batch, grid, max_points, max_voxels);
}

extern "C" int toda_voxelize_hard(const float *points, int64_t n, int stride, int xyz_col, int feat_col, int F,
                                  const int32_t *frame_offsets, int batch, const float *range, const float *vsize,
                                  const int *grid, int K, int max_voxels, int order, float *voxels, int32_t *coords,
                                  int32_t *num_points, int32_t *voxel_counts, void *workspace, size_t workspace_bytes,
                                  void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    TODA_CHECK_ARG(n >= 0 && n < (1ll << 31) - 64, "voxelize: n_points=%lld out of range", (long long)n);
    TODA_CHECK_ARG(batch > 0 && batch <= 1024 && frame_offsets, "voxelize: bad batch/frame_offsets");
    TODA_CHECK_ARG(range && vsize && grid && K > 0 && max_voxels > 0, "voxelize: bad geometry args");
    TODA_CHECK_ARG(stride >= 3 && xyz_col >= 0 && xyz_col + 3 <= stride && feat_col >= 0 && F > 0 &&
                       feat_col + F <= stride, "voxelize: column layout does not fit point_stride=%d", stride);
    TODA_CHECK_ARG(order == TODA_ORDER_FIRST_APPEARANCE || order == TODA_ORDER_CANONICAL, "voxelize: bad order %d", order);
    TODA_CHECK_ARG(voxels && coords && num_points && voxel_counts && workspace, "voxelize: null output/workspace");
    TODA_CHECK_ARG((long long)batch * max_voxels * K < (1ll << 31), "voxelize: batch*max_voxels*max_points too large");
    for (int a = 0; a < 3; ++a) TODA_CHECK_ARG(grid[a] > 0 && vsize[a] > 0.f, "voxelize: bad grid/vsize on axis %d", a);
    long long cells = index_frame_stride(grid[2], grid[1], grid[0]) * batch;
    TODA_CHECK_ARG(cells < (1ll << 32) - 1, "voxelize: %lld cells exceed the 32-bit cell id range", cells);
    int64_t n_eff = n > 0 ? n : 1;
    VoxWork w;
    size_t need = layout(&w, workspace, n_eff, batch, grid, K, max_voxels);
    if (workspace_bytes < need) {
        toda_set_error("voxelize: workspace %zu < required %zu bytes", workspace_bytes, need);
        return TODA_ERR_WORKSPACE;
    }
    VoxGeom geo;
    for (int a = 0; a < 3; ++a) { geo.lo[a] = range[a]; geo.vs[a] = vsize[a]; geo.grid[a] = grid[a]; }

    // the two bitmaps must be zero on entry.  They are left zero on exit (vox_release_kernel), but the
    // caller-owned workspace may be fresh, so clear them here; it is 2 bits per 64 cells ~ a few MB/frame.
    size_t zero_bytes = (size_t)((char *)w.gi.rank0 - (char *)w.gi.bits0);
    TODA_CUDA_OK(cudaMemsetAsync(w.gi.bits0, 0, zero_bytes, st));
    TODA_CUDA_OK(cudaMemsetAsync(w.pflags, 0, (size_t)(n_eff / 32 + 1) * 4, st));
    if (order == TODA_ORDER_CANONICAL) TODA_CUDA_OK(cudaMemsetAsync(w.kflags, 0, (size_t)(n_eff / 32 + 1) * 4, st));

    if (n > 0) {
        size_t smem = (size_t)kBlock * stride * sizeof(float) + 16;
        TODA_CHECK_ARG(smem <= 48 * 1024, "voxelize: point_stride %d too large", stride);
        vox_cells_kernel<<<wave_grid(n, kBlock), kBlock, smem, st>>>(points, n, stride, xyz_col, frame_offsets, batch, geo,
                                                                    w.gi, w.pt_cell);
        TODA_LAUNCH_OK();
    }
    // ranks + cid -> cell table + per-frame voxel totals (counts[0]=Vall, counts[1..B])
    if (int rc = index_build_ranks(w.gi, nullptr, (int)n_eff, w.cid_cell, w.counts, st)) return rc;
    vox_frames_kernel<<<1, 32, 0, st>>>(w.counts, batch, max_voxels, voxel_counts);
    TODA_LAUNCH_OK();
    if (n > 0) {
        int g_v = wave_grid(n, kBlock);
        vox_init_first_kernel<<<g_v, kBlock, 0, st>>>(w.first, w.counts);
        TODA_LAUNCH_OK();
        vox_first_kernel<<<g_v, kBlock, 0, st>>>(w.gi, w.pt_cell, n, w.first);
        TODA_LAUNCH_OK();
        vox_flag_first_kernel<<<g_v, kBlock, 0, st>>>(w.first, w.counts, w.pflags);
        TODA_LAUNCH_OK();
        int nwords = (int)(n / 32 + 1);
        if (int rc = scan_exclusive(LoadPopc32{w.pflags}, nwords, w.pprefix, w.scan_tmp, nullptr, st)) return rc;
        vox_assign_kernel<<<g_v, kBlock, 0, st>>>(w.first, w.counts, batch, max_voxels, w.pflags, w.pprefix, order,
                                                  w.row_of_cid, w.kflags);
        TODA_LAUNCH_OK();
        if (order == TODA_ORDER_CANONICAL) {
            if (int rc = scan_exclusive(LoadPopc32{w.kflags}, nwords, w.kprefix, w.scan_tmp, nullptr, st)) return rc;
            vox_rows_canonical_kernel<<<g_v, kBlock, 0, st>>>(w.counts, w.kflags, w.kprefix, w.row_of_cid);
            TODA_LAUNCH_OK();
        }
        int g_s = wave_grid((int64_t)batch * max_voxels * K, kBlock);
        vox_init_slots_kernel<<<g_s, kBlock, 0, st>>>(w.slots, voxel_counts, batch, K);
        TODA_LAUNCH_OK();
        vox_insert_kernel<<<g_v, kBlock, 0, st>>>(w.pt_cell, n, w.row_of_cid, w.slots, K);
        TODA_LAUNCH_OK();
        vox_write_kernel<<<g_s, kBlock, 0, st>>>(points, stride, feat_col, F, w.slots, K, voxel_counts, batch, voxels);
        TODA_LAUNCH_OK();
        vox_meta_kernel<<<g_v, kBlock, 0, st>>>(w.gi, w.cid_cell, w.counts, w.row_of_cid, w.slots, K, (int4 *)coords,
                                                num_points);
        TODA_LAUNCH_OK();
        vox_release_kernel<<<g_v, kBlock, 0, st>>>(w.gi, w.cid_cell, w.counts);
        TODA_LAUNCH_OK();
    }
    return TODA_OK;
}

extern "C" size_t toda_voxelize_dynamic_workspace_bytes(int64_t n_points, int batch, const int *grid) {
    if (n_points < 0 || batch <= 0 || !grid) return 0;
    return layout_dynamic(nullptr, nullptr, n_points > 0 ? n_points : 1, batch, grid);
}

extern "C" int toda_voxelize_dynamic(const float *points, int64_t n, int stride, int xyz_col, int feat_col, int F,
                                     const int32_t *frame_offsets, int batch, const float *range, const float *vsize,
                                     const int *grid, float *features, int32_t *coords, int32_t *voxel_counts,
                                     void *workspace, size_t workspace_bytes, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    TODA_CHECK_ARG(n >= 0 && n < (1ll << 31) - 64, "voxelize_dynamic: n_points=%lld out of range", (long long)n);
    TODA_CHECK_ARG(batch > 0 && batch <= 1024 && frame_offsets, "voxelize_dynamic: bad batch/frame_offsets");
    TODA_CHECK_ARG(range && vsize && grid, "voxelize_dynamic: bad geometry args");
    TODA_CHECK_ARG(stride >= 3 && xyz_col >= 0 && xyz_col + 3 <= stride && feat_col >= 0 && F > 0 &&
                       feat_col + F <= stride, "voxelize_dynamic: column layout does not fit point_stride=%d", stride);
    TODA_CHECK_ARG(features && coords && voxel_counts && workspace, "voxelize_dynamic: null output/workspace");
    for (int a = 0; a < 3; ++a)
        TODA_CHECK_ARG(grid[a] > 0 && vsize[a] > 0.f, "voxelize_dynamic: bad grid/vsize on axis %d", a);
    long long cells = index_frame_stride(grid[2], grid[1], grid[0]) * batch;
    TODA_CHECK_ARG(cells < (1ll << 32) - 1, "voxelize_dynamic: %lld cells exceed the 32-bit cell id range", cells);
    size_t smem = (size_t)kBlock * stride * sizeof(float) + 16;
    TODA_CHECK_ARG(smem <= 48 * 1024, "voxelize_dynamic: point_stride %d too large", stride);
    int64_t n_eff = n > 0 ? n : 1;
    DynWork w;
    size_t need = layout_dynamic(&w, workspace, n_eff, batch, grid);
    if (workspace_bytes < need) {
        toda_set_error("voxelize_dynamic: workspace %zu < required %zu bytes", workspace_bytes, need);
        return TODA_ERR_WORKSPACE;
    }
    VoxGeom geo;
    for (int a = 0; a < 3; ++a) { geo.lo[a] = range[a]; geo.vs[a] = vsize[a]; geo.grid[a] = grid[a]; }
    int *n_long = w.counts + 3 * batch + 8;

    size_t zero_bytes = (size_t)((char *)w.gi.rank0 - (char *)w.gi.bits0);
    TODA_CUDA_OK(cudaMemsetAsync(w.gi.bits0, 0, zero_bytes, st));
    TODA_CUDA_OK(cudaMemsetAsync(w.cnt, 0, (size_t)n_eff * 4, st));
    TODA_CUDA_OK(cudaMemsetAsync(n_long, 0, sizeof(int), st));
    if (n > 0) {
        vox_cells_kernel<<<wave_grid(n, kBlock), kBlock, smem, st>>>(points, n, stride, xyz_col, frame_offsets, batch, geo,
                                                                    w.gi, w.pt_cell);
        TODA_LAUNCH_OK();
    }
    // every voxel is kept, so the canonical rank (cid) is the output row
    if (int rc = index_build_ranks(w.gi, nullptr, (int)n_eff, w.cid_cell, w.counts, st)) return rc;
    vox_frames_kernel<<<1, 32, 0, st>>>(w.counts, batch, 0x7fffffff, voxel_counts);
    TODA_LAUNCH_OK();
    if (n > 0) {
        int g_v = wave_grid(n, kBlock);
        dyn_count_kernel<<<g_v, kBlock, 0, st>>>(w.gi, w.pt_cell, n, w.cnt);
        TODA_LAUNCH_OK();
        if (int rc = scan_exclusive(LoadInt{w.cnt}, (int)n, w.seg, w.scan_tmp, nullptr, st)) return rc;
        dyn_place_kernel<<<g_v, kBlock, 0, st>>>(w.pt_cell, n, w.seg, w.members);
        TODA_LAUNCH_OK();
        dyn_mean_short_kernel<<<g_v, kBlock, 0, st>>>(points, stride, feat_col, F, w.gi, w.cid_cell, w.counts, w.cnt, w.seg,
                                                      w.members, w.long_cids, n_long, features, (int4 *)coords);
        TODA_LAUNCH_OK();
        dyn_mean_long_kernel<<<kLongGrid, kBlock, 0, st>>>(points, stride, feat_col, F, w.gi, w.cid_cell, frame_offsets, batch,
                                                          n, w.cnt, w.seg, w.members, w.long_cids, n_long, (int *)w.pt_cell,
                                                          features);
        TODA_LAUNCH_OK();
        vox_release_kernel<<<g_v, kBlock, 0, st>>>(w.gi, w.cid_cell, w.counts);
        TODA_LAUNCH_OK();
    }
    return TODA_OK;
}

extern "C" int toda_mean_vfe_fwd(const float *voxels, const void *num_points, int num_is_float, int n_voxels, int K,
                                 int F, float *out, void *stream) {
    TODA_CHECK_ARG(n_voxels >= 0 && K > 0 && F > 0, "mean_vfe_fwd: bad sizes");
    if (n_voxels == 0) return TODA_OK;
    TODA_CHECK_ARG(voxels && num_points && out, "mean_vfe_fwd: null pointer");
    long long total = (long long)n_voxels * F;
    int grid = wave_grid(total, kBlock);
    if (num_is_float)
        mean_vfe_fwd_kernel<true><<<grid, kBlock, 0, (cudaStream_t)stream>>>(voxels, num_points, total, K, F, out);
    else
        mean_vfe_fwd_kernel<false><<<grid, kBlock, 0, (cudaStream_t)stream>>>(voxels, num_points, total, K, F, out);
    TODA_LAUNCH_OK();
    return TODA_OK;
}

extern "C" int toda_mean_vfe_bwd(const float *dout, const void *num_points, int num_is_float, int n_voxels, int K, int F,
                                 float *dvoxels, void *stream) {
    TODA_CHECK_ARG(n_voxels >= 0 && K > 0 && F > 0, "mean_vfe_bwd: bad sizes");
    if (n_voxels == 0) return TODA_OK;
    TODA_CHECK_ARG(dout && num_points && dvoxels, "mean_vfe_bwd: null pointer");
    long long total = (long long)n_voxels * K * F;
    int grid = wave_grid(total, kBlock);
    if (num_is_float)
        mean_vfe_bwd_kernel<true><<<grid, kBlock, 0, (cudaStream_t)stream>>>(dout, num_points, total, K, F, dvoxels);
    else
        mean_vfe_bwd_kernel<false><<<grid, kBlock, 0, (cudaStream_t)stream>>>(dout, num_points, total, K, F, dvoxels);
    TODA_LAUNCH_OK();
    return TODA_OK;
}
