// K5/K6 sparse convolution on the 5th-generation tensor cores (TODA_CONV_BF16):
//   y[o, :] = bias + sum_{k, ci} x[nbr[k,o], ci] * w[k, ci, :]        bf16 operands, fp32 accumulate in TMEM
//
// Implicit GEMM, output-stationary.  One CTA owns 128 output rows (UMMA M = 128, cta_group::1, which runs the
// tensor pipe at full rate) and all Cout columns (UMMA N = Cout).  The reduction dimension is the flattened
// (kernel offset, input channel) axis, K = kvol*Cin, walked in chunks of 64 bf16 = one 128-byte swizzle row:
//   A chunk [128 rows x 64]  : gathered -- for every row the neighbour named by the table, 16 bytes per
//                              cp.async, written straight into the SWIZZLE_128B K-major layout tcgen05 reads;
//                              missing neighbours (-1) are zero-filled by the same instruction (src-size 0)
//   B chunk [Cout rows x 64] : the weights, K-major ([Cout][kvol*Cin] bf16), same layout
// Warps 0-3 (128 threads) produce both chunks into a ring of shared-memory stages and later run the epilogue;
// warp 4 allocates TMEM and one of its threads issues the tcgen05.mma stream.  Stage hand-off is by mbarrier:
// full[s] completes when the 128 producers' cp.asyncs have landed (cp.async.mbarrier.arrive.noinc), empty[s]
// when the MMAs that read the stage have retired (tcgen05.commit).  Epilogue: tcgen05.ld (32 lanes x 32 bit),
// + bias, fp32 rows to global.
//
// No scatter and no atomics: every output row is written once.  dgrad is the same kernel on the
// input-stationary table with transposed weights.
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"
#include "conv.cuh"
#include "epilogue.cuh"
#include "table_slice.cuh"
#include "tcgen05.cuh"

namespace {

constexpr int kTileM = 128;
constexpr int kChunkK = 64;                       // bf16 elements per K chunk (128 bytes)
constexpr int kStages = 3;
constexpr int kProducers = 128;
constexpr int kThreadsTC = kProducers + 32;
constexpr int kABytes = kTileM * kChunkK * 2;     // 16 KB
constexpr int kBBytesMax = 128 * kChunkK * 2;     // 16 KB (Cout <= 128)
constexpr int kStageBytes = kABytes + kBBytesMax;
constexpr int kMaxKvol = 27;
constexpr int kIdxBytes = kMaxKvol * kTileM * 4;  // this tile's slice of the neighbour table (13.5 KB)
constexpr uint32_t kMaxSpins = 1u << 24;          // mbarrier probes before a wait traps (tcgen05.cuh)

__device__ __forceinline__ void cp_async_16(uint32_t dst, const void *src, uint32_t src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void st_shared_zero16(uint32_t dst) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(dst), "r"(0u) : "memory");
}
// ---- forward / dgrad kernel: persistent, warp-specialised --------------------------------------------------
//   warps 0-7   producers : gather A + copy B for every K chunk into the stage ring (cp.async, SWIZZLE_128B)
//   warp  8     MMA       : one thread issues tcgen05.mma; accumulators double-buffered in TMEM
//   warps 9-12  epilogue  : tcgen05.ld -> + bias -> fp32 rows to global, overlapped with the next tile's MMAs
//   warp  13    indexer   : streams the next tile's slice of the neighbour table into shared memory
// A CTA stays resident (grid = #SMs) and walks tiles t = blockIdx.x, blockIdx.x + gridDim.x, ...
// The producer loop is the critical path (ncu: it is issue-bound, not memory-bound), so everything in it is a
// compile-time constant or hoisted: CIN is a template parameter (no divisions), swizzled shared-memory offsets
// are per-thread constants, and the table slice is read from shared memory.
constexpr int kProdThreads = 256;
constexpr int kFwdThreads = kProdThreads + 32 + 128 + 32;   // 448
constexpr int kFwdSmemBudget = 200 * 1024;
// KB = 64-element K blocks per chunk.  Small-N MMAs are cheap, so the per-chunk barrier round trip and issue overhead
// dominate: layers with Cout <= 64 use KB = 2 (8 MMAs per round trip), Cout = 128 keeps KB = 1 (more stages).
template <int COUT, int KB> struct FwdCfg {
    static constexpr int kABlock = kTileM * kChunkK * 2;     // 16 KB per K block
    static constexpr int kBBlock = COUT * kChunkK * 2;
    static constexpr int kATile = KB * kABlock, kBTile = KB * kBBlock;
    static constexpr int kStage = kATile + kBTile;
    static constexpr int kStagesRaw = (kFwdSmemBudget - 2 * kIdxBytes) / kStage;
    static constexpr int kStages = kStagesRaw > 8 ? 8 : kStagesRaw;
    static constexpr int kSmem = kStages * kStage + 1024 + 256 + 2 * kIdxBytes;
    static constexpr int kTmemCols = 2 * COUT < 32 ? 32 : 2 * COUT;
    static_assert(kStages >= 3, "need at least 3 stages");
};

template <int CIN, int COUT, int KB>
__global__ void __launch_bounds__(kFwdThreads, 1) conv_tc_fwd_kernel(const __nv_bfloat16 *__restrict__ xb,
                                                                     const int *__restrict__ nbr, int n_out, int kvol,
                                                                     const __grid_constant__ CUtensorMap map_w /*[COUT][kvol*CIN] bf16*/,
                                                                     const float *__restrict__ bias, const float *__restrict__ addend /* optional */,
                                                                     float *__restrict__ y,
                                                                     const int *__restrict__ out_rows /* optional */,
                                                                     const uint32_t *__restrict__ tile_masks /* optional */,
                                                                     double *__restrict__ bn_sums, int num_tiles) {
    static_assert(COUT % 16 == 0 && COUT >= 16 && COUT <= 128, "UMMA N");
    static_assert(CIN == 16 || CIN == 32 || CIN == 64 || CIN == 128, "row = 32..256 bytes of bf16");
    using C = FwdCfg<COUT, KB>;
    constexpr int S = C::kStages;
    constexpr int kChunkElems = KB * kChunkK;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;   // SWIZZLE_128B tiles need 1024-byte alignment
    const uint32_t bar_base = base + S * C::kStage;
    const uint32_t full_bar = bar_base, empty_bar = bar_base + 8 * S;
    const uint32_t acc_full = bar_base + 16 * S, acc_empty = acc_full + 16;
    const uint32_t idx_full = acc_full + 32, idx_empty = acc_full + 48;
    const uint32_t tmem_slot = acc_full + 64;
    const uint32_t idx_base = bar_base + 256;
    volatile uint32_t *tmem_slot_ptr = (volatile uint32_t *)(smem_raw + (tmem_slot - raw));

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int ktot = kvol * CIN;
    const int nchunks = (ktot + kChunkElems - 1) / kChunkElems;
    // K chunks of tile t that hold at least one real neighbour (bit c = chunk c), from the tile's offset mask.  Every role
    // derives the same list, so the stage ring stays in step.  Without masks every chunk is walked.  A tile with no
    // neighbour at all still walks chunk 0 (all zero rows) so that its accumulator is defined.
    auto chunk_mask_of = [&](int t) -> unsigned long long {
        if (!tile_masks) return nchunks >= 64 ? ~0ull : ((1ull << nchunks) - 1ull);
        const uint32_t om = __ldg(tile_masks + t);
        unsigned long long cm = 0ull;
        if (CIN <= kChunkElems) {
            constexpr int kOpc = CIN <= kChunkElems ? kChunkElems / CIN : 1;       // offsets per chunk
            for (int c = 0; c < nchunks; ++c)
                if ((om >> (c * kOpc)) & ((1u << kOpc) - 1u)) cm |= 1ull << c;
        } else {
            constexpr int kCpo = CIN > kChunkElems ? CIN / kChunkElems : 1;        // chunks per offset
            for (int c = 0; c < nchunks; ++c)
                if ((om >> (c / kCpo)) & 1u) cm |= 1ull << c;
        }
        return cm ? cm : 1ull;
    };

    if (tid == 0) {
        for (int s = 0; s < S; ++s) {
            // one releasing arrival per producer warp (gathered A rows, cp.async) + one arrive.expect_tx for the weight
            // tile, which the TMA writes and completes by transaction bytes
            mbar_init(full_bar + 8 * s, kProdThreads / 32 + 1);
            mbar_init(empty_bar + 8 * s, 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(acc_full + 8 * b, 1);
            mbar_init(acc_empty + 8 * b, 128);
            mbar_init(idx_full + 8 * b, 64);
            mbar_init(idx_empty + 8 * b, kProdThreads);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 8) tmem_alloc<C::kTmemCols>(tmem_slot);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot_ptr;

    if (warp < 8) {
        // ------------------------------------------------------------------ producers (256 threads)
        const int p = tid & 7;          // 16-byte piece of the 128-byte chunk row
        const int rbase = tid >> 3;     // rows rbase + 32*i, i = 0..3  (all share r & 7 == rbase & 7)
        const uint32_t piece_off = (uint32_t)(rbase * 128 + ((p ^ (rbase & 7)) << 4));   // + i * 4096 per row step
        // which kernel offset / channel this thread's piece belongs to, per chunk c:
        //   CIN=16: k = 4c + p/2, ci = (p&1)*8      CIN=32: k = 2c + p/4, ci = (p&3)*8
        //   CIN=64: k = c,        ci = p*8          CIN=128: k = c/2,     ci = (c&1)*64 + p*8
        constexpr int kOffsPerChunk = CIN >= 64 ? 1 : 64 / CIN;
        const int k_sub = CIN >= 64 ? 0 : p / (CIN / 8);
        const int ci_lo = CIN >= 64 ? p * 8 : (p % (CIN / 8)) * 8;
        const char *xbytes = (const char *)xb + ci_lo * 2;
        const uint32_t idx_lane = idx_base + 4 * rbase;
        constexpr int kLag = S - 2;     // chunks a producer runs ahead of its completion signal
        int g = 0, it = 0;              // global chunk counter (stage ring position), tile counter
        for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
            const int ib = it & 1;
            mbar_wait<kMaxSpins>(idx_full + 8 * ib, (it >> 1) & 1);
            const uint32_t idx_tile = idx_lane + ib * kIdxBytes;
            for (unsigned long long cm = chunk_mask_of(t); cm; cm &= cm - 1, ++g) {
                const int c = __ffsll((long long)cm) - 1;
                const int s = g % S, use = g / S;
                if (use > 0) mbar_wait<kMaxSpins>(empty_bar + 8 * s, (use - 1) & 1);
                const uint32_t a_dst0 = base + s * C::kStage + piece_off;
#pragma unroll
                for (int kb = 0; kb < KB; ++kb) {
                    const int cb = c * KB + kb;                       // 64-element block index on the flattened K axis
                    const uint32_t a_dst = a_dst0 + kb * C::kABlock;
                    const int k = CIN == 128 ? (cb >> 1) : cb * kOffsPerChunk + k_sub;
                    const bool k_ok = k < kvol;      // only the K tail can miss
                    const int ci_hi = CIN == 128 ? (cb & 1) * 64 : 0;
                    int src[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        src[i] = -1;
                        if (k_ok) asm volatile("ld.shared.b32 %0, [%1];" : "=r"(src[i]) : "r"(idx_tile + 4 * (k * kTileM + 32 * i)));
                    }
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        // missing neighbour: plain zero store (a zero-size cp.async would still send a request per piece)
                        if (src[i] >= 0) cp_async_16(a_dst + i * 4096, xbytes + ((size_t)(unsigned)src[i] * CIN + ci_hi) * 2, 16u);
                        else st_shared_zero16(a_dst + i * 4096);
                    }
                }
                // weights of this chunk: one TMA tile per K block ([COUT rows][64] bf16, hardware SWIZZLE_128B; the part of
                // the box beyond K = kvol*CIN is zero-filled by the TMA)
                if (tid == 0) {
                    const int left = ktot - c * kChunkElems;                       // K elements left from this chunk on
                    const int nblk = left >= kChunkElems ? KB : (left + kChunkK - 1) / kChunkK;   // blocks that hold data
                    mbar_arrive_expect_tx(full_bar + 8 * s, nblk * C::kBBlock);
                    const uint32_t b_tile = base + s * C::kStage + C::kATile;
                    for (int kb = 0; kb < nblk; ++kb)
                        tma_load_2d(b_tile + kb * C::kBBlock, &map_w, (c * KB + kb) * kChunkK, 0, full_bar + 8 * s);
                }
                // Completion is signalled per WARP, kLag chunks later: 8 arrivals per stage instead of 512 (arrivals
                // on one mbarrier serialise lane by lane).  wait_group<kLag> returns once this thread's copies of chunk
                // g-kLag have landed; the proxy fence then also covers that chunk's zero stores.
                asm volatile("cp.async.commit_group;" ::: "memory");
                if (g >= kLag) {
                    asm volatile("cp.async.wait_group %0;" ::"n"(kLag) : "memory");
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) mbar_arrive(full_bar + 8 * ((g - kLag) % S));
                }
            }
            mbar_arrive(idx_empty + 8 * ib);   // this tile's table slice has been consumed
        }
        // drain: signal the last kLag chunks
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0)
            for (int j = (g > kLag ? g - kLag : 0); j < g; ++j) mbar_arrive(full_bar + 8 * (j % S));
    } else if (warp == 8) {
        // ------------------------------------------------------------------ MMA issuer
        // The whole warp walks the loop (warp-uniform control flow keeps descriptors in uniform registers); one elected
        // lane issues.  The issuing thread is the serial bottleneck of small-N layers, so the next stage's barrier is
        // probed (non-blocking) before the current chunk's MMAs are issued: its latency overlaps the issue.
        {
            constexpr uint32_t idesc = make_idesc_bf16(kTileM, COUT);
            int g = 0, it = 0;
            uint32_t ready = 0;
            for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
                const int ab = it & 1, ause = it >> 1;
                if (ause > 0) mbar_wait<kMaxSpins>(acc_empty + 8 * ab, (ause - 1) & 1);   // epilogue has drained this accumulator
                const uint32_t d_tmem = tmem_base + ab * COUT;
                uint32_t accumulate = 0;
                for (unsigned long long cm = chunk_mask_of(t); cm; cm &= cm - 1, ++g) {
                    const int c = __ffsll((long long)cm) - 1;
                    const int s = g % S, use = g / S;
                    if (!ready) mbar_wait<kMaxSpins>(full_bar + 8 * s, use & 1);
                    const int sn = (g + 1) % S, usen = (g + 1) / S;
                    ready = mbar_test(full_bar + 8 * sn, usen & 1);            // look one stage ahead
                    // (the producers fence their generic-proxy zero stores before signalling; no proxy fence needed here)
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t a_tile = base + s * C::kStage, b_tile = a_tile + C::kATile;
                    const int ksteps = min(kChunkElems, ktot - c * kChunkElems) / 16;     // UMMA K = 16 bf16 = 32 bytes
                    if (elect_one()) {
                        // one descriptor per operand per chunk; a K-step advances the start-address field by 32 B (>>4 = 2),
                        // the second 64-element K block starts one A / B block further
                        const uint64_t ad0 = make_desc_k_sw128(a_tile), bd0 = make_desc_k_sw128(b_tile);
                        umma_bf16(d_tmem, ad0, bd0, idesc, accumulate);
                        for (int j = 1; j < ksteps; ++j) {
                            const uint32_t blk = j >> 2, st = j & 3;
                            umma_bf16(d_tmem, ad0 + blk * (C::kABlock >> 4) + 2 * st, bd0 + blk * (C::kBBlock >> 4) + 2 * st, idesc, 1u);
                        }
                        umma_commit(empty_bar + 8 * s);        // stage reusable once these MMAs have read it
                    }
                    accumulate = 1u;
                    __syncwarp();
                }
                if (elect_one()) umma_commit(acc_full + 8 * ab);            // accumulator of this tile complete
                __syncwarp();
            }
        }
    } else if (warp < 13) {
        // ------------------------------------------------------------------ epilogue (warps 9..12)
        const int q = warp & 3;                                  // TMEM lane quarter this warp may access
        float acc_s[COUT / 16], acc_q[COUT / 16];                // running per-channel sum / sum of squares (BatchNorm)
#pragma unroll
        for (int i = 0; i < COUT / 16; ++i) acc_s[i] = acc_q[i] = 0.f;
        int it = 0;
        for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
            const int ab = it & 1;
            mbar_wait<kMaxSpins>(acc_full + 8 * ab, (it >> 1) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const int row = t * kTileM + q * 32 + lane;          // TMEM lane = tile row
            drain_accumulator<COUT>(tmem_base + ((uint32_t)(q * 32) << 16), ab, row, n_out, out_rows, bias, addend, y, bn_sums, acc_s,
                                    acc_q, lane);
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            mbar_arrive(acc_empty + 8 * ab);
        }
        flush_bn_sums<COUT>(bn_sums, acc_s, acc_q, lane);
    } else {
        // ------------------------------------------------------------------ indexer (warp 13)
        index_tiles<kTileM, kMaxSpins>(idx_base, kIdxBytes, idx_full, idx_empty, nbr, n_out, kvol, num_tiles, lane);
    }
    __syncthreads();
    if (warp == 8) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        tmem_dealloc<C::kTmemCols>(tmem_base);
    }
}

__global__ void f32_to_bf16_kernel(const float *__restrict__ in, long long n4, __nv_bfloat16 *__restrict__ out) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
        float4 v = __ldg((const float4 *)in + i);
        __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
        uint2 o;
        o.x = *(uint32_t *)&lo;
        o.y = *(uint32_t *)&hi;
        ((uint2 *)out)[i] = o;
    }
}

// x [n][cin] fp32 -> xb [n][cpad] bf16, channels >= cin zero (the 4/5-channel input layer is padded to UMMA K = 16)
__global__ void f32_to_bf16_pad_kernel(const float *__restrict__ in, long long n, int cin, int cpad,
                                       __nv_bfloat16 *__restrict__ out) {
    long long total = n * cpad;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        long long r = e / cpad;
        int c = (int)(e - r * cpad);
        out[e] = __float2bfloat16_rn(c < cin ? __ldg(in + r * cin + c) : 0.f);
    }
}

// w [kvol][cin][cout] fp32  ->  wb [cout][kvol*cpad] bf16 (K-major rows for the B operand; padded channels zero)
__global__ void weight_to_kmajor_bf16_kernel(const float *__restrict__ w, int kvol, int cin, int cpad, int cout,
                                             __nv_bfloat16 *__restrict__ wb) {
    size_t per = (size_t)kvol * cpad * cout;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < per; e += (size_t)gridDim.x * blockDim.x) {
        size_t kc = e % ((size_t)kvol * cpad);
        int co = (int)(e / ((size_t)kvol * cpad));
        int k = (int)(kc / cpad), ci = (int)(kc % cpad);
        wb[e] = __float2bfloat16_rn(ci < cin ? __ldg(w + ((size_t)k * cin + ci) * cout + co) : 0.f);
    }
}

// masks[t] bit k = some row of tile t (128 rows) has a neighbour under offset k.  One warp per tile.
__global__ void table_tile_masks_kernel(const int *__restrict__ nbr, int n_out, int kvol, int num_tiles, uint32_t *__restrict__ masks) {
    const int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (t >= num_tiles) return;
    const int row0 = t * kTileM;
    uint32_t m = 0;
    for (int k = 0; k < kvol; ++k) {
        const int *src = nbr + (size_t)k * n_out + row0;
        int any = 0;
#pragma unroll
        for (int j = 0; j < kTileM / 32; ++j) {
            const int r = lane + 32 * j;
            if (row0 + r < n_out) any |= (__ldg(src + r) >= 0);
        }
        if (__any_sync(0xffffffffu, any)) m |= 1u << k;
    }
    if (lane == 0) masks[t] = m;
}

}  // namespace

extern "C" int toda_table_tile_masks(const int32_t *nbr, int n_out, int kvol, uint32_t *masks, void *stream) {
    TODA_CHECK_ARG(n_out >= 0 && kvol > 0 && kvol <= 32, "table_tile_masks: bad sizes n_out=%d kvol=%d", n_out, kvol);
    if (n_out == 0) return TODA_OK;
    TODA_CHECK_ARG(nbr && masks, "table_tile_masks: null pointer");
    const int num_tiles = ceil_div(n_out, kTileM);
    table_tile_masks_kernel<<<ceil_div(num_tiles * 32, 256), 256, 0, (cudaStream_t)stream>>>(nbr, n_out, kvol, num_tiles, masks);
    TODA_LAUNCH_OK();
    return TODA_OK;
}

// w [kvol][cin][cout] fp32 -> [cout][kvol*max(cin,16)] bf16, the B operand of the tensor-core kernels (cacheable by the caller)
extern "C" int toda_weight_kmajor_bf16(const float *w, int kvol, int cin, int cout, void *w_bf16, void *stream) {
    TODA_CHECK_ARG(w && w_bf16 && kvol > 0 && cin > 0 && cout > 0, "weight_kmajor_bf16: bad args");
    const int cp = pad16(cin);
    weight_to_kmajor_bf16_kernel<<<wave_grid((int64_t)kvol * cp * cout, 256), 256, 0, (cudaStream_t)stream>>>(w, kvol, cin, cp, cout,
                                                                                                            (__nv_bfloat16 *)w_bf16);
    TODA_LAUNCH_OK();
    return TODA_OK;
}

bool conv_tc_supported(int cin, int cout, int kvol) {
    bool cin_ok = (cin >= 1 && cin < 16) || cin == 16 || cin == 32 || cin == 64 || cin == 128;
    return cin_ok && kvol <= kMaxKvol && (cout == 16 || cout == 32 || cout == 64 || cout == 128);
}

size_t conv_tc_fwd_workspace_bytes(int n_in, int cin, int cout, int kvol) {
    int cp = pad16(cin);
    return align_up((size_t)n_in * cp * 2 + 16, 256) + align_up((size_t)kvol * cp * cout * 2, 256) + 256;
}

int conv_tc_fwd(const float *x, const void *x_bf16, int n_in, int cin, const int32_t *nbr, int n_out, int kvol, const float *w,
                int cout, const float *bias, float *y, const int32_t *out_rows, const uint32_t *tile_masks, double *bn_sums,
                void *workspace, size_t workspace_bytes,
                cudaStream_t st, const TilePlan *plan, const float *addend, const void *w_bf16) {
    size_t need = conv_tc_fwd_workspace_bytes(n_in, cin, cout, kvol);
    if (!workspace || workspace_bytes < need) {
        toda_set_error("spconv_fwd(bf16): workspace %zu < required %zu bytes", workspace_bytes, need);
        return TODA_ERR_WORKSPACE;
    }
    const int cp = pad16(cin);
    __nv_bfloat16 *xb = (__nv_bfloat16 *)workspace;
    __nv_bfloat16 *wb = (__nv_bfloat16 *)((char *)workspace + align_up((size_t)n_in * cp * 2 + 16, 256));
    if (cp == cin && x_bf16) {
        xb = (__nv_bfloat16 *)x_bf16;       // caller already holds the bf16 copy (written by the BN-apply pass)
    } else if (cp == cin) {
        long long n4 = (long long)n_in * cin / 4;
        if (n4 > 0) {
            f32_to_bf16_kernel<<<wave_grid(n4, 256), 256, 0, st>>>(x, n4, xb);
            TODA_LAUNCH_OK();
        }
    } else if (n_in > 0) {
        f32_to_bf16_pad_kernel<<<wave_grid((int64_t)n_in * cp, 256), 256, 0, st>>>(x, n_in, cin, cp, xb);
        TODA_LAUNCH_OK();
    }
    if (w_bf16) {
        wb = (__nv_bfloat16 *)w_bf16;      // caller caches the K-major bf16 weights (toda_weight_kmajor_bf16)
    } else {
        weight_to_kmajor_bf16_kernel<<<wave_grid((int64_t)kvol * cp * cout, 256), 256, 0, st>>>(w, kvol, cin, cp, cout, wb);
        TODA_LAUNCH_OK();
    }
    cin = cp;
    if (bn_sums) TODA_CUDA_OK(cudaMemsetAsync(bn_sums, 0, 2 * (size_t)cout * sizeof(double), st));
    // with a tile plan (toda_table_tile_plan) the row-cache / TMEM-operand kernel takes every supported shape
    if (conv_ts_supported(cin, cout, kvol, plan))
        return conv_ts_fwd(xb, n_in, cin, nbr, n_out, kvol, *plan, wb, cout, bias, addend, y, out_rows, tile_masks, bn_sums, st);
    // otherwise the operand feed is chosen by shape from measurements on B200 (profiles/r01_feed_ab.md): TMA (gather4 rows +
    // tiled weights, conv_tma.cu) wins when rows are 256 bytes (Cin = Cout = 128); gather4 costs ~20-50 cycles per
    // instruction whatever the row width, so the cp.async producers below are faster for narrower rows.
    if (cin == 128 && cout == 128) {
        // (raster-order masks skip ~17 % of the 128-channel chunks but measured slower on this kernel -- the skipped chunks
        // unbalance the round-robin of its four issuing warps; class-sorted dgrad rows, where most chunks vanish, keep them)
        return conv_tma_fwd(xb, n_in, cin, nbr, n_out, kvol, wb, cout, bias, addend, y, out_rows, out_rows ? tile_masks : nullptr, bn_sums, st);
    }
    int num_tiles = ceil_div(n_out, kTileM);
    int grid = num_tiles < kNumSMs ? num_tiles : kNumSMs;   // persistent: one CTA per SM walks the tiles
    CUtensorMap map_w;
    if (int rc = make_tensor_map_bf16(&map_w, wb, (uint64_t)cout, (uint64_t)kvol * cin, (uint32_t)cout, kChunkK)) return rc;
    // K blocks per chunk: 2 for Cout <= 64 (8 MMAs per barrier round trip), 1 for Cout = 128 (more stages); the A/B is in
    // profiles/r01_feed_ab.md
#define LAUNCH_TC(CI, CO)                                                                                                    \
    do {                                                                                                                     \
        constexpr int KB_ = (CO) <= 64 ? 2 : 1;                                                                              \
        constexpr int smem = FwdCfg<CO, KB_>::kSmem;                                                                         \
        static bool attr_set = false;                                                                                        \
        if (!attr_set) {                                                                                                     \
            TODA_CUDA_OK(cudaFuncSetAttribute(conv_tc_fwd_kernel<CI, CO, KB_>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); \
            attr_set = true;                                                                                                 \
        }                                                                                                                    \
        conv_tc_fwd_kernel<CI, CO, KB_><<<grid, kFwdThreads, smem, st>>>(xb, nbr, n_out, kvol, map_w, bias, addend, y, out_rows, tile_masks, bn_sums, num_tiles); \
    } while (0)
#define LAUNCH_TC_CO(CI)                                                                                 \
    switch (cout) {                                                                                      \
        case 16: LAUNCH_TC(CI, 16); break;                                                               \
        case 32: LAUNCH_TC(CI, 32); break;                                                               \
        case 64: LAUNCH_TC(CI, 64); break;                                                               \
        case 128: LAUNCH_TC(CI, 128); break;                                                             \
        default: toda_set_error("conv_tc_fwd: unsupported cout %d", cout); return TODA_ERR_UNSUPPORTED;  \
    }
    switch (cin) {
        case 16: LAUNCH_TC_CO(16); break;
        case 32: LAUNCH_TC_CO(32); break;
        case 64: LAUNCH_TC_CO(64); break;
        case 128:                       // (Cout = 128 went to conv_tma_fwd above)
            switch (cout) {
                case 16: LAUNCH_TC(128, 16); break;
                case 32: LAUNCH_TC(128, 32); break;
                case 64: LAUNCH_TC(128, 64); break;
                default: toda_set_error("conv_tc_fwd: unsupported cout %d", cout); return TODA_ERR_UNSUPPORTED;
            }
            break;
        default: toda_set_error("conv_tc_fwd: unsupported cin %d", cin); return TODA_ERR_UNSUPPORTED;
    }
#undef LAUNCH_TC_CO
#undef LAUNCH_TC
    TODA_LAUNCH_OK();
    return TODA_OK;
}

namespace {

// ---------------------------------------------------------------------------------------------------------------
// K7 weight gradient on tensor cores:  dw[k][ci][co] = sum_o x[nbr[k,o], ci] * dy[o, co]
// The reduction runs over output rows, so both operands are "MN-major" for tcgen05: shared-memory tiles are
// [row][channel] with channels contiguous (exactly how rows are gathered), rows being the UMMA K dimension.
//   A tile [64 rows][128 M-slots]: M = (128/Cin) kernel offsets x Cin channels -- small-channel layers stack several
//                                  offsets on the M axis so that every MMA is a full M=128 instruction
//   B tile [64 rows][NPAD]       : dy rows (NPAD = max(64, Cout); columns >= Cout are zero)
// One "pass" = one group of 128/Cin offsets = one [128 x NPAD] fp32 accumulator in TMEM; a CTA keeps up to
// 512/NPAD passes resident and owns a slice of the rows (split-K over rows); partial results go to a workspace
// and are reduced in a fixed order (deterministic) into the parameter layout.
// ---------------------------------------------------------------------------------------------------------------
// Per-launch geometry of the wgrad kernel.  ROWS = reduction rows per item (ROWS/16 UMMA K-steps): 128 for N <= 64
// (small-N MMAs are cheap, so the per-item barrier / issue overhead dominates and bigger items pay), 64 for N = 128.
template <int NPAD, int ROWS> struct WCfg {
    static constexpr int kATile = 2 * ROWS * 128;              // two 64-wide M blocks
    static constexpr int kBTile = (NPAD / 64) * ROWS * 128;    // one or two 64-wide N blocks
    static constexpr int kIdx = 32 * ROWS * 4;                 // table slice of one row chunk: <= 32 offset slots
    static constexpr int kBBufs = ROWS == 128 ? 2 : 3;         // dy tiles in flight
    static constexpr int kStages = ROWS == 128 ? 4 : 8;        // A ring
    static constexpr int kLag = ROWS == 128 ? 2 : 3;           // items a producer runs ahead of its completion signal
    static constexpr int kSmem = kStages * kATile + kBBufs * kBTile + 2 * kIdx + 1024 + 256;
};
constexpr int kWgradThreads = kProdThreads + 32 + 128 + 32;

// MN-major SWIZZLE_128B descriptor: 64 channels (128 B) contiguous, next 64-channel block at `lbo` bytes,
// groups of 8 rows 1024 B apart.
__device__ __forceinline__ uint64_t make_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3fff);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

// Live passes (bit ps) of row chunk c (rows c*rows ..) for the npass passes of opp offsets from offset k0: those with a
// neighbour under one of their offsets in the 128-row tile that encloses the chunk (a 64-row chunk reads its tile's word,
// which may claim more than the chunk holds but never misses a neighbour).  No masks: every pass.
__device__ __forceinline__ uint32_t wgrad_live_passes(const uint32_t *__restrict__ tile_masks, int c, int rows, int k0, int npass,
                                                      int opp) {
    if (!tile_masks) return (1u << npass) - 1u;
    const uint32_t om = __ldg(tile_masks + ((c * rows) >> 7)) >> k0;
    uint32_t lm = 0;
    for (int ps = 0; ps < npass; ++ps)
        if ((om >> (ps * opp)) & ((1u << opp) - 1u)) lm |= 1u << ps;
    return lm;
}

// Row chunks [c_begin, c_end) of split `split` of one offset group: the group's chunks cut into `splits` contiguous ranges
// with equal shares of its live items.  Split s starts at the first chunk c whose preceding chunks hold at least
// floor(s*T/splits) of the T live items (the last split ends at the last chunk).  The boundaries depend only on the
// masks, so the partition of the fp32 partial sums -- and the result -- is the same on every run.  Called by the whole
// block; scratch: blockDim.x + 2 ints of shared memory.
__device__ void wgrad_split_chunks(const uint32_t *__restrict__ tile_masks, int n_out, int rows, int k0, int npass, int opp,
                                   int split, int splits, int *scratch, int &c_begin, int &c_end) {
    const int tid = threadIdx.x, nt = blockDim.x;
    const int nch = (n_out + rows - 1) / rows;
    const int per = (nch + nt - 1) / nt, c0 = min(nch, tid * per), c1 = min(nch, c0 + per);
    int local = 0;
    for (int c = c0; c < c1; ++c) local += __popc(wgrad_live_passes(tile_masks, c, rows, k0, npass, opp));
    if (tid == 0) scratch[nt] = scratch[nt + 1] = 0;
    scratch[tid] = local;
    __syncthreads();
    for (int off = 1; off < nt; off <<= 1) {           // inclusive scan of the per-thread counts
        const int v = tid >= off ? scratch[tid - off] : 0;
        __syncthreads();
        scratch[tid] += v;
        __syncthreads();
    }
    const long long total = scratch[nt - 1];
    const long long ta = (long long)split * total / splits, tb = (long long)(split + 1) * total / splits;
    int run = scratch[tid] - local, na = 0, nb = 0;    // live items before chunk c
    for (int c = c0; c < c1; ++c) {
        na += run < ta;
        nb += run < tb;
        run += __popc(wgrad_live_passes(tile_masks, c, rows, k0, npass, opp));
    }
    if (na) atomicAdd(scratch + nt, na);
    if (nb) atomicAdd(scratch + nt + 1, nb);
    __syncthreads();
    c_begin = split == 0 ? 0 : scratch[nt];
    c_end = split + 1 == splits ? nch : scratch[nt + 1];
}

// Roles as in the forward kernel: warps 0-7 produce (gather x rows per pass into the A ring; dy rows once per row
// chunk into a double-buffered B tile), warp 8 issues the MMAs, warps 9-12 drain TMEM at the end, warp 13 streams
// the table slice of the next row chunk into shared memory.  The row range of the CTA is computed first, by the whole
// block (wgrad_split_chunks, gridDim.x splits per offset group).
template <int CIN, int NPAD, int ROWS>
__global__ void __launch_bounds__(kWgradThreads, 1) conv_tc_wgrad_kernel(const __nv_bfloat16 *__restrict__ xb,
                                                                         const int *__restrict__ nbr, int n_out, int kvol,
                                                                         const __nv_bfloat16 *__restrict__ dyb, int cout,
                                                                         const uint32_t *__restrict__ tile_masks /* optional */,
                                                                         int passes_per_cta, float *__restrict__ partial) {
    using W = WCfg<NPAD, ROWS>;
    constexpr int kOffsPerPass = 128 / CIN;
    constexpr int S = W::kStages;
    constexpr int kRowsW = ROWS, kATileW = W::kATile, kBTileW = W::kBTile, kIdxW = W::kIdx, kBBufsW = W::kBBufs;
    constexpr int kRowIters = ROWS / 32;            // rows per producer thread per 64-wide block
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    const uint32_t b_base = base + S * kATileW;
    const uint32_t idx_base = b_base + kBBufsW * kBTileW;
    const uint32_t bar_base = idx_base + 2 * kIdxW;
    const uint32_t a_full = bar_base, a_empty = bar_base + 8 * S;
    const uint32_t b_full = bar_base + 16 * S, b_empty = b_full + 32;
    const uint32_t idx_full = b_full + 64, idx_empty = b_full + 80;
    const uint32_t accum_bar = b_full + 96, tmem_slot = b_full + 104;
    volatile uint32_t *tmem_slot_ptr = (volatile uint32_t *)(smem_raw + (tmem_slot - raw));

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int split = blockIdx.x, group = blockIdx.y;
    const int total_passes = (kvol + kOffsPerPass - 1) / kOffsPerPass;
    const int pass0 = group * passes_per_cta;
    const int npass = min(passes_per_cta, total_passes - pass0);
    const int k0 = pass0 * kOffsPerPass;                         // first kernel offset of this CTA
    const int noffs = min(npass * kOffsPerPass, kvol - k0);      // offsets this CTA really owns
    int c_begin, c_end;     // scratch: the A ring, which nothing uses before the __syncthreads below
    wgrad_split_chunks(tile_masks, n_out, kRowsW, k0, npass, kOffsPerPass, split, gridDim.x, (int *)(smem_raw + (base - raw)),
                       c_begin, c_end);
    const int r_begin = c_begin * kRowsW;
    const int r_end = min(n_out, c_end * kRowsW);
    const int nchunks = c_end - c_begin;
    // An item = a live (chunk, pass) pair; every role derives the same item sequence from the same mask words, so the
    // rings stay in step.  Chunks without a live pass are skipped whole (no dy rows, no table slice).
    auto live_of = [&](int rc) -> uint32_t {
        return wgrad_live_passes(tile_masks, c_begin + rc, kRowsW, k0, npass, kOffsPerPass);
    };

    if (tid == 0) {
        for (int s = 0; s < S; ++s) {
            mbar_init(a_full + 8 * s, kProdThreads / 32);
            mbar_init(a_empty + 8 * s, 1);
        }
        for (int b = 0; b < kBBufsW; ++b) {
            mbar_init(b_full + 8 * b, kProdThreads / 32);
            mbar_init(b_empty + 8 * b, 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(idx_full + 8 * b, 64);
            mbar_init(idx_empty + 8 * b, kProdThreads);
        }
        mbar_init(accum_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // TMEM columns: one [128 x NPAD] accumulator per resident pass, rounded up to a power of two
    uint32_t tmem_cols = 32;
    while ((int)tmem_cols < passes_per_cta * NPAD) tmem_cols <<= 1;
    if (warp == 8) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot_ptr;

    if (warp < 8) {
        // ------------------------------------------------------------------ producers
        const int p = tid & 7, rbase = tid >> 3;       // 16-byte piece; rows rbase, rbase + 32
        const uint32_t piece_off = (uint32_t)(rbase * 128 + ((p ^ (rbase & 7)) << 4));
        // M slot m = mb*64 + p*8 -> (offset within the pass, channel)
        //   CIN=128: (0, mb*64+p*8)  CIN=64: (mb, p*8)  CIN=32: (2mb + p/4, (p%4)*8)  CIN=16: (4mb + p/2, (p%2)*8)
        const int off_lo = CIN >= 64 ? 0 : p / (CIN / 8);
        const int ci_lo = CIN >= 64 ? p * 8 : (p % (CIN / 8)) * 8;
        // Completion of item j is signalled kLagW items later (per warp, see the forward kernel); the dy tile of a live
        // chunk joins the cp.async group of the chunk's first item and is signalled (b_full) with it.
        // Hang freedom.  (a) A ring: before item g overwrites stage g % S the MMAs of item g-S must be done, and they need
        // the signals of items <= g-S; signalled are items < g-kLagW, so kLagW <= S-1 suffices (4/2, 8/3), whatever the
        // chunks.  (b) dy ring: before live chunk lc overwrites dy buffer lc % kBBufsW, the MMA warp must have finished live
        // chunk lc-kBBufsW, i.e. every item of it must be signalled: signalled >= first item of live chunk
        // lc-kBBufsW+1.  With a fixed npass items per chunk that held for kLagW <= (kBBufsW-1)*npass; with a variable
        // number of live passes per chunk it can fail (chunks of one live item), so it is tested here and, where it fails,
        // the producer drains: waits for all of its copies and signals every pending item before it waits on b_empty.
        // (c) The table-slice ring involves only the indexer and the producers.
        constexpr int kLagW = W::kLag;
        int g = 0, signalled = 0;       // items issued / items signalled
        int lc = 0, bsig = 0;           // live chunks started / dy tiles signalled
        int first1 = 0, first2 = 0;     // first item of live chunk lc-1 / lc-2
        uint32_t pend_first = 0;        // bit i: pending item signalled+i is the first of its chunk (carries its dy tile)
        auto signal_next = [&]() {
            if (lane == 0) {
                if (pend_first & 1u) mbar_arrive(b_full + 8 * (bsig % kBBufsW));
                mbar_arrive(a_full + 8 * (signalled % S));
            }
            bsig += pend_first & 1u;
            pend_first >>= 1;
            ++signalled;
        };
        for (int rc = 0; rc < nchunks; ++rc) {
            const uint32_t lm = live_of(rc);
            if (!lm) continue;
            const int ib = lc & 1, use_i = lc >> 1;
            const int bb = lc % kBBufsW, use_b = lc / kBBufsW;
            const int row_base = r_begin + rc * kRowsW;
            if (use_b > 0 && signalled < (kBBufsW == 2 ? first1 : first2)) {
                asm volatile("cp.async.wait_group 0;" ::: "memory");
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                while (signalled < g) signal_next();
            }
            first2 = first1;
            first1 = g;
            // dy rows of this chunk (shared by every pass)
            if (use_b > 0) mbar_wait<kMaxSpins>(b_empty + 8 * bb, (use_b - 1) & 1);
            {
                const uint32_t b_dst = b_base + bb * kBTileW + piece_off;
#pragma unroll
                for (int nb = 0; nb < NPAD / 64; ++nb) {
                    const int co = nb * 64 + p * 8;
#pragma unroll
                    for (int i = 0; i < kRowIters; ++i) {
                        const int row = row_base + rbase + 32 * i;
                        const uint32_t dst = b_dst + nb * (kRowsW * 128) + i * 4096;
                        if (row < r_end && co < cout) cp_async_16(dst, dyb + (size_t)row * cout + co, 16u);
                        else st_shared_zero16(dst);
                    }
                }
            }
            mbar_wait<kMaxSpins>(idx_full + 8 * ib, use_i & 1);
            const uint32_t idx_tile = idx_base + ib * kIdxW + 4 * rbase;
            for (uint32_t m = lm; m; m &= m - 1, ++g) {
                const int ps = __ffs(m) - 1;
                if (m == lm) pend_first |= 1u << (g - signalled);
                const int s = g % S, use = g / S;
                if (use > 0) mbar_wait<kMaxSpins>(a_empty + 8 * s, (use - 1) & 1);
                const uint32_t a_dst = base + s * kATileW + piece_off;
#pragma unroll
                for (int mb = 0; mb < 2; ++mb) {
                    const int koff = ps * kOffsPerPass + (CIN == 128 ? 0 : (CIN == 64 ? mb : mb * (kOffsPerPass / 2) + off_lo));
                    const int ci = CIN == 128 ? mb * 64 + ci_lo : ci_lo;
                    const bool k_ok = koff < noffs;
                    int src[kRowIters];
#pragma unroll
                    for (int i = 0; i < kRowIters; ++i) {
                        src[i] = -1;
                        if (k_ok) asm volatile("ld.shared.b32 %0, [%1];" : "=r"(src[i]) : "r"(idx_tile + 4 * (koff * kRowsW + 32 * i)));
                    }
#pragma unroll
                    for (int i = 0; i < kRowIters; ++i) {
                        const uint32_t dst = a_dst + mb * (kRowsW * 128) + i * 4096;
                        if (src[i] >= 0) cp_async_16(dst, xb + (size_t)(unsigned)src[i] * CIN + ci, 16u);
                        else st_shared_zero16(dst);
                    }
                }
                asm volatile("cp.async.commit_group;" ::: "memory");
                if (g - signalled >= kLagW) {
                    // the copies of item signalled (= g - kLagW) have landed
                    asm volatile("cp.async.wait_group %0;" ::"n"(kLagW) : "memory");
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    signal_next();
                }
            }
            mbar_arrive(idx_empty + 8 * ib);
            ++lc;
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        while (signalled < g) signal_next();
    } else if (warp == 8) {
        // ------------------------------------------------------------------ MMA issuer (warp-uniform loop, one elected lane issues)
        if (nchunks > 0) {
            // D = A(MN-major) x B(MN-major): bits 15 / 16 of the instruction descriptor select MN-major operands
            constexpr uint32_t idesc = make_idesc_bf16(128, NPAD) | (1u << 15) | (1u << 16);
            int g = 0, lc = 0;
            uint32_t ready = 0, started = 0;     // bit ps: pass ps's accumulator holds its first live item
            for (int rc = 0; rc < nchunks; ++rc) {
                const uint32_t lm = live_of(rc);
                if (!lm) continue;
                const int ib = lc % kBBufsW;
                mbar_wait<kMaxSpins>(b_full + 8 * ib, (lc / kBBufsW) & 1);
                const uint32_t b_tile = b_base + ib * kBTileW;
                for (uint32_t m = lm; m; m &= m - 1, ++g) {
                    const int ps = __ffs(m) - 1;
                    const int s = g % S, use = g / S;
                    if (!ready) mbar_wait<kMaxSpins>(a_full + 8 * s, use & 1);
                    ready = mbar_test(a_full + 8 * ((g + 1) % S), ((g + 1) / S) & 1);   // look one stage ahead
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t a_tile = base + s * kATileW;
                    if (elect_one()) {
#pragma unroll
                        // UMMA K = 16 rows = 2 swizzle atoms of 8 rows = 2048 B: a K-step adds 128 to the start-address field
                        const uint64_t ad0 = make_desc_mn_sw128(a_tile, kRowsW * 128), bd0 = make_desc_mn_sw128(b_tile, kRowsW * 128);
                        umma_bf16(tmem_base + ps * NPAD, ad0, bd0, idesc, (started >> ps) & 1u);
                        for (int j = 1; j < kRowsW / 16; ++j)
                            umma_bf16(tmem_base + ps * NPAD, ad0 + 128 * j, bd0 + 128 * j, idesc, 1u);
                        umma_commit(a_empty + 8 * s);
                    }
                    __syncwarp();
                }
                started |= lm;
                if (elect_one()) umma_commit(b_empty + 8 * ib);      // dy tile reusable once every live pass of this chunk has read it
                __syncwarp();
                ++lc;
            }
            if (g > 0) {
                if (elect_one()) umma_commit(accum_bar);
                __syncwarp();
            }
        }
    } else if (warp < 13) {
        // ------------------------------------------------------------------ epilogue: TMEM lane = M slot (offset, ci)
        const int q = warp & 3;
        uint32_t used = 0;                                       // passes with at least one live item (written TMEM)
        for (int rc = 0; rc < nchunks; ++rc) used |= live_of(rc);
        if (used) {
            mbar_wait<kMaxSpins>(accum_bar, 0);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        }
        const int m = q * 32 + lane;
        for (int ps = 0; ps < npass; ++ps) {
            const int k = (pass0 + ps) * kOffsPerPass + m / CIN, ci = m % CIN;
            float *dst = partial + (((size_t)split * kvol + k) * CIN + ci) * cout;
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + ps * NPAD;
            for (int n0 = 0; n0 < cout; n0 += 16) {
                uint32_t v[16];
                if ((used >> ps) & 1u) {
                    asm volatile(
                        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                        : "r"(taddr + n0));
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                } else {
#pragma unroll
                    for (int qq = 0; qq < 16; ++qq) v[qq] = 0u;      // no live item of this pass in this split: its partial is zero
                }
                if (k < kvol) {
#pragma unroll
                    for (int qq = 0; qq < 4; ++qq)
                        *(float4 *)(dst + n0 + 4 * qq) = make_float4(__uint_as_float(v[4 * qq]), __uint_as_float(v[4 * qq + 1]),
                                                                     __uint_as_float(v[4 * qq + 2]), __uint_as_float(v[4 * qq + 3]));
                }
            }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    } else {
        // ------------------------------------------------------------------ indexer (warp 13)
        for (int rc = 0, lc = 0; rc < nchunks; ++rc) {
            if (!live_of(rc)) continue;
            const int ib = lc & 1, use = lc >> 1;
            ++lc;
            if (use > 0) mbar_wait<kMaxSpins>(idx_empty + 8 * ib, (use - 1) & 1);
            const uint32_t dst0 = idx_base + ib * kIdxW;
            const int row_base = r_begin + rc * kRowsW;
            load_table_slice<ROWS>(dst0, nbr + (size_t)k0 * n_out, n_out, row_base, r_end, noffs, lane);
            cp_async_arrive_noinc(idx_full + 8 * ib);
            mbar_arrive(idx_full + 8 * ib);
        }
    }
    __syncthreads();
    if (warp == 8) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
    }
}

// fixed-order reduction over splits into the parameter layout (Cout, kvol, Cin)
// partial: [splits][kvol][cpad][cout].  Block = 32 consecutive source elements (coalesced 128-byte reads) x 8 split
// subsets, combined through shared memory in a fixed tree (deterministic); the transposing write is the small side.
__global__ void __launch_bounds__(256) wgrad_tc_reduce_kernel(const float *__restrict__ partial, int splits, int kvol, int cin,
                                                              int cpad, int cout, float *__restrict__ dw_param) {
    __shared__ float red[8][33];
    const size_t per_pad = (size_t)kvol * cpad * cout;
    const int x = threadIdx.x & 31, y = threadIdx.x >> 5;
    for (size_t e0 = (size_t)blockIdx.x * 32; e0 < per_pad; e0 += (size_t)gridDim.x * 32) {
        const size_t e = e0 + x;
        float s = 0.f;
        if (e < per_pad) {
#pragma unroll 4
            for (int sp = y; sp < splits; sp += 8) s += __ldg(partial + sp * per_pad + e);
        }
        red[y][x] = s;
        __syncthreads();
        if (y == 0 && e < per_pad) {
            s = ((red[0][x] + red[1][x]) + (red[2][x] + red[3][x])) + ((red[4][x] + red[5][x]) + (red[6][x] + red[7][x]));
            const int co = (int)(e % cout);
            const size_t t = e / cout;
            const int ci = (int)(t % cpad), k = (int)(t / cpad);
            if (ci < cin) dw_param[((size_t)co * kvol + k) * cin + ci] = s;
        }
        __syncthreads();
    }
}

struct WgradPlan {
    int passes_per_cta, groups, splits, rows;
    size_t xb_bytes, dyb_bytes, partial_bytes;
};

WgradPlan wgrad_plan(int n_in, int n_out, int kvol, int cin, int cout) {
    WgradPlan p;
    int npad = cout <= 64 ? 64 : 128;
    const int kRowsW = npad == 64 ? 128 : 64;
    int offs = 128 / cin;
    int total_passes = (kvol + offs - 1) / offs;
    p.passes_per_cta = total_passes < 512 / npad ? total_passes : 512 / npad;
    p.groups = (total_passes + p.passes_per_cta - 1) / p.passes_per_cta;
    int want = kNumSMs / p.groups;   // one resident CTA per SM, a single wave
    if (want < 1) want = 1;
    int max_by_rows = (n_out + 4 * kRowsW - 1) / (4 * kRowsW);
    p.splits = want < max_by_rows ? want : max_by_rows;
    if (p.splits < 1) p.splits = 1;
    p.rows = kRowsW;
    p.xb_bytes = align_up((size_t)n_in * cin * 2 + 16, 256);
    p.dyb_bytes = align_up((size_t)n_out * cout * 2 + 16, 256);
    p.partial_bytes = align_up((size_t)p.splits * kvol * cin * cout * 4, 256);
    return p;
}

// first row of every (offset group, split) of a wgrad launch: row_begin[group * splits + split]
__global__ void __launch_bounds__(kWgradThreads) wgrad_row_splits_kernel(const uint32_t *__restrict__ tile_masks, int n_out,
                                                                         int kvol, int opp, int rows, int passes_per_cta,
                                                                         int32_t *__restrict__ row_begin) {
    __shared__ int scratch[kWgradThreads + 2];
    const int total_passes = (kvol + opp - 1) / opp, pass0 = blockIdx.y * passes_per_cta;
    int c_begin, c_end;
    wgrad_split_chunks(tile_masks, n_out, rows, pass0 * opp, min(passes_per_cta, total_passes - pass0), opp, blockIdx.x, gridDim.x,
                       scratch, c_begin, c_end);
    if (threadIdx.x == 0) row_begin[blockIdx.y * gridDim.x + blockIdx.x] = min(n_out, c_begin * rows);
}

}  // namespace

extern "C" int toda_spconv_wgrad_row_splits(const uint32_t *tile_masks, int n_out, int kvol, int cin, int cout, int *groups,
                                            int *splits, int32_t *row_begin, void *stream) {
    TODA_CHECK_ARG(n_out > 0 && kvol > 0 && kvol <= kMaxKvol && groups && splits && conv_tc_wgrad_supported(cin, cout, kvol),
                   "spconv_wgrad_row_splits: bad args");
    const int cp = pad16(cin);
    WgradPlan p = wgrad_plan(0, n_out, kvol, cp, cout);
    *groups = p.groups;
    *splits = p.splits;
    if (!row_begin) return TODA_OK;
    wgrad_row_splits_kernel<<<dim3(p.splits, p.groups), kWgradThreads, 0, (cudaStream_t)stream>>>(tile_masks, n_out, kvol, 128 / cp,
                                                                                                  p.rows, p.passes_per_cta, row_begin);
    TODA_LAUNCH_OK();
    return TODA_OK;
}

bool conv_tc_wgrad_supported(int cin, int cout, int kvol) {
    // (the kernel's shared-memory table slice holds at most 32 offsets: larger kernels take the fp32 wgrad)
    return kvol <= kMaxKvol && ((cin >= 1 && cin <= 16) || cin == 32 || cin == 64 || cin == 128) && (cout == 16 || cout == 32 || cout == 64 || cout == 128);
}

size_t conv_tc_wgrad_workspace_bytes(int n_in, int n_out, int kvol, int cin, int cout) {
    WgradPlan p = wgrad_plan(n_in, n_out, kvol, pad16(cin), cout);
    return p.xb_bytes + p.dyb_bytes + p.partial_bytes + 256;
}

int conv_tc_wgrad(const float *x, const void *x_bf16, int n_in, int cin, const int32_t *nbr, int n_out, int kvol,
                  const uint32_t *tile_masks, const float *dy, const void *dy_bf16, int cout, float *dw_param, void *workspace,
                  size_t workspace_bytes, cudaStream_t st) {
    const int cin_real = cin;
    cin = pad16(cin);
    WgradPlan p = wgrad_plan(n_in, n_out, kvol, cin, cout);
    size_t need = p.xb_bytes + p.dyb_bytes + p.partial_bytes;
    if (!workspace || workspace_bytes < need) {
        toda_set_error("spconv_wgrad(bf16): workspace %zu < required %zu bytes", workspace_bytes, need);
        return TODA_ERR_WORKSPACE;
    }
    __nv_bfloat16 *xb = (__nv_bfloat16 *)workspace;
    __nv_bfloat16 *dyb = (__nv_bfloat16 *)((char *)workspace + p.xb_bytes);
    float *partial = (float *)((char *)workspace + p.xb_bytes + p.dyb_bytes);
    long long n4 = (long long)n_in * cin / 4;
    if (cin_real != cin) {
        if (n_in > 0) {
            f32_to_bf16_pad_kernel<<<wave_grid((int64_t)n_in * cin, 256), 256, 0, st>>>(x, n_in, cin_real, cin, xb);
            TODA_LAUNCH_OK();
        }
    } else if (x_bf16) {
        xb = (__nv_bfloat16 *)x_bf16;
    } else if (n4 > 0) {
        f32_to_bf16_kernel<<<wave_grid(n4, 256), 256, 0, st>>>(x, n4, xb);
        TODA_LAUNCH_OK();
    }
    if (dy_bf16) {
        dyb = (__nv_bfloat16 *)dy_bf16;
    } else {
        n4 = (long long)n_out * cout / 4;
        f32_to_bf16_kernel<<<wave_grid(n4, 256), 256, 0, st>>>(dy, n4, dyb);
        TODA_LAUNCH_OK();
    }
    dim3 grid(p.splits, p.groups);
#define LAUNCH_W(CI, NP, RW)                                                                                              \
    do {                                                                                                                   \
        constexpr int smem = WCfg<NP, RW>::kSmem;                                                                          \
        static bool attr_set = false;                                                                                      \
        if (!attr_set) {                                                                                                   \
            TODA_CUDA_OK(cudaFuncSetAttribute(conv_tc_wgrad_kernel<CI, NP, RW>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); \
            attr_set = true;                                                                                               \
        }                                                                                                                  \
        conv_tc_wgrad_kernel<CI, NP, RW><<<grid, kWgradThreads, smem, st>>>(xb, nbr, n_out, kvol, dyb, cout, tile_masks,       \
                                                                           p.passes_per_cta, partial);                      \
    } while (0)
    const bool wide = cout > 64;
    switch (cin) {
        case 16: if (wide) LAUNCH_W(16, 128, 64); else LAUNCH_W(16, 64, 128); break;
        case 32: if (wide) LAUNCH_W(32, 128, 64); else LAUNCH_W(32, 64, 128); break;
        case 64: if (wide) LAUNCH_W(64, 128, 64); else LAUNCH_W(64, 64, 128); break;
        case 128: if (wide) LAUNCH_W(128, 128, 64); else LAUNCH_W(128, 64, 128); break;
        default: toda_set_error("conv_tc_wgrad: unsupported cin %d", cin); return TODA_ERR_UNSUPPORTED;
    }
#undef LAUNCH_W
    TODA_LAUNCH_OK();
    size_t per_pad = (size_t)kvol * cin * cout;
    wgrad_tc_reduce_kernel<<<wave_grid(per_pad * 8, 256), 256, 0, st>>>(partial, p.splits, kvol, cin_real, cin, cout, dw_param);
    TODA_LAUNCH_OK();
    return TODA_OK;
}
