// K5/K6 sparse convolution, TMA-fed variant of the tcgen05 implicit GEMM (see conv_tc.cu for the structure).
//
// Both operands are moved by the Tensor Memory Accelerator, so the producer side shrinks from ~1000 cp.async per
// 128x64 chunk to 33 bulk-tensor instructions issued by one warp:
//   A chunk [128 rows][ROW bytes] : 32 x cp.async.bulk.tensor.2d ... tile::gather4 -- each gathers the 4 input rows named
//                                   by the neighbour table (rows without a neighbour are pointed one past the end of
//                                   the tensor, which the TMA fills with zeros) and writes them, hardware-swizzled,
//                                   into the K-major layout tcgen05 reads
//   B chunk [Cout rows][ROW bytes]: one tiled cp.async.bulk.tensor.2d from the K-major bf16 weights [Cout][kvol*Cin]
// A chunk is ONE kernel offset (Cin <= 64: ROW = 2*Cin bytes, swizzle 32/64/128B) or half of one (Cin = 128).
// Completion is by transaction bytes on the stage's full-barrier (mbarrier.arrive.expect_tx by the issuing warp).
// Roles: warps 0-3 producers (round-robin over chunks), warp 4 MMA issuer, warps 5-8 epilogue, warp 9 table indexer.
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"
#include "epilogue.cuh"
#include "table_slice.cuh"

namespace {

constexpr int kTileM = 128;
constexpr int kMaxKvol = 27;
constexpr int kIdxBytes = kMaxKvol * kTileM * 4;
constexpr int kProdWarps = 4;
constexpr int kThreads = (kProdWarps + 1 + 4 + 1) * 32;   // 320
constexpr int kSmemBudget = 200 * 1024;

template <int CIN, int COUT> struct Cfg {
    static constexpr int kRowElems = CIN < 64 ? CIN : 64;          // K elements per chunk
    static constexpr int kRowBytes = kRowElems * 2;                // 32 / 64 / 128
    static constexpr int kABytes = kTileM * kRowBytes;
    static constexpr int kBBytes = COUT * kRowBytes;
    static constexpr int kStage = ((kABytes + kBBytes + 1023) / 1024) * 1024;
    static constexpr int kStagesRaw = (kSmemBudget - 2 * kIdxBytes) / kStage;
    static constexpr int kStages = kStagesRaw > 12 ? 12 : kStagesRaw;
    static constexpr int kSmem = kStages * kStage + 1024 + 512 + 2 * kIdxBytes;
    static constexpr int kTmemCols = 2 * COUT < 32 ? 32 : 2 * COUT;
    static constexpr int kChunksPerOffset = CIN / kRowElems;       // 1, or 2 for CIN = 128
    static constexpr int kKSteps = kRowElems / 16;                 // UMMA K = 16
    // UMMA / TMA swizzle mode for this row width
    static constexpr int kLayoutType = kRowBytes == 128 ? 2 : (kRowBytes == 64 ? 4 : 6);
    static constexpr int kSBO = 8 * kRowBytes;                     // bytes between 8-row groups
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0, spins = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (!done && ++spins > (1u << 24)) __trap();   // a lost arrival must not hang the GPU box
    }
}
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
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async_4(uint32_t dst, const void *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_arrive_noinc(uint32_t bar) {
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tma_gather4(uint32_t dst, const CUtensorMap *map, int col, int r0, int r1, int r2, int r3,
                                            uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile::gather4.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];"
        ::"r"(dst), "l"(map), "r"(col), "r"(r0), "r"(r1), "r"(r2), "r"(r3), "r"(bar)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, int c0, int c1, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// K-major swizzled matrix descriptor (cute::UMMA::SmemDescriptor): start>>4 | LBO(1)<<16 | (SBO>>4)<<32 | version 1<<46 |
// layout type<<61 (2 = SWIZZLE_128B, 4 = SWIZZLE_64B, 6 = SWIZZLE_32B)
__device__ __forceinline__ uint64_t make_desc_k(uint32_t smem_addr, int sbo_bytes, int layout_type) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3fff);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3fff) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)layout_type << 61;
    return d;
}
__host__ __device__ constexpr uint32_t make_idesc_bf16(int m, int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

template <int CIN, int COUT>
__global__ void __launch_bounds__(kThreads, 1) conv_tma_fwd_kernel(const __grid_constant__ CUtensorMap map_x,
                                                                   const __grid_constant__ CUtensorMap map_w,
                                                                   const int *__restrict__ nbr, int n_in, int n_out, int kvol,
                                                                   const float *__restrict__ bias, const float *__restrict__ addend /* optional */,
                                                                   float *__restrict__ y,
                                                                   const int *__restrict__ out_rows /* optional */,
                                                                   const uint32_t *__restrict__ tile_masks /* optional */,
                                                                   double *__restrict__ bn_sums, int num_tiles) {
    using C = Cfg<CIN, COUT>;
    constexpr int S = C::kStages;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    const uint32_t bar_base = base + S * C::kStage;
    const uint32_t full_bar = bar_base, empty_bar = bar_base + 8 * S;          // S <= 12 -> 192 bytes
    const uint32_t acc_full = bar_base + 256, acc_empty = acc_full + 16;
    const uint32_t idx_full = acc_full + 32, idx_empty = acc_full + 48;
    const uint32_t tmem_slot = acc_full + 64;
    const uint32_t idx_base = bar_base + 512;
    volatile uint32_t *tmem_slot_ptr = (volatile uint32_t *)(smem_raw + (tmem_slot - raw));

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nchunks = kvol * C::kChunksPerOffset;
    // chunks of tile t that hold at least one real neighbour (see conv_tc.cu): bit c = chunk c; every role derives the
    // same list from the tile's offset mask, an all-empty tile still walks chunk 0 so that its accumulator is defined
    auto chunk_mask_of = [&](int t) -> unsigned long long {
        if (!tile_masks) return nchunks >= 64 ? ~0ull : ((1ull << nchunks) - 1ull);
        const uint32_t om = __ldg(tile_masks + t);
        unsigned long long cm = 0ull;
        for (int c = 0; c < nchunks; ++c)
            if ((om >> (c / C::kChunksPerOffset)) & 1u) cm |= 1ull << c;
        return cm ? cm : 1ull;
    };

    if (tid == 0) {
        for (int s = 0; s < S; ++s) {
            mbar_init(full_bar + 8 * s, 1);       // one arrive.expect_tx by the issuing producer; TMA completes the bytes
            mbar_init(empty_bar + 8 * s, 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(acc_full + 8 * b, 1);
            mbar_init(acc_empty + 8 * b, 128);
            mbar_init(idx_full + 8 * b, 64);
            mbar_init(idx_empty + 8 * b, kProdWarps);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == kProdWarps) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(C::kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w) : "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot_ptr;

    if (warp < kProdWarps) {
        // ------------------------------------------------------------------ producers: warp w owns chunks g = w (mod 4)
        int it = 0;
        int g0 = 0;                       // global index of this tile's first chunk
        for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
            const int ib = it & 1;
            mbar_wait(idx_full + 8 * ib, (it >> 1) & 1);
            const uint32_t idx_tile = idx_base + ib * kIdxBytes + 16 * lane;     // rows 4*lane .. 4*lane+3 of every offset
            const unsigned long long cm0 = chunk_mask_of(t);
            int g = g0;
            for (unsigned long long cm = cm0; cm; cm &= cm - 1, ++g) {
                if (g % kProdWarps != warp) continue;                            // chunks are dealt round-robin to the warps
                const int c = __ffsll((long long)cm) - 1;
                const int s = g % S, use = g / S;
                if (use > 0) mbar_wait(empty_bar + 8 * s, (use - 1) & 1);
                const uint32_t a_tile = base + s * C::kStage, b_tile = a_tile + C::kABytes;
                const int k = c / C::kChunksPerOffset;
                const int col = (c % C::kChunksPerOffset) * C::kRowElems;
                int r0, r1, r2, r3;
                asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
                             : "r"(idx_tile + 4 * k * kTileM));
                // no neighbour -> first row past the end of x: out of bounds, filled with zeros by the TMA
                r0 = r0 < 0 ? n_in : r0; r1 = r1 < 0 ? n_in : r1; r2 = r2 < 0 ? n_in : r2; r3 = r3 < 0 ? n_in : r3;
                if (lane == 0) {
                    mbar_arrive_expect_tx(full_bar + 8 * s, C::kABytes + C::kBBytes);
                    tma_load_2d(b_tile, &map_w, k * CIN + col, 0, full_bar + 8 * s);
                }
                __syncwarp();
                tma_gather4(a_tile + lane * 4 * C::kRowBytes, &map_x, col, r0, r1, r2, r3, full_bar + 8 * s);
            }
            g0 = g;
            __syncwarp();
            if (lane == 0) mbar_arrive(idx_empty + 8 * ib);   // this warp is done with the tile's table slice
        }
    } else if (warp == kProdWarps) {
        // ------------------------------------------------------------------ MMA issuer (warp-uniform loop, one elected lane issues)
        {
            constexpr uint32_t idesc = make_idesc_bf16(kTileM, COUT);
            int g = 0, it = 0;
            uint32_t ready = 0;
            for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
                const int ab = it & 1, ause = it >> 1;
                if (ause > 0) mbar_wait(acc_empty + 8 * ab, (ause - 1) & 1);
                const uint32_t d_tmem = tmem_base + ab * COUT;
                uint32_t accumulate = 0;
                for (unsigned long long cm = chunk_mask_of(t); cm; cm &= cm - 1, ++g) {
                    const int s = g % S, use = g / S;
                    if (!ready) mbar_wait(full_bar + 8 * s, use & 1);
                    ready = mbar_test(full_bar + 8 * ((g + 1) % S), ((g + 1) / S) & 1);   // look one stage ahead
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t a_tile = base + s * C::kStage, b_tile = a_tile + C::kABytes;
                    if (elect_one()) {
#pragma unroll
                        for (int j = 0; j < C::kKSteps; ++j) {
                            uint64_t ad = make_desc_k(a_tile + j * 32, C::kSBO, C::kLayoutType);
                            uint64_t bd = make_desc_k(b_tile + j * 32, C::kSBO, C::kLayoutType);
                            umma_bf16(d_tmem, ad, bd, idesc, accumulate | (uint32_t)(j != 0));
                        }
                        umma_commit(empty_bar + 8 * s);
                    }
                    accumulate = 1u;
                    __syncwarp();
                }
                if (elect_one()) umma_commit(acc_full + 8 * ab);
                __syncwarp();
            }
        }
    } else if (warp < kProdWarps + 5) {
        // ------------------------------------------------------------------ epilogue (4 warps)
        const int q = warp & 3;                                  // TMEM lane quarter this warp may access
        float acc_s[COUT / 16], acc_q[COUT / 16];                // running per-channel sum / sum of squares (BatchNorm)
#pragma unroll
        for (int i = 0; i < COUT / 16; ++i) acc_s[i] = acc_q[i] = 0.f;
        int it = 0;
        for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
            const int ab = it & 1;
            mbar_wait(acc_full + 8 * ab, (it >> 1) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const int row = t * kTileM + q * 32 + lane;          // TMEM lane = tile row
            const int orow = (out_rows && row < n_out) ? __ldg(out_rows + row) : row;    // see conv_tc.cu
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + ab * COUT;
#pragma unroll
            for (int n0 = 0; n0 < COUT; n0 += 16) {
                uint32_t v[16];
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                    : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
                      "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                    : "r"(taddr + n0));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                float o[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) o[j] = __uint_as_float(v[j]) + (bias ? __ldg(bias + n0 + j) : 0.f);
                if (row < n_out) {
                    if (addend) {
                        const float4 *ad = (const float4 *)(addend + (size_t)orow * COUT + n0);
#pragma unroll
                        for (int qq = 0; qq < 4; ++qq) {
                            const float4 a4 = __ldg(ad + qq);
                            o[4 * qq] += a4.x; o[4 * qq + 1] += a4.y; o[4 * qq + 2] += a4.z; o[4 * qq + 3] += a4.w;
                        }
                    }
                    float4 *dst = (float4 *)(y + (size_t)orow * COUT + n0);
#pragma unroll
                    for (int qq = 0; qq < 4; ++qq) dst[qq] = make_float4(o[4 * qq], o[4 * qq + 1], o[4 * qq + 2], o[4 * qq + 3]);
                }
                if (bn_sums) {
                    // statistics of the rows just produced, for the BatchNorm that follows: no second pass over y
                    float sq[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        o[j] = row < n_out ? o[j] : 0.f;
                        sq[j] = o[j] * o[j];
                    }
                    acc_s[n0 / 16] += warp_colsum16(o, lane);
                    acc_q[n0 / 16] += warp_colsum16(sq, lane);
                }
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            mbar_arrive(acc_empty + 8 * ab);
        }
        if (bn_sums && !(lane & 1)) {
            // lane l (even) owns column n0 + ((l >> 1) & 15); one fp64 atomic per CTA-warp and channel
            const int col = (lane >> 1) & 15;
#pragma unroll
            for (int i = 0; i < COUT / 16; ++i) {
                atomicAdd(bn_sums + i * 16 + col, (double)acc_s[i]);
                atomicAdd(bn_sums + COUT + i * 16 + col, (double)acc_q[i]);
            }
        }
    } else {
        // ------------------------------------------------------------------ indexer
        int it = 0;
        for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
            const int ib = it & 1, use = it >> 1;
            if (use > 0) mbar_wait(idx_empty + 8 * ib, (use - 1) & 1);
            const uint32_t dst0 = idx_base + ib * kIdxBytes;
            const int row0 = t * kTileM;
            load_table_slice<kTileM>(dst0, nbr, n_out, row0, n_out, kvol, lane);
            cp_async_arrive_noinc(idx_full + 8 * ib);
            mbar_arrive(idx_full + 8 * ib);
        }
    }
    __syncthreads();
    if (warp == kProdWarps) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(C::kTmemCols) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

// 2-D bf16 row-major tensor [rows][cols]; box = [box_rows][box_cols]; swizzle by the box's row bytes
int make_map(CUtensorMap *m, const void *ptr, uint64_t rows, uint64_t cols, uint32_t box_rows, uint32_t box_cols) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) { toda_set_error("cuTensorMapEncodeTiled is not available in this driver"); return TODA_ERR_CUDA; }
    cuuint64_t gdim[2] = {cols, rows};
    cuuint64_t gstr[1] = {cols * 2};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    uint32_t row_bytes = box_cols * 2;
    CUtensorMapSwizzle sw = row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : (row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void *)ptr, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { toda_set_error("cuTensorMapEncodeTiled failed with code %d", (int)r); return TODA_ERR_CUDA; }
    return TODA_OK;
}

template <int CIN, int COUT>
int launch(const __nv_bfloat16 *xb, int n_in, const int32_t *nbr, int n_out, int kvol, const __nv_bfloat16 *wb, const float *bias,
           const float *addend, float *y, const int32_t *out_rows, const uint32_t *tile_masks, double *bn_sums, cudaStream_t st) {
    using C = Cfg<CIN, COUT>;
    CUtensorMap mx, mw;
    if (int rc = make_map(&mx, xb, (uint64_t)n_in, CIN, 1, C::kRowElems)) return rc;              // gather4: box = one row
    if (int rc = make_map(&mw, wb, COUT, (uint64_t)kvol * CIN, COUT, C::kRowElems)) return rc;
    int num_tiles = ceil_div(n_out, kTileM);
    int grid = num_tiles < kNumSMs ? num_tiles : kNumSMs;
    static bool attr_set = false;      // per <CIN, COUT> instantiation
    if (!attr_set) {
        TODA_CUDA_OK(cudaFuncSetAttribute(conv_tma_fwd_kernel<CIN, COUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::kSmem));
        attr_set = true;
    }
    conv_tma_fwd_kernel<CIN, COUT><<<grid, kThreads, C::kSmem, st>>>(mx, mw, nbr, n_in, n_out, kvol, bias, addend, y, out_rows, tile_masks, bn_sums, num_tiles);
    TODA_LAUNCH_OK();
    return TODA_OK;
}

}  // namespace

int conv_tma_make_map(CUtensorMap *m, const void *ptr, uint64_t rows, uint64_t cols, uint32_t box_rows, uint32_t box_cols) {
    return make_map(m, ptr, rows, cols, box_rows, box_cols);
}

// xb: bf16 [n_in][128], wb: bf16 [128][kvol*128].  Only Cin = Cout = 128 is built: narrower rows go to conv_tc.cu's
// cp.async producers, which are faster for them (profiles/r01_feed_ab.md).
int conv_tma_fwd(const void *xb, int n_in, int cin, const int32_t *nbr, int n_out, int kvol, const void *wb, int cout,
                 const float *bias, const float *addend, float *y, const int32_t *out_rows, const uint32_t *tile_masks, double *bn_sums,
                 cudaStream_t st) {
    if (cin != 128 || cout != 128) {
        toda_set_error("conv_tma_fwd: only cin=cout=128 is built, got cin=%d cout=%d", cin, cout);
        return TODA_ERR_UNSUPPORTED;
    }
    return launch<128, 128>((const __nv_bfloat16 *)xb, n_in, nbr, n_out, kvol, (const __nv_bfloat16 *)wb, bias, addend, y, out_rows,
                            tile_masks, bn_sums, st);
}
