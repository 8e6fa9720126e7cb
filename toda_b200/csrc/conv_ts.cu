// K5/K6 sparse convolution, row-cache + TMEM-operand variant of the tcgen05 implicit GEMM ("TS" kernel).
//
//   y[o, :] = bias + sum_{k, ci} x[nbr[k,o], ci] * w[k, ci, :]  (+ addend[o, :])      bf16 operands, fp32 accumulate
//
// Why another kernel: conv_tc.cu / conv_tma.cu gather every A row from L2 once per (offset, output row) -- in raster
// order the same input row is fetched 2.5-4 times per 128-row tile (profiles/r01_feed_ab.md) -- and every A byte crosses
// the shared-memory port twice more (written by the copy, read by the MMA).  Here
//   * a plan-time pass (tile_plan_kernel) lists, per tile and per kz-group of offsets, the DISTINCT 16-row blocks of x the
//     tile touches and rewrites the neighbour table into 16-bit slot numbers into that list;
//   * two loader warps bring each listed block in with ONE tiled TMA box copy (hardware swizzle) into a slab, up to four
//     offset groups ahead of their use (only the first warp talks to the slab barriers, the second follows it through a
//     named barrier); the tile's slot table arrives by cp.async.bulk, a tile ahead;
//   * the gather warpgroups (thread = output row = TMEM lane; 4 x 32 or 2 x 64 data registers, TsCfg) read their row's
//     neighbour out of the slab (predicated 16-byte ld.shared: a row without a neighbour stays zero registers) and write
//     it with tcgen05.st straight into TENSOR MEMORY, where tcgen05.mma takes its A operand from (the ".ts" form: A in
//     TMEM, lane = row, two bf16 per 32-bit column).  The A tile never exists in shared memory;
//   * B (weights, K-major SWIZZLE_128B) arrives by tiled TMA (resident for the life of the CTA when all K blocks fit in
//     56 KB); accumulators are double-buffered in TMEM and drained by four epilogue warps (bias, optional addend,
//     BatchNorm statistics) while the next tile is multiplied.
// TMEM map (512 columns): [0, 2*COUT) two accumulators, then a ring of 4-6 A slots of 2 x 32 columns (ARing).
// OPT-IN (TODA_TILE_PLANS=1): see ops.py and profiles/r02_conv_ts.md section 5 for the deadlock history of this kernel and
// why every wait uses the plain mbarrier.try_wait.
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"
#include "conv.cuh"
#include "epilogue.cuh"
#include "tcgen05.cuh"

namespace {

constexpr int kTileM = 128;
constexpr int kMaxKvol = 27;
constexpr int kLidxBytes = 7168;                  // >= 27 * 128 * 2, 1024-multiple
constexpr uint32_t kLidxNone = 0xFFFFu;           // no neighbour under this offset
constexpr uint32_t kLidxGlobal = 0xFFFEu;         // neighbour exists but is not in the slab: read it from global memory
// Gather warps: kWGs warpgroups (per instantiation, TsCfg).  What bounds the gather is the number of dependent shared-memory
// round trips per pair -- in the bursts where every gather warp loads at once a round trip costs ~500 cycles (timeline in
// profiles/r02_conv_ts.md) -- and how many pairs are in flight.  Two variants, measured per layer width:
//   * 4 warpgroups x 32 data registers: the two K blocks of a pair go through the same registers one after the other (768
//     threads leave 80 registers per thread);
//   * 2 warpgroups x 64 data registers: both blocks of a pair in flight at once (512 threads, up to 128 registers).
// Same bytes in flight per SM either way; the second is ahead for 256-byte rows, the first for the narrow layers.
// the warp scheduler favours high warp ids: the latency-critical gather warps get them
constexpr int kWarpMma = 4, kWarpLoader = 5, kWarpB = 6, kWarpLoader2 = 7, kWarpGather0 = 8;
// A ring: pair slots of 2 x 32 TMEM columns (2 x 64 K elements) behind the two accumulators
// Pair gp is produced by warpgroup gp % 4 into slot gp % kSlots.  Its barriers are NOT per slot but per pair index modulo
// 16 (a_full / a_empty[gp & 15]): every barrier is then waited on by one warpgroup only, which sees each of its phases in turn
// -- a parity wait by a thread that is two phases behind would pass at once (this hung the kernel when barriers were per slot
// and a warpgroup without work in a few sparse tiles ran ahead).
template <int COUT> struct ARing { static constexpr int kSlots = COUT <= 64 ? 6 : 4; static constexpr int kCol0 = COUT <= 64 ? 128 : 256; };
constexpr int kABars = 16;
constexpr int kPlanWindow = 32768;                // block-id window of the plan kernel's bitmap
constexpr uint32_t kMaxSpins = 1u << 26;          // mbarrier probes before a wait traps (tcgen05.cuh)

// wait of a role that is not on the critical path (epilogue, weight producer): probe, then really sleep -- a spinning warp
// takes issue slots from the gather warp it shares a scheduler with (the epilogue's wait alone was 12 % of all instructions)
__device__ __forceinline__ void mbar_wait_relaxed(uint32_t bar, uint32_t parity) {
    uint32_t done = 0, spins = 0;
    while (true) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (done) break;
        __nanosleep(256);
        if (++spins > kMaxSpins) {
#ifdef TODA_TS_VERBOSE_TIMEOUT
            printf("conv_ts: mbarrier timeout (relaxed) smem=0x%x parity=%u block=%d warp=%d\n", bar, parity, (int)blockIdx.x, (int)(threadIdx.x >> 5));
#endif
            __trap();
        }
    }
}
__device__ __forceinline__ void bulk_copy_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar)
                 : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]: A = 128 lanes x 8 columns (16 bf16 per lane), B = K-major SWIZZLE_128B descriptor
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void lds128(uint32_t addr, uint32_t &a, uint32_t &b, uint32_t &c, uint32_t &d) {
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(addr));
}
// predicated 16-byte load: lanes without a neighbour keep their zeros and take no part in the access (no wavefront, no
// bank conflict with the lanes that do read)
__device__ __forceinline__ void lds128_if(uint32_t addr, uint32_t on, uint32_t &a, uint32_t &b, uint32_t &c, uint32_t &d) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.u32 p, %5, 0;\n\t"
        "@p ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];\n\t}"
        : "+r"(a), "+r"(b), "+r"(c), "+r"(d)
        : "r"(addr), "r"(on));
}
__device__ __forceinline__ uint32_t lds_u16(uint32_t addr) {
    uint16_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(addr));
    return (uint32_t)v;
}

template <int CIN, int COUT> struct TsCfg {
    static constexpr int kWGs = CIN >= 128 ? 2 : 4;            // gather warpgroups
    static constexpr bool kBoth = kWGs == 2;                   // both K blocks of a pair in flight (64 data registers)
    static constexpr int kGatherWarps = 4 * kWGs;
    static constexpr int kThreads = (8 + kGatherWarps) * 32;
    static constexpr int kRowBytes = CIN * 2;
    static constexpr int kRB = kRowBytes < 128 ? kRowBytes : 128;   // bytes of a row inside one swizzled slab half
    static constexpr int kHalves = kRowBytes / kRB;                  // 2 for 256-byte rows (two 128-byte column halves)
    // a slab caches 16-row BLOCKS of x (rows 16 b .. 16 b + 15), each brought in by one TMA box copy
    static constexpr int kCap = CIN == 128 ? 16 : (CIN == 64 ? 20 : 32);   // blocks per slab (<= 32: one loader lane per block)
    static constexpr int kHalfSlab = kCap * 16 * kRB;
    static constexpr int kSlab = kHalfSlab * kHalves;          // 16 / 32 / 40 / 64 KB
    static constexpr int kBStage = COUT * 128;                 // [COUT rows][64 bf16]
    static constexpr int kNkbMax = (kMaxKvol * CIN + 63) / 64;
    // small layers keep ALL their weights in shared memory for the lifetime of the (persistent) CTA: no per-tile re-fetch
    // (at 32->32 the weights were more than half of the L2->SM bytes of a tile)
    static constexpr bool kBRes = kNkbMax * kBStage <= 57344;
    static constexpr int kSB = kBRes ? kNkbMax : (COUT == 128 ? 4 : (COUT == 64 ? 6 : 8));
    static constexpr int kParts = CIN >= 64 ? 1 : 64 / CIN;    // kernel offsets per 64-element K block
    static constexpr int kPV = (CIN >= 64 ? 64 : CIN) / 8;     // 16-byte vectors per part
    // slab buffers (offset groups in flight): as many as fit, up to 4.  With 3 groups per tile and 3 buffers, group 0 of the next
    // tile can only be fetched once every warp has let go of group 0 of this one; a 4th buffer takes that off the critical path.
    static constexpr int kFixed = 1024 + kSB * kBStage + 2 * kLidxBytes + 640 + 256;
    static constexpr int kNB = kFixed + 4 * kSlab <= 232448 ? 4 : (kFixed + 3 * kSlab <= 232448 ? 3 : 2);
    static constexpr int kSmemRaw = kFixed + kNB * kSlab;
    // the kernel allocates all 512 TMEM columns: never let two CTAs share an SM (the second would wait in tcgen05.alloc)
    static constexpr int kSmem = kSmemRaw < 120 * 1024 ? 120 * 1024 : kSmemRaw;
    static_assert(kCap <= 32 && kSlab % 1024 == 0 && kBStage % 1024 == 0, "slab layout");
    static_assert(2 * COUT <= ARing<COUT>::kCol0 && ARing<COUT>::kCol0 + 64 * ARing<COUT>::kSlots <= 512, "TMEM map");
    static constexpr int kBBars = kBRes ? 1 : kSB;             // resident weights arrive on one barrier, once
    static_assert(kBBars <= 14, "barrier area");
    static_assert(!kBRes || kNkbMax <= 32, "the MMA warp peels a 32-bit K-block mask when the weights are resident");
    // TMA swizzle of a slab row (hardware XORs the 16-byte chunk index with address bits 7..9 / 7..8 / 7): chunk q of slot s
    // lives at s * kRB + ((q ^ swz(s)) << 4); eight consecutive slots then hit eight different 16-byte bank groups
    __device__ static __forceinline__ uint32_t swz(uint32_t s) { return kRB == 128 ? (s & 7u) : (kRB == 64 ? ((s >> 1) & 3u) : ((s >> 2) & 1u)); }
};

#define TS_STTM_X32(addr, v)                                                                                                        \
    asm volatile(                                                                                                                   \
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,"     \
        "%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"                                                                         \
        ::"r"(addr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),  \
          "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]),   \
          "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]),   \
          "r"(v[30]), "r"(v[31])                                                                                                    \
        : "memory")

// Roles: warps 0-3 epilogue, 4 MMA issuer, 5 + 7 slab loaders, 6 weight producer, 8.. gather (TsCfg::kWGs warpgroups,
// thread = tile row = TMEM lane).
template <int CIN, int COUT>
__global__ void __launch_bounds__((TsCfg<CIN, COUT>::kThreads), 1) conv_ts_fwd_kernel(const __nv_bfloat16 *__restrict__ xb, const int *__restrict__ nbr,
                                                                  int n_out, int kvol, const uint16_t *__restrict__ lidx,
                                                                  const int *__restrict__ prow, const int *__restrict__ pcnt,
                                                                  int ngroups, int cap,
                                                                  const __grid_constant__ CUtensorMap map_x /*[n_in][CIN] bf16, box 16 rows*/,
                                                                  const __grid_constant__ CUtensorMap map_w /*[COUT][kvol*CIN] bf16*/,
                                                                  const float *__restrict__ bias, const float *__restrict__ addend,
                                                                  float *__restrict__ y, const int *__restrict__ out_rows,
                                                                  const uint32_t *__restrict__ tile_masks,
                                                                  double *__restrict__ bn_sums, int num_tiles) {
    using C = TsCfg<CIN, COUT>;
    constexpr int NB = C::kNB, SB = C::kSB, PARTS = C::kParts, PV = C::kPV;
    constexpr bool BRES = C::kBRes;
    constexpr int kASlots = ARing<COUT>::kSlots, kACol0 = ARing<COUT>::kCol0;
    extern __shared__ uint8_t smem_raw[];
    uint32_t raw;     // (volatile: the compiler otherwise re-derives the shared window base from SR_CgaCtaId at every use)
    asm volatile("mov.u32 %0, %1;" : "=r"(raw) : "r"(smem_u32(smem_raw)));
    const uint32_t base = (raw + 1023u) & ~1023u;          // B stages: SWIZZLE_128B tiles need 1024-byte alignment
    const uint32_t slab_base = base + SB * C::kBStage;
    const uint32_t lidx_base = slab_base + NB * C::kSlab;
    const uint32_t bar_base = lidx_base + 2 * kLidxBytes;
    const uint32_t a_full = bar_base, a_empty = bar_base + 128;              // 16 + 16
    const uint32_t b_full = bar_base + 256, b_empty = bar_base + 368;         // 14 + 14
    const uint32_t acc_full = bar_base + 480, acc_empty = bar_base + 496;     // 2 + 2
    const uint32_t slab_full = bar_base + 512, slab_empty = bar_base + 544;   // 4 + 4
    const uint32_t lidx_full = bar_base + 576, lidx_empty = bar_base + 592;   // 2 + 2
    const uint32_t tmem_slot = bar_base + 608;
    const uint32_t zero_base = bar_base + 640;               // 256 zero bytes: the row read for a missing neighbour
    volatile uint32_t *tmem_slot_ptr = (volatile uint32_t *)(smem_raw + (tmem_slot - raw));

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nkb = (kvol * CIN + 63) / 64;                // 64-element K blocks
    const int gs = kvol / ngroups, gs2 = 2 * gs;           // offsets per group; group of offset k = (k >= gs) + (k >= 2 gs)
    // K blocks of tile t that hold at least one real neighbour (bit c = K block c); every role derives the same list.
    // A tile without any neighbour still walks block 0 (all-zero rows) so that its accumulator is defined.
    // (the offset mask of the NEXT tile is fetched while the current tile is processed: load_om / kb_mask_from)
    auto load_om = [&](int t) -> uint32_t { return (tile_masks && t < num_tiles) ? __ldg(tile_masks + t) : 0xffffffffu; };
    // (warp-collective: lane c tests K block c (and c + 32), two ballots give the mask -- the 14..54-iteration scalar loop this
    // replaces sat on every role's critical path at each tile start)
    auto kb_mask_from = [&](uint32_t om) -> unsigned long long {
        if (!tile_masks) return nkb >= 64 ? ~0ull : ((1ull << nkb) - 1ull);
        const int c0 = lane, c1 = lane + 32;
        bool b0, b1;
        if (CIN <= 64) {
            b0 = c0 < nkb && ((om >> (c0 * PARTS)) & ((1u << PARTS) - 1u)) != 0u;
            b1 = false;
        } else {
            b0 = c0 < nkb && ((om >> (c0 >> 1)) & 1u) != 0u;
            b1 = c1 < nkb && ((om >> (c1 >> 1)) & 1u) != 0u;
        }
        const unsigned lo = __ballot_sync(0xffffffffu, b0);
        const unsigned hi = CIN <= 64 ? 0u : __ballot_sync(0xffffffffu, b1);
        const unsigned long long cm = (unsigned long long)lo | ((unsigned long long)hi << 32);
        return cm ? cm : 1ull;
    };
    auto kb_mask_of = [&](int t) -> unsigned long long { return kb_mask_from(load_om(t)); };
    // Active K blocks as a list held across the warp: lane r keeps the K block of rank r (and r + 32 when a tile can have more
    // than 32 K blocks).  The roles used to peel the mask bit by bit -- ~42 instructions of 64-bit arithmetic per pair, run by
    // every gather warp for all the pairs it skips as well: 18 % of all instructions the kernel issued and most of the gather
    // warps' latency per pair (ncu source view, profiles/r02_conv_ts.md).  Now a pair costs two shuffles.
    auto kb_list = [&](unsigned long long cm, int &p0, int &p1) {
        const uint32_t lo = (uint32_t)cm, hi = (uint32_t)(cm >> 32);
        const int nlo = __popc(lo);
        p0 = lane < nlo ? (int)__fns(lo, 0, lane + 1) : -1;
        p1 = -1;
        if (CIN > 64) {
            const int nhi = __popc(hi);
            if (lane >= nlo && lane - nlo < nhi) p0 = 32 + (int)__fns(hi, 0, lane - nlo + 1);
            const int r1 = lane + 32 - nlo;
            if (r1 >= 0 && r1 < nhi) p1 = 32 + (int)__fns(hi, 0, r1 + 1);
        }
    };
    auto kb_at = [&](int p0, int p1, int rank) -> int {
        if (CIN > 64) {
            const int a = __shfl_sync(0xffffffffu, p0, rank & 31), b = __shfl_sync(0xffffffffu, p1, rank & 31);
            return rank < 32 ? a : b;
        }
        return __shfl_sync(0xffffffffu, p0, rank);
    };

    if (tid == 0) {
        for (int s = 0; s < kABars; ++s) {
            mbar_init(a_full + 8 * s, 4);          // the four warps of the gathering warpgroup
            mbar_init(a_empty + 8 * s, 1);         // tcgen05.commit
        }
        for (int s = 0; s < C::kBBars; ++s) {
            mbar_init(b_full + 8 * s, 1);          // arrive.expect_tx; the TMA completes the bytes
            mbar_init(b_empty + 8 * s, 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(acc_full + 8 * b, 1);
            mbar_init(acc_empty + 8 * b, 4);       // the four epilogue warps
            mbar_init(lidx_full + 8 * b, 1);
            mbar_init(lidx_empty + 8 * b, C::kGatherWarps);
        }
        for (int b = 0; b < NB; ++b) {
            mbar_init(slab_full + 8 * b, 1);       // arrive.expect_tx by the first loader warp; the TMA box copies complete the bytes
            mbar_init(slab_empty + 8 * b, C::kGatherWarps);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == kWarpMma) tmem_alloc<512>(tmem_slot);
    if (warp == kWarpB && lane == 0) asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w) : "memory");
    if (tid < 16) asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(zero_base + tid * 16), "r"(0u) : "memory");
    if (warp == kWarpLoader && lane == 0) asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot_ptr;

    if (warp >= kWarpGather0) {
        // ------------------------------------------------------------------ gather warps: thread = tile row = TMEM lane
        // The active K blocks of a tile are dealt out in pairs, pair gp to warpgroup gp % 4.  A pair costs one round of barrier
        // waits / tcgen05.wait::st / arrivals and keeps 2 x 128 bytes per thread in flight.  This loop is instruction-latency
        // bound (the warps share four schedulers at ~57 % issue utilisation, profiles/r02_conv_ts.md), so everything that does
        // not depend on the pair is computed once per tile: unsigned arithmetic only, no division by the ring sizes, barrier
        // addresses and phases of the tile's slabs kept in registers.
        const uint32_t wg = (uint32_t)(warp - kWarpGather0) >> 2;
        const uint32_t row = (uint32_t)(warp & 3) * 32u + (uint32_t)lane;
        const uint32_t t_lane = tmem_base + (((uint32_t)(warp & 3) * 32u) << 16) + kACol0;
        const uint32_t ugs = (uint32_t)gs, ugs2 = (uint32_t)gs2, ukvol = (uint32_t)kvol;
        uint32_t gpbase = 0, it = 0;                    // global index of this tile's first pair
        uint32_t uq = 0, ur = 0;                        // the tile's first (tile, group) unit is number uq * NB + ur of this CTA
        uint32_t om_next = load_om(blockIdx.x);
        for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
            const uint32_t ib = it & 1u;
            const uint32_t om = om_next;
            om_next = load_om(t + gridDim.x);
            mbar_wait<kMaxSpins>(lidx_full + 8 * ib, (it >> 1) & 1u);
            const uint32_t lidx_tile = lidx_base + ib * kLidxBytes + 2u * row;
            // slab buffer, barrier offset and phase parity of the tile's (up to three) offset groups
            uint32_t sbuf[3], sbar[3], spar[3];
#pragma unroll
            for (int g = 0; g < 3; ++g) {
                uint32_t r = ur + (uint32_t)g;
                const uint32_t wrap = r >= (uint32_t)NB ? 1u : 0u;
                r -= wrap * (uint32_t)NB;
                sbuf[g] = slab_base + r * (uint32_t)C::kSlab;
                sbar[g] = 8u * r;
                spar[g] = (uq + wrap) & 1u;
            }
            uint32_t gwait = 0, gdone = 0;              // groups of this tile whose slab this warp has waited for / released
            auto wait_group = [&](uint32_t grp) {       // the slabs of groups 0..grp have landed
                if (gwait > grp) return;
#pragma unroll
                for (int g = 0; g < 3; ++g)
                    if ((uint32_t)g >= gwait && (uint32_t)g <= grp) mbar_wait<kMaxSpins>(slab_full + sbar[g], spar[g]);
                gwait = grp + 1u;
            };
            auto release_below = [&](uint32_t grp_end) {
                // (a warp waits for a slab before releasing it even if it never read it: its arrival must not land in
                // the barrier phase of the slab's previous use.  One group at a time: with fewer buffers than groups the
                // slab of a later group is only fetched once an earlier one has been handed back.)
                if (gdone >= grp_end) return;
#pragma unroll
                for (int g = 0; g < 3; ++g)
                    if ((uint32_t)g >= gdone && (uint32_t)g < grp_end) {
                        if ((uint32_t)g >= gwait) {
                            mbar_wait<kMaxSpins>(slab_full + sbar[g], spar[g]);
                            gwait = (uint32_t)g + 1u;
                        }
                        __syncwarp();
                        if (lane == 0) mbar_arrive(slab_empty + sbar[g]);
                    }
                gdone = grp_end;
            };
            // Branch-free fast path: the table entries of both blocks of a pair are fetched first (load_li), then every
            // 16-byte piece of both blocks by predicated loads (load_data): a row without a neighbour keeps zero registers and
            // issues no shared-memory access -- 44 % of the entries of a stride-1 table are empty.  load_data returns true if
            // some entry must be read from global memory instead (fix_block).
            auto load_li = [&](uint32_t kb, bool on, uint32_t (&li)[PARTS]) {
#pragma unroll
                for (int part = 0; part < PARTS; ++part) {
                    const uint32_t k = CIN == 128 ? (kb >> 1) : kb * PARTS + part;
                    li[part] = kLidxNone;
                    if (on && (PARTS == 1 || k < ukvol)) li[part] = lds_u16(lidx_tile + k * (kTileM * 2));
                }
            };
            auto load_data = [&](uint32_t kb, const uint32_t (&li)[PARTS], uint32_t (&v)[32]) -> bool {
                bool fix = false;
#pragma unroll
                for (int part = 0; part < PARTS; ++part) {
                    const uint32_t k = CIN == 128 ? (kb >> 1) : kb * PARTS + part;
                    const uint32_t sl = li[part];
                    const bool hit = sl < kLidxGlobal;
                    uint32_t buf = k >= ugs2 ? sbuf[2] : (k >= ugs ? sbuf[1] : sbuf[0]);
                    if (CIN == 128) buf += (kb & 1u) * (uint32_t)C::kHalfSlab;
                    // chunk q of slot s lives at s * kRB + ((q ^ swz(s)) << 4); the row start is kRB-aligned, so the swizzle
                    // is one XOR of the row address per 16-byte piece
                    const uint32_t src = buf + sl * (uint32_t)C::kRB + (C::swz(sl) << 4);
                    const uint32_t on = hit ? 1u : 0u;
#pragma unroll
                    for (int q = 0; q < PV; ++q) {
                        uint32_t &r0 = v[(part * PV + q) * 4], &r1 = v[(part * PV + q) * 4 + 1], &r2 = v[(part * PV + q) * 4 + 2],
                                 &r3 = v[(part * PV + q) * 4 + 3];
                        r0 = r1 = r2 = r3 = 0u;
                        lds128_if(src ^ ((uint32_t)q << 4), on, r0, r1, r2, r3);
                    }
                    fix |= sl == kLidxGlobal;
                }
                return fix;
            };
            auto fix_block = [&](uint32_t kb, const uint32_t (&li)[PARTS], uint32_t (&v)[32]) {
#pragma unroll
                for (int part = 0; part < PARTS; ++part) {
                    const uint32_t k = CIN == 128 ? (kb >> 1) : kb * PARTS + part;
                    const uint32_t half = CIN == 128 ? (kb & 1u) * 128u : 0u;
                    if (li[part] == kLidxGlobal) {
                        const int gi = __ldg(nbr + (size_t)k * n_out + (size_t)t * kTileM + row);
                        const uint4 *src = (const uint4 *)((const char *)xb + (size_t)gi * C::kRowBytes + half);
#pragma unroll
                        for (int q = 0; q < PV; ++q) {
                            const uint4 r = __ldg(src + q);
                            v[(part * PV + q) * 4] = r.x; v[(part * PV + q) * 4 + 1] = r.y;
                            v[(part * PV + q) * 4 + 2] = r.z; v[(part * PV + q) * 4 + 3] = r.w;
                        }
                    }
                }
            };
            const unsigned long long cm = kb_mask_from(om);
            const uint32_t nact = (uint32_t)__popcll(cm), npairs = (nact + 1u) >> 1;
            int kl0, kl1;
            kb_list(cm, kl0, kl1);
            // this warpgroup's pairs of the tile: global pair index gp = gpbase + pj with gp % kWGs == wg (kWGs is 2 or 4)
            for (uint32_t pj = (wg - gpbase) & (uint32_t)(C::kWGs - 1); pj < npairs; pj += (uint32_t)C::kWGs) {
                const uint32_t kbA = (uint32_t)kb_at(kl0, kl1, (int)(2u * pj));
                const uint32_t kbB = (uint32_t)kb_at(kl0, kl1, (int)((2u * pj + 1u) & 63u));
                const bool two = 2u * pj + 1u < nact;
                const uint32_t gp = gpbase + pj;        // global pair index: A slot gp % kASlots (two 32-column blocks)
                const uint32_t aslot = gp % (uint32_t)kASlots;
                uint32_t liA[PARTS], liB[PARTS];
                load_li(kbA, true, liA);
                load_li(kbB, two, liB);
                const uint32_t k_first = CIN == 128 ? (kbA >> 1) : kbA * PARTS;
                const uint32_t g_first = (k_first >= ugs ? 1u : 0u) + (k_first >= ugs2 ? 1u : 0u);
                const uint32_t kb_last = two ? kbB : kbA;
                const uint32_t k_last = min(CIN == 128 ? (kb_last >> 1) : kb_last * PARTS + PARTS - 1, ukvol - 1u);
                const uint32_t g_last = (k_last >= ugs ? 1u : 0u) + (k_last >= ugs2 ? 1u : 0u);
                release_below(g_first);                 // slabs of earlier groups are no longer read by this warp
                // With two slab buffers (256-byte rows) groups 0 and 2 of a tile share a buffer: a pair whose blocks lie in
                // those two groups (group 1 fully masked out) cannot have both resident -- it is walked one block at a time,
                // the first group handed back in between.  (Waiting for both deadlocked the CTA on such a tile.)
                const bool apart = NB < 3 && g_last >= g_first + (uint32_t)NB;
                wait_group(apart ? g_first : g_last);
                // (the A slot is waited for while the loads are in flight: the barrier probe overlaps them)
                uint32_t va[32];
                bool fixA = load_data(kbA, liA, va);
                if (C::kBoth && !apart) {
                    uint32_t vb[32];
                    bool fixB = load_data(kbB, liB, vb);
                    if (gp >= (uint32_t)kASlots) {      // the pair that used this slot before (gp - kASlots) has been consumed
                        const uint32_t pg = gp - (uint32_t)kASlots;
                        mbar_wait<kMaxSpins>(a_empty + 8u * (pg & (kABars - 1)), (pg / kABars) & 1u);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    }
                    if (__any_sync(0xffffffffu, fixA || fixB)) {
                        fix_block(kbA, liA, va);
                        fix_block(kbB, liB, vb);
                    }
                    __syncwarp();
                    TS_STTM_X32(t_lane + aslot * 64u, va);
                    if (two) TS_STTM_X32(t_lane + aslot * 64u + 32u, vb);
                } else {
                    if (gp >= (uint32_t)kASlots) {
                        const uint32_t pg = gp - (uint32_t)kASlots;
                        mbar_wait<kMaxSpins>(a_empty + 8u * (pg & (kABars - 1)), (pg / kABars) & 1u);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    }
                    if (__any_sync(0xffffffffu, fixA)) fix_block(kbA, liA, va);
                    __syncwarp();
                    TS_STTM_X32(t_lane + aslot * 64u, va);
                    if (two) {                          // (the table entries of block B were fetched with those of block A)
                        if (apart) {
                            release_below(g_last);
                            wait_group(g_last);
                        }
                        fixA = load_data(kbB, liB, va);
                        if (__any_sync(0xffffffffu, fixA)) fix_block(kbB, liB, va);
                        __syncwarp();
                        TS_STTM_X32(t_lane + aslot * 64u + 32u, va);
                    }
                }
                asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(a_full + 8u * (gp & (kABars - 1)));
            }
            gpbase += npairs;
            release_below((uint32_t)ngroups);
            ur += (uint32_t)ngroups;
            while (ur >= (uint32_t)NB) { ur -= (uint32_t)NB; ++uq; }
            __syncwarp();
            if (lane == 0) mbar_arrive(lidx_empty + 8 * ib);
        }
    } else if (warp < kWarpMma) {
        // ------------------------------------------------------------------ epilogue (warps 0..3)
        const int q = warp & 3;                                  // TMEM lane quarter this warp may access
        float acc_s[COUT / 16], acc_q[COUT / 16];                // running per-channel sum / sum of squares (BatchNorm)
#pragma unroll
        for (int i = 0; i < COUT / 16; ++i) acc_s[i] = acc_q[i] = 0.f;
        int it = 0;
        for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
            const int ab = it & 1;
            mbar_wait_relaxed(acc_full + 8 * ab, (it >> 1) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const int row = t * kTileM + q * 32 + lane;          // TMEM lane = tile row
            drain_accumulator<COUT>(tmem_base + ((uint32_t)(q * 32) << 16), ab, row, n_out, out_rows, bias, addend, y, bn_sums, acc_s,
                                    acc_q, lane);
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(acc_empty + 8 * ab);
        }
        flush_bn_sums<COUT>(bn_sums, acc_s, acc_q, lane);
    } else if (warp == kWarpMma) {
        // ------------------------------------------------------------------ MMA issuer.  The single issuing thread is the serial
        // resource of the kernel (a tcgen05.mma costs ~45 cycles of issue whatever its N: scripts/ubench/commit_lat.cu), so the
        // loop around it is kept minimal: ONE full-barrier per pair of K blocks, warp-uniform waits, 8 MMAs + 1-2 commits.
        constexpr uint32_t idesc = make_idesc_bf16(kTileM, COUT);
        if (BRES) mbar_wait<kMaxSpins>(b_full, 0);
        int gbase = 0, gp = 0, it = 0;
        uint32_t om_next = load_om(blockIdx.x);
        for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
            const int ab = it & 1, ause = it >> 1;
            const uint32_t om = om_next;
            om_next = load_om(t + gridDim.x);
            if (ause > 0) mbar_wait<kMaxSpins>(acc_empty + 8 * ab, (ause - 1) & 1);   // epilogue has drained this accumulator
            const uint32_t d_tmem = tmem_base + ab * COUT;
            uint32_t accumulate = 0;
            const unsigned long long cm = kb_mask_from(om);
            const int nact = __popcll(cm), npairs = (nact + 1) >> 1;
            // resident weights are addressed by K block (at most 14 of them: a 32-bit mask peeled with two instructions per
            // block), streamed ones by ring position.  No shuffles here: they queue behind the gather warps' shared-memory loads.
            uint32_t m32 = (uint32_t)cm;
            for (int pj = 0; pj < npairs; ++pj) {
                const int gA = gbase + 2 * pj;
                const int n = 2 * pj + 1 < nact ? 2 : 1;
                int kbA = 0, kbB = 0;
                if (BRES) {
                    kbA = __ffs((int)m32) - 1;
                    m32 &= m32 - 1u;
                    kbB = __ffs((int)m32) - 1;
                    m32 &= m32 - 1u;
                }
                const int aslot = gp % kASlots;
                mbar_wait<kMaxSpins>(a_full + 8 * (gp & (kABars - 1)), (gp / kABars) & 1);
                if (!BRES) {
                    mbar_wait<kMaxSpins>(b_full + 8 * (gA % SB), (gA / SB) & 1);
                    if (n == 2) mbar_wait<kMaxSpins>(b_full + 8 * ((gA + 1) % SB), ((gA + 1) / SB) & 1);
                }
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                if (elect_one()) {
#pragma unroll
                    for (int i = 0; i < 2; ++i) {
                        if (i < n) {
                            const int g = gA + i, kb = i ? kbB : kbA;
                            const int stage = BRES ? kb : g % SB;
                            const uint64_t bd0 = make_desc_k_sw128(base + stage * C::kBStage);
                            const uint32_t a0 = tmem_base + kACol0 + aslot * 64 + i * 32;
                            umma_bf16_ts(d_tmem, a0, bd0, idesc, accumulate);
#pragma unroll
                            for (int jj = 1; jj < 4; ++jj) umma_bf16_ts(d_tmem, a0 + 8 * jj, bd0 + 2 * jj, idesc, 1u);   // K = 16: 8 columns / 32 bytes
                            accumulate = 1u;
                            if (!BRES) umma_commit(b_empty + 8 * stage);
                        }
                    }
                    umma_commit(a_empty + 8 * (gp & (kABars - 1)));
                }
                accumulate = 1u;
                __syncwarp();
                ++gp;
            }
            gbase += nact;
            if (elect_one()) umma_commit(acc_full + 8 * ab);
            __syncwarp();
        }
    } else if (warp == kWarpLoader || warp == kWarpLoader2) {
        // ------------------------------------------------------------------ loaders (two warps: even / odd blocks; issuing a TMA costs
        // ~65 cycles): table slice + row slabs, up to NB groups ahead.
        // One TMA box copy (16 rows, hardware-swizzled) per cached block, lane i issuing block i of the unit.  The block list of
        // unit u+1 is fetched while unit u is issued (a list read is two dependent L2 round trips).
        const int L = warp == kWarpLoader ? 0 : 1;
        int bid_n = -1, nb_n = 0;
        auto fetch_unit = [&](int t, int grp) {
            if (t < num_tiles) {
                nb_n = __ldg(pcnt + (size_t)t * ngroups + grp);
                bid_n = lane < nb_n ? __ldg(prow + ((size_t)t * ngroups + grp) * cap + lane) : -1;
            }
        };
        fetch_unit(blockIdx.x, 0);
        int it = 0;
        for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
            const int ib = it & 1;
            if (L == 0 && lane == 0) {
                if (it >= 2) mbar_wait<kMaxSpins>(lidx_empty + 8 * ib, ((it >> 1) - 1) & 1);
                const uint32_t bytes = (uint32_t)kvol * (kTileM * 2);
                mbar_arrive_expect_tx(lidx_full + 8 * ib, bytes);
                bulk_copy_g2s(lidx_base + ib * kLidxBytes, lidx + (size_t)t * kvol * kTileM, bytes, lidx_full + 8 * ib);
            }
            __syncwarp();
            for (int grp = 0; grp < ngroups; ++grp) {
                const int u = it * ngroups + grp, buf = u % NB, use = u / NB;
                const int bid = bid_n, nb = nb_n;
                if (grp + 1 < ngroups) fetch_unit(t, grp + 1);
                else fetch_unit(t + gridDim.x, 0);
                // Only the first loader warp talks to the slab barriers; the second follows it unit by unit through a named
                // hardware barrier.  (When both warps waited on slab_empty themselves, a unit in which the second warp had no
                // block to fetch completed without it; that warp could then fall two uses of a buffer behind, where its
                // parity wait never passes again: a deadlock seen a few times in ten runs on one rank's frames.)
                if (L == 0) {
                    if (use > 0) mbar_wait<kMaxSpins>(slab_empty + 8 * buf, (use - 1) & 1);
                    if (lane == 0) {
                        if (nb > 0) mbar_arrive_expect_tx(slab_full + 8 * buf, (uint32_t)nb * 16u * C::kRowBytes);
                        else mbar_arrive(slab_full + 8 * buf);
                    }
                }
                __syncwarp();
                asm volatile("barrier.sync 1, 64;" ::: "memory");
                if (bid >= 0 && (lane & 1) == L) {
                    const uint32_t dst = slab_base + buf * C::kSlab + lane * (16 * C::kRB);
#pragma unroll
                    for (int h = 0; h < C::kHalves; ++h)
                        tma_load_2d(dst + h * C::kHalfSlab, &map_x, h * 64, bid * 16, slab_full + 8 * buf);
                }
            }
        }
    } else if (warp == kWarpB) {
        // ------------------------------------------------------------------ weight producer (the warp walks the tiles together: the
        // K-block mask is a warp-collective; lane 0 issues the TMA copies)
        if (BRES) {
            if (lane == 0) {
                // every K block once, resident for the lifetime of the CTA
                mbar_arrive_expect_tx(b_full, (uint32_t)nkb * C::kBStage);
                for (int kb = 0; kb < nkb; ++kb) tma_load_2d(base + kb * C::kBStage, &map_w, kb * 64, 0, b_full);
            }
        } else {
            int g = 0;
            for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
                const unsigned long long cm0 = kb_mask_of(t);
                if (lane == 0) {
                    int gg = g;
                    for (unsigned long long cm = cm0; cm; cm &= cm - 1, ++gg) {
                        const int kb = __ffsll((long long)cm) - 1;
                        const int stage = gg % SB, use = gg / SB;
                        if (use > 0) mbar_wait_relaxed(b_empty + 8 * stage, (use - 1) & 1);
                        mbar_arrive_expect_tx(b_full + 8 * stage, C::kBStage);
                        tma_load_2d(base + stage * C::kBStage, &map_w, kb * 64, 0, b_full + 8 * stage);
                    }
                }
                g += __popcll(cm0);
                __syncwarp();
            }
        }
    }
    __syncthreads();
    if (warp == kWarpMma) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        tmem_dealloc<512>(tmem_base);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Plan: one CTA (128 threads = the tile's rows) per (tile, offset group).  The cache unit is a BLOCK of 16 consecutive rows
// of x (one TMA box).  The distinct blocks the group touches are found with a shared-memory bitmap over the window
// [min block, min block + 32768): set bits, prefix popcount = slot of every block in ascending order; a table entry
// becomes 16 * block slot + (row & 15).  Rows outside the window or beyond the slab capacity are flagged kLidxGlobal and
// read from global memory by the conv kernel.  Deterministic.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kPlanWords = kPlanWindow / 32;       // 1024
__global__ void __launch_bounds__(128) tile_plan_kernel(const int *__restrict__ nbr, int n_out, int kvol, int ngroups, int cap,
                                                        uint16_t *__restrict__ lidx, int *__restrict__ prow, int *__restrict__ pcnt) {
    __shared__ uint32_t bits[kPlanWords];
    __shared__ uint16_t pref[kPlanWords];
    __shared__ int red[4];
    __shared__ int wsum[4];
    const int tile = blockIdx.x / ngroups, grp = blockIdx.x % ngroups;
    const int gs = kvol / ngroups;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int row = tile * kTileM + tid;
    int v[9];
    int mn = 0x7fffffff;
#pragma unroll
    for (int j = 0; j < 9; ++j) {
        v[j] = -1;
        if (j < gs && row < n_out) v[j] = __ldg(nbr + (size_t)(grp * gs + j) * n_out + row);
        if (v[j] >= 0) mn = min(mn, v[j] >> 4);
    }
    for (int w = tid; w < kPlanWords; w += 128) bits[w] = 0u;
    for (int o = 16; o; o >>= 1) mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    if (lane == 0) red[warp] = mn;
    __syncthreads();
    const int base = min(min(red[0], red[1]), min(red[2], red[3]));
#pragma unroll
    for (int j = 0; j < 9; ++j) {
        if (v[j] >= 0) {
            const unsigned d = (unsigned)((v[j] >> 4) - base);
            if (d < (unsigned)kPlanWindow) atomicOr(&bits[d >> 5], 1u << (d & 31));
        }
    }
    __syncthreads();
    // exclusive prefix of popcounts over the 1024 words: 8 consecutive words per thread
    int cnt8[8], s = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        cnt8[j] = s;
        s += __popc(bits[tid * 8 + j]);
    }
    int incl = s;
    for (int o = 1; o < 32; o <<= 1) {
        const int nb = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += nb;
    }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    int woff = 0;
    for (int w = 0; w < warp; ++w) woff += wsum[w];
    const int excl = woff + incl - s;
    const int total = wsum[0] + wsum[1] + wsum[2] + wsum[3];
#pragma unroll
    for (int j = 0; j < 8; ++j) pref[tid * 8 + j] = (uint16_t)min(excl + cnt8[j], 0xFFFF);
    // the row list: every set bit, in ascending order
    int *rows = prow + ((size_t)tile * ngroups + grp) * cap;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        uint32_t wbits = bits[tid * 8 + j];
        int slot = excl + cnt8[j];
        while (wbits) {
            const int b = __ffs(wbits) - 1;
            wbits &= wbits - 1;
            if (slot < cap) rows[slot] = base + (tid * 8 + j) * 32 + b;
            ++slot;
        }
    }
    if (tid == 0) pcnt[(size_t)tile * ngroups + grp] = min(total, cap);
    __syncthreads();
    uint16_t *lt = lidx + ((size_t)tile * kvol + (size_t)grp * gs) * kTileM + tid;
#pragma unroll
    for (int j = 0; j < 9; ++j) {
        if (j < gs) {
            uint32_t li = kLidxNone;
            if (v[j] >= 0) {
                const unsigned d = (unsigned)((v[j] >> 4) - base);
                li = kLidxGlobal;
                if (d < (unsigned)kPlanWindow) {
                    const int slot = (int)pref[d >> 5] + __popc(bits[d >> 5] & ((1u << (d & 31)) - 1u));
                    if (slot < cap) li = (uint32_t)(slot * 16 + (v[j] & 15));
                }
            }
            lt[(size_t)j * kTileM] = (uint16_t)li;
        }
    }
}

template <int CIN, int COUT>
int launch_ts(const __nv_bfloat16 *xb, int n_in, const int32_t *nbr, int n_out, int kvol, const TilePlan &plan, const __nv_bfloat16 *wb,
              const float *bias, const float *addend, float *y, const int32_t *out_rows, const uint32_t *tile_masks, double *bn_sums,
              cudaStream_t st) {
    using C = TsCfg<CIN, COUT>;
    if (plan.cap > C::kCap) {
        toda_set_error("conv_ts_fwd: plan capacity %d exceeds the slab capacity %d of Cin=%d", plan.cap, C::kCap, CIN);
        return TODA_ERR_INVALID;
    }
    CUtensorMap map_w, map_x;
    if (int rc = make_tensor_map_bf16(&map_w, wb, (uint64_t)COUT, (uint64_t)kvol * CIN, (uint32_t)COUT, 64)) return rc;
    if (int rc = make_tensor_map_bf16(&map_x, xb, (uint64_t)n_in, (uint64_t)CIN, 16u, (uint32_t)(CIN < 64 ? CIN : 64))) return rc;
    const int num_tiles = ceil_div(n_out, kTileM);
    const int grid = num_tiles < kNumSMs ? num_tiles : kNumSMs;
    static bool attr_set = false;      // per <CIN, COUT> instantiation
    if (!attr_set) {
        TODA_CUDA_OK(cudaFuncSetAttribute(conv_ts_fwd_kernel<CIN, COUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::kSmem));
        attr_set = true;
    }
    conv_ts_fwd_kernel<CIN, COUT><<<grid, C::kThreads, C::kSmem, st>>>(xb, nbr, n_out, kvol, plan.lidx, plan.rows, plan.cnt, plan.ngroups,
                                                                   plan.cap, map_x, map_w, bias, addend, y, out_rows, tile_masks, bn_sums,
                                                                   num_tiles);
    TODA_LAUNCH_OK();
    return TODA_OK;
}

}  // namespace

int conv_ts_slab_capacity(int cin) {
    switch (pad16(cin)) {
        case 16: return TsCfg<16, 16>::kCap;
        case 32: return TsCfg<32, 32>::kCap;
        case 64: return TsCfg<64, 64>::kCap;
        case 128: return TsCfg<128, 128>::kCap;
    }
    return 0;
}

bool conv_ts_supported(int cin, int cout, int kvol, const TilePlan *plan) {
    if (!plan || !plan->lidx || !plan->rows || !plan->cnt) return false;
    if (plan->ngroups < 1 || plan->ngroups > 3 || kvol % plan->ngroups != 0 || kvol / plan->ngroups > 9 || kvol > kMaxKvol) return false;
    const int cp = pad16(cin);
    if (!(cp == 16 || cp == 32 || cp == 64 || cp == 128)) return false;
    if (!(cout == 16 || cout == 32 || cout == 64 || cout == 128)) return false;
    return plan->cap >= 1 && plan->cap <= conv_ts_slab_capacity(cp);
}

// xb: bf16 [n_in][cin], wb: bf16 [cout][kvol*cin]; cin, cout in {16,32,64,128}
int conv_ts_fwd(const void *xb, int n_in, int cin, const int32_t *nbr, int n_out, int kvol, const TilePlan &plan, const void *wb,
                int cout, const float *bias, const float *addend, float *y, const int32_t *out_rows, const uint32_t *tile_masks,
                double *bn_sums, cudaStream_t st) {
    const __nv_bfloat16 *x = (const __nv_bfloat16 *)xb, *w = (const __nv_bfloat16 *)wb;
#define CASE_CO(CI)                                                                                                          \
    switch (cout) {                                                                                                          \
        case 16: return launch_ts<CI, 16>(x, n_in, nbr, n_out, kvol, plan, w, bias, addend, y, out_rows, tile_masks, bn_sums, st);   \
        case 32: return launch_ts<CI, 32>(x, n_in, nbr, n_out, kvol, plan, w, bias, addend, y, out_rows, tile_masks, bn_sums, st);   \
        case 64: return launch_ts<CI, 64>(x, n_in, nbr, n_out, kvol, plan, w, bias, addend, y, out_rows, tile_masks, bn_sums, st);   \
        case 128: return launch_ts<CI, 128>(x, n_in, nbr, n_out, kvol, plan, w, bias, addend, y, out_rows, tile_masks, bn_sums, st); \
    }                                                                                                                        \
    break;
    switch (cin) {
        case 16: CASE_CO(16)
        case 32: CASE_CO(32)
        case 64: CASE_CO(64)
        case 128: CASE_CO(128)
    }
#undef CASE_CO
    toda_set_error("conv_ts_fwd: unsupported cin=%d cout=%d", cin, cout);
    return TODA_ERR_UNSUPPORTED;
}

extern "C" int toda_tile_plan_capacity(int channels) { return conv_ts_slab_capacity(channels); }

extern "C" int toda_table_tile_plan(const int32_t *nbr, int n_out, int kvol, int ngroups, int cap, uint16_t *lidx, int32_t *rows,
                                    int32_t *cnt, void *stream) {
    TODA_CHECK_ARG(n_out >= 0 && kvol > 0 && kvol <= kMaxKvol, "table_tile_plan: bad sizes n_out=%d kvol=%d", n_out, kvol);
    TODA_CHECK_ARG(ngroups >= 1 && ngroups <= 3 && kvol % ngroups == 0 && kvol / ngroups <= 9, "table_tile_plan: bad groups %d", ngroups);
    TODA_CHECK_ARG(cap >= 1 && cap <= 32, "table_tile_plan: bad capacity %d", cap);
    if (n_out == 0) return TODA_OK;
    TODA_CHECK_ARG(nbr && lidx && rows && cnt, "table_tile_plan: null pointer");
    const int num_tiles = ceil_div(n_out, kTileM);
    tile_plan_kernel<<<num_tiles * ngroups, 128, 0, (cudaStream_t)stream>>>(nbr, n_out, kvol, ngroups, cap, lidx, rows, cnt);
    TODA_LAUNCH_OK();
    return TODA_OK;
}
