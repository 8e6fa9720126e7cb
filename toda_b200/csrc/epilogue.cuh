// Accumulator epilogue of the tcgen05 forward / dgrad kernels (conv_tc.cu, conv_tma.cu, conv_ts.cu): TMEM -> + bias
// (+ addend) -> fp32 rows of y, and the per-channel sums of those rows for the following BatchNorm.  Each kernel keeps its
// own accumulator barrier protocol around drain_accumulator.
#pragma once
#include <cstdint>

// v[16] = this lane's row, 16 consecutive columns.  Returns, on every lane, the sum over the warp's 32 rows of column
// ((lane >> 1) & 15): a butterfly that halves the number of live columns at every step (8+4+2+1+1 = 16 shuffles
// instead of 16 x 5 for sixteen independent warp reductions).
__device__ __forceinline__ float warp_colsum16(const float (&v)[16], int lane) {
    float a[8], b[4], c[2], d;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        float keep = (lane & 16) ? v[j + 8] : v[j];
        float send = (lane & 16) ? v[j] : v[j + 8];
        a[j] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        float keep = (lane & 8) ? a[j + 4] : a[j];
        float send = (lane & 8) ? a[j] : a[j + 4];
        b[j] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        float keep = (lane & 4) ? b[j + 2] : b[j];
        float send = (lane & 4) ? b[j] : b[j + 2];
        c[j] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    }
    {
        float keep = (lane & 2) ? c[1] : c[0];
        float send = (lane & 2) ? c[0] : c[1];
        d = keep + __shfl_xor_sync(0xffffffffu, send, 2);
    }
    d += __shfl_xor_sync(0xffffffffu, d, 1);
    return d;
}

// An epilogue warp drains its 32 TMEM lanes (lane = tile row `row`; `tmem_lane` addresses the warp's first lane, column 0)
// of the fp32 accumulator ab of a double-buffered pair (TMEM columns [ab * COUT, (ab + 1) * COUT)):
// y[orow] = acc + bias (+ addend[orow]) for row < n_out, where orow = out_rows[row] if given (class-sorted dgrad launches
// scatter back to canonical rows), else row.  With bn_sums, the column sums of the rows just produced are added to acc_s /
// acc_q (sum / sum of squares, column n0 + ((lane >> 1) & 15) of every 16-column group n0): no second pass over y.
template <int COUT>
__device__ __forceinline__ void drain_accumulator(uint32_t tmem_lane, int ab, int row, int n_out, const int *__restrict__ out_rows,
                                                  const float *__restrict__ bias, const float *__restrict__ addend,
                                                  float *__restrict__ y, const double *bn_sums, float (&acc_s)[COUT / 16],
                                                  float (&acc_q)[COUT / 16], int lane) {
    const int orow = (out_rows && row < n_out) ? __ldg(out_rows + row) : row;
    const uint32_t taddr = tmem_lane + ab * COUT;
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
}

// After the last tile: adds an epilogue warp's sums to bn_sums ([0, COUT) sums, [COUT, 2 COUT) sums of squares).  Lane l
// (even) owns column n0 + ((l >> 1) & 15); one fp64 atomic per CTA-warp and channel.
template <int COUT>
__device__ __forceinline__ void flush_bn_sums(double *bn_sums, const float (&acc_s)[COUT / 16], const float (&acc_q)[COUT / 16],
                                              int lane) {
    if (bn_sums && !(lane & 1)) {
        const int col = (lane >> 1) & 15;
#pragma unroll
        for (int i = 0; i < COUT / 16; ++i) {
            atomicAdd(bn_sums + i * 16 + col, (double)acc_s[i]);
            atomicAdd(bn_sums + COUT + i * 16 + col, (double)acc_q[i]);
        }
    }
}
