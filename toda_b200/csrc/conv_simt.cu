// K5/K6/K7 sparse convolution, fp32 FFMA path (TODA_CONV_FP32): the parity path.
// Output-stationary gather-GEMM: a CTA owns a tile of output rows, loops over the kernel offsets,
// gathers the neighbour rows named by the table into shared memory and accumulates in registers.
// No scatter, no atomics: every output row is written exactly once (deterministic).
// The tcgen05 path (conv_tc.cu) has the same structure with the accumulator in TMEM.
#include "common.cuh"
#include "conv.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int BK = 16;

// y[o, col0:col0+BN] = bias + sum_k x[nbr[k,o], :] @ w[k][:, col0:col0+BN]
template <int BM, int BN>
__global__ void __launch_bounds__(kThreads) conv_fwd_f32_kernel(const float *__restrict__ x, int cin,
                                                                const int *__restrict__ nbr, int n_out, int kvol,
                                                                const float *__restrict__ w, int cout,
                                                                const float *__restrict__ bias, float *__restrict__ y,
                                                                const int *__restrict__ out_rows /* optional */,
                                                                const float *__restrict__ addend /* optional */) {
    static_assert((BM / 4) * (BN / 4) == kThreads, "4x4 micro-tiles must cover the CTA tile");
    __shared__ __align__(16) float As[BK][BM + 4];
    __shared__ __align__(16) float Bs[BK][BN + 4];
    __shared__ int rows[BM];
    const int tid = threadIdx.x;
    const int tx = tid % (BN / 4), ty = tid / (BN / 4);
    const int row0 = blockIdx.x * BM, col0 = blockIdx.y * BN;
    const bool vec = (cin % 4) == 0;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    for (int k = 0; k < kvol; ++k) {
        int any = 0;
        for (int m = tid; m < BM; m += kThreads) {
            int r = row0 + m;
            int src = (r < n_out) ? __ldg(nbr + (size_t)k * n_out + r) : -1;
            rows[m] = src;
            any |= (src >= 0);
        }
        any = __syncthreads_or(any);  // also publishes rows[]
        if (!any) continue;           // CTA-uniform: no row of this tile has a neighbour at offset k
        for (int c0 = 0; c0 < cin; c0 += BK) {
            // gathered A tile, stored transposed (As[kk][m]) so the FFMA loop reads float4 along m
            if (vec) {
                for (int e = tid; e < BM * (BK / 4); e += kThreads) {
                    int m = e / (BK / 4), q = e % (BK / 4);
                    int src = rows[m];
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (src >= 0 && c0 + q * 4 < cin) v = __ldg((const float4 *)(x + (size_t)src * cin + c0 + q * 4));
                    As[q * 4 + 0][m] = v.x; As[q * 4 + 1][m] = v.y; As[q * 4 + 2][m] = v.z; As[q * 4 + 3][m] = v.w;
                }
            } else {
                for (int e = tid; e < BM * BK; e += kThreads) {
                    int m = e / BK, kk = e % BK;
                    int src = rows[m];
                    As[kk][m] = (src >= 0 && c0 + kk < cin) ? __ldg(x + (size_t)src * cin + c0 + kk) : 0.f;
                }
            }
            for (int e = tid; e < BK * BN; e += kThreads) {
                int kk = e / BN, nn = e % BN;
                Bs[kk][nn] = (c0 + kk < cin && col0 + nn < cout) ? __ldg(w + ((size_t)k * cin + c0 + kk) * cout + col0 + nn) : 0.f;
            }
            __syncthreads();
#pragma unroll
            for (int kk = 0; kk < BK; ++kk) {
                float4 a = *(const float4 *)&As[kk][ty * 4];
                float4 b = *(const float4 *)&Bs[kk][tx * 4];
                float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
            }
            __syncthreads();
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        int r = row0 + ty * 4 + i;
        if (r >= n_out) continue;
        const int orow = out_rows ? __ldg(out_rows + r) : r;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int c = col0 + tx * 4 + j;
            if (c < cout) y[(size_t)orow * cout + c] = acc[i][j] + (bias ? __ldg(bias + c) : 0.f) + (addend ? __ldg(addend + (size_t)orow * cout + c) : 0.f);
        }
    }
}

// dw partial[split][k][ci][co] = sum over this split's rows of x[nbr[k,o], ci] * dy[o, co].
// Rows without a neighbour at offset k are compacted away on the fly (ballot + prefix in shared memory),
// so the FFMA loop only sees real pairs -- at stride 1 only ~14% of (row, offset) slots are pairs.
constexpr int WT = 64;  // weight tile WT x WT per CTA (4x4 per thread)
__global__ void __launch_bounds__(kThreads) conv_wgrad_f32_kernel(const float *__restrict__ x, int cin,
                                                                  const int *__restrict__ nbr, int n_out, int kvol,
                                                                  const float *__restrict__ dy, int cout, int rows_per_split,
                                                                  float *__restrict__ partial) {
    __shared__ __align__(16) float As[BK][WT + 4];
    __shared__ __align__(16) float Bs[BK][WT + 4];
    __shared__ int pin[kThreads], pout[kThreads];
    __shared__ int warp_cnt[kThreads / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tx = tid % (WT / 4), ty = tid / (WT / 4);
    const int ci_tiles = (cin + WT - 1) / WT, co_tiles = (cout + WT - 1) / WT;
    int bx = blockIdx.x;
    const int co_t = bx % co_tiles; bx /= co_tiles;
    const int ci_t = bx % ci_tiles; bx /= ci_tiles;
    const int k = bx;
    const int split = blockIdx.y;
    const int ci0 = ci_t * WT, co0 = co_t * WT;
    const int r_begin = split * rows_per_split;
    const int r_end = min(n_out, r_begin + rows_per_split);
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    for (int r0 = r_begin; r0 < r_end; r0 += kThreads) {
        int r = r0 + tid;
        int src = (r < r_end) ? __ldg(nbr + (size_t)k * n_out + r) : -1;
        unsigned bal = __ballot_sync(0xffffffffu, src >= 0);
        if (lane == 0) warp_cnt[warp] = __popc(bal);
        __syncthreads();
        int woff = 0, total = 0;
#pragma unroll
        for (int wi = 0; wi < kThreads / 32; ++wi) {
            int c = warp_cnt[wi];
            if (wi < warp) woff += c;
            total += c;
        }
        if (src >= 0) {
            int pos = woff + __popc(bal & ((1u << lane) - 1u));
            pin[pos] = src;
            pout[pos] = r;
        }
        __syncthreads();
        for (int g0 = 0; g0 < total; g0 += BK) {
            for (int e = tid; e < BK * WT; e += kThreads) {
                int kk = e / WT, c = e % WT;
                bool ok = g0 + kk < total;
                As[kk][c] = (ok && ci0 + c < cin) ? __ldg(x + (size_t)pin[ok ? g0 + kk : 0] * cin + ci0 + c) : 0.f;
                Bs[kk][c] = (ok && co0 + c < cout) ? __ldg(dy + (size_t)pout[ok ? g0 + kk : 0] * cout + co0 + c) : 0.f;
            }
            __syncthreads();
#pragma unroll
            for (int kk = 0; kk < BK; ++kk) {
                float4 a = *(const float4 *)&As[kk][ty * 4];
                float4 b = *(const float4 *)&Bs[kk][tx * 4];
                float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
            }
            __syncthreads();
        }
    }
    float *dst = partial + ((size_t)split * kvol + k) * cin * cout;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        int ci = ci0 + ty * 4 + i;
        if (ci >= cin) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int co = co0 + tx * 4 + j;
            if (co < cout) dst[(size_t)ci * cout + co] = acc[i][j];
        }
    }
}

// fixed-order reduction over splits, written in the parameter layout (Cout, kvol, Cin)
// fixed-order reduction over splits, written in the parameter layout (Cout, kvol, Cin)
__global__ void wgrad_reduce_kernel(const float *__restrict__ partial, int splits, int kvol, int cin, int cout,
                                    float *__restrict__ dw_param) {
    size_t per = (size_t)kvol * cin * cout;
    const int sub = threadIdx.x & 7;   // 8 lanes per element walk the splits; fixed shuffle tree => deterministic
    for (size_t e = (blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 3; e < ((per + 31) & ~(size_t)31);
         e += ((size_t)gridDim.x * blockDim.x) >> 3) {
        float s = 0.f;
        if (e < per) {
            // e indexes the parameter layout: (co, k, ci)
            int ci = (int)(e % cin);
            size_t t = e / cin;
            int k = (int)(t % kvol);
            int co = (int)(t / kvol);
            size_t src = ((size_t)k * cin + ci) * cout + co;
            for (int sp = sub; sp < splits; sp += 8) s += partial[sp * per + src];
        }
        s += __shfl_xor_sync(0xffffffffu, s, 1);
        s += __shfl_xor_sync(0xffffffffu, s, 2);
        s += __shfl_xor_sync(0xffffffffu, s, 4);
        if (e < per && sub == 0) dw_param[e] = s;
    }
}

__global__ void weight_repack_kernel(const float *__restrict__ w_param, int kvol, int cin, int cout, int transpose,
                                     int mirror, float *__restrict__ w_out) {
    size_t per = (size_t)kvol * cin * cout;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < per; e += (size_t)gridDim.x * blockDim.x) {
        // e indexes the output: [k][ci][co] or (transpose) [k][co][ci]
        int inner = (int)(e % (transpose ? cin : cout));
        size_t t = e / (transpose ? cin : cout);
        int mid = (int)(t % (transpose ? cout : cin));
        int k = (int)(t / (transpose ? cout : cin));
        int ci = transpose ? inner : mid, co = transpose ? mid : inner;
        int ks = mirror ? kvol - 1 - k : k;
        w_out[e] = __ldg(w_param + ((size_t)co * kvol + ks) * cin + ci);
    }
}

__global__ void gather_rows_kernel(const float *__restrict__ in, const int *__restrict__ rows, long long total, int c,
                                   float *__restrict__ out) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        long long i = e / c;
        int r = __ldg(rows + i);
        out[e] = r >= 0 ? __ldg(in + (long long)r * c + (e - i * c)) : 0.f;
    }
}

int wgrad_splits(int n_out, int kvol, int cin, int cout) {
    int tiles = kvol * ((cin + WT - 1) / WT) * ((cout + WT - 1) / WT);
    int want = (4 * kNumSMs + tiles - 1) / tiles;  // ~4 CTAs per SM in flight
    int max_by_rows = (n_out + 4 * kThreads - 1) / (4 * kThreads);
    int s = want < max_by_rows ? want : max_by_rows;
    return s < 1 ? 1 : s;
}

}  // namespace

extern "C" int toda_weight_repack(const float *w_param, int kvol, int cin, int cout, int transpose, int mirror_k,
                                  float *w_out, void *stream) {
    TODA_CHECK_ARG(w_param && w_out && kvol > 0 && cin > 0 && cout > 0, "weight_repack: bad args");
    size_t per = (size_t)kvol * cin * cout;
    weight_repack_kernel<<<wave_grid(per, 256), 256, 0, (cudaStream_t)stream>>>(w_param, kvol, cin, cout, transpose,
                                                                              mirror_k, w_out);
    TODA_LAUNCH_OK();
    return TODA_OK;
}

// 1 when toda_spconv_fwd(precision) runs the tensor-core kernel for this shape (and can therefore fuse the BN statistics)
extern "C" int toda_spconv_uses_tensor_cores(int cin, int cout, int kvol, int precision) {
    return (precision == TODA_CONV_BF16 || precision == TODA_CONV_BF16X3) && conv_tc_supported(cin, cout, kvol) ? 1 : 0;
}

extern "C" int toda_spconv_wgrad_uses_tensor_cores(int cin, int cout, int kvol, int precision) {
    return (precision == TODA_CONV_BF16 || precision == TODA_CONV_BF16X3) && conv_tc_wgrad_supported(cin, cout, kvol) ? 1 : 0;
}

extern "C" size_t toda_spconv_fwd_workspace_bytes(int n_in, int cin, int cout, int kvol, int precision) {
    if (precision == TODA_CONV_BF16 && n_in >= 0 && cin > 0 && cout > 0 && kvol > 0 && conv_tc_supported(cin, cout, kvol))
        return conv_tc_fwd_workspace_bytes(n_in, cin, cout, kvol);
    if (precision == TODA_CONV_BF16X3 && n_in >= 0 && cin > 0 && cout > 0 && kvol > 0 && conv_tc_supported(cin, cout, kvol))
        return conv_x3_fwd_workspace_bytes(n_in, cin, cout, kvol);
    return 0;
}

extern "C" int toda_spconv_fwd(const float *x, const void *x_bf16, int n_in, int cin, const int32_t *nbr, int n_out, int kvol,
                               const float *w, int cout, const float *bias, const float *addend, float *y,
                               const int32_t *out_rows, const uint32_t *tile_masks, const uint16_t *plan_lidx,
                               const int32_t *plan_rows, const int32_t *plan_cnt, int plan_groups, int plan_cap, double *bn_sums,
                               const void *w_bf16, int precision, void *workspace, size_t workspace_bytes, void *stream) {
    TODA_CHECK_ARG(n_in >= 0 && n_out >= 0 && cin > 0 && cout > 0 && kvol > 0, "spconv_fwd: bad sizes");
    if (n_out == 0) return TODA_OK;
    TODA_CHECK_ARG(x && nbr && w && y, "spconv_fwd: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    TODA_CHECK_ARG(precision == TODA_CONV_FP32 || precision == TODA_CONV_BF16 || precision == TODA_CONV_BF16X3,
                   "spconv_fwd: unknown precision %d", precision);
    const TilePlan plan_data{plan_lidx, plan_rows, plan_cnt, plan_groups, plan_cap};
    const TilePlan *plan = plan_lidx ? &plan_data : nullptr;
    if (precision == TODA_CONV_BF16X3 && conv_tc_supported(cin, cout, kvol))
        return conv_x3_fwd(x, n_in, cin, nbr, n_out, kvol, w, cout, bias, y, out_rows, tile_masks, bn_sums, workspace, workspace_bytes, st,
                           plan, addend);
    // kernel selection by shape: the tensor-core kernel covers Cin in {<=16 (zero-padded to 16), 32, 64, 128} and
    // Cout in {16,32,64,128}; anything else (e.g. the dgrad of the 4/5-channel input layer) runs on the FFMA kernel.
    if (precision == TODA_CONV_BF16 && conv_tc_supported(cin, cout, kvol))
        return conv_tc_fwd(x, x_bf16, n_in, cin, nbr, n_out, kvol, w, cout, bias, y, out_rows, tile_masks, bn_sums, workspace,
                           workspace_bytes, st, plan, addend, w_bf16);
    TODA_CHECK_ARG(!bn_sums, "spconv_fwd: fused BatchNorm statistics need the tensor-core kernel for this shape");
    if (cout <= 16) {
        dim3 grid(ceil_div(n_out, 256), ceil_div(cout, 16));
        conv_fwd_f32_kernel<256, 16><<<grid, kThreads, 0, st>>>(x, cin, nbr, n_out, kvol, w, cout, bias, y, out_rows, addend);
    } else if (cout <= 32) {
        dim3 grid(ceil_div(n_out, 128), ceil_div(cout, 32));
        conv_fwd_f32_kernel<128, 32><<<grid, kThreads, 0, st>>>(x, cin, nbr, n_out, kvol, w, cout, bias, y, out_rows, addend);
    } else {
        dim3 grid(ceil_div(n_out, 64), ceil_div(cout, 64));
        conv_fwd_f32_kernel<64, 64><<<grid, kThreads, 0, st>>>(x, cin, nbr, n_out, kvol, w, cout, bias, y, out_rows, addend);
    }
    TODA_LAUNCH_OK();
    return TODA_OK;
}

extern "C" size_t toda_spconv_wgrad_workspace_bytes(int n_in, int n_out, int kvol, int cin, int cout, int precision) {
    if (n_in < 0 || n_out < 0 || kvol <= 0 || cin <= 0 || cout <= 0) return 0;
    if (precision == TODA_CONV_BF16 && conv_tc_wgrad_supported(cin, cout, kvol))
        return conv_tc_wgrad_workspace_bytes(n_in, n_out, kvol, cin, cout);
    if (precision == TODA_CONV_BF16X3 && conv_tc_wgrad_supported(cin, cout, kvol))
        return conv_x3_wgrad_workspace_bytes(n_in, n_out, kvol, cin, cout);
    int splits = wgrad_splits(n_out, kvol, cin, cout);
    return align_up((size_t)splits * kvol * cin * cout * sizeof(float), 256);
}

extern "C" int toda_spconv_wgrad(const float *x, const void *x_bf16, int n_in, int cin, const int32_t *nbr, int n_out,
                                 int kvol, const uint32_t *tile_masks, const float *dy, const void *dy_bf16, int cout,
                                 float *dw_param, void *workspace, size_t workspace_bytes, int precision, void *stream) {
    TODA_CHECK_ARG(n_in >= 0 && n_out >= 0 && cin > 0 && cout > 0 && kvol > 0, "spconv_wgrad: bad sizes");
    TODA_CHECK_ARG(dw_param, "spconv_wgrad: null dw");
    cudaStream_t st = (cudaStream_t)stream;
    if (n_out == 0) {
        TODA_CUDA_OK(cudaMemsetAsync(dw_param, 0, (size_t)kvol * cin * cout * sizeof(float), st));
        return TODA_OK;
    }
    TODA_CHECK_ARG(x && nbr && dy && workspace, "spconv_wgrad: null pointer");
    TODA_CHECK_ARG(precision == TODA_CONV_FP32 || precision == TODA_CONV_BF16 || precision == TODA_CONV_BF16X3,
                   "spconv_wgrad: unknown precision %d", precision);
    if (precision == TODA_CONV_BF16X3 && conv_tc_wgrad_supported(cin, cout, kvol))
        return conv_x3_wgrad(x, n_in, cin, nbr, n_out, kvol, tile_masks, dy, cout, dw_param, workspace, workspace_bytes, st);
    if (precision == TODA_CONV_BF16 && conv_tc_wgrad_supported(cin, cout, kvol))
        return conv_tc_wgrad(x, x_bf16, n_in, cin, nbr, n_out, kvol, tile_masks, dy, dy_bf16, cout, dw_param, workspace,
                             workspace_bytes, st);
    int splits = wgrad_splits(n_out, kvol, cin, cout);
    size_t need = (size_t)splits * kvol * cin * cout * sizeof(float);
    if (workspace_bytes < need) {
        toda_set_error("spconv_wgrad: workspace %zu < required %zu bytes", workspace_bytes, need);
        return TODA_ERR_WORKSPACE;
    }
    int rows_per_split = ceil_div(n_out, splits);
    rows_per_split = ceil_div(rows_per_split, kThreads) * kThreads;
    int tiles = kvol * ((cin + WT - 1) / WT) * ((cout + WT - 1) / WT);
    dim3 grid(tiles, splits);
    conv_wgrad_f32_kernel<<<grid, kThreads, 0, st>>>(x, cin, nbr, n_out, kvol, dy, cout, rows_per_split, (float *)workspace);
    TODA_LAUNCH_OK();
    size_t per = (size_t)kvol * cin * cout;
    wgrad_reduce_kernel<<<wave_grid(per * 8, 256), 256, 0, st>>>((const float *)workspace, splits, kvol, cin, cout, dw_param);
    TODA_LAUNCH_OK();
    return TODA_OK;
}

extern "C" int toda_gather_rows(const float *in, const int32_t *rows, int n, int channels, float *out, void *stream) {
    TODA_CHECK_ARG(n >= 0 && channels > 0, "gather_rows: bad sizes");
    if (n == 0) return TODA_OK;
    TODA_CHECK_ARG(in && rows && out, "gather_rows: null pointer");
    long long total = (long long)n * channels;
    gather_rows_kernel<<<wave_grid(total, 256), 256, 0, (cudaStream_t)stream>>>(in, rows, total, channels, out);
    TODA_LAUNCH_OK();
    return TODA_OK;
}
