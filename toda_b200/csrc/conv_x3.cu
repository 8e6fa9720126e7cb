// TODA_CONV_BF16X3: a tensor-core path at fp32-class accuracy (VERDICT r01 "missing" #3; the reference computes in fp32,
// spconv_backbone.py L73 / L187).  Every fp32 operand is split into two bf16 terms, v = hi + lo with hi = bf16(v) and
// lo = bf16(v - hi) (|v - hi - lo| <= 2^-17 |v|), and the product is evaluated as hi*hi + hi*lo + lo*hi on the SAME tcgen05
// kernels as the bf16 path (three launches chained through the epilogue's addend; fp32 accumulation in TMEM).  The
// dropped lo*lo term is 2^-16 relative: the result agrees with the fp32 FFMA path to ~1e-5, i.e. inside the rtol 1e-4 the
// north star asks of fp32, at 3x the bf16 cost instead of the ~12x of the FFMA kernels.
#include <cuda_bf16.h>

#include "common.cuh"
#include "conv.cuh"

namespace {

__device__ __forceinline__ void split_bf16(float v, __nv_bfloat16 &hi, __nv_bfloat16 &lo) {
    hi = __float2bfloat16_rn(v);
    lo = __float2bfloat16_rn(v - __bfloat162float(hi));
}

// x [n][cin] fp32 -> hi, lo [n][cpad] bf16 (channels >= cin zero)
__global__ void split_rows_kernel(const float *__restrict__ in, long long n, int cin, int cpad, __nv_bfloat16 *__restrict__ hi,
                                  __nv_bfloat16 *__restrict__ lo) {
    const long long total = n * cpad;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long r = e / cpad;
        const int c = (int)(e - r * cpad);
        __nv_bfloat16 h, l;
        split_bf16(c < cin ? __ldg(in + r * cin + c) : 0.f, h, l);
        hi[e] = h;
        lo[e] = l;
    }
}

// w [kvol][cin][cout] fp32 -> hi, lo [cout][kvol*cpad] bf16 (the K-major B operand)
__global__ void split_weights_kernel(const float *__restrict__ w, int kvol, int cin, int cpad, int cout, __nv_bfloat16 *__restrict__ hi,
                                     __nv_bfloat16 *__restrict__ lo) {
    const size_t per = (size_t)kvol * cpad * cout;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < per; e += (size_t)gridDim.x * blockDim.x) {
        const size_t kc = e % ((size_t)kvol * cpad);
        const int co = (int)(e / ((size_t)kvol * cpad));
        const int k = (int)(kc / cpad), ci = (int)(kc % cpad);
        __nv_bfloat16 h, l;
        split_bf16(ci < cin ? __ldg(w + ((size_t)k * cin + ci) * cout + co) : 0.f, h, l);
        hi[e] = h;
        lo[e] = l;
    }
}

// dw[co][k][ci] = t1 + t2 + t3 over [co][k][cpad] partial results, dropping the padded channels
__global__ void sum3_unpad_kernel(const float *__restrict__ t1, const float *__restrict__ t2, const float *__restrict__ t3, size_t rows,
                                  int cpad, int cin, float *__restrict__ dw) {
    const size_t total = rows * cin;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const size_t r = e / cin;
        const int c = (int)(e - r * cin);
        const size_t s = r * cpad + c;
        dw[e] = (t1[s] + t2[s]) + t3[s];
    }
}

struct X3Fwd { size_t x_bytes, w_bytes, inner; };
X3Fwd x3_fwd_layout(int n_in, int cin, int cout, int kvol) {
    const int cp = pad16(cin);
    X3Fwd l;
    l.x_bytes = align_up((size_t)(n_in > 0 ? n_in : 1) * cp * 2 + 16, 256);
    l.w_bytes = align_up((size_t)kvol * cp * cout * 2, 256);
    l.inner = conv_tc_fwd_workspace_bytes(n_in, cp, cout, kvol);
    return l;
}

struct X3Wgrad { size_t x_bytes, dy_bytes, t_bytes, inner; };
X3Wgrad x3_wgrad_layout(int n_in, int n_out, int kvol, int cin, int cout) {
    const int cp = pad16(cin);
    X3Wgrad l;
    l.x_bytes = align_up((size_t)(n_in > 0 ? n_in : 1) * cp * 2 + 16, 256);
    l.dy_bytes = align_up((size_t)(n_out > 0 ? n_out : 1) * cout * 2 + 16, 256);
    l.t_bytes = align_up((size_t)kvol * cp * cout * 4, 256);
    l.inner = conv_tc_wgrad_workspace_bytes(n_in, n_out, kvol, cp, cout);
    return l;
}

}  // namespace

size_t conv_x3_fwd_workspace_bytes(int n_in, int cin, int cout, int kvol) {
    X3Fwd l = x3_fwd_layout(n_in, cin, cout, kvol);
    return 2 * l.x_bytes + 2 * l.w_bytes + l.inner + 256;
}

int conv_x3_fwd(const float *x, int n_in, int cin, const int32_t *nbr, int n_out, int kvol, const float *w, int cout, const float *bias,
                float *y, const int32_t *out_rows, const uint32_t *tile_masks, double *bn_sums, void *workspace, size_t workspace_bytes,
                cudaStream_t st, const TilePlan *plan, const float *addend) {
    const size_t need = conv_x3_fwd_workspace_bytes(n_in, cin, cout, kvol);
    if (!workspace || workspace_bytes < need) {
        toda_set_error("spconv_fwd(bf16x3): workspace %zu < required %zu bytes", workspace_bytes, need);
        return TODA_ERR_WORKSPACE;
    }
    const int cp = pad16(cin);
    X3Fwd l = x3_fwd_layout(n_in, cin, cout, kvol);
    char *p = (char *)workspace;
    __nv_bfloat16 *xh = (__nv_bfloat16 *)p, *xl = (__nv_bfloat16 *)(p + l.x_bytes);
    __nv_bfloat16 *wh = (__nv_bfloat16 *)(p + 2 * l.x_bytes), *wl = (__nv_bfloat16 *)(p + 2 * l.x_bytes + l.w_bytes);
    void *inner = p + 2 * l.x_bytes + 2 * l.w_bytes;
    if (n_in > 0) {
        split_rows_kernel<<<wave_grid((int64_t)n_in * cp, 256), 256, 0, st>>>(x, n_in, cin, cp, xh, xl);
        TODA_LAUNCH_OK();
    }
    split_weights_kernel<<<wave_grid((int64_t)kvol * cp * cout, 256), 256, 0, st>>>(w, kvol, cin, cp, cout, wh, wl);
    TODA_LAUNCH_OK();
    // hi*hi (+ bias, + the caller's addend), then the two cross terms accumulated through the epilogue's addend (in place:
    // every output element is read and rewritten by the same thread); the BatchNorm statistics ride on the last launch
    int rc = conv_tc_fwd(x, xh, n_in, cp, nbr, n_out, kvol, w, cout, bias, y, out_rows, tile_masks, nullptr, inner, l.inner, st, plan, addend, wh);
    if (rc) return rc;
    rc = conv_tc_fwd(x, xh, n_in, cp, nbr, n_out, kvol, w, cout, nullptr, y, out_rows, tile_masks, nullptr, inner, l.inner, st, plan, y, wl);
    if (rc) return rc;
    return conv_tc_fwd(x, xl, n_in, cp, nbr, n_out, kvol, w, cout, nullptr, y, out_rows, tile_masks, bn_sums, inner, l.inner, st, plan, y, wh);
}

size_t conv_x3_wgrad_workspace_bytes(int n_in, int n_out, int kvol, int cin, int cout) {
    X3Wgrad l = x3_wgrad_layout(n_in, n_out, kvol, cin, cout);
    return 2 * l.x_bytes + 2 * l.dy_bytes + 3 * l.t_bytes + l.inner + 256;
}

int conv_x3_wgrad(const float *x, int n_in, int cin, const int32_t *nbr, int n_out, int kvol, const uint32_t *tile_masks,
                  const float *dy, int cout, float *dw_param, void *workspace, size_t workspace_bytes, cudaStream_t st) {
    const size_t need = conv_x3_wgrad_workspace_bytes(n_in, n_out, kvol, cin, cout);
    if (!workspace || workspace_bytes < need) {
        toda_set_error("spconv_wgrad(bf16x3): workspace %zu < required %zu bytes", workspace_bytes, need);
        return TODA_ERR_WORKSPACE;
    }
    const int cp = pad16(cin);
    X3Wgrad l = x3_wgrad_layout(n_in, n_out, kvol, cin, cout);
    char *p = (char *)workspace;
    __nv_bfloat16 *xh = (__nv_bfloat16 *)p, *xl = (__nv_bfloat16 *)(p + l.x_bytes);
    __nv_bfloat16 *dh = (__nv_bfloat16 *)(p + 2 * l.x_bytes), *dl = (__nv_bfloat16 *)(p + 2 * l.x_bytes + l.dy_bytes);
    float *t1 = (float *)(p + 2 * l.x_bytes + 2 * l.dy_bytes), *t2 = (float *)((char *)t1 + l.t_bytes), *t3 = (float *)((char *)t2 + l.t_bytes);
    void *inner = (char *)t3 + l.t_bytes;
    split_rows_kernel<<<wave_grid((int64_t)n_in * cp, 256), 256, 0, st>>>(x, n_in, cin, cp, xh, xl);
    TODA_LAUNCH_OK();
    split_rows_kernel<<<wave_grid((int64_t)n_out * cout, 256), 256, 0, st>>>(dy, n_out, cout, cout, dh, dl);
    TODA_LAUNCH_OK();
    int rc = conv_tc_wgrad(x, xh, n_in, cp, nbr, n_out, kvol, tile_masks, dy, dh, cout, t1, inner, l.inner, st);
    if (rc) return rc;
    rc = conv_tc_wgrad(x, xh, n_in, cp, nbr, n_out, kvol, tile_masks, dy, dl, cout, t2, inner, l.inner, st);
    if (rc) return rc;
    rc = conv_tc_wgrad(x, xl, n_in, cp, nbr, n_out, kvol, tile_masks, dy, dh, cout, t3, inner, l.inner, st);
    if (rc) return rc;
    const size_t rows = (size_t)cout * kvol;
    sum3_unpad_kernel<<<wave_grid((int64_t)rows * cin, 256), 256, 0, st>>>(t1, t2, t3, rows, cp, cin, dw_param);
    TODA_LAUNCH_OK();
    return TODA_OK;
}
