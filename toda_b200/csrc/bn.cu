// K8 BatchNorm1d (+ReLU, +residual) over (N_active, C) rows, and column sums (bias gradient).
// All passes are HBM-bound streams over (N, C) fp32; reductions use fixed-size per-CTA partials reduced
// in a fixed order, so results are run-to-run deterministic.
#include <cuda_bf16.h>

#include "common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kPartials = 2 * kNumSMs;  // CTAs in the reduction grids
// CTAs of a resident streaming grid at most (2048 threads per SM): the backward apply pass leaves one partial column sum
// per CTA for the bias gradient
constexpr int kApplyPartials = 2048 / kThreads * kNumSMs;

// per-CTA partial sums of up to two quantities per channel; C % 4 == 0 path: one thread owns 4 channels (float4
// loads) and walks rows with four independent loads in flight per array.
// mode 0: (y, y*y)      mode 1: (g, g*xhat) with g = da*(a>0)     mode 2: (dy, -)
template <int MODE>
__global__ void __launch_bounds__(kThreads) col_reduce_vec_kernel(const float *__restrict__ p0, const float *__restrict__ p1,
                                                                  const float *__restrict__ p2, int n, int c,
                                                                  const float *__restrict__ mean, const float *__restrict__ rstd,
                                                                  int relu, double *__restrict__ partial) {
    __shared__ double s0[kThreads * 4], s1[kThreads * 4];
    const int tpr = c >> 2;                       // threads per row
    const int rpi = kThreads / tpr;               // rows per CTA iteration
    const int tx = threadIdx.x % tpr, ty = threadIdx.x / tpr;
    double a0[4] = {0, 0, 0, 0}, a1[4] = {0, 0, 0, 0};
    float4 m4 = make_float4(0, 0, 0, 0), r4 = make_float4(0, 0, 0, 0);
    if (MODE == 1) { m4 = __ldg((const float4 *)mean + tx); r4 = __ldg((const float4 *)rstd + tx); }
    const long long stride = (long long)gridDim.x * rpi;
    const bool active = ty < rpi;
    constexpr int U = 4;                          // rows in flight per thread and array
    for (long long r = (long long)blockIdx.x * rpi + ty; active && r < n; r += U * stride) {
        float4 v0[U], v1[U], v2[U];
        bool ok[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            long long rr = r + u * stride;
            ok[u] = rr < n;
            size_t e = ok[u] ? (size_t)rr * tpr + tx : 0;
            v0[u] = __ldg((const float4 *)p0 + e);
            if (MODE == 1) { v1[u] = __ldg((const float4 *)p1 + e); v2[u] = __ldg((const float4 *)p2 + e); }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (!ok[u]) continue;
            float x[4] = {v0[u].x, v0[u].y, v0[u].z, v0[u].w};
            if (MODE == 0) {
#pragma unroll
                for (int q = 0; q < 4; ++q) { a0[q] += x[q]; a1[q] += (double)x[q] * x[q]; }
            } else if (MODE == 1) {
                float av[4] = {v1[u].x, v1[u].y, v1[u].z, v1[u].w}, yv[4] = {v2[u].x, v2[u].y, v2[u].z, v2[u].w};
                float mm[4] = {m4.x, m4.y, m4.z, m4.w}, rs[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    float g = (relu && !(av[q] > 0.f)) ? 0.f : x[q];
                    float xh = (yv[q] - mm[q]) * rs[q];
                    a0[q] += g; a1[q] += (double)g * xh;
                }
            } else {
#pragma unroll
                for (int q = 0; q < 4; ++q) a0[q] += x[q];
            }
        }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) { s0[threadIdx.x * 4 + q] = a0[q]; s1[threadIdx.x * 4 + q] = a1[q]; }
    __syncthreads();
    if ((int)threadIdx.x < c) {
        // channel ch = threadIdx.x lives in thread tx = ch/4, slot ch%4 of every row lane ty
        int ch = threadIdx.x, txx = ch >> 2, q = ch & 3;
        double t0 = 0.0, t1 = 0.0;
        for (int j = 0; j < rpi; ++j) { t0 += s0[(j * tpr + txx) * 4 + q]; t1 += s1[(j * tpr + txx) * 4 + q]; }
        partial[((size_t)blockIdx.x * 2 + 0) * c + ch] = t0;
        partial[((size_t)blockIdx.x * 2 + 1) * c + ch] = t1;
    }
}

// scalar fallback for channel counts that are not a multiple of 4 (e.g. the 5 point features)
template <int MODE>
__global__ void __launch_bounds__(kThreads) col_reduce_kernel(const float *__restrict__ p0, const float *__restrict__ p1,
                                                              const float *__restrict__ p2, int n, int c,
                                                              const float *__restrict__ mean, const float *__restrict__ rstd,
                                                              int relu, double *__restrict__ partial) {
    __shared__ double s0[kThreads], s1[kThreads];
    const int cpad = c <= 16 ? 16 : (c <= 32 ? 32 : (c <= 64 ? 64 : (c <= 128 ? 128 : 256)));
    const int rows_per_iter = kThreads / cpad;
    const int tx = threadIdx.x % cpad, ty = threadIdx.x / cpad;
    double a0 = 0.0, a1 = 0.0;
    float m = 0.f, rs = 0.f;
    if (MODE == 1 && tx < c) { m = mean[tx]; rs = rstd[tx]; }
    for (long long r = (long long)blockIdx.x * rows_per_iter + ty; r < n; r += (long long)gridDim.x * rows_per_iter) {
        if (tx < c) {
            size_t e = (size_t)r * c + tx;
            if (MODE == 0) {
                float v = __ldg(p0 + e);
                a0 += v; a1 += (double)v * v;
            } else if (MODE == 1) {
                float g = __ldg(p0 + e);
                if (relu && !(__ldg(p1 + e) > 0.f)) g = 0.f;
                float xh = (__ldg(p2 + e) - m) * rs;
                a0 += g; a1 += (double)g * xh;
            } else {
                a0 += __ldg(p0 + e);
            }
        }
    }
    s0[threadIdx.x] = a0; s1[threadIdx.x] = a1;
    __syncthreads();
    if (threadIdx.x < cpad && threadIdx.x < c) {
        double t0 = 0.0, t1 = 0.0;
        for (int j = 0; j < rows_per_iter; ++j) { t0 += s0[j * cpad + threadIdx.x]; t1 += s1[j * cpad + threadIdx.x]; }
        partial[((size_t)blockIdx.x * 2 + 0) * c + threadIdx.x] = t0;
        partial[((size_t)blockIdx.x * 2 + 1) * c + threadIdx.x] = t1;
    }
}

// A thread of the float4 kernels owns four channels; with kThreads a multiple of C/4, so is every grid stride, and a
// thread keeps its channels over the whole grid-stride loop.
static bool vec_channels(int c) { return c % 4 == 0 && kThreads % (c / 4) == 0; }

template <int MODE>
static void launch_col_reduce(const float *p0, const float *p1, const float *p2, int n, int c, const float *mean,
                              const float *rstd, int relu, double *partial, cudaStream_t st) {
    if (vec_channels(c))
        col_reduce_vec_kernel<MODE><<<kPartials, kThreads, 0, st>>>(p0, p1, p2, n, c, mean, rstd, relu, partial);
    else
        col_reduce_kernel<MODE><<<kPartials, kThreads, 0, st>>>(p0, p1, p2, n, c, mean, rstd, relu, partial);
}

// fixed-order sum of the per-CTA partials of one channel: one warp per channel, lanes stride over the partials.
// All loads of a lane are issued before the first add (the loop used to be a chain of ~10 dependent L2 round trips,
// which made this tiny kernel take as long as a third of the streaming pass next to it).  A CTA left ROWS rows of c
// partials (quantity q in row q; ss is only summed when ROWS = 2), at most MAX_BLOCKS CTAs.
template <int MAX_BLOCKS = kPartials, int ROWS = 2>
__device__ __forceinline__ void warp_sum_partials(const double *__restrict__ partial, int nblocks, int c, int ch, double &s,
                                                  double &ss) {
    const int lane = threadIdx.x & 31;
    constexpr int kPerLane = (MAX_BLOCKS + 31) / 32;
    double va[kPerLane], vb[kPerLane];
#pragma unroll
    for (int i = 0; i < kPerLane; ++i) {
        const int j = lane + 32 * i;
        const bool ok = j < nblocks;
        va[i] = ok ? partial[((size_t)j * ROWS) * c + ch] : 0.0;
        vb[i] = ok && ROWS == 2 ? partial[((size_t)j * ROWS + 1) * c + ch] : 0.0;
    }
    double a = 0.0, b = 0.0;
#pragma unroll
    for (int i = 0; i < kPerLane; ++i) { a += va[i]; b += vb[i]; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
    s = a; ss = b;
}

// BatchNorm coefficients of one channel from its sums (fp64), with explicit roundings: every training-mode coefficient
// of the library is derived here.
__device__ __forceinline__ void bn_coeffs(double s, double ss, int n, float g, float bt, float eps, float &scale, float &shift,
                                          float &meanf, float &rstd, double &var) {
    const double mean = n > 0 ? s / n : 0.0;
    var = n > 0 ? ss / n - mean * mean : 0.0;
    if (var < 0.0) var = 0.0;
    rstd = (float)(1.0 / sqrt(var + (double)eps));
    meanf = (float)mean;
    scale = __fmul_rn(g, rstd);
    shift = __fsub_rn(bt, __fmul_rn(__fmul_rn(meanf, g), rstd));
}

__device__ __forceinline__ void bn_update_running(float *running_mean, float *running_var, int ch, float momentum, float meanf,
                                                  double var, int n) {
    if (running_mean) running_mean[ch] = __fadd_rn(__fmul_rn(1.f - momentum, running_mean[ch]), __fmul_rn(momentum, meanf));
    if (running_var) {
        const double unbiased = n > 1 ? var * n / (n - 1) : var;
        running_var[ch] = __fadd_rn(__fmul_rn(1.f - momentum, running_var[ch]), __fmul_rn(momentum, (float)unbiased));
    }
}

// out = [sum(y) | sum(y*y)] per channel: from the per-CTA partials (partial != NULL), copied from `src` (the convolution
// epilogue's sums; src == out: in place) or zeros (no rows).  `count` (optional) receives the row count: written here, on
// the device, so that a count all-reduced with the sums never has to pass through the host.
__global__ void bn_local_sums_kernel(const double *partial, int nblocks, const double *src, int n, int c, double *out,
                                     double *count) {
    if (count && blockIdx.x == 0 && threadIdx.x == 0) *count = (double)n;
    int ch = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (ch >= c) return;
    double s = 0.0, ss = 0.0;
    if (partial) warp_sum_partials(partial, nblocks, c, ch, s, ss);
    else if (src) { s = src[ch]; ss = src[c + ch]; }
    if ((threadIdx.x & 31) != 0) return;
    out[ch] = s;
    out[c + ch] = ss;
}

__global__ void bn_eval_coeffs_kernel(const float *gamma, const float *beta, const float *rm, const float *rv, float eps,
                                      int c, float *scale, float *shift) {
    int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= c) return;
    float rstd = 1.0f / sqrtf(rv[ch] + eps);
    float g = gamma ? gamma[ch] : 1.f, bt = beta ? beta[ch] : 0.f;
    scale[ch] = g * rstd;
    shift[ch] = bt - rm[ch] * g * rstd;
}

// bf16 copy of four consecutive outputs (element group e of a float4 stream): the next convolution's tensor-core operand
__device__ __forceinline__ void store_bf16x4(__nv_bfloat16 *__restrict__ dst, long long e, float4 o) {
    __nv_bfloat162 lo = __floats2bfloat162_rn(o.x, o.y), hi = __floats2bfloat162_rn(o.z, o.w);
    uint2 pk;
    pk.x = *(uint32_t *)&lo;
    pk.y = *(uint32_t *)&hi;
    ((uint2 *)dst)[e] = pk;
}

// Where the coefficients of an apply pass come from.  Training (sums != NULL): sums = [sum(y) | sum(y*y)] (fp64) of the
// whole batch and its row count (*count, or n when count is NULL); block 0 publishes scale / shift / save_mean /
// save_rstd and updates the running statistics (not on an empty batch).  Eval (sums == NULL): scale / shift as
// toda_bn_eval_coeffs wrote them.
struct BnCoeffs {
    const double *sums; const double *count; int n;
    const float *gamma, *beta; float eps, momentum;
    float *running_mean, *running_var, *scale, *shift, *save_mean, *save_rstd;
};

// a = act(y*scale + shift (+ residual)): every CTA first fills the coefficients of all channels into shared memory
// (scale[c] | shift[c]), then streams its rows.  VEC (vec_channels(c)): float4 rows, a thread's four coefficients held
// in registers.  A process with no rows still runs block 0: its running statistics must follow the other ranks'.
template <bool VEC>
__global__ void __launch_bounds__(kThreads) bn_apply_kernel(const float *__restrict__ y, long long total, int c, BnCoeffs k,
                                                            const float *__restrict__ residual, int relu, float *__restrict__ a,
                                                            __nv_bfloat16 *__restrict__ a_bf16) {
    extern __shared__ __align__(16) float s_coef[];
    float *s_sc = s_coef, *s_sh = s_coef + c;
    const int n = k.count ? (int)*k.count : k.n;
    for (int ch = threadIdx.x; ch < c; ch += blockDim.x) {
        if (!k.sums) {
            s_sc[ch] = k.scale[ch];
            s_sh[ch] = k.shift[ch];
            continue;
        }
        float meanf, rstd;
        double var;
        bn_coeffs(k.sums[ch], k.sums[c + ch], n, k.gamma ? k.gamma[ch] : 1.f, k.beta ? k.beta[ch] : 0.f, k.eps, s_sc[ch], s_sh[ch],
                  meanf, rstd, var);
        if (blockIdx.x == 0) {
            k.scale[ch] = s_sc[ch];
            k.shift[ch] = s_sh[ch];
            if (k.save_mean) k.save_mean[ch] = meanf;
            if (k.save_rstd) k.save_rstd[ch] = rstd;
            if (n > 0) bn_update_running(k.running_mean, k.running_var, ch, k.momentum, meanf, var, n);
        }
    }
    __syncthreads();
    const long long stride = (long long)gridDim.x * blockDim.x;
    long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (VEC) {
        const long long tv = total >> 2;
        const int ch = (int)((e << 2) % c);
        const float4 sc = *(const float4 *)(s_sc + ch), sh = *(const float4 *)(s_sh + ch);
        for (; e < tv; e += stride) {
            const float4 v = __ldg((const float4 *)y + e);
            float4 o = make_float4(fmaf(v.x, sc.x, sh.x), fmaf(v.y, sc.y, sh.y), fmaf(v.z, sc.z, sh.z), fmaf(v.w, sc.w, sh.w));
            if (residual) {
                const float4 r = __ldg((const float4 *)residual + e);
                o.x += r.x; o.y += r.y; o.z += r.z; o.w += r.w;
            }
            if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
            ((float4 *)a)[e] = o;
            if (a_bf16) store_bf16x4(a_bf16, e, o);
        }
    } else {
        for (; e < total; e += stride) {
            const int ch = (int)(e % c);
            float o = fmaf(__ldg(y + e), s_sc[ch], s_sh[ch]);
            if (residual) o += __ldg(residual + e);
            if (relu) o = fmaxf(o, 0.f);
            a[e] = o;
            if (a_bf16) a_bf16[e] = __float2bfloat16_rn(o);
        }
    }
}

// sums = [sum g | sum g*xhat] (fp64) of the per-CTA partials, and the same rounded to float as dbeta / dgamma
__global__ void bn_bwd_finalize_kernel(const double *__restrict__ partial, int nblocks, int c, float *dgamma, float *dbeta,
                                       double *sums) {
    int ch = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (ch >= c) return;
    double s, sx;
    warp_sum_partials(partial, nblocks, c, ch, s, sx);
    if ((threadIdx.x & 31) != 0) return;
    if (dbeta) dbeta[ch] = (float)s;
    if (dgamma) dgamma[ch] = (float)sx;
    sums[ch] = s;
    sums[c + ch] = sx;
}

// dy = gamma*rstd*(g - sum_g/N - xhat*sum_gx/N)   (training)   |   dy = gamma*rstd*g   (eval)
// Per channel this is dy = A*g + B*y + C with A = gamma*rstd, B = -gamma*rstd^2*sum_gx/N,
// C = -A*sum_g/N - B*mean: coefficients are computed once per thread (4 channels), rows stream as float4.
// The sums are bn_bwd_finalize_kernel's (all-reduced over the processes of a synchronized BatchNorm), rounded to float;
// N is *count (the global count of a synchronized BatchNorm, device memory) or n when count is NULL.
// db_partial (optional): the column sums of dy -- the gradient of the bias of the convolution before the BatchNorm -- as
// fixed-order fp64 partials, one row of c per CTA in dynamic shared memory of kThreads*4 doubles (col_sum_finalize_kernel
// sums them).  Every thread keeps the same
// channels over its whole grid-stride loop: VEC, because kThreads is a multiple of c/4; scalar, because the stride is
// rounded down to a multiple of c (the few threads past it idle).  At most 48 registers: the 5 CTAs per SM this
// HBM-bound pass had before it also summed dy.
template <bool VEC>
__global__ void __launch_bounds__(kThreads, 5) bn_bwd_apply_kernel(const float *__restrict__ da, const float *__restrict__ a,
                                                                const float *__restrict__ y, long long total, int c, int n,
                                                                const double *__restrict__ count, const float *__restrict__ gamma,
                                                                const float *__restrict__ mean, const float *__restrict__ rstd,
                                                                const double *__restrict__ sums, int relu, int training,
                                                                float *__restrict__ dy, float *__restrict__ dres,
                                                                __nv_bfloat16 *__restrict__ dy_bf16, double *__restrict__ db_partial) {
    extern __shared__ double s_db[];
    double db[4] = {0.0, 0.0, 0.0, 0.0};       // this thread's sums of dy (VEC: its 4 channels; scalar: db[0])
    if (count) n = (int)*count;
    auto sum = [&](int i) -> float { return (float)sums[i]; };
    const float inv_n = n > 0 ? 1.0f / (float)n : 0.f;
    const long long threads = (long long)gridDim.x * blockDim.x;
    const long long stride = VEC ? threads : threads / c * c;
    long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (VEC) {
        const long long tv = total >> 2;
        const int ch = (int)((e << 2) % c);
        float A[4], B[4], C[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            float gm = gamma ? gamma[ch + q] : 1.f, rs = rstd[ch + q];
            A[q] = gm * rs;
            B[q] = training ? -gm * rs * rs * sum(c + ch + q) * inv_n : 0.f;
            C[q] = training ? -A[q] * sum(ch + q) * inv_n - B[q] * mean[ch + q] : 0.f;
        }
        for (; e < tv; e += stride) {
            float4 g4 = __ldg((const float4 *)da + e);
            float4 y4 = training ? __ldg((const float4 *)y + e) : make_float4(0.f, 0.f, 0.f, 0.f);
            if (relu) {
                float4 a4 = __ldg((const float4 *)a + e);
                g4.x = a4.x > 0.f ? g4.x : 0.f; g4.y = a4.y > 0.f ? g4.y : 0.f;
                g4.z = a4.z > 0.f ? g4.z : 0.f; g4.w = a4.w > 0.f ? g4.w : 0.f;
            }
            if (dres) ((float4 *)dres)[e] = g4;
            float4 o;
            o.x = fmaf(A[0], g4.x, fmaf(B[0], y4.x, C[0]));
            o.y = fmaf(A[1], g4.y, fmaf(B[1], y4.y, C[1]));
            o.z = fmaf(A[2], g4.z, fmaf(B[2], y4.z, C[2]));
            o.w = fmaf(A[3], g4.w, fmaf(B[3], y4.w, C[3]));
            if (dy) ((float4 *)dy)[e] = o;
            if (dy_bf16) store_bf16x4(dy_bf16, e, o);
            if (db_partial) { db[0] += o.x; db[1] += o.y; db[2] += o.z; db[3] += o.w; }
        }
    } else {
        for (e = e < stride ? e : total; e < total; e += stride) {
            int ch = (int)(e % c);
            float g = __ldg(da + e);
            if (relu && !(__ldg(a + e) > 0.f)) g = 0.f;
            if (dres) dres[e] = g;
            float gm = gamma ? gamma[ch] : 1.f;
            float rs = rstd[ch];
            float o;
            if (training) {
                float xh = (__ldg(y + e) - mean[ch]) * rs;
                o = gm * rs * (g - sum(ch) * inv_n - xh * sum(c + ch) * inv_n);
            } else {
                o = gm * rs * g;
            }
            if (dy) dy[e] = o;
            if (dy_bf16) dy_bf16[e] = __float2bfloat16_rn(o);
            if (db_partial) db[0] += o;
        }
    }
    if (!db_partial) return;
    // CTA sum per channel in a fixed order: thread t < c takes channel t's slots
    constexpr int kSlots = VEC ? 4 : 1;
#pragma unroll
    for (int q = 0; q < kSlots; ++q) s_db[threadIdx.x * kSlots + q] = db[q];
    __syncthreads();
    if ((int)threadIdx.x < c) {
        // VEC: thread t holds channels 4*(t % (c/4)) + q; scalar: channel (blockIdx.x*kThreads + t) % c
        const int units = VEC ? c / 4 : c;
        const int u = VEC ? (int)threadIdx.x >> 2 : (int)threadIdx.x, q = VEC ? (int)threadIdx.x & 3 : 0;
        double t = 0.0;
        for (int j = u; j < kThreads; j += units) t += s_db[j * kSlots + q];
        const int ch = VEC ? (int)threadIdx.x : (int)(((long long)blockIdx.x * kThreads + threadIdx.x) % c);
        db_partial[(size_t)blockIdx.x * c + ch] = t;
    }
}

// out[ch] = the fixed-order sum of the first quantity of the per-CTA partials (col_reduce: two rows per CTA; the
// backward apply pass's bias sums: one row per CTA)
template <int MAX_BLOCKS, int ROWS>
__global__ void col_sum_finalize_kernel(const double *__restrict__ partial, int nblocks, int c, float *out) {
    int ch = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (ch >= c) return;
    double s, unused;
    warp_sum_partials<MAX_BLOCKS, ROWS>(partial, nblocks, c, ch, s, unused);
    if ((threadIdx.x & 31) == 0) out[ch] = (float)s;
}

// workspace: the per-CTA partials (two rows of c per reduction CTA, or one per backward-apply CTA), then the 2c reduced
// backward sums of toda_bn_bwd
size_t partials_bytes(int c) {
    return (size_t)(2 * kPartials > kApplyPartials ? 2 * kPartials : kApplyPartials) * c * sizeof(double);
}
size_t bn_ws_bytes(int c) { return align_up(partials_bytes(c) + 2 * c * sizeof(double), 256); }

// Grid of a grid-stride streaming kernel over `items` work items: exactly the CTAs that are resident at once (occupancy x
// SMs, queried once per kernel), never more than the work.  A grid that is 1.3-1.6 waves (what a fixed 8 CTAs/SM gave for
// the 34- and 41-register kernels) leaves most SMs idle during the second, partial wave.
template <auto Kernel> int resident_grid(int64_t items) {
    static const int64_t cap = [] {
        int per_sm = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, Kernel, kThreads, 0) != cudaSuccess || per_sm < 1) per_sm = 4;
        return (int64_t)per_sm * kNumSMs;
    }();
    const int64_t need = (items + kThreads - 1) / kThreads;
    return (int)(need < 1 ? 1 : (need < cap ? need : cap));
}

int launch_bn_apply(const float *y, int n, int c, const BnCoeffs &k, const float *residual, int relu, float *a, void *a_bf16,
                    cudaStream_t st) {
    const long long total = (long long)n * c;
    const size_t smem = 2 * (size_t)c * sizeof(float);
    if (vec_channels(c))
        bn_apply_kernel<true><<<resident_grid<bn_apply_kernel<true>>(total / 4), kThreads, smem, st>>>(
            y, total, c, k, residual, relu, a, (__nv_bfloat16 *)a_bf16);
    else
        bn_apply_kernel<false><<<resident_grid<bn_apply_kernel<false>>(total), kThreads, smem, st>>>(
            y, total, c, k, residual, relu, a, (__nv_bfloat16 *)a_bf16);
    TODA_LAUNCH_OK();
    return TODA_OK;
}

}  // namespace

extern "C" size_t toda_bn_workspace_bytes(int channels) { return channels > 0 ? bn_ws_bytes(channels) : 0; }

double *bn_workspace_red(void *workspace, int c) { return (double *)((char *)workspace + partials_bytes(c)); }

extern "C" int toda_bn_local_sums(const float *y, const double *epilogue_sums, int n, int c, double *sums, double *count,
                                  void *workspace, size_t workspace_bytes, void *stream) {
    TODA_CHECK_ARG(n >= 0 && c > 0 && c <= 256 && sums, "bn_local_sums: bad args n=%d c=%d", n, c);
    if (n > 0 && epilogue_sums == sums && !count) return TODA_OK;      // already in place, and no count wanted
    cudaStream_t st = (cudaStream_t)stream;
    const double *partial = nullptr;
    if (n > 0 && !epilogue_sums) {
        TODA_CHECK_ARG(y && workspace, "bn_local_sums: null pointer");
        if (workspace_bytes < bn_ws_bytes(c)) { toda_set_error("bn_local_sums: workspace too small"); return TODA_ERR_WORKSPACE; }
        launch_col_reduce<0>(y, nullptr, nullptr, n, c, nullptr, nullptr, 0, (double *)workspace, st);
        TODA_LAUNCH_OK();
        partial = (const double *)workspace;
    }
    bn_local_sums_kernel<<<ceil_div(c * 32, 128), 128, 0, st>>>(partial, kPartials, n > 0 ? epilogue_sums : nullptr, n, c, sums,
                                                              count);
    TODA_LAUNCH_OK();
    return TODA_OK;
}

extern "C" int toda_bn_eval_coeffs(const float *gamma, const float *beta, const float *running_mean, const float *running_var,
                                   float eps, int c, float *scale, float *shift, void *stream) {
    TODA_CHECK_ARG(c > 0 && running_mean && running_var && scale && shift, "bn_eval_coeffs: bad args");
    bn_eval_coeffs_kernel<<<ceil_div(c, 128), 128, 0, (cudaStream_t)stream>>>(gamma, beta, running_mean, running_var, eps, c,
                                                                             scale, shift);
    TODA_LAUNCH_OK();
    return TODA_OK;
}

extern "C" int toda_bn_apply(const float *y, int n, int c, const float *scale, const float *shift, const float *residual,
                             int relu, float *a, void *a_bf16, void *stream) {
    TODA_CHECK_ARG(n >= 0 && c > 0, "bn_apply: bad sizes");
    if (n == 0) return TODA_OK;
    TODA_CHECK_ARG(y && scale && shift && a, "bn_apply: null pointer");
    BnCoeffs k{};
    k.scale = (float *)scale;
    k.shift = (float *)shift;
    return launch_bn_apply(y, n, c, k, residual, relu, a, a_bf16, (cudaStream_t)stream);
}

extern "C" int toda_bn_apply_sums(const float *y, int n, int c, const double *sums, const double *count, const float *gamma,
                                  const float *beta, float eps, float momentum, float *running_mean, float *running_var,
                                  float *scale, float *shift, float *save_mean, float *save_rstd, const float *residual, int relu,
                                  float *a, void *a_bf16, void *stream) {
    TODA_CHECK_ARG(n >= 0 && c > 0 && sums && scale && shift, "bn_apply_sums: bad args");
    TODA_CHECK_ARG(n == 0 || (y && a), "bn_apply_sums: null pointer");
    const BnCoeffs k{sums, count, n, gamma, beta, eps, momentum, running_mean, running_var, scale, shift, save_mean, save_rstd};
    return launch_bn_apply(y, n, c, k, residual, relu, a, a_bf16, (cudaStream_t)stream);
}

extern "C" int toda_bn_bwd_reduce(const float *da, const float *a, const float *y, int n, int c, const float *save_mean,
                                  const float *save_rstd, int relu, double *local_red, float *dgamma, float *dbeta, void *workspace,
                                  size_t workspace_bytes, void *stream) {
    TODA_CHECK_ARG(n >= 0 && c > 0 && c <= 256, "bn_bwd_reduce: unsupported sizes n=%d c=%d", n, c);
    TODA_CHECK_ARG(save_mean && save_rstd && workspace && local_red && (n == 0 || (da && y)) && (!relu || a || n == 0),
                   "bn_bwd_reduce: null pointer");
    if (workspace_bytes < bn_ws_bytes(c)) { toda_set_error("bn_bwd_reduce: workspace too small"); return TODA_ERR_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    double *partial = (double *)workspace;
    launch_col_reduce<1>(da, a, y, n, c, save_mean, save_rstd, relu, partial, st);
    TODA_LAUNCH_OK();
    bn_bwd_finalize_kernel<<<ceil_div(c * 32, 128), 128, 0, st>>>(partial, kPartials, c, dgamma, dbeta, local_red);
    TODA_LAUNCH_OK();
    return TODA_OK;
}

extern "C" int toda_bn_bwd_finish(const float *da, const float *a, const float *y, int n, int c, const float *gamma,
                                  const float *save_mean, const float *save_rstd, int relu, int training, const double *red,
                                  const double *count, float *dy, void *dy_bf16, float *dresidual, float *dbias, void *workspace,
                                  size_t workspace_bytes, void *stream) {
    TODA_CHECK_ARG(n >= 0 && c > 0 && c <= 256, "bn_bwd_finish: unsupported sizes n=%d c=%d", n, c);
    // dy may be NULL when dy_bf16 is given: the fp32 gradient is then not stored (a caller whose consumers -- tensor-core
    // dgrad and wgrad -- only read the bf16 copy saves 4 of the ~30 bytes per element this pass moves)
    TODA_CHECK_ARG(save_mean && save_rstd && (red || !training) && (n == 0 || (da && y && (dy || dy_bf16))) &&
                   (!relu || a || n == 0) && (!dbias || workspace), "bn_bwd_finish: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    if (dbias && workspace_bytes < bn_ws_bytes(c)) { toda_set_error("bn_bwd_finish: workspace too small"); return TODA_ERR_WORKSPACE; }
    if (n == 0) {
        if (dbias) TODA_CUDA_OK(cudaMemsetAsync(dbias, 0, sizeof(float) * c, st));
        return TODA_OK;
    }
    const long long total = (long long)n * c;
    double *db_partial = dbias ? (double *)workspace : nullptr;
    const size_t smem = dbias ? kThreads * 4 * sizeof(double) : 0;    // the CTA's column sums, only with a bias gradient
    int grid;
    if (vec_channels(c)) {
        grid = resident_grid<bn_bwd_apply_kernel<true>>(total / 4);
        grid = grid < kApplyPartials ? grid : kApplyPartials;
        bn_bwd_apply_kernel<true><<<grid, kThreads, smem, st>>>(da, a, y, total, c, n, count, gamma, save_mean, save_rstd, red, relu,
                                                               training, dy, dresidual, (__nv_bfloat16 *)dy_bf16, db_partial);
    } else {
        grid = resident_grid<bn_bwd_apply_kernel<false>>(total);
        grid = grid < kApplyPartials ? grid : kApplyPartials;
        bn_bwd_apply_kernel<false><<<grid, kThreads, smem, st>>>(da, a, y, total, c, n, count, gamma, save_mean, save_rstd, red,
                                                                relu, training, dy, dresidual, (__nv_bfloat16 *)dy_bf16, db_partial);
    }
    TODA_LAUNCH_OK();
    if (dbias) {
        col_sum_finalize_kernel<kApplyPartials, 1><<<ceil_div(c * 32, 128), 128, 0, st>>>(db_partial, grid, c, dbias);
        TODA_LAUNCH_OK();
    }
    return TODA_OK;
}

extern "C" int toda_bn_bwd(const float *da, const float *a, const float *y, int n, int c, const float *gamma,
                           const float *save_mean, const float *save_rstd, int relu, int training, float *dy, void *dy_bf16,
                           float *dresidual, float *dgamma, float *dbeta, float *dbias, void *workspace, size_t workspace_bytes,
                           void *stream) {
    TODA_CHECK_ARG(workspace, "bn_bwd: null workspace");
    double *red = bn_workspace_red(workspace, c);
    int rc = toda_bn_bwd_reduce(da, a, y, n, c, save_mean, save_rstd, relu, red, dgamma, dbeta, workspace, workspace_bytes, stream);
    if (rc) return rc;
    return toda_bn_bwd_finish(da, a, y, n, c, gamma, save_mean, save_rstd, relu, training, red, nullptr, dy, dy_bf16, dresidual,
                              dbias, workspace, workspace_bytes, stream);
}

extern "C" int toda_col_sum(const float *dy, int n, int c, float *out, void *workspace, size_t workspace_bytes, void *stream) {
    TODA_CHECK_ARG(n >= 0 && c > 0 && c <= 256 && out && workspace, "col_sum: bad args");
    if (workspace_bytes < bn_ws_bytes(c)) { toda_set_error("col_sum: workspace too small"); return TODA_ERR_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    double *partial = (double *)workspace;
    launch_col_reduce<2>(dy, nullptr, nullptr, n, c, nullptr, nullptr, 0, partial, st);
    TODA_LAUNCH_OK();
    col_sum_finalize_kernel<kPartials, 2><<<ceil_div(c * 32, 128), 128, 0, st>>>(partial, kPartials, c, out);
    TODA_LAUNCH_OK();
    return TODA_OK;
}
