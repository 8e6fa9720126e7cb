// K8 BatchNorm1d (+ReLU, +residual) over (N_active, C) rows, and column sums (bias gradient).
// All passes are HBM-bound streams over (N, C) fp32; reductions use fixed-size per-CTA partials reduced
// in a fixed order, so results are run-to-run deterministic.
#include <cuda_bf16.h>

#include "common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kPartials = 2 * kNumSMs;  // CTAs in the reduction grids

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

template <int MODE>
static void launch_col_reduce(const float *p0, const float *p1, const float *p2, int n, int c, const float *mean,
                              const float *rstd, int relu, double *partial, cudaStream_t st) {
    if (c % 4 == 0 && kThreads % (c / 4) == 0)
        col_reduce_vec_kernel<MODE><<<kPartials, kThreads, 0, st>>>(p0, p1, p2, n, c, mean, rstd, relu, partial);
    else
        col_reduce_kernel<MODE><<<kPartials, kThreads, 0, st>>>(p0, p1, p2, n, c, mean, rstd, relu, partial);
}

// fixed-order sum of the per-CTA partials of one channel: one warp per channel, lanes stride over the partials.
// All loads of a lane are issued before the first add (the loop used to be a chain of ~10 dependent L2 round trips,
// which made this tiny kernel take as long as a third of the streaming pass next to it).
__device__ __forceinline__ void warp_sum_partials(const double *__restrict__ partial, int nblocks, int c, int ch, double &s,
                                                  double &ss) {
    const int lane = threadIdx.x & 31;
    constexpr int kPerLane = (kPartials + 31) / 32;
    double va[kPerLane], vb[kPerLane];
#pragma unroll
    for (int i = 0; i < kPerLane; ++i) {
        const int j = lane + 32 * i;
        const bool ok = j < nblocks;
        va[i] = ok ? partial[((size_t)j * 2) * c + ch] : 0.0;
        vb[i] = ok ? partial[((size_t)j * 2 + 1) * c + ch] : 0.0;
    }
    double a = 0.0, b = 0.0;
#pragma unroll
    for (int i = 0; i < kPerLane; ++i) { a += va[i]; b += vb[i]; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
    s = a; ss = b;
}

// BatchNorm coefficients of one channel from its sums (fp64).  One definition for the finalize kernel and for the fused
// statistics+apply kernel below, with explicit roundings so that both produce the same bits.
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

__global__ void bn_finalize_kernel(const double *__restrict__ partial, int nblocks, int n, int c,
                                   const float *__restrict__ gamma, const float *__restrict__ beta, float eps, float momentum,
                                   float *running_mean, float *running_var, float *scale, float *shift, float *save_mean,
                                   float *save_rstd) {
    int ch = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (ch >= c) return;
    double s, ss;
    warp_sum_partials(partial, nblocks, c, ch, s, ss);
    if ((threadIdx.x & 31) != 0) return;
    float sc, sh, meanf, rstd;
    double var;
    bn_coeffs(s, ss, n, gamma ? gamma[ch] : 1.f, beta ? beta[ch] : 0.f, eps, sc, sh, meanf, rstd, var);
    scale[ch] = sc;
    shift[ch] = sh;
    if (save_mean) save_mean[ch] = meanf;
    if (save_rstd) save_rstd[ch] = rstd;
    bn_update_running(running_mean, running_var, ch, momentum, meanf, var, n);
}

// Local statistics of a BatchNorm whose batch spans several processes: out = [sum(y) | sum(y*y) | n], the fp64 buffer
// that is all-reduced across ranks.  From the per-CTA partials (partial != NULL: the same fixed-order sums as
// bn_finalize_kernel) or copied from `src` (the convolution epilogue's sums; src == out: count only; NULL: zeros).
// The count is written here, on the device, so the host never has to provide or read it.
__global__ void bn_local_sums_kernel(const double *partial, int nblocks, const double *src, int n, int c, double *out) {
    if (blockIdx.x == 0 && threadIdx.x == 0) out[2 * c] = (double)n;
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

// a = act(y*scale + shift (+ residual)); C % 4 == 0 -> float4 path
template <bool VEC>
__global__ void __launch_bounds__(kThreads) bn_apply_kernel(const float *__restrict__ y, long long total, int c,
                                                            const float *__restrict__ scale, const float *__restrict__ shift,
                                                            const float *__restrict__ residual, int relu, float *__restrict__ a,
                                                            __nv_bfloat16 *__restrict__ a_bf16) {
    if (VEC) {
        long long tv = total >> 2;
        for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < tv; e += (long long)gridDim.x * blockDim.x) {
            int ch = (int)((e << 2) % c);
            float4 v = __ldg((const float4 *)y + e);
            float4 sc = __ldg((const float4 *)(scale + ch)), sh = __ldg((const float4 *)(shift + ch));
            float4 o = make_float4(fmaf(v.x, sc.x, sh.x), fmaf(v.y, sc.y, sh.y), fmaf(v.z, sc.z, sh.z), fmaf(v.w, sc.w, sh.w));
            if (residual) {
                float4 r = __ldg((const float4 *)residual + e);
                o.x += r.x; o.y += r.y; o.z += r.z; o.w += r.w;
            }
            if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
            ((float4 *)a)[e] = o;
            if (a_bf16) {   // bf16 shadow for the tensor-core operands of the next convolution
                __nv_bfloat162 lo = __floats2bfloat162_rn(o.x, o.y), hi = __floats2bfloat162_rn(o.z, o.w);
                uint2 pk;
                pk.x = *(uint32_t *)&lo;
                pk.y = *(uint32_t *)&hi;
                ((uint2 *)a_bf16)[e] = pk;
            }
        }
    } else {
        for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
            int ch = (int)(e % c);
            float o = fmaf(__ldg(y + e), scale[ch], shift[ch]);
            if (residual) o += __ldg(residual + e);
            if (relu) o = fmaxf(o, 0.f);
            a[e] = o;
            if (a_bf16) a_bf16[e] = __float2bfloat16_rn(o);
        }
    }
}

// Training-mode BatchNorm whose statistics arrive as per-channel sums from the producing convolution's epilogue: every
// thread derives the coefficients of its four channels itself (grid x block is a multiple of C/4: a thread keeps its
// channels over the grid stride), so the finalize launch between the convolution and this pass disappears; the first C/4
// threads of block 0 also publish scale / shift / mean / rstd for the backward pass and update the running statistics.
__global__ void __launch_bounds__(kThreads) bn_apply_sums_kernel(const float *__restrict__ y, long long total, int c, int n,
                                                                 const double *__restrict__ sums, const float *__restrict__ gamma,
                                                                 const float *__restrict__ beta, float eps, float momentum,
                                                                 float *running_mean, float *running_var, float *scale_out,
                                                                 float *shift_out, float *save_mean, float *save_rstd,
                                                                 const float *__restrict__ residual, int relu, float *__restrict__ a,
                                                                 __nv_bfloat16 *__restrict__ a_bf16) {
    const long long tv = total >> 2;
    const long long stride = (long long)gridDim.x * blockDim.x;
    long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const int ch = (int)((e << 2) % c);
    float sc[4], sh[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        float meanf, rstd;
        double var;
        bn_coeffs(sums[ch + q], sums[c + ch + q], n, gamma ? gamma[ch + q] : 1.f, beta ? beta[ch + q] : 0.f, eps, sc[q], sh[q], meanf,
                  rstd, var);
        if (e < (c >> 2)) {          // block 0, one thread per group of four channels
            scale_out[ch + q] = sc[q];
            shift_out[ch + q] = sh[q];
            if (save_mean) save_mean[ch + q] = meanf;
            if (save_rstd) save_rstd[ch + q] = rstd;
            bn_update_running(running_mean, running_var, ch + q, momentum, meanf, var, n);
        }
    }
    for (; e < tv; e += stride) {
        const float4 v = __ldg((const float4 *)y + e);
        float4 o = make_float4(fmaf(v.x, sc[0], sh[0]), fmaf(v.y, sc[1], sh[1]), fmaf(v.z, sc[2], sh[2]), fmaf(v.w, sc[3], sh[3]));
        if (residual) {
            const float4 r = __ldg((const float4 *)residual + e);
            o.x += r.x; o.y += r.y; o.z += r.z; o.w += r.w;
        }
        if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
        ((float4 *)a)[e] = o;
        if (a_bf16) {
            __nv_bfloat162 lo = __floats2bfloat162_rn(o.x, o.y), hi = __floats2bfloat162_rn(o.z, o.w);
            uint2 pk;
            pk.x = *(uint32_t *)&lo;
            pk.y = *(uint32_t *)&hi;
            ((uint2 *)a_bf16)[e] = pk;
        }
    }
}

// Training-mode BatchNorm from statistics all-reduced over several processes: sums = [sum(y) | sum(y*y) | n] of the
// union batch (bn_local_sums_kernel's layout).  Every CTA derives the coefficients of all channels into shared memory
// (the same bn_coeffs as the finalize kernels, so the same bits), block 0 publishes scale / shift / mean / rstd and
// updates the running statistics with the global count; then the rows of this process stream as in bn_apply_kernel.
// A process with no rows still runs block 0: its running statistics must follow the other ranks'.
template <bool VEC>
__global__ void __launch_bounds__(kThreads) bn_apply_global_kernel(const float *__restrict__ y, long long total, int c,
                                                                   const double *__restrict__ sums, const float *__restrict__ gamma,
                                                                   const float *__restrict__ beta, float eps, float momentum,
                                                                   float *running_mean, float *running_var, float *scale_out,
                                                                   float *shift_out, float *save_mean, float *save_rstd,
                                                                   const float *__restrict__ residual, int relu, float *__restrict__ a,
                                                                   __nv_bfloat16 *__restrict__ a_bf16) {
    __shared__ __align__(16) float s_sc[256], s_sh[256];
    const int n = (int)sums[2 * c];
    for (int ch = threadIdx.x; ch < c; ch += blockDim.x) {
        float meanf, rstd;
        double var;
        bn_coeffs(sums[ch], sums[c + ch], n, gamma ? gamma[ch] : 1.f, beta ? beta[ch] : 0.f, eps, s_sc[ch], s_sh[ch], meanf, rstd, var);
        if (blockIdx.x == 0) {
            scale_out[ch] = s_sc[ch];
            shift_out[ch] = s_sh[ch];
            if (save_mean) save_mean[ch] = meanf;
            if (save_rstd) save_rstd[ch] = rstd;
            if (n > 0) bn_update_running(running_mean, running_var, ch, momentum, meanf, var, n);
        }
    }
    __syncthreads();
    if (VEC) {
        const long long tv = total >> 2;
        for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < tv; e += (long long)gridDim.x * blockDim.x) {
            const int ch = (int)((e << 2) % c);
            const float4 v = __ldg((const float4 *)y + e);
            const float4 sc = *(const float4 *)(s_sc + ch), sh = *(const float4 *)(s_sh + ch);
            float4 o = make_float4(fmaf(v.x, sc.x, sh.x), fmaf(v.y, sc.y, sh.y), fmaf(v.z, sc.z, sh.z), fmaf(v.w, sc.w, sh.w));
            if (residual) {
                const float4 r = __ldg((const float4 *)residual + e);
                o.x += r.x; o.y += r.y; o.z += r.z; o.w += r.w;
            }
            if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
            ((float4 *)a)[e] = o;
            if (a_bf16) {
                __nv_bfloat162 lo = __floats2bfloat162_rn(o.x, o.y), hi = __floats2bfloat162_rn(o.z, o.w);
                uint2 pk;
                pk.x = *(uint32_t *)&lo;
                pk.y = *(uint32_t *)&hi;
                ((uint2 *)a_bf16)[e] = pk;
            }
        }
    } else {
        for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
            const int ch = (int)(e % c);
            float o = fmaf(__ldg(y + e), s_sc[ch], s_sh[ch]);
            if (residual) o += __ldg(residual + e);
            if (relu) o = fmaxf(o, 0.f);
            a[e] = o;
            if (a_bf16) a_bf16[e] = __float2bfloat16_rn(o);
        }
    }
}

// T = float: the sums bn_bwd_apply_kernel reads in the same call; T = double: the local sums a multi-process BatchNorm
// all-reduces before its bn_bwd_apply_kernel<., true> (which rounds them to float exactly as this kernel does for float).
template <typename T>
__global__ void bn_bwd_finalize_kernel(const double *__restrict__ partial, int nblocks, int c, float *dgamma, float *dbeta,
                                       T *sums /* [2c]: sum_g, sum_g_xhat */) {
    int ch = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (ch >= c) return;
    double s, sx;
    warp_sum_partials(partial, nblocks, c, ch, s, sx);
    if ((threadIdx.x & 31) != 0) return;
    if (dbeta) dbeta[ch] = (float)s;
    if (dgamma) dgamma[ch] = (float)sx;
    sums[ch] = (T)s;
    sums[c + ch] = (T)sx;
}

// dy = gamma*rstd*(g - sum_g/N - xhat*sum_gx/N)   (training)   |   dy = gamma*rstd*g   (eval)
// Per channel this is dy = A*g + B*y + C with A = gamma*rstd, B = -gamma*rstd^2*sum_gx/N,
// C = -A*sum_g/N - B*mean: coefficients are computed once per thread (4 channels), rows stream as float4.
// GLOBAL: the sums are the fp64 ones all-reduced over the processes of a synchronized BatchNorm (`gsums`) and N is the
// global count (`gcount`, device memory); both are rounded exactly as the single-process path rounds them.
template <bool VEC, bool GLOBAL>
__global__ void __launch_bounds__(kThreads) bn_bwd_apply_kernel(const float *__restrict__ da, const float *__restrict__ a,
                                                                const float *__restrict__ y, long long total, int c, int n_local,
                                                                const float *__restrict__ gamma, const float *__restrict__ mean,
                                                                const float *__restrict__ rstd, const float *__restrict__ fsums,
                                                                const double *__restrict__ gsums, const double *__restrict__ gcount,
                                                                int relu, int training, float *__restrict__ dy,
                                                                float *__restrict__ dres, __nv_bfloat16 *__restrict__ dy_bf16) {
    const int n = GLOBAL ? (int)*gcount : n_local;
    auto sums = [&](int i) -> float { return GLOBAL ? (float)gsums[i] : fsums[i]; };
    const float inv_n = n > 0 ? 1.0f / (float)n : 0.f;
    if (VEC) {
        const long long tv = total >> 2;
        const long long stride = (long long)gridDim.x * blockDim.x;      // multiple of c/4 (host guarantees it)
        long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
        const int ch = (int)((e << 2) % c);
        float A[4], B[4], C[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            float gm = gamma ? gamma[ch + q] : 1.f, rs = rstd[ch + q];
            A[q] = gm * rs;
            B[q] = training ? -gm * rs * rs * sums(c + ch + q) * inv_n : 0.f;
            C[q] = training ? -A[q] * sums(ch + q) * inv_n - B[q] * mean[ch + q] : 0.f;
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
            if (dy_bf16) {
                __nv_bfloat162 lo = __floats2bfloat162_rn(o.x, o.y), hi = __floats2bfloat162_rn(o.z, o.w);
                uint2 pk;
                pk.x = *(uint32_t *)&lo;
                pk.y = *(uint32_t *)&hi;
                ((uint2 *)dy_bf16)[e] = pk;
            }
        }
    } else {
        for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
            int ch = (int)(e % c);
            float g = __ldg(da + e);
            if (relu && !(__ldg(a + e) > 0.f)) g = 0.f;
            if (dres) dres[e] = g;
            float gm = gamma ? gamma[ch] : 1.f;
            float rs = rstd[ch];
            float o;
            if (training) {
                float xh = (__ldg(y + e) - mean[ch]) * rs;
                o = gm * rs * (g - sums(ch) * inv_n - xh * sums(c + ch) * inv_n);
            } else {
                o = gm * rs * g;
            }
            if (dy) dy[e] = o;
            if (dy_bf16) dy_bf16[e] = __float2bfloat16_rn(o);
        }
    }
}

__global__ void col_sum_finalize_kernel(const double *__restrict__ partial, int nblocks, int c, float *out) {
    int ch = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (ch >= c) return;
    double s, unused;
    warp_sum_partials(partial, nblocks, c, ch, s, unused);
    if ((threadIdx.x & 31) == 0) out[ch] = (float)s;
}

size_t bn_ws_bytes(int c) { return align_up((size_t)kPartials * 2 * c * sizeof(double) + 2 * c * sizeof(float), 256); }

}  // namespace

extern "C" size_t toda_bn_workspace_bytes(int channels) { return channels > 0 ? bn_ws_bytes(channels) : 0; }

extern "C" int toda_bn_stats(const float *y, int n, int c, const float *gamma, const float *beta, float eps, float momentum,
                             float *running_mean, float *running_var, float *scale, float *shift, float *save_mean,
                             float *save_rstd, void *workspace, size_t workspace_bytes, void *stream) {
    TODA_CHECK_ARG(n >= 0 && c > 0 && c <= 256, "bn_stats: unsupported sizes n=%d c=%d", n, c);
    TODA_CHECK_ARG((y || n == 0) && scale && shift && workspace, "bn_stats: null pointer");
    if (workspace_bytes < bn_ws_bytes(c)) { toda_set_error("bn_stats: workspace too small"); return TODA_ERR_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    double *partial = (double *)workspace;
    launch_col_reduce<0>(y, nullptr, nullptr, n, c, nullptr, nullptr, 0, partial, st);
    TODA_LAUNCH_OK();
    // an empty batch has no statistics: the running statistics stay as they are (torch.nn.BatchNorm1d does the same)
    bn_finalize_kernel<<<ceil_div(c * 32, 128), 128, 0, st>>>(partial, kPartials, n, c, gamma, beta, eps, momentum,
                                                        n > 0 ? running_mean : nullptr, n > 0 ? running_var : nullptr,
                                                        scale, shift, save_mean, save_rstd);
    TODA_LAUNCH_OK();
    return TODA_OK;
}

extern "C" int toda_bn_finalize_sums(const double *sums, int n, int c, const float *gamma, const float *beta, float eps,
                                     float momentum, float *running_mean, float *running_var, float *scale, float *shift,
                                     float *save_mean, float *save_rstd, void *stream) {
    TODA_CHECK_ARG(n >= 0 && c > 0 && sums && scale && shift, "bn_finalize_sums: bad args");
    // `sums` = [sum(y) per channel | sum(y*y) per channel]: the layout of one partial block of toda_bn_stats.  An empty
    // batch leaves the running statistics unchanged, as in toda_bn_stats.
    bn_finalize_kernel<<<ceil_div(c * 32, 128), 128, 0, (cudaStream_t)stream>>>(sums, 1, n, c, gamma, beta, eps, momentum,
                                                                            n > 0 ? running_mean : nullptr,
                                                                            n > 0 ? running_var : nullptr, scale, shift,
                                                                            save_mean, save_rstd);
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

// Grid of a grid-stride streaming kernel: exactly the CTAs that are resident at once (occupancy x SMs), never more than
// the work.  A grid that is 1.3-1.6 waves (what a fixed 8 CTAs/SM gave for the 34- and 41-register kernels) leaves most
// SMs idle during the second, partial wave.
template <typename K> static int resident_grid(K kernel, int64_t items) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kThreads, 0) != cudaSuccess || per_sm < 1) per_sm = 4;
    int64_t need = (items + kThreads - 1) / kThreads;
    int64_t cap = (int64_t)per_sm * kNumSMs;
    return (int)(need < 1 ? 1 : (need < cap ? need : cap));
}

extern "C" int toda_bn_apply(const float *y, int n, int c, const float *scale, const float *shift, const float *residual,
                             int relu, float *a, void *a_bf16, void *stream) {
    TODA_CHECK_ARG(n >= 0 && c > 0, "bn_apply: bad sizes");
    if (n == 0) return TODA_OK;
    TODA_CHECK_ARG(y && scale && shift && a, "bn_apply: null pointer");
    long long total = (long long)n * c;
    cudaStream_t st = (cudaStream_t)stream;
    static int per_sm_vec = 0, per_sm_scalar = 0;     // resident CTAs per SM of the two variants (queried once)
    if (!per_sm_vec) {
        per_sm_vec = resident_grid(bn_apply_kernel<true>, (int64_t)1 << 40) / kNumSMs;
        per_sm_scalar = resident_grid(bn_apply_kernel<false>, (int64_t)1 << 40) / kNumSMs;
    }
    auto grid_for = [](int64_t items, int per_sm) {
        int64_t need = (items + kThreads - 1) / kThreads, cap = (int64_t)per_sm * kNumSMs;
        return (int)(need < 1 ? 1 : (need < cap ? need : cap));
    };
    if (c % 4 == 0)
        bn_apply_kernel<true><<<grid_for(total / 4, per_sm_vec), kThreads, 0, st>>>(y, total, c, scale, shift, residual, relu, a, (__nv_bfloat16 *)a_bf16);
    else
        bn_apply_kernel<false><<<grid_for(total, per_sm_scalar), kThreads, 0, st>>>(y, total, c, scale, shift, residual, relu, a, (__nv_bfloat16 *)a_bf16);
    TODA_LAUNCH_OK();
    return TODA_OK;
}

extern "C" int toda_bn_apply_sums(const float *y, int n, int c, const double *sums, const float *gamma, const float *beta, float eps,
                                  float momentum, float *running_mean, float *running_var, float *scale, float *shift,
                                  float *save_mean, float *save_rstd, const float *residual, int relu, float *a, void *a_bf16,
                                  void *stream) {
    TODA_CHECK_ARG(n >= 0 && c > 0 && sums && scale && shift, "bn_apply_sums: bad args");
    cudaStream_t st = (cudaStream_t)stream;
    // the fused kernel needs a thread to keep its four channels over the grid stride; other shapes (none in these backbones)
    // and empty inputs (coefficients only: the running statistics are left unchanged) take the two-launch route
    if (n == 0 || c % 4 != 0 || kThreads % (c / 4) != 0) {
        int rc = toda_bn_finalize_sums(sums, n, c, gamma, beta, eps, momentum, running_mean, running_var, scale, shift, save_mean,
                                       save_rstd, stream);
        if (rc) return rc;
        return toda_bn_apply(y, n, c, scale, shift, residual, relu, a, a_bf16, stream);
    }
    TODA_CHECK_ARG(y && a, "bn_apply_sums: null pointer");
    const long long total = (long long)n * c;
    static int per_sm = 0;
    if (!per_sm) per_sm = resident_grid(bn_apply_sums_kernel, (int64_t)1 << 40) / kNumSMs;
    const int64_t need = (total / 4 + kThreads - 1) / kThreads, cap = (int64_t)per_sm * kNumSMs;
    const int grid = (int)(need < 1 ? 1 : (need < cap ? need : cap));
    bn_apply_sums_kernel<<<grid, kThreads, 0, st>>>(y, total, c, n, sums, gamma, beta, eps, momentum, running_mean, running_var, scale,
                                                    shift, save_mean, save_rstd, residual, relu, a, (__nv_bfloat16 *)a_bf16);
    TODA_LAUNCH_OK();
    return TODA_OK;
}

// The streaming pass of the BatchNorm backward (bn_bwd_apply_kernel) over n > 0 rows.  GLOBAL: the reductions and the
// count come from device memory (fp64, all-reduced over the processes of a synchronized BatchNorm) instead of `fsums`/`n`.
template <bool GLOBAL>
static void launch_bn_bwd_apply(const float *da, const float *a, const float *y, int n, int c, const float *gamma,
                                const float *save_mean, const float *save_rstd, const float *fsums, const double *gsums,
                                const double *gcount, int relu, int training, float *dy, float *dresidual, void *dy_bf16,
                                cudaStream_t st) {
    long long total = (long long)n * c;
    static int per_sm_vec = 0, per_sm_scalar = 0;
    if (!per_sm_vec) {
        per_sm_vec = resident_grid(bn_bwd_apply_kernel<true, GLOBAL>, (int64_t)1 << 40) / kNumSMs;
        per_sm_scalar = resident_grid(bn_bwd_apply_kernel<false, GLOBAL>, (int64_t)1 << 40) / kNumSMs;
    }
    auto grid_for = [](int64_t items, int per_sm) {
        int64_t need = (items + kThreads - 1) / kThreads, cap = (int64_t)per_sm * kNumSMs;
        return (int)(need < 1 ? 1 : (need < cap ? need : cap));
    };
    if (c % 4 == 0 && kThreads % (c / 4) == 0)   // grid*block is then a multiple of c/4: a thread keeps its 4 channels
        bn_bwd_apply_kernel<true, GLOBAL><<<grid_for(total / 4, per_sm_vec), kThreads, 0, st>>>(
            da, a, y, total, c, n, gamma, save_mean, save_rstd, fsums, gsums, gcount, relu, training, dy, dresidual,
            (__nv_bfloat16 *)dy_bf16);
    else
        bn_bwd_apply_kernel<false, GLOBAL><<<grid_for(total, per_sm_scalar), kThreads, 0, st>>>(
            da, a, y, total, c, n, gamma, save_mean, save_rstd, fsums, gsums, gcount, relu, training, dy, dresidual,
            (__nv_bfloat16 *)dy_bf16);
}

extern "C" int toda_bn_bwd(const float *da, const float *a, const float *y, int n, int c, const float *gamma,
                           const float *save_mean, const float *save_rstd, int relu, int training, float *dy, void *dy_bf16,
                           float *dresidual, float *dgamma, float *dbeta, void *workspace, size_t workspace_bytes, void *stream) {
    TODA_CHECK_ARG(n >= 0 && c > 0 && c <= 256, "bn_bwd: unsupported sizes n=%d c=%d", n, c);
    // dy may be NULL when dy_bf16 is given: the fp32 gradient is then not stored (a caller whose consumers -- tensor-core
    // dgrad and wgrad -- only read the bf16 copy saves 4 of the ~30 bytes per element this pass moves)
    TODA_CHECK_ARG(save_mean && save_rstd && workspace && (n == 0 || (da && y && (dy || dy_bf16))) && (!relu || a || n == 0),
                   "bn_bwd: null pointer");
    if (workspace_bytes < bn_ws_bytes(c)) { toda_set_error("bn_bwd: workspace too small"); return TODA_ERR_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    double *partial = (double *)workspace;
    float *sums = (float *)((char *)workspace + (size_t)kPartials * 2 * c * sizeof(double));
    launch_col_reduce<1>(da, a, y, n, c, save_mean, save_rstd, relu, partial, st);
    TODA_LAUNCH_OK();
    bn_bwd_finalize_kernel<float><<<ceil_div(c * 32, 128), 128, 0, st>>>(partial, kPartials, c, dgamma, dbeta, sums);
    TODA_LAUNCH_OK();
    if (n > 0) {
        launch_bn_bwd_apply<false>(da, a, y, n, c, gamma, save_mean, save_rstd, sums, nullptr, nullptr, relu, training, dy,
                                   dresidual, dy_bf16, st);
        TODA_LAUNCH_OK();
    }
    return TODA_OK;
}

// ---- BatchNorm over a batch split across processes (torch.nn.SyncBatchNorm): each phase that needs the other ranks'
// statistics is split at the all-reduce.  Forward: toda_bn_local_sums -> all-reduce SUM -> toda_bn_apply_global.
// Backward: toda_bn_bwd_reduce -> all-reduce SUM -> toda_bn_bwd_finish.  Given its own local buffers unreduced, each
// pair computes exactly what the single-process call computes (toda_bn_stats + toda_bn_apply / toda_bn_apply_sums,
// toda_bn_bwd), bit for bit.

extern "C" int toda_bn_local_sums(const float *y, const double *epilogue_sums, int n, int c, double *local_sums, void *workspace,
                                  size_t workspace_bytes, void *stream) {
    TODA_CHECK_ARG(n >= 0 && c > 0 && c <= 256 && local_sums, "bn_local_sums: bad args n=%d c=%d", n, c);
    cudaStream_t st = (cudaStream_t)stream;
    const double *partial = nullptr;
    if (n > 0 && !epilogue_sums) {
        TODA_CHECK_ARG(y && workspace, "bn_local_sums: null pointer");
        if (workspace_bytes < bn_ws_bytes(c)) { toda_set_error("bn_local_sums: workspace too small"); return TODA_ERR_WORKSPACE; }
        launch_col_reduce<0>(y, nullptr, nullptr, n, c, nullptr, nullptr, 0, (double *)workspace, st);
        TODA_LAUNCH_OK();
        partial = (const double *)workspace;
    }
    bn_local_sums_kernel<<<ceil_div(c * 32, 128), 128, 0, st>>>(partial, kPartials, n > 0 ? epilogue_sums : nullptr, n, c,
                                                              local_sums);
    TODA_LAUNCH_OK();
    return TODA_OK;
}

extern "C" int toda_bn_apply_global(const float *y, int n, int c, const double *global_sums, const float *gamma, const float *beta,
                                    float eps, float momentum, float *running_mean, float *running_var, float *scale, float *shift,
                                    float *save_mean, float *save_rstd, const float *residual, int relu, float *a, void *a_bf16,
                                    void *stream) {
    TODA_CHECK_ARG(n >= 0 && c > 0 && c <= 256 && global_sums && scale && shift, "bn_apply_global: bad args");
    TODA_CHECK_ARG(n == 0 || (y && a), "bn_apply_global: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const long long total = (long long)n * c;
    static int per_sm_vec = 0, per_sm_scalar = 0;
    if (!per_sm_vec) {
        per_sm_vec = resident_grid(bn_apply_global_kernel<true>, (int64_t)1 << 40) / kNumSMs;
        per_sm_scalar = resident_grid(bn_apply_global_kernel<false>, (int64_t)1 << 40) / kNumSMs;
    }
    auto grid_for = [](int64_t items, int per_sm) {
        int64_t need = (items + kThreads - 1) / kThreads, cap = (int64_t)per_sm * kNumSMs;
        return (int)(need < 1 ? 1 : (need < cap ? need : cap));
    };
    if (c % 4 == 0)
        bn_apply_global_kernel<true><<<grid_for(total / 4, per_sm_vec), kThreads, 0, st>>>(
            y, total, c, global_sums, gamma, beta, eps, momentum, running_mean, running_var, scale, shift, save_mean, save_rstd,
            residual, relu, a, (__nv_bfloat16 *)a_bf16);
    else
        bn_apply_global_kernel<false><<<grid_for(total, per_sm_scalar), kThreads, 0, st>>>(
            y, total, c, global_sums, gamma, beta, eps, momentum, running_mean, running_var, scale, shift, save_mean, save_rstd,
            residual, relu, a, (__nv_bfloat16 *)a_bf16);
    TODA_LAUNCH_OK();
    return TODA_OK;
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
    bn_bwd_finalize_kernel<double><<<ceil_div(c * 32, 128), 128, 0, st>>>(partial, kPartials, c, dgamma, dbeta, local_red);
    TODA_LAUNCH_OK();
    return TODA_OK;
}

extern "C" int toda_bn_bwd_finish(const float *da, const float *a, const float *y, int n, int c, const float *gamma,
                                  const float *save_mean, const float *save_rstd, int relu, const double *global_red,
                                  const double *global_count, float *dy, void *dy_bf16, float *dresidual, void *stream) {
    TODA_CHECK_ARG(n >= 0 && c > 0 && c <= 256, "bn_bwd_finish: unsupported sizes n=%d c=%d", n, c);
    TODA_CHECK_ARG(save_mean && save_rstd && global_red && global_count && (n == 0 || (da && y && (dy || dy_bf16))) &&
                   (!relu || a || n == 0), "bn_bwd_finish: null pointer");
    if (n == 0) return TODA_OK;
    launch_bn_bwd_apply<true>(da, a, y, n, c, gamma, save_mean, save_rstd, nullptr, global_red, global_count, relu, 1, dy,
                              dresidual, dy_bf16, (cudaStream_t)stream);
    TODA_LAUNCH_OK();
    return TODA_OK;
}

extern "C" int toda_col_sum(const float *dy, int n, int c, float *out, void *workspace, size_t workspace_bytes, void *stream) {
    TODA_CHECK_ARG(n >= 0 && c > 0 && c <= 256 && out && workspace, "col_sum: bad args");
    if (workspace_bytes < bn_ws_bytes(c)) { toda_set_error("col_sum: workspace too small"); return TODA_ERR_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    double *partial = (double *)workspace;
    launch_col_reduce<2>(dy, nullptr, nullptr, n, c, nullptr, nullptr, 0, partial, st);
    TODA_LAUNCH_OK();
    col_sum_finalize_kernel<<<ceil_div(c * 32, 128), 128, 0, st>>>(partial, kPartials, c, out);
    TODA_LAUNCH_OK();
    return TODA_OK;
}
