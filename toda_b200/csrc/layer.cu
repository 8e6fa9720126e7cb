// One C-ABI call per backbone layer (and per layer backward): conv -> BatchNorm1d (+ residual) (+ ReLU), i.e. the unit
// `post_act_block` / `SparseBasicBlock` repeat 21 times (pcdet/models/backbones_3d/spconv_backbone.py L8-27, L30-66).
// The host side of a training step was ~9 ms of Python / ctypes / allocator work for ~10 ms of GPU work (VERDICT r01,
// weak #6): the same kernels, launched from here in sequence, cost the interpreter one call instead of three (forward) or
// four (backward).  No new device code: this file only sequences the entry points of conv_*.cu and bn.cu.
#include "common.cuh"

static int layer_conv(const toda_layer_fwd_args *p, double *bn_sums, void *stream) {
    return toda_spconv_fwd(p->x, p->x_bf16, p->n_in, p->cin, p->nbr, p->n_out, p->kvol, p->w, p->cout, p->bias, nullptr, p->y,
                           nullptr, p->tile_masks, p->plan_lidx, p->plan_rows, p->plan_cnt, p->plan_groups, p->plan_cap,
                           bn_sums, p->w_bf16, p->precision, p->conv_ws, p->conv_ws_bytes, stream);
}

// Training forward up to the BatchNorm's statistics: the convolution, then sum(y) | sum(y*y) of its output in `sums` (in
// tensor-core mode the convolution's epilogue accumulates them straight into the buffer) and the row count in `count`
// when given.
static int layer_fwd_stats(const toda_layer_fwd_args *p, double *sums, double *count, void *stream) {
    const int c = p->cout, n = p->n_out;
    const bool tc = n > 0 && toda_spconv_uses_tensor_cores(p->cin, c, p->kvol, p->precision);
    int rc = layer_conv(p, tc ? sums : nullptr, stream);
    if (rc) return rc;
    return toda_bn_local_sums(p->y, tc ? sums : nullptr, n, c, sums, count, p->bn_ws, p->bn_ws_bytes, stream);
}

// The BatchNorm (+ residual) (+ ReLU) from the batch's sums and row count (`count`, or n_out when NULL): coefficients,
// save_mean / save_rstd and running statistics are derived and applied in one launch.
static int layer_fwd_apply(const toda_layer_fwd_args *p, const double *sums, const double *count, void *stream) {
    const int c = p->cout;
    float *scale = p->stats, *shift = p->stats + c, *mean = p->stats + 2 * c, *rstd = p->stats + 3 * c;
    return toda_bn_apply_sums(p->y, p->n_out, c, sums, count, p->gamma, p->beta, p->eps, p->momentum, p->running_mean,
                              p->running_var, scale, shift, mean, rstd, p->residual, p->relu, p->a, p->a_bf16, stream);
}

extern "C" int toda_layer_fwd(const toda_layer_fwd_args *p, void *stream) {
    TODA_CHECK_ARG(p, "layer_fwd: null args");
    const int c = p->cout, n = p->n_out;
    // an empty tensor's storage pointer is NULL: y and a are only required when there are rows to write
    TODA_CHECK_ARG(c > 0 && n >= 0 && p->stats && (n == 0 || (p->y && p->a)) && (!p->training || p->sums),
                   "layer_fwd: bad sizes / null outputs");
    if (n == 0) return layer_conv(p, nullptr, stream);   // no rows, running statistics unchanged (as torch.nn.BatchNorm1d)
    int rc;
    if (p->training) {
        rc = layer_fwd_stats(p, p->sums, nullptr, stream);
        return rc ? rc : layer_fwd_apply(p, p->sums, nullptr, stream);
    }
    float *scale = p->stats, *shift = p->stats + c;
    if ((rc = layer_conv(p, nullptr, stream))) return rc;
    if ((rc = toda_bn_eval_coeffs(p->gamma, p->beta, p->running_mean, p->running_var, p->eps, c, scale, shift, stream))) return rc;
    return toda_bn_apply(p->y, n, c, scale, shift, p->residual, p->relu, p->a, p->a_bf16, stream);
}

// Backward of an empty layer: zero parameter gradients (BatchNorm's too when `bn_grads`), dx = the residual-branch addend.
static int layer_bwd_empty(const toda_layer_bwd_args *p, bool bn_grads, cudaStream_t st) {
    const int c = p->cout;
    if (bn_grads && p->dgamma) TODA_CUDA_OK(cudaMemsetAsync(p->dgamma, 0, sizeof(float) * c, st));
    if (bn_grads && p->dbeta) TODA_CUDA_OK(cudaMemsetAsync(p->dbeta, 0, sizeof(float) * c, st));
    if (p->need_db && p->db) TODA_CUDA_OK(cudaMemsetAsync(p->db, 0, sizeof(float) * c, st));
    if (p->need_dw && p->dw) TODA_CUDA_OK(cudaMemsetAsync(p->dw, 0, sizeof(float) * (size_t)p->kvol * p->cin * c, st));
    if (p->need_dx && p->dx && p->n_in > 0) {
        if (p->addend) TODA_CUDA_OK(cudaMemcpyAsync(p->dx, p->addend, sizeof(float) * (size_t)p->n_in * p->cin, cudaMemcpyDeviceToDevice, st));
        else TODA_CUDA_OK(cudaMemsetAsync(p->dx, 0, sizeof(float) * (size_t)p->n_in * p->cin, st));
    }
    return TODA_OK;
}

// The fp32 copy of the gradient between BatchNorm and the convolution is only written when something reads it: the
// tensor-core dgrad / wgrad take the bf16 copy the same pass writes (4 of ~30 bytes per element of this HBM-bound pass),
// and the bias gradient is summed by that pass itself.
static bool layer_bwd_reads_dy_f32(const toda_layer_bwd_args *p) {
    const int c = p->cout;
    return !p->dy_bf16 || p->precision != TODA_CONV_BF16 ||
           (p->need_dx && !toda_spconv_uses_tensor_cores(c, p->cin, p->kvol, p->precision)) ||
           (p->need_dw && !toda_spconv_wgrad_uses_tensor_cores(p->cin, c, p->kvol, p->precision));
}

// The convolution's part of the layer backward, from dy: dgrad (+ residual-branch addend), wgrad.
static int layer_bwd_conv(const toda_layer_bwd_args *p, void *stream) {
    const int c = p->cout, n = p->n_out;
    int rc;
    if (p->need_dx) {
        // dgrad = the forward kernel on the input-stationary table with transposed (SubM: mirrored) weights; `addend` is the
        // gradient that reaches the same tensor through the block's residual branch (spconv_backbone.py L63)
        rc = toda_spconv_fwd(p->dy, p->dy_bf16, n, c, p->dgrad_nbr, p->n_in, p->kvol, p->wt, p->cin, nullptr, p->addend, p->dx,
                             p->dgrad_out_rows, p->dgrad_masks, p->dplan_lidx, p->dplan_rows, p->dplan_cnt, p->dplan_groups,
                             p->dplan_cap, nullptr, p->wt_bf16, p->precision, p->conv_ws, p->conv_ws_bytes, stream);
        if (rc) return rc;
    }
    if (p->need_dw) {
        rc = toda_spconv_wgrad(p->x, p->x_bf16, p->n_in, p->cin, p->nbr_fwd, n, p->kvol, p->fwd_masks, p->dy, p->dy_bf16, c, p->dw,
                               p->wgrad_ws, p->wgrad_ws_bytes, p->precision, stream);
        if (rc) return rc;
    }
    return TODA_OK;
}

static int layer_bwd_reduce(const toda_layer_bwd_args *p, double *red, void *stream) {
    return toda_bn_bwd_reduce(p->da, p->a_mask, p->y, p->n_out, p->cout, p->mean, p->rstd, p->relu, red, p->dgamma, p->dbeta,
                              p->bn_ws, p->bn_ws_bytes, stream);
}

// The layer backward from the BatchNorm's reduced sums on: dy (+ dres, + the bias gradient) from `red` and the row count
// (`count`, or n_out when NULL), then the convolution's part.
static int layer_bwd_finish(const toda_layer_bwd_args *p, const double *red, const double *count, void *stream) {
    const int c = p->cout, n = p->n_out;
    if (n == 0) return layer_bwd_empty(p, false, (cudaStream_t)stream);   // dgamma / dbeta: written by the reduce phase
    int rc = toda_bn_bwd_finish(p->da, p->a_mask, p->y, n, c, p->gamma, p->mean, p->rstd, p->relu, p->training, red, count,
                                layer_bwd_reads_dy_f32(p) ? p->dy : nullptr, p->dy_bf16, p->dres, p->need_db ? p->db : nullptr,
                                p->bn_ws, p->bn_ws_bytes, stream);
    return rc ? rc : layer_bwd_conv(p, stream);
}

extern "C" int toda_layer_bwd(const toda_layer_bwd_args *p, void *stream) {
    TODA_CHECK_ARG(p, "layer_bwd: null args");
    TODA_CHECK_ARG(p->cout > 0 && p->n_out >= 0, "layer_bwd: bad sizes");
    if (p->n_out == 0) return layer_bwd_empty(p, true, (cudaStream_t)stream);
    TODA_CHECK_ARG(p->bn_ws, "layer_bwd: null workspace");
    double *red = bn_workspace_red(p->bn_ws, p->cout);
    int rc = layer_bwd_reduce(p, red, stream);
    return rc ? rc : layer_bwd_finish(p, red, nullptr, stream);
}

// ---- The same layer with its BatchNorm synchronized over several processes (torch.nn.SyncBatchNorm): each direction is
// split at its all-reduce (include/toda_b200.h).  Training mode only; eval mode needs no exchange.

extern "C" int toda_layer_fwd_stats(const toda_layer_fwd_args *p, double *local_sums, void *stream) {
    TODA_CHECK_ARG(p && local_sums, "layer_fwd_stats: null args");
    const int c = p->cout, n = p->n_out;
    TODA_CHECK_ARG(c > 0 && n >= 0 && p->training && (n == 0 || p->y), "layer_fwd_stats: bad sizes / not training / null y");
    return layer_fwd_stats(p, local_sums, local_sums + 2 * c, stream);
}

extern "C" int toda_layer_fwd_apply(const toda_layer_fwd_args *p, const double *global_sums, void *stream) {
    TODA_CHECK_ARG(p && global_sums, "layer_fwd_apply: null args");
    const int c = p->cout, n = p->n_out;
    TODA_CHECK_ARG(c > 0 && n >= 0 && p->training && p->stats && (n == 0 || (p->y && p->a)),
                   "layer_fwd_apply: bad sizes / not training / null outputs");
    return layer_fwd_apply(p, global_sums, global_sums + 2 * c, stream);
}

extern "C" int toda_layer_bwd_reduce(const toda_layer_bwd_args *p, double *local_red, void *stream) {
    TODA_CHECK_ARG(p && local_red, "layer_bwd_reduce: null args");
    TODA_CHECK_ARG(p->cout > 0 && p->n_out >= 0 && p->training, "layer_bwd_reduce: bad sizes / not training");
    return layer_bwd_reduce(p, local_red, stream);
}

extern "C" int toda_layer_bwd_finish(const toda_layer_bwd_args *p, const double *global_red, const double *global_count,
                                     void *stream) {
    TODA_CHECK_ARG(p && global_red && global_count, "layer_bwd_finish: null args");
    TODA_CHECK_ARG(p->cout > 0 && p->n_out >= 0 && p->training, "layer_bwd_finish: bad sizes / not training");
    return layer_bwd_finish(p, global_red, global_count, stream);
}
