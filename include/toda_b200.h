/*
 * toda_b200.h -- C ABI of libtoda_b200.so: the B200 (sm_100a) implementation of TODA's
 * data-parallel LiDAR hot path (SURVEY.md section 8).
 *
 * Conventions (SURVEY.md section 8b, row "C-ABI"):
 *   - extern "C", plain pointers + sizes, no torch types.
 *   - every pointer is a DEVICE pointer unless the parameter name ends in `_host`.
 *   - no allocation or ownership inside the library: the caller (PyTorch on the host side)
 *     allocates inputs, outputs and workspaces; `*_bytes()` functions size the workspaces.
 *   - every entry point enqueues work on `stream` (a cudaStream_t passed as void*) and
 *     returns without synchronising.
 *   - return value: 0 = TODA_OK, negative = error; the message is in toda_last_error()
 *     (thread-local).  There is no CPU fallback: without a CUDA device every call fails.
 *   - entry points are re-entrant and stateless (state = caller-owned buffers).
 *
 * Each function cites the reference interface it replaces (file:line in rasd3/TODA).
 */
#ifndef TODA_B200_H
#define TODA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TODA_OK 0
#define TODA_ERR_INVALID (-1)
#define TODA_ERR_CUDA (-2)
#define TODA_ERR_WORKSPACE (-3)
#define TODA_ERR_UNSUPPORTED (-4)

#define TODA_ORDER_FIRST_APPEARANCE 0 /* voxel rows in the reference's order (order of first point) */
#define TODA_ORDER_CANONICAL 1        /* voxel rows sorted by (b,z,y,x) */

const char *toda_last_error(void);
int toda_version(void);
/* number of kernels this library has launched in the calling process (bench.py reports the per-run delta as gpu_launches) */
long long toda_launch_count(void);
/* number of SMs / compute capability of the current device; fails when there is no CUDA device. */
int toda_device_info(int *sm_count_host, int *cc_major_host, int *cc_minor_host);

/* ------------------------------------------------------------------------------------------
 * Occupancy index: a two-level bitmap over the (batch, D, H, W) cell grid plus per-word ranks.
 * It is the "hash table" of this implementation: a perfect (collision-free) hash whose
 * enumeration order IS the canonical (b,z,y,x) order, so dedup, canonical sort and
 * coordinate -> row lookup are one structure.  Replaces the hash tables inside the un-vendored
 * spconv package (call sites: pcdet/models/backbones_3d/spconv_backbone.py L141-146, L254-259).
 * The buffer must be all-zero before the first insert; toda_index_release() re-zeroes exactly
 * the words that inserts touched, so a buffer can be reused without a full memset.
 * ------------------------------------------------------------------------------------------ */
size_t toda_index_bytes(int batch, int D, int H, int W);
/* mark coords[n,4] = (b,z,y,x) int32 */
int toda_index_insert(void *index, int batch, int D, int H, int W, const int32_t *coords, int n, void *stream);
/* mark every output cell reachable from in_coords under a conv (k,s,p): o*s = p_in + pad - k */
int toda_index_insert_strided(void *index_out, int batch, int oD, int oH, int oW, const int32_t *in_coords, int n_in,
                              const int *ksize_host, const int *stride_host, const int *pad_host, void *stream);
/* ranks every marked cell; writes the sorted coordinate list (up to `cap` rows) and the number of
 * marked cells to n_out[0] (device int32).  per-frame counts go to n_out[1..batch]. */
int toda_index_build(void *index, int batch, int D, int H, int W, int32_t *out_coords, int cap, int32_t *n_out,
                     void *stream);
/* rows[i] = canonical row of coords[i], or -1 */
int toda_index_rows(const void *index, int batch, int D, int H, int W, const int32_t *coords, int n, int32_t *rows,
                    void *stream);
int toda_index_release(void *index, int batch, int D, int H, int W, const int32_t *coords, int n, void *stream);

/* ------------------------------------------------------------------------------------------
 * K0 point-stream selection (order-preserving compaction under a per-point predicate).  Replaces, for the points of a
 * whole batch of frames in one call, the boolean-mask indexing of
 *   mode TODA_SELECT_RANGE_XY  common_utils.mask_points_by_range (pcdet/utils/common_utils.py L60-63) as used by
 *        DataProcessor.mask_points_and_boxes_outside_range (data_processor.py L78-91): lo <= x,y <= hi, no z test;
 *        params_host = {lo_x, lo_y, hi_x, hi_y} (compared in float32, as the reference's float32 range array is)
 *   mode TODA_SELECT_RECT_XY   the crop of inter_domain_point_cutmix (inter_domain_point_cutmix.py L45-55): strict
 *        min < x,y < max with float64 thresholds; params_host = {min_x, min_y, max_x, max_y}
 *   mode TODA_SELECT_SECTOR    the sector of PolarMix swap / swap_with_range (inter_domain_point_polarmix.py L76-80,
 *        L103-119): start < -arctan2(y,x) < end in float32; params_host = {start, end, dis_th, dis_mode} with
 *        dis_mode 0 = no distance test, 1 = also sqrt(x^2+y^2) < dis_th, 2 = also > dis_th
 *   mode TODA_SELECT_BOXES     augmentor_utils.get_points_in_box (pcdet/datasets/augmentor/augmentor_utils.py L474-491)
 *        OR-ed over M <= 96 boxes: the point is rotated by -rz about the box centre; |z - cz| <= dz/2 and
 *        |local x|, |local y| <= half size + margin, all in float32 as numpy evaluates it; with invert != 0 this is the
 *        point filter of intra_domain_point_mixup_cd (intra_domain_point_mixup.py L50-59).  Needs a z column (x_col + 2).
 *        params_host = {M, margin, M x (cx, cy, cz, dx, dy, dz, rz)}
 * invert != 0 keeps the complement (np.delete / ~mask).  Kept rows keep their input order (what numpy's mask indexing
 * gives).  add_batch_col != 0 prepends the frame index as a float column (collate_batch, dataset.py L173-178), so raw
 * (N,F) frames can be shipped and collated on the device.
 *   points [n][stride] fp32, x at column x_col and y at x_col+1; frame_offsets int32[batch+1] device or NULL
 *   out [>= n][stride + (add_batch_col?1:0)]; out_offsets int32[batch+1] device (kept rows before each frame start,
 *   last entry = total kept) or int32[1] = total when frame_offsets is NULL.
 * ------------------------------------------------------------------------------------------ */
#define TODA_SELECT_RANGE_XY 0
#define TODA_SELECT_RECT_XY 1
#define TODA_SELECT_SECTOR 2
#define TODA_SELECT_BOXES 3   /* params = [M, margin, M x (cx,cy,cz,dx,dy,dz,rz)]: inside ANY box (augmentor_utils.py L474-491), M <= 96 */
size_t toda_points_select_workspace_bytes(int n);
int toda_points_select(const float *points, int n, int stride, int x_col, const int32_t *frame_offsets, int batch, int mode,
                       const double *params_host, int invert, int add_batch_col, float *out, int32_t *out_offsets,
                       void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------
 * K0 world augmentations: the point side of DataAugmentor.random_world_flip / random_world_rotation /
 * random_world_scaling (pcdet/datasets/augmentor/data_augmentor.py L43-80, augmentor_utils.py L8-82; OpenPCDet v0.5.2)
 * for a whole batch of frames in one elementwise launch.  The random draws are made on the host; each step carries
 * per-frame parameters, params_host[(step * nb + b) * 2 + {0, 1}] with nb = batch (1 when frame_offsets is NULL):
 *   TODA_WORLD_FLIP_X  {enabled, -}: negate y (random_flip_along_x)     TODA_WORLD_FLIP_Y  {enabled, -}: negate x
 *   TODA_WORLD_ROTATE  {cos, sin}: common_utils.rotate_points_along_z with cos / sin of the float32 angle as torch.cos /
 *        torch.sin give them; the product is rounded as torch.matmul on the CPU rounds it, which depends on the frame's
 *        row count off[b+1] - off[b]: unfused products and sums from a zero accumulator for <= 44 rows (ATen's naive bmm),
 *        a chain of fmas for >= 45 (BLAS).  The 0 and 1 entries of the rotation matrix take part in both.
 *   TODA_WORLD_SCALE   {noise, -}: points[:, :3] *= noise, i.e. x * float32(noise)
 * Steps apply in list order (n_steps <= 4), float32 op by op, so the result is bit-identical to the reference's.  A
 * scaling step whose range is narrower than 1e-3 draws nothing in the reference and is left out of the list.
 *   points [n][stride] fp32, x, y, z at columns x_col..x_col+2; frame_offsets int32[batch+1] device or NULL (one frame),
 *   batch <= 64; out [n][stride]: every other column copied bit for bit.  No workspace, deterministic.
 * ------------------------------------------------------------------------------------------ */
#define TODA_WORLD_FLIP_X 0
#define TODA_WORLD_FLIP_Y 1
#define TODA_WORLD_ROTATE 2
#define TODA_WORLD_SCALE 3
int toda_points_world_transform(const float *points, int n, int stride, int x_col, const int32_t *frame_offsets, int batch,
                                int n_steps, const int *kinds_host, const float *params_host, float *out, void *stream);

/* ------------------------------------------------------------------------------------------
 * K0 gt_sampling: the device side of DataBaseSampler.__call__ / add_sampled_boxes_to_scene
 * (pcdet/datasets/augmentor/database_sampler.py; OpenPCDet v0.5.2) for a whole batch of frames.  The database samples
 * are drawn on the host; the collision test, the scene-point removal and the paste run on `stream` in four launches
 * without a host synchronisation.
 *
 * toda_gt_sampling_pack_boxes (host only): boxes_host float32 [n][7] (x, y, z, dx, dy, dz, heading) ->
 * packed_host float32 [n][16] = {x, y, z, dx, dy, dz, cosf(h), sinf(h), cosf(-h), sinf(-h), dx + w0, dy + w1, dz + w2, 0,
 * 0, 0} with libm cosf / sinf (what the compiled ops iou3d_cpu.cpp / roiaware_pool3d.cpp evaluate) and the enlarged sizes
 * of box_utils.enlarge_box3d in float32 (w = extra_width_host[3], or 0 when it is NULL).
 *
 * toda_gt_sampling:
 *   points [n][stride] fp32 frames back to back, frame_offsets int32[batch+1] device, batch <= 64; x_col 0 (raw frames)
 *     or 1 (collated, column 0 = batch index); stride = x_col + db_features.
 *   exist_boxes packed [E][16]: every frame's unmasked gt_boxes, frame b at exist_offsets_host[b..b+1).
 *   samp_boxes packed [S][16] (enlarged by REMOVE_EXTRA_WIDTH): frame by frame, within a frame class by class in
 *     SAMPLE_GROUPS order; group_sizes_host[b * n_groups + g] samples of group g in frame b (n_groups <= 16, at most 1024
 *     samples per frame, else TODA_ERR_UNSUPPORTED).
 *   samp_rows int64 [S][2] (first row, row count) of each sample's object points in db_points [R][db_features];
 *   samp_shift float64 [S][3]: the database box centre box3d_lidar[:3]; shift_f64 != 0 when the database stores float64
 *     boxes (object xyz = float32(double(p) + c)), 0 for float32 boxes (float32 add).
 * A sample is accepted iff every iou_bev against the frame's gt boxes, the samples accepted for earlier classes and
 * the other samples of its class is exactly 0 (boxes_bev_iou_cpu, iou1.max + iou2.max == 0); accepted int32 [S] gets
 * 1 / 0.  Scene rows inside an accepted box (points_in_boxes_cpu with the enlarged box) are removed.  out [>= n + sum of
 * the sample row counts][stride]: frame b = the object rows of its accepted samples in sample order, xyz shifted by the box
 * centre (batch column = b when x_col == 1), then its kept scene rows in input order; out_offsets int32[batch+1].
 * Deterministic, no atomics.  The workspace is toda_gt_sampling_workspace_bytes(n, batch, S) bytes.
 * ------------------------------------------------------------------------------------------ */
int toda_gt_sampling_pack_boxes(const float *boxes_host, int n, const float *extra_width_host, float *packed_host);
size_t toda_gt_sampling_workspace_bytes(int n, int batch, int n_samples);
int toda_gt_sampling(const float *points, int n, int stride, int x_col, const int32_t *frame_offsets, int batch,
                     const float *exist_boxes, const int *exist_offsets_host, const float *samp_boxes, const int *group_sizes_host,
                     int n_groups, const float *db_points, int db_features, const int64_t *samp_rows, const double *samp_shift,
                     int shift_f64, float *out, int32_t *out_offsets, int32_t *accepted, void *workspace, size_t workspace_bytes,
                     void *stream);

/* ------------------------------------------------------------------------------------------
 * K1 hard voxelizer.  Replaces spconv.utils.Point2VoxelCPU3d.point_to_voxel as called from
 * pcdet/datasets/processor/data_processor.py L36-42, L54 (VoxelGeneratorWrapper) /
 * L115-143 (transform_points_to_voxels), for a whole batch of frames in one call.
 *   points: row i = point_stride floats; x,y,z at columns xyz_col..xyz_col+2; the num_features
 *           columns starting at feat_col are copied into `voxels`.  (collated `points` of
 *           pcdet/datasets/dataset.py L173-178: stride 1+F, xyz_col = feat_col = 1.)
 *   frame_offsets: int32[batch+1], points of frame b are rows [off[b], off[b+1]).
 *   range_host[6] = xmin,ymin,zmin,xmax,ymax,zmax; vsize_host[3] = x,y,z; grid_host[3] = x,y,z
 *           (= round((hi-lo)/vsize), data_processor.py L117-118).
 * Semantics = spconv 2.x loop (SURVEY.md Appendix C.1): c = floor((p-lo)/vsize) in fp32 with true
 * division; a point outside [0,grid) on any axis is dropped; voxels are numbered in order of first
 * appearance; once max_voxels exist in a frame, points of further voxels are dropped; the first
 * max_points points (input order) of a voxel are kept.
 * Outputs (capacity batch*max_voxels rows, frames packed back to back as np.concatenate does in
 * dataset.py L171-178): voxels [V,max_points,F] zero padded, coords [V,4] = (b,z,y,x),
 * num_points [V]; voxel_counts int32[batch+1] = per-frame V_b then the total V.
 * ------------------------------------------------------------------------------------------ */
size_t toda_voxelize_workspace_bytes(int64_t n_points, int batch, const int *grid_host, int max_points,
                                     int max_voxels);
int toda_voxelize_hard(const float *points, int64_t n_points, int point_stride, int xyz_col, int feat_col,
                       int num_features, const int32_t *frame_offsets, int batch, const float *range_host,
                       const float *vsize_host, const int *grid_host, int max_points, int max_voxels, int order,
                       float *voxels, int32_t *coords, int32_t *num_points, int32_t *voxel_counts, void *workspace,
                       size_t workspace_bytes, void *stream);

/* K2 MeanVFE.  pcdet/models/backbones_3d/vfe/mean_vfe.py L25-29: sum over all K slots / max(num,1).
 * num_points is int32 when num_is_float == 0, float32 otherwise (load_data_to_gpu casts it,
 * pcdet/models/__init__.py L34). */
int toda_mean_vfe_fwd(const float *voxels, const void *num_points, int num_is_float, int n_voxels, int max_points,
                      int num_features, float *voxel_features, void *stream);
int toda_mean_vfe_bwd(const float *d_voxel_features, const void *num_points, int num_is_float, int n_voxels,
                      int max_points, int num_features, float *d_voxels, void *stream);

/* ------------------------------------------------------------------------------------------
 * K3 / K4 rulebooks, as neighbour tables: nbr[k*n_out + o] = input row paired with output row o
 * under kernel offset k = (kz*KH+ky)*KW+kx, or -1.  The pair list of spconv is the set of
 * non-negative entries.  coords must be in canonical order (toda_index_build output).
 *   SubMConv3d  (spconv_backbone.py L12, L38-45, L78, L192): outputs == inputs.
 *   SparseConv3d (L14-15, L90/97/104/113, L205/212/219/228): outputs from toda_index_insert_strided
 *   + toda_index_build; nbr_fwd[kvol,n_out] gathers inputs for each output, nbr_bwd[kvol,n_in]
 *   gives for each input the output it feeds under offset k (used by dgrad).
 * ------------------------------------------------------------------------------------------ */
int toda_rulebook_subm(const void *index, int batch, int D, int H, int W, const int32_t *coords, int n,
                       const int *ksize_host, int32_t *nbr, void *stream);
int toda_rulebook_sparse(const void *index_in, int iD, int iH, int iW, const void *index_out, int oD, int oH, int oW,
                         int batch, const int32_t *in_coords, int n_in, const int32_t *out_coords, int n_out,
                         const int *ksize_host, const int *stride_host, const int *pad_host, int32_t *nbr_fwd,
                         int32_t *nbr_bwd, void *stream);

/* Parity order of the input rows of a strided convolution: rows sorted by ((z+pz)%sz, (y+py)%sy, (x+px)%sx), canonical
 * order kept inside a class (stable, deterministic); order[i] = canonical row at sorted position i, pos_of_row (optional)
 * its inverse.  coords int32 (n,4) = (b,z,y,x).  At most 8 classes (strides <= 2).  Used by the dgrad of SparseConv3d
 * (see out_rows / tile_masks of toda_spconv_fwd). */
size_t toda_parity_order_workspace_bytes(int n);
int toda_parity_order(const int32_t *coords, int n, const int *stride_host, const int *pad_host, int32_t *order,
                      int32_t *pos_of_row, void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------
 * K5/K6/K7 sparse convolution on neighbour tables (every `conv(x)` in spconv_backbone.py).
 *   fwd :  y[o,:]  = bias + sum_k x[nbr[k,o],:] @ w[k]        w: [kvol, Cin, Cout]
 *   dgrad: the same entry point with dy as x, the transposed weights [kvol, Cout, Cin] and the
 *          input-stationary table (SubM: the same table with k mirrored -- toda_weight_repack does it;
 *          SparseConv3d: nbr_bwd).
 *   wgrad: dw[k] = sum_o x[nbr[k,o],:]^T @ dy[o,:], written in the parameter layout
 *          (Cout, kvol, Cin) of spconv 2.x, which pcdet/models/detectors/detector3d_template.py
 *          L341-348 accepts.
 * precision: TODA_CONV_FP32 = fp32 FFMA (parity path, rtol 1e-4 vs the oracle);
 *            TODA_CONV_BF16 = bf16 operands, fp32 accumulate on tcgen05 tensor cores.
 *            TODA_CONV_BF16X3 = the same tensor-core kernels at fp32-class accuracy: every operand is split into two
 *            bf16 terms and each product is three launches (hi*hi + hi*lo + lo*hi, ~2^-16 relative; x_bf16 / dy_bf16 /
 *            w_bf16 are ignored: the kernels split the fp32 tensors themselves). */
#define TODA_CONV_FP32 0
#define TODA_CONV_BF16 1
#define TODA_CONV_BF16X3 2
/* param (Cout,kvol,Cin) -> [kvol,Cin,Cout] (transpose=0) or [kvol,Cout,Cin] with optional k mirroring */
int toda_weight_repack(const float *w_param, int kvol, int cin, int cout, int transpose, int mirror_k, float *w_out,
                       void *stream);
size_t toda_spconv_fwd_workspace_bytes(int n_in, int cin, int cout, int kvol, int precision);
/* tile_masks: uint32[ceil(n_out/128)], bit k set when some row of that 128-row tile has a neighbour under offset k. */
int toda_table_tile_masks(const int32_t *nbr, int n_out, int kvol, uint32_t *masks, void *stream);
int toda_spconv_uses_tensor_cores(int cin, int cout, int kvol, int precision);
/* the same question for toda_spconv_wgrad */
int toda_spconv_wgrad_uses_tensor_cores(int cin, int cout, int kvol, int precision);
/* Tile plan (row cache of the TODA_CONV_BF16 kernel): for every 128-row tile of a neighbour table and every group of
 * kvol/ngroups consecutive offsets (ngroups = kz: the neighbours of one group lie in one z plane), the ascending list of
 * DISTINCT input rows the tile gathers (`rows`: int32, `cap` entries reserved per (tile, group); `cnt`: int32 per
 * (tile, group), entries used) and the table rewritten as 16-bit slots into that list (`lidx`: uint16
 * [tiles][kvol][128]; 0xFFFF = no neighbour, 0xFFFE = not in the list, read the row through `nbr`).
 * cap = toda_tile_plan_capacity(channels of the gathered rows) (<= 512). */
int toda_tile_plan_capacity(int channels);
int toda_table_tile_plan(const int32_t *nbr, int n_out, int kvol, int ngroups, int cap, uint16_t *lidx, int32_t *rows,
                         int32_t *cnt, void *stream);
/* The convolution.  Every argument below is optional (NULL, or plan_lidx NULL for no plan):
 * x_bf16 / dy_bf16: an existing bf16 copy of x / dy ([rows][channels], same values rounded to nearest) that the
 *   TODA_CONV_BF16 kernels use instead of converting x / dy themselves.
 * addend: [n_out][cout] fp32, added to y in the epilogue (every kernel): the residual-branch gradient in
 *   SparseBasicBlock's backward, spconv_backbone.py L63.
 * out_rows: int32[n_out]; output row o of this call is written to y[out_rows[o], :] instead of y[o, :].  Used by the
 *   dgrad of strided convolutions: with stride s only the offsets k = (in + pad) mod s (per axis) can reach an input
 *   voxel, so its rows are processed in s_z*s_y*s_x parity classes, each with the compact table of its own 1..kvol
 *   offsets: the caller sorts the rows (and the table's columns) by class and they are scattered back to canonical rows
 *   here; with tile_masks the K blocks that are structurally empty for a class are skipped (in canonical order every
 *   tile mixes all classes and the [27] table is ~85 % structural padding).
 * tile_masks: the toda_table_tile_masks words of `nbr`; the tensor-core kernels then walk only the K blocks that hold
 *   data (the FFMA kernel tests this per tile itself).
 * plan_lidx / plan_rows / plan_cnt / plan_groups / plan_cap: a tile plan of `nbr` (toda_table_tile_plan).  With a plan
 *   the tensor-core convolution loads each distinct row once per tile into shared memory and feeds tcgen05.mma's A
 *   operand from tensor memory; the FFMA kernel ignores it.
 * bn_sums (tensor-core kernels only, see toda_spconv_uses_tensor_cores): double[2*cout] receiving sum(y) and sum(y*y)
 *   per output channel, accumulated in the epilogue, for toda_bn_apply_sums -- the BatchNorm that follows the
 *   convolution (spconv_backbone.py L23-24) then needs no statistics pass over y.
 * w_bf16: see toda_weight_kmajor_bf16. */
int toda_spconv_fwd(const float *x, const void *x_bf16, int n_in, int cin, const int32_t *nbr, int n_out, int kvol,
                    const float *w, int cout, const float *bias, const float *addend, float *y,
                    const int32_t *out_rows, const uint32_t *tile_masks, const uint16_t *plan_lidx,
                    const int32_t *plan_rows, const int32_t *plan_cnt, int plan_groups, int plan_cap, double *bn_sums,
                    const void *w_bf16, int precision, void *workspace, size_t workspace_bytes, void *stream);
/* w_bf16 (optional, may be NULL): the weights already converted for the tensor-core kernels by toda_weight_kmajor_bf16
 * ([cout][kvol*max(cin,16)] bf16), so that a caller that caches them per optimizer step saves the conversion per call. */
int toda_weight_kmajor_bf16(const float *w, int kvol, int cin, int cout, void *w_bf16, void *stream);
size_t toda_spconv_wgrad_workspace_bytes(int n_in, int n_out, int kvol, int cin, int cout, int precision);
/* tile_masks (optional, may be NULL): the toda_table_tile_masks words of `nbr`.  The tensor-core weight gradient then
 * skips, per 128-row tile, the groups of kernel offsets that have no neighbour there; NULL: every group is computed. */
int toda_spconv_wgrad(const float *x, const void *x_bf16, int n_in, int cin, const int32_t *nbr, int n_out, int kvol,
                      const uint32_t *tile_masks, const float *dy, const void *dy_bf16, int cout, float *dw_param,
                      void *workspace, size_t workspace_bytes, int precision, void *stream);
/* How the tensor-core weight gradient splits the rows of one call: it runs groups x splits CTAs (one offset group, one
 * row range each) and cuts each group's rows into `splits` ranges of whole row chunks (128 rows, 64 when cout = 128)
 * holding equal shares of the group's live (chunk, offset group) items, computed on the device from tile_masks (NULL:
 * every item live).  Writes *groups and *splits and, when row_begin (device int32[groups*splits]) is given, the first
 * row of every range at row_begin[group*splits + split] (a range ends where the next begins, the last at n_out). */
int toda_spconv_wgrad_row_splits(const uint32_t *tile_masks, int n_out, int kvol, int cin, int cout, int *groups,
                                 int *splits, int32_t *row_begin, void *stream);

/* ------------------------------------------------------------------------------------------
 * K8 BatchNorm1d(eps, momentum) + ReLU (+ residual) over (N_active, C) rows
 * (spconv_backbone.py L23-24, L54-64, L73/L187).
 *   training: fp64 sums of y (sum(y) | sum(y*y) per channel), all-reduced across processes when the BatchNorm is
 *             synchronized (torch.nn.SyncBatchNorm), then one apply pass that derives from them scale = gamma*rstd,
 *             shift = beta - mean*scale, save_mean, save_rstd and the running stats update (unbiased var, momentum).
 *             An empty batch (count 0) leaves the running stats unchanged, as torch.nn.BatchNorm1d does.
 *   eval    : scale / shift from the running stats (toda_bn_eval_coeffs), then the same apply pass (toda_bn_apply).
 *   apply   : a = act(y*scale + shift (+ residual)).
 *   bwd     : g = da * (a>0 if relu); dgamma = sum g*xhat; dbeta = sum g;
 *             dy = scale*(g - dbeta/N - xhat*dgamma/N); dresidual = g.
 * Each phase that needs the other processes' statistics is split at the all-reduce (SUM, done by the caller):
 *   forward : toda_bn_local_sums -> all-reduce sums (+ count) -> toda_bn_apply_sums
 *   backward: toda_bn_bwd_reduce -> all-reduce red            -> toda_bn_bwd_finish
 * A single process passes its own buffers through and the row count n (count = NULL); toda_bn_bwd is its backward in
 * one call.  A process of a synchronized BatchNorm with no rows still makes every call.
 * ------------------------------------------------------------------------------------------ */
size_t toda_bn_workspace_bytes(int channels);
/* sums: double[2*channels] = sum(y) | sum(y*y) per channel, from the per-CTA fixed-order partials of y, or from the
 * convolution epilogue's `epilogue_sums` (optional; y is then not read, and it may be `sums` itself).  count (optional):
 * receives the row count, written on the device (&sums[2*channels] when the count is all-reduced with the sums). */
int toda_bn_local_sums(const float *y, const double *epilogue_sums, int n, int channels, double *sums, double *count,
                       void *workspace, size_t workspace_bytes, void *stream);
int toda_bn_eval_coeffs(const float *gamma, const float *beta, const float *running_mean, const float *running_var,
                        float eps, int channels, float *scale, float *shift, void *stream);
/* a_bf16 / dy_bf16 (optional, may be NULL): bf16 copies written by the same pass, consumed as tensor-core operands. */
int toda_bn_apply(const float *y, int n, int channels, const float *scale, const float *shift, const float *residual,
                  int relu, float *a, void *a_bf16, void *stream);
/* Training-mode apply: coefficients, save_mean / save_rstd and the running statistics from `sums` (toda_bn_local_sums'
 * layout, all-reduced or not) and the row count *count (the global count of a synchronized BatchNorm) or n when count is
 * NULL, applied in the same launch; scale / shift are written for the backward pass. */
int toda_bn_apply_sums(const float *y, int n, int channels, const double *sums, const double *count, const float *gamma,
                       const float *beta, float eps, float momentum, float *running_mean, float *running_var, float *scale,
                       float *shift, float *save_mean, float *save_rstd, const float *residual, int relu, float *a,
                       void *a_bf16, void *stream);
/* red: double[2*channels] = sum g | sum g*xhat (g = da after the ReLU mask); dgamma / dbeta are this process's own sums
 * (torch leaves their averaging to the gradient all-reduce).  count: as in toda_bn_apply_sums (the forward's).  training
 * = 0 (eval-mode gradient): dy = scale*g, red is not read. */
int toda_bn_bwd_reduce(const float *da, const float *a, const float *y, int n, int channels, const float *save_mean,
                       const float *save_rstd, int relu, double *red, float *dgamma, float *dbeta, void *workspace,
                       size_t workspace_bytes, void *stream);
/* dbias (optional, may be NULL): sum_rows dy[:,c], the gradient of a bias added before the BatchNorm, summed in the same
 * pass from fixed-order fp64 partials (workspace: toda_bn_workspace_bytes(channels), needed only with dbias). */
int toda_bn_bwd_finish(const float *da, const float *a, const float *y, int n, int channels, const float *gamma,
                       const float *save_mean, const float *save_rstd, int relu, int training, const double *red,
                       const double *count, float *dy, void *dy_bf16, float *dresidual, float *dbias, void *workspace,
                       size_t workspace_bytes, void *stream);
int toda_bn_bwd(const float *da, const float *a, const float *y, int n, int channels, const float *gamma,
                const float *save_mean, const float *save_rstd, int relu, int training, float *dy, void *dy_bf16,
                float *dresidual, float *dgamma, float *dbeta, float *dbias, void *workspace, size_t workspace_bytes,
                void *stream);
/* column sums: dbias[c] = sum_rows dy[:,c] (the bias gradient of a convolution with no BatchNorm after it) */
int toda_col_sum(const float *dy, int n, int channels, float *out, void *workspace, size_t workspace_bytes,
                 void *stream);

/* ------------------------------------------------------------------------------------------
 * One call per backbone layer: conv -> BatchNorm1d (+ residual) (+ ReLU) forward, and its backward
 * (BN backward -> dgrad (+ residual-branch gradient) -> wgrad -> bias gradient): `post_act_block` /
 * `SparseBasicBlock` (spconv_backbone.py L8-27, L30-66) as the host sees them.  Same kernels as the
 * individual entry points above, sequenced in C so that the Python host pays one call per layer.
 *   stats: float[4*cout] = scale, shift, save_mean, save_rstd (mean / rstd rows unused in eval mode)
 *   sums : double[2*cout] scratch for the BatchNorm's sums of y (training mode): accumulated by the conv epilogue
 *          (tensor-core kernel) or by toda_bn_local_sums (FFMA kernel)
 * Pointers marked optional may be NULL; with n_out = 0 the output pointers may be NULL too (the forward then leaves the
 * running statistics unchanged, the backward writes zero parameter gradients).
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    const float *x; const void *x_bf16; int n_in, cin; const int32_t *nbr; int n_out, kvol;
    const float *w; const void *w_bf16 /* optional */; int cout; const float *bias /* optional */;
    const uint32_t *tile_masks /* optional */;
    const uint16_t *plan_lidx /* optional */; const int32_t *plan_rows; const int32_t *plan_cnt; int plan_groups, plan_cap;
    int precision; void *conv_ws; size_t conv_ws_bytes;
    const float *gamma; const float *beta; float eps, momentum; float *running_mean; float *running_var; int training;
    const float *residual /* optional */; int relu;
    float *y; double *sums; float *stats; float *a; void *a_bf16 /* optional */;
    void *bn_ws; size_t bn_ws_bytes;
} toda_layer_fwd_args;
typedef struct {
    const float *da; const float *a_mask; const float *y; int n_out, cout; const float *gamma; const float *mean; const float *rstd;
    int relu, training; float *dy; void *dy_bf16 /* optional */; float *dres /* optional */; float *dgamma; float *dbeta;
    void *bn_ws; size_t bn_ws_bytes;
    const float *x; const void *x_bf16 /* optional */; int n_in, cin, kvol;
    int need_dx; const int32_t *dgrad_nbr; const float *wt; const void *wt_bf16 /* optional */;
    const int32_t *dgrad_out_rows /* optional */; const uint32_t *dgrad_masks /* optional */;
    const uint16_t *dplan_lidx /* optional */; const int32_t *dplan_rows; const int32_t *dplan_cnt; int dplan_groups, dplan_cap;
    const float *addend /* optional */; float *dx;
    int need_dw; const int32_t *nbr_fwd; const uint32_t *fwd_masks /* optional: tile masks of nbr_fwd */; float *dw;
    void *wgrad_ws; size_t wgrad_ws_bytes;
    int need_db; float *db;
    int precision; void *conv_ws; size_t conv_ws_bytes;
} toda_layer_bwd_args;
int toda_layer_fwd(const toda_layer_fwd_args *args, void *stream);
int toda_layer_bwd(const toda_layer_bwd_args *args, void *stream);
/* The same layer split at the all-reduces of a BatchNorm synchronized across processes (training mode), as the
 * toda_bn_* calls above: toda_layer_fwd_stats (conv + sums, double[2*cout+1] with the row count) -> all-reduce ->
 * toda_layer_fwd_apply (stats, a, a_bf16, running statistics from global_sums); toda_layer_bwd_reduce (red,
 * double[2*cout], and this process's dgamma / dbeta) -> all-reduce -> toda_layer_bwd_finish (dy, dres, dgrad, wgrad,
 * bias gradient; global_count = &global_sums[2*cout] of the forward).  `sums` of the forward args is not used.
 * toda_layer_fwd / toda_layer_bwd are the two phases back to back on the layer's own buffers, with the count n_out. */
int toda_layer_fwd_stats(const toda_layer_fwd_args *args, double *local_sums, void *stream);
int toda_layer_fwd_apply(const toda_layer_fwd_args *args, const double *global_sums, void *stream);
int toda_layer_bwd_reduce(const toda_layer_bwd_args *args, double *local_red, void *stream);
int toda_layer_bwd_finish(const toda_layer_bwd_args *args, const double *global_red, const double *global_count, void *stream);

/* ------------------------------------------------------------------------------------------
 * K9 HeightCompression: pcdet/models/backbones_2d/map_to_bev/height_compression.py L20-25
 * (SparseConvTensor.dense() + view).  out[b, c*D+z, y, x] = features[n, c]; zero elsewhere.
 * ------------------------------------------------------------------------------------------ */
int toda_bev_scatter_fwd(const float *features, const int32_t *coords, int n, int channels, int batch, int D, int H,
                         int W, float *out, void *stream);
int toda_bev_scatter_bwd(const float *d_out, const int32_t *coords, int n, int channels, int batch, int D, int H,
                         int W, float *d_features, void *stream);

/* row gather used when a SparseConvTensor arrives in non-canonical order: out[i,:] = in[rows[i],:] */
int toda_gather_rows(const float *in, const int32_t *rows, int n, int channels, float *out, void *stream);

#ifdef __cplusplus
}
#endif
#endif
