/*
 * cf_b200.h -- C ABI of libcf_b200.so: the B200 (sm_100a) continuous-fusion hot path and the
 * rotated-box post-process, as bound by the Python host layer (ctypes) or any other FFI.
 *
 * Conventions (SURVEY.md 8b)
 *   - every pointer named d_* is a DEVICE pointer owned by the caller (PyTorch's caching allocator);
 *     kernels never allocate or free.  Workspaces are caller-provided, sized by cf_*_workspace_bytes.
 *   - `stream` is a cudaStream_t passed as void* (torch.cuda.current_stream().cuda_stream);
 *     calls only enqueue work, they never synchronise.
 *   - return value: 0 = CF_OK, negative = error class; cf_last_error() gives the thread-local text.
 *   - a device that is not compute capability 10.x is a hard error (CF_ERR_ARCH): there is no fallback.
 *   - tensors are dense row-major fp32 unless a stride argument says otherwise.
 *
 * Each entry point cites the reference interface it stands behind (file:line in the upstream tree)
 * or, for the fusion layer the reference leaves as a TODO (model.py:199-203), the slot it fills.
 */
#ifndef CF_B200_H
#define CF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define CF_API __attribute__((visibility("default")))
#else
#define CF_API
#endif

#define CF_ABI_VERSION 2

#define CF_OK 0
#define CF_ERR_ARG (-1)         /* bad shape / null pointer / unsupported size */
#define CF_ERR_ALIGN (-2)       /* pointer not aligned as documented            */
#define CF_ERR_ARCH (-3)        /* no CUDA device, or device is not sm_100       */
#define CF_ERR_LAUNCH (-4)      /* CUDA launch / runtime error                   */
#define CF_ERR_UNSUPPORTED (-5) /* valid request this build does not implement   */

#define CF_MAX_K 16 /* neighbours per BEV cell */

/* MLP arithmetic of cf_fusion_fwd */
#define CF_MODE_FP32 0      /* fp32-accurate: split-bf16 x3 on tcgen05 (or FFMA), fp32 accumulate */
#define CF_MODE_BF16 1      /* bf16 operands on tcgen05, fp32 accumulate / pool / add            */
#define CF_MODE_FP32_SIMT 2 /* CUDA-core FFMA path (bring-up / cross-check path)                  */
#define CF_MODE_BF16_TABLES 3 /* CF_MODE_BF16 with the layer-1 tables T stored as bf16 (inference only):
                               * cf_point_mlp1 / cf_point_mlp1_multi write bf16 rows into d_T / h_T[s], cf_fusion_fwd
                               * reads them; halves the table traffic, doubles the rounding error of CF_MODE_BF16
                               * (still within its 1e-2 tolerance); cf_fusion_bwd rejects it                  */

CF_API int cf_abi_version(void);
CF_API const char *cf_last_error(void);
/* 0 if the current device can run this library (compute capability 10.x). */
CF_API int cf_device_check(void);
/* number of kernels this library has launched in this process (bench.py reports it as gpu_launches). */
CF_API long long cf_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * K-1  point bucketing: counting sort of the valid LiDAR points of each frame into a uniform BEV
 * grid (histogram -> warp-scan exclusive prefix -> scatter).  Once per frame, shared by all scales.
 *   d_points      (B,N,3) fp32, sample["pointcloud_raw"]   data_import_carla.py:263-264,71,79
 *   d_num_points  (B) int64,   sample["num_points_raw"]    data_import_carla.py:262,73,81 (collated)
 *   grid: bucket (bx,by) covers [gx0+bx*cell, +cell) x [gy0+by*cell, +cell); points outside are
 *         clamped into the border buckets.
 *   d_bucket_start (B, nbx*nby+1) int32 out; d_sorted (B,N,4) fp32 out = (x, y, z, bits(idx)).
 *   d_workspace    cf_bucket_workspace_bytes(B, nbx, nby) bytes.
 * ------------------------------------------------------------------------------------------- */
CF_API size_t cf_bucket_workspace_bytes(int32_t B, int32_t nbx, int32_t nby);
CF_API int cf_bucket_points(const float *d_points, const int64_t *d_num_points, int32_t B, int32_t N, float gx0,
                     float gy0, float cell, int32_t nbx, int32_t nby, int32_t *d_bucket_start,
                     float *d_sorted, void *d_workspace, void *stream);

/* ---------------------------------------------------------------------------------------------
 * K-2  bounded-radius top-K query per BEV cell (SURVEY Appendix A1-A5).  Fills the KNN half of the
 * TODO at model.py:199-203 for the feature map produced at model.py:74-78.
 *   cell (i,j) centre: cx = x0 + (float)i*dx, cy = y0 + (float)j*dy (fp32, separately rounded);
 *   d2 = (px-cx)^2 + (py-cy)^2 fp32 without FMA; keep d2 <= radius*radius; ascending (d2, idx).
 *   d_knn_idx (B,H,W,K) int32 out, -1 = empty slot.  1 <= K <= CF_MAX_K.
 * ------------------------------------------------------------------------------------------- */
CF_API int cf_knn_query(const int32_t *d_bucket_start, const float *d_sorted, int32_t B, int32_t N, float gx0,
                 float gy0, float cell, int32_t nbx, int32_t nby, int32_t H, int32_t W, float x0, float y0,
                 float dx, float dy, float radius, int32_t K, int32_t *d_knn_idx, void *stream);

/* The cell centres of a 2^m-times coarser scale are bit-identical to every 2^m-th centre of a finer scale
 * (same x0,y0; dx,dy scaled by a power of two), so its KNN table is a strided copy of the finer one:
 *   d_coarse[b,i,j,:] = d_fine[b, i*step, j*step, :]. */
CF_API int cf_knn_subsample(const int32_t *d_fine, int32_t B, int32_t Hf, int32_t Wf, int32_t step,
                     int32_t *d_coarse, int32_t Hc, int32_t Wc, int32_t K, void *stream);

/* ---------------------------------------------------------------------------------------------
 * K-3  projection + bilinear gather, once per frame (Appendix A6, A7).
 *   d_img_feat  camera feature map, logical (B,Ci,Hf,Wf) fp32 with ELEMENT strides sb,sc,sh,sw
 *               (NCHW contiguous or channels_last both accepted; Ci % 4 == 0)
 *   uv source   exactly one of: d_uv (B,N,2) = sample["projected_loc_uv"], data_import_carla.py:265-266;
 *               or h_calib, 12 HOST floats = CRT_tensor (4,3), data_import_carla.py:31-34,199-200
 *   d_feat      (B,N,Ci) fp32 out; rows >= num_points[b] are zero filled
 *   d_workspace cf_gather_workspace_bytes(...) bytes (pixel-major copy of the map when sc != 1)
 * cf_point_gather_bf16: the same with a bf16 camera map (any element strides; channels_last: every pixel 8-byte
 *   aligned; same workspace, an upper bound for its bf16 pixel-major copy).  Each tap is widened exactly to fp32 and the
 *   blend is the fp32 sequence of cf_point_gather, so the result equals cf_point_gather on the widened map; d_feat is fp32.
 * ------------------------------------------------------------------------------------------- */
CF_API size_t cf_gather_workspace_bytes(int32_t B, int32_t Ci, int32_t Hf, int32_t Wf, int64_t sc);
CF_API int cf_point_gather(const float *d_img_feat, int64_t sb, int64_t sc, int64_t sh, int64_t sw, int32_t B,
                    int32_t Ci, int32_t Hf, int32_t Wf, const float *d_points, const float *d_uv,
                    const float *h_calib, const int64_t *d_num_points, int32_t N, float img_w, float img_h,
                    float *d_feat, void *d_workspace, void *stream);
CF_API int cf_point_gather_bf16(const void *d_img_feat, int64_t sb, int64_t sc, int64_t sh, int64_t sw, int32_t B,
                         int32_t Ci, int32_t Hf, int32_t Wf, const float *d_points, const float *d_uv,
                         const float *h_calib, const int64_t *d_num_points, int32_t N, float img_w, float img_h,
                         float *d_feat, void *d_workspace, void *stream);

/* ---------------------------------------------------------------------------------------------
 * K-4a per-point half of MLP layer 1 (exact factorisation of Appendix A8/A9):
 *   T[b,p,:] = W1[:, :Ci] f_p + W1[:, Ci:Ci+3] (px,py,pz) + b1        so that for BEV cell centre c
 *   relu(W1 [f_p, p - (cx,cy,0)] + b1) = relu(T[b,p,:] - W1[:,Ci]*cx - W1[:,Ci+1]*cy)
 *   d_W1 (C, Ci+3) fp32 row-major (nn.Linear.weight layout), d_b1 (C).  d_T (B,N,C) fp32 out.
 *   mode CF_MODE_FP32 / CF_MODE_BF16: tcgen05 GEMM over the Ci image channels (needs the workspace);
 *   CF_MODE_FP32_SIMT, or shapes without a tensor-core instantiation: FFMA kernel.
 * ------------------------------------------------------------------------------------------- */
CF_API size_t cf_point_mlp1_workspace_bytes(int32_t Ci, int32_t C, int32_t mode);
CF_API int cf_point_mlp1(const float *d_feat, const float *d_points, const int64_t *d_num_points, int32_t B,
                  int32_t N, int32_t Ci, int32_t C, const float *d_W1, const float *d_b1, float *d_T,
                  int32_t mode, const void *d_packed, void *d_workspace, void *stream);
/* Optional: the tensor-core paths consume weights re-packed into the UMMA operand image.  A caller whose weights do
 * not change between calls (inference) packs them once into a buffer of cf_point_mlp1_workspace_bytes /
 * cf_fusion_packed_bytes bytes and passes it as d_packed; with d_packed == NULL every call packs into d_workspace. */
CF_API int cf_point_mlp1_pack_weights(const float *d_W1, int32_t Ci, int32_t C, int32_t mode, void *d_packed, void *stream);
/* K-4a for several scales in one launch: the point features are packed into the tensor-core operand once and
 * multiplied by every scale's W1.  h_* are HOST arrays of n_scales entries (channel counts and DEVICE pointers):
 * h_W1[s] (C_s, Ci+3), h_b1[s] (C_s), h_T[s] (B,N,C_s) out, h_packed[s] from cf_point_mlp1_pack_weights (required).
 * Same result as n_scales calls of cf_point_mlp1 in the same mode.  Ci % 32 == 0, C_s % 32 == 0, n_scales <= 8;
 * CF_ERR_UNSUPPORTED if the shapes do not fit (call cf_point_mlp1 per scale instead). */
CF_API int cf_point_mlp1_multi(const float *d_feat, const float *d_points, const int64_t *d_num_points, int32_t B,
                        int32_t N, int32_t Ci, int32_t n_scales, const int32_t *h_C, const float *const *h_W1,
                        const float *const *h_b1, float *const *h_T, int32_t mode, const void *const *h_packed,
                        void *stream);
CF_API size_t cf_fusion_packed_bytes(int32_t C, int32_t mode);
CF_API int cf_fusion_pack_weights(const float *d_W2, const float *d_W3, int32_t C, int32_t mode, void *d_packed,
                           void *stream);

/* ---------------------------------------------------------------------------------------------
 * K-4  per-neighbour MLP layers 1b/2/3 + K-sum-pool + BEV add for one scale (Appendix A9, A10);
 * the result replaces `x` after a residual group in ResnetCustomed.forward (model.py:74-78).
 *   out[b,:,i,j] = bev[b,:,i,j] + W3 * sum_k relu(W2 relu(T[b,idx_k,:] - e_ij) + b2) + n_valid*b3
 *   d_bev/d_out (B,C,H,W) fp32 NCHW contiguous (may alias: in place); C % 16 == 0, 16 <= C <= 256; d_T 32-byte aligned.
 *   mode: CF_MODE_*.   d_workspace: cf_fusion_workspace_bytes(C, mode, B, H, W) bytes (packed weights and the
 *   compacted list of cells that have a neighbour).  B <= 64 frames per call.
 *   mode | CF_IO_BF16: d_bev and d_out are bf16 (B,C,H,W) NCHW maps (may alias, as for fp32).  bev is widened exactly to
 *   fp32, everything else is computed as without the flag and out is rounded once to bf16 (nearest even) when stored:
 *   the result equals the fp32 call on the widened map, rounded.  T, weights and the workspace size are unchanged.
 *   The opt-in segment-tile kernel (CF_SEG=1) is fp32-only and is skipped with this flag.
 * Every function that takes a `mode` ignores the flag bits (CF_IO_BF16, CF_BWD_DETERMINISTIC) when it picks the
 * arithmetic, the operand layout or a workspace size.
 * ------------------------------------------------------------------------------------------- */
#define CF_IO_BF16 0x200 /* OR-ed into `mode` of cf_fusion_fwd (bf16 bev / out) and cf_fusion_bwd (bf16 d_gout) */
CF_API size_t cf_fusion_workspace_bytes(int32_t C, int32_t mode, int32_t B, int32_t H, int32_t W);
CF_API int cf_fusion_fwd(const float *d_bev, const float *d_T, const int32_t *d_knn_idx, int32_t B, int32_t N,
                  int32_t C, int32_t H, int32_t W, int32_t K, float x0, float y0, float dx, float dy,
                  const float *d_W1, int32_t Ci, const float *d_W2, const float *d_b2, const float *d_W3,
                  const float *d_b3, float *d_out, int32_t mode, const void *d_packed, void *d_workspace,
                  void *stream);

/* ---------------------------------------------------------------------------------------------
 * K-4b backward of cf_point_mlp1 + cf_fusion_fwd for one scale (training only).  d_gout = dL/d out (B,C,H,W);
 * dL/d bev is d_gout itself.  mode | CF_IO_BF16: d_gout is bf16 (widened exactly on load; combines with
 * CF_BWD_DETERMINISTIC, and with it the gradients equal those of the fp32 call on the widened d_gout).  Gradients are ACCUMULATED into d_gW1 (C,Ci+3), d_gb1 (C), d_gW2 (C,C), d_gb2,
 * d_gW3, d_gb3 and d_gfeat (B,N,Ci) -- zero them first (d_gfeat collects every scale's contribution).
 * The forward saves only indices, inputs and weights (and, optionally, its table: d_T = the output of
 * cf_point_mlp1, NULL = recompute it); H1/H2/pooled are recomputed into the workspace
 * (cf_fusion_bwd_workspace_bytes), for the (cell, k) slots that hold a neighbour only.
 * mode CF_MODE_FP32 / CF_MODE_BF16: the GEMMs run on tcgen05 (fp32 operands split into bf16 hi + lo, three MMAs,
 * fp32 accumulate -- gradients are fp32-accurate in both modes); CF_MODE_FP32_SIMT, or shapes without a
 * tensor-core instantiation: FFMA kernels.
 * Two summation paths:
 *   default            the live-cell / live-row lists are placed with atomics and the reductions over rows (dW, db,
 *                      dT, d img) use float atomics: reproducible to rounding, not bit for bit.
 *   deterministic      mode | CF_BWD_DETERMINISTIC, workspace cf_fusion_bwd_det_workspace_bytes: the lists come from
 *                      device-wide scans (grid order), every row reduction writes per-split partials that are summed in
 *                      a fixed order (the splits depend on shapes and on the device-side live counts only, not on the
 *                      GPU's SM count), dT is a gather over each point's rows in ascending row order.  Identical inputs
 *                      give bit-identical gradients on sm_100, in every mode and at every width; still no host
 *                      synchronisation (capturable in a CUDA graph).
 * cf_point_gather_bwd is the adjoint of cf_point_gather: d_gimg (+)= bilinear scatter of d_gfeat; d_gimg has the
 * camera map's logical shape and the given element strides.  cf_point_gather_bwd_det computes the same with a fixed
 * order: the (point, tap) contributions are listed per pixel (counting sort, each list in ascending (point, tap)) and
 * one thread per (pixel, channel) sums its list and adds the sum into d_gimg; workspace
 * cf_point_gather_bwd_det_workspace_bytes(B, N, Hf, Wf).  d_gimg is fp32; for a bf16 camera map accumulate into an fp32
 * buffer and round it once (summing the taps in bf16 would lose precision and the fixed order's guarantee).
 * ------------------------------------------------------------------------------------------- */
#define CF_BWD_DETERMINISTIC 0x100 /* OR-ed into `mode` of cf_fusion_bwd */
CF_API size_t cf_fusion_bwd_workspace_bytes(int32_t B, int32_t N, int32_t C, int32_t Ci, int32_t H, int32_t W,
                                            int32_t K);
CF_API size_t cf_fusion_bwd_det_workspace_bytes(int32_t B, int32_t N, int32_t C, int32_t Ci, int32_t H, int32_t W,
                                                int32_t K);
CF_API int cf_fusion_bwd(const float *d_gout, const float *d_feat, const float *d_points,
                  const int64_t *d_num_points, const int32_t *d_knn_idx, int32_t B, int32_t N, int32_t C,
                  int32_t H, int32_t W, int32_t K, float x0, float y0, float dx, float dy,
                  const float *d_W1, const float *d_b1, int32_t Ci, const float *d_W2, const float *d_b2,
                  const float *d_W3, const float *d_T, float *d_gW1, float *d_gb1, float *d_gW2, float *d_gb2,
                  float *d_gW3, float *d_gb3, float *d_gfeat, int32_t mode, void *d_workspace, void *stream);
CF_API int cf_point_gather_bwd(const float *d_gfeat, float *d_gimg, int64_t sb, int64_t sc, int64_t sh, int64_t sw,
                        int32_t B, int32_t Ci, int32_t Hf, int32_t Wf, const float *d_points,
                        const float *d_uv, const float *h_calib, const int64_t *d_num_points, int32_t N,
                        float img_w, float img_h, void *stream);
CF_API size_t cf_point_gather_bwd_det_workspace_bytes(int32_t B, int32_t N, int32_t Hf, int32_t Wf);
CF_API int cf_point_gather_bwd_det(const float *d_gfeat, float *d_gimg, int64_t sb, int64_t sc, int64_t sh, int64_t sw,
                            int32_t B, int32_t Ci, int32_t Hf, int32_t Wf, const float *d_points,
                            const float *d_uv, const float *h_calib, const int64_t *d_num_points, int32_t N,
                            float img_w, float img_h, void *d_workspace, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Dataset side on the device (SURVEY 8f-2): CarlaDataset.Voxelization_Projection + .Projection,
 * data_import_carla.py:196-267, for a batch of raw sweeps.  Produces every tensor the model consumes:
 *   d_raw (B,Nraw,3) fp32 LiDAR xyz, d_num_raw (B) int64 valid rows per frame
 *   h_range  6 HOST floats (x_lo, x_hi, y_lo, y_hi, z_lo, z_hi): keep lo < v < hi   (:214-226; hi = max - delta)
 *   h_vox    6 HOST floats (x_scale, y_scale, z_scale, x_off, y_off, z_off) of pc_to_voxel_indice (:35-43)
 *   h_calib  12 HOST floats = CRT_tensor (4,3);  0 < u < u_hi (image_height) and 0 < v < v_hi (image_width) [sic :202-205]
 *   d_voxel  (B,Z,X,Y) fp32 out = sample["pointcloud"]: trilinear splat; of the points that share a voxel inside one of
 *            the 8 `voxel[idx] += w` statements only the LAST counts (index_put_ without accumulation, :249-256)
 *   d_points (B,max_num_pc,3), d_uv (B,max_num_pc,2) fp32 out, zero padded; d_num_points (B) int64 out
 *            = sample["pointcloud_raw"], ["projected_loc_uv"], ["num_points_raw"] (:261-267); input order is kept
 *   d_workspace cf_voxelize_workspace_bytes(...) bytes.  B <= 64, lidar_x_min >= 0.
 * ------------------------------------------------------------------------------------------- */
CF_API size_t cf_voxelize_workspace_bytes(int32_t B, int32_t Nraw, int32_t Z, int32_t X, int32_t Y);
CF_API int cf_voxelize_project(const float *d_raw, const int64_t *d_num_raw, int32_t B, int32_t Nraw,
                        const float *h_range, const float *h_vox, int32_t Z, int32_t X, int32_t Y,
                        const float *h_calib, float u_hi, float v_hi, int32_t max_num_pc, float *d_voxel,
                        float *d_points, float *d_uv, int64_t *d_num_points, void *d_workspace, void *stream);

/* ---------------------------------------------------------------------------------------------
 * SURVEY 8(f-4)  target assignment of LossTotal on device: getPositionOfPositive (loss.py:74-110) and
 * getPositionOfNegative (loss.py:112-127) for every frame of the batch, no host loop and no host list.
 *   d_ref_boxes (B,M,ref_stride) fp32 = object_data (x at [0], y at [1]); d_num_ref (B) int64
 *   centre cell: int((x*x_scale + x_offset)/reduced_scale), int((y*y_scale + y_offset)/reduced_scale) in
 *   fp32, truncated toward zero (loss.py:86-87); window positive_range^2 clipped to the (H,W) map.
 *   RNG contract (the caller supplies the draws, so the reference run with the same draws can be compared):
 *     d_shuffle_keys (B, M*R*R) fp32: the positive list of length n is reordered by the stable ascending
 *       order of its first n keys (stands for np.random.shuffle, loss.py:106), then cut to pos_threshold;
 *     d_candidates (B,L,2) int32: the (x,y) draws of the rejection loop (loss.py:116-126) in order; the
 *       first neg_threshold+1 that are not in the cut positive list are kept.
 *   out: d_pos_cells (B,pos_threshold) / d_neg_cells (B,neg_threshold+1) int32 linear cells x*W+y, -1 padded;
 *        d_pos_count / d_neg_count (B) int32; d_reg_cells (B,M,R*R) int32: the regression cells of every box
 *        in window order (whole window for regress_type 0, centre only otherwise), -1 = none.
 * ------------------------------------------------------------------------------------------- */
CF_API int cf_loss_targets(const float *d_ref_boxes, const int64_t *d_num_ref, int32_t B, int32_t M, int32_t ref_stride,
                    int32_t H, int32_t W, float x_scale, float y_scale, float x_offset, float y_offset,
                    float reduced_scale, int32_t positive_range, int32_t regress_type, int32_t pos_threshold,
                    int32_t neg_threshold, const float *d_shuffle_keys, const int32_t *d_candidates, int32_t L,
                    int32_t *d_pos_cells, int32_t *d_pos_count, int32_t *d_neg_cells, int32_t *d_neg_count,
                    int32_t *d_reg_cells, void *stream);

/* ---------------------------------------------------------------------------------------------
 * P-1  Test.get_bboxes (test.py:88-108) on device: per frame, anchor 0 then anchor 1, cells in
 * row-major order with cls[b,2a+1] > thr; gathers the 7 decoded channels [7a,7a+7).
 *   d_pred_cls (B,4,H,W), d_pred_box (B,14,H,W) fp32; d_boxes (B,cap,7) out; d_counts (B) int32 out
 *   (counts are clamped to cap; d_counts_raw, if non-null, receives the unclamped totals).
 * ------------------------------------------------------------------------------------------- */
CF_API int cf_get_bboxes(const float *d_pred_cls, const float *d_pred_box, int32_t B, int32_t H, int32_t W,
                  float thr, int32_t cap, float *d_boxes, int32_t *d_counts, int32_t *d_counts_raw,
                  void *stream);

/* ---------------------------------------------------------------------------------------------
 * P-2..P-4  Test.NMS_SAT (test.py:142-175) with get_vertice_rect / separating_axis_theorem
 * (separation_axis_theorem.py:82-94, 66-80): greedy in input order, box i is kept iff it overlaps no
 * previously kept box.  fp32 arithmetic mirrors the reference under numpy >= 2 (see DESIGN.md).
 *   d_boxes (B,cap,7) fp32 [x,y,z,l,w,h,yaw]; d_counts (B) int32
 *   d_keep_idx (B,cap) int32 out, ascending kept input indices, -1 padded; d_keep_count (B) int32 out
 *   d_workspace cf_nms_workspace_bytes(B,cap) bytes.
 * P-7  Test.NMS_IOU (test.py:110-140): same rule with predicate iou3d > thr (kept box nudged +1e-4).
 * ------------------------------------------------------------------------------------------- */
CF_API size_t cf_nms_workspace_bytes(int32_t B, int32_t cap);
CF_API int cf_nms_sat(const float *d_boxes, const int32_t *d_counts, int32_t B, int32_t cap, int32_t *d_keep_idx,
               int32_t *d_keep_count, void *d_workspace, void *stream);
CF_API int cf_nms_iou(const float *d_boxes, const int32_t *d_counts, int32_t B, int32_t cap, float thr,
               int32_t *d_keep_idx, int32_t *d_keep_count, void *d_workspace, void *stream);
/* the (cap x cap) overlap predicate of one frame as a dense uint8 matrix, for mask-level parity tests */
CF_API int cf_sat_matrix(const float *d_boxes, int32_t n, uint8_t *d_matrix, void *stream);

/* ---------------------------------------------------------------------------------------------
 * P-5/P-6  get_3d_box + box3d_iou (IOU.py:127-155, 91-120) for every pair (a_i, b_j), with the
 * reference's axis convention (rotation about axis 1; BEV polygon on axes (0,2); height on axis 1).
 *   d_boxes_a (na,7), d_boxes_b (nb,7) fp32; d_iou3d, d_iou2d (na,nb) fp64 out; nudge_b as test.py:129.
 * ------------------------------------------------------------------------------------------- */
CF_API int cf_box_iou(const float *d_boxes_a, int32_t na, const float *d_boxes_b, int32_t nb, float nudge_b,
               double *d_iou3d, double *d_iou2d, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Self-test of the tcgen05 building blocks (operand packing, shared-memory descriptors, TMEM):
 *   D (128,N) fp32 = A (128,K) * B (N,K)^T, bf16 operands (split != 0: bf16 hi/lo, three products).
 *   N in {32,64,128,192,256}, K % 16 == 0.  Not part of the reference-facing surface.
 * ------------------------------------------------------------------------------------------- */
CF_API int cf_debug_umma_gemm(const float *d_A, const float *d_B, int32_t N, int32_t K, int32_t split, float *d_D,
                       void *stream);

/* ---------------------------------------------------------------------------------------------
 * Self-tests of the two tcgen05 GEMM shapes behind cf_fusion_bwd (fp32 operands split into bf16 hi + lo):
 *   nn: Out (R,N) = epi( X (R,Kd) * B^T ),  B = W (N,Kd) [transpose 0] or W^T with W (Kd,N) [transpose 1];
 *       epi 0 store, 1 accumulate, 2 relu(. + aux[N]), 3 zero where aux (R,N) <= 0.  Kd, N % 32 == 0.
 *   tn: dW (M, N+n2) += X (R,M)^T * [Y (R,N) | Y2 (R,n2)],  db (M) += X^T * (wcol or 1);  M, N % 32 == 0, n2 <= 15.
 *   d_R (device int32, may be NULL) clamps R without a host synchronisation.
 * ------------------------------------------------------------------------------------------- */
CF_API size_t cf_debug_bwd_packed_bytes(int32_t N, int32_t Kd);
CF_API int cf_debug_bwd_gemm_nn(const float *d_X, int64_t R, const int32_t *d_R, int32_t Kd, int32_t N, const float *d_W,
                         int32_t transpose, float *d_Out, int32_t epi, const float *d_aux, void *d_packed,
                         void *stream);
CF_API int cf_debug_bwd_gemm_tn(const float *d_X, int32_t M, const float *d_Y, int32_t N, const float *d_Y2, int32_t n2,
                         const float *d_wcol, int64_t R, const int32_t *d_R, float *d_dW, float *d_db, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* CF_B200_H */
