/* gsx.h — C ABI of libgsx.so, the B200 (sm_100a) engine behind gradslam's PointFusion / ICPSLAM hot path.
 *
 * gradslam (reference @44470ee) is pure Python on PyTorch tensor ops: it has no FFI/plugin layer of its
 * own.  The boundary a maintainer would bind is therefore the set of tensor-op chains listed below; each
 * entry point names the reference function(s) (file:line under /root/reference) whose arithmetic it
 * replaces.  INTEGRATION.md shows the ctypes stub a gradslam maintainer would add at each site.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no torch / C++ types.  All pointers are DEVICE pointers
 *     (float32 data, int32/int64 tables) owned by the caller and borrowed for the duration of the call.
 *   - `stream` is a cudaStream_t passed as void*; every call only ENQUEUES work on it (no device
 *     synchronisation) unless the doc says it returns a host-visible count.
 *   - return 0 on success, non-zero on invalid argument / launch failure; gsx_last_error() returns a
 *     thread-local message for the last failure.
 *   - images are channels-last: depth (B,L,H,W,1), rgb/vertex/normal (B,L,H,W,3).  Per-frame calls take
 *     a base pointer for the frame plus the element stride (`*_bstride`, in floats) between batch elements,
 *     so frame s of a (B,L,H,W,C) tensor is addressed without a copy.
 *   - the surfel map has a fixed capacity and SECTOR-PACKED rows: map_geometry (B,cap,8) float32 rows
 *     (px,py,pz,nx,ny,nz,ccount,0) - exactly one 32-byte DRAM sector per surfel - and map_colors (B,cap,4) rows
 *     (r,g,b,0); both 16-byte aligned, every row access is a 128-bit load / store.  counts int32 (B,).  Rows
 *     >= counts[b] are never read.  (gradslam's padded tensors points / normals / colors / features are the
 *     strided views [..., 0:3], [..., 3:6], colours [..., 0:3], [..., 6:7] of these two arrays.)
 *   - arithmetic is IEEE fp32 with a fixed association order and no fused multiply-add, except the normal
 *     estimate's cross product and length, which are fused exactly as the reference's CPU build fuses them
 *     (see DESIGN.md "canonical arithmetic"), so every decision (threshold, pixel rounding, arg-min key) is
 *     bit-exact against the CPU oracle.
 */
#ifndef GSX_H_
#define GSX_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GSX_VERSION 201 /* 0.2.1: single-cloud gsx_icp_normal_eq_fwd/bwd, gsx_rigid_transform_fwd/bwd removed */

int gsx_version(void);
const char *gsx_last_error(void);

/* ------------------------------------------------------------------------------------------------
 * K1  depth -> vertex / normal maps (+ posed "global" maps)
 * replaces RGBDImages._compute_vertex_map / _compute_normal_map / _compute_global_vertex_map /
 *          _compute_global_normal_map   gradslam/structures/rgbdimages.py:643-762
 *          and projutils.inverse_intrinsics   gradslam/geometry/projutils.py:405-450
 * depth (B,L,H,W) with element stride depth_bstride between b and H*W between l;
 * intrinsics: B matrices 4x4 row-major, stride K_bstride; poses: B*L matrices, strides pose_bstride
 * (between b) and 16 (between l), or NULL (global maps = local maps).  Any output may be NULL.
 * Outputs are dense (B,L,H,W,3). */
int gsx_backproject_normals_fwd(const float *depth, int64_t depth_bstride, const float *intrinsics,
                                int64_t K_bstride, const float *poses, int64_t pose_bstride, int B, int L,
                                int H, int W, float *vertex, float *normal, float *gvertex, float *gnormal,
                                void *stream);

/* backward of K1: from the upstream gradients of any of the four maps (dense (B,L,H,W,3), NULL = zero)
 * computes d(loss)/d(depth) (B,L,H,W) and, if g_poses != NULL and poses != NULL, d(loss)/d(poses)
 * (B*L,4,4) (top 3x4 block; bottom row zero).  Autograd counterpart of the op chain above (the reference
 * obtains it from PyTorch's tape).  Gradients w.r.t. the intrinsics are not produced.  Deterministic: no
 * atomics; pose gradients are reduced per tile then summed in tile order.
 * scratch: gsx_backproject_normals_bwd_scratch_bytes(B,L,H,W) bytes (only needed for g_poses). */
int64_t gsx_backproject_normals_bwd_scratch_bytes(int B, int L, int H, int W);
int gsx_backproject_normals_bwd(const float *depth, int64_t depth_bstride, const float *intrinsics,
                                int64_t K_bstride, const float *poses, int64_t pose_bstride, int B, int L,
                                int H, int W, const float *g_vertex, const float *g_normal,
                                const float *g_gvertex, const float *g_gnormal, float *g_depth,
                                float *g_poses, void *scratch, int64_t scratch_bytes, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Fused PointFusion map update, one live frame for all B elements: three kernels
 *   K1r  gsx_fusion_frame_records    per pixel: world vertex, world normal, confidence weight, depth -> one
 *                                    32-byte record; re-arms the workspace for this frame
 *   K2   gsx_fusion_project_select   per map row: projection, tests, per-pixel 128-bit arg-min
 *   K4   gsx_fusion_merge_append     per pixel: merge the selected row or append a new surfel
 * replaces update_map_fusion = find_active_map_points + find_similar_map_points +
 *          find_best_unique_correspondences + fuse_with_map (+ Pointclouds.append_points)
 *          gradslam/slam/fusionutils.py:198-287, 290-411, 414-546, 580-722, 761-789;
 *          gradslam/structures/pointclouds.py:526-614, 1117-1237
 *
 * Workspace: gsx_fusion_workspace_bytes(B,H,W) bytes, 16-byte aligned.  Nothing in it has to survive from one frame
 * to the next: gsx_fusion_frame_records re-arms everything the other two kernels consume, so no zero-fill and no
 * epoch bookkeeping is needed and an abandoned frame cannot poison the next one.  (Only the statistics below
 * accumulate; zero them once if they are read.)                                                            */
int64_t gsx_fusion_workspace_bytes(int B, int H, int W);
/* byte offset inside the workspace of uint64 stats[B][2] = running totals of {map points inside the
 * live frustum ("active"), map points merged}; used for the roofline's algorithmic-byte count. */
int64_t gsx_fusion_workspace_stats_offset(int B, int H, int W);

/* K1r: frame records of the live frame.
 * replaces, per pixel, RGBDImages.global_vertex_map / global_normal_map (gradslam/structures/rgbdimages.py:643-762)
 *          and get_alpha on the camera-frame vertex (gradslam/slam/fusionutils.py:16-73, :657)
 * Either evaluate everything from the depth image (gvertex = gnormal = vertex = NULL; intrinsics required; poses =
 * camera-to-world, or NULL for "world frame == camera frame"), or pack already materialised maps: gvertex / gnormal /
 * vertex (B,H,W,3) (outputs of gsx_backproject_normals_fwd, used by the differentiable mode; intrinsics / poses are
 * then ignored).  Same arithmetic either way, bit for bit. */
int gsx_fusion_frame_records(const float *depth, int64_t depth_bstride, const float *intrinsics, int64_t K_bstride,
                             const float *poses, int64_t pose_bstride, const float *gvertex, const float *gnormal,
                             const float *vertex, int B, int H, int W, double sigma, void *workspace, void *stream);

/* K2+K3: project every map point into the live camera, keep points that are in the frustum, close to
 * the frame vertex they land on and with a similar normal, and reduce per pixel to the best candidate
 * (largest confidence count, then smallest ray distance, then smallest index) with a 128-bit atomic
 * min.  max_count = host upper bound on counts[b] (sizes the grid).  The frame records of the live frame must be in
 * the workspace (gsx_fusion_frame_records). */
int gsx_fusion_project_select(const float *map_geometry, const int32_t *counts, int64_t capacity, int64_t max_count,
                              const float *poses, int64_t pose_bstride, const float *intrinsics, int64_t K_bstride,
                              int B, int H, int W, float dist_th, float dot_th, void *workspace, void *stream);

/* K4: per pixel, merge the selected map point with the frame sample (confidence-weighted mean) or, for
 * valid pixels without a match, append a new surfel in row-major pixel order (stable single-pass scan).
 * counts_in -> counts_out (may not alias).  with_ccounts = 0 for maps without confidence counts
 * (ICPSLAM aggregation, gradslam/slam/fusionutils.py:725-758): then nothing is merged, every valid
 * pixel is appended and the ccount slot of the new rows is 0.  overflow_flag (int32, device) is set to 1 if capacity
 * was exceeded (the surplus points are dropped).  rgb: live colours (B,H,W,3), element stride rgb_bstride.
 * assoc_out: NULL, or int32 (B,H,W) zero-filled by the caller that receives where every pixel went: +(row+1) appended
 * as `row`, -(row+1) merged into `row`, 0 dropped (the differentiable mode's forward: the caller runs the kernel on
 * a COPY of the map so that the pre-merge rows survive for the backward). */
int gsx_fusion_merge_append(float *map_geometry, float *map_colors, int with_ccounts, const int32_t *counts_in,
                            int32_t *counts_out, int64_t capacity, const float *rgb, int64_t rgb_bstride, int B, int H,
                            int W, void *workspace, int32_t *overflow_flag, int32_t *assoc_out, void *stream);

/* Backward of K4 (autograd.Function backward of the differentiable mode).
 * replaces the tape PyTorch builds through fuse_with_map   gradslam/slam/fusionutils.py:654-720 (merge),
 *          :702-720 + gradslam/structures/pointclouds.py:1117-1237 (append), get_alpha :16-73
 * upstream gradients of the updated map in the packed row layout (B,capacity_out,8 / 4) (either may be NULL = zero)
 * -> gradients of the pre-merge map (B,capacity_in,8 / 4) (every row written; padding rows and padding slots zero) and
 * of the frame values: world vertex / normal maps, colours and - through the confidence weight alpha - the
 * camera-frame vertex map, all (B,H,W,3). */
int gsx_fusion_merge_append_bwd(const int32_t *assoc, const int32_t *counts_in, const float *map_geometry,
                                const float *map_colors, int with_ccounts, int64_t capacity_in,
                                const float *g_geometry, const float *g_colors, int64_t capacity_out,
                                const float *gvertex, const float *gnormal, const float *rgb, const float *vertex,
                                int B, int H, int W, double sigma, float *d_map_geometry, float *d_map_colors,
                                float *d_gvertex, float *d_gnormal, float *d_rgb, float *d_vertex, void *stream);

/* Whole-sequence driver with ground-truth poses: for s in [s_begin,s_end): K1r -> K2/K3 -> K4, no host sync.
 * replaces ICPSLAM.forward with odom='gt' + PointFusion._map   gradslam/slam/icpslam.py:99-138,
 *          gradslam/slam/pointfusion.py:107-112
 * depth (B,L,H,W), rgb (B,L,H,W,3) dense; poses (B,L,4,4) dense; intrinsics (B,4,4) dense.
 * counts: int32 (2,B) ping-pong buffer; row (s_begin & 1) holds the current sizes on entry; on return the
 * current sizes are in row (s_end & 1).  max_count0 = host upper bound of the sizes on entry.
 * Splitting a sequence into several calls (s_begin..s_end chunks) lets the caller overlap host->device copies of
 * later frames with the fusion of earlier ones.  On a launch failure the internal streams are still joined to
 * `stream` before the error is returned. */
/* number of independent batch groups gsx_pointfusion_sequence_gt runs on concurrent internal streams for a batch of
 * B (default 2, environment GSX_SEQ_GROUPS = 1..4 overrides; never more than B).  Kernel launches per call =
 * groups * (3 * frames - [map empty on entry]). */
int gsx_pointfusion_sequence_groups(int B);
/* workspace of the sequence driver: two frame workspaces used alternately (the records of frame s+1 are computed on a
 * side stream while frame s is fused), 16-byte aligned, no initialisation needed */
int64_t gsx_pointfusion_sequence_workspace_bytes(int B, int H, int W);
int gsx_pointfusion_sequence_gt(float *map_geometry, float *map_colors, int32_t *counts, int64_t capacity,
                                int64_t max_count0, const float *depth, const float *rgb, const float *intrinsics,
                                const float *poses, int B, int L, int s_begin, int s_end, int H, int W, float dist_th,
                                float dot_th, double sigma, void *workspace, int32_t *overflow_flag, void *stream);
/* test hook: the next gsx_pointfusion_sequence_gt call reports a launch failure at frame s (once); -1 = off */
void gsx_debug_fail_at_frame(int s);

/* ------------------------------------------------------------------------------------------------
 * Map exchange between the GPUs of a node through peer memory (SURVEY.md section 8e "Collective": the variable-length
 * all-gather of the finished maps; the reference has no multi-GPU code - this is the exchange its DataParallel-style
 * use would need).  One process per GPU.  The owner exports the allocation behind a store pointer as a CUDA IPC handle,
 * peers open it (mappings are cached per process; gsx_peer_close_all drops them - call it before the owners free their
 * allocations back to the driver) and pull row blocks with pitched device-to-device copies on the copy engines:
 * block b of n_blocks moves width_bytes from src + b*src_pitch_bytes to dst + b*dst_pitch_bytes.  Ordering between the
 * processes is the caller's (gradslam_b200/parallel.py).  Return 0, or non-zero with gsx_last_error(). */
#define GSX_IPC_HANDLE_BYTES 64
int gsx_peer_export(const void *ptr, unsigned char *handle /* [GSX_IPC_HANDLE_BYTES] */, int64_t *offset,
                    int64_t *allocation_bytes /* optional */);
int gsx_peer_open(const unsigned char *handle, int64_t offset, void **ptr_out);
int gsx_peer_close_all(void);
int gsx_peer_copy_rows(void *dst, int64_t dst_pitch_bytes, const void *src, int64_t src_pitch_bytes,
                       int64_t width_bytes, int64_t n_blocks, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Dataset-native ingest (SURVEY.md §8f.2): 8-bit colour (n_pixels,3) and 16-bit depth (n_pixels) as stored by
 * ICL-NUIM / TUM / ScanNet -> float32 colour and depth on the device, bit-identical to the reference loaders'
 * host-side conversion: colour = float(u8) [/ 255 if normalize_color], depth = float32(float64(u16) /
 * depth_scaling_factor)   (gradslam/datasets/icl.py:467-513; tum.py and scannet.py alike).  16-byte aligned
 * buffers take the vectorised path.  The image resize the loaders can also perform is not covered (pass frames at their final size). */
int gsx_ingest_raw(const uint8_t *rgb_u8, const uint16_t *depth_u16, int64_t n_pixels, double depth_scaling_factor,
                   int normalize_color, float *rgb_out, float *depth_out, void *stream);

/* The arithmetic part of the loaders' calibration contract, on the device (either half may be skipped with NULL outputs):
 *   intrinsics_out[i] = intrinsics[i] with fx, cx scaled by w_ratio and fy, cy by h_ratio, in float32
 *                       (gradslam/datasets/datautils.py:73-122 scale_intrinsics; n_intrinsics matrices of
 *                       intrinsics_dim x intrinsics_dim, 3 or 4);
 *   poses_out[b][l]   = compose(inverse(poses[b][0]), poses[b][l]) with the bottom row forced to 0 0 0 1
 *                       (gradslam/datasets/icl.py:515-533 _preprocess_poses = geometryutils.relative_transformation with
 *                       a general 4x4 inverse); *singular_flag (int32, may be NULL) is set to 1 if a first pose is singular. */
int gsx_ingest_calibration(const float *intrinsics, int64_t n_intrinsics, int intrinsics_dim, double h_ratio,
                           double w_ratio, float *intrinsics_out, const float *poses, int B, int L, float *poses_out,
                           int32_t *singular_flag, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Table-returning association steps (API parity with gradslam's module-level helpers; the fused path
 * above never materialises these tables).  Tables are int64 (rows,4) with rows [b, n, h, w].
 * replaces find_active_map_points gradslam/slam/fusionutils.py:198-287 (gsx_active_eval + compaction),
 *          find_similar_map_points :290-411 (gsx_similar_eval + compaction),
 *          find_best_unique_correspondences :414-546 (gsx_unique_select + compaction, replacing the
 *          torch.unique(dim=0) row sort), and the scatter of fuse_with_map :659-676, 702-704
 *          (gsx_records_from_table, followed by gsx_fusion_merge_append).                              */

/* stable compaction: ascending indices i with flags[i] != 0 -> out_idx, their number -> *out_count (int64,
 * device).  scratch: gsx_compact_scratch_bytes(n) bytes, zero-filled by the caller; epoch >= 1, unique per
 * call on the same scratch. */
int64_t gsx_compact_scratch_bytes(int64_t n);
int gsx_compact_indices(const uint8_t *flags, int64_t n, int64_t *out_idx, int64_t *out_count, void *scratch,
                        uint32_t epoch, void *stream);

/* per map slot (b, n < width): 1 if the point is a valid map point inside the live frustum; hw = h*W + w
 * of the pixel it rounds to.  flags, hw: (B, width). */
int gsx_active_eval(const float *map_geometry, const int32_t *counts, int64_t capacity, int64_t width,
                    const float *poses, int64_t pose_bstride, const float *intrinsics, int64_t K_bstride, int B,
                    int H, int W, uint8_t *flags, int32_t *hw, void *stream);

/* per table row: 1 if ||frame vertex - map point|| < dist_th and <frame normal, map normal> > dot_th. */
int gsx_similar_eval(const int64_t *table, int64_t rows, const float *map_geometry, int64_t capacity,
                     const float *gvertex, const float *gnormal, int B, int H, int W, float dist_th, float dot_th,
                     uint8_t *flags, void *stream);

/* per pixel winner among the table rows (largest ccount, then smallest ray distance, then smallest n):
 * pixel_flags (B*H*W) and pixel_n (B*H*W, -1 if none).  records: scratch of B*H*W 16-byte records, 16-byte
 * aligned (cleared by the call). */
int gsx_unique_select(const int64_t *table, int64_t rows, const float *map_geometry, int64_t capacity,
                      const float *gvertex, int B, int H, int W, void *records, uint8_t *pixel_flags,
                      int64_t *pixel_n, void *stream);

/* stores every table row as its pixel's winner in the fusion workspace: call it AFTER gsx_fusion_frame_records
 * (which re-arms the workspace) and BEFORE gsx_fusion_merge_append. */
int gsx_records_from_table(const int64_t *table, int64_t rows, int64_t capacity, int B, int H, int W,
                           void *workspace, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Point-to-plane ICP / gradICP odometry (K5 exact 1-NN, K6 residual+Jacobian rows and the 6x6 normal
 * equations, K7 damped solve + se3_exp + LM / gradLM update), batched over B, no host synchronisation.
 * replaces chamferdist.chamfer.knn_points (third party, call site gradslam/odometry/icputils.py:200),
 *          gauss_newton_solve :93-232, solve_linear_system :22-90, point_to_plane_ICP :235-367,
 *          point_to_plane_gradICP :370-545, se3utils.se3_exp gradslam/geometry/se3utils.py:77-115,
 *          transform_pointcloud gradslam/geometry/geometryutils.py:737-794 and the per-element Python loops
 *          of ICPOdometryProvider.provide / GradICPOdometryProvider.provide (odometry/icp.py:84-97,
 *          odometry/gradicp.py:105-122).
 *
 * Clouds are padded (B, stride, 3) float32 with int32 (B) sizes.  mode 0 = LM accept/reject (ICP),
 * mode 1 = gradLM (gradICP; lambda_max, B, B2, nu as in the reference).  use_dist_thresh = 0 means
 * dist_thresh=None; otherwise the SQUARED nn distance is compared with dist_thresh exactly as the
 * reference does (icputils.py:206).  Exact 1-NN ties resolve to the lowest target index.            */

/* exact nearest neighbour of every source point: idx_out int64 (B, ns_stride) (-1 for rows >= size or an
 * empty target), d2_out squared distance (may be NULL).  scratch: gsx_knn1_scratch_bytes bytes.
 * Target clouds with nt_stride > 4096 are binned into a uniform grid and searched ring by ring with an exact
 * termination bound (full scan as the fallback); smaller ones are scanned from shared memory.  Both return
 * the same (distance, index): candidates are ordered by (squared distance, index).
 * build_grid: 1 = bin the target into `scratch` first; 0 = `scratch` still holds the grid that an earlier call built
 * for the same target (the ICP loop queries one target 2 x numiters times). */
int64_t gsx_knn1_scratch_bytes(int B, int ns_stride, int nt_stride);
int gsx_knn1(const float *src_points, const int32_t *src_count, int ns_stride, const float *tgt_points,
             const int32_t *tgt_count, int nt_stride, int B, int64_t *idx_out, float *d2_out, void *scratch,
             int64_t scratch_bytes, int build_grid, void *stream);

/* K6 as a differentiable op on padded clouds (B, stride, 3) with int32 sizes (NULL = all rows): for a GIVEN
 * association nn_idx (int64 (B, ns_stride), -1 = row unused) reduce the point-to-plane rows A_i = [n, s x n],
 * r_i = n.(p - s) (gauss_newton_solve, icputils.py:210-230) to the 28 sums (B,28)
 * [upper triangle of A^T A (21, row-major), A^T r (6), r^T r] (the matmuls of solve_linear_system, icputils.py:85-90).
 * Backward: from d(loss)/d(sums) the gradient w.r.t. every source point (B, ns_stride, 3) and, per SOURCE row,
 * w.r.t. its associated target point and normal (B, ns_stride, 3 each; the caller scatter-adds them through nn_idx).
 * One launch for all elements (the differentiable mode's op chain is recorded ONCE for the batch instead of once per
 * element, which is what the reference's providers do, odometry/icp.py:84-97); a single cloud is B = 1.  Padding rows
 * get zero outputs / zero gradients.  Deterministic, no atomics.
 * scratch: B * gsx_icp_normal_eq_scratch_bytes(ns_stride) bytes. */
int64_t gsx_icp_normal_eq_scratch_bytes(int ns);
int gsx_icp_normal_eq_batched_fwd(const float *src_points, const int32_t *src_count, int ns_stride,
                                  const float *tgt_points, const float *tgt_normals, int nt_stride, int B,
                                  const int64_t *nn_idx, float *sums_out, void *scratch, int64_t scratch_bytes,
                                  void *stream);
int gsx_icp_normal_eq_batched_bwd(const float *src_points, const int32_t *src_count, int ns_stride,
                                  const float *tgt_points, const float *tgt_normals, int nt_stride, int B,
                                  const int64_t *nn_idx, const float *g_sums, float *g_src, float *g_tgt_points_rows,
                                  float *g_tgt_normals_rows, void *stream);

/* K7 as differentiable ops (n independent problems; every array is dense float32, device):
 * _solve_: xi = (A^T A + damp I)^-1 A^T b from the 28 sums of gsx_icp_normal_eq_batched_fwd and damp (n), then
 *          dT = se3_exp(xi).
 *          replaces solve_linear_system   gradslam/odometry/icputils.py:22-90  and  se3_exp  geometry/se3utils.py:77-115
 * _update_: mode 0 = LM accept / reject (icputils.py:356-365): new_err < err -> applied step se3_exp(xi), damp / 2,
 *          else identity, damp * 2;  mode 1 = gradLM gates (icputils.py:519-543): diff = clamp(new_err - err, +-70),
 *          damp * (1/lambda_max + (lambda_max - 1/lambda_max) / (1 + exp(-B diff))), applied step
 *          se3_exp(xi / (1 + exp(-B2 diff))^(1/nu)).  Outputs: new damp (n), applied step (n,16), T_out = step * T (n,16).
 * The backward entries take the forward inputs again plus the upstream gradients (any may be NULL = zero) and write
 * the gradient of every forward input (same arithmetic evaluated on dual numbers, one lane per input). */
int gsx_icp_solve_fwd(const float *sums, const float *damp, int n, float *xi_out, float *dT_out, void *stream);
int gsx_icp_solve_bwd(const float *sums, const float *damp, int n, const float *g_xi, const float *g_dT,
                      float *g_sums, float *g_damp, void *stream);
int gsx_icp_update_fwd(const float *xi, const float *err, const float *new_err, const float *damp, const float *T,
                       int n, int mode, float lambda_max, float B, float B2, float nu, float *damp_out,
                       float *dT_out, float *T_out, void *stream);
int gsx_icp_update_bwd(const float *xi, const float *err, const float *new_err, const float *damp, const float *T,
                       int n, int mode, float lambda_max, float B, float B2, float nu, const float *g_damp_out,
                       const float *g_dT_out, const float *g_T_out, float *g_xi, float *g_err, float *g_new_err,
                       float *g_damp, float *g_T, void *stream);

/* out = R p + t for padded clouds points (B, stride, 3) with int32 sizes counts (B) (NULL = all rows) and T (B,4,4);
 * padding rows are written as zeros.  backward: g_points = R^T g (zero on padding rows), g_T = sum_i g_i (x) [p_i; 1]
 * (fixed-order reduction; bottom row zero).  scratch: B * gsx_rigid_transform_bwd_scratch_bytes(stride) bytes.
 *          replaces transform_pointcloud   gradslam/geometry/geometryutils.py:737-794 */
int64_t gsx_rigid_transform_bwd_scratch_bytes(int64_t n);
int gsx_rigid_transform_batched_fwd(const float *points, const int32_t *counts, int64_t stride, int B, const float *T,
                                    float *out, void *stream);
int gsx_rigid_transform_batched_bwd(const float *points, const int32_t *counts, int64_t stride, int B, const float *T,
                                    const float *g_out, float *g_points, float *g_T, void *scratch,
                                    int64_t scratch_bytes, void *stream);

/* full ICP / gradICP on given clouds.  initial_transform (B,16) or NULL (identity).  transform_out (B,16).
 * nn_idx_out optional int64 (B, ns_stride): association of the last iteration (-1 = filtered out).
 * scratch: gsx_icp_align_scratch_bytes(B, ns_stride, nt_stride) bytes. */
int64_t gsx_icp_align_scratch_bytes(int B, int ns_stride, int nt_stride);
int gsx_icp_align(const float *src_points, const int32_t *src_count, int ns_stride, const float *tgt_points,
                  const float *tgt_normals, const int32_t *tgt_count, int nt_stride, int B,
                  const float *initial_transform, int mode, int numiters, float damp, int use_dist_thresh,
                  float dist_thresh, float lambda_max, float Bp, float B2p, float nu, float *transform_out,
                  int64_t *nn_idx_out, void *scratch, int64_t scratch_bytes, void *stream);

/* ICPSLAM._localize for odom in {icp, gradicp} (gradslam/slam/icpslam.py:238-247) as one call:
 * source cloud = live depth on the ds-lattice placed at the previous pose (downsample_rgbdimages,
 * icputils.py:623-669); target cloud = map points inside the previous frame's frustum that land on the
 * ds-lattice (find_active_map_points + downsample_pointclouds, fusionutils.py:198-287,
 * icputils.py:548-620); ICP loop; poses_out[b] = T_icp[b] * prev_poses[b].
 * tgt_scratch: gsx_icp_tgt_scratch_bytes(B, tgt_capacity) bytes (target points, normals, search grid);
 * *overflow_flag is set to 1 if a target cloud did not fit tgt_capacity (surplus dropped).  workspace:
 * gsx_icp_workspace_bytes(B,H,W,ds,workspace_map_capacity) bytes zero-filled once (pass the same
 * workspace_map_capacity >= max_count on every call: it fixes the layout); `epoch` increases by one per
 * call on the same workspace, starting at 1. */
int64_t gsx_icp_workspace_bytes(int B, int H, int W, int ds, int64_t map_capacity);
int64_t gsx_icp_tgt_scratch_bytes(int B, int64_t tgt_capacity);
int gsx_icp_localize(const float *map_geometry, const int32_t *counts, int64_t capacity, int64_t max_count, const float *depth, int64_t depth_bstride, const float *intrinsics,
                     int64_t K_bstride, const float *prev_poses, int64_t prev_pose_bstride, int B, int H, int W,
                     int ds, int mode, int numiters, float damp, int use_dist_thresh, float dist_thresh,
                     float lambda_max, float Bp, float B2p, float nu, void *tgt_scratch, int64_t tgt_capacity,
                     float *poses_out, int64_t poses_out_bstride, void *workspace,
                     int64_t workspace_map_capacity, uint32_t epoch, int32_t *overflow_flag, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* GSX_H_ */
