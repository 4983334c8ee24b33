/* d3d_b200.h -- C ABI of the B200-native d3d hot path (libd3d_b200.so).
 *
 * Drop-in boundary for the three data-parallel geometry operators of cmpute/d3d.  Every entry point
 * replaces one native function the reference's Python packages import from their pybind11 modules
 * (cited per function as reference file:line).  Conventions:
 *   - plain pointers and sizes only; all data pointers are DEVICE pointers unless the name says host;
 *   - the library never allocates user-visible memory: outputs and scratch ("workspace") are caller
 *     provided, `*_workspace_bytes` tells how much scratch a call needs;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*), re-entrant, no globals;
 *   - return value: D3D_OK or a D3D_ERR_* code (never exit(), unlike reference d3d/common.h:33-46);
 *     d3d_error_string() names the code; d3d_last_cuda_error() returns the CUDA error text of the
 *     calling thread's last D3D_ERR_CUDA.
 *   - box rows are (x, y, w, h, r) contiguous, row-major, like reference d3d/box/__init__.py:184-185.
 * Built for sm_100a only; there is no CPU fallback.
 */
#ifndef D3D_B200_H
#define D3D_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define D3D_B200_ABI_VERSION 5   /* 5: + d3d_aligned_scatter_*_ws (tile path); 4: + differentiable IoU family, soft-NMS, d3d_nms2d_batch_*, d3d_pdist2dr_*, d3d_match_greedy_f32, voxel algo TILES */

enum d3d_status {
    D3D_OK = 0,
    D3D_ERR_INVALID_ARGUMENT = 1, /* reference raises ValueError / py::value_error */
    D3D_ERR_CUDA = 2,             /* a CUDA runtime call failed */
    D3D_ERR_WORKSPACE = 3,        /* workspace smaller than *_workspace_bytes() */
    D3D_ERR_UNSUPPORTED = 4,      /* e.g. FARTHEST_SAMPLING (reference throws, voxelize.cpp:468-471) */
    D3D_ERR_RANGE = 5             /* voxel grid too large for the 63-bit voxel key */
};

/* reference d3d/box/common.h:5-10 (same integer values) */
enum d3d_iou_type { D3D_IOU_NA = 0, D3D_IOU_BOX = 1, D3D_IOU_RBOX = 2, D3D_IOU_GBOX = 3, D3D_IOU_GRBOX = 4, D3D_IOU_DBOX = 5, D3D_IOU_DRBOX = 6 };
enum d3d_supression_type { D3D_SUP_HARD = 0, D3D_SUP_LINEAR = 1, D3D_SUP_GAUSSIAN = 2 };
/* reference d3d/voxel/voxelize.h:5-7 */
enum d3d_reduction_type { D3D_RED_NONE = 0, D3D_RED_MEAN = 1, D3D_RED_MAX = 2, D3D_RED_MIN = 3 };
enum d3d_max_points_filter { D3D_PF_NONE = 0, D3D_PF_TRIM = 1, D3D_PF_FARTHEST_SAMPLING = 2 };
enum d3d_max_voxels_filter { D3D_VF_NONE = 0, D3D_VF_TRIM = 1, D3D_VF_DESCENDING = 2 };
/* reference d3d/point/scatter.h:37 */
enum d3d_align_type { D3D_ALIGN_DROP = 0, D3D_ALIGN_MEAN = 1, D3D_ALIGN_LINEAR = 2, D3D_ALIGN_MAX = 3, D3D_ALIGN_NEAREST = 4 };
enum d3d_dtype { D3D_F32 = 0, D3D_F64 = 1 };
/* voxelization back ends: a software pipeline of streaming tiles (default fast path: sparse, no voxel cap, TRIM up
 * to 8 points per voxel), one thread-block cluster per frame with a hash table, or the sort / segmented-scan
 * pipeline (general).  All produce identical, deterministic outputs. */
enum d3d_voxel_algo { D3D_VOXEL_AUTO = 0, D3D_VOXEL_SORT = 1, D3D_VOXEL_CLUSTER = 2, D3D_VOXEL_TILES = 3,
                      D3D_VOXEL_AUTO_NO_TILES = 4 /* AUTO restricted to the cluster and sort back ends (A/B runs, tests) */ };

int d3d_abi_version(void);
const char *d3d_error_string(int status);
const char *d3d_last_cuda_error(void);
/* Tuning knobs force one of the back ends that produce identical results (names = the environment variables D3D_B200_NMS_PATH
 * (tiles | dense), D3D_B200_NMS_FIX (0 | 1: resolve by the block walk | the pulled parallel fixpoint; batched NMS: 2 = rounds over the
 * edge list), D3D_B200_NMS_BATCH_PATH (dense), D3D_B200_SORT_COOP (0 | 1 | 2), D3D_B200_CROP_PATH (brute | grid), D3D_B200_SCATTER_PATH
 * (gather | tiles), D3D_B200_VOX_ROUTE (0), and D3D_B200_NMS_STOP, which truncates d3d_nms2d_* after a phase for phase timing and so
 * is the one knob that changes a result).  The environment is read once, at the first use of a knob; this call overrides (set != 0) or
 * clears (set == 0) a knob afterwards -- tests and tuning tools use it instead of changing the environment of a running process.
 * An unknown name returns D3D_ERR_INVALID_ARGUMENT. */
int d3d_tuning_set(const char *name, int value, int set);
/* number of kernels this library has launched in the calling process (bench.py's gpu_launches) */
int64_t d3d_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * Pairwise IoU.  ious is [n, m] row-major with leading dimension ld (elements, ld >= m).
 * d3d_iou2dr_*: rotated IoU, replaces iou2dr_forward[_cuda] (reference d3d/box/iou.h:14-16,
 *   iou.cpp:94-141, iou_cuda.cu:99-151).  The backward-only outputs nx/xflags are not produced (d3d_iou2dr_backward_* recomputes).
 * d3d_iou2d_*: IoU of the axis-aligned bounding boxes of the rotated boxes, replaces
 *   iou2d_forward[_cuda] (iou.h:7-9, iou.cpp:11-46, iou_cuda.cu:9-48).
 * Row-block sharding (multi-GPU): pass a slice of boxes1 and the matching slab of ious.
 * ---------------------------------------------------------------------------------------------- */
size_t d3d_iou_workspace_bytes(int64_t n, int64_t m, int dtype);
int d3d_iou2dr_f32(const float *boxes1, int64_t n, const float *boxes2, int64_t m, float *ious, int64_t ld,
                   void *workspace, size_t workspace_bytes, void *stream);
int d3d_iou2dr_f64(const double *boxes1, int64_t n, const double *boxes2, int64_t m, double *ious, int64_t ld,
                   void *workspace, size_t workspace_bytes, void *stream);
int d3d_iou2d_f32(const float *boxes1, int64_t n, const float *boxes2, int64_t m, float *ious, int64_t ld,
                  void *workspace, size_t workspace_bytes, void *stream);
int d3d_iou2d_f64(const double *boxes1, int64_t n, const double *boxes2, int64_t m, double *ious, int64_t ld,
                  void *workspace, size_t workspace_bytes, void *stream);
/* Differentiable IoU family (SURVEY.md 8(a) row A2, 8(f) row f2).
 * d3d_giou2dr_* / d3d_diou2dr_*: rotated generalized / distance IoU, [n, m] with leading dimension ld; replace giou2dr_forward[_cuda] /
 *   diou2dr_forward[_cuda] (reference d3d/box/iou.h:24-26, 34-36, iou.cpp:202-243, 311-352; dgal::giou / diou geometry.hpp:1232-1291:
 *   GIoU = I/U + U/M - 1 with M the area of the convex hull of both boxes, DIoU = I/U - |c1 - c2|^2 / D^2 with D the largest vertex distance).
 *   The backward-only outputs (nxm / nxd, flags) are not produced: the backward recomputes what it needs.
 * d3d_*_backward_*: gradients of sum(grad * value) with respect to both box arrays; replace iou2d_backward, iou2dr_backward,
 *   giou2dr_backward, diou2dr_backward [_cuda] (iou.h:10-12, 17-20, 27-30, 37-40, iou.cpp:48-92, 143-200, 245-309, 354-419; dgal::iou_grad /
 *   giou_grad / diou_grad, geometry_grad.hpp:327-606).  grad [n, m] with leading dimension ld; grad_boxes1 [n,5] and grad_boxes2 [m,5] are
 *   WRITTEN (not accumulated).  One warp owns one box and sums its row / column in a fixed order: results are deterministic, there is no
 *   atomic and no race (the reference adds pair gradients into the box rows from all threads, iou_cuda.cu:184-185). */
int d3d_giou2dr_f32(const float *boxes1, int64_t n, const float *boxes2, int64_t m, float *out, int64_t ld, void *stream);
int d3d_giou2dr_f64(const double *boxes1, int64_t n, const double *boxes2, int64_t m, double *out, int64_t ld, void *stream);
int d3d_diou2dr_f32(const float *boxes1, int64_t n, const float *boxes2, int64_t m, float *out, int64_t ld, void *stream);
int d3d_diou2dr_f64(const double *boxes1, int64_t n, const double *boxes2, int64_t m, double *out, int64_t ld, void *stream);
int d3d_iou2d_backward_f32(const float *boxes1, int64_t n, const float *boxes2, int64_t m, const float *grad, int64_t ld, float *grad_boxes1,
                           float *grad_boxes2, void *stream);
int d3d_iou2d_backward_f64(const double *boxes1, int64_t n, const double *boxes2, int64_t m, const double *grad, int64_t ld, double *grad_boxes1,
                           double *grad_boxes2, void *stream);
int d3d_iou2dr_backward_f32(const float *boxes1, int64_t n, const float *boxes2, int64_t m, const float *grad, int64_t ld, float *grad_boxes1,
                            float *grad_boxes2, void *stream);
int d3d_iou2dr_backward_f64(const double *boxes1, int64_t n, const double *boxes2, int64_t m, const double *grad, int64_t ld, double *grad_boxes1,
                            double *grad_boxes2, void *stream);
int d3d_giou2dr_backward_f32(const float *boxes1, int64_t n, const float *boxes2, int64_t m, const float *grad, int64_t ld, float *grad_boxes1,
                             float *grad_boxes2, void *stream);
int d3d_giou2dr_backward_f64(const double *boxes1, int64_t n, const double *boxes2, int64_t m, const double *grad, int64_t ld, double *grad_boxes1,
                             double *grad_boxes2, void *stream);
int d3d_diou2dr_backward_f32(const float *boxes1, int64_t n, const float *boxes2, int64_t m, const float *grad, int64_t ld, float *grad_boxes1,
                             float *grad_boxes2, void *stream);
int d3d_diou2dr_backward_f64(const double *boxes1, int64_t n, const double *boxes2, int64_t m, const double *grad, int64_t ld, double *grad_boxes1,
                             double *grad_boxes2, void *stream);
/* Frame-batched differentiable IoU family (a detector computes it once per frame of every training batch: target assignment, IoU / GIoU /
 * DIoU losses).  Frames are packed back to back: boxes1 T[total1,5] / boxes2 T[total2,5] with DEVICE offsets1 / offsets2 i64[nframes+1]
 * (frame f owns rows [offsets[f], offsets[f+1]), n_f and m_f of them).  out_offsets DEVICE i64[nframes+1]: frame f's block is the row-major
 * [n_f, m_f] matrix at out + out_offsets[f] (leading dimension m_f), usually at the running sum of n_f * m_f.  iou_type: D3D_IOU_BOX (IoU of
 * the axis-aligned bounding boxes), D3D_IOU_RBOX, D3D_IOU_GRBOX or D3D_IOU_DRBOX; anything else: D3D_ERR_INVALID_ARGUMENT.  Per frame, the
 * block equals d3d_iou2d_* / d3d_iou2dr_* / d3d_giou2dr_* / d3d_diou2dr_* on that frame bit for bit, and the backward's gradients equal
 * d3d_*_backward_* on that frame bit for bit: the frames run the same per-pair code, and the backward the same warp per owned box with the
 * same summation order.  max_frame1 / max_frame2: HARD UPPER BOUNDS of n_f / m_f (0 = unknown, assume total1 / total2); they size the launch
 * grid.  The RBOX forward skips a frame beyond them (n_f > max_frame1 or m_f > max_frame2): its block is not written, so a caller can pass
 * the bounds of the frames that fit the tile grid and run d3d_iou2dr_* on the others.  Elsewhere a frame beyond them may be written only
 * in part.  No limit on nframes below 2^31, nor on the frame sizes except for RBOX.
 * Forward: "box" and "rbox" two box preparations and one IoU launch, "grbox" / "drbox" one launch and no workspace (may be NULL).  Workspace
 * below d3d_box2d_iou_batch_workspace_bytes for BOX / RBOX: D3D_ERR_WORKSPACE.  RBOX frames over 65535 tiles of 64 rows or of 128 (fp32) /
 * 64 (fp64) columns: D3D_ERR_UNSUPPORTED (call d3d_iou2dr_* on such frames).  Negative sizes: D3D_ERR_INVALID_ARGUMENT; nframes == 0 or an
 * empty side: no-op.
 * Backward: two launches, no workspace.  grad T has the layout of out; grad_boxes1 T[total1,5] / grad_boxes2 T[total2,5] are WRITTEN (not
 * accumulated), every box included: the boxes of a frame whose other side is empty get exact zeros. */
size_t d3d_box2d_iou_batch_workspace_bytes(int64_t total1, int64_t total2, int64_t nframes, int dtype);
int d3d_box2d_iou_batch_f32(const float *boxes1, int64_t total1, const int64_t *offsets1, const float *boxes2, int64_t total2,
                            const int64_t *offsets2, int64_t nframes, int64_t max_frame1, int64_t max_frame2, int iou_type,
                            const int64_t *out_offsets, float *out, void *workspace, size_t workspace_bytes, void *stream);
int d3d_box2d_iou_batch_f64(const double *boxes1, int64_t total1, const int64_t *offsets1, const double *boxes2, int64_t total2,
                            const int64_t *offsets2, int64_t nframes, int64_t max_frame1, int64_t max_frame2, int iou_type,
                            const int64_t *out_offsets, double *out, void *workspace, size_t workspace_bytes, void *stream);
int d3d_box2d_iou_batch_backward_f32(const float *boxes1, int64_t total1, const int64_t *offsets1, const float *boxes2, int64_t total2,
                                     const int64_t *offsets2, int64_t nframes, int64_t max_frame1, int64_t max_frame2, int iou_type,
                                     const int64_t *out_offsets, const float *grad, float *grad_boxes1, float *grad_boxes2, void *stream);
int d3d_box2d_iou_batch_backward_f64(const double *boxes1, int64_t total1, const int64_t *offsets1, const double *boxes2, int64_t total2,
                                     const int64_t *offsets2, int64_t nframes, int64_t max_frame1, int64_t max_frame2, int iou_type,
                                     const int64_t *out_offsets, const double *grad, double *grad_boxes1, double *grad_boxes2, void *stream);
/* Fused max-IoU reduction (target assignment: each anchor / proposal's best ground truth and each ground truth's best anchor), without
 * the IoU matrix.  Boxes, offsets, max_frame1 / max_frame2 and iou_type as for d3d_box2d_iou_batch_*, except that iou_type is D3D_IOU_BOX
 * or D3D_IOU_RBOX only.  Outputs: max1 [total1] / idx1 i64[total1] and max2 [total2] / idx2 i64[total2] (DEVICE), of dtype out_dtype:
 * D3D_F32, or D3D_F64 for the f64 entry (fp32 boxes computed in fp64 and rounded to fp32: pass fp64 boxes and D3D_F32).  For box i of
 * frame f, max1[i] / idx1[i] are the value and FRAME-LOCAL column index that torch.max(block, dim=1) returns for frame f's block of
 * d3d_box2d_iou_batch_* rounded to out_dtype; max2 / idx2 those of dim=0.  So ties (+0 against -0 included) go to the lower index, and
 * NaN is the maximum, at the first NaN's index.  A box whose frame's other side is empty gets (0, -1).  Rows and columns reduce inside
 * the tiles and combine across tiles through atomics on an order-preserving (value, index) key; the result does not depend on the
 * schedule.  Every frame size works: frames of more than 65535 tiles on an axis take more than one tile launch.  An init, two box
 * preparations, the tile launches (one per 65535 x 65535 tiles of the largest frame) and a finalise, whatever the number of frames.
 * max_frame1 / max_frame2 are HARD UPPER BOUNDS (0 = unknown, assume total1 / total2); a frame beyond them has undefined results.
 * Invalid iou_type or out_dtype, or negative sizes: D3D_ERR_INVALID_ARGUMENT; workspace below d3d_box2d_iou_max_batch_workspace_bytes
 * (dtype = the boxes' dtype): D3D_ERR_WORKSPACE; nframes > 2^31 - 1, or a D3D_F32 output with a frame of 2^32 boxes or more:
 * D3D_ERR_UNSUPPORTED.  nframes == 0 or no box: no-op. */
size_t d3d_box2d_iou_max_batch_workspace_bytes(int64_t total1, int64_t total2, int64_t nframes, int dtype);
int d3d_box2d_iou_max_batch_f32(const float *boxes1, int64_t total1, const int64_t *offsets1, const float *boxes2, int64_t total2,
                                const int64_t *offsets2, int64_t nframes, int64_t max_frame1, int64_t max_frame2, int iou_type, int out_dtype,
                                void *max1, int64_t *idx1, void *max2, int64_t *idx2, void *workspace, size_t workspace_bytes, void *stream);
int d3d_box2d_iou_max_batch_f64(const double *boxes1, int64_t total1, const int64_t *offsets1, const double *boxes2, int64_t total2,
                                const int64_t *offsets2, int64_t nframes, int64_t max_frame1, int64_t max_frame2, int iou_type, int out_dtype,
                                void *max1, int64_t *idx1, void *max2, int64_t *idx2, void *workspace, size_t workspace_bytes, void *stream);
/* Detection-evaluation distance matrix (SURVEY.md 8(f) row f1): dist[i][j] = 1 - iou2d(BEV boxes) * ziou, fp32,
 * for 3-D boxes [n,7] / [m,7] with rows (x, y, z, lx, ly, lz, rz).  rotated != 0: rotated BEV IoU, replaces the pair
 * loop over box3dr_iou in ScoreMatcher.prepare_boxes (reference d3d/tracking/matcher.pyx:66-76, d3d/dgal_wrap.h:45-68);
 * rotated == 0: IoU of the BEV axis-aligned boxes, replaces the loop over box3d_iou (matcher.pyx:55-65,
 * dgal_wrap.h:70-91).  Same tile kernel as the IoU matrix; the z factor is applied to the clipped candidate pairs only
 * (a rejected pair is the constant 1), which costs ~19 % over the plain IoU matrix. */
size_t d3d_iou3d_distance_workspace_bytes(int64_t n, int64_t m);
int d3d_iou3d_distance_f32(const float *boxes1, int64_t n, const float *boxes2, int64_t m, int rotated, float *dist,
                           int64_t ld, void *workspace, size_t workspace_bytes, void *stream);
/* Greedy score-ordered matching over a distance matrix (SURVEY.md 8(f) row f1): replaces the pair walk of ScoreMatcher.match +
 * BaseMatcher.match_by_order (reference d3d/tracking/matcher.pyx:93-122, 138-162) that the detection evaluator repeats for every score
 * threshold (d3d/benchmarks.pyx:220-238).  dist f32[n, m] with leading dimension ld (the matrix d3d_iou3d_distance_f32 writes);
 * src_order i32[n] = source indices from the best score down; src_tag i32[n], dst_tag i32[m] = category indices in [0, ncat);
 * thresholds f32[nsets, ncat]: set t matches a pair when dist <= thresholds[t][category].  Outputs (device) src_assign i32[nsets, n],
 * dst_assign i32[nsets, m]: the partner's index or -1.  Each source takes the closest free destination of its category within the
 * threshold; equal distances go to the lower destination index.  One CTA per threshold set. */
int d3d_match_greedy_f32(const float *dist, int64_t n, int64_t m, int64_t ld, const int32_t *src_order, const int32_t *src_tag,
                         const int32_t *dst_tag, const float *thresholds, int32_t nsets, int32_t ncat, int32_t *src_assign,
                         int32_t *dst_assign, void *stream);
/* Frame-batched evaluator distance matrix and matching (the detection evaluator runs both once per frame of a validation set).
 * Frames are packed back to back: boxes1 f32[total1,7] / boxes2 f32[total2,7] with DEVICE offsets1 / offsets2 i64[nframes+1]
 * (frame f owns rows [offsets[f], offsets[f+1]), n_f and m_f of them).  dist_offsets DEVICE i64[nframes+1]: frame f's block is the
 * row-major [n_f, m_f] matrix at dist + dist_offsets[f] (leading dimension m_f); the caller chooses the layout, usually the running sum
 * of n_f * m_f.  max_frame1 / max_frame2: HARD UPPER BOUNDS of n_f / m_f (0 = unknown, assume total1 / total2); they size the launch
 * grid, and the part of a frame beyond them is not written.  Per frame, the block equals d3d_iou3d_distance_f32 on that frame bit for bit,
 * for rotated != 0 and rotated == 0: the frames run the same tile body, reject test and clip.  One prep launch per box set and one
 * distance launch for the whole batch (rotated == 0: one per 65535 rows of the largest frame).  nframes == 0 or an empty box set: no-op.
 * Negative sizes: D3D_ERR_INVALID_ARGUMENT; workspace below d3d_iou3d_distance_batch_workspace_bytes: D3D_ERR_WORKSPACE;
 * nframes > 2^31 - 1, rotated frames over 65535 tiles (64 rows / 128 columns) or axis-aligned frames over 65535 x 1024 columns:
 * D3D_ERR_UNSUPPORTED. */
size_t d3d_iou3d_distance_batch_workspace_bytes(int64_t total1, int64_t total2, int64_t nframes);
int d3d_iou3d_distance_batch_f32(const float *boxes1, int64_t total1, const int64_t *offsets1, const float *boxes2, int64_t total2,
                                 const int64_t *offsets2, int64_t nframes, int64_t max_frame1, int64_t max_frame2, int rotated,
                                 const int64_t *dist_offsets, float *dist, void *workspace, size_t workspace_bytes, void *stream);
/* d3d_match_greedy_f32 on every frame of a packed batch in one launch: dist and dist_offsets as written by d3d_iou3d_distance_batch_f32,
 * src_offsets / dst_offsets DEVICE i64[nframes+1] (total_src = src_offsets[nframes], total_dst = dst_offsets[nframes]).  src_order i32
 * [total_src] holds, per frame, the FRAME-LOCAL source indices from the best score down; src_tag i32[total_src] / dst_tag i32[total_dst]
 * are packed like the boxes; thresholds f32[nsets, ncat] are shared by all frames.  Outputs src_assign i32[nsets, total_src] /
 * dst_assign i32[nsets, total_dst]: the frame-local partner index or -1.  Per frame and threshold set, the result equals
 * d3d_match_greedy_f32 on the frame's block (d <= threshold, so a NaN distance never matches; equal distances go to the lower
 * destination index; a source whose tag is outside [0, ncat) matches nothing).  One warp per (frame, threshold set) with its taken flags
 * as a bitmask in shared memory.  max_frame_dst: HARD UPPER BOUND of the frames' destination counts; more than 4096:
 * D3D_ERR_UNSUPPORTED (call d3d_match_greedy_f32 per frame); a frame over 4096 destinations despite the bound stays unmatched.
 * Negative sizes or ncat < 1: D3D_ERR_INVALID_ARGUMENT; nframes == 0 or nsets == 0: no-op. */
int d3d_match_greedy_batch_f32(const float *dist, const int64_t *dist_offsets, const int64_t *src_offsets, const int64_t *dst_offsets,
                               int64_t nframes, int64_t max_frame_dst, const int32_t *src_order, const int32_t *src_tag,
                               const int32_t *dst_tag, const float *thresholds, int32_t nsets, int32_t ncat, int32_t *src_assign,
                               int32_t *dst_assign, void *stream);
/* Point-in-rotated-box mask (SURVEY.md 8(f) row f4): mask u8[m boxes, n points] row-major, 1 where the point lies inside
 * the box.  points [n,2], boxes [m,5] (x, y, w, h, r).  Replaces crop_2dr (reference d3d/box/utils.h:45, utils.cpp:10-47,
 * bound at d3d/box/impl.cpp:26 and called by box2dr_crop / box3dp_crop, d3d/box/__init__.py:278-314); the reference
 * has no CUDA version.  Same decision rule as dgal: open AABB test, then no edge with a negative cross product.
 * Large problems bin the points into a grid first and zero-fill the mask; the result does not depend on the back end. */
size_t d3d_crop2dr_workspace_bytes(int64_t n, int64_t m, int dtype);
int d3d_crop2dr_f32(const float *points, int64_t n, const float *boxes, int64_t m, uint8_t *mask, void *workspace,
                    size_t workspace_bytes, void *stream);
int d3d_crop2dr_f64(const double *points, int64_t n, const double *boxes, int64_t m, uint8_t *mask, void *workspace,
                    size_t workspace_bytes, void *stream);
/* Signed distance from points to rotated boxes (SURVEY.md 8(f) row f4): dist T[m boxes, n points] row-major, positive inside;
 * iedge u8[m, n] (may be NULL) = edge of the box that realises the distance (edge k runs from vertex k to vertex k+1 of
 * dgal::poly2_from_xywhr).  points [n,2], boxes [m,5].  Replaces pdist2dr_forward[_cuda] (reference d3d/box/dist.h:7-9,16-18,
 * dist.cpp:11-47, dist_cuda.cu:9-50; dgal::distance geometry.hpp:453-497) behind box2dr_pdist / box3dr_pdist
 * (d3d/box/__init__.py:149-166, 330-381).  The backward replaces pdist2dr_backward[_cuda] (dist.h:10-12,19-21, dist.cpp:49-110):
 * grad T[m, n]; grad_boxes T[m,5] and grad_points T[n,2] are ACCUMULATED into (caller zero-fills them, like the reference's
 * zeros_like). */
int d3d_pdist2dr_f32(const float *points, int64_t n, const float *boxes, int64_t m, float *dist, uint8_t *iedge, void *stream);
int d3d_pdist2dr_f64(const double *points, int64_t n, const double *boxes, int64_t m, double *dist, uint8_t *iedge, void *stream);
int d3d_pdist2dr_backward_f32(const float *points, int64_t n, const float *boxes, int64_t m, const float *grad, float *grad_boxes,
                              float *grad_points, void *stream);
int d3d_pdist2dr_backward_f64(const double *points, int64_t n, const double *boxes, int64_t m, const double *grad, double *grad_boxes,
                              double *grad_points, void *stream);
/* Frame-batched point-to-box mask and distance (a training batch or a dataset pass computes them once per frame).  Frames are packed back
 * to back: points T[total_points, P] and boxes T[total_boxes, B] with DEVICE offsets point_offsets / box_offsets i64[nframes+1] (frame f
 * owns rows [offsets[f], offsets[f+1]), n_f points and m_f boxes).  out_offsets DEVICE i64[nframes+1] (mask_offsets / dist_offsets): frame
 * f's result is the row-major [m_f boxes, n_f points] block at out + out_offsets[f], usually at the running sum of m_f * n_f.
 * project_axis -1: P = 2, B = 5 (x, y, w, h, r), per frame the result of d3d_crop2dr_* / d3d_pdist2dr_*.  project_axis 0, 1 or 2: P = 3,
 * B = 7 (x, y, z, lx, ly, lz, r), projected to that axis like box3dp_crop / box3dr_pdist (d3d_b200.box): the 2-D operator runs on point
 * columns (a, b) and box columns (a, b, 3 + a, 3 + b, 6), where a < b are the two other axes; the mask also requires
 * p - d / 2 < c < p + d / 2 along the axis (point coordinate p, box centre c and extent d), the distance combines the 2-D distance d2 with
 * the axial distance dp = min(c + d / 2 - p, p - c + d / 2) (the branch on p > c): min(d2, dp) inside the prism, d2 or dp where only one of
 * them is positive, -sqrt(d2^2 + dp^2) outside both.  Every operation is rounded like torch's elementwise operators, so per frame the
 * values equal the Python functions' bit for bit.
 * max_frame_points / max_frame_boxes: HARD UPPER BOUNDS of n_f / m_f (0 = unknown, assume the totals); they size the launch grid.  No limit
 * on nframes below 2^31.  Negative sizes or project_axis outside -1..2: D3D_ERR_INVALID_ARGUMENT; nframes == 0 or an empty side: no-op.
 * d3d_crop2dr_batch_*: one box preparation and one mask launch.  A frame with n_f * m_f >= d3d_crop2dr_grid_min_pairs() is NOT written
 * (neither are the bounds required to cover it): run d3d_crop2dr_* on it, whose grid path is faster there, then apply the axis test for
 * project_axis >= 0.  Workspace below d3d_crop2dr_batch_workspace_bytes: D3D_ERR_WORKSPACE.
 * d3d_pdist2dr_batch_*: one launch, no workspace, no iedge output.  The backward ACCUMULATES into grad_boxes T[total_boxes, B] and
 * grad_points T[total_points, P] (caller zero-fills them); grad T has the layout of dist.  The 3-D gradient is the analytic gradient of the
 * combination: where d2 == dp > 0 each gets half, and on the corner branch (d2, dp) get -(d2, dp) / sqrt(d2^2 + dp^2), 0 where both are 0. */
int64_t d3d_crop2dr_grid_min_pairs(void);
size_t d3d_crop2dr_batch_workspace_bytes(int64_t total_boxes, int dtype);
int d3d_crop2dr_batch_f32(const float *points, int64_t total_points, const int64_t *point_offsets, const float *boxes, int64_t total_boxes,
                          const int64_t *box_offsets, int64_t nframes, int64_t max_frame_points, int64_t max_frame_boxes, int project_axis,
                          const int64_t *mask_offsets, uint8_t *mask, void *workspace, size_t workspace_bytes, void *stream);
int d3d_crop2dr_batch_f64(const double *points, int64_t total_points, const int64_t *point_offsets, const double *boxes, int64_t total_boxes,
                          const int64_t *box_offsets, int64_t nframes, int64_t max_frame_points, int64_t max_frame_boxes, int project_axis,
                          const int64_t *mask_offsets, uint8_t *mask, void *workspace, size_t workspace_bytes, void *stream);
/* Fused reductions of the point-in-box mask, without the mask: point_box i64[points] is the lowest FRAME-LOCAL index of a box whose mask
 * entry for the point is 1, or -1 if there is none; box_npoints i64[boxes] is the number of points inside each box.  The decision per pair
 * is that of d3d_crop2dr_* / d3d_crop2dr_batch_* (same points, boxes and project_axis convention), so per frame the outputs equal
 * where(mask.any(0), mask.argmax(0), -1) and mask.sum(1) exactly.
 * d3d_crop2dr_assign_*: one frame, n points, m boxes (project_axis -1: rows [n,2] / [m,5]; 0, 1, 2: rows [n,3] / [m,7]).  It initialises
 * point_box[0, n) and box_npoints[0, m) itself and then computes them; like d3d_crop2dr_* it bins the points into a grid when
 * n * m >= d3d_crop2dr_grid_min_pairs() (D3D_B200_CROP_PATH=brute | grid forces a back end); the result does not depend on the back end.
 * Workspace below d3d_crop2dr_assign_workspace_bytes (needed when n and m are both positive): D3D_ERR_WORKSPACE; n >= 2^32 or m >= 2^31:
 * D3D_ERR_INVALID_ARGUMENT.
 * d3d_crop2dr_assign_batch_*: the arguments of d3d_crop2dr_batch_* with the two outputs in place of mask_offsets and mask.  It initialises
 * ALL of point_box [total_points] (to -1) and box_npoints [total_boxes] (to 0), including the slices of the frames it skips, then makes
 * one box preparation and one tile launch, whatever the number of frames.  Like the mask batch entry, it does not compute a frame with
 * n_f * m_f >= d3d_crop2dr_grid_min_pairs() (the bounds need not cover it): call d3d_crop2dr_assign_* on that frame's slices AFTER the batch
 * call on the same stream, which would otherwise overwrite them.  Workspace below d3d_crop2dr_assign_batch_workspace_bytes:
 * D3D_ERR_WORKSPACE; nframes > 2^31 - 1: D3D_ERR_UNSUPPORTED.
 * Both: negative sizes or project_axis outside -1..2: D3D_ERR_INVALID_ARGUMENT; no point and no box (or nframes == 0): no-op.  A null
 * pointer is allowed only for an empty side.  Argument errors return before any CUDA call. */
size_t d3d_crop2dr_assign_workspace_bytes(int64_t n, int64_t m, int dtype);
int d3d_crop2dr_assign_f32(const float *points, int64_t n, const float *boxes, int64_t m, int project_axis, int64_t *point_box,
                           int64_t *box_npoints, void *workspace, size_t workspace_bytes, void *stream);
int d3d_crop2dr_assign_f64(const double *points, int64_t n, const double *boxes, int64_t m, int project_axis, int64_t *point_box,
                           int64_t *box_npoints, void *workspace, size_t workspace_bytes, void *stream);
size_t d3d_crop2dr_assign_batch_workspace_bytes(int64_t total_boxes, int dtype);
int d3d_crop2dr_assign_batch_f32(const float *points, int64_t total_points, const int64_t *point_offsets, const float *boxes,
                                 int64_t total_boxes, const int64_t *box_offsets, int64_t nframes, int64_t max_frame_points,
                                 int64_t max_frame_boxes, int project_axis, int64_t *point_box, int64_t *box_npoints, void *workspace,
                                 size_t workspace_bytes, void *stream);
int d3d_crop2dr_assign_batch_f64(const double *points, int64_t total_points, const int64_t *point_offsets, const double *boxes,
                                 int64_t total_boxes, const int64_t *box_offsets, int64_t nframes, int64_t max_frame_points,
                                 int64_t max_frame_boxes, int project_axis, int64_t *point_box, int64_t *box_npoints, void *workspace,
                                 size_t workspace_bytes, void *stream);
int d3d_pdist2dr_batch_f32(const float *points, int64_t total_points, const int64_t *point_offsets, const float *boxes, int64_t total_boxes,
                           const int64_t *box_offsets, int64_t nframes, int64_t max_frame_points, int64_t max_frame_boxes, int project_axis,
                           const int64_t *dist_offsets, float *dist, void *stream);
int d3d_pdist2dr_batch_f64(const double *points, int64_t total_points, const int64_t *point_offsets, const double *boxes, int64_t total_boxes,
                           const int64_t *box_offsets, int64_t nframes, int64_t max_frame_points, int64_t max_frame_boxes, int project_axis,
                           const int64_t *dist_offsets, double *dist, void *stream);
int d3d_pdist2dr_batch_backward_f32(const float *points, int64_t total_points, const int64_t *point_offsets, const float *boxes,
                                    int64_t total_boxes, const int64_t *box_offsets, int64_t nframes, int64_t max_frame_points,
                                    int64_t max_frame_boxes, int project_axis, const int64_t *dist_offsets, const float *grad,
                                    float *grad_boxes, float *grad_points, void *stream);
int d3d_pdist2dr_batch_backward_f64(const double *points, int64_t total_points, const int64_t *point_offsets, const double *boxes,
                                    int64_t total_boxes, const int64_t *box_offsets, int64_t nframes, int64_t max_frame_points,
                                    int64_t max_frame_boxes, int project_axis, const int64_t *dist_offsets, const double *grad,
                                    double *grad_boxes, double *grad_points, void *stream);

/* ------------------------------------------------------------------------------------------------
 * NMS, replaces nms2d[_cuda] (reference d3d/box/nms.h:6-10, nms.cpp:98-119, nms_cuda.cu:217-244).
 * boxes [n,5], scores [n]; suppressed u8[n] (1 = suppressed) in ORIGINAL box order -- the Python
 * front door returns ~suppressed (d3d/box/__init__.py:272).  Order = stable descending sort of
 * scores (ties keep the lower original index first).  iou > (T)(float)iou_threshold, strict.
 * Score rule: every box with score <= score_threshold is suppressed (reference CUDA rule,
 * nms_cuda.cu:223).  iou_type: D3D_IOU_BOX or D3D_IOU_RBOX; supression_type: D3D_SUP_HARD, or D3D_SUP_LINEAR / D3D_SUP_GAUSSIAN
 * (soft-NMS, nms.cpp:33-94: a suppressed box's score is multiplied by 1 - iou^supression_param / exp(-iou^2 / supression_param) and
 * the box is dropped once its score falls below score_threshold; the order is re-established after every box exactly like the
 * reference's insertion sort, so the walk is sequential: one CTA, no dense N x N coefficient matrix).
 * ---------------------------------------------------------------------------------------------- */
size_t d3d_nms2d_workspace_bytes(int64_t n, int dtype);
int d3d_nms2d_f32(const float *boxes, const float *scores, int64_t n, int iou_type, int supression_type,
                  float iou_threshold, float score_threshold, float supression_param, uint8_t *suppressed,
                  void *workspace, size_t workspace_bytes, void *stream);
int d3d_nms2d_f64(const double *boxes, const double *scores, int64_t n, int iou_type, int supression_type,
                  float iou_threshold, float score_threshold, float supression_param, uint8_t *suppressed,
                  void *workspace, size_t workspace_bytes, void *stream);

/* Frame-batched hard NMS (BASELINE.json config 5; the reference has no batch form): boxes [total,5] / scores [total] of all frames
 * back to back, frame_offsets DEVICE i64[nframes+1] as in the voxel ABI, suppressed u8[total] in the ORIGINAL order of every frame;
 * per frame exactly the result of d3d_nms2d_* (same order, thresholds and score rule).  max_frame_boxes: HARD UPPER BOUND of the frame
 * sizes (0 = unknown, assume `total`); frames of up to 8192 boxes are supported (more: D3D_ERR_UNSUPPORTED, use d3d_nms2d_* per frame);
 * supression_type: D3D_SUP_HARD only (soft-NMS is sequential in the scores).  Rotated boxes with a threshold >= 0: every frame is sorted
 * along a Morton curve through its box centres, tiles of two 64-box blocks whose bounding rectangles do not meet are skipped, the
 * surviving pairs are clipped from one flat candidate list, and the keep mask is the fixpoint of keep / suppress rounds over the
 * resulting edge list (one CTA per frame).  Axis-aligned boxes, negative thresholds and frames whose edge list overflows (device flag)
 * take the dense form: per-frame sort by score in shared memory, 64x64 tiles of the upper triangle, one resolve CTA per frame.  Both
 * forms give the keep mask of d3d_nms2d_* called per frame (D3D_B200_NMS_BATCH_PATH=dense forces the second). */
size_t d3d_nms2d_batch_workspace_bytes(int64_t total, int64_t nframes, int64_t max_frame_boxes, int dtype);
int d3d_nms2d_batch_f32(const float *boxes, const float *scores, int64_t total, const int64_t *frame_offsets, int64_t nframes,
                        int64_t max_frame_boxes, int iou_type, int supression_type, float iou_threshold, float score_threshold,
                        uint8_t *suppressed, void *workspace, size_t workspace_bytes, void *stream);
int d3d_nms2d_batch_f64(const double *boxes, const double *scores, int64_t total, const int64_t *frame_offsets, int64_t nframes,
                        int64_t max_frame_boxes, int iou_type, int supression_type, float iou_threshold, float score_threshold,
                        uint8_t *suppressed, void *workspace, size_t workspace_bytes, void *stream);

/* Frame-batched soft-NMS: supression_type D3D_SUP_LINEAR or D3D_SUP_GAUSSIAN (D3D_SUP_HARD or anything else: D3D_ERR_INVALID_ARGUMENT;
 * hard NMS is d3d_nms2d_batch_*).  Same packing, offsets, max_frame_boxes bound, 8192-box frame limit (D3D_ERR_UNSUPPORTED beyond)
 * and nframes <= 65535 as d3d_nms2d_batch_*; per frame exactly the keep mask of d3d_nms2d_* with the same arguments.  One CTA walks
 * each frame with the walk state in shared memory.  For iou_threshold >= 0 the pairs of a frame that may overlap above the threshold
 * (bounding circles / AABBs meet) are listed first and a kept box decays only its listed neighbours; a frame whose list overflows
 * (more than 32 x max_frame_boxes pairs) and every frame under a negative threshold decay all boxes behind the kept one. */
size_t d3d_nms2d_batch_soft_workspace_bytes(int64_t total, int64_t nframes, int64_t max_frame_boxes, int dtype);
int d3d_nms2d_batch_soft_f32(const float *boxes, const float *scores, int64_t total, const int64_t *frame_offsets, int64_t nframes,
                             int64_t max_frame_boxes, int iou_type, int supression_type, float iou_threshold, float score_threshold,
                             float supression_param, uint8_t *suppressed, void *workspace, size_t workspace_bytes, void *stream);
int d3d_nms2d_batch_soft_f64(const double *boxes, const double *scores, int64_t total, const int64_t *frame_offsets, int64_t nframes,
                             int64_t max_frame_boxes, int iou_type, int supression_type, float iou_threshold, float score_threshold,
                             float supression_param, uint8_t *suppressed, void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Voxelization of a BATCH of frames (one frame = one reference VoxelGenerator.__call__).
 * points f32[total, nfeat] (first 3 columns xyz); frame_offsets DEVICE i64[nframes+1], ascending,
 * frame f owns points [frame_offsets[f], frame_offsets[f+1]).
 * Sparse outputs are PACKED across frames in frame order: the kept points of frame f occupy rows
 * [frame_rows[f][0], frame_rows[f+1][0]) of out_points / out_mask / out_mapping and its voxels rows
 * [frame_rows[f][1], frame_rows[f+1][1]) of out_npoints / out_coords, where frame_rows is the DEVICE
 * i64[nframes+1, 2] array the call fills (entry nframes = totals).  One contiguous device-to-host copy
 * per array therefore moves a whole batch.  Dense outputs keep the regular [nframes, max_voxels, ...]
 * layout and report counts[f] = {0, voxels V_f} (device i64[nframes, 2]).
 * ---------------------------------------------------------------------------------------------- */
typedef struct d3d_voxel_params {
    /* sparse path (reference voxelize.cpp:288-484 through d3d/voxel/__init__.py:96-103) */
    float size[3];      /* _size: f32 (hi-lo)/shape, coordinate = floor(p/size)            */
    int64_t vlo[3];     /* _vbounds[:,0]: keep voxels with vlo <= coord < vhi              */
    int64_t vhi[3];     /* _vbounds[:,1]                                                   */
    int32_t offset[3];  /* _offset: coords_out = coord - offset                            */
    int32_t min_points; /* voxel filter: npoints >= min_points                             */
    int32_t max_points; /* TRIM: first max_points points per voxel; dense: slots per voxel */
    int32_t max_voxels; /* TRIM / DESCENDING cap; dense: voxel capacity per frame          */
    int32_t max_points_filter; /* d3d_max_points_filter */
    int32_t max_voxels_filter; /* d3d_max_voxels_filter */
    /* dense path (reference voxelize.cpp:45-199) */
    float bound[6];     /* xmin,xmax,ymin,ymax,zmin,zmax; idx = (int)((p-lo)/((hi-lo)/shape)) */
    int32_t shape[3];
    int32_t reduction;  /* d3d_reduction_type */
    /* execution parameters */
    int32_t algo;              /* d3d_voxel_algo: AUTO picks the fastest back end that supports the configuration (no effect on results) */
    int64_t max_frame_points;  /* HARD UPPER BOUND of the frame lengths of the batch (the host knows the offsets); 0 = unknown,
                                * assume `total`.  It sizes the per-frame scratch and the launch geometry of the fast paths: a
                                * frame longer than this bound is cut to its first max_frame_points points.  With 0 a multi-frame
                                * batch runs with scratch sized for one frame of `total` points (slower, never wrong). */
} d3d_voxel_params;

/* max_frame_points: largest frame of the batch (0 = unknown): bounds the per-frame scratch of the cluster path */
size_t d3d_voxelize_workspace_bytes(int64_t total_points, int64_t nframes, int64_t max_frame_points);
/* sparse + filter fused; replaces voxelize_3d_sparse + voxelize_3d_filter (voxelize.h:14-25).
 * Capacities: out_points f32[total,nfeat], out_mask i64[total] (index of the surviving point INSIDE its
 * frame), out_mapping i64[total] (voxel id inside the frame), out_npoints i32[total], out_coords i64[total,3];
 * frame_rows i64[nframes+1,2] as described above. */
int d3d_voxelize_sparse_f32(const float *points, int64_t total, int32_t nfeat, const int64_t *frame_offsets,
                            int64_t nframes, const d3d_voxel_params *params, float *out_points, int64_t *out_mask,
                            int64_t *out_mapping, int32_t *out_npoints, int64_t *out_coords, int64_t *frame_rows,
                            void *workspace, size_t workspace_bytes, void *stream);
/* dense; replaces voxelize_3d_dense (voxelize.h:9-12).  Per frame f the outputs live at
 * voxels f32[nframes,max_voxels,max_points,nfeat], coords i64[nframes,max_voxels,3],
 * pmask u8[nframes,max_voxels,max_points] (0 where the reference leaves memory uninitialised),
 * npoints i32[nframes,max_voxels], aggregates f32[nframes,max_voxels,nfeat] (NULL when reduction NONE);
 * counts[f] = {points stored, voxels V_f}.  The call zero-fills voxels/pmask/npoints itself. */
int d3d_voxelize_dense_f32(const float *points, int64_t total, int32_t nfeat, const int64_t *frame_offsets,
                           int64_t nframes, const d3d_voxel_params *params, float *voxels, int64_t *coords,
                           uint8_t *pmask, int32_t *npoints, float *aggregates, int64_t *counts, void *workspace,
                           size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------------
 * aligned_scatter, replaces aligned_scatter_forward/backward[_cuda] (reference d3d/point/scatter.h:39-45,
 * scatter.cpp:79-201, scatter_cuda.cu:91-241).  coord T[n,1+dim] (col 0 = batch index), image
 * T[nbatch,nchan,dims[0..dim)], out T[n,nchan]; align: D3D_ALIGN_MEAN or D3D_ALIGN_LINEAR; dim in 1..3.
 * backward accumulates into image_grad (caller zero-fills it, d3d/point/__init__.py:32).
 * ---------------------------------------------------------------------------------------------- */
int d3d_aligned_scatter_forward(const void *coord, int64_t n, int32_t dim, const void *image, int64_t nbatch,
                                int64_t nchan, const int64_t *dims_host, int align, int dtype, void *out, void *stream);
int d3d_aligned_scatter_backward(const void *coord, int64_t n, int32_t dim, const void *grad, int64_t nbatch,
                                 int64_t nchan, const int64_t *dims_host, int align, int dtype, void *image_grad,
                                 void *stream);
/* The same two operators with a caller-provided workspace (d3d_aligned_scatter_workspace_bytes; 0 = none needed).  With a workspace,
 * 2-D fp32 maps whose points are dense (n >= cells / 16) take the tile path: the points are binned by 8 x 64-cell tile and every tile is
 * staged once in shared memory, instead of one 32-byte sector per neighbour row and channel plane.  Forward outputs are bit-identical to
 * the gather path; backward sums in a different (still unspecified) order.  A point whose batch index lies outside [0, nbatch) -- for
 * which the gather path, like the reference, reads outside the map -- is skipped by the tile path (its output row is not written).
 * reuse_plan != 0: the workspace still holds the binning of an earlier call with the same coord / n / nbatch / dims (the backward pass
 * after its forward pass: the autograd function keeps the workspace) and the three binning launches are skipped.
 * The entry points without workspace always gather. */
size_t d3d_aligned_scatter_workspace_bytes(int64_t n, int32_t dim, int64_t nbatch, const int64_t *dims_host);
int d3d_aligned_scatter_forward_ws(const void *coord, int64_t n, int32_t dim, const void *image, int64_t nbatch,
                                   int64_t nchan, const int64_t *dims_host, int align, int dtype, void *out,
                                   void *workspace, size_t workspace_bytes, int reuse_plan, void *stream);
int d3d_aligned_scatter_backward_ws(const void *coord, int64_t n, int32_t dim, const void *grad, int64_t nbatch,
                                    int64_t nchan, const int64_t *dims_host, int align, int dtype, void *image_grad,
                                    void *workspace, size_t workspace_bytes, int reuse_plan, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Measurement helper: FMA-chain microbenchmark used as the measured FP32/FP64 ALU peak for the IoU
 * roofline (SURVEY.md 8(d)).  Runs `iters` dependent FMAs x 16 independent chains per thread on a full
 * grid (fp32: packed FFMA2, the instruction the IoU clip uses; fp64: DFMA); writes the number of FLOPs
 * executed to *flops_host.  Time it with CUDA events on `stream`.
 * ---------------------------------------------------------------------------------------------- */
int d3d_fma_peak_probe(int dtype, int64_t iters, float *sink, double *flops_host, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* D3D_B200_H */
