/*
 * fnp.h -- C ABI of libfnp_sm100.so, the B200-native (sm_100a) Greedy Box Seeker path.
 *
 * Drop-in boundary for the native side of findnpropagate's pcdet.ops on this path
 * (reference paths relative to the reference tree):
 *
 *   reference pybind symbol (file:line)                     replaced by
 *   ------------------------------------------------------  ---------------------------
 *   roiaware_pool3d_cuda.points_in_boxes_gpu
 *     (roiaware_pool3d/src/roiaware_pool3d.cpp:98,175)       fnp_points_in_boxes
 *   iou3d_nms_cuda.boxes_overlap_bev_gpu
 *     (iou3d_nms/src/iou3d_nms.cpp:49, iou3d_nms_api.cpp:12) fnp_boxes_overlap_bev
 *   iou3d_nms_cuda.boxes_aligned_overlap_bev_gpu
 *     (iou3d_nms.cpp:71, iou3d_nms_api.cpp:13)               fnp_boxes_aligned_overlap_bev
 *   iou3d_nms_cuda.boxes_iou_bev_gpu
 *     (iou3d_nms.cpp:93, iou3d_nms_api.cpp:14)               fnp_boxes_iou_bev
 *   iou3d_nms_cuda.nms_gpu
 *     (iou3d_nms.cpp:113, iou3d_nms_api.cpp:15)              fnp_nms_rotated
 *   iou3d_nms_cuda.nms_normal_gpu
 *     (iou3d_nms.cpp:162, iou3d_nms_api.cpp:16)              fnp_nms_normal
 *   the per-hypothesis loop of FrustumProposerOG.get_proposals
 *     (models/dense_heads/frustum_proposals_v1.py:582-1053)  fnp_seeker_* (fused stages)
 *
 * Conventions (differences from the reference are deliberate, see INTEGRATION.md):
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless the
 *     parameter name ends in _host;
 *   - the caller owns all memory, including workspaces (no cudaMalloc in any call);
 *   - `stream` is a cudaStream_t passed as void*; work is enqueued on it, and no call
 *     synchronises the device or the stream (the reference uses the legacy default
 *     stream and a blocking cudaMemcpy inside NMS);
 *   - return value: 0 on success, otherwise a cudaError_t (> 0) or an FNP_E* code (< 0).
 *     Nothing ever calls exit() (the reference does, roiaware_pool3d_kernel.cu:350-354).
 *   - all floating point data is fp32, boxes are [x, y, z, dx, dy, dz, heading] (7 floats).
 */
#ifndef FNP_H_
#define FNP_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FNP_OK 0
#define FNP_EINVAL (-1)   /* bad argument (null pointer, negative size, misalignment) */
#define FNP_EWORKSPACE (-2) /* workspace too small */

/* Library / build identification: returns e.g. "fnp-sm100a 0.1". */
const char *fnp_version(void);

/* ------------------------------------------------------------------ op-level API */

/* First containing box per point (k ascending) or -1.
 * boxes (B,T,7), pts (B,M,3) contiguous, out (B,M) int32 -- every entry is written. */
int fnp_points_in_boxes(const float *boxes, const float *pts, int32_t *out, int B, int T, int M,
                        void *stream);

/* Per-box point counts over packed segments: for segment s (one frustum), points
 * pts4[pt_start[s] .. pt_start[s+1]) (float4 x,y,z,_) are tested against boxes
 * boxes[box_start[s] .. box_start[s+1]) (7 floats each); counts[] is indexed like boxes.
 * Same predicate as fnp_points_in_boxes; count = what the reference obtains with one
 * points_in_boxes_gpu call + (idx >= 0).sum() per box (frustum_proposals_v1.py:930-932).
 * There is no cap on the points or boxes of a segment: every count is written. */
int fnp_count_in_boxes(const float *pts4, const int32_t *pt_start, const float *boxes,
                       const int32_t *box_start, int n_segments, int32_t *counts, void *stream);

/* Points of every box, cropped out of a batch of ragged frames (the crop of create_groundtruth_database,
 * nuscenes_dataset.py:346-390: pts[box_idxs_of_pts == i], then xyz minus the box centre).
 *   pts (n_points, n_cols) f32, n_cols >= 3, x y z first; frame f's rows are row_start[f] .. row_start[f+1]
 *   (int64, n_frames+1, row_start[0] = 0, row_start[n_frames] = n_points);
 *   boxes (n_boxes, 7) f32 and centres (n_boxes, 3) f64, frame f's boxes box_start[f] .. box_start[f+1] (int64,
 *   the same rule with n_boxes).
 * Each point goes to the FIRST box of its frame that contains it, by the predicate of fnp_points_in_boxes
 * (prep_box / in_box), so the assignment is that op's bit for bit.  Outputs, caller-allocated:
 *   counts (n_boxes) int32, starts (n_boxes+1) int64 (exclusive scan of counts), rows (n_points, n_cols) f32 of
 *   which rows starts[b] .. starts[b]+counts[b] are box b's points in input order, x y z as
 *   (float)((double)p - centre) (numpy's f32_rows[:, :3] -= f64_centre) and the other columns copied.
 * Each point lands in at most one box, so rows never needs more than n_points rows; there is no cap on points or
 * boxes per frame.  The order is fixed by per-tile counts, a scan and a per-tile ordered scatter: no atomic picks a
 * position, and two runs give the same bytes.
 * workspace: 16-byte aligned, at least fnp_crop_workspace_bytes(host copies of row_start, box_start, n_frames)
 * bytes (4 bytes per point plus 4 per (1024-point tile, box) pair of each frame); FNP_EWORKSPACE when it cannot
 * hold the per-point part.  Starts that do not end at n_points / n_boxes, or a workspace too small for the
 * per-tile part, leave every count 0 and write no row (checked on the device).  FNP_EINVAL: n_cols < 3, a
 * negative size, frames without n_frames, a missing pointer.  Build record (nvcc 12.9, -Xptxas -v, sm_100a), no
 * stack, no spills: crop_plan_kernel 1024 threads, 32 registers; crop_assign_kernel 256 threads, 48 registers;
 * crop_prefix_kernel 128 threads, 61 registers; crop_starts_kernel 1024 threads, 30 registers;
 * crop_scatter_kernel 32 threads (one warp per tile), 64 registers. */
int fnp_crop_points_in_boxes(const float *pts, int n_cols, const int64_t *row_start, long long n_points,
                             const float *boxes, const double *centres, const int64_t *box_start, int n_boxes,
                             int n_frames, int32_t *counts, int64_t *starts, float *rows, void *workspace,
                             size_t workspace_bytes, void *stream);
/* HOST pointers: row_start_host, box_start_host as passed (on the device) to fnp_crop_points_in_boxes; 0 for a
 * negative n_frames or a missing pointer. */
size_t fnp_crop_workspace_bytes(const int64_t *row_start_host, const int64_t *box_start_host, int n_frames);

/* Every-box crop, by the predicate of points_in_boxes_cpu (the crop of KittiDataset.create_groundtruth_database:
 * points[point_indices[i] > 0], then xyz minus the box centre).  A point is written once for every box of its own
 * frame that contains it, so the number of rows is known only after counting: two calls, on one stream, with the
 * same arguments and workspace (sized by fnp_crop_workspace_bytes, left untouched between them).
 *   pts, row_start, box_start, centres: as for fnp_crop_points_in_boxes.
 *   box_prep (n_boxes, 8) f32 device = fnp_host_prep_boxes_cpu of the boxes cast to float32; each (point, box)
 *   test gives the bits of fnp_points_in_boxes_matrix.
 * fnp_crop_all_count writes counts (n_boxes) int32 and starts (n_boxes+1) int64, starts[n_boxes] = the rows needed.
 * fnp_crop_all_scatter then writes rows (rows_cap, n_cols) f32: box b's points are rows starts[b] ..
 * starts[b]+counts[b], in input order, x y z as (float)((double)p - centre), the other columns copied; no row at
 * or past rows_cap is written.  Positions come from per-(tile, box) counts summed from warp ballots, a scan over
 * the tiles, and a ballot rank in row order: no atomic picks one, and two runs give the same bytes.  No cap on
 * points or boxes per frame.  Starts that do not end at n_points / n_boxes, or a workspace too small for the
 * per-tile part, leave every count 0 and write no row (checked on the device).  FNP_EINVAL / FNP_EWORKSPACE as for
 * fnp_crop_points_in_boxes, and for a negative rows_cap or a missing rows with rows_cap > 0, before any launch.
 * Build record (nvcc 12.9, -Xptxas -v, sm_100a), no stack, no spills: crop_all_count_kernel 256 threads,
 * 33 registers, 16384 bytes of shared memory; crop_all_scatter_kernel 256 threads (one warp per box of the
 * tile), 40 registers, 12288 bytes of shared memory.  The plan, prefix and starts kernels are
 * fnp_crop_points_in_boxes'. */
int fnp_crop_all_count(const float *pts, int n_cols, const int64_t *row_start, long long n_points,
                       const float *box_prep, const int64_t *box_start, int n_boxes, int n_frames,
                       int32_t *counts, int64_t *starts, void *workspace, size_t workspace_bytes, void *stream);
int fnp_crop_all_scatter(const float *pts, int n_cols, const int64_t *row_start, long long n_points,
                         const float *box_prep, const double *centres, const int64_t *box_start, int n_boxes,
                         int n_frames, const int64_t *starts, float *rows, long long rows_cap,
                         void *workspace, size_t workspace_bytes, void *stream);

/* The (N, P) 0/1 matrix of the reference's CPU op points_in_boxes_cpu (roiaware_pool3d.cpp:121-168): NOT
 * the GPU predicate -- the margin is 1e-2 instead of 1e-5 and the products are rounded individually, with
 * the host libm's cosf / sinf.  box_prep (N,8) device = fnp_host_prep_boxes_cpu(boxes) uploaded (the per-box
 * constants are formed on the host, where the reference forms them); pts (P,3); out (N,P) int32, every
 * entry written. */
int fnp_points_in_boxes_matrix(const float *box_prep, const float *pts, int32_t *out, int N, int P,
                               void *stream);
/* HOST pointers: boxes_host (N,7) -> prep_host (N,8) = cx, cy, cz, hz, cosa, sina, tx, ty. */
int fnp_host_prep_boxes_cpu(const float *boxes_host, float *prep_host, int N);

/* 3D IoU (iou3d_nms_utils.py:48-81 boxes_iou3d_gpu / :83-117 boxes_aligned_iou3d_gpu): rotated BEV overlap
 * x height overlap over the union volume, every step rounded like the reference's torch expressions, in ONE
 * kernel.  (N,7) x (M,7) -> (N,M);  aligned: (N,7),(N,7) -> (N). */
int fnp_boxes_iou3d(const float *boxes_a, const float *boxes_b, float *out, int N, int M, void *stream);
int fnp_boxes_aligned_iou3d(const float *boxes_a, const float *boxes_b, float *out, int N, void *stream);

/* Rotated BEV overlap area / IoU, (N,7) x (M,7) -> (N,M). */
int fnp_boxes_overlap_bev(const float *boxes_a, const float *boxes_b, float *out, int N, int M,
                          void *stream);
int fnp_boxes_iou_bev(const float *boxes_a, const float *boxes_b, float *out, int N, int M,
                      void *stream);
/* Aligned pairs, (N,7),(N,7) -> (N). */
int fnp_boxes_aligned_overlap_bev(const float *boxes_a, const float *boxes_b, float *out, int N,
                                  void *stream);

/* NMS over boxes already sorted by descending score.  keep (N) int64 and num_keep (1) int32
 * are written on the device; entries keep[*num_keep..N) are left untouched.
 * workspace: fnp_nms_workspace_bytes(N) bytes, 8-byte aligned. */
size_t fnp_nms_workspace_bytes(int N);
int fnp_nms_rotated(const float *boxes_sorted, int N, float thresh, int64_t *keep,
                    int32_t *num_keep, void *workspace, size_t workspace_bytes, void *stream);
int fnp_nms_normal(const float *boxes_sorted, int N, float thresh, int64_t *keep,
                   int32_t *num_keep, void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------- fused seeker stages
 *
 * One call sequence processes a BATCH of frames.  Units: `cand` = one candidate frustum
 * (a 2D box that survived the 2D NMS and the score threshold, in reference order:
 * frame, then camera order [2,0,1,5,3,4], then 2D-NMS order); F = total candidates.
 */

typedef struct fnp_seeker_cfg {
    int32_t num_mags;        /* M depth steps                    (PARAMS num_mags)      */
    int32_t num_yaw_size;    /* J = num_rotations * num_sizes                           */
    int32_t n_classes;       /* A rows of the prior tables                               */
    int32_t clamp_bottom;    /* PARAMS clamp_bottom                                      */
    float img_w, img_h;      /* 1600, 900  (frustum_proposals_v1.py:203)                 */
    float lq, uq, cq;        /* depth quantiles                                          */
    float frustum_min;       /* 2.0       (frustum_proposals_v1.py:240)                  */
    float max_dist;          /* 50                                                       */
    float min_cam_iou;       /* 0.3                                                      */
    float dns_w, iou_w;      /* score weights                                            */
    /* ---- optional terms of FrustumProposerOG (SURVEY.md 8 row f3); all zero = the shipped YAML ---- */
    float dst_w;             /* weight of dists_ranked (frustum_proposals_v1.py:889-893,996-999)           */
    float ego_w;             /* weight of |centre| / max |centre| (:1016-1020)                              */
    float occl_w;            /* weight of 1 - fail / (max fail + 1e-6), calc_occl_scores (:408-477,1007-1014) */
    float search_depth;      /* PARAMS search_depth (:619-623,841-842); <= 0: not set                       */
    int32_t flags;           /* FNP_SEEKER_MULT | FNP_SEEKER_OCCL_MULT | FNP_SEEKER_MULTICAM_IOU            */
    int32_t topk;            /* proposals per frustum (:1040-1046); 0 and 1 both mean the single best one  */
    float nms_normal;        /* axis-aligned BEV IoU threshold of the per-frustum NMS (:1030); only matters
                                for topk > 1 (the first survivor is the arg-max whatever the threshold)    */
    int32_t variant;         /* FNP_VARIANT_NUSCENES (FrustumProposerOG, frustum_proposals_v1.py) or
                                FNP_VARIANT_KITTI (FrustumProposerOGKITTI, frustum_proposals_v1_kitti.py:38):
                                KITTI calibration arithmetic (calibration_kitti.py:128-216), no on-image test,
                                first-match point counts normalised by their sum, additive score (:646-654)  */
} fnp_seeker_cfg;

#define FNP_VARIANT_NUSCENES 0
#define FNP_VARIANT_KITTI 1
/* FNP_VARIANT_KITTI: one camera (index 0); the 144 floats of a frame in cam_mats hold
 *   [0..11]  M1  = V2C.T @ R0.T, (4,3) row-major      (lidar_to_rect, calibration_kitti.py:171-182)
 *   [12..23] P2T = P2.T, (4,3) row-major               (rect_to_img, :184-194)
 *   [24..29] cu, cv, fu, fv, tx, ty                    (img_to_rect, :205-216)
 *   [32..47] Minv = inverse((R0_ext @ V2C_ext).T), (4,4) row-major   (rect_to_lidar, :151-169)
 * each formed by the caller with the reference's own torch calls.  The matmuls are restated in the
 * accumulation order torch uses on B200 for >= 33 rows (tools/probe_kitti.py): an fma chain over k = 0..3. */

#define FNP_SEEKER_MULT 1          /* MODEL.DENSE_HEAD.MULT: product of the score terms (:998-999)             */
#define FNP_SEEKER_OCCL_MULT 2     /* OCCL_MULT: score = density * iou * occlusion fail score (:1022-1026)      */
#define FNP_SEEKER_MULTICAM_IOU 4  /* MULTICAM_IOU: 2D IoU averaged over the frame's same-label boxes (:1413-1429) */

typedef struct fnp_seeker_batch {
    /* ---- inputs ---- */
    int32_t n_frames;
    int32_t n_cands;                 /* F */
    int32_t n_tiles;                 /* point tiles over all frames (FNP_CULL_TILE rows each) */
    int32_t max_cands_per_frame;
    const float *points;             /* rows of point_stride floats, xyz at xyz_offset     */
    int32_t point_stride, xyz_offset;
    const int64_t *frame_row_start;  /* (n_frames+1) first row of each frame               */
    const int32_t *tile_frame;       /* (n_tiles) frame of each tile                       */
    const int32_t *tile_row0;        /* (n_tiles) first row (within the frame) of each tile */
    const int32_t *frame_tile_start; /* (n_frames+1) first tile of each frame              */
    const float *cam_mats;           /* (n_frames,6,24): lidar2image rows 0..2 (12),
                                        combine = cam2lidar_R inv(K) (9), cam2lidar_t (3)  */
    const int32_t *frame_cand_start; /* (n_frames+1) first candidate of each frame         */
    const int32_t *cam_cand_start;   /* (n_frames*6+1) first candidate of (frame, camera rank r):
                                        within a frame candidates are grouped by camera in the
                                        order [2,0,1,5,3,4]; rank r is position r of that list  */
    const int32_t *cand_frame;       /* (F) */
    const int32_t *cand_cam;         /* (F) 0..5 */
    const int32_t *cand_label;       /* (F) 1..A */
    const float *cand_box2d;         /* (F,4) x1,y1,x2,y2 */
    const float *base_boxes;         /* (A,J,7)   constructor tables                       */
    const float *base_corners;       /* (A,J,8,3)                                          */
    const float *mags;               /* (M) linspace(0,1,M)                                */
    /* ---- workspaces / intermediates (caller allocated) ---- */
    uint32_t *cell_masks;            /* fnp_seeker_cell_mask_bytes(): per (frame, camera rank, 64-px
                                        image cell) the bitmask (mask_words words) of the rank's
                                        candidates whose 2D box touches the cell            */
    int32_t mask_words;              /* = fnp_seeker_mask_words(max_cands_per_frame)        */
    int32_t *cand_npts;              /* (F)   P_f: the frustum's fill counter while stage 1 runs, its
                                        point count afterwards                              */
    int32_t *page_tab;               /* (F, page_tab_stride) page of point block k of frustum f, + 1
                                        (0: not handed out, < 0: pool exhausted); zeroed by stage 1 */
    int32_t page_tab_stride;         /* >= ceil(largest frame's points / FNP_PAGE_POINTS) + 1 */
    int32_t page_planes;             /* 4: x | y | z | d per page; 5: + source row within the frame
                                        (debug)                                             */
    float *frustum_pts;              /* the page pool: (pts_capacity / FNP_PAGE_POINTS pages, page_planes,
                                        FNP_PAGE_POINTS) -- point i of frustum f is slot i % 256 of
                                        page page_tab[f][i / 256] - 1; xyz of the unprojected point and
                                        its camera depth, SoA inside the page.  The ORDER of a
                                        frustum's points is unspecified (whatever order the tiles
                                        reached it in); no output depends on it                */
    int64_t pts_capacity;            /* points the pool holds; a multiple of FNP_PAGE_POINTS */
    float *cand_stats;               /* (F,40): [0]dmin [1]dmax [2]dcentre [3..5]pmin [6..8]pmax
                                        [9]n_points [10..12] weighted_centre_xyz [13]/[14] min/max of
                                        hyp_dist over the hypotheses within max_dist
                                        [16..39] clamped frustum corners (8,3).  [2] and [10..14] are
                                        formed only when hyp_dist != NULL (the distance term is their
                                        only reader; without it the cq quantile is not selected)  */
    float *centres;                  /* (F,M,3) */
    float *hyp_prep;                 /* (F,H,8) compacted valid hypotheses, H = M*J:
                                        cx,cy,cz,hz, cosa,sina,tx,ty                       */
    int32_t *hyp_index;              /* (F,H) original hypothesis index of each compacted one */
    float *hyp_iou;                  /* (F,H) its 2D IoU                                   */
    int32_t *hyp_nvalid;             /* (F)                                                */
    float *hyp_boxes_dbg;            /* (F,H,7) all hypothesis boxes by original index, or NULL */
    float *hyp_iou_dbg;              /* (F,H) or NULL                                      */
    uint8_t *hyp_valid_dbg;          /* (F,H) or NULL                                      */
    int32_t split_points;            /* points per scoring work item (point split); a multiple of
                                        FNP_PAGE_POINTS                                     */
    int32_t max_items;               /* capacity of `items`                                */
    int32_t *cand_item_start;        /* (F+1) first work item of each frustum              */
    int32_t *items;                  /* (max_items,4) work items: frustum, first hypothesis, split,
                                        hypotheses per thread (1..4)                         */
    int32_t *counts;                 /* (F,H) point count of every compacted hypothesis (zeroed by
                                        fnp_seeker_score, accumulated per point split)      */
    int32_t score_mode;              /* FNP_SCORE_AUTO / FNP_SCORE_DIRECT / FNP_SCORE_SWEEP */
    float *sweep_cols;               /* (F,J,FNP_SWEEP_COL_FLOATS) per (frustum, yaw-size column) depth-
                                        sweep parameters; required for the sweep mode       */
    /* ---- outputs (T = max(cfg.topk, 1) slots per candidate, in NMS order: slot f*T + k) ---- */
    float *out_boxes;                /* (F*T,7) selected boxes per candidate               */
    float *out_score;                /* (F*T)   their second-stage scores                  */
    int32_t *out_best;               /* (F*T)   compacted index of the hypothesis, -1 for an unused slot */
    int32_t *out_count;              /* (F*T)   its point count                            */
    int32_t *status;                 /* (8)   [0] bit0: page pool overflow (capacity needed, in points,
                                        in [1]), bit1: items overflow ([2] items needed);
                                        [4] work-item counter of the scoring kernel; [5] page
                                        cursor of stage 1; [6..7] spare                     */
    /* ---- workspaces of the optional terms (may be NULL when the term is off) ---- */
    float *hyp_dist;                 /* (F,H) |front - weighted_centre_xyz| of each compacted hypothesis;
                                        required iff dst_w != 0 or FNP_SEEKER_MULT          */
    int32_t *hyp_nfar;               /* (F,H) frustum points beyond the nearest corner of each compacted
                                        hypothesis; required iff occl_w > 0 or FNP_SEEKER_OCCL_MULT */
    float *hyp_score;                /* (F,H) second-stage score of each compacted hypothesis; required iff
                                        topk > 1 (needs H <= 32768)                          */
} fnp_seeker_batch;

#ifndef FNP_CULL_TILE
#define FNP_CULL_TILE 1024      /* rows of a stage-1 point tile (one CTA); fnp_seeker_cull_tile() reports the built value */
#endif
#define FNP_PAGE_POINTS 256
/* Scoring modes (fnp_seeker_batch.score_mode).  Both produce the same counts, bit for bit.
 *   DIRECT: every valid hypothesis tests every frustum point (P_f * nv_f in-box predicates).
 *   SWEEP : the M hypotheses of one (yaw, size) column share rotation and size and their centres
 *           advance along the centre line, so a point is inside for one contiguous range of depth
 *           steps; the range is solved per (point, column) with a conservative error bound, added
 *           to a per-column difference array, and only the depth steps within the error bound
 *           of a range end take the exact predicate.  Work: P_f * J range solves instead of
 *           P_f * M * J predicates.
 *   AUTO  : SWEEP when num_mags >= FNP_SWEEP_MIN_MAGS, sweep_cols != NULL and its shared
 *           memory fits; DIRECT otherwise. */
#define FNP_SCORE_AUTO 0
#define FNP_SCORE_DIRECT 1
#define FNP_SCORE_SWEEP 2
#define FNP_SWEEP_MIN_MAGS 16
#define FNP_SWEEP_COL_FLOATS 20
/* Rows of a stage-1 point tile in this build of the library (the host's tile table must use it). */
int fnp_seeker_cull_tile(void);
/* Words of the per-point candidate mask for a batch whose busiest frame has that many
 * candidates: 1, 2, 4, 8, 16 or 32 (-1: more than 1024 candidates per frame are not supported -- the limit of
 * the stage-4 NMS, FNP_SEG_NMS_MAX). */
int fnp_seeker_mask_words(int max_cands_per_frame);
/* Bytes of fnp_seeker_batch.cell_masks for a batch (0 on bad arguments). */
size_t fnp_seeker_cell_mask_bytes(const fnp_seeker_cfg *cfg, int n_frames, int max_cands_per_frame);

/* Stage 1: fused LiDAR->camera projection + per-2D-box frustum cull + compaction into pages.
 * Cell table, then ONE pass over the points: membership, a reservation per (tile, candidate) on the
 * frustum's fill counter, member points written to their final page slots.  No counting pass, no
 * scan, no reordering pass, no host sync. */
int fnp_seeker_cull(const fnp_seeker_cfg *cfg, const fnp_seeker_batch *b, void *stream);
/* Stage 1b: per-frustum depth quantiles, point AABB, frustum corners, centre line. */
int fnp_seeker_frustum_stats(const fnp_seeker_cfg *cfg, const fnp_seeker_batch *b, void *stream);
/* Stage 2a: hypothesis grid, softmin front shift, distance + 2D-IoU filters, compaction. */
int fnp_seeker_hypotheses(const fnp_seeker_cfg *cfg, const fnp_seeker_batch *b, void *stream);
/* Stage 2b: points-in-boxes scoring.  DIRECT: TMA-staged point tiles against register-resident
 * hypotheses; SWEEP: per-(point, column) depth-range solve + difference arrays in shared memory. */
int fnp_seeker_score(const fnp_seeker_cfg *cfg, const fnp_seeker_batch *b, void *stream);
/* The scoring kernel fnp_seeker_score runs for this batch: FNP_SCORE_DIRECT or FNP_SCORE_SWEEP
 * (FNP_EINVAL if the requested mode cannot run).  Host-only query, enqueues nothing. */
int fnp_seeker_score_mode(const fnp_seeker_cfg *cfg, const fnp_seeker_batch *b);
/* Optional stage 2c (occl_w > 0 or FNP_SEEKER_OCCL_MULT; a no-op otherwise): hyp_nfar.  The reference's
 * occlusion score of a hypothesis is hyp_nfar * (P_f - count) (calc_occl_scores broadcasts a (P,1)
 * against a (P,) mask, :453); fnp_seeker_select forms the product. */
int fnp_seeker_occlusion(const fnp_seeker_cfg *cfg, const fnp_seeker_batch *b, void *stream);
/* Stage 3: second-stage score (density + IoU and the optional terms) and greedy argmax per frustum. */
int fnp_seeker_select(const fnp_seeker_cfg *cfg, const fnp_seeker_batch *b, void *stream);
/* All stages back to back on `stream`. */
int fnp_seeker_run(const fnp_seeker_cfg *cfg, const fnp_seeker_batch *b, void *stream);

/* Stage 3 for many "select-level" settings at once, for tuning the score.  Stages 1-2c do not read the score weights,
 * a hypothesis's point count does not depend on which other hypotheses are valid, and min_cam_iou only removes
 * hypotheses; so settings that differ only in the fields below can share one execution of stages 1-2c and differ in
 * stage 3 alone.  For every setting s and candidate f the call writes what fnp_seeker_select writes at topk = 1 when
 * the stages run with s's values in cfg, bit for bit:
 *   out_boxes (S,F,7), out_score (S,F), out_best (S,F) and out_count (S,F), slot s*F + f.  out_best is the
 *   index among b's compacted hypotheses (b->hyp_index maps it to the original one), -1 when no hypothesis of the
 *   frustum is valid for s; such a slot has a zero box, score 0 and count 0.
 * Setting s's valid set is the compacted hypotheses with hyp_iou > s.min_cam_iou; the count, occlusion and ego
 * normalisers are maxima over that set, while the distance term keeps cand_stats[13..14] (every hypothesis within
 * max_dist, whatever its IoU).  Ties go to the lowest index.
 * Call it after fnp_seeker_run (or the stages up to fnp_seeker_occlusion) on the same b.  settings_host is a HOST
 * array of n_settings (1..FNP_SELECT_MAX_SETTINGS) entries, passed by value as kernel parameters (256 x 32 B = 8 KB
 * of the 32 KB parameter space; the library allocates nothing).  Each CTA stages a frustum's counts and IoUs, plus
 * the distance, occlusion and centre-norm planes when some setting reads them: 4 H bytes per plane, at most 200 KB
 * (6-15 KB at H = 768).  A caller with more settings makes one call per 256 over the same stages 1-2c.
 * FNP_VARIANT_KITTI: that head's counts are first-match counts over the valid set, so they hold for a setting only
 * when its valid set is the one stages 1-2c compacted: every setting must have cfg->min_cam_iou, bit for bit, no
 * flags and no ego_w / occl_w (not terms of that score).  The count normaliser is then the SUM of the frustum's
 * compacted counts + 1e-8, the distance plane is always staged, and the score is that head's additive one
 * (dns_w + density + iou_w iou + dst_w dist), as fnp_seeker_select forms it for a KITTI cfg.
 * Build record (nvcc 12.9, -Xptxas -v, sm_100a), 256 threads, no static shared memory: select_multi_kernel<false>
 * (nuScenes) 48 registers, 8-byte stack frame, 4 bytes of spill stores / loads, 2672 SASS instructions;
 * select_multi_kernel<true> (KITTI) 40 registers, no stack, no spills, 1760 SASS instructions.
 * FNP_EINVAL: cfg->topk > 1; a KITTI setting outside the rule above; a flag other than
 * FNP_SEEKER_MULT / FNP_SEEKER_OCCL_MULT; a setting's min_cam_iou below cfg->min_cam_iou (the compaction was done
 * at cfg's threshold); a setting that needs hyp_dist (dst_w != 0, MULT, the KITTI variant) or hyp_nfar (occl_w > 0,
 * OCCL_MULT) on a batch without it -- hyp_nfar is formed by fnp_seeker_occlusion, which runs only when cfg itself turns
 * occlusion on. */
#define FNP_SELECT_MAX_SETTINGS 256
typedef struct fnp_select_setting {
    float dns_w, iou_w, dst_w, ego_w, occl_w, min_cam_iou;
    int32_t flags;           /* FNP_SEEKER_MULT | FNP_SEEKER_OCCL_MULT */
    int32_t reserved;
} fnp_select_setting;
int fnp_seeker_select_multi(const fnp_seeker_cfg *cfg, const fnp_seeker_batch *b, const fnp_select_setting *settings_host,
                            int n_settings, float *out_boxes, float *out_score, int32_t *out_best, int32_t *out_count,
                            void *stream);

/* Stage 4: batched rotated-BEV bitmask NMS in shared memory.  Segment s covers boxes
 * [seg_start[s], seg_start[s+1]) (<= max_seg_boxes <= FNP_SEG_NMS_MAX each, in priority order: an earlier
 * kept box suppresses later ones with IoU > thresh, and if label != NULL only boxes of the
 * same label interact).  order (n_boxes, nullable): entry i of a segment is box order[i]
 * (gather; lets the caller impose a score order without moving boxes).  valid (nullable,
 * indexed like boxes): entries < 0 are not boxes (never kept, never suppress).
 * keep_mask (n_boxes) uint8, indexed like boxes, is written. */
#define FNP_SEG_NMS_MAX 1024
int fnp_seg_nms_rotated(const float *boxes, const int32_t *label, const int32_t *order,
                        const int32_t *valid, const int32_t *seg_start, int n_segments,
                        int max_seg_boxes, float thresh, uint8_t *keep_mask, void *stream);

/* Recall counters (Detector3DTemplate.generate_recall_record): per frame, IoU3D of the
 * proposals vs GT, per-GT max, thresholded.  pred (sum K,7) with pred_start (n_frames+1),
 * pred_valid (nullable): rows with pred_valid[i] < 0 are skipped;
 * gt (sum G,8) = box7 + class label with gt_start (n_frames+1); thresh (n_thresh<=8).
 * counters (int64): [0]=gt, [1]=num_3known, [2]=num_6known, [3]=num_4unknown,
 * [4]=num_7unknown, then per threshold t: [5+5t+0]=rcnn, +1 = 3known, +2 = 6known,
 * +3 = 4unknown, +4 = 7unknown.  Counters are ACCUMULATED (caller zeroes them).
 * max_pred_per_frame / max_gt_per_frame: upper bounds of the per-frame row counts (they size
 * the shared memory of the kernel; 64 (max_pred + max_gt) + 4 max_gt bytes must fit in 200 KB). */
int fnp_recall_counters(const float *pred, const int32_t *pred_valid, const int32_t *pred_start, const float *gt,
                        const int32_t *gt_start, int n_frames, int max_pred_per_frame, int max_gt_per_frame,
                        const float *thresh_host, int n_thresh, long long *counters, void *stream);

/* Precision counters, the companion of fnp_recall_counters with the same arguments: recall counts the GT boxes some
 * proposal finds, this counts the proposals that find something -- what a looser filter costs.  counters (int64):
 * [0] = valid proposals (pred_valid[i] >= 0, or every row when pred_valid is NULL), then per threshold t:
 * [1+t] = valid proposals whose largest IoU3D over their frame's GT boxes is > thresh[t] (the IoU of
 * fnp_recall_counters, box_overlap + iou3d_from_overlap).  ACCUMULATED (caller zeroes them).  Shared memory:
 * 64 (max_pred + max_gt) + 4 max_pred bytes, at most 200 KB.  Build record (nvcc 12.9, -Xptxas -v, sm_100a):
 * precision_kernel 256 threads, 73 registers, 304-byte stack frame (box_overlap's vertex arrays), no spills. */
int fnp_precision_counters(const float *pred, const int32_t *pred_valid, const int32_t *pred_start, const float *gt,
                           const int32_t *gt_start, int n_frames, int max_pred_per_frame, int max_gt_per_frame,
                           const float *thresh_host, int n_thresh, long long *counters, void *stream);

/* Quality counters: recall and precision per class and per BEV range bin, for n_settings sets of proposals over the
 * same frames and GT, in one launch.  The IoU of a (GT, proposal) pair is that of fnp_recall_counters, bit for bit,
 * and each pair is computed once.
 *   pred: setting s's rows start at pred + 7 * s * pred_setting_stride (0: every setting reads the same rows);
 *   pred_valid (nullable): setting s's flags at pred_valid + s * valid_setting_stride, rows < 0 are not proposals;
 *   pred_label (1-based class), pred_start (n_frames+1): shared by every setting;
 *   gt (sum G,8) = box7 + 1-based class with gt_start (n_frames+1); trailing all-zero GT rows of a frame are dropped
 *   as in fnp_recall_counters.
 * Range: r = sqrt(x*x + y*y) of the box centre, each operation rounded in fp32; bin b = number of range edges <= r
 * (edges strictly increasing, > 0).  A GT box is binned by its centre, a proposal by its own.
 * T = n_thresh <= 8, R = n_edges + 1 <= 8, C = n_classes <= 32, W = 1 + 2T.  counters (int64), ACCUMULATED (caller
 * zeroes them), 2 C R W per setting: setting s starts at counters + 2 C R W s, then
 *   recall    [c][b][w], c = GT class - 1, b = GT bin:   w = 0 GT boxes;  1+t: best IoU over all valid proposals of
 *             the frame > thresh[t];  1+T+t: the same over the proposals with the GT's label;
 *   precision [c][b][w], c = label - 1, b = proposal bin: w = 0 valid proposals;  1+t: best IoU over the frame's GT
 *             > thresh[t];  1+T+t: the same over the GT boxes of the proposal's class.
 * Labels must lie in 1..C (the caller checks them; a box with another label is not counted).  Shared memory:
 * fnp_quality_smem_bytes(...) <= 200 KB.  FNP_EINVAL: T, R or C out of range, bad edges, shared memory, a negative
 * size or stride, a missing pointer.  Build record (nvcc 12.9, -Xptxas -v, sm_100a): quality_kernel 256 threads,
 * 71 registers, 272-byte stack frame (box_overlap's vertex arrays), no spills; one CTA per (frame, 8 settings). */
int fnp_quality_counters(const float *pred, long long pred_setting_stride, const int32_t *pred_valid,
                         long long valid_setting_stride, const int32_t *pred_label, const int32_t *pred_start,
                         int n_settings, const float *gt, const int32_t *gt_start, int n_frames, int max_pred_per_frame,
                         int max_gt_per_frame, int n_classes, const float *range_edges_host, int n_edges,
                         const float *thresh_host, int n_thresh, long long *counters, void *stream);
size_t fnp_quality_smem_bytes(int max_pred_per_frame, int max_gt_per_frame, int n_classes, int n_edges, int n_thresh);

/* ------------------------------------------------------------- host-side planning
 * (runs on the CPU, touches no device memory: every pointer here is a HOST pointer)
 *
 * Candidate frustums of a batch in reference order: frame, then cameras [2,0,1,5,3,4], then
 * torchvision.ops.batched_nms order (descending score), dropping score < score_thr
 * (frustum_proposals_v1.py:582-595).  det_* describe all n_dets GLIP boxes of the batch
 * (boxes (n_dets,4) xyxy fp32, labels/frame/cam int64).  Writes cand_det (capacity n_dets):
 * indices into det_* of the candidates, and frame_cand_start (n_frames+1).
 * Returns the number of candidates (>= 0) or FNP_EINVAL. */
int fnp_host_select_candidates(const float *det_boxes, const int64_t *det_labels,
                               const float *det_scores, const int64_t *det_frame,
                               const int64_t *det_cam, int n_dets, int n_frames, float nms_2d,
                               float score_thr, int32_t *cand_det, int32_t *frame_cand_start);

/* Whole-batch planning in one call: everything SeekerEngine.plan contributes to a batch.  One
 * fnp_host_frame per frame points at the frame's own host arrays (nothing is concatenated by the
 * caller); every output array is caller-allocated with the capacities fnp_host_plan_sizes reports
 * (sizes3 = {detections, point tiles, point rows} of the batch): arrays indexed by candidate have
 * room for `detections` entries, tile arrays for `point tiles`.  box_xywh: the 2D boxes are x, y, w, h
 * (BOX_FORMAT other than 'xyxy', frustum_proposals_v1.py:597-601: the 2D NMS runs on the raw numbers,
 * the corner is formed afterwards).  topk > 1 also fills frame_prop_start / prop_order (slot tables of
 * stage 4).  Returns FNP_OK / FNP_EINVAL. */
typedef struct fnp_host_frame {
    int64_t n_rows;              /* points of the frame                                    */
    const float *det_boxes;      /* (n_dets,4) fp32                                        */
    const int64_t *det_labels;   /* (n_dets) 1..A                                          */
    const float *det_scores;     /* (n_dets)                                               */
    const int64_t *det_cam;      /* (n_dets) 0..5                                          */
    const float *cam_mats;       /* (6,24): lidar2image rows 0..2 | combine | cam2lidar_t  */
    int32_t n_dets;
    int32_t reserved;
} fnp_host_frame;

typedef struct fnp_host_plan_out {
    /* the batch metadata the device reads (fnp_seeker_batch fields of the same names) */
    int64_t *frame_row_start;    /* (n_frames+1)   */
    int32_t *tile_frame;         /* (tiles)        */
    int32_t *tile_row0;          /* (tiles)        */
    int32_t *frame_tile_start;   /* (n_frames+1)   */
    float *cam_mats;             /* (n_frames,6,24)*/
    int32_t *frame_cand_start;   /* (n_frames+1)   */
    int32_t *cam_cand_start;     /* (6 n_frames+1) */
    int32_t *cand_frame;         /* (detections)   */
    int32_t *cand_cam;
    int32_t *cand_label;
    float *cand_box2d;           /* (detections,4) */
    int32_t *nms_order;          /* (detections) stage-4 priority order                    */
    int32_t *frame_prop_start;   /* (n_frames+1), topk > 1 only (else may be NULL)         */
    int32_t *prop_order;         /* (detections * topk), topk > 1 only                     */
    /* host-side bookkeeping */
    float *cand_score;           /* (detections) 2D score of each candidate                */
    int32_t *cand_det;           /* (detections) index of each candidate among the batch's detections, frames
                                    back to back                                           */
    /* written by the call */
    int32_t n_cands, n_tiles, max_cands_per_frame, reserved;
    int64_t total_rows;
} fnp_host_plan_out;

int fnp_host_plan_sizes(const fnp_host_frame *frames, int n_frames, int64_t *sizes3);
int fnp_host_plan(const fnp_host_frame *frames, int n_frames, float nms_2d, float score_thr, int box_xywh,
                  int topk, fnp_host_plan_out *out);

/* Stage-4 priority order: inside every frame the candidates by descending 2D score, ties by
 * candidate index.  cand_score (F), frame_cand_start (n_frames+1), order (F) out. */
int fnp_host_nms_order(const float *cand_score, const int32_t *frame_cand_start, int n_frames,
                       int32_t *order);

/* Column gather of the point table on the host: x, y, z of `rows` rows of `stride` floats (xyz at
 * column xyz_offset) into dst_host (rows,3), so that only the 12 B/point the path reads cross PCIe
 * (the reference uploads every column: pcdet/models/__init__.py:23-36).  n_threads worker threads
 * split the rows.  _begin returns a ticket (>= 0) at once and gathers in the background;
 * fnp_host_pack_wait(ticket) blocks until that gather is complete (FNP_EWORKSPACE: more than 16
 * gathers in flight).  dst_host is typically pinned memory the next H2D copy reads. */
int fnp_host_pack_xyz(const float *src_host, int64_t rows, int stride, int xyz_offset, float *dst_host,
                      int n_threads);
int fnp_host_pack_xyz_begin(const float *src_host, int64_t rows, int stride, int xyz_offset, float *dst_host,
                            int n_threads);
int fnp_host_pack_wait(int ticket);
/* The same for a table that lies in n_segments pieces on the host (one per frame, as a data loader
 * leaves them): segment s has seg_rows[s] rows at seg_src_host[s]; the pieces are gathered back to
 * back into dst_host, so no concatenated copy of the full-width rows is ever made. */
int fnp_host_pack_xyz_multi_begin(const float *const *seg_src_host, const int64_t *seg_rows, int n_segments,
                                  int stride, int xyz_offset, float *dst_host, int n_threads);

/* Host->device upload of a small block by a kernel instead of the copy engine: src is pinned,
 * UVA-mapped host memory (cudaHostAlloc / torch pin_memory), dst device memory, both 16-byte
 * aligned, bytes a multiple of 16.  The per-batch metadata goes this way so that it cannot queue
 * behind a large point copy of another stream in the H2D engine. */
int fnp_upload_from_pinned(void *dst, const void *src_pinned_host, size_t bytes, void *stream);

/* Tuning / test switches, process-wide; not part of the stable surface.  "cull_sectors" (default 1): stage 1
 * consults the per-frame azimuth-sector table to skip cameras that cannot see a point (0: every camera for
 * every point -- same results, the tests compare the two).  Returns FNP_EINVAL for an unknown name. */
int fnp_set_option(const char *name, int value);

/* Test hook: out (4,n) = sinf(x), cosf(x), atan2f(y,x), fnp_exp(x) as evaluated on the
 * device by this library's build (checked against the oracle's restatements). */
int fnp_dbg_math(const float *x, const float *y, float *out, int n, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* FNP_H_ */
