"""ctypes binding of libfnp_sm100.so (the C ABI declared in include/fnp.h).

There is no CPU fallback: importing this module fails loudly when the CUDA library has not
been built (python -m findnpropagate_b200.build), and every compute entry point needs a
CUDA device.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("FNP_LIB_PATH") or os.path.join(HERE, "libfnp_sm100.so")   # override: A/B builds

if not os.path.exists(SO_PATH):
    raise ImportError(
        "findnpropagate_b200: %s is missing -- build it with `python -m findnpropagate_b200.build` "
        "(nvcc, sm_100a). There is no CPU fallback." % SO_PATH)

lib = C.CDLL(SO_PATH)

_vp = C.c_void_p
_i = C.c_int
_f = C.c_float


class SeekerCfg(C.Structure):
    _fields_ = [("num_mags", C.c_int32), ("num_yaw_size", C.c_int32), ("n_classes", C.c_int32),
                ("clamp_bottom", C.c_int32), ("img_w", _f), ("img_h", _f), ("lq", _f), ("uq", _f),
                ("cq", _f), ("frustum_min", _f), ("max_dist", _f), ("min_cam_iou", _f),
                ("dns_w", _f), ("iou_w", _f),
                ("dst_w", _f), ("ego_w", _f), ("occl_w", _f), ("search_depth", _f), ("flags", C.c_int32),
                ("topk", C.c_int32), ("nms_normal", _f), ("variant", C.c_int32)]


class SeekerBatch(C.Structure):
    _fields_ = [
        ("n_frames", C.c_int32), ("n_cands", C.c_int32), ("n_tiles", C.c_int32),
        ("max_cands_per_frame", C.c_int32),
        ("points", _vp), ("point_stride", C.c_int32), ("xyz_offset", C.c_int32),
        ("frame_row_start", _vp), ("tile_frame", _vp), ("tile_row0", _vp), ("frame_tile_start", _vp),
        ("cam_mats", _vp), ("frame_cand_start", _vp), ("cam_cand_start", _vp), ("cand_frame", _vp), ("cand_cam", _vp),
        ("cand_label", _vp), ("cand_box2d", _vp), ("base_boxes", _vp), ("base_corners", _vp),
        ("mags", _vp),
        ("cell_masks", _vp), ("mask_words", C.c_int32), ("cand_npts", _vp), ("page_tab", _vp),
        ("page_tab_stride", C.c_int32), ("page_planes", C.c_int32), ("frustum_pts", _vp),
        ("pts_capacity", C.c_int64), ("cand_stats", _vp), ("centres", _vp),
        ("hyp_prep", _vp), ("hyp_index", _vp), ("hyp_iou", _vp), ("hyp_nvalid", _vp),
        ("hyp_boxes_dbg", _vp), ("hyp_iou_dbg", _vp), ("hyp_valid_dbg", _vp),
        ("split_points", C.c_int32), ("max_items", C.c_int32),
        ("cand_item_start", _vp), ("items", _vp), ("counts", _vp),
        ("score_mode", C.c_int32), ("sweep_cols", _vp),
        ("out_boxes", _vp), ("out_score", _vp), ("out_best", _vp), ("out_count", _vp),
        ("status", _vp),
        ("hyp_dist", _vp), ("hyp_nfar", _vp), ("hyp_score", _vp),
    ]


class SelectSetting(C.Structure):
    _fields_ = [("dns_w", _f), ("iou_w", _f), ("dst_w", _f), ("ego_w", _f), ("occl_w", _f), ("min_cam_iou", _f),
                ("flags", C.c_int32), ("reserved", C.c_int32)]


class HostFrame(C.Structure):
    _fields_ = [("n_rows", C.c_int64), ("det_boxes", _vp), ("det_labels", _vp), ("det_scores", _vp), ("det_cam", _vp),
                ("cam_mats", _vp), ("n_dets", C.c_int32), ("reserved", C.c_int32)]


class HostPlanOut(C.Structure):
    _fields_ = [("frame_row_start", _vp), ("tile_frame", _vp), ("tile_row0", _vp), ("frame_tile_start", _vp),
                ("cam_mats", _vp), ("frame_cand_start", _vp), ("cam_cand_start", _vp), ("cand_frame", _vp),
                ("cand_cam", _vp), ("cand_label", _vp), ("cand_box2d", _vp), ("nms_order", _vp),
                ("frame_prop_start", _vp), ("prop_order", _vp), ("cand_score", _vp), ("cand_det", _vp),
                ("n_cands", C.c_int32), ("n_tiles", C.c_int32), ("max_cands_per_frame", C.c_int32),
                ("reserved", C.c_int32), ("total_rows", C.c_int64)]


lib.fnp_seeker_cull_tile.restype = C.c_int
lib.fnp_seeker_cull_tile.argtypes = []
CULL_TILE = int(lib.fnp_seeker_cull_tile())
PAGE_POINTS = 256
SCORE_AUTO, SCORE_DIRECT, SCORE_SWEEP = 0, 1, 2
VARIANT_NUSCENES, VARIANT_KITTI = 0, 1
SEEKER_MULT, SEEKER_OCCL_MULT, SEEKER_MULTICAM_IOU = 1, 2, 4
SWEEP_MIN_MAGS = 16
SWEEP_COL_FLOATS = 20
SEG_NMS_MAX = 1024
STATS_FLOATS = 40

lib.fnp_version.restype = C.c_char_p
lib.fnp_version.argtypes = []
lib.fnp_points_in_boxes.restype = _i
lib.fnp_points_in_boxes.argtypes = [_vp, _vp, _vp, _i, _i, _i, _vp]
lib.fnp_count_in_boxes.restype = _i
lib.fnp_count_in_boxes.argtypes = [_vp, _vp, _vp, _vp, _i, _vp, _vp]
lib.fnp_crop_points_in_boxes.restype = _i
lib.fnp_crop_points_in_boxes.argtypes = [_vp, _i, _vp, C.c_longlong, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp,
                                         C.c_size_t, _vp]
lib.fnp_crop_workspace_bytes.restype = C.c_size_t
lib.fnp_crop_all_count.restype = _i
lib.fnp_crop_all_count.argtypes = [_vp, _i, _vp, C.c_longlong, _vp, _vp, _i, _i, _vp, _vp, _vp, C.c_size_t, _vp]
lib.fnp_crop_all_scatter.restype = _i
lib.fnp_crop_all_scatter.argtypes = [_vp, _i, _vp, C.c_longlong, _vp, _vp, _vp, _i, _i, _vp, _vp, C.c_longlong, _vp,
                                     C.c_size_t, _vp]
lib.fnp_crop_workspace_bytes.argtypes = [_vp, _vp, _i]
for _n in ("fnp_boxes_overlap_bev", "fnp_boxes_iou_bev"):
    getattr(lib, _n).restype = _i
    getattr(lib, _n).argtypes = [_vp, _vp, _vp, _i, _i, _vp]
lib.fnp_boxes_iou3d.restype = _i
lib.fnp_boxes_iou3d.argtypes = [_vp, _vp, _vp, _i, _i, _vp]
lib.fnp_boxes_aligned_iou3d.restype = _i
lib.fnp_boxes_aligned_iou3d.argtypes = [_vp, _vp, _vp, _i, _vp]
lib.fnp_points_in_boxes_matrix.restype = _i
lib.fnp_points_in_boxes_matrix.argtypes = [_vp, _vp, _vp, _i, _i, _vp]
lib.fnp_host_prep_boxes_cpu.restype = _i
lib.fnp_host_prep_boxes_cpu.argtypes = [_vp, _vp, _i]
lib.fnp_boxes_aligned_overlap_bev.restype = _i
lib.fnp_boxes_aligned_overlap_bev.argtypes = [_vp, _vp, _vp, _i, _vp]
lib.fnp_nms_workspace_bytes.restype = C.c_size_t
lib.fnp_nms_workspace_bytes.argtypes = [_i]
for _n in ("fnp_nms_rotated", "fnp_nms_normal"):
    getattr(lib, _n).restype = _i
    getattr(lib, _n).argtypes = [_vp, _i, _f, _vp, _vp, _vp, C.c_size_t, _vp]
for _n in ("fnp_seeker_cull", "fnp_seeker_frustum_stats", "fnp_seeker_hypotheses", "fnp_seeker_score",
           "fnp_seeker_occlusion", "fnp_seeker_select", "fnp_seeker_run"):
    getattr(lib, _n).restype = _i
    getattr(lib, _n).argtypes = [C.POINTER(SeekerCfg), C.POINTER(SeekerBatch), _vp]
lib.fnp_seeker_score_mode.restype = _i
lib.fnp_seeker_score_mode.argtypes = [C.POINTER(SeekerCfg), C.POINTER(SeekerBatch)]
lib.fnp_seeker_mask_words.restype = _i
lib.fnp_seeker_mask_words.argtypes = [_i]
lib.fnp_seeker_cell_mask_bytes.restype = C.c_size_t
lib.fnp_seeker_cell_mask_bytes.argtypes = [C.POINTER(SeekerCfg), _i, _i]
lib.fnp_seg_nms_rotated.restype = _i
lib.fnp_seg_nms_rotated.argtypes = [_vp, _vp, _vp, _vp, _vp, _i, _i, _f, _vp, _vp]
SEG_NMS_MAX_THRESH = 8
lib.fnp_seg_nms_rotated_multi.restype = _i
lib.fnp_seg_nms_rotated_multi.argtypes = [_vp, C.c_longlong, _vp, C.c_longlong, _vp, _vp, _i, _i, _i, C.POINTER(_f), _i,
                                          _vp, C.c_longlong, _vp]
SELECT_MAX_SETTINGS = 256
lib.fnp_seeker_select_multi.restype = _i
lib.fnp_seeker_select_multi.argtypes = [C.POINTER(SeekerCfg), C.POINTER(SeekerBatch), C.POINTER(SelectSetting), _i,
                                        _vp, _vp, _vp, _vp, _vp]
for _n in ("fnp_recall_counters", "fnp_precision_counters"):
    getattr(lib, _n).restype = _i
    getattr(lib, _n).argtypes = [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, C.POINTER(_f), _i, _vp, _vp]
lib.fnp_quality_counters.restype = _i
lib.fnp_quality_counters.argtypes = [_vp, C.c_longlong, _vp, C.c_longlong, _vp, _vp, _i, _vp, _vp, _i, _i, _i, _i,
                                     C.POINTER(_f), _i, C.POINTER(_f), _i, _vp, _vp]
lib.fnp_quality_smem_bytes.restype = C.c_size_t
lib.fnp_quality_smem_bytes.argtypes = [_i, _i, _i, _i, _i]

lib.fnp_host_select_candidates.restype = _i
lib.fnp_host_select_candidates.argtypes = [_vp, _vp, _vp, _vp, _vp, _i, _i, _f, _f, _vp, _vp]

lib.fnp_host_plan_sizes.restype = _i
lib.fnp_host_plan_sizes.argtypes = [_vp, _i, _vp]
lib.fnp_host_plan.restype = _i
lib.fnp_host_plan.argtypes = [_vp, _i, _f, _f, _i, _i, C.POINTER(HostPlanOut)]
lib.fnp_host_nms_order.restype = _i
lib.fnp_host_nms_order.argtypes = [_vp, _vp, _i, _vp]
for _n in ("fnp_host_pack_xyz", "fnp_host_pack_xyz_begin"):
    getattr(lib, _n).restype = _i
    getattr(lib, _n).argtypes = [_vp, C.c_int64, _i, _i, _vp, _i]
lib.fnp_host_pack_xyz_multi_begin.restype = _i
lib.fnp_host_pack_xyz_multi_begin.argtypes = [_vp, _vp, _i, _i, _i, _vp, _i]
lib.fnp_host_pack_wait.restype = _i
lib.fnp_host_pack_wait.argtypes = [_i]

lib.fnp_upload_from_pinned.restype = _i
lib.fnp_upload_from_pinned.argtypes = [_vp, _vp, C.c_size_t, _vp]

lib.fnp_set_option.restype = _i
lib.fnp_set_option.argtypes = [C.c_char_p, _i]
lib.fnp_dbg_math.restype = _i
lib.fnp_dbg_math.argtypes = [_vp, _vp, _vp, _i, _vp]

EXPORTED = [
    "fnp_dbg_math", "fnp_upload_from_pinned",
    "fnp_version", "fnp_points_in_boxes", "fnp_count_in_boxes", "fnp_crop_points_in_boxes", "fnp_crop_workspace_bytes",
    "fnp_crop_all_count", "fnp_crop_all_scatter",
    "fnp_boxes_overlap_bev",
    "fnp_boxes_iou_bev", "fnp_boxes_aligned_overlap_bev", "fnp_nms_workspace_bytes", "fnp_nms_rotated",
    "fnp_nms_normal", "fnp_seeker_cull", "fnp_seeker_frustum_stats", "fnp_seeker_hypotheses",
    "fnp_seeker_score", "fnp_seeker_score_mode", "fnp_seeker_occlusion", "fnp_seeker_select", "fnp_seeker_run", "fnp_seg_nms_rotated", "fnp_seg_nms_rotated_multi", "fnp_seeker_mask_words", "fnp_seeker_cell_mask_bytes",
    "fnp_recall_counters", "fnp_precision_counters", "fnp_quality_counters", "fnp_quality_smem_bytes",
    "fnp_seeker_select_multi", "fnp_host_select_candidates", "fnp_host_pack_xyz", "fnp_host_pack_xyz_begin",
    "fnp_host_pack_wait", "fnp_host_nms_order", "fnp_host_pack_xyz_multi_begin", "fnp_host_plan_sizes", "fnp_host_plan",
    "fnp_points_in_boxes_matrix", "fnp_host_prep_boxes_cpu", "fnp_boxes_iou3d", "fnp_boxes_aligned_iou3d", "fnp_set_option", "fnp_seeker_cull_tile",
]


def check(rc, what):
    """Turn a C-ABI return code into an exception (the reference prints and exit(-1)s)."""
    if rc == 0:
        return
    if rc == -1:
        raise ValueError("%s: invalid argument" % what)
    if rc == -2:
        raise ValueError("%s: workspace too small" % what)
    raise RuntimeError("%s: CUDA error %d" % (what, rc))


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("findnpropagate_b200 ops run on CUDA tensors only (no CPU fallback); got %s"
                               % t.device)


def current_stream(device=None):
    import torch
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
