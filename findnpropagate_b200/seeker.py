"""Greedy Box Seeker, B200-native.

Host-side mirror of ``FrustumProposerOG`` (reference:
pcdet/models/dense_heads/frustum_proposals_v1.py:142-1573) for the option set of
tools/cfgs/nuscenes_box_seeker_proposals.yaml: same constructor arguments / PARAMS keys,
same ``get_proposals`` / ``get_bboxes`` / ``forward`` contract and output format, with the
per-frame Python loop replaced by five fused CUDA stages over a *batch* of frames
(libfnp_sm100.so, include/fnp.h):

    host  : 2D NMS + score threshold (nms2d.py), camera matrices, tile/candidate tables
    GPU 1 : projection x cameras + per-2D-box frustum cull + ordered compaction
    GPU 1b: depth quantiles, point AABB, frustum corners, centre line
    GPU 2a: hypothesis grid, softmin front shift, distance + 2D-IoU filters
    GPU 2b: points-in-boxes scoring (TMA-staged point tiles)
    GPU 3 : density + IoU score, greedy argmax
    GPU 4 : (optional) rotated-BEV NMS of the frame's proposals, recall counters

There is no CPU compute path: the engine raises if CUDA or the extension is missing.
"""
import ctypes as C
import math
import time
from dataclasses import dataclass
from typing import List, Optional

import numpy as np
import torch

from . import _lib, nms2d

ANCHORS = [[4.63, 1.97, 1.74], [6.93, 2.51, 2.84], [6.37, 2.85, 3.19], [10.5, 2.94, 3.47],
           [12.29, 2.90, 3.87], [0.50, 2.53, 0.98], [2.11, 0.77, 1.47], [1.70, 0.60, 1.28],
           [0.73, 0.67, 1.77], [0.41, 0.41, 1.07]]          # frustum_proposals_v1.py:270-281
IMAGE_SIZE = (900, 1600)                                     # frustum_proposals_v1.py:203
FRUSTUM_MIN = 2.0                                            # frustum_proposals_v1.py:240
# FrustumProposerOGKITTI (frustum_proposals_v1_kitti.py:157-166): car, tram, truck, van, person sitting, cyclist,
# pedestrian; same constructor defaults except max_dist = 70 (:44); image_size and frustum_min as above (:108, :141)
ANCHORS_KITTI = [[3.9, 1.6, 1.56], [6.37, 2.85, 3.19], [6.93, 2.51, 2.84], [6.93, 2.51, 2.84], [0.8, 0.6, 1.73],
                 [1.76, 0.6, 1.73], [0.8, 0.6, 1.73]]

# constructor defaults, frustum_proposals_v1.py:146-148
DEFAULTS = dict(lq=0.336, uq=0.356, iou_w=0.95, dst_w=0.226, dns_w=0.05, min_cam_iou=0.3,
                size_min=0.957, size_max=1.2, ry_min=0.0, ry_max=float(torch.pi), cq=0.46, num_mags=6,
                max_dist=50, num_sizes=4, num_rotations=10, topk=1, nms_2d=0.7, nms_3d=1.0,
                score_thr=0.1, nms_normal=0.7, clamp_bottom=0)

RECALL_KEYS = ["gt", "num_3known", "num_6known", "num_4unknown", "num_7unknown"]
RECALL_PER_THRESH = ["rcnn", "rcnn_3known", "rcnn_6known", "rcnn_4unknown", "rcnn_7unknown"]


FLAG_KEYS = ("MULT", "OCCL_MULT", "MULTICAM_IOU")     # MODEL.DENSE_HEAD switches, frustum_proposals_v1.py:154-156
# the parameters only stage 3 reads (with min_cam_iou, which only removes hypotheses): settings that differ in these
# alone share stages 1-2c (SeekerEngine.evaluate_settings, fnp_seeker_select_multi)
SELECT_KEYS = ("dns_w", "iou_w", "dst_w", "ego_w", "occl_w", "min_cam_iou", "MULT", "OCCL_MULT")
# the KITTI head's: its counts are first-match counts over the valid set, which min_cam_iou changes
SELECT_KEYS_KITTI = ("dns_w", "iou_w", "dst_w")


def resolve_params(params: Optional[dict], variant: str = "nuscenes") -> dict:
    """PARAMS of the head (frustum_proposals_v1.py:167-195) over the constructor defaults.  Besides the
    shipped option set, the optional terms of SURVEY.md 8 row f3 are supported: dst_w, ego_w, occl_w,
    search_depth and the switches MULT / OCCL_MULT / MULTICAM_IOU (keys of the same dict).
    variant "kitti": FrustumProposerOGKITTI (frustum_proposals_v1_kitti.py:38-98), whose score has the density, IoU
    and distance terms only."""
    p = dict(DEFAULTS)
    if variant == "kitti":
        p["max_dist"] = 70
    p.update(ego_w=0, occl_w=0, aln_w=0, rand_center=False, search_depth=None)      # :160-165
    p.update({k: False for k in FLAG_KEYS})
    if params:
        p.update(params)
    # rand_center (:844-847; frustum_proposals_v1_kitti.py:568-571): the hypothesis centres of a frustum are
    # weighted_centre_xyz + torch.randn((num_mags, 3)) drawn from the device's default generator, one draw per frustum
    # with points, in frustum order -- reproduced draw for draw (same generator, same shapes, same order), so a run
    # seeded like the reference's gives the reference's centres.
    unsupported = []
    if int(p["topk"]) < 1:
        unsupported.append("topk < 1")
    if p["nms_3d"] != 0:
        unsupported.append("nms_3d != 0 (the reference asserts it too, :209)")
    if p.get("aln_w"):
        unsupported.append("aln_w (it cannot run in the reference either: frustum_proposals_v1.py:987 indexes the (P,3) points "
                           "with a (1,P) mask and raises IndexError as soon as a hypothesis holds more than 3 points)")
    if p.get("rand_center") and int(p["num_mags"]) < 1:
        unsupported.append("rand_center with num_mags < 1")
    if p["search_depth"] is not None and not p["search_depth"] > 0:
        unsupported.append("search_depth <= 0")
    if variant == "kitti":
        for k in ("ego_w", "occl_w") + FLAG_KEYS:      # read by that constructor, never used in its score (:650-654)
            if p.get(k):
                unsupported.append("%s with the KITTI head (not a term of its score)" % k)
    if unsupported:
        raise NotImplementedError("Box Seeker options outside the supported set: " + ", ".join(unsupported))
    return p


def select_setting(p: dict) -> "_lib.SelectSetting":
    """The fnp_select_setting of a parameter dict (its SELECT_KEYS; the head's defaults for those it leaves out)."""
    p = dict(dict(DEFAULTS, ego_w=0, occl_w=0, MULT=False, OCCL_MULT=False), **{k: p[k] for k in SELECT_KEYS if k in p})
    return _lib.SelectSetting(dns_w=float(p["dns_w"]), iou_w=float(p["iou_w"]), dst_w=float(p["dst_w"]),
                              ego_w=float(p["ego_w"] or 0), occl_w=float(p["occl_w"] or 0),
                              min_cam_iou=float(p["min_cam_iou"]),
                              flags=(_lib.SEEKER_MULT if p["MULT"] else 0) | (_lib.SEEKER_OCCL_MULT if p["OCCL_MULT"] else 0),
                              reserved=0)


def build_tables(p: dict, anchors=None):
    """base_boxes (A,J,7), base_corners (A,J,8,3) -- the constructor tables of
    frustum_proposals_v1.py:282-298 (+ box_utils.boxes_to_corners_3d, box_utils.py:28-52),
    built with the same torch calls on the host."""
    anchors = torch.tensor(ANCHORS if anchors is None else anchors, dtype=torch.float32)
    A, R, S = anchors.shape[0], int(p["num_rotations"]), int(p["num_sizes"])
    size_variations = torch.linspace(p["size_min"], p["size_max"], steps=S)
    base_rotations = torch.linspace(p["ry_min"], p["ry_max"], steps=R)
    base = torch.zeros((A, R, S, 7))
    base[..., 3:6] = anchors[:, None, None, :]
    base[..., 6] = base_rotations[None, :, None]
    base[..., 3:6] = base[..., 3:6] * size_variations[None, None, :, None]
    flat = base.reshape(-1, 7)
    template = flat.new_tensor(([1, 1, -1], [1, -1, -1], [-1, -1, -1], [-1, 1, -1],
                                [1, 1, 1], [1, -1, 1], [-1, -1, 1], [-1, 1, 1])) / 2
    corners = flat[:, None, 3:6].repeat(1, 8, 1) * template[None, :, :]
    cosa, sina = torch.cos(flat[:, 6]), torch.sin(flat[:, 6])
    zeros, ones = torch.zeros_like(cosa), torch.ones_like(cosa)
    rot = torch.stack((cosa, sina, zeros, -sina, cosa, zeros, zeros, zeros, ones), dim=1).view(-1, 3, 3)
    corners = torch.matmul(corners, rot) + flat[:, None, 0:3]
    return base.reshape(A, R * S, 7).contiguous(), corners.reshape(A, R * S, 8, 3).contiguous()


def camera_matrices(lidar2image, camera2lidar, camera_intrinsics):
    """(B,6,24) f32: lidar2image rows 0..2 | combine = cam2lidar_R @ inverse(K) | cam2lidar_t
    (frustum_proposals_v1.py:1442-1452 and :1512-1535), computed with torch on the host."""
    l2i = torch.as_tensor(np.asarray(lidar2image), dtype=torch.float32)
    c2l = torch.as_tensor(np.asarray(camera2lidar), dtype=torch.float32)
    K = torch.as_tensor(np.asarray(camera_intrinsics), dtype=torch.float32)[..., :3, :3]
    combine = c2l[..., :3, :3].matmul(torch.inverse(K))
    out = torch.cat([l2i[..., :3, :].reshape(*l2i.shape[:-2], 12), combine.reshape(*combine.shape[:-2], 9),
                     c2l[..., :3, 3]], dim=-1)
    return out.numpy()


@dataclass
class FrameInput:
    """What the engine needs of one frame (host memory)."""
    points: np.ndarray            # (N, C>=3) f32, xyz in columns xyz_offset..+3
    lidar2image: np.ndarray       # (6,4,4)
    camera2lidar: np.ndarray      # (6,4,4)
    camera_intrinsics: np.ndarray  # (6,4,4)
    det_boxes: np.ndarray         # (D,4) xyxy
    det_labels: np.ndarray        # (D,) 1..10
    det_scores: np.ndarray        # (D,)
    det_cam_idx: np.ndarray       # (D,) 0..5
    gt_boxes: Optional[np.ndarray] = None   # (G,>=8): box7 ... class label last
    _prep: Optional[dict] = None            # per-frame host preparation (prepare()); assigning any field drops it

    def __setattr__(self, name, value):
        object.__setattr__(self, name, value)
        if name != "_prep":
            object.__setattr__(self, "_prep", None)

    def prepare(self):
        """Per-FRAME host work, done once (by the loader's worker threads, or lazily by the first plan()):
        typed contiguous detection arrays, the frame's (6,24) camera-matrix block (inverse(K), combine --
        frustum_proposals_v1.py:1442-1452, 1512-1535) and the fnp_host_frame record fnp_host_plan reads.
        SeekerEngine.plan() then only joins the records of a batch and makes one C call."""
        if self._prep is None:
            boxes = np.ascontiguousarray(self.det_boxes, np.float32).reshape(-1, 4)
            labels = np.ascontiguousarray(self.det_labels, np.int64).reshape(-1)
            scores = np.ascontiguousarray(self.det_scores, np.float32).reshape(-1)
            cam = np.ascontiguousarray(self.det_cam_idx, np.int64).reshape(-1)
            assert boxes.shape[0] == labels.shape[0] == scores.shape[0] == cam.shape[0]
            cm = np.ascontiguousarray(camera_matrices(self.lidar2image, self.camera2lidar, self.camera_intrinsics), np.float32)
            assert cm.shape == (6, 24)
            rec = _lib.HostFrame(n_rows=int(self.points.shape[0]), det_boxes=boxes.ctypes.data, det_labels=labels.ctypes.data,
                                 det_scores=scores.ctypes.data, det_cam=cam.ctypes.data, cam_mats=cm.ctypes.data,
                                 n_dets=int(scores.shape[0]), reserved=0)
            self._prep = dict(blob=bytes(rec), keep=(boxes, labels, scores, cam, cm))
        return self._prep


_KITTI_BLOCKS = {}      # calibration repeats from frame to frame (it is fixed per drive): block by content


def kitti_camera_block(P2, R0, V2C, device):
    """The 144 floats of a frame for FNP_VARIANT_KITTI (include/fnp.h): M1 = V2C.T @ R0.T | P2.T | cu cv fu fv tx ty |
    inverse((R0_ext @ V2C_ext).T) -- formed with the calls CalibrationTorch makes (calibration_kitti.py:128-169), on
    the device the reference forms them on, so that the bits are its bits."""
    key = (str(device), np.asarray(P2, np.float32).tobytes(), np.asarray(R0, np.float32).tobytes(),
           np.asarray(V2C, np.float32).tobytes())
    hit = _KITTI_BLOCKS.get(key)
    if hit is not None:
        return hit
    if len(_KITTI_BLOCKS) > 256:
        _KITTI_BLOCKS.clear()
    _KITTI_BLOCKS[key] = out = _kitti_camera_block(P2, R0, V2C, device)
    return out


def _kitti_camera_block(P2, R0, V2C, device):
    P2 = torch.as_tensor(np.asarray(P2, np.float32), device=device)
    R0 = torch.as_tensor(np.asarray(R0, np.float32), device=device)
    V2C = torch.as_tensor(np.asarray(V2C, np.float32), device=device)
    m1 = V2C.T @ R0.T                                                   # (4,3)
    cu, cv, fu, fv = P2[0, 2], P2[1, 2], P2[0, 0], P2[1, 1]
    tx, ty = P2[0, 3] / (-fu), P2[1, 3] / (-fv)
    r0e = torch.cat((torch.cat((R0, R0.new_zeros((3, 1))), dim=1), R0.new_zeros((1, 4))), dim=0)
    r0e[3, 3] = 1
    v2ce = torch.cat((V2C, V2C.new_zeros((1, 4))), dim=0)
    v2ce[3, 3] = 1
    minv = torch.inverse(torch.matmul(r0e, v2ce).T)                     # (4,4)
    out = torch.zeros(144, dtype=torch.float32, device=device)
    out[0:12] = m1.reshape(-1)
    out[12:24] = P2.T.reshape(-1)
    out[24:30] = torch.stack((cu, cv, fu, fv, tx, ty))
    out[32:48] = minv.reshape(-1)
    return out.cpu().numpy().reshape(6, 24)


@dataclass
class KittiFrameInput:
    """One KITTI frame for SeekerEngine(variant="kitti"): LiDAR points, the calibration (P2 (3,4), R0 (3,3),
    Tr_velo2cam (3,4) -- pcdet.utils.calibration_kitti.Calibration) and the 2D detections of the one camera as
    x, y, w, h boxes (PreprocessedDetector on one COCO result file, frustum_proposals_v1_kitti.py:150)."""
    points: np.ndarray            # (N, C>=3) f32
    P2: np.ndarray
    R0: np.ndarray
    V2C: np.ndarray
    det_boxes: np.ndarray         # (D,4) x, y, w, h
    det_labels: np.ndarray        # (D,) 1..7
    det_scores: np.ndarray        # (D,)
    gt_boxes: Optional[np.ndarray] = None
    device: str = "cuda"
    _prep: Optional[dict] = None

    def prepare(self):
        if self._prep is None:
            boxes = np.ascontiguousarray(self.det_boxes, np.float32).reshape(-1, 4)
            labels = np.ascontiguousarray(self.det_labels, np.int64).reshape(-1)
            scores = np.ascontiguousarray(self.det_scores, np.float32).reshape(-1)
            cam = np.zeros(scores.shape[0], np.int64)                   # c = 0 (:336)
            cm = np.ascontiguousarray(kitti_camera_block(self.P2, self.R0, self.V2C, self.device), np.float32)
            rec = _lib.HostFrame(n_rows=int(self.points.shape[0]), det_boxes=boxes.ctypes.data, det_labels=labels.ctypes.data,
                                 det_scores=scores.ctypes.data, det_cam=cam.ctypes.data, cam_mats=cm.ctypes.data,
                                 n_dets=int(scores.shape[0]), reserved=0)
            self._prep = dict(blob=bytes(rec), keep=(boxes, labels, scores, cam, cm))
        return self._prep


class _Arena:
    """Grow-only device/pinned scratch so that steady-state batches allocate nothing."""

    def __init__(self, device):
        self.device = device
        self.bufs = {}

    def get(self, name, nbytes, pinned=False):
        nbytes = int(max(nbytes, 256))
        t = self.bufs.get(name)
        if t is None or t.numel() < nbytes:
            cap = int(nbytes * 1.25) + 256
            if pinned:
                t = torch.empty(cap, dtype=torch.uint8, pin_memory=True)
            else:
                t = torch.empty(cap, dtype=torch.uint8, device=self.device)
            self.bufs[name] = t
        return t


class _FrameResults:
    """Per-frame results of a batch as a read-only sequence: frame b -> dict(pred_boxes (K,7) f32, pred_scores (K) f32,
    pred_labels (K) int32[, nms_keep (K) bool]) -- the reference's per-frame output (frustum_proposals_v1.py:1554-1573).
    The dicts are views of the batch's compacted arrays, made when a frame is asked for: a 256-frame batch whose
    consumer only wants the packed arrays (the frame-sharded exchange) pays nothing per frame."""

    def __init__(self, boxes, scores, labels, keep, start):
        self._b, self._s, self._l, self._k, self._st = boxes, scores, labels, keep, start

    def __len__(self):
        return len(self._st) - 1

    def __getitem__(self, b):
        if isinstance(b, slice):
            return [self[i] for i in range(*b.indices(len(self)))]
        if b < 0:
            b += len(self)
        if not 0 <= b < len(self):
            raise IndexError(b)
        lo, hi = int(self._st[b]), int(self._st[b + 1])
        d = dict(pred_boxes=self._b[lo:hi], pred_scores=self._s[lo:hi], pred_labels=self._l[lo:hi])
        if self._k is not None:
            d["nms_keep"] = self._k[lo:hi]
        return d

    def __iter__(self):
        return (self[b] for b in range(len(self)))


def _align(x, a=256):
    return (x + a - 1) // a * a


_F32, _I32, _I64, _U8 = (np.dtype(t) for t in (np.float32, np.int32, np.int64, np.uint8))


class OutLayout:
    """The output block of one execute(), which comes back in one D2H: its regions in this order, each at the next
    offset aligned for its dtype.  Per proposal slot (F*T of them, T = topk slots per candidate): boxes, score, best
    (compacted hypothesis index, -1: unused), count; per candidate: npts, nvalid; status (include/fnp.h: 8 int32);
    the recall counters; the stage-4 keep flags.  Then, for S settings of evaluate_settings: boxes, score, best, count
    per setting and candidate, the recall and the precision counters per setting, and n_quality quality counters per
    setting (quality.QualitySpec.n_counters)."""

    def __init__(self, F, T=1, S=0, n_quality=0):
        FT, NC, NP = F * T, SeekerEngine.N_COUNTERS, SeekerEngine.N_PRECISION
        self.regions, end = {}, 0            # name -> (byte offset, dtype, shape)
        for name, dt, shape in (
                ("boxes", _F32, (FT, 7)), ("score", _F32, (FT,)), ("best", _I32, (FT,)), ("count", _I32, (FT,)),
                ("npts", _I32, (F,)), ("nvalid", _I32, (F,)), ("status", _I32, (8,)), ("recall", _I64, (NC,)),
                ("keep", _U8, (FT,)), ("sel_boxes", _F32, (S, F, 7)), ("sel_score", _F32, (S, F)),
                ("sel_best", _I32, (S, F)), ("sel_count", _I32, (S, F)), ("sel_recall", _I64, (S, NC)),
                ("sel_precision", _I64, (S, NP)), ("quality", _I64, (S, n_quality))):
            off = _align(end, dt.itemsize)
            self.regions[name] = (off, dt, shape)
            end = off + dt.itemsize * math.prod(shape)
        self.nbytes = end

    def span(self, first, last=None):
        """Byte range of region `first`, or of the regions `first` through `last`."""
        off, dt, shape = self.regions[last or first]
        return slice(self.regions[first][0], off + dt.itemsize * math.prod(shape))

    def ptr(self, base, name, row=0):
        """Device address of region `name` (or of its row `row` along the first axis) in the block at `base`."""
        off, dt, shape = self.regions[name]
        return base + off + row * dt.itemsize * math.prod(shape[1:])

    def view(self, raw, name):
        """Region `name` of a host copy of the block (a uint8 array) as a shaped numpy array."""
        _, dt, shape = self.regions[name]
        return raw[self.span(name)].view(dt).reshape(shape)


class SeekerEngine:
    """Batched Box Seeker on one GPU."""

    def __init__(self, params=None, device=None, debug=False, split_points=None, score_mode="auto", box_format="xyxy",
                 host_cache=True, variant="nuscenes"):
        if not torch.cuda.is_available():
            raise RuntimeError("findnpropagate_b200.SeekerEngine needs a CUDA device (no CPU fallback)")
        assert variant in ("nuscenes", "kitti")
        self.variant = variant
        self.p = resolve_params(params, variant)
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.debug = debug
        self.M = max(int(self.p["num_mags"]), 1)
        self.J = int(self.p["num_rotations"]) * int(self.p["num_sizes"])
        self.H = self.M * self.J
        bb, bc = build_tables(self.p, ANCHORS_KITTI if variant == "kitti" else None)
        self.base_boxes_host, self.base_corners_host = bb, bc
        self.base_boxes = bb.to(self.device)
        self.base_corners = bc.to(self.device)
        mags = torch.linspace(0.0, 1.0, self.p["num_mags"]) if self.p["num_mags"] > 0 else torch.zeros(1)
        self.mags = mags.to(self.device)
        self.cfg = _lib.SeekerCfg(
            num_mags=self.M, num_yaw_size=self.J, n_classes=bb.shape[0], clamp_bottom=int(self.p["clamp_bottom"]),
            img_w=float(IMAGE_SIZE[1]), img_h=float(IMAGE_SIZE[0]), lq=float(self.p["lq"]), uq=float(self.p["uq"]),
            cq=float(self.p["cq"]), frustum_min=FRUSTUM_MIN, max_dist=float(self.p["max_dist"]),
            min_cam_iou=float(self.p["min_cam_iou"]), dns_w=float(self.p["dns_w"]), iou_w=float(self.p["iou_w"]),
            dst_w=float(self.p["dst_w"]), ego_w=float(self.p["ego_w"] or 0), occl_w=float(self.p["occl_w"] or 0),
            search_depth=float(self.p["search_depth"] or 0),
            flags=(_lib.SEEKER_MULT if self.p["MULT"] else 0) | (_lib.SEEKER_OCCL_MULT if self.p["OCCL_MULT"] else 0)
            | (_lib.SEEKER_MULTICAM_IOU if self.p["MULTICAM_IOU"] else 0),
            topk=int(self.p["topk"]), nms_normal=float(self.p["nms_normal"]),
            variant=_lib.VARIANT_KITTI if variant == "kitti" else _lib.VARIANT_NUSCENES)
        self.T = int(self.p["topk"])       # proposal slots per candidate frustum (NMS order), :1040-1046
        # workspaces of the optional score terms (include/fnp.h: hyp_dist, hyp_nfar)
        self.rand_center = bool(self.p.get("rand_center"))
        # the KITTI head always ranks distances; rand_center needs the weighted centre, which rides on the same workspace
        self.use_dist = self.cfg.dst_w != 0 or bool(self.p["MULT"]) or variant == "kitti" or self.rand_center
        self.use_occl = self.cfg.occl_w > 0 or bool(self.p["OCCL_MULT"])
        self.arena = _Arena(self.device)
        self.fixed_split_points = split_points
        # "auto" | "direct" | "sweep": which stage-2b kernel counts the points (same counts either way)
        self.score_mode = {"auto": _lib.SCORE_AUTO, "direct": _lib.SCORE_DIRECT, "sweep": _lib.SCORE_SWEEP}[score_mode]
        if self.rand_center:      # random centres are no line: the depth sweep would only take exact predicates
            self.score_mode = _lib.SCORE_DIRECT
        self.last_score_mode = None
        # MODEL.DENSE_HEAD.BOX_FORMAT (frustum_proposals_v1.py:252,597-601): 'xyxy', anything else means
        # x, y, w, h -- the 2D NMS runs on the raw numbers (as in the reference), the corner x+w, y+h is
        # formed afterwards in fp32
        self.box_format = box_format
        self.pts_factor = 2.0
        self.n_sms = torch.cuda.get_device_properties(self.device).multi_processor_count
        self.launches = 0          # kernels of ours launched (bench bookkeeping)
        self._cam_cache, self._tile_cache = {}, {}
        # host_cache=False: plan() recomputes the tile table and the camera matrices of every batch (a sweep
        # over distinct frames never hits these caches; bench.py measures that case)
        self.host_cache = bool(host_cache)
        self.host_s = dict(plan=0.0, execute=0.0, finish=0.0)   # host time spent per call kind (bench bookkeeping)

    # ------------------------------------------------------------------ host planning
    @classmethod
    def host_planner(cls, params=None, box_format="xyxy"):
        """The planning half only (plan / plan_flat / plan_arrays), without a device: for loaders that plan ahead
        of the GPU process, and for the CPU tests."""
        self = object.__new__(cls)
        self.p = resolve_params(params)
        self.T, self.box_format = int(self.p["topk"]), box_format
        self._cam_cache, self._tile_cache, self.host_cache = {}, {}, True
        self.host_s = dict(plan=0.0, execute=0.0, finish=0.0)
        return self

    def _cam_mats(self, frames):
        """(B,6,24) camera matrices; calibration repeats from frame to frame (it is fixed per
        scene), so the torch.inverse/matmul result is cached by the content of its inputs."""
        out = np.empty((len(frames), 6, 24), np.float32)
        miss = []
        keys = []
        for b, f in enumerate(frames):
            k = (np.asarray(f.lidar2image, np.float32).tobytes(), np.asarray(f.camera2lidar, np.float32).tobytes(),
                 np.asarray(f.camera_intrinsics, np.float32).tobytes())
            keys.append(k)
            m = self._cam_cache.get(k) if self.host_cache else None
            if m is None:
                miss.append(b)
            else:
                out[b] = m
        if miss:
            mm = camera_matrices(np.stack([frames[b].lidar2image for b in miss]),
                                 np.stack([frames[b].camera2lidar for b in miss]),
                                 np.stack([frames[b].camera_intrinsics for b in miss]))
            if len(self._cam_cache) > 4096:
                self._cam_cache.clear()
            for i, b in enumerate(miss):
                out[b] = mm[i]
                self._cam_cache[keys[b]] = mm[i].copy()
        return out

    def plan(self, frames: List[FrameInput], xyz_offset=0, stride=None):
        """Everything the host contributes to a batch, as numpy arrays.  stride / xyz_offset describe
        the DEVICE point table handed to execute() (default: the frames' own row layout; (3, 0) for
        a table gathered by HostPointFeeder).  One call into the C-ABI library (fnp_host_plan) over the
        frames' prepared records; the arrays are views of one block that execute() uploads as it is."""
        t0 = time.perf_counter()
        B = len(frames)
        if stride is None:
            stride = int(frames[0].points.shape[1]) if B else 5
        blob = b"".join([f.prepare()["blob"] for f in frames])
        sz = (C.c_int64 * 3)()
        _lib.check(_lib.lib.fnp_host_plan_sizes(blob, B, sz), "fnp_host_plan_sizes")
        D, n_tiles = int(sz[0]), int(sz[1])
        T = self.T
        spec = [("frame_row_start", np.int64, B + 1), ("tile_frame", np.int32, n_tiles), ("tile_row0", np.int32, n_tiles),
                ("frame_tile_start", np.int32, B + 1), ("cam_mats", np.float32, B * 144), ("frame_cand_start", np.int32, B + 1),
                ("cam_cand_start", np.int32, 6 * B + 1), ("cand_frame", np.int32, D), ("cand_cam", np.int32, D),
                ("cand_label", np.int32, D), ("cand_box2d", np.float32, 4 * D), ("nms_order", np.int32, D)]
        if T > 1:
            spec += [("frame_prop_start", np.int32, B + 1), ("prop_order", np.int32, D * T)]
        n_dev = len(spec)
        spec += [("cand_score", np.float32, D), ("cand_det", np.int32, D)]        # host-side bookkeeping, not uploaded
        offs, total, dev_bytes = {}, 0, 0
        for i, (k, dt, n) in enumerate(spec):
            offs[k] = total
            total = _align(total + np.dtype(dt).itemsize * max(n, 1))
            if i + 1 == n_dev:
                dev_bytes = total
        block = np.empty(total, np.uint8)
        base = block.ctypes.data
        out = _lib.HostPlanOut(**{k: base + offs[k] for k, _, _ in spec})
        _lib.check(_lib.lib.fnp_host_plan(blob, B, float(self.p["nms_2d"]), float(self.p["score_thr"]),
                                          int(self.box_format != "xyxy"), T, C.byref(out)), "fnp_host_plan")
        F = int(out.n_cands)

        def view(k, dt, n):
            return block[offs[k]:offs[k] + np.dtype(dt).itemsize * n].view(dt)
        plan = dict(B=B, F=F, n_tiles=int(out.n_tiles), stride=int(stride), xyz_offset=int(xyz_offset),
                    total_rows=int(out.total_rows), max_cands=int(out.max_cands_per_frame),
                    meta_block=block, meta_offs=offs, meta_dev_bytes=dev_bytes)
        for k, dt, n in spec:
            n_used = F if k.startswith("cand_") or k == "nms_order" else F * T if k == "prop_order" else n
            plan[k] = view(k, dt, n_used)
        plan["cand_box2d"] = view("cand_box2d", np.float32, 4 * F).reshape(F, 4)
        plan["cam_mats"] = plan["cam_mats"].reshape(B, 6, 24)
        self.host_s["plan"] += time.perf_counter() - t0
        return plan

    def plan_flat(self, frames: List[FrameInput], xyz_offset=0, stride=None):
        """The same plan from flat numpy arrays (plan_arrays): the path FrustumProposerOG.get_proposals takes with
        the detections of a collated batch_dict.  Kept equal to plan() by tests/test_host_cpu.py."""
        B = len(frames)
        n_rows = np.array([f.points.shape[0] for f in frames], dtype=np.int64)
        frame_row_start = np.zeros(B + 1, np.int64)
        np.cumsum(n_rows, out=frame_row_start[1:])
        if stride is None:
            stride = int(frames[0].points.shape[1]) if B else 5
        n_det = [len(f.det_scores) for f in frames]
        det_frame = np.repeat(np.arange(B, dtype=np.int64), n_det)
        if B:
            det_boxes = np.concatenate([np.asarray(f.det_boxes, np.float32).reshape(-1, 4) for f in frames])
            det_labels = np.concatenate([np.asarray(f.det_labels, np.int64) for f in frames])
            det_scores = np.concatenate([np.asarray(f.det_scores, np.float32) for f in frames])
            det_cam = np.concatenate([np.asarray(f.det_cam_idx, np.int64) for f in frames])
            cam_mats = self._cam_mats(frames)
        else:
            det_boxes, det_labels = np.zeros((0, 4), np.float32), np.zeros(0, np.int64)
            det_scores, det_cam = np.zeros(0, np.float32), np.zeros(0, np.int64)
            cam_mats = np.zeros((0, 6, 24), np.float32)
        return self.plan_arrays(frame_row_start, stride, xyz_offset, cam_mats, det_boxes, det_labels, det_scores,
                                det_frame, det_cam)

    def _tiles(self, frame_row_start):
        key = frame_row_start.tobytes()
        t = self._tile_cache.get(key) if self.host_cache else None
        if t is None:
            B = frame_row_start.shape[0] - 1
            n_rows = np.diff(frame_row_start)
            tiles_per_frame = (n_rows + _lib.CULL_TILE - 1) // _lib.CULL_TILE
            frame_tile_start = np.zeros(B + 1, np.int32)
            np.cumsum(tiles_per_frame, out=frame_tile_start[1:])
            n_tiles = int(frame_tile_start[-1])
            tile_frame = np.repeat(np.arange(B, dtype=np.int32), tiles_per_frame)
            tile_row0 = ((np.arange(n_tiles, dtype=np.int64)
                          - np.repeat(frame_tile_start[:-1].astype(np.int64), tiles_per_frame))
                         * _lib.CULL_TILE).astype(np.int32)
            if len(self._tile_cache) > 64:
                self._tile_cache.clear()
            t = self._tile_cache[key] = (n_tiles, tile_frame, tile_row0, frame_tile_start)
        return t

    def plan_arrays(self, frame_row_start, stride, xyz_offset, cam_mats, det_boxes, det_labels, det_scores,
                    det_frame, det_cam):
        B = frame_row_start.shape[0] - 1
        sel, frame_cand_start = nms2d.frustum_candidates(det_boxes, det_labels, det_scores, det_frame, det_cam,
                                                         self.p["nms_2d"], self.p["score_thr"], n_frames=B,
                                                         return_starts=True)
        F = int(sel.shape[0])
        cand_frame = det_frame[sel].astype(np.int32)
        cand_cam = det_cam[sel].astype(np.int32)
        # first candidate of every (frame, camera rank): candidates are already in that order
        cam_cand_start = np.zeros(B * 6 + 1, np.int32)
        if F:
            np.cumsum(np.bincount(cand_frame.astype(np.int64) * 6 + nms2d.CAM_RANK[cand_cam], minlength=B * 6),
                      out=cam_cand_start[1:])
        n_tiles, tile_frame, tile_row0, frame_tile_start = self._tiles(np.ascontiguousarray(frame_row_start, np.int64))
        cand_score = np.ascontiguousarray(det_scores[sel], np.float32)
        # stage-4 priority order inside each frame: descending 2D score, stable (= np.lexsort((index,
        # -score, frame)); in C: the lexsort was 1.1 of plan's 3.9 ms per 256 frames)
        nms_order = np.empty(max(F, 1), np.int32)[:F]
        fcs32 = np.ascontiguousarray(frame_cand_start, np.int32)
        _lib.check(_lib.lib.fnp_host_nms_order(cand_score.ctypes.data, fcs32.ctypes.data, B, nms_order.ctypes.data),
                   "fnp_host_nms_order")
        extra = {}
        if self.T > 1:
            # topk > 1: every candidate owns T consecutive proposal slots; per-frame slot ranges and the
            # stage-4 order over slots (a candidate's slots stay together, best first)
            T = self.T
            extra = dict(frame_prop_start=(fcs32 * T).astype(np.int32),
                         prop_order=(nms_order[:, None] * T + np.arange(T, dtype=np.int32)[None, :]).reshape(-1).astype(np.int32))
        return dict(
            **extra,
            B=B, F=F, n_tiles=n_tiles, stride=int(stride), xyz_offset=int(xyz_offset),
            total_rows=int(frame_row_start[-1]),
            max_cands=int(np.diff(frame_cand_start).max()) if B else 0,
            frame_row_start=frame_row_start.astype(np.int64), tile_frame=tile_frame, tile_row0=tile_row0,
            frame_tile_start=frame_tile_start, cam_mats=np.ascontiguousarray(cam_mats, np.float32),
            frame_cand_start=frame_cand_start, cam_cand_start=cam_cand_start, cand_frame=cand_frame,
            cand_cam=cand_cam, cand_label=det_labels[sel].astype(np.int32),
            cand_box2d=self._cand_boxes(det_boxes[sel]),
            cand_score=cand_score, cand_det=sel, nms_order=nms_order)

    def _cand_boxes(self, boxes):
        b = np.ascontiguousarray(boxes, np.float32).reshape(-1, 4)
        if self.box_format != "xyxy":
            b = b.copy()
            b[:, 2:] += b[:, 0:2]
        return b

    # ------------------------------------------------------------------ device execution
    _META = ["frame_row_start", "tile_frame", "tile_row0", "frame_tile_start", "cam_mats", "frame_cand_start",
             "cam_cand_start", "cand_frame", "cand_cam", "cand_label", "cand_box2d", "nms_order"]

    def _upload_meta(self, plan, stream, slot=0):
        if "meta_block" in plan:       # plan(): the arrays already lie in one block with these offsets
            total = int(plan["meta_dev_bytes"])
            host = self.arena.get("meta_host%d" % slot, total, pinned=True)
            host.numpy()[:total] = plan["meta_block"][:total]
            dev = self.arena.get("meta_dev%d" % slot, total)
            _lib.check(_lib.lib.fnp_upload_from_pinned(dev.data_ptr(), host.data_ptr(), total, stream),
                       "fnp_upload_from_pinned")
            self.launches += 1
            base = dev.data_ptr()
            return {k: base + o for k, o in plan["meta_offs"].items()}
        offs, total = {}, 0
        keys = self._META + (["frame_prop_start", "prop_order"] if self.T > 1 else [])
        for k in keys:
            offs[k] = total
            total = _align(total + plan[k].nbytes)
        host = self.arena.get("meta_host%d" % slot, total, pinned=True)
        hv = host.numpy()
        for k in keys:
            a = plan[k]
            hv[offs[k]:offs[k] + a.nbytes] = a.reshape(-1).view(np.uint8)
        dev = self.arena.get("meta_dev%d" % slot, total)
        # by a kernel reading the pinned block, not by the copy engine: an H2D memcpy here can be
        # served after the NEXT step's 200 MB point copy and stall this step's kernels behind it
        _lib.check(_lib.lib.fnp_upload_from_pinned(dev.data_ptr(), host.data_ptr(), total, stream),
                   "fnp_upload_from_pinned")
        self.launches += 1
        base = dev.data_ptr()
        return {k: base + o for k, o in offs.items()}

    def execute(self, plan, points_dev, nms_thresh=None, gt=None, recall_thresh=(0.3, 0.5, 0.7), slot=0,
                points_ready=None, settings=None, quality=None):
        """Enqueue the whole batch on the current stream.  points_dev: CUDA float32 tensor
        holding the rows of all frames back to back.  points_ready: optional CUDA event the
        kernels must wait for (the H2D copy of the points on another stream); the small
        metadata upload is issued *before* that wait so that it does not queue behind the
        next step's point copy in the H2D engine.  settings, quality: see evaluate_settings.  Returns a
        handle for `finish`."""
        t0 = time.perf_counter()
        _lib.require_cuda(points_dev)
        assert points_dev.dtype == torch.float32 and points_dev.is_contiguous()
        F, B, H, M = plan["F"], plan["B"], self.H, self.M
        S = len(settings) if settings is not None else 0
        if S:
            sel = [select_setting(dict(self.p, **s)) for s in settings]     # left-out keys: this engine's values
            # the workspaces any setting reads, whether or not this engine's own score reads them
            use_dist = self.use_dist or any(s.dst_w != 0 or s.flags & _lib.SEEKER_MULT for s in sel)
            use_occl = self.use_occl or any(s.occl_w > 0 or s.flags & _lib.SEEKER_OCCL_MULT for s in sel)
        else:
            use_dist, use_occl = self.use_dist, self.use_occl
        dev = self.device
        with torch.cuda.device(dev):
            stream = _lib.current_stream(dev)
            meta = self._upload_meta(plan, stream, slot)
            if points_ready is not None:
                torch.cuda.current_stream(dev).wait_event(points_ready)
            chunks = -(-H // 512)      # hypothesis chunks per frustum (csrc: score_chunks)
            PG = _lib.PAGE_POINTS
            # page pool: pts_factor x the batch's rows, plus the half-empty last page of every frustum
            cap = (int(max(plan["total_rows"] * self.pts_factor, 4096)) + PG * (F + 1) + PG - 1) // PG * PG
            max_rows = int(np.diff(plan["frame_row_start"]).max()) if B else 0
            tab_stride = (max_rows + PG - 1) // PG + 1
            planes = 5 if self.debug else 4
            if self.fixed_split_points is not None:
                sp = max(PG, (int(self.fixed_split_points) + PG - 1) // PG * PG)      # splits are whole pages
            else:
                # point splits small enough to balance the persistent CTAs (measured on cfg2, 32 frames,
                # direct kernel: 2048 -> 0.737 ms, 512 -> 0.666 ms, 256 -> 0.663 ms), large enough to amortise
                # an item; the sweep kernel stages a whole split in shared memory: 256 cfg2 frames per step, whole
                # step / score stage alone: 512 -> 4.02 / 1.83 ms, 1024 -> 3.80 / 1.64, 1536 -> 3.73 / 1.60,
                # 2048 -> 3.69 / 1.62 (profiles/r02s_ab_sweep_split_and_queue.txt; round 1's kernel was best at 1024)
                sp = plan["total_rows"] // (self.n_sms * 128)
                sp = int(min(2048, max(256, 1 << max(sp, 1).bit_length() - 1)))
            max_items = (cap // sp + F + 1) * chunks
            Cmax = max(plan["max_cands"], 1)
            W = _lib.lib.fnp_seeker_mask_words(Cmax)
            if W < 0:
                raise ValueError("more than 1024 candidate frustums in one frame (%d) are not supported" % Cmax)
            if self.variant == "kitti" and W > 4:
                raise ValueError("the KITTI variant takes up to 128 candidate frustums per frame (%d)" % Cmax)
            sizes = dict(
                page_tab=4 * max(F, 1) * tab_stride, cell_masks=_lib.lib.fnp_seeker_cell_mask_bytes(C.byref(self.cfg), B, Cmax),
                frustum_pts=4 * planes * cap,
                cand_stats=4 * _lib.STATS_FLOATS * F, centres=12 * M * F, hyp_prep=32 * H * F, hyp_index=4 * H * F,
                hyp_iou=4 * H * F, counts=4 * H * F, items=16 * max_items,
                cand_item_start=4 * (F + 1), sweep_cols=4 * _lib.SWEEP_COL_FLOATS * self.J * F,
                )
            if self.T > 1:
                sizes["hyp_score"] = 4 * H * F
            if use_dist:
                sizes["hyp_dist"] = 4 * H * F
            if use_occl:
                sizes["hyp_nfar"] = 4 * H * F
            if self.debug:
                sizes.update(hyp_boxes_dbg=28 * H * F, hyp_iou_dbg=4 * H * F, hyp_valid_dbg=H * F)
            # every slot owns its intermediates, so that batches of different slots may be in flight on
            # different streams at the same time (slot 0 keeps the plain names: debug_views reads them)
            sfx = "" if slot == 0 else "@%d" % slot
            ptr = {k: self.arena.get(k + sfx, v).data_ptr() for k, v in sizes.items()}
            lay = OutLayout(F, self.T, S, quality.n_counters if quality is not None else 0)
            out_dev = self.arena.get("out%d" % slot, lay.nbytes)
            ob = out_dev.data_ptr()
            b = _lib.SeekerBatch(
                n_frames=B, n_cands=F, n_tiles=plan["n_tiles"], max_cands_per_frame=Cmax,
                points=points_dev.data_ptr(), point_stride=plan["stride"], xyz_offset=plan["xyz_offset"],
                frame_row_start=meta["frame_row_start"], tile_frame=meta["tile_frame"], tile_row0=meta["tile_row0"],
                frame_tile_start=meta["frame_tile_start"], cam_mats=meta["cam_mats"],
                frame_cand_start=meta["frame_cand_start"], cam_cand_start=meta["cam_cand_start"],
                cand_frame=meta["cand_frame"], cand_cam=meta["cand_cam"],
                cand_label=meta["cand_label"], cand_box2d=meta["cand_box2d"],
                base_boxes=self.base_boxes.data_ptr(), base_corners=self.base_corners.data_ptr(),
                mags=self.mags.data_ptr(),
                cell_masks=ptr["cell_masks"], mask_words=W, cand_npts=lay.ptr(ob, "npts"), page_tab=ptr["page_tab"],
                page_tab_stride=tab_stride, page_planes=planes, frustum_pts=ptr["frustum_pts"], pts_capacity=cap,
                cand_stats=ptr["cand_stats"], centres=ptr["centres"], hyp_prep=ptr["hyp_prep"],
                hyp_index=ptr["hyp_index"], hyp_iou=ptr["hyp_iou"], hyp_nvalid=lay.ptr(ob, "nvalid"),
                hyp_boxes_dbg=ptr.get("hyp_boxes_dbg"), hyp_iou_dbg=ptr.get("hyp_iou_dbg"),
                hyp_valid_dbg=ptr.get("hyp_valid_dbg"),
                split_points=sp, max_items=max_items,
                cand_item_start=ptr["cand_item_start"], items=ptr["items"],
                counts=ptr["counts"], score_mode=self.score_mode, sweep_cols=ptr["sweep_cols"],
                out_boxes=lay.ptr(ob, "boxes"), out_score=lay.ptr(ob, "score"), out_best=lay.ptr(ob, "best"),
                out_count=lay.ptr(ob, "count"), status=lay.ptr(ob, "status"),
                hyp_dist=ptr.get("hyp_dist"), hyp_nfar=ptr.get("hyp_nfar"), hyp_score=ptr.get("hyp_score"))
            if self.rand_center and F and plan["n_tiles"]:
                self._run_rand_center(b, stream, F, M, out_dev[lay.span("npts")].view(torch.int32),
                                      self.arena.bufs["cand_stats" + sfx], self.arena.bufs["centres" + sfx])
            else:
                rc = _lib.lib.fnp_seeker_run(C.byref(self.cfg), C.byref(b), stream)
                _lib.check(rc, "fnp_seeker_run")
            mode = _lib.lib.fnp_seeker_score_mode(C.byref(self.cfg), C.byref(b))
            self.last_score_mode = {_lib.SCORE_DIRECT: "direct", _lib.SCORE_SWEEP: "sweep"}.get(mode)
            self.launches += (9 + (mode == _lib.SCORE_SWEEP) + self.use_occl) if F and plan["n_tiles"] else 0
            handle = dict(plan=plan, batch=b, sp=sp, cap=cap, out_dev=out_dev, layout=lay, meta=meta,
                          tab_stride=tab_stride, planes=planes, has_nms=False, has_recall=False,
                          recall_thresh=tuple(recall_thresh), n_settings=S, quality=None,
                          args=dict(plan=plan, points_dev=points_dev, nms_thresh=nms_thresh, gt=gt,
                                    recall_thresh=recall_thresh, slot=slot, points_ready=points_ready,
                                    settings=settings, quality=quality))
            if S and F:
                self._select_multi(handle, b, sel, use_occl, gt, recall_thresh, stream)
                if quality is not None and gt is not None:
                    self._quality(handle, gt, quality, stream)
                    handle["quality"] = quality
            if nms_thresh is not None and F:
                self._stage4_nms(handle, float(nms_thresh), stream)
                handle["has_nms"] = True
            if gt is not None and F:
                self._recall(handle, gt, recall_thresh, stream)
                handle["has_recall"] = True
            host = self.arena.get("out_host%d" % slot, lay.nbytes, pinned=True)
            host[:lay.nbytes].copy_(out_dev[:lay.nbytes], non_blocking=True)
            handle["out_host"] = host
            handle["event"] = torch.cuda.Event()
            handle["event"].record()
        self.host_s["execute"] += time.perf_counter() - t0
        return handle

    N_COUNTERS = 5 + 5 * 3          # generate_recall_record counters for 3 IoU thresholds

    def _stage4_nms(self, handle, thresh, stream):
        """Rotated-BEV NMS of each frame's proposals in 2D-score order (the dedup
        PseudoLoader applies later on the CPU, pseudo_loader.py:29-55,755)."""
        plan, meta, lay, ob, T = handle["plan"], handle["meta"], handle["layout"], handle["out_dev"].data_ptr(), self.T
        if plan["max_cands"] * T > _lib.SEG_NMS_MAX:
            raise ValueError("stage-4 NMS handles at most %d proposals per frame" % _lib.SEG_NMS_MAX)
        rc = _lib.lib.fnp_seg_nms_rotated(lay.ptr(ob, "boxes"), None, meta["nms_order" if T == 1 else "prop_order"],
                                          lay.ptr(ob, "best"),
                                          meta["frame_cand_start" if T == 1 else "frame_prop_start"], plan["B"],
                                          int(min(max(plan["max_cands"] * T, 1), _lib.SEG_NMS_MAX)), thresh,
                                          lay.ptr(ob, "keep"), stream)
        _lib.check(rc, "fnp_seg_nms_rotated")
        self.launches += 1

    def _recall(self, handle, gt, thresh, stream):
        plan, meta, lay, out_dev = handle["plan"], handle["meta"], handle["layout"], handle["out_dev"]
        ob = out_dev.data_ptr()
        gt_boxes, gt_start, max_gt = gt
        assert len(thresh) == 3
        out_dev[lay.span("recall")].zero_()
        th = (C.c_float * len(thresh))(*[float(t) for t in thresh])
        rc = _lib.lib.fnp_recall_counters(lay.ptr(ob, "boxes"), lay.ptr(ob, "best"),
                                          meta["frame_cand_start" if self.T == 1 else "frame_prop_start"],
                                          gt_boxes.data_ptr(), gt_start.data_ptr(), plan["B"],
                                          max(plan["max_cands"] * self.T, 1), int(max_gt), th, len(thresh),
                                          lay.ptr(ob, "recall"), stream)
        _lib.check(rc, "fnp_recall_counters")
        self.launches += 1

    N_PRECISION = 1 + 3             # valid proposals, then hits at 3 IoU thresholds (fnp_precision_counters)

    def _select_multi(self, handle, b, sel, use_occl, gt, thresh, stream):
        """Stage 3 once per setting over this execution's stages 1-2c, then each setting's recall and precision."""
        plan, meta, lay, out_dev = handle["plan"], handle["meta"], handle["layout"], handle["out_dev"]
        L, ob, S = _lib.lib, out_dev.data_ptr(), len(sel)
        if use_occl and not self.use_occl:      # this engine's own cfg leaves stage 2c off
            cfg = _lib.SeekerCfg.from_buffer_copy(self.cfg)
            cfg.flags |= _lib.SEEKER_OCCL_MULT
            _lib.check(L.fnp_seeker_occlusion(C.byref(cfg), C.byref(b), stream), "fnp_seeker_occlusion")
            self.launches += 1
        # one launch per FNP_SELECT_MAX_SETTINGS settings (the kernel-parameter block), all over the same stages 1-2c
        for c0 in range(0, S, _lib.SELECT_MAX_SETTINGS):
            n = min(_lib.SELECT_MAX_SETTINGS, S - c0)
            chunk = (_lib.SelectSetting * n)(*sel[c0:c0 + n])
            rows = [lay.ptr(ob, k, c0) for k in ("sel_boxes", "sel_score", "sel_best", "sel_count")]
            _lib.check(L.fnp_seeker_select_multi(C.byref(self.cfg), C.byref(b), chunk, n, *rows, stream),
                       "fnp_seeker_select_multi")
            self.launches += 1
        if gt is None:
            return
        gt_boxes, gt_start, max_gt = gt
        out_dev[lay.span("sel_recall", "sel_precision")].zero_()
        th = (C.c_float * len(thresh))(*[float(t) for t in thresh])
        for s in range(S):
            for fn, counters in ((L.fnp_recall_counters, "sel_recall"), (L.fnp_precision_counters, "sel_precision")):
                rc = fn(lay.ptr(ob, "sel_boxes", s), lay.ptr(ob, "sel_best", s), meta["frame_cand_start"],
                        gt_boxes.data_ptr(), gt_start.data_ptr(), plan["B"], max(plan["max_cands"], 1), int(max_gt), th,
                        len(thresh), lay.ptr(ob, counters, s), stream)
                _lib.check(rc, fn.__name__)
        self.launches += 2 * S

    def _quality(self, handle, gt, spec, stream):
        """One fnp_quality_counters launch over every setting's proposals (the boxes and flags _select_multi wrote);
        labels are the candidates' 2D labels, shared by the settings."""
        from . import quality
        plan, meta, lay, out_dev = handle["plan"], handle["meta"], handle["layout"], handle["out_dev"]
        ob, F = out_dev.data_ptr(), plan["F"]
        gt_boxes, gt_start, max_gt = gt
        out_dev[lay.span("quality")].zero_()
        quality.launch(spec, lay.ptr(ob, "sel_boxes"), meta["cand_label"], meta["frame_cand_start"], gt_boxes, gt_start,
                       plan["B"], max(plan["max_cands"], 1), int(max_gt), lay.ptr(ob, "quality"),
                       n_settings=handle["n_settings"], pred_valid=lay.ptr(ob, "sel_best"), pred_stride=F,
                       valid_stride=F, stream=stream)
        self.launches += 1

    def evaluate_settings(self, plan, points_dev, gt, settings, recall_thresh=(0.3, 0.5, 0.7), quality=None):
        """Scores several select-level settings on one batch: stages 1-2c run once with this engine's parameters, then
        stage 3 once per setting (fnp_seeker_select_multi), and its recall and precision counters.  settings: dicts of
        SELECT_KEYS (a key a setting leaves out takes this engine's value), any number of them: stage 3 runs for up to
        256 settings per launch; each min_cam_iou must be at least this engine's, whose compaction every setting
        filters further -- for the KITTI variant each must equal this engine's, and a setting holds SELECT_KEYS_KITTI
        (first-match counts depend on the valid set).  plan / points_dev / gt as for execute (gt from
        upload_gt).  Returns finish()'s dict, whose "settings" holds per setting: proposals, recall (recall_dict),
        precision (proposals, then "hits_<t>": proposals with a GT IoU3D > t), and per candidate cand_best (index among
        the compacted hypotheses, -1: none), cand_score2, cand_count, cand_boxes.  quality (a quality.QualitySpec): one
        more launch, fnp_quality_counters over every setting, and each setting gains "quality", its flat counters
        (quality.tables reads them).  One D2H; on a page-pool overflow the pool grows and the batch runs again."""
        if self.T != 1 or self.rand_center:
            raise NotImplementedError("evaluate_settings runs with topk = 1 and no rand_center")
        if not settings:
            raise ValueError("evaluate_settings needs at least one setting")
        for s in settings:
            iou = np.float32(s.get("min_cam_iou", self.p["min_cam_iou"]))
            if iou < np.float32(self.p["min_cam_iou"]):
                raise ValueError("setting %r: min_cam_iou below the engine's %s" % (s, self.p["min_cam_iou"]))
            if self.variant == "kitti" and iou != np.float32(self.p["min_cam_iou"]):
                raise ValueError("setting %r: the KITTI head's min_cam_iou must be the engine's %s (its first-match "
                                 "counts depend on the valid set)" % (s, self.p["min_cam_iou"]))
        if quality is not None:
            from .quality import check_labels
            check_labels(quality, plan["cand_label"], gt[0].cpu().numpy(), gt[1].cpu().numpy())
            quality.check_size(plan["max_cands"], gt[2], "the largest frame of the batch")
        return self.result(self.execute(plan, points_dev, gt=gt, recall_thresh=recall_thresh, settings=settings,
                                         quality=quality))

    def result(self, handle):
        """finish(handle), recovering from a page pool too small for the batch: the pool grows (pts_factor) and the
        batch runs again with execute()'s original arguments until it fits.  The handle is updated in place, so that
        afterwards it describes the run whose results are returned."""
        while True:
            try:
                return self.finish(handle)
            except OverflowError as e:
                need = int(e.args[0])
                self.pts_factor = max(self.pts_factor * 1.5, 1.25 * need / max(handle["plan"]["total_rows"], 1))
                handle.update(self.execute(**handle["args"]))

    def finish(self, handle):
        """Wait for the batch and assemble per-frame results (reference output format)."""
        handle["event"].synchronize()
        t0 = time.perf_counter()
        plan = handle["plan"]
        F, B = plan["F"], plan["B"]
        raw, lay, T = handle["out_host"].numpy(), handle["layout"], self.T
        boxes, score, best, count, npts, nvalid, status = (lay.view(raw, k) for k in (
            "boxes", "score", "best", "count", "npts", "nvalid", "status"))
        if status[0] & 1:
            raise OverflowError(int(status[1]))
        if status[0] & 2:
            raise RuntimeError("scoring work-item table overflowed (%d items)" % status[2])
        ok = best >= 0
        fcs = plan["frame_cand_start"]
        # compact once, then hand every frame a slice (views of the compacted arrays: no per-frame
        # boolean indexing -- 128 frames: 1.4 ms -> 0.4 ms of host time per batch)
        idx = np.flatnonzero(ok)
        cand_of = idx if T == 1 else idx // T      # slot -> candidate: 2D score and label repeat (:1048-1052)
        c_boxes, c_scores = boxes[idx], plan["cand_score"][cand_of]
        c_labels = plan["cand_label"][cand_of].astype(np.int32)
        c_keep = lay.view(raw, "keep")[idx].astype(bool) if handle["has_nms"] else None
        frames = _FrameResults(c_boxes, c_scores, c_labels, c_keep, np.searchsorted(idx, fcs * T))
        # per-candidate views: the best proposal of each (slot 0); cand_topk has every slot
        res = dict(frames=frames, cand_valid=ok[::T].copy(), cand_best=best[::T].copy(), cand_score2=score[::T].copy(),
                   cand_count=count[::T].copy(), cand_npts=npts.copy(), cand_nvalid=nvalid.copy(),
                   cand_boxes=boxes[::T].copy())
        if T > 1:
            res["cand_topk"] = dict(best=best.reshape(F, T).copy(), score2=score.reshape(F, T).copy(),
                                    boxes=boxes.reshape(F, T, 7).copy(), count=count.reshape(F, T).copy())
        if handle["has_recall"]:
            res["recall"] = self.recall_dict(lay.view(raw, "recall"), handle["recall_thresh"])
        S = handle["n_settings"]
        if S:
            sb, ss, sbest, scount, rec, prec, qc = (lay.view(raw, k) for k in (
                "sel_boxes", "sel_score", "sel_best", "sel_count", "sel_recall", "sel_precision", "quality"))
            th = handle["recall_thresh"]
            spec = handle.get("quality")
            res["settings"] = []
            for s in range(S):
                d = dict(proposals=int((sbest[s] >= 0).sum()), cand_best=sbest[s].copy(), cand_score2=ss[s].copy(),
                         cand_count=scount[s].copy(), cand_boxes=sb[s].copy())
                if handle["has_recall"]:
                    d["recall"] = self.recall_dict(rec[s], th)
                    d["precision"] = dict(proposals=int(prec[s, 0]),
                                          **{"hits_%s" % t: int(prec[s, 1 + i]) for i, t in enumerate(th)})
                if spec is not None:
                    d["quality"] = qc[s].copy()
                res["settings"].append(d)
        self.host_s["finish"] += time.perf_counter() - t0
        return res

    @staticmethod
    def recall_dict(counters, thresh=(0.3, 0.5, 0.7)):
        d = {k: int(counters[i]) for i, k in enumerate(RECALL_KEYS)}
        for t, th in enumerate(thresh):
            for j, k in enumerate(RECALL_PER_THRESH):
                d["%s_%s" % (k, th)] = int(counters[5 + 5 * t + j])
        return d

    def _run_rand_center(self, b, stream, F, M, npts_dev, stats_buf, centres_buf):
        """The stages one by one, with the reference's random centres put in between (rand_center): after stage 1b the
        population and the weighted centre of every frustum are known; the host then draws torch.randn((M, 3)) per
        frustum WITH points, in frustum order, exactly as frustum_proposals_v1.py:844-847 does, and overwrites the
        centre line.  One device round trip per batch: an option for experiments, not for throughput."""
        L, cfg = _lib.lib, C.byref(self.cfg)
        _lib.check(L.fnp_seeker_cull(cfg, C.byref(b), stream), "fnp_seeker_cull")
        _lib.check(L.fnp_seeker_frustum_stats(cfg, C.byref(b), stream), "fnp_seeker_frustum_stats")

        npts = npts_dev.cpu().numpy()                                                   # synchronises
        stats = stats_buf[:4 * F * _lib.STATS_FLOATS].view(torch.float32).view(F, _lib.STATS_FLOATS)
        centres = centres_buf[:12 * F * M].view(torch.float32).view(F, M, 3)
        for f in np.flatnonzero(npts > 0):
            centres[f] = stats[f, 10:13].reshape(1, 3) + torch.randn((M, 3), dtype=torch.float32, device=self.device)
        for name in ("fnp_seeker_hypotheses", "fnp_seeker_score", "fnp_seeker_occlusion", "fnp_seeker_select"):
            _lib.check(getattr(L, name)(cfg, C.byref(b), stream), name)

    def run(self, frames: List[FrameInput], points_dev=None, nms_thresh=None, with_recall=False, xyz_offset=0):
        """Plan + H2D + execute + finish for a list of frames; grows the frustum-point
        buffer and retries on overflow."""
        plan = self.plan(frames, xyz_offset=xyz_offset)
        if points_dev is None:
            points_dev = self.upload_points(frames)
        gt = self.upload_gt(frames) if with_recall else None
        return self.result(self.execute(plan, points_dev, nms_thresh=nms_thresh, gt=gt))

    def upload_points(self, frames):
        rows = sum(f.points.shape[0] for f in frames)
        stride = frames[0].points.shape[1] if frames else 5
        buf = self.arena.get("points", 4 * rows * stride)
        pts = buf[:4 * rows * stride].view(torch.float32).view(rows, stride)
        r = 0
        for f in frames:
            n = f.points.shape[0]
            src = f.points if isinstance(f.points, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(f.points, np.float32))
            pts[r:r + n].copy_(src, non_blocking=True)
            r += n
        return pts

    def upload_gt(self, frames):
        g, start = [], [0]
        for f in frames:
            gb = np.zeros((0, 8), np.float32) if f.gt_boxes is None else np.asarray(f.gt_boxes, np.float32)
            if gb.shape[0]:
                gb = np.concatenate([gb[:, :7], gb[:, -1:]], 1)
            g.append(gb.reshape(-1, 8))
            start.append(start[-1] + gb.shape[0])
        gt = torch.from_numpy(np.ascontiguousarray(np.concatenate(g) if g else np.zeros((0, 8), np.float32)))
        max_gt = int(np.diff(start).max()) if len(start) > 1 else 0
        return gt.to(self.device), torch.tensor(start, dtype=torch.int32).to(self.device), max_gt

    # ------------------------------------------------------------------ debug views
    def debug_views(self, handle):
        """Intermediate tensors of the last batch (only with debug=True): per candidate the
        frustum points, source rows, stats, centres, hypothesis boxes / iou / valid, counts."""
        assert self.debug
        torch.cuda.synchronize(self.device)
        plan, F, H, M = handle["plan"], handle["plan"]["F"], self.H, self.M

        def view(name, dtype, shape):
            n = int(np.prod(shape)) * torch.tensor([], dtype=dtype).element_size()
            return self.arena.bufs[name][:n].view(dtype).view(*shape).cpu().numpy()
        # the page pool -> one (x, y, z, d) row per point, frustum by frustum, sorted by source row (stage 1 fills
        # a frustum in whatever order the tiles reach it; no result depends on that order, this view fixes one)
        PG, planes, ts = _lib.PAGE_POINTS, handle["planes"], handle["tab_stride"]
        npts = handle["layout"].view(handle["out_host"].numpy(), "npts")
        tab = view("page_tab", torch.int32, (F, ts))
        n_pages = int(tab.max()) if F else 0
        pool = view("frustum_pts", torch.float32, (max(n_pages, 1), planes, PG))
        rows_l, idx_l = [], []
        for f in range(F):
            n = int(npts[f])
            k = (n + PG - 1) // PG
            pg = pool[tab[f, :k] - 1]                                   # (k, planes, PG)
            xyzd = pg[:, :4].transpose(0, 2, 1).reshape(-1, 4)[:n]
            src = pg[:, 4].reshape(-1)[:n].view(np.int32)
            o = np.argsort(src, kind="stable")
            rows_l.append(xyzd[o])
            idx_l.append(src[o])
        rows = np.concatenate(rows_l + [np.zeros((0, 4), np.float32)])
        idx = np.concatenate(idx_l + [np.zeros(0, np.int32)])
        pt_start = np.concatenate([[0], np.cumsum(npts)]).astype(np.int32)
        extra = {}
        if self.use_dist:
            extra["hyp_dist"] = view("hyp_dist", torch.float32, (F, H))
        if self.use_occl:
            extra["hyp_nfar"] = view("hyp_nfar", torch.int32, (F, H))
        return dict(
            **extra,
            pt_start=pt_start,
            frustum_pts=np.ascontiguousarray(rows),
            frustum_idx=np.ascontiguousarray(idx),
            stats=view("cand_stats", torch.float32, (F, _lib.STATS_FLOATS)),
            centres=view("centres", torch.float32, (F, M, 3)),
            hyp_boxes=view("hyp_boxes_dbg", torch.float32, (F, H, 7)),
            hyp_iou=view("hyp_iou_dbg", torch.float32, (F, H)),
            hyp_valid=view("hyp_valid_dbg", torch.uint8, (F, H)).astype(bool),
            hyp_index=view("hyp_index", torch.int32, (F, H)),
            hyp_prep=view("hyp_prep", torch.float32, (F, H, 8)),
            counts=view("counts", torch.int32, (F, H)),
        )


class HostPointFeeder:
    """Host buffers -> device point table for SeekerEngine.execute, double buffered.

    The reference uploads every column of the point table (pcdet/models/__init__.py:23-36) although
    the seeker reads xyz only.  submit() starts a threaded gather of x, y, z into a pinned staging
    slot on the host (fnp_host_pack_xyz_begin: returns at once, the workers do not hold the GIL);
    upload() waits for it and enqueues the H2D copy of the 12 B/point table on the copy stream.
    Slots alternate, so the gather of batch k+1 runs while batch k crosses PCIe and batch k-1 is in
    the kernels.  With pack=False the rows are uploaded as they are (all columns)."""

    def __init__(self, engine: "SeekerEngine", pack=True, n_threads=None, slots=2):
        import os
        self.eng, self.pack, self.slots = engine, bool(pack), int(slots)
        self.n_threads = int(n_threads) if n_threads else max(1, min(16, len(os.sched_getaffinity(0)) - 1))
        self.copy_stream = torch.cuda.Stream(device=engine.device)
        self.ready = [torch.cuda.Event() for _ in range(self.slots)]       # H2D of the slot complete
        self.consumed = [torch.cuda.Event() for _ in range(self.slots)]    # kernels done with the slot
        for e in self.consumed:
            e.record()
        self.ticket = [None] * self.slots
        self.host = [None] * self.slots
        self.dev = [None] * self.slots
        self.src = [None] * self.slots
        self.rows, self.width = [0] * self.slots, [0] * self.slots
        self.copied = [torch.cuda.Event() for _ in range(self.slots)]      # staging slot read by the DMA
        self.copied_valid = [False] * self.slots

    @property
    def layout(self):
        """(stride, xyz_offset) of the device table, for SeekerEngine.plan."""
        return (3, 0) if self.pack else (None, None)

    def close(self):
        """Waits for every gather still in flight and releases its ticket (the C side has 16 of them and
        its worker threads write into this object's pinned slots).  Safe to call more than once."""
        for slot, t in enumerate(self.ticket):
            if t is not None:
                try:
                    _lib.lib.fnp_host_pack_wait(t)
                finally:
                    self.ticket[slot] = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
        return False

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def submit(self, slot, points_host, xyz_offset=0):
        """Starts the gather of one batch into staging slot `slot`.  points_host: one (rows, C)
        float32 CPU tensor, or a list of per-frame (n_i, C) float32 arrays / tensors as a data loader
        leaves them (gathered back to back: no concatenated copy of the full-width rows is made).
        With pack=False a list is concatenated into a pinned slot instead (one full-width copy)."""
        segs = points_host if isinstance(points_host, (list, tuple)) else [points_host]
        segs = [torch.from_numpy(np.ascontiguousarray(p, np.float32)) if isinstance(p, np.ndarray) else p for p in segs]
        for p in segs:
            assert p.dtype == torch.float32 and p.is_contiguous() and not p.is_cuda and p.dim() == 2
        C_ = int(segs[0].shape[1])
        assert all(int(p.shape[1]) == C_ for p in segs)
        rows = int(sum(int(p.shape[0]) for p in segs))
        self.rows[slot], self.width[slot] = rows, C_
        if self.copied_valid[slot]:
            self.copied[slot].synchronize()          # the DMA has read the previous contents of the slot
        if not self.pack:
            if len(segs) == 1:
                self.src[slot] = segs[0]
                return
            nbytes = rows * C_ * 4
            if self.host[slot] is None or self.host[slot].numel() < nbytes:
                self.host[slot] = torch.empty(int(nbytes * 1.25) + 256, dtype=torch.uint8, pin_memory=True)
            dst = self.host[slot][:nbytes].view(torch.float32).view(rows, C_)
            r = 0
            for p in segs:
                dst[r:r + p.shape[0]] = p
                r += int(p.shape[0])
            self.src[slot] = dst
            return
        if self.ticket[slot] is not None:            # a gather submitted to this slot and never uploaded
            _lib.lib.fnp_host_pack_wait(self.ticket[slot])
            self.ticket[slot] = None
        self.src[slot] = segs                        # keep the sources alive until the gather is done
        nbytes = rows * 12
        if self.host[slot] is None or self.host[slot].numel() < nbytes:
            self.host[slot] = torch.empty(int(nbytes * 1.25) + 256, dtype=torch.uint8, pin_memory=True)
        ptrs = (C.c_void_p * len(segs))(*[p.data_ptr() for p in segs])
        nrow = (C.c_int64 * len(segs))(*[int(p.shape[0]) for p in segs])
        t = _lib.lib.fnp_host_pack_xyz_multi_begin(ptrs, nrow, len(segs), C_, xyz_offset, self.host[slot].data_ptr(),
                                                   self.n_threads)
        if t < 0:
            _lib.check(t, "fnp_host_pack_xyz_multi_begin")
        self.ticket[slot] = t

    def upload(self, slot):
        """Waits for the slot's gather, enqueues its H2D copy; returns (device table, ready event)."""
        src = self.src[slot]
        rows, C_ = self.rows[slot], self.width[slot]
        if self.pack:
            _lib.check(_lib.lib.fnp_host_pack_wait(self.ticket[slot]), "fnp_host_pack_wait")
            self.ticket[slot] = None
            width, host = 3, self.host[slot][:rows * 12].view(torch.float32).view(rows, 3)
        else:
            width, host = C_, src
        if self.dev[slot] is None or self.dev[slot].numel() < rows * width:
            self.dev[slot] = torch.empty(int(rows * width * 1.25) + 64, dtype=torch.float32, device=self.eng.device)
        dev = self.dev[slot][:rows * width].view(rows, width)
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(self.consumed[slot])
            dev.copy_(host, non_blocking=True)
            self.ready[slot].record(self.copy_stream)
            self.copied[slot].record(self.copy_stream)
            self.copied_valid[slot] = True
        return dev, self.ready[slot]

    def mark_consumed(self, slot):
        """Call on the compute stream after the kernels that read the slot's device table."""
        self.consumed[slot].record()
