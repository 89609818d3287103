"""Synthetic nuScenes-shaped frames for the Greedy Box Seeker path.

No nuScenes data exists in this environment, so this module emits the *same boundary
objects* the reference's loader hands to the seeker:

  * the per-frame ``batch_dict`` entries of ``NuScenesDataset.__getitem__`` /
    ``load_camera_info`` / ``collate_batch`` (reference:
    pcdet/datasets/nuscenes/nuscenes_dataset.py:172-279, pcdet/datasets/dataset.py:222-344):
    ``points (N,5) [x,y,z,intensity,time]`` (collated to ``(sum N, 1+5)`` with a leading
    batch index), ``lidar2image``, ``camera_intrinsics``, ``camera2lidar`` ``(6,4,4)``,
    ``lidar_aug_matrix (4,4)`` = identity, ``gt_boxes (G,10)``, ``image_paths``,
    ``metadata['token']``, ``frame_id``;
  * the 2D detections of ``PreprocessedGLIP`` (pcdet/models/preprocessed_detector.py:47-106):
    ``boxes (D,4) xyxy px``, ``labels (D) 1..10``, ``scores (D)``, ``cam_idx (D)``.

Frame ``i`` is generated from ``numpy.random.Generator(PCG64(1000 + i))`` (SURVEY.md 8d).
Geometry is ray-cast: a spinning LiDAR against a ground plane, class-prior sized cuboids
and a far wall, so frustums contain object + background points like real data.
"""
from dataclasses import dataclass, field
from typing import Dict, List

import numpy as np
import torch

CLASS_NAMES = ['car', 'truck', 'construction_vehicle', 'bus', 'trailer',
               'barrier', 'motorcycle', 'bicycle', 'pedestrian', 'traffic_cone']

# class prior sizes (l, w, h), reference: frustum_proposals_v1.py:270-281
PRIORS = np.array([
    [4.63, 1.97, 1.74], [6.93, 2.51, 2.84], [6.37, 2.85, 3.19], [10.5, 2.94, 3.47],
    [12.29, 2.90, 3.87], [0.50, 2.53, 0.98], [2.11, 0.77, 1.47], [1.70, 0.60, 1.28],
    [0.73, 0.67, 1.77], [0.41, 0.41, 1.07]], dtype=np.float64)

# camera index order of the nuScenes loader: FRONT, FRONT_RIGHT, FRONT_LEFT, BACK,
# BACK_LEFT, BACK_RIGHT (reference: pcdet/datasets/nuscenes/nuscenes_utils.py:364-371)
CAM_NAMES = ['CAM_FRONT', 'CAM_FRONT_RIGHT', 'CAM_FRONT_LEFT', 'CAM_BACK', 'CAM_BACK_LEFT', 'CAM_BACK_RIGHT']
CAM_YAW_DEG = [0.0, -55.0, 55.0, 180.0, 110.0, -110.0]
IMG_W, IMG_H = 1600, 900
GROUND_Z = -1.84


@dataclass
class SynthConfig:
    name: str = "cfg1"
    beams: int = 32
    azimuths: int = 1085
    sweeps: int = 1
    n_boxes2d: int = 20          # target number of surviving 2D boxes per frame
    num_mags: int = 6            # depth steps      (seeker PARAMS)
    num_rotations: int = 10      # yaw bins
    num_sizes: int = 1
    n_objects: int = 0           # 0 -> derived from n_boxes2d


CONFIGS: Dict[str, SynthConfig] = {
    # BASELINE.json configs[0]: one sweep, ~34k points, 20 GLIP boxes, shipped H = 6*10*1
    "cfg1": SynthConfig("cfg1", 32, 1085, 1, 20, 6, 10, 1),
    # configs[1..3]: 10 sweeps, ~300k points, 60 boxes, H = 64*12*1 = 768
    "cfg2": SynthConfig("cfg2", 32, 1085, 10, 60, 64, 12, 1),
    # configs[4]: 1M points, 200 boxes, H = 128*24*1 = 3072
    "cfg5": SynthConfig("cfg5", 128, 7812, 1, 200, 128, 24, 1),
    # tiny case for unit tests
    "tiny": SynthConfig("tiny", 16, 360, 1, 8, 4, 6, 1),
}


@dataclass
class Frame:
    """One frame at the seeker's input boundary (host memory, numpy)."""
    frame_id: str
    token: str
    points: np.ndarray                 # (N,5) f32  x,y,z,intensity,time
    lidar2image: np.ndarray            # (6,4,4) f32
    camera_intrinsics: np.ndarray      # (6,4,4) f32
    camera2lidar: np.ndarray           # (6,4,4) f32
    lidar_aug_matrix: np.ndarray       # (4,4) f32
    gt_boxes: np.ndarray               # (G,10) f32  x,y,z,dx,dy,dz,ry,vx,vy,cls
    image_paths: List[str]
    det_boxes: np.ndarray              # (D,4) f32 xyxy
    det_labels: np.ndarray             # (D,) int64 1..10
    det_scores: np.ndarray             # (D,) f32
    det_cam_idx: np.ndarray            # (D,) int64 0..5
    meta: dict = field(default_factory=dict)


def make_cameras():
    """6 pinhole cameras -> (lidar2image, camera_intrinsics, camera2lidar), each (6,4,4) f32,
    assembled exactly as load_camera_info does (nuscenes_dataset.py:180-213)."""
    l2i, intr, c2l = [], [], []
    for c, yaw_deg in enumerate(CAM_YAW_DEG):
        yaw = np.deg2rad(yaw_deg)
        # camera frame: z forward, x right, y down.  Columns = camera axes in lidar frame.
        fwd = np.array([np.cos(yaw), np.sin(yaw), 0.0])
        right = np.array([np.sin(yaw), -np.cos(yaw), 0.0])
        down = np.array([0.0, 0.0, -1.0])
        # small fixed mounting tilt so the matrices are not axis-aligned
        tilt = np.deg2rad(0.6 + 0.2 * c)
        fwd_t = np.cos(tilt) * fwd + np.sin(tilt) * down
        down_t = -np.sin(tilt) * fwd + np.cos(tilt) * down
        R = np.stack([right, down_t, fwd_t], axis=1)            # sensor2lidar_rotation
        t = np.array([0.75 * np.cos(yaw), 0.75 * np.sin(yaw) + 0.05 * (c - 2.5), -0.3])
        if c == 3:
            K = np.array([[809.2, 0, 829.2], [0, 809.2, 481.8], [0, 0, 1.0]])
        else:
            K = np.array([[1266.4, 0, 816.3], [0, 1266.4, 491.5], [0, 0, 1.0]])
        lidar2camera_r = np.linalg.inv(R)
        lidar2camera_t = t @ lidar2camera_r.T
        rt = np.eye(4).astype(np.float32)
        rt[:3, :3] = lidar2camera_r.T
        rt[3, :3] = -lidar2camera_t
        K4 = np.eye(4).astype(np.float32)
        K4[:3, :3] = K
        l2i.append(K4 @ rt.T)
        intr.append(K4)
        m = np.eye(4).astype(np.float32)
        m[:3, :3] = R
        m[:3, 3] = t
        c2l.append(m)
    return (np.stack(l2i).astype(np.float32), np.stack(intr).astype(np.float32),
            np.stack(c2l).astype(np.float32))


def _box_corners(b):
    """(G,7) -> (G,8,3) float64, corner order of box_utils.boxes_to_corners_3d."""
    tpl = np.array([[1, 1, -1], [1, -1, -1], [-1, -1, -1], [-1, 1, -1],
                    [1, 1, 1], [1, -1, 1], [-1, -1, 1], [-1, 1, 1]], dtype=np.float64) / 2
    c = b[:, None, 3:6] * tpl[None]
    ca, sa = np.cos(b[:, 6]), np.sin(b[:, 6])
    x = c[..., 0] * ca[:, None] - c[..., 1] * sa[:, None]
    y = c[..., 0] * sa[:, None] + c[..., 1] * ca[:, None]
    return np.stack([x, y, c[..., 2]], -1) + b[:, None, 0:3]


def _raycast(origins, dirs, boxes, device, wall_r):
    """Nearest hit distance of each ray against ground / cuboids / far wall (torch, f64)."""
    o = torch.as_tensor(origins, dtype=torch.float64, device=device)
    d = torch.as_tensor(dirs, dtype=torch.float64, device=device)
    bx = torch.as_tensor(boxes, dtype=torch.float64, device=device)
    out = torch.empty(o.shape[0], dtype=torch.float64, device=device)
    ca, sa = torch.cos(bx[:, 6]), torch.sin(bx[:, 6])
    half = bx[:, 3:6] / 2
    CH = 1 << 16
    inf = torch.tensor(float('inf'), dtype=torch.float64, device=device)
    for s in range(0, o.shape[0], CH):
        oo, dd = o[s:s + CH], d[s:s + CH]
        # ground
        tg = torch.where(dd[:, 2] < -1e-6, (GROUND_Z - oo[:, 2]) / dd[:, 2], inf)
        # wall: vertical cylinder of radius wall_r around the origin (ray from near the axis)
        hn = torch.sqrt(dd[:, 0] ** 2 + dd[:, 1] ** 2).clamp_min(1e-9)
        tw = wall_r[s:s + CH] / hn
        t = torch.minimum(tg, tw)
        # cuboids: slab test in each box's frame
        rel = oo[:, None, :] - bx[None, :, 0:3]
        lox = rel[..., 0] * ca + rel[..., 1] * sa
        loy = -rel[..., 0] * sa + rel[..., 1] * ca
        ldx = dd[:, None, 0] * ca + dd[:, None, 1] * sa
        ldy = -dd[:, None, 0] * sa + dd[:, None, 1] * ca
        lo = torch.stack([lox, loy, rel[..., 2]], -1)
        ld = torch.stack([ldx, ldy, dd[:, None, 2].expand_as(ldx)], -1)
        ld = torch.where(ld.abs() < 1e-12, torch.full_like(ld, 1e-12), ld)
        t1 = (-half[None] - lo) / ld
        t2 = (half[None] - lo) / ld
        tn = torch.minimum(t1, t2).amax(-1)
        tf = torch.maximum(t1, t2).amin(-1)
        hit = (tf >= tn) & (tn > 0.5)
        tb = torch.where(hit, tn, inf).amin(1) if bx.shape[0] else inf.expand(oo.shape[0])
        out[s:s + CH] = torch.minimum(t, tb)
    return out.cpu().numpy()


def make_frame(index: int, cfg: SynthConfig, device: str = "cpu") -> Frame:
    rng = np.random.Generator(np.random.PCG64(1000 + index))
    l2i, intr, c2l = make_cameras()

    # ---- objects ---------------------------------------------------------------
    G = cfg.n_objects or int(np.ceil(cfg.n_boxes2d * 1.7)) + 4
    cls = rng.integers(0, 10, size=G)
    dims = PRIORS[cls] * rng.uniform(0.9, 1.1, size=(G, 3))
    rad = rng.uniform(5.0, 50.0, size=G)
    az = rng.uniform(-np.pi, np.pi, size=G)
    yaw = rng.uniform(-np.pi, np.pi, size=G)
    gt = np.zeros((G, 10), dtype=np.float64)
    gt[:, 0] = rad * np.cos(az)
    gt[:, 1] = rad * np.sin(az)
    gt[:, 2] = GROUND_Z + dims[:, 2] / 2
    gt[:, 3:6] = dims
    gt[:, 6] = yaw
    gt[:, 7:9] = rng.normal(0, 1.0, size=(G, 2))
    gt[:, 9] = cls + 1
    keep = (np.abs(gt[:, 0]) < 52) & (np.abs(gt[:, 1]) < 52)
    gt = gt[keep]

    # ---- LiDAR -----------------------------------------------------------------
    elev = np.deg2rad(np.linspace(-30.67, 10.67, cfg.beams))
    azim = np.linspace(-np.pi, np.pi, cfg.azimuths, endpoint=False)
    ee, aa = np.meshgrid(elev, azim, indexing='ij')
    dirs1 = np.stack([np.cos(ee) * np.cos(aa), np.cos(ee) * np.sin(aa), np.sin(ee)], -1).reshape(-1, 3)
    pts = []
    for k in range(cfg.sweeps):
        origin = np.array([-0.25 * k, 0.0, 0.0])
        o = np.ascontiguousarray(np.broadcast_to(origin, dirs1.shape))
        wall = 45.0 + 9.0 * (0.5 + 0.5 * np.sin(3.0 * np.arctan2(dirs1[:, 1], dirs1[:, 0]) + 0.7 * k))
        t = _raycast(o, dirs1, gt[:, :7], device, torch.as_tensor(wall, dtype=torch.float64, device=device))
        t = t + rng.normal(0.0, 0.02, size=t.shape)
        ok = np.isfinite(t) & (t > 0.8) & (t < 75.0)
        p = o[ok] + dirs1[ok] * t[ok, None]
        ok2 = (np.abs(p[:, 0]) < 54.0) & (np.abs(p[:, 1]) < 54.0) & (p[:, 2] > -5.0) & (p[:, 2] < 3.0)
        p = p[ok2]
        feat = np.stack([rng.uniform(0, 255, size=p.shape[0]), np.full(p.shape[0], 0.05 * k)], -1)
        pts.append(np.concatenate([p, feat], -1))
    points = np.concatenate(pts, 0).astype(np.float32)

    # ---- 2D detections -----------------------------------------------------------
    corners = _box_corners(gt[:, :7])                                   # (G,8,3)
    hom = np.concatenate([corners, np.ones(corners.shape[:2] + (1,))], -1)
    cand = []
    for c in range(6):
        w = hom @ l2i[c].astype(np.float64).T                           # (G,8,4)
        front = (w[..., 2] > 0.5).all(1)
        u = w[..., 0] / np.maximum(w[..., 2], 1e-5)
        v = w[..., 1] / np.maximum(w[..., 2], 1e-5)
        x1, x2, y1, y2 = u.min(1), u.max(1), v.min(1), v.max(1)
        x1c, x2c = np.clip(x1, 0, IMG_W), np.clip(x2, 0, IMG_W)
        y1c, y2c = np.clip(y1, 0, IMG_H), np.clip(y2, 0, IMG_H)
        area = (x2c - x1c) * (y2c - y1c)
        full = np.maximum((x2 - x1) * (y2 - y1), 1e-6)
        vis = front & (area > 150.0) & (area / full > 0.35)
        for g in np.nonzero(vis)[0]:
            cand.append((c, g, x1c[g], y1c[g], x2c[g], y2c[g]))
    order = rng.permutation(len(cand))
    cand = [cand[i] for i in order][:cfg.n_boxes2d]
    boxes, labels, scores, cams = [], [], [], []
    for (c, g, x1, y1, x2, y2) in cand:
        j = rng.normal(0, 5.0, size=4)
        b = np.array([np.clip(x1 + j[0], 0, IMG_W - 2), np.clip(y1 + j[1], 0, IMG_H - 2),
                      np.clip(x2 + j[2], 0, IMG_W), np.clip(y2 + j[3], 0, IMG_H)])
        b[2] = max(b[2], b[0] + 2.0)
        b[3] = max(b[3], b[1] + 2.0)
        s = rng.uniform(0.45, 0.95)
        boxes.append(b); labels.append(int(gt[g, 9])); scores.append(s); cams.append(c)
        r = rng.uniform()
        if r < 0.15:      # near-duplicate, lower score, same label: removed by the 2D NMS
            boxes.append(b + rng.normal(0, 1.5, size=4)); labels.append(int(gt[g, 9]))
            scores.append(s * rng.uniform(0.6, 0.98)); cams.append(c)
        elif r < 0.30:    # distractor below the score threshold
            bb = b + rng.normal(0, 40.0, size=4)
            bb = np.array([min(bb[0], bb[2]), min(bb[1], bb[3]), max(bb[0], bb[2]) + 2, max(bb[1], bb[3]) + 2])
            boxes.append(bb); labels.append(int(rng.integers(1, 11)))
            scores.append(rng.uniform(0.05, 0.44)); cams.append(c)
    D = len(boxes)
    perm = rng.permutation(D) if D else np.zeros((0,), dtype=np.int64)
    det_boxes = np.asarray(boxes, dtype=np.float32).reshape(-1, 4)[perm]
    det_labels = np.asarray(labels, dtype=np.int64)[perm]
    det_scores = np.asarray(scores, dtype=np.float32)[perm]
    det_cams = np.asarray(cams, dtype=np.int64)[perm]
    # PreprocessedGLIP concatenates camera 0..5 in order (preprocessed_detector.py:60-93)
    o2 = np.argsort(det_cams, kind='stable')
    det_boxes, det_labels, det_scores, det_cams = det_boxes[o2], det_labels[o2], det_scores[o2], det_cams[o2]

    fid = "n%03d-synth-%s__LIDAR_TOP__%010d.pcd" % (index % 1000, cfg.name, 1000 + index)
    return Frame(
        frame_id=fid, token="tok%08d" % (1000 + index), points=points,
        lidar2image=l2i, camera_intrinsics=intr, camera2lidar=c2l,
        lidar_aug_matrix=np.eye(4, dtype=np.float32), gt_boxes=gt.astype(np.float32),
        image_paths=["samples/%s/%s__%s.jpg" % (n, fid, n) for n in CAM_NAMES],
        det_boxes=det_boxes, det_labels=det_labels, det_scores=det_scores, det_cam_idx=det_cams,
        meta=dict(index=index, cfg=cfg.name))


def collate(frames: List[Frame]) -> dict:
    """The batch_dict of DatasetTemplate.collate_batch (dataset.py:222-344) as numpy/host
    objects: points get a leading batch-index column, gt_boxes are zero-padded."""
    B = len(frames)
    pts = []
    for b, f in enumerate(frames):
        pts.append(np.concatenate([np.full((f.points.shape[0], 1), b, np.float32), f.points], 1))
    G = max([f.gt_boxes.shape[0] for f in frames] + [1])
    gt = np.zeros((B, G, 10), np.float32)
    for b, f in enumerate(frames):
        gt[b, :f.gt_boxes.shape[0]] = f.gt_boxes
    return dict(
        batch_size=B,
        points=np.concatenate(pts, 0),
        lidar2image=np.stack([f.lidar2image for f in frames]),
        camera_intrinsics=np.stack([f.camera_intrinsics for f in frames]),
        camera2lidar=np.stack([f.camera2lidar for f in frames]),
        lidar_aug_matrix=np.stack([f.lidar_aug_matrix for f in frames]),
        gt_boxes=gt,
        image_paths=[list(f.image_paths) for f in frames],
        metadata=[dict(token=f.token) for f in frames],
        frame_id=np.array([f.frame_id for f in frames]),
    )


def seeker_params(cfg: SynthConfig) -> dict:
    """MODEL.DENSE_HEAD.PARAMS of tools/cfgs/nuscenes_box_seeker_proposals.yaml:83 with the
    hypothesis-grid sizes of the synthetic config."""
    return dict(lq=0.0, uq=0.25, cq=1.0, iou_w=1.0, nms_normal=1.0, dst_w=0.0, dns_w=1.0,
                min_cam_iou=0.3, score_thr=0.45, nms_2d=0.4, nms_3d=0.0, clamp_bottom=1,
                num_sizes=cfg.num_sizes, num_mags=cfg.num_mags, num_rotations=cfg.num_rotations)


def write_nuscenes_tree(root, frames):
    """Write synthetic frames as a nuScenes-format tree (LiDAR .bin files of 5 floats per point,
    no sweeps) and return the matching info dicts (the fields NuScenesDataset reads,
    nuscenes_dataset.py:105-233) -- the on-disk input of findnpropagate_b200.nuscenes_feed."""
    import os
    infos = []
    names = ["CAM_FRONT", "CAM_FRONT_RIGHT", "CAM_FRONT_LEFT", "CAM_BACK", "CAM_BACK_LEFT", "CAM_BACK_RIGHT"]
    for f in frames:
        rel = os.path.join("samples", "LIDAR_TOP", f.frame_id + ".bin")
        os.makedirs(os.path.join(root, os.path.dirname(rel)), exist_ok=True)
        np.ascontiguousarray(f.points, np.float32).tofile(os.path.join(root, rel))
        cams = {}
        for c, name in enumerate(names):
            cams[name] = dict(data_path=f.image_paths[c], sensor2lidar_rotation=f.camera2lidar[c, :3, :3].astype(np.float64),
                              sensor2lidar_translation=f.camera2lidar[c, :3, 3].astype(np.float64),
                              camera_intrinsics=f.camera_intrinsics[c, :3, :3].astype(np.float64),
                              sensor2ego_rotation=[1.0, 0.0, 0.0, 0.0], sensor2ego_translation=[0.0, 0.0, 0.0])
        gt = np.asarray(f.gt_boxes, np.float32)
        infos.append(dict(lidar_path=rel, token=f.token, sweeps=[], cams=cams, gt_boxes=gt[:, :9].copy(),
                          gt_names=np.array([CLASS_NAMES[int(c) - 1] for c in gt[:, -1]]),
                          num_lidar_pts=np.full(gt.shape[0], 10)))
    return infos


def write_glip_predictions(frames, pred_pth, meta_coco):
    """Write the detections of synthetic frames as the GLIP prediction file (a pickled list of BoxList, one per camera
    image) and its COCO meta json (``images`` with ``token`` and ``file_name``) that proposer.PreprocessedGLIP
    reads (preprocessed_detector.py:11-45)."""
    import json
    import os
    from .proposer import BoxList, install_boxlist_shim
    install_boxlist_shim()
    lists, images = [], []
    for f in frames:
        for c in range(6):
            m = np.asarray(f.det_cam_idx) == c
            bl = BoxList(torch.from_numpy(np.asarray(f.det_boxes, np.float32)[m].reshape(-1, 4)), (IMG_W, IMG_H))
            bl.extra_fields = dict(scores=torch.from_numpy(np.asarray(f.det_scores, np.float32)[m]),
                                   labels=torch.from_numpy(np.asarray(f.det_labels, np.int64)[m]))
            lists.append(bl)
            images.append(dict(id=len(images), token=f.token, file_name=str(f.image_paths[c])))
    for p in (pred_pth, meta_coco):
        os.makedirs(os.path.dirname(os.path.abspath(p)), exist_ok=True)
    torch.save(lists, pred_pth)
    with open(meta_coco, "w") as fh:
        json.dump(dict(images=images, categories=[dict(id=i + 1, name=n) for i, n in enumerate(CLASS_NAMES)]), fh)


# class names of the synthetic KITTI tree (write_kitti_tree), one per anchor of the KITTI head, in label order
KITTI_CLASS_NAMES = ['Car', 'Truck', 'Van', 'Tram', 'Pedestrian', 'Cyclist', 'Person_sitting']
KITTI_IMAGE_SHAPE = (375, 1242)


def make_kitti_frame(index, with_gt=False, cfg=None, full_scan=False):
    """A KITTI-shaped frame: points in front of the sensor, P2 / R0 / Tr_velo2cam, x-y-w-h 2D boxes of the visible
    synthetic objects, labels 1..7 (the KITTI head's seven anchors).  with_gt: also the frame's (G,10) LiDAR-frame GT
    (make_frame's).  cfg: the scan (default 32 beams x 900 azimuths); full_scan: every point of the scan, not only
    those in front of the sensor (what a velodyne file holds before the FOV filter)."""
    cfg = cfg or SynthConfig("kitti", 32, 900, 1, 12, 4, 6, 1)
    f = make_frame(index, cfg)
    pts = (f.points if full_scan else f.points[f.points[:, 0] > 1.0])[:, :4].copy()
    V2C = np.array([[0.0, -1.0, 0.0, 0.004], [0.0, 0.0, -1.0, -0.076], [1.0, 0.0, 0.0, -0.272]], np.float32)
    a = 0.01
    R0 = np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]], np.float32)
    P2 = np.array([[721.54, 0, 609.56, 44.857], [0, 721.54, 172.85, 0.2163], [0, 0, 1, 0.002746]], np.float32)
    boxes, labels, scores = [], [], []
    rng = np.random.default_rng(index)
    for g in f.gt_boxes:
        if g[0] < 4 or abs(g[1]) > g[0]:
            continue
        c = _box_corners(g[None, :7].astype(np.float64))[0]
        rect = (np.c_[c, np.ones(8)] @ (np.vstack([V2C, [0, 0, 0, 1]]).T))[:, :3] @ R0.T
        img = np.c_[rect, np.ones(8)] @ P2.T
        u, v = img[:, 0] / rect[:, 2], img[:, 1] / rect[:, 2]
        x1, x2 = np.clip(u.min(), 0, 1242), np.clip(u.max(), 0, 1242)
        y1, y2 = np.clip(v.min(), 0, 375), np.clip(v.max(), 0, 375)
        if x2 - x1 < 8 or y2 - y1 < 8:
            continue
        boxes.append([x1, y1, x2 - x1, y2 - y1])
        labels.append(1 + int(rng.integers(0, 7)))
        scores.append(float(rng.uniform(0.5, 0.9)))
    out = (pts, {'P2': P2, 'R0': R0, 'Tr_velo2cam': V2C}, np.asarray(boxes, np.float32).reshape(-1, 4),
           np.asarray(labels, np.int64), np.asarray(scores, np.float32))
    return out + (f.gt_boxes,) if with_gt else out


def write_kitti_tree(root, frames, class_names=KITTI_CLASS_NAMES, coco_path=None):
    """Write make_kitti_frame(i, with_gt=True) frames as an OpenPCDet KITTI tree under ``root`` (DATA_PATH), frame k
    with id ``%06d % k``: ``training/velodyne/<id>.bin`` (float32 x, y, z, intensity), ``training/calib/<id>.txt``
    (P0..P3, R0_rect, Tr_velo_to_cam, Tr_imu_to_velo), ``kitti_infos_train.pkl`` (point_cloud.lidar_idx,
    image.image_shape, annos with name / dimensions (l, h, w) / location / rotation_y in the rectified camera frame:
    every GT box, out of range ones included, plus one DontCare row per frame) and, at ``coco_path`` (default
    ``root/kitti_coco_results.json``), the COCO result file of the 2D boxes that proposer.PreprocessedDetector reads
    (images ``<id>.png``, category k + 1 = class_names[k]).  Returns the info dicts."""
    import json
    import os
    import pickle
    split = os.path.join(str(root), "training")
    for sub in ("velodyne", "calib"):
        os.makedirs(os.path.join(split, sub), exist_ok=True)
    infos, images, anns = [], [], []
    for k, (pts, cal, boxes, labels, scores, gt) in enumerate(frames):
        idx = "%06d" % k
        np.ascontiguousarray(pts, np.float32).tofile(os.path.join(split, "velodyne", idx + ".bin"))
        P2, R0, V2C = (np.asarray(cal[n], np.float32) for n in ("P2", "R0", "Tr_velo2cam"))
        rows = [("P0", P2), ("P1", P2), ("P2", P2), ("P3", P2), ("R0_rect", R0), ("Tr_velo_to_cam", V2C),
                ("Tr_imu_to_velo", V2C)]
        with open(os.path.join(split, "calib", idx + ".txt"), "w") as fh:
            fh.write("".join("%s: %s\n" % (n, " ".join(repr(float(v)) for v in m.reshape(-1))) for n, m in rows))
        g = np.asarray(gt, np.float64)
        bottom = np.c_[g[:, 0:2], g[:, 2] - g[:, 5] / 2, np.ones(len(g))]
        loc = (bottom @ np.vstack([V2C, [0, 0, 0, 1]]).astype(np.float64).T)[:, :3] @ R0.astype(np.float64).T
        names = [class_names[(int(c) - 1) % len(class_names)] for c in g[:, 9]] + ["DontCare"]
        annos = dict(name=np.array(names),
                     dimensions=np.r_[g[:, [3, 5, 4]], [[-1.0, -1.0, -1.0]]].astype(np.float32),
                     location=np.r_[loc, [[-1000.0, -1000.0, -1000.0]]].astype(np.float32),
                     rotation_y=np.r_[-g[:, 6] - np.pi / 2, [-10.0]].astype(np.float32))
        infos.append(dict(point_cloud=dict(num_features=4, lidar_idx=idx),
                          image=dict(image_idx=idx, image_shape=np.array(KITTI_IMAGE_SHAPE, np.int32)),
                          calib=dict(P2=P2, R0_rect=R0, Tr_velo_to_cam=V2C), annos=annos))
        images.append(dict(id=k, file_name=idx + ".png"))
        for b, lab, sc in zip(boxes, labels, scores):
            anns.append(dict(id=len(anns), image_id=k, category_id=int(lab), score=float(sc),
                             bbox=[float(v) for v in b]))
    with open(os.path.join(str(root), "kitti_infos_train.pkl"), "wb") as fh:
        pickle.dump(infos, fh)
    with open(coco_path or os.path.join(str(root), "kitti_coco_results.json"), "w") as fh:
        json.dump(dict(images=images, annotations=anns,
                       categories=[dict(id=i + 1, name=n) for i, n in enumerate(class_names)]), fh)
    return infos
