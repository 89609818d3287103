"""Drop-in for the reference's ``FrustumProposerOG`` dense head and its 2D-box feeder.

Reference: pcdet/models/dense_heads/frustum_proposals_v1.py:142-318 (constructor),
:523-1067 (get_proposals), :1547-1573 (forward / get_bboxes) and
pcdet/models/preprocessed_detector.py:7-106 (PreprocessedGLIP), :111-290 (PreprocessedDetector).

Same class names, constructor arguments, ``model_cfg.PARAMS`` keys, method names, return
types and devices; the work is done by :class:`findnpropagate_b200.seeker.SeekerEngine`.
"""
import json
import os
import sys
import types

import numpy as np
import torch
from torch import nn

from .seeker import DEFAULTS, SeekerEngine


def _cfg_get(cfg, key, default=None):
    if cfg is None:
        return default
    if isinstance(cfg, dict):
        return cfg.get(key, default)
    return getattr(cfg, key, default) if not hasattr(cfg, "get") else cfg.get(key, default)


# PARAMS keys the head reads besides the constructor's own (:160-165)
EXTRA_PARAMS = ('aln_w', 'ego_w', 'occl_w', 'rand_center', 'search_depth')


def head_params(model_cfg, defaults=None):
    """The parameters FrustumProposerOG runs with: ``defaults`` (the constructor's, DEFAULTS when None), overridden by
    ``model_cfg.PARAMS`` (:167-196), plus the model_cfg-level switches MULTICAM_IOU / OCCL_MULT / MULT (:154-156)."""
    p = dict(DEFAULTS if defaults is None else defaults)
    params = _cfg_get(model_cfg, 'PARAMS')
    if params is not None:
        for k in list(DEFAULTS) + list(EXTRA_PARAMS):
            if k in params:
                p[k] = params[k]
    if _cfg_get(model_cfg, 'SAVE_BLEND', False):
        raise NotImplementedError("SAVE_BLEND (Blender visualisation dumps) is outside the Box Seeker path")
    for flag in ('MULTICAM_IOU', 'OCCL_MULT', 'MULT'):
        p[flag] = bool(_cfg_get(model_cfg, flag, False))
    return p


# ----------------------------------------------------------------------------- feeders
class BoxList:
    """Unpickling shim for maskrcnn_benchmark.structures.bounding_box.BoxList (GLIP's
    prediction container; un-vendored dependency of the reference): only the attributes
    PreprocessedGLIP reads -- ``bbox`` (D,4) xyxy and ``extra_fields['scores'|'labels']``."""

    def __init__(self, bbox=None, image_size=None, mode="xyxy"):
        self.bbox = bbox
        self.size = image_size
        self.mode = mode
        self.extra_fields = {}


def install_boxlist_shim():
    """Make ``torch.load`` of a GLIP prediction file work without maskrcnn_benchmark."""
    if "maskrcnn_benchmark.structures.bounding_box" in sys.modules:
        return
    pkg = types.ModuleType("maskrcnn_benchmark")
    sub = types.ModuleType("maskrcnn_benchmark.structures")
    mod = types.ModuleType("maskrcnn_benchmark.structures.bounding_box")
    mod.BoxList = BoxList
    BoxList.__module__ = mod.__name__
    pkg.structures, sub.bounding_box = sub, mod
    sys.modules.update({pkg.__name__: pkg, sub.__name__: sub, mod.__name__: mod})


class PreprocessedGLIP:
    """Loads the pickled GLIP predictions + COCO-style meta json and returns, per batch, the
    5 CPU tensors (boxes xyxy, labels 1..10, scores, batch_idx, cam_idx) --
    preprocessed_detector.py:7-106."""

    def __init__(self, pred_pth='../data/training_pred/nuscenes_glip_train_pred.pth',
                 meta_coco='../data/training_pred/nuscenes_infos_train_mono3d.coco.json', class_names=None):
        self.all_class_names = ['car', 'truck', 'construction_vehicle', 'bus', 'trailer',
                                'barrier', 'motorcycle', 'bicycle', 'pedestrian', 'traffic_cone']
        self.class_names = self.all_class_names if class_names is None else class_names
        install_boxlist_shim()
        self.glip_bboxes = torch.load(pred_pth, weights_only=False)
        with open(meta_coco, 'r') as f:
            self.meta_info = json.load(f)
        self.map_catid = {(i + 1): (i + 1) for i in range(len(self.all_class_names))}
        self.token_to_id, self.path_to_id = {}, {}
        for img_id, image in enumerate(self.meta_info['images']):
            self.token_to_id[image['token']] = img_id
            self.path_to_id[image['file_name']] = img_id

    def has_image(self, path) -> bool:
        """Whether ``infer_nusc`` finds the camera image ``path`` in the prediction file."""
        return str(path) in self.path_to_id

    def infer_nusc(self, batch_dict):
        labels, boxes, scores, idx, cam_idx = [], [], [], [], []
        for b in range(batch_dict['batch_size']):
            cur_paths = batch_dict['image_paths'][b]
            for c in range(6):
                img_id = self.path_to_id[str(cur_paths[c])]
                assert batch_dict['metadata'][b]['token'] == self.meta_info['images'][img_id]['token']
                assert str(cur_paths[c]) == self.meta_info['images'][img_id]['file_name']
                bl = self.glip_bboxes[img_id]
                c_boxes = bl.bbox.reshape(-1, 4)
                c_scores = bl.extra_fields['scores'].reshape(-1)
                c_labels = bl.extra_fields['labels'].reshape(-1).clone()
                for i, lbl in enumerate(c_labels):
                    c_labels[i] = self.map_catid[lbl.item()]
                boxes.append(c_boxes); labels.append(c_labels); scores.append(c_scores)
                idx.extend([b] * len(c_boxes)); cam_idx.extend([c] * len(c_boxes))
        return (torch.cat(boxes, dim=0), torch.cat(labels, dim=0), torch.cat(scores, dim=0),
                torch.tensor(idx), torch.tensor(cam_idx))

    def __call__(self, batch_dict):
        if 'image_paths' in batch_dict:
            return self.infer_nusc(batch_dict)
        raise TypeError('need kitti / nusc batch dict!')


class PreprocessedDetector:
    """The head's other feeder: COCO-format result files, one per camera view (``PREDS_PATHS`` / ``PREDS_PATH`` +
    camera name, frustum_proposals_v1.py:262-268), served per batch with the same 5-tensor contract --
    pcdet/models/preprocessed_detector.py:111-290.

    The files are indexed once: per image name the boxes / class ids / scores of the wanted categories as
    arrays, in annotation order (file after file), so that a batch is a handful of concatenations.  Boxes are
    handed out as they are stored (COCO x, y, w, h: such configs set ``BOX_FORMAT`` accordingly)."""

    def __init__(self, cam_jsons=(), class_names=None):
        assert len(cam_jsons) > 0
        self.infer_cam = len(cam_jsons) == 1
        self.categories = None
        views = []
        for path in cam_jsons:
            with open(path, 'r') as f:
                d = json.load(f)
            assert self.categories is None or self.categories == d['categories'], 'categories differ!'
            self.categories = d['categories']
            views.append(d)
        self.class_names = [c['name'] for c in self.categories] if not class_names else list(class_names)
        cat_ids = {c['id'] for c in self.categories}
        # category id -> class id (1-based position of the category's name in class_names); other categories
        # are dropped (:149-150)
        self.catid_to_classid = {c['id']: i + 1 for c in self.categories
                                 for i, n in enumerate(self.class_names) if n == c['name']}
        self.wanted_catids = list(self.catid_to_classid)
        if not self.catid_to_classid:
            raise ValueError("none of the class names %r is a category of the result files" % (self.class_names,))
        rows = {}                       # image name -> list of (bbox, class id, score)
        for d in views:
            name_of = {}
            for img in d['images']:
                name = img['name'] if 'name' in img else os.path.basename(img['file_name'])     # :132-135
                name_of[img['id']] = name
                rows.setdefault(name, [])
            for ann in d['annotations']:
                cat = ann['category_id']
                if cat not in cat_ids:                      # files with 1-based ids over 0-based categories (:176-177)
                    cat -= 1
                assert cat in cat_ids, '%r not valid' % (ann,)
                if cat in self.catid_to_classid:
                    rows[name_of[ann['image_id']]].append(
                        (ann['bbox'], self.catid_to_classid[cat], 1.0 if 'score' not in ann else ann['score']))
        self.img_names = set(rows)
        first = next(iter(rows))
        self.incl_ext = '.jpg' in first or '.png' in first
        self.by_name = {n: (np.asarray([r[0] for r in v], np.float32).reshape(-1, 4),
                            np.asarray([r[1] for r in v], np.int64), np.asarray([r[2] for r in v], np.float32))
                        for n, v in rows.items()}

    def _collect(self, names_per_frame, cams_per_frame, strict=False):
        boxes, labels, scores, idx, cam = [], [], [], [], []
        for b, (names, cams) in enumerate(zip(names_per_frame, cams_per_frame)):
            for name, c in zip(names, cams):
                ent = self.by_name.get(name)
                if ent is None:
                    if strict:
                        raise ValueError('frame_id=%s did not exist in preprocessing' % name)
                    continue
                boxes.append(ent[0]); labels.append(ent[1]); scores.append(ent[2])
                idx.append(np.full(ent[1].shape[0], b, np.int64)); cam.append(np.full(ent[1].shape[0], c, np.int64))
        if not boxes or sum(x.shape[0] for x in labels) == 0:
            # the reference builds its tensors from empty lists here: five float tensors of shape (0,)
            return tuple(torch.tensor([]) for _ in range(5))
        return (torch.from_numpy(np.concatenate(boxes)), torch.from_numpy(np.concatenate(labels)),
                torch.from_numpy(np.concatenate(scores)), torch.from_numpy(np.concatenate(idx)),
                torch.from_numpy(np.concatenate(cam)))

    def _image_name(self, path) -> str:
        return os.path.basename(str(path)) if self.incl_ext else os.path.splitext(os.path.basename(str(path)))[0]

    def has_image(self, path) -> bool:
        """Whether the result files list the camera image ``path``."""
        return self._image_name(path) in self.by_name

    def infer_nusc(self, batch_dict):
        names = [[self._image_name(p) for p in batch_dict['image_paths'][b]] for b in range(batch_dict['batch_size'])]
        return self._collect(names, [range(len(n)) for n in names])

    def infer_kitti(self, batch_dict):
        names = [[(batch_dict['frame_id'][b] + '.png') if self.incl_ext else batch_dict['frame_id'][b]]
                 for b in range(batch_dict['batch_size'])]
        return self._collect(names, [[0]] * len(names), strict=True)

    def __call__(self, batch_dict):
        if 'image_paths' in batch_dict:
            return self.infer_nusc(batch_dict)
        if 'frame_id' in batch_dict:
            return self.infer_kitti(batch_dict)
        raise TypeError('need kitti / nusc batch dict!')


class SyntheticGLIP:
    """Feeder with the PreprocessedGLIP return contract over synthetic frames
    (findnpropagate_b200.synth.Frame), keyed by the first image path of each frame."""

    def __init__(self, frames=(), class_names=None):
        self.by_path = {str(f.image_paths[0]): f for f in frames}

    def add(self, frame):
        self.by_path[str(frame.image_paths[0])] = frame

    def __call__(self, batch_dict):
        if 'image_paths' not in batch_dict:
            raise TypeError('need kitti / nusc batch dict!')
        boxes, labels, scores, idx, cam = [], [], [], [], []
        for b in range(batch_dict['batch_size']):
            f = self.by_path[str(batch_dict['image_paths'][b][0])]
            boxes.append(torch.from_numpy(np.asarray(f.det_boxes, np.float32)).reshape(-1, 4))
            labels.append(torch.from_numpy(np.asarray(f.det_labels, np.int64)))
            scores.append(torch.from_numpy(np.asarray(f.det_scores, np.float32)))
            cam.append(torch.from_numpy(np.asarray(f.det_cam_idx, np.int64)))
            idx.extend([b] * len(f.det_scores))
        return (torch.cat(boxes), torch.cat(labels), torch.cat(scores), torch.tensor(idx, dtype=torch.long),
                torch.cat(cam))


# ----------------------------------------------------------------------------- the head
class FrustumProposerOG(nn.Module):
    """Greedy Box Seeker head with the reference's constructor signature
    (frustum_proposals_v1.py:143-149).  ``image_detector`` may be passed explicitly; otherwise
    ``PREDS_PATH == 'PreprocessedGLIP'`` builds the GLIP feeder as the reference does."""

    def __init__(self, model_cfg=None, input_channels=None, num_class=None, class_names=None, grid_size=None,
                 point_cloud_range=None, voxel_size=None, predict_boxes_when_training=True,
                 lq=0.336, uq=0.356, iou_w=0.95, dst_w=0.226, dns_w=0.05, min_cam_iou=0.3, size_min=0.957,
                 size_max=1.2, ry_min=0.0, ry_max=torch.pi, cq=0.46, num_mags=6, max_dist=50, num_sizes=4,
                 num_rotations=10, topk=1, nms_2d=0.7, nms_3d=1.0, score_thr=0.1, nms_normal=0.7, clamp_bottom=0,
                 image_detector=None, device=None):
        super().__init__()
        p = dict(lq=lq, uq=uq, iou_w=iou_w, dst_w=dst_w, dns_w=dns_w, min_cam_iou=min_cam_iou, size_min=size_min,
                 size_max=size_max, ry_min=ry_min, ry_max=float(ry_max), cq=cq, num_mags=num_mags, max_dist=max_dist,
                 num_sizes=num_sizes, num_rotations=num_rotations, topk=topk, nms_2d=nms_2d, nms_3d=nms_3d,
                 score_thr=score_thr, nms_normal=nms_normal, clamp_bottom=clamp_bottom)
        p = head_params(model_cfg, p)
        assert p['nms_3d'] == 0, 'DO NOT USE!'          # the reference's own assertion (:209)
        self.params = p
        self.box_fmt = _cfg_get(model_cfg, 'BOX_FORMAT', 'xyxy')
        self.image_order = [2, 0, 1, 5, 3, 4]
        self.image_size = [900, 1600]
        self.topk, self.score_thr, self.max_dist = p['topk'], p['score_thr'], p['max_dist']
        self.num_mags, self.num_sizes, self.num_rotations = p['num_mags'], p['num_sizes'], p['num_rotations']
        if image_detector is not None:
            self.image_detector = image_detector
        else:
            preds_path = _cfg_get(model_cfg, 'PREDS_PATH', 'PreprocessedGLIP')
            if 'PreprocessedGLIP' in preds_path:
                self.image_detector = PreprocessedGLIP(class_names=class_names)
            else:      # one COCO result file per camera view (:262-268)
                camera_names = ['CAM_BACK', 'CAM_BACK_LEFT', 'CAM_BACK_RIGHT', 'CAM_FRONT', 'CAM_FRONT_LEFT',
                                'CAM_FRONT_RIGHT']
                preds_paths = _cfg_get(model_cfg, 'PREDS_PATHS', [preds_path + "%s.json" % c for c in camera_names])
                self.image_detector = PreprocessedDetector(preds_paths, class_names=class_names)
        self.engine = SeekerEngine(p, device=device, box_format=self.box_fmt)
        self._cal_cache = {}
        self.anchors = torch.tensor(__import__('findnpropagate_b200.seeker', fromlist=['ANCHORS']).ANCHORS,
                                    dtype=torch.float32, device=self.engine.device)
        self.base_boxes = self.engine.base_boxes
        self.base_corners = self.engine.base_corners

    # -- helpers ---------------------------------------------------------------
    @staticmethod
    def _np(x):
        return x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)

    def get_proposals(self, batch_dict):
        """-> (proposal_boxes (K,7) f32 on the GPU, frust_labels (K) int64 CPU, frust_scores (K)
        f32 CPU, frust_batch_idx (K) int64 CPU), exactly as frustum_proposals_v1.py:1055-1067."""
        if 'img_aug_matrix' in batch_dict:
            raise NotImplementedError("img_aug_matrix (image_calibrate) is disabled in the shipped config")
        B = int(batch_dict['batch_size'])
        det_boxes, det_labels, det_scores, det_batch_idx, det_cam_idx = self.image_detector(batch_dict)
        pts = batch_dict['points']
        dev = self.engine.device
        if isinstance(pts, np.ndarray):
            pts = torch.from_numpy(np.ascontiguousarray(pts, np.float32))
        if not pts.is_cuda:
            # host table (the collate output before load_data_to_gpu): frame bounds from the batch
            # column on the host, then only x, y, z cross PCIe (threaded gather, fnp_host_pack_xyz)
            pts = pts.to(torch.float32).contiguous()
            bcol = pts[:, 0].numpy()
            if bcol.size > 1 and not bool((bcol[1:] >= bcol[:-1]).all()):
                raise ValueError("batch_dict['points'] must be grouped by batch index (collate_batch order)")
            bounds = np.searchsorted(bcol, np.arange(B + 1, dtype=np.float32))
            rows = int(pts.shape[0])
            stage = self.engine.arena.get("head_xyz_host", rows * 12, pinned=True)[:rows * 12].view(torch.float32).view(rows, 3)
            from . import _lib
            _lib.check(_lib.lib.fnp_host_pack_xyz(pts.data_ptr(), rows, int(pts.shape[1]), 1, stage.data_ptr(),
                                                  max(1, min(16, len(os.sched_getaffinity(0)) - 1))),
                       "fnp_host_pack_xyz")
            pts = self.engine.arena.get("head_xyz_dev", rows * 12)[:rows * 12].view(torch.float32).view(rows, 3)
            pts.copy_(stage, non_blocking=True)
            stride, xyz_offset = 3, 0
        else:
            pts = pts.to(dev, dtype=torch.float32, non_blocking=True).contiguous()
            if B == 1:
                # the reference's operating point (tools/extract_pseudo_labels.py:36 asserts batch size 1): one
                # frame, every row belongs to it -- no device round trip for the frame bounds
                bounds = np.array([0, int(pts.shape[0])], np.int64)
            else:
                bidx = pts[:, 0].contiguous()
                q = torch.searchsorted(bidx, torch.arange(B + 1, device=dev, dtype=torch.float32))
                ordered = (bidx[1:] >= bidx[:-1]).all() if bidx.numel() > 1 else torch.ones((), dtype=torch.bool, device=dev)
                got = torch.cat([q, ordered.reshape(1).to(q.dtype)]).cpu().numpy()      # one device round trip
                if not got[-1]:
                    raise ValueError("batch_dict['points'] must be grouped by batch index (collate_batch order)")
                bounds = got[:-1]
            stride, xyz_offset = int(pts.shape[1]), 1
        from .seeker import camera_matrices
        cal = [batch_dict['lidar2image'], batch_dict['camera2lidar'], batch_dict['camera_intrinsics']]
        aug = batch_dict['lidar_aug_matrix']
        if all(isinstance(c, torch.Tensor) and c.is_cuda for c in cal + [aug]):
            # four small device tensors: one concatenation, one copy back
            flat = torch.cat([c.reshape(B, -1).to(torch.float32) for c in cal + [aug]], dim=1).cpu().numpy()
            cal = [flat[:, 96 * i:96 * (i + 1)].reshape(B, 6, 4, 4) for i in range(3)]
            aug = flat[:, 288:304]
        else:
            cal = [self._np(c) for c in cal]
            aug = self._np(aug)
        aug = aug.reshape(B, 4, 4)
        if not np.array_equal(aug, np.broadcast_to(np.eye(4, dtype=aug.dtype), aug.shape)):
            raise NotImplementedError("lidar_aug_matrix must be the identity (augmentation is disabled on this path)")
        key = b"".join(np.ascontiguousarray(c, np.float32).tobytes() for c in cal)
        cam_mats = self._cal_cache.get(key)
        if cam_mats is None:          # calibration repeats from frame to frame within a scene
            cam_mats = camera_matrices(*cal)
            if len(self._cal_cache) > 256:
                self._cal_cache.clear()
            self._cal_cache[key] = cam_mats
        plan = self.engine.plan_arrays(
            bounds.astype(np.int64), stride, xyz_offset, cam_mats, self._np(det_boxes).astype(np.float32).reshape(-1, 4),
            self._np(det_labels).astype(np.int64), self._np(det_scores).astype(np.float32),
            self._np(det_batch_idx).astype(np.int64), self._np(det_cam_idx).astype(np.int64))
        res = self.engine.result(self.engine.execute(plan, pts))
        boxes, labels, scores, bi = [], [], [], []
        for b, fr in enumerate(res["frames"]):
            boxes.append(fr["pred_boxes"]); labels.append(fr["pred_labels"]); scores.append(fr["pred_scores"])
            bi.append(np.full(fr["pred_labels"].shape[0], b, np.int64))
        proposal_boxes = torch.from_numpy(np.concatenate(boxes).reshape(-1, 7)).to(dev)
        return (proposal_boxes, torch.from_numpy(np.concatenate(labels).astype(np.int64)),
                torch.from_numpy(np.concatenate(scores).astype(np.float32)), torch.from_numpy(np.concatenate(bi)))

    def get_bboxes(self, batch_dict):
        boxes, labels, scores, bidx = self.get_proposals(batch_dict)
        ret = []
        for k in range(batch_dict['batch_size']):
            mask = (bidx == k)
            ret.append(dict(pred_boxes=boxes[mask.to(boxes.device)], pred_scores=scores[mask],
                            pred_labels=labels[mask].int()))
        return ret

    def forward(self, batch_dict):
        batch_dict['final_box_dicts'] = self.get_bboxes(batch_dict)
        assert not self.training, "not trainable!"
        return batch_dict


class FrustumProposerOGKITTI(nn.Module):
    """The KITTI single-camera Greedy Box Seeker head with the reference's constructor signature and
    ``get_proposals`` / ``get_bboxes`` / ``forward`` contract (frustum_proposals_v1_kitti.py:38-48, 292-690, 709-740),
    on the fused stages in their KITTI variant (include/fnp.h FNP_VARIANT_KITTI): CalibrationTorch's two-step
    projection without an on-image test, x-y-w-h boxes, seven anchors, max_dist 70, ONE batched first-match
    ``points_in_boxes_gpu`` per frustum, densities over their sum, ``score = dns_w + density + iou_w iou + dst_w dist``,
    ``nms_normal`` + ``topk``.  ``batch_dict``: ``points`` (N, 1+3+) with the batch index in column 0, ``calib`` a list
    of objects with ``P2``, ``R0``, ``V2C`` (pcdet.utils.calibration_kitti.Calibration), ``batch_size``."""

    def __init__(self, model_cfg=None, input_channels=None, num_class=None, class_names=None, grid_size=None,
                 point_cloud_range=None, voxel_size=None, predict_boxes_when_training=True,
                 lq=0.336, uq=0.356, iou_w=0.95, dst_w=0.226, dns_w=0.05, min_cam_iou=0.3, size_min=0.957,
                 size_max=1.2, ry_min=0.0, ry_max=torch.pi, cq=0.46, num_mags=6, max_dist=70, num_sizes=4,
                 num_rotations=10, topk=1, nms_2d=0.7, nms_3d=1.0, score_thr=0.1, nms_normal=0.7, clamp_bottom=0,
                 image_detector=None, device=None):
        super().__init__()
        p = dict(lq=lq, uq=uq, iou_w=iou_w, dst_w=dst_w, dns_w=dns_w, min_cam_iou=min_cam_iou, size_min=size_min,
                 size_max=size_max, ry_min=ry_min, ry_max=float(ry_max), cq=cq, num_mags=num_mags, max_dist=max_dist,
                 num_sizes=num_sizes, num_rotations=num_rotations, topk=topk, nms_2d=nms_2d, nms_3d=nms_3d,
                 score_thr=score_thr, nms_normal=nms_normal, clamp_bottom=0)      # the argument is ignored (:62)
        params = _cfg_get(model_cfg, 'PARAMS')
        if params is not None:                       # PARAMS override the defaults (:68-98)
            for k in list(DEFAULTS) + ['aln_w', 'ego_w', 'occl_w', 'rand_center', 'search_depth']:
                if k in params:
                    p[k] = params[k]
        if _cfg_get(model_cfg, 'SAVE_BLEND', False):
            raise NotImplementedError("SAVE_BLEND (Blender visualisation dumps) is outside the Box Seeker path")
        assert p['nms_3d'] == 0, 'DO NOT USE!'          # the reference's own assertion (:114)
        # aln_w / ego_w / occl_w and the MULT / OCCL_MULT / MULTICAM_IOU switches are read by that constructor and never
        # used by its get_proposals: ignored here as there
        p['aln_w'] = p['ego_w'] = p['occl_w'] = 0
        self.params = p
        self.image_size = [900, 1600]
        self.topk, self.score_thr, self.max_dist = p['topk'], p['score_thr'], p['max_dist']
        self.num_mags, self.num_sizes, self.num_rotations = p['num_mags'], p['num_sizes'], p['num_rotations']
        if image_detector is not None:
            self.image_detector = image_detector
        else:
            preds_path = _cfg_get(model_cfg, 'PREDS_PATH', '/home/uqdetche/GLIP/OWL_PREDEFINED_MMDETCOCO_val_kitti.coco.json')
            self.image_detector = PreprocessedDetector([preds_path], class_names=class_names)
        self.engine = SeekerEngine(p, device=device, box_format='xywh', variant='kitti')
        self.base_boxes = self.engine.base_boxes
        self.base_corners = self.engine.base_corners

    def get_proposals(self, batch_dict):
        """-> (proposal_boxes (K,7) f32 on the GPU, frust_labels (K) int64 CPU, frust_scores (K) f32 CPU,
        frust_batch_idx (K) int64 CPU), as frustum_proposals_v1_kitti.py:676-690."""
        from .seeker import KittiFrameInput
        B = int(batch_dict['batch_size'])
        det_boxes, det_labels, det_scores, det_batch_idx, det_cam_idx = self.image_detector(batch_dict)
        det_boxes, det_labels = FrustumProposerOG._np(det_boxes), FrustumProposerOG._np(det_labels)
        det_scores, det_batch_idx = FrustumProposerOG._np(det_scores), FrustumProposerOG._np(det_batch_idx)
        det_cam_idx = FrustumProposerOG._np(det_cam_idx)
        pts = batch_dict['points']
        dev = self.engine.device
        if isinstance(pts, np.ndarray):
            pts = torch.from_numpy(np.ascontiguousarray(pts, np.float32))
        pts = pts.to(dev, dtype=torch.float32).contiguous()
        bidx = pts[:, 0].contiguous()
        if bidx.numel() > 1 and not bool((bidx[1:] >= bidx[:-1]).all()):
            raise ValueError("batch_dict['points'] must be grouped by batch index (collate_batch order)")
        bounds = torch.searchsorted(bidx, torch.arange(B + 1, device=dev, dtype=torch.float32)).cpu().numpy()
        frames = []
        for b in range(B):
            cal = batch_dict['calib'][b]
            m = (det_batch_idx == b) & (det_cam_idx == 0)           # c = 0 only (:336-337)
            n = int(bounds[b + 1] - bounds[b])
            frames.append(KittiFrameInput(points=np.empty((n, int(pts.shape[1])), np.float32), P2=cal.P2, R0=cal.R0, V2C=cal.V2C,
                                          det_boxes=det_boxes[m], det_labels=det_labels[m], det_scores=det_scores[m],
                                          device=str(dev)))
        plan = self.engine.plan(frames, xyz_offset=1, stride=int(pts.shape[1]))
        res = self.engine.result(self.engine.execute(plan, pts))
        boxes, labels, scores, bi = [], [], [], []
        for b, fr in enumerate(res["frames"]):
            boxes.append(fr["pred_boxes"]); labels.append(fr["pred_labels"]); scores.append(fr["pred_scores"])
            bi.append(np.full(fr["pred_labels"].shape[0], b, np.int64))
        proposal_boxes = torch.from_numpy(np.concatenate(boxes).reshape(-1, 7)).to(dev)
        return (proposal_boxes, torch.from_numpy(np.concatenate(labels).astype(np.int64)),
                torch.from_numpy(np.concatenate(scores).astype(np.float32)), torch.from_numpy(np.concatenate(bi)))

    def get_bboxes(self, batch_dict):
        boxes, labels, scores, bidx = self.get_proposals(batch_dict)
        ret = []
        for k in range(batch_dict['batch_size']):
            mask = (bidx == k)
            ret.append(dict(pred_boxes=boxes[mask.to(boxes.device)], pred_scores=scores[mask],
                            pred_labels=labels[mask].int()))
        return ret

    def forward(self, batch_dict):
        batch_dict['final_box_dicts'] = self.get_bboxes(batch_dict)
        assert not self.training, "not trainable!"
        return batch_dict
