"""KITTI batch_dict producer for the KITTI Box Seeker head (``FrustumProposerOGKITTI``), the counterpart of
``nuscenes_feed.NuScenesFeed``: what OpenPCDet v0.6's ``KittiDataset`` hands to the head in the mode the reference's
tools/extract_pseudo_labels.py builds its loader in (training=True, an empty augmentation list), produced from the
same files (``kitti_infos_<split>.pkl``, ``<split root>/velodyne/<idx>.bin``, ``<split root>/calib/<idx>.txt``).

reference (OpenPCDet v0.6)                                          here
------------------------------------------------------------------  ---------------------------------------
kitti_dataset.py KittiDataset.__init__ / root_split_path           KittiFeed.__init__ (training / testing)
KittiDataset.get_lidar                                              KittiFeed.lidar
KittiDataset.get_calib, calibration_kitti.get_calib_from_file      KittiFeed.calib, get_calib_from_file
calibration_kitti.Calibration (numpy: lidar_to_rect, rect_to_img,  Calibration
  rect_to_lidar)
KittiDataset.get_fov_flag (FOV_POINTS_ONLY)                         fov_flag
common_utils.drop_info_with_name (DontCare)                        KittiFeed._load_gt
box_utils.boxes3d_kitti_camera_to_lidar                             boxes3d_kitti_camera_to_lidar
box_utils.boxes3d_lidar_to_kitti_camera,                            boxes3d_lidar_to_kitti_camera,
  boxes3d_to_corners3d_kitti_camera,                                  boxes3d_to_corners3d_kitti_camera,
  boxes3d_kitti_camera_to_imageboxes                                  boxes3d_kitti_camera_to_imageboxes
KittiDataset.__getitem__                                            KittiFeed.__getitem__
DatasetTemplate.prepare_data, training mode with an empty           KittiFeed._prepare_gt (NuScenesFeed's)
  augmentation list: heading wrap, class filter, class column,        and __getitem__: x / y range mask of the
  REMOVE_OUTSIDE_BOXES by centre, SKIP_NO_GT re-draw                  points, SKIP_NO_GT
DatasetTemplate.collate_batch                                       nuscenes_feed.collate_batch

The FOV filter stays on the host, in numpy float32 with the numpy Calibration's arithmetic: the reference forms it
with numpy's float32 BLAS, and a restatement on the device could not promise the same bits for points on the image
border.  The KITTI head has no on-image test of its own (DESIGN.md section 4) and relies on this filter.

``shuffle_points`` (DataProcessor, enabled for training in the KITTI dataset configs) is not applied: no output of
the seeker depends on the order of the points (DESIGN.md sections 2 and 3), so the frames are served in file order.
"""
import copy
import pickle
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path
from typing import Iterable, Sequence

import numpy as np

from .nuscenes_feed import NuScenesFeed, mask_points_by_range

CLASS_NAMES = ['Car', 'Pedestrian', 'Cyclist']                     # OpenPCDet's KITTI configs
POINT_CLOUD_RANGE = [0, -40, -3, 70.4, 40, 1]                       # kitti_dataset.yaml


def get_calib_from_file(calib_file) -> dict:
    """calibration_kitti.get_calib_from_file: lines 2 / 3 / 4 / 5 of the file (0-based) are P2, P3 (3,4), R0_rect (3,3)
    and Tr_velo_to_cam (3,4), each after its ``name:`` field, float32."""
    with open(calib_file) as f:
        lines = f.readlines()
    rows = [np.array(lines[k].strip().split(' ')[1:], dtype=np.float32) for k in (2, 3, 4, 5)]
    return {'P2': rows[0].reshape(3, 4), 'P3': rows[1].reshape(3, 4), 'R0': rows[2].reshape(3, 3),
            'Tr_velo2cam': rows[3].reshape(3, 4)}


class Calibration:
    """calibration_kitti.Calibration, the numpy methods the loader calls, with its float32 arithmetic."""

    def __init__(self, calib):
        calib = calib if isinstance(calib, dict) else get_calib_from_file(calib)
        self.P2, self.R0, self.V2C = calib['P2'], calib['R0'], calib['Tr_velo2cam']

    @staticmethod
    def cart_to_hom(pts):
        return np.hstack((pts, np.ones((pts.shape[0], 1), dtype=np.float32)))

    def lidar_to_rect(self, pts_lidar):
        return np.dot(self.cart_to_hom(pts_lidar), np.dot(self.V2C.T, self.R0.T))

    def rect_to_img(self, pts_rect):
        """(u, v) (N,2) and the depth in the rectified camera frame (N,)."""
        hom = self.cart_to_hom(pts_rect)
        pts_2d = np.dot(hom, self.P2.T)
        return (pts_2d[:, 0:2].T / hom[:, 2]).T, pts_2d[:, 2] - self.P2.T[3, 2]

    def rect_to_lidar(self, pts_rect):
        r0 = np.vstack((np.hstack((self.R0, np.zeros((3, 1), dtype=np.float32))), np.zeros((1, 4), dtype=np.float32)))
        r0[3, 3] = 1
        v2c = np.vstack((self.V2C, np.zeros((1, 4), dtype=np.float32)))
        v2c[3, 3] = 1
        return np.dot(self.cart_to_hom(pts_rect), np.linalg.inv(np.dot(r0, v2c).T))[:, 0:3]


def fov_flag(points: np.ndarray, img_shape, calib: Calibration) -> np.ndarray:
    """KittiDataset.get_fov_flag on calib.lidar_to_rect(points[:, :3]): 0 <= u < W, 0 <= v < H and depth >= 0, with
    (H, W) = img_shape."""
    pts_img, depth = calib.rect_to_img(calib.lidar_to_rect(points[:, 0:3]))
    on_img = (pts_img[:, 0] >= 0) & (pts_img[:, 0] < img_shape[1]) & (pts_img[:, 1] >= 0) & (pts_img[:, 1] < img_shape[0])
    return on_img & (depth >= 0)


def boxes3d_kitti_camera_to_lidar(boxes3d_camera: np.ndarray, calib: Calibration) -> np.ndarray:
    """(N,7) [x, y, z, l, h, w, ry] in the rectified camera frame (z at the bottom) -> (N,7) [x, y, z, l, w, h, heading]
    in the LiDAR frame (z at the centre)."""
    b = copy.deepcopy(boxes3d_camera)
    xyz, r = b[:, 0:3], b[:, 6:7]
    l, h, w = b[:, 3:4], b[:, 4:5], b[:, 5:6]
    xyz_lidar = calib.rect_to_lidar(xyz)
    xyz_lidar[:, 2] += h[:, 0] / 2
    return np.concatenate([xyz_lidar, l, w, h, -(r + np.pi / 2)], axis=-1)


def boxes3d_lidar_to_kitti_camera(boxes3d_lidar: np.ndarray, calib: Calibration) -> np.ndarray:
    """box_utils.boxes3d_lidar_to_kitti_camera, the inverse of boxes3d_kitti_camera_to_lidar: (N,7) [x, y, z, dx, dy,
    dz, heading] in the LiDAR frame -> (N,7) [x, y, z, l, h, w, ry] in the rectified camera frame, z at the bottom."""
    b = copy.deepcopy(boxes3d_lidar)
    xyz_lidar = b[:, 0:3]
    l, w, h = b[:, 3:4], b[:, 4:5], b[:, 5:6]
    r = b[:, 6:7]
    xyz_lidar[:, 2] -= h.reshape(-1) / 2
    xyz_cam = calib.lidar_to_rect(xyz_lidar)
    r = -r - np.pi / 2
    return np.concatenate([xyz_cam, l, h, w, r], axis=-1)


def boxes3d_to_corners3d_kitti_camera(boxes3d: np.ndarray) -> np.ndarray:
    """box_utils.boxes3d_to_corners3d_kitti_camera (bottom_center=True): (N,7) camera boxes -> (N,8,3) float32."""
    n = boxes3d.shape[0]
    l, h, w = boxes3d[:, 3], boxes3d[:, 4], boxes3d[:, 5]
    x_corners = np.array([l / 2., l / 2., -l / 2., -l / 2., l / 2., l / 2., -l / 2., -l / 2], dtype=np.float32).T
    z_corners = np.array([w / 2., -w / 2., -w / 2., w / 2., w / 2., -w / 2., -w / 2., w / 2.], dtype=np.float32).T
    y_corners = np.zeros((n, 8), dtype=np.float32)
    y_corners[:, 4:8] = -h.reshape(n, 1).repeat(4, axis=1)
    ry = boxes3d[:, 6]
    zeros, ones = np.zeros(ry.size, dtype=np.float32), np.ones(ry.size, dtype=np.float32)
    rot_list = np.array([[np.cos(ry), zeros, -np.sin(ry)],
                         [zeros, ones, zeros],
                         [np.sin(ry), zeros, np.cos(ry)]])                      # (3, 3, N)
    R_list = np.transpose(rot_list, (2, 0, 1))                                   # (N, 3, 3)
    temp_corners = np.concatenate((x_corners.reshape(-1, 8, 1), y_corners.reshape(-1, 8, 1),
                                   z_corners.reshape(-1, 8, 1)), axis=2)         # (N, 8, 3)
    rotated = np.matmul(temp_corners, R_list)
    x = boxes3d[:, 0].reshape(-1, 1) + rotated[:, :, 0].reshape(-1, 8)
    y = boxes3d[:, 1].reshape(-1, 1) + rotated[:, :, 1].reshape(-1, 8)
    z = boxes3d[:, 2].reshape(-1, 1) + rotated[:, :, 2].reshape(-1, 8)
    corners = np.concatenate((x.reshape(-1, 8, 1), y.reshape(-1, 8, 1), z.reshape(-1, 8, 1)), axis=2)
    return corners.astype(np.float32)


def boxes3d_kitti_camera_to_imageboxes(boxes3d: np.ndarray, calib: Calibration, image_shape=None) -> np.ndarray:
    """box_utils.boxes3d_kitti_camera_to_imageboxes: the (N,4) [u1, v1, u2, v2] image box around the eight corners of
    each (N,7) camera box; with image_shape (H, W), u clipped to [0, W-1] and v to [0, H-1]."""
    corners3d = boxes3d_to_corners3d_kitti_camera(boxes3d)
    pts_img, _ = calib.rect_to_img(corners3d.reshape(-1, 3))
    corners_in_image = pts_img.reshape(-1, 8, 2)
    boxes2d_image = np.concatenate([np.min(corners_in_image, axis=1), np.max(corners_in_image, axis=1)], axis=1)
    if image_shape is not None:
        boxes2d_image[:, 0] = np.clip(boxes2d_image[:, 0], a_min=0, a_max=image_shape[1] - 1)
        boxes2d_image[:, 1] = np.clip(boxes2d_image[:, 1], a_min=0, a_max=image_shape[0] - 1)
        boxes2d_image[:, 2] = np.clip(boxes2d_image[:, 2], a_min=0, a_max=image_shape[1] - 1)
        boxes2d_image[:, 3] = np.clip(boxes2d_image[:, 3], a_min=0, a_max=image_shape[0] - 1)
    return boxes2d_image


class KittiFeed:
    """Map-style producer of the KITTI head's per-frame ``data_dict`` in training mode (the extraction tool's):
    GT headings wrapped to [-pi, pi), GT outside the classes or with its centre outside POINT_CLOUD_RANGE dropped, and
    a frame left without GT replaced by a randomly drawn one (SKIP_NO_GT)."""

    def __init__(self, root_path, infos, split: str = 'train', class_names: Sequence[str] = CLASS_NAMES,
                 point_cloud_range=POINT_CLOUD_RANGE, fov_points_only: bool = True, training: bool = True,
                 skip_no_gt: bool = True, rng=None, device=None):
        """root_path: DATA_PATH; infos: list of info dicts, or path(s) of kitti_infos_*.pkl files relative to it.
        split: DATA_SPLIT['train'] ('test' reads testing/, anything else training/).  device: where the frames'
        calibration blocks are formed (the engine's device; None: the current CUDA device).  rng: private generator
        for the SKIP_NO_GT re-draw (None: numpy's global one, as in the reference)."""
        self.root = Path(root_path)
        self.root_split_path = self.root / ('training' if split != 'test' else 'testing')
        if isinstance(infos, (str, Path)):
            infos = [infos]
        if len(infos) and isinstance(infos[0], (str, Path)):
            loaded = []
            for p in infos:
                with open(p if Path(p).is_absolute() else self.root / p, 'rb') as f:
                    loaded.extend(pickle.load(f))
            infos = loaded
        self.infos = list(infos)
        self.class_names = list(class_names)
        self.range = np.asarray(point_cloud_range, dtype=np.float32)
        self.fov_points_only = bool(fov_points_only)
        self.training, self.skip_no_gt = bool(training), bool(skip_no_gt)
        self.rng = rng
        self.device = device

    # the training-mode GT steps are NuScenesFeed's (limit_period, mask_boxes_outside_range) on the same attributes:
    # training, class_names, range
    _prepare_gt = NuScenesFeed._prepare_gt

    def __len__(self):
        return len(self.infos)

    @staticmethod
    def frame_id(info: dict) -> str:
        return info['point_cloud']['lidar_idx']

    def lidar_path(self, idx: str) -> Path:
        return self.root_split_path / 'velodyne' / ('%s.bin' % idx)

    def calib_path(self, idx: str) -> Path:
        return self.root_split_path / 'calib' / ('%s.txt' % idx)

    def lidar(self, idx: str) -> np.ndarray:
        return np.fromfile(str(self.lidar_path(idx)), dtype=np.float32).reshape(-1, 4)

    def calib(self, idx: str) -> Calibration:
        return Calibration(str(self.calib_path(idx)))

    def _load_gt(self, info: dict, calib: Calibration, d: dict):
        """The info's annotations without DontCare, in the LiDAR frame, into d."""
        if 'annos' not in info:
            return
        annos = info['annos']
        keep = [i for i, n in enumerate(annos['name']) if n != 'DontCare']
        annos = {k: v[keep] for k, v in annos.items()}
        boxes_camera = np.concatenate([annos['location'], annos['dimensions'], annos['rotation_y'][..., np.newaxis]],
                                      axis=1).astype(np.float32)
        d['gt_names'] = annos['name']
        d['gt_boxes'] = boxes3d_kitti_camera_to_lidar(boxes_camera, calib)

    def __getitem__(self, index: int) -> dict:
        info = copy.deepcopy(self.infos[index])
        idx = self.frame_id(info)
        img_shape = info['image']['image_shape']
        calib = self.calib(idx)
        d = {'frame_id': idx, 'calib': calib}
        self._load_gt(info, calib, d)
        points = self.lidar(idx)
        if self.fov_points_only:
            points = points[fov_flag(points, img_shape, calib)]
        d['points'] = points
        self._prepare_gt(d)
        d['use_lead_xyz'] = True
        d['points'] = d['points'][mask_points_by_range(d['points'], self.range)]
        if self.training and len(d['gt_boxes']) == 0 and self.skip_no_gt:    # dataset.py:213-215
            return self[int((np.random if self.rng is None else self.rng).randint(len(self)))]
        d.pop('gt_names', None)
        d['image_shape'] = img_shape
        return d

    def gt_boxes(self, index: int) -> np.ndarray:
        """The frame's (G,8) gt_boxes as ``self[index]`` produces them, reading its calibration but not its velodyne
        file.  A frame left without GT gives an empty array: no other frame is drawn in its place (SKIP_NO_GT), because
        a caller that scores frame by frame must see this frame's GT."""
        info = self.infos[index]
        if 'annos' not in info:
            return np.zeros((0, 8), np.float32)
        d = {}
        self._load_gt(info, self.calib(self.frame_id(info)), d)
        self._prepare_gt(d)
        return d['gt_boxes']

    # ---------------------------------------------------------------- seeker inputs
    def frame_input(self, index: int, detector, xyz_only: bool = False):
        """One frame as SeekerEngine(variant="kitti") wants it: a KittiFrameInput of ``self[index]`` with the 2D boxes
        ``detector`` (proposer.PreprocessedDetector) gives its frame id (infer_kitti), on ``self.device``."""
        import torch
        from .seeker import KittiFrameInput
        d = self[index]
        if xyz_only:
            d['points'] = np.ascontiguousarray(d['points'][:, :3], np.float32)
        boxes, labels, scores, _, _ = detector({'batch_size': 1, 'frame_id': [d['frame_id']]})
        cal = d['calib']
        device = self.device if self.device is not None else torch.device('cuda', torch.cuda.current_device())
        fi = KittiFrameInput(points=np.ascontiguousarray(d['points'], np.float32), P2=cal.P2, R0=cal.R0, V2C=cal.V2C,
                             det_boxes=np.asarray(boxes, np.float32).reshape(-1, 4),
                             det_labels=np.asarray(labels, np.int64).reshape(-1),
                             det_scores=np.asarray(scores, np.float32).reshape(-1), gt_boxes=d['gt_boxes'],
                             device=str(device))
        return fi, d['frame_id'], {'frame_id': d['frame_id']}

    def prefetch(self, indices: Iterable[int], detector, batch_frames: int = 32, workers: int = 4,
                 xyz_only: bool = False):
        """Yields (frame_inputs, frame_ids, metadata) per batch of ``batch_frames`` frames, loading the next batch on
        worker threads while the caller runs the current one (NuScenesFeed.prefetch)."""
        idx = list(indices)
        batches = [idx[i:i + batch_frames] for i in range(0, len(idx), batch_frames)]
        if not batches:
            return
        with ThreadPoolExecutor(max_workers=max(1, workers)) as pool:
            def submit(b):
                return [pool.submit(self.frame_input, i, detector, xyz_only) for i in b]
            pending = submit(batches[0])
            for k in range(len(batches)):
                nxt = submit(batches[k + 1]) if k + 1 < len(batches) else None
                got = [f.result() for f in pending]
                yield [g[0] for g in got], [g[1] for g in got], [g[2] for g in got]
                pending = nxt
