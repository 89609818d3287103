"""nuScenes batch_dict producer for the Box Seeker path (SURVEY.md section 8, row f2).

The step immediately before the path: what the reference's dataset / collate code hands to
``FrustumProposerOG.get_proposals``, produced from the same files (``nuscenes_infos_*.pkl`` info
dicts, ``samples/LIDAR_TOP/*.bin`` point files, camera calibration), for the option set of
tools/cfgs/nuscenes_box_seeker_proposals.yaml + cfgs/dataset_configs/nuscenes_dataset.yaml
(test mode: no augmentation, no shuffling, CAM_WITHOUT_IMAGE).

reference                                                          here
-----------------------------------------------------------------  --------------------------
NuScenesDataset.get_sweep (nuscenes_dataset.py:85-103)             load_sweep
NuScenesDataset.get_lidar_with_sweeps (:105-124)                   lidar_with_sweeps
NuScenesDataset.load_camera_info (:172-233, CAM_WITHOUT_IMAGE)     camera_info
NuScenesDataset.__getitem__ (:241-279)                             NuScenesFeed.__getitem__
DatasetTemplate.prepare_data (dataset.py:159-220)                  NuScenesFeed._prepare
  test mode, and the mode the extraction tool really runs in:        training=True
  tools/extract_pseudo_labels.py:47-58 builds its loader with
  training=True and an EMPTY augmentation list, so that
  DataAugmentor.forward (data_augmentor.py:362-395) only wraps the
  headings, REMOVE_OUTSIDE_BOXES drops GT whose centre is outside
  POINT_CLOUD_RANGE (data_processor.py:88-93, box_utils.py:93-114)
  and frames left without GT are re-drawn (SKIP_NO_GT, dataset.py:
  23,213-215)
  DataProcessor.mask_points_and_boxes_outside_range                  (data_processor.py:80-94,
  (shuffle disabled, yaml:46-50)                                      common_utils.py:78-81)
DatasetTemplate.collate_batch (dataset.py:222-344)                 collate_batch
load_data_to_gpu (pcdet/models/__init__.py:23-36)                  seeker.HostPointFeeder

Everything here is host-side file reading and numpy bookkeeping (the reference does it in
DataLoader worker processes); ``prefetch`` overlaps it with the GPU by loading the next batch
of frames on worker threads.  The device side starts at SeekerEngine / HostPointFeeder.
"""
import copy
import pickle
from collections import defaultdict
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path
from typing import Iterable, List, Optional, Sequence

import numpy as np

CLASS_NAMES = ['car', 'truck', 'construction_vehicle', 'bus', 'trailer', 'barrier', 'motorcycle', 'bicycle',
               'pedestrian', 'traffic_cone']                       # nuscenes_box_seeker_proposals.yaml:1-2
POINT_CLOUD_RANGE = [-54.0, -54.0, -5.0, 54.0, 54.0, 3.0]          # yaml:8


def quaternion_rotation_matrix(q: Sequence[float]) -> np.ndarray:
    """Rotation matrix of a (w, x, y, z) quaternion, normalised first -- what
    ``pyquaternion.Quaternion(q).rotation_matrix`` returns (nuscenes_dataset.py:209-211)."""
    q = np.asarray(q, dtype=np.float64)
    q = q / np.linalg.norm(q)
    w, x, y, z = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def remove_ego_points(points: np.ndarray, center_radius: float = 1.0) -> np.ndarray:
    """nuscenes_dataset.py:88-91."""
    mask = ~((np.abs(points[:, 0]) < center_radius) & (np.abs(points[:, 1]) < center_radius))
    return points[mask]


def load_sweep(root: Path, sweep_info: dict):
    """One earlier sweep in the key frame's LiDAR frame: (n,4) points and (n,1) time lags
    (nuscenes_dataset.py:85-103)."""
    pts = np.fromfile(str(root / sweep_info['lidar_path']), dtype=np.float32, count=-1).reshape([-1, 5])[:, :4]
    pts = remove_ego_points(pts).T
    if sweep_info['transform_matrix'] is not None:
        n = pts.shape[1]
        pts[:3, :] = sweep_info['transform_matrix'].dot(np.vstack((pts[:3, :], np.ones(n))))[:3, :]
    times = sweep_info['time_lag'] * np.ones((1, pts.shape[1]))
    return pts.T, times.T


def draw_sweeps(info: dict, max_sweeps: int = 1, rng=None) -> np.ndarray:
    """Indices into ``info['sweeps']`` of the max_sweeps - 1 earlier sweeps a frame reads, drawn without replacement
    (nuscenes_dataset.py:105-124; the reference draws from the global numpy generator, pass ``rng`` for a private one)."""
    rng = np.random if rng is None else rng
    return rng.choice(len(info['sweeps']), max_sweeps - 1, replace=False)


def read_lidar_with_sweeps(root: Path, info: dict, sweep_ids) -> np.ndarray:
    """(N,5) float32 [x, y, z, intensity, time]: the key frame followed by the sweeps ``sweep_ids`` (draw_sweeps)."""
    points = np.fromfile(str(root / info['lidar_path']), dtype=np.float32, count=-1).reshape([-1, 5])[:, :4]
    pts_list = [points]
    times_list = [np.zeros((points.shape[0], 1))]
    for k in sweep_ids:
        p, t = load_sweep(root, info['sweeps'][k])
        pts_list.append(p)
        times_list.append(t)
    points = np.concatenate(pts_list, axis=0)
    times = np.concatenate(times_list, axis=0).astype(points.dtype)
    return np.concatenate((points, times), axis=1)


def lidar_with_sweeps(root: Path, info: dict, max_sweeps: int = 1, rng=None) -> np.ndarray:
    """(N,5) float32 [x, y, z, intensity, time]: the key frame followed by max_sweeps - 1 earlier
    sweeps drawn without replacement (nuscenes_dataset.py:105-124; the reference draws from the
    global numpy generator, pass ``rng`` for a private one)."""
    return read_lidar_with_sweeps(root, info, draw_sweeps(info, max_sweeps, rng))


def camera_info(info: dict) -> dict:
    """Camera matrices of a frame, one (4,4) float32 per camera in ``info['cams']`` order
    (nuscenes_dataset.py:172-218); no images are opened (CAM_WITHOUT_IMAGE, yaml:17)."""
    out = {k: [] for k in ("image_paths", "lidar2camera", "lidar2image", "camera2ego", "camera_intrinsics",
                           "camera2lidar")}
    for _, cam in info["cams"].items():
        out["image_paths"].append(cam["data_path"])
        lidar2camera_r = np.linalg.inv(cam["sensor2lidar_rotation"])
        lidar2camera_t = cam["sensor2lidar_translation"] @ lidar2camera_r.T
        lidar2camera_rt = np.eye(4).astype(np.float32)
        lidar2camera_rt[:3, :3] = lidar2camera_r.T
        lidar2camera_rt[3, :3] = -lidar2camera_t
        out["lidar2camera"].append(lidar2camera_rt.T)
        K = np.eye(4).astype(np.float32)
        K[:3, :3] = cam["camera_intrinsics"]
        out["camera_intrinsics"].append(K)
        out["lidar2image"].append(K @ lidar2camera_rt.T)
        camera2ego = np.eye(4).astype(np.float32)
        camera2ego[:3, :3] = quaternion_rotation_matrix(cam["sensor2ego_rotation"])
        camera2ego[:3, 3] = cam["sensor2ego_translation"]
        out["camera2ego"].append(camera2ego)
        camera2lidar = np.eye(4).astype(np.float32)
        camera2lidar[:3, :3] = cam["sensor2lidar_rotation"]
        camera2lidar[:3, 3] = cam["sensor2lidar_translation"]
        out["camera2lidar"].append(camera2lidar)
    return out


def mask_points_by_range(points: np.ndarray, limit_range) -> np.ndarray:
    """x / y window, both ends included (common_utils.py:78-81)."""
    return (points[:, 0] >= limit_range[0]) & (points[:, 0] <= limit_range[3]) \
        & (points[:, 1] >= limit_range[1]) & (points[:, 1] <= limit_range[4])


def collate_batch(batch_list: List[dict]) -> dict:
    """DatasetTemplate.collate_batch (dataset.py:222-344) for the keys this path produces:
    points get a leading batch-index column, gt_boxes are zero-padded to the longest frame,
    img_process_infos are concatenated, everything else is stacked."""
    data = defaultdict(list)
    for sample in batch_list:
        for k, v in sample.items():
            data[k].append(v)
    ret = {}
    for key, val in data.items():
        if key == 'points':
            ret[key] = np.concatenate([np.pad(p, ((0, 0), (1, 0)), mode='constant', constant_values=i)
                                       for i, p in enumerate(val)], axis=0)
        elif key == 'gt_boxes':
            max_gt = max(len(x) for x in val)
            out = np.zeros((len(batch_list), max_gt, val[0].shape[-1]), dtype=np.float32)
            for k in range(len(batch_list)):
                out[k, :len(val[k]), :] = val[k]
            ret[key] = out
        elif key == 'img_process_infos':
            ret[key] = [x for v in val for x in v]
        else:
            ret[key] = np.stack(val, axis=0)
    ret['batch_size'] = len(batch_list)
    return ret


def limit_period(val: np.ndarray, offset: float = 0.5, period: float = np.pi) -> np.ndarray:
    """common_utils.py:21-24 (the reference computes it through a float32 torch tensor; so does this)."""
    import torch
    v = torch.from_numpy(np.ascontiguousarray(val)).float()
    return (v - torch.floor(v / period + offset) * period).numpy()


def mask_boxes_outside_range(boxes: np.ndarray, limit_range) -> np.ndarray:
    """box_utils.mask_boxes_outside_range_numpy with USE_CENTER_TO_FILTER (its default, box_utils.py:93-107):
    keep a box when its centre lies inside the range, both ends included."""
    c = boxes[:, 0:3]
    return ((c >= limit_range[0:3]) & (c <= limit_range[3:6])).all(axis=-1)


class NuScenesFeed:
    """Map-style producer of the seeker's per-frame ``data_dict``.

    training=False is the reference's test mode; training=True is the mode tools/extract_pseudo_labels.py
    builds its loader in (:47-58, with an empty augmentation list): GT headings are wrapped to [-pi, pi), GT
    boxes whose centre is outside POINT_CLOUD_RANGE are dropped, and a frame left without GT is replaced by
    a randomly drawn one (SKIP_NO_GT).  The points and camera matrices -- everything the proposals depend on --
    are the same in both modes; what changes is the gt_boxes the recall counters see."""

    def __init__(self, root_path, infos, class_names: Sequence[str] = CLASS_NAMES, max_sweeps: int = 1,
                 point_cloud_range=POINT_CLOUD_RANGE, filter_min_points_in_gt: int = 1, pred_velocity: bool = True,
                 set_nan_velocity_to_zeros: bool = True, final_dim=(900, 1600), resize_lim_test=(1.0, 1.0), rng=None,
                 training: bool = False, skip_no_gt: bool = True):
        """infos: list of info dicts, or path(s) of nuscenes_infos_*.pkl files (nuscenes_dataset.py:39-51).
        max_sweeps: MAX_SWEEPS (1 in the seeker yaml:12, 10 in the dataset base config).
        rng: private generator for the sweep draw and the SKIP_NO_GT re-draw (None: numpy's global one, as in
        the reference)."""
        self.training, self.skip_no_gt = bool(training), bool(skip_no_gt)
        self.root = Path(root_path)
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
        self.max_sweeps = int(max_sweeps)
        self.range = np.asarray(point_cloud_range, dtype=np.float32)
        self.filter_min_points_in_gt = filter_min_points_in_gt
        self.pred_velocity = pred_velocity
        self.set_nan_velocity_to_zeros = set_nan_velocity_to_zeros
        self.final_dim, self.resize_lim_test = tuple(final_dim), tuple(resize_lim_test)
        self.rng = rng

    def __len__(self):
        return len(self.infos)

    def _load_gt(self, info: dict, d: dict):
        """The info's GT with the min-points filter (nuscenes_dataset.py:252-258) into d."""
        if 'gt_boxes' in info:
            mask = (info['num_lidar_pts'] > self.filter_min_points_in_gt - 1) if self.filter_min_points_in_gt else None
            d['gt_names'] = info['gt_names'] if mask is None else info['gt_names'][mask]
            d['gt_boxes'] = info['gt_boxes'] if mask is None else info['gt_boxes'][mask]

    def _prepare_gt(self, d: dict):
        """The GT part of _prepare: class filter, class column, and in training mode the heading wrap and the range
        filter."""
        if self.training:
            assert 'gt_boxes' in d, 'gt_boxes should be provided for training'      # dataset.py:182
            # DataAugmentor.forward with an empty queue (data_augmentor.py:380-394): headings wrapped, then the
            # class mask computed at dataset.py:183 applied
            keep = np.array([n in self.class_names for n in d['gt_names']], dtype=np.bool_)
            d['gt_boxes'][:, 6] = limit_period(d['gt_boxes'][:, 6], offset=0.5, period=2 * np.pi)
            d['gt_boxes'], d['gt_names'] = d['gt_boxes'][keep], d['gt_names'][keep]
        if d.get('gt_boxes', None) is not None:
            sel = np.array([i for i, n in enumerate(d['gt_names']) if n in self.class_names], dtype=np.int64)
            d['gt_boxes'] = d['gt_boxes'][sel]
            d['gt_names'] = d['gt_names'][sel]
            cls = np.array([self.class_names.index(n) + 1 for n in d['gt_names']], dtype=np.int32)
            d['gt_boxes'] = np.concatenate((d['gt_boxes'], cls.reshape(-1, 1).astype(np.float32)), axis=1)
        if self.training and d.get('gt_boxes', None) is not None:          # REMOVE_OUTSIDE_BOXES, data_processor.py:88-93
            d['gt_boxes'] = d['gt_boxes'][mask_boxes_outside_range(d['gt_boxes'], self.range)]

    def _finish_gt(self, info: dict, d: dict):
        """NaN velocities zeroed, and the velocity columns dropped without PRED_VELOCITY (nuscenes_dataset.py:269-277)."""
        if self.set_nan_velocity_to_zeros and 'gt_boxes' in info:
            g = d['gt_boxes']
            g[np.isnan(g)] = 0
            d['gt_boxes'] = g
        if not self.pred_velocity and 'gt_boxes' in d:
            d['gt_boxes'] = d['gt_boxes'][:, [0, 1, 2, 3, 4, 5, 6, -1]]

    def _prepare(self, d: dict) -> dict:
        """DatasetTemplate.prepare_data (dataset.py:159-220); returns None when the frame has to be re-drawn."""
        self._prepare_gt(d)
        d['lidar_aug_matrix'] = np.eye(4)                                   # set_lidar_aug_matrix, no augmentation
        d['use_lead_xyz'] = True                                            # absolute_coordinates_encoding
        d['points'] = d['points'][mask_points_by_range(d['points'], self.range)]
        if self.training and len(d['gt_boxes']) == 0 and self.skip_no_gt:   # dataset.py:213-215
            return None
        d.pop('gt_names', None)
        return d

    def __getitem__(self, index: int) -> dict:
        info = copy.deepcopy(self.infos[index])
        d = {'points': lidar_with_sweeps(self.root, info, self.max_sweeps, self.rng),
             'frame_id': Path(info['lidar_path']).stem, 'metadata': {'token': info['token']}}
        self._load_gt(info, d)
        d.update(camera_info(info))
        fH, fW = self.final_dim
        d['ori_shape'] = [fW, fH]
        d['img_process_infos'] = [[float(np.mean(self.resize_lim_test)), (0, 0, fW, fH), False, 0] for _ in range(6)]
        d = self._prepare(d)
        if d is None:        # SKIP_NO_GT: the reference returns another, randomly drawn frame in this one's place
            d = self[int((np.random if self.rng is None else self.rng).randint(len(self)))]
        self._finish_gt(info, d)
        return d

    def gt_boxes(self, index: int) -> np.ndarray:
        """The frame's gt_boxes as ``self[index]`` produces them, without reading its LiDAR file.  A frame left
        without GT gives an empty array here: no other frame is drawn in its place (SKIP_NO_GT), because a caller
        that scores frame by frame must see this frame's GT.  A frame whose info has no GT gives a (0, 8) array."""
        info = self.infos[index]
        if 'gt_boxes' not in info:
            return np.zeros((0, 8), np.float32)
        d = {k: copy.deepcopy(info[k]) for k in ('gt_boxes', 'gt_names', 'num_lidar_pts') if k in info}
        self._load_gt(d, d)
        self._prepare_gt(d)
        self._finish_gt(info, d)
        return d['gt_boxes']

    # ---------------------------------------------------------------- seeker inputs
    def frame_input(self, index: int, detector, xyz_only: bool = False):
        """One frame as the engine wants it: the data_dict of ``__getitem__`` plus the frame's
        GLIP boxes.  ``detector`` has the reference feeder's contract (preprocessed_detector.py:47-106,
        e.g. ``proposer.PreprocessedGLIP``): called with a batch_dict holding ``batch_size``,
        ``image_paths`` and ``metadata`` it returns (boxes, labels, scores, batch_idx, cam_idx)."""
        from .seeker import FrameInput
        d = self[index]
        if xyz_only:
            # the seeker reads x, y, z only: split the columns here, on the loader's worker thread, so that the
            # host table that crosses PCIe is 12 B/point and no separate gather pass over full rows is needed
            d['points'] = np.ascontiguousarray(d['points'][:, :3], np.float32)
        boxes, labels, scores, _, cam_idx = detector(
            {'batch_size': 1, 'image_paths': [d['image_paths']], 'metadata': [d['metadata']]})
        fi = FrameInput(points=np.ascontiguousarray(d['points'], np.float32),
                        lidar2image=np.stack(d['lidar2image']).astype(np.float32),
                        camera2lidar=np.stack(d['camera2lidar']).astype(np.float32),
                        camera_intrinsics=np.stack(d['camera_intrinsics']).astype(np.float32),
                        det_boxes=np.asarray(boxes, np.float32).reshape(-1, 4), det_labels=np.asarray(labels, np.int64),
                        det_scores=np.asarray(scores, np.float32), det_cam_idx=np.asarray(cam_idx, np.int64),
                        gt_boxes=d.get('gt_boxes'))
        return fi, d['frame_id'], d['metadata']

    def prefetch(self, indices: Iterable[int], detector, batch_frames: int = 32, workers: int = 4,
                 xyz_only: bool = False):
        """Yields (frame_inputs, frame_ids, metadata) per batch of ``batch_frames`` frames, loading
        the NEXT batch on worker threads while the caller runs the current one on the GPU (file
        reads and numpy release the GIL).  The reference gets the same overlap from DataLoader
        worker processes."""
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
