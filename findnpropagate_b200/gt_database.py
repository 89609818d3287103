"""Ground-truth database creation: the other caller of batched first-match ``points_in_boxes_gpu`` on this path
(SURVEY.md section 8 row f4).

Reference: ``NuScenesDataset.create_groundtruth_database`` (pcdet/datasets/nuscenes/nuscenes_dataset.py:346-390):
per frame, every point is assigned to the FIRST GT box that contains it (one ``points_in_boxes_gpu`` call over all
of the frame's boxes), the points of each box are written to ``gt_database_<S>sweeps_withvelo/<frame>_<name>_<i>.bin``
relative to the box centre, and one info dict per box goes into ``nuscenes_dbinfos_<S>sweeps_withvelo.pkl``.

Here the frames of a batch are uploaded together and cropped by ONE ``fnp_crop_points_in_boxes`` call: the first-match
assignment of ``fnp_points_in_boxes``, then every box's points in input order with the centre subtracted, on the
device.  Only the counts and the rows in boxes come back.  The rest is the same host-side bookkeeping and the same
files, byte for byte.

KITTI: ``KittiDataset.create_groundtruth_database`` (pcdet/datasets/kitti/kitti_dataset.py) crops by
``points_in_boxes_cpu`` instead: the CPU op's predicate, and every box that contains a point gets it.
``create_groundtruth_database_kitti`` does that through ``crop_points_in_boxes_all`` (``crop_frames(every_box=True)``),
again one crop per batch with no (boxes, points) matrix formed or copied back.
"""
import pickle
from pathlib import Path
from typing import Optional, Sequence

import numpy as np
import torch

from .nuscenes_feed import lidar_with_sweeps


def _starts(name, starts, total):
    a = starts.numpy() if isinstance(starts, torch.Tensor) else np.asarray(starts)
    if a.ndim != 1 or a.shape[0] < 1 or not np.issubdtype(a.dtype, np.integer):
        raise ValueError("%s must be a 1-D integer array of n_frames + 1 entries" % name)
    a = a.astype(np.int64)
    if a[0] != 0 or a[-1] != total or (np.diff(a) < 0).any():
        raise ValueError("%s must rise from 0 to %d, got %s .. %s" % (name, total, a[0], a[-1]))
    return a


def _crop_args(points, row_start, boxes, centres, box_start):
    """The crop launchers' argument checks; (N, C, G, row_start, box_start) with the starts as int64 numpy arrays."""
    for name, t, dt, w in (("points", points, torch.float32, None), ("boxes", boxes, torch.float32, 7),
                           ("centres", centres, torch.float64, 3)):
        if not isinstance(t, torch.Tensor):
            raise ValueError("%s must be a tensor, got %s" % (name, type(t).__name__))
        if t.dtype != dt or t.dim() != 2 or (t.shape[1] != w if w else t.shape[1] < 3) or not t.is_contiguous():
            raise ValueError("%s must be a contiguous (rows, %s) %s tensor, got %s %s"
                             % (name, w or ">= 3", dt, t.dtype, tuple(t.shape)))
    if boxes.shape[0] != centres.shape[0]:
        raise ValueError("boxes and centres differ in length: %d and %d" % (boxes.shape[0], centres.shape[0]))
    if any(isinstance(t, torch.Tensor) and t.is_cuda for t in (row_start, box_start)):
        raise ValueError("row_start and box_start are host arrays")
    N, C, G = points.shape[0], points.shape[1], boxes.shape[0]
    rs, bs = _starts("row_start", row_start, N), _starts("box_start", box_start, G)
    if rs.shape != bs.shape:
        raise ValueError("row_start and box_start differ in length: %d and %d" % (rs.shape[0], bs.shape[0]))
    dev = points.device
    if not points.is_cuda or boxes.device != dev or centres.device != dev:
        raise ValueError("points, boxes and centres must be on one CUDA device, got %s, %s, %s"
                         % (points.device, boxes.device, centres.device))
    return N, C, G, rs, bs


def crop_points_in_boxes(points, row_start, boxes, centres, box_start):
    """Every box's points, cropped on the device in one fnp_crop_points_in_boxes call.

    points (N, C) float32 CUDA, C >= 3, x y z first; boxes (G, 7) float32 and centres (G, 3) float64 on the same
    device; all contiguous.  row_start / box_start: host integer arrays (or CPU tensors) of n_frames + 1 entries,
    frame f owning points row_start[f] .. row_start[f+1] and boxes box_start[f] .. box_start[f+1].
    Each point goes to the first box of its frame that contains it (fnp_points_in_boxes' predicate).  Returns device
    tensors counts (G,) int32, starts (G+1,) int64 and rows (N, C) float32: box g's points are rows
    starts[g] .. starts[g] + counts[g], in input order, x y z as float32(float64(p) - centre).  ValueError for a bad
    argument."""
    from . import _lib
    N, C, G, rs, bs = _crop_args(points, row_start, boxes, centres, box_start)
    dev = points.device
    F = rs.shape[0] - 1
    ws_bytes = int(_lib.lib.fnp_crop_workspace_bytes(rs.ctypes.data, bs.ctypes.data, F))
    d_starts = torch.from_numpy(np.concatenate([rs, bs])).to(dev)
    counts = torch.empty(G, dtype=torch.int32, device=dev)
    starts = torch.empty(G + 1, dtype=torch.int64, device=dev)
    rows = torch.empty((N, C), dtype=torch.float32, device=dev)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        rc = _lib.lib.fnp_crop_points_in_boxes(points.data_ptr(), C, d_starts.data_ptr(), N, boxes.data_ptr(),
                                               centres.data_ptr(), d_starts[F + 1:].data_ptr(), G, F,
                                               counts.data_ptr(), starts.data_ptr(), rows.data_ptr(), ws.data_ptr(),
                                               ws_bytes, _lib.current_stream(dev))
    _lib.check(rc, "fnp_crop_points_in_boxes")
    return counts, starts, rows


def crop_points_in_boxes_all(points, row_start, boxes, centres, box_start):
    """Every box's points by points_in_boxes_cpu's rule, cropped on the device: a point goes to EVERY box of its frame
    that contains it (``points[point_indices[i] > 0]``), tested with the CPU op's predicate (margin 1e-2, rounded
    products, the host libm's trig: fnp_host_prep_boxes_cpu + fnp_crop_all_count / fnp_crop_all_scatter).

    Arguments as for crop_points_in_boxes; the boxes are copied to the host for their per-box constants.  Returns
    device tensors counts (G,) int32, starts (G+1,) int64 and rows (starts[G], C) float32: box g's points are rows
    starts[g] .. starts[g] + counts[g], in input order, x y z as float32(float64(p) - centre).  The only read back
    before the rows are written is starts[G] (8 bytes), which sizes rows exactly.  ValueError for a bad argument."""
    import ctypes
    from . import _lib
    N, C, G, rs, bs = _crop_args(points, row_start, boxes, centres, box_start)
    dev = points.device
    F = rs.shape[0] - 1
    b_host = boxes.cpu()
    prep = torch.empty((G, 8), dtype=torch.float32)
    _lib.check(_lib.lib.fnp_host_prep_boxes_cpu(ctypes.c_void_p(b_host.data_ptr()), ctypes.c_void_p(prep.data_ptr()),
                                                G), "fnp_host_prep_boxes_cpu")
    ws_bytes = int(_lib.lib.fnp_crop_workspace_bytes(rs.ctypes.data, bs.ctypes.data, F))
    d_starts = torch.from_numpy(np.concatenate([rs, bs])).to(dev)
    prep = prep.to(dev)
    counts = torch.empty(G, dtype=torch.int32, device=dev)
    starts = torch.empty(G + 1, dtype=torch.int64, device=dev)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        rc = _lib.lib.fnp_crop_all_count(points.data_ptr(), C, d_starts.data_ptr(), N, prep.data_ptr(),
                                         d_starts[F + 1:].data_ptr(), G, F, counts.data_ptr(), starts.data_ptr(),
                                         ws.data_ptr(), ws_bytes, _lib.current_stream(dev))
        _lib.check(rc, "fnp_crop_all_count")
        total = int(starts[G].item())
        rows = torch.empty((total, C), dtype=torch.float32, device=dev)
        rc = _lib.lib.fnp_crop_all_scatter(points.data_ptr(), C, d_starts.data_ptr(), N, prep.data_ptr(),
                                           centres.data_ptr(), d_starts[F + 1:].data_ptr(), G, F, starts.data_ptr(),
                                           rows.data_ptr(), total, ws.data_ptr(), ws_bytes, _lib.current_stream(dev))
    _lib.check(rc, "fnp_crop_all_scatter")
    return counts, starts, rows


def crop_frames(points_list, boxes_list, device=None, every_box=False):
    """Per frame, the list of its boxes' points (n_i, C) float32, box-centred: ``pts[box_of_pt == i]`` then
    ``[:, :3] -= boxes[i, :3]`` in the boxes' own precision, as create_groundtruth_database crops them.
    points_list[b]: (N_b, C >= 3) float32 arrays; boxes_list[b]: (G_b, >= 7) float32 or float64 arrays.  One upload,
    one crop call; the counts come back first, then only the rows that lie in a box.
    every_box: KITTI's rule instead (``points_in_boxes_cpu`` on the boxes cast to float32, then
    ``pts[point_indices[i] > 0]``): a point goes to every box that contains it (crop_points_in_boxes_all)."""
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if not points_list:
        return []
    C = points_list[0].shape[1]
    pts = np.concatenate([np.asarray(p, np.float32).reshape(-1, C) for p in points_list])
    box = np.concatenate([np.asarray(b)[:, :7] for b in boxes_list])
    rs = np.concatenate([[0], np.cumsum([p.shape[0] for p in points_list])]).astype(np.int64)
    bs = np.concatenate([[0], np.cumsum([len(b) for b in boxes_list])]).astype(np.int64)
    if every_box:
        counts, starts, rows = crop_points_in_boxes_all(
            torch.from_numpy(pts).to(dev), rs, torch.from_numpy(np.ascontiguousarray(box, np.float32)).to(dev),
            torch.from_numpy(np.ascontiguousarray(box[:, :3], np.float64)).to(dev), bs)
        counts, starts, rows = counts.cpu().numpy(), starts.cpu().numpy(), rows.cpu().numpy()
        return [[rows[starts[g]:starts[g] + counts[g]] for g in range(bs[b], bs[b + 1])]
                for b in range(len(points_list))]
    counts, starts, rows = crop_points_in_boxes(
        torch.from_numpy(pts).to(dev), rs, torch.from_numpy(np.ascontiguousarray(box, np.float32)).to(dev),
        torch.from_numpy(np.ascontiguousarray(box[:, :3], np.float64)).to(dev), bs)
    counts = counts.cpu().numpy()
    total = int(counts.sum())
    rows = rows[:total].cpu().numpy()
    ends = np.cumsum(counts)
    out = []
    for b in range(len(points_list)):
        out.append([rows[ends[g] - counts[g]:ends[g]] for g in range(bs[b], bs[b + 1])])
    return out


def create_groundtruth_database(root_path, infos: Sequence[dict], used_classes: Optional[Sequence[str]] = None,
                                max_sweeps: int = 10, batch_frames: int = 16, device=None, rng=None):
    """nuscenes_dataset.py:346-390 for a list of info dicts under ``root_path``; returns the db-info dict that is
    also pickled.  ``rng``: private generator for the sweep draw (None: numpy's global one, like the reference)."""
    root = Path(root_path)
    db_dir = root / ('gt_database_%dsweeps_withvelo' % max_sweeps)
    db_info_path = root / ('nuscenes_dbinfos_%dsweeps_withvelo.pkl' % max_sweeps)
    db_dir.mkdir(parents=True, exist_ok=True)
    all_db_infos = {}
    for s in range(0, len(infos), batch_frames):
        chunk = list(range(s, min(s + batch_frames, len(infos))))
        points = [lidar_with_sweeps(root, infos[i], max_sweeps, rng) for i in chunk]       # the reference's order of draws
        cropped = crop_frames(points, [infos[i]['gt_boxes'] for i in chunk], device=device)
        for k, idx in enumerate(chunk):
            info = infos[idx]
            gt_boxes, gt_names = info['gt_boxes'], info['gt_names']
            for i in range(gt_boxes.shape[0]):
                filepath = db_dir / ('%s_%s_%d.bin' % (idx, gt_names[i], i))
                gt_points = cropped[k][i]
                with open(filepath, 'w') as f:
                    gt_points.tofile(f)
                if (used_classes is None) or gt_names[i] in used_classes:
                    db_info = {'name': gt_names[i], 'path': str(filepath.relative_to(root)), 'image_idx': idx, 'gt_idx': i,
                               'box3d_lidar': gt_boxes[i], 'num_points_in_gt': gt_points.shape[0]}
                    all_db_infos.setdefault(gt_names[i], []).append(db_info)
    with open(db_info_path, 'wb') as f:
        pickle.dump(all_db_infos, f)
    return all_db_infos


def kitti_split_root(root, split):
    """``<root>/training`` unless the split is ``test`` (KittiDataset's root_split_path, KittiFeed's rule)."""
    return Path(root) / ('training' if split != 'test' else 'testing')


def create_groundtruth_database_kitti(root_path, infos: Sequence[dict], used_classes: Optional[Sequence[str]] = None,
                                      split: str = 'train', batch_frames: int = 16, device=None):
    """OpenPCDet v0.6's ``KittiDataset.create_groundtruth_database`` for a list of info dicts under ``root_path``
    (DATA_PATH); returns the db-info dict that is also pickled to ``kitti_dbinfos_<split>.pkl``.

    Per info: the whole velodyne scan ``<split root>/velodyne/<lidar_idx>.bin`` as (N, 4) float32, the first
    ``len(annos['gt_boxes_lidar'])`` rows of ``name``, ``difficulty`` and ``bbox`` (DontCare rows come last), every
    box's points by ``points_in_boxes_cpu``'s rule (a point in two boxes goes to both) written to
    ``gt_database[_<split>]/<lidar_idx>_<name>_<i>.bin``, and for the used classes one info with ``name``, ``path``,
    ``image_idx`` (the lidar_idx string), ``gt_idx``, ``box3d_lidar``, ``num_points_in_gt``, ``difficulty``, ``bbox``
    and ``score``.  The frames of a batch of ``batch_frames`` are cropped by one crop_frames(every_box=True) call."""
    root = Path(root_path)
    split_root = kitti_split_root(root, split)
    db_dir = root / ('gt_database' if split == 'train' else 'gt_database_%s' % split)
    db_info_path = root / ('kitti_dbinfos_%s.pkl' % split)
    db_dir.mkdir(parents=True, exist_ok=True)
    all_db_infos = {}
    for s in range(0, len(infos), batch_frames):
        chunk = infos[s:s + batch_frames]
        ids = [info['point_cloud']['lidar_idx'] for info in chunk]
        points = [np.fromfile(str(split_root / 'velodyne' / ('%s.bin' % idx)), dtype=np.float32).reshape(-1, 4)
                  for idx in ids]
        cropped = crop_frames(points, [info['annos']['gt_boxes_lidar'] for info in chunk], device=device,
                              every_box=True)
        for k, (info, sample_idx) in enumerate(zip(chunk, ids)):
            annos = info['annos']
            names, difficulty, bbox = annos['name'], annos['difficulty'], annos['bbox']
            gt_boxes = annos['gt_boxes_lidar']
            for i in range(gt_boxes.shape[0]):
                filepath = db_dir / ('%s_%s_%d.bin' % (sample_idx, names[i], i))
                gt_points = cropped[k][i]
                with open(filepath, 'w') as f:
                    gt_points.tofile(f)
                if (used_classes is None) or names[i] in used_classes:
                    db_info = {'name': names[i], 'path': str(filepath.relative_to(root)), 'image_idx': sample_idx,
                               'gt_idx': i, 'box3d_lidar': gt_boxes[i], 'num_points_in_gt': gt_points.shape[0],
                               'difficulty': difficulty[i], 'bbox': bbox[i], 'score': annos['score'][i]}
                    all_db_infos.setdefault(names[i], []).append(db_info)
    with open(db_info_path, 'wb') as f:
        pickle.dump(all_db_infos, f)
    return all_db_infos
