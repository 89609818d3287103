"""A KITTI GT-sampling database of pseudo-labelled instances, for self-training:

    python -m findnpropagate_b200.create_kitti_pseudo_database --cfg_file cfgs/kitti_box_seeker_proposals.yaml --folder out/

reads the ``.pth`` pseudo-labels of every frame of the config's train info list as self-training's loader reads them
(``pseudo_loader.load_pseudos(folder, lidar_idx, labels, nms_thresh)``), crops every box's points out of the frame's
whole velodyne scan on the GPU by ``points_in_boxes_cpu``'s rule (``gt_database.crop_frames(every_box=True)``: a point
goes to every box that contains it, input order, box-centred) and writes the database OpenPCDet's ``DataBaseSampler``
reads, in the format of ``KittiDataset.create_groundtruth_database``, under ``DATA_PATH``:

  * ``pseudo_database[_<split>]/<lidar_idx>_<class>_<gt_idx>.bin``: float32 ``[x, y, z, intensity]`` rows relative to
    the box centre (an empty file for a box without points);
  * ``kitti_pseudo_dbinfos_<split>.pkl``: ``{class: [info, ...]}`` with the GT database's keys: ``name``, ``path``
    (relative to ``DATA_PATH``), ``image_idx`` (the lidar_idx string), ``gt_idx`` (the row of load_pseudos' array),
    ``box3d_lidar`` (the box's 7 float32 values), ``num_points_in_gt``, ``difficulty`` (0: a pseudo-label has no
    occlusion or truncation to grade, and the KITTI configs' ``filter_by_difficulty`` drops only -1), ``bbox`` (the
    image box of the box's eight corners through the frame's calibration, clipped to the image) and ``score``.

The split is ``DATA_SPLIT['train']``; its points are the whole scan (no FOV or range filter: the GT database's rule).
A frame without a ``.pth`` file has no boxes; a frame whose velodyne or calib file is missing is logged and skipped.
Files are read and written on ``--workers`` threads, and two runs write the same bytes.  Every refusal (existing
output, missing folder, a label outside the classes, ``WORLD_SIZE`` > 1, a frame over the NMS's box limit, a nuScenes
config) exits with status 1 before anything is written.
"""
import argparse
import os
import pickle
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np


def parse_args(argv=None):
    p = argparse.ArgumentParser(prog="python -m findnpropagate_b200.create_kitti_pseudo_database",
                                description="Build a KITTI GT-sampling database from a folder of pseudo-labels.")
    p.add_argument("--cfg_file", required=True, help="head config, e.g. cfgs/kitti_box_seeker_proposals.yaml")
    p.add_argument("--folder", required=True, help="folder of per-frame .pth pseudo-labels")
    p.add_argument("--labels", type=int, nargs="+", default=None,
                   help="keep only these 1-based class labels (load_pseudos(labels=...))")
    p.add_argument("--nms_thresh", type=float, default=None,
                   help="rotated BEV NMS of each frame's boxes at this threshold (load_pseudos(nms_thresh=...))")
    p.add_argument("--batch_frames", type=int, default=16, help="frames per crop call on the GPU")
    p.add_argument("--workers", type=int, default=4, help="file reader and writer threads")
    p.add_argument("--set", dest="set_cfgs", default=None, nargs=argparse.REMAINDER, metavar="KEY VALUE",
                   help="config overrides, e.g. --set DATA_CONFIG.DATA_SPLIT.train val")
    return p.parse_args(argv)


def _fail(msg):
    print(msg, file=sys.stderr)
    raise SystemExit(1)


def output_paths(root, split):
    """(database folder, db-info pickle) under DATA_PATH for the split (KittiDataset's naming of the GT database)."""
    root = Path(root)
    return (root / ("pseudo_database" if split == "train" else "pseudo_database_%s" % split),
            root / ("kitti_pseudo_dbinfos_%s.pkl" % split))


def image_boxes(boxes, calib, image_shape):
    """(K,4) float32 image boxes of (K,>=7) LiDAR boxes: LiDAR -> rect -> image through ``calib``, clipped to the
    image (OpenPCDet's boxes3d_lidar_to_kitti_camera + boxes3d_kitti_camera_to_imageboxes)."""
    from .kitti_feed import boxes3d_kitti_camera_to_imageboxes, boxes3d_lidar_to_kitti_camera
    if len(boxes) == 0:
        return np.zeros((0, 4), np.float32)
    cam = boxes3d_lidar_to_kitti_camera(np.asarray(boxes, np.float32)[:, :7], calib)
    return boxes3d_kitti_camera_to_imageboxes(cam, calib, image_shape).astype(np.float32)


def main(argv=None):
    """Runs the command; returns dict(frames, boxes {class: count}, missing, skipped, skipped_frames)."""
    args = parse_args(argv)
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        _fail("create_kitti_pseudo_database runs in one process (it is bound by file reads): start it without torchrun")
    if not os.path.isdir(args.folder):
        _fail("%s does not exist or is not a folder" % args.folder)
    if args.batch_frames < 1 or args.workers < 1:
        _fail("--batch_frames and --workers must be at least 1")
    from .extract_pseudo_labels import FAILURES, build_feed, check_frame, frame_id, is_kitti, load_config
    try:
        cfg = load_config(args.cfg_file, args.set_cfgs)
    except (OSError, KeyError, ValueError) as e:
        _fail(e.args[-1] if isinstance(e, KeyError) else e)
    if not is_kitti(cfg):
        _fail("DATA_CONFIG.DATASET %s is not supported: this command writes KITTI's database layout; "
              "python -m findnpropagate_b200.create_pseudo_database writes the nuScenes one" % cfg.DATA_CONFIG.DATASET)
    feed = build_feed(cfg)
    names = list(feed.class_names)
    if args.labels is not None:
        bad = [c for c in args.labels if not 1 <= c <= len(names)]
        if bad:
            _fail("--labels %s: outside the classes 1..%d" % (" ".join(map(str, bad)), len(names)))
    split = cfg.DATA_CONFIG.get("DATA_SPLIT", {}).get("train", "train")
    db_dir, db_info_path = output_paths(feed.root, split)
    for p in (db_dir, db_info_path):
        if os.path.exists(p):
            _fail("%s already exists (nothing was written)" % p)
    from .create_pseudo_database import _load_boxes
    from .gt_database import crop_frames
    n = len(feed)
    codes = [check_frame(feed, None, feed.infos[i]) for i in range(n)]
    skipped = [(frame_id(feed.infos[i]), FAILURES[c]) for i, c in enumerate(codes) if c]
    for fid, why in skipped:
        print("skipped frame %s: %s" % (fid, why))
    run = [i for i in range(n) if not codes[i]]
    with ThreadPoolExecutor(max_workers=args.workers) as pool:
        loaded = dict(zip(run, _load_boxes(args, feed, run, len(names), pool)))
        missing = sum(v is None for v in loaded.values())
        db_dir.mkdir(parents=True)
        all_db_infos = {}
        written = {}
        todo_all = [i for i in run if loaded[i] is not None and len(loaded[i][0])]
        for s in range(0, len(todo_all), args.batch_frames):
            todo = todo_all[s:s + args.batch_frames]
            ids = [frame_id(feed.infos[i]) for i in todo]
            points = list(pool.map(feed.lidar, ids))
            calibs = list(pool.map(feed.calib, ids))
            cropped = crop_frames(points, [loaded[i][0] for i in todo], every_box=True)
            files = []
            for k, (idx, sample_idx) in enumerate(zip(todo, ids)):
                boxes, scores = loaded[idx]
                bbox = image_boxes(boxes, calibs[k], feed.infos[idx]["image"]["image_shape"])
                for j in range(boxes.shape[0]):
                    name = names[int(boxes[j, 7]) - 1]
                    path = db_dir / ("%s_%s_%d.bin" % (sample_idx, name, j))
                    files.append((path, cropped[k][j]))
                    all_db_infos.setdefault(name, []).append(
                        {'name': name, 'path': str(path.relative_to(feed.root)), 'image_idx': sample_idx, 'gt_idx': j,
                         'box3d_lidar': boxes[j, :7].copy(), 'num_points_in_gt': cropped[k][j].shape[0],
                         'difficulty': 0, 'bbox': bbox[j], 'score': float(scores[j])})
                    written[name] = written.get(name, 0) + 1
            list(pool.map(lambda f: f[1].tofile(str(f[0])), files))
    with open(db_info_path, "wb") as f:
        pickle.dump(all_db_infos, f)
    print("frames: %d, missing files: %d, skipped frames: %d" % (len(run), missing, len(skipped)))
    print("boxes written: %s (%s)" % (", ".join("%s %d" % (c, written[c]) for c in names if c in written) or "none",
                                      db_dir))
    return dict(frames=len(run), boxes=written, missing=missing, skipped=len(skipped), skipped_frames=skipped)


if __name__ == "__main__":
    main()
