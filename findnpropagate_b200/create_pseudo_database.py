"""A GT-sampling database of pseudo-labelled instances, for self-training:

    python -m findnpropagate_b200.create_pseudo_database --cfg_file cfgs/nuscenes_box_seeker_proposals.yaml --folder out/

reads the ``.pth`` pseudo-labels of every frame of the config's train info list as self-training's loader reads them
(``pseudo_loader.load_pseudos(folder, frame_id, labels, nms_thresh)``), crops every box's points out of the frame's
LiDAR sweeps on the GPU (``gt_database.crop_frames``: first containing box, input order, box-centred) and writes the
database OpenPCDet's ``DataBaseSampler`` reads, in the format of ``create_groundtruth_database``, under
``DATA_PATH/VERSION``:

  * ``pseudo_database_<S>sweeps_withvelo/<info index>_<class>_<gt_idx>.bin``: float32 ``[x, y, z, intensity, time]``
    rows relative to the box centre (an empty file for a box without points);
  * ``nuscenes_pseudo_dbinfos_<S>sweeps_withvelo.pkl``: ``{class: [info, ...]}`` with ``name``, ``path`` (relative to
    ``DATA_PATH/VERSION``), ``image_idx``, ``gt_idx`` (the row of load_pseudos' array), ``box3d_lidar`` (the box
    padded with zero velocity to the width and dtype of the infos' ``gt_boxes``), ``num_points_in_gt`` and ``score``.

The points are ``lidar_with_sweeps(root, info, MAX_SWEEPS, RandomState(--seed))`` without range filter or ego-point
removal on the key frame (the GT database's rule).  The sweeps are drawn on the main thread once per frame of the info
list, in order, and the files are read on ``--workers`` threads, so two runs write the same bytes.  Every refusal
(existing output, missing folder, a label outside the classes, ``WORLD_SIZE`` > 1, a frame over the NMS's box limit, a
KITTI config: KITTI's ``kitti_dbinfos`` / ``gt_database`` layout is another format) exits with status 1 before anything
is written.
"""
import argparse
import os
import pickle
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np


def parse_args(argv=None):
    p = argparse.ArgumentParser(prog="python -m findnpropagate_b200.create_pseudo_database",
                                description="Build a GT-sampling database from a folder of pseudo-labels.")
    p.add_argument("--cfg_file", required=True, help="head config, e.g. cfgs/nuscenes_box_seeker_proposals.yaml")
    p.add_argument("--folder", required=True, help="folder of per-frame .pth pseudo-labels")
    p.add_argument("--labels", type=int, nargs="+", default=None,
                   help="keep only these 1-based class labels (load_pseudos(labels=...))")
    p.add_argument("--nms_thresh", type=float, default=None,
                   help="rotated BEV NMS of each frame's boxes at this threshold (load_pseudos(nms_thresh=...))")
    p.add_argument("--seed", type=int, default=0, help="seed of the sweep draw (numpy RandomState)")
    p.add_argument("--batch_frames", type=int, default=16, help="frames per crop call on the GPU")
    p.add_argument("--workers", type=int, default=4, help="file reader and writer threads")
    p.add_argument("--set", dest="set_cfgs", default=None, nargs=argparse.REMAINDER, metavar="KEY VALUE",
                   help="config overrides, e.g. --set DATA_CONFIG.MAX_SWEEPS 10")
    return p.parse_args(argv)


def _fail(msg):
    print(msg, file=sys.stderr)
    raise SystemExit(1)


def output_paths(root, max_sweeps):
    """(database folder, db-info pickle) under the dataset root."""
    root = Path(root)
    return (root / ("pseudo_database_%dsweeps_withvelo" % max_sweeps),
            root / ("nuscenes_pseudo_dbinfos_%dsweeps_withvelo.pkl" % max_sweeps))


def _load_boxes(args, feed, frames, n_classes, pool):
    """Per frame of ``frames`` (info indices): (boxes (K,8) [box7, label], scores (K,)) as load_pseudos returns them,
    or None for a missing file.  Exits for a label outside the classes or a frame too large for the NMS."""
    from ._lib import SEG_NMS_MAX
    from .extract_pseudo_labels import frame_id
    from .pseudo_loader import pseudo_path, read_pseudos, seg_nms_keep
    ids = [frame_id(feed.infos[i]) for i in frames]
    got = list(pool.map(lambda fid: read_pseudos(pseudo_path(args.folder, fid)), ids))
    out = []
    for fid, g in zip(ids, got):
        if g is None:
            out.append(None)
            continue
        boxes, scores, lab = g
        bad = (lab < 1) | (lab > n_classes)
        if bad.any():
            _fail("frame %s: label %s outside the %d classes" % (fid, lab[bad][0], n_classes))
        if args.labels is not None:
            m = np.isin(lab, np.asarray(args.labels))
            boxes, scores, lab = boxes[m], scores[m], lab[m]
        if args.nms_thresh is not None and boxes.shape[0] > SEG_NMS_MAX:
            _fail("frame %s: %d boxes, the NMS takes at most %d per frame" % (fid, boxes.shape[0], SEG_NMS_MAX))
        b8 = np.zeros((boxes.shape[0], 8), np.float32)
        b8[:, :7] = boxes
        b8[:, 7] = lab
        out.append((b8, scores))
    if args.nms_thresh is not None:
        live = [k for k, o in enumerate(out) if o is not None]
        keeps = seg_nms_keep([out[k][0] for k in live], [out[k][1] for k in live], args.nms_thresh)
        for k, keep in zip(live, keeps):
            out[k] = (out[k][0][keep], out[k][1][keep])
    return out


def main(argv=None):
    """Runs the command; returns dict(frames, boxes {class: count}, missing, skipped, skipped_frames)."""
    args = parse_args(argv)
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        _fail("create_pseudo_database runs in one process (it is bound by file reads): start it without torchrun")
    if not os.path.isdir(args.folder):
        _fail("%s does not exist or is not a folder" % args.folder)
    if args.batch_frames < 1 or args.workers < 1:
        _fail("--batch_frames and --workers must be at least 1")
    from .extract_pseudo_labels import FAILURES, build_feed, check_frame, is_kitti, load_config
    try:
        cfg = load_config(args.cfg_file, args.set_cfgs)
    except (OSError, KeyError, ValueError) as e:
        _fail(e.args[-1] if isinstance(e, KeyError) else e)
    if is_kitti(cfg):
        _fail("DATA_CONFIG.DATASET KittiDataset is not supported: this command writes the nuScenes database layout "
              "(KITTI's kitti_dbinfos / gt_database format is not written)")
    feed = build_feed(cfg)
    names = list(feed.class_names)
    if args.labels is not None:
        bad = [c for c in args.labels if not 1 <= c <= len(names)]
        if bad:
            _fail("--labels %s: outside the classes 1..%d" % (" ".join(map(str, bad)), len(names)))
    db_dir, db_info_path = output_paths(feed.root, feed.max_sweeps)
    for p in (db_dir, db_info_path):
        if os.path.exists(p):
            _fail("%s already exists (nothing was written)" % p)
    from .gt_database import crop_frames
    from .nuscenes_feed import draw_sweeps, read_lidar_with_sweeps
    n = len(feed)
    codes = [check_frame(feed, None, feed.infos[i]) for i in range(n)]
    skipped = [(Path(feed.infos[i]["lidar_path"]).stem, FAILURES[c]) for i, c in enumerate(codes) if c]
    for fid, why in skipped:
        print("skipped frame %s: %s" % (fid, why))
    run = [i for i in range(n) if not codes[i]]
    with ThreadPoolExecutor(max_workers=args.workers) as pool:
        loaded = dict(zip(run, _load_boxes(args, feed, run, len(names), pool)))
        missing = sum(v is None for v in loaded.values())
        rng = np.random.RandomState(args.seed)
        db_dir.mkdir(parents=True)
        all_db_infos = {}
        written = {}
        for s in range(0, n, args.batch_frames):
            chunk = range(s, min(s + args.batch_frames, n))
            picks = {i: draw_sweeps(feed.infos[i], feed.max_sweeps, rng) for i in chunk}
            todo = [i for i in chunk if loaded.get(i) is not None and len(loaded[i][0])]
            points = list(pool.map(lambda i: read_lidar_with_sweeps(feed.root, feed.infos[i], picks[i]), todo))
            cropped = crop_frames(points, [loaded[i][0] for i in todo])
            files = []
            for k, idx in enumerate(todo):
                boxes, scores = loaded[idx]
                gt = feed.infos[idx]["gt_boxes"]
                for j in range(boxes.shape[0]):
                    name = names[int(boxes[j, 7]) - 1]
                    path = db_dir / ("%d_%s_%d.bin" % (idx, name, j))
                    files.append((path, cropped[k][j]))
                    box = np.zeros(gt.shape[1], gt.dtype)
                    box[:7] = boxes[j, :7]
                    all_db_infos.setdefault(name, []).append(
                        {'name': name, 'path': str(path.relative_to(feed.root)), 'image_idx': idx, 'gt_idx': j,
                         'box3d_lidar': box, 'num_points_in_gt': cropped[k][j].shape[0], 'score': float(scores[j])})
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
