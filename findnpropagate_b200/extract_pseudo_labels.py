"""Pseudo-label extraction from the reference's config files, on the batched pipeline:

    python -m findnpropagate_b200.extract_pseudo_labels --cfg_file cfgs/nuscenes_box_seeker_proposals.yaml --folder out/

is tools/extract_pseudo_labels.py of the reference with ``extract.extract_nuscenes`` in place of its batch-size-1
loop.  Run it from the directory the reference runs from (``tools/``): the config's relative paths
(``_BASE_CONFIG_``, ``DATA_PATH``, the GLIP prediction files of ``PreprocessedGLIP``) are read as there.

  * config: ``DATA_CONFIG.DATASET`` NuScenesDataset with ``MODEL.DENSE_HEAD.NAME`` FrustumProposerOG, or KittiDataset
    with FrustumProposerOGKITTI; the head's options are read by its own constructor (``proposer``); frames come from
    ``NuScenesFeed`` / ``KittiFeed`` in the mode the reference tool runs its loader in (training=True, augmentation
    list emptied, extract_pseudo_labels.py:47-58);
  * output: one ``.pth`` per frame in ``--folder``, which must not exist yet (:80-84);
  * failed frames: a frame whose LiDAR file, one of whose sweep files (MAX_SWEEPS > 1) or one of whose six camera
    images is missing from the detector's predictions is skipped, logged and counted (``check_frame``); for KITTI a
    frame whose velodyne or calib file is missing, or whose ``<frame_id>.png`` is not in the predictions;
  * several GPUs: under torchrun (``WORLD_SIZE`` > 1) each process runs on ``cuda:LOCAL_RANK`` over NCCL and takes
    frames ``rank::world``; rank 0 prints.
"""
import argparse
import json
import os
import sys
from pathlib import Path

from .config import cfg_from_list, cfg_from_yaml_file

# the dataset each supported head runs on
PAIRS = {"NuScenesDataset": "FrustumProposerOG", "KittiDataset": "FrustumProposerOGKITTI"}
DATASETS = tuple(PAIRS)
HEADS = tuple(PAIRS.values())

LIDAR_MISSING, SWEEP_MISSING, IMAGE_NOT_PREDICTED, CALIB_MISSING = 1, 2, 3, 4
FAILURES = {LIDAR_MISSING: "LiDAR file missing", SWEEP_MISSING: "sweep file missing",
            IMAGE_NOT_PREDICTED: "camera image not in the detector's predictions",
            CALIB_MISSING: "calibration file missing"}


def parse_args(argv=None):
    p = argparse.ArgumentParser(prog="python -m findnpropagate_b200.extract_pseudo_labels",
                                description="Box Seeker pseudo-label extraction from an OpenPCDet config.")
    p.add_argument("--cfg_file", required=True, help="head config, e.g. cfgs/nuscenes_box_seeker_proposals.yaml")
    p.add_argument("--folder", required=True, help="output folder for the .pth files; must not exist")
    p.add_argument("--batch_frames", type=int, default=64, help="frames per batch on the GPU")
    p.add_argument("--workers", type=int, default=4, help="loader threads")
    p.add_argument("--nms_thresh", type=float, default=None,
                   help="per-frame rotated NMS of the proposals (default: none, proposals are written raw)")
    p.add_argument("--set", dest="set_cfgs", default=None, nargs=argparse.REMAINDER, metavar="KEY VALUE",
                   help="config overrides, e.g. --set DATA_CONFIG.MAX_SWEEPS 1")
    return p.parse_args(argv)


def load_config(cfg_file, set_cfgs=None):
    """The config with the ``--set`` overrides applied; ValueError when it is not a supported one."""
    cfg = cfg_from_yaml_file(cfg_file)
    if set_cfgs:
        cfg_from_list(set_cfgs, cfg)
    dataset = cfg.get("DATA_CONFIG", {}).get("DATASET")
    if dataset not in DATASETS:
        raise ValueError("DATA_CONFIG.DATASET %r is not supported: this command reads %s" % (dataset, ", ".join(DATASETS)))
    head = cfg.get("MODEL", {}).get("DENSE_HEAD", {}).get("NAME")
    if head != PAIRS[dataset]:
        raise ValueError("DATA_CONFIG.DATASET %r with MODEL.DENSE_HEAD.NAME %r is not supported: this command reads %s, "
                         "and runs %s" % (dataset, head, " and ".join(DATASETS),
                                          ", ".join("%s on %s" % (h, d) for d, h in PAIRS.items())))
    return cfg


def is_kitti(cfg) -> bool:
    return cfg.DATA_CONFIG.DATASET == "KittiDataset"


def build_head(cfg, device=None):
    """The config's head, built by its own constructor from MODEL.DENSE_HEAD and CLASS_NAMES."""
    from . import proposer
    cls = proposer.FrustumProposerOGKITTI if is_kitti(cfg) else proposer.FrustumProposerOG
    return cls(model_cfg=cfg.MODEL.DENSE_HEAD, class_names=cfg.get("CLASS_NAMES"), device=device)


def frame_id(info: dict) -> str:
    """The frame id of an info dict of either dataset (the name of its .pth file, before '.' -> '_')."""
    return info["point_cloud"]["lidar_idx"] if "point_cloud" in info else Path(info["lidar_path"]).stem


def build_feed(cfg, infos=None, device=None):
    """NuScenesFeed over ``DATA_PATH / VERSION`` (the NuScenesDataset rule), or KittiFeed over ``DATA_PATH`` and
    ``DATA_SPLIT['train']`` (``device``: where its frames' calibration blocks are formed), of ``INFO_PATH['train']``
    (or ``infos``), training=True; keys the config leaves out keep the feed's defaults."""
    d = cfg.DATA_CONFIG
    if is_kitti(cfg):
        from .kitti_feed import KittiFeed
        kw = {arg: d[key] for key, arg in (("POINT_CLOUD_RANGE", "point_cloud_range"),
                                           ("FOV_POINTS_ONLY", "fov_points_only")) if key in d}
        if "CLASS_NAMES" in cfg:
            kw["class_names"] = cfg.CLASS_NAMES
        return KittiFeed(d.DATA_PATH, d.INFO_PATH["train"] if infos is None else infos,
                         split=d.get("DATA_SPLIT", {}).get("train", "train"), training=True, device=device, **kw)
    from .nuscenes_feed import NuScenesFeed
    kw = {arg: d[key] for key, arg in (("MAX_SWEEPS", "max_sweeps"), ("POINT_CLOUD_RANGE", "point_cloud_range"),
                                       ("FILTER_MIN_POINTS_IN_GT", "filter_min_points_in_gt"),
                                       ("PRED_VELOCITY", "pred_velocity"),
                                       ("SET_NAN_VELOCITY_TO_ZEROS", "set_nan_velocity_to_zeros")) if key in d}
    image = (d.get("CAMERA_CONFIG") or {}).get("IMAGE") or {}
    if "FINAL_DIM" in image:
        kw["final_dim"] = image["FINAL_DIM"]
    if "RESIZE_LIM_TEST" in image:
        kw["resize_lim_test"] = image["RESIZE_LIM_TEST"]
    if "CLASS_NAMES" in cfg:
        kw["class_names"] = cfg.CLASS_NAMES
    return NuScenesFeed(Path(d.DATA_PATH) / d.VERSION, d.INFO_PATH["train"] if infos is None else infos,
                        training=True, **kw)


def check_frame(feed, detector, info) -> int:
    """0, or why the frame cannot run: its LiDAR file is missing; MAX_SWEEPS > 1 and a sweep file its info lists is
    missing (which sweeps the feed reads is drawn only at load time); one of its camera images is not in the
    detector's predictions (not checked when ``detector`` is None).  KITTI: its velodyne file or its calib file is
    missing; ``<frame_id>.png`` is not in the detector's predictions."""
    if "point_cloud" in info:
        fid = frame_id(info)
        if not feed.lidar_path(fid).is_file():
            return LIDAR_MISSING
        if not feed.calib_path(fid).is_file():
            return CALIB_MISSING
        if detector is not None and not detector.has_image(fid + ".png"):
            return IMAGE_NOT_PREDICTED
        return 0
    if not (feed.root / info["lidar_path"]).is_file():
        return LIDAR_MISSING
    if feed.max_sweeps > 1 and not all((feed.root / s["lidar_path"]).is_file() for s in info["sweeps"]):
        return SWEEP_MISSING
    if detector is not None and not all(detector.has_image(cam["data_path"]) for cam in info["cams"].values()):
        return IMAGE_NOT_PREDICTED
    return 0


def main(argv=None):
    """Runs the command; returns dict(frames, failed, failed_frames, recall, ar)."""
    args = parse_args(argv)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    folder_exists = os.path.exists(args.folder)
    if world == 1 and folder_exists:
        print("%s already exists: pass a new --folder (nothing was written)" % args.folder)
        raise SystemExit(1)
    import torch
    import torch.distributed as dist
    device = None
    if world > 1:
        device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
        torch.cuda.set_device(device)
        dist.init_process_group("nccl", device_id=device)
    try:
        if world > 1:
            # every rank has looked before any rank creates the folder
            flag = torch.tensor([int(folder_exists)], device=device)
            dist.all_reduce(flag, op=dist.ReduceOp.MAX)
            if flag.item():
                if rank == 0:
                    print("%s already exists: pass a new --folder (nothing was written)" % args.folder)
                raise SystemExit(1)
        return _run(args, rank, world, device)
    finally:
        if world > 1:
            dist.destroy_process_group()


def _run(args, rank, world, device):
    import numpy as np
    import torch
    import torch.distributed as dist
    from . import extract
    log = print if rank == 0 else (lambda *a, **k: None)
    try:
        cfg = load_config(args.cfg_file, args.set_cfgs)
    except (OSError, KeyError, ValueError) as e:      # unreadable or unsupported config, bad --set
        if rank == 0:
            print(e.args[-1] if isinstance(e, KeyError) else e, file=sys.stderr)
        raise SystemExit(1)
    head = build_head(cfg, device=device)
    all_frames = build_feed(cfg, device=head.engine.device)
    n = len(all_frames)
    # each rank checks its own shard; the failure codes are then combined so that every rank runs the same frame list
    codes = np.zeros(n, np.int32)
    for i in extract.shard_indices(n, rank, world):
        codes[i] = check_frame(all_frames, head.image_detector, all_frames.infos[i])
    if world > 1:
        t = torch.from_numpy(codes).to(device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        codes = t.cpu().numpy()
    failed = [(frame_id(all_frames.infos[i]), FAILURES[int(codes[i])]) for i in np.flatnonzero(codes)]
    for fid, why in failed:
        log("skipped frame %s: %s" % (fid, why))
    feed = build_feed(cfg, infos=[all_frames.infos[i] for i in np.flatnonzero(codes == 0)], device=head.engine.device)
    _, recall, ar = extract.extract_nuscenes(feed, head.image_detector, head.engine, folder=args.folder,
                                             batch_frames=args.batch_frames, rank=rank, world=world,
                                             nms_thresh=args.nms_thresh, workers=args.workers,
                                             device=head.engine.device)
    log("frames written: %d (%s)" % (len(feed), args.folder))
    log("failed frames: %d" % len(failed))
    log("recall counters: %s" % json.dumps(recall))
    log("  ".join("AR@%s: %.4f" % (t, ar["rcnn_%s" % t]) for t in extract.THRESH))
    return dict(frames=len(feed), failed=len(failed), failed_frames=failed, recall=recall, ar=ar)


if __name__ == "__main__":
    main()
