"""End-to-end throughput of the commands on a KITTI config: ``extract_pseudo_labels`` over a synthetic KITTI tree,
and the tuner's shared pass against separate runs for 64 KITTI select-level settings.

Writes a reference-like tree (tools/cfgs, data/kitti) of --frames KITTI-sized synthetic frames under /dev/shm when it
has room: a 64-beam full scan of about 120k velodyne points per frame, of which the FOV filter keeps about an eighth,
P2 / R0 / Tr_velo2cam, and the COCO result file of the 2D boxes.  The frames are --distinct generated frames repeated
under distinct frame ids; each copy's velodyne and calib files are hard links of its frame's (they are read from the
page cache either way).

1. Extraction: the command's ``main`` in this process, a warm-up pass over --warmup frames, then the timed pass over
   every frame, the clock stopped when ``main`` returns (after the last .pth is written): frames/s of the whole
   command and of the pipeline alone (extract.extract_nuscenes).
2. Tuning: --tune_frames frames loaded once, then for the 64 settings dns_w x iou_w x dst_w (4 x 4 x 4, one group)
   per batch of --batch_frames: the shared path (one SeekerEngine.evaluate_settings) and the separate path (one
   engine per setting, execute with its recall counters), alternated --reps times in this process; the recall
   counters of every setting are checked equal.

Prints one JSON line with the GPU's name and power limit read in the same run.

    python tools/kitti_cli_e2e.py [--frames 4096] [--distinct 16] [--batch_frames 64] [--workers 4]
"""
import argparse
import contextlib
import copy
import json
import os
import pickle
import shutil
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from extract_cli_e2e import power_limit_w  # noqa: E402


def write_tree(root, pool, n):
    """root (DATA_PATH): n frames cycling through ``pool`` (make_kitti_frame(..., with_gt=True) tuples)."""
    from findnpropagate_b200 import synth
    coco_path = os.path.join(root, "kitti_coco_results.json")
    pool_infos = synth.write_kitti_tree(root, pool)
    coco = json.load(open(coco_path))
    by_image = {}
    for a in coco["annotations"]:
        by_image.setdefault(a["image_id"], []).append(a)
    infos = list(pool_infos)
    split = os.path.join(root, "training")
    for k in range(len(pool), n):
        j, idx = k % len(pool), "%06d" % k
        for sub, ext in (("velodyne", ".bin"), ("calib", ".txt")):
            os.link(os.path.join(split, sub, "%06d%s" % (j, ext)), os.path.join(split, sub, idx + ext))
        info = copy.deepcopy(pool_infos[j])
        info["point_cloud"]["lidar_idx"] = info["image"]["image_idx"] = idx
        infos.append(info)
        coco["images"].append(dict(id=k, file_name=idx + ".png"))
        coco["annotations"] += [dict(a, id=len(coco["annotations"]) + i, image_id=k) for i, a in enumerate(by_image.get(j, []))]
    with open(os.path.join(root, "kitti_infos_train.pkl"), "wb") as f:
        pickle.dump(infos, f)
    with open(coco_path, "w") as f:
        json.dump(coco, f)
    return infos


def tune(cli, cfg, frames_n, batch_frames, workers, reps):
    """(shared seconds per pass, separate seconds per pass, counters equal) over the first frames_n frames."""
    import numpy as np
    import torch
    from findnpropagate_b200 import tune_params
    from findnpropagate_b200.extract import THRESH
    from findnpropagate_b200.seeker import SeekerEngine
    head = cli.build_head(cfg)
    feed = cli.build_feed(cfg, device=head.engine.device)
    batches = [b[0] for b in feed.prefetch(range(frames_n), head.image_detector, batch_frames=batch_frames,
                                           workers=workers, xyz_only=True)]
    settings = [dict(dns_w=d, iou_w=i, dst_w=t) for d in (0.0, 0.05, 0.5, 1.0) for i in (0.25, 0.5, 0.95, 2.0)
                for t in (0.0, 0.1, 0.226, 0.5)]
    groups = tune_params.group_settings(head.params, settings, "kitti")
    assert len(groups) == 1 and len(groups[0]["settings"]) == 64
    shared_eng = SeekerEngine(groups[0]["params"], device=head.engine.device, box_format="xywh", variant="kitti")
    engines = [SeekerEngine(s, device=head.engine.device, box_format="xywh", variant="kitti") for s in groups[0]["settings"]]

    def shared():
        out = [None] * len(settings)
        for frames in batches:
            pts = torch.from_numpy(np.concatenate([f.points for f in frames])).to(shared_eng.device)
            gt = shared_eng.upload_gt(frames)
            res = shared_eng.evaluate_settings(shared_eng.plan(frames), pts, gt, groups[0]["settings"],
                                               recall_thresh=THRESH)["settings"]
            out = [r["recall"] if o is None else {k: o[k] + r["recall"][k] for k in o} for o, r in zip(out, res)]
        return out

    def separate():
        out = []
        for eng in engines:
            tot = None
            for frames in batches:
                pts = torch.from_numpy(np.concatenate([f.points for f in frames])).to(eng.device)
                r = eng.result(eng.execute(eng.plan(frames), pts, gt=eng.upload_gt(frames), recall_thresh=THRESH))["recall"]
                tot = r if tot is None else {k: tot[k] + r[k] for k in tot}
            out.append(tot)
        return out

    a, b = shared(), separate()          # warm-up, and the check
    equal = a == b
    ts, tp = [], []
    for _ in range(reps):
        for fn, acc in ((shared, ts), (separate, tp)):
            torch.cuda.synchronize()
            t = time.perf_counter()
            got = fn()
            torch.cuda.synchronize()
            acc.append(time.perf_counter() - t)
            equal = equal and got == a
    return min(ts), min(tp), equal, sum(len(b) for b in batches), a[0]["gt"]


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--frames", type=int, default=4096)
    ap.add_argument("--distinct", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=256)
    ap.add_argument("--batch_frames", type=int, default=64)
    ap.add_argument("--workers", type=int, default=4)
    ap.add_argument("--tune_frames", type=int, default=512)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    import numpy as np
    import torch
    import yaml
    if not torch.cuda.is_available():
        raise SystemExit("kitti_cli_e2e needs a CUDA device")
    from findnpropagate_b200 import extract, synth
    from findnpropagate_b200 import extract_pseudo_labels as cli

    scan = synth.SynthConfig("kitti64", 64, 2200, 1, 12, 4, 6, 1)
    need = a.distinct * 4 * 2 ** 20 + 2 ** 30
    shm = os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > need
    base = tempfile.mkdtemp(prefix="fnp_kitti_e2e_", dir="/dev/shm" if shm else None)
    cwd = os.getcwd()
    try:
        pool = [synth.make_kitti_frame(i, with_gt=True, cfg=scan, full_scan=True) for i in range(a.distinct)]
        root = os.path.join(base, "data", "kitti")
        infos = write_tree(root, pool, a.frames)
        with open(os.path.join(root, "kitti_infos_warm.pkl"), "wb") as f:
            pickle.dump(infos[:a.warmup], f)
        tools = os.path.join(base, "tools")
        os.makedirs(os.path.join(tools, "cfgs"))
        head = dict(CLASS_NAMES=list(synth.KITTI_CLASS_NAMES),
                    DATA_CONFIG=dict(DATASET="KittiDataset", DATA_PATH="../data/kitti", DATA_SPLIT=dict(train="train"),
                                     INFO_PATH=dict(train=["kitti_infos_train.pkl"]), FOV_POINTS_ONLY=True,
                                     POINT_CLOUD_RANGE=[0, -40, -3, 70.4, 40, 1]),
                    MODEL=dict(NAME="Seeker", DENSE_HEAD=dict(NAME="FrustumProposerOGKITTI",
                                                              PREDS_PATH="../data/kitti/kitti_coco_results.json",
                                                              PARAMS=dict(nms_3d=0.0, score_thr=0.45, nms_2d=0.4))))
        with open(os.path.join(tools, "cfgs", "e2e.yaml"), "w") as f:
            yaml.safe_dump(head, f)
        os.chdir(tools)
        args = ["--cfg_file", "cfgs/e2e.yaml", "--batch_frames", str(a.batch_frames), "--workers", str(a.workers)]

        spans = []
        run_pipeline = extract.extract_nuscenes

        def timed_pipeline(*p, **k):
            t = time.perf_counter()
            out = run_pipeline(*p, **k)
            torch.cuda.synchronize()
            spans.append(time.perf_counter() - t)
            return out
        extract.extract_nuscenes = timed_pipeline
        with contextlib.redirect_stdout(sys.stderr):         # the command's own log; stdout carries the JSON line
            cli.main(args + ["--folder", "../out_warm", "--set", "DATA_CONFIG.INFO_PATH.train", "['kitti_infos_warm.pkl']"])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = cli.main(args + ["--folder", "../out"])
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
        extract.extract_nuscenes = run_pipeline
        written = len(os.listdir(os.path.join(base, "out")))
        assert res["frames"] == a.frames and res["failed"] == 0 and written == a.frames, (res["frames"], written)
        feed = cli.build_feed(cli.load_config("cfgs/e2e.yaml"), device="cuda:0")
        kept = [feed[k]["points"].shape[0] for k in range(a.distinct)]
        with contextlib.redirect_stdout(sys.stderr):
            t_shared, t_separate, equal, tuned, tune_gt = tune(cli, cli.load_config("cfgs/e2e.yaml"),
                                                               min(a.tune_frames, a.frames), a.batch_frames, a.workers,
                                                               a.reps)
        print(json.dumps(dict(
            metric="kitti_extract_cli_frames_per_s", value=round(a.frames / wall, 1),
            pipeline_frames_per_s=round(a.frames / spans[-1], 1), wall_s=round(wall, 3), pipeline_s=round(spans[-1], 3),
            frames=a.frames, distinct_frames=a.distinct, velodyne_points_per_frame=int(np.mean([p[0].shape[0] for p in pool])),
            fov_points_per_frame=int(np.mean(kept)), batch_frames=a.batch_frames, workers=a.workers,
            tree_on="/dev/shm" if shm else tempfile.gettempdir(), gt=res["recall"]["gt"], ar_0_5=round(res["ar"]["rcnn_0.5"], 4),
            tune_settings=64, tune_frames=tuned, tune_shared_s=round(t_shared, 4), tune_separate_s=round(t_separate, 4),
            tune_speedup=round(t_separate / t_shared, 2), tune_counters_equal=bool(equal), tune_gt=tune_gt,
            host_cores=len(os.sched_getaffinity(0)), gpu=torch.cuda.get_device_name(), power_limit_w=power_limit_w())))
    finally:
        os.chdir(cwd)
        shutil.rmtree(base, ignore_errors=True)


if __name__ == "__main__":
    main()
