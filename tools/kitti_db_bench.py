"""Throughput of the KITTI databases: the every-box crop of gt_database.crop_frames(every_box=True) against the matrix
path it replaces, and the whole create_kitti_pseudo_database command from files.

Inputs: --distinct synthetic 64-beam full KITTI scans (SynthConfig("kitti64", 64, 2200, ...), about 123k points each,
no FOV filter), each with 30 boxes: its GT boxes, jittered copies of some of them (overlapping the originals), then
boxes of 1-5 m centred on random points of the scan.

  * crop step, per batch of --batch frames from host arrays to per-box host arrays: the new path (fnp_crop_all_count,
    one 8-byte read, fnp_crop_all_scatter, then only the rows in boxes back) against the matrix path, the reference's
    per frame: points_in_boxes_cpu (here on the device: the (G, N) int32 matrix), its D2H, then
    ``pts[mask[i] > 0]`` and the centre subtraction per box on the host.  The two alternate over --reps repetitions
    (host clock; both end in a D2H, which synchronises).  Exit status 1 when any box's bytes differ.  The device time
    of the crop calls alone on resident inputs is timed with CUDA events.
  * the command: a tree on /dev/shm (when it has room) of --frames frames (scan k is scan k % --distinct), one .pth
    of the scan's 30 boxes per frame; a warm-up run over --batch frames, then the timed run over all frames, which
    ends after the pickle is written.

Prints one JSON line with frames/s of both crop paths, the crop calls' device time, the command's frames/s, the GPU's
name and its power limit.

    python tools/kitti_db_bench.py [--distinct 16] [--frames 256] [--batch 16] [--reps 20] [--workers 4]
"""
import argparse
import contextlib
import json
import os
import pickle
import shutil
import sys
import tempfile
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

N_BOXES = 30


def make_boxes(pts, gt, rng, n=N_BOXES):
    """(n, 7) float32 and labels 1..7: the GT boxes (up to a third of n), jittered copies of them, then boxes of
    1-5 m centred on random points of the scan."""
    import numpy as np
    g = np.asarray(gt, np.float32)[:n // 3, :7]
    jit = g + rng.normal(0, 0.3, g.shape).astype(np.float32) * [1, 1, 0.1, 0.2, 0.2, 0.1, 0.3]
    k = n - 2 * g.shape[0]
    c = pts[rng.integers(0, pts.shape[0], k), :3]
    rnd = np.concatenate([c, rng.uniform(1, 5, (k, 3)), rng.uniform(-3, 3, (k, 1))], 1)
    boxes = np.concatenate([g, jit, rnd]).astype(np.float32)
    return boxes, rng.integers(1, 8, n).astype(np.int32)


def matrix_crop(points_list, boxes_list):
    """The reference's crop, per frame: points_in_boxes_cpu's (G, N) matrix, then pts[mask[i] > 0] per box."""
    from findnpropagate_b200.pcdet_ops import roiaware_pool3d_utils
    out = []
    for pts, boxes in zip(points_list, boxes_list):
        mask = roiaware_pool3d_utils.points_in_boxes_cpu(pts[:, 0:3], boxes[:, 0:7])
        per = []
        for i in range(boxes.shape[0]):
            g = pts[mask[i] > 0]
            g[:, :3] -= boxes[i, :3]
            per.append(g)
        out.append(per)
    return out


def write_tree(base, scans, cals, boxes, labels, n):
    """base/data/kitti (training/velodyne, training/calib, kitti_infos_*.pkl), base/pseudo, base/tools/cfgs."""
    import numpy as np
    import yaml
    from findnpropagate_b200 import extract, synth
    root = os.path.join(base, "data", "kitti")
    for sub in ("velodyne", "calib"):
        os.makedirs(os.path.join(root, "training", sub))
    os.makedirs(os.path.join(base, "pseudo"))
    infos = []
    for k in range(n):
        s = k % len(scans)
        idx = "%06d" % k
        scans[s].tofile(os.path.join(root, "training", "velodyne", idx + ".bin"))
        P2, R0, V2C = (np.asarray(cals[s][m], np.float32) for m in ("P2", "R0", "Tr_velo2cam"))
        rows = [("P0", P2), ("P1", P2), ("P2", P2), ("P3", P2), ("R0_rect", R0), ("Tr_velo_to_cam", V2C),
                ("Tr_imu_to_velo", V2C)]
        with open(os.path.join(root, "training", "calib", idx + ".txt"), "w") as fh:
            fh.write("".join("%s: %s\n" % (m, " ".join(repr(float(v)) for v in a.reshape(-1))) for m, a in rows))
        infos.append(dict(point_cloud=dict(num_features=4, lidar_idx=idx),
                          image=dict(image_idx=idx, image_shape=np.array(synth.KITTI_IMAGE_SHAPE, np.int32))))
        extract.save_frame(os.path.join(base, "pseudo"), idx,
                           dict(pred_boxes=boxes[s], pred_scores=np.linspace(1, 0.5, N_BOXES, dtype=np.float32),
                                pred_labels=labels[s]))
    for name, part in (("kitti_infos_train.pkl", infos), ("kitti_infos_warm.pkl", infos[:16])):
        with open(os.path.join(root, name), "wb") as fh:
            pickle.dump(part, fh)
    cfg = dict(CLASS_NAMES=list(synth.KITTI_CLASS_NAMES),
               DATA_CONFIG=dict(DATASET="KittiDataset", DATA_PATH="../data/kitti", DATA_SPLIT=dict(train="train"),
                                INFO_PATH=dict(train=["kitti_infos_train.pkl"])),
               MODEL=dict(NAME="Seeker", DENSE_HEAD=dict(NAME="FrustumProposerOGKITTI")))
    os.makedirs(os.path.join(base, "tools", "cfgs"))
    with open(os.path.join(base, "tools", "cfgs", "db.yaml"), "w") as fh:
        yaml.safe_dump(cfg, fh)
    return root


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--distinct", type=int, default=16)
    ap.add_argument("--frames", type=int, default=256)
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--workers", type=int, default=4)
    a = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("kitti_db_bench.py measures on a CUDA device; none is available")
    from extract_cli_e2e import power_limit_w
    from findnpropagate_b200 import gt_database, synth
    from findnpropagate_b200 import create_kitti_pseudo_database as cli

    scan = synth.SynthConfig("kitti64", 64, 2200, 1, 12, 4, 6, 1)
    rng = np.random.default_rng(0)
    scans, cals, boxes, labels = [], [], [], []
    for i in range(a.distinct):
        pts, cal, _, _, _, gt = synth.make_kitti_frame(i, with_gt=True, cfg=scan, full_scan=True)
        pts = np.ascontiguousarray(pts, np.float32)
        b, lab = make_boxes(pts, gt, rng)
        scans.append(pts)
        cals.append(cal)
        boxes.append(b)
        labels.append(lab)
    pts_b = [scans[k % a.distinct] for k in range(a.batch)]
    box_b = [boxes[k % a.distinct] for k in range(a.batch)]

    new = gt_database.crop_frames(pts_b, box_b, every_box=True)
    old = matrix_crop(pts_b, box_b)
    same = all(x.tobytes() == y.tobytes() for pn, po in zip(new, old) for x, y in zip(pn, po))
    if not same:
        print(json.dumps(dict(error="crop outputs differ")))
        sys.exit(1)
    rows_in_boxes = sum(x.shape[0] for per in new for x in per)
    t_new, t_old = [], []
    for _ in range(a.reps):
        for fn, acc in ((lambda p, b: gt_database.crop_frames(p, b, every_box=True), t_new), (matrix_crop, t_old)):
            torch.cuda.synchronize()
            t = time.perf_counter()
            fn(pts_b, box_b)
            acc.append(time.perf_counter() - t)

    # the two crop calls alone on resident inputs (the host-side box prep and the 8-byte read included)
    d_pts = torch.from_numpy(np.concatenate(pts_b)).cuda()
    bcat = np.concatenate(box_b)
    d_box, d_cen = torch.from_numpy(bcat).cuda(), torch.from_numpy(bcat[:, :3].astype(np.float64)).cuda()
    rs = np.concatenate([[0], np.cumsum([p.shape[0] for p in pts_b])])
    bs = np.concatenate([[0], np.cumsum([b.shape[0] for b in box_b])])
    gt_database.crop_points_in_boxes_all(d_pts, rs, d_box, d_cen, bs)
    dev_ms = []
    for _ in range(a.reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        gt_database.crop_points_in_boxes_all(d_pts, rs, d_box, d_cen, bs)
        e1.record()
        e1.synchronize()
        dev_ms.append(e0.elapsed_time(e1))
    matrix_bytes = sum(4 * p.shape[0] * b.shape[0] for p, b in zip(pts_b, box_b))

    need = sum(s.nbytes for s in scans) * (a.frames // a.distinct + 1) * 3 + 2 ** 30
    shm = os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > need
    base = tempfile.mkdtemp(prefix="fnp_kitti_db_", dir="/dev/shm" if shm else None)
    cwd = os.getcwd()
    try:
        root = write_tree(base, scans, cals, boxes, labels, a.frames)
        os.chdir(os.path.join(base, "tools"))
        args = ["--cfg_file", "cfgs/db.yaml", "--folder", "../pseudo", "--workers", str(a.workers),
                "--batch_frames", str(a.batch)]
        with contextlib.redirect_stdout(sys.stderr):
            cli.main(args + ["--set", "DATA_CONFIG.INFO_PATH.train", "['kitti_infos_warm.pkl']"])
            for p in cli.output_paths(root, "train"):
                shutil.rmtree(p) if os.path.isdir(p) else os.remove(p)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = cli.main(args)
            wall = time.perf_counter() - t0
        assert res["frames"] == a.frames and sum(res["boxes"].values()) == N_BOXES * a.frames, res
    finally:
        os.chdir(cwd)
        shutil.rmtree(base, ignore_errors=True)
    med_new, med_old = float(np.median(t_new)), float(np.median(t_old))
    print(json.dumps(dict(
        distinct_scans=a.distinct, frames=a.frames, batch=a.batch, boxes_per_frame=N_BOXES,
        points_per_frame=int(np.mean([s.shape[0] for s in scans])), rows_in_boxes_per_batch=int(rows_in_boxes),
        matrix_mb_per_batch=round(matrix_bytes / 2 ** 20, 1), outputs_equal=True,
        crop_new_frames_per_s=round(a.batch / med_new, 1), crop_matrix_frames_per_s=round(a.batch / med_old, 1),
        crop_speedup=round(med_old / med_new, 2), crop_new_ms=round(1e3 * med_new, 2),
        crop_matrix_ms=round(1e3 * med_old, 2), crop_calls_device_ms=round(float(np.median(dev_ms)), 3),
        command_frames_per_s=round(a.frames / wall, 1), command_wall_s=round(wall, 3),
        tree_on="/dev/shm" if shm else tempfile.gettempdir(), workers=a.workers,
        host_cores=len(os.sched_getaffinity(0)), gpu=torch.cuda.get_device_name(), power_limit_w=power_limit_w())),
        flush=True)


if __name__ == "__main__":
    main()
