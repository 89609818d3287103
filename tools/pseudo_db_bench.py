"""Throughput of the pseudo-label database: the crop step of gt_database.crop_frames against the path it replaced, and
the whole create_pseudo_database command from files.

Inputs: --frames synthetic cfg2 frames (BASELINE.json configs[1]: ten sweeps, about 330k points per frame), each with
50 boxes (its GT boxes, then random boxes around its points), generated on the GPU and kept in host memory.

  * crop step, per batch of --batch frames from host arrays to per-box host arrays: the new path (one
    fnp_crop_points_in_boxes call: H2D, kernels, the counts and then only the rows in boxes back) against the path it
    replaced, restated here: host-side padding to (B, M, 3) / (B, T, 7), one padded points_in_boxes_gpu launch, the
    D2H of the (B, M) box indices, then ``pts[box_of_pt == i]`` and the centre subtraction per box on the host.  The
    two alternate over --reps repetitions (host clock; both end in a D2H, which synchronises).  Exit status 1 when any
    box's bytes differ.  The device time of the crop call alone on resident inputs is timed with CUDA events; the
    JSON line says whether those inputs fit in the 126 MB L2.
  * the command: a tree on /dev/shm (when it has room) whose key frames hold a tenth of each frame's points and
    whose nine listed sweeps (identity transforms) hold the rest, one .pth of the frame's 50 boxes per frame,
    MAX_SWEEPS 10; a warm-up run over --batch frames, then the timed run over all frames, which ends after the pickle
    is written.

Prints one JSON line with frames/s of both crop paths, the crop call's device time, the command's frames/s, the
GPU's name and its power limit.

    python tools/pseudo_db_bench.py [--frames 64] [--batch 16] [--reps 20] [--workers 4]
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

L2_BYTES = 126 * 2 ** 20


def make_boxes(f, rng, n=50):
    """(n, 7) float32: the frame's GT boxes, then boxes of 1-5 m centred on random points of the frame; labels 1..10."""
    import numpy as np
    gt = np.asarray(f.gt_boxes, np.float32)[:n]
    k = n - gt.shape[0]
    c = f.points[rng.integers(0, f.points.shape[0], k), :3]
    rnd = np.concatenate([c, rng.uniform(1, 5, (k, 3)), rng.uniform(-3, 3, (k, 1))], 1)
    boxes = np.concatenate([gt[:, :7], rnd]).astype(np.float32)
    labels = np.concatenate([gt[:, -1], rng.integers(1, 11, k)]).astype(np.int32)
    return boxes, labels


def old_crop(points_list, boxes_list):
    """The crop of create_groundtruth_database before fnp_crop_points_in_boxes."""
    import numpy as np
    import torch
    from findnpropagate_b200.pcdet_ops import roiaware_pool3d_utils
    B = len(points_list)
    M = max(max(p.shape[0] for p in points_list), 1)
    T = max(max(g.shape[0] for g in boxes_list), 1)
    pts = np.full((B, M, 3), 1.0e6, np.float32)
    boxes = np.zeros((B, T, 7), np.float32)
    boxes[:, :, 0:3] = -1.0e6
    for b in range(B):
        pts[b, :points_list[b].shape[0]] = points_list[b][:, 0:3]
        boxes[b, :boxes_list[b].shape[0]] = boxes_list[b][:, 0:7]
    idx = roiaware_pool3d_utils.points_in_boxes_gpu(torch.from_numpy(pts).cuda(), torch.from_numpy(boxes).cuda())
    idx = idx.long().cpu().numpy()
    out = []
    for b in range(B):
        box_of_pt = idx[b, :points_list[b].shape[0]]
        per = []
        for i in range(boxes_list[b].shape[0]):
            g = points_list[b][box_of_pt == i]
            g[:, :3] -= boxes_list[b][i, :3]
            per.append(g)
        out.append(per)
    return out


def write_tree(base, frames, boxes, labels):
    """base/data/nuscenes/v1.0-trainval with ten files per frame, base/pseudo with one .pth per frame, base/tools/cfgs."""
    import numpy as np
    import yaml
    from findnpropagate_b200 import extract, synth
    root = os.path.join(base, "data", "nuscenes", "v1.0-trainval")
    parts = [np.array_split(f.points, 10) for f in frames]
    keys = [synth.Frame(**dict(f.__dict__, points=p[0])) for f, p in zip(frames, parts)]
    infos = synth.write_nuscenes_tree(root, keys)
    for f, p, info in zip(frames, parts, infos):
        info["sweeps"] = []
        for k in range(1, 10):
            rel = os.path.join("sweeps", "LIDAR_TOP", "%s_%d.bin" % (f.frame_id, k))
            os.makedirs(os.path.join(root, os.path.dirname(rel)), exist_ok=True)
            np.ascontiguousarray(p[k], np.float32).tofile(os.path.join(root, rel))
            info["sweeps"].append(dict(lidar_path=rel, transform_matrix=np.eye(4), time_lag=0.05 * k))
    for name, part in (("infos_all.pkl", infos), ("infos_warm.pkl", infos[:4])):
        with open(os.path.join(root, name), "wb") as fh:
            pickle.dump(part, fh)
    os.makedirs(os.path.join(base, "pseudo"))
    for f, b, lab in zip(frames, boxes, labels):
        extract.save_frame(os.path.join(base, "pseudo"), f.frame_id,
                           dict(pred_boxes=b, pred_scores=np.linspace(1, 0.5, b.shape[0], dtype=np.float32),
                                pred_labels=lab))
    cfg = dict(CLASS_NAMES=list(synth.CLASS_NAMES),
               DATA_CONFIG=dict(DATASET="NuScenesDataset", DATA_PATH="../data/nuscenes", VERSION="v1.0-trainval",
                                MAX_SWEEPS=10, INFO_PATH=dict(train=["infos_all.pkl"])),
               MODEL=dict(NAME="TransFusion", DENSE_HEAD=dict(NAME="FrustumProposerOG")))
    os.makedirs(os.path.join(base, "tools", "cfgs"))
    with open(os.path.join(base, "tools", "cfgs", "db.yaml"), "w") as fh:
        yaml.safe_dump(cfg, fh)
    return root


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--workers", type=int, default=4)
    a = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("pseudo_db_bench.py measures on a CUDA device; none is available")
    from extract_cli_e2e import power_limit_w
    from findnpropagate_b200 import gt_database, synth
    from findnpropagate_b200 import create_pseudo_database as cli

    rng = np.random.default_rng(0)
    frames = []
    for i in range(a.frames):
        f = synth.make_frame(i, synth.CONFIGS["cfg2"], device="cuda:0")
        f.points = np.ascontiguousarray(f.points, np.float32)
        frames.append(f)
    boxes, labels = zip(*[make_boxes(f, rng) for f in frames])
    pts_b, box_b = [f.points for f in frames[:a.batch]], list(boxes[:a.batch])

    new = gt_database.crop_frames(pts_b, box_b)
    old = old_crop(pts_b, box_b)
    same = all(x.tobytes() == y.tobytes() for pn, po in zip(new, old) for x, y in zip(pn, po))
    if not same:
        print(json.dumps(dict(error="crop outputs differ")))
        sys.exit(1)
    t_new, t_old = [], []
    for _ in range(a.reps):
        for fn, acc in ((gt_database.crop_frames, t_new), (old_crop, t_old)):
            torch.cuda.synchronize()
            t = time.perf_counter()
            fn(pts_b, box_b)
            acc.append(time.perf_counter() - t)

    # the crop call alone on resident inputs
    d_pts = torch.from_numpy(np.concatenate(pts_b)).cuda()
    bcat = np.concatenate(box_b)
    d_box, d_cen = torch.from_numpy(bcat).cuda(), torch.from_numpy(bcat[:, :3].astype(np.float64)).cuda()
    rs = np.concatenate([[0], np.cumsum([p.shape[0] for p in pts_b])])
    bs = np.concatenate([[0], np.cumsum([b.shape[0] for b in box_b])])
    gt_database.crop_points_in_boxes(d_pts, rs, d_box, d_cen, bs)
    dev_ms = []
    for _ in range(a.reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        counts, _, _ = gt_database.crop_points_in_boxes(d_pts, rs, d_box, d_cen, bs)
        e1.record()
        e1.synchronize()
        dev_ms.append(e0.elapsed_time(e1))
    in_bytes = d_pts.numel() * 4 + d_box.numel() * 4 + d_cen.numel() * 8

    need = sum(f.points.nbytes for f in frames) * 3 + 2 ** 30
    shm = os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > need
    base = tempfile.mkdtemp(prefix="fnp_pseudo_db_", dir="/dev/shm" if shm else None)
    cwd = os.getcwd()
    try:
        root = write_tree(base, frames, boxes, labels)
        os.chdir(os.path.join(base, "tools"))
        args = ["--cfg_file", "cfgs/db.yaml", "--folder", "../pseudo", "--workers", str(a.workers),
                "--batch_frames", str(a.batch)]
        with contextlib.redirect_stdout(sys.stderr):
            cli.main(args + ["--set", "DATA_CONFIG.INFO_PATH.train", "['infos_warm.pkl']"])
            for p in cli.output_paths(root, 10):
                shutil.rmtree(p) if os.path.isdir(p) else os.remove(p)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = cli.main(args)
            wall = time.perf_counter() - t0
        assert res["frames"] == a.frames and sum(res["boxes"].values()) == 50 * a.frames, res
    finally:
        os.chdir(cwd)
        shutil.rmtree(base, ignore_errors=True)
    med_new, med_old = float(np.median(t_new)), float(np.median(t_old))
    print(json.dumps(dict(
        frames=a.frames, batch=a.batch, boxes_per_frame=50,
        points_per_frame=int(np.mean([f.points.shape[0] for f in frames])),
        points_in_boxes_per_batch=int(counts.sum().item()), outputs_equal=True,
        crop_new_frames_per_s=round(a.batch / med_new, 1), crop_old_frames_per_s=round(a.batch / med_old, 1),
        crop_speedup=round(med_old / med_new, 2), crop_new_ms=round(1e3 * med_new, 2), crop_old_ms=round(1e3 * med_old, 2),
        crop_call_device_ms=round(float(np.median(dev_ms)), 3), crop_call_inputs_mb=round(in_bytes / 2 ** 20, 1),
        crop_call_inputs_fit_l2=in_bytes < L2_BYTES,
        command_frames_per_s=round(a.frames / wall, 1), command_wall_s=round(wall, 3),
        tree_on="/dev/shm" if shm else tempfile.gettempdir(), workers=a.workers,
        host_cores=len(os.sched_getaffinity(0)), gpu=torch.cuda.get_device_name(), power_limit_w=power_limit_w())),
        flush=True)


if __name__ == "__main__":
    main()
