"""End-to-end throughput of ``python -m findnpropagate_b200.extract_pseudo_labels`` from nuScenes-format files.

Writes a reference-like tree (tools/cfgs, data/nuscenes/v1.0-trainval, data/training_pred) of --frames cfg2-sized
synthetic frames (BASELINE.json configs[1]: ten sweeps, about 330k points and 60 GLIP boxes per frame, the 64 x 12
hypothesis grid) under /dev/shm when it has room, with the GLIP prediction file and COCO meta file for them.  The
frames are --distinct generated frames repeated under distinct frame ids, tokens and image paths; each copy's .bin is
a hard link of its frame's file, which keeps the tree small (the files are read from the page cache either way).

Runs the command's ``main`` in this process: a warm-up pass over --warmup frames into one folder, then the timed pass
over all frames into another, the clock stopped when ``main`` returns (after the last .pth is written).  Prints one
JSON line: frames/s of the whole command (config, GLIP file, info file, frame check, pipeline) and of the pipeline
alone (extract.extract_nuscenes: file reads, H2D, kernels, .pth writes), with the configuration, the host's core
count and the GPU's name and power limit read in the same run.

    python tools/extract_cli_e2e.py [--frames 8192] [--batch_frames 64] [--workers 4]
"""
import argparse
import contextlib
import dataclasses
import json
import os
import pickle
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def power_limit_w():
    """The current device's power limit in W (nvidia-smi query by UUID), None when it cannot be read."""
    import torch
    try:
        uuid = "GPU-%s" % torch.cuda.get_device_properties(torch.cuda.current_device()).uuid
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", uuid],
                             capture_output=True, text=True, timeout=60)
        return float(out.stdout.strip().splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        return None


def write_tree(base, pool, n):
    """base/data/...: n frames cycling through ``pool``; returns the info dicts."""
    from findnpropagate_b200 import synth
    root = os.path.join(base, "data", "nuscenes", "v1.0-trainval")
    pool_infos = synth.write_nuscenes_tree(root, pool)
    frames, infos = [], []
    for k in range(n):
        j = k % len(pool)
        if k < len(pool):
            f, info = pool[j], pool_infos[j]
        else:
            fid = "n%03d-e2e__LIDAR_TOP__%010d.pcd" % (k % 1000, k)
            f = dataclasses.replace(pool[j], frame_id=fid, token="e2e%08d" % k,
                                    image_paths=["samples/%s/%s__%s.jpg" % (c, fid, c) for c in synth.CAM_NAMES])
            rel = os.path.join("samples", "LIDAR_TOP", fid + ".bin")
            os.link(os.path.join(root, pool_infos[j]["lidar_path"]), os.path.join(root, rel))
            cams = {name: dict(cam, data_path=f.image_paths[c]) for c, (name, cam) in enumerate(pool_infos[j]["cams"].items())}
            info = dict(pool_infos[j], lidar_path=rel, token=f.token, cams=cams)
        frames.append(f)
        infos.append(info)
    synth.write_glip_predictions(frames, os.path.join(base, "data", "training_pred", "nuscenes_glip_train_pred.pth"),
                                 os.path.join(base, "data", "training_pred", "nuscenes_infos_train_mono3d.coco.json"))
    return infos


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--frames", type=int, default=8192)
    ap.add_argument("--distinct", type=int, default=64)
    ap.add_argument("--warmup", type=int, default=256)
    ap.add_argument("--batch_frames", type=int, default=64)
    ap.add_argument("--workers", type=int, default=4)
    a = ap.parse_args()
    import torch
    import yaml
    if not torch.cuda.is_available():
        raise SystemExit("extract_cli_e2e needs a CUDA device")
    from findnpropagate_b200 import extract, synth
    from findnpropagate_b200 import extract_pseudo_labels as cli

    cfg = synth.CONFIGS["cfg2"]
    need = a.distinct * 8 * 2 ** 20 + 2 ** 30
    shm = os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > need
    base = tempfile.mkdtemp(prefix="fnp_extract_e2e_", dir="/dev/shm" if shm else None)
    cwd = os.getcwd()
    try:
        pool = [synth.make_frame(i, cfg, device="cuda:0") for i in range(a.distinct)]
        infos = write_tree(base, pool, a.frames)
        root = os.path.join(base, "data", "nuscenes", "v1.0-trainval")
        for name, part in (("nuscenes_infos_e2e_train.pkl", infos), ("nuscenes_infos_e2e_warm.pkl", infos[:a.warmup])):
            with open(os.path.join(root, name), "wb") as f:
                pickle.dump(part, f)
        tools = os.path.join(base, "tools")
        os.makedirs(os.path.join(tools, "cfgs"))
        head = dict(CLASS_NAMES=list(synth.CLASS_NAMES),
                    DATA_CONFIG=dict(DATASET="NuScenesDataset", DATA_PATH="../data/nuscenes", VERSION="v1.0-trainval",
                                     MAX_SWEEPS=1, INFO_PATH=dict(train=["nuscenes_infos_e2e_train.pkl"]),
                                     POINT_CLOUD_RANGE=[-54.0, -54.0, -5.0, 54.0, 54.0, 3.0]),
                    MODEL=dict(NAME="TransFusion", DENSE_HEAD=dict(NAME="FrustumProposerOG", PREDS_PATH="PreprocessedGLIP",
                                                                   BOX_FORMAT="xyxy", PARAMS=synth.seeker_params(cfg))))
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
            cli.main(args + ["--folder", "../out_warm", "--set", "DATA_CONFIG.INFO_PATH.train",
                             "['nuscenes_infos_e2e_warm.pkl']"])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = cli.main(args + ["--folder", "../out"])
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
        extract.extract_nuscenes = run_pipeline
        written = len(os.listdir(os.path.join(base, "out")))
        assert res["frames"] == a.frames and res["failed"] == 0 and written == a.frames, (res["frames"], written)
        print(json.dumps(dict(
            metric="extract_cli_e2e_frames_per_s", value=round(a.frames / wall, 1),
            pipeline_frames_per_s=round(a.frames / spans[-1], 1), wall_s=round(wall, 3), pipeline_s=round(spans[-1], 3),
            frames=a.frames, distinct_frames=a.distinct, config="cfg2", points_per_frame=int(sum(f.points.shape[0] for f in pool) / len(pool)),
            batch_frames=a.batch_frames, workers=a.workers, nms_thresh=None, tree_on="/dev/shm" if shm else tempfile.gettempdir(),
            host_cores=len(os.sched_getaffinity(0)), gpu=torch.cuda.get_device_name(), power_limit_w=power_limit_w(),
            gt=res["recall"]["gt"], ar_0_5=round(res["ar"]["rcnn_0.5"], 4))))
    finally:
        os.chdir(cwd)
        shutil.rmtree(base, ignore_errors=True)


if __name__ == "__main__":
    main()
