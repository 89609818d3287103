"""Throughput of scoring a grid of head settings: the shared path (stages 1-2c once per group of settings,
SeekerEngine.evaluate_settings) against one full SeekerEngine execution + recall counters per setting, on the same
resident points, timed alternately in one process.

Inputs: --frames distinct synthetic cfg2 frames (BASELINE.json configs[1]: ten sweeps, ~330k points, 60 GLIP boxes,
the 64 x 12 hypothesis grid), generated on the GPU and kept there, one batch.  Grids: (a) 64 settings that differ in
select-level values only (one group); (b) the same 64 settings at num_mags 64 and 48 (two groups).  The recall
counters and proposal counts of the two paths must be equal (exit status 1 otherwise).  Prints one JSON line per grid
with settings x frames / s of both paths, their ratio, the GPU's name and its power limit.

    python tools/tune_bench.py [--frames 256] [--reps 3] [--profile]
"""
import argparse
import itertools
import json
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)


def grid_a():
    terms = [dict(), dict(dst_w=0.2), dict(ego_w=0.1, occl_w=0.2), dict(MULT=True, dst_w=0.5)]
    return [dict(t, dns_w=d, iou_w=i, min_cam_iou=m)
            for d, i, m, t in itertools.product((0.5, 1.0, 2.0, 4.0), (0.5, 1.0), (0.3, 0.4), terms)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=256)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--profile", action="store_true",
                    help="after the timing, one shared pass of each grid under torch.profiler: device time per kernel")
    a = ap.parse_args()
    import numpy as np
    import torch
    from extract_cli_e2e import power_limit_w
    from findnpropagate_b200 import synth, tune_params
    from findnpropagate_b200.seeker import FrameInput, SeekerEngine, _Arena
    if not torch.cuda.is_available():
        sys.exit("tune_bench.py measures on a CUDA device; none is available")
    cfg = synth.CONFIGS["cfg2"]
    frames = []
    for i in range(a.frames):
        f = synth.make_frame(i, cfg, device="cuda:0")
        frames.append(FrameInput(points=f.points, lidar2image=f.lidar2image, camera2lidar=f.camera2lidar,
                                 camera_intrinsics=f.camera_intrinsics, det_boxes=f.det_boxes, det_labels=f.det_labels,
                                 det_scores=f.det_scores, det_cam_idx=f.det_cam_idx, gt_boxes=f.gt_boxes))
    base = synth.seeker_params(cfg)
    points = torch.from_numpy(np.concatenate([f.points for f in frames])).cuda()
    n_points = int(points.shape[0])
    for name, settings in (("a", grid_a()), ("b", [dict(s, num_mags=m) for m in (64, 48) for s in grid_a()])):
        groups = tune_params.group_settings(base, settings)
        shared = [SeekerEngine(g["params"], device="cuda:0") for g in groups]
        plans = [e.plan(frames) for e in shared]
        gt = shared[0].upload_gt(frames)
        arena = _Arena(torch.device("cuda:0"))       # the separate engines run one after another: one scratch
        separate = []
        for gi, g in enumerate(groups):
            for s in g["settings"]:
                e = SeekerEngine(s, device="cuda:0")
                e.arena = arena
                separate.append((gi, e))

        def run_shared():
            out = [None] * len(settings)
            for g, e, plan in zip(groups, shared, plans):
                res = e.evaluate_settings(plan, points, gt, g["settings"])
                for i, r in zip(g["members"], res["settings"]):
                    out[i] = (r["proposals"], r.get("recall"))
            return out

        def run_separate():
            out = [None] * len(settings)
            order = [i for g in groups for i in g["members"]]
            for i, (gi, e) in zip(order, separate):
                res = e.result(e.execute(plans[gi], points, gt=gt))
                out[i] = (int(res["cand_valid"].sum()), res.get("recall"))
            return out

        def timed(fn):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = fn()
            torch.cuda.synchronize()
            return time.perf_counter() - t0, r

        ref_shared, ref_separate = run_shared(), run_separate()          # warm-up: every shape, every allocation
        if ref_shared != ref_separate:
            bad = [settings[i] for i in range(len(settings)) if ref_shared[i] != ref_separate[i]]
            print(json.dumps(dict(grid=name, error="counters differ", settings=bad[:4])))
            sys.exit(1)
        t_sh, t_sep = [], []
        for _ in range(a.reps):
            dt, r = timed(run_shared)
            assert r == ref_shared
            t_sh.append(dt)
            dt, r = timed(run_separate)
            assert r == ref_separate
            t_sep.append(dt)
        work = len(settings) * a.frames
        sh, sep = work / min(t_sh), work / min(t_sep)
        print(json.dumps(dict(grid=name, settings=len(settings), groups=len(groups), frames=a.frames, points=n_points,
                              shared_setting_frames_per_s=round(sh, 1), separate_setting_frames_per_s=round(sep, 1),
                              ratio=round(sh / sep, 2), shared_s=[round(t, 4) for t in t_sh],
                              separate_s=[round(t, 4) for t in t_sep], counters_equal=True,
                              gpu=torch.cuda.get_device_name(), power_limit_w=power_limit_w())), flush=True)
        if a.profile:       # a run of its own, after the timed ones: tracing slows the host
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                dt, _ = timed(run_shared)
            kernels = {}
            for e in prof.key_averages():
                us = getattr(e, "self_device_time_total", None)
                us = getattr(e, "self_cuda_time_total", 0) if us is None else us
                if us > 0:
                    kernels[e.key] = dict(calls=e.count, ms=round(us / 1e3, 3))
            print(json.dumps(dict(grid=name, profiled_wall_s=round(dt, 4),
                                  device_ms_total=round(sum(k["ms"] for k in kernels.values()), 3),
                                  kernels=dict(sorted(kernels.items(), key=lambda kv: -kv[1]["ms"])))), flush=True)
        del shared, separate, arena
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
