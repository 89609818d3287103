"""Per-stage device times of the fused seeker pipeline (CUDA events, warm, run under gpurun).

    python tools/stage_times.py [--config cfg2] [--frames 32] [--iters 10]

Each C-ABI stage entry point is timed alone on the current stream over the same batch;
host-side planning (2D NMS, camera matrices, tables) is timed with perf_counter.
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, ROOT)
from bench import make_frames  # noqa: E402
from findnpropagate_b200 import _lib  # noqa: E402
from findnpropagate_b200.seeker import SeekerEngine  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="cfg2")
    ap.add_argument("--frames", type=int, default=32)
    ap.add_argument("--distinct", type=int, default=8)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--split-points", type=int, default=None)
    ap.add_argument("--score-mode", default="auto", choices=["auto", "direct", "sweep"])
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    frames, params = make_frames(a.config, 0, a.distinct, str(dev))
    batch = [frames[i % a.distinct] for i in range(a.frames)]
    eng = SeekerEngine(params, device=dev, split_points=a.split_points, score_mode=a.score_mode)
    t0 = time.perf_counter()
    for _ in range(5):
        plan = eng.plan(batch)
    host_plan_ms = (time.perf_counter() - t0) / 5 * 1e3
    pts = eng.upload_points(batch)
    gt = eng.upload_gt(batch)
    h = eng.execute(plan, pts, nms_thresh=0.1, gt=gt)
    t0 = time.perf_counter()
    res = eng.finish(h)
    host_finish_ms = (time.perf_counter() - t0) * 1e3
    stream = _lib.current_stream(dev)
    cfg, b = C.byref(eng.cfg), C.byref(h["batch"])
    L = _lib.lib
    stages = [("cull", L.fnp_seeker_cull), ("frustum_stats", L.fnp_seeker_frustum_stats),
              ("hypotheses", L.fnp_seeker_hypotheses), ("score", L.fnp_seeker_score), ("select", L.fnp_seeker_select),
              ("run(all five)", L.fnp_seeker_run)]
    out = {"config": a.config, "frames": a.frames, "score_mode": eng.last_score_mode, "split_points": h["sp"], "F": plan["F"], "H": eng.H, "host_plan_ms": host_plan_ms,
           "host_finish_ms": host_finish_ms, "sum_P_f": int(res["cand_npts"].sum()),
           "valid_hyps": int(res["cand_nvalid"].sum()),
           "tests": int((res["cand_npts"].astype(np.int64) * res["cand_nvalid"]).sum()), "stages_ms": {}}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for name, fn in stages:
        for _ in range(2):
            fn(cfg, b, stream)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(a.iters):
            rc = fn(cfg, b, stream)
            assert rc == 0
        e1.record()
        torch.cuda.synchronize()
        out["stages_ms"][name] = e0.elapsed_time(e1) / a.iters
    # stage 4 + recall, timed through the engine helpers
    for name, fn in (("seg_nms", lambda: eng._stage4_nms(h, 0.1, stream)),
                     ("recall", lambda: eng._recall(h, gt, (0.3, 0.5, 0.7), stream))):
        fn(); torch.cuda.synchronize()
        e0.record()
        for _ in range(a.iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        out["stages_ms"][name] = e0.elapsed_time(e1) / a.iters
    # H2D bandwidth of the point buffer from pinned memory
    pin = torch.empty(pts.shape, dtype=torch.float32, pin_memory=True)
    pts.copy_(pin); torch.cuda.synchronize()
    e0.record()
    for _ in range(5):
        pts.copy_(pin, non_blocking=True)
    e1.record(); torch.cuda.synchronize()
    out["h2d_GBps"] = pts.numel() * 4 * 5 / (e0.elapsed_time(e1) * 1e-3) / 1e9
    out["points_bytes"] = pts.numel() * 4
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
