"""Device time of the per-class / per-range quality counters against the per-setting counters the tuner launches today:
one fnp_quality_counters launch over all settings, against one fnp_recall_counters and one fnp_precision_counters
launch per setting (SeekerEngine._select_multi), on the same per-setting proposals, timed with CUDA events and
alternated in one process.

Inputs: the tune_bench.py setup -- --frames distinct synthetic cfg2 frames (BASELINE.json configs[1]) resident on the
GPU, one batch, and its 64 select-level settings (one group); the per-setting proposals are those of
SeekerEngine.execute(settings=...).  Exit status 1 when the tables' sums differ from the per-setting counters.
Prints one JSON line with both times, their ratio, the GPU's name and its power limit.

    python tools/quality_bench.py [--frames 256] [--reps 20]
"""
import argparse
import ctypes as C
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=256)
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    import numpy as np
    import torch
    from extract_cli_e2e import power_limit_w
    from tune_bench import grid_a
    from findnpropagate_b200 import _lib, quality, synth, tune_params
    from findnpropagate_b200.seeker import FrameInput, SeekerEngine
    if not torch.cuda.is_available():
        sys.exit("quality_bench.py measures on a CUDA device; none is available")
    cfg = synth.CONFIGS["cfg2"]
    frames = []
    for i in range(a.frames):
        f = synth.make_frame(i, cfg, device="cuda:0")
        frames.append(FrameInput(points=f.points, lidar2image=f.lidar2image, camera2lidar=f.camera2lidar,
                                 camera_intrinsics=f.camera_intrinsics, det_boxes=f.det_boxes, det_labels=f.det_labels,
                                 det_scores=f.det_scores, det_cam_idx=f.det_cam_idx, gt_boxes=f.gt_boxes))
    groups = tune_params.group_settings(synth.seeker_params(cfg), grid_a())
    assert len(groups) == 1
    settings = groups[0]["settings"]
    S = len(settings)
    eng = SeekerEngine(groups[0]["params"], device="cuda:0")
    plan = eng.plan(frames)
    points = torch.from_numpy(np.concatenate([f.points for f in frames])).cuda()
    gt_boxes, gt_start, max_gt = gt = eng.upload_gt(frames)
    spec = quality.QualitySpec(synth.CLASS_NAMES)
    quality.check_labels(spec, plan["cand_label"], gt_boxes.cpu().numpy(), gt_start.cpu().numpy())
    while True:     # the per-setting proposals stay in the engine's output block
        h = eng.execute(plan, points, gt=gt, settings=settings)
        try:
            res = eng.finish(h)
            break
        except OverflowError as err:
            eng.pts_factor = max(eng.pts_factor * 1.5, 1.25 * int(err.args[0]) / plan["total_rows"])
    F, B, meta = plan["F"], plan["B"], h["meta"]
    ob = h["out_dev"].data_ptr() + h["off_sel"]
    boxes, best = ob, ob + 32 * S * F
    max_k = max(plan["max_cands"], 1)
    stream = _lib.current_stream()
    th = (C.c_float * 3)(*spec.thresh)
    q_out = torch.zeros((S, spec.n_counters), dtype=torch.int64, device="cuda")
    rec_out = torch.zeros((S, 20), dtype=torch.int64, device="cuda")
    prec_out = torch.zeros((S, 4), dtype=torch.int64, device="cuda")

    def one_launch():
        q_out.zero_()
        quality.launch(spec, boxes, meta["cand_label"], meta["frame_cand_start"], gt_boxes, gt_start, B, max_k, max_gt,
                       q_out, n_settings=S, pred_valid=best, pred_stride=F, valid_stride=F, stream=stream)

    def per_setting():
        rec_out.zero_()
        prec_out.zero_()
        for s in range(S):
            for fn, out in ((_lib.lib.fnp_recall_counters, rec_out), (_lib.lib.fnp_precision_counters, prec_out)):
                _lib.check(fn(boxes + 28 * s * F, best + 4 * s * F, meta["frame_cand_start"], gt_boxes.data_ptr(),
                              gt_start.data_ptr(), B, max_k, int(max_gt), th, 3, out[s].data_ptr(), stream), fn.__name__)

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1)

    one_launch(), per_setting()             # warm-up
    torch.cuda.synchronize()
    q, rc, pc = q_out.cpu().numpy(), rec_out.cpu().numpy(), prec_out.cpu().numpy()
    for s in range(S):
        p = quality.precision_dict(q[s], spec)
        if (quality.recall_dict(q[s], spec) != SeekerEngine.recall_dict(rc[s]) or
                [p["proposals"], p["hits_0.3"], p["hits_0.5"], p["hits_0.7"]] != pc[s].tolist() or
                SeekerEngine.recall_dict(rc[s]) != res["settings"][s]["recall"]):
            print(json.dumps(dict(error="counters differ", setting=settings[s])))
            sys.exit(1)
    t_one, t_per = [], []
    for _ in range(a.reps):
        t_one.append(timed(one_launch))
        t_per.append(timed(per_setting))
    print(json.dumps(dict(settings=S, frames=a.frames, proposals=int(sum(r["proposals"] for r in res["settings"])),
                          gt_boxes=int(gt_boxes.shape[0]), quality_ms=round(float(np.median(t_one)), 3),
                          quality_ms_min=round(min(t_one), 3), recall_precision_ms=round(float(np.median(t_per)), 3),
                          recall_precision_ms_min=round(min(t_per), 3),
                          ratio=round(float(np.median(t_per) / np.median(t_one)), 2), counters_equal=True,
                          gpu=torch.cuda.get_device_name(), power_limit_w=power_limit_w())), flush=True)


if __name__ == "__main__":
    main()
