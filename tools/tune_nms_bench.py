"""Cost of scoring tuning settings after load_pseudos' NMS: the NMS + counters step of evaluate_settings(nms_thresh=...)
-- one fnp_seg_nms_rotated_multi launch over every setting and threshold, then one fnp_quality_counters launch per
threshold -- against the straightforward one: S x n_thresh fnp_seg_nms_rotated calls, each keep mask turned into 0 / -1
flags, and the same quality launches.  Both are timed with CUDA events, alternately, in one process, on the
proposals one shared execution left on the device; their counters must be equal (exit status 1 otherwise).  Then the
whole evaluate_settings pass (stages 1-3, the counters, the one D2H) with and without the thresholds.

Inputs: the tools/tune_bench.py setup -- --frames distinct synthetic cfg2 frames (ten sweeps, 60 GLIP boxes, the
64 x 12 hypothesis grid) resident on the GPU, one batch, the 64 select-level settings of grid_a (one group) -- with the
thresholds {0.1} and {0.1, 0.3, 0.5}.  The NMS step reads each setting's boxes and flags (S x F x 32 bytes, printed as
nms_input_bytes), which stay in the 126 MB L2 between repetitions: the step is timed warm, as evaluate_settings runs
it right after stage 3 wrote those arrays.  Prints one JSON line per threshold set with the GPU's name and power limit.

    python tools/tune_nms_bench.py [--frames 256] [--reps 20]
"""
import argparse
import json
import os
import sys
import time

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
    from findnpropagate_b200.extract import THRESH
    from findnpropagate_b200.seeker import FrameInput, SeekerEngine
    if not torch.cuda.is_available():
        sys.exit("tune_nms_bench.py measures on a CUDA device; none is available")
    cfg = synth.CONFIGS["cfg2"]
    frames = []
    for i in range(a.frames):
        f = synth.make_frame(i, cfg, device="cuda:0")
        frames.append(FrameInput(points=f.points, lidar2image=f.lidar2image, camera2lidar=f.camera2lidar,
                                 camera_intrinsics=f.camera_intrinsics, det_boxes=f.det_boxes, det_labels=f.det_labels,
                                 det_scores=f.det_scores, det_cam_idx=f.det_cam_idx, gt_boxes=f.gt_boxes))
    points = torch.from_numpy(np.concatenate([f.points for f in frames])).cuda()
    (g,) = tune_params.group_settings(synth.seeker_params(cfg), grid_a())
    spec = quality.QualitySpec(synth.CLASS_NAMES)
    eng = SeekerEngine(g["params"], device="cuda:0")
    plan, gt = eng.plan(frames), eng.upload_gt(frames)
    F, B, S, L = plan["F"], plan["B"], len(g["settings"]), _lib.lib
    stream = _lib.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def events(fn, n=1):
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    for thresh in ((0.1,), (0.1, 0.3, 0.5)):
        NT = len(thresh)
        h = eng.execute(plan, points, gt=gt, recall_thresh=THRESH, settings=g["settings"], quality=spec,
                        settings_nms=thresh)
        eng.result(h)
        lay, out_dev, meta = h["layout"], h["out_dev"], h["meta"]
        ob = out_dev.data_ptr()
        new_counters = out_dev[lay.span("nms_quality")].view(torch.int64)

        def multi():
            eng._settings_nms(h, gt, spec, thresh, "", stream)

        keep = torch.empty((S, F), dtype=torch.uint8, device="cuda")
        valid = torch.empty((NT, S, F), dtype=torch.int32, device="cuda")
        old_counters = torch.zeros((NT, S, spec.n_counters), dtype=torch.int64, device="cuda")

        def single_calls():
            for t, th in enumerate(thresh):
                for s in range(S):
                    _lib.check(L.fnp_seg_nms_rotated(lay.ptr(ob, "sel_boxes", s), None, meta["nms_order"],
                                                     lay.ptr(ob, "sel_best", s), meta["frame_cand_start"], B,
                                                     max(plan["max_cands"], 1), th, keep[s].data_ptr(), stream),
                               "fnp_seg_nms_rotated")
                torch.sub(keep.to(torch.int32), 1, out=valid[t])
            old_counters.zero_()
            for t in range(NT):
                quality.launch(spec, lay.ptr(ob, "sel_boxes"), meta["cand_label"], meta["frame_cand_start"], gt[0],
                               gt[1], B, max(plan["max_cands"], 1), int(gt[2]), old_counters[t], n_settings=S,
                               pred_valid=valid[t], pred_stride=F, valid_stride=F, stream=stream)

        multi(); single_calls(); torch.cuda.synchronize()          # warm-up: every launch shape
        if not torch.equal(new_counters.view(NT, S, -1), old_counters):
            print(json.dumps(dict(thresh=thresh, error="counters differ")))
            sys.exit(1)
        t_new, t_old = [], []
        for _ in range(a.reps):
            t_new.append(events(multi))
            t_old.append(events(single_calls))
        if not torch.equal(new_counters.view(NT, S, -1), old_counters):
            print(json.dumps(dict(thresh=thresh, error="counters differ after the timed runs")))
            sys.exit(1)

        def whole(nms):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            eng.evaluate_settings(plan, points, gt, g["settings"], recall_thresh=THRESH, quality=spec, nms_thresh=nms)
            torch.cuda.synchronize()
            return (time.perf_counter() - t0) * 1e3

        whole(()); whole(thresh)
        w_plain, w_nms = [], []
        for _ in range(max(3, a.reps // 4)):
            w_plain.append(whole(()))
            w_nms.append(whole(thresh))
        print(json.dumps(dict(
            thresh=list(thresh), frames=a.frames, settings=S, candidates=F, nms_input_bytes=S * F * 32,
            nms_counters_ms=dict(multi=round(float(np.median(t_new)), 4), single_calls=round(float(np.median(t_old)), 4),
                                 speedup=round(float(np.median(t_old) / np.median(t_new)), 2)),
            evaluate_settings_ms=dict(without_nms=round(float(np.median(w_plain)), 3),
                                      with_nms=round(float(np.median(w_nms)), 3)),
            counters_equal=True, gpu=torch.cuda.get_device_name(), power_limit_w=power_limit_w())), flush=True)


if __name__ == "__main__":
    main()
