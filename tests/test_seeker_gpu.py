"""GPU parity tests of the fused seeker pipeline (through SeekerEngine -> C ABI) against the
CPU oracle stage by stage (bit-exact), against the golden vectors of the reference's own
get_proposals (1e-5 relative on boxes), and size-independent properties at full size."""
import glob
import json
import os

import numpy as np
import pytest
import torch

import oracle as O
import seeker_oracle as SO
from findnpropagate_b200 import synth
from findnpropagate_b200.seeker import FrameInput, SeekerEngine

pytestmark = pytest.mark.gpu
GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "seeker_*.npz")))


def _frame_from_golden(g):
    return FrameInput(points=g["points"], lidar2image=g["lidar2image"], camera2lidar=g["camera2lidar"],
                      camera_intrinsics=g["camera_intrinsics"], det_boxes=g["det_boxes"], det_labels=g["det_labels"],
                      det_scores=g["det_scores"], det_cam_idx=g["det_cam_idx"], gt_boxes=g["gt_boxes"])


def _frame_from_synth(f):
    return FrameInput(points=f.points, lidar2image=f.lidar2image, camera2lidar=f.camera2lidar,
                      camera_intrinsics=f.camera_intrinsics, det_boxes=f.det_boxes, det_labels=f.det_labels,
                      det_scores=f.det_scores, det_cam_idx=f.det_cam_idx, gt_boxes=f.gt_boxes)


def _oracle(fi, params, eng):
    return SO.seek_frame(fi.points, fi.lidar2image, fi.camera2lidar, fi.camera_intrinsics,
                         (fi.det_boxes, fi.det_labels, fi.det_scores, fi.det_cam_idx), params,
                         tables=(eng.base_boxes_host.numpy(), eng.base_corners_host.numpy()), keep_intermediates=True,
                         box_format=eng.box_format)


def _bits(a):
    """Bit patterns with every NaN mapped to one value: a degenerate frustum (clamped to a point, so that
    search_depth divides 0 by 0) is NaN in the reference, the oracle and the kernels alike, but the
    default NaN of x86 (0xffc00000) and of the GPU (0x7fffffff) differ in their payload."""
    a = np.ascontiguousarray(a, np.float32)
    return np.where(np.isnan(a), np.uint32(0x7fc00000), a.view(np.uint32))


def _check_against_oracle(eng, frames, params):
    plan = eng.plan(frames)
    pts = eng.upload_points(frames)
    h = eng.execute(plan, pts)
    res = eng.finish(h)
    dbg = eng.debug_views(h)
    fcs = plan["frame_cand_start"]
    n_checked = 0
    for b, fi in enumerate(frames):
        ora = _oracle(fi, params, eng)
        cands = ora["frustums"]
        assert len(cands) == fcs[b + 1] - fcs[b]
        for j, rec in enumerate(cands):
            f = fcs[b] + j
            assert rec["cam"] == plan["cand_cam"][f] and rec["label"] == plan["cand_label"][f]
            assert np.array_equal(rec["box2d"], plan["cand_box2d"][f])
            # --- stage 1: frustum membership (bit-exact, ordered) and unprojected points
            p0, p1 = dbg["pt_start"][f], dbg["pt_start"][f + 1]
            assert res["cand_npts"][f] == rec["n_points"] == p1 - p0
            if rec["n_points"] == 0:
                assert not res["cand_valid"][f]
                continue
            assert np.array_equal(dbg["frustum_idx"][p0:p1], rec["idx"])
            assert np.array_equal(dbg["frustum_pts"][p0:p1, :3].view(np.uint32), rec["xyz"].view(np.uint32))
            assert np.array_equal(dbg["frustum_pts"][p0:p1, 3].view(np.uint32), rec["uvd"][:, 2].view(np.uint32))
            # --- stage 1b: depth quantiles, corners, centre line
            st = dbg["stats"][f]
            assert st[0].tobytes() == np.float32(rec["dmin"]).tobytes()
            assert st[1].tobytes() == np.float32(rec["dmax"]).tobytes()
            assert np.array_equal(st[16:40].reshape(8, 3).view(np.uint32), rec["corners"].view(np.uint32))
            assert np.array_equal(_bits(dbg["centres"][f]), _bits(rec["centres"]))
            # --- stage 2a: hypotheses
            assert np.array_equal(dbg["hyp_valid"][f], rec["valid"])
            assert np.array_equal(_bits(dbg["hyp_boxes"][f]), _bits(rec["hyp_boxes"]))
            assert np.array_equal(_bits(dbg["hyp_iou"][f]), _bits(rec["iou"]))
            nv = int(rec["valid"].sum())
            assert res["cand_nvalid"][f] == nv
            assert np.array_equal(dbg["hyp_index"][f, :nv], np.flatnonzero(rec["valid"]))
            # --- stage 2b: per-hypothesis counts (bit-exact)
            assert np.array_equal(dbg["counts"][f, :nv], rec["counts"][rec["valid"]])
            # --- optional terms (row f3): distance to the weighted centre, occlusion n_far
            if eng.use_dist:
                assert np.array_equal(st[10:13].view(np.uint32), rec["wc"].view(np.uint32))
                assert np.array_equal(dbg["hyp_dist"][f, :nv].view(np.uint32), rec["dist"][rec["valid"]].view(np.uint32))
                if rec["near"].any():
                    assert st[13] == rec["dist"][rec["near"]].min() and st[14] == rec["dist"][rec["near"]].max()
            if eng.use_occl:
                assert np.array_equal(dbg["hyp_nfar"][f, :nv], rec["nfar"][rec["valid"]])
            # --- stage 3: greedy argmax
            if rec["best"] < 0:
                assert not res["cand_valid"][f]
            else:
                assert dbg["hyp_index"][f, res["cand_best"][f]] == rec["best"]
                assert res["cand_score2"][f].tobytes() == np.float32(rec["best_score"]).tobytes()
                assert np.array_equal(res["cand_boxes"][f].view(np.uint32), rec["hyp_boxes"][rec["best"]].view(np.uint32))
                if eng.T > 1:    # topk > 1: the first T survivors of the per-frustum nms_normal, in order
                    tk, want = res["cand_topk"]["best"][f], rec["topk"]
                    assert np.array_equal(dbg["hyp_index"][f, tk[:len(want)]], want) and (tk[len(want):] == -1).all()
                    assert np.array_equal(res["cand_topk"]["boxes"][f, :len(want)].view(np.uint32),
                                          rec["hyp_boxes"][want].view(np.uint32))
                    assert np.array_equal(res["cand_topk"]["score2"][f, :len(want)].view(np.uint32),
                                          rec["scores"][want].view(np.uint32))
            n_checked += 1
        out = res["frames"][b]
        assert np.array_equal(out["pred_boxes"].view(np.uint32), ora["pred_boxes"].view(np.uint32))
        assert np.array_equal(out["pred_labels"], ora["pred_labels"])
        assert np.array_equal(out["pred_scores"], ora["pred_scores"])
    return res, n_checked


@pytest.mark.parametrize("path", GOLDEN)
def test_pipeline_vs_oracle_and_reference_golden(path):
    g = np.load(path)
    params = synth.seeker_params(synth.CONFIGS[str(g["cfg"])])
    opts = json.loads(str(g["opts"])) if "opts" in g else {}      # row f3 option sets (tools/gen_golden.py)
    params.update(opts)
    tol = 1e-5 if not opts else 3e-5
    eng = SeekerEngine(params, device="cuda:0", debug=True,
                       box_format=str(g["box_format"]) if "box_format" in g else "xyxy")     # one fixture is x, y, w, h
    fi = _frame_from_golden(g)
    res, n = _check_against_oracle(eng, [fi], params)
    assert n > 0
    out = res["frames"][0]
    # versus the reference's own get_proposals (golden): same K / labels / scores, boxes 1e-5
    assert out["pred_boxes"].shape == g["ref_boxes"].shape
    assert out["pred_boxes"].dtype == np.float32 and out["pred_labels"].dtype == np.int32
    assert np.array_equal(out["pred_labels"], g["ref_labels"])
    assert np.array_equal(out["pred_scores"], g["ref_scores"])
    rel = np.abs(out["pred_boxes"] - g["ref_boxes"]) / np.maximum(np.abs(g["ref_boxes"]), 1e-3)
    for k in range(rel.shape[0]):
        if rel[k].max() > tol:   # yaw 0 / pi twin (documented tie, SURVEY 7.5)
            assert rel[k, :6].max() <= tol
            assert abs(abs(out["pred_boxes"][k, 6] - g["ref_boxes"][k, 6]) - np.pi) < 1e-5


def test_batch_of_frames_equals_frame_by_frame_and_splits_are_invariant():
    cfg = synth.CONFIGS["cfg1"]
    params = synth.seeker_params(cfg)
    frames = [_frame_from_synth(synth.make_frame(i, cfg)) for i in range(3)]
    empty = _frame_from_synth(synth.make_frame(7, synth.CONFIGS["tiny"]))
    empty.det_boxes = np.zeros((0, 4), np.float32)
    empty.det_labels = np.zeros(0, np.int64)
    empty.det_scores = np.zeros(0, np.float32)
    empty.det_cam_idx = np.zeros(0, np.int64)
    frames.insert(1, empty)                                     # a frame without detections
    eng = SeekerEngine(params, device="cuda:0", debug=True)
    res, n = _check_against_oracle(eng, frames, params)
    assert res["frames"][1]["pred_boxes"].shape == (0, 7)
    for sp in (1 << 20, 333, 64):
        e2 = SeekerEngine(params, device="cuda:0", split_points=sp)
        r2 = e2.run(frames)
        v = res["cand_valid"]
        assert np.array_equal(r2["cand_count"][v], res["cand_count"][v])
        assert np.array_equal(r2["cand_best"], res["cand_best"])
        for a, b in zip(r2["frames"], res["frames"]):
            assert np.array_equal(a["pred_boxes"], b["pred_boxes"])
    # no frames at all / no candidates at all
    r0 = eng.run([empty])
    assert r0["frames"][0]["pred_boxes"].shape == (0, 7)


@pytest.mark.parametrize("n_boxes", [40, 100, 150])
def test_many_candidates_per_frame_mask_words(n_boxes):
    """Frames with more than 32 / 64 / 128 candidate frustums: the per-point membership mask
    of stage 1 takes 2 / 4 / 8 words; results stay bit-exact against the oracle."""
    cfg = synth.SynthConfig("many%d" % n_boxes, 16, 720, 1, n_boxes, 4, 6, 1)
    params = synth.seeker_params(cfg)
    frames = [_frame_from_synth(synth.make_frame(i, cfg)) for i in range(2)]
    eng = SeekerEngine(params, device="cuda:0", debug=True)
    plan = eng.plan(frames)
    assert plan["max_cands"] > (32 if n_boxes == 40 else 64 if n_boxes == 100 else 128)
    res, n = _check_against_oracle(eng, frames, params)
    assert n > n_boxes // 2


def test_dense_overlapping_boxes_take_the_direct_pass_of_stage_one():
    """Nested 2D boxes in every label: a point is a member of dozens of candidates, so the members of a
    1024-point tile exceed the shared-memory member list of stage 1 and the tile repeats its membership pass
    with direct writes.  Bit-exact against the oracle like any other frame."""
    cfg = synth.SynthConfig("nested", 16, 720, 1, 8, 4, 6, 1)
    params = synth.seeker_params(cfg)
    frames = []
    for i in range(2):
        f = _frame_from_synth(synth.make_frame(i, cfg))
        boxes, labels, scores, cams = [], [], [], []
        for cam in range(6):
            for lab in range(1, 11):
                for k, w in enumerate((35.0, 90.0, 240.0, 620.0, 1600.0)):  # mutual IoU < 0.4: all survive the 2D NMS
                    boxes.append([0.0, 0.0, w, 900.0 - 3.0 * lab])
                    labels.append(lab); scores.append(0.5 + 0.01 * k + 0.001 * lab); cams.append(cam)
        f.det_boxes, f.det_labels = np.asarray(boxes, np.float32), np.asarray(labels, np.int64)
        f.det_scores, f.det_cam_idx = np.asarray(scores, np.float32), np.asarray(cams, np.int64)
        frames.append(f)
    eng = SeekerEngine(params, device="cuda:0", debug=True)
    eng.pts_factor = 64.0                       # a point is a member of up to 40 frustums here
    plan = eng.plan(frames)
    assert plan["max_cands"] == 300             # more than 256 candidates in a frame: 16 mask words per image cell
    res, n = _check_against_oracle(eng, frames, params)
    assert n > 250
    per_tile = res["cand_npts"].sum() / plan["n_tiles"]
    assert per_tile > 1280, per_tile           # more members per tile than the list holds (csrc: kCullList)


def test_sector_table_only_skips_cameras_that_cannot_see_the_point():
    """Stage 1 projects a point only into the cameras its azimuth sector lists (csrc: sector_sees).  The table
    must be a superset of the truth: with the table switched off (every camera for every point) stage 1 must
    give the same members, and both must equal the oracle -- on a frame salted with the points the table could
    get wrong: behind a camera on the thin tube that still lands on the image through the depth clamp, closer to
    the sensor than the table's minimum radius, far above / below it, exactly on sector borders."""
    from findnpropagate_b200 import _lib
    cfg = synth.SynthConfig("sect", 16, 720, 1, 8, 4, 6, 1)
    params = synth.seeker_params(cfg)
    sf = synth.make_frame(3, cfg)
    extra = []
    for c in range(6):
        L = sf.lidar2image[c][:3].astype(np.float64)
        for t in np.linspace(0.3, 70.0, 160):           # wz = -t: behind camera c, wx and wy inside [0, 1600e-5) x [0, 900e-5)
            for a, b in ((0.005, 0.004), (0.0, 0.0), (0.0155, 0.0085), (0.012, 0.001)):
                extra.append(np.linalg.solve(L[:, :3], np.array([a, b, -t]) - L[:, 3]))
    rng = np.random.default_rng(11)
    near = rng.uniform(-3.5, 3.5, (600, 3)); near[:, 2] = rng.uniform(-2, 2, 600)            # inside the minimum radius
    tall = rng.uniform(-40, 40, (600, 3)); tall[:, 2] = rng.choice([-30.0, 17.0, 16.0, -16.0, 60.0], 600)
    r = rng.uniform(3.0, 60.0, 400)
    ang = rng.choice(np.arctan2(np.arange(17) / 16.0, 1 - np.arange(17) / 16.0), 400) * rng.choice([1, -1], 400) \
        + rng.choice([0, np.pi], 400)                                                         # exactly on sector borders
    border = np.stack([r * np.cos(ang), r * np.sin(ang), rng.uniform(-2, 1, 400)], 1)
    axes = np.array([[5, 0, 0], [-5, 0, 0], [0, 5, 0], [0, -5, 0], [-0.0, 7, 0], [7, -0.0, 0], [3, 0, 0], [0, 3, 0]], float)
    add = np.concatenate([np.asarray(extra), near, tall, border, axes]).astype(np.float32)
    pts = np.concatenate([sf.points, np.concatenate([add, np.zeros((add.shape[0], 2), np.float32)], 1)]).astype(np.float32)
    fi = _frame_from_synth(sf)
    fi.points = pts
    boxes, labels, scores, cams = [fi.det_boxes], [fi.det_labels], [fi.det_scores], [fi.det_cam_idx]
    for c in range(6):      # one box over the whole image of every camera: every on-image point is a member
        boxes.append(np.array([[0, 0, 1600, 900]], np.float32)); labels.append(np.array([1 + c])); scores.append(np.array([0.9], np.float32))
        cams.append(np.array([c]))
    fi.det_boxes, fi.det_labels = np.concatenate(boxes).astype(np.float32), np.concatenate(labels).astype(np.int64)
    fi.det_scores, fi.det_cam_idx = np.concatenate(scores).astype(np.float32), np.concatenate(cams).astype(np.int64)
    out = {}
    try:
        for mode in (1, 0):
            assert _lib.lib.fnp_set_option(b"cull_sectors", mode) == 0
            eng = SeekerEngine(params, device="cuda:0", debug=True)
            eng.pts_factor = 8.0
            if mode == 1:
                res, n = _check_against_oracle(eng, [fi], params)
                assert n >= 6
            plan = eng.plan([fi])
            h = eng.execute(plan, eng.upload_points([fi]))
            r_ = eng.finish(h)
            d_ = eng.debug_views(h)
            v_ = r_["cand_valid"]
            out[mode] = (r_["cand_npts"].copy(), d_["frustum_idx"].copy(), d_["frustum_pts"].copy(), d_["counts"].copy(),
                         v_.copy(), r_["cand_boxes"][v_].copy(), r_["cand_count"][v_].copy())
    finally:
        _lib.lib.fnp_set_option(b"cull_sectors", 1)
    for a, b in zip(out[1], out[0]):
        assert np.array_equal(a.view(np.uint32) if a.dtype == np.float32 else a, b.view(np.uint32) if b.dtype == np.float32 else b)
    # the salted points did reach frustums (among them points BEHIND their camera)
    n_base = sf.points.shape[0]
    assert (out[1][1] >= n_base).sum() > 300
    assert _lib.lib.fnp_set_option(b"no_such_option", 1) != 0


def test_full_size_properties_cfg2():
    """cfg2 (300k points, 60 boxes, H = 768): properties that do not need the slow oracle on
    every hypothesis -- run twice = identical; membership ordered/unique; counts equal the
    op-level count kernel and a sample of them equals the oracle; capacity overflow path."""
    import ctypes as C
    from findnpropagate_b200 import _lib
    cfg = synth.CONFIGS["cfg2"]
    params = synth.seeker_params(cfg)
    frames = [_frame_from_synth(synth.make_frame(i, cfg, device="cuda:0")) for i in range(2)]
    eng = SeekerEngine(params, device="cuda:0", debug=True)
    plan = eng.plan(frames)
    pts = eng.upload_points(frames)
    h = eng.execute(plan, pts, nms_thresh=0.1, gt=eng.upload_gt(frames))
    res = eng.finish(h)
    dbg = eng.debug_views(h)
    F, H = plan["F"], eng.H
    assert H == 768 and F > 60
    # membership: strictly increasing source rows per frustum, inside the frame
    for f in range(F):
        idx = dbg["frustum_idx"][dbg["pt_start"][f]:dbg["pt_start"][f + 1]]
        assert np.all(np.diff(idx) > 0)
    # counts of every valid hypothesis through the independent op-level kernel
    nv = res["cand_nvalid"]
    hb = np.concatenate([dbg["hyp_boxes"][f][dbg["hyp_index"][f, :nv[f]]] for f in range(F)])
    bstart = np.concatenate([[0], np.cumsum(nv)]).astype(np.int32)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0")
    tb, tbs, tps = d(hb), d(bstart), d(dbg["pt_start"])
    tp = d(dbg["frustum_pts"])
    cnt = torch.zeros(hb.shape[0], dtype=torch.int32, device="cuda:0")
    rc = _lib.lib.fnp_count_in_boxes(tp.data_ptr(), tps.data_ptr(), tb.data_ptr(), tbs.data_ptr(), F, cnt.data_ptr(),
                                     _lib.current_stream())
    assert rc == 0
    cnt = cnt.cpu().numpy()
    for f in range(F):
        assert np.array_equal(cnt[bstart[f]:bstart[f + 1]], dbg["counts"][f, :nv[f]])
    # oracle on a sample of frustums (all hypotheses of each)
    for f in list(range(0, F, 9))[:8]:
        p = dbg["frustum_pts"][dbg["pt_start"][f]:dbg["pt_start"][f + 1], :3]
        if nv[f] and p.shape[0]:
            assert np.array_equal(O.count_in_boxes(p, hb[bstart[f]:bstart[f + 1]]), dbg["counts"][f, :nv[f]])
    # whole-frame oracle for frame 0 (bit-exact boxes)
    ora = _oracle(frames[0], params, eng)
    assert np.array_equal(res["frames"][0]["pred_boxes"].view(np.uint32), ora["pred_boxes"].view(np.uint32))
    # recall counters and stage-4 NMS vs oracle
    exp = None
    for b, fi in enumerate(frames):
        rd = SO.recall_record(res["frames"][b]["pred_boxes"], fi.gt_boxes)
        exp = rd if exp is None else {k: exp[k] + rd[k] for k in rd}
        fr = res["frames"][b]
        kept = O.nms_rotated(fr["pred_boxes"], fr["pred_scores"], 0.1)
        m = np.zeros(fr["pred_boxes"].shape[0], bool)
        m[kept] = True
        assert np.array_equal(fr["nms_keep"], m)
    assert res["recall"] == exp
    # idempotence
    res2 = eng.finish(eng.execute(plan, pts))
    v = res["cand_valid"]
    assert np.array_equal(res2["cand_valid"], v) and np.array_equal(res2["cand_count"][v], res["cand_count"][v])
    assert np.array_equal(res2["cand_boxes"][v], res["cand_boxes"][v])
    # frustum-point buffer overflow is detected and recovered from
    e3 = SeekerEngine(params, device="cuda:0")
    e3.pts_factor = 0.05
    r3 = e3.run(frames)
    assert e3.pts_factor > 0.05
    assert np.array_equal(r3["cand_count"][v], res["cand_count"][v])


def test_stress_cfg5_whole_frame_vs_oracle(monkeypatch):
    """BASELINE.json configs[4]: 1M-point frame, 200 2D boxes, 128 x 24 = 3072 hypotheses per
    frustum.  The whole-frame oracle runs on it stage by stage; to keep it to seconds, oracle
    count calls above 2e7 point-box tests are answered by the op-level count kernel
    (fnp_count_in_boxes, itself pinned bit-exact against the oracle and the reference kernel in
    test_ops_gpu.py), smaller ones by the C oracle.  Also checks stage-4 NMS and recall."""
    from findnpropagate_b200 import _lib
    cfg = synth.CONFIGS["cfg5"]
    params = synth.seeker_params(cfg)
    frames = [_frame_from_synth(synth.make_frame(0, cfg, device="cuda:0"))]
    assert frames[0].points.shape[0] > 900_000
    eng = SeekerEngine(params, device="cuda:0", debug=True)
    assert eng.H == 3072
    c_oracle = O.count_in_boxes
    calls = {"oracle": 0, "gpu": 0}

    def count(points, boxes):
        if points.shape[0] * boxes.shape[0] <= 2e7:
            calls["oracle"] += 1
            return c_oracle(points, boxes)
        calls["gpu"] += 1
        p4 = np.zeros((points.shape[0], 4), np.float32)
        p4[:, :3] = points[:, :3]
        d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0")
        tp, tb = d(p4), d(np.ascontiguousarray(boxes, np.float32))
        ps, bs = d(np.array([0, points.shape[0]], np.int32)), d(np.array([0, boxes.shape[0]], np.int32))
        cnt = torch.zeros(boxes.shape[0], dtype=torch.int32, device="cuda:0")
        assert _lib.lib.fnp_count_in_boxes(tp.data_ptr(), ps.data_ptr(), tb.data_ptr(), bs.data_ptr(), 1, cnt.data_ptr(),
                                           _lib.current_stream()) == 0
        return cnt.cpu().numpy()

    monkeypatch.setattr(O, "count_in_boxes", count)
    res, n = _check_against_oracle(eng, frames, params)
    assert n > 100 and calls["oracle"] > 0 and calls["gpu"] > 0
    r2 = eng.run(frames, nms_thresh=0.1, with_recall=True)
    fr = r2["frames"][0]
    kept = O.nms_rotated(fr["pred_boxes"], fr["pred_scores"], 0.1)
    m = np.zeros(fr["pred_boxes"].shape[0], bool)
    m[kept] = True
    assert np.array_equal(fr["nms_keep"], m)
    assert r2["recall"] == SO.recall_record(fr["pred_boxes"], frames[0].gt_boxes)


def test_reference_compatible_head_and_extraction(tmp_path):
    """FrustumProposerOG drop-in: same call contract / return types as the reference head
    (frustum_proposals_v1.py:1055-1067,1554-1573) and the extraction output format."""
    from findnpropagate_b200 import extract, proposer
    cfg = synth.CONFIGS["cfg1"]
    params = synth.seeker_params(cfg)
    sf = [synth.make_frame(i, cfg) for i in range(3)]
    feeder = proposer.SyntheticGLIP(sf)
    head = proposer.FrustumProposerOG(model_cfg=dict(PARAMS=params, PREDS_PATH="PreprocessedGLIP", BOX_FORMAT="xyxy"),
                                      class_names=synth.CLASS_NAMES, image_detector=feeder).eval()
    bd = synth.collate(sf)
    for k, v in list(bd.items()):
        if isinstance(v, np.ndarray) and v.dtype.kind == "f":
            bd[k] = torch.from_numpy(v).cuda()              # load_data_to_gpu (models/__init__.py:23-36)
    boxes, labels, scores, bidx = head.get_proposals(bd)
    assert boxes.is_cuda and boxes.dtype == torch.float32 and boxes.shape[1] == 7
    assert labels.dtype == torch.int64 and not labels.is_cuda and scores.dtype == torch.float32
    assert bidx.dtype == torch.int64 and boxes.shape[0] == labels.shape[0] == scores.shape[0] == bidx.shape[0]
    out = head(bd)["final_box_dicts"]
    assert len(out) == 3 and out[0]["pred_labels"].dtype == torch.int32
    # a page pool too small for the batch: the head grows it, runs the batch again and gives the same proposals
    starved = proposer.FrustumProposerOG(model_cfg=dict(PARAMS=params, PREDS_PATH="PreprocessedGLIP", BOX_FORMAT="xyxy"),
                                         class_names=synth.CLASS_NAMES, image_detector=feeder).eval()
    starved.engine.pts_factor = 0.05
    got = starved.get_proposals(bd)
    assert starved.engine.pts_factor > 0.05
    assert all(torch.equal(g, w) for g, w in zip(got, (boxes, labels, scores, bidx)))
    eng = SeekerEngine(params, device="cuda:0")
    for b, f in enumerate(sf):
        ora = _oracle(_frame_from_synth(f), params, eng)
        assert np.array_equal(out[b]["pred_boxes"].cpu().numpy().view(np.uint32), ora["pred_boxes"].view(np.uint32))
        assert np.array_equal(out[b]["pred_labels"].numpy(), ora["pred_labels"])
    # numpy batch_dict works too, and options outside the shipped config fail loudly
    boxes2, _, _, _ = head.get_proposals(synth.collate(sf))
    assert torch.equal(boxes2, boxes)
    with pytest.raises(NotImplementedError):
        proposer.FrustumProposerOG(model_cfg=dict(PARAMS=dict(params, aln_w=0.2)), image_detector=feeder)
    with pytest.raises(NotImplementedError):
        proposer.FrustumProposerOG(model_cfg=dict(PARAMS=dict(params), SAVE_BLEND=True), image_detector=feeder)
    # the optional settings of the head (row f3) reach the engine: PARAMS keys and model_cfg switches
    p3 = dict(params, topk=3, nms_normal=0.5, dst_w=0.2)
    head3 = proposer.FrustumProposerOG(model_cfg=dict(PARAMS=p3, MULTICAM_IOU=True), image_detector=feeder)
    out3 = head3.get_bboxes(bd)
    p3["MULTICAM_IOU"] = True
    for b, f in enumerate(sf):
        ora = _oracle(_frame_from_synth(f), p3, eng)
        assert np.array_equal(out3[b]["pred_boxes"].cpu().numpy().view(np.uint32), ora["pred_boxes"].view(np.uint32))
        assert np.array_equal(out3[b]["pred_labels"].numpy(), ora["pred_labels"])
    assert sum(o["pred_boxes"].shape[0] for o in out3) > sum(o["pred_boxes"].shape[0] for o in out)
    # the head's other feeder: one COCO result file per camera view (PREDS_PATHS, x, y, w, h boxes ->
    # BOX_FORMAT), preprocessed_detector.py:111-290
    import json
    names = ['car', 'truck', 'construction_vehicle', 'bus', 'trailer', 'barrier', 'motorcycle', 'bicycle',
             'pedestrian', 'traffic_cone']
    files = []
    for c in range(6):
        images, anns = [], []
        for b, f in enumerate(sf):
            images.append({"id": b, "file_name": f.image_paths[c]})
            for k in np.flatnonzero(f.det_cam_idx == c):
                x1, y1, x2, y2 = (float(v) for v in f.det_boxes[k])
                anns.append({"id": len(anns), "image_id": b, "category_id": int(f.det_labels[k]) - 1,
                             "bbox": [x1, y1, x2 - x1, y2 - y1], "score": float(f.det_scores[k])})
        files.append(str(tmp_path / ("OWL_%d.json" % c)))
        json.dump({"images": images, "annotations": anns,
                   "categories": [{"id": i, "name": n} for i, n in enumerate(names)]}, open(files[-1], "w"))
    head4 = proposer.FrustumProposerOG(model_cfg=dict(PARAMS=params, PREDS_PATH=str(tmp_path / "OWL_"), PREDS_PATHS=files,
                                                      BOX_FORMAT='xywh'), class_names=names)
    assert isinstance(head4.image_detector, proposer.PreprocessedDetector)
    out4 = head4.get_bboxes(bd)
    db, dl, ds, di, dc = head4.image_detector(bd)
    e4 = SeekerEngine(params, device="cuda:0", box_format="xywh")
    for b, f in enumerate(sf):
        m = (di == b).numpy()
        ora = SO.seek_frame(f.points, f.lidar2image, f.camera2lidar, f.camera_intrinsics,
                            (db.numpy()[m], dl.numpy()[m], ds.numpy()[m], dc.numpy()[m]), params,
                            tables=(e4.base_boxes_host.numpy(), e4.base_corners_host.numpy()), box_format="xywh")
        assert ora["pred_boxes"].shape[0] > 0
        assert np.array_equal(out4[b]["pred_boxes"].cpu().numpy().view(np.uint32), ora["pred_boxes"].view(np.uint32))
        assert np.array_equal(out4[b]["pred_labels"].numpy(), ora["pred_labels"])
    # extraction driver: one .pth per frame, reference format, recall counters
    frames = [_frame_from_synth(f) for f in sf]
    merged, total, ar = extract.extract(frames, lambda fs: eng.run(fs, with_recall=True), folder=str(tmp_path),
                                        batch_frames=2, frame_ids=[f.frame_id for f in sf])
    exp = None
    for b, f in enumerate(sf):
        rd = SO.recall_record(merged[b]["pred_boxes"], f.gt_boxes)
        exp = rd if exp is None else {k: exp[k] + rd[k] for k in rd}
        saved = torch.load(str(tmp_path / (f.frame_id.replace(".", "_") + ".pth")), map_location="cpu")
        assert np.array_equal(saved[0]["pred_boxes"].numpy(), merged[b]["pred_boxes"])
    assert {k: total[k] for k in exp} == exp and 0.0 <= ar["rcnn_0.3"] <= 1.0


@pytest.mark.parametrize("cfg_name,override,n_frames,split", [
    ("tiny", None, 3, None), ("cfg1", None, 3, 64), ("cfg1", dict(num_mags=40, num_sizes=2), 2, 333),
    ("cfg2", None, 2, None), ("cfg2", dict(num_mags=17, num_rotations=5), 1, 2048),
])
def test_sweep_and_direct_scoring_give_identical_counts(cfg_name, override, n_frames, split):
    """Stage 2b has two kernels (include/fnp.h FNP_SCORE_*): DIRECT tests every (point, valid
    hypothesis) pair, SWEEP solves one depth range per (point, yaw-size column) and takes the
    exact predicate only next to the range ends.  Their (F, H) count tables must be the same
    integers, for every hypothesis, whatever the point split, and match the oracle."""
    cfg = synth.CONFIGS[cfg_name]
    params = synth.seeker_params(cfg)
    if override:
        params.update(override)
    frames = [_frame_from_synth(synth.make_frame(i, cfg, device="cuda:0" if cfg_name == "cfg2" else "cpu"))
              for i in range(n_frames)]
    out = {}
    for mode in ("direct", "sweep"):
        eng = SeekerEngine(params, device="cuda:0", debug=True, score_mode=mode, split_points=split)
        plan = eng.plan(frames)
        h = eng.execute(plan, eng.upload_points(frames))
        res = eng.finish(h)
        assert eng.last_score_mode == mode
        dbg = eng.debug_views(h)
        nv = res["cand_nvalid"]
        out[mode] = (res, [dbg["counts"][f, :nv[f]].copy() for f in range(plan["F"])], dbg)
    (rd, cd, dbg), (rs, cs, _) = out["direct"], out["sweep"]
    assert sum(int(c.sum()) for c in cd) > 0
    for f, (a, b) in enumerate(zip(cd, cs)):
        assert np.array_equal(a, b), "frustum %d: sweep counts differ from direct counts" % f
    assert np.array_equal(rd["cand_best"], rs["cand_best"])
    v = rd["cand_valid"]
    assert np.array_equal(rd["cand_boxes"][v].view(np.uint32), rs["cand_boxes"][v].view(np.uint32))
    # and the oracle on a few frustums (all valid hypotheses of each)
    nv = rd["cand_nvalid"]
    checked = 0
    for f in range(0, len(cd), max(1, len(cd) // 6)):
        p = dbg["frustum_pts"][dbg["pt_start"][f]:dbg["pt_start"][f + 1], :3]
        if nv[f] and p.shape[0] and p.shape[0] * nv[f] < 3e7:
            hb = dbg["hyp_boxes"][f][dbg["hyp_index"][f, :nv[f]]]
            assert np.array_equal(O.count_in_boxes(p, hb), cs[f])
            checked += 1
    assert checked > 0


@pytest.mark.parametrize("opts,override,mode", [
    (dict(dst_w=0.226, iou_w=0.95, dns_w=0.05, ego_w=0.1), None, "direct"),
    (dict(occl_w=0.4, MULTICAM_IOU=True, search_depth=5.0), None, "direct"),
    (dict(MULT=True, dst_w=0.6, OCCL_MULT=True), None, "direct"),
    (dict(dst_w=0.3, ego_w=0.2, occl_w=0.5, MULTICAM_IOU=True), dict(num_mags=24, num_sizes=2), "sweep"),
    (dict(MULT=True, dst_w=0.8, search_depth=7.5), dict(num_mags=17), "sweep"),
    (dict(topk=3, nms_normal=0.5), None, "direct"),
    (dict(topk=4, nms_normal=0.3, occl_w=0.2, dst_w=0.1), dict(num_mags=20), "sweep"),
])
def test_optional_score_terms_vs_oracle(opts, override, mode):
    """SURVEY.md 8 row f3: dst_w / ego_w / occl_w / search_depth and MULT / OCCL_MULT / MULTICAM_IOU
    (frustum_proposals_v1.py:408-477,619-623,841-842,889-893,994-1026,1413-1429) through the fused
    pipeline, bit-exact against the oracle on a batch of frames: weighted centre, distances, n_far,
    multi-view IoUs, second-stage scores and the selected boxes."""
    cfg = synth.CONFIGS["cfg1"]
    params = synth.seeker_params(cfg)
    params.update(opts)
    if override:
        params.update(override)
    frames = [_frame_from_synth(synth.make_frame(i, cfg)) for i in range(3)]
    eng = SeekerEngine(params, device="cuda:0", debug=True, score_mode=mode)
    res, n = _check_against_oracle(eng, frames, params)
    assert eng.last_score_mode == mode and n > 10
    # the terms change the outcome: at least one frustum selects another box than the shipped scoring
    p0 = synth.seeker_params(cfg)
    if override:
        p0.update(override)
    r0 = SeekerEngine(p0, device="cuda:0").run(frames)
    if "search_depth" not in opts and "MULTICAM_IOU" not in opts:
        assert np.array_equal(r0["cand_nvalid"], res["cand_nvalid"])
        if set(opts) & {"dst_w", "ego_w", "occl_w", "MULT", "OCCL_MULT"}:
            assert not np.array_equal(r0["cand_best"], res["cand_best"])
        else:
            assert np.array_equal(r0["cand_best"], res["cand_best"])
    if eng.T > 1:
        # more than one proposal per frustum comes out, and stage-4 NMS / recall run over all of them
        assert sum(f["pred_boxes"].shape[0] for f in res["frames"]) > sum(f["pred_boxes"].shape[0] for f in r0["frames"])
        r2 = eng.run(frames, nms_thresh=0.1, with_recall=True)
        exp = None
        for b, fr in enumerate(r2["frames"]):
            assert np.array_equal(fr["pred_boxes"], res["frames"][b]["pred_boxes"])
            kept = O.nms_rotated(fr["pred_boxes"], fr["pred_scores"], 0.1)
            m = np.zeros(fr["pred_boxes"].shape[0], bool)
            m[kept] = True
            assert np.array_equal(fr["nms_keep"], m)
            rd = SO.recall_record(fr["pred_boxes"], frames[b].gt_boxes)
            exp = rd if exp is None else {k: exp[k] + rd[k] for k in rd}
        assert r2["recall"] == exp


@pytest.mark.parametrize("cfg_name,quant,n_frames", [
    ("cfg1", dict(lq=0.336, uq=0.356, cq=0.46, dst_w=0.226), 3),      # the KITTI head's defaults (frustum_proposals_v1_kitti.py:41)
    ("cfg1", dict(lq=0.1, uq=0.9, cq=0.5), 3),                          # far apart: two bins, two lists
    ("cfg1", dict(lq=0.5, uq=0.5, cq=0.0, dst_w=0.1), 2),               # the same rank twice
    ("cfg1", dict(lq=0.0, uq=1.0, cq=1.0), 2),                          # both ends trivial
    ("cfg2", dict(lq=0.05, uq=0.3, cq=0.7, dst_w=0.2), 1),              # frustums of > 4096 points stream their depth planes
])
def test_interior_depth_quantiles_vs_oracle(cfg_name, quant, n_frames):
    """torch.quantile at interior positions (frustum_proposals_v1.py:616-648): the near and the far quantile come from
    ONE histogram pass and ONE collect pass of the radix select (select_two), the centre quantile -- selected only
    when the distance term reads it -- from the single-rank select; dmin / dmax / weighted centre and everything
    downstream bit-exact against the oracle.  The shipped YAML (lq 0, uq 0.25, cq 1) needs one interior rank only."""
    cfg = synth.CONFIGS[cfg_name]
    params = synth.seeker_params(cfg)
    params.update(quant)
    frames = [_frame_from_synth(synth.make_frame(10 + i, cfg)) for i in range(n_frames)]
    eng = SeekerEngine(params, device="cuda:0", debug=True)
    res, n = _check_against_oracle(eng, frames, params)
    assert n > 10


def test_optional_score_terms_full_size_frame():
    """The same on a cfg2 frame (BASELINE.json configs[1]: ~322k points, 58 frustums of up to 1e4 points,
    768 hypotheses each): occl_kernel runs several point tiles and hypothesis blocks per frustum, the
    per-frustum NMS works on hundreds of valid hypotheses."""
    cfg = synth.CONFIGS["cfg2"]
    params = synth.seeker_params(cfg)
    params.update(occl_w=0.3, dst_w=0.2, ego_w=0.1, topk=3, nms_normal=0.6, MULTICAM_IOU=True)
    frames = [_frame_from_synth(synth.make_frame(1, cfg, device="cuda:0"))]
    eng = SeekerEngine(params, device="cuda:0", debug=True)
    res, n = _check_against_oracle(eng, frames, params)
    assert eng.last_score_mode == "sweep" and n > 30
    assert res["cand_npts"].max() > 4096 and res["cand_nvalid"].max() > 256
    assert (res["cand_topk"]["best"][:, 1] >= 0).sum() > 2      # the axis-aligned IoU ignores yaw: few survivors


def test_unsupported_options_raise():
    for bad in (dict(aln_w=0.1), dict(topk=0), dict(nms_3d=0.5), dict(search_depth=0.0)):
        with pytest.raises(NotImplementedError):
            SeekerEngine(dict(synth.seeker_params(synth.CONFIGS["tiny"]), **bad), device="cuda:0")


def test_score_mode_auto_picks_sweep_for_deep_grids_only():
    from findnpropagate_b200 import _lib
    for name, want in (("cfg1", "direct"), ("cfg2", "sweep")):
        cfg = synth.CONFIGS[name]
        eng = SeekerEngine(synth.seeker_params(cfg), device="cuda:0")
        eng.run([_frame_from_synth(synth.make_frame(0, cfg, device="cuda:0" if name == "cfg2" else "cpu"))])
        assert eng.last_score_mode == want
        assert (eng.M >= _lib.SWEEP_MIN_MAGS) == (want == "sweep")


@pytest.mark.parametrize("pack_xyz,loader_xyz", [(True, True), (False, True), (True, False), (False, False)])
def test_nuscenes_feed_to_pth_pipeline(tmp_path, pack_xyz, loader_xyz):
    """Row f2 end to end: nuScenes-format files -> NuScenesFeed (prefetch threads) -> HostPointFeeder
    (threaded x,y,z gather, double-buffered H2D) -> the five stages -> one .pth per frame.  The
    pipelined driver must give what the plain per-batch path gives on the same frames, bit for
    bit, with and without the host-side column gather."""
    from findnpropagate_b200 import extract, nuscenes_feed, proposer
    cfg = synth.CONFIGS["cfg1"]
    params = synth.seeker_params(cfg)
    sf = [synth.make_frame(i, cfg) for i in range(5)]
    infos = synth.write_nuscenes_tree(str(tmp_path / "nusc"), sf)
    feed = nuscenes_feed.NuScenesFeed(tmp_path / "nusc", infos, max_sweeps=1)
    glip = proposer.SyntheticGLIP(sf)
    eng = SeekerEngine(params, device="cuda:0")
    out_dir = tmp_path / "pl"
    merged, total, ar = extract.extract_nuscenes(feed, glip, eng, folder=str(out_dir), batch_frames=2, nms_thresh=0.1,
                                                 pack_xyz=pack_xyz, workers=2, loader_xyz=loader_xyz)
    assert len(merged) == 5
    frames = [feed.frame_input(i, glip)[0] for i in range(5)]
    ref = SeekerEngine(params, device="cuda:0").run(frames, with_recall=True, nms_thresh=0.1)
    assert {k: total[k] for k in ref["recall"]} == ref["recall"]
    for i, f in enumerate(sf):
        assert np.array_equal(merged[i]["pred_boxes"].view(np.uint32), ref["frames"][i]["pred_boxes"].view(np.uint32))
        assert np.array_equal(merged[i]["pred_labels"], ref["frames"][i]["pred_labels"])
        saved = torch.load(str(out_dir / (f.frame_id.replace(".", "_") + ".pth")), map_location="cpu")
        assert isinstance(saved, list) and len(saved) == 1
        assert np.array_equal(saved[0]["pred_boxes"].numpy(), merged[i]["pred_boxes"])
        assert saved[0]["pred_labels"].dtype == torch.int32
    # a page pool too small for a batch: the pipeline runs that batch again in a grown pool, with the same results
    starved = SeekerEngine(params, device="cuda:0")
    starved.pts_factor = 0.05
    merged2, total2, _ = extract.extract_nuscenes(feed, glip, starved, batch_frames=2, nms_thresh=0.1, pack_xyz=pack_xyz,
                                                  workers=2, loader_xyz=loader_xyz)
    assert starved.pts_factor > 0.05 and total2 == total
    for a, b in zip(merged2, merged):
        assert set(a) == set(b) and all(np.array_equal(a[k], b[k]) for k in a)
    # the feed reproduces the generator's frames: same points after the range filter, same detections
    assert np.array_equal(frames[0].points, sf[0].points[nuscenes_feed.mask_points_by_range(sf[0].points, nuscenes_feed.POINT_CLOUD_RANGE)])
    assert sum(m["pred_boxes"].shape[0] for m in merged) > 0
