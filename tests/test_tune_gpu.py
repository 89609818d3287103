"""Scoring many head settings over one execution of stages 1-2c (SeekerEngine.evaluate_settings,
fnp_seeker_select_multi, fnp_precision_counters) and the tune_params command, against separate engines and the
extraction command."""
import json

import numpy as np
import pytest
import torch

from findnpropagate_b200 import synth, tune_params
from findnpropagate_b200.seeker import FrameInput, SeekerEngine

from test_extract_cli import HEAD, _frames, _write_tree, _write_yaml

pytestmark = pytest.mark.gpu

THRESH = (0.3, 0.5, 0.7)
# every select-level key: a min_cam_iou above the base, MULT, OCCL_MULT, ego_w, occl_w, dst_w of both signs
SELECT = [dict(), dict(dns_w=0.5), dict(iou_w=0.7, min_cam_iou=0.5), dict(dst_w=0.3), dict(dst_w=-0.2, min_cam_iou=0.4),
          dict(ego_w=0.2), dict(occl_w=0.3), dict(MULT=True, dst_w=0.5), dict(OCCL_MULT=True),
          dict(occl_w=0.1, ego_w=0.1, dst_w=0.2, min_cam_iou=0.45), dict(MULT=True, dst_w=1.0, min_cam_iou=0.6),
          dict(min_cam_iou=0.9)]
# a cfg2-shaped hypothesis grid (64 depth steps x 12 yaws: H = 768, the sweep kernel) on fewer points
CFG2_SMALL = synth.SynthConfig("cfg2_small", 32, 1085, 2, 60, 64, 12, 1)


def _inputs(name, n):
    cfg = synth.CONFIGS.get(name, CFG2_SMALL)
    dev = "cuda:0" if cfg.num_mags > 16 else "cpu"
    return cfg, [FrameInput(points=f.points, lidar2image=f.lidar2image, camera2lidar=f.camera2lidar,
                            camera_intrinsics=f.camera_intrinsics, det_boxes=f.det_boxes, det_labels=f.det_labels,
                            det_scores=f.det_scores, det_cam_idx=f.det_cam_idx, gt_boxes=f.gt_boxes)
                 for f in (synth.make_frame(i, cfg, device=dev) for i in range(n))]


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _precision(frames, res):
    """fnp_precision_counters restated with the op-level boxes_iou3d_gpu: per frame the row max over the GT boxes."""
    from findnpropagate_b200.pcdet_ops import iou3d_nms_utils
    out = np.zeros(1 + len(THRESH), np.int64)
    for f, pred in zip(frames, res["frames"]):
        k = pred["pred_boxes"].shape[0]
        out[0] += k
        if k == 0 or f.gt_boxes is None or len(f.gt_boxes) == 0:
            continue
        iou = iou3d_nms_utils.boxes_iou3d_gpu(torch.from_numpy(np.ascontiguousarray(pred["pred_boxes"])).cuda(),
                                              torch.from_numpy(np.ascontiguousarray(f.gt_boxes[:, :7], np.float32)).cuda())
        best = iou.max(dim=1).values.cpu().numpy()
        for t, th in enumerate(THRESH):
            out[1 + t] += int((best > th).sum())
    return out


@pytest.mark.parametrize("name,n_frames,split", [("cfg1", 4, dict(lq=0.05)), ("cfg2_small", 2, dict(num_mags=48))])
def test_shared_path_equals_separate_engines(name, n_frames, split):
    cfg, frames = _inputs(name, n_frames)
    base = synth.seeker_params(cfg)
    settings = [dict(s) for s in SELECT] + [dict(s, **split) for s in SELECT]
    groups = tune_params.group_settings(base, settings)
    assert [g["members"] for g in groups] == [list(range(12)), list(range(12, 24))]
    checked = 0
    for g in groups:
        eng = SeekerEngine(g["params"], device="cuda:0", debug=True)
        plan = eng.plan(frames)
        pts, gt = eng.upload_points(frames), eng.upload_gt(frames)
        with pytest.raises(ValueError):          # below the compaction threshold of the shared execution
            eng.evaluate_settings(plan, pts, gt, [dict(min_cam_iou=0.2)])
        h = eng.execute(plan, pts, gt=gt, settings=g["settings"])
        res = eng.finish(h)
        hyp_index = eng.debug_views(h)["hyp_index"]
        F = plan["F"]
        # the group's own cfg is its first setting: select_kernel's out_* of the same execution
        own = res["settings"][0]
        assert np.array_equal(own["cand_best"], res["cand_best"])
        v = res["cand_valid"]
        assert np.array_equal(_bits(own["cand_score2"][v]), _bits(res["cand_score2"][v]))
        assert np.array_equal(_bits(own["cand_boxes"][v]), _bits(res["cand_boxes"][v]))
        assert own["recall"] == res["recall"]
        for i, got in zip(g["members"], res["settings"]):
            p = dict(base)
            p.update(settings[i])
            ref_eng = SeekerEngine(p, device="cuda:0", debug=True)
            rh = ref_eng.execute(ref_eng.plan(frames), pts, gt=gt)
            ref = ref_eng.finish(rh)
            ref_index = ref_eng.debug_views(rh)["hyp_index"]
            valid = ref["cand_valid"]
            assert np.array_equal(got["cand_best"] >= 0, valid), settings[i]
            rows = np.flatnonzero(valid)
            assert np.array_equal(hyp_index[rows, got["cand_best"][rows]], ref_index[rows, ref["cand_best"][rows]]), settings[i]
            assert np.array_equal(_bits(got["cand_score2"][rows]), _bits(ref["cand_score2"][rows])), settings[i]
            assert np.array_equal(got["cand_count"][rows], ref["cand_count"][rows])
            assert np.array_equal(_bits(got["cand_boxes"][rows]), _bits(ref["cand_boxes"][rows]))
            assert not got["cand_boxes"][~valid].any() and not got["cand_score2"][~valid].any()
            # per frame: the proposals in order, with their labels and 2D scores
            fcs = plan["frame_cand_start"]
            for b, pred in enumerate(ref["frames"]):
                sel = [c for c in range(fcs[b], fcs[b + 1]) if got["cand_best"][c] >= 0]
                assert np.array_equal(_bits(got["cand_boxes"][sel]), _bits(pred["pred_boxes"]))
                assert np.array_equal(plan["cand_label"][sel], pred["pred_labels"])
                assert np.array_equal(_bits(plan["cand_score"][sel]), _bits(pred["pred_scores"]))
            assert got["recall"] == ref["recall"], settings[i]
            assert got["proposals"] == int(valid.sum()) == got["precision"]["proposals"]
            prec = _precision(frames, ref)
            assert [got["precision"]["proposals"]] + [got["precision"]["hits_%s" % t] for t in THRESH] == prec.tolist()
            checked += int(valid.sum())
        assert F > 0
    assert checked > 20


def test_select_terms_change_the_choice():
    """The grid is not degenerate: the settings above pick different hypotheses and proposal counts."""
    cfg, frames = _inputs("cfg1", 4)
    g = tune_params.group_settings(synth.seeker_params(cfg), SELECT)[0]
    eng = SeekerEngine(g["params"], device="cuda:0")
    res = eng.evaluate_settings(eng.plan(frames), eng.upload_points(frames), eng.upload_gt(frames), g["settings"])
    best = np.stack([s["cand_best"] for s in res["settings"]])
    assert len({b.tobytes() for b in best}) >= 6
    assert len({s["proposals"] for s in res["settings"]}) >= 3


@pytest.fixture
def cfg1_tree(tmp_path, monkeypatch):
    frames = _frames("cfg1", 5)
    tools = _write_tree(tmp_path, frames)
    monkeypatch.chdir(tools)
    return tmp_path, frames


GRID = {"MODEL.DENSE_HEAD.PARAMS.dns_w": [1.0, 0.2], "MODEL.DENSE_HEAD.PARAMS.min_cam_iou": [0.3, 0.5],
        "MODEL.DENSE_HEAD.PARAMS.num_mags": [6, 4]}


def test_command_equals_extraction_per_setting(cfg1_tree, capsys):
    from findnpropagate_b200 import extract_pseudo_labels as cli
    base, frames = cfg1_tree
    _write_yaml(str(base / "tools" / "grid.yaml"), GRID)
    lines = tune_params.main(["--cfg_file", HEAD, "--grid", "grid.yaml", "--batch_frames", "2", "--out", "../res.jsonl"])
    out = capsys.readouterr().out
    assert "8 settings in 2 groups" in out and "frames scored: 5, failed frames: 0" in out
    assert [json.loads(t) for t in open(base / "res.jsonl")] == lines
    ar = [d["ar"]["0.5"] for d in lines]
    assert ar == sorted(ar, reverse=True) and len(lines) == 8
    assert {d["group"] for d in lines} == {0, 1}
    assert "--set" in out.split("best setting:")[1]
    for k, d in enumerate(lines):
        sets = [x for key, v in d["setting"].items() for x in (key, repr(v))]
        got = cli.main(["--cfg_file", HEAD, "--folder", "../out%d" % k, "--batch_frames", "3", "--set"] + sets)
        assert d["recall"] == got["recall"], d["setting"]
        assert d["recall"]["gt"] > 0
        for t in THRESH:
            assert d["ar"][str(t)] == got["ar"]["rcnn_%s" % t]
    # batch independence: one frame per batch gives the same lines
    assert tune_params.main(["--cfg_file", HEAD, "--grid", "grid.yaml", "--batch_frames", "1"]) == lines
    assert tune_params.main(["--cfg_file", HEAD, "--grid", "grid.yaml", "--batch_frames", "64"]) == lines


def test_every_and_keys_missing_from_the_config(cfg1_tree, capsys):
    base, frames = cfg1_tree
    _write_yaml(str(base / "tools" / "grid.yaml"), {"MODEL.DENSE_HEAD.OCCL_MULT": [False, True],
                                                    "MODEL.DENSE_HEAD.PARAMS.ego_w": [0.0, 0.3]})
    lines = tune_params.main(["--cfg_file", HEAD, "--grid", "grid.yaml", "--every", "2"])
    out = capsys.readouterr().out
    assert "frames scored: 3" in out and "4 settings in 1 groups" in out
    assert "add OCCL_MULT" in out and "add ego_w" in out
    # against the library on frames 0, 2, 4 with each setting
    params = synth.seeker_params(synth.CONFIGS["cfg1"])
    for d in lines:
        p = dict(params, OCCL_MULT=d["setting"]["MODEL.DENSE_HEAD.OCCL_MULT"],
                 ego_w=d["setting"]["MODEL.DENSE_HEAD.PARAMS.ego_w"])
        ref = _library_run_every(base, frames, p)
        assert d["recall"] == ref["recall"], d["setting"]


def _library_run_every(base, frames, params):
    import os
    from findnpropagate_b200 import nuscenes_feed, proposer
    from test_extract_cli import GLIP_META, GLIP_PTH, INFOS, NUSC
    feed = nuscenes_feed.NuScenesFeed(os.path.join(str(base), NUSC), INFOS, max_sweeps=1, training=True)
    det = proposer.PreprocessedGLIP(os.path.join(str(base), GLIP_PTH), os.path.join(str(base), GLIP_META))
    eng = SeekerEngine(params, device="cuda:0")
    return eng.run([feed.frame_input(i, det)[0] for i in range(0, len(frames), 2)], with_recall=True)


def _big_grid():
    return [dict(dns_w=d, iou_w=i, dst_w=t, min_cam_iou=m, MULT=u) for d in (0.05, 0.5, 1.0, 2.0, 4.0)
            for i in (0.25, 0.5, 1.0, 2.0) for t in (0.0, 0.1, 0.2, 0.4) for m in (0.3, 0.5) for u in (False, True)]


def _same(a, b):
    assert a["recall"] == b["recall"] and a["precision"] == b["precision"] and a["proposals"] == b["proposals"]
    assert np.array_equal(a["cand_best"], b["cand_best"]) and np.array_equal(a["cand_count"], b["cand_count"])
    assert np.array_equal(_bits(a["cand_score2"]), _bits(b["cand_score2"]))
    assert np.array_equal(_bits(a["cand_boxes"]), _bits(b["cand_boxes"]))


def test_more_settings_than_one_launch():
    """320 settings in one group: stage 3 runs in launches of 256 over the same stages 1-2c, with the results of
    smaller calls and of separate engines; a key a setting leaves out takes the engine's value."""
    cfg, frames = _inputs("cfg1", 4)
    base = synth.seeker_params(cfg)
    settings = _big_grid()
    g = tune_params.group_settings(base, settings)
    assert len(g) == 1 and len(g[0]["settings"]) == 320
    eng = SeekerEngine(g[0]["params"], device="cuda:0")
    plan, pts, gt = eng.plan(frames), eng.upload_points(frames), eng.upload_gt(frames)
    whole = eng.evaluate_settings(plan, pts, gt, g[0]["settings"])["settings"]
    halves = (eng.evaluate_settings(plan, pts, gt, g[0]["settings"][:160])["settings"]
              + eng.evaluate_settings(plan, pts, gt, g[0]["settings"][160:])["settings"])
    for a, b in zip(whole, halves):
        _same(a, b)
    for i in (0, 255, 256, 257, 319):
        ref = SeekerEngine(dict(base, **settings[i]), device="cuda:0").run(frames, with_recall=True)
        assert whole[i]["recall"] == ref["recall"], settings[i]
        assert np.array_equal(whole[i]["cand_best"] >= 0, ref["cand_valid"])
        v = ref["cand_valid"]
        assert np.array_equal(_bits(whole[i]["cand_score2"][v]), _bits(ref["cand_score2"][v]))
    partial = eng.evaluate_settings(plan, pts, gt, [dict(dns_w=0.5)])["settings"][0]
    _same(partial, eng.evaluate_settings(plan, pts, gt, [dict(g[0]["params"], dns_w=0.5)])["settings"][0])


def test_command_with_more_settings_than_one_launch(cfg1_tree, capsys):
    base, frames = cfg1_tree
    grid = {"MODEL.DENSE_HEAD.PARAMS.dns_w": [0.05, 0.5, 1.0, 2.0, 4.0], "MODEL.DENSE_HEAD.PARAMS.iou_w": [0.25, 0.5, 1.0, 2.0],
            "MODEL.DENSE_HEAD.PARAMS.dst_w": [0.0, 0.1, 0.2, 0.4], "MODEL.DENSE_HEAD.PARAMS.min_cam_iou": [0.3, 0.5],
            "MODEL.DENSE_HEAD.PARAMS.num_mags": [6, 4]}
    _write_yaml(str(base / "tools" / "grid.yaml"), grid)
    lines = tune_params.main(["--cfg_file", HEAD, "--grid", "grid.yaml", "--every", "2"])
    assert "320 settings in 2 groups" in capsys.readouterr().out
    assert len(lines) == 320 and lines[0]["recall"]["gt"] > 0
