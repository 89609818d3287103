"""The commands on a KITTI config, on the GPU: extract_pseudo_labels against FrustumProposerOGKITTI.get_bboxes fed one
collated KittiFeed frame at a time, the shared tuning pass for the KITTI head (select_multi_kernel<true>) against
separate engines, fnp_seeker_select_multi's KITTI rule called through the C entry, and eval_pseudo_labels on the
extracted folder against a restatement on boxes_iou3d_gpu."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from findnpropagate_b200 import _lib, quality, synth, tune_params
from findnpropagate_b200.seeker import SeekerEngine

from test_kitti_feed_cpu import KITTI_DATA, KITTI_HEAD, _kitti_frames, write_kitti_tree
from test_quality_gpu import restate
from test_tune_gpu import THRESH, _bits

pytestmark = pytest.mark.gpu

N_FRAMES = 6


@pytest.fixture
def kitti_tree(tmp_path, monkeypatch):
    """Six frames; frame 3 is not in the predictions."""
    tools = write_kitti_tree(tmp_path, _kitti_frames(N_FRAMES), predicted=[k for k in range(N_FRAMES) if k != 3])
    monkeypatch.chdir(tools)
    return tmp_path


def _setup():
    from findnpropagate_b200 import extract_pseudo_labels as cli
    cfg = cli.load_config(KITTI_HEAD)
    head = cli.build_head(cfg, device="cuda:0")
    return cli, cfg, head, cli.build_feed(cfg, device=head.engine.device)


def _assert_file(folder, fid, pred):
    s = torch.load(os.path.join(str(folder), fid + ".pth"), map_location="cpu")
    assert isinstance(s, list) and len(s) == 1
    s = s[0]
    assert s["pred_labels"].dtype == torch.int32
    assert np.array_equal(_bits(s["pred_boxes"].numpy()), _bits(np.asarray(pred["pred_boxes"]).reshape(-1, 7)))
    assert np.array_equal(_bits(s["pred_scores"].numpy()), _bits(pred["pred_scores"]))
    assert np.array_equal(s["pred_labels"].numpy(), np.asarray(pred["pred_labels"]))


def test_extraction_equals_the_head_frame_by_frame(kitti_tree, capsys):
    from findnpropagate_b200 import extract
    from findnpropagate_b200.nuscenes_feed import collate_batch
    base = kitti_tree
    os.remove(base / KITTI_DATA / "training" / "velodyne" / "000001.bin")
    cli, cfg, head, feed = _setup()
    got = cli.main(["--cfg_file", KITTI_HEAD, "--folder", "../out", "--batch_frames", "2", "--workers", "2"])
    out = capsys.readouterr().out
    assert got["frames"] == N_FRAMES - 2 and got["failed"] == 2
    assert got["failed_frames"] == [("000001", cli.FAILURES[cli.LIDAR_MISSING]),
                                    ("000003", cli.FAILURES[cli.IMAGE_NOT_PREDICTED])]
    assert "skipped frame 000001" in out and "skipped frame 000003" in out
    ok = [k for k in range(N_FRAMES) if k not in (1, 3)]
    assert sorted(os.listdir(base / "out")) == ["%06d.pth" % k for k in ok]
    n_boxes, frames = 0, []
    for k in ok:
        d = feed[k]
        assert d["frame_id"] == "%06d" % k
        ref = head.get_bboxes(collate_batch([d]))[0]          # the reference's batch size: one frame
        ref = {n: v.cpu().numpy() for n, v in ref.items()}
        _assert_file(base / "out", d["frame_id"], ref)
        n_boxes += ref["pred_boxes"].shape[0]
        frames.append(feed.frame_input(k, head.image_detector)[0])
    assert n_boxes > 5
    # the summed recall counters: the engine over the same frames, with their GT
    eng = SeekerEngine(head.params, device="cuda:0", box_format="xywh", variant="kitti")
    ref = eng.run(frames, with_recall=True)["recall"]
    assert {k: got["recall"][k] for k in ref} == ref and ref["gt"] > 0
    assert got["ar"] == {"rcnn_%s" % t: ref["rcnn_%s" % t] / ref["gt"] for t in extract.THRESH}
    # --nms_thresh: the stage-4 NMS is run as extract_nuscenes runs it
    got = cli.main(["--cfg_file", KITTI_HEAD, "--folder", "../nms", "--nms_thresh", "0.1", "--batch_frames", "3"])
    live = cli.build_feed(cfg, infos=[feed.infos[k] for k in ok], device=head.engine.device)
    merged, total, ar = extract.extract_nuscenes(live, head.image_detector, eng, batch_frames=3, nms_thresh=0.1)
    assert got["recall"] == total and got["ar"] == ar
    for k, pred in zip(ok, merged):
        assert "nms_keep" in pred
        _assert_file(base / "nms", "%06d" % k, pred)


def _kitti_frames_on_gpu(n=N_FRAMES):
    _, cfg, head, feed = _setup()
    return head, [feed.frame_input(k, head.image_detector)[0] for k in range(n) if k != 3]


def _same_setting(got, ref):
    assert np.array_equal(got["cand_best"], ref["cand_best"])
    assert np.array_equal(_bits(got["cand_score2"]), _bits(ref["cand_score2"]))
    assert np.array_equal(got["cand_count"], ref["cand_count"])
    assert np.array_equal(_bits(got["cand_boxes"]), _bits(ref["cand_boxes"]))
    assert got["recall"] == ref["recall"] and got["precision"] == ref["precision"]
    assert got["proposals"] == ref["proposals"]
    assert np.array_equal(got["quality"], ref["quality"])


@pytest.mark.parametrize("min_cam_iou", [[None], [0.3, 0.5]])
def test_tuning_equals_separate_engines(kitti_tree, min_cam_iou):
    head, frames = _kitti_frames_on_gpu()
    base = dict(head.params)
    settings = [dict(dns_w=d, iou_w=i, dst_w=t) for d in (0.05, 0.5, 2.0) for i in (0.5, 0.95) for t in (0.0, 0.226, -0.3)]
    if min_cam_iou != [None]:
        settings = [dict(s, min_cam_iou=m) for m in min_cam_iou for s in settings]
    groups = tune_params.group_settings(base, settings, "kitti")
    assert len(groups) == len(min_cam_iou)
    spec = quality.QualitySpec(synth.KITTI_CLASS_NAMES)
    distinct = set()
    for g in groups:
        eng = SeekerEngine(g["params"], device="cuda:0", box_format="xywh", variant="kitti")
        plan = eng.plan(frames)
        pts, gt = eng.upload_points(frames), eng.upload_gt(frames)
        res = eng.evaluate_settings(plan, pts, gt, g["settings"], recall_thresh=THRESH, quality=spec)["settings"]
        with pytest.raises(ValueError, match="KITTI"):
            eng.evaluate_settings(plan, pts, gt, [dict(min_cam_iou=0.9)])
        for i, got in zip(g["members"], res):
            ref_eng = SeekerEngine(dict(base, **settings[i]), device="cuda:0", box_format="xywh", variant="kitti")
            ref_plan = ref_eng.plan(frames)
            own = ref_eng.finish(ref_eng.execute(ref_plan, pts, gt=gt, recall_thresh=THRESH))     # select_kernel<true>
            alone = ref_eng.evaluate_settings(ref_plan, pts, gt, [{}], recall_thresh=THRESH, quality=spec)["settings"][0]
            v = own["cand_valid"]
            assert np.array_equal(got["cand_best"] >= 0, v), settings[i]
            assert np.array_equal(got["cand_best"], own["cand_best"]), settings[i]
            assert np.array_equal(_bits(got["cand_score2"][v]), _bits(own["cand_score2"][v])), settings[i]
            assert np.array_equal(got["cand_count"][v], own["cand_count"][v])
            assert np.array_equal(_bits(got["cand_boxes"][v]), _bits(own["cand_boxes"][v]))
            assert got["recall"] == own["recall"], settings[i]
            _same_setting(got, alone)
            distinct.add(got["cand_best"].tobytes())
    assert len(distinct) >= 4


def test_c_entry_kitti_rule(kitti_tree):
    """fnp_seeker_select_multi on a KITTI cfg: accepted when every setting keeps cfg's min_cam_iou bit for bit with no
    flags; FNP_EINVAL for another min_cam_iou, a flag, ego_w / occl_w, and topk > 1."""
    head, frames = _kitti_frames_on_gpu()
    eng = SeekerEngine(head.params, device="cuda:0", box_format="xywh", variant="kitti")
    plan = eng.plan(frames)
    h = eng.execute(plan, eng.upload_points(frames))
    own = eng.finish(h)
    F = plan["F"]
    L, stream = _lib.lib, _lib.current_stream(eng.device)
    boxes = torch.zeros((4, F, 7), dtype=torch.float32, device=eng.device)
    score = torch.zeros((4, F), dtype=torch.float32, device=eng.device)
    best = torch.zeros((4, F), dtype=torch.int32, device=eng.device)
    count = torch.zeros((4, F), dtype=torch.int32, device=eng.device)

    def call(sel, cfg=eng.cfg):
        arr = (_lib.SelectSetting * len(sel))(*sel)
        return L.fnp_seeker_select_multi(C.byref(cfg), C.byref(h["batch"]), arr, len(sel), boxes.data_ptr(),
                                         score.data_ptr(), best.data_ptr(), count.data_ptr(), stream)

    def setting(**kw):
        p = dict(dns_w=float(eng.p["dns_w"]), iou_w=float(eng.p["iou_w"]), dst_w=float(eng.p["dst_w"]), ego_w=0.0,
                 occl_w=0.0, min_cam_iou=eng.cfg.min_cam_iou, flags=0, reserved=0)
        p.update(kw)
        return _lib.SelectSetting(**p)

    assert call([setting(), setting(dns_w=2.0), setting(dst_w=0.0)]) == 0
    torch.cuda.synchronize()
    assert np.array_equal(best[0].cpu().numpy(), own["cand_best"])
    assert np.array_equal(_bits(score[0].cpu().numpy()), _bits(own["cand_score2"]))
    assert np.array_equal(count[0].cpu().numpy(), own["cand_count"])
    above = float(np.nextafter(np.float32(eng.cfg.min_cam_iou), np.float32(1)))
    for bad in (setting(min_cam_iou=0.5), setting(min_cam_iou=above), setting(flags=_lib.SEEKER_MULT),
                setting(ego_w=0.1), setting(occl_w=0.1)):
        assert call([setting(), bad]) != 0
    topk = _lib.SeekerCfg.from_buffer_copy(eng.cfg)
    topk.topk = 2
    assert call([setting()], topk) != 0


def test_eval_on_the_extracted_folder(kitti_tree, capsys):
    from findnpropagate_b200 import eval_pseudo_labels as ev
    from findnpropagate_b200.pseudo_loader import load_pseudos
    base = kitti_tree
    cli, cfg, head, feed = _setup()
    ext = cli.main(["--cfg_file", KITTI_HEAD, "--folder", "../out", "--batch_frames", "4"])
    capsys.readouterr()
    lines = ev.main(["--cfg_file", KITTI_HEAD, "--folder", "../out", "--nms_thresh", "0.1", "--batch_frames", "2"])
    spec = quality.QualitySpec(synth.KITTI_CLASS_NAMES)
    assert lines[0]["frames"] == N_FRAMES and lines[0]["missing_files"] == 1        # frame 3 was not extracted
    assert lines[0]["proposals"] > 0
    for d, t in zip(lines, (None, 0.1)):
        frames = []
        for k in range(N_FRAMES):
            g = feed.gt_boxes(k)
            g = np.concatenate([g[:, :7], g[:, -1:]], 1)
            if k == 3:
                b = np.zeros((0, 8), np.float32)
            else:
                b, _ = load_pseudos(base / "out", "%06d" % k, nms_thresh=t)
            frames.append((b[:, :7], b[:, 7].astype(np.int32), np.ones(len(b), bool), g))
        ref = restate(spec, frames)
        assert d["classes"] == quality.tables(ref, spec), t
        assert d["recall"] == quality.recall_dict(ref, spec)
    assert lines[0]["recall"]["gt"] == ext["recall"]["gt"] + len(feed.gt_boxes(3))
