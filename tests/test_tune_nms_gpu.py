"""Scoring tuning settings after load_pseudos' NMS: fnp_seg_nms_rotated_multi against one fnp_seg_nms_rotated call per
(setting, threshold), SeekerEngine.evaluate_settings(nms_thresh=...) against separate engines run with execute(nms_thresh),
and tune_params --nms_thresh against extract_pseudo_labels + eval_pseudo_labels --nms_thresh on the extracted folders
(nuScenes and KITTI)."""
import ctypes as C
import json

import numpy as np
import pytest
import torch

from findnpropagate_b200 import _lib, quality, synth, tune_params
from findnpropagate_b200.seeker import SeekerEngine

from test_extract_cli import HEAD, _frames, _write_tree, _write_yaml
from test_kitti_feed_cpu import KITTI_HEAD, _kitti_cfg, _kitti_frames, write_kitti_tree
from test_tune_gpu import SELECT, _inputs

pytestmark = pytest.mark.gpu

# ------------------------------------------------------------------------------------------------- 1: the kernel
def _segment_boxes(rng, n):
    """n rotated boxes packed so that many overlap (about 0.3 boxes per 4 m^2), some exact duplicates."""
    side = max(2.0, np.sqrt(n * 4.0 / 0.3))
    b = np.zeros((n, 7), np.float32)
    b[:, 0:2] = rng.uniform(0, side, (n, 2))
    b[:, 2] = rng.uniform(-1, 1, n)
    b[:, 3:6] = rng.uniform(0.5, 4.5, (n, 3))
    b[:, 6] = rng.uniform(-np.pi, np.pi, n)
    if n > 3:
        dup = rng.choice(n, n // 8 + 1, replace=False)
        b[dup] = b[rng.choice(n, dup.size)]
    return b


def _case(sizes, S, seed=0):
    """Boxes (S, N, 7), valid (S, N), the shared order and seg_start.  Settings jitter some boxes and flags; the scores
    have ties (one decimal), resolved by row as fnp_host_nms_order resolves them."""
    rng = np.random.default_rng(seed)
    base = np.concatenate([_segment_boxes(rng, n) for n in sizes]) if sum(sizes) else np.zeros((0, 7), np.float32)
    N = base.shape[0]
    boxes = np.repeat(base[None], S, 0)
    valid = np.zeros((S, N), np.int32)
    for s in range(S):
        if s:
            moved = rng.random(N) < 0.3
            boxes[s, moved, :2] += rng.normal(0, 0.3, (moved.sum(), 2)).astype(np.float32)
        valid[s, rng.random(N) < 0.15] = -1
    seg = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    score = np.round(rng.random(N), 1).astype(np.float32)
    frame = np.repeat(np.arange(len(sizes)), sizes)
    order = np.lexsort((np.arange(N), -score, frame)).astype(np.int32)
    return boxes, valid, order, seg


def _multi(boxes, valid, order, seg, thresh, max_seg=None):
    S, N = valid.shape
    dev = "cuda"
    tb, tv = torch.from_numpy(boxes).to(dev), torch.from_numpy(valid).to(dev)
    to, ts = torch.from_numpy(order).to(dev), torch.from_numpy(seg).to(dev)
    out = torch.full((len(thresh), S, max(N, 1)), 7, dtype=torch.int32, device=dev)
    th = (C.c_float * len(thresh))(*thresh)
    max_seg = int(np.diff(seg).max(initial=0)) if max_seg is None else max_seg
    rc = _lib.lib.fnp_seg_nms_rotated_multi(tb.data_ptr(), N, tv.data_ptr(), N, to.data_ptr(), ts.data_ptr(),
                                            len(seg) - 1, S, max(max_seg, 1), th, len(thresh), out.data_ptr(),
                                            out.shape[2], _lib.current_stream())
    assert rc == 0
    return out.cpu().numpy()[:, :, :N]


def _single(boxes, valid, order, seg, t):
    """fnp_seg_nms_rotated of one setting, its keep_mask mapped to 0 (kept) / -1."""
    N = valid.shape[0]
    tb, tv = torch.from_numpy(np.ascontiguousarray(boxes)).cuda(), torch.from_numpy(np.ascontiguousarray(valid)).cuda()
    to, ts = torch.from_numpy(order).cuda(), torch.from_numpy(seg).cuda()
    keep = torch.full((max(N, 1),), 9, dtype=torch.uint8, device="cuda")
    rc = _lib.lib.fnp_seg_nms_rotated(tb.data_ptr(), None, to.data_ptr(), tv.data_ptr(), ts.data_ptr(), len(seg) - 1,
                                      max(int(np.diff(seg).max(initial=0)), 1), float(t), keep.data_ptr(),
                                      _lib.current_stream())
    assert rc == 0
    k = keep.cpu().numpy()[:N]
    assert set(np.unique(k)) <= {0, 1}
    return np.where(k == 1, 0, -1).astype(np.int32)


def _pair_iou(boxes, valid, order, seg):
    """The IoU iou_bev gives a pair of valid boxes of the first large segment (earlier one first), between 0.05 and
    0.9: a threshold equal to it bit for bit."""
    for g in range(len(seg) - 1):
        idx = order[seg[g]:seg[g + 1]]
        idx = idx[valid[idx] >= 0]
        if idx.size < 8:
            continue
        a = torch.from_numpy(boxes[idx]).cuda()
        out = torch.empty((idx.size, idx.size), dtype=torch.float32, device="cuda")
        assert _lib.lib.fnp_boxes_iou_bev(a.data_ptr(), a.data_ptr(), out.data_ptr(), idx.size, idx.size,
                                          _lib.current_stream()) == 0
        iou = np.triu(out.cpu().numpy(), 1)
        hit = np.argwhere((iou > 0.05) & (iou < 0.9))
        if len(hit):
            return float(iou[tuple(hit[0])])
    raise AssertionError("no overlapping pair")


SIZES = [0, 1, 63, 64, 65, 1023, 1024]


@pytest.mark.parametrize("sizes,S,extra", [
    (SIZES, 1, ()),
    (SIZES, 3, (-0.2,)),                 # a negative threshold: no pre-filter for any threshold of the launch
    ([0, 1, 63, 64, 65, 200], 300, ()),  # more settings than one select_multi launch takes
    ([5, 300, 512, 130], 2, (0.0, 0.05, 0.2, 0.4, 0.7)),       # 8 thresholds at 512 boxes: chunks of 6 and 2
    (SIZES, 2, (0.0, 0.05, 0.2, 0.4, 0.7)),                    # 8 thresholds at 1024 boxes: one at a time
])
def test_kernel_equals_single_calls(sizes, S, extra):
    boxes, valid, order, seg = _case(sizes, S, seed=S)
    thresh = [0.1, 0.3, 0.5] + list(extra)
    if S < 300:
        thresh[1] = _pair_iou(boxes[0], valid[0], order, seg)        # an IoU the kernel meets exactly
    got = _multi(boxes, valid, order, seg, thresh)
    suppressed = 0
    for s in range(S):
        for t, th in enumerate(thresh):
            ref = _single(boxes[s], valid[s], order, seg, th)
            assert np.array_equal(got[t, s], ref), (s, th)
            suppressed += int(((ref < 0) & (valid[s] >= 0)).sum())
    assert suppressed > 0


def test_kernel_refusals():
    boxes, valid, order, seg = _case([10, 20], 2)
    tb, tv = torch.from_numpy(boxes).cuda(), torch.from_numpy(valid).cuda()
    to, ts = torch.from_numpy(order).cuda(), torch.from_numpy(seg).cuda()
    out = torch.zeros((8, 2, 30), dtype=torch.int32, device="cuda")
    st = _lib.current_stream()

    def call(n_thresh=1, b=tb.data_ptr(), bs=30, v=tv.data_ptr(), vs=30, o=to.data_ptr(), s=ts.data_ptr(), nseg=2,
             nset=2, cap=20, th=(C.c_float * 9)(*([0.1] * 9)), k=out.data_ptr(), ks=30):
        return _lib.lib.fnp_seg_nms_rotated_multi(b, bs, v, vs, o, s, nseg, nset, cap, th, n_thresh, k, ks, st)

    assert call() == 0 and call(n_thresh=8) == 0
    for bad in (dict(n_thresh=0), dict(n_thresh=9), dict(bs=-1), dict(vs=-1), dict(ks=-1), dict(nseg=-1),
                dict(nset=-1), dict(cap=-1), dict(cap=_lib.SEG_NMS_MAX + 1), dict(b=None), dict(v=None), dict(o=None),
                dict(s=None), dict(k=None), dict(th=None)):
        assert call(**bad) == -1, bad
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------- 2: the engine
NMS = (0.1, 0.3, 0.5)


def test_evaluate_settings_equals_separate_engines():
    cfg, frames = _inputs("cfg1", 4)
    base = synth.seeker_params(cfg)
    groups = tune_params.group_settings(base, [dict(s) for s in SELECT])
    spec = quality.QualitySpec(synth.CLASS_NAMES)
    suppressed = 0
    for g in groups:
        eng = SeekerEngine(g["params"], device="cuda:0")
        plan, pts, gt = eng.plan(frames), eng.upload_points(frames), eng.upload_gt(frames)
        with pytest.raises(ValueError, match="quality"):
            eng.evaluate_settings(plan, pts, gt, g["settings"], nms_thresh=NMS)
        res = eng.evaluate_settings(plan, pts, gt, g["settings"], quality=spec, nms_thresh=NMS)
        F, S = plan["F"], len(g["settings"])
        planes = eng.arena.bufs["nms_keep"][:4 * len(NMS) * S * F].view(torch.int32).view(len(NMS), S, F).cpu().numpy()
        plain = eng.evaluate_settings(plan, pts, gt, g["settings"], quality=spec)
        for a, b in zip(plain["settings"], res["settings"]):
            b = dict(b)
            assert len(b.pop("nms")) == len(NMS)
            assert set(a) == set(b)
            for k in a:
                assert np.array_equal(a[k], b[k]) if isinstance(a[k], np.ndarray) else a[k] == b[k], k
        fcs = plan["frame_cand_start"]
        for i, got in zip(g["members"], res["settings"]):
            ref_eng = SeekerEngine(dict(base, **SELECT[i]), device="cuda:0")
            ref_plan = ref_eng.plan(frames)
            assert np.array_equal(ref_plan["frame_cand_start"], fcs)
            for t, th in enumerate(NMS):
                ref = ref_eng.finish(ref_eng.execute(ref_plan, pts, nms_thresh=th))
                kept = np.zeros(F, bool)
                kept[np.flatnonzero(ref["cand_valid"])] = np.concatenate(
                    [f["nms_keep"] for f in ref["frames"]]).astype(bool)
                s = g["members"].index(i)
                assert np.array_equal(planes[t, s] == 0, kept), (SELECT[i], th)
                assert np.array_equal(planes[t, s] < 0, ~kept)
                suppressed += int(ref["cand_valid"].sum() - kept.sum())
                # the counters: fnp_quality_counters over that engine's kept proposals
                counters = torch.zeros(spec.n_counters, dtype=torch.int64, device="cuda")
                quality.launch(spec, torch.from_numpy(ref["cand_boxes"]).cuda(),
                               torch.from_numpy(plan["cand_label"].astype(np.int32)).cuda(),
                               torch.from_numpy(fcs.astype(np.int32)).cuda(), gt[0], gt[1], len(frames),
                               max(plan["max_cands"], 1), int(gt[2]), counters,
                               pred_valid=torch.from_numpy(np.where(kept, 0, -1).astype(np.int32)).cuda())
                assert np.array_equal(got["nms"][t], counters.cpu().numpy()), (SELECT[i], th)
    assert suppressed > 0


# ------------------------------------------------------------------------------------------------- 3, 4: the command
@pytest.fixture
def cfg1_tree(tmp_path, monkeypatch):
    frames = _frames("cfg1", 5)
    tools = _write_tree(tmp_path, frames)
    monkeypatch.chdir(tools)
    return tmp_path, frames


GRID = {"MODEL.DENSE_HEAD.PARAMS.dns_w": [1.0, 0.2], "MODEL.DENSE_HEAD.PARAMS.min_cam_iou": [0.3, 0.5],
        "MODEL.DENSE_HEAD.PARAMS.num_mags": [6, 4]}
FIELDS = ("proposals", "recall", "ar", "precision", "classes")


def _against_eval(cfg_file, lines, thresh):
    """Every line's nms entries against eval_pseudo_labels --nms_thresh on the folder extract_pseudo_labels writes
    with the line's setting."""
    from findnpropagate_b200 import eval_pseudo_labels as ev
    from findnpropagate_b200 import extract_pseudo_labels as cli
    for k, d in enumerate(lines):
        sets = [x for key, v in d["setting"].items() for x in (key, repr(v))]
        cli.main(["--cfg_file", cfg_file, "--folder", "../nms_out%d" % k, "--set"] + sets)
        got = ev.main(["--cfg_file", cfg_file, "--folder", "../nms_out%d" % k, "--nms_thresh"] + [str(t) for t in thresh])
        assert [e["nms"] for e in got] == ["none"] + list(thresh)
        for e, t in zip(got[1:], thresh):
            for f in FIELDS:
                assert d["nms"][str(t)][f] == e[f], (d["setting"], t, f)
        assert d["proposals"] == got[0]["proposals"] and d["recall"] == got[0]["recall"]


def _pre_nms(d):
    return {k: v for k, v in d.items() if k not in ("nms", "classes")}


def test_command_equals_eval_on_extracted_folders(cfg1_tree, capsys):
    base, frames = cfg1_tree
    _write_yaml(str(base / "tools" / "grid.yaml"), GRID)
    args = ["--cfg_file", HEAD, "--grid", "grid.yaml", "--nms_thresh", "0.1", "0.3", "--breakdown"]
    lines = tune_params.main(args + ["--batch_frames", "2"])
    out = capsys.readouterr().out
    assert "8 settings in 2 groups" in out and "after the NMS at 0.1" in out.split("best setting")[1]
    ar = [d["nms"]["0.1"]["ar"]["0.5"] for d in lines]
    assert ar == sorted(ar, reverse=True) and len(lines) == 8
    assert all(set(d["nms"]) == {"0.1", "0.3"} for d in lines)
    assert any(d["nms"]["0.1"]["proposals"] < d["proposals"] for d in lines)
    plain = {json.dumps(d["setting"]): d for d in tune_params.main(["--cfg_file", HEAD, "--grid", "grid.yaml"])}
    for d in lines:
        assert _pre_nms(d) == plain[json.dumps(d["setting"])]
    assert tune_params.main(args + ["--batch_frames", "1"]) == lines
    assert tune_params.main(args + ["--batch_frames", "64"]) == lines
    _against_eval(HEAD, lines, (0.1, 0.3))


def test_command_equals_eval_on_kitti(tmp_path, monkeypatch):
    cfg = _kitti_cfg(params=dict(nms_3d=0.0, score_thr=0.45, nms_2d=0.4, dns_w=1.0))
    tools = write_kitti_tree(tmp_path, _kitti_frames(6), cfg=cfg)
    monkeypatch.chdir(tools)
    _write_yaml(str(tmp_path / "tools" / "grid.yaml"), {"MODEL.DENSE_HEAD.PARAMS.dns_w": [1.0, 0.2, 3.0]})
    lines = tune_params.main(["--cfg_file", KITTI_HEAD, "--grid", "grid.yaml", "--nms_thresh", "0.1", "--breakdown",
                              "--batch_frames", "4"])
    assert len(lines) == 3 and lines[0]["recall"]["gt"] > 0
    ar = [d["nms"]["0.1"]["ar"]["0.5"] for d in lines]
    assert ar == sorted(ar, reverse=True)
    _against_eval(KITTI_HEAD, lines, (0.1,))
