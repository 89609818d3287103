"""fnp_quality_counters against a restatement with the op-level boxes_iou3d_gpu and numpy float32 range bins, against
fnp_recall_counters / fnp_precision_counters, over many settings; SeekerEngine.evaluate_settings(quality=...), the
eval_pseudo_labels command and tune_params --breakdown."""
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch

from findnpropagate_b200 import _lib, quality, synth, tune_params
from findnpropagate_b200.seeker import SeekerEngine

from test_extract_cli import HEAD, _frames, _write_tree, _write_yaml
from test_tune_gpu import GRID, SELECT, _inputs

pytestmark = pytest.mark.gpu

CLASSES = tuple(synth.CLASS_NAMES)
SPEC = quality.QualitySpec(CLASSES)


# ------------------------------------------------------------------------------------------------- restatement
def restate(spec, frames):
    """frames: per frame (boxes (K,7), labels (K,), valid (K,) bool, gt (G,8)).  The counters of one setting."""
    from findnpropagate_b200.pcdet_ops import iou3d_nms_utils
    R, W, T = spec.n_bins, spec.width, len(spec.thresh)
    out = np.zeros((2, len(spec.class_names), R, W), np.int64)
    edges = np.asarray(spec.range_edges, np.float32)
    th = np.asarray(spec.thresh, np.float32)

    def bins(b):
        x, y = b[:, 0].astype(np.float32), b[:, 1].astype(np.float32)
        r = np.sqrt((x * x).astype(np.float32) + (y * y).astype(np.float32)).astype(np.float32)
        return (edges[None, :] <= r[:, None]).sum(1) if len(edges) else np.zeros(len(r), np.int64)

    for boxes, labels, valid, gt in frames:
        g = quality.strip_gt(gt)
        p, pl = np.asarray(boxes, np.float32).reshape(-1, 7)[valid], np.asarray(labels)[valid]
        gl = g[:, 7].astype(np.int64)
        if len(p) and len(g):
            iou = iou3d_nms_utils.boxes_iou3d_gpu(torch.from_numpy(np.ascontiguousarray(p)).cuda(),
                                                  torch.from_numpy(np.ascontiguousarray(g[:, :7])).cuda()).cpu().numpy()
        else:
            iou = np.zeros((len(p), len(g)), np.float32)
        same = pl[:, None] == gl[None, :]
        masked = np.where(same, iou, -1.0)
        for blk, lab, bn, best_any, best_lab in (
                (0, gl, bins(g), iou.max(0, initial=-1.0), masked.max(0, initial=-1.0)),
                (1, pl, bins(p), iou.max(1, initial=-1.0), masked.max(1, initial=-1.0))):
            for i in range(len(lab)):
                c = out[blk, lab[i] - 1, bn[i]]
                c[0] += 1
                c[1:1 + T] += best_any[i] > th
                c[1 + T:] += best_lab[i] > th
    return out.reshape(-1)


def _device(frames, n_settings=1):
    """Concatenated device inputs of per-frame (boxes, labels, valid, gt); the valid flags as 0 / -1."""
    ks = [len(f[1]) for f in frames]
    gs = [len(f[3]) for f in frames]
    cat = lambda xs, shape, dt: np.ascontiguousarray(np.concatenate([np.asarray(x, dt).reshape(shape) for x in xs]))
    d = dict(pred=torch.from_numpy(cat([f[0] for f in frames], (-1, 7), np.float32)).cuda(),
             label=torch.from_numpy(cat([f[1] for f in frames], (-1,), np.int32)).cuda(),
             valid=torch.from_numpy(np.where(cat([f[2] for f in frames], (-1,), bool), 0, -1).astype(np.int32)).cuda(),
             pstart=torch.tensor(np.concatenate([[0], np.cumsum(ks)]), dtype=torch.int32).cuda(),
             gt=torch.from_numpy(cat([f[3] for f in frames], (-1, 8), np.float32)).cuda(),
             gstart=torch.tensor(np.concatenate([[0], np.cumsum(gs)]), dtype=torch.int32).cuda(),
             n=len(frames), max_k=max(ks + [0]), max_g=max(gs + [0]))
    return d


def _run(spec, d, n_settings=1, pred=None, valid=None, pred_stride=0, valid_stride=0):
    out = torch.zeros((n_settings, spec.n_counters), dtype=torch.int64, device="cuda")
    quality.launch(spec, d["pred"] if pred is None else pred, d["label"], d["pstart"], d["gt"], d["gstart"], d["n"],
                   d["max_k"], d["max_g"], out, n_settings=n_settings, pred_valid=d["valid"] if valid is None else valid,
                   pred_stride=pred_stride, valid_stride=valid_stride)
    return out.cpu().numpy()


def _old_counters(d, thresh=(0.3, 0.5, 0.7)):
    """fnp_recall_counters and fnp_precision_counters on the same inputs."""
    th = (C.c_float * len(thresh))(*thresh)
    rec = torch.zeros(5 + 5 * len(thresh), dtype=torch.int64, device="cuda")
    prec = torch.zeros(1 + len(thresh), dtype=torch.int64, device="cuda")
    for fn, out in ((_lib.lib.fnp_recall_counters, rec), (_lib.lib.fnp_precision_counters, prec)):
        _lib.check(fn(d["pred"].data_ptr(), d["valid"].data_ptr(), d["pstart"].data_ptr(), d["gt"].data_ptr(),
                      d["gstart"].data_ptr(), d["n"], max(d["max_k"], 1), d["max_g"], th, len(thresh), out.data_ptr(),
                      _lib.current_stream()), fn.__name__)
    return SeekerEngine.recall_dict(rec.cpu().numpy(), thresh), prec.cpu().numpy()


def _check_against_old(spec, d, counters):
    rec, prec = _old_counters(d, spec.thresh)
    assert quality.recall_dict(counters, spec) == rec
    p = quality.precision_dict(counters, spec)
    assert [p["proposals"]] + [p["hits_%s" % t] for t in spec.thresh] == prec.tolist()


# ------------------------------------------------------------------------------------------------- inputs
def _cfg1_frames():
    """cfg1 extraction results: the proposals of SeekerEngine.run with their labels, and the frames' GT."""
    cfg, frames = _inputs("cfg1", 4)
    res = SeekerEngine(synth.seeker_params(cfg), device="cuda:0").run(frames, with_recall=True)
    out = []
    for f, p in zip(frames, res["frames"]):
        g = np.asarray(f.gt_boxes, np.float32)
        out.append((p["pred_boxes"], p["pred_labels"], np.ones(len(p["pred_labels"]), bool),
                    np.concatenate([g[:, :7], g[:, -1:]], 1)))
    assert sum(len(o[1]) for o in out) > 10
    return out, res["recall"]


def _random_box(rng, n, spread=45.0):
    b = np.zeros((n, 7), np.float32)
    b[:, 0:2] = rng.uniform(-spread, spread, (n, 2))
    b[:, 2] = rng.uniform(-1, 1, n)
    b[:, 3:6] = rng.uniform(0.5, 5.0, (n, 3))
    b[:, 6] = rng.uniform(-np.pi, np.pi, n)
    return b


def _random_frames(seed=0, n=12):
    """Overlapping rotated boxes, proposals identical to GT boxes and to each other (ties), frames without
    proposals and without GT, trailing all-zero GT rows, invalid rows, centres exactly on a range edge."""
    rng = np.random.RandomState(seed)
    frames = []
    for f in range(n):
        G = 0 if f % 5 == 1 else int(rng.randint(1, 12))
        K = 0 if f % 5 == 2 else int(rng.randint(1, 30))
        gt = np.zeros((G, 8), np.float32)
        gt[:, :7] = _random_box(rng, G)
        gt[:, 7] = rng.randint(1, len(CLASSES) + 1, G)
        boxes = _random_box(rng, K)
        if G and K:
            j = rng.randint(0, G, K)
            near = rng.rand(K) < 0.7             # proposals near a GT box: jitter, or an exact copy
            boxes[near] = gt[j[near], :7] + rng.normal(0, 0.3, (near.sum(), 7)).astype(np.float32) * (rng.rand(near.sum(), 1) < 0.6)
        if K > 2:
            boxes[1] = boxes[0]                  # two identical proposals
        labels = rng.randint(1, len(CLASSES) + 1, K).astype(np.int32)
        if G and K:                              # some proposals share their GT's label
            same = rng.rand(K) < 0.5
            labels[same] = gt[rng.randint(0, G, K)[same], 7]
        if f == 3 and G and K:                   # centres exactly on the 20 m edge: (20, 0) and (12, 16)
            gt[0, :2] = (20.0, 0.0)
            boxes[0, :2] = (12.0, 16.0)
        if f % 4 == 0:                           # trailing all-zero GT rows (collate padding)
            gt = np.concatenate([gt, np.zeros((2, 8), np.float32)])
        valid = rng.rand(K) > 0.2
        frames.append((boxes, labels, valid, gt))
    return frames


# ------------------------------------------------------------------------------------------------- 1, 2
@pytest.mark.parametrize("spec", [SPEC, quality.QualitySpec(CLASSES, range_edges=(10, 20, 25, 30, 40, 45, 50),
                                                             thresh=(0.1, 0.3, 0.5, 0.7, 0.9, 1.0, 0.0, 0.55))])
def test_kernel_equals_restatement_on_random_boxes(spec):
    frames = _random_frames()
    d = _device(frames)
    got = _run(spec, d)[0]
    assert np.array_equal(got, restate(spec, frames))
    tab = quality.tables(got, spec)
    assert sum(tab[c]["all"]["gt"] for c in CLASSES) > 40
    assert sum(tab[c]["all"]["recall_label"][str(spec.thresh[0])] for c in CLASSES) > 0
    if spec is SPEC:
        _check_against_old(spec, d, got)


def test_threshold_tie_at_an_exact_iou():
    """A threshold equal to a pair's IoU bit for bit: not above it, so not counted; one ulp lower: counted.  The IoU
    of two identical boxes is the clipped polygon's area over the box area in fp32, not always exactly 1.0, so the
    tie is taken from the op-level IoU of the pair itself."""
    from findnpropagate_b200.pcdet_ops import iou3d_nms_utils
    box = np.array([[23.5, -7.25, 0.3, 4.1, 1.8, 1.6, 0.7]], np.float32)
    v = iou3d_nms_utils.boxes_iou3d_gpu(torch.from_numpy(box).cuda(), torch.from_numpy(box).cuda()).cpu().numpy()[0, 0]
    below = np.nextafter(v, np.float32(-1))
    spec = quality.QualitySpec(CLASSES, thresh=(float(v), float(below)))
    frames = [(box, np.array([2], np.int32), np.ones(1, bool), np.concatenate([box, [[2]]], 1).astype(np.float32))]
    got = _run(spec, _device(frames))[0]
    assert np.array_equal(got, restate(spec, frames))
    e = quality.tables(got, spec)["truck"]["20-30"]
    assert e["gt"] == 1 and e["proposals"] == 1
    for k in ("recall_any", "recall_label", "precision_any", "precision_label"):
        assert e[k] == {str(float(v)): 0, str(float(below)): 1}, k


def test_kernel_equals_restatement_on_cfg1_results():
    frames, recall = _cfg1_frames()
    d = _device(frames)
    got = _run(SPEC, d)[0]
    assert np.array_equal(got, restate(SPEC, frames))
    assert quality.recall_dict(got, SPEC) == recall
    _check_against_old(SPEC, d, got)


def test_range_bin_on_the_edge():
    frames = [(np.array([[12, 16, 0, 2, 2, 2, 0], [19.5, 0, 0, 2, 2, 2, 0]], np.float32), np.array([1, 1], np.int32),
               np.ones(2, bool), np.array([[20, 0, 0, 2, 2, 2, 0, 2]], np.float32))]
    tab = quality.tables(_run(SPEC, _device(frames))[0], SPEC)
    assert tab["truck"]["20-30"]["gt"] == 1 and tab["car"]["20-30"]["proposals"] == 1
    assert tab["car"]["0-20"]["proposals"] == 1


# ------------------------------------------------------------------------------------------------- 3
def test_many_settings_equal_single_calls():
    frames = _random_frames(seed=1, n=6)
    d = _device(frames)
    rng = np.random.RandomState(2)
    S, N = 300, d["pred"].shape[0]
    preds = d["pred"].unsqueeze(0).repeat(S, 1, 1)
    preds += torch.from_numpy(rng.normal(0, 0.2, (S, N, 7)).astype(np.float32)).cuda() * \
        torch.from_numpy((rng.rand(S, N, 1) < 0.5).astype(np.float32)).cuda()
    valid = torch.from_numpy(np.where(rng.rand(S, N) < 0.8, 0, -1).astype(np.int32)).cuda()
    whole = _run(SPEC, d, S, pred=preds, valid=valid, pred_stride=N, valid_stride=N)
    for s in range(S):
        one = _run(SPEC, d, 1, pred=preds[s].contiguous(), valid=valid[s].contiguous())
        assert np.array_equal(whole[s], one[0]), s
    assert len({w.tobytes() for w in whole}) > 100
    # stride 0: every setting reads the same rows, equal to the rows copied per setting
    shared = _run(SPEC, d, 20, valid=valid[:20].contiguous(), pred_stride=0, valid_stride=N)
    copied = _run(SPEC, d, 20, pred=d["pred"].unsqueeze(0).repeat(20, 1, 1).contiguous(), valid=valid[:20].contiguous(),
                  pred_stride=N, valid_stride=N)
    assert np.array_equal(shared, copied)


# ------------------------------------------------------------------------------------------------- 4
def _c_call(d, n_classes=10, edges=(20.0, 30.0, 40.0), thresh=(0.5,), max_k=None, max_g=None):
    e = (C.c_float * max(len(edges), 1))(*edges)
    t = (C.c_float * max(len(thresh), 1))(*thresh)
    out = torch.zeros(100000, dtype=torch.int64, device="cuda")
    return _lib.lib.fnp_quality_counters(d["pred"].data_ptr(), 0, None, 0, d["label"].data_ptr(), d["pstart"].data_ptr(),
                                         1, d["gt"].data_ptr(), d["gstart"].data_ptr(), d["n"],
                                         d["max_k"] if max_k is None else max_k, d["max_g"] if max_g is None else max_g,
                                         n_classes, e, len(edges), t, len(thresh), out.data_ptr(), _lib.current_stream())


def test_refusals():
    frames = _random_frames(seed=3, n=3)
    d = _device(frames)
    assert _c_call(d) == 0
    bad = dict(d, label=d["label"].clone())
    bad["label"][0] = 11
    with pytest.raises(ValueError, match="label"):
        _run(SPEC, bad)
    bad["label"][0] = 0
    with pytest.raises(ValueError, match="label"):
        _run(SPEC, bad)
    with pytest.raises(ValueError, match="edges"):
        quality.QualitySpec(CLASSES, range_edges=(20, 20))
    assert _c_call(d, edges=(20.0, 20.0)) == -1            # FNP_EINVAL
    assert _c_call(d, edges=(30.0, 20.0)) == -1 and _c_call(d, edges=(0.0,)) == -1
    with pytest.raises(ValueError, match="thresholds"):
        quality.QualitySpec(CLASSES, thresh=[0.1] * 9)
    assert _c_call(d, thresh=[0.1] * 9) == -1
    with pytest.raises(ValueError, match="bins"):
        quality.QualitySpec(CLASSES, range_edges=range(1, 9))
    assert _c_call(d, edges=[float(x) for x in range(1, 9)]) == -1
    assert _c_call(d, n_classes=33) == -1 and _c_call(d, n_classes=0) == -1
    with pytest.raises(ValueError, match="shared memory"):
        quality.launch(SPEC, d["pred"], d["label"], d["pstart"], d["gt"], d["gstart"], d["n"], 2000, 2000,
                       torch.zeros(SPEC.n_counters, dtype=torch.int64, device="cuda"))
    assert _c_call(d, max_k=2000, max_g=2000) == -1


# ------------------------------------------------------------------------------------------------- 5
def test_evaluate_settings_quality():
    cfg, frames = _inputs("cfg1", 4)
    base = synth.seeker_params(cfg)
    settings = [dict(s) for s in SELECT] + [dict(s, lq=0.05) for s in SELECT]
    groups = tune_params.group_settings(base, settings)
    assert len(groups) == 2
    checked = 0
    for g in groups:
        eng = SeekerEngine(g["params"], device="cuda:0")
        plan, pts, gt = eng.plan(frames), eng.upload_points(frames), eng.upload_gt(frames)
        plain = eng.evaluate_settings(plan, pts, gt, g["settings"])
        res = eng.evaluate_settings(plan, pts, gt, g["settings"], quality=SPEC)
        fcs = plan["frame_cand_start"]
        gts = [np.concatenate([np.asarray(f.gt_boxes, np.float32)[:, :7], np.asarray(f.gt_boxes, np.float32)[:, -1:]], 1)
               for f in frames]
        for a, b in zip(plain["settings"], res["settings"]):
            q = b.pop("quality")
            assert set(a) == set(b)
            for k in a:
                assert np.array_equal(a[k], b[k]) if isinstance(a[k], np.ndarray) else a[k] == b[k], k
            per_frame = [(b["cand_boxes"][fcs[i]:fcs[i + 1]], plan["cand_label"][fcs[i]:fcs[i + 1]],
                          b["cand_best"][fcs[i]:fcs[i + 1]] >= 0, gts[i]) for i in range(len(frames))]
            assert np.array_equal(q, restate(SPEC, per_frame))
            assert quality.recall_dict(q, SPEC) == b["recall"]
            assert quality.precision_dict(q, SPEC) == b["precision"]
            checked += b["proposals"]
        for k in ("cand_best", "cand_score2", "cand_boxes", "cand_count", "cand_npts"):
            assert np.array_equal(plain[k], res[k])
        assert plain.get("recall") == res.get("recall")
    assert checked > 20


# ------------------------------------------------------------------------------------------------- 6, 7
@pytest.fixture
def cfg1_tree(tmp_path, monkeypatch):
    frames = _frames("cfg1", 5)
    tools = _write_tree(tmp_path, frames)
    monkeypatch.chdir(tools)
    return tmp_path, frames


def _folder_frames(base, frames, nms_thresh=None):
    """What load_pseudos gives self-training, with the frames' GT from NuScenesFeed.gt_boxes."""
    from findnpropagate_b200 import extract_pseudo_labels as cli
    from findnpropagate_b200.pseudo_loader import load_pseudos
    feed = cli.build_feed(cli.load_config(HEAD))
    out = []
    for i, f in enumerate(frames):
        b, _ = load_pseudos(base / "out", f.frame_id, nms_thresh=nms_thresh)
        g = feed.gt_boxes(i)
        out.append((b[:, :7], b[:, 7].astype(np.int32), np.ones(len(b), bool), np.concatenate([g[:, :7], g[:, -1:]], 1)))
    return out


def test_command_on_an_extracted_folder(cfg1_tree, capsys):
    from findnpropagate_b200 import eval_pseudo_labels as ev
    from findnpropagate_b200 import extract_pseudo_labels as cli
    base, frames = cfg1_tree
    ext = cli.main(["--cfg_file", HEAD, "--folder", "../out", "--batch_frames", "2"])
    capsys.readouterr()
    lines = ev.main(["--cfg_file", HEAD, "--folder", "../out", "--nms_thresh", "0.1", "0.3", "--batch_frames", "2",
                     "--out", "../q.jsonl"])
    assert [json.loads(t) for t in open(base / "q.jsonl")] == lines
    assert [d["nms"] for d in lines] == ["none", 0.1, 0.3]
    assert lines[0]["recall"] == ext["recall"] and ext["recall"]["gt"] > 0
    assert all(d["frames"] == 5 and d["missing_files"] == 0 for d in lines)
    assert lines[0]["proposals"] >= lines[1]["proposals"] > 0
    for d, t in zip(lines, (None, 0.1, 0.3)):
        ref = restate(SPEC, _folder_frames(base, frames, t))
        assert d["classes"] == quality.tables(ref, SPEC), t
        assert d["recall"] == quality.recall_dict(ref, SPEC)
    # a deleted file: no proposals for that frame, its GT counted as not found
    os.remove(base / "out" / (frames[1].frame_id.replace(".", "_") + ".pth"))
    got = ev.main(["--cfg_file", HEAD, "--folder", "../out"])[0]
    assert got["missing_files"] == 1 and "missing files: 1" in capsys.readouterr().out
    ref = restate(SPEC, _folder_frames(base, frames))
    assert got["classes"] == quality.tables(ref, SPEC) and got["recall"]["gt"] == lines[0]["recall"]["gt"]
    assert got["recall"]["rcnn_0.3"] <= lines[0]["recall"]["rcnn_0.3"]
    # --every and the range edges
    got = ev.main(["--cfg_file", HEAD, "--folder", "../out", "--every", "2", "--range_edges", "25"])[0]
    assert got["frames"] == 3 and list(got["classes"]["car"]) == ["0-25", "25+", "all"]


def _table_sums(classes):
    tot = {"gt": 0}
    for c in classes.values():
        tot["gt"] += c["all"]["gt"]
        for t, v in c["all"]["recall_any"].items():
            tot["rcnn_%s" % t] = tot.get("rcnn_%s" % t, 0) + v
    return tot


def test_tune_params_breakdown(cfg1_tree, capsys):
    base, frames = cfg1_tree
    _write_yaml(str(base / "tools" / "grid.yaml"), GRID)
    plain = tune_params.main(["--cfg_file", HEAD, "--grid", "grid.yaml", "--batch_frames", "2"])
    broken = tune_params.main(["--cfg_file", HEAD, "--grid", "grid.yaml", "--batch_frames", "2", "--breakdown"])
    assert len(plain) == len(broken) == 8
    for a, b in zip(plain, broken):
        classes = b.pop("classes")
        assert a == b
        sums = _table_sums(classes)
        assert sums == {k: b["recall"][k] for k in sums}
        assert sum(c["all"]["proposals"] for c in classes.values()) == b["proposals"]
    assert all("classes" not in a for a in plain)
