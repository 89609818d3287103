"""fnp_crop_points_in_boxes against points_in_boxes_gpu plus numpy (rows[box_of_pt == i], centre subtracted in
float64) byte for byte; the GT database on float64 infos; the create_pseudo_database command against a serial
restatement (load_pseudos + lidar_with_sweeps(RandomState(seed)) + the GT database's loop)."""
import os
import pickle
from pathlib import Path

import numpy as np
import pytest
import torch

from findnpropagate_b200 import gt_database, synth
from findnpropagate_b200 import create_pseudo_database as cli
from findnpropagate_b200.pcdet_ops import roiaware_pool3d_utils

from test_extract_cli import HEAD, INFOS, NUSC, _frames
from test_pseudo_db_cpu import write_pseudos, write_sweep_tree

pytestmark = pytest.mark.gpu


def _box_of_pt(pts, boxes):
    if boxes.shape[0] == 0 or pts.shape[0] == 0:
        return np.full(pts.shape[0], -1, np.int64)
    out = roiaware_pool3d_utils.points_in_boxes_gpu(
        torch.from_numpy(np.ascontiguousarray(pts[None, :, :3], np.float32)).cuda(),
        torch.from_numpy(np.ascontiguousarray(boxes[None, :, :7], np.float32)).cuda())
    return out.long().squeeze(0).cpu().numpy()


def _expected(pts, boxes, centres):
    """Per box: pts[box_of_pt == i] with xyz minus the float64 centre, rounded to float32 (numpy's in-place rule)."""
    idx = _box_of_pt(pts, boxes)
    out = []
    for i in range(boxes.shape[0]):
        e = pts[idx == i].copy()
        e[:, :3] -= centres[i]
        out.append(e)
    return out


def _check(frames):
    """frames: list of (points (N,5) f32, boxes (G,7) f32, centres (G,3) f64): one crop call against the restatement,
    and a second call for the same bytes."""
    pts = np.concatenate([f[0] for f in frames]).astype(np.float32).reshape(-1, 5)
    boxes = np.concatenate([f[1] for f in frames]).astype(np.float32).reshape(-1, 7)
    cen = np.concatenate([f[2] for f in frames]).astype(np.float64).reshape(-1, 3)
    rs = np.concatenate([[0], np.cumsum([f[0].shape[0] for f in frames])])
    bs = np.concatenate([[0], np.cumsum([f[1].shape[0] for f in frames])])
    args = (torch.from_numpy(pts).cuda(), rs, torch.from_numpy(boxes).cuda(), torch.from_numpy(cen).cuda(), bs)
    counts, starts, rows = gt_database.crop_points_in_boxes(*args)
    counts, starts, rows = counts.cpu().numpy(), starts.cpu().numpy(), rows.cpu().numpy()
    assert starts[0] == 0 and np.array_equal(np.diff(starts), counts)
    g = 0
    for f in frames:
        for e in _expected(*f):
            assert counts[g] == e.shape[0]
            assert rows[starts[g]:starts[g + 1]].tobytes() == e.tobytes(), "box %d" % g
            g += 1
    again = [t.cpu().numpy() for t in gt_database.crop_points_in_boxes(*args)]
    total = starts[-1]
    assert np.array_equal(again[0], counts) and again[2][:total].tobytes() == rows[:total].tobytes()
    return counts


def _cloud(rng, n, spread=40.0):
    p = np.zeros((n, 5), np.float32)
    p[:, :2] = rng.uniform(-spread, spread, (n, 2))
    p[:, 2] = rng.uniform(-2, 2, n)
    p[:, 3] = rng.uniform(0, 255, n)
    p[:, 4] = rng.choice([0.0, 0.05, 0.1], n)
    return p


def _boxes(rng, g, spread=40.0):
    b = np.concatenate([rng.uniform(-spread, spread, (g, 2)), rng.uniform(-1, 1, (g, 1)), rng.uniform(1, 8, (g, 2)),
                        rng.uniform(1, 3, (g, 1)), rng.uniform(-np.pi, np.pi, (g, 1))], 1).astype(np.float32)
    return b, b[:, :3].astype(np.float64)


def test_crop_overlapping_empty_and_size_mixed_frames():
    rng = np.random.default_rng(0)
    frames = []
    # overlapping boxes: big boxes around the same centres, first match wins
    b, c = _boxes(rng, 30, 10.0)
    b = np.concatenate([b, b * [1, 1, 1, 2, 2, 2, 1]]).astype(np.float32)
    frames.append((_cloud(rng, 20000, 12.0), b, b[:, :3].astype(np.float64)))
    frames.append((_cloud(rng, 500), np.zeros((0, 7), np.float32), np.zeros((0, 3))))      # no boxes
    b, c = _boxes(rng, 5)
    frames.append((np.zeros((0, 5), np.float32), b, c))                                     # no points
    b, c = _boxes(rng, 8)
    b[:, :2] += 500.0                                                                       # boxes with no points
    frames.append((_cloud(rng, 3000), b, b[:, :3].astype(np.float64)))
    b, c = _boxes(rng, 40, 50.0)
    frames.append((_cloud(rng, 310000, 50.0), b, c))                                        # a 10-sweep-size frame
    b, c = _boxes(rng, 3, 3.0)
    frames.append((_cloud(rng, 7, 3.0), b, c))                                              # a tiny one
    counts = _check(frames)
    assert (counts == 0).sum() >= 13 and counts.max() > 1000


def test_crop_points_on_box_faces():
    rng = np.random.default_rng(1)
    b = np.array([[1.0, 2.0, 0.5, 4.0, 2.0, 1.5, 0.0], [10.0, -3.0, 0.0, 3.0, 3.0, 2.0, 0.7],
                  [-5.0, 5.0, 0.0, 1.0, 1.0, 1.0, np.pi / 2]], np.float32)
    pts = []
    for box in b:
        c, s = np.cos(box[6]), np.sin(box[6])
        for fx, fy, fz in [(0.5, 0, 0), (-0.5, 0, 0), (0, 0.5, 0), (0, -0.5, 0), (0, 0, 0.5), (0, 0, -0.5),
                           (0.5, 0.5, 0.5), (0.4999999, 0, 0), (0.5000001, 0, 0)]:
            lx, ly = fx * box[3], fy * box[4]
            pts.append([box[0] + lx * c - ly * s, box[1] + lx * s + ly * c, box[2] + fz * box[5], 1, 0])
    pts = np.array(pts, np.float32)
    pts = np.concatenate([pts, pts + np.float32(1e-6), _cloud(rng, 2000, 12.0)]).astype(np.float32)
    _check([(pts, b, b[:, :3].astype(np.float64))])


def test_crop_more_than_1024_boxes_in_a_frame():
    rng = np.random.default_rng(2)
    xs, ys = np.meshgrid(np.arange(40) * 2.0 - 40, np.arange(30) * 2.0 - 30)
    g = xs.size
    assert g > 1024
    b = np.stack([xs.ravel(), ys.ravel(), np.zeros(g), np.full(g, 1.5), np.full(g, 1.5), np.full(g, 2.0),
                  rng.uniform(-3, 3, g)], 1).astype(np.float32)
    counts = _check([(_cloud(rng, 60000, 42.0), b, b[:, :3].astype(np.float64)),
                     (_cloud(rng, 1000), b[:100], b[:100, :3].astype(np.float64))])
    assert (counts[:g] > 0).sum() > 1000


def test_crop_float64_centres_round_once():
    """Centres off the float32 grid: float32(float64(p) - c) is kept, which differs from p - float32(c)."""
    rng = np.random.default_rng(3)
    b, _ = _boxes(rng, 20, 20.0)
    c = b[:, :3].astype(np.float64) + rng.uniform(-1e-3, 1e-3, (20, 3)) + 1.2345678901234e-7
    pts = _cloud(rng, 50000, 22.0)
    _check([(pts, b, c)])
    idx = _box_of_pt(pts, b)
    m = idx >= 0
    one = (pts[m, :3] - c[idx[m]]).astype(np.float32)
    two = pts[m, :3] - c[idx[m]].astype(np.float32)
    assert (one != two).any()


def test_gt_database_on_float64_infos(tmp_path):
    """create_groundtruth_database on infos whose gt_boxes are float64 (as nuScenes' are), with centres off the float32
    grid: the .bin files are the numpy procedure's, byte for byte."""
    cfg = synth.SynthConfig("gtdb", 16, 720, 1, 8, 4, 6, 1)
    sf = [synth.make_frame(i, cfg) for i in range(4)]
    infos = synth.write_nuscenes_tree(str(tmp_path / "nusc"), sf)
    rng = np.random.default_rng(4)
    for info in infos:
        g = info["gt_boxes"].astype(np.float64)
        g[:, :3] += rng.uniform(-1e-3, 1e-3, (g.shape[0], 3)) + 3.3e-8
        info["gt_boxes"] = g
    got = gt_database.create_groundtruth_database(tmp_path / "nusc", infos, max_sweeps=1, batch_frames=3)
    db = tmp_path / "nusc" / "gt_database_1sweeps_withvelo"
    differ = False
    for idx, info in enumerate(infos):
        pts = np.fromfile(str(tmp_path / "nusc" / info["lidar_path"]), np.float32).reshape(-1, 5)[:, :4]
        pts = np.concatenate([pts, np.zeros((pts.shape[0], 1), np.float32)], 1)
        g = info["gt_boxes"]
        box_of_pt = _box_of_pt(pts, g[:, :7].astype(np.float32))
        for i in range(g.shape[0]):
            e = pts[box_of_pt == i]
            differ |= bool(((e[:, :3] - g[i, :3]).astype(np.float32) != e[:, :3] - g[i, :3].astype(np.float32)).any())
            e[:, :3] -= g[i, :3]
            path = db / ("%d_%s_%d.bin" % (idx, info["gt_names"][i], i))
            assert path.read_bytes() == e.tobytes()
    assert differ
    assert sum(len(v) for v in got.values()) == sum(i["gt_boxes"].shape[0] for i in infos)
    assert all(d["box3d_lidar"].dtype == np.float64 for v in got.values() for d in v)


# ---------------------------------------------------------------------------------------------------- the command
def restate(base, folder, max_sweeps, seed=0, labels=None, nms_thresh=None):
    """The database the command writes, serially: {relative path: bytes} and {class: [info]}."""
    from findnpropagate_b200.nuscenes_feed import lidar_with_sweeps
    from findnpropagate_b200.pseudo_loader import load_pseudos, pseudo_path
    root = base / NUSC
    with open(root / INFOS, "rb") as f:
        infos = pickle.load(f)
    rng = np.random.RandomState(seed)
    files, dbinfos, missing, skipped = {}, {}, 0, 0
    for idx, info in enumerate(infos):
        if not (root / info["lidar_path"]).is_file() or (
                max_sweeps > 1 and not all((root / s["lidar_path"]).is_file() for s in info["sweeps"])):
            rng.choice(len(info["sweeps"]), max_sweeps - 1, replace=False)
            skipped += 1
            continue
        fid = Path(info["lidar_path"]).stem
        missing += not os.path.exists(pseudo_path(folder, fid))
        boxes, scores = load_pseudos(folder, fid, labels=labels, nms_thresh=nms_thresh)
        pts = lidar_with_sweeps(root, info, max_sweeps, rng)
        box_of_pt = _box_of_pt(pts, boxes[:, :7])
        for i in range(boxes.shape[0]):
            name = synth.CLASS_NAMES[int(boxes[i, 7]) - 1]
            rel = "pseudo_database_%dsweeps_withvelo/%d_%s_%d.bin" % (max_sweeps, idx, name, i)
            e = pts[box_of_pt == i]
            e[:, :3] -= boxes[i, :3]
            files[rel] = e.tobytes()
            box = np.zeros(info["gt_boxes"].shape[1], info["gt_boxes"].dtype)
            box[:7] = boxes[i, :7]
            dbinfos.setdefault(name, []).append(dict(name=name, path=rel, image_idx=idx, gt_idx=i, box3d_lidar=box,
                                                     num_points_in_gt=e.shape[0], score=float(scores[i])))
    return files, dbinfos, missing, skipped


def _compare(base, sweeps, want, result):
    files, dbinfos, missing, skipped = want
    root = base / NUSC
    db, pkl = cli.output_paths(root, sweeps)
    assert sorted(str(p.relative_to(root)) for p in db.iterdir()) == sorted(files)
    for rel, data in files.items():
        assert (root / rel).read_bytes() == data, rel
    with open(pkl, "rb") as f:
        got = pickle.load(f)
    assert list(got) == list(dbinfos)
    for name in dbinfos:
        assert len(got[name]) == len(dbinfos[name])
        for g, w in zip(got[name], dbinfos[name]):
            assert sorted(g) == sorted(w)
            assert g["box3d_lidar"].dtype == w["box3d_lidar"].dtype
            assert g["box3d_lidar"].tobytes() == w["box3d_lidar"].tobytes()
            assert all(g[k] == w[k] for k in w if k != "box3d_lidar")
            # DataBaseSampler's read-back: the path relative to the root, 5 floats per point, the box's width
            pts = np.fromfile(str(root / g["path"]), np.float32).reshape(-1, 5)
            assert pts.shape[0] == g["num_points_in_gt"] and g["box3d_lidar"].shape[0] == 9
    assert result["missing"] == missing and result["skipped"] == skipped
    assert result["boxes"] == {n: len(v) for n, v in dbinfos.items()}


@pytest.mark.parametrize("opts", [dict(), dict(labels=[1, 9]), dict(nms_thresh=0.1), dict(labels=[1], nms_thresh=0.2)])
def test_command_matches_the_serial_restatement(tmp_path, monkeypatch, opts):
    frames = _frames("tiny", 5)
    tools = write_sweep_tree(tmp_path, frames, n_sweeps=9)
    folder = tmp_path / "pseudo"
    write_pseudos(str(folder), frames)
    os.remove(folder / ("%s.pth" % frames[1].frame_id.replace(".", "_")))         # a missing .pth
    os.remove(tmp_path / NUSC / "samples" / "LIDAR_TOP" / ("%s.bin" % frames[3].frame_id))   # a missing LiDAR file
    monkeypatch.chdir(tools)
    argv = ["--cfg_file", HEAD, "--folder", str(folder), "--seed", "7", "--batch_frames", "2"]
    if "labels" in opts:
        argv += ["--labels"] + [str(x) for x in opts["labels"]]
    if "nms_thresh" in opts:
        argv += ["--nms_thresh", str(opts["nms_thresh"])]
    res = cli.main(argv + ["--set", "DATA_CONFIG.MAX_SWEEPS", "10"])
    want = restate(tmp_path, folder, 10, seed=7, **opts)
    assert want[2] == 1 and want[3] == 1 and sum(len(v) for v in want[1].values()) > (0 if "labels" in opts else 20)
    _compare(tmp_path, 10, want, res)
    # the 1-sweep database of the same folder is written beside the 10-sweep one
    res1 = cli.main(argv)
    _compare(tmp_path, 1, restate(tmp_path, folder, 1, seed=7, **opts), res1)
