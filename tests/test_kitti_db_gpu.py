"""The every-box crop and the KITTI databases on the GPU: crop_frames(every_box=True) against points_in_boxes_cpu plus
numpy (``pts[mask[i] > 0]``, centre subtracted in the boxes' precision) byte for byte, and against the
reference-compiled op where it was built; create_groundtruth_database_kitti against a serial restatement of
KittiDataset.create_groundtruth_database; create_kitti_pseudo_database against a serial restatement (load_pseudos +
the whole velodyne scan + the matrix crop), read back as DataBaseSampler reads it."""
import os
import pickle
import shutil

import numpy as np
import pytest
import torch

from findnpropagate_b200 import gt_database, kitti_feed, synth
from findnpropagate_b200 import create_kitti_pseudo_database as cli
from findnpropagate_b200.kitti_feed import Calibration
from findnpropagate_b200.pcdet_ops import roiaware_pool3d_utils as RP
from findnpropagate_b200.pseudo_loader import load_pseudos

from test_kitti_db_cpu import add_db_annos, write_kitti_pseudos
from test_kitti_feed_cpu import KITTI_DATA, KITTI_HEAD, write_kitti_tree

pytestmark = pytest.mark.gpu


def _mask(pts, boxes, ref_ops=None):
    """points_in_boxes_cpu's (G, N) matrix on the boxes cast to float32, checked against the reference-compiled op
    where it exists."""
    b32 = np.ascontiguousarray(np.asarray(boxes)[:, :7], np.float32)
    p3 = np.ascontiguousarray(pts[:, :3], np.float32)
    m = RP.points_in_boxes_cpu(p3, b32)
    if ref_ops is not None and b32.shape[0] and p3.shape[0]:
        want = torch.zeros((b32.shape[0], p3.shape[0]), dtype=torch.int32)
        ref_ops[0].points_in_boxes_cpu(torch.from_numpy(b32), torch.from_numpy(p3), want)
        assert np.array_equal(m, want.numpy())
    return m


def _matrix_crop(pts, boxes, ref_ops=None):
    """Per box: pts[mask[i] > 0], then [:, :3] -= boxes[i, :3] (numpy's in-place rule, in the boxes' dtype)."""
    m = _mask(pts, boxes, ref_ops)
    out = []
    for i in range(len(boxes)):
        e = pts[m[i] > 0]
        e[:, :3] -= boxes[i, :3]
        out.append(e)
    return out


def _overlap_frame(rng, C, n):
    """n points, most in a nest of 2..5 boxes around the same centres, some boxes empty."""
    centres = rng.uniform([-30, -30, -1.5], [30, 30, 0.5], (6, 3))
    boxes = []
    for ci, c in enumerate(centres):
        for k in range(2 + ci % 4):                       # nested and rotated: a point lies in 2 .. 5 of them
            d = np.array([4.0, 2.0, 1.6]) * (1 + 0.3 * k)
            boxes.append(np.r_[c + rng.normal(0, 0.2, 3), d, rng.uniform(-np.pi, np.pi)])
    boxes.append([80.0, 80.0, 0.0, 1.0, 1.0, 1.0, 0.3])   # no points
    boxes = np.array(boxes)
    near = centres[rng.integers(0, 6, n)] + rng.normal(0, 1.5, (n, 3))
    far = rng.uniform(-40, 40, (n, 3))
    xyz = np.where(rng.random((n, 1)) < 0.7, near, far)
    return np.c_[xyz, rng.uniform(0, 1, (n, C - 3))].astype(np.float32), boxes


def _face_frame(rng, C):
    """Rotated, separate boxes with points placed 1e-5 .. 1e-2 outside a face (inside by the CPU op's margin, outside
    by the GPU op's), and points a few ulp around the CPU margin."""
    n_box = 40
    boxes = np.c_[np.arange(n_box) % 8 * 12.0 - 40, np.arange(n_box) // 8 * 12.0 - 25, rng.uniform(-1, 0, n_box),
                  rng.uniform(1, 5, (n_box, 3)), rng.uniform(-np.pi, np.pi, n_box)]
    b = boxes.astype(np.float32).astype(np.float64)
    n = 4000
    k = rng.integers(0, n_box, n)
    eps = np.concatenate([10 ** rng.uniform(-5, -2, n // 2), 0.01 + rng.integers(-6, 7, n - n // 2) * 1e-7])
    sign, axis = rng.choice([-1.0, 1.0], n), rng.integers(0, 3, n)
    lx = np.where(axis == 0, sign * (b[k, 3] / 2 + eps), rng.uniform(-0.4, 0.4, n) * b[k, 3])
    ly = np.where(axis == 1, sign * (b[k, 4] / 2 + eps), rng.uniform(-0.4, 0.4, n) * b[k, 4])
    lz = np.where(axis == 2, sign * (b[k, 5] / 2 + eps), rng.uniform(-0.4, 0.4, n) * b[k, 5])
    ca, sa = np.cos(b[k, 6]), np.sin(b[k, 6])
    xyz = np.stack([b[k, 0] + lx * ca - ly * sa, b[k, 1] + lx * sa + ly * ca, b[k, 2] + lz], 1)
    return np.c_[xyz, rng.uniform(0, 1, (n, C - 3))].astype(np.float32), boxes


def _cases(C, seed=0):
    rng = np.random.default_rng(seed + C)
    frames = [_overlap_frame(rng, C, 3000), _overlap_frame(rng, C, 1023)]
    frames.append((rng.uniform(-20, 20, (1500, C)).astype(np.float32), np.zeros((0, 7))))          # no boxes
    frames.append((np.zeros((0, C), np.float32), _overlap_frame(rng, C, 10)[1]))                     # no points
    many = np.c_[rng.uniform(-30, 30, (1100, 2)), rng.uniform(-1, 0, 1100), rng.uniform(0.5, 4, (1100, 3)),
                 rng.uniform(-np.pi, np.pi, 1100)]                                                   # > 1024 boxes
    frames.append((np.c_[rng.uniform([-30, -30, -2], [30, 30, 1], (2049, 3)),
                         rng.uniform(0, 1, (2049, C - 3))].astype(np.float32), many))
    frames.append(_face_frame(rng, C))
    frames.append(_overlap_frame(rng, C, 1025))
    return frames


@pytest.mark.parametrize("C", [3, 4, 5])
@pytest.mark.parametrize("box_dtype", [np.float32, np.float64])
def test_every_box_crop_equals_the_matrix_crop(ref_ops, C, box_dtype):
    frames = _cases(C)
    pts_list = [f[0] for f in frames]
    boxes_list = [np.asarray(f[1], box_dtype) for f in frames]
    got = gt_database.crop_frames(pts_list, boxes_list, every_box=True)
    assert len(got) == len(frames)
    multi = 0
    for p, b, g in zip(pts_list, boxes_list, got):
        want = _matrix_crop(p, b, ref_ops)
        assert len(g) == len(want) == len(b)
        for i, (x, y) in enumerate(zip(g, want)):
            assert x.dtype == np.float32 and x.shape == y.shape, "box %d" % i
            assert x.tobytes() == y.tobytes(), "box %d" % i
        if len(b) and len(p):
            multi = max(multi, int(_mask(p, b).sum(0).max()))
    assert multi >= 4                                   # points really are in several boxes
    assert sum(len(x) == 0 for x in got[0]) >= 1        # and some boxes are empty
    # the face points separate the two predicates: the GPU op puts some of them in no box
    p, b = frames[5]
    cpu_in = _mask(p, b).any(0)
    gpu_idx = RP.points_in_boxes_gpu(torch.from_numpy(p[None, :, :3].copy()).cuda(),
                                     torch.from_numpy(np.asarray(b, np.float32)[None]).cuda()).cpu().numpy()[0]
    assert (cpu_in & (gpu_idx < 0)).sum() > 100
    # the default crop is unchanged by the option: first match only
    first = gt_database.crop_frames(pts_list[:1], boxes_list[:1])[0]
    idx = RP.points_in_boxes_gpu(torch.from_numpy(pts_list[0][None, :, :3].copy()).cuda(),
                                 torch.from_numpy(np.asarray(boxes_list[0], np.float32)[None]).cuda()).cpu().numpy()[0]
    assert sum(len(x) for x in first) == int((idx >= 0).sum())


def test_every_box_crop_is_deterministic_and_sized_exactly():
    frames = _cases(4, seed=7)
    pts = torch.from_numpy(np.concatenate([f[0] for f in frames])).cuda()
    box = np.concatenate([np.asarray(f[1], np.float64) for f in frames])
    rs = np.concatenate([[0], np.cumsum([f[0].shape[0] for f in frames])])
    bs = np.concatenate([[0], np.cumsum([len(f[1]) for f in frames])])
    args = (pts, rs, torch.from_numpy(box.astype(np.float32)).cuda(), torch.from_numpy(box[:, :3].copy()).cuda(), bs)
    a = [t.cpu().numpy() for t in gt_database.crop_points_in_boxes_all(*args)]
    b = [t.cpu().numpy() for t in gt_database.crop_points_in_boxes_all(*args)]
    assert all(x.tobytes() == y.tobytes() for x, y in zip(a, b))
    counts, starts, rows = a
    assert starts[0] == 0 and np.array_equal(np.diff(starts), counts) and rows.shape == (starts[-1], 4)
    assert starts[-1] > 1000


def test_crop_with_inconsistent_starts_writes_nothing():
    """row_start that does not end at n_points: every count 0, starts all 0 (checked on the device)."""
    from findnpropagate_b200 import _lib
    p, b = _overlap_frame(np.random.default_rng(1), 4, 2000)
    pts = torch.from_numpy(p).cuda()
    b32 = np.ascontiguousarray(b, np.float32)
    prep = torch.empty((len(b), 8))
    _lib.check(_lib.lib.fnp_host_prep_boxes_cpu(b32.ctypes.data, prep.data_ptr(), len(b)), "prep")
    prep = prep.cuda()
    rs, bs = np.array([0, 1999], np.int64), np.array([0, len(b)], np.int64)
    d = torch.from_numpy(np.concatenate([rs, bs])).cuda()
    ws_bytes = int(_lib.lib.fnp_crop_workspace_bytes(np.array([0, 2000], np.int64).ctypes.data, bs.ctypes.data, 1))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    counts = torch.full((len(b),), 7, dtype=torch.int32, device="cuda")
    starts = torch.full((len(b) + 1,), 7, dtype=torch.int64, device="cuda")
    rc = _lib.lib.fnp_crop_all_count(pts.data_ptr(), 4, d.data_ptr(), 2000, prep.data_ptr(), d[2:].data_ptr(), len(b),
                                     1, counts.data_ptr(), starts.data_ptr(), ws.data_ptr(), ws_bytes, None)
    assert rc == 0
    rows = torch.full((64, 4), 5.0, device="cuda")
    rc = _lib.lib.fnp_crop_all_scatter(pts.data_ptr(), 4, d.data_ptr(), 2000, prep.data_ptr(),
                                       torch.zeros((len(b), 3), dtype=torch.float64, device="cuda").data_ptr(),
                                       d[2:].data_ptr(), len(b), 1, starts.data_ptr(), rows.data_ptr(), 64,
                                       ws.data_ptr(), ws_bytes, None)
    assert rc == 0
    torch.cuda.synchronize()
    assert int(counts.abs().sum()) == 0 and int(starts.abs().sum()) == 0 and bool((rows == 5.0).all())


# --------------------------------------------------------------------------------------------------- GT database
N_FRAMES = 5


@pytest.fixture(scope="module")
def full_frames():
    return [synth.make_kitti_frame(i, with_gt=True, full_scan=True) for i in range(N_FRAMES)]


def _gt_db_restated(root, infos, used_classes):
    """KittiDataset.create_groundtruth_database, frame by frame, into memory: ({relative path: bytes}, db infos)."""
    files, db = {}, {}
    for info in infos:
        idx = info["point_cloud"]["lidar_idx"]
        points = np.fromfile(os.path.join(root, "training", "velodyne", idx + ".bin"), np.float32).reshape(-1, 4)
        annos = info["annos"]
        gt_boxes = annos["gt_boxes_lidar"]
        point_indices = RP.points_in_boxes_cpu(torch.from_numpy(points[:, 0:3]), torch.from_numpy(gt_boxes)).numpy()
        for i in range(gt_boxes.shape[0]):
            path = os.path.join("gt_database", "%s_%s_%d.bin" % (idx, annos["name"][i], i))
            gt_points = points[point_indices[i] > 0]
            gt_points[:, :3] -= gt_boxes[i, :3]
            files[path] = gt_points.tobytes()
            if used_classes is None or annos["name"][i] in used_classes:
                db.setdefault(annos["name"][i], []).append(
                    {"name": annos["name"][i], "path": path, "image_idx": idx, "gt_idx": i, "box3d_lidar": gt_boxes[i],
                     "num_points_in_gt": gt_points.shape[0], "difficulty": annos["difficulty"][i],
                     "bbox": annos["bbox"][i], "score": annos["score"][i]})
    return files, db


def _files(base, sub):
    d = os.path.join(base, sub)
    return {os.path.join(sub, f): open(os.path.join(d, f), "rb").read() for f in sorted(os.listdir(d))}


def _assert_infos_equal(got, want):
    assert list(got) == list(want)
    for name in want:
        assert len(got[name]) == len(want[name])
        for g, w in zip(got[name], want[name]):
            assert list(g) == list(w)
            for k in w:
                if isinstance(w[k], np.ndarray):
                    assert g[k].dtype == w[k].dtype and g[k].tobytes() == w[k].tobytes(), k
                else:
                    assert type(g[k]) is type(w[k]) and g[k] == w[k], k


@pytest.mark.parametrize("box_dtype", [np.float32, np.float64])
def test_gt_database_equals_the_serial_restatement(tmp_path, full_frames, box_dtype):
    root = str(tmp_path)
    synth.write_kitti_tree(root, full_frames)
    infos = add_db_annos(root)
    for info in infos:
        info["annos"]["gt_boxes_lidar"] = info["annos"]["gt_boxes_lidar"].astype(box_dtype)
    assert sum(len(i["annos"]["gt_boxes_lidar"]) for i in infos) > 20
    for used, batch in ((None, 1), (None, 16), (["Car", "Van", "Pedestrian"], 2)):
        want_files, want_db = _gt_db_restated(root, infos, used)
        got_db = gt_database.create_groundtruth_database_kitti(root, infos, used_classes=used, batch_frames=batch)
        with open(os.path.join(root, "kitti_dbinfos_train.pkl"), "rb") as f:
            pickled = pickle.load(f)
        assert _files(root, "gt_database") == want_files
        _assert_infos_equal(got_db, want_db)
        _assert_infos_equal(pickled, want_db)
        shutil.rmtree(os.path.join(root, "gt_database"))
    # another split: gt_database_<split>, kitti_dbinfos_<split>.pkl
    gt_database.create_groundtruth_database_kitti(root, infos[:2], split="val")
    assert os.path.isdir(os.path.join(root, "gt_database_val"))
    assert os.path.isfile(os.path.join(root, "kitti_dbinfos_val.pkl"))


# ------------------------------------------------------------------------------------------------------- command
@pytest.fixture
def cmd_tree(tmp_path, monkeypatch, full_frames):
    tools = write_kitti_tree(tmp_path, full_frames)
    write_kitti_pseudos(str(tmp_path / "pseudo"), full_frames)
    monkeypatch.chdir(tools)
    return tmp_path


def _cmd_restated(base, labels, nms_thresh):
    """Serial restatement: per frame with a velodyne file, load_pseudos, the whole scan, the matrix crop."""
    root = os.path.join(str(base), KITTI_DATA)
    with open(os.path.join(root, "kitti_infos_train.pkl"), "rb") as f:
        infos = pickle.load(f)
    names = list(synth.KITTI_CLASS_NAMES)
    files, db = {}, {}
    for info in infos:
        idx = info["point_cloud"]["lidar_idx"]
        velo = os.path.join(root, "training", "velodyne", idx + ".bin")
        if not os.path.exists(velo):
            continue
        boxes, scores = load_pseudos(str(base / "pseudo"), idx, labels, nms_thresh)
        if len(boxes) == 0:
            continue
        pts = np.fromfile(velo, np.float32).reshape(-1, 4)
        crops = _matrix_crop(pts, boxes[:, :7])
        cal = Calibration(os.path.join(root, "training", "calib", idx + ".txt"))
        cam = kitti_feed.boxes3d_lidar_to_kitti_camera(boxes[:, :7].copy(), cal)
        bbox = kitti_feed.boxes3d_kitti_camera_to_imageboxes(cam, cal, info["image"]["image_shape"])
        for j in range(len(boxes)):
            name = names[int(boxes[j, 7]) - 1]
            path = os.path.join("pseudo_database", "%s_%s_%d.bin" % (idx, name, j))
            files[path] = crops[j].tobytes()
            db.setdefault(name, []).append(
                {"name": name, "path": path, "image_idx": idx, "gt_idx": j, "box3d_lidar": boxes[j, :7],
                 "num_points_in_gt": crops[j].shape[0], "difficulty": 0, "bbox": bbox[j].astype(np.float32),
                 "score": float(scores[j])})
    return files, db


def _run(base, extra):
    root = os.path.join(str(base), KITTI_DATA)
    got = cli.main(["--cfg_file", KITTI_HEAD, "--folder", "../pseudo", "--batch_frames", "2", "--workers", "3"] + extra)
    files = _files(root, "pseudo_database")
    with open(os.path.join(root, "kitti_pseudo_dbinfos_train.pkl"), "rb") as f:
        db = pickle.load(f)
    return got, files, db


def _clean(base):
    root = os.path.join(str(base), KITTI_DATA)
    shutil.rmtree(os.path.join(root, "pseudo_database"))
    os.remove(os.path.join(root, "kitti_pseudo_dbinfos_train.pkl"))


def test_command_equals_the_serial_restatement(cmd_tree, capsys):
    base = cmd_tree
    root = base / KITTI_DATA
    os.remove(root / "training" / "velodyne" / "000002.bin")
    os.remove(base / "pseudo" / "000004.pth")
    for labels, nms in ((None, None), ([1, 2, 5], None), (None, 0.3), ([1, 3, 4, 6], 0.1)):
        extra = (["--labels"] + [str(c) for c in labels] if labels else []) + (["--nms_thresh", str(nms)] if nms else [])
        got, files, db = _run(base, extra)
        out = capsys.readouterr().out
        assert "skipped frame 000002" in out
        assert got["frames"] == N_FRAMES - 1 and got["missing"] == 1 and got["skipped"] == 1
        assert got["skipped_frames"] == [("000002", "LiDAR file missing")]
        want_files, want_db = _cmd_restated(base, labels, nms)
        assert files == want_files and len(files) > 10
        _assert_infos_equal(db, want_db)
        assert got["boxes"] == {k: len(v) for k, v in want_db.items()}
        # read back as DataBaseSampler reads it
        for infos in db.values():
            for info in infos:
                pts = np.fromfile(str(root / info["path"]), np.float32).reshape(-1, 4)
                assert pts.shape[0] == info["num_points_in_gt"]
                assert info["difficulty"] == 0 and info["bbox"].shape == (4,) and isinstance(info["score"], float)
        assert sum(i["num_points_in_gt"] for v in db.values() for i in v) > 100
        _clean(base)
    # two runs write the same bytes
    a = _run(base, ["--nms_thresh", "0.2"])
    _clean(base)
    b = _run(base, ["--nms_thresh", "0.2"])
    assert a[1] == b[1]
    assert pickle.dumps(a[2]) == pickle.dumps(b[2])
