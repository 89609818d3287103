"""python -m findnpropagate_b200.create_kitti_pseudo_database on the host: --help, the output names, every refusal
(nothing is written), the argument checks of the every-box crop (the C entries without a device, and
gt_database.crop_points_in_boxes_all), and the image-box helpers of kitti_feed against a float64 restatement.

``add_db_annos`` gives the synthetic KITTI tree what real info files carry for the GT database (``gt_boxes_lidar``,
``difficulty``, ``bbox``, ``score``); the GPU tests and tools/kitti_db_bench.py use it too."""
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest
import torch
import yaml

from findnpropagate_b200 import _lib, extract, gt_database, kitti_feed
from findnpropagate_b200 import create_kitti_pseudo_database as cli
from findnpropagate_b200.kitti_feed import Calibration

from test_extract_cli import ROOT
from test_kitti_feed_cpu import KITTI_DATA, KITTI_HEAD, _kitti_cfg, _kitti_frames, _snapshot, write_kitti_tree
from test_pseudo_db_cpu import _crop_args

N_CLASSES = 7


def add_db_annos(root, seed=0, split="training"):
    """Add to every info of ``root/kitti_infos_train.pkl`` the annotations KittiDataset.get_infos writes for the GT
    database: ``gt_boxes_lidar`` (the non-DontCare rows, converted as KittiFeed converts them), and ``difficulty``,
    ``bbox`` and ``score`` with one row per annotation, DontCare included.  Returns the infos."""
    path = os.path.join(str(root), "kitti_infos_train.pkl")
    with open(path, "rb") as f:
        infos = pickle.load(f)
    rng = np.random.default_rng(seed)
    for info in infos:
        annos = info["annos"]
        n = len(annos["name"])
        keep = annos["name"] != "DontCare"
        cal = Calibration(os.path.join(str(root), split, "calib", "%s.txt" % info["point_cloud"]["lidar_idx"]))
        cam = np.concatenate([annos["location"][keep], annos["dimensions"][keep],
                              annos["rotation_y"][keep][:, None]], 1).astype(np.float32)
        annos["gt_boxes_lidar"] = kitti_feed.boxes3d_kitti_camera_to_lidar(cam, cal)
        annos["difficulty"] = np.where(keep, rng.integers(0, 3, n), -1).astype(np.int32)
        annos["bbox"] = np.sort(rng.uniform(0, 1200, (n, 4)), 1).astype(np.float32)
        annos["score"] = np.round(rng.uniform(-1, 1, n), 2)
    with open(path, "wb") as f:
        pickle.dump(infos, f)
    return infos


def write_kitti_pseudos(folder, frames, seed=0, extra=None):
    """One .pth per frame ``%06d``: each GT box, a jittered copy (overlapping it), and random boxes, tied scores,
    labels 1..7; ``extra`` {frame index: (boxes, scores, labels)} replaces a frame's content."""
    os.makedirs(folder, exist_ok=True)
    rng = np.random.default_rng(seed)
    for k, fr in enumerate(frames):
        if extra and k in extra:
            b, s, l = extra[k]
        else:
            gt = np.asarray(fr[5], np.float32)
            jit = gt[:, :7] + rng.normal(0, 0.1, (gt.shape[0], 7)).astype(np.float32) * [1, 1, 0.2, 0.1, 0.1, 0.1, 0.1]
            rnd = np.concatenate([rng.uniform(5, 40, (4, 1)), rng.uniform(-15, 15, (4, 1)), rng.uniform(-1.5, 0, (4, 1)),
                                  rng.uniform(0.5, 5, (4, 3)), rng.uniform(-3, 3, (4, 1))], 1)
            b = np.concatenate([gt[:, :7], jit, rnd]).astype(np.float32)
            s = np.round(rng.uniform(0, 1, b.shape[0]), 1).astype(np.float32)
            l = rng.integers(1, N_CLASSES + 1, b.shape[0]).astype(np.int32)
        extract.save_frame(str(folder), "%06d" % k, dict(pred_boxes=b, pred_scores=s, pred_labels=l))


@pytest.fixture
def db_tree(tmp_path, monkeypatch):
    frames = _kitti_frames(3)
    tools = write_kitti_tree(tmp_path, frames)
    add_db_annos(tmp_path / KITTI_DATA)
    write_kitti_pseudos(str(tmp_path / "pseudo"), frames)
    monkeypatch.chdir(tools)
    return tmp_path


def test_help_runs_without_a_gpu():
    r = subprocess.run([sys.executable, "-m", "findnpropagate_b200.create_kitti_pseudo_database", "--help"], cwd=ROOT,
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    for flag in ("--cfg_file", "--folder", "--labels", "--nms_thresh", "--batch_frames", "--workers", "--set"):
        assert flag in r.stdout


def test_output_names(tmp_path):
    assert cli.output_paths(tmp_path, "train") == (tmp_path / "pseudo_database",
                                                   tmp_path / "kitti_pseudo_dbinfos_train.pkl")
    assert cli.output_paths(tmp_path, "val") == (tmp_path / "pseudo_database_val",
                                                 tmp_path / "kitti_pseudo_dbinfos_val.pkl")


def _refused(base, argv, capsys, match):
    before = _snapshot(base)
    with pytest.raises(SystemExit) as e:
        cli.main(argv)
    assert e.value.code == 1
    assert match in capsys.readouterr().err
    assert _snapshot(base) == before


ARGS = ["--cfg_file", KITTI_HEAD, "--folder", "../pseudo"]


def test_refusals_write_nothing(db_tree, capsys, monkeypatch):
    _refused(db_tree, ["--cfg_file", KITTI_HEAD, "--folder", "../nowhere"], capsys, "../nowhere does not exist")
    for bad in (["0"], ["3", "8"]):
        _refused(db_tree, ARGS + ["--labels"] + bad, capsys, "outside the classes")
    for bad in (["--batch_frames", "0"], ["--workers", "0"]):
        _refused(db_tree, ARGS + bad, capsys, "must be at least 1")
    _refused(db_tree, ARGS + ["--set", "DATA_CONFIG.NOPE", "1"], capsys, "DATA_CONFIG.NOPE")
    monkeypatch.setenv("WORLD_SIZE", "2")
    _refused(db_tree, ARGS, capsys, "one process")
    monkeypatch.delenv("WORLD_SIZE")


def test_a_nuscenes_config_is_refused(db_tree, capsys):
    cfg = _kitti_cfg()
    cfg["DATA_CONFIG"]["DATASET"] = "NuScenesDataset"
    cfg["MODEL"]["DENSE_HEAD"]["NAME"] = "FrustumProposerOG"
    with open("cfgs/nusc.yaml", "w") as f:
        yaml.safe_dump(cfg, f)
    _refused(db_tree, ["--cfg_file", "cfgs/nusc.yaml", "--folder", "../pseudo"], capsys, "create_pseudo_database")


@pytest.mark.parametrize("split", ["train", "val"])
@pytest.mark.parametrize("which", [0, 1])
def test_existing_output_is_refused(db_tree, capsys, which, split):
    target = cli.output_paths(db_tree / KITTI_DATA, split)[which]
    (target.mkdir() if which == 0 else target.write_bytes(b"x"))
    _refused(db_tree, ARGS + ["--set", "DATA_CONFIG.DATA_SPLIT.train", split], capsys, "already exists")
    assert not cli.output_paths(db_tree / KITTI_DATA, split)[1 - which].exists()


def test_bad_label_in_a_file_names_the_frame(db_tree, capsys):
    b = np.asarray(_kitti_frames(3)[1][5], np.float32)[:2, :7]
    write_kitti_pseudos(str(db_tree / "pseudo"), _kitti_frames(3),
                        extra={1: (b, np.ones(2, np.float32), np.array([3, 8], np.int32))})
    _refused(db_tree, ARGS, capsys, "frame 000001: label 8")


def test_frame_over_the_nms_limit_is_refused(db_tree, capsys):
    n = _lib.SEG_NMS_MAX + 1
    b = np.tile(np.array([[10, 0, -1, 2, 2, 1.5, 0]], np.float32), (n, 1))
    write_kitti_pseudos(str(db_tree / "pseudo"), _kitti_frames(3),
                        extra={2: (b, np.ones(n, np.float32), np.ones(n, np.int32))})
    _refused(db_tree, ARGS + ["--nms_thresh", "0.1"], capsys, "frame 000002: %d boxes" % n)


# ------------------------------------------------------------------------------------------------ the crop's checks
def _entry_args(**kw):
    """Arguments of fnp_crop_all_count / fnp_crop_all_scatter that pass every check: fake, aligned device addresses
    (nothing is launched when a check fails, so they are never dereferenced)."""
    a = dict(pts=0x1000, n_cols=4, row_start=0x2000, n_points=2048, box_prep=0x3000, centres=0x4000,
             box_start=0x5000, n_boxes=3, n_frames=2, counts=0x6000, starts=0x7000, rows=0x8000, rows_cap=10,
             ws=0x10000, ws_bytes=1 << 20)
    a.update(kw)
    return a


def _count(a):
    return _lib.lib.fnp_crop_all_count(a["pts"], a["n_cols"], a["row_start"], a["n_points"], a["box_prep"],
                                       a["box_start"], a["n_boxes"], a["n_frames"], a["counts"], a["starts"], a["ws"],
                                       a["ws_bytes"], None)


def _scatter(a):
    return _lib.lib.fnp_crop_all_scatter(a["pts"], a["n_cols"], a["row_start"], a["n_points"], a["box_prep"],
                                         a["centres"], a["box_start"], a["n_boxes"], a["n_frames"], a["starts"],
                                         a["rows"], a["rows_cap"], a["ws"], a["ws_bytes"], None)


EINVAL, EWORKSPACE = -1, -2


@pytest.mark.parametrize("entry", [_count, _scatter])
@pytest.mark.parametrize("change, rc", [
    (dict(n_cols=2), EINVAL), (dict(n_points=-1), EINVAL), (dict(n_boxes=-1), EINVAL), (dict(n_frames=-1), EINVAL),
    (dict(n_frames=0), EINVAL), (dict(pts=None), EINVAL), (dict(row_start=None), EINVAL),
    (dict(box_start=None), EINVAL), (dict(box_prep=None), EINVAL), (dict(starts=None), EINVAL),
    (dict(ws=None), EINVAL), (dict(ws=0x10008), EINVAL), (dict(ws_bytes=64), EWORKSPACE),
    (dict(n_points=1 << 20, ws_bytes=(1 << 22) + 16), EWORKSPACE),
])
def test_crop_all_entries_refuse_bad_arguments(entry, change, rc):
    assert entry(_entry_args(**change)) == rc


def test_crop_all_entry_specific_refusals():
    assert _count(_entry_args(counts=None)) == EINVAL
    assert _scatter(_entry_args(centres=None)) == EINVAL
    assert _scatter(_entry_args(rows_cap=-1)) == EINVAL
    assert _scatter(_entry_args(rows=None)) == EINVAL


@pytest.mark.parametrize("change, match", [
    (dict(points=np.zeros((10, 5), np.float32)), "points must be a tensor"),
    (dict(points=torch.zeros((10, 5), dtype=torch.float64)), "points must be a contiguous"),
    (dict(points=torch.zeros((10, 2))), "points must be a contiguous"),
    (dict(points=torch.zeros((5, 10)).t()), "points must be a contiguous"),
    (dict(boxes=torch.zeros((2, 9))), "boxes must be a contiguous"),
    (dict(centres=torch.zeros((2, 3))), "centres must be a contiguous"),
    (dict(centres=torch.zeros((3, 3), dtype=torch.float64)), "differ in length"),
    (dict(row_start=np.array([0, 4, 9])), "row_start must rise from 0 to 10"),
    (dict(row_start=np.array([0, 6, 4, 10])), "row_start must rise"),
    (dict(row_start=np.array([0.0, 10.0])), "row_start must be a 1-D integer array"),
    (dict(box_start=np.array([1, 2])), "box_start must rise from 0 to 2"),
    (dict(box_start=np.array([0, 2])), "differ in length"),
    (dict(), "one CUDA device"),
])
def test_crop_all_launcher_refusals(change, match):
    kw = _crop_args()
    kw.update(change)
    with pytest.raises(ValueError, match=match):
        gt_database.crop_points_in_boxes_all(**kw)


# ------------------------------------------------------------------------------------------------------ image boxes
def _image_boxes_f64(boxes, cal, shape):
    """OpenPCDet's procedure in float64: the box's bottom centre to the rectified camera frame, its eight corners there
    (l = dx along x, w = dy along z, h = dz up along -y, rotated by ry = -heading - pi/2 about y), projected with P2,
    min / max, then clipped."""
    V2C = np.vstack([cal.V2C.astype(np.float64), [0, 0, 0, 1]])
    R0 = cal.R0.astype(np.float64)
    P2 = cal.P2.astype(np.float64)
    out = []
    for b in np.asarray(boxes, np.float64):
        x, y, z, dx, dy, dz, h = b[:7]
        loc = (V2C @ [x, y, z - dz / 2, 1])[:3] @ R0.T
        ry = -h - np.pi / 2
        cx = np.array([1, 1, -1, -1, 1, 1, -1, -1]) * dx / 2
        cz = np.array([1, -1, -1, 1, 1, -1, -1, 1]) * dy / 2
        cy = np.array([0, 0, 0, 0, -1, -1, -1, -1]) * dz
        rect = np.stack([cx * np.cos(ry) + cz * np.sin(ry), cy, -cx * np.sin(ry) + cz * np.cos(ry)], 1) + loc
        img = np.c_[rect, np.ones(8)] @ P2.T
        u, v = img[:, 0] / rect[:, 2], img[:, 1] / rect[:, 2]          # rect_to_img divides by the rect depth
        out.append([np.clip(u.min(), 0, shape[1] - 1), np.clip(v.min(), 0, shape[0] - 1),
                    np.clip(u.max(), 0, shape[1] - 1), np.clip(v.max(), 0, shape[0] - 1)])
    return np.array(out).reshape(-1, 4)


def test_image_boxes_match_a_float64_restatement():
    from findnpropagate_b200.synth import KITTI_IMAGE_SHAPE
    _, cal, *_ = _kitti_frames(1)[0]
    cal = Calibration(cal)
    rng = np.random.default_rng(3)
    n = 400
    # in front of the camera, many across the left / right / top / bottom borders of the image
    boxes = np.concatenate([rng.uniform(4, 40, (n, 1)), rng.uniform(-30, 30, (n, 1)), rng.uniform(-2, 3, (n, 1)),
                            rng.uniform(0.5, 6, (n, 3)), rng.uniform(-np.pi, np.pi, (n, 1))], 1).astype(np.float32)
    boxes = boxes[boxes[:, 0] - np.hypot(boxes[:, 3], boxes[:, 4]) > 1.0]
    got = cli.image_boxes(boxes, cal, KITTI_IMAGE_SHAPE)
    want = _image_boxes_f64(boxes, cal, KITTI_IMAGE_SHAPE)
    assert got.dtype == np.float32 and got.shape == want.shape
    assert np.abs(got - want).max() < 1e-3
    H, W = KITTI_IMAGE_SHAPE
    assert (want[:, 0] == 0).sum() > 10 and (want[:, 2] == W - 1).sum() > 10 and (want[:, 1] == 0).sum() > 10
    assert (want[:, 3] == H - 1).sum() > 10 and ((want[:, 0] > 0) & (want[:, 2] < W - 1)).sum() > 10
    # the two helpers one by one: the camera box round-trips through boxes3d_kitti_camera_to_lidar
    cam = kitti_feed.boxes3d_lidar_to_kitti_camera(boxes, cal)
    back = kitti_feed.boxes3d_kitti_camera_to_lidar(cam, cal)
    assert np.abs(back[:, :6] - boxes[:, :6]).max() < 1e-3
    assert np.abs(np.cos(back[:, 6] - boxes[:, 6]) - 1).max() < 1e-6
    assert cli.image_boxes(np.zeros((0, 7), np.float32), cal, KITTI_IMAGE_SHAPE).shape == (0, 4)
