"""KittiFeed (findnpropagate_b200.kitti_feed) and the KITTI configs of the commands, without a GPU: the calibration
parse, the FOV rule at the image borders and at depth 0, the GT conversion and its training-mode filters, the
SKIP_NO_GT re-draw, the dataset / head pairing, the failed-frame check, the database refusal and the tuner's grouping
and refusals for the KITTI head."""
import functools
import os
import pickle

import numpy as np
import pytest
import yaml

from findnpropagate_b200 import kitti_feed, synth
from findnpropagate_b200.kitti_feed import Calibration, KittiFeed

KITTI_HEAD = "cfgs/kitti_box_seeker_proposals.yaml"
KITTI_DATA = "data/kitti"
P = "MODEL.DENSE_HEAD.PARAMS."


@functools.lru_cache(maxsize=None)
def _kitti_frames(n):
    return tuple(synth.make_kitti_frame(i, with_gt=True) for i in range(n))


def _kitti_cfg(params=None, **data):
    d = dict(DATASET="KittiDataset", DATA_PATH="../" + KITTI_DATA, DATA_SPLIT=dict(train="train", test="val"),
             INFO_PATH=dict(train=["kitti_infos_train.pkl"], test=["kitti_infos_val.pkl"]),
             POINT_CLOUD_RANGE=[0, -40, -3, 70.4, 40, 1], FOV_POINTS_ONLY=True)
    d.update(data)
    head = dict(NAME="FrustumProposerOGKITTI", PREDS_PATH="../%s/kitti_coco_results.json" % KITTI_DATA,
                PARAMS=dict(params or dict(nms_3d=0.0, score_thr=0.45, nms_2d=0.4)))
    return dict(CLASS_NAMES=list(synth.KITTI_CLASS_NAMES), DATA_CONFIG=d, MODEL=dict(NAME="Seeker", DENSE_HEAD=head))


def write_kitti_tree(base, frames, cfg=None, predicted=None):
    """base/tools/cfgs/kitti_box_seeker_proposals.yaml and base/data/kitti/... (write_kitti_tree); returns base/tools.
    predicted: indices of the frames the COCO result file lists (default: all)."""
    tools = os.path.join(str(base), "tools")
    path = os.path.join(tools, KITTI_HEAD)
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "w") as f:
        yaml.safe_dump(cfg or _kitti_cfg(), f)
    root = os.path.join(str(base), KITTI_DATA)
    synth.write_kitti_tree(root, frames)
    if predicted is not None:
        import json
        coco = os.path.join(root, "kitti_coco_results.json")
        d = json.load(open(coco))
        d["images"] = [im for im in d["images"] if im["id"] in predicted]
        d["annotations"] = [a for a in d["annotations"] if a["image_id"] in predicted]
        json.dump(d, open(coco, "w"))
    return tools


@pytest.fixture
def kitti_tools(tmp_path, monkeypatch):
    tools = write_kitti_tree(tmp_path, _kitti_frames(3))
    monkeypatch.chdir(tools)
    return tmp_path


# --------------------------------------------------------------------------------------------------- calibration
def test_calib_file_parse(tmp_path):
    p = tmp_path / "000007.txt"
    p.write_text("P0: 1 0 0 0 0 1 0 0 0 0 1 0\n"
                 "P1: 2 0 0 0 0 2 0 0 0 0 1 0\n"
                 "P2: 7.215377e+02 0.000000e+00 6.095593e+02 4.485728e+01 0.000000e+00 7.215377e+02 1.728540e+02 "
                 "2.163791e-01 0.000000e+00 0.000000e+00 1.000000e+00 2.745884e-03\n"
                 "P3: 3 0 0 0 0 3 0 0 0 0 1 0\n"
                 "R0_rect: 9.999239e-01 9.837760e-03 -7.445048e-03 -9.869795e-03 9.999421e-01 -4.278459e-03 "
                 "7.402527e-03 4.351614e-03 9.999631e-01\n"
                 "Tr_velo_to_cam: 7.533745e-03 -9.999714e-01 -6.166020e-04 -4.069766e-03 1.480249e-02 7.280733e-04 "
                 "-9.998902e-01 -7.631618e-02 9.998621e-01 7.523790e-03 1.480755e-02 -2.717806e-01\n"
                 "Tr_imu_to_velo: 1 0 0 0 0 1 0 0 0 0 1 0\n")
    c = kitti_feed.get_calib_from_file(str(p))
    assert {k: v.dtype for k, v in c.items()} == dict(P2=np.float32, P3=np.float32, R0=np.float32, Tr_velo2cam=np.float32)
    assert c["P2"].shape == (3, 4) and c["R0"].shape == (3, 3) and c["Tr_velo2cam"].shape == (3, 4)
    assert c["P2"][0].tolist() == np.float32([721.5377, 0.0, 609.5593, 44.85728]).tolist()
    assert c["P2"][1, 3] == np.float32(0.2163791) and c["P2"][2, 3] == np.float32(0.002745884)
    assert c["P3"][0, 0] == 3
    assert c["R0"][2].tolist() == np.float32([0.007402527, 0.004351614, 0.9999631]).tolist()
    assert c["Tr_velo2cam"][:, 3].tolist() == np.float32([-0.004069766, -0.07631618, -0.2717806]).tolist()
    cal = Calibration(str(p))
    assert cal.P2 is not None and np.array_equal(cal.V2C, c["Tr_velo2cam"])


def _axis_calib():
    """LiDAR (x forward, y left, z up) -> camera (x right, y down, z forward) with P2 = [I | 0]: u = -y / x, v = -z / x,
    depth = x, all exact in float32."""
    V2C = np.array([[0, -1, 0, 0], [0, 0, -1, 0], [1, 0, 0, 0]], np.float32)
    P2 = np.array([[1, 0, 0, 0], [0, 1, 0, 0], [0, 0, 1, 0]], np.float32)
    return Calibration(dict(P2=P2, R0=np.eye(3, dtype=np.float32), Tr_velo2cam=V2C))


def test_fov_rule_at_the_borders():
    H, W = 375.0, 1242.0
    below_w, below_h = float(np.nextafter(np.float32(W), np.float32(0))), float(np.nextafter(np.float32(H), np.float32(0)))
    e = 2.0 ** -20
    # (x, y, z) -> kept?  u = -y / x, v = -z / x, depth = x
    cases = [((1, 0, -5), True),                  # u = 0
             ((1, e, -5), False),                 # u just below 0
             ((1, -W, -5), False),                # u = W
             ((1, -below_w, -5), True),           # the float below W
             ((1, -5, 0), True),                  # v = 0
             ((1, -5, e), False),                 # v just below 0
             ((1, -5, -H), False),                # v = H
             ((1, -5, -below_h), True),           # the float below H
             ((0, -5, -5), False),                # depth 0: u and v are infinite
             ((e, -5 * e, -5 * e), True),         # depth just above 0, u = v = 5
             ((-e, 5 * e, 5 * e), False),         # depth just below 0, u = v = 5
             ((-10, 50, 50), False)]              # behind the camera, u = v = 5
    pts = np.array([c[0] + (0.0,) for c in cases], np.float32)
    got = kitti_feed.fov_flag(pts, (int(H), int(W)), _axis_calib())
    assert got.tolist() == [c[1] for c in cases]


def test_fov_rule_agrees_with_float64_away_from_the_borders():
    pts, cal = synth.make_kitti_frame(0, full_scan=True)[:2]
    rng = np.random.default_rng(0)
    pts = np.concatenate([pts, rng.uniform([-20, -40, -3, 0], [60, 40, 3, 1], size=(20000, 4)).astype(np.float32)])
    c = Calibration(cal)
    H, W = synth.KITTI_IMAGE_SHAPE
    V2C, R0, P2 = (np.asarray(m, np.float64) for m in (c.V2C, c.R0, c.P2))
    rect = np.c_[pts[:, :3].astype(np.float64), np.ones(len(pts))] @ V2C.T @ R0.T
    img = np.c_[rect, np.ones(len(pts))] @ P2.T
    u, v, depth = img[:, 0] / rect[:, 2], img[:, 1] / rect[:, 2], img[:, 2] - P2[2, 3]
    ref = (u >= 0) & (u < W) & (v >= 0) & (v < H) & (depth >= 0)
    far = (np.minimum.reduce([np.abs(u), np.abs(u - W), np.abs(v), np.abs(v - H)]) > 1e-2) & (np.abs(depth) > 1e-3)
    got = kitti_feed.fov_flag(pts, (H, W), c)
    assert far.sum() > 0.99 * len(pts) and 0.1 * len(pts) < ref.sum() < 0.9 * len(pts)
    assert np.array_equal(got[far], ref[far])


# --------------------------------------------------------------------------------------------------- GT
def _restated_lidar_boxes(annos, cal):
    """boxes3d_kitti_camera_to_lidar in float64, written out: the bottom centre through inverse(R0_ext V2C_ext), then
    z up by h / 2, (l, w, h) and heading -(ry + pi / 2)."""
    r0e, v2ce = np.eye(4), np.eye(4)
    r0e[:3, :3] = cal.R0
    v2ce[:3, :] = cal.V2C
    xyz = (np.linalg.inv(r0e @ v2ce) @ np.c_[annos["location"], np.ones(len(annos["name"]))].T).T[:, :3]
    l, h, w = annos["dimensions"][:, 0], annos["dimensions"][:, 1], annos["dimensions"][:, 2]
    return np.c_[xyz[:, 0], xyz[:, 1], xyz[:, 2] + h / 2, l, w, h, -(annos["rotation_y"] + np.pi / 2)]


def test_camera_to_lidar_agrees_with_a_restatement():
    c = Calibration(_kitti_frames(3)[1][1])
    rng = np.random.default_rng(1)
    annos = dict(name=np.array(["Car"] * 50), location=rng.uniform([-20, -2, 1], [20, 3, 70], (50, 3)).astype(np.float32),
                 dimensions=rng.uniform(0.5, 6, (50, 3)).astype(np.float32),
                 rotation_y=rng.uniform(-np.pi, np.pi, 50).astype(np.float32))
    cam = np.c_[annos["location"], annos["dimensions"], annos["rotation_y"]].astype(np.float32)
    got = kitti_feed.boxes3d_kitti_camera_to_lidar(cam, c)
    assert got.dtype == np.float32
    assert np.allclose(got, _restated_lidar_boxes(annos, c), rtol=1e-5, atol=1e-5)


def _tree_feed(base, **kw):
    return KittiFeed(os.path.join(str(base), KITTI_DATA), "kitti_infos_train.pkl",
                     class_names=kw.pop("class_names", synth.KITTI_CLASS_NAMES), device="cpu", **kw)


def test_gt_filters_and_heading_wrap(tmp_path):
    frames = list(_kitti_frames(3))
    write_kitti_tree(tmp_path, frames)
    feed = _tree_feed(tmp_path)
    info = feed.infos[0]
    assert "DontCare" in list(info["annos"]["name"])
    cal = feed.calib(info["point_cloud"]["lidar_idx"])
    keep = info["annos"]["name"] != "DontCare"
    ref = _restated_lidar_boxes({k: v[keep] for k, v in info["annos"].items()}, cal)
    ref[:, 6] = ref[:, 6] - np.floor(ref[:, 6] / (2 * np.pi) + 0.5) * 2 * np.pi
    inside = (ref[:, :3] >= feed.range[:3]).all(1) & (ref[:, :3] <= feed.range[3:]).all(1)
    assert 0 < inside.sum() < len(ref)                   # the tree holds GT out of range
    got = feed.gt_boxes(0)
    assert got.shape == (inside.sum(), 8)
    assert np.allclose(got[:, :7], ref[inside], rtol=1e-5, atol=1e-4)
    assert (got[:, 6] >= -np.pi).all() and (got[:, 6] < np.pi).all()
    names = info["annos"]["name"][keep][inside]
    assert got[:, 7].tolist() == [synth.KITTI_CLASS_NAMES.index(n) + 1 for n in names]
    # the boxes are the synthetic LiDAR boxes the tree was written from
    src = np.asarray(frames[0][5], np.float64)
    src_in = src[(src[:, :3] >= feed.range[:3]).all(1) & (src[:, :3] <= feed.range[3:]).all(1)]
    assert np.allclose(got[:, :6], src_in[:, :6], atol=1e-4)
    # __getitem__: the same GT, the points inside the x / y range and on the image
    d = feed[0]
    assert np.array_equal(d["gt_boxes"], got) and d["frame_id"] == "000000"
    assert d["points"].dtype == np.float32 and d["points"].shape[1] == 4
    assert (d["points"][:, 0] >= 0).all() and (d["points"][:, 0] <= 70.4).all()
    assert len(d["points"]) < len(frames[0][0])
    # the class filter: a feed of two classes keeps only theirs, with their own column
    two = _tree_feed(tmp_path, class_names=["Van", "Car"])
    g2 = two.gt_boxes(0)
    sel = np.isin(names, ["Van", "Car"])
    assert g2[:, 7].tolist() == [["Van", "Car"].index(n) + 1 for n in names[sel]]
    assert np.array_equal(g2[:, :7], got[sel, :7])
    # FOV_POINTS_ONLY off: the range mask alone
    raw = _tree_feed(tmp_path, fov_points_only=False)[0]["points"]
    p0 = frames[0][0]
    assert len(raw) == int(((p0[:, 0] >= 0) & (p0[:, 0] <= 70.4) & (p0[:, 1] >= -40) & (p0[:, 1] <= 40)).sum())


class _Draw:
    def __init__(self, k):
        self.k, self.calls = k, 0

    def randint(self, n):
        self.calls += 1
        return self.k


def test_skip_no_gt_redraws_in_getitem_only(tmp_path):
    write_kitti_tree(tmp_path, _kitti_frames(3))
    root = tmp_path / KITTI_DATA
    infos = pickle.load(open(root / "kitti_infos_train.pkl", "rb"))
    a = infos[1]["annos"]
    a["location"][:, 0] = -30.0                          # every box of frame 1 left of the range (x < 0 in LiDAR)
    a["location"][:, 2] = -5.0
    pickle.dump(infos, open(root / "kitti_infos_train.pkl", "wb"))
    draw = _Draw(2)
    feed = _tree_feed(tmp_path, rng=draw)
    d = feed[1]
    assert draw.calls == 1 and d["frame_id"] == "000002"
    assert np.array_equal(d["gt_boxes"], feed.gt_boxes(2))
    for f in (root / "training" / "velodyne").iterdir():
        f.unlink()
    assert feed.gt_boxes(1).shape == (0, 8) and draw.calls == 1
    assert len(feed.gt_boxes(0)) > 0


# --------------------------------------------------------------------------------------------------- commands
def test_kitti_pair_is_accepted_and_mixed_pairs_are_refused(kitti_tools):
    from findnpropagate_b200 import extract_pseudo_labels as cli
    cfg = cli.load_config(KITTI_HEAD)
    assert cli.is_kitti(cfg)
    feed = cli.build_feed(cfg)
    assert isinstance(feed, KittiFeed) and feed.training and len(feed) == 3 and feed.fov_points_only
    assert os.path.samefile(feed.root_split_path, kitti_tools / KITTI_DATA / "training")
    assert feed.range.tolist() == [0, -40, -3, np.float32(70.4), 40, 1]
    assert feed.class_names == synth.KITTI_CLASS_NAMES
    assert cli.build_feed(cli.load_config(KITTI_HEAD, ["DATA_CONFIG.FOV_POINTS_ONLY", "False"])).fov_points_only is False
    for key, value in (("MODEL.DENSE_HEAD.NAME", "FrustumProposerOG"), ("DATA_CONFIG.DATASET", "NuScenesDataset")):
        with pytest.raises(ValueError) as e:
            cli.load_config(KITTI_HEAD, [key, value])
        assert value in str(e.value) and "FrustumProposerOGKITTI on KittiDataset" in str(e.value)
    with pytest.raises(ValueError, match="WaymoDataset"):
        cli.load_config(KITTI_HEAD, ["DATA_CONFIG.DATASET", "WaymoDataset"])


def test_check_frame_reports_each_failure(tmp_path, monkeypatch):
    from findnpropagate_b200 import extract_pseudo_labels as cli
    from findnpropagate_b200.proposer import PreprocessedDetector
    tools = write_kitti_tree(tmp_path, _kitti_frames(4), predicted=[0, 1, 3])
    monkeypatch.chdir(tools)
    root = tmp_path / KITTI_DATA / "training"
    os.remove(root / "velodyne" / "000000.bin")
    os.remove(root / "calib" / "000001.txt")
    feed = cli.build_feed(cli.load_config(KITTI_HEAD))
    det = PreprocessedDetector([str(tmp_path / KITTI_DATA / "kitti_coco_results.json")], synth.KITTI_CLASS_NAMES)
    assert [cli.check_frame(feed, det, info) for info in feed.infos] == [cli.LIDAR_MISSING, cli.CALIB_MISSING,
                                                                          cli.IMAGE_NOT_PREDICTED, 0]
    assert [cli.check_frame(feed, None, info) for info in feed.infos] == [cli.LIDAR_MISSING, cli.CALIB_MISSING, 0, 0]
    assert [cli.frame_id(info) for info in feed.infos] == ["000000", "000001", "000002", "000003"]


def _snapshot(base):
    return sorted((os.path.relpath(os.path.join(d, f), str(base)), os.stat(os.path.join(d, f)).st_mtime_ns)
                  for d, _, fs in os.walk(str(base)) for f in fs)


def test_pseudo_database_refuses_a_kitti_config(kitti_tools, capsys):
    from findnpropagate_b200 import create_pseudo_database
    os.makedirs("../pseudo")
    before = _snapshot(kitti_tools)
    with pytest.raises(SystemExit) as e:
        create_pseudo_database.main(["--cfg_file", KITTI_HEAD, "--folder", "../pseudo"])
    assert e.value.code == 1
    assert "KittiDataset" in capsys.readouterr().err
    assert _snapshot(kitti_tools) == before


def _grid(d, path="grid.yaml"):
    with open(path, "w") as f:
        yaml.safe_dump(d, f, sort_keys=False)
    return path


@pytest.mark.parametrize("key,values", [(P + "ego_w", [0.0]), (P + "occl_w", [0.0, 0.2]), ("MODEL.DENSE_HEAD.MULT", [True]),
                                        ("MODEL.DENSE_HEAD.OCCL_MULT", [False]), ("MODEL.DENSE_HEAD.MULTICAM_IOU", [True]),
                                        (P + "topk", [1, 2]), (P + "rand_center", [True])])
def test_tuner_refuses_keys_the_kitti_head_does_not_read(kitti_tools, capsys, monkeypatch, key, values):
    from findnpropagate_b200 import tune_params
    monkeypatch.setattr(tune_params, "build_feed", lambda *a, **k: pytest.fail("read frames"))
    monkeypatch.setattr(tune_params, "build_head", lambda *a, **k: pytest.fail("built the head"))
    with pytest.raises(SystemExit) as e:
        tune_params.main(["--cfg_file", KITTI_HEAD, "--grid", _grid({P + "dns_w": [0.5, 1.0], key: values})])
    assert e.value.code == 1
    err = capsys.readouterr().err
    assert "setting {" in err and key.split(".")[-1] in err


def test_kitti_grouping(kitti_tools):
    from findnpropagate_b200 import tune_params
    from findnpropagate_b200.extract_pseudo_labels import load_config
    from findnpropagate_b200.proposer import kitti_head_params
    base = kitti_head_params(load_config(KITTI_HEAD).MODEL.DENSE_HEAD)
    assert base["max_dist"] == 70 and base["score_thr"] == 0.45
    axes = [("a", "dns_w", True, [0.05, 0.5, 1.0]), ("b", "iou_w", True, [0.5, 1.0]), ("c", "dst_w", True, [0.0, 0.2])]
    flat = [{k: v for k, v in zip(("dns_w", "iou_w", "dst_w"), s.values())} for s in tune_params.expand_grid(axes)]
    groups = tune_params.group_settings(base, flat, "kitti")
    assert [g["members"] for g in groups] == [list(range(12))]
    assert groups[0]["params"]["min_cam_iou"] == base["min_cam_iou"]
    two = [dict(s, min_cam_iou=m) for m in (0.3, 0.5) for s in flat]
    groups = tune_params.group_settings(base, two, "kitti")
    assert [g["members"] for g in groups] == [list(range(12)), list(range(12, 24))]
    assert [g["params"]["min_cam_iou"] for g in groups] == [0.3, 0.5]
    # the nuScenes rule on the same settings: min_cam_iou is select-level there
    assert len(tune_params.group_settings(base, two)) == 1
