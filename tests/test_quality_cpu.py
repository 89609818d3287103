"""Per-class / per-range quality counters on the host: NuScenesFeed.gt_boxes, the table layout of quality.tables and
recall_dict, and the refusals of the eval_pseudo_labels command."""
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest

from findnpropagate_b200 import quality
from findnpropagate_b200.nuscenes_feed import NuScenesFeed

from test_extract_cli import HEAD, INFOS, NUSC, ROOT, _frames, _write_tree

CLASSES = ("car", "truck", "construction_vehicle", "bus", "trailer", "barrier", "motorcycle", "bicycle", "pedestrian",
           "traffic_cone")


@pytest.fixture
def tree(tmp_path, monkeypatch):
    tools = _write_tree(tmp_path, _frames("tiny", 3))
    monkeypatch.chdir(tools)
    return tmp_path


@pytest.mark.parametrize("kw", [dict(training=True), dict(training=False), dict(training=True, pred_velocity=False),
                                dict(training=True, filter_min_points_in_gt=0, point_cloud_range=[-20, -20, -5, 20, 20, 3])])
def test_gt_boxes_equals_getitem_without_lidar(tree, kw):
    infos = pickle.load(open(tree / NUSC / INFOS, "rb"))
    infos[1]["gt_boxes"][0, 7:9] = np.nan            # NaN velocity: zeroed
    feed = NuScenesFeed(tree / NUSC, infos, max_sweeps=1, **kw)
    want = [feed[i]["gt_boxes"] for i in range(len(feed))]
    assert sum(len(w) for w in want) > 0
    for i in range(len(feed)):
        os.remove(tree / NUSC / infos[i]["lidar_path"])
    for i, w in enumerate(want):
        got = feed.gt_boxes(i)
        assert got.dtype == w.dtype and got.shape == w.shape and np.array_equal(got, w)
    # gt_boxes works on a copy: the infos are not changed by it
    assert np.array_equal(feed.gt_boxes(0), want[0])


def test_gt_boxes_of_a_frame_left_without_gt_is_empty(tree):
    infos = pickle.load(open(tree / NUSC / INFOS, "rb"))
    infos[0]["gt_boxes"][:, 0] = 500.0                   # every centre outside the range: training mode drops them
    feed = NuScenesFeed(tree / NUSC, infos, max_sweeps=1, training=True, rng=np.random.RandomState(0))
    g = feed.gt_boxes(0)
    assert g.shape[0] == 0 and g.shape[1] == feed.gt_boxes(1).shape[1]
    assert len(feed[0]["gt_boxes"]) > 0                   # __getitem__ draws another frame in its place


def _hand_counters(spec):
    """Counters with a distinct value per entry, laid out as fnp.h documents: [block][class][bin][w]."""
    C, R, W = len(spec.class_names), spec.n_bins, spec.width
    return np.arange(2 * C * R * W, dtype=np.int64).reshape(2, C, R, W), C, R, W


def test_tables_layout_and_bins():
    spec = quality.QualitySpec(CLASSES)
    assert spec.bin_names() == ["0-20", "20-30", "30-40", "40+"]
    assert quality.QualitySpec(CLASSES, range_edges=(12.5,)).bin_names() == ["0-12.5", "12.5+"]
    assert quality.QualitySpec(CLASSES, range_edges=()).bin_names() == ["0+"]
    c, C, R, W = _hand_counters(spec)
    assert spec.n_counters == c.size == 2 * 10 * 4 * 7
    tab = quality.tables(c.reshape(-1), spec)
    assert list(tab) == list(CLASSES) and list(tab["bus"]) == ["0-20", "20-30", "30-40", "40+", "all"]
    e = tab["bus"]["30-40"]                      # class 4 -> index 3, bin 2
    assert e["gt"] == c[0, 3, 2, 0] and e["proposals"] == c[1, 3, 2, 0]
    assert e["recall_any"] == {"0.3": c[0, 3, 2, 1], "0.5": c[0, 3, 2, 2], "0.7": c[0, 3, 2, 3]}
    assert e["recall_label"] == {"0.3": c[0, 3, 2, 4], "0.5": c[0, 3, 2, 5], "0.7": c[0, 3, 2, 6]}
    assert e["precision_any"]["0.5"] == c[1, 3, 2, 2] and e["precision_label"]["0.7"] == c[1, 3, 2, 6]
    a = tab["pedestrian"]["all"]
    assert a["gt"] == c[0, 8, :, 0].sum() and a["precision_label"]["0.3"] == c[1, 8, :, 4].sum()


def test_recall_dict_known_unknown_sums():
    from findnpropagate_b200.extract import recall_keys
    spec = quality.QualitySpec(CLASSES)
    c, C, R, W = _hand_counters(spec)
    r = quality.recall_dict(c.reshape(-1), spec)
    assert list(r) == recall_keys()
    gt = c[0, :, :, 0].sum(1)                    # per class
    k3, k6 = [0, 7, 8], [0, 2, 4, 5, 7, 8]
    assert r["gt"] == gt.sum() and r["num_3known"] == gt[k3].sum() and r["num_6known"] == gt[k6].sum()
    assert r["num_4unknown"] == gt.sum() - gt[k6].sum() and r["num_7unknown"] == gt.sum() - gt[k3].sum()
    for t, th in enumerate((0.3, 0.5, 0.7)):
        hit = c[0, :, :, 1 + t].sum(1)
        assert r["rcnn_%s" % th] == hit.sum() and r["rcnn_3known_%s" % th] == hit[k3].sum()
        assert r["rcnn_6known_%s" % th] == hit[k6].sum() and r["rcnn_4unknown_%s" % th] == hit.sum() - hit[k6].sum()
        assert r["rcnn_7unknown_%s" % th] == hit.sum() - hit[k3].sum()
    p = quality.precision_dict(c.reshape(-1), spec)
    assert p["proposals"] == c[1, :, :, 0].sum() and p["hits_0.5"] == c[1, :, :, 2].sum()


@pytest.mark.parametrize("edges", [(30, 20), (20, 20), (0, 10), (-5,), tuple(range(1, 9))])
def test_spec_refuses_bad_edges(edges):
    with pytest.raises(ValueError):
        quality.QualitySpec(CLASSES, range_edges=edges)


def test_spec_refuses_too_many_thresholds_and_classes():
    with pytest.raises(ValueError):
        quality.QualitySpec(CLASSES, thresh=[0.1 * i for i in range(9)])
    with pytest.raises(ValueError):
        quality.QualitySpec(["c%d" % i for i in range(33)])
    quality.QualitySpec(CLASSES, range_edges=tuple(range(1, 8)), thresh=[0.1 * i for i in range(8)])


def test_check_labels_after_stripping_zero_rows():
    spec = quality.QualitySpec(CLASSES)
    gt = np.zeros((3, 8), np.float32)
    gt[0] = [1, 2, 0, 4, 2, 1.5, 0, 3]
    quality.check_labels(spec, np.array([1, 10]), gt, np.array([0, 3]))    # rows 1, 2: trailing zeros, dropped
    with pytest.raises(ValueError, match="proposal label"):
        quality.check_labels(spec, np.array([0]), gt, np.array([0, 3]))
    with pytest.raises(ValueError, match="proposal label"):
        quality.check_labels(spec, np.array([11]), gt, np.array([0, 3]))
    gt[2, 0] = 1.0                                # a non-zero last row: row 1 (label 0) is now inside the frame
    with pytest.raises(ValueError, match="GT class"):
        quality.check_labels(spec, np.array([1]), gt, np.array([0, 3]))
    assert quality.strip_gt(np.zeros((2, 8))).shape == (0, 8)


def _eval(argv):
    from findnpropagate_b200 import eval_pseudo_labels as cli
    return cli.main(argv)


def test_command_refusals(tree, capsys, monkeypatch):
    with pytest.raises(SystemExit) as e:
        _eval(["--cfg_file", HEAD, "--folder", "../nowhere"])
    assert e.value.code == 1 and "../nowhere does not exist" in capsys.readouterr().err
    os.makedirs("../out")
    for edges in (["30", "20"], ["0"], ["1", "2", "3", "4", "5", "6", "7", "8"]):
        with pytest.raises(SystemExit) as e:
            _eval(["--cfg_file", HEAD, "--folder", "../out", "--range_edges"] + edges)
        assert e.value.code == 1 and "edges" in capsys.readouterr().err
    with pytest.raises(SystemExit) as e:
        _eval(["--cfg_file", HEAD, "--folder", "../out", "--set", "DATA_CONFIG.NOPE", "1"])
    assert e.value.code == 1 and "DATA_CONFIG.NOPE" in capsys.readouterr().err
    monkeypatch.setenv("WORLD_SIZE", "2")
    with pytest.raises(SystemExit) as e:
        _eval(["--cfg_file", HEAD, "--folder", "../out"])
    assert e.value.code == 1 and "one process" in capsys.readouterr().err


def test_help_runs_without_a_gpu():
    for mod, flags in (("eval_pseudo_labels", ("--cfg_file", "--folder", "--nms_thresh", "--range_edges", "--every",
                                               "--batch_frames", "--workers", "--out", "--set")),
                       ("tune_params", ("--breakdown", "--range_edges"))):
        r = subprocess.run([sys.executable, "-m", "findnpropagate_b200." + mod, "--help"], cwd=ROOT,
                           capture_output=True, text=True, timeout=120)
        assert r.returncode == 0, r.stderr
        for flag in flags:
            assert flag in r.stdout
