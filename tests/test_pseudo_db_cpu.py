"""python -m findnpropagate_b200.create_pseudo_database on the host: --help, the output names, every refusal (nothing is
written), and the argument checks of gt_database.crop_points_in_boxes.  ``write_sweep_tree`` builds the reference-like
tree of test_extract_cli with earlier sweeps (files, ``transform_matrix``, ``time_lag``) in every info, which the GPU
tests of the command and tools/pseudo_db_bench.py also use."""
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest
import torch

from findnpropagate_b200 import extract, gt_database
from findnpropagate_b200 import create_pseudo_database as cli

from test_extract_cli import HEAD, INFOS, NUSC, ROOT, _frames, _write_tree


def write_sweep_tree(base, frames, n_sweeps=9, seed=0):
    """_write_tree plus ``n_sweeps`` earlier sweeps per frame: each a random half of the frame's points, moved by a
    small rigid transform, under samples/SWEEPS; returns base/tools."""
    tools = _write_tree(base, frames)
    nusc = os.path.join(str(base), NUSC)
    with open(os.path.join(nusc, INFOS), "rb") as f:
        infos = pickle.load(f)
    rng = np.random.default_rng(seed)
    for info, fr in zip(infos, frames):
        info["sweeps"] = []
        for k in range(n_sweeps):
            rel = os.path.join("samples", "SWEEPS", "%s_%d.bin" % (fr.frame_id, k))
            os.makedirs(os.path.join(nusc, os.path.dirname(rel)), exist_ok=True)
            pts = np.asarray(fr.points, np.float32)
            np.ascontiguousarray(pts[rng.random(pts.shape[0]) < 0.5]).tofile(os.path.join(nusc, rel))
            a = rng.uniform(-0.02, 0.02)
            tm = np.eye(4)
            tm[:2, :2] = [[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]]
            tm[:3, 3] = rng.uniform(-0.5, 0.5, 3)
            info["sweeps"].append(dict(lidar_path=rel, transform_matrix=tm, time_lag=0.05 * (k + 1)))
    with open(os.path.join(nusc, INFOS), "wb") as f:
        pickle.dump(infos, f)
    return tools


def write_pseudos(folder, frames, seed=0, extra=None):
    """One .pth per frame (extract.save_frame): each GT box twice (jittered, so the NMS has work), random boxes,
    tied scores, labels 1..10; ``extra`` {frame index: (boxes, scores, labels)} replaces a frame's content."""
    os.makedirs(folder, exist_ok=True)
    rng = np.random.default_rng(seed)
    for i, fr in enumerate(frames):
        gt = np.asarray(fr.gt_boxes, np.float32)
        if extra and i in extra:
            b, s, l = extra[i]
        else:
            jit = gt[:, :7] + rng.normal(0, 0.1, (gt.shape[0], 7)).astype(np.float32) * [1, 1, 0.2, 0.1, 0.1, 0.1, 0.1]
            rnd = np.concatenate([rng.uniform(-30, 30, (6, 2)), rng.uniform(-1.5, 0, (6, 1)), rng.uniform(0.5, 5, (6, 3)),
                                  rng.uniform(-3, 3, (6, 1))], 1)
            b = np.concatenate([gt[:, :7], jit, rnd]).astype(np.float32)
            s = np.round(rng.uniform(0, 1, b.shape[0]), 1).astype(np.float32)        # ties
            l = np.concatenate([gt[:, -1], gt[:, -1], rng.integers(1, 11, 6)]).astype(np.int32)
        extract.save_frame(str(folder), fr.frame_id, dict(pred_boxes=b, pred_scores=s, pred_labels=l))


@pytest.fixture
def tree(tmp_path, monkeypatch):
    frames = _frames("tiny", 3)
    tools = write_sweep_tree(tmp_path, frames, n_sweeps=2)
    write_pseudos(str(tmp_path / "pseudo"), frames)
    monkeypatch.chdir(tools)
    return tmp_path


def _outputs(base, sweeps=1):
    return cli.output_paths(base / NUSC, sweeps)


def _refused(argv, capsys, base, match):
    with pytest.raises(SystemExit) as e:
        cli.main(argv)
    assert e.value.code == 1
    assert match in capsys.readouterr().err
    assert not any(p.exists() for p in _outputs(base)) and not any(p.exists() for p in _outputs(base, 10))


def test_help_runs_without_a_gpu():
    r = subprocess.run([sys.executable, "-m", "findnpropagate_b200.create_pseudo_database", "--help"], cwd=ROOT,
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    for flag in ("--cfg_file", "--folder", "--labels", "--nms_thresh", "--seed", "--batch_frames", "--workers", "--set"):
        assert flag in r.stdout


def test_output_names(tmp_path):
    d, p = cli.output_paths(tmp_path, 10)
    assert d == tmp_path / "pseudo_database_10sweeps_withvelo"
    assert p == tmp_path / "nuscenes_pseudo_dbinfos_10sweeps_withvelo.pkl"


def test_refusals_write_nothing(tree, capsys, monkeypatch):
    args = ["--cfg_file", HEAD, "--folder", "../pseudo"]
    _refused(["--cfg_file", HEAD, "--folder", "../nowhere"], capsys, tree, "../nowhere does not exist")
    for bad in (["0"], ["3", "11"]):
        _refused(args + ["--labels"] + bad, capsys, tree, "outside the classes")
    _refused(args + ["--set", "DATA_CONFIG.NOPE", "1"], capsys, tree, "DATA_CONFIG.NOPE")
    monkeypatch.setenv("WORLD_SIZE", "2")
    _refused(args, capsys, tree, "one process")
    monkeypatch.delenv("WORLD_SIZE")


@pytest.mark.parametrize("which", [0, 1])
def test_existing_output_is_refused(tree, capsys, which):
    target = _outputs(tree, 10)[which]
    (target.mkdir() if which == 0 else target.write_bytes(b"x"))
    with pytest.raises(SystemExit) as e:
        cli.main(["--cfg_file", HEAD, "--folder", "../pseudo", "--set", "DATA_CONFIG.MAX_SWEEPS", "10"])
    assert e.value.code == 1 and "already exists" in capsys.readouterr().err
    other = _outputs(tree, 10)[1 - which]
    assert not other.exists()
    assert (not any(target.iterdir())) if which == 0 else target.read_bytes() == b"x"


def test_bad_label_in_a_file_names_the_frame(tree, capsys):
    frames = _frames("tiny", 3)
    b = np.asarray(frames[1].gt_boxes, np.float32)[:2, :7]
    write_pseudos(str(tree / "pseudo"), frames, extra={1: (b, np.ones(2, np.float32), np.array([3, 11], np.int32))})
    _refused(["--cfg_file", HEAD, "--folder", "../pseudo"], capsys, tree, "frame %s: label 11" % frames[1].frame_id)


def test_frame_over_the_nms_limit_is_refused(tree, capsys):
    from findnpropagate_b200._lib import SEG_NMS_MAX
    frames = _frames("tiny", 3)
    n = SEG_NMS_MAX + 1
    b = np.tile(np.array([[5, 5, -1, 2, 2, 1.5, 0]], np.float32), (n, 1))
    write_pseudos(str(tree / "pseudo"), frames, extra={2: (b, np.ones(n, np.float32), np.ones(n, np.int32))})
    _refused(["--cfg_file", HEAD, "--folder", "../pseudo", "--nms_thresh", "0.1"], capsys, tree,
             "frame %s: %d boxes" % (frames[2].frame_id, n))


def _crop_args(n=10, g=2, c=5):
    return dict(points=torch.zeros((n, c)), row_start=np.array([0, 4, n]), boxes=torch.zeros((g, 7)),
                centres=torch.zeros((g, 3), dtype=torch.float64), box_start=np.array([0, 1, g]))


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
def test_crop_launcher_refusals(change, match):
    kw = _crop_args()
    kw.update(change)
    with pytest.raises(ValueError, match=match):
        gt_database.crop_points_in_boxes(**kw)
