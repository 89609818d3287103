"""python -m findnpropagate_b200.tune_params without a GPU: grid expansion, the grid refusals, the grouping of settings
that share stages 1-2c, the refusals of unsupported settings before any frame is read, --help."""
import os
import subprocess
import sys

import pytest
import yaml

from findnpropagate_b200 import synth, tune_params
from findnpropagate_b200.proposer import head_params

from test_extract_cli import HEAD, _write_tree, _frames

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = "MODEL.DENSE_HEAD.PARAMS."


@pytest.fixture
def tools_dir(tmp_path, monkeypatch):
    tools = _write_tree(tmp_path, _frames("tiny", 2))
    monkeypatch.chdir(tools)
    return tools


def _grid(d, path="grid.yaml"):
    with open(path, "w") as f:
        yaml.safe_dump(d, f, sort_keys=False)
    return path


def _axes(d):
    from findnpropagate_b200.extract_pseudo_labels import load_config
    return tune_params.load_grid(_grid(d), load_config(HEAD))


def test_grid_expands_in_cartesian_order(tools_dir):
    axes = _axes({P + "dns_w": [0.5, 1], "MODEL.DENSE_HEAD.MULT": [False, True], P + "ego_w": [0.0, 0.25]})
    assert [(k, n, y) for k, n, y, _ in axes] == [(P + "dns_w", "dns_w", True), ("MODEL.DENSE_HEAD.MULT", "MULT", False),
                                                  (P + "ego_w", "ego_w", False)]
    got = tune_params.expand_grid(axes)
    assert len(got) == 8
    assert [tuple(s.values()) for s in got] == [(a, b, c) for a in (0.5, 1.0) for b in (False, True) for c in (0.0, 0.25)]
    assert isinstance(got[-1][P + "dns_w"], float)        # an int where the config has a float: --set's rule


@pytest.mark.parametrize("grid,needle", [
    ({P + "nope": [1]}, P + "nope"),
    ({"DATA_CONFIG.MAX_SWEEPS": [1, 2]}, "DATA_CONFIG.MAX_SWEEPS"),
    ({"MODEL.DENSE_HEAD.NAME": ["x"]}, "MODEL.DENSE_HEAD.NAME"),
    ({P + "dns_w": 0.5}, P + "dns_w"),
    ({P + "dns_w": []}, P + "dns_w"),
    ({P + "num_mags": [4, "many"]}, P + "num_mags"),
    ({P + "ego_w": [True]}, P + "ego_w"),
    ({}, "empty"),
])
def test_grid_refusals_exit_1_and_name_the_key(tools_dir, capsys, monkeypatch, grid, needle):
    monkeypatch.setattr(tune_params, "build_feed", lambda *a, **k: pytest.fail("read frames"))
    with pytest.raises(SystemExit) as e:
        tune_params.main(["--cfg_file", HEAD, "--grid", _grid(grid)])
    assert e.value.code == 1
    assert needle in capsys.readouterr().err


def test_group_settings_shares_select_level_keys_only(tools_dir):
    from findnpropagate_b200.extract_pseudo_labels import load_config
    base = head_params(load_config(HEAD).MODEL.DENSE_HEAD)
    select = [dict(dns_w=0.5), dict(iou_w=0.2, min_cam_iou=0.5), dict(dst_w=0.3), dict(ego_w=0.1), dict(occl_w=0.2),
              dict(MULT=True), dict(OCCL_MULT=True), dict(min_cam_iou=0.4, dns_w=2.0)]
    groups = tune_params.group_settings(base, select)
    assert [g["members"] for g in groups] == [list(range(len(select)))]
    assert groups[0]["params"]["min_cam_iou"] == base["min_cam_iou"] == 0.3
    assert tune_params.group_settings(base, select[1:2])[0]["params"]["min_cam_iou"] == 0.5
    # a routine cartesian grid beyond one kernel launch's 256 settings stays one group
    axes = [(P + "dns_w", "dns_w", True, [0.05, 0.5, 1.0, 2.0, 4.0]), (P + "iou_w", "iou_w", True, [0.25, 0.5, 1.0, 2.0]),
            (P + "dst_w", "dst_w", True, [0.0, 0.1, 0.2, 0.4]), (P + "min_cam_iou", "min_cam_iou", True, [0.3, 0.5]),
            ("MODEL.DENSE_HEAD.MULT", "MULT", False, [False, True])]
    big = [{k.split(".")[-1]: v for k, v in s.items()} for s in tune_params.expand_grid(axes)]
    assert len(big) == 320
    assert [g["members"] for g in tune_params.group_settings(base, big)] == [list(range(320))]
    for split in (dict(num_mags=5), dict(lq=0.1), dict(nms_2d=0.5), dict(MULTICAM_IOU=True)):
        groups = tune_params.group_settings(base, [dict(dns_w=0.5), dict(split, dns_w=0.7), dict(dns_w=0.9)])
        assert [g["members"] for g in groups] == [[0, 2], [1]], split


@pytest.mark.parametrize("key,values,needle", [(P + "topk", [1, 2], "topk > 1"),
                                               (P + "rand_center", [False, True], "rand_center"),
                                               (P + "aln_w", [0.0, 0.5], "aln_w")])
def test_unsupported_settings_are_refused_before_any_frame_is_read(tools_dir, capsys, monkeypatch, key, values, needle):
    monkeypatch.setattr(tune_params, "build_feed", lambda *a, **k: pytest.fail("read frames"))
    with pytest.raises(SystemExit) as e:
        tune_params.main(["--cfg_file", HEAD, "--grid", _grid({key: values})])
    assert e.value.code == 1
    err = capsys.readouterr().err
    assert needle in err and "setting {" in err


def test_several_processes_are_refused(tools_dir, capsys, monkeypatch):
    monkeypatch.setenv("WORLD_SIZE", "2")
    with pytest.raises(SystemExit) as e:
        tune_params.main(["--cfg_file", HEAD, "--grid", _grid({P + "dns_w": [1.0]})])
    assert e.value.code == 1 and "one process" in capsys.readouterr().err


def test_help_runs_without_a_gpu():
    r = subprocess.run([sys.executable, "-m", "findnpropagate_b200.tune_params", "--help"], cwd=ROOT,
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    for flag in ("--cfg_file", "--grid", "--every", "--batch_frames", "--workers", "--set", "--out"):
        assert flag in r.stdout
