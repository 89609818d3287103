"""python -m findnpropagate_b200.extract_pseudo_labels: config loading (_BASE_CONFIG_ includes, --set), the supported
config check, the folder and failed-frame rules, and on the GPU the files it writes against the library calls it wires
up.  The fixtures lay out a tree like the reference's: configs under tools/cfgs, the nuScenes files under
data/nuscenes/v1.0-trainval and the GLIP predictions under data/training_pred, and run from tools/, so that the
relative paths of the config and of PreprocessedGLIP's defaults are the ones exercised."""
import functools
import json
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest
import torch
import yaml

from findnpropagate_b200 import synth
from findnpropagate_b200.config import cfg_from_list, cfg_from_yaml_file

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEAD = "cfgs/nuscenes_box_seeker_proposals.yaml"
DATASET = "cfgs/dataset_configs/nuscenes_dataset.yaml"
NUSC = "data/nuscenes/v1.0-trainval"
INFOS = "nuscenes_infos_10sweeps_train.pkl"
GLIP_PTH = "data/training_pred/nuscenes_glip_train_pred.pth"
GLIP_META = "data/training_pred/nuscenes_infos_train_mono3d.coco.json"


@functools.lru_cache(maxsize=None)
def _frames(name, n):
    return tuple(synth.make_frame(i, synth.CONFIGS[name]) for i in range(n))


def _dataset_cfg():
    """The part of cfgs/dataset_configs/nuscenes_dataset.yaml the command reads, and some it does not."""
    return dict(DATASET="NuScenesDataset", DATA_PATH="../data/nuscenes", VERSION="v1.0-trainval", MAX_SWEEPS=10,
                PRED_VELOCITY=True, SET_NAN_VELOCITY_TO_ZEROS=True, FILTER_MIN_POINTS_IN_GT=1,
                INFO_PATH=dict(train=[INFOS], test=["nuscenes_infos_10sweeps_val.pkl"]),
                POINT_CLOUD_RANGE=[-51.2, -51.2, -5.0, 51.2, 51.2, 3.0],
                CAMERA_CONFIG=dict(USE_CAMERA=True, IMAGE=dict(FINAL_DIM=[256, 704], RESIZE_LIM_TRAIN=[0.38, 0.55],
                                                               RESIZE_LIM_TEST=[0.48, 0.48])),
                DATA_AUGMENTOR=dict(DISABLE_AUG_LIST=["placeholder"], AUG_CONFIG_LIST=[dict(NAME="random_world_flip")]))


def _head_cfg(params, **dense_head):
    head = dict(NAME="FrustumProposerOG", PREDS_PATH="PreprocessedGLIP", BOX_FORMAT="xyxy", PARAMS=dict(params))
    head.update(dense_head)
    return dict(CLASS_NAMES=list(synth.CLASS_NAMES),
                DATA_CONFIG=dict(_BASE_CONFIG_=DATASET, POINT_CLOUD_RANGE=[-54.0, -54.0, -5.0, 54.0, 54.0, 3.0],
                                 MAX_SWEEPS=1, CAMERA_CONFIG=dict(IMAGE=dict(FINAL_DIM=[900, 1600],
                                                                             RESIZE_LIM_TEST=[1.0, 1.0]))),
                MODEL=dict(NAME="TransFusion", DENSE_HEAD=head))


def _write_yaml(path, d):
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "w") as f:
        yaml.safe_dump(d, f)


def _write_tree(base, frames, head=None, glip_frames=None):
    """base/tools/cfgs/..., base/data/nuscenes/v1.0-trainval/..., base/data/training_pred/...; returns base/tools."""
    tools = os.path.join(str(base), "tools")
    _write_yaml(os.path.join(tools, DATASET), _dataset_cfg())
    _write_yaml(os.path.join(tools, HEAD), head or _head_cfg(synth.seeker_params(synth.CONFIGS["cfg1"])))
    infos = synth.write_nuscenes_tree(os.path.join(str(base), NUSC), frames)
    with open(os.path.join(str(base), NUSC, INFOS), "wb") as f:
        pickle.dump(infos, f)
    synth.write_glip_predictions(frames if glip_frames is None else glip_frames, os.path.join(str(base), GLIP_PTH),
                                 os.path.join(str(base), GLIP_META))
    return tools


@pytest.fixture
def tools_dir(tmp_path, monkeypatch):
    """A reference-like tree of three tiny frames, the current directory set to its tools/."""
    tools = _write_tree(tmp_path, _frames("tiny", 3))
    monkeypatch.chdir(tools)
    return tools


# --------------------------------------------------------------------------------------------------- config (CPU)
def test_base_config_merges_at_a_nested_level(tools_dir):
    cfg = cfg_from_yaml_file(HEAD)
    d = cfg.DATA_CONFIG
    # from the base file, included under DATA_CONFIG
    assert d.DATASET == "NuScenesDataset" and d.VERSION == "v1.0-trainval" and d.INFO_PATH.train == [INFOS]
    assert d.CAMERA_CONFIG.USE_CAMERA is True and d.CAMERA_CONFIG.IMAGE.RESIZE_LIM_TRAIN == [0.38, 0.55]
    # the head's own keys at the top level, untouched by the include
    assert cfg.MODEL.DENSE_HEAD.NAME == "FrustumProposerOG" and cfg.CLASS_NAMES == list(synth.CLASS_NAMES)
    assert "DATASET" not in cfg


def test_including_file_overrides_its_base(tools_dir):
    d = cfg_from_yaml_file(HEAD).DATA_CONFIG
    assert d.MAX_SWEEPS == 1                                              # scalar replaced (base: 10)
    assert d.POINT_CLOUD_RANGE == [-54.0, -54.0, -5.0, 54.0, 54.0, 3.0]   # list replaced, not merged
    assert d.CAMERA_CONFIG.IMAGE.FINAL_DIM == [900, 1600]                 # dicts merged key by key
    assert d.CAMERA_CONFIG.IMAGE.RESIZE_LIM_TEST == [1.0, 1.0]
    assert d.CAMERA_CONFIG.IMAGE.RESIZE_LIM_TRAIN == [0.38, 0.55]


def test_set_overrides(tools_dir):
    cfg = cfg_from_yaml_file(HEAD)
    cfg_from_list(["DATA_CONFIG.MAX_SWEEPS", "3", "MODEL.DENSE_HEAD.PARAMS.score_thr", "0.3",
                   "MODEL.DENSE_HEAD.PARAMS.lq", "0", "DATA_CONFIG.DATA_PATH", "/data/nuscenes",
                   "DATA_CONFIG.INFO_PATH.train", "['a.pkl', 'b.pkl']", "DATA_CONFIG.POINT_CLOUD_RANGE", "-50,-50,-4,50,50,2"],
                  cfg)
    assert cfg.DATA_CONFIG.MAX_SWEEPS == 3 and cfg.MODEL.DENSE_HEAD.PARAMS.score_thr == 0.3
    assert cfg.MODEL.DENSE_HEAD.PARAMS.lq == 0.0 and isinstance(cfg.MODEL.DENSE_HEAD.PARAMS.lq, float)
    assert cfg.DATA_CONFIG.DATA_PATH == "/data/nuscenes"          # not a Python literal: kept as the string
    assert cfg.DATA_CONFIG.INFO_PATH.train == ["a.pkl", "b.pkl"]
    assert cfg.DATA_CONFIG.POINT_CLOUD_RANGE == [-50, -50, -4, 50, 50, 2]
    with pytest.raises(KeyError, match="MODEL.DENSE_HEAD.NOPE"):
        cfg_from_list(["MODEL.DENSE_HEAD.NOPE.x", "1"], cfg)
    with pytest.raises(KeyError, match="DATA_CONFIG.MAX_SWEPS"):
        cfg_from_list(["DATA_CONFIG.MAX_SWEPS", "1"], cfg)
    with pytest.raises(ValueError, match="MAX_SWEEPS"):
        cfg_from_list(["DATA_CONFIG.MAX_SWEEPS", "ten"], cfg)
    with pytest.raises(ValueError):
        cfg_from_list(["DATA_CONFIG.MAX_SWEEPS"], cfg)


def test_base_config_path_fallbacks(tmp_path, monkeypatch):
    cfgs = tmp_path / "tools" / "cfgs"
    _write_yaml(str(cfgs / "dataset_configs" / "ds.yaml"), dict(A=1, B=dict(C=2, D=3)))
    # 1. as written, relative to the current directory (OpenPCDet runs from tools/)
    _write_yaml(str(cfgs / "cwd.yaml"), dict(X=dict(_BASE_CONFIG_="cfgs/dataset_configs/ds.yaml", B=dict(D=4))))
    monkeypatch.chdir(tmp_path / "tools")
    assert cfg_from_yaml_file("cfgs/cwd.yaml").X == dict(_BASE_CONFIG_="cfgs/dataset_configs/ds.yaml", A=1,
                                                         B=dict(C=2, D=4))
    # 2. not found from the current directory: relative to the including file
    _write_yaml(str(cfgs / "beside.yaml"), dict(_BASE_CONFIG_="dataset_configs/ds.yaml", A=5))
    monkeypatch.chdir(tmp_path)
    cfg = cfg_from_yaml_file(str(cfgs / "beside.yaml"))
    assert cfg.A == 5 and cfg.B.C == 2
    # neither: the error names both paths it tried
    _write_yaml(str(cfgs / "broken.yaml"), dict(_BASE_CONFIG_="cfgs/dataset_configs/none.yaml"))
    with pytest.raises(FileNotFoundError) as e:
        cfg_from_yaml_file(str(cfgs / "broken.yaml"))
    assert str(tmp_path / "cfgs" / "dataset_configs" / "none.yaml") in str(e.value)
    assert str(cfgs / "cfgs" / "dataset_configs" / "none.yaml") in str(e.value)


# --------------------------------------------------------------------------------------------------- command (CPU)
@pytest.mark.parametrize("key,value,supported", [("DATA_CONFIG.DATASET", "KittiDataset", "NuScenesDataset"),
                                                 ("MODEL.DENSE_HEAD.NAME", "FrustumProposerOGKITTI", "FrustumProposerOG")])
def test_unsupported_configs_are_refused(tools_dir, capsys, key, value, supported):
    from findnpropagate_b200 import extract_pseudo_labels as cli
    with pytest.raises(SystemExit) as e:
        cli.main(["--cfg_file", HEAD, "--folder", "out", "--set", key, value])
    assert e.value.code == 1
    err = capsys.readouterr().err
    assert value in err and ("runs %s on" % supported in err or "reads %s" % supported in err), err
    assert not os.path.exists("out")


def test_unknown_set_key_exits_with_its_name(tools_dir, capsys):
    from findnpropagate_b200 import extract_pseudo_labels as cli
    with pytest.raises(SystemExit) as e:
        cli.main(["--cfg_file", HEAD, "--folder", "out", "--set", "DATA_CONFIG.NOPE", "1"])
    assert e.value.code == 1 and "no key DATA_CONFIG.NOPE" in capsys.readouterr().err
    assert not os.path.exists("out")


def test_existing_folder_exits_before_loading_anything(tools_dir, capsys):
    from findnpropagate_b200 import extract_pseudo_labels as cli
    os.makedirs("out")
    with open("out/keep.txt", "w") as f:
        f.write("x")
    before = os.stat("out/keep.txt").st_mtime_ns
    # a config that does not exist: the folder check comes first
    with pytest.raises(SystemExit) as e:
        cli.main(["--cfg_file", "cfgs/missing.yaml", "--folder", "out"])
    assert e.value.code == 1
    assert "out already exists" in capsys.readouterr().out
    assert os.listdir("out") == ["keep.txt"] and os.stat("out/keep.txt").st_mtime_ns == before


def test_failed_frame_check(tmp_path, monkeypatch):
    """A deleted LiDAR file, a frame missing from the GLIP predictions and (MAX_SWEEPS > 1) a missing sweep file."""
    from findnpropagate_b200 import extract_pseudo_labels as cli
    from findnpropagate_b200 import proposer
    frames = _frames("tiny", 4)
    tools = _write_tree(tmp_path, frames, glip_frames=[f for i, f in enumerate(frames) if i != 2])
    monkeypatch.chdir(tools)
    nusc = tmp_path / NUSC
    infos = pickle.load(open(nusc / INFOS, "rb"))
    infos[3]["sweeps"] = [dict(lidar_path="samples/LIDAR_TOP/gone.bin", transform_matrix=None, time_lag=0.05)]
    pickle.dump(infos, open(nusc / INFOS, "wb"))
    os.remove(nusc / infos[0]["lidar_path"])
    glip = proposer.PreprocessedGLIP()             # the reference's default paths, relative to tools/
    feed = cli.build_feed(cli.load_config(HEAD))
    assert [cli.check_frame(feed, glip, info) for info in feed.infos] == [cli.LIDAR_MISSING, 0, cli.IMAGE_NOT_PREDICTED, 0]
    feed = cli.build_feed(cli.load_config(HEAD, ["DATA_CONFIG.MAX_SWEEPS", "2"]))
    assert feed.max_sweeps == 2
    assert [cli.check_frame(feed, glip, info) for info in feed.infos] == [cli.LIDAR_MISSING, 0, cli.IMAGE_NOT_PREDICTED,
                                                                           cli.SWEEP_MISSING]


def test_build_feed_reads_the_config(tools_dir):
    from findnpropagate_b200 import extract_pseudo_labels as cli
    feed = cli.build_feed(cli.load_config(HEAD))
    assert feed.training and len(feed) == 3 and feed.max_sweeps == 1
    assert os.path.samefile(feed.root, os.path.join(tools_dir, "..", NUSC))
    assert feed.range.tolist() == [-54.0, -54.0, -5.0, 54.0, 54.0, 3.0]
    assert feed.final_dim == (900, 1600) and feed.resize_lim_test == (1.0, 1.0)


def test_help_runs_without_a_gpu():
    r = subprocess.run([sys.executable, "-m", "findnpropagate_b200.extract_pseudo_labels", "--help"], cwd=ROOT,
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    for flag in ("--cfg_file", "--folder", "--batch_frames", "--workers", "--set", "--nms_thresh"):
        assert flag in r.stdout


# --------------------------------------------------------------------------------------------------- GPU
def _library_run(base, frames, params, detector=None, box_format="xyxy", nms_thresh=None):
    """What the command wires up, called directly: SeekerEngine.run over the training-mode feed's frames."""
    from findnpropagate_b200 import nuscenes_feed, proposer
    from findnpropagate_b200.seeker import SeekerEngine
    feed = nuscenes_feed.NuScenesFeed(os.path.join(str(base), NUSC), INFOS, max_sweeps=1, training=True)
    det = detector or proposer.PreprocessedGLIP(os.path.join(str(base), GLIP_PTH), os.path.join(str(base), GLIP_META))
    eng = SeekerEngine(params, device="cuda:0", box_format=box_format)
    return eng.run([feed.frame_input(i, det)[0] for i in range(len(frames))], with_recall=True, nms_thresh=nms_thresh)


def _load(folder, frame):
    return torch.load(os.path.join(str(folder), frame.frame_id.replace(".", "_") + ".pth"), map_location="cpu")


def _assert_file_equals(folder, frame, pred):
    saved = _load(folder, frame)
    assert isinstance(saved, list) and len(saved) == 1
    s = saved[0]
    assert s["pred_boxes"].dtype == torch.float32 and s["pred_scores"].dtype == torch.float32
    assert s["pred_labels"].dtype == torch.int32
    assert np.array_equal(s["pred_boxes"].numpy().view(np.uint32), np.asarray(pred["pred_boxes"], np.float32).reshape(-1, 7).view(np.uint32))
    assert np.array_equal(s["pred_scores"].numpy().view(np.uint32), np.asarray(pred["pred_scores"], np.float32).view(np.uint32))
    assert np.array_equal(s["pred_labels"].numpy(), pred["pred_labels"])


@pytest.fixture
def cfg1_tree(tmp_path, monkeypatch):
    frames = _frames("cfg1", 5)
    tools = _write_tree(tmp_path, frames)
    monkeypatch.chdir(tools)
    return tmp_path, frames


@pytest.mark.gpu
def test_command_equals_the_library(cfg1_tree, capsys):
    from findnpropagate_b200 import extract_pseudo_labels as cli
    base, frames = cfg1_tree
    ref = _library_run(base, frames, synth.seeker_params(synth.CONFIGS["cfg1"]))
    got = cli.main(["--cfg_file", HEAD, "--folder", "../out", "--batch_frames", "2", "--workers", "2"])
    assert got["frames"] == 5 and got["failed"] == 0
    assert {k: got["recall"][k] for k in ref["recall"]} == ref["recall"] and got["recall"]["gt"] > 0
    for f, pred in zip(frames, ref["frames"]):
        _assert_file_equals(base / "out", f, pred)
    assert len(os.listdir(base / "out")) == 5
    assert sum(p["pred_boxes"].shape[0] for p in ref["frames"]) > 0
    out = capsys.readouterr().out
    assert "frames written: 5" in out and "failed frames: 0" in out and "AR@0.5" in out
    assert json.loads(out.split("recall counters: ")[1].splitlines()[0]) == got["recall"]


@pytest.mark.gpu
def test_missing_lidar_file_is_skipped_and_counted(cfg1_tree, capsys):
    from findnpropagate_b200 import extract_pseudo_labels as cli
    base, frames = cfg1_tree
    ref = _library_run(base, frames, synth.seeker_params(synth.CONFIGS["cfg1"]))
    os.remove(base / NUSC / "samples" / "LIDAR_TOP" / (frames[2].frame_id + ".bin"))
    got = cli.main(["--cfg_file", HEAD, "--folder", "../out", "--batch_frames", "2"])
    assert got["frames"] == 4 and got["failed"] == 1
    assert got["failed_frames"] == [(frames[2].frame_id, cli.FAILURES[cli.LIDAR_MISSING])]
    assert "skipped frame %s" % frames[2].frame_id in capsys.readouterr().out
    assert not os.path.exists(base / "out" / (frames[2].frame_id.replace(".", "_") + ".pth"))
    assert len(os.listdir(base / "out")) == 4
    for i, (f, pred) in enumerate(zip(frames, ref["frames"])):
        if i != 2:
            _assert_file_equals(base / "out", f, pred)


@pytest.mark.gpu
def test_per_camera_coco_results_xywh(cfg1_tree):
    """PREDS_PATHS: one COCO result file per camera view, BOX_FORMAT xywh (PreprocessedDetector)."""
    from findnpropagate_b200 import extract_pseudo_labels as cli
    from findnpropagate_b200 import proposer
    base, frames = cfg1_tree
    paths = []
    for c, cam in enumerate(synth.CAM_NAMES):
        images, anns = [], []
        for f in frames:
            images.append(dict(id=len(images), file_name=f.image_paths[c]))
            for b, l, s in zip(f.det_boxes[f.det_cam_idx == c], f.det_labels[f.det_cam_idx == c],
                               f.det_scores[f.det_cam_idx == c]):
                anns.append(dict(id=len(anns), image_id=images[-1]["id"], category_id=int(l), score=float(s),
                                 bbox=[float(b[0]), float(b[1]), float(b[2] - b[0]), float(b[3] - b[1])]))
        paths.append(str(base / "data" / "coco" / ("results_%s.json" % cam)))
        os.makedirs(os.path.dirname(paths[-1]), exist_ok=True)
        json.dump(dict(images=images, annotations=anns,
                       categories=[dict(id=i + 1, name=n) for i, n in enumerate(synth.CLASS_NAMES)]), open(paths[-1], "w"))
    params = synth.seeker_params(synth.CONFIGS["cfg1"])
    _write_yaml(HEAD, _head_cfg(params, PREDS_PATH="../data/coco/results_", PREDS_PATHS=paths, BOX_FORMAT="xywh"))
    got = cli.main(["--cfg_file", HEAD, "--folder", "../out", "--batch_frames", "3"])
    ref = _library_run(base, frames, params, detector=proposer.PreprocessedDetector(paths, synth.CLASS_NAMES),
                       box_format="xywh")
    assert got["frames"] == 5 and got["failed"] == 0
    assert {k: got["recall"][k] for k in ref["recall"]} == ref["recall"]
    for f, pred in zip(frames, ref["frames"]):
        _assert_file_equals(base / "out", f, pred)
    assert sum(p["pred_boxes"].shape[0] for p in ref["frames"]) > 0


@pytest.mark.gpu
def test_nms_thresh_equals_extract_nuscenes(cfg1_tree, monkeypatch):
    from findnpropagate_b200 import extract, extract_pseudo_labels as cli, nuscenes_feed, proposer
    from findnpropagate_b200.seeker import SeekerEngine
    base, frames = cfg1_tree
    params = synth.seeker_params(synth.CONFIGS["cfg1"])
    run, seen = extract.extract_nuscenes, []

    def spy(*a, **k):
        seen.append(k.get("nms_thresh"))
        return run(*a, **k)
    monkeypatch.setattr(extract, "extract_nuscenes", spy)
    got = cli.main(["--cfg_file", HEAD, "--folder", "../out", "--nms_thresh", "0.1", "--batch_frames", "2"])
    assert seen == [0.1]
    feed = nuscenes_feed.NuScenesFeed(base / NUSC, INFOS, max_sweeps=1, training=True)
    merged, total, ar = run(feed, proposer.PreprocessedGLIP(), SeekerEngine(params, device="cuda:0"), batch_frames=2,
                            nms_thresh=0.1)
    assert got["recall"] == total and got["ar"] == ar
    for f, pred in zip(frames, merged):
        _assert_file_equals(base / "out", f, pred)


@pytest.mark.gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_processes_under_nccl(cfg1_tree):
    from findnpropagate_b200 import extract_pseudo_labels as cli
    base, frames = cfg1_tree
    one = cli.main(["--cfg_file", HEAD, "--folder", "../one", "--batch_frames", "2"])
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT] + [p for p in [os.environ.get("PYTHONPATH")] if p]))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc_per_node", "2", "-m",
                        "findnpropagate_b200.extract_pseudo_labels", "--cfg_file", HEAD, "--folder", "../two",
                        "--batch_frames", "2"], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.count("frames written: 5") == 1             # rank 0 prints, rank 1 does not
    assert json.loads(r.stdout.split("recall counters: ")[1].splitlines()[0]) == one["recall"]
    assert sorted(os.listdir(base / "two")) == sorted(os.listdir(base / "one")) and len(os.listdir(base / "one")) == 5
    for f in frames:
        a, b = _load(base / "one", f)[0], _load(base / "two", f)[0]
        for k in ("pred_boxes", "pred_scores", "pred_labels"):
            assert a[k].dtype == b[k].dtype and np.array_equal(a[k].numpy().view(np.uint8), b[k].numpy().view(np.uint8))
