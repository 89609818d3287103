"""CPU tests of the host-side logic and of the C-ABI library surface (no compute calls)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from findnpropagate_b200 import nms2d, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_and_exports_every_declared_symbol():
    from findnpropagate_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "fnp.h")).read()
    declared = set(re.findall(r"^(?:int|size_t|const char \*)\s*(fnp_[a-z0-9_]+)\s*\(", hdr, re.M))
    assert declared, "no declarations parsed"
    for name in sorted(declared):
        assert hasattr(_lib.lib, name), "libfnp_sm100.so does not export %s" % name
    assert set(_lib.EXPORTED) == declared
    assert _lib.lib.fnp_version().startswith(b"fnp-sm100a")
    assert _lib.lib.fnp_nms_workspace_bytes(1000) >= 1000 * 16 * 8


def test_struct_layout_matches_header():
    from findnpropagate_b200 import _lib
    # 22 x 4-byte fields, in the header's order
    assert ctypes.sizeof(_lib.SeekerCfg) == 88
    hdr = open(os.path.join(ROOT, "include", "fnp.h")).read()
    cbody = hdr[hdr.index("typedef struct fnp_seeker_cfg"):hdr.index("} fnp_seeker_cfg;")]
    cbody = re.sub(r"/\*.*?\*/", "", cbody, flags=re.S)
    cnames = [n for grp in re.findall(r"(?:int32_t|float)\s+([a-z_0-9,\s]+);", cbody) for n in re.split(r",\s*", grp.strip())]
    assert cnames == [f[0] for f in _lib.SeekerCfg._fields_]
    body = hdr[hdr.index("typedef struct fnp_seeker_batch"):hdr.index("} fnp_seeker_batch;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = re.findall(r"[\*\s]([a-z_0-9]+)(?:,\s*([a-z_0-9]+))?;", body)
    flat = [n for pair in names for n in pair if n]
    assert flat == [f[0] for f in _lib.SeekerBatch._fields_]


def test_ops_refuse_cpu_tensors():
    from findnpropagate_b200.pcdet_ops import iou3d_nms_utils, roiaware_pool3d_utils
    with pytest.raises(RuntimeError):
        roiaware_pool3d_utils.points_in_boxes_gpu(torch.zeros(1, 4, 3), torch.zeros(1, 2, 7))
    with pytest.raises(RuntimeError):
        iou3d_nms_utils.boxes_iou_bev(torch.zeros(2, 7), torch.zeros(2, 7))
    from findnpropagate_b200.seeker import SeekerEngine
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):
            SeekerEngine(synth.seeker_params(synth.CONFIGS["tiny"]))


def test_nms2d_matches_torchvision():
    from torchvision.ops import batched_nms
    rng = np.random.default_rng(0)
    for trial in range(60):
        D = int(rng.integers(0, 40))
        b = rng.uniform(0, 1500, (D, 2)).astype(np.float32)
        boxes = np.concatenate([b, b + rng.uniform(2, 400, (D, 2)).astype(np.float32)], 1)
        for _ in range(D // 3):
            i, j = rng.integers(0, D, 2)
            boxes[j] = boxes[i] + rng.normal(0, 3, 4).astype(np.float32)
        scores = rng.uniform(0, 1, D).astype(np.float32)
        if D > 4:
            scores[1] = scores[3]
        labels = rng.integers(1, 4, D)
        cam = rng.integers(0, 6, D)
        frame = rng.integers(0, 3, D)
        got = list(nms2d.frustum_candidates(boxes, labels, scores, frame, cam, 0.4, 0.45))
        ref = []
        for f in range(3):
            for c in nms2d.IMAGE_ORDER:
                m = np.flatnonzero((cam == c) & (frame == f))
                if len(m) == 0:
                    continue
                sel = batched_nms(torch.from_numpy(boxes[m]), torch.from_numpy(scores[m]),
                                  torch.from_numpy(labels[m]), 0.4).numpy()
                ref += [m[s] for s in sel if not (scores[m][s] < np.float32(0.45))]
        assert got == ref


def test_tables_match_reference_constructor(golden_dir):
    from findnpropagate_b200 import seeker
    g = np.load(os.path.join(golden_dir, "seeker_cfg1_0.npz"))
    bb, bc = seeker.build_tables(seeker.resolve_params(synth.seeker_params(synth.CONFIGS["cfg1"])))
    assert np.array_equal(bb.numpy(), g["base_boxes"])
    assert np.array_equal(bc.numpy(), g["base_corners"])


def test_synth_frame_is_deterministic_and_well_formed(golden_dir):
    g = np.load(os.path.join(golden_dir, "seeker_tiny_0.npz"))
    f = synth.make_frame(0, synth.CONFIGS["tiny"])
    assert f.points.dtype == np.float32 and f.points.shape[1] == 5
    assert f.lidar2image.shape == (6, 4, 4) and f.det_boxes.shape[1] == 4
    assert np.allclose(f.points, g["points"], atol=1e-4)
    assert np.array_equal(f.det_labels, g["det_labels"])
    bd = synth.collate([f, f])
    assert bd["points"].shape == (2 * f.points.shape[0], 6) and bd["batch_size"] == 2
    assert set(np.unique(bd["points"][:, 0])) == {0.0, 1.0}


def test_unsupported_options_raise():
    from findnpropagate_b200 import seeker
    with pytest.raises(NotImplementedError):
        seeker.resolve_params(dict(topk=0, nms_3d=0, dst_w=0))
    for bad in (dict(aln_w=0.1), dict(nms_3d=0.5), dict(search_depth=0.0)):
        with pytest.raises(NotImplementedError):
            seeker.resolve_params(dict(dict(nms_3d=0), **bad))
    # the optional terms of SURVEY.md 8 row f3 are accepted
    p = seeker.resolve_params(dict(nms_3d=0, dst_w=0.2, ego_w=0.1, occl_w=0.3, search_depth=4.0, MULT=True,
                                   OCCL_MULT=True, MULTICAM_IOU=True))
    assert p["MULT"] and p["search_depth"] == 4.0


def test_host_pack_xyz_gathers_the_columns():
    """fnp_host_pack_xyz[_begin/_wait]: x,y,z of every row into a contiguous (rows,3) table, any
    stride / offset / thread count, empty input, and bad arguments rejected."""
    from findnpropagate_b200 import _lib
    rng = np.random.default_rng(3)
    for rows, stride, off, nt in ((0, 5, 0, 4), (1, 3, 0, 1), (1001, 5, 0, 3), (4097, 6, 1, 16), (50000, 5, 0, 7)):
        src = rng.random((rows, stride), dtype=np.float32)
        dst = np.full((rows, 3), -1, np.float32)
        assert _lib.lib.fnp_host_pack_xyz(src.ctypes.data, rows, stride, off, dst.ctypes.data, nt) == 0
        assert np.array_equal(dst, src[:, off:off + 3])
    src = rng.random((1000, 5), dtype=np.float32)
    a, b = np.empty((1000, 3), np.float32), np.empty((1000, 3), np.float32)
    t1 = _lib.lib.fnp_host_pack_xyz_begin(src.ctypes.data, 1000, 5, 0, a.ctypes.data, 2)
    t2 = _lib.lib.fnp_host_pack_xyz_begin(src.ctypes.data, 1000, 5, 2, b.ctypes.data, 2)
    assert t1 >= 0 and t2 >= 0 and t1 != t2
    assert _lib.lib.fnp_host_pack_wait(t2) == 0 and _lib.lib.fnp_host_pack_wait(t1) == 0
    assert np.array_equal(a, src[:, :3]) and np.array_equal(b, src[:, 2:5])
    assert _lib.lib.fnp_host_pack_wait(t1) == -1                       # already collected
    assert _lib.lib.fnp_host_pack_xyz(src.ctypes.data, 10, 2, 0, a.ctypes.data, 1) == -1      # stride < 3
    assert _lib.lib.fnp_host_pack_xyz(src.ctypes.data, 10, 5, 3, a.ctypes.data, 1) == -1      # columns past the row
    assert _lib.lib.fnp_host_pack_xyz(None, 10, 5, 0, a.ctypes.data, 1) == -1


def test_host_nms_order_equals_lexsort():
    """fnp_host_nms_order: per frame, descending score, ties by index."""
    from findnpropagate_b200 import _lib
    rng = np.random.default_rng(5)
    for n_frames in (0, 1, 7, 64):
        counts = rng.integers(0, 40, n_frames)
        fcs = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
        F = int(fcs[-1])
        score = rng.choice(np.linspace(0.45, 0.95, 23).astype(np.float32), F)       # many ties
        frame = np.repeat(np.arange(n_frames), counts)
        order = np.full(max(F, 1), -7, np.int32)
        assert _lib.lib.fnp_host_nms_order(score.ctypes.data, fcs.ctypes.data, n_frames, order.ctypes.data) == 0
        ref = np.lexsort((np.arange(F), -score.astype(np.float64), frame)).astype(np.int32)
        assert np.array_equal(order[:F], ref)


def test_host_pack_xyz_multi_gathers_segments_back_to_back():
    """fnp_host_pack_xyz_multi_begin: per-frame pieces of the point table -> one (rows,3) table,
    including empty pieces, pieces shorter than a thread share, and odd alignments."""
    import ctypes as C
    from findnpropagate_b200 import _lib
    rng = np.random.default_rng(11)
    for sizes, stride, off, nt in (([5, 0, 1, 1000, 3, 77], 5, 0, 4), ([4096, 4097, 1], 5, 1, 7), ([0, 0], 5, 0, 2),
                                   ([333] * 9, 6, 2, 16), ([2], 3, 0, 5)):
        segs = [rng.random((n, stride), dtype=np.float32) for n in sizes]
        rows = sum(sizes)
        dst = np.full((max(rows, 1), 3), -1, np.float32)
        ptrs = (C.c_void_p * len(segs))(*[s.ctypes.data for s in segs])
        nrow = (C.c_int64 * len(segs))(*sizes)
        t = _lib.lib.fnp_host_pack_xyz_multi_begin(ptrs, nrow, len(segs), stride, off, dst.ctypes.data, nt)
        assert t >= 0 and _lib.lib.fnp_host_pack_wait(t) == 0
        ref = np.concatenate([s[:, off:off + 3] for s in segs]) if rows else np.zeros((0, 3), np.float32)
        assert np.array_equal(dst[:rows], ref)


def test_batch_planner_in_c_equals_the_numpy_path():
    """SeekerEngine.plan (one fnp_host_plan call over the frames' prepared records) against plan_flat (numpy +
    fnp_host_select_candidates on flat arrays): every array of the plan, for xyxy / xywh boxes, topk 1 and 3,
    frames without detections, and an empty batch."""
    from findnpropagate_b200.seeker import FrameInput, SeekerEngine
    cfg = synth.SynthConfig("plan", 8, 180, 1, 40, 16, 6, 1)
    sf = [synth.make_frame(i, cfg) for i in range(6)]
    fis = [FrameInput(points=f.points, lidar2image=f.lidar2image, camera2lidar=f.camera2lidar,
                      camera_intrinsics=f.camera_intrinsics, det_boxes=f.det_boxes, det_labels=f.det_labels,
                      det_scores=f.det_scores, det_cam_idx=f.det_cam_idx, gt_boxes=f.gt_boxes) for f in sf]
    fis[2].det_boxes, fis[2].det_labels = np.zeros((0, 4), np.float32), np.zeros(0, np.int64)
    fis[2].det_scores, fis[2].det_cam_idx = np.zeros(0, np.float32), np.zeros(0, np.int64)
    batch = [fis[i % 6] for i in range(17)]
    for topk, fmt in ((1, "xyxy"), (3, "xywh")):
        eng = SeekerEngine.host_planner(dict(synth.seeker_params(cfg), topk=topk), box_format=fmt)
        for frames in (batch, batch[:1], [fis[2]], []):
            a, b = eng.plan(frames, stride=3), eng.plan_flat(frames, stride=3)
            assert a["F"] == b["F"] and (a["F"] > 0 or len(frames) < 2)
            for k, vb in b.items():
                va = a[k]
                if isinstance(vb, np.ndarray):
                    assert np.array_equal(np.asarray(va), vb), k
                    assert va.dtype == vb.dtype or k == "cand_det", (k, va.dtype, vb.dtype)
                else:
                    assert va == vb, (k, va, vb)
    # the prepared record follows the fields: assigning one drops it
    p0 = fis[0].prepare()
    assert fis[0].prepare() is p0
    fis[0].det_scores = fis[0].det_scores.copy()
    assert fis[0]._prep is None and fis[0].prepare() is not p0


def test_cpu_op_box_constants_reproduce_the_reference_cpu_op(ref_ops, golden_dir):
    """fnp_host_prep_boxes_cpu (the host half of the device-executed points_in_boxes_cpu): with its constants, the
    rounded fp32 arithmetic the device kernel performs -- emulated here in numpy, one rounding per operation --
    gives the reference-compiled CPU op's matrix bit for bit, also for points within a few ulp of dx/2 + 1e-2.
    Without the compiled op: its matrix on the stored inputs (tests/golden), and the oracle's port of it on these."""
    import ctypes as C
    import oracle as O
    from findnpropagate_b200 import _lib

    def emulated(boxes, pts):
        n = boxes.shape[0]
        prep = np.zeros((n, 8), np.float32)
        assert _lib.lib.fnp_host_prep_boxes_cpu(C.c_void_p(boxes.ctypes.data), C.c_void_p(prep.ctypes.data), n) == 0
        f = np.float32
        sx = (pts[None, :, 0] - prep[:, None, 0]).astype(f)
        sy = (pts[None, :, 1] - prep[:, None, 1]).astype(f)
        sz = (pts[None, :, 2] - prep[:, None, 2]).astype(f)
        cosa, sina = prep[:, None, 4], prep[:, None, 5]
        lxx = ((sx * cosa).astype(f) + (sy * -sina).astype(f)).astype(f)
        lyy = ((sx * sina).astype(f) + (sy * cosa).astype(f)).astype(f)
        inside = ~(np.abs(sz) > prep[:, None, 3]) & (np.abs(lxx) <= prep[:, None, 6]) & (np.abs(lyy) <= prep[:, None, 7])
        return inside.astype(np.int32)

    g = np.load(os.path.join(golden_dir, "ops_cpu_reference.npz"))
    assert np.array_equal(emulated(np.ascontiguousarray(g["boxes"]), g["pts"]), g["pib_cpu"])
    rng = np.random.default_rng(3)
    n = 40
    boxes = np.zeros((n, 7), np.float32)
    boxes[:, :3] = rng.uniform(-20, 20, (n, 3))
    boxes[:, 3:6] = rng.uniform(0.3, 12, (n, 3))
    boxes[:, 6] = rng.uniform(-7, 7, n)
    k = rng.integers(0, n, 4000)
    b = boxes[k].astype(np.float64)
    eps = np.concatenate([rng.uniform(-0.012, 0.012, 2000), 0.01 + rng.integers(-6, 7, 2000) * 1e-7])
    sgn = rng.choice([-1.0, 1.0], 4000)
    lx, ly = sgn * (b[:, 3] / 2 + eps), rng.uniform(-0.45, 0.45, 4000) * b[:, 4]
    ca, sa = np.cos(b[:, 6]), np.sin(b[:, 6])
    pts = np.stack([b[:, 0] + lx * ca - ly * sa, b[:, 1] + lx * sa + ly * ca, b[:, 2] + rng.uniform(-0.5, 0.5, 4000) * b[:, 5]], 1)
    pts = np.concatenate([pts, rng.uniform(-25, 25, (4000, 3))]).astype(np.float32)
    if ref_ops is not None:
        want = torch.zeros((n, pts.shape[0]), dtype=torch.int32)
        ref_ops[0].points_in_boxes_cpu(torch.from_numpy(boxes), torch.from_numpy(pts), want)
        want = want.numpy()
    else:
        want = O.points_in_boxes_cpu(pts, boxes)
    got = emulated(boxes, pts)
    assert np.array_equal(got, want), int((got != want).sum())
    assert want.sum() > 2000


def test_shipped_yaml_params_equal_the_hard_coded_ones():
    """MODEL.DENSE_HEAD.PARAMS of the reference's tools/cfgs/nuscenes_box_seeker_proposals.yaml against
    synth.seeker_params (the option set every test and the bench run), the head's constructor defaults
    (frustum_proposals_v1.py:146-148) filling the keys the YAML leaves out.  Needs the reference tree: runs in the
    build container, skipped on the GPU box."""
    import yaml
    from findnpropagate_b200.seeker import DEFAULTS, resolve_params
    path = "/root/reference/tools/cfgs/nuscenes_box_seeker_proposals.yaml"
    if not os.path.exists(path):
        pytest.skip("reference tree not present")
    head = yaml.safe_load(open(path))["MODEL"]["DENSE_HEAD"]
    assert head["NAME"] == "FrustumProposerOG" and head["PREDS_PATH"] == "PreprocessedGLIP" and head["BOX_FORMAT"] == "xyxy"
    shipped = head["PARAMS"]
    cfg1 = synth.CONFIGS["cfg1"]                     # BASELINE.json configs[0]: the shipped grid
    mine = synth.seeker_params(cfg1)
    for k, v in shipped.items():
        assert mine[k] == v, (k, mine[k], v)
    # keys the YAML omits fall back to the constructor defaults, as in the reference (:167-196)
    for k in ("num_mags", "num_rotations"):
        assert k not in shipped and mine[k] == DEFAULTS[k]
    full = resolve_params(shipped)
    assert (full["num_mags"], full["num_rotations"], full["num_sizes"]) == (cfg1.num_mags, cfg1.num_rotations, cfg1.num_sizes)
    assert full["max_dist"] == 50 and full["topk"] == 1


@pytest.mark.skipif(not os.path.isdir("/root/reference/pcdet"), reason="needs the reference tree (build container only)")
def test_aln_w_raises_in_the_reference_itself():
    """PARAMS aln_w is refused by this build (seeker.resolve_params) because it cannot run in the reference:
    frustum_proposals_v1.py:987 indexes the (P,3) frustum points with a (1,P) mask.  The reference head (CPU run of
    tools/ref_seeker.py, own process: it registers the reference modules globally) raises IndexError."""
    import subprocess
    import sys
    code = ("import sys; sys.path[:0] = [%r, %r, %r]\n"
            "import ref_seeker\nfrom findnpropagate_b200 import synth\n"
            "cfg = synth.CONFIGS['tiny']\n"
            "try:\n    ref_seeker.run([synth.make_frame(0, cfg)], dict(synth.seeker_params(cfg), aln_w=0.1), capture=False)\n"
            "    print('RAN')\nexcept IndexError as e:\n    print('INDEXERROR', e)\n") % (
        os.path.join(ROOT, "tools"), ROOT, os.path.join(ROOT, "oracle"))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300).stdout
    assert "INDEXERROR" in out and "shape of the mask" in out, out
