"""Every op-level kernel against the float64 geometry of fp64_geometry.py, at the sizes where the kernels' tiling
changes: the 256-box tile of points_in_boxes, 4096 boxes per segment in count_in_boxes, 16-box pairwise tiles, more
NMS mask words than scan threads above 16384 boxes, FNP_SEG_NMS_MAX boxes in one stage-4 segment, and the largest
frames the counters' shared memory takes.

Where the fp32 ops may round either way the inputs are kept out of it: points within UNDECIDED of a face are not
compared, and NMS and counter inputs are resampled until no float64 IoU lies within DELTA (plus the pair's fp32 bound)
of a threshold and no pair has a corner in the 1 cm margin band of the other box."""
import ctypes as C

import numpy as np
import pytest
import torch

import fp64_geometry as G
from findnpropagate_b200 import _lib, quality
from findnpropagate_b200.seeker import SeekerEngine
from test_ops_gpu import _boxes, _pair_boxes

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
UNDECIDED = 1e-4          # m: points this close to a face of a box that decides them are not compared
DELTA = 1e-3              # IoU: inputs are kept this far (plus the pair's fp32 bound) from every threshold
FNP_EINVAL = -1
THRESH = (0.3, 0.5, 0.7)
EDGES = (20.0, 30.0, 40.0)
N_CLASSES = 10


def _d(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _stream():
    return _lib.current_stream()


def _small_boxes(rng, n, half=48.0):
    """Boxes of 0.3 - 1.5 m by 0.3 - 1.5 m (dz 0.5 - 2 m) with centres in a (2 half)^2 m square at the origin."""
    b = np.zeros((n, 7))
    b[:, :2] = rng.uniform(-half, half, (n, 2))
    b[:, 2] = rng.uniform(-1, 1, n)
    b[:, 3:5] = rng.uniform(0.3, 1.5, (n, 2))
    b[:, 5] = rng.uniform(0.5, 2.0, n)
    b[:, 6] = rng.uniform(-np.pi, np.pi, n)
    return b.astype(np.float32).astype(np.float64)


def _wide_boxes(rng, n, half=45.0):
    """Boxes of the seeker's class priors with centres in a (2 half)^2 m square at the origin."""
    return _boxes(rng, n, centre=(0.0, 0.0, -0.5), spread=2 * half).astype(np.float64)


def _jitter(rng, src, pos=0.25, rel=0.15, yaw=0.15):
    """Copies of src moved, resized and turned a little: pairs with IoUs spread over (0, 1)."""
    b = src.copy()
    b[:, :3] += rng.normal(0, pos, (len(b), 3)) * [1, 1, 0.5]
    b[:, 3:6] *= rng.uniform(1 - rel, 1 + rel, (len(b), 3))
    b[:, 6] += rng.normal(0, yaw, len(b))
    return b.astype(np.float32).astype(np.float64)


def _bad_pairs(a, b, i, j, thresholds, three_d=False, normal=False):
    """Mask over the pairs (a[i], b[j]) whose fp32 result may fall on either side of a threshold: a corner in the
    margin band, or an IoU within DELTA plus its fp32 bound of one of the thresholds."""
    ov, m = G.overlap_bev(a[i], b[j])
    v = G.iou_from_overlap(a[i], b[j], ov, three_d)
    tol = DELTA + G.iou_tol(a[i], b[j], ov, three_d)
    bad = m | (np.abs(v[:, None] - np.asarray(thresholds)[None]) <= tol[:, None]).any(1)
    if normal:
        vn = G.iou_normal(a[i], b[j])
        bad |= (np.abs(vn[:, None] - np.asarray(thresholds)[None]) <= DELTA).any(1)
    return bad


def _resample_self(rng, boxes, thresholds, normal=False, half=48.0):
    """Redraw (anywhere in the square) a box of every bad pair within boxes until there is none; after the first
    pass only the pairs of redrawn boxes are evaluated again."""
    i, j = G.near_pairs(boxes)
    redo = np.unique(j[_bad_pairs(boxes, boxes, i, j, thresholds, normal=normal)])
    for _ in range(100):
        if not len(redo):
            return boxes
        boxes[redo] = _small_boxes(rng, len(redo), half)
        ri, j = G.near_pairs(boxes[redo], boxes)
        i = redo[ri]
        i, j = i[i != j], j[i != j]
        redo = np.unique(i[_bad_pairs(boxes, boxes, i, j, thresholds, normal=normal)])
    raise AssertionError("resampling did not converge")


# ------------------------------------------------------------------------------------------------ points in boxes
@pytest.mark.parametrize("T", [1, 255, 256, 257, 513])
def test_points_in_boxes_count_and_crop_vs_fp64(T):
    """points_in_boxes_gpu, fnp_count_in_boxes and fnp_crop_points_in_boxes on B = 3 frames of M = 3001 points (not a
    multiple of 256) and T boxes, across the 256-box tile and its early exit; overlapping boxes test first-match."""
    from findnpropagate_b200 import gt_database
    from findnpropagate_b200.pcdet_ops import roiaware_pool3d_utils as RP
    rng = np.random.default_rng(100 + T)
    B, M = 3, 3001
    boxes = np.stack([_boxes(rng, T) for _ in range(B)])
    k = T // 4
    boxes[:, T // 2:T // 2 + k] = boxes[:, :k] * [1, 1, 1, 0.8, 1.2, 1, 1]     # later boxes overlapping earlier ones
    pts = (rng.uniform(-0.5, 0.5, (B, M, 3)) * [10, 10, 3] + [14, 0, -0.5]).astype(np.float32)
    got = RP.points_in_boxes_gpu(_d(pts), _d(boxes)).cpu().numpy()
    tp4 = _d(np.concatenate([pts.reshape(-1, 3), np.zeros((B * M, 1), np.float32)], 1))
    tps, tbs = _d(np.arange(B + 1, dtype=np.int32) * M), _d(np.arange(B + 1, dtype=np.int32) * T)
    tb = _d(boxes.reshape(-1, 7))
    counts = torch.full((B * T,), -7, dtype=torch.int32, device=DEV)
    assert _lib.lib.fnp_count_in_boxes(tp4.data_ptr(), tps.data_ptr(), tb.data_ptr(), tbs.data_ptr(), B,
                                       counts.data_ptr(), _stream()) == 0
    counts = counts.cpu().numpy().reshape(B, T)
    crop, _, _ = gt_database.crop_points_in_boxes(_d(pts.reshape(-1, 3)), np.arange(B + 1) * M, tb,
                                                  _d(boxes.reshape(-1, 7)[:, :3].astype(np.float64)), np.arange(B + 1) * T)
    crop = crop.cpu().numpy().reshape(B, T)
    n_undecided = n_hit = n_box_decided = 0
    for f in range(B):
        idx, margin = G.points_in_boxes(pts[f], boxes[f])
        decided = np.abs(margin) > UNDECIDED
        n_undecided += int((~decided).sum())
        n_hit += int((idx[decided] >= 0).sum())
        assert np.array_equal(got[f][decided], idx[decided]), int((got[f] != idx)[decided].sum())
        # the crop assigns by the same predicate, first match, bit for bit
        assert np.array_equal(crop[f], np.bincount(got[f][got[f] >= 0], minlength=T))
        m = G.face_margin(pts[f], boxes[f])
        box_decided = (np.abs(m) > UNDECIDED).all(0)
        n_box_decided += int(box_decided.sum())
        assert np.array_equal(counts[f][box_decided], (m >= 0).sum(0)[box_decided])
    assert n_undecided < 0.001 * B * M and n_hit > 0.1 * B * M and n_box_decided >= 0.9 * B * T - 1


def test_count_in_boxes_covers_every_box_of_large_segments():
    """Segments of 4095, 4096, 4097 and 8193 boxes (the launch has 32 x 128 threads per segment) beside small and empty
    ones: every count is written (the sentinel is gone) and equals the float64 count where no point is undecided."""
    rng = np.random.default_rng(7)
    seg_box = [4095, 5, 4096, 0, 4097, 3, 8193]
    seg_pts = [400, 300, 0, 50, 350, 0, 500]
    boxes = [_boxes(rng, n) for n in seg_box]
    pts = [(rng.uniform(-0.5, 0.5, (n, 3)) * [10, 10, 3] + [14, 0, -0.5]).astype(np.float32) for n in seg_pts]
    tp4 = _d(np.concatenate([np.concatenate([p, np.zeros((len(p), 1), np.float32)], 1) for p in pts]))
    bs = np.cumsum([0] + seg_box).astype(np.int32)
    tps, tb, tbs = _d(np.cumsum([0] + seg_pts).astype(np.int32)), _d(np.concatenate(boxes)), _d(bs)
    counts = torch.full((int(bs[-1]),), -7, dtype=torch.int32, device=DEV)
    assert _lib.lib.fnp_count_in_boxes(tp4.data_ptr(), tps.data_ptr(), tb.data_ptr(), tbs.data_ptr(), len(seg_box),
                                       counts.data_ptr(), _stream()) == 0
    got = counts.cpu().numpy()
    unwritten = np.flatnonzero(got == -7)
    assert unwritten.size == 0, "%d boxes never written, the first at %d" % (unwritten.size, unwritten[:1].sum())
    for s in range(len(seg_box)):
        g = got[bs[s]:bs[s + 1]]
        if not seg_pts[s] or not seg_box[s]:
            assert (g == 0).all()
            continue
        m = G.face_margin(pts[s], boxes[s])
        decided = (np.abs(m) > UNDECIDED).all(0)
        assert decided.mean() > 0.95 and (g[decided] > 0).sum() > seg_box[s] // 4
        assert np.array_equal(g[decided], (m >= 0).sum(0)[decided])


# ------------------------------------------------------------------------------------------------ BEV overlap / IoU
def _overlap_case(n, m, seed):
    rng = np.random.default_rng(seed)
    a, b = _pair_boxes(rng, max(n, m, 16))
    a[:, 2] += rng.uniform(-1, 1, len(a)).astype(np.float32)
    return a[:n], b[:m]


def _check_bounds(a, b, got, exact, in_margin, three_d, what, record):
    """fp32 op values got against the float64 exact overlap of the pairs (a, b) (broadcast: a[:, None] with b[None],
    or aligned rows): the overlap itself when three_d is None, else the BEV (False) or 3D (True) IoU."""
    got = np.asarray(got, np.float64)
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    perim = np.maximum(2 * (a[..., 3] + a[..., 4]), 2 * (b[..., 3] + b[..., 4]))
    if three_d is None:
        want, tol = exact, G.overlap_tol(exact)
        hi = exact + 0.01 * perim + tol
    else:
        want, tol = G.iou_from_overlap(a, b, exact, three_d), G.iou_tol(a, b, exact, three_d)
        hi = G.iou_from_overlap(a, b, exact + 0.01 * perim + G.overlap_tol(exact), three_d) + 1e-6
    dev = got - want
    ok = ~in_margin
    assert (np.abs(dev) <= tol)[ok].all(), "%s: max deviation %g" % (what, np.abs(dev)[ok].max())
    assert (got <= hi)[in_margin].all() and (dev >= -tol)[in_margin].all(), what
    record[what] = max(record.get(what, 0.0), float(np.abs(dev)[ok].max(initial=0)))


_SIZES = [(1, 1), (1, 257), (257, 1), (15, 16), (16, 17), (17, 15), (255, 257), (257, 255), (16, 16), (2000, 1500)]


def test_pairwise_and_aligned_overlap_iou_vs_fp64():
    """fnp_boxes_overlap_bev, _iou_bev, _iou3d and the aligned overlap / IoU3D on the CPU test's inputs (identical,
    shifted and yaw 0 / pi/2 pairs among random ones), N, M in {1, 15, 16, 17, 255, 257} across the 16-box tiles, and
    one 2000 x 1500 call.  Pairs without in_margin lie within the fp64_geometry bounds; in_margin pairs no more than
    1 cm x the larger perimeter above the exact area.  Largest deviations from float64 (pairs without in_margin) seen on
    a B200 at 1000 W, printed with -s: overlap 3.6e-5 m^2, BEV IoU 1.0e-5, IoU3D 8.4e-6, aligned overlap 1.6e-5 m^2,
    aligned IoU3D 8.4e-6."""
    record = {}
    L = _lib.lib
    for s, (n, m) in enumerate(_SIZES):
        a, b = _overlap_case(n, m, 50 + s)
        exact, in_margin = G.pairwise(G.overlap_bev, a, b)
        ta, tb = _d(a), _d(b)
        for fn, three_d, what in ((L.fnp_boxes_overlap_bev, None, "overlap"), (L.fnp_boxes_iou_bev, False, "iou_bev"),
                                  (L.fnp_boxes_iou3d, True, "iou3d")):
            out = torch.full((n, m), -1.0, device=DEV)
            assert fn(ta.data_ptr(), tb.data_ptr(), out.data_ptr(), n, m, _stream()) == 0
            _check_bounds(a[:, None], b[None], out.cpu().numpy(), exact, in_margin, three_d, what, record)
        k = min(n, m)
        ov, in_margin = G.overlap_bev(a[:k], b[:k])
        for fn, three_d, what in ((L.fnp_boxes_aligned_overlap_bev, None, "aligned overlap"),
                                  (L.fnp_boxes_aligned_iou3d, True, "aligned iou3d")):
            out = torch.full((k,), -1.0, device=DEV)
            assert fn(ta.data_ptr(), tb.data_ptr(), out.data_ptr(), k, _stream()) == 0
            _check_bounds(a[:k], b[:k], out.cpu().numpy(), ov, in_margin, three_d, what, record)
    print("largest float64 deviations:", record)


# ------------------------------------------------------------------------------------------------ NMS
NMS_THRESH = (0.01, 0.1, 0.5)


@pytest.fixture(scope="module")
def nms_sets():
    """Per N: boxes in score order (a third are jittered copies of earlier boxes, so suppression chains form) with no
    rotated or axis-aligned IoU near a threshold, their near pairs with both IoUs, and a permutation to feed them in."""
    cache = {}

    def get(n):
        if n not in cache:
            rng = np.random.default_rng(n)
            sb = _small_boxes(rng, n)
            k = n // 3
            sb[n - k:] = _jitter(rng, sb[rng.integers(0, n - k, k)])
            sb = _resample_self(rng, sb, NMS_THRESH, normal=True)
            i, j = G.near_pairs(sb)
            cache[n] = (sb, i, j, G.iou_bev(sb[i], sb[j])[0], G.iou_normal(sb[i], sb[j]), rng.permutation(n))
        return cache[n]
    return get


@pytest.mark.parametrize("n", [16383, 16384, 16385, 20000])
@pytest.mark.parametrize("rotated", [True, False])
def test_nms_at_scale_vs_fp64_greedy(nms_sets, n, rotated):
    """nms_gpu / nms_normal_gpu at N around 16384, where the greedy scan has more mask words than its 256 threads,
    at thresholds 0.01, 0.1 and 0.5: the keep list equals the float64 greedy NMS exactly.  nms_normal_gpu is also
    checked against the C oracle (its rotated NMS is O(N^2) polygon clips: minutes at this size)."""
    import oracle as O
    from findnpropagate_b200.pcdet_ops import iou3d_nms_utils as IU
    sb, i, j, rot, nrm, perm = nms_sets(n)
    inv = np.argsort(perm)                           # input row of each score position
    boxes = np.ascontiguousarray(sb[perm], np.float32)
    scores = ((n - np.arange(n)) / n).astype(np.float32)[perm]
    tb, ts = _d(boxes), _d(scores)
    rows = G.sparse_rows(i, j, rot if rotated else nrm)
    for thr in NMS_THRESH:
        keep, _ = (IU.nms_gpu if rotated else IU.nms_normal_gpu)(tb, ts, thr)
        keep = keep.cpu().numpy()
        exp = inv[G.greedy_nms(rows, n, thr)]
        assert len(keep) == len(exp) and np.array_equal(keep, exp), (thr, len(keep), len(exp))
        assert len(exp) < n
        if not rotated and thr == 0.1:
            assert np.array_equal(O.nms_normal(boxes, scores, thr), exp)


def test_seg_nms_at_its_cap_vs_fp64_greedy():
    """fnp_seg_nms_rotated in one launch over segments of 0, 1, 63, 64, 65, 1023 and 1024 boxes with max_seg_boxes =
    FNP_SEG_NMS_MAX = 1024 (about 201 KB of shared memory), a score order and rows with valid = -1, as SeekerEngine
    passes them: each segment keeps what the float64 greedy NMS keeps.  1025 is refused."""
    rng = np.random.default_rng(11)
    segs = [0, 1, 63, 64, 65, 1023, 1024]
    thr_list = (0.1, 0.5)
    parts = []
    for n in segs:
        b = _small_boxes(rng, n, half=16.0)
        k = n // 3
        if k:
            b[n - k:] = _jitter(rng, b[rng.integers(0, n - k, k)])
        parts.append(_resample_self(rng, b, thr_list, half=16.0))
    boxes = np.concatenate(parts)
    start = np.cumsum([0] + segs)
    valid = np.where(rng.uniform(size=len(boxes)) < 0.15, -1, 0).astype(np.int32)
    scores = rng.permutation(len(boxes))
    order = np.concatenate([start[s] + np.argsort(-scores[start[s]:start[s + 1]], kind="stable")
                            for s in range(len(segs))]).astype(np.int32)
    tb, to, tv, ts = _d(boxes.astype(np.float32)), _d(order), _d(valid), _d(start.astype(np.int32))
    keep = torch.full((len(boxes),), 9, dtype=torch.uint8, device=DEV)
    call = lambda cap, thr: _lib.lib.fnp_seg_nms_rotated(tb.data_ptr(), None, to.data_ptr(), tv.data_ptr(), ts.data_ptr(),
                                                         len(segs), cap, C.c_float(thr), keep.data_ptr(), _stream())
    assert call(1025, 0.1) == FNP_EINVAL
    for thr in thr_list:
        assert call(1024, thr) == 0
        got = keep.cpu().numpy()
        n_removed = 0
        for s, n in enumerate(segs):
            src = order[start[s]:start[s + 1]]
            live = src[valid[src] >= 0]                 # in priority order
            i, j = G.near_pairs(boxes[live])
            v = G.iou_bev(boxes[live][i], boxes[live][j])[0]
            want = np.zeros(len(boxes), np.uint8)
            want[live[G.greedy_nms(G.sparse_rows(i, j, v), len(live), thr)]] = 1
            assert np.array_equal(got[start[s]:start[s + 1]], want[start[s]:start[s + 1]]), (thr, n)
            n_removed += len(live) - int(want.sum())
        assert n_removed > 50


# ------------------------------------------------------------------------------------------------ counters
def _near_edge(b):
    r = np.hypot(b[:, 0], b[:, 1])
    return (np.abs(r[:, None] - np.asarray(EDGES)[None]) <= 1e-3).any(1)


def _counter_frame(rng, K, n_gt):
    """One frame: (proposals (K, 7), labels (K,), valid (K,) bool, GT (n_gt, 8)).  Half the proposals are jittered
    copies of GT boxes (half of those with the GT's label); a proposal is redrawn while its 3D IoU with a GT box is
    near a threshold, a corner lies in the margin band, or its centre is within 1e-3 m of a range edge."""
    gt = np.zeros((n_gt, 8))
    gt[:, :7] = _wide_boxes(rng, n_gt)
    while _near_edge(gt).any():
        gt[_near_edge(gt), :7] = _wide_boxes(rng, int(_near_edge(gt).sum()))
    gt[:, 7] = rng.integers(1, N_CLASSES + 1, n_gt)
    src = rng.integers(0, n_gt, K)
    pred = _jitter(rng, gt[src, :7])
    rand = rng.uniform(size=K) < 0.5
    pred[rand] = _wide_boxes(rng, int(rand.sum()))
    label = np.where(rng.uniform(size=K) < 0.5, gt[src, 7], rng.integers(1, N_CLASSES + 1, K)).astype(np.int32)
    redo = np.arange(K)
    for _ in range(100):
        ri, j = G.near_pairs(pred[redo], gt)
        bad = redo[ri[_bad_pairs(pred[redo], gt, ri, j, THRESH, three_d=True)]]
        redo = np.union1d(bad, redo[_near_edge(pred[redo])])
        if not len(redo):
            return pred, label, rng.uniform(size=K) >= 0.1, gt
        pred[redo] = _wide_boxes(rng, len(redo))
    raise AssertionError("resampling did not converge")


def _upload(frames):
    cat = lambda xs, dt: np.ascontiguousarray(np.concatenate(xs), dt)
    return dict(pred=_d(cat([f[0] for f in frames], np.float32)), label=_d(cat([f[1] for f in frames], np.int32)),
                valid=_d(np.where(cat([f[2] for f in frames], bool), 0, -1).astype(np.int32)),
                pstart=_d(np.cumsum([0] + [len(f[1]) for f in frames]).astype(np.int32)),
                gt=_d(cat([f[3] for f in frames], np.float32)),
                gstart=_d(np.cumsum([0] + [len(f[3]) for f in frames]).astype(np.int32)))


def _fp64_ious(frames):
    return [G.pairwise(G.iou3d, f[0][f[2]], f[3][:, :7])[0] for f in frames]


@pytest.fixture(scope="module")
def counter_frames():
    cache = {}

    def get(K):
        if K not in cache:
            rng = np.random.default_rng(K)
            frames = [_counter_frame(rng, K, 200), _counter_frame(rng, 5, 3)]
            cache[K] = frames, _upload(frames), _fp64_ious(frames)
        return cache[K]
    return get


def _launch_old(fn, d, max_pred, max_gt, out):
    th = (C.c_float * len(THRESH))(*THRESH)
    return fn(d["pred"].data_ptr(), d["valid"].data_ptr(), d["pstart"].data_ptr(), d["gt"].data_ptr(),
              d["gstart"].data_ptr(), len(d["pstart"]) - 1, max_pred, max_gt, th, len(THRESH), out.data_ptr(), _stream())


def _launch_quality(spec, d, max_pred, max_gt, out):
    e = (C.c_float * len(spec.range_edges))(*spec.range_edges)
    th = (C.c_float * len(spec.thresh))(*spec.thresh)
    return _lib.lib.fnp_quality_counters(d["pred"].data_ptr(), 0, d["valid"].data_ptr(), 0, d["label"].data_ptr(),
                                         d["pstart"].data_ptr(), 1, d["gt"].data_ptr(), d["gstart"].data_ptr(),
                                         len(d["pstart"]) - 1, max_pred, max_gt, len(spec.class_names), e,
                                         len(spec.range_edges), th, len(spec.thresh), out.data_ptr(), _stream())


def _quality_spec():
    return quality.QualitySpec(["c%d" % k for k in range(1, N_CLASSES + 1)], EDGES, THRESH)


def test_recall_counters_at_the_shared_memory_limit(counter_frames):
    """(K + G) 64 + 4 G + 16 <= 200 KB: with G = 200, K = 2987 is accepted and 2988 refused.  The counters of a frame
    of that size equal the float64 restatement."""
    K, n_gt = 2987, 200
    assert (K + n_gt) * 64 + 4 * n_gt + 16 <= 200 * 1024 < (K + 1 + n_gt) * 64 + 4 * n_gt + 16
    frames, d, ious = counter_frames(K)
    out = torch.zeros(5 + 5 * len(THRESH), dtype=torch.int64, device=DEV)
    assert _launch_old(_lib.lib.fnp_recall_counters, d, K + 1, n_gt, out) == FNP_EINVAL
    assert _launch_old(_lib.lib.fnp_recall_counters, d, K, n_gt, out) == 0
    exp = G.recall_dict([(iou, f[3][:, 7]) for iou, f in zip(ious, frames)], THRESH)
    assert SeekerEngine.recall_dict(out.cpu().numpy(), THRESH) == exp
    assert 0 < exp["rcnn_0.7"] < exp["rcnn_0.3"] < exp["gt"]


def test_precision_counters_at_the_shared_memory_limit(counter_frames):
    """(K + G) 64 + 4 K + 16 <= 200 KB: with G = 200, K = 2823 is accepted and 2824 refused."""
    K, n_gt = 2823, 200
    assert (K + n_gt) * 64 + 4 * K + 16 <= 200 * 1024 < (K + 1 + n_gt) * 64 + 4 * (K + 1) + 16
    frames, d, ious = counter_frames(K)
    out = torch.zeros(1 + len(THRESH), dtype=torch.int64, device=DEV)
    assert _launch_old(_lib.lib.fnp_precision_counters, d, K + 1, n_gt, out) == FNP_EINVAL
    assert _launch_old(_lib.lib.fnp_precision_counters, d, K, n_gt, out) == 0
    exp = G.precision_counts(ious, THRESH)
    assert out.cpu().numpy().tolist() == exp.tolist()
    assert 0 < exp[3] < exp[1] < exp[0]


def test_quality_counters_at_the_shared_memory_limit(counter_frames):
    """fnp_quality_smem_bytes = 80 K + 76 G + 8 C R W + 16 <= 200 KB: with G = 200, 10 classes, 4 range bins and 3
    thresholds, K = 2341 is accepted and 2342 refused."""
    K, n_gt = 2341, 200
    spec = _quality_spec()
    assert spec.smem_bytes(K, n_gt) == 80 * K + 76 * n_gt + 8 * 10 * 4 * 7 + 16
    assert spec.smem_bytes(K, n_gt) <= 200 * 1024 < spec.smem_bytes(K + 1, n_gt)
    frames, d, ious = counter_frames(K)
    out = torch.zeros(spec.n_counters, dtype=torch.int64, device=DEV)
    assert _launch_quality(spec, d, K + 1, n_gt, out) == FNP_EINVAL
    assert _launch_quality(spec, d, K, n_gt, out) == 0
    exp = G.quality_counts([(iou, f[1][f[2]], f[0][f[2], :2], f[3][:, 7], f[3][:, :2]) for iou, f in zip(ious, frames)],
                           THRESH, EDGES, N_CLASSES)
    got = out.cpu().numpy()
    assert np.array_equal(got, exp)
    c = exp.reshape(2, N_CLASSES, len(EDGES) + 1, -1)
    assert (c[:, :, :, 0].sum(1) > 0).all() and c[0, :, :, 1 + len(THRESH):].sum() > 0


# ------------------------------------------------------------------------------------------------ degenerate sizes
def test_negative_and_zero_sizes_match_the_unfiltered_iou():
    """Rows with dx <= 0 or dy <= 0 among normal ones.  The counters and the stage-4 NMS dismiss far pairs with a
    bounding-circle test; for such rows they must still give what the same restatements give from boxes_iou3d_gpu /
    boxes_iou_bev, which clip every pair."""
    from findnpropagate_b200.pcdet_ops import iou3d_nms_utils as IU
    rng = np.random.default_rng(21)
    frames = []
    exposed = 0
    for f in range(3):
        n_gt, K = 30, 90
        gt = np.zeros((n_gt, 8))
        gt[:, :7] = _wide_boxes(rng, n_gt, half=30.0)
        gt[:, 7] = rng.integers(1, N_CLASSES + 1, n_gt)
        src = rng.integers(0, n_gt, K)
        pred = _jitter(rng, gt[src, :7])
        odd = np.arange(K) % 3 == 0
        ang = rng.uniform(-np.pi, np.pi, K)
        dist = rng.uniform(1.5, 3.5, K)
        pred[odd, 0] += (dist * np.cos(ang))[odd]
        pred[odd, 1] += (dist * np.sin(ang))[odd]
        kind = rng.integers(0, 4, K)
        pred[odd & (kind == 0), 3] *= -1
        pred[odd & (kind == 1), 4] *= -1
        pred[odd & (kind == 2), 3] = 0
        pred[odd & (kind == 3), 3:5] *= -1
        for b in (gt, pred):
            b[_near_edge(b), :2] *= 1.001
        label = rng.integers(1, N_CLASSES + 1, K).astype(np.int32)
        valid = rng.uniform(size=K) >= 0.1
        frames.append((pred, label, valid, gt))
        # pairs the old radius, tx + ty = dx/2 + dy/2 + 2e-2 (negative for dx < 0), dismissed though they overlap
        p32, g32 = pred.astype(np.float32), gt[:, :7].astype(np.float32)
        iou = IU.boxes_iou3d_gpu(_d(p32), _d(g32)).cpu().numpy()
        r = (p32[:, 3:4] + p32[:, 4:5]) / 2 + 0.02 + ((g32[:, 3] + g32[:, 4]) / 2 + 0.02)[None] + 0.1
        d2 = (p32[:, 0:1] - g32[None, :, 0]) ** 2 + (p32[:, 1:2] - g32[None, :, 1]) ** 2
        exposed += int(((d2 > 1.0001 * r * r) & (iou != 0) & valid[:, None]).sum())
    assert exposed >= 5
    d = _upload(frames)
    n_pred, n_gt = max(len(f[1]) for f in frames), max(len(f[3]) for f in frames)
    ious = []
    for p, lab, v, g in frames:
        iou = IU.boxes_iou3d_gpu(_d(p[v].astype(np.float32)), _d(g[:, :7].astype(np.float32))).cpu().numpy()
        ious.append(np.where(iou >= 0, iou, -1.0))         # the counters skip IoUs that are not >= 0
    rec = torch.zeros(5 + 5 * len(THRESH), dtype=torch.int64, device=DEV)
    prec = torch.zeros(1 + len(THRESH), dtype=torch.int64, device=DEV)
    assert _launch_old(_lib.lib.fnp_recall_counters, d, n_pred, n_gt, rec) == 0
    assert _launch_old(_lib.lib.fnp_precision_counters, d, n_pred, n_gt, prec) == 0
    assert SeekerEngine.recall_dict(rec.cpu().numpy(), THRESH) == G.recall_dict(
        [(iou, f[3][:, 7]) for iou, f in zip(ious, frames)], THRESH)
    assert prec.cpu().numpy().tolist() == G.precision_counts(ious, THRESH).tolist()
    spec = _quality_spec()
    q = torch.zeros(spec.n_counters, dtype=torch.int64, device=DEV)
    assert _launch_quality(spec, d, n_pred, n_gt, q) == 0
    exp = G.quality_counts([(iou, f[1][f[2]], f[0][f[2], :2], f[3][:, 7], f[3][:, :2]) for iou, f in zip(ious, frames)],
                           THRESH, EDGES, N_CLASSES)
    assert np.array_equal(q.cpu().numpy(), exp)
    # stage-4 NMS over each frame's proposals in a score order, with its invalid rows
    boxes = np.concatenate([f[0] for f in frames]).astype(np.float32)
    valid = np.concatenate([np.where(f[2], 0, -1) for f in frames]).astype(np.int32)
    start = np.cumsum([0] + [len(f[1]) for f in frames])
    order = np.concatenate([start[s] + rng.permutation(start[s + 1] - start[s]) for s in range(3)]).astype(np.int32)
    tb, to, tv, ts = _d(boxes), _d(order), _d(valid), _d(start.astype(np.int32))
    keep = torch.full((len(boxes),), 9, dtype=torch.uint8, device=DEV)
    assert _lib.lib.fnp_seg_nms_rotated(tb.data_ptr(), None, to.data_ptr(), tv.data_ptr(), ts.data_ptr(), 3,
                                        int(np.diff(start).max()), C.c_float(0.1), keep.data_ptr(), _stream()) == 0
    want = np.zeros(len(boxes), np.uint8)
    for s in range(3):
        live = order[start[s]:start[s + 1]]
        live = live[valid[live] >= 0]
        m = IU.boxes_iou_bev(_d(boxes[live]), _d(boxes[live])).cpu().numpy()
        rows = lambda i: (np.arange(i + 1, len(live)), m[i, i + 1:])
        want[live[G.greedy_nms(rows, len(live), 0.1)]] = 1
    assert np.array_equal(keep.cpu().numpy(), want)
