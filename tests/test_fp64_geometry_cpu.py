"""The float64 geometry of fp64_geometry.py against closed forms, and the C oracle (the fp32 arithmetic of the kernels,
restated) against it within the bounds test_ops_fp64_gpu.py holds the kernels to.  No GPU needed."""
import numpy as np

import fp64_geometry as G
import oracle as O
from test_ops_gpu import _boxes, _pair_boxes


def _perimeter(a, b):
    """(N, M) larger perimeter of the two boxes of each pair."""
    return np.maximum(2 * (a[:, 3:4] + a[:, 4:5]), 2 * (b[:, 3] + b[:, 4])[None]).astype(np.float64)


def _check_overlap_bounds(exact, in_margin, got, perimeter):
    got = np.asarray(got, np.float64)
    ok = ~in_margin
    assert (np.abs(got - exact)[ok] <= G.overlap_tol(exact[ok])).all(), np.abs(got - exact)[ok].max()
    # a corner within 1 cm outside the other box counts as inside: the fp32 area may exceed the exact one there only
    assert ((got - exact) <= 0.01 * perimeter + G.overlap_tol(exact))[in_margin].all()
    assert ((exact - got)[in_margin] <= G.overlap_tol(exact[in_margin])).all()


def _special_pairs():
    """Closed-form pairs: identical boxes, boxes sharing an edge, same-yaw shifted boxes, yaw 0 against yaw pi/2, all
    as (a, b, exact BEV overlap)."""
    rng = np.random.default_rng(3)
    a = _boxes(rng, 64, spread=20.0).astype(np.float64)
    sx, sy = rng.uniform(-0.45, 0.45, (2, 64))
    c, s = np.cos(a[:, 6]), np.sin(a[:, 6])
    out = [(a, a.copy(), a[:, 3] * a[:, 4])]
    edge = a.copy()                                   # neighbour along the box's own x axis
    edge[:, 0] += a[:, 3] * c
    edge[:, 1] += a[:, 3] * s
    out.append((a, edge, np.zeros(64)))
    shifted = a.copy()                                # same yaw, shifted by (sx dx, sy dy) in the box's frame
    shifted[:, 0] += sx * a[:, 3] * c - sy * a[:, 4] * s
    shifted[:, 1] += sx * a[:, 3] * s + sy * a[:, 4] * c
    out.append((a, shifted, (1 - np.abs(sx)) * a[:, 3] * (1 - np.abs(sy)) * a[:, 4]))
    a0, b90 = a.copy(), a.copy()                      # yaw 0 against yaw pi/2: rectangles (dx, dy) and (dy', dx')
    a0[:, 6] = 0.0
    b90[:, 6] = np.pi / 2
    b90[:, :2] += rng.uniform(-1.5, 1.5, (64, 2))
    b90[:, 3:5] = rng.permutation(a[:, 3:5])
    w = np.maximum(np.minimum(a0[:, 0] + a0[:, 3] / 2, b90[:, 0] + b90[:, 4] / 2) -
                   np.maximum(a0[:, 0] - a0[:, 3] / 2, b90[:, 0] - b90[:, 4] / 2), 0)
    h = np.maximum(np.minimum(a0[:, 1] + a0[:, 4] / 2, b90[:, 1] + b90[:, 3] / 2) -
                   np.maximum(a0[:, 1] - a0[:, 4] / 2, b90[:, 1] - b90[:, 3] / 2), 0)
    out.append((a0, b90, w * h))
    return out


def test_fp64_overlap_matches_closed_forms():
    for a, b, exact in _special_pairs():
        ov, _ = G.overlap_bev(a, b)
        assert np.allclose(ov, exact, rtol=1e-12, atol=1e-9), np.abs(ov - exact).max()
        ov_t, _ = G.overlap_bev(b, a)
        assert np.allclose(ov_t, exact, rtol=1e-12, atol=1e-9)
    # disjoint, and one box inside another
    box = np.array([[1.0, 2.0, 0.0, 4.0, 2.0, 1.5, 0.3]])
    far, small = box.copy(), box.copy()
    far[0, 0] += 10
    small[0, 3:5] = [1.0, 0.5]
    assert G.overlap_bev(box, far)[0][0] == 0 and np.isclose(G.overlap_bev(box, small)[0][0], 0.5)
    assert np.isclose(G.iou_bev(box, small)[0][0], 0.5 / 8)
    assert np.isclose(G.iou3d(box, small)[0][0], 0.5 * 1.5 / (12 + 0.75 - 0.75))
    # the dense form equals the aligned one everywhere, far pairs included
    rng = np.random.default_rng(4)
    a, b = _boxes(rng, 40, spread=30.0), _boxes(rng, 30, spread=30.0)
    dense, dm = G.pairwise(G.overlap_bev, a, b)
    ii, jj = np.meshgrid(np.arange(40), np.arange(30), indexing="ij")
    al, am = G.overlap_bev(a[ii.ravel()], b[jj.ravel()])
    assert np.array_equal(dense.ravel(), al) and np.array_equal(dm.ravel(), am)


def test_fp64_points_in_boxes_matches_the_definition():
    box = np.array([[0.0, 0.0, 0.0, 4.0, 2.0, 2.0, np.pi / 2], [0.0, 0.0, 0.0, 10.0, 10.0, 10.0, 0.0]])
    pts = np.array([[0.0, 1.9, 0.0], [1.9, 0.0, 0.0], [0.0, 0.0, 0.99], [0.0, 0.0, 1.01], [6.0, 6.0, 0.0]])
    idx, margin = G.points_in_boxes(pts, box)
    assert idx.tolist() == [0, 1, 0, 1, -1]
    assert np.allclose(margin, [0.1, -0.9, 0.01, -0.01, -1.0])


def test_oracle_overlap_and_iou_within_the_fp64_bounds():
    """The C oracle's BEV overlap (the kernels' fp32 arithmetic) on random boxes with identical, shifted and
    axis-aligned pairs: within OVERLAP_ABS_TOL + OVERLAP_REL_TOL x area of the exact area for pairs without
    in_margin, and no more than 1 cm x the larger perimeter above it for in_margin pairs."""
    rng = np.random.default_rng(5)
    a, b = _pair_boxes(rng, 640)
    b = b[:500]
    exact, in_margin = G.pairwise(G.overlap_bev, a, b)
    assert (exact > 0).sum() > 50000 and in_margin.sum() > 1000
    _check_overlap_bounds(exact, in_margin, O.boxes_overlap_bev(a, b), _perimeter(a, b))
    ok = ~in_margin
    for fn_o, three_d in ((O.boxes_iou_bev, False), (O.boxes_iou3d, True)):
        exact_iou = G.pairwise(G.iou3d if three_d else G.iou_bev, a, b)[0]
        assert np.allclose(exact_iou, G.iou_from_overlap(a[:, None], b[None], exact, three_d), rtol=1e-14, atol=0)
        dev = np.abs(fn_o(a, b) - exact_iou)
        assert (dev <= G.iou_tol(a[:, None], b[None], exact, three_d))[ok].all(), dev[ok].max()
    for x, y, ex in _special_pairs():
        ov, m = G.overlap_bev(x, y)
        assert np.allclose(ov, ex, rtol=1e-12, atol=1e-9)
        got = np.array([O.boxes_overlap_bev(x[i:i + 1], y[i:i + 1])[0, 0] for i in range(len(x))])
        _check_overlap_bounds(ov, m, got, np.maximum(2 * (x[:, 3] + x[:, 4]), 2 * (y[:, 3] + y[:, 4])))


def test_oracle_points_in_boxes_and_nms_agree_with_fp64_where_decided():
    rng = np.random.default_rng(6)
    boxes = _boxes(rng, 40)
    boxes[20:25] = boxes[:5] * [1, 1, 1, 0.9, 1.1, 1, 1]          # overlapping boxes: first match decides
    pts = (rng.uniform(-0.5, 0.5, (20000, 3)) * [10, 10, 3] + [14, 0, -0.5]).astype(np.float32)
    idx, margin = G.points_in_boxes(pts, boxes)
    decided = np.abs(margin) > 1e-4
    assert decided.mean() > 0.99 and (idx[decided] >= 0).sum() > 1000
    assert np.array_equal(O.points_in_boxes_gpu(pts[None], boxes[None])[0][decided], idx[decided])
    # NMS: no pair IoU within 1e-3 of the threshold -> the oracle keeps what the float64 greedy keeps
    boxes = _boxes(rng, 300, spread=30.0)
    scores = rng.permutation(300).astype(np.float32)
    order = np.argsort(-scores, kind="stable")
    sb = boxes[order].astype(np.float64)
    i, j = G.near_pairs(sb)
    ran = 0
    for thr in (0.1, 0.5):
        for fn, fn_o in ((lambda x, y: G.iou_bev(x, y)[0], O.nms_rotated), (G.iou_normal, O.nms_normal)):
            v = fn(sb[i], sb[j])
            if (np.abs(v - thr) <= 1e-3).any():
                continue
            exp = order[G.greedy_nms(G.sparse_rows(i, j, v), 300, thr)]
            assert np.array_equal(fn_o(boxes, scores, thr), exp)
            assert 0 < len(exp) < 300
            ran += 1
    assert ran >= 2


def test_counter_restatements_match_the_recall_oracle():
    """recall_dict on float64 IoUs against seeker_oracle.recall_record, on frames with no IoU within 1e-3 of a
    threshold."""
    import seeker_oracle as SO
    rng = np.random.default_rng(7)
    done = 0
    for f in range(12):
        g = np.zeros((9, 8), np.float32)
        g[:, :7] = _boxes(rng, 9, spread=10.0)
        g[:, 7] = rng.integers(1, 11, 9)
        p = np.concatenate([g[:6, :7] + rng.normal(0, 0.15, (6, 7)).astype(np.float32) * [1, 1, 0, 0.2, 0.2, 0, 0.2],
                            _boxes(rng, 5, spread=10.0)])
        iou = G.pairwise(G.iou3d, p, g[:, :7])[0]
        if (np.abs(iou[..., None] - [0.3, 0.5, 0.7]) <= 1e-3).any():
            continue
        exp = SO.recall_record(p, np.concatenate([g[:, :7], np.zeros((9, 2), np.float32), g[:, 7:]], 1))
        assert G.recall_dict([(iou, g[:, 7])]) == exp
        done += 1
    assert done >= 8
