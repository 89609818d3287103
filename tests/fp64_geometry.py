"""A plain float64 statement of the box geometry behind the op-level kernels, written from the geometry itself and not
from the kernels or the C oracle: numpy only.  The fp32 ops are bounded against it by test_fp64_geometry_cpu.py (the
oracle) and test_ops_fp64_gpu.py (the kernels).

Boxes are rows [x, y, z, dx, dy, dz, heading] (further columns are ignored): (x, y, z) is the centre, (dx, dy, dz) the
full sizes along the box's own axes, and the heading turns the box counter-clockwise about +z.  Sizes are taken to be
positive; the clipper assumes counter-clockwise corners.
"""
import numpy as np

# The reference's check_in_box2d counts a corner up to 1 cm outside a box as inside (tx = dx/2 + 1e-2).  Only a pair
# with a corner of one box in the band (0, MARGIN_BAND] outside the other may get more than the true area from the
# fp32 op; the band is twice the 1 cm so that rounding cannot move a corner across its outer end.
MARGIN_BAND = 0.02

# How far the fp32 BEV overlap of a pair without in_margin may lie from the exact area, for boxes within ~50 m of the
# origin: corners and edge crossings are rounded to a few ulp of their coordinates (ulp(32) = 3.8e-6 m), which moves
# the area by at most the intersection's perimeter (< 40 m here) times that.  The largest deviation seen on the C
# oracle over 3M pairs of test_ops_gpu._pair_boxes was 2.7e-5 m^2, and 4.6e-6 m^2 above 1e-5 relative.
OVERLAP_ABS_TOL, OVERLAP_REL_TOL = 1e-4, 1e-5

# generate_recall_record's known-class sets, as 1-based labels
KNOWN3 = (1, 8, 9)
KNOWN6 = (1, 3, 5, 6, 8, 9)


def _rows(boxes):
    b = np.asarray(boxes, np.float64)
    return b.reshape(-1, b.shape[-1]) if b.size else b.reshape(0, 7)


def box_corners(boxes):
    """(N, 4, 2) BEV corners, counter-clockwise from the (-dx/2, -dy/2) corner in the box's frame."""
    b = _rows(boxes)
    lx = np.array([-0.5, 0.5, 0.5, -0.5])[None] * b[:, 3:4]
    ly = np.array([-0.5, -0.5, 0.5, 0.5])[None] * b[:, 4:5]
    c, s = np.cos(b[:, 6:7]), np.sin(b[:, 6:7])
    return np.stack([b[:, 0:1] + lx * c - ly * s, b[:, 1:2] + lx * s + ly * c], -1)


def _to_local(x, y, b):
    """Offsets of the points (x, y) (broadcast against b's rows) along box b's own x and y axes."""
    sx, sy = x - b[..., 0], y - b[..., 1]
    c, s = np.cos(b[..., 6]), np.sin(b[..., 6])
    return sx * c + sy * s, -sx * s + sy * c


# ------------------------------------------------------------------------------------------------ points in boxes
def face_margin(pts, boxes):
    """(M, T): for point m and box t, the least over the three axes of (half size - |offset along the axis|): > 0
    inside the true box, < 0 outside it.  A point with |margin| > eps changes sides only if it moves more than eps."""
    p = np.asarray(pts, np.float64).reshape(-1, 3)
    b = _rows(boxes)[None]
    lx, ly = _to_local(p[:, 0:1], p[:, 1:2], b)
    lz = p[:, 2:3] - b[..., 2]
    return np.minimum(np.minimum(b[..., 3] / 2 - np.abs(lx), b[..., 4] / 2 - np.abs(ly)), b[..., 5] / 2 - np.abs(lz))


def points_in_boxes(pts, boxes, chunk=2048):
    """First box (in row order) whose true box contains each point, or -1; and per point the signed face margin
    (face_margin) of smallest magnitude over the boxes that decide the answer: every box before the first containing
    one, and that box (all boxes for -1).  Callers treat points with |margin| <= a tolerance as undecided."""
    p = np.asarray(pts, np.float64).reshape(-1, 3)
    T = _rows(boxes).shape[0]
    idx = np.full(p.shape[0], -1, np.int64)
    margin = np.full(p.shape[0], np.inf)
    if T == 0:
        return idx, margin
    for r0 in range(0, p.shape[0], chunk):
        m = face_margin(p[r0:r0 + chunk], boxes)
        inside = m >= 0
        hit = inside.any(1)
        first = np.where(hit, inside.argmax(1), -1)
        deciding = np.arange(T)[None] <= np.where(hit, first, T - 1)[:, None]
        k = np.where(deciding, np.abs(m), np.inf).argmin(1)
        idx[r0:r0 + chunk] = first
        margin[r0:r0 + chunk] = m[np.arange(m.shape[0]), k]
    return idx, margin


# ------------------------------------------------------------------------------------------------ BEV overlap
def _clip(poly, n, e0, e1):
    """Sutherland-Hodgman step: convex polygons poly (P, W, 2) with n (P,) vertices, clipped to the half-plane left of
    the directed edge e0 -> e1 (P, 2).  Returns the clipped polygons and their vertex counts."""
    P, W, _ = poly.shape
    j = np.arange(W)[None]
    live = j < n[:, None]
    q = np.take_along_axis(poly, np.where(j + 1 < n[:, None], j + 1, 0)[..., None], 1)
    d = (e1 - e0)[:, None]
    side = lambda v: d[..., 0] * (v[..., 1] - e0[:, None, 1]) - d[..., 1] * (v[..., 0] - e0[:, None, 0])
    sp, sq = side(poly), side(q)
    pin = sp >= 0
    crossing = live & (pin != (sq >= 0))
    t = sp / np.where(crossing, sp - sq, 1.0)
    x = poly + t[..., None] * (q - poly)
    # for each edge p -> q: p if it is inside, then the crossing point if the edge crosses the line
    cand = np.stack([poly, x], 2).reshape(P, 2 * W, 2)
    keep = np.stack([live & pin, crossing], 2).reshape(P, 2 * W)
    m = keep.sum(1)
    cand = np.take_along_axis(cand, np.argsort(~keep, axis=1, kind="stable")[..., None], 1)
    return cand[:, :max(int(m.max(initial=0)), 1)], m


def _polygon_area(poly, n):
    j = np.arange(poly.shape[1])[None]
    q = np.take_along_axis(poly, np.where(j + 1 < n[:, None], j + 1, 0)[..., None], 1)
    cr = poly[..., 0] * q[..., 1] - poly[..., 1] * q[..., 0]
    return 0.5 * np.abs(np.where(j < n[:, None], cr, 0.0).sum(1))


def _corner_outside(corners, b):
    """(P, 4): how far each corner lies outside box b along the box's axes (<= 0: inside or on the boundary)."""
    lx, ly = _to_local(corners[..., 0], corners[..., 1], b[:, None])
    return np.maximum(np.abs(lx) - b[:, None, 3] / 2, np.abs(ly) - b[:, None, 4] / 2)


def overlap_bev(a, b):
    """Aligned pairs (P, 7), (P, 7): the exact BEV intersection area of a[i] and b[i] (clipping a's rectangle against
    each edge of b's), and in_margin (P,): a corner of either box lies in (0, MARGIN_BAND] m outside the other."""
    a, b = _rows(a)[:, :7], _rows(b)[:, :7]
    P = a.shape[0]
    if P == 0:
        return np.zeros(0), np.zeros(0, bool)
    shift = np.concatenate([a[:, :2], np.zeros((P, 5))], 1)   # clip around a's centre
    ca, cb = box_corners(a - shift), box_corners(b - shift)
    poly, n = ca, np.full(P, 4)
    for k in range(4):
        poly, n = _clip(poly, n, cb[:, k], cb[:, (k + 1) % 4])
    area = _polygon_area(poly, n)
    out = np.concatenate([_corner_outside(ca, b - shift), _corner_outside(cb, a - shift)], 1)
    in_margin = ((out > 0) & (out <= MARGIN_BAND)).any(1)
    return area, in_margin


def _height_overlap(a, b):
    return np.maximum(np.minimum(a[..., 2] + a[..., 5] / 2, b[..., 2] + b[..., 5] / 2) -
                      np.maximum(a[..., 2] - a[..., 5] / 2, b[..., 2] - b[..., 5] / 2), 0.0)


def iou_from_overlap(a, b, overlap, three_d=False):
    """BEV IoU overlap / max(area_a + area_b - overlap, 1e-8), or with three_d the 3D IoU: overlap x height overlap
    over max(volume_a + volume_b - that, 1e-6).  a, b and overlap broadcast against each other (a[:, None] with
    b[None] and an (N, M) overlap gives the dense matrix)."""
    a, b, ov = np.asarray(a, np.float64), np.asarray(b, np.float64), np.asarray(overlap, np.float64)
    if not three_d:
        return ov / np.maximum(a[..., 3] * a[..., 4] + b[..., 3] * b[..., 4] - ov, 1e-8)
    ov3 = ov * _height_overlap(a, b)
    return ov3 / np.maximum(np.prod(a[..., 3:6], -1) + np.prod(b[..., 3:6], -1) - ov3, 1e-6)


def overlap_tol(exact):
    """The bound |fp32 overlap - exact| <= OVERLAP_ABS_TOL + OVERLAP_REL_TOL * exact of a pair without in_margin."""
    return OVERLAP_ABS_TOL + OVERLAP_REL_TOL * np.asarray(exact)


def iou_tol(a, b, exact_overlap, three_d=False):
    """The IoU bound that overlap_tol implies for pairs without in_margin (broadcast like iou_from_overlap): IoU =
    v / (S - v) moves by at most tol * S / (S - v - tol)^2 when v moves by tol, plus 1e-6 for the fp32 rounding of
    the division itself."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    ov, tol = np.asarray(exact_overlap, np.float64), overlap_tol(exact_overlap)
    if three_d:
        h = _height_overlap(a, b)
        ov, tol, s = ov * h, tol * h, np.prod(a[..., 3:6], -1) + np.prod(b[..., 3:6], -1)
    else:
        s = a[..., 3] * a[..., 4] + b[..., 3] * b[..., 4]
    return tol * s / np.maximum(s - ov - tol, 1e-8) ** 2 + 1e-6


def iou_bev(a, b):
    """Aligned pairs: (BEV IoU, in_margin)."""
    ov, m = overlap_bev(a, b)
    return iou_from_overlap(_rows(a), _rows(b), ov), m


def iou3d(a, b):
    """Aligned pairs: (3D IoU, in_margin)."""
    ov, m = overlap_bev(a, b)
    return iou_from_overlap(_rows(a), _rows(b), ov, three_d=True), m


def iou_normal(a, b):
    """Aligned pairs: BEV IoU of the axis-aligned rectangles (heading ignored), union clamped to 1e-8."""
    a, b = _rows(a), _rows(b)
    w = np.maximum(np.minimum(a[:, 0] + a[:, 3] / 2, b[:, 0] + b[:, 3] / 2) -
                   np.maximum(a[:, 0] - a[:, 3] / 2, b[:, 0] - b[:, 3] / 2), 0.0)
    h = np.maximum(np.minimum(a[:, 1] + a[:, 4] / 2, b[:, 1] + b[:, 4] / 2) -
                   np.maximum(a[:, 1] - a[:, 4] / 2, b[:, 1] - b[:, 4] / 2), 0.0)
    inter = w * h
    return inter / np.maximum(a[:, 3] * a[:, 4] + b[:, 3] * b[:, 4] - inter, 1e-8)


def near_pairs(a, b=None, chunk=512):
    """(i, j) of the pairs that can touch, or come within MARGIN_BAND: centres no further apart than the sum of the
    half diagonals plus twice the band.  b=None: the pairs i < j within a.  Every other pair has overlap 0, IoU 0 and
    no in_margin flag.  Rows are visited in x order, each chunk against the boxes within reach in x."""
    a = _rows(a)
    bb = a if b is None else _rows(b)
    ra, rb = np.hypot(a[:, 3], a[:, 4]) / 2, np.hypot(bb[:, 3], bb[:, 4]) / 2
    reach = ra.max(initial=0) + rb.max(initial=0) + 2 * MARGIN_BAND
    oa, ob = np.argsort(a[:, 0], kind="stable"), np.argsort(bb[:, 0], kind="stable")
    bx = bb[ob, 0]
    out_i, out_j = [np.zeros(0, np.int64)], [np.zeros(0, np.int64)]
    for r0 in range(0, a.shape[0], chunk):
        rows = oa[r0:r0 + chunk]
        cols = ob[np.searchsorted(bx, a[rows, 0].min() - reach):np.searchsorted(bx, a[rows, 0].max() + reach, "right")]
        d = np.hypot(a[rows, 0:1] - bb[None, cols, 0], a[rows, 1:2] - bb[None, cols, 1])
        near = d <= ra[rows, None] + rb[None, cols] + 2 * MARGIN_BAND
        if b is None:
            near &= cols[None] > rows[:, None]
        i, j = np.nonzero(near)
        out_i.append(rows[i])
        out_j.append(cols[j])
    return np.concatenate(out_i), np.concatenate(out_j)


def pairwise(fn, a, b, chunk=1 << 15):
    """The (N, M) matrices of an aligned-pair function fn (returning one array or a tuple of them) over every pair
    of a x b, evaluated on near_pairs only; the other entries are 0 / False."""
    a, b = _rows(a), _rows(b)
    i, j = near_pairs(a, b)
    parts = [fn(a[i[k:k + chunk]], b[j[k:k + chunk]]) for k in range(0, len(i), chunk)] or [fn(a[:0], b[:0])]
    single = not isinstance(parts[0], tuple)
    outs = []
    for col in zip(*([(p,) for p in parts] if single else parts)):
        v = np.concatenate(col)
        m = np.zeros((a.shape[0], b.shape[0]), v.dtype)
        m[i, j] = v
        outs.append(m)
    return outs[0] if single else tuple(outs)


# ------------------------------------------------------------------------------------------------ NMS
def greedy_nms(iou_rows, n, thresh):
    """Greedy NMS over n boxes already in score order (position 0 is the best): a box is kept unless a kept box
    before it has IoU > thresh with it.  iou_rows(i) -> (j, iou): the boxes j > i that may overlap box i with their
    IoUs (a pair left out has IoU 0).  Returns the kept positions in order."""
    removed = np.zeros(n, bool)
    keep = []
    for i in range(n):
        if removed[i]:
            continue
        keep.append(i)
        j, v = iou_rows(i)
        removed[j[v > thresh]] = True
    return np.asarray(keep, np.int64)


def sparse_rows(i, j, v):
    """iou_rows for greedy_nms from lists of unordered pairs (i[k], j[k]) (i != j, each pair once) with IoU v[k]."""
    lo, hi = np.minimum(i, j), np.maximum(i, j)
    o = np.argsort(lo, kind="stable")
    lo, hi, v = lo[o], hi[o], np.asarray(v)[o]

    def rows(k):
        s, e = np.searchsorted(lo, k), np.searchsorted(lo, k, "right")
        return hi[s:e], v[s:e]
    return rows


# ------------------------------------------------------------------------------------------------ counters
def recall_dict(frames, thresh=(0.3, 0.5, 0.7)):
    """generate_recall_record's counters, keyed as SeekerEngine.recall_dict keys them, from per-frame
    (iou (K, G) of the frame's valid proposals against its GT boxes, GT labels (G,)).  A GT box counts for threshold
    t when its best IoU over the proposals is > t; the known / unknown splits use KNOWN3 and KNOWN6."""
    names = ["", "_3known", "_6known", "_4unknown", "_7unknown"]
    d = dict.fromkeys(["gt", "num_3known", "num_6known", "num_4unknown", "num_7unknown"], 0)
    d.update(("rcnn%s_%s" % (s, t), 0) for t in thresh for s in names)
    for iou, lab in frames:
        lab = np.asarray(lab).astype(np.int64)
        k3, k6 = np.isin(lab, KNOWN3), np.isin(lab, KNOWN6)
        split = [np.ones_like(k3), k3, k6, ~k6, ~k3]
        best = np.asarray(iou).reshape(-1, len(lab)).max(0, initial=-1.0)
        for key, m in zip(["gt", "num_3known", "num_6known", "num_4unknown", "num_7unknown"], split):
            d[key] += int(m.sum())
        for t in thresh:
            for s, m in zip(names, split):
                d["rcnn%s_%s" % (s, t)] += int((m & (best > t)).sum())
    return d


def precision_counts(frames, thresh=(0.3, 0.5, 0.7)):
    """fnp_precision_counters' layout from per-frame iou (K, G) of the valid proposals against the GT: [proposals,
    then per threshold the proposals whose best IoU over the frame's GT is > t]."""
    out = np.zeros(1 + len(thresh), np.int64)
    for iou in frames:
        iou = np.asarray(iou)
        best = iou.max(1, initial=-1.0)
        out[0] += iou.shape[0]
        out[1:] += [(best > t).sum() for t in thresh]
    return out


def quality_counts(frames, thresh, edges, n_classes):
    """One setting of fnp_quality_counters (layout [recall | precision][class - 1][range bin][1 + 2T], flat) from
    per-frame (iou (K, G), proposal labels (K,), proposal centres (K, 2), GT labels (G,), GT centres (G, 2)) of the
    valid proposals.  The bin of a centre is the number of edges <= its distance from the origin; for each box, w = 0
    counts it, 1 + t counts a best IoU > t over all boxes of the other kind, 1 + T + t over those of the same label."""
    T, R = len(thresh), len(edges) + 1
    out = np.zeros((2, n_classes, R, 1 + 2 * T), np.int64)
    th = np.asarray(thresh, np.float64)
    for iou, pl, pxy, gl, gxy in frames:
        pl, gl = np.asarray(pl).astype(np.int64), np.asarray(gl).astype(np.int64)
        iou = np.asarray(iou, np.float64).reshape(len(pl), len(gl))
        same = np.where(pl[:, None] == gl[None], iou, -1.0)
        for blk, lab, xy, best_any, best_lab in ((0, gl, gxy, iou.max(0, initial=-1.0), same.max(0, initial=-1.0)),
                                                 (1, pl, pxy, iou.max(1, initial=-1.0), same.max(1, initial=-1.0))):
            xy = np.asarray(xy, np.float64).reshape(-1, 2)
            bins = (np.asarray(edges, np.float64)[None] <= np.hypot(xy[:, 0], xy[:, 1])[:, None]).sum(1)
            for k in range(len(lab)):
                c = out[blk, lab[k] - 1, bins[k]]
                c[0] += 1
                c[1:1 + T] += best_any[k] > th
                c[1 + T:] += best_lab[k] > th
    return out.reshape(-1)
