"""Frustums built to reach every path of stage 2b, the per-hypothesis point counts (csrc/fnp_seeker.cu: score_kernel,
the DIRECT mode; sweep_prep_kernel + sweep_score_kernel, the SWEEP mode; firstmatch_kernel, the KITTI variant), shared by
test_score_cases_cpu.py (the host model of the sweep, the oracle and a float64 bracket) and test_score_stage_gpu.py (the
kernels, driven through fnp_seeker_score on a hand-built page pool).

A case is one fnp_seeker_score call: J yaw-size columns x M depth steps, a point split and a few frustums.  A frustum
holds its points and its valid hypotheses in compacted order: 7-dof boxes, their prep rows (the arithmetic of prep_box,
tools/sweep_model/model.prep_boxes) and hyp_index (ascending m*J + j).  The hypotheses of a column share size and
heading, so their rotation and thresholds agree bit for bit, as prep_box guarantees in the pipeline.

Each case names the part of the kernels it reaches; test_score_cases_cpu.py checks that it does.
"""
import functools
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (os.path.join(ROOT, "tools", "sweep_model"), os.path.join(ROOT, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)
import model as SM  # noqa: E402
import oracle as O  # noqa: E402

PG = 256                       # FNP_PAGE_POINTS: points per page of the pool
SWEEP_WARPS, SWEEP_QUEUE = 8, 384   # kSweepThreads / 32 warps, each with a queue of kSweepQueue (point, steps) entries
SWEEP_COL_BYTES = 80           # sizeof(SweepCol)
SMEM_LIMIT = 200 * 1024        # the sweep kernel's dynamic shared memory bound (resolve_score_mode)
SCORE_CHUNK = 512              # kScoreThreads * kScoreKMax: hypotheses of a full DIRECT chunk


def sweep_smem_bytes(SP, H, J):
    """Dynamic shared memory of sweep_score_kernel (sweep_smem_bytes in fnp_seeker.cu):
    80 J (columns) + 8 * 384 * 8 (queues) + 12 SP (the split's x, y, z) + 4 H (difference arrays)
    + 2 ceil4(H) (the short slot table) + 16 + 128 (control words, one scratch word per lane)."""
    return SWEEP_COL_BYTES * J + SWEEP_WARPS * SWEEP_QUEUE * 8 + 12 * SP + 4 * H + 2 * ((H + 3) & ~3) + 144


def sweep_admits(J, M, SP):
    """Whether resolve_score_mode lets the sweep run (the `fits` bound).  H <= 32767 is what the short slot table
    needs; under the shared-memory bound it is never the one that binds: at J = 1 and SP = 256 that bound already
    stops at H = 29 488."""
    H = J * M
    return H <= 32767 and M <= 255 and SP <= 65536 and sweep_smem_bytes(SP, H, J) <= SMEM_LIMIT and 60 * J <= 48 * 1024


def items_needed(case, sweep):
    """Work items fnp_seeker_score plans (plan_items_kernel): per frustum with points and valid hypotheses,
    ceil(n / split) point splits, times ceil(nv / 512) hypothesis chunks in DIRECT mode."""
    tot = 0
    for fr in case.frustums:
        if fr.n > 0 and fr.nv > 0:
            tot += -(-fr.n // case.split) * (1 if sweep else -(-fr.nv // SCORE_CHUNK))
    return tot


class Frustum:
    def __init__(self, pts, boxes, hidx):
        self.pts = np.ascontiguousarray(pts, np.float32).reshape(-1, 3)
        self.boxes = np.ascontiguousarray(boxes, np.float32).reshape(-1, 7)
        self.hidx = np.ascontiguousarray(hidx, np.int32)
        assert np.all(np.diff(self.hidx) > 0)
        self.prep = SM.prep_boxes(self.boxes, O.cosf, O.sinf) if self.nv else np.zeros((0, 8), np.float32)
        self._bracket = None

    @property
    def n(self):
        return self.pts.shape[0]

    @property
    def nv(self):
        return self.hidx.shape[0]

    def bracket(self):
        if self._bracket is None:
            self._bracket = bracket(self.pts, self.boxes)
        return self._bracket


class Case:
    def __init__(self, name, J, M, split, frustums, kind="count", benign=True):
        self.name, self.J, self.M, self.split, self.frustums = name, J, M, split, frustums
        self.kind = kind          # "count": every valid hypothesis counts its points; "kitti": first match
        self.benign = benign      # False: points sit on faces on purpose, the float64 bracket is loose there

    @property
    def H(self):
        return self.J * self.M


# ---------------------------------------------------------------------------------------------- the float64 bracket
def bracket(pts, boxes, pairs_per_chunk=1 << 21):
    """Per hypothesis (lo, hi): lo = points certainly inside, hi = lo + points too close to a face to call.

    The predicate is restated in float64 from the fp32 inputs: local coordinates lx = sx cos h + sy sin h,
    ly = -sx sin h + sy cos h, lz = z - cz, inside iff |lx| < dx/2 + 1e-5, |ly| < dy/2 + 1e-5, |lz| <= dz/2.  The fp32
    chain of the kernels (the rounded differences, cosf / sinf, the product and the fma) moves a local coordinate by
    less than 2^-21 (|sx| + |sy|) + 2^-24 |l| <= 2^-19 (2 maxabs + half extent), with maxabs the largest |coordinate|
    of the frustum's points and centres; that is the margin.  A pair is decided inside when every face is farther
    than the margin on the inner side, decided outside when some face is farther than the margin on the outer side."""
    p = np.asarray(pts, np.float64).reshape(-1, 3)
    b = np.asarray(boxes, np.float64).reshape(-1, 7)
    nv = b.shape[0]
    lo = np.zeros(nv, np.int64)
    und = np.zeros(nv, np.int64)
    if nv == 0 or p.shape[0] == 0:
        return lo, lo.copy()
    maxabs = max(np.abs(p).max(), np.abs(b[:, :3]).max())
    t = np.stack([b[:, 3] * 0.5 + np.float64(np.float32(1e-5)), b[:, 4] * 0.5 + np.float64(np.float32(1e-5)),
                  b[:, 5] * 0.5], 1)
    margin = 2.0 ** -19 * (2 * maxabs + t.max(1))
    c, s = np.cos(b[:, 6]), np.sin(b[:, 6])
    step = max(1, pairs_per_chunk // nv)
    for i0 in range(0, p.shape[0], step):
        q = p[i0:i0 + step]
        sx, sy = q[:, 0:1] - b[:, 0], q[:, 1:2] - b[:, 1]
        d = np.stack([t[:, 0] - np.abs(sx * c + sy * s), t[:, 1] - np.abs(-sx * s + sy * c),
                      t[:, 2] - np.abs(q[:, 2:3] - b[:, 2])], -1)       # (points, nv, 3): > 0 inside the face
        inside = (d > margin[:, None]).all(-1)
        outside = (d < -margin[:, None]).any(-1)
        lo += inside.sum(0)
        und += (~inside & ~outside).sum(0)
    return lo, lo + und


# ---------------------------------------------------------------------------------------------- geometry helpers
def _unit(rng):
    d = rng.normal(size=3)
    return d / np.linalg.norm(d)


def _grid(rng, J, M, origin, direction, step, jitter, dims, yaw, valid):
    """Hypotheses of the valid (m, j) of a (M, J) mask: centre origin + direction * step * m + N(0, jitter) per axis
    (jitter a scalar or (J,) per column), size dims[j], heading yaw[j].  -> boxes (nv, 7), hidx (nv,)"""
    mm, jj = np.nonzero(valid)
    order = np.argsort(mm * J + jj, kind="stable")
    mm, jj = mm[order], jj[order]
    jit = np.broadcast_to(np.asarray(jitter, np.float64), (J,))[jj]
    c = origin[None] + direction[None] * (step * mm)[:, None] + rng.normal(size=(mm.size, 3)) * jit[:, None]
    boxes = np.concatenate([c, dims[jj], yaw[jj, None]], 1).astype(np.float32)
    return boxes, (mm * J + jj).astype(np.int32)


def _points_in(rng, prep, n, spread=1.2, face_p=0.0):
    """n points around the boxes of `prep` rows: local offsets uniform in +-spread half sizes, a share face_p of them
    moved onto a face, a few ulp either side."""
    b = prep[rng.integers(0, prep.shape[0], n)].astype(np.float64)
    half = b[:, [6, 7, 3]]
    l = rng.uniform(-spread, spread, (n, 3)) * half
    on = rng.random(n) < face_p
    k = rng.integers(0, 3, n)
    ulp = 1 + rng.integers(-4, 5, n) * 6e-8
    r = np.arange(n)
    l[r[on], k[on]] = np.sign(l[r[on], k[on]] + 1e-30) * half[r[on], k[on]] * ulp[on]
    ca, sa = b[:, 4], b[:, 5]
    # local = Rot(-yaw)(p - c)  =>  p = c + Rot(yaw) local;  cosa = cos(-yaw), sina = sin(-yaw)
    x = b[:, 0] + l[:, 0] * ca + l[:, 1] * sa
    y = b[:, 1] - l[:, 0] * sa + l[:, 1] * ca
    return np.stack([x, y, b[:, 2] + l[:, 2]], 1).astype(np.float32)


def _mix(rng, parts):
    pts = np.concatenate([np.asarray(p, np.float32).reshape(-1, 3) for p in parts])
    return pts[rng.permutation(pts.shape[0])]


def _line_frustum(rng, J, M, n, valid, origin=None, direction=None, step=0.2, jitter=1e-3, dims=None, yaw=None,
                  spread=1.2, bg=0.1):
    """A seeker-like frustum: columns of boxes on one centre line, points around the boxes plus a little background."""
    origin = rng.uniform(-30, 30, 3) if origin is None else np.asarray(origin, np.float64)
    direction = _unit(rng) if direction is None else np.asarray(direction, np.float64)
    dims = rng.uniform(0.8, 5.0, (J, 3)) if dims is None else dims
    yaw = rng.uniform(-np.pi, np.pi, J) if yaw is None else yaw
    boxes, hidx = _grid(rng, J, M, origin, direction, step, jitter, dims, yaw, valid)
    if hidx.size == 0 or n == 0:
        pts = origin[None] + rng.normal(size=(n, 3)) * 5
        return Frustum(pts, boxes, hidx)
    prep = SM.prep_boxes(boxes, O.cosf, O.sinf)
    nb = int(round(n * bg))
    pts = _mix(rng, [_points_in(rng, prep, n - nb, spread), origin[None] + rng.normal(size=(nb, 3)) * 5])
    return Frustum(pts, boxes, hidx)


# ---------------------------------------------------------------------------------------------- the cases
def _adversarial(seed):
    """test_sweep_model_cpu's adversarial columns on the device: offsets up to 1 km, steps 0 - 0.5 m, jitter 0 - 0.5 m,
    70 % of the points within +-4 ulp of a face, validity 0.2 / 0.7 / 1; several frustums of different sizes in one
    call, so that the pieces of different frustums share the persistent CTAs."""
    rng = np.random.default_rng(900 + seed)
    J = int(rng.integers(1, 9))
    M = int(rng.choice([1, 2, 5, 16, 64, 100, 255]))
    split = int(rng.choice([256, 768, 2048]))
    frs = []
    for k in range(3):
        scale = float(rng.choice([1.0, 50.0, 200.0, 1000.0]))
        step = float(rng.choice([0.0, 1e-7, 1e-5, 1e-3, 2e-2, 0.5]))
        jitter = float(rng.choice([0.0, 1e-6, 1e-4, 1e-2, 0.5]))
        valid_p = float(rng.choice([0.2, 0.7, 1.0]))
        n = int(rng.choice([1, 300, 1000, 3000])) if k else 2500
        origin = rng.uniform(-1, 1, 3) * scale
        direction = _unit(rng)
        if rng.random() < 0.3:
            direction[rng.integers(0, 3)] = 0.0       # no travel along one world axis
        dims = rng.uniform(0.3, 12.0, (J, 3))
        yaw = rng.uniform(-np.pi, np.pi, J)
        valid = rng.random((M, J)) < valid_p
        valid[rng.integers(0, M), rng.integers(0, J)] = True
        boxes, hidx = _grid(rng, J, M, origin, direction, step, jitter, dims, yaw, valid)
        prep = SM.prep_boxes(boxes, O.cosf, O.sinf)
        nb = int(n * 0.2)
        pts = _mix(rng, [_points_in(rng, prep, n - nb, 1.2, 0.7), origin[None] + rng.normal(size=(nb, 3)) * 5])
        frs.append(Frustum(pts, boxes, hidx))
    return Case("adversarial_%02d" % seed, J, M, split, frs, benign=False)


def _queue():
    """Queue overflow and full packed bytes: M = 255 (D = 254).  Six columns have boxes far smaller than the jitter of
    their centres (t < dl: no pair has a definite range, so every pair near the line is all uncertain steps and a2 =
    B + 1 reaches 255); two have large boxes and mild jitter (a definite range plus uncertain ends).  Every point
    lies near the centre line, so every piece of every column pushes its 256 entries and the warp drains before
    each piece, between REDs of the definite columns into the difference array."""
    rng = np.random.default_rng(7001)
    J, M = 8, 255
    dims = np.concatenate([rng.uniform(0.2, 0.5, (6, 3)), rng.uniform([3.5, 3.0, 2.5], [4.5, 4.0, 3.0], (2, 3))])
    jitter = np.array([1.0] * 6 + [0.12] * 2)
    yaw = rng.uniform(-np.pi, np.pi, J)
    frs = []
    for n, sp in ((2600, 0.25), (700, 0.15)):
        origin, direction = rng.uniform(-20, 20, 3), _unit(rng)
        boxes, hidx = _grid(rng, J, M, origin, direction, 0.02, jitter, dims, yaw, np.ones((M, J), bool))
        m = rng.uniform(0, M - 1, n)
        pts = origin[None] + direction[None] * 0.02 * m[:, None] + rng.normal(size=(n, 3)) * sp
        frs.append(Frustum(pts, boxes, hidx))
    return Case("queue_overflow", J, M, 2048, frs, benign=False)


def _sparse():
    """Sparse columns: a column without a valid step (m1 < m0), single valid steps at m = 0, 17 and M - 1 (D = 0),
    a column of 2 % validity with gaps inside it, a full column; and a frustum of 2 % validity over the whole grid."""
    rng = np.random.default_rng(7002)
    J, M = 6, 40
    frs = []
    for n, whole in ((900, False), (2000, False), (1500, True)):
        valid = np.zeros((M, J), bool)
        if whole:
            valid = rng.random((M, J)) < 0.02
            valid[[2, 25], [1, 1]] = True
        else:
            valid[17, 1] = valid[0, 2] = valid[M - 1, 3] = True
            valid[:, 4] = rng.random(M) < 0.02
            valid[[3, 30], 4] = True
            valid[:, 5] = True
        frs.append(_line_frustum(rng, J, M, n, valid))
    return Case("sparse_columns", J, M, 768, frs)


def _single_step():
    """M = 1: every column is one depth step (D = 0); one column empty."""
    rng = np.random.default_rng(7003)
    J, M = 7, 1
    valid = np.ones((M, J), bool)
    valid[0, 3] = False
    frs = [_line_frustum(rng, J, M, n, valid) for n in (1000, 257)]
    return Case("single_step", J, M, 512, frs)


def point_count_list(SP):
    return [1, 2, 63, 64, 65, 255, 256, 257, 511, 513, SP - 1, SP, SP + 1, 3 * SP + 17, 0]


def _point_counts(SP):
    """Every tail modulo 64 (sweep passes) and 256 (pages, far padding) that matters, a TMA stage of one page, several
    splits adding into one row, a frustum without points.  The centre line passes through the origin, so that a
    padding point at (0, 0, 0) would be counted."""
    rng = np.random.default_rng(7100 + SP)
    J, M = 4, 32
    direction = _unit(rng)
    origin = -direction * 0.2 * 11.3          # the origin sits between steps 11 and 12 of every column
    dims = rng.uniform(1.5, 4.0, (J, 3))
    yaw = rng.uniform(-np.pi, np.pi, J)
    frs = []
    for n in point_count_list(SP):
        valid = rng.random((M, J)) < 0.8
        valid[11:13] = True
        frs.append(_line_frustum(rng, J, M, n, valid, origin=origin, direction=direction, dims=dims, yaw=yaw))
    return Case("point_counts_sp%d" % SP, J, M, SP, frs)


DIRECT_NV = [1, 127, 128, 129, 383, 384, 385, 511, 512, 513, 640, 1025]


def _direct_chunks():
    """DIRECT's hypothesis chunks: K = 1..4 per thread, the remainder chunk, more than two chunks, all with odd point
    counts (the last point of a page taken on its own)."""
    rng = np.random.default_rng(7200)
    J, M = 12, 100
    ns = [257, 511, 1025, 333, 777, 1, 3, 515, 999, 1537, 129, 2049]
    frs = []
    for nv, n in zip(DIRECT_NV, ns):
        valid = np.zeros(J * M, bool)
        valid[rng.choice(J * M, nv, replace=False)] = True
        frs.append(_line_frustum(rng, J, M, n, valid.reshape(M, J), step=0.1))
    return Case("direct_chunks", J, M, 768, frs)


def _smem(J, M, SP, ns, valid_p):
    rng = np.random.default_rng(7300 + J + SP)
    frs = []
    for n, vp in zip(ns, valid_p):
        valid = rng.random((M, J)) < vp
        frs.append(_line_frustum(rng, J, M, n, valid, step=0.05))
    return Case("smem_J%d_M%d_sp%d" % (J, M, SP), J, M, SP, frs)


def _kitti():
    """KITTI's first match: heavily overlapping hypotheses, frustums across the kernel's 4096-point splits."""
    rng = np.random.default_rng(7400)
    J, M = 6, 20
    frs = []
    for n in (4095, 4096, 4097, 9000):
        valid = rng.random((M, J)) < 0.6
        frs.append(_line_frustum(rng, J, M, n, valid, step=0.1, spread=1.0))
    return Case("kitti_first_match", J, M, 256, frs, kind="kitti")


_BUILDERS = dict(
    [("adversarial_%02d" % s, functools.partial(_adversarial, s)) for s in range(12)] +
    [("queue_overflow", _queue), ("sparse_columns", _sparse), ("single_step", _single_step)] +
    [("point_counts_sp%d" % sp, functools.partial(_point_counts, sp)) for sp in (256, 768, 2048)] +
    [("direct_chunks", _direct_chunks),
     # the largest hypothesis table the sweep takes (J = 109 at M = 255, SP = 256) and the largest split (J = 1, M = 16)
     ("smem_J109_M255_sp256", functools.partial(_smem, 109, 255, 256, (600, 257), (0.7, 0.3))),
     ("smem_J1_M16_sp14848", functools.partial(_smem, 1, 16, 14848, (2 * 14848 + 17, 14848, 14847), (1.0, 0.7, 1.0))),
     # one step past each: the sweep refuses them, AUTO runs DIRECT
     ("smem_J110_M255_sp256", functools.partial(_smem, 110, 255, 256, (300,), (0.3,))),
     ("smem_J1_M16_sp15104", functools.partial(_smem, 1, 16, 15104, (2 * 15104 + 5,), (1.0,))),
     ("kitti_first_match", _kitti)])
NAMES = list(_BUILDERS)
COUNT_NAMES = [n for n in NAMES if n != "kitti_first_match"]


@functools.lru_cache(maxsize=None)
def case(name):
    return _BUILDERS[name]()


def first_match_counts(fr):
    """KITTI reference: bincount of points_in_boxes_gpu's first-match index over the compacted hypotheses."""
    idx = O.points_in_boxes_gpu(fr.pts[None], fr.boxes[None])[0]
    return np.bincount(idx[idx >= 0], minlength=fr.nv).astype(np.int32)
