"""Stage 1b's depth quantiles (csrc/fnp_seeker.cu: stats_kernel, select_pair, select_two) against exact order
statistics, on the depth distributions of depth_select_cases.py that drive the radix select down each of its paths:
refinement levels, the successor key of an earlier level's bin, narrow ranges, ties, select_two's fallback, and
frustums that stream their depth planes from the pages.

(a) fnp_seeker_frustum_stats alone, on a hand-built page pool: every case is one frustum of one launch, its pages
shuffled inside a larger pool whose unused slots and pages hold keys that would move min, max or a quantile if read.
Each quantile must equal torch.quantile of the same fp32 depths on the GPU (the reference's call,
frustum_proposals_v1.py:616-629) and the C oracle bit for bit, and pass the float64 check of depth_select_cases.

(b) Through the real stages: a cfg1 frame salted with walls of points, points behind the camera clamped to depth 1e-5,
and its rows stacked ten times, compared with the oracle stage by stage."""
import ctypes as C

import numpy as np
import pytest
import torch

import depth_select_cases as DS
import oracle as O
import seeker_oracle as SO
from findnpropagate_b200 import _lib, synth
from findnpropagate_b200.seeker import SeekerEngine, camera_matrices
from test_seeker_gpu import _check_against_oracle, _frame_from_synth

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
PG = _lib.PAGE_POINTS
POISON_D = (np.float32(1e-30), np.float32(3e30))        # depths below 1e-5 and above 1e5
POISON_X = (np.float32(-1e30), np.float32(1e30))
CASES = DS.build_cases()


def _d(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


class Pool:
    """The cases as frustums of one stats launch: points in pages of `planes` planes, pages at shuffled places of a
    pool with spare pages; every slot no frustum owns holds poison."""

    def __init__(self, cases, planes, seed):
        rng = np.random.default_rng(seed)
        self.n = np.array([len(c.depths) for c in cases], np.int32)
        npg = (self.n + PG - 1) // PG
        spare = 9
        total = int(npg.sum()) + spare
        alt = np.arange(total * PG).reshape(total, PG) % 2
        pool = np.empty((total, planes, PG), np.float32)
        pool[:, 0:3] = np.where(alt, POISON_X[1], POISON_X[0])[:, None, :]
        pool[:, 3] = np.where(alt, POISON_D[1], POISON_D[0])
        if planes == 5:
            pool[:, 4] = np.int32(-1).view(np.float32)
        place = rng.permutation(total)
        self.stride = int(npg.max()) + 2
        tab = np.zeros((len(cases), self.stride), np.int32)
        tab[:] = place[-1] + 1                             # entries past a frustum's pages name a poison page
        self.xyz = []
        p = 0
        for f, c in enumerate(cases):
            n = len(c.depths)
            order = rng.permutation(n)                     # the ABI leaves the order of a frustum's points open
            xyz = np.random.default_rng(f).uniform(-60, 60, (n, 3)).astype(np.float32)
            self.xyz.append(xyz)
            for k in range(npg[f]):
                sl = order[k * PG:(k + 1) * PG]
                pg = place[p]
                pool[pg, 0:3, :len(sl)] = xyz[sl].T
                pool[pg, 3, :len(sl)] = c.depths[sl]
                tab[f, k] = pg + 1
                p += 1
        self.pool, self.tab, self.planes = _d(pool), _d(tab), planes
        self.npts = _d(self.n)
        self.cap = total * PG

    def run(self, ctx, lq, uq, cq, search_depth=0.0, with_cq=True):
        F, eng = len(self.n), ctx["eng"]
        cfg = _lib.SeekerCfg.from_buffer_copy(eng.cfg)
        cfg.lq, cfg.uq, cfg.cq = lq, uq, cq
        cfg.frustum_min, cfg.max_dist, cfg.search_depth = 0.0, float("inf"), search_depth
        stats = torch.zeros((F, _lib.STATS_FLOATS), dtype=torch.float32, device=DEV)
        centres = torch.zeros((F, eng.M, 3), dtype=torch.float32, device=DEV)
        hyp_dist = torch.zeros(16, dtype=torch.float32, device=DEV)
        status = torch.zeros(8, dtype=torch.int32, device=DEV)            # the kernel skips every frustum otherwise
        b = _lib.SeekerBatch(
            n_frames=1, n_cands=F, n_tiles=0, max_cands_per_frame=F, cam_mats=ctx["mats"].data_ptr(),
            cand_frame=ctx["frame"].data_ptr(), cand_cam=ctx["cam"].data_ptr(),
            cand_box2d=ctx["box"].data_ptr(), mags=eng.mags.data_ptr(), cand_npts=self.npts.data_ptr(),
            page_tab=self.tab.data_ptr(), page_tab_stride=self.stride, page_planes=self.planes,
            frustum_pts=self.pool.data_ptr(), pts_capacity=self.cap, cand_stats=stats.data_ptr(),
            centres=centres.data_ptr(), split_points=PG, max_items=0, status=status.data_ptr(),
            hyp_dist=hyp_dist.data_ptr() if with_cq else None)
        _lib.check(_lib.lib.fnp_seeker_frustum_stats(C.byref(cfg), C.byref(b), _lib.current_stream()),
                   "fnp_seeker_frustum_stats")
        torch.cuda.synchronize()
        return stats.cpu().numpy(), centres.cpu().numpy()


@pytest.fixture(scope="module")
def ctx():
    """A valid cfg (SeekerEngine.cfg) and the per-candidate inputs the corner and centre-line part of the kernel
    reads: one cfg1 frame's cameras, a 2D box per frustum."""
    cfg = synth.CONFIGS["cfg1"]
    sf = synth.make_frame(0, cfg)
    F = len(CASES)
    return dict(eng=SeekerEngine(synth.seeker_params(cfg), device=DEV),
                mats=_d(camera_matrices(sf.lidar2image[None], sf.camera2lidar[None], sf.camera_intrinsics[None])),
                frame=_d(np.zeros(F, np.int32)), cam=_d((np.arange(F) % 6).astype(np.int32)),
                box=_d(np.tile(np.array([[500.0, 300.0, 900.0, 600.0]], np.float32), (F, 1))))


_REF = {}


def _reference(f, q):
    """(torch.quantile on the GPU, C oracle) of case f at q, bit patterns; cached across launches."""
    key = (f, np.float32(q).tobytes())
    if key not in _REF:
        d = CASES[f].depths
        t = torch.quantile(_d(d), q).item()
        _REF[key] = (np.float32(t), O.quantile(d, q))
    return _REF[key]


def _check_quantiles(stats, lq, uq, cq, what):
    bad = []
    for f, c in enumerate(CASES):
        for j, q in ((0, lq), (1, uq), (2, cq)):
            got = stats[f, j]
            t, o = _reference(f, q)
            if got.tobytes() != t.tobytes() or got.tobytes() != o.tobytes():
                bad.append("%s %s [%d] q=%r: kernel %r, torch.quantile %r, oracle %r" % (what, c.name, j, q, got, t, o))
                continue
            err = DS.fp64_check(c.depths, q, got)
            if err:
                bad.append("%s %s [%d]: %s" % (what, c.name, j, err))
    assert not bad, "\n".join(bad[:20])


SETTINGS = DS.SETTINGS + [("target:" + c.name, *c.setting) for c in CASES]


@pytest.mark.parametrize("planes", [4, 5])
def test_frustum_stats_quantiles_are_exact_order_statistics(ctx, planes):
    pool = Pool(CASES, planes, seed=planes)
    for name, lq, uq, cq in SETTINGS:
        stats, _ = pool.run(ctx, lq, uq, cq)
        _check_quantiles(stats, lq, uq, cq, "%s/planes %d:" % (name, planes))
        if name == "shipped":
            for f, c in enumerate(CASES):        # the point AABB and the count
                xyz = pool.xyz[f]
                assert np.array_equal(_bits(stats[f, 3:6]), _bits(xyz.min(0))), c.name
                assert np.array_equal(_bits(stats[f, 6:9]), _bits(xyz.max(0))), c.name
                assert stats[f, 9] == len(c.depths), c.name


def test_frustum_stats_do_not_depend_on_point_or_page_order(ctx):
    """Shuffling the points within a frustum's pages and the pages within the pool gives the same bits, all of them."""
    a, b = Pool(CASES, 4, seed=11), Pool(CASES, 4, seed=12)
    for _, lq, uq, cq in DS.SETTINGS[:2]:
        sa, ca = a.run(ctx, lq, uq, cq)
        sb, cb = b.run(ctx, lq, uq, cq)
        assert np.array_equal(_bits(sa), _bits(sb)) and np.array_equal(_bits(ca), _bits(cb))


def test_frustum_stats_search_depth_and_without_the_centre_quantile(ctx):
    pool = Pool(CASES, 5, seed=3)
    lq, uq, cq = 0.336, 0.356, 0.46
    ref, _ = pool.run(ctx, lq, uq, cq)
    # hyp_dist = NULL: the cq quantile is not selected; the near and far ones are unchanged
    st, _ = pool.run(ctx, lq, uq, cq, with_cq=False)
    assert np.array_equal(_bits(st[:, 0:2]), _bits(ref[:, 0:2]))
    # search_depth > 0: the far end is the near quantile + depth, and the near quantile is selected on its own
    for sd in (5.0, 0.75):
        st, _ = pool.run(ctx, lq, uq, cq, search_depth=sd)
        assert np.array_equal(_bits(st[:, 0]), _bits(ref[:, 0]))
        assert np.array_equal(_bits(st[:, 1]), _bits(st[:, 0] + np.float32(sd)))
        assert np.array_equal(_bits(st[:, 2]), _bits(ref[:, 2]))


# ---------------------------------------------------------------------------------------------- (b) the real stages
def _salted_frame():
    """A cfg1 frame with two walls in 2D boxes of their own -- a truck's rear at 10 m (3000 points within +-5 cm, 200
    background points at 2 - 50 m) and a small one within +-2 cm of 10.05 m (250 + 25) -- points behind the camera that land on
    the box through the 1e-5 depth clamp, and every row stacked ten times.  The large wall's frustum streams its
    depth planes (> 4096 points), the small one's stays in the shared-memory cache."""
    cfg = synth.CONFIGS["cfg1"]
    sf = synth.make_frame(4, cfg)
    fi = _frame_from_synth(sf)
    cm = camera_matrices(sf.lidar2image, sf.camera2lidar, sf.camera_intrinsics)
    rng = np.random.default_rng(7)
    extra, boxes = [], []
    for cam, box, n_wall, n_bg, at, half in ((0, (620.0, 320.0, 980.0, 580.0), 3000, 200, 10.0, 0.05),
                                             (3, (740.0, 430.0, 820.0, 490.0), 250, 25, 10.05, 0.02)):
        u = rng.uniform(box[0] + 1, box[2] - 1, n_wall + n_bg)
        v = rng.uniform(box[1] + 1, box[3] - 1, n_wall + n_bg)
        d = np.concatenate([at + rng.uniform(-half, half, n_wall), rng.uniform(2.0, 50.0, n_bg)])
        for k in range(n_wall + n_bg):
            extra.append(O.unproject(cm[cam, 12:21], cm[cam, 21:24], u[k], v[k], d[k]))
        L = sf.lidar2image[cam][:3].astype(np.float64)
        for t in np.linspace(0.3, 30.0, 120 if cam == 0 else 8):     # behind the camera: wz = -t, (wx, wy) / 1e-5 in the box
            for a in (0.3, 0.5, 0.7):
                uv = np.array([box[0] + a * (box[2] - box[0]), box[1] + (1 - a) * (box[3] - box[1])]) * 1e-5
                extra.append(np.linalg.solve(L[:, :3], np.array([uv[0], uv[1], -t]) - L[:, 3]))
        boxes.append((cam, box))
    add = np.asarray(extra, np.float32)
    pts = np.concatenate([sf.points, np.concatenate([add, np.zeros((add.shape[0], sf.points.shape[1] - 3), np.float32)], 1)])
    fi.points = np.ascontiguousarray(np.tile(pts.astype(np.float32), (10, 1)))
    fi.det_boxes = np.concatenate([fi.det_boxes, np.array([b for _, b in boxes], np.float32)]).astype(np.float32)
    fi.det_labels = np.concatenate([fi.det_labels, [1, 2]]).astype(np.int64)
    fi.det_scores = np.concatenate([fi.det_scores, [0.99, 0.99]]).astype(np.float32)
    fi.det_cam_idx = np.concatenate([fi.det_cam_idx, [c for c, _ in boxes]]).astype(np.int64)
    return fi


@pytest.mark.parametrize("quant", [dict(), dict(lq=0.336, uq=0.356, cq=0.46, dst_w=0.226), dict(lq=0.25, search_depth=5.0)],
                         ids=["shipped", "kitti_interior", "search_depth"])
def test_salted_frame_through_the_stages_vs_oracle(quant, monkeypatch):
    cfg = synth.CONFIGS["cfg1"]
    params = synth.seeker_params(cfg)
    params.update(quant)
    fi = _salted_frame()
    recs = []
    seek = SO.seek_frame

    def recording(*a, **k):
        out = seek(*a, **k)
        recs.extend(out["frustums"])
        return out
    monkeypatch.setattr(SO, "seek_frame", recording)
    eng = SeekerEngine(params, device=DEV, debug=True)
    eng.pts_factor = 4.0
    res, n = _check_against_oracle(eng, [fi], params)
    assert n > 10
    p = dict(synth.seeker_params(cfg), **quant)
    deep = {"cached": 0, "streamed": 0}
    clamped = 0
    for r in recs:
        if r["n_points"] == 0:
            continue
        d = r["uvd"][:, 2]
        clamped += int((d == DS.DEPTH_MIN).sum())
        lvl = DS.deepest_level(d, p["lq"], p["uq"], p["cq"], p.get("search_depth") or 0.0, with_cq=eng.use_dist)
        if lvl >= 2:
            deep["streamed" if len(d) > DS.STATS_CACHE else "cached"] += 1
    assert deep["cached"] >= 1 and deep["streamed"] >= 1, deep
    assert clamped > 0
