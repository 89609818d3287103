"""Stage 2b's kernels (csrc/fnp_seeker.cu: score_kernel in DIRECT mode, sweep_prep_kernel + sweep_score_kernel in SWEEP
mode, firstmatch_kernel in the KITTI variant) on the frustums of score_cases.py, driven through fnp_seeker_score
alone on a page pool this file builds: every frustum's pages lie at shuffled places of the pool, between spare pages
and behind page-table entries that hold points inside the frustum's hypotheses, and so do the unused slots of a
frustum's last page, so that any read past a frustum's points changes a count.

Every valid hypothesis must count exactly what the oracle's count_in_boxes counts (first-match counts in the KITTI
variant), in DIRECT mode and, wherever fnp_seeker_score_mode admits it, in SWEEP mode.  test_score_cases_cpu.py holds
the same cases against the host model and a float64 bracket.  Run with -s for the uncertain-pair share of the queue
case, the boundary configurations and the largest case's time."""
import ctypes as C

import numpy as np
import pytest
import torch

import oracle as O
import score_cases as SC
from findnpropagate_b200 import _lib

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
PG = _lib.PAGE_POINTS
MODES = {"direct": _lib.SCORE_DIRECT, "sweep": _lib.SCORE_SWEEP, "auto": _lib.SCORE_AUTO}


def _d(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


class Stage:
    """One fnp_seeker_score call over the frustums of a case.  seed: placement of the pages in the pool;
    permute: also shuffle each frustum's points across its pages."""

    def __init__(self, case, seed=0, permute=False, stride=None):
        rng = np.random.default_rng(seed)
        self.case = case
        F, H = len(case.frustums), case.H
        n = np.array([fr.n for fr in case.frustums], np.int64)
        npg = (n + PG - 1) // PG
        spare = 3
        total = int(npg.sum()) + spare
        # poison: centres of the case's hypotheses, inside them by construction
        centres = np.concatenate([fr.boxes[:, :3] for fr in case.frustums if fr.nv])
        pool = np.zeros((total, 4, PG), np.float32)
        pool[:, :3] = centres[rng.integers(0, centres.shape[0], (total, PG))].transpose(0, 2, 1)
        place = rng.permutation(total)
        self.stride = int(stride if stride is not None else npg.max() + 1)
        tab = np.full((F, self.stride), place[-1] + 1, np.int32)        # past a frustum's pages: a poison page
        p = 0
        for f, fr in enumerate(case.frustums):
            order = rng.permutation(fr.n) if permute else np.arange(fr.n)
            own = fr.boxes[:, :3] if fr.nv else centres
            for k in range(int(npg[f])):
                sl = order[k * PG:(k + 1) * PG]
                pg = place[p]
                pool[pg, :3] = own[rng.integers(0, own.shape[0], PG)].T    # the tail of the last page: poison too
                pool[pg, :3, :len(sl)] = fr.pts[sl].T
                tab[f, k] = pg + 1
                p += 1
        stats = np.zeros((F, _lib.STATS_FLOATS), np.float32)
        prep = np.tile(np.array([0, 0, 0, 1e30, 1, 0, 1e30, 1e30], np.float32), (F, H, 1))   # contains everything
        hidx = np.zeros((F, H), np.int32)
        for f, fr in enumerate(case.frustums):
            if fr.n:
                stats[f, 3:6], stats[f, 6:9], stats[f, 9] = fr.pts.min(0), fr.pts.max(0), fr.n
            prep[f, :fr.nv] = fr.prep
            hidx[f, :fr.nv] = fr.hidx
        self.t = dict(pool=_d(pool), tab=_d(tab), npts=_d(n.astype(np.int32)), stats=_d(stats), prep=_d(prep),
                      hidx=_d(hidx), nvalid=_d(np.array([fr.nv for fr in case.frustums], np.int32)),
                      cols=torch.zeros((F, case.J, _lib.SWEEP_COL_FLOATS), dtype=torch.float32, device=DEV),
                      counts=torch.zeros((F, H), dtype=torch.int32, device=DEV),
                      item_start=torch.zeros(F + 1, dtype=torch.int32, device=DEV),
                      status=torch.zeros(8, dtype=torch.int32, device=DEV))
        self.cap = total * PG

    def batch(self, mode, max_items):
        t = self.t
        t["items"] = torch.zeros((max(max_items, 1), 4), dtype=torch.int32, device=DEV)
        return _lib.SeekerBatch(
            n_frames=1, n_cands=len(self.case.frustums), n_tiles=0, max_cands_per_frame=len(self.case.frustums),
            cand_npts=t["npts"].data_ptr(), page_tab=t["tab"].data_ptr(), page_tab_stride=self.stride, page_planes=4,
            frustum_pts=t["pool"].data_ptr(), pts_capacity=self.cap, cand_stats=t["stats"].data_ptr(),
            hyp_prep=t["prep"].data_ptr(), hyp_index=t["hidx"].data_ptr(), hyp_nvalid=t["nvalid"].data_ptr(),
            split_points=self.case.split, max_items=max_items, cand_item_start=t["item_start"].data_ptr(),
            items=t["items"].data_ptr(), counts=t["counts"].data_ptr(), score_mode=MODES[mode],
            sweep_cols=t["cols"].data_ptr(), status=t["status"].data_ptr())

    def cfg(self):
        kitti = self.case.kind == "kitti"
        return _lib.SeekerCfg(num_mags=self.case.M, num_yaw_size=self.case.J,
                              variant=_lib.VARIANT_KITTI if kitti else _lib.VARIANT_NUSCENES)

    def mode_of(self, mode):
        return _lib.lib.fnp_seeker_score_mode(C.byref(self.cfg()), C.byref(self.batch(mode, 1)))

    def run(self, mode, max_items=None, timed=False):
        """-> counts (F, H), status (8), milliseconds of the call (timed) or None"""
        if max_items is None:
            max_items = SC.items_needed(self.case, self.mode_of(mode) == _lib.SCORE_SWEEP)
        cfg, b = self.cfg(), self.batch(mode, max_items)
        self.t["counts"].fill_(-7)          # fnp_seeker_score zeroes the table itself
        self.t["status"].zero_()
        ms = None
        if timed:
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            ev[0].record()
        _lib.check(_lib.lib.fnp_seeker_score(C.byref(cfg), C.byref(b), _lib.current_stream()), "fnp_seeker_score")
        if timed:
            ev[1].record()
        torch.cuda.synchronize()
        if timed:
            ms = ev[0].elapsed_time(ev[1])
        return self.t["counts"].cpu().numpy(), self.t["status"].cpu().numpy(), ms


_ORACLE = {}


def _oracle(case):
    if case.name not in _ORACLE:
        ref = SC.first_match_counts if case.kind == "kitti" else (lambda fr: O.count_in_boxes(fr.pts, fr.boxes))
        _ORACLE[case.name] = [ref(fr) if fr.nv else np.zeros(0, np.int32) for fr in case.frustums]
    return _ORACLE[case.name]


def _check(case, counts, what):
    bad = []
    for f, (fr, want) in enumerate(zip(case.frustums, _oracle(case))):
        got = counts[f, :fr.nv]
        if not np.array_equal(got, want):
            i = np.nonzero(got != want)[0]
            bad.append("%s %s frustum %d (n %d, nv %d): %d hypotheses differ, e.g. slot %s: %s != oracle %s" % (
                case.name, what, f, fr.n, fr.nv, i.size, i[:4], got[i[:4]], want[i[:4]]))
    assert not bad, "\n".join(bad)


def _modes(stage):
    out = ["direct"]
    if stage.mode_of("sweep") == _lib.SCORE_SWEEP:
        out.append("sweep")
    return out


@pytest.mark.parametrize("name", [n for n in SC.COUNT_NAMES if not n.startswith("smem_")])
def test_counts_equal_the_oracle_in_both_modes(name):
    case = SC.case(name)
    st = Stage(case, seed=SC.NAMES.index(name))
    modes = _modes(st)
    assert "sweep" in modes, name
    got = {}
    for mode in modes:
        counts, status, _ = st.run(mode)
        assert status[0] == 0 and status[2] == SC.items_needed(case, mode == "sweep")
        _check(case, counts, mode)
        got[mode] = counts
    assert np.array_equal(got["direct"], got["sweep"])
    if name == "queue_overflow":
        lib = SC.SM.build()
        pairs = unc = 0
        for fr in case.frustums:
            _, _, s = SC.SM.run_frustum(lib, fr.pts, fr.prep, fr.hidx, case.J, case.M, split=case.split)
            pairs, unc = pairs + s["pairs"], unc + s["pairs_uncertain"]
        print("\n%s: uncertain (point, column) pairs %d of %d = %.3f" % (name, unc, pairs, unc / pairs))


def test_counts_do_not_depend_on_page_or_point_order():
    for name in ("adversarial_00", "queue_overflow", "direct_chunks", "point_counts_sp768"):
        case = SC.case(name)
        a, b = Stage(case, seed=1), Stage(case, seed=2, permute=True)
        for mode in ("direct", "sweep"):
            ca, cb = a.run(mode)[0], b.run(mode)[0]
            for f, fr in enumerate(case.frustums):
                assert np.array_equal(ca[f, :fr.nv], cb[f, :fr.nv]), (name, mode, f)


def test_shared_memory_boundary_of_the_sweep():
    """sweep_smem_bytes(SP, H, J) = 80 J + 24 576 + 12 SP + 4 H + 2 ceil4(H) + 144 must stay <= 204 800 B.  The largest
    accepted table (J = 109, M = 255, SP = 256: H = 27 795, 203 284 B) and the largest accepted split (J = 1, M = 16,
    SP = 14 848) run in SWEEP and in DIRECT; one step past each (J = 110: 204 896 B; SP = 15 104) SWEEP is refused with
    FNP_EINVAL and AUTO runs DIRECT.  The H <= 32767 guard of the short slot table cannot be reached under this bound
    (J = 1, SP = 256 already stops at H = 29 488)."""
    for name, admit in (("smem_J109_M255_sp256", True), ("smem_J1_M16_sp14848", True),
                        ("smem_J110_M255_sp256", False), ("smem_J1_M16_sp15104", False)):
        case = SC.case(name)
        st = Stage(case, seed=5)
        smem = SC.sweep_smem_bytes(case.split, case.H, case.J)
        m_sweep, m_auto = st.mode_of("sweep"), st.mode_of("auto")
        print("\n%s: H %d, %d B of shared memory: SWEEP request -> %d, AUTO -> %d (%s)" % (
            name, case.H, smem, m_sweep, m_auto, "accepted" if admit else "refused"))
        assert (smem <= SC.SMEM_LIMIT) == admit == SC.sweep_admits(case.J, case.M, case.split)
        if admit:
            assert m_sweep == _lib.SCORE_SWEEP and m_auto == _lib.SCORE_SWEEP
            cs, status, _ = st.run("sweep")
            assert status[0] == 0
            _check(case, cs, "sweep")
            cd, _, _ = st.run("direct")
            _check(case, cd, "direct")
            assert np.array_equal(cs, cd)
        else:
            assert m_sweep == -1                 # FNP_EINVAL
            assert m_auto == _lib.SCORE_DIRECT
            rc = _lib.lib.fnp_seeker_score(C.byref(st.cfg()), C.byref(st.batch("sweep", 1)), _lib.current_stream())
            assert rc == -1
            ca, status, _ = st.run("auto")
            assert status[0] == 0
            _check(case, ca, "auto")


@pytest.mark.parametrize("mode", ["direct", "sweep"])
def test_item_capacity_one_short_and_exact(mode):
    case = SC.case("direct_chunks")
    st = Stage(case, seed=3)
    need = SC.items_needed(case, mode == "sweep")
    assert need > 2
    counts, status, _ = st.run(mode, max_items=need - 1)
    assert status[0] & 2 and status[2] == need
    assert not counts.any()
    counts, status, _ = st.run(mode, max_items=need)
    assert status[0] == 0 and status[2] == need
    _check(case, counts, mode)


def test_kitti_first_match_counts():
    """firstmatch_kernel: a point counts for the first hypothesis, in compacted order, that contains it; frustums of
    4095 - 9000 points with page_tab_stride at its least allowed value, ceil(largest / 256) + 1."""
    case = SC.case("kitti_first_match")
    st = Stage(case, seed=4, stride=-(-max(fr.n for fr in case.frustums) // PG) + 1)
    assert st.stride == 37
    counts, status, _ = st.run("direct", max_items=1)
    _check(case, counts, "kitti")
    assert not counts[:, max(fr.nv for fr in case.frustums):].any()


def test_largest_case_time():
    """The time of fnp_seeker_score on the largest table (J = 109, M = 255), after a warm-up call, in both modes."""
    case = SC.case("smem_J109_M255_sp256")
    st = Stage(case, seed=6)
    for mode in ("sweep", "direct"):
        st.run(mode)
        _, _, ms = st.run(mode, timed=True)
        print("\n%s %s: %.3f ms (%d points x %d valid hypotheses)" % (
            case.name, mode, ms, sum(fr.n for fr in case.frustums), sum(fr.nv for fr in case.frustums)))


def test_sweep_columns_share_size_and_heading_on_a_pipeline_frame():
    """sweep_prep_kernel reads a column's rotation and size from its first valid hypothesis only: on a cfg2 frame with
    clamp_bottom and search_depth, every valid hypothesis of a column carries the same dx, dy, dz and heading bits."""
    from findnpropagate_b200 import synth
    from findnpropagate_b200.seeker import SeekerEngine
    from test_seeker_gpu import _frame_from_synth
    cfg = synth.CONFIGS["cfg2"]
    params = dict(synth.seeker_params(cfg), clamp_bottom=1, search_depth=5.0)
    frames = [_frame_from_synth(synth.make_frame(3, cfg, device=DEV))]
    eng = SeekerEngine(params, device=DEV, debug=True)
    h = eng.execute(eng.plan(frames), eng.upload_points(frames))
    res = eng.finish(h)
    assert eng.last_score_mode == "sweep"
    dbg = eng.debug_views(h)
    J, nv = eng.J, res["cand_nvalid"]
    checked = 0
    for f in range(nv.shape[0]):
        idx = dbg["hyp_index"][f, :nv[f]]
        bits = np.ascontiguousarray(dbg["hyp_boxes"][f][idx][:, 3:7], np.float32).view(np.uint32)
        for j in np.unique(idx % J):
            rows = bits[idx % J == j]
            assert (rows == rows[0]).all(), "frustum %d column %d" % (f, j)
            checked += rows.shape[0] > 1
    assert checked > 100
