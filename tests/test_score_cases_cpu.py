"""The stage 2b cases of score_cases.py without a GPU: on every frustum the host model's sweep (tools/sweep_model, the
arithmetic of fnp_sweep.cuh) equals its brute force equals the oracle's count_in_boxes, the counts lie inside the
float64 bracket, and every case reaches the path of the kernels it is named for.  test_score_stage_gpu.py runs the
same cases through the kernels."""
import ctypes as C

import numpy as np
import pytest

import oracle as O
import score_cases as SC
from score_cases import SM

# SweepCol as floats: cosa sina tx ty | m0 m1 pseudo_mask (int) eps | c0[3] inv_s[3] w_in[3] w_p[3]
COL_M0, COL_M1, COL_C0, COL_INV, COL_WIN, COL_WP = 4, 5, 8, 11, 14, 17


@pytest.fixture(scope="module")
def lib():
    return SM.build()


_RUNS = {}


def _run(lib, name):
    """Per frustum: host-model sweep and brute-force counts, statistics, column parameters; cached per case."""
    if name not in _RUNS:
        c = SC.case(name)
        out = []
        for fr in c.frustums:
            cols = np.zeros((c.J, 20), np.float32)
            cs, cb, st = SM.run_frustum(lib, fr.pts, fr.prep, fr.hidx, c.J, c.M, split=c.split, cols_out=cols)
            out.append((cs, cb, st, cols))
        _RUNS[name] = out
    return _RUNS[name]


def _possible_range(col, pts):
    """float64 restatement of sweep_solve's possible range [plo, phi] (before rounding to steps) of every point."""
    p = pts.astype(np.float64)
    ca, sa = np.float64(col[0]), np.float64(col[1])
    P = np.stack([p[:, 0] * ca - p[:, 1] * sa, p[:, 1] * ca + p[:, 0] * sa, p[:, 2]], 1)
    q = (P - col[COL_C0:COL_C0 + 3].astype(np.float64)) * col[COL_INV:COL_INV + 3].astype(np.float64)
    wp = col[COL_WP:COL_WP + 3].astype(np.float64)
    return (q - wp).max(1), (q + wp).min(1)


@pytest.mark.parametrize("name", SC.COUNT_NAMES)
def test_host_sweep_brute_force_oracle_and_bracket_agree(lib, name):
    c = SC.case(name)
    total = loose = decided = undecided_pairs = pairs = 0
    for f, (fr, (cs, cb, st, _)) in enumerate(zip(c.frustums, _run(lib, name))):
        co = O.count_in_boxes(fr.pts, fr.boxes) if fr.nv else np.zeros(0, np.int32)
        assert np.array_equal(cb, co), "%s frustum %d: brute force with in_box() differs from the oracle" % (name, f)
        assert np.array_equal(cs, cb), "%s frustum %d: sweep differs from brute force %s" % (name, f, st)
        lo, hi = fr.bracket()
        bad = np.nonzero((co < lo) | (co > hi))[0]
        assert bad.size == 0, "%s frustum %d: counts %s outside the float64 bracket [%s, %s]" % (
            name, f, co[bad[:5]], lo[bad[:5]], hi[bad[:5]])
        total += int(co.sum())
        loose += int((lo != hi).sum())
        decided += int((lo == hi).sum())
        undecided_pairs += int((hi - lo).sum())
        pairs += fr.n * fr.nv
    assert total > 0
    if c.benign:
        # the bracket has teeth: almost every pair is decided, and most hypotheses have all of theirs decided (not
        # where a frustum of > 10 000 points is counted by a single column: every hypothesis meets a face point there)
        assert undecided_pairs <= 1e-3 * pairs, (name, undecided_pairs, pairs)
        if max(fr.n for fr in c.frustums) < 10000:
            assert decided >= 0.8 * (decided + loose), (name, decided, loose)


def test_adversarial_cases_vary(lib):
    """The 12 adversarial cases cover the ranges they are ported for."""
    Ms, Js, splits = set(), set(), set()
    pairs = unc = 0
    for s in range(12):
        c = SC.case("adversarial_%02d" % s)
        Ms.add(c.M), Js.add(c.J), splits.add(c.split)
        assert len({fr.n for fr in c.frustums}) >= 2 or len(c.frustums) == 1
        for cs, cb, st, _ in _run(lib, c.name):
            pairs += st["pairs"]
            unc += st["pairs_uncertain"]
    assert len(Ms) >= 4 and len(Js) >= 4 and splits == {256, 768, 2048}
    assert unc > 0.05 * pairs


def test_queue_case_overflows_the_queue_with_full_packed_bytes(lib):
    c = SC.case("queue_overflow")
    assert c.M == 255
    pairs = unc = definite = 0
    full = both = 0
    for fr, (cs, cb, st, cols) in zip(c.frustums, _run(lib, c.name)):
        pairs += st["pairs"]
        unc += st["pairs_uncertain"]
        definite += st["pairs_definite"]
        ci = cols.view(np.int32)
        for j in range(c.J):
            assert ci[j, COL_M0] == 0 and ci[j, COL_M1] == 254        # D = 254
            if np.isneginf(cols[j, COL_WIN:COL_WIN + 3]).any():      # t < dl: no definite range in this column
                plo, phi = _possible_range(cols[j], fr.pts)
                full += int(((phi > 255.0) & (plo < 253.0)).sum())     # B = D = 254, so a2 = B + 1 = 255
            else:
                both += 1
        assert fr.n > SC.PG          # several pieces per column: drains before each piece after the first
    assert unc > 0.9 * pairs, "uncertain share %.3f" % (unc / pairs)
    assert definite > 0 and both >= 2 and full > 100


def test_sparse_cases_reach_empty_and_single_step_columns(lib):
    m1_lt_m0 = d0 = gaps = 0
    for name in ("sparse_columns", "single_step"):
        c = SC.case(name)
        for fr, (cs, cb, st, cols) in zip(c.frustums, _run(lib, name)):
            ci = cols.view(np.int32)
            m0, m1 = ci[:, COL_M0], ci[:, COL_M1]
            m1_lt_m0 += int((m1 < m0).sum())
            d0 += int((m1 == m0).sum())
            for j in range(c.J):
                steps = fr.hidx[fr.hidx % c.J == j] // c.J
                if steps.size >= 2 and steps.size < steps[-1] - steps[0] + 1:
                    gaps += 1
    assert SC.case("single_step").M == 1
    assert m1_lt_m0 >= 2 and d0 >= 4 and gaps >= 2
    assert any(fr.nv <= 0.03 * SC.case("sparse_columns").H for fr in SC.case("sparse_columns").frustums)


@pytest.mark.parametrize("SP", [256, 768, 2048])
def test_point_count_cases_cover_the_tails(SP):
    c = SC.case("point_counts_sp%d" % SP)
    ns = [fr.n for fr in c.frustums]
    assert ns == SC.point_count_list(SP) and c.split == SP
    assert {n % 64 for n in ns} >= {0, 1, 2, 63} and {n % 256 for n in ns} >= {0, 1, 255}
    assert max(ns) > 3 * SP                      # several splits add into one row
    # the origin lies inside hypotheses of every frustum with any: a split tail padded with (0, 0, 0) would count
    for fr in c.frustums:
        if fr.nv:
            assert O.count_in_boxes(np.zeros((1, 3), np.float32), fr.boxes).sum() > 0


def test_direct_chunk_case_covers_every_chunk_shape():
    c = SC.case("direct_chunks")
    nvs = [fr.nv for fr in c.frustums]
    assert nvs == SC.DIRECT_NV and all(fr.n % 2 == 1 for fr in c.frustums)
    rem = {(nv % SC.SCORE_CHUNK + 127) // 128 for nv in nvs if nv % SC.SCORE_CHUNK}
    assert rem == {1, 2, 3, 4} and any(nv > 2 * SC.SCORE_CHUNK for nv in nvs)


def test_sweep_shared_memory_formula_and_score_mode():
    """sweep_smem_bytes = 80 J + 24 576 + 12 SP + 4 H + 2 ceil4(H) + 144 <= 204 800: the boundary cases sit on either
    side of it, and fnp_seeker_score_mode agrees with the formula around them."""
    assert SC.sweep_smem_bytes(256, 109 * 255, 109) == 203284 and SC.sweep_admits(109, 255, 256)
    assert SC.sweep_smem_bytes(256, 110 * 255, 110) == 204896 and not SC.sweep_admits(110, 255, 256)
    assert SC.sweep_admits(1, 16, 14848) and not SC.sweep_admits(1, 16, 15104)
    # H <= 32767 (the short slot table) never binds: at the smallest J and split the shared memory refuses H = 29 489
    assert SC.sweep_smem_bytes(256, 29488, 1) <= SC.SMEM_LIMIT < SC.sweep_smem_bytes(256, 29489, 1)
    from findnpropagate_b200 import _lib
    cols = np.zeros(16, np.float32)
    for J, M, SP in [(109, 255, 256), (110, 255, 256), (1, 16, 14848), (1, 16, 15104), (1, 255, 256), (128, 255, 256),
                     (600, 50, 256), (819, 1, 256), (820, 1, 256), (8, 64, 65536), (3, 16, 13056), (3, 16, 13312)]:
        cfg = _lib.SeekerCfg(num_mags=M, num_yaw_size=J)
        b = _lib.SeekerBatch(split_points=SP, sweep_cols=cols.ctypes.data)
        for req, want in ((_lib.SCORE_SWEEP, _lib.SCORE_SWEEP if SC.sweep_admits(J, M, SP) else -1),
                          (_lib.SCORE_AUTO, _lib.SCORE_SWEEP if SC.sweep_admits(J, M, SP) and M >= 16 else _lib.SCORE_DIRECT),
                          (_lib.SCORE_DIRECT, _lib.SCORE_DIRECT)):
            b.score_mode = req
            assert _lib.lib.fnp_seeker_score_mode(C.byref(cfg), C.byref(b)) == want, (J, M, SP, req)


def test_kitti_case_overlaps_and_straddles_the_splits():
    """First-match counts by the oracle, checked against the float64 first match where every deciding box is far
    enough from the point to call; the hypotheses overlap, so first match and plain counts differ."""
    import fp64_geometry as FG
    c = SC.case("kitti_first_match")
    assert [fr.n for fr in c.frustums] == [4095, 4096, 4097, 9000]
    for fr in c.frustums:
        idx = O.points_in_boxes_gpu(fr.pts[None], fr.boxes[None])[0]
        want, margin = FG.points_in_boxes(fr.pts, fr.boxes)
        tol = 2.0 ** -19 * (2 * max(np.abs(fr.pts).max(), np.abs(fr.boxes[:, :3]).max()) + fr.boxes[:, 3:6].max() / 2) + 2e-5
        sure = np.abs(margin) > tol
        assert sure.mean() > 0.99 and np.array_equal(idx[sure], want[sure])
        fm = SC.first_match_counts(fr)
        assert fm.sum() == (idx >= 0).sum() and O.count_in_boxes(fr.pts, fr.boxes).sum() > 1.5 * fm.sum()
