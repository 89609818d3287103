"""The depth-select cases of depth_select_cases.py without a GPU: every case reaches the path it is named for according
to the path model, and the C oracle's quantile (sort plus torch.quantile's fma lerp) passes the float64 check on every
case and setting.  The GPU side is test_depth_select_gpu.py."""
import numpy as np
import pytest

import depth_select_cases as DS
import oracle as O

CASES = DS.build_cases()

# every path the select has, as named by DS.path_tags
PATHS = ["no_select", "all_equal", "level1_shift0", "level1_shift1",
         "refine1_k1_same_bin", "refine1_k1_next_bin", "refine1_k1_above", "refine2_shift0_k1_above", "three_levels",
         "dup_k_first", "dup_k_middle", "dup_k_last", "cached_refine", "streamed_refine",
         "two_same_bin", "two_adjacent_bins", "two_total_496", "two_total_497", "two_same_bin_496", "two_same_bin_497",
         "two_two_lists", "two_fallback", "two_shift0", "two_skipped_lq_gt_uq"]


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_case_reaches_its_path(case):
    tags = DS.path_tags(case)
    assert case.expect <= tags, "%s reaches %s, not %s" % (case.name, sorted(tags), sorted(case.expect - tags))
    d = case.depths
    assert d.dtype == np.float32 and d.min() >= DS.DEPTH_MIN and d.max() <= DS.DEPTH_MAX


def test_every_path_is_reached(capsys):
    by_path = {p: [c.name for c in CASES if p in DS.path_tags(c)] for p in PATHS}
    with capsys.disabled():
        print()
        for p in PATHS:
            print("  %-24s %s" % (p, ", ".join(by_path[p]) or "-"))
    assert all(by_path.values()), [p for p, v in by_path.items() if not v]
    sizes = {len(c.depths) for c in CASES}
    assert {1, 2, 3, 5, 4095, 4096, 4097} <= sizes and max(sizes) > 200_000
    assert any(n > DS.STATS_CACHE and n % 4 and n % 256 for n in sizes)


def test_settings_cover_the_weights():
    """Across cases and settings: interior positions with w = 0, 0 < w < 0.5 and w >= 0.5, and the ends q = 0, 1."""
    seen = set()
    for c in CASES:
        for _, lq, uq, cq in DS.SETTINGS:
            seen |= {DS.weight_class(len(c.depths), q) for q in (lq, uq, cq)}
    assert {"w0", "w_lt_half", "w_ge_half", None} <= seen


def test_path_model_on_hand_checked_keys():
    """The model itself, on keys whose bins are worked out by hand."""
    k = DS.K10
    # range 2^24 - 1 -> shift 13; 600 keys k .. k + 599 in level-1 bin 1024, refined by 4-ulp bins (shift 2)
    d = DS.depths_of(np.concatenate([[k - (1 << 23), k + (1 << 23) - 1], k + np.arange(600)]))
    p = DS.select_pair_path(d, 600)          # key k + 599: the last of the crowded bin, its successor is kmax
    assert p == dict(exit="rank_count", levels=[dict(shift=13, bin=1024, count=600, next="next_bin"),
                                                dict(shift=2, bin=149, count=4, next="above")])
    p = DS.select_pair_path(d, 598)          # key k + 597: its successor is in the same 4-ulp bin
    assert p["levels"][1] == dict(shift=2, bin=149, count=4, next="same_bin")
    p = DS.select_pair_path(d, 596)          # key k + 595: the last of 4-ulp bin 148
    assert p["levels"][1] == dict(shift=2, bin=148, count=4, next="next_bin")
    # narrow: 2047 ulps -> shift 0, one key per bin
    d = DS.depths_of(k + np.array([0, 5, 2047]))
    assert DS.select_pair_path(d, 1) == dict(exit="exact", levels=[dict(shift=0, bin=5, count=1, next="next_bin")])
    assert DS.select_two_path(d, 0, 1)["exit"] == "exact"
    # the kernel's dispatch: lq = 0 is the minimum, lq > uq selects per rank
    sel = DS.stats_selects(DS.depths_of(k + np.arange(100)), 0.0, 0.25, 1.0)
    assert [(r, kind) for r, kind, _ in sel] == [("lq", "min"), ("uq", "pair"), ("cq", "max")]
    sel = DS.stats_selects(DS.depths_of(k + np.arange(100)), 0.6, 0.4, 0.5, with_cq=False)
    assert [(r, kind) for r, kind, _ in sel] == [("lq", "pair"), ("uq", "pair")]
    sel = DS.stats_selects(DS.depths_of(k + np.arange(100)), 0.3, 0.4, 0.5, search_depth=2.0)
    assert [(r, kind) for r, kind, _ in sel] == [("lq", "pair"), ("cq", "pair")]


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_oracle_quantile_passes_the_fp64_check(case):
    d = case.depths
    qs = {q for _, lq, uq, cq in DS.SETTINGS for q in (lq, uq, cq)} | set(case.setting)
    for q in sorted(qs):
        err = DS.fp64_check(d, q, O.quantile(d, q))
        assert err is None, err
