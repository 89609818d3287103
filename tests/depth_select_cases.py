"""Depth distributions that drive stage 1b's radix select (csrc/fnp_seeker.cu: select_pair, select_two,
block_quantile, stats_kernel) down each of its paths, and a model of the select's decisions.

The model restates which bins the kernel picks, when it refines, where it finds the (k+1)-th key and which exit it
takes.  It is used only to prove that a case reaches the path it is named for; the expected values of the tests are
torch.quantile, the C oracle's sort, and the float64 check `fp64_check`.

Keys are the bit patterns of the fp32 depths.  The cull clamps depths to [1e-5, 1e5], so they are positive and their
bit patterns order like the values."""
from dataclasses import dataclass, field

import numpy as np

SEL_BITS, SEL_BINS = 11, 2048
SEL_LIST = 512                 # kSelList: a bin of at most this many keys is finished by rank counting
TWO_LIST = SEL_LIST - 16       # select_two finishes both ranks when its lists hold at most this many keys
STATS_CACHE = 4096             # kStatsCache: larger frustums stream every pass from the pages' depth planes
DEPTH_MIN, DEPTH_MAX = np.float32(1e-5), np.float32(1e5)

# (name, lq, uq, cq) run on every case
SETTINGS = [
    ("shipped", 0.0, 0.25, 1.0),           # tools/cfgs/nuscenes_box_seeker_proposals.yaml
    ("kitti", 0.336, 0.356, 0.46),         # frustum_proposals_v1_kitti.py:41
    ("ends", 0.0, 1.0, 0.5),               # q = 0, 1 and 0.5
    ("half", 0.5, 0.5, 0.0),               # the same rank twice; w = 0 for odd n
    ("reversed", 0.6, 0.4, 0.75),          # lq > uq: the kernel selects each rank on its own
    ("spread", 0.1, 0.9, 0.3),
]


def keys_of(depths):
    return np.ascontiguousarray(depths, np.float32).view(np.uint32).astype(np.int64)


def depths_of(keys):
    return np.asarray(keys, np.int64).astype(np.uint32).view(np.float32)


def position(n, q):
    """torch.quantile's position in fp32: (rank below, rank above, weight)."""
    pos = np.float32(q) * np.float32(n - 1)
    lo, hi = np.floor(pos), np.ceil(pos)
    return int(lo), int(hi), np.float32(pos - lo)


def q_for_rank(n, k, frac=0.5):
    """An fp32 q whose position q * (n - 1) lies strictly between k and k + 1."""
    q = np.float32((k + frac) / (n - 1))
    klo, khi, w = position(n, q)
    assert klo == k and khi == k + 1 and 0 < w < 1, (n, k, q)
    return float(q)


# ---------------------------------------------------------------------------------------------- path model
def select_pair_path(depths, k):
    """select_pair's decisions for rank k: per level the shift, the bin holding the rank, its count and where the
    (k+1)-th key is ("same_bin", "next_bin" of this level, "above" = the next bin of an earlier level, "none"), then
    the exit ("all_equal", "exact" when a bin is one key, "rank_count")."""
    keys = keys_of(depths)
    kmin, kmax = int(keys.min()), int(keys.max())
    if kmin == kmax:
        return dict(exit="all_equal", levels=[])
    rel = keys - kmin
    shift = max(0, (kmax - kmin).bit_length() - SEL_BITS)
    pshift, lo_rel, rank = 32, 0, k
    pending, above = None, False
    levels = []
    while True:
        inset = np.ones(rel.shape, bool) if pshift == 32 else (rel >> pshift) == (lo_rel >> pshift)
        if pending is not None:                       # the kernel takes its minimum in this level's histogram pass
            nb_lo, nb_shift = pending
            assert ((rel >> nb_shift) == (nb_lo >> nb_shift)).any()
            above, pending = True, None
        hist = np.bincount((rel[inset] >> shift) & (SEL_BINS - 1), minlength=SEL_BINS)
        cum = np.cumsum(hist)
        B = int(np.searchsorted(cum, rank, side="right"))
        below, cB = int(cum[B] - hist[B]), int(hist[B])
        nz = np.flatnonzero(hist[B + 1:])
        Bn = B + 1 + int(nz[0]) if nz.size else None
        rank -= below
        hi_part = 0 if pshift == 32 else (lo_rel >> pshift) << pshift
        nxt = "same_bin" if rank + 1 < cB else "next_bin" if Bn is not None else "above" if above else "none"
        levels.append(dict(shift=shift, bin=B, count=cB, next=nxt))
        if shift == 0:
            return dict(exit="exact", levels=levels)
        if cB <= SEL_LIST:
            return dict(exit="rank_count", levels=levels)
        if Bn is not None:
            pending = (hi_part | (Bn << shift), shift)
        lo_rel, pshift, shift = hi_part | (B << shift), shift, max(0, shift - SEL_BITS)


def select_two_path(depths, k1, k2):
    """select_two's decisions for ranks k1 <= k2 (level 1 only): the bins, their counts, and whether the two lists fit
    (exit "two_lists") or the kernel falls back to select_pair per rank ("fallback")."""
    keys = keys_of(depths)
    kmin, kmax = int(keys.min()), int(keys.max())
    if kmin == kmax:
        return dict(exit="all_equal")
    shift = max(0, (kmax - kmin).bit_length() - SEL_BITS)
    hist = np.bincount(((keys - kmin) >> shift) & (SEL_BINS - 1), minlength=SEL_BINS)
    cum = np.cumsum(hist)
    B1, B2 = (int(np.searchsorted(cum, k, side="right")) for k in (k1, k2))
    c1, c2 = int(hist[B1]), int(hist[B2])
    same = B1 == B2
    total = c1 if same else c1 + c2
    out = dict(shift=shift, same=same, adjacent=B2 == B1 + 1, c1=c1, c2=c2, total=total)
    if shift == 0:
        return dict(out, exit="exact")
    return dict(out, exit="fallback" if total > TWO_LIST else "two_lists")


def stats_selects(depths, lq, uq, cq, search_depth=0.0, with_cq=True):
    """The selects stats_kernel runs for one frustum: a list of (role, kind, detail).  kind "two" is select_two on
    (lq, uq), "pair" select_pair on one rank, "min"/"max" an end of the range that needs no select."""
    n = len(depths)
    out = []
    both = False
    if not search_depth > 0:
        klo1, khi1, _ = position(n, lq)
        klo2, khi2, _ = position(n, uq)
        if khi1 != 0 and klo1 != n - 1 and khi2 != 0 and klo2 != n - 1 and klo1 <= klo2:
            p = select_two_path(depths, klo1, klo2)
            out.append(("lq+uq", "two", p))
            both = p["exit"] != "fallback"

    def single(role, q):
        klo, khi, _ = position(n, q)
        if khi == 0:
            return (role, "min", None)
        if klo == n - 1:
            return (role, "max", None)
        return (role, "pair", select_pair_path(depths, klo))
    if not both:
        out.append(single("lq", lq))
        if not search_depth > 0:
            out.append(single("uq", uq))
    if with_cq:
        out.append(single("cq", cq))
    return out


def deepest_level(depths, lq, uq, cq, search_depth=0.0, with_cq=True):
    """The most levels a select_pair of the frustum runs (0 when none runs)."""
    sel = stats_selects(depths, lq, uq, cq, search_depth, with_cq)
    return max([len(p["levels"]) for _, kind, p in sel if kind == "pair"], default=0)


def run_position(depths, k):
    """Where rank k lies in its run of equal keys: "single", "first", "middle" or "last"."""
    s = np.sort(np.asarray(depths, np.float32))
    lo = int(np.searchsorted(s, s[k], side="left"))
    hi = int(np.searchsorted(s, s[k], side="right")) - 1
    if lo == hi:
        return "single"
    return "first" if k == lo else "last" if k == hi else "middle"


def path_tags(case):
    """The named paths a case reaches under its own setting, according to the model."""
    d, (lq, uq, cq) = case.depths, case.setting
    n = len(d)
    tags = set()
    for role, kind, p in stats_selects(d, lq, uq, cq):
        if kind == "pair":
            lv = p["levels"]
            if p["exit"] == "all_equal":
                tags.add("all_equal")
                continue
            if len(lv) == 1 and lv[0]["shift"] == 0:
                tags.add("level1_shift0")
            if lv[0]["shift"] == 1:
                tags.add("level1_shift1")
            if len(lv) == 2 and p["exit"] == "rank_count":
                tags.add("refine1_k1_" + lv[-1]["next"])
            if len(lv) >= 3 and lv[-1]["shift"] == 0 and lv[-1]["next"] == "above":
                tags.add("refine2_shift0_k1_above")
            if len(lv) >= 3:
                tags.add("three_levels")
            if len(lv) >= 2:
                tags.add("streamed_refine" if n > STATS_CACHE else "cached_refine")
            klo = position(n, {"lq": lq, "uq": uq, "cq": cq}[role])[0]
            rp = run_position(d, klo)
            if rp != "single":
                tags.add("dup_k_" + rp)
        elif kind == "two":
            if p["exit"] == "all_equal":
                tags.add("all_equal")
                continue
            if p["exit"] == "exact":
                tags.add("two_shift0")
                continue
            if p["same"]:
                tags.add("two_same_bin")
                if p["total"] in (TWO_LIST, TWO_LIST + 1):
                    tags.add("two_same_bin_%d" % p["total"])
            else:
                if p["adjacent"]:
                    tags.add("two_adjacent_bins")
                if p["total"] in (TWO_LIST, TWO_LIST + 1):
                    tags.add("two_total_%d" % p["total"])
            tags.add("two_" + p["exit"])
    klo1, khi1, _ = position(n, lq)
    klo2, khi2, _ = position(n, uq)
    if klo1 > klo2 and khi2 != 0 and klo1 != n - 1:
        tags.add("two_skipped_lq_gt_uq")
    if not any(kind == "pair" or kind == "two" for _, kind, _ in stats_selects(d, lq, uq, cq)):
        tags.add("no_select")
    return tags


def weight_class(n, q):
    """"w0", "w_lt_half" or "w_ge_half" for an interior position, None at an end of the range."""
    klo, khi, w = position(n, q)
    if khi == 0 or klo == n - 1:
        return None
    return "w0" if w == 0 else "w_lt_half" if w < 0.5 else "w_ge_half"


# ---------------------------------------------------------------------------------------------- float64 check
def fp64_check(depths, q, got):
    """The fp32 result of quantile q must lie between the two exactly sorted keys around the fp32 position and within
    one fp32 ulp of their float64 lerp.  Returns an error message, or None."""
    s = np.sort(np.asarray(depths, np.float32).astype(np.float64))
    klo, khi, w = position(len(s), q)
    exact = s[klo] + float(w) * (s[khi] - s[klo])
    g = float(np.float32(got))
    if not s[klo] <= g <= s[khi]:
        return "q=%r: %r outside [s[%d], s[%d]] = [%r, %r]" % (q, g, klo, khi, s[klo], s[khi])
    ulp = float(np.spacing(np.float32(abs(exact))))
    if abs(g - exact) > ulp:
        return "q=%r: %r is %.3g ulp from the float64 lerp %r" % (q, g, abs(g - exact) / ulp, exact)
    return None


# ---------------------------------------------------------------------------------------------- cases
@dataclass
class Case:
    name: str
    depths: np.ndarray                       # float32, shuffled
    setting: tuple                           # (lq, uq, cq) that drives the case down its path
    expect: set = field(default_factory=set)  # path tags the case must reach


K10 = int(np.float32(10.0).view(np.uint32))


def _mk(rng, keys):
    d = depths_of(rng.permutation(np.asarray(keys, np.int64)))
    assert d.min() >= DEPTH_MIN and d.max() <= DEPTH_MAX and np.isfinite(d).all()
    return d


def _single(name, rng, keys, k, expect, frac=0.5):
    """A case whose uq (and cq) target rank k of the sorted keys; lq = 0 is the minimum, as shipped."""
    keys = np.sort(np.asarray(keys, np.int64))
    q = q_for_rank(len(keys), k, frac)
    return Case(name, _mk(rng, keys), (0.0, q, q), set(expect))


def _two(name, rng, keys, k1, k2, expect, cq=0.5):
    keys = np.sort(np.asarray(keys, np.int64))
    n = len(keys)
    return Case(name, _mk(rng, keys), (q_for_rank(n, k1), q_for_rank(n, k2), cq), set(expect))


def _background(rng, kmin, kmax, n, avoid=None):
    """n keys spread over [kmin, kmax] (both ends included), none in the key range `avoid` = (lo, hi)."""
    b = rng.integers(kmin, kmax + 1, 4 * n)
    if avoid is not None:
        b = b[(b < avoid[0]) | (b >= avoid[1])]
    return np.concatenate([[kmin, kmax], b[:n - 2]])


def _wall(rng, n_wall, n_bg, half=0.05, centre=10.0, near=2.0, far=50.0):
    """A wall or a truck's rear: n_wall depths within +-half of `centre`, n_bg background depths in [near, far]."""
    w = np.float32(centre) + rng.uniform(-half, half, n_wall).astype(np.float32)
    b = rng.uniform(near, far, n_bg).astype(np.float32)
    return keys_of(np.concatenate([w, b]))


def build_cases(seed=20261021):
    rng = np.random.default_rng(seed)
    cases = []
    # ---- all keys equal; n = 1 selects nothing (every rank is an end of the range)
    for n in (1, 2, 3, 5):
        cases.append(Case("equal_n%d" % n, np.full(n, np.float32(7.25)), (0.0, 0.5, 0.5),
                          {"no_select"} if n == 1 else {"all_equal"}))
    # ---- narrow ranges: every key within 2047 ulps (shift 0 at level 1), 2048 and 4095 ulps (shift 1)
    for r, tag in ((2047, "level1_shift0"), (2048, "level1_shift1"), (4095, "level1_shift1")):
        keys = np.sort(_background(rng, K10, K10 + r, 700))
        cases.append(_single("narrow_%d" % r, rng, keys, 350, {tag}))
    # ---- one crowded level-1 bin (8192 ulps: range 2^24 - 1, shift 13), refined once by 4-ulp bins (shift 2) holding
    # 3 keys each; the rank's successor in the same 4-ulp bin, in the next one, or in the next level-1 bin (`above`)
    kmin = K10 - (1 << 23)
    kmax = kmin + (1 << 24) - 1
    lo = kmin + 1024 * 8192
    clus = (lo + 4 * np.arange(300)[:, None] + np.arange(3)[None, :]).reshape(-1)          # 900 keys
    bg = _background(rng, kmin, kmax, 300, avoid=(lo, lo + 8192))
    keys = np.sort(np.concatenate([clus, bg]))
    below = int((bg < lo).sum())
    cases.append(_single("refine1_same_bin", rng, keys, below + 3 * 150, {"refine1_k1_same_bin", "cached_refine"}))
    cases.append(_single("refine1_next_bin", rng, keys, below + 3 * 150 + 2, {"refine1_k1_next_bin"}))
    cases.append(_single("refine1_above", rng, keys, below + 899, {"refine1_k1_above"}))
    # ---- crowded twice: 600 keys within one 4-ulp bin, refined to shift 0; the successor of the bin's last key is the
    # minimum of the next level-1 bin (above_l1) or of the next 4-ulp bin (above_l2), found lazily a level later
    dense = lo + 4 * 700 + rng.integers(0, 4, 600)
    dense[:4] = lo + 4 * 700 + np.arange(4)
    for name, extra in (("refine2_above_l1", np.zeros(0, np.int64)), ("refine2_above_l2", lo + 4 * 700 + 4 + 4 * np.arange(50))):
        keys = np.sort(np.concatenate([dense, extra, bg]))
        cases.append(_single(name, rng, keys, below + 599, {"refine2_shift0_k1_above", "three_levels"}))
    # ---- the clamp values 1e-5 and 1e5 at both ends of a dense cluster: 2^28 ulps, three levels
    k_lo, k_hi = int(DEPTH_MIN.view(np.uint32)), int(DEPTH_MAX.view(np.uint32))
    clus = K10 + rng.integers(0, 100, 1500)
    keys = np.sort(np.concatenate([[k_lo] * 7, clus, [k_hi] * 5]))
    cases.append(_single("clamp_ends", rng, keys, 7 + 700, {"three_levels"}, frac=0.3))
    cases.append(_single("clamp_ends_last", rng, keys, 7 + 1499, {"three_levels"}, frac=0.7))
    # ---- long runs of exact duplicates (more keys than a list holds: refined down to shift 0) and short ones
    vals = np.sort(rng.choice(np.arange(K10 - 5_000_000, K10 + 5_000_000), 30, replace=False))
    runs = np.repeat(vals, 40)
    long_run = np.concatenate([runs, np.full(700, vals[10] + 7)])
    keys = np.sort(long_run)
    first = int(np.searchsorted(keys, vals[10] + 7))
    for pos, off in (("first", 0), ("middle", 350), ("last", 699)):
        cases.append(_single("dup_long_%s" % pos, rng, keys, first + off, {"dup_k_%s" % pos}))
    for pos, off in (("first", 0), ("middle", 17), ("last", 39)):
        cases.append(_single("dup_short_%s" % pos, rng, runs, 40 * 12 + off, {"dup_k_%s" % pos}))
    # ---- ten identical copies of a frustum's depths (duplicated rows)
    keys = np.tile(_wall(rng, 300, 40, half=0.02), 10)
    cases.append(_single("ten_copies", rng, np.sort(keys), int(0.25 * (len(keys) - 1)), {"cached_refine"}))
    # ---- sizes around the shared-memory key cache and far beyond it, each with a crowded bin; n % 4 != 0 and
    # n % 256 != 0 except 4096, so the last vector and the last page are partial
    for n in (4095, 4096, 4097, 20001, 200003):
        nw = int(n * 0.6)
        keys = np.sort(_wall(rng, nw, n - nw))
        cases.append(_single("size_%d" % n, rng, keys, int(0.25 * (n - 1)) + 1,
                             {"streamed_refine" if n > STATS_CACHE else "cached_refine"}, frac=0.6))
    # streamed with the successor in the next level-1 bin
    clus = lo + rng.integers(0, 8192, 1200)
    bg = _background(rng, kmin, kmax, 18803, avoid=(lo, lo + 8192))
    keys = np.sort(np.concatenate([clus, bg]))
    cases.append(_single("streamed_above", rng, keys, int((bg < lo).sum()) + 1199, {"refine1_k1_above", "streamed_refine"}))
    # ---- select_two: both ranks in one bin, in adjacent bins (k1 the last key of its bin), lists of 496 / 497 keys
    # together or in one bin, a narrow range (shift 0)
    bins = lambda b, c: kmin + 8192 * b + np.sort(rng.integers(0, 8192, c))
    bg = _background(rng, kmin, kmax, 400, avoid=(kmin + 8192 * 900, kmin + 8192 * 1200))
    nb = int((bg < kmin + 8192 * 900).sum())
    keys = np.concatenate([bg, bins(1000, 300)])
    cases.append(_two("two_same_bin", rng, keys, nb + 40, nb + 250, {"two_same_bin", "two_two_lists"}))
    keys = np.concatenate([bg, bins(1000, 200), bins(1001, 200)])
    cases.append(_two("two_adjacent_bins", rng, keys, nb + 199, nb + 300, {"two_adjacent_bins", "two_two_lists"}))
    for tot in (TWO_LIST, TWO_LIST + 1):
        keys = np.concatenate([bg, bins(1000, 248), bins(1100, tot - 248)])
        exit_ = "two_two_lists" if tot == TWO_LIST else "two_fallback"
        cases.append(_two("two_total_%d" % tot, rng, keys, nb + 247, nb + 400, {"two_total_%d" % tot, exit_}))
        keys = np.concatenate([bg, bins(1000, tot)])
        cases.append(_two("two_same_bin_%d" % tot, rng, keys, nb + 100, nb + tot - 1, {"two_same_bin_%d" % tot, exit_}))
    keys = np.sort(_background(rng, K10, K10 + 1500, 900))
    cases.append(_two("two_shift0", rng, keys, 300, 320, {"two_shift0"}))
    keys = np.sort(_wall(rng, 900, 300))
    n = len(keys)
    cases.append(Case("two_lq_gt_uq", _mk(rng, keys), (q_for_rank(n, 700), q_for_rank(n, 400), 0.5), {"two_skipped_lq_gt_uq"}))
    return cases
