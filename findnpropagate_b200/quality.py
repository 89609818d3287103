"""Pseudo-label quality per class and per range: recall and precision counters binned by class and by the BEV distance
of the box centre from the LiDAR origin (fnp_quality_counters), and the tables the commands print from them.

The reference's only quality signal is generate_recall_record (detectors/detector3d_template.py:315-399):
class-agnostic recall over all ranges.  The counters here contain it -- ``recall_dict`` rebuilds its counters from the
table exactly -- and add, per (class, range bin):
  * recall: GT boxes, and those whose best IoU3D over the frame's proposals is above each threshold, over all
    proposals (the reference's rule) and over the proposals with the GT's label only;
  * precision: proposals, and those whose best IoU3D over the frame's GT is above each threshold, over all GT and
    over the GT of the proposal's class only.
"""
import ctypes as C
from dataclasses import dataclass
from typing import Sequence

import numpy as np

from .extract import THRESH, recall_keys

MAX_THRESH, MAX_BINS, MAX_CLASSES = 8, 8, 32
SHARED_MEMORY_LIMIT = 200 * 1024
# generate_recall_record's known / unknown splits, as 1-based class positions (recall_kernel)
KNOWN3 = (1, 8, 9)
KNOWN6 = (1, 3, 5, 6, 8, 9)


@dataclass(frozen=True)
class QualitySpec:
    """class_names: 1-based labels index them; range_edges: strictly increasing, > 0, at most 7 (bins [0, e0),
    [e0, e1), ..., [e_last, inf)); thresh: IoU3D thresholds, at most 8."""
    class_names: Sequence[str]
    range_edges: Sequence[float] = (20, 30, 40)
    thresh: Sequence[float] = THRESH

    def __post_init__(self):
        object.__setattr__(self, "class_names", tuple(self.class_names))
        object.__setattr__(self, "range_edges", tuple(float(e) for e in self.range_edges))
        object.__setattr__(self, "thresh", tuple(float(t) for t in self.thresh))
        e = np.asarray(self.range_edges, np.float32)
        if len(e) + 1 > MAX_BINS:
            raise ValueError("at most %d range bins (%d edges), got %d edges" % (MAX_BINS, MAX_BINS - 1, len(e)))
        if len(e) and (not (e > 0).all() or not (np.diff(e) > 0).all()):
            raise ValueError("range edges must be > 0 and strictly increasing, got %s" % list(self.range_edges))
        if len(self.thresh) > MAX_THRESH:
            raise ValueError("at most %d IoU thresholds, got %d" % (MAX_THRESH, len(self.thresh)))
        if not 1 <= len(self.class_names) <= MAX_CLASSES:
            raise ValueError("1 to %d classes, got %d" % (MAX_CLASSES, len(self.class_names)))

    @property
    def n_bins(self):
        return len(self.range_edges) + 1

    @property
    def width(self):
        return 1 + 2 * len(self.thresh)

    @property
    def n_counters(self):
        """int64 counters per setting: a recall block and a precision block."""
        return 2 * len(self.class_names) * self.n_bins * self.width

    def bin_names(self):
        e = ["%g" % x for x in self.range_edges]
        lo = ["0"] + e
        return ["%s-%s" % (a, b) for a, b in zip(lo, e)] + ["%s+" % lo[-1]]

    def smem_bytes(self, max_pred, max_gt):
        from . import _lib
        return int(_lib.lib.fnp_quality_smem_bytes(int(max_pred), int(max_gt), len(self.class_names),
                                                   len(self.range_edges), len(self.thresh)))

    def check_size(self, max_pred, max_gt, what="a frame"):
        if self.smem_bytes(max_pred, max_gt) > SHARED_MEMORY_LIMIT:
            raise ValueError("%s has too many boxes for fnp_quality_counters (%d proposals, %d GT boxes: more than "
                             "%d KB of shared memory)" % (what, max_pred, max_gt, SHARED_MEMORY_LIMIT // 1024))


def strip_gt(gt):
    """The rows of one frame's (G, 8) GT the counters see: trailing all-zero rows dropped (recall_kernel's rule)."""
    g = np.asarray(gt, np.float32).reshape(-1, 8)
    n = g.shape[0]
    while n > 0:
        s = np.float32(0)
        for v in g[n - 1]:              # the kernel's sequential fp32 sum
            s = np.float32(s + v)
        if s != 0:
            break
        n -= 1
    return g[:n]


def check_labels(spec, pred_label, gt, gt_start):
    """ValueError unless every proposal label and every GT class (after strip_gt, per frame) lies in 1..C.  Host
    arrays: pred_label (K,), gt (sum G, 8), gt_start (n_frames+1)."""
    C_ = len(spec.class_names)
    pl = np.asarray(pred_label).reshape(-1)
    if pl.size and (pl.min() < 1 or pl.max() > C_):
        raise ValueError("proposal label outside 1..%d: %s" % (C_, sorted(set(pl[(pl < 1) | (pl > C_)].tolist()))[:5]))
    gt = np.asarray(gt, np.float32).reshape(-1, 8)
    gs = np.asarray(gt_start)
    for f in range(len(gs) - 1):
        lab = strip_gt(gt[gs[f]:gs[f + 1]])[:, 7]
        if lab.size and (lab.min() < 1 or lab.max() > C_):
            raise ValueError("GT class outside 1..%d in frame %d: %s" % (C_, f, sorted(set(lab.tolist()))[:5]))


def _ptr(x):
    if x is None:
        return None
    return x.data_ptr() if hasattr(x, "data_ptr") else int(x)


def launch(spec, pred, pred_label, pred_start, gt, gt_start, n_frames, max_pred, max_gt, counters, n_settings=1,
           pred_valid=None, pred_stride=0, valid_stride=0, stream=None):
    """One fnp_quality_counters launch (counters are ADDED to ``counters``: (n_settings, spec.n_counters) int64).
    Array arguments are CUDA tensors, or device addresses (int) of the same layouts; labels given as tensors are
    checked here (one small D2H), callers passing addresses check theirs with check_labels.
      pred (rows, 7) f32 per setting, setting s at row s * pred_stride (0: shared); pred_valid (rows) int32 per setting
      at s * valid_stride (None: every row); pred_label, pred_start (n_frames+1), gt (sum G, 8), gt_start: shared.
    ValueError for labels outside 1..C and a frame too large for the kernel's shared memory."""
    from . import _lib
    import torch
    spec.check_size(max_pred, max_gt, "the largest frame")
    if isinstance(pred_label, torch.Tensor) and isinstance(gt, torch.Tensor):
        check_labels(spec, pred_label.cpu().numpy(), gt.cpu().numpy(), gt_start.cpu().numpy())
    for t in (pred, pred_label, pred_start, gt, gt_start, pred_valid, counters):
        if isinstance(t, torch.Tensor):
            _lib.require_cuda(t)
    if isinstance(counters, torch.Tensor):
        assert counters.dtype == torch.int64 and counters.numel() >= n_settings * spec.n_counters
    edges = (C.c_float * max(len(spec.range_edges), 1))(*spec.range_edges)
    th = (C.c_float * max(len(spec.thresh), 1))(*spec.thresh)
    if stream is None:
        stream = _lib.current_stream()
    rc = _lib.lib.fnp_quality_counters(_ptr(pred), int(pred_stride), _ptr(pred_valid), int(valid_stride),
                                       _ptr(pred_label), _ptr(pred_start), int(n_settings), _ptr(gt), _ptr(gt_start),
                                       int(n_frames), int(max_pred), int(max_gt), len(spec.class_names), edges,
                                       len(spec.range_edges), th, len(spec.thresh), _ptr(counters), stream)
    _lib.check(rc, "fnp_quality_counters")


def tables(counters, spec):
    """The flat counters of one setting as {class: {bin: dict(gt, recall_any, recall_label, proposals,
    precision_any, precision_label)}}: counts, the *_any / *_label entries keyed by threshold ("0.5"), bins named
    "0-20", ..., "40+", and per class an "all" entry summed over the bins."""
    c = np.asarray(counters, np.int64).reshape(2, len(spec.class_names), spec.n_bins, spec.width)
    T = len(spec.thresh)
    keys = [str(t) for t in spec.thresh]
    out = {}
    for ci, name in enumerate(spec.class_names):
        rows = {}
        for bi, b in enumerate(spec.bin_names() + ["all"]):
            r = c[0, ci].sum(0) if b == "all" else c[0, ci, bi]
            p = c[1, ci].sum(0) if b == "all" else c[1, ci, bi]
            rows[b] = dict(gt=int(r[0]), recall_any={k: int(r[1 + t]) for t, k in enumerate(keys)},
                           recall_label={k: int(r[1 + T + t]) for t, k in enumerate(keys)},
                           proposals=int(p[0]), precision_any={k: int(p[1 + t]) for t, k in enumerate(keys)},
                           precision_label={k: int(p[1 + T + t]) for t, k in enumerate(keys)})
        out[name] = rows
    return out


def recall_dict(counters, spec):
    """The generate_recall_record counters (extract.recall_keys(spec.thresh)) rebuilt from the table of ``counters``:
    gt and rcnn_<t> summed over every class and bin, the known splits over the classes KNOWN3 / KNOWN6."""
    tab = tables(counters, spec)
    keys = [str(t) for t in spec.thresh]

    def total(labels, field, t=None):
        return sum((tab[n]["all"][field] if t is None else tab[n]["all"][field][t])
                   for i, n in enumerate(spec.class_names) if labels is None or i + 1 in labels)
    out = {}
    for prefix, field, t in [("", "gt", None)] + [("rcnn", "recall_any", k) for k in keys]:
        every, k3, k6 = total(None, field, t), total(KNOWN3, field, t), total(KNOWN6, field, t)
        vals = [every, k3, k6, every - k6, every - k3]
        names = (["gt", "num_3known", "num_6known", "num_4unknown", "num_7unknown"] if t is None else
                 ["rcnn_%s" % t, "rcnn_3known_%s" % t, "rcnn_6known_%s" % t, "rcnn_4unknown_%s" % t,
                  "rcnn_7unknown_%s" % t])
        out.update(zip(names, vals))
    assert list(out) == recall_keys(spec.thresh)
    return out


def precision_dict(counters, spec):
    """fnp_precision_counters' counters rebuilt from the table: proposals and hits_<t>, summed over classes and bins."""
    tab = tables(counters, spec)
    out = dict(proposals=sum(tab[n]["all"]["proposals"] for n in spec.class_names))
    for t in spec.thresh:
        out["hits_%s" % t] = sum(tab[n]["all"]["precision_any"][str(t)] for n in spec.class_names)
    return out


def summary(counters, spec):
    """What the commands print per setting besides the tables: proposals, recall counters, AR and precision."""
    rec, prec = recall_dict(counters, spec), precision_dict(counters, spec)
    n_gt, n_prop = max(rec["gt"], 1), max(prec["proposals"], 1)
    return dict(proposals=prec["proposals"], recall=rec,
                ar={str(t): rec["rcnn_%s" % t] / n_gt for t in spec.thresh},
                precision={str(t): prec["hits_%s" % t] / n_prop for t in spec.thresh})
