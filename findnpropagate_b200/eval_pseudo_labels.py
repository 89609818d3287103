"""Scoring a folder of pseudo-labels per class and per range, on the GPU:

    python -m findnpropagate_b200.eval_pseudo_labels --cfg_file cfgs/nuscenes_box_seeker_proposals.yaml --folder out/

reads the ``.pth`` file of every frame of the config's info list (``<folder>/<frame_id with . -> _>.pth``, the format
``extract_pseudo_labels`` and the reference's tool write, read as ``pseudo_loader.load_pseudos`` reads it) and scores
it against the frame's GT as the extraction tool's loader produces it (``NuScenesFeed.gt_boxes`` or
``KittiFeed.gt_boxes``, training mode; the LiDAR files are not read), with the classes of the config's CLASS_NAMES.  ``--nms_thresh T ...`` also scores the folder as self-training reads it after
``load_pseudos(nms_thresh=T)``; every threshold is one more setting of the same fnp_quality_counters launch.

Per NMS setting it prints one JSON line: ``nms``, ``frames``, ``missing_files``, ``proposals``, ``recall`` (the
counters of ``extract.recall_keys``), ``ar`` and ``precision`` at the IoU thresholds, and ``classes``
(``quality.tables``: per class and range bin).
"""
import argparse
import json
import os
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np


def parse_args(argv=None):
    p = argparse.ArgumentParser(prog="python -m findnpropagate_b200.eval_pseudo_labels",
                                description="Score a folder of pseudo-labels per class and per range.")
    p.add_argument("--cfg_file", required=True, help="head config, e.g. cfgs/nuscenes_box_seeker_proposals.yaml")
    p.add_argument("--folder", required=True, help="folder of per-frame .pth files")
    p.add_argument("--nms_thresh", type=float, nargs="*", default=[],
                   help="also score after a rotated BEV NMS at each of these thresholds (as load_pseudos(nms_thresh=T))")
    p.add_argument("--range_edges", type=float, nargs="*", default=[20.0, 30.0, 40.0],
                   help="BEV range bin edges in metres, strictly increasing (default: 20 30 40)")
    p.add_argument("--every", type=int, default=1, help="score frames 0, K, 2K, ... of the info list")
    p.add_argument("--batch_frames", type=int, default=256, help="frames per batch on the GPU")
    p.add_argument("--workers", type=int, default=4, help="file reader threads")
    p.add_argument("--out", default=None, help="also write the JSON lines to this file")
    p.add_argument("--set", dest="set_cfgs", default=None, nargs=argparse.REMAINDER, metavar="KEY VALUE",
                   help="config overrides, e.g. --set DATA_CONFIG.MAX_SWEEPS 1")
    return p.parse_args(argv)


def _fail(msg):
    print(msg, file=sys.stderr)
    raise SystemExit(1)


def _pack(arrays):
    """The arrays back to back in one byte block, each at a 16-byte boundary: (block, offsets)."""
    offs, total = [], 0
    for a in arrays:
        offs.append(total)
        total = (total + a.nbytes + 15) // 16 * 16
    block = np.zeros(max(total, 16), np.uint8)
    for a, o in zip(arrays, offs):
        block[o:o + a.nbytes] = np.ascontiguousarray(a).reshape(-1).view(np.uint8)
    return block, offs


def _sub_batches(frames, spec):
    """Splits a batch where the largest proposal count and the largest GT count of the frames so far would exceed the
    kernel's shared memory together (each frame fits on its own)."""
    from .quality import SHARED_MEMORY_LIMIT
    out, cur, mk, mg = [], [], 0, 0
    for f in frames:
        k, g = f[1].shape[0], f[3].shape[0]
        if cur and spec.smem_bytes(max(mk, k), max(mg, g)) > SHARED_MEMORY_LIMIT:
            out.append(cur)
            cur, mk, mg = [], 0, 0
        cur.append(f)
        mk, mg = max(mk, k), max(mg, g)
    if cur:
        out.append(cur)
    return out


def _score(frames, spec, nms, counters, device):
    """One H2D, the NMS of every threshold, one fnp_quality_counters launch over every setting.  frames: list of
    (frame_id, boxes (K,7), labels (K,), gt (G,8), scores (K,))."""
    import torch
    from . import _lib, quality
    n = len(frames)
    ks = np.array([f[1].shape[0] for f in frames], np.int64)
    gs = np.array([f[3].shape[0] for f in frames], np.int64)
    pred_start = np.concatenate([[0], np.cumsum(ks)]).astype(np.int32)
    gt_start = np.concatenate([[0], np.cumsum(gs)]).astype(np.int32)
    boxes = np.concatenate([f[1] for f in frames]).astype(np.float32).reshape(-1, 7)
    labels = np.concatenate([f[2] for f in frames]).astype(np.int32).reshape(-1)
    scores = np.concatenate([f[4] for f in frames]).astype(np.float32).reshape(-1)
    gt = np.concatenate([f[3] for f in frames]).astype(np.float32).reshape(-1, 8)
    quality.check_labels(spec, labels, gt, gt_start)
    # stage-4 priority order of load_pseudos' NMS: per frame by descending score, ties by row (a stable sort)
    order = np.lexsort((-scores, np.repeat(np.arange(n), ks))).astype(np.int32)
    N, S = boxes.shape[0], len(nms)
    block, offs = _pack([boxes, labels, order, pred_start, gt, gt_start])
    dev = torch.from_numpy(block).to(device)
    view = [dev[o:o + a.nbytes] for a, o in zip((boxes, labels, order, pred_start, gt, gt_start), offs)]
    d_boxes, d_labels, d_order, d_pstart, d_gt, d_gstart = [v.view(torch.float32 if i in (0, 4) else torch.int32)
                                                            for i, v in enumerate(view)]
    valid = torch.zeros((S, max(N, 1)), dtype=torch.int32, device=device)
    max_k, max_g = int(ks.max(initial=0)), int(gs.max(initial=0))
    stream = _lib.current_stream(device)
    if N:
        keep = torch.empty(N, dtype=torch.uint8, device=device)
        for s, t in enumerate(nms):
            if t is None:
                continue
            _lib.check(_lib.lib.fnp_seg_nms_rotated(d_boxes.data_ptr(), None, d_order.data_ptr(), None,
                                                    d_pstart.data_ptr(), n, max(max_k, 1), float(t), keep.data_ptr(),
                                                    stream), "fnp_seg_nms_rotated")
            valid[s, :N] = keep.to(torch.int32) - 1          # kept: 0, removed: -1
    quality.launch(spec, d_boxes if N else None, d_labels.data_ptr() if N else None, d_pstart, d_gt.data_ptr(),
                   d_gstart, n, max_k, max_g, counters, n_settings=S, pred_valid=valid, pred_stride=0,
                   valid_stride=valid.shape[1], stream=stream)


def main(argv=None):
    """Runs the command; returns the JSON lines as dicts, one per NMS setting ("none" first)."""
    args = parse_args(argv)
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        _fail("eval_pseudo_labels runs in one process (it is bound by file reads): start it without torchrun")
    if not os.path.isdir(args.folder):
        _fail("%s does not exist or is not a folder" % args.folder)
    if args.every < 1 or args.batch_frames < 1:
        _fail("--every and --batch_frames must be at least 1")
    from .extract_pseudo_labels import build_feed, frame_id, load_config
    from .quality import QualitySpec
    try:
        cfg = load_config(args.cfg_file, args.set_cfgs)
    except (OSError, KeyError, ValueError) as e:
        _fail(e.args[-1] if isinstance(e, KeyError) else e)
    feed = build_feed(cfg)
    try:
        spec = QualitySpec(feed.class_names, range_edges=args.range_edges)
    except ValueError as e:
        _fail(e)
    import torch
    from . import _lib, quality
    from .pseudo_loader import pseudo_path, read_pseudos
    nms = [None] + [float(t) for t in args.nms_thresh]
    device = torch.device("cuda", torch.cuda.current_device())
    counters = torch.zeros((len(nms), spec.n_counters), dtype=torch.int64, device=device)
    picked = list(range(0, len(feed), args.every))
    missing = []

    def load(i):
        fid = frame_id(feed.infos[i])
        got = read_pseudos(pseudo_path(args.folder, fid))
        absent = got is None
        if absent:          # no proposals
            got = (np.zeros((0, 7), np.float32), np.zeros((0,), np.float32), np.zeros((0,), np.int32))
        g = np.asarray(feed.gt_boxes(i), np.float32)
        g = np.concatenate([g[:, :7], g[:, -1:]], 1) if g.shape[0] else np.zeros((0, 8), np.float32)
        return (fid, got[0], got[2], quality.strip_gt(g), got[1]), absent

    with ThreadPoolExecutor(max_workers=max(1, args.workers)) as pool:
        for b0 in range(0, len(picked), args.batch_frames):
            frames = []
            for f, absent in pool.map(load, picked[b0:b0 + args.batch_frames]):
                if absent:
                    missing.append(f[0])
                k = f[1].shape[0]
                if len(nms) > 1 and k > _lib.SEG_NMS_MAX:
                    _fail("frame %s: %d proposals, the NMS takes at most %d per frame" % (f[0], k, _lib.SEG_NMS_MAX))
                try:
                    spec.check_size(k, f[3].shape[0], "frame %s" % f[0])
                except ValueError as e:
                    _fail(e)
                frames.append(f)
            try:
                for sub in _sub_batches(frames, spec):
                    _score(sub, spec, nms, counters, device)
            except ValueError as e:
                _fail(e)
    c = counters.cpu().numpy()
    print("frames scored: %d, missing files: %d" % (len(picked), len(missing)))
    lines = []
    for s, t in enumerate(nms):
        d = dict(nms="none" if t is None else t, frames=len(picked), missing_files=len(missing))
        d.update(quality.summary(c[s], spec))
        d["classes"] = quality.tables(c[s], spec)
        lines.append(d)
    text = [json.dumps(d) for d in lines]
    for t in text:
        print(t)
    if args.out:
        with open(args.out, "w") as f:
            f.write("".join(t + "\n" for t in text))
    return lines


if __name__ == "__main__":
    main()
