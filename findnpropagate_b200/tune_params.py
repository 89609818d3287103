"""Tuning the Box Seeker's head settings: score a grid of settings in one pass over the frames.

    python -m findnpropagate_b200.tune_params --cfg_file cfgs/nuscenes_box_seeker_proposals.yaml --grid grid.yaml

``grid.yaml`` maps ``--set``-style keys of the head (``MODEL.DENSE_HEAD.PARAMS.<k>``, ``MODEL.DENSE_HEAD.MULT``,
``…OCCL_MULT``, ``…MULTICAM_IOU``) to lists of values; the settings are their cartesian product, in file order.  Every
frame is read and uploaded once.  Settings that differ only in the select-level parameters (seeker.SELECT_KEYS: the
score weights, ``min_cam_iou``, ``MULT``, ``OCCL_MULT``) form one group and share stages 1-2c of the seeker; only
stage 3 and the counters run per setting (SeekerEngine.evaluate_settings).  Every other parameter splits groups.

A KITTI config (KittiDataset, FrustumProposerOGKITTI) is tuned the same way, with that head's rule: its counts are
first-match counts over the valid set, so ``min_cam_iou`` splits groups and only ``dns_w``, ``iou_w`` and ``dst_w``
(seeker.SELECT_KEYS_KITTI) share stages 1-2c; the keys that head does not read (``ego_w``, ``occl_w``, ``MULT``,
``OCCL_MULT``, ``MULTICAM_IOU``) are refused, and ``topk`` stays 1.

For each setting the command prints one JSON line -- its values and group, the proposals, the recall counters, AR and
precision at 0.3 / 0.5 / 0.7 -- sorted by AR@0.5, then the ``--set`` arguments that give the best setting to
``extract_pseudo_labels``.  The config, its refusals and the failed-frame rule are those of ``extract_pseudo_labels``.

Self-training reads the proposals through ``load_pseudos(nms_thresh=T)``, a class-agnostic rotated BEV NMS in 2D-score
order.  ``--nms_thresh T ...`` (up to 8 thresholds) scores every setting that way too: each line gains ``nms``, per
threshold the proposals, recall counters, AR and precision ``eval_pseudo_labels --nms_thresh`` would print for the
folder the setting extracts, and the lines are ranked by AR@0.5 after the first threshold's NMS.
"""
import argparse
import copy
import itertools
import json
import math
import os
import sys

import yaml

from .config import cfg_from_list
from .extract_pseudo_labels import build_feed, build_head, check_frame, frame_id, is_kitti, load_config, FAILURES

HEAD = ("MODEL", "DENSE_HEAD")


def _head_keys():
    """name -> default of every PARAMS key and switch the head reads, the weights that default to 0 as floats (the
    default's type is the type a grid value must have, config.cfg_from_list's rule)."""
    from .proposer import EXTRA_PARAMS
    from .seeker import DEFAULTS, FLAG_KEYS
    params = dict(DEFAULTS, aln_w=0.0, ego_w=0.0, occl_w=0.0, rand_center=False, search_depth=None)
    assert set(params) == set(DEFAULTS) | set(EXTRA_PARAMS)
    return params, {k: False for k in FLAG_KEYS}


def load_grid(path, cfg):
    """The grid file as a list of axes (key, name, in_yaml, values): ``name`` is the head parameter the key sets,
    ``in_yaml`` whether the config has the key (else --set cannot pass it).  ValueError, naming the key, for a key
    outside MODEL.DENSE_HEAD, an unknown key, a value that is not a non-empty list or of the wrong type, and for an
    empty grid."""
    with open(path) as f:
        grid = yaml.safe_load(f)
    if not grid:
        raise ValueError("%s: the grid is empty" % path)
    if not isinstance(grid, dict):
        raise ValueError("%s: the grid must map keys to lists of values" % path)
    params, switches = _head_keys()
    head = cfg.MODEL.DENSE_HEAD
    axes = []
    for key, values in grid.items():
        key = str(key)
        parts = key.split(".")
        if tuple(parts[:2]) != HEAD or len(parts) < 3:
            raise ValueError("grid key %s is outside MODEL.DENSE_HEAD: it would change the frames" % key)
        rest = parts[2:]
        if len(rest) == 1 and rest[0] in switches:
            name, node, known = rest[0], head, switches
        elif len(rest) == 2 and rest[0] == "PARAMS":
            name, node, known = rest[1], head.get("PARAMS"), params
        else:
            raise ValueError("grid key %s is unknown: the grid takes MODEL.DENSE_HEAD.PARAMS.<key> and the switches %s"
                             % (key, ", ".join("MODEL.DENSE_HEAD." + s for s in switches)))
        in_yaml = isinstance(node, dict) and name in node
        if not in_yaml and name not in known:
            raise ValueError("grid key %s is unknown: the config has no such key and the head reads no such parameter"
                             % key)
        if not isinstance(values, list) or not values:
            raise ValueError("grid key %s: the values must be a non-empty list, got %r" % (key, values))
        # each value goes through --set's type rule, against the config's value or the head's default
        scratch = {"MODEL": {"DENSE_HEAD": {"PARAMS": {}}}}
        leaf = scratch["MODEL"]["DENSE_HEAD"] if len(rest) == 1 else scratch["MODEL"]["DENSE_HEAD"]["PARAMS"]
        checked = []
        for v in values:
            leaf[name] = copy.deepcopy(node[name] if in_yaml else known[name])
            try:
                cfg_from_list([key, repr(v)], scratch)
            except ValueError as e:
                raise ValueError("grid key %s: %s" % (key, e)) from None
            checked.append(leaf[name])
        axes.append((key, name, in_yaml, checked))
    return axes


def expand_grid(axes):
    """The cartesian product of the axes, the first axis varying slowest: a list of {key: value}."""
    keys = [a[0] for a in axes]
    return [dict(zip(keys, vals)) for vals in itertools.product(*[a[3] for a in axes])]


def group_settings(base_params, settings, variant="nuscenes"):
    """Groups of settings that can share stages 1-2c.  base_params: the head's parameters (proposer.head_params, or
    proposer.kitti_head_params for variant "kitti"); settings: dicts of parameter overrides.  Each setting is checked by
    seeker.resolve_params; topk > 1, rand_center and aln_w are refused, and for the KITTI head the keys it does not
    read (ValueError naming the setting).  Settings are grouped on every resolved parameter except seeker.SELECT_KEYS
    (seeker.SELECT_KEYS_KITTI for the KITTI head).  Returns a list of dict(params, members): members are indices into
    settings, params the engine parameters of the group -- its first member's, at the group's loosest min_cam_iou."""
    from .seeker import FLAG_KEYS, SELECT_KEYS, SELECT_KEYS_KITTI, resolve_params
    kitti = variant == "kitti"
    resolved = []
    for s in settings:
        unused = [k for k in ("ego_w", "occl_w") + FLAG_KEYS if k in s] if kitti else []
        if unused:
            raise ValueError("setting %s: %s not read by the KITTI head" % (s, ", ".join(unused)))
        p = dict(base_params)
        p.update(s)
        try:
            r = resolve_params(p, variant)
        except NotImplementedError as e:
            raise ValueError("setting %s: %s" % (s, e)) from None
        if int(r["topk"]) > 1:
            raise ValueError("setting %s: topk > 1 is not supported by the tuner (one proposal per frustum)" % (s,))
        if r.get("rand_center"):
            raise ValueError("setting %s: rand_center is not supported by the tuner (the centres are random)" % (s,))
        resolved.append(r)
    select = SELECT_KEYS_KITTI if kitti else SELECT_KEYS
    groups = {}
    for i, r in enumerate(resolved):
        key = tuple(sorted((k, repr(v)) for k, v in r.items() if k not in select))
        groups.setdefault(key, []).append(i)
    out = []
    for members in groups.values():
        params = dict(resolved[members[0]])
        params["min_cam_iou"] = min(resolved[i]["min_cam_iou"] for i in members)
        out.append(dict(params=params, members=members, settings=[resolved[i] for i in members]))
    return out


def evaluate_grid(feed, detector, base_params, settings, batch_frames=64, workers=4, box_format="xyxy", device=None,
                  quality=None, variant="nuscenes", nms_thresh=()):
    """Scores every setting over every frame of ``feed``: each batch is read once (NuScenesFeed / KittiFeed.prefetch)
    and uploaded once, then every group of ``group_settings`` runs on it (variant: the head's, as for SeekerEngine).  Returns (per setting dict(proposals, recall, precision)
    summed over the frames, groups).  quality (a quality.QualitySpec): each setting's dict also holds "quality", its
    summed fnp_quality_counters counters.  nms_thresh (needs quality): and "nms", its summed counters after the NMS at
    each threshold (SeekerEngine.evaluate_settings)."""
    import numpy as np
    import torch
    from .extract import THRESH, recall_keys
    from .seeker import SeekerEngine
    groups = group_settings(base_params, settings, variant)
    engines = [SeekerEngine(g["params"], device=device, box_format=box_format, variant=variant) for g in groups]
    # the groups run one after another and evaluate_settings waits for its results: one scratch arena serves them all,
    # so device memory does not grow with the number of groups
    for e in engines[1:]:
        e.arena = engines[0].arena
    prec_keys = ["proposals"] + ["hits_%s" % t for t in THRESH]
    totals = [dict(proposals=0, recall=dict.fromkeys(recall_keys(), 0), precision=dict.fromkeys(prec_keys, 0))
              for _ in settings]
    if quality is not None:
        for t in totals:
            t["quality"] = np.zeros(quality.n_counters, np.int64)
            t["nms"] = np.zeros((len(nms_thresh), quality.n_counters), np.int64)
    for frames, _, _ in feed.prefetch(range(len(feed)), detector, batch_frames=batch_frames, workers=workers,
                                      xyz_only=True):
        points = torch.from_numpy(np.concatenate([f.points for f in frames])).to(engines[0].device)
        gt = engines[0].upload_gt(frames)
        for g, eng in zip(groups, engines):
            res = eng.evaluate_settings(eng.plan(frames), points, gt, g["settings"], recall_thresh=THRESH, quality=quality,
                                        nms_thresh=nms_thresh)
            for i, r in zip(g["members"], res["settings"]):
                t = totals[i]
                t["proposals"] += r["proposals"]
                for k, v in r.get("recall", {}).items():       # no candidate in the batch: no counters, as in extract
                    t["recall"][k] += v
                for k, v in r.get("precision", {}).items():
                    t["precision"][k] += v
                if "quality" in r:
                    t["quality"] += r["quality"]
                if "nms" in r:
                    t["nms"] += np.stack(r["nms"])
    return totals, groups


def parse_args(argv=None):
    p = argparse.ArgumentParser(prog="python -m findnpropagate_b200.tune_params",
                                description="Score a grid of Box Seeker head settings in one pass over the frames.")
    p.add_argument("--cfg_file", required=True, help="head config, e.g. cfgs/nuscenes_box_seeker_proposals.yaml")
    p.add_argument("--grid", required=True,
                   help="YAML mapping MODEL.DENSE_HEAD.PARAMS.<key> / MODEL.DENSE_HEAD.<switch> to lists of values")
    p.add_argument("--every", type=int, default=1, help="score frames 0, K, 2K, ... of the info list")
    p.add_argument("--batch_frames", type=int, default=64, help="frames per batch on the GPU")
    p.add_argument("--workers", type=int, default=4, help="loader threads")
    p.add_argument("--out", default=None, help="also write the JSON lines to this file")
    p.add_argument("--breakdown", action="store_true",
                   help="add per class and range bin counters to each line (classes; see eval_pseudo_labels)")
    p.add_argument("--range_edges", type=float, nargs="*", default=[20.0, 30.0, 40.0],
                   help="with --breakdown: BEV range bin edges in metres (default: 20 30 40)")
    p.add_argument("--nms_thresh", type=float, nargs="*", default=[],
                   help="also score each setting after a rotated BEV NMS at each of these thresholds (as "
                        "load_pseudos(nms_thresh=T)), at most 8; the lines are then ranked by AR@0.5 after the first")
    p.add_argument("--set", dest="set_cfgs", default=None, nargs=argparse.REMAINDER, metavar="KEY VALUE",
                   help="config overrides applied to every setting, e.g. --set DATA_CONFIG.MAX_SWEEPS 1")
    return p.parse_args(argv)


def _fail(msg):
    print(msg, file=sys.stderr)
    raise SystemExit(1)


def main(argv=None):
    """Runs the command; returns the JSON lines as dicts, best first."""
    args = parse_args(argv)
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        _fail("tune_params runs in one process: start it without torchrun")
    if args.every < 1:
        _fail("--every must be at least 1")
    nms = [float(t) for t in args.nms_thresh]
    from ._lib import SEG_NMS_MAX_THRESH
    if len(nms) > SEG_NMS_MAX_THRESH:
        _fail("--nms_thresh takes at most %d thresholds, got %d: %s" % (SEG_NMS_MAX_THRESH, len(nms), nms))
    for i, t in enumerate(nms):
        if not math.isfinite(t):
            _fail("--nms_thresh %s: the thresholds must be finite" % t)
        if t in nms[:i]:
            _fail("--nms_thresh %s is given twice" % t)
    from .proposer import head_params, kitti_head_params
    try:
        cfg = load_config(args.cfg_file, args.set_cfgs)
        axes = load_grid(args.grid, cfg)
        grid = expand_grid(axes)
        names = {key: name for key, name, _, _ in axes}
        settings = [{names[k]: v for k, v in s.items()} for s in grid]
        kitti = is_kitti(cfg)
        variant = "kitti" if kitti else "nuscenes"
        base = (kitti_head_params if kitti else head_params)(cfg.MODEL.DENSE_HEAD)
        groups = group_settings(base, settings, variant)
        spec = None
        if args.breakdown or nms:
            from .kitti_feed import CLASS_NAMES as KITTI_CLASS_NAMES
            from .nuscenes_feed import CLASS_NAMES
            from .quality import QualitySpec
            spec = QualitySpec(cfg.get("CLASS_NAMES") or (KITTI_CLASS_NAMES if kitti else CLASS_NAMES),
                               range_edges=args.range_edges)
    except (OSError, KeyError, ValueError, NotImplementedError) as e:
        _fail(e.args[-1] if isinstance(e, KeyError) else e)
    print("%d settings in %d groups" % (len(settings), len(groups)))
    from . import extract
    head = build_head(cfg)
    device = head.engine.device
    all_frames = build_feed(cfg, device=device)
    picked = list(range(0, len(all_frames), args.every))
    codes = [check_frame(all_frames, head.image_detector, all_frames.infos[i]) for i in picked]
    for i, c in zip(picked, codes):
        if c:
            print("skipped frame %s: %s" % (frame_id(all_frames.infos[i]), FAILURES[c]))
    feed = build_feed(cfg, infos=[all_frames.infos[i] for i, c in zip(picked, codes) if c == 0], device=device)
    print("frames scored: %d, failed frames: %d" % (len(feed), sum(1 for c in codes if c)))
    totals, groups = evaluate_grid(feed, head.image_detector, base, settings, batch_frames=args.batch_frames,
                                   workers=args.workers, box_format=head.engine.box_format, device=device,
                                   quality=spec, variant=variant, nms_thresh=nms)
    group_of = {i: gi for gi, g in enumerate(groups) for i in g["members"]}
    from .quality import summary, tables
    lines = []
    for i, (s, t) in enumerate(zip(grid, totals)):
        rec, n_gt, n_prop = t["recall"], max(t["recall"]["gt"], 1), max(t["proposals"], 1)
        lines.append(dict(setting=s, group=group_of[i], proposals=t["proposals"], recall=rec,
                          ar={str(th): rec["rcnn_%s" % th] / n_gt for th in extract.THRESH},
                          precision={str(th): t["precision"]["hits_%s" % th] / n_prop for th in extract.THRESH}))
        if args.breakdown:
            lines[-1]["classes"] = tables(t["quality"], spec)
        if nms:
            lines[-1]["nms"] = {}
            for th, c in zip(nms, t["nms"]):
                d = lines[-1]["nms"][str(th)] = summary(c, spec)
                if args.breakdown:
                    d["classes"] = tables(c, spec)
    # stable: equal AR keeps grid order; with --nms_thresh, the AR self-training sees after the first threshold's NMS
    if nms:
        lines.sort(key=lambda d: -d["nms"][str(nms[0])]["ar"]["0.5"])
    else:
        lines.sort(key=lambda d: -d["ar"]["0.5"])
    text = [json.dumps(d) for d in lines]
    for t in text:
        print(t)
    if args.out:
        with open(args.out, "w") as f:
            f.write("".join(t + "\n" for t in text))
    best = lines[0]["setting"]
    set_args = list(args.set_cfgs or [])
    for key, name, in_yaml, _ in axes:
        if in_yaml:
            set_args += [key, repr(best[key])]
        else:
            print("best %s = %r: the config has no %s, add %s: %r to it (--set cannot add a key)"
                  % (key, best[key], key, name, best[key]))
    print("best setting%s: python -m findnpropagate_b200.extract_pseudo_labels --cfg_file %s --folder <folder>%s"
          % (" (ranked by AR@0.5 after the NMS at %s)" % nms[0] if nms else "", args.cfg_file,
             (" --set " + " ".join('"%s"' % a for a in set_args)) if set_args else ""))
    return lines


if __name__ == "__main__":
    main()
