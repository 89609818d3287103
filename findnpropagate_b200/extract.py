"""Pseudo-label extraction driver: the frame loop of tools/extract_pseudo_labels.py
(reference :113-146) batched, frame-sharded across ranks, with the reference's output
format and recall bookkeeping.

  * output: ``<folder>/<frame_id with '.' -> '_'>.pth`` = ``torch.save`` of a list of length 1
    holding ``{pred_boxes (K,7) f32, pred_scores (K) f32, pred_labels (K) int32}``
    (reference :133-137; consumer pcdet/datasets/augmentor/pseudo_loader.py:561-679);
  * sharding: rank r of W takes frames r, r+W, ... (the reference's own rule for
    distributed evaluation, pcdet/datasets/__init__.py:43-48);
  * the only exchange: one all_gather of fixed-stride packed proposals and one all_reduce
    (SUM) of the int64 recall-counter vector per run -- NCCL over NVLink on GPUs, gloo in
    the CPU tests -- replacing the reference's pickle-on-shared-disk merge
    (pcdet/utils/common_utils.py:229-248).
"""
import os
from typing import Callable, Iterable, List, Optional

import numpy as np
import torch
import torch.distributed as dist

from .seeker import RECALL_KEYS, RECALL_PER_THRESH

THRESH = (0.3, 0.5, 0.7)


def recall_keys(thresh=THRESH):
    keys = list(RECALL_KEYS)
    for t in thresh:
        keys += ["%s_%s" % (k, t) for k in RECALL_PER_THRESH]
    return keys


def shard_indices(n_frames: int, rank: int, world: int) -> List[int]:
    return list(range(rank, n_frames, world))


def save_frame(folder: str, frame_id: str, pred: dict) -> str:
    """One .pth per frame in the reference's format."""
    path = os.path.join(folder, "%s.pth" % frame_id.replace('.', '_'))
    out = [dict(pred_boxes=torch.from_numpy(np.ascontiguousarray(pred["pred_boxes"], np.float32)).reshape(-1, 7),
                pred_scores=torch.from_numpy(np.ascontiguousarray(pred["pred_scores"], np.float32)),
                pred_labels=torch.from_numpy(np.ascontiguousarray(pred["pred_labels"], np.int32)))]
    torch.save(out, path)
    return path


def pack_proposals(preds: List[dict], kmax: int) -> (np.ndarray, np.ndarray):
    """(n,kmax,9) f32 [box7, score, label] + (n,) int32 counts."""
    pack = np.zeros((len(preds), kmax, 9), np.float32)
    cnt = np.zeros((len(preds),), np.int32)
    for i, p in enumerate(preds):
        k = p["pred_boxes"].shape[0]
        pack[i, :k, :7] = p["pred_boxes"]
        pack[i, :k, 7] = p["pred_scores"]
        pack[i, :k, 8] = p["pred_labels"]
        cnt[i] = k
    return pack, cnt


def unpack_proposals(pack: np.ndarray, cnt: np.ndarray) -> List[dict]:
    return [dict(pred_boxes=pack[i, :cnt[i], :7].copy(), pred_scores=pack[i, :cnt[i], 7].copy(),
                 pred_labels=pack[i, :cnt[i], 8].astype(np.int32)) for i in range(pack.shape[0])]


def gather_shards(local_preds: List[dict], local_recall: dict, n_frames: int, rank: int, world: int, device="cpu"):
    """All ranks receive every frame's proposals (in dataset order) and the summed recall
    counters.  One all_gather (+ its count vector) and one all_reduce."""
    keys = recall_keys()
    rc = torch.tensor([int(local_recall.get(k, 0)) for k in keys], dtype=torch.int64, device=device)
    if world == 1:
        return local_preds, dict(zip(keys, rc.tolist()))
    per_rank = (n_frames + world - 1) // world
    kmax = torch.tensor([max([p["pred_boxes"].shape[0] for p in local_preds] + [1])], dtype=torch.int64, device=device)
    dist.all_reduce(kmax, op=dist.ReduceOp.MAX)
    kmax = int(kmax.item())
    pack, cnt = pack_proposals(local_preds, kmax)
    pad = per_rank - pack.shape[0]
    if pad:
        pack = np.concatenate([pack, np.zeros((pad, kmax, 9), np.float32)])
        cnt = np.concatenate([cnt, np.full((pad,), -1, np.int32)])
    tp, tc = torch.from_numpy(pack).to(device), torch.from_numpy(cnt).to(device)
    allp = torch.empty((world * per_rank, kmax, 9), dtype=tp.dtype, device=device)
    allc = torch.empty((world * per_rank,), dtype=tc.dtype, device=device)
    dist.all_gather_into_tensor(allp, tp)
    dist.all_gather_into_tensor(allc, tc)
    dist.all_reduce(rc)
    allp = allp.cpu().numpy().reshape(world, per_rank, kmax, 9)
    allc = allc.cpu().numpy().reshape(world, per_rank)
    merged = [None] * n_frames
    for r in range(world):
        idx = shard_indices(n_frames, r, world)
        un = unpack_proposals(allp[r][:len(idx)], allc[r][:len(idx)])
        for j, i in enumerate(idx):
            merged[i] = un[j]
    return merged, dict(zip(keys, rc.tolist()))


def extract(frames, compute_fn: Callable, folder: Optional[str] = None, batch_frames: int = 32, rank: int = 0,
            world: int = 1, device="cpu", frame_ids: Optional[List[str]] = None):
    """Run the seeker over ``frames`` (any indexable of frame inputs), sharded by rank.

    compute_fn(list_of_frames) -> dict(frames=[per-frame pred dict], recall=dict) -- normally
    ``lambda fs: engine.run(fs, with_recall=True)``.
    Returns (all_preds in dataset order, summed recall dict, running AR per threshold)."""
    n = len(frames)
    mine = shard_indices(n, rank, world)
    local, recall = [], {}
    if folder is not None:
        os.makedirs(folder, exist_ok=True)
    for s in range(0, len(mine), batch_frames):
        idx = mine[s:s + batch_frames]
        res = compute_fn([frames[i] for i in idx])
        for j, i in enumerate(idx):
            local.append(res["frames"][j])
            if folder is not None:
                fid = frame_ids[i] if frame_ids is not None else getattr(frames[i], "frame_id", "frame_%06d" % i)
                save_frame(folder, fid, res["frames"][j])
        for k, v in res.get("recall", {}).items():
            recall[k] = recall.get(k, 0) + int(v)
    merged, total = gather_shards(local, recall, n, rank, world, device=device)
    ar = {("rcnn_%s" % t): (total.get("rcnn_%s" % t, 0) / max(total.get("gt", 0), 1)) for t in THRESH}
    return merged, total, ar


def extract_nuscenes(feed, detector, engine, folder: Optional[str] = None, batch_frames: int = 32, rank: int = 0,
                     world: int = 1, nms_thresh: Optional[float] = None, workers: int = 4, pack_xyz: bool = True,
                     device=None, loader_xyz: bool = True):
    """tools/extract_pseudo_labels.py:113-146 over a nuScenes info list, pipelined end to end:

        worker threads   NuScenesFeed.prefetch: read + transform + filter the next batch of frames
        host threads     HostPointFeeder: gather x,y,z of the batch into a pinned slot
        copy stream      H2D of the 12 B/point table
        compute stream   the five seeker stages (+ stage-4 NMS, recall counters), one D2H per batch
        this thread      per-frame .pth files (``save_frame``), recall bookkeeping

    Batch k+1 is read, gathered and uploaded while batch k is in the kernels.  Frames are sharded
    by rank as in ``extract``; returns (all_preds in dataset order, recall dict, AR per threshold).

    loader_xyz: the loader's worker threads hand over x, y, z as their own (n,3) arrays (the seeker reads
    nothing else), so the host threads only concatenate 12 B/point instead of gathering columns out of full rows.
    For the recall numbers the reference tool logs, build ``feed`` with ``training=True`` -- the mode
    tools/extract_pseudo_labels.py:47-58 runs its loader in (see NuScenesFeed)."""
    import torch
    from .seeker import HostPointFeeder
    n = len(feed)
    mine = shard_indices(n, rank, world)
    if folder is not None:
        os.makedirs(folder, exist_ok=True)
    feeder = HostPointFeeder(engine, pack=pack_xyz)
    stride, _ = feeder.layout
    local, recall = [], {}

    def finish(job):
        h, ids = job
        res = engine.result(h)
        for j, fid in enumerate(ids):
            local.append(res["frames"][j])
            if folder is not None:
                save_frame(folder, fid, res["frames"][j])
        for k, v in res.get("recall", {}).items():
            recall[k] = recall.get(k, 0) + int(v)

    def stage(slot, frames):
        feeder.submit(slot, [f.points for f in frames])      # per-frame arrays, gathered back to back

    prev, k = None, 0
    batches = feed.prefetch(mine, detector, batch_frames=batch_frames, workers=workers, xyz_only=loader_xyz)
    try:
        cur = next(batches, None)
        if cur is not None:
            stage(0, cur[0])
        prev = _pipeline(cur, batches, feeder, engine, stride, stage, finish, nms_thresh)
    finally:
        feeder.close()          # an exception between submit and upload must not leak a gather ticket
    if prev is not None:
        finish(prev)
    merged, total = gather_shards(local, recall, n, rank, world, device=device or "cpu")
    ar = {("rcnn_%s" % t): (total.get("rcnn_%s" % t, 0) / max(total.get("gt", 0), 1)) for t in THRESH}
    return merged, total, ar


def _pipeline(cur, batches, feeder, engine, stride, stage, finish, nms_thresh):
    """The steady state of extract_nuscenes; returns the last job in flight (not yet finished)."""
    prev, k = None, 0
    while cur is not None:
        frames, ids, _ = cur
        slot = k % 2
        pts, ready = feeder.upload(slot)
        nxt = next(batches, None)
        if nxt is not None:
            stage((k + 1) % 2, nxt[0])                      # gathered while this batch runs
        plan = engine.plan(frames, stride=stride)
        gt = engine.upload_gt(frames)
        h = engine.execute(plan, pts, nms_thresh=nms_thresh, gt=gt, slot=slot, points_ready=ready)
        feeder.mark_consumed(slot)
        if prev is not None:
            finish(prev)                                    # overlaps the kernels of this batch
        prev, cur, k = (h, ids), nxt, k + 1
    return prev
