#!/usr/bin/env python
"""Headline benchmark: Greedy Box Seeker frames/s (and hypotheses/s) on synthetic
nuScenes-shaped frames -- BASELINE.json configs[1] frames (10 sweeps ~300k points, 6
cameras, ~60 GLIP boxes, 64 depths x 12 yaws = 768 hypotheses per frustum), a batch of
such frames per step.

    python bench.py --gpus N --steps K --warmup W          # ours (CUDA, sm_100a)
    python bench.py --impl reference ...                    # reference CPU path on host cores
    python bench.py ... --dump-outputs DIR                  # + the last timed step's results as DIR/<name>.npy

One JSON line on stdout (rank 0).  See DESIGN.md "Measurement" for the definition of every
field.  Nothing here reads the reference's source tree; the CPU arms use oracle/_ref (the
reference's own ops, prebuilt) and the oracle restatement of the seeker loop.
"""
import argparse
import collections
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 20)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2")
    ap.add_argument("--frames", type=int, default=256, help="frames per step per GPU (BASELINE.json configs[2]: batches of 256 frames)")
    ap.add_argument("--pool-offset", type=int, default=0, help="weak scaling: rank r works on block r + offset of the synthetic "
                    "frames (diagnosis of per-rank differences: which block is more work)")
    ap.add_argument("--distinct", type=int, default=256, help="distinct synthetic frames per rank (weak scaling) / in the pool (--total-frames)")
    ap.add_argument("--total-frames", type=int, default=0,
                    help="strong scaling, BASELINE.json configs[3]: this many frames in all, sharded rank::world "
                         "(6019 = the nuScenes val sweep); steps = ceil(shard / frames), so --steps is refused")
    ap.add_argument("--layout", default="xyz", choices=["xyz", "rows"],
                    help="point table the loader hands over: x,y,z as its own array (12 B/point, no gather) or the "
                         "reference's rows (5 columns; the e2e arm gathers x,y,z on the host)")
    ap.add_argument("--cpu-sample-frames", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--score-mode", default="auto", choices=["auto", "direct", "sweep"],
                    help="stage-2b kernel (include/fnp.h FNP_SCORE_*); both give the same counts")
    ap.add_argument("--split-points", type=int, default=None)
    ap.add_argument("--pack-threads", type=int, default=None)
    ap.add_argument("--slots", type=int, default=3, help="batches in flight on the device (streams + arenas), resident arm")
    ap.add_argument("--opt", action="append", default=[], help="name=value tuning switch (fnp_set_option), A/B runs only")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step of the timed (resident) run returned -- "
                         "proposals, per-candidate results, recall counters -- as DIR/<name>.npy (float32 / float64, "
                         "rank 0), to compare two builds output for output; a seeded sample of the frames above 64 MB")
    a = ap.parse_args()
    if a.total_frames > 0 and a.steps is not None:
        ap.error("--total-frames sets the number of timed steps; leave out --steps")
    if a.impl == "reference" and a.dump_outputs:
        ap.error("--dump-outputs writes the results of the CUDA path (--impl ours)")
    a.steps = 20 if a.steps is None else a.steps
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return a


# --------------------------------------------------------------------------- outputs
def dump_outputs(out_dir, res, plan, limit=64 << 20):
    """SeekerEngine.finish's result of one batch as .npy files: per proposal (frames back to back) boxes, 2D scores,
    labels, stage-4 keep flags; per candidate frustum validity, point / valid-hypothesis counts and the best
    hypothesis (zero where invalid; with topk > 1 these hold slot 0, the per-proposal arrays every slot); the recall
    counters in the engine's order (RECALL_KEYS, then RECALL_PER_THRESH per IoU threshold).  Integers are stored as
    float64 (exact).  Above `limit` bytes, the frames are a seeded sample (frame_index says which); the recall
    counters always count the whole batch."""
    n_frames = len(res["frames"])
    fcs = plan["frame_cand_start"]

    def arrays(frames):
        fr = [res["frames"][b] for b in frames]
        cand = np.concatenate([np.arange(fcs[b], fcs[b + 1]) for b in frames]).astype(np.int64)
        valid = res["cand_valid"][cand]
        f64 = lambda x: np.asarray(x, np.float64)                               # noqa: E731
        out = {
            "frame_index": f64(frames),
            "frame_pred_count": f64([f["pred_boxes"].shape[0] for f in fr]),
            "frame_cand_count": f64(np.diff(fcs)[frames]),
            "pred_boxes": np.concatenate([f["pred_boxes"] for f in fr]).astype(np.float32).reshape(-1, 7),
            "pred_scores": np.concatenate([f["pred_scores"] for f in fr]).astype(np.float32),
            "pred_labels": f64(np.concatenate([f["pred_labels"] for f in fr])),
            "cand_valid": valid.astype(np.float32),
            "cand_npts": f64(res["cand_npts"][cand]),
            "cand_nvalid": f64(res["cand_nvalid"][cand]),
            "cand_boxes": np.where(valid[:, None], res["cand_boxes"][cand], 0).astype(np.float32),
            "cand_score2": np.where(valid, res["cand_score2"][cand], 0).astype(np.float32),
            "cand_best": f64(np.where(valid, res["cand_best"][cand], 0)),
            "cand_count": f64(np.where(valid, res["cand_count"][cand], 0)),
        }
        if fr and "nms_keep" in fr[0]:
            out["pred_nms_keep"] = np.concatenate([f["nms_keep"] for f in fr]).astype(np.float32)
        if "recall" in res:
            out["recall"] = f64(list(res["recall"].values()))
        return out

    frames = np.arange(n_frames)
    out = arrays(frames)
    rng = np.random.default_rng(0)
    while sum(v.nbytes for v in out.values()) > limit and len(frames) > 1:
        frames = np.sort(rng.choice(n_frames, len(frames) // 2, replace=False))
        out = arrays(frames)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed regions.  NVML in a thread (a few
    ms per sample, so that even a 20 ms timed region is covered); nvidia-smi -lms as fallback."""
    BAD = (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20))

    def __init__(self, index=0, period_s=0.004):
        self.index, self.period, self.rows = index, period_s, []
        self.stop_flag, self.thread, self.proc, self.nvml = False, None, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.nvml = pynvml
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            q = "clocks.sm,clocks.max.sm,clocks_event_reasons.active"
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read_smi, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll_nvml(self):
        n = self.nvml
        mx = n.nvmlDeviceGetMaxClockInfo(self.h, n.NVML_CLOCK_SM)
        get_reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop_flag:
            try:
                self.rows.append((float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)), float(mx),
                                  int(get_reasons(self.h)), n.nvmlDeviceGetUtilizationRates(self.h).gpu))
            except Exception:
                pass
            time.sleep(self.period)

    def _read_smi(self):
        for line in self.proc.stdout:
            r = [x.strip() for x in line.split(",")]
            try:
                self.rows.append((float(r[0]), float(r[1]), int(r[2], 16), 100))
            except Exception:
                continue

    def stop(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        if self.thread:
            self.thread.join(timeout=2)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(r[0] for r in self.rows)
        top = sm[len(sm) // 2:]                  # samples under load = upper half
        bits = 0
        for r in self.rows:
            bits |= r[2]
        reasons = sorted(name for name, bit in self.BAD if bits & bit)
        return {"sm_mhz": float(np.median(top)), "sm_max_mhz": float(max(r[1] for r in self.rows)), "reasons": reasons,
                "samples": len(sm), "source": "nvml" if self.nvml else "nvidia-smi"}


# --------------------------------------------------------------------------- data
def _synth_standalone():
    """The synthetic-frame generator loaded from its file, WITHOUT importing the findnpropagate_b200 package:
    the reference arm must not map the product's library (synth.py itself needs numpy and torch only)."""
    import importlib.util
    name = "fnp_bench_synth"
    if name in sys.modules:
        return sys.modules[name]
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, "findnpropagate_b200", "synth.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def make_frames(cfg_name, first_index, n, device, standalone=False):
    if standalone:
        import types
        synth = _synth_standalone()
        FrameInput = lambda **kw: types.SimpleNamespace(**kw)      # noqa: E731
    else:
        from findnpropagate_b200 import synth
        from findnpropagate_b200.seeker import FrameInput
    cfg = synth.CONFIGS[cfg_name]
    out = []
    for i in range(n):
        f = synth.make_frame(first_index + i, cfg, device=device)
        out.append(FrameInput(points=f.points, lidar2image=f.lidar2image, camera2lidar=f.camera2lidar,
                              camera_intrinsics=f.camera_intrinsics, det_boxes=f.det_boxes, det_labels=f.det_labels,
                              det_scores=f.det_scores, det_cam_idx=f.det_cam_idx, gt_boxes=f.gt_boxes))
        if not standalone:
            out[-1].prepare()      # per-frame loader work (typed arrays, camera matrices), once per frame
    return out, synth.seeker_params(cfg)


# --------------------------------------------------------------------------- CPU arms
def _cpu_frame(args):
    """Reference CPU path for one frame: the seeker loop restated with numpy/torch-CPU
    calling the reference-compiled points_in_boxes_cpu for the per-hypothesis counts."""
    fi, params, kind = args
    import oracle as O
    import seeker_oracle as SO
    if kind == "reference":
        import build_ref
        import torch
        rp = build_ref.load("roiaware_pool3d_cuda")

        def count(points, boxes):
            out = torch.zeros((boxes.shape[0], points.shape[0]), dtype=torch.int32)
            rp.points_in_boxes_cpu(torch.from_numpy(np.ascontiguousarray(boxes, np.float32)),
                                   torch.from_numpy(np.ascontiguousarray(points[:, :3], np.float32)), out)
            return out.sum(1).numpy().astype(np.int32)
        O_count, O.count_in_boxes = O.count_in_boxes, count
    try:
        r = SO.seek_frame(fi.points, fi.lidar2image, fi.camera2lidar, fi.camera_intrinsics,
                          (fi.det_boxes, fi.det_labels, fi.det_scores, fi.det_cam_idx), params)
    finally:
        if kind == "reference":
            O.count_in_boxes = O_count
    return r["pred_boxes"].shape[0]


def cpu_kind():
    try:
        import build_ref
        build_ref.load("roiaware_pool3d_cuda")
        return "reference"
    except Exception:
        return "port"


def cpu_baseline(frames, params, n_frames):
    kind = cpu_kind()
    import oracle as O
    O.lib()
    t = time.perf_counter()
    for fi in frames[:n_frames]:
        _cpu_frame((fi, params, kind))
    dt = time.perf_counter() - t
    return {"value": n_frames / dt, "unit": "frames/s", "cores": 1, "kind": kind,
            "sample": "%d frame(s) of the same workload, single thread: seeker loop restated on the host + "
                      "reference points_in_boxes_cpu (oracle/_ref)" % n_frames if kind == "reference" else
                      "%d frame(s), single thread, oracle port" % n_frames}


_REF = {}


def _ref_init(frames, params, kind):
    """Pool initializer (spawned process): single-threaded torch, frames of the workload."""
    os.environ["OMP_NUM_THREADS"] = "1"
    import torch
    torch.set_num_threads(1)
    _REF.update(frames=frames, params=params, kind=kind)
    import oracle as O
    O.lib()
    if kind == "reference":
        import build_ref
        build_ref.load("roiaware_pool3d_cuda")


def _ref_job(i):
    return _cpu_frame((_REF["frames"][i % len(_REF["frames"])], _REF["params"], _REF["kind"]))


def run_reference_arm(a):
    """bench.py --impl reference: the reference's CPU implementation of the path on all host
    cores (frame-parallel, one frame per process).  Processes are SPAWNED, not forked: forking
    after torch has started its thread pools deadlocks the children."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = len(os.sched_getaffinity(0))
    kind = cpu_kind()
    procs = max(1, min(cores, 16))
    frames, params = make_frames(a.config, 0, min(a.distinct, procs), "cpu", standalone=True)
    assert not any("findnpropagate_b200" in m for m in sys.modules), "the reference arm must not import the product"
    per_step = procs                              # bounded sample: one frame per process and step
    ctx = mp.get_context("spawn")
    with ctx.Pool(processes=procs, initializer=_ref_init, initargs=(frames, params, kind)) as pool:
        for _ in range(a.warmup):
            pool.map(_ref_job, range(per_step), chunksize=1)
        t = time.perf_counter()
        for _ in range(a.steps):
            pool.map(_ref_job, range(per_step), chunksize=1)
        dt = time.perf_counter() - t
    fps = per_step * a.steps / dt
    H = params["num_mags"] * params["num_rotations"] * params["num_sizes"]
    line = {
        "impl": "reference", "metric": "box_seeker_frames_per_s", "value": fps, "unit": "frames/s",
        "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * dt / a.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "%s frames (BASELINE.json configs[1] shape), %d hypotheses/frustum; bounded sample: "
                               "%d frames per step" % (a.config, H, per_step)},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": procs, "kind": kind,
                         "sample": "%d frames per step, frame-parallel over %d processes (host has %d cores)"
                                   % (per_step, procs, cores)},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- ours
def bind_numa(local):
    """Pins this rank's threads to the CPUs of the NUMA node its GPU hangs off, BEFORE any pinned host memory
    is allocated (first touch), so that the H2D DMA of every rank reads node-local DRAM.  Best effort."""
    info = {"node": None, "cpus": None}
    try:
        import torch
        bus = torch.cuda.get_device_properties(local).pci_bus_id
        dom = torch.cuda.get_device_properties(local).pci_domain_id
        dev_id = torch.cuda.get_device_properties(local).pci_device_id
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (dom, bus, dev_id)
        node = int(open(path).read().strip())
        if node < 0:
            return info
        cl = open("/sys/devices/system/node/node%d/cpulist" % node).read().strip()
        cpus = set()
        for part in cl.split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
            info = {"node": node, "cpus": len(allowed)}
    except Exception as e:          # containers without sysfs / a restricted cpuset: leave the affinity alone
        info["error"] = type(e).__name__
    return info


def run_ours(a):
    import torch
    import torch.distributed as dist
    from findnpropagate_b200 import _lib
    from findnpropagate_b200.seeker import HostPointFeeder, SeekerEngine

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (ours) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_numa(local) if world > 1 else {"node": None, "cpus": None}
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    for o in a.opt:
        name, _, val = o.partition("=")
        _lib.check(_lib.lib.fnp_set_option(name.encode(), int(val)), "fnp_set_option(%s)" % o)
    B, D = a.frames, a.distinct
    strong = a.total_frames > 0
    if strong:
        # BASELINE.json configs[3]: a FIXED set of frames sharded rank::world (extract.shard_indices, the reference's
        # rule, pcdet/datasets/__init__.py:43-48), fill/drain, the ragged last batch and the gather inside the timing.
        # Global frame i carries synthetic frame i % D; every rank generates the pool, so that rank 0 can re-run any
        # other rank's frames for the gather check.  (W B) % D == 0 makes every batch of a rank the same table.
        assert (world * B) % D == 0, "--total-frames needs (world * frames) % distinct == 0"
        pool, params = make_frames(a.config, 0, D, str(dev))
        n_mine = len(range(rank, a.total_frames, world))
        n_steps = max(1, -(-n_mine // B))
        tail = n_mine - (n_steps - 1) * B

        def content(r, j):
            return (r + world * j) % D
    else:
        # weak scaling: the same NUMBER of frames per rank and step, but every rank works on its own D distinct
        # synthetic frames (indices rank D .. rank D + D - 1)
        pool, params = make_frames(a.config, (rank + a.pool_offset) * D, D, str(dev))
        n_steps, tail = a.steps, B

        def content(r, j):
            return j % D
    batch = [pool[content(rank, j)] for j in range(B)]
    eng = SeekerEngine(params, device=dev, score_mode=a.score_mode, split_points=a.split_points, host_cache=False)
    H = eng.H
    # ---- the batch's point table on the host (pinned) and on the device, two copies of each (A/B) so that
    # consecutive steps never touch the same HBM lines; each is B x ~4 MB, well above the 126 MB L2.
    # layout "xyz": the loader keeps x, y, z as their own (rows,3) array (nuscenes_feed.py emits it while it
    # concatenates the sweeps), so 12 B/point cross PCIe with no gather pass; "rows": the reference's full rows
    # (5 columns) on the host, gathered to 12 B/point by HostPointFeeder's threads (round-1 path).
    width = 3 if a.layout == "xyz" else batch[0].points.shape[1]
    row_end = np.zeros(B + 1, np.int64)
    np.cumsum([f.points.shape[0] for f in batch], out=row_end[1:])
    rows = int(row_end[-1])
    pinned = []
    for s in range(2):
        t = torch.empty((rows, width), dtype=torch.float32, pin_memory=True)
        for j, f in enumerate(batch):
            t[row_end[j]:row_end[j + 1]] = torch.from_numpy(np.ascontiguousarray(f.points[:, :width]))
        pinned.append(t)
    dev_pts = [p.to(dev) for p in pinned]
    gt = eng.upload_gt(batch)
    in_bytes = pinned[0].numel() * 4

    comp = [torch.cuda.Stream(device=dev) for _ in range(max(2, a.slots))]
    feeder = HostPointFeeder(eng, pack=(a.layout == "rows"), n_threads=a.pack_threads)
    copy_stream = feeder.copy_stream

    def nf_of(k):
        """frames of timed step k: full batches, then the ragged tail of the shard (strong scaling only)"""
        return B if k < n_steps - 1 else tail

    from concurrent.futures import ThreadPoolExecutor
    planner = ThreadPoolExecutor(max_workers=1)      # plan of batch k+1 (one C call, GIL released) under execute of batch k
    planned = {}

    def get_plan(k, nf, nf_next, stride):
        fut = planned.pop((k, nf), None)
        plan = fut.result() if fut is not None else eng.plan(batch if nf == B else batch[:nf], stride=stride, xyz_offset=0)
        if nf_next is not None:
            planned[(k + 1, nf_next)] = planner.submit(eng.plan, batch if nf_next == B else batch[:nf_next],
                                                       stride=stride, xyz_offset=0)
        return plan

    def step(k, resident, prev, nf=B, nf_next=None):
        """One pass of the hot path over one batch of nf frames; nf_next: frames of the step after it (None: this is
        the last one).  Returns the result of the oldest batch in flight, if any."""
        fk = batch if nf == B else batch[:nf]
        slot = k % len(comp) if resident else k % 2
        if resident:
            pts, ready = dev_pts[k % 2][:row_end[len(fk)]], None
            plan = get_plan(k, nf, nf_next, width)
        else:
            # this step's points come from (pinned) host memory inside the timed region, H2D on a copy stream so
            # that it overlaps the previous step's kernels
            pts, ready = feeder.upload(k % 2)
            if nf_next is not None:
                feeder.submit((k + 1) % 2, pinned[(k + 1) % 2][:row_end[nf_next]])
            plan = get_plan(k, nf, nf_next, 3)
        with torch.cuda.stream(comp[slot]):
            h = eng.execute(plan, pts, nms_thresh=0.1, gt=gt, slot=slot, points_ready=ready)
            if not resident:
                feeder.mark_consumed(k % 2)
        prev.append(h)
        res = None
        if len(prev) >= (len(comp) if resident else 2):           # the oldest batch in flight: its result is
            old = prev.popleft()                                  # assembled under the GPU work of the newer ones
            res = eng.finish(old)
            if world > 1:
                exchange_add(res, old["plan"])
        return res

    exchange_ms = [0.0]     # host + device time of that exchange in the last timed run (it is inside the timing)
    ms_by_rank = {}         # per-rank ms/step of the last timed runs (the reported time is their maximum)
    xbuf = {}               # exchange slabs (pinned host + device), sized before the timing starts

    def exchange_setup(n):
        cap = B * 64
        xbuf["n"], xbuf["cap"], xbuf["i"] = n, cap, 0
        xbuf["pack"] = eng.arena.get("gather_pack", n * cap * 9 * 4, pinned=True)[:n * cap * 9 * 4] \
            .view(torch.float32).view(n, cap, 9)
        xbuf["cnt"] = eng.arena.get("gather_cnt", n * B * 4, pinned=True)[:n * B * 4].view(torch.int32).view(n, B)
        xbuf["cnt"].zero_()
        xbuf["tp"] = eng.arena.get("gather_pack_dev", n * cap * 9 * 4)[:n * cap * 9 * 4].view(torch.float32).view(n, cap, 9)
        xbuf["tc"] = eng.arena.get("gather_cnt_dev", n * B * 4)[:n * B * 4].view(torch.int32).view(n, B)
        xbuf["allp"] = eng.arena.get("gather_all_pack", world * n * cap * 9 * 4)[:world * n * cap * 9 * 4] \
            .view(torch.float32).view(world, n, cap, 9)
        xbuf["allc"] = eng.arena.get("gather_all_cnt", world * n * B * 4)[:world * n * B * 4] \
            .view(torch.int32).view(world, n, B)
        xbuf["recall"] = None

    def exchange_add(res, plan):
        """Pack one step's proposals into the slab as soon as they are on the host (this overlaps the
        kernels of the next step): [box7, score, label] rows back to back, per-frame counts beside."""
        i = xbuf["i"]
        m = res["cand_valid"]
        n = int(m.sum())
        assert n <= xbuf["cap"] and i < xbuf["n"]
        pk = xbuf["pack"].numpy()
        pk[i, :n, :7] = res["cand_boxes"][m]
        pk[i, :n, 7] = plan["cand_score"][m]
        pk[i, :n, 8] = plan["cand_label"][m]
        csum = np.concatenate([[0], np.cumsum(m)])
        per_frame = np.diff(csum[plan["frame_cand_start"]])
        xbuf["cnt"].numpy()[i, :per_frame.shape[0]] = per_frame
        rc = res["recall"]
        xbuf["recall"] = dict(rc) if xbuf["recall"] is None else {k: xbuf["recall"][k] + rc[k] for k in rc}
        xbuf["i"] = i + 1

    def gather_results():
        # frame-sharded run: ONE all_gather of fixed-stride packed proposals (+ per-frame counts) and
        # ONE all_reduce of the recall counters for the whole shard (NCCL over NVLink), as in
        # findnpropagate_b200.extract.gather_shards; fixed-capacity slabs, so no sizes are negotiated.
        xbuf["tp"].copy_(xbuf["pack"], non_blocking=True)
        xbuf["tc"].copy_(xbuf["cnt"], non_blocking=True)
        dist.all_gather_into_tensor(xbuf["allp"], xbuf["tp"])
        dist.all_gather_into_tensor(xbuf["allc"], xbuf["tc"])
        keys = sorted(xbuf["recall"]) if xbuf["recall"] else []
        rc = torch.tensor([xbuf["recall"][k] for k in keys], dtype=torch.int64, device=dev)
        dist.all_reduce(rc)
        return xbuf["allp"], xbuf["allc"], rc

    def drain(prev):
        """Finishes the batches still in flight; returns (result, plan) of the newest one."""
        last = None
        while prev:
            old = prev.popleft()
            last = eng.finish(old), old["plan"]
            if world > 1:
                exchange_add(last[0], old["plan"])
        return last

    gathered = {}

    def timed(resident, steps, warmup):
        prev = collections.deque()
        if world > 1:
            exchange_setup(max(warmup, 1))
        if not resident and warmup > 0:
            feeder.submit(0, pinned[0])
        for k in range(warmup):
            step(k, resident, prev, B, B if k + 1 < warmup else None)
        if prev:
            drain(prev)
            if world > 1:
                gather_results()           # warm-up of the exchange too (NCCL connects lazily per collective)
        if world > 1:
            exchange_setup(steps)          # the slabs at their final size, outside the timing
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = eng.launches
        cur = torch.cuda.current_stream(dev)
        e0.record()
        for st in comp + [copy_stream]:
            st.wait_event(e0)                  # nothing of the timed region starts before e0
        t_host = time.perf_counter()
        h0 = dict(eng.host_s)
        if not resident:
            feeder.submit(0, pinned[0][:row_end[nf_of(0)]])   # the first upload is inside the timed region too
        for k in range(steps):
            step(k, resident, prev, nf_of(k), nf_of(k + 1) if k + 1 < steps else None)
        last = drain(prev)
        ms_pre = 0.0
        if world > 1:
            # this rank's own time up to the exchange (the ranks leave the timed region together, through the collective:
            # the per-rank totals below are equal by construction, these are not)
            for st in comp + [copy_stream]:
                st.synchronize()
            ms_pre = 1e3 * (time.perf_counter() - t_host)
            t_x = time.perf_counter()
            g = gather_results()
            torch.cuda.synchronize()
            exchange_ms[0] = 1e3 * (time.perf_counter() - t_x)
        for st in comp + [copy_stream]:
            cur.wait_stream(st)                # e1 after everything the timed region enqueued
        e1.record()
        torch.cuda.synchronize()
        ms = max(e0.elapsed_time(e1), 1e3 * (time.perf_counter() - t_host) if not resident else 0.0)
        if world > 1 and resident:      # kept for the gather check (outside the timing: the product path does not read them back)
            gathered["allp"], gathered["allc"] = g[0].cpu().numpy().copy(), g[1].cpu().numpy().copy()
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            every = torch.empty(world, dtype=torch.float64, device=dev)
            dist.all_gather_into_tensor(every, t)
            ms_by_rank[("resident" if resident else "e2e")] = [round(float(x) / steps, 4) for x in every.tolist()]
            t = torch.tensor([ms_pre], dtype=torch.float64, device=dev)
            dist.all_gather_into_tensor(every, t)
            ms_by_rank[("resident" if resident else "e2e") + "_before_exchange"] = [round(float(x) / steps, 4) for x in every.tolist()]
            ms = float(every.max().item())
            dist.barrier()
        host_ms = {k: 1e3 * (eng.host_s[k] - h0[k]) / steps for k in h0}
        return ms, last, eng.launches - l0, host_ms

    def gather_check():
        """Rank 0 re-runs frames of every rank's shard alone (one batch, same engine code) and compares them with
        what arrived through the all_gather: boxes bit for bit, 2D scores, labels, per-frame counts."""
        checked = 0
        chk = SeekerEngine(params, device=dev, score_mode=a.score_mode)
        for r in range(world):
            pos = list(range(0, B, max(1, B // 16))) if strong else [0, D // 2, D - 1]
            if strong:      # frames of rank r's first batch
                pos = [j for j in pos if j < min(B, len(range(r, a.total_frames, world)))]
            if strong:
                fr = [pool[content(r, j)] for j in pos]
            elif r == rank:
                fr = [pool[j % D] for j in pos]
            else:
                fr = [make_frames(a.config, (r + a.pool_offset) * D + (j % D), 1, str(dev))[0][0] for j in pos]
            res = chk.run(fr, nms_thresh=0.1, with_recall=True)
            cnt = gathered["allc"][r, 0]
            off = np.concatenate([[0], np.cumsum(cnt)])
            for i, j in enumerate(pos):
                got = gathered["allp"][r, 0, off[j]:off[j + 1]]
                want = res["frames"][i]
                if got.shape[0] != want["pred_boxes"].shape[0] or \
                        not np.array_equal(got[:, :7].view(np.uint32), want["pred_boxes"].view(np.uint32)) or \
                        not np.array_equal(got[:, 7], want["pred_scores"]) or \
                        not np.array_equal(got[:, 8].astype(np.int32), want["pred_labels"]):
                    return "MISMATCH rank %d frame %d" % (r, j)
                checked += 1
        return "ok (%d frames of %d ranks re-run on rank 0, bit-equal to the gathered proposals)" % (checked, world)

    def h2d_ceiling(iters=4):
        """Pinned -> device copies of this rank's point table, all ranks at the same time: what the link (and the
        host memory behind it) delivers with nothing else going on."""
        dst = torch.empty_like(dev_pts[0])
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(copy_stream):
            dst.copy_(pinned[0], non_blocking=True)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        with torch.cuda.stream(copy_stream):
            e0.record(copy_stream)
            for i in range(iters):
                dst.copy_(pinned[i % 2], non_blocking=True)
            e1.record(copy_stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        per_rank = [ms]
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            every = torch.empty(world, dtype=torch.float64, device=dev)
            dist.all_gather_into_tensor(every, t)
            per_rank = every.tolist()
        gbs = [in_bytes * iters / (m * 1e-3) / 1e9 for m in per_rank]
        return {"per_rank_gbs": [round(g, 2) for g in gbs], "aggregate_gbs": world * in_bytes * iters / (max(per_rank) * 1e-3) / 1e9}

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_res, last, launches, host_res = timed(True, n_steps, a.warmup)
    ms_e2e, _, _, host_e2e = timed(False, n_steps, a.warmup)
    clocks = sampler.stop() if rank == 0 else None
    check = None
    if world > 1:
        check = gather_check() if rank == 0 else None
        dist.barrier()
    ceiling = h2d_ceiling()

    # ---- the two heaviest stages in isolation, CUDA events on the launching stream, L2 flushed
    plan = eng.plan(batch, stride=width, xyz_offset=0)
    h = eng.execute(plan, dev_pts[0])
    res = eng.finish(h)
    score_mode = eng.last_score_mode
    stream = _lib.current_stream(dev)
    import ctypes as C
    scr = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def stage_ms(fn, iters=10):
        for _ in range(3):
            fn(C.byref(eng.cfg), C.byref(h["batch"]), stream)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tot = 0.0
        for _ in range(iters):
            scr.zero_()                                   # flush L2 (256 MB > 126 MB)
            e0.record()
            rc = fn(C.byref(eng.cfg), C.byref(h["batch"]), stream)
            e1.record()
            torch.cuda.synchronize()
            assert rc == 0
            tot += e0.elapsed_time(e1)
        return tot / iters

    cull_ms = stage_ms(_lib.lib.fnp_seeker_cull)          # later stages read what cull leaves: run it first
    stats_ms = stage_ms(_lib.lib.fnp_seeker_frustum_stats)
    hyp_ms = stage_ms(_lib.lib.fnp_seeker_hypotheses)
    score_ms = stage_ms(_lib.lib.fnp_seeker_score)
    select_ms = stage_ms(_lib.lib.fnp_seeker_select)
    npts = res["cand_npts"].astype(np.int64)
    nval = res["cand_nvalid"].astype(np.int64)
    n_rows = int(plan["total_rows"])
    n_dets = sum(len(f.det_scores) for f in batch)
    # algorithmic bytes per launch, SURVEY.md section 8(d): stage 1 = 16 N + 16 sum P_f + 16 D;
    # stage 2 = 16 sum P_f + 28 nv + 4 nv (+ 4 nv for the 2D IoU the score needs) over the valid hypotheses
    alg = {"cull": float(16 * n_rows + 16 * npts.sum() + 16 * n_dets),
           "score": float(16 * npts[nval > 0].sum() + 36 * nval.sum())}
    tests = float((npts * nval).sum())
    J = int(params["num_rotations"] * params["num_sizes"])
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 (of fallback)"
    traffic = {}
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "kernel_traffic.json")))
        if tj.get("config") == a.config and tj.get("frames") == B and tj.get("layout") == a.layout:
            traffic = tj.get("dram_bytes_per_launch", {})
    except Exception:
        pass
    score_kernel = "fnp::sweep_score_kernel" if score_mode == "sweep" else "fnp::score_kernel"

    def roof(name, kernel, ms, note):
        ach = alg[name] / (ms * 1e-3) / 1e9
        return {"kernel": kernel, "stage": name, "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                "frac": ach / hbm_peak, "traffic": traffic.get(kernel), "peak_source": peak_src, "ms_per_launch": ms,
                "algorithmic_bytes_per_launch": alg[name], "note": note}
    roofs = {
        "score": roof("score", score_kernel, score_ms,
                      "stage 2b (per-hypothesis point counts), timed through fnp_seeker_score (includes its small "
                      "planning kernels).  Bound by instruction issue, not HBM (DESIGN.md section 4): the sweep kernel "
                      "solves one depth range per (point, column) pair instead of testing every (point, hypothesis) pair"
                      if score_mode == "sweep" else
                      "stage 2b, direct kernel: bound by the SM's ALU/FMA pipes, not by HBM (DESIGN.md section 4)"),
        "cull": roof("cull", "fnp::cull_kernel", cull_ms,
                     "stage 1 (projection + frustum cull + ordered compaction), timed through fnp_seeker_cull (all its "
                     "launches); HBM-bound by design, instruction-issue-bound as measured"),
    }
    dominant = "score" if score_ms >= cull_ms else "cull"
    other = "cull" if dominant == "score" else "score"
    roofs["score"].update({
        "score_mode": score_mode, "point_box_tests_equivalent_per_launch": tests,
        "point_column_range_solves_per_launch": float(npts[nval > 0].sum() * J) if score_mode == "sweep" else None})

    if rank == 0:
        total = a.total_frames if strong else B * world * n_steps
        F_step = plan["F"]
        cpu = None if (a.no_cpu_baseline or world > 1) else cpu_baseline(batch, params, a.cpu_sample_frames)
        h2d_step = int(n_rows * 12 + sum(plan[k].nbytes for k in eng._META))
        # bytes this rank really uploaded in the timed e2e run (the last batch of a strong-scaling shard is ragged)
        h2d_run = sum(int(row_end[nf_of(k)]) * 12 for k in range(n_steps)) + n_steps * sum(plan[k].nbytes for k in eng._META)
        e2e_fps = total / (ms_e2e * 1e-3)
        line = {
            "metric": "box_seeker_frames_per_s", "value": total / (ms_res * 1e-3), "unit": "frames/s",
            "n_gpus": world, "steps": n_steps, "warmup": a.warmup, "ms_per_step": ms_res / n_steps,
            "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {
                "workload": "%s frames (%s: ~%dk points, 6 cameras, ~%d 2D boxes, "
                            "%d depths x %d yaws = %d hypotheses/frustum), batch of %d frames per step per GPU"
                            % (a.config, {"cfg1": "BASELINE.json configs[0] shape, 1 sweep",
                                          "cfg2": "BASELINE.json configs[1] shape, 10 sweeps",
                                          "cfg5": "BASELINE.json configs[4] shape, 128 beams"}.get(a.config, "custom"),
                               int(np.mean([f.points.shape[0] for f in batch]) / 1000), F_step // B,
                               params["num_mags"], params["num_rotations"] * params["num_sizes"], H, B)
                            + ("; BASELINE.json configs[3]: %d frames in all, sharded rank::world, ragged last batch, "
                               "fill/drain and the gather inside the timing" % a.total_frames if strong else ""),
                "frames_per_step_per_gpu": B,
                "distinct_frames": ("%d in the pool, global frame i = pool[i %% %d]" % (D, D)) if strong else
                                   "%d per rank, different on every rank (synthetic indices rank*%d ..)" % (D, D),
                "host_planning": "per frame, once, by the loader: typed detection arrays + camera matrices (FrameInput."
                                 "prepare); per batch: one fnp_host_plan call (2D NMS, candidate order, tile table), for "
                                 "batch k+1 on a worker thread while batch k is enqueued",
                "point_layout": "x,y,z as its own (rows,3) array on the host and on the device (the loader splits the "
                                "columns while it concatenates the sweeps)" if a.layout == "xyz" else
                                "reference rows (5 columns) on the host and on the device",
                "l2_policy": "inputs larger than L2: %.0f MB of points per step, two alternating input sets" % (in_bytes / 1e6),
                "sharding": ("frame-wise, no data-path collective; one all_gather of packed proposals + one "
                             "all_reduce of recall counters per run, inside the timed region (%.2f ms of the run)"
                             % exchange_ms[0]) if world > 1 else "single GPU",
                "numa": numa},
            "hypotheses_per_s": (total / B) * F_step * H / (ms_res * 1e-3),
            "point_box_tests_equivalent_per_s_scoring_stage": tests / (score_ms * 1e-3),
            "e2e": {"value": e2e_fps, "unit": "frames/s",
                    "h2d_bytes_per_step": h2d_step,
                    "d2h_bytes_per_step": int(4 * (12 * plan["F"] + 8) + plan["F"]),
                    "ms_per_step": ms_e2e / n_steps,
                    "host_input_bytes_per_step": int(in_bytes),
                    "host_pack": ("rows on the host: x,y,z gathered by %d threads (fnp_host_pack_xyz), 12 B/point uploaded"
                                  % feeder.n_threads) if feeder.pack else
                                 "none: the loader's (rows,3) x,y,z array is uploaded as is, 12 B/point, same at every N",
                    "h2d_ceiling": ceiling,
                    "frac_of_h2d_ceiling": (world * h2d_run / (ms_e2e * 1e-3) / 1e9) / ceiling["aggregate_gbs"]},
            "gpu_launches": int(launches),
            "gather_check": check,
            "ms_per_step_by_rank": ms_by_rank if world > 1 else None,
            "host_ms_per_step": {"resident": host_res, "e2e": host_e2e,
                                 "note": "main-thread time in SeekerEngine.plan / execute / finish (after its event wait) per step"},
            "stage_ms": {"cull": cull_ms, "frustum_stats": stats_ms, "hypotheses": hyp_ms, "score": score_ms,
                         "select": select_ms, "note": "each stage alone through its C-ABI call, L2 flushed, CUDA events"},
            "clocks": clocks,
            "roofline": roofs[dominant],
            "roofline_second_kernel": roofs[other],
        }
        ref_gpu = os.path.join(ROOT, "profiles", "r02_reference_gpu.json")
        if os.path.exists(ref_gpu):
            try:
                rg = json.load(open(ref_gpu))
                line["reference_gpu"] = {
                    "source": "profiles/r02_reference_gpu.json (tools/ref_gpu_bench.py: the reference's own head + "
                              "kernels compiled for sm_100a, run on a B200 of this pool)",
                    "frames_per_s": {hd["config"]: hd["reference_gpu_frames_per_s"] for hd in rg.get("heads", [])}}
            except Exception:
                pass
        if cpu is not None:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, *last)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)
