#!/usr/bin/env python
"""Benchmark of the SSD box-geometry hot path (BASELINE.json metric: images/sec for
target-assign + loss + NMS, SSD300 / 8732 priors) -- one JSON line on stdout.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference          # the reference's own CPU code on the host cores
    python bench.py --dump-outputs DIR        # also save the last timed step's results as DIR/*.npy

A step is one pass of the chain over one synthetic batch per GPU (weak scaling: the per-GPU batch is fixed;
``--scaling strong --global-batch G`` fixes the total instead).  ``value`` is measured with the inputs resident in HBM,
rotating over two distinct resident batches; ``e2e`` goes through the public host API
(ssdgeom.pipeline.HotPath.submit) with pinned host buffers and the copies inside the timed region.

Besides the headline, the same invocation records under ``detail`` (BASELINE.json configs 4/5 and the north-star
scaling target, SURVEY.md section 8d):
    sustained              >= 2 s of steps over the two resident batches, clocks sampled inside that window
    strong_ssd300_b1024    SSD300, GLOBAL batch 1024 split over the N GPUs (per-shard mining), with the one-GPU
                           time of the same 1024 images measured in the same run -> strong-scaling efficiency
    ssd512_b1024           config 4: SSD512 (24 564 priors), global batch 1024 over the N GPUs
    ssd512_t500_b2048      config 5 (N = 8, or --detail-config5): SSD512, 500 GT per image, global batch 2048
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "ssd-object-detection_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "images/sec for target-assign+loss+NMS (SSD300, 8732 anchors)"
CLASSES = 81


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="images per GPU (weak scaling)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--global-batch", type=int, default=1024, help="total images with --scaling strong")
    ap.add_argument("--table", default="ssd300", choices=["ssd300", "ssd512"])
    ap.add_argument("--max-gt", type=int, default=100)
    ap.add_argument("--gt-mode", default="max", choices=["max", "coco"])
    ap.add_argument("--cpu-images", type=int, default=0, help="images in the CPU sample per step (0 = 2 x host cores)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-detail", action="store_true", help="skip the extra detail records (sustained, configs 4/5, strong scaling)")
    ap.add_argument("--detail-config5", action="store_true", help="record config 5 (SSD512, T=500, global batch 2048) at any N")
    ap.add_argument("--sustained-seconds", type=float, default=2.0)
    ap.add_argument("--depth", type=int, default=2, choices=[1, 2, 3],
                    help="steps in flight (HotPath depth): 2 = consecutive steps use alternate buffers and overlap")
    ap.add_argument("--pipeline", default="split", choices=["split", "two-stream"],
                    help="split: NMS and loss on their own streams (loss outranks NMS); two-stream: one stream per branch")
    ap.add_argument("--no-fused", action="store_true",
                    help="loss streams the logits itself (ce_kernel) instead of reusing the filter pass's row statistics")
    ap.add_argument("--mining", default="shard", choices=["shard", "global"],
                    help="hard-negative threshold over this rank's batch (reference split-batch semantics) or "
                         "over all ranks' batches (exact-global, staged all-reduces)")
    ap.add_argument("--exchange", default="ssdg", choices=["ssdg", "torch"],
                    help="data-parallel exchange through the library's own ssdg_comm_* (NCCL) or torch.distributed")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returns to its caller (loss result block, kept lists, counts; "
                         "rank 0's shard) as DIR/<name>.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the GPU path (--impl ours)")
    return args


# ---------------------------------------------------------------------------------------------------------
# CPU arm.  When the reference's own modules are importable (from /root/reference in the build container, else
# from oracle/_ref: the same modules byte-compiled by oracle/build_ref.py) the arm runs THE REFERENCE:
#   match_bbox + apply_anchor_box per image (utils/bbox.py:44-101 as chained by models/ssd_model.py:211-215) and
#   _ssd_loss (models/ssd_model.py:341-396) over a NumPy stand-in for the dozen TensorFlow ops it calls
#   (oracle/tf_shim.py; TensorFlow is not installed) -- kind "reference";
# otherwise the NumPy port oracle/ssd_oracle.py (kind "port").  The reference has no NMS: that stage is always the
# builder's restatement (oracle.ssd_oracle.detect, vectorised over classes) and is reported separately.
# ---------------------------------------------------------------------------------------------------------
_W = {}


def _worker_state(table):
    if "ref" not in _W:
        from oracle import ref_loader
        _W["ref"] = ref_loader.load() if ref_loader.available() else None
    if table not in _W:
        from oracle import ssd_oracle as O
        from ssdgeom import synth
        t = synth.TABLES[table]
        _W[table] = O.build_prior_box(t["sizes"], t["s_k_refer"], t["aspect_ratio"], t["input_size"])
    return _W["ref"], _W[table]


def _cpu_assign(task):
    (table, cls, boxes) = task
    ref, priors = _worker_state(table)
    t0 = time.perf_counter()
    if ref is not None:      # models/ssd_model.py:211-215 with the casts of the output_signature :219-224
        lab, box, mask = ref.match_bbox(cls, boxes, priors, 0.5)
        loc = ref.apply_anchor_box(box, priors)
        lab, loc, mask = np.asarray(lab, np.int32), np.asarray(loc, np.float32), np.asarray(mask, bool)
    else:
        from oracle import ssd_oracle as O
        lab, loc, mask = O.assign_encode(cls, boxes, priors, 0.5, sweeps=True)
    return lab, loc, mask, time.perf_counter() - t0


def _cpu_nms(task):
    (table, pred_cls, pred_box) = task
    from oracle import ssd_oracle as O
    _, priors = _worker_state(table)
    t0 = time.perf_counter()
    _, count, _, _ = O.detect(pred_cls, pred_box, priors)
    return int(count.sum()), time.perf_counter() - t0


def _cpu_loss(task):
    """_ssd_loss on one slice of the batch: the reference's shipped configuration calls it per `split_batch` slice
    of 4 images and averages (models/ssd_model.py:235-256, config/default.yml:40-42)."""
    (table, lo, hi, y_true) = task
    ref, _ = _worker_state(table)
    pred_box, pred_cls = _W["pred"]
    t0 = time.perf_counter()
    if ref is not None:
        total, _ = ref.ssd_loss(y_true, (pred_box[lo:hi], pred_cls[lo:hi]))              # models/ssd_model.py:341-396
    else:
        from oracle import ssd_oracle as O
        total, _ = O.ssd_loss(y_true, (pred_box[lo:hi], pred_cls[lo:hi]))
    return float(np.asarray(total)), time.perf_counter() - t0


SPLIT_BATCH = 4          # config/default.yml:40-42


class CpuArm:
    def __init__(self, args, images):
        import multiprocessing as mp
        from oracle import ref_loader
        from ssdgeom import synth
        self.cores = os.cpu_count() or 1
        self.images = images if images > 0 else 2 * self.cores
        self.table, self.args = args.table, args
        self.kind = "reference" if ref_loader.available() else "port"
        a = synth.num_priors(synth.TABLES[args.table])
        boxes, cls, off = synth.make_gt(1234, self.images, args.max_gt, args.gt_mode)
        pred_cls, pred_box = synth.make_predictions(1234, self.images, a)
        self.t_assign = [(args.table, cls[off[i]:off[i + 1]], boxes[off[i]:off[i + 1]]) for i in range(self.images)]
        self.t_nms = [(args.table, pred_cls[i], pred_box[i]) for i in range(self.images)]
        _W["pred"] = (pred_box, pred_cls)            # inherited by the forked workers
        self.procs = min(self.cores, self.images)
        self.pool = mp.get_context("fork").Pool(self.procs)
        self.wall = {"assign": 0.0, "loss": 0.0, "nms": 0.0}
        self.cpu = {"assign": 0.0, "loss": 0.0, "nms": 0.0}
        self.steps = 0

    def step(self, record=True):
        ref, _ = _worker_state(self.table)
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_assign, self.t_assign, chunksize=1)
        t1 = time.perf_counter()
        y_true = tuple(np.stack([r[k] for r in res]) for k in range(3))
        slices = [(self.table, lo, min(lo + SPLIT_BATCH, self.images), tuple(v[lo:lo + SPLIT_BATCH] for v in y_true))
                  for lo in range(0, self.images, SPLIT_BATCH)]
        losses = self.pool.map(_cpu_loss, slices, chunksize=1)
        total = float(np.mean([l[0] for l in losses]))                                # accumulate-and-average, :251-256
        t2 = time.perf_counter()
        det = self.pool.map(_cpu_nms, self.t_nms, chunksize=1)
        t3 = time.perf_counter()
        if record:
            self.steps += 1
            self.wall["assign"] += t1 - t0; self.wall["loss"] += t2 - t1; self.wall["nms"] += t3 - t2
            self.cpu["assign"] += sum(r[3] for r in res); self.cpu["loss"] += sum(l[1] for l in losses); self.cpu["nms"] += sum(d[1] for d in det)
        return float(np.asarray(total))

    def close(self):
        self.pool.close()
        self.pool.join()

    def describe(self):
        n = self.images * max(self.steps, 1)
        wall_all = sum(self.wall.values())
        wall_ref = self.wall["assign"] + self.wall["loss"]
        src = ("the reference's own match_bbox + apply_anchor_box per image and _ssd_loss per split_batch slice of 4 "
               "images, averaged (models/ssd_model.py:235-256, config/default.yml:40-42) (unmodified modules, "
               "byte-compiled from the reference tree; TensorFlow is absent, so its dozen ops run on a NumPy stand-in, "
               "oracle/tf_shim.py)") if self.kind == "reference" else \
              "NumPy port of match_bbox + apply_anchor_box (the reference's arg-max sweeps) and _ssd_loss per slice of 4 images (oracle/ssd_oracle.py)"
        return {"value": n / wall_all if wall_all else 0.0, "unit": "images/s", "cores": self.procs, "kind": self.kind,
                "sample": "%d %s images per step x %d steps (GT mode %s, <=%d GT): %s in a %d-process pool; plus the "
                          "builder-written decode + per-class NMS restatement (the reference has no NMS)" %
                          (self.images, self.table, self.steps, self.args.gt_mode, self.args.max_gt, src, self.procs),
                # seconds of CPU per image and stage (one core), and the same arm restricted to what the reference has
                "parts_s_per_image": {k: self.cpu[k] / n for k in ("assign", "loss", "nms")},
                "parts_wall_share": {k: self.wall[k] / wall_all for k in ("assign", "loss", "nms")} if wall_all else None,
                "reference_only": {"value": n / wall_ref if wall_ref else 0.0, "unit": "images/s",
                                   "stages": "assign + loss (utils/bbox.py:44-101, models/ssd_model.py:341-396); no NMS"},
                "nms_stage_kind": "port (builder-defined spec; parity unpinned)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    arm = CpuArm(args, args.cpu_images)
    for _ in range(max(args.warmup, 0)):
        arm.step(record=False)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        arm.step()
    dt = time.perf_counter() - t0
    arm.close()
    value = arm.images * args.steps / dt
    cb = arm.describe()
    cb["value"] = value
    line = base_line(args, value, dt / args.steps * 1e3, n_gpus=args.gpus, per_gpu=per_gpu_batch(args, args.gpus))
    line.update({"impl": "reference", "dtype": "f64", "cpu_baseline": cb, "gpu_launches": 0,
                 "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
    from ssdgeom import synth
    line["config"]["priors"] = synth.num_priors(synth.TABLES[args.table])
    line["config"]["l2"] = "inputs larger than L2 (logits %.0f MB per GPU)" % (
        per_gpu_batch(args, args.gpus) * line["config"]["priors"] * CLASSES * 4 / 1e6)
    print(json.dumps(line), flush=True)


def per_gpu_batch(args, world):
    if args.scaling == "strong":
        if args.global_batch % world:
            raise SystemExit("--global-batch must be a multiple of the number of GPUs")
        return args.global_batch // world
    return args.batch


def workload_name(args, per_gpu):
    return "%s chained assign+encode -> multibox loss (3:1 mining) | decode+per-class NMS, batch %d/GPU, %d classes, " \
           "GT %s<=%d" % (args.table.upper(), per_gpu, CLASSES, args.gt_mode, args.max_gt)


def base_line(args, value, ms, n_gpus, per_gpu):
    return {"metric": METRIC, "value": value, "unit": "images/s", "n_gpus": n_gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic",
            "config": {"workload": workload_name(args, per_gpu), "global_batch": per_gpu * n_gpus, "priors": None,
                       "l2": "inputs larger than L2 (logits %.0f MB per GPU)" % 0.0, "parallelism": "dp%d" % n_gpus,
                       "mining": "per-shard" if getattr(args, "mining", "shard") == "shard" else "exact-global"}}


# ---------------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1, load0=None, load1=None):
        """Median SM clock and throttle reasons over the timed window [t0, t1]; when that window is too
        short for three samples, over the whole period the GPU was under this benchmark's load."""
        out = self._summary(t0 - 0.02, t1 + 0.02)
        out["window"] = "timed region"
        if out["samples"] < 3 and load0 is not None:
            out = self._summary(load0, load1)
            out["window"] = "whole loaded period (timed region shorter than 3 samples)"
        return out

    def _summary(self, t0, t1):
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, row in self.rows:
            if t < t0 or t > t1:
                continue
            f = [x.strip() for x in row.split(",")]
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except Exception:
                continue
            try:
                pw.append(float(f[3]))
            except Exception:
                pass
            for name, v in zip(names, f[5:9]):
                if v == "Active":
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_min_mhz": min(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(pw) if pw else None}


class Ranks:
    """torch.distributed is the launcher-side plumbing only: rendezvous, barrier, max-over-ranks of a time."""

    def __init__(self):
        import torch
        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
        torch.cuda.set_device(self.local_rank)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
            self.dist = dist

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max(self, v):
        if self.dist is None:
            return v
        t = self.torch.tensor([v], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def bcast_bytes(self, payload):
        if self.dist is None:
            return payload
        box = [payload]
        self.dist.broadcast_object_list(box, src=0)
        return box[0]

    def close(self):
        if self.dist is not None:
            self.dist.destroy_process_group()


def device_predictions(torch, hp, seed):
    """Second and further resident batches are drawn on the device (same distribution as synth.make_predictions:
    logits N(0,1) with the background column +7, box regressions N(0,1) * 0.5) straight into the pipeline's buffers."""
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    pc = torch.as_tensor(hp.pred_cls, device="cuda")
    pb = torch.as_tensor(hp.pred_box, device="cuda")
    rows = max(1, (1 << 27) // (hp.A * hp.classes))        # draw in slices: normal_ needs no extra memory this way
    for i in range(0, hp.batch, rows):
        pc[i:i + rows].normal_(generator=g)
    pc[..., -1] += 7.0
    pb.normal_(generator=g)
    pb *= 0.5
    torch.cuda.synchronize()


def upload_gt(hp, boxes, cls, off):
    from ssdgeom import _native as N, device as D
    for dst, src in ((hp.gt_boxes, boxes), (hp.gt_cls, cls), (hp.gt_off, off)):
        src = np.ascontiguousarray(src)
        N.check(N.lib().ssdg_memcpy_h2d(dst.ptr, src.ctypes.data, src.nbytes, D.stream_handle(hp.s_main)), "h2d")
    hp.s_main.sync()


def chain_bytes_per_image(a, c, fused=True):
    # logits (once when the loss reuses the filter pass) + pred_box (x2 readers) + gt targets out/in + detections' decoded boxes
    return a * (c * 4 * (1 if fused else 2) + 16 * 3 + 4 + 1 + 4 + 16 + 1)


def make_comm(R, args):
    """The library's own NCCL communicator (ssdg_comm_*); the 128-byte id travels over the launcher's channel."""
    if R.world == 1 or args.exchange != "ssdg":
        return None
    from ssdgeom import comm as CM
    uid = R.bcast_bytes(CM.unique_id() if R.rank == 0 else None)
    return CM.Comm(uid, R.world, R.rank)


def torch_exchange(R, hp):
    """--exchange torch: the same sums through torch.distributed (kept for A/B against ssdg_comm)."""
    torch, dist = R.torch, R.dist
    res_t = torch.as_tensor(hp.loss["result"], device="cuda")
    streams = {}

    def exchange_on(stream):
        if stream.handle not in streams:
            streams[stream.handle] = torch.cuda.ExternalStream(stream.handle)
        with torch.cuda.stream(streams[stream.handle]):
            dist.all_reduce(res_t[4:11])

    views = {}

    def allreduce_on(buf, stream):
        key = (buf.ptr, stream.handle)
        if key not in views:
            views[key] = (torch.as_tensor(buf, device="cuda"), torch.cuda.ExternalStream(stream.handle))
        t, ts = views[key]
        with torch.cuda.stream(ts):
            dist.all_reduce(t)

    return exchange_on, allreduce_on


def build_hotpath(R, args, table_name, b, max_gt, gt_mode, comm, seed0, n_sets=1, host_set0=False, solo=False):
    """HotPath with `n_sets` resident batches.  Set 0 comes from the seeded NumPy generator when `host_set0` (the
    headline workload: also the source of the end-to-end copies), else everything is drawn on the device.
    solo: a single-process run inside a multi-process job (no exchange)."""
    from ssdgeom import device as D, synth
    from ssdgeom.pipeline import HotPath
    table = synth.TABLES[table_name]
    world = 1 if solo else R.world
    gts = [synth.make_gt(seed0 + 7 * k + R.rank * 131, b, max_gt, gt_mode) for k in range(n_sets)]
    total_gt = max(g[0].shape[0] for g in gts)
    a = synth.num_priors(table)
    kw = {}
    if world > 1 and args.mining == "global":
        kw = dict(mining="global", global_priors=b * world * a)
    use_comm = comm if world > 1 else None
    via_torch = world > 1 and comm is None          # --exchange torch
    late = {}
    hp = HotPath(table, batch=b, max_gt=max(int(np.diff(g[2]).max()) for g in gts), total_gt=total_gt, comm=use_comm,
                 allreduce=(lambda buf, st: late["allreduce"](buf, st)) if via_torch else None,
                 depth=1 if via_torch else getattr(args, "depth", 2), **kw)
    if via_torch:
        ex, late["allreduce"] = torch_exchange(R, hp)
        if args.mining == "shard":
            hp.loss_exchange = ex
    hp.split = args.pipeline == "split"
    hp.fused = not args.no_fused and hp.split
    host = None
    for k in range(n_sets):
        if k:
            hp.add_input_set()
        hp.use_set(k)
        boxes, cls, off = gts[k]
        if boxes.shape[0] < total_gt:      # sets share the buffer size: pad the CSR arrays (rows beyond off[-1] are unused)
            boxes = np.concatenate([boxes, np.zeros((total_gt - boxes.shape[0], 4), np.float32)])
            cls = np.concatenate([cls, np.zeros((total_gt - cls.shape[0],), np.float32)])
        if k == 0 and host_set0:
            c = hp.classes
            host = {"gt_boxes": D.PinnedArray(boxes.shape, np.float32), "gt_cls": D.PinnedArray(cls.shape, np.float32),
                    "gt_off": D.PinnedArray(off.shape, np.int32), "pred_cls": D.PinnedArray((b, a, c), np.float32),
                    "pred_box": D.PinnedArray((b, a, 4), np.float32)}
            host["gt_boxes"].array[...] = boxes; host["gt_cls"].array[...] = cls; host["gt_off"].array[...] = off
            for i in range(0, b, 16):               # generate in chunks to bound host memory
                n = min(16, b - i)
                pc, pb = synth.make_predictions(1000 * R.rank + i, n, a, c)
                host["pred_cls"].array[i:i + n] = pc; host["pred_box"].array[i:i + n] = pb
            hp.upload(*[host[k2].array for k2 in ("gt_boxes", "gt_cls", "gt_off", "pred_cls", "pred_box")])
            hp.s_main.sync()
        else:
            upload_gt(hp, boxes, cls, off)
            device_predictions(R.torch, hp, 4242 + 17 * k + R.rank)
    hp.use_set(0)
    return hp, host, gts


def timed_steps(R, hp, steps, warmup, n_sets=1, solo=False):
    """`warmup` untimed steps, then exactly `steps` steps between CUDA events on the pipeline's main stream, bracketed
    by a barrier + device synchronisation on both sides; returns (ms per step as the max over ranks, wall window)."""
    from ssdgeom import device as D
    for i in range(max(warmup, 3)):
        hp.use_set(i % n_sets)
        hp.step()
    hp.s_main.sync()
    ev0, ev1 = D.Event(), D.Event()
    if solo:
        R.torch.cuda.synchronize()
    else:
        R.barrier()
    t0 = time.perf_counter()
    ev0.record(hp.s_main)
    for i in range(steps):
        hp.use_set(i % n_sets)
        hp.step()
    hp.join()                     # (with two steps in flight s_main has not waited for them yet)
    hp.finish_exchange()          # the last step's loss exchange belongs to the timed region
    ev1.record(hp.s_main)
    hp.s_main.sync()
    if solo:
        R.torch.cuda.synchronize()
    else:
        R.barrier()
    t1 = time.perf_counter()
    ms = ev0.elapsed_ms(ev1)
    hp.check_status(sync=True)
    return (ms if solo else R.max(ms)) / steps, (t0, t1)


def detail_config(R, args, comm, table_name, global_batch, max_gt, steps=10, warmup=3, with_solo=False):
    """One extra workload inside the same invocation: `global_batch` images split over the ranks."""
    from ssdgeom import synth
    if global_batch % R.world:
        return {"skipped": "global batch %d is not a multiple of %d GPUs" % (global_batch, R.world)}
    b = global_batch // R.world
    a = synth.num_priors(synth.TABLES[table_name])
    out = {"table": table_name, "global_batch": global_batch, "per_gpu_batch": b, "max_gt": max_gt, "priors": a,
           "n_gpus": R.world, "steps": steps, "warmup": warmup, "mining": "per-shard" if args.mining == "shard" else "exact-global",
           "inputs": "device-resident, drawn on the device (logits N(0,1), background +7; boxes N(0,1)*0.5); GT from the seeded NumPy generator"}
    hp, _, _ = build_hotpath(R, args, table_name, b, max_gt, "max", comm, seed0=300, n_sets=1)
    ms, _ = timed_steps(R, hp, steps, warmup)
    out["ms_per_step"] = ms
    out["value"] = global_batch / (ms * 1e-3)
    out["unit"] = "images/s"
    peak = peaks().get("hbm_gbs", 6650.0)
    bpi = chain_bytes_per_image(a, CLASSES, hp.fused)
    out["chain_bytes_per_image"] = bpi
    out["hbm_roofline_frac"] = bpi * b / (ms * 1e-3) / 1e9 / peak        # per GPU
    del hp
    gc.collect()
    if with_solo and R.world > 1:
        # strong-scaling reference point measured in the same run: all `global_batch` images on ONE GPU (rank 0
        # alone; the other ranks wait at the barrier).  efficiency = T(1) / (N * T(N)).
        solo_ms = 0.0
        if R.rank == 0:
            hp1, _, _ = build_hotpath(R, args, table_name, global_batch, max_gt, "max", None, seed0=300, n_sets=1, solo=True)
            solo_ms, _ = timed_steps(R, hp1, steps, warmup, solo=True)
            del hp1
            gc.collect()
        solo_ms = R.max(solo_ms)
        out["one_gpu_ms_per_step_same_run"] = solo_ms
        out["one_gpu_value_same_run"] = global_batch / (solo_ms * 1e-3)
        out["efficiency"] = solo_ms / (R.world * ms)
        out["limiter"] = ("per-GPU latency, not the exchange: at %d images per GPU the step is two chains of latency-bound "
                          "kernels (filter -> NMS; row search -> per-image matching, one CTA per image -> loss) whose "
                          "per-image / per-row latencies do not shrink with the batch; the 56-byte all-reduce runs on a "
                          "stream nobody waits for inside the step (DESIGN.md section 5)" % (global_batch // R.world))
        out["scaling"] = "strong"
    elif with_solo:
        out["efficiency"] = 1.0
        out["scaling"] = "strong"
    return out


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def profile_json(name):
    try:
        return json.load(open(os.path.join(ROOT, "profiles", name)))
    except Exception:
        return None


DUMP_LIMIT_BYTES = 64 << 20


def write_outputs(path, outputs):
    """Save the last timed step's results as float64 (loss result block) and float32 (kept prior indices, -1 padded,
    and counts: exact below 2**24).  Kept lists and counts are per image; if together they would pass
    DUMP_LIMIT_BYTES, a fixed seeded sample of images is written instead, its indices in images.npy."""
    os.makedirs(path, exist_ok=True)
    arrays = {"loss_result": outputs["loss_result"].astype(np.float64), "kept": outputs["kept"].astype(np.float32),
              "count": outputs["count"].astype(np.float32)}
    batch = arrays["count"].shape[0]
    per_image = (arrays["kept"].nbytes + arrays["count"].nbytes) // batch + 8        # + its index in images.npy
    room = (DUMP_LIMIT_BYTES - arrays["loss_result"].nbytes - 4 * 4096) // per_image     # (.npy headers)
    if room < batch:
        images = np.sort(np.random.default_rng(0).choice(batch, room, replace=False))
        arrays["kept"], arrays["count"] = arrays["kept"][images], arrays["count"][images]
        arrays["images"] = images.astype(np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def run_ours(args):
    from ssdgeom import _native as N, device as D, synth
    R = Ranks()
    rank, world = R.rank, R.world
    N.check(N.lib().ssdg_set_device(R.local_rank), "set_device")
    comm = make_comm(R, args)
    b = per_gpu_batch(args, world)

    sampler = ClockSampler(R.local_rank)
    sampler.start()
    time.sleep(0.2)
    M = headline(R, args, comm, sampler, b)            # its buffers are released on return

    # ---- the other configurations of BASELINE.json, recorded by the same invocation -----------------------------
    gc.collect()
    detail_cfg = {}
    if not args.no_detail:
        detail_cfg["strong_ssd300_b1024"] = detail_config(R, args, comm, "ssd300", 1024, 100, with_solo=True)
        detail_cfg["ssd512_b1024"] = detail_config(R, args, comm, "ssd512", 1024, 100)
        if world == 8 or args.detail_config5:
            detail_cfg["ssd512_t500_b2048"] = detail_config(R, args, comm, "ssd512", 2048, 500, steps=5)
    sampler.stop()

    if rank != 0:
        if comm is not None:
            comm.close()
        R.close()
        return
    line = report(args, R, comm, b, M, detail_cfg)
    print(json.dumps(line), flush=True)
    if args.dump_outputs:
        write_outputs(args.dump_outputs, M["outputs"])
    if comm is not None:
        comm.close()
    R.close()


def headline(R, args, comm, sampler, b):
    """The headline workload (BASELINE.json configs 2+3 chained behind the assignment of config 1's shape): resident
    value, sustained window, per-stage / per-kernel times, end to end.  Returns plain numbers only."""
    from ssdgeom import _native as N, device as D
    world = R.world
    t_load0 = time.perf_counter()
    n_sets = 2
    hp, host, gts = build_hotpath(R, args, args.table, b, args.max_gt, args.gt_mode, comm, seed0=100, n_sets=n_sets,
                                  host_set0=True)
    a, c = hp.A, hp.classes
    off = gts[0][2]
    host_in = [host[k].array for k in ("gt_boxes", "gt_cls", "gt_off", "pred_cls", "pred_box")]
    o = {"result": D.PinnedArray((N.LOSS_RESULT_LEN,), np.float64), "kept": D.PinnedArray((b, c - 1, hp.top_k), np.int32),
         "count": D.PinnedArray((b, c - 1), np.int32)}
    host_out = [o[k].array for k in ("result", "kept", "count")]

    # ---- timed region: device-resident chain, rotating over the resident batches -----------------------------
    ms_step, (t0, t1) = timed_steps(R, hp, args.steps, args.warmup, n_sets=n_sets)
    value = b * world * 1e3 / ms_step
    hp.use_set((args.steps - 1) % n_sets)
    res = hp.loss["result"].to_host()
    # the buffers HotPath.download reads hold the last timed step's results until the next step runs
    outputs = {"loss_result": res, "kept": hp.det["kept"].to_host(), "count": hp.det["count"].to_host()} \
        if args.dump_outputs else None
    clocks = sampler.summary(t0, t1, t_load0, time.perf_counter())
    # the same steps as closed units (each joined before the next starts): the latency of one step
    depth, closed_ms = hp.depth, ms_step
    if depth > 1 and not args.no_detail:
        hp.depth = 1
        closed_ms, _ = timed_steps(R, hp, args.steps, args.warmup, n_sets=n_sets)
        hp.depth = depth

    # ---- sustained: >= sustained_seconds of steps over the resident batches, clocks sampled inside the window -----
    sustained = None
    if not args.no_detail and args.sustained_seconds > 0:
        chunk = 25
        n_chunks = max(4, int(args.sustained_seconds * 1e3 / (ms_step * chunk)) + 1)
        evs = [D.Event() for _ in range(n_chunks + 1)]
        R.barrier()
        ts0 = time.perf_counter()
        evs[0].record(hp.s_main)
        k = 0
        for ci in range(n_chunks):
            for _ in range(chunk):
                hp.use_set(k % n_sets)
                hp.step()
                k += 1
            hp.join()
            evs[ci + 1].record(hp.s_main)
        hp.finish_exchange()
        hp.s_main.sync()
        R.barrier()
        ts1 = time.perf_counter()
        per = [evs[i].elapsed_ms(evs[i + 1]) / chunk for i in range(n_chunks)]
        tot_ms = R.max(evs[0].elapsed_ms(evs[n_chunks]))
        sustained = {"seconds": tot_ms * 1e-3, "steps": n_chunks * chunk, "resident_batches": n_sets,
                     "value": b * world * n_chunks * chunk / (tot_ms * 1e-3), "unit": "images/s",
                     "ms_per_step_mean": tot_ms / (n_chunks * chunk), "ms_per_step_median_of_chunks": statistics.median(per),
                     "ms_per_step_min_of_chunks": min(per), "ms_per_step_max_of_chunks": max(per), "chunk_steps": chunk,
                     "clocks": sampler.summary(ts0, ts1), "vs_value": None}
        sustained["vs_value"] = sustained["value"] / value
    hp.use_set(0)

    # ---- per-stage serial timing + dominant-kernel durations (CUDA events on the launch stream) ---------
    N.lib().ssdg_profile_enable(1)
    import ctypes as C
    stages = {}
    kernel_ms = {}

    def time_stage(name, fn, prof_ids):
        for _ in range(3):
            fn(hp.s_main)
        hp.s_main.sync()
        tot, ksum = 0.0, {k: 0.0 for k in prof_ids}
        a0, a1 = D.Event(), D.Event()
        for _ in range(args.steps):
            a0.record(hp.s_main)
            fn(hp.s_main)
            a1.record(hp.s_main)
            tot += a0.elapsed_ms(a1)
            for k in prof_ids:
                ms = C.c_float(0)
                N.lib().ssdg_profile_last_ms(k, C.byref(ms))
                ksum[k] += ms.value
        stages[name] = tot / args.steps
        for k in prof_ids:
            kernel_ms[k] = ksum[k] / args.steps

    time_stage("assign_ms", hp.assign, [N.PROF_MATCH, N.PROF_SEARCH])
    # work counter of the matcher: 32-prior tiles evaluated exactly by the search kernel in the last call
    head = hp._match_out["_match_ws"].view((8,), np.uint32).to_host(hp.s_main)
    tiles_evaluated = int(head[3])
    time_stage("loss_ms", hp.loss_stage, [N.PROF_CE, N.PROF_LOSS_TAIL])
    time_stage("detect_ms", hp.detect_stage, [N.PROF_FILTER, N.PROF_NMS])
    ce_alone_ms, filter_alone_ms = kernel_ms.get(N.PROF_CE, 0.0), kernel_ms.get(N.PROF_FILTER, 0.0)
    if hp.fused:   # the variants the chained step actually launches
        time_stage("detect_with_row_stats_ms", lambda s: hp.detect_stage(s, stats=True), [N.PROF_FILTER, N.PROF_NMS])
        time_stage("loss_from_row_stats_ms", lambda s: hp.loss_stage(s, stats=True), [N.PROF_CE, N.PROF_LOSS_TAIL])
    grad_ms = None
    if not args.no_detail and world == 1:
        # the backward of the loss (SURVEY 8f row 1): d total / d logits is one more logits-sized write
        from ssdgeom import ops
        gout = {"result": D.empty((N.LOSS_RESULT_LEN,), np.float64), "grad_box": D.empty((b, a, 4), np.float32),
                "grad_cls": D.empty((b, a, c), np.float32)}

        def loss_with_grad(s):
            ops.multibox_loss(hp.tgt["cls"], hp.tgt["loc"], hp.tgt["mask"], hp.pred_box, hp.pred_cls, hp.neg_ratio,
                              want_grad=True, out=gout, stream=s, pool=hp.pool)
        time_stage("loss_with_grad_ms", loss_with_grad, [N.PROF_GRAD])
        grad_ms = kernel_ms.get(N.PROF_GRAD)
        del gout
    N.lib().ssdg_profile_enable(0)

    # ---- end to end through the host API -------------------------------------------------------------------
    e2e = None
    if not args.no_e2e:
        pipelined = args.mining == "shard"   # double-buffered inputs: the H2D of step k+1 runs under step k
        def e2e_step():
            if pipelined:
                hp.submit(host_in, host_out)
            else:
                hp.step_host(*host_in, *host_out)
        for _ in range(2):
            e2e_step()
        hp.drain()
        R.barrier()
        e0, e1 = D.Event(), D.Event()
        e0.record(hp.s_main)
        if pipelined:
            D.stream_wait_event(hp.s_copy, e0)   # the first timed copy starts inside the timed region
        for _ in range(args.steps):
            e2e_step()
        e1.record(hp.s_main)
        hp.drain()
        R.barrier()
        e_ms = R.max(e0.elapsed_ms(e1))
        # the ceiling of this path: the bare pinned host -> device copy of one step's inputs, all ranks at once
        R.barrier()
        c0, c1 = D.Event(), D.Event()
        c0.record(hp.s_main)
        n_copy = 5
        for _ in range(n_copy):
            hp.upload(*host_in)
        c1.record(hp.s_main)
        hp.s_main.sync()
        R.barrier()
        c_ms = R.max(c0.elapsed_ms(c1)) / n_copy
        ceiling_gbs = hp.h2d_bytes / (c_ms * 1e-3) / 1e9
        ceiling_ips = b * world / (c_ms * 1e-3)
        e_val = b * world * args.steps / (e_ms * 1e-3)
        e2e = {"value": e_val, "unit": "images/s", "h2d_bytes_per_step": hp.h2d_bytes,
               "d2h_bytes_per_step": hp.d2h_bytes, "ms_per_step": e_ms / args.steps,
               "mode": "HotPath.submit: double-buffered inputs, H2D of step k+1 under compute + D2H of step k" if pipelined
               else "HotPath.step_host: serial H2D, compute, D2H",
               "h2d_ceiling_gbs_per_gpu": ceiling_gbs, "h2d_ceiling_images_per_s": ceiling_ips,
               "frac_of_h2d_ceiling": e_val / ceiling_ips,
               "h2d_ceiling_how": "bare cudaMemcpyAsync of one step's inputs from the same pinned buffers, all %d ranks "
                                  "concurrently, max over ranks" % world}
    return dict(a=a, c=c, ms_step=ms_step, value=value, res=res, clocks=clocks, sustained=sustained, stages=stages,
                depth=depth, closed_ms=closed_ms,
                kernel_ms=kernel_ms, tiles_evaluated=tiles_evaluated, ce_alone_ms=ce_alone_ms,
                filter_alone_ms=filter_alone_ms, grad_ms=grad_ms, e2e=e2e, launches=hp.kernel_launches_per_step,
                memsets=hp.memsets_per_step, fused=bool(hp.fused), logits_mb=hp.pred_cls.nbytes / 1e6,
                gt_rows=float(np.diff(off).sum()), outputs=outputs)


def report(args, R, comm, b, M, detail_cfg):
    from ssdgeom import _native as N
    world = R.world
    a, c, ms_step, value, res, clocks = M["a"], M["c"], M["ms_step"], M["value"], M["res"], M["clocks"]
    sustained, stages, kernel_ms, tiles_evaluated = M["sustained"], M["stages"], M["kernel_ms"], M["tiles_evaluated"]
    ce_alone_ms, filter_alone_ms, grad_ms, e2e = M["ce_alone_ms"], M["filter_alone_ms"], M["grad_ms"], M["e2e"]
    launches, memsets, fused, logits_mb, gt_rows = M["launches"], M["memsets"], M["fused"], M["logits_mb"], M["gt_rows"]
    # ---- roofline of the dominant kernel (the step's one pass over the logits) -------------------------------
    pk = peaks()
    peak = float(pk.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in pk else "fallback"

    def traffic_of(name):   # dram__bytes_read.sum + dram__bytes_write.sum of one launch (ncu --set full), same shape only
        cap = profile_json(name)
        if cap and cap.get("batch") == b and cap.get("priors") == a and cap.get("classes") == c:
            return cap["dram_bytes_per_launch"]
        return None

    if fused:
        # the one pass over the logits: in logits + pred_box, out decoded boxes (16 B) + row statistics (12 B) per prior
        k_name, k_ms = "filter_kernel (softmax filter + decode + loss row statistics)", kernel_ms.get(N.PROF_FILTER, 0.0)
        k_bytes = b * a * (c * 4 + 16 + 16 + 12)
        traffic = traffic_of("filter_kernel_traffic.json")
    else:
        k_name, k_ms = "ce_kernel", ce_alone_ms
        k_bytes = b * a * (c * 4 + 16 + 16 + 4 + 1)            # logits + pred_box + gt_box + gt_cls + mask
        traffic = traffic_of("ce_kernel_traffic.json")
    achieved = k_bytes / (k_ms * 1e-3) / 1e9 if k_ms > 0 else 0.0
    roof = {"bound": "hbm", "kernel": k_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src, "kernel_ms": k_ms,
            "algorithmic_bytes_per_launch": k_bytes,
            "frac_input_bytes_only": (b * a * (c * 4 + 16) / (k_ms * 1e-3) / 1e9 / peak) if k_ms > 0 else None}
    ce_ms = ce_alone_ms
    f_ms = filter_alone_ms
    m_ms = kernel_ms.get(N.PROF_MATCH) or 0.0
    mcap = profile_json("matcher_ncu.json") or {}
    matcher = {"candidate_pairs_per_s": gt_rows * a / (m_ms * 1e-3) if m_ms else None,
               "evaluated_pairs_per_s": tiles_evaluated * 32 / (m_ms * 1e-3) if m_ms else None,
               "evaluated_fraction": tiles_evaluated * 32 / (gt_rows * a) if gt_rows else None,
               "search_kernel_ms": kernel_ms.get(N.PROF_SEARCH), "search_plus_match_ms": m_ms,
               "algorithmic_bytes_per_launch": b * (2000 + a * (4 + 16 + 1)) + a * 32,
               "hbm_frac": (b * (2000 + a * (4 + 16 + 1)) + a * 32) / (m_ms * 1e-3) / 1e9 / peak if m_ms else None,
               "fp64_pipe_pct_of_peak": mcap.get("fp64_pipe_pct_of_peak"), "ncu_source": mcap.get("source"),
               "bound": "memory latency / instruction issue (fp64 pipe <= 11 % of its peak, DRAM < 4 %): see profiles/"}
    extra = {"stages_ms": stages, "fused_logits_pass": fused,
             "ce_kernel_gbs_standalone": b * a * (c * 4 + 16 + 16 + 4 + 1) / (ce_ms * 1e-3) / 1e9 if ce_ms > 0 else None,
             "kernels_ms": {"match_kernel": m_ms, "search_kernel": kernel_ms.get(N.PROF_SEARCH), "ce_kernel": ce_ms,
                            "filter_kernel": f_ms, "nms_kernel": kernel_ms.get(N.PROF_NMS),
                            "bucket_kernel": None,   # gone: the filter appends straight to the class lists
                            "loss_tail": kernel_ms.get(N.PROF_LOSS_TAIL),
                            "filter_kernel_with_row_stats": kernel_ms.get(N.PROF_FILTER) if fused else None,
                            "lossprep_kernel": kernel_ms.get(N.PROF_CE) if fused else None,
                            "grad_kernel": grad_ms},
             "grad_kernel_gbs": (b * a * (c * 4 * 2 + 16 * 3 + 4 + 1 + 4) / (grad_ms * 1e-3) / 1e9) if grad_ms else None,
             "filter_kernel_gbs": b * a * (c * 4 + 16) / (f_ms * 1e-3) / 1e9 if f_ms > 0 else None,
             "match_pairs_per_s": matcher["candidate_pairs_per_s"],
             "matcher_roofline": matcher,
             "steps_in_flight": {"depth": M["depth"],
                                 "how": "consecutive steps use alternate sets of every per-step buffer (targets, row "
                                        "statistics, candidate lists, workspaces, results), so a step's filter pass and row "
                                        "search run under the NMS and loss tail of the step before; all K steps complete "
                                        "inside the timed region",
                                 "closed_step_ms": M["closed_ms"],
                                 "closed_step_value": b * R.world * 1e3 / M["closed_ms"] if M["closed_ms"] else None},
             "chain_bytes_per_image": chain_bytes_per_image(a, c, fused),
             "chain_hbm_roofline_frac": chain_bytes_per_image(a, c, fused) * b / (ms_step * 1e-3) / 1e9 / peak,
             "sustained": sustained,
             "exchange": ("ssdg_comm (libssdgeom NCCL entry points)" if comm is not None else "torch.distributed") if world > 1 else None,
             "loss": ({"total": res[0], "num_pos": res[4], "num_neg": res[5], "status": res[7],
                       "scope": "this rank" if world == 1 else "total: this rank's shard; num_pos / num_neg: pooled over the ranks by the exchange"}
                      if args.mining == "shard" or world == 1 else
                      {"total": (res[8] + res[10]) / res[11] + res[9] / res[5], "num_pos": res[11], "num_neg": res[5],
                       "status": res[7], "scope": "all ranks (exact-global mining)"})}
    extra.update(detail_cfg)

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        arm = CpuArm(args, args.cpu_images)
        arm.step(record=False)                       # warm the pool
        for _ in range(2):
            arm.step()
        arm.close()
        cpu = arm.describe()

    line = base_line(args, value, ms_step, world, b)
    line["config"]["priors"] = a
    line["config"]["steps_in_flight"] = M["depth"]
    line["config"]["l2"] = "inputs larger than L2 (logits %.0f MB per GPU, two resident batches in rotation)" % logits_mb
    line.update({"clocks": clocks, "e2e": e2e, "gpu_launches": launches * args.steps,
                 "gpu_memsets": memsets * args.steps,
                 "roofline": roof, "cpu_baseline": cpu, "detail": extra, "impl": "ours"})
    return line


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
