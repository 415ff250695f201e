"""Cost of the detection evaluation on one GPU; prints one JSON line (and writes it to --out).

    python tools/eval_bench.py [--batch 256] [--launches 200] [--steps 200] [--rounds 4] [--out FILE]

  accumulate_ms      ssdg_eval_accumulate alone (CUDA events around --launches launches) at SSD300, C=81, top_k 200,
                     max_dets 100, on the kept lists of ops.detect for the default synthetic predictions (the ones
                     bench.py times) and for trained-like ones (synth.make_trained_predictions: AP is meaningful)
  step_ms            the depth-2 HotPath step (bench.py's chained step, inputs of bench.py) without and with an
                     evaluator, alternated in --rounds rounds of --steps steps in the same process
  finalize_ms        ssdg_eval_finalize over a 5 000-image state filled with trained-like batches
  oracle_host_ms     the NumPy restatement (tests/coco_eval_oracle.py) for ONE batch, for scale
The card's name and power limit are read in the same run."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "ssd-object-detection_b200"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)

from ssdgeom import _native as N, device as D, ops, synth   # noqa: E402
from ssdgeom.evaluate import DetectionEvaluator      # noqa: E402
from ssdgeom.models import ssd_model as M            # noqa: E402
from ssdgeom.pipeline import HotPath                 # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def timed(fn, n, stream):
    a, b = D.Event(), D.Event()
    a.record(stream)
    for _ in range(n):
        fn()
    b.record(stream)
    return a.elapsed_ms(b) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--images", type=int, default=5000)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    b, max_gt = args.batch, 100
    rec = {"card": card(), "batch": b, "classes": 81, "top_k": 200, "max_dets": 100, "table": "ssd300"}
    priors = M.build_prior_box(synth.SSD300["sizes"])
    a = priors.shape[0]
    st = D.Stream()

    # inputs of bench.py (seed 1234, T = 100 per image) and trained-like predictions from their targets
    gt, gcls, off = synth.make_gt(1234, b, max_gt, "max")
    pc_default, pb_default = synth.make_predictions(1234, b, a)
    t = ops.match_encode(gt, gcls, off, priors, b, max_gt, 0.5)
    pc_trained, pb_trained = synth.make_trained_predictions(1234, t["cls"].to_host(), t["loc"].to_host(),
                                                            t["mask"].to_host())
    acc = {}
    for name, pc, pb in (("default", pc_default, pb_default), ("trained", pc_trained, pb_trained)):
        det = ops.detect(pc, pb, priors, want_scores=True, want_boxes=True, stream=st)
        ev = DetectionEvaluator(max_images=b, max_gt=max_gt)
        g = (D.to_device(gt), D.to_device(gcls), D.to_device(off))
        ev.add(det, *g, image_base=0, stream=st)
        # the raw entry point with prepared arguments, so that the launches queue up ahead of the device
        thr = ev.iou_thresholds
        cargs = (det["kept"].ptr, det["count"].ptr, det["kept_score"].ptr, 200, det["boxes"].ptr, b, a, 81, g[0].ptr,
                 g[1].ptr, g[2].ptr, max_gt, thr.ctypes.data_as(C.POINTER(C.c_double)), thr.size, 100, 0, b,
                 ev.state.ptr, ev.state.nbytes, D.stream_handle(st))
        fn = N.lib().ssdg_eval_accumulate
        call = lambda: fn(*cargs)
        timed(call, 10, st)
        acc[name] = timed(call, args.launches, st)
        acc[name + "_detections"] = int(det["count"].to_host().clip(max=100).sum())
        acc[name + "_AP"] = ev.summarize(st)["AP"]
    rec["accumulate_ms"] = acc

    # the chained depth-2 step without / with the evaluator, alternated
    hps = {}
    for name, ev in (("without", None), ("with", DetectionEvaluator(max_images=b, max_gt=max_gt))):
        hp = HotPath(synth.SSD300, batch=b, max_gt=max_gt, total_gt=gt.shape[0], depth=2, evaluator=ev)
        hp.upload(gt, gcls, off, pc_default, pb_default)
        hp.s_main.sync()
        hps[name] = hp

    def run(hp, n):
        ev0, ev1 = D.Event(), D.Event()
        ev0.record(hp.s_main)
        for _ in range(n):
            hp.step(image_base=0) if hp.evaluator is not None else hp.step()
        hp.join()
        ev1.record(hp.s_main)
        return ev0.elapsed_ms(ev1) / n

    for hp in hps.values():
        run(hp, 20)
    per = {k: [] for k in hps}
    for _ in range(args.rounds):
        for k, hp in hps.items():
            per[k].append(run(hp, args.steps))
    rec["step_ms"] = {k: {"median": float(np.median(v)), "all": v} for k, v in per.items()}
    rec["step_overhead_pct"] = 100.0 * (rec["step_ms"]["with"]["median"] / rec["step_ms"]["without"]["median"] - 1.0)
    del hps

    # finalize over a state of --images images (trained-like batches, the last one partial)
    ev = DetectionEvaluator(max_images=args.images, max_gt=max_gt)
    det = ops.detect(pc_trained, pb_trained, priors, want_scores=True, want_boxes=True, stream=st)
    g = (D.to_device(gt), D.to_device(gcls), D.to_device(off))
    base = 0
    while base + b <= args.images:
        ev.add(det, *g, image_base=base, stream=st)
        base += b
    if base < args.images:
        n = args.images - base
        part = ops.detect(pc_trained[:n], pb_trained[:n], priors, want_scores=True, want_boxes=True, stream=st)
        ev.add(part, gt[:off[n]], gcls[:off[n]], off[:n + 1], image_base=base, stream=st)
    fin = lambda: ops.eval_finalize(ev.state, ev.recall_thresholds, st, ev.pool)
    keep = fin()                        # warm-up; each timed call below is bracketed on its own (its outputs are
    rec["finalize_ms"] = float(np.median([timed(fin, 1, st) for _ in range(5)]))   # allocated and freed per call)
    del keep
    rec["finalize_images"] = args.images
    rec["finalize_state_mb"] = ev.state.nbytes / 1e6
    res = ev.summarize(st)
    rec["finalize_AP"], rec["finalize_detections"] = res["AP"], int(res["n_det"].sum())

    # the host restatement for one batch of the same evaluation
    import coco_eval_oracle as E
    host = {k: det[k].to_host() for k in ("kept", "count", "kept_score", "boxes")}
    t0 = time.perf_counter()
    r = E.evaluate_batch(host["kept"], host["count"], host["kept_score"], host["boxes"], gt, gcls, off, 0)
    E.coco_accumulate(*r, 81)
    rec["oracle_host_ms"] = {"images": b, "ms": 1e3 * (time.perf_counter() - t0)}
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
