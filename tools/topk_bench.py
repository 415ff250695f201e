"""Cost of the per-image keep_top_k on one GPU; prints one JSON line (and writes it to --out).

    python tools/topk_bench.py [--batch 256] [--launches 200] [--steps 200] [--rounds 5] [--out FILE]

  kernel_ms   ssdg_detect_keep_top_k alone (CUDA events around --launches launches, after warm-up) at SSD300, C=81,
              top_k 200, K = 100 and 200, on the kept lists of ops.detect for the default synthetic predictions (the
              ones bench.py times) and for trained-like ones (synth.make_trained_predictions), with the mean and
              maximum candidates per image.  The larger batch (4 x --batch) repeats the --batch images' lists 4 times:
              the work per image is the same, only the host-side generation of the predictions is saved.
  step_ms     the depth-2 HotPath step (bench.py's chained step, inputs of bench.py) without and with
              keep_top_k=200, alternated in --rounds rounds of --steps steps in the same process: median and spread
The card's name and power limit are read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "ssd-object-detection_b200")):
    sys.path.insert(0, p)

from ssdgeom import _native as N, device as D, ops, synth   # noqa: E402
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
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if N.device_count() < 1:
        raise SystemExit("topk_bench: no CUDA device")
    b, max_gt, top_k = args.batch, 100, 200
    rec = {"card": card(), "batch": b, "classes": 81, "top_k": top_k, "table": "ssd300"}
    priors = M.build_prior_box(synth.SSD300["sizes"])
    a = priors.shape[0]
    st = D.Stream()

    # inputs of bench.py (seed 1234, T = 100 per image) and trained-like predictions from their targets
    gt, gcls, off = synth.make_gt(1234, b, max_gt, "max")
    pc_default, pb_default = synth.make_predictions(1234, b, a)
    t = ops.match_encode(gt, gcls, off, priors, b, max_gt, 0.5)
    pc_trained, pb_trained = synth.make_trained_predictions(1234, t["cls"].to_host(), t["loc"].to_host(),
                                                            t["mask"].to_host())
    kern = {}
    for name, pc, pb in (("default", pc_default, pb_default), ("trained", pc_trained, pb_trained)):
        det = ops.detect(pc, pb, priors, want_scores=True, want_boxes=True, stream=st)
        host = {k: det[k].to_host(st) for k in ("kept", "count", "kept_score", "boxes")}
        cand = np.clip(host["count"], 0, top_k).sum(axis=1)
        kern[name] = {"candidates_per_image_mean": float(cand.mean()), "candidates_per_image_max": int(cand.max())}
        for reps in (1, 4):
            d = {k: D.to_device(np.concatenate([v] * reps)) for k, v in host.items()}
            bb = b * reps
            for K in (100, 200):
                top = ops.keep_top_k(d, K, stream=st)
                # the raw entry point with prepared arguments, so that the launches queue up ahead of the device
                cargs = (d["kept"].ptr, d["count"].ptr, d["kept_score"].ptr, top_k, d["boxes"].ptr, bb, a, 81, K,
                         top["prior"].ptr, top["class"].ptr, top["score"].ptr, top["box"].ptr, top["n"].ptr,
                         top["count"].ptr, D.stream_handle(st))
                fn = N.lib().ssdg_detect_keep_top_k
                call = lambda: N.check(fn(*cargs), "keep_top_k")
                timed(call, 20, st)
                kern[name]["B%d_K%d" % (bb, K)] = timed(call, args.launches, st)
    rec["kernel_ms"] = kern

    # the chained depth-2 step without / with keep_top_k=200, alternated
    hps = {}
    for name, keep in (("without", None), ("with", 200)):
        hp = HotPath(synth.SSD300, batch=b, max_gt=max_gt, total_gt=gt.shape[0], depth=2, keep_top_k=keep)
        hp.upload(gt, gcls, off, pc_default, pb_default)
        hp.s_main.sync()
        hps[name] = hp

    def run(hp, n):
        ev0, ev1 = D.Event(), D.Event()
        ev0.record(hp.s_main)
        for _ in range(n):
            hp.step()
        hp.join()
        ev1.record(hp.s_main)
        return ev0.elapsed_ms(ev1) / n

    for hp in hps.values():
        run(hp, 20)
    per = {k: [] for k in hps}
    for _ in range(args.rounds):
        for k, hp in hps.items():
            per[k].append(run(hp, args.steps))
    rec["step_ms"] = {k: {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v)), "all": v}
                      for k, v in per.items()}
    rec["step_overhead_pct"] = 100.0 * (rec["step_ms"]["with"]["median"] / rec["step_ms"]["without"]["median"] - 1.0)
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
