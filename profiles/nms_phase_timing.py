"""Where nms_kernel's cycles go: per-phase clocks and the counts each phase scales with, on bench.py's workload (SSD300,
B=256, 80 class lists per image, score > 0.01, top_k 200, IoU 0.45).  Builds the library variant "nms_timing" with
-DSSDG_NMS_TIMING (detect.cu, NmsTiming) and runs the post-processing on it; the default build is not touched.
usage: python profiles/nms_phase_timing.py [repeats]
Phase clocks are read by thread 0 of each CTA at the barrier that ends the phase: they are the wall cycles of a list
while 11 other lists share its SM, not issue cycles.  The join passes A and B have no barrier between them and are
clocked per warp (cycles summed over the warps of a list)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np

root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [root, os.path.join(root, "ssd-object-detection_b200")]
os.environ["SSDG_EXTRA_NVCC_FLAGS"] = (os.environ.get("SSDG_EXTRA_NVCC_FLAGS", "") + " -DSSDG_NMS_TIMING").strip()
import build_native  # noqa: E402

os.environ["SSDGEOM_LIB"] = build_native.build(variant="nms_timing")
from ssdgeom import _native as N, device as D, ops, synth  # noqa: E402

PHASES = ["key load + histogram", "select / single-bucket rebuild", "scan + scatter", "rank + box + registration",
          "running OR", "join (passes A + B)", "resolution", "output"]
COUNTS = ["lists", "keys", "lists through the select", "rows (top_k of the list)", "count-loop steps (threads)",
          "count-loop trips (warps)", "pass-A words (per row group)", "pass-B candidate pairs", "pass-B trips (warps)",
          "pass-B (row, word)s with candidates", "suppressing pairs", "open rows", "resolution rounds"]
RANK_PARTS = ["  rank: key + count loop", "  rank: box + preparation + registration"]
NT_SLOTS = 32

repeats = int(sys.argv[1]) if len(sys.argv) > 1 else 5
b = 256
table = synth.TABLES["ssd300"]
pri = ops.prior_boxes(table["sizes"], table["s_k_refer"], table["aspect_ratio"], table["input_size"])
a = synth.num_priors(table)
pred_cls = np.empty((b, a, 81), np.float32)
pred_box = np.empty((b, a, 4), np.float32)
for i in range(0, b, 16):   # bench.py's headline batch (rank 0, drawn in chunks of 16 images)
    pred_cls[i:i + 16], pred_box[i:i + 16] = synth.make_predictions(i, 16, a, 81)
pc, pb = D.as_device(pred_cls), D.as_device(pred_box)
fn = N.lib().ssdg_nms_timing
fn.argtypes = [C.POINTER(C.c_ulonglong), C.c_int32]
buf = (C.c_ulonglong * NT_SLOTS)()
ops.detect(pc, pb, pri, 0.01, 200, 0.45, want_scores=True)   # warm-up
D.sync()
N.check(fn(buf, NT_SLOTS), "nms_timing")
for _ in range(repeats):
    ops.detect(pc, pb, pri, 0.01, 200, 0.45, want_scores=True)
D.sync()
N.check(fn(buf, NT_SLOTS), "nms_timing")
t = np.array(buf[:], np.float64)

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
print("GPU: %s" % (gpu[0] if gpu else "unknown"))
lists = t[10]
print("nms_kernel phase attribution, SSD300 B=%d, %d launches, %.0f lists" % (b, repeats, lists))
tot = t[:8].sum()
print("%-34s %12s %8s" % ("phase (CTA wall cycles)", "per list", "share"))
for k, name in enumerate(PHASES):
    print("%-34s %12.0f %7.1f%%" % (name, t[k] / lists, 100 * t[k] / tot))
print("%-34s %12.0f" % ("all phases", tot / lists))
print("%-34s %12.0f   (warp cycles, summed over the 4 warps)" % ("  join pass A", t[8] / lists))
print("%-34s %12.0f   (warp cycles, summed over the 4 warps)" % ("  join pass B", t[9] / lists))
for k, name in enumerate(RANK_PARTS):
    print("%-34s %12.0f   (warp cycles, summed over the 4 warps)" % (name, t[23 + k] / lists))
print("%-34s %12s" % ("count", "per list"))
for k, name in enumerate(COUNTS):
    print("%-34s %12.2f" % (name, t[10 + k] / lists))
