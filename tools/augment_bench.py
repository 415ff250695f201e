"""Cost of the SSD training augmentation (ops.augment) on one GPU; prints one JSON line (and writes it to --out).

    python tools/augment_bench.py [--batch 256] [--size 300] [--launches 200] [--host-images 512] [--out FILE]

  boxes_ms    ssdg_augment_boxes (sampling + scan + compaction), CUDA events around --launches launches after warm-up
  images_ms   ssdg_augment_images alone, the same way; bytes model: B*H*W*12 written + at most as much read (every
              source pixel is fetched through L2, neighbouring output pixels share their taps)
  augment_ms  the whole ops.augment call from device inputs (both entry points and the host wrapper)
  copy        a device-to-device copy of the same image bytes (torch copy_), timed the same way: the copy peak that
              images_bytes_per_s is divided by
  host        torchvision v2 RandomZoomOut -> RandomIoUCrop -> RandomHorizontalFlip -> Resize per image on all host cores
              (a process pool, one torch thread each), in images/s; images without ground truth are skipped there (the
              crop never terminates on them).  Absent when torchvision is not importable.
Workload: SSD300-sized images, B = 256, 300 x 300 x 3 float32, synthetic ground truth with T = 100 in "coco" mode, the
default recipe.  The batch's images (276 MB) exceed the 126 MB L2.  The card's name and power limit are read in the same
run."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "ssd-object-detection_b200")):
    sys.path.insert(0, p)

from ssdgeom import _native as N, device as D, ops, synth   # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def timed(fn, n, stream):
    fn()
    a, b = D.Event(), D.Event()
    for _ in range(10):
        fn()
    a.record(stream)
    for _ in range(n):
        fn()
    b.record(stream)
    return a.elapsed_ms(b) / n


_HOST = {}


def _host_init(h, w):
    import torch
    from torchvision.transforms import v2
    torch.set_num_threads(1)
    fill = tuple(float(v) for v in ops.AUGMENT_DEFAULTS["fill"])
    _HOST["t"] = v2.Compose([v2.RandomZoomOut(fill=fill, side_range=(1.0, 4.0), p=0.5), v2.RandomIoUCrop(),
                             v2.RandomHorizontalFlip(0.5), v2.Resize((h, w), antialias=False)])


def _host_one(item):
    import torch
    from torchvision import tv_tensors
    img, boxes = item
    h, w = img.shape[:2]
    x = tv_tensors.Image(torch.from_numpy(img).permute(2, 0, 1))
    b = torch.from_numpy(boxes) * torch.tensor([w, h, w, h], dtype=torch.float32)
    bb = tv_tensors.BoundingBoxes(b, format="CXCYWH", canvas_size=(h, w))
    out = _HOST["t"](x, bb)
    return int(out[1].shape[0])


def host_arm(images, boxes, off, n_images):
    try:
        import torchvision  # noqa: F401
    except Exception:
        return None
    from multiprocessing import get_context
    b = images.shape[0]
    items = [(images[i % b], boxes[off[i % b]:off[i % b + 1]]) for i in range(n_images) if off[i % b + 1] > off[i % b]]
    procs = os.cpu_count() or 1
    with get_context("spawn").Pool(procs, initializer=_host_init, initargs=images.shape[1:3]) as pool:
        pool.map(_host_one, items[:procs * 2])           # warm-up: imports in every worker
        t0 = time.perf_counter()
        pool.map(_host_one, items, chunksize=4)
        dt = time.perf_counter() - t0
    return {"processes": procs, "images": len(items), "seconds": dt, "images_per_s": len(items) / dt}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--size", type=int, default=300)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--host-images", type=int, default=512)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if N.device_count() < 1:
        raise SystemExit("augment_bench: no CUDA device")
    import torch
    b, h, w, max_t = args.batch, args.size, args.size, 100
    rec = {"card": card(), "batch": b, "height": h, "width": w, "max_t": max_t, "gt_mode": "coco",
           "config": {k: list(v) if isinstance(v, tuple) else v for k, v in ops.AUGMENT_DEFAULTS.items()}}
    st = D.Stream()
    boxes, cls, off = synth.make_gt(1234, b, max_t, "coco")
    images = np.random.default_rng(1234).random((b, h, w, 3), dtype=np.float32)
    d_img, d_boxes, d_cls = D.to_device(images), D.to_device(boxes), D.to_device(cls)
    d_off = D.to_device(off)
    max_gt = int(np.diff(off).max())
    out = ops.augment(d_img, d_boxes, d_cls, d_off, 7, max_gt=max_gt, stream=st)
    tr = out["transform"].to_host(st)
    rec["rows_in"], rec["rows_out"] = int(off[-1]), int(out["offsets"].to_host(st)[-1])
    rec["records"] = {"zoomed": int((tr[:, 0] > w).sum()), "cropped": int((tr[:, 6] < tr[:, 0]).sum()),
                      "flipped": int(tr[:, 8].sum()), "round_cap": int((tr[:, 9] == -1).sum()),
                      "rounds_mean": float(tr[tr[:, 9] > 0, 9].mean())}

    cfg = ops.AUGMENT_DEFAULTS
    opts = np.ascontiguousarray(cfg["min_ious"], np.float64)
    lib, sh = N.lib(), D.stream_handle(st)
    import ctypes as C
    bargs = (d_boxes.ptr, d_cls.ptr, d_off.ptr, b, max_gt, h, w, 7, 0, cfg["zoom_p"], cfg["side_range"][0],
             cfg["side_range"][1], opts.ctypes.data_as(C.POINTER(C.c_double)), opts.size, cfg["min_scale"],
             cfg["max_scale"], cfg["min_aspect"], cfg["max_aspect"], cfg["trials"], cfg["max_rounds"], cfg["flip_p"],
             out["boxes"].ptr, out["cls"].ptr, out["offsets"].ptr, out["src_row"].ptr, out["transform"].ptr, sh)
    fill = (C.c_float * 3)(*cfg["fill"])
    iargs = (d_img.ptr, out["transform"].ptr, b, h, w, fill, out["images"].ptr, sh)
    rec["boxes_ms"] = timed(lambda: N.check(lib.ssdg_augment_boxes(*bargs), "augment_boxes"), args.launches, st)
    rec["images_ms"] = timed(lambda: N.check(lib.ssdg_augment_images(*iargs), "augment_images"), args.launches, st)
    rec["augment_ms"] = timed(lambda: ops.augment(d_img, d_boxes, d_cls, d_off, 7, max_gt=max_gt, stream=st, out=out),
                              args.launches, st)
    # the copy peak: a device-to-device copy of the same bytes, on the same stream
    src = torch.as_tensor(d_img, device="cuda")
    dst = torch.empty_like(src)
    ts = torch.cuda.ExternalStream(sh)
    with torch.cuda.stream(ts):
        rec["copy_ms"] = timed(lambda: dst.copy_(src), args.launches, st)
    nbytes = b * h * w * 12
    rec["images_bytes_model"] = 2 * nbytes
    rec["images_bytes_per_s"] = 2 * nbytes / (rec["images_ms"] * 1e-3)
    rec["copy_bytes_per_s"] = 2 * nbytes / (rec["copy_ms"] * 1e-3)
    rec["images_of_copy_peak"] = rec["images_bytes_per_s"] / rec["copy_bytes_per_s"]
    rec["device_images_per_s"] = b / (rec["augment_ms"] * 1e-3)
    rec["host"] = host_arm(images, boxes, off, args.host_images)
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
