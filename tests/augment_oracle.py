"""NumPy restatement of the SSD training augmentation spec (include/ssdgeom.h, A13): Philox4x32-10, torchvision's
RandomZoomOut -> RandomIoUCrop -> RandomHorizontalFlip as a sequential per-image loop, the box transform and a float64
bilinear resample, so that the device results can be compared bit for bit (images within rounding).  The checker
only: product code never imports it."""
from __future__ import annotations

import numpy as np

MASK = 0xFFFFFFFF
DEFAULTS = dict(zoom_p=0.5, side_range=(1.0, 4.0), min_ious=(0.0, 0.1, 0.3, 0.5, 0.7, 0.9, 1.0), min_scale=0.3,
                max_scale=1.0, min_aspect=0.5, max_aspect=2.0, trials=40, max_rounds=50, flip_p=0.5,
                fill=(123 / 255, 117 / 255, 104 / 255))
RECORD = ("canvas_w", "canvas_h", "pad_left", "pad_top", "left", "top", "width", "height", "flip", "rounds")
f32 = np.float32


def philox4x32(ctr, key):
    """Philox4x32-10 of four 32-bit counter words and a 64-bit key (Random123)."""
    c = [int(v) & MASK for v in ctr]
    k0, k1 = key & MASK, (key >> 32) & MASK
    for _ in range(10):
        p0, p1 = 0xD2511F53 * c[0], 0xCD9E8D57 * c[2]
        c = [((p1 >> 32) ^ c[1] ^ k0) & MASK, p1 & MASK, ((p0 >> 32) ^ c[3] ^ k1) & MASK, p0 & MASK]
        k0, k1 = (k0 + 0x9E3779B9) & MASK, (k1 + 0xBB67AE85) & MASK
    return c


def draw(seed, g, stream, index):
    return philox4x32((g & MASK, (g >> 32) & MASK, stream, index), seed & (2**64 - 1))


def unif(x):
    """u = (x >> 8) * 2^-24, float32 in [0, 1)."""
    return f32(x >> 8) * f32(2.0 ** -24)


def option_index(x, n):
    return (x * n) >> 32


class Uniforms:
    """Every draw of one image at its fixed address, in the terms torchvision's make_params consumes them."""

    def __init__(self, seed, g):
        self.seed, self.g = seed, g

    def zoom(self):            # gate, r, left, top
        return [unif(x) for x in draw(self.seed, self.g, 0, 0)]

    def flip(self):
        return unif(draw(self.seed, self.g, 0, 1)[0])

    def option(self, q, n):
        return option_index(draw(self.seed, self.g, 1, q)[0], n)

    def trial(self, q, t):     # scale w, scale h, left, top
        return [unif(x) for x in draw(self.seed, self.g, 2 + q, t)]


def canvas_corners(boxes, width, height, pl, pt):
    """float64 pixel corners (x0, y0, x1, y1) of relative cxcywh float32 rows on the canvas."""
    b = np.asarray(boxes, np.float32).reshape(-1, 4).astype(np.float64)
    hw, hh = 0.5 * b[:, 2], 0.5 * b[:, 3]
    return np.stack([(b[:, 0] - hw) * width + pl, (b[:, 1] - hh) * height + pt,
                     (b[:, 0] + hw) * width + pl, (b[:, 1] + hh) * height + pt], axis=1)


def within(k, l, t, w, h):
    cx, cy = 0.5 * (k[:, 0] + k[:, 2]), 0.5 * (k[:, 1] + k[:, 3])
    with np.errstate(invalid="ignore"):
        return (l < cx) & (cx < l + w) & (t < cy) & (cy < t + h)


def box_iou_crop(k, l, t, w, h):
    """torchvision's box_iou of rows against the crop, in float64."""
    area1 = (k[:, 2] - k[:, 0]) * (k[:, 3] - k[:, 1])
    area2 = float(w) * float(h)
    ex = np.maximum(np.minimum(k[:, 2], float(l + w)) - np.maximum(k[:, 0], float(l)), 0.0)
    ey = np.maximum(np.minimum(k[:, 3], float(t + h)) - np.maximum(k[:, 1], float(t)), 0.0)
    inter = ex * ey
    with np.errstate(invalid="ignore", divide="ignore"):
        return inter / ((area1 + area2) - inter)


def crop_trial(u, cw, ch, cfg):
    """(left, top, new_w, new_h, ok) of a trial from its four uniforms."""
    lo, d = f32(cfg["min_scale"]), f32(cfg["max_scale"] - cfg["min_scale"])
    nw, nh = int(f32(cw) * (lo + u[0] * d)), int(f32(ch) * (lo + u[1] * d))
    left, top = int(f32(cw - nw) * u[2]), int(f32(ch - nh) * u[3])
    ok = nw != 0 and nh != 0 and cfg["min_aspect"] <= nw / nh <= cfg["max_aspect"]
    return left, top, nw, nh, ok


def sample(boxes, seed, g, height, width, cfg):
    """The transform record (RECORD order) of one image and its within mask (None without a crop)."""
    u = Uniforms(seed, g)
    z = u.zoom()
    cw, ch, pl, pt = width, height, 0, 0
    if z[0] < f32(cfg["zoom_p"]):
        lo, hi = cfg["side_range"]
        r = f32(lo) + z[1] * f32(hi - lo)
        cw, ch = int(f32(width) * r), int(f32(height) * r)
        pl, pt = int(f32(cw - width) * z[2]), int(f32(ch - height) * z[3])
    k = canvas_corners(boxes, width, height, pl, pt)
    opts = list(cfg["min_ious"])
    crop, mask, rounds = (0, 0, cw, ch), None, (-1 if opts else 0)
    for q in range(cfg["max_rounds"] if opts else 0):
        m = float(opts[u.option(q, len(opts))])
        if m >= 1.0:
            rounds = q + 1
            break
        for t in range(cfg["trials"]):
            left, top, nw, nh, ok = crop_trial(u.trial(q, t), cw, ch, cfg)
            if not ok:
                continue
            inside = within(k, left, top, nw, nh)
            if not inside.any():
                continue
            with np.errstate(invalid="ignore"):
                if not (~(box_iou_crop(k[inside], left, top, nw, nh) < m)).any():
                    continue
            crop, mask, rounds = (left, top, nw, nh), inside, q + 1
            break
        if mask is not None:
            break
    flip = int(u.flip() < f32(cfg["flip_p"]))
    return np.array([cw, ch, pl, pt, *crop, flip, rounds], np.int32), mask


def map_rows(boxes, rec, width, height, cropped):
    """Rows through a record: shift into the crop, clamp when cropped, relative cxcywh of the crop, flip; float64,
    rounded once to float32."""
    k = canvas_corners(boxes, width, height, rec[2], rec[3])
    l, t, w, h = (float(v) for v in rec[4:8])
    x0, y0, x1, y1 = k[:, 0] - l, k[:, 1] - t, k[:, 2] - l, k[:, 3] - t
    if cropped:
        x0, x1 = np.minimum(np.maximum(x0, 0.0), w), np.minimum(np.maximum(x1, 0.0), w)
        y0, y1 = np.minimum(np.maximum(y0, 0.0), h), np.minimum(np.maximum(y1, 0.0), h)
    with np.errstate(invalid="ignore"):
        cx = ((x0 + x1) * 0.5) / w
        if rec[8]:
            cx = 1.0 - cx
        return np.stack([cx, ((y0 + y1) * 0.5) / h, (x1 - x0) / w, (y1 - y0) / h], axis=1).astype(np.float32)


def source_coords(n_out, n_in):
    """F.interpolate(bilinear, align_corners=False) source taps in float32: (i0, i1, lambda1)."""
    s = np.maximum(f32(0), (f32(n_in) / f32(n_out)) * (np.arange(n_out, dtype=np.float32) + f32(0.5)) - f32(0.5))
    i0 = s.astype(np.int64)
    i1 = i0 + (i0 < n_in - 1)
    return i0, i1, s - i0.astype(np.float32)


def resample(image, rec, fill):
    """Output image f32[H,W,3] of one record: bilinear over the crop of the virtual canvas, float64 blend."""
    image = np.asarray(image, np.float32)
    h_img, w_img = image.shape[:2]
    x0, x1, lx = source_coords(w_img, int(rec[6]))
    y0, y1, ly = source_coords(h_img, int(rec[7]))
    ox, oy = int(rec[4]) - int(rec[2]), int(rec[5]) - int(rec[3])
    fillv = np.asarray(fill, np.float32).astype(np.float64)

    def tap(ys, xs):
        yy, xx = ys[:, None] + oy, xs[None, :] + ox
        ok = (yy >= 0) & (yy < h_img) & (xx >= 0) & (xx < w_img)
        v = image[np.clip(yy, 0, h_img - 1), np.clip(xx, 0, w_img - 1)].astype(np.float64)
        return np.where(ok[..., None], v, fillv)

    lx, ly = lx.astype(np.float64)[None, :, None], ly.astype(np.float64)[:, None, None]
    hx, hy = (1 - lx.astype(np.float32)).astype(np.float64), (1 - ly.astype(np.float32)).astype(np.float64)
    out = hy * (hx * tap(y0, x0) + lx * tap(y0, x1)) + ly * (hx * tap(y1, x0) + lx * tap(y1, x1))
    if rec[8]:
        out = out[:, ::-1]
    return out.astype(np.float32)


def augment(images, boxes, cls, offsets, seed, image_base=0, size=None, **config):
    """A13 for a batch: returns dict(images, boxes, cls, offsets, src_row, transform) laid out as the device writes
    them (rows past offsets[B]: zero / -1).  images None: the boxes only, for images of ``size`` (H, W)."""
    cfg = dict(DEFAULTS, **config)
    boxes = np.asarray(boxes, np.float32).reshape(-1, 4)
    cls = np.asarray(cls, np.float32).reshape(-1)
    offsets = np.asarray(offsets, np.int64)
    b = offsets.size - 1
    height, width = (images.shape[1], images.shape[2]) if images is not None else size
    rows = boxes.shape[0]
    out = dict(boxes=np.zeros((rows, 4), np.float32), cls=np.zeros(rows, np.float32),
               src_row=np.full(rows, -1, np.int32), offsets=np.zeros(b + 1, np.int32),
               transform=np.zeros((b, len(RECORD)), np.int32))
    o = 0
    for i in range(b):
        r0, r1 = int(offsets[i]), int(offsets[i + 1])
        rec, mask = sample(boxes[r0:r1], seed, image_base + i, height, width, cfg)
        keep = np.arange(r0, r1) if mask is None else r0 + np.flatnonzero(mask)
        n = keep.size
        out["boxes"][o:o + n] = map_rows(boxes[keep], rec, width, height, mask is not None)
        out["cls"][o:o + n] = cls[keep]
        out["src_row"][o:o + n] = keep
        o += n
        out["offsets"][i + 1] = o
        out["transform"][i] = rec
    if images is not None:
        out["images"] = np.stack([resample(images[i], out["transform"][i], cfg["fill"]) for i in range(b)])
    return out
