"""Seeded synthetic "COCO-shaped" inputs for the SSD box-geometry hot path.

NumPy only (no torch, no CUDA): used by the parity tests, by ``bench.py`` and by
the oracle's golden-vector generator, so every consumer sees identical bytes.

The generator follows SURVEY.md section 8(d):

* ground truth per image: ``cx, cy ~ U(0,1)``, ``w, h = exp(U(ln 0.02, ln 0.9))``,
  float32 relative cxcywh (the contract of the reference data adapter,
  data_loaders/ssd/make_dataset.py:37-46), class ids ``U{0..79}`` stored as
  float32 (data_loaders/ssd/make_dataset.py:57);
* two T modes: ``max`` (every image has ``max_t`` boxes) and ``coco``
  (``clip(round(lognormal(ln 4.5, 1)), 1, max_t)``, mean about 7);
* logits ``N(0,1)`` float32 with the background column (last class, the
  reference's convention at models/ssd_model.py:365) shifted by ``bg_bias``;
* box regressions ``N(0,1) * 0.5`` float32.
"""
from __future__ import annotations

import math

import numpy as np

# The reference's SSD300 table (models/ssd_model.py:153,176-177) and the SSD512
# extension SURVEY.md 8(a) row A1 prescribes (same rule, 7 levels).
SSD300 = dict(
    input_size=300,
    sizes=[(38, 38), (19, 19), (10, 10), (5, 5), (3, 3), (1, 1)],
    s_k_refer=[21, 45, 99, 153, 207, 261, 315],
    aspect_ratio=[[2], [2, 3], [2, 3], [2, 3], [2], [2]],
)
SSD512 = dict(
    input_size=512,
    sizes=[(64, 64), (32, 32), (16, 16), (8, 8), (4, 4), (2, 2), (1, 1)],
    s_k_refer=[20.48, 51.2, 133.12, 215.04, 296.96, 378.88, 460.8, 542.72],
    aspect_ratio=[[2], [2, 3], [2, 3], [2, 3], [2, 3], [2], [2]],
)
TABLES = {"ssd300": SSD300, "ssd512": SSD512}


def num_priors(table) -> int:
    return sum(h * w * (2 + 2 * len(r)) for (h, w), r in zip(table["sizes"], table["aspect_ratio"]))


def gt_counts(rng: np.random.Generator, batch: int, max_t: int, mode: str) -> np.ndarray:
    if mode == "max":
        return np.full((batch,), max_t, dtype=np.int32)
    if mode == "coco":
        t = np.rint(rng.lognormal(mean=math.log(4.5), sigma=1.0, size=batch))
        return np.clip(t, 1, max_t).astype(np.int32)
    raise ValueError("mode must be 'max' or 'coco'")


def make_gt(seed: int, batch: int, max_t: int = 100, mode: str = "max", num_fg: int = 80):
    """CSR-packed ground truth: boxes f32[sum T,4], cls f32[sum T], offsets i32[B+1]."""
    rng = np.random.default_rng(seed)
    counts = gt_counts(rng, batch, max_t, mode)
    offsets = np.zeros((batch + 1,), dtype=np.int32)
    np.cumsum(counts, out=offsets[1:])
    n = int(offsets[-1])
    cxcy = rng.uniform(0.0, 1.0, size=(n, 2))
    wh = np.exp(rng.uniform(math.log(0.02), math.log(0.9), size=(n, 2)))
    boxes = np.concatenate([cxcy, wh], axis=1).astype(np.float32)
    cls = rng.integers(0, num_fg, size=n).astype(np.float32)
    return boxes, cls, offsets


def make_predictions(seed: int, batch: int, num_anchors: int, num_classes: int = 81,
                     bg_bias: float = 7.0):
    """pred_cls f32[B,A,C] ("trained-like": background column shifted) and pred_box f32[B,A,4]."""
    rng = np.random.default_rng(seed + 7919)
    pred_cls = rng.standard_normal(size=(batch, num_anchors, num_classes), dtype=np.float32)
    pred_cls[..., -1] += np.float32(bg_bias)
    pred_box = rng.standard_normal(size=(batch, num_anchors, 4), dtype=np.float32) * np.float32(0.5)
    return pred_cls, pred_box


def make_trained_predictions(seed: int, tgt_cls, tgt_loc, tgt_mask, num_classes: int = 81, bg_bias: float = 7.0,
                             max_noise: float = 0.25, boost=(3.0, 12.0)):
    """Predictions of a partly trained detector, built from the matcher's targets (cls i32[B,A], loc f32[B,A,4], mask
    [B,A]) so that AP is meaningful: every positive prior gets its encoded target plus N(0, s^2) noise with s ~
    U(0, max_noise) per prior (IoUs spread over all COCO thresholds) and its ground-truth logit raised by U(boost);
    everything else is ``make_predictions``."""
    tgt_cls, tgt_loc = np.asarray(tgt_cls), np.asarray(tgt_loc, np.float32)
    pos = np.asarray(tgt_mask).astype(bool)
    b, a = pos.shape
    pred_cls, pred_box = make_predictions(seed, b, a, num_classes, bg_bias)
    rng = np.random.default_rng(seed + 104729)
    n = int(pos.sum())
    sigma = rng.uniform(0.0, max_noise, size=(n, 1))
    pred_box[pos] = (tgt_loc[pos] + rng.standard_normal(size=(n, 4)) * sigma).astype(np.float32)
    bi, ai = np.nonzero(pos)
    pred_cls[bi, ai, tgt_cls[pos]] += rng.uniform(boost[0], boost[1], size=n).astype(np.float32)
    return pred_cls, pred_box
