"""NumPy restatement of the per-image keep_top_k spec (include/ssdgeom.h, A12): the kept lists of the per-class NMS
ranked across classes and capped at K, written as one lexsort per image so that the device results can be compared
bit for bit.  The checker only: product code never imports it."""
from __future__ import annotations

import numpy as np


def keep_top_k(kept, count, kept_score, boxes, K):
    """A12 for a batch: ``kept`` int32 [B,C-1,top_k], ``count`` [B,C-1], ``kept_score`` float32 [B,C-1,top_k], decoded
    ``boxes`` float32 [B,A,4] or None.  The candidates of an image are the first clamp(count, 0, top_k) entries of
    every class list, ranked by score descending (as float values: -0 == +0), class ascending, position ascending; the
    first min(K, total) are kept.  Returns (prior int32 [B,K] -1 padded, class int32 [B,K] -1 padded, score float32
    [B,K] 0 padded, box float32 [B,K,4] 0 padded -- zeros for a prior outside [0, A) -- or None, n int32 [B],
    count int32 [B,C-1] survivors per class)."""
    kept = np.asarray(kept, np.int32)
    kept_score = np.asarray(kept_score, np.float32)
    b, k, top_k = kept.shape
    cnt = np.clip(np.asarray(count, np.int64).reshape(b, k), 0, top_k)
    prior, cls = np.full((b, K), -1, np.int32), np.full((b, K), -1, np.int32)
    score, n, out_count = np.zeros((b, K), np.float32), np.zeros((b,), np.int32), np.zeros((b, k), np.int32)
    box = None if boxes is None else np.zeros((b, K, 4), np.float32)
    for i in range(b):
        c = np.repeat(np.arange(k), cnt[i])
        pos = np.arange(c.size) - np.repeat(np.cumsum(cnt[i]) - cnt[i], cnt[i])
        s = kept_score[i, c, pos]
        order = np.lexsort((pos, c, -s.astype(np.float64)))[:K]
        m = order.size
        n[i] = m
        prior[i, :m] = kept[i, c[order], pos[order]]
        cls[i, :m] = c[order]
        score[i, :m] = s[order]
        out_count[i] = np.bincount(c[order], minlength=k)
        if box is not None:
            p = prior[i, :m]
            ok = (p >= 0) & (p < boxes.shape[1])
            box[i, :m][ok] = np.asarray(boxes, np.float32)[i, p[ok]]
    return prior, cls, score, box, n, out_count
