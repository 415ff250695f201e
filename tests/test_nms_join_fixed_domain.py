"""The candidate pairs of nms_kernel's interval join (detect.cu) -- slabs fixed over [0, 1] and clamped, size classes
against the fixed reference width 1, and a box whose corner extents do not reproduce its area (inexact) registered
unshrunk and in every size class -- restated with the kernel's float32 arithmetic: the join may only prune pairs the
IoU formula keeps below the threshold, wherever the boxes lie and whichever of them are inexact."""
import numpy as np
import pytest

from oracle import ssd_oracle as O

f = np.float32
N_SLABS, N_SIZE = 32, 16


def join_candidates(boxes, thr):
    """(i, j, keep) over the lower triangle i > j: keep marks the pairs the join passes to the pair test."""
    b = np.asarray(boxes, f)
    with np.errstate(all="ignore"):
        hw, hh = b[:, 2] * f(0.5), b[:, 3] * f(0.5)
        x1, y1, x2, y2 = b[:, 0] - hw, b[:, 1] - hh, b[:, 0] + hw, b[:, 1] + hh
        area = b[:, 2] * b[:, 3]
        sane = (b[:, 2] > 0) & (b[:, 3] > 0) & np.isfinite(x1) & np.isfinite(y1) & np.isfinite(x2) & np.isfinite(y2) \
            & np.isfinite(area)
        q = f(thr) / (f(1) + f(thr))
        pr = (x2 - x1) * (y2 - y1)
        exact = (area >= f(0.999) * pr) & (area <= f(1.001) * pr)
        tq = np.where(exact, min(f(0.98) * q, f(0.49)), f(0)).astype(f)

        def slab(v):
            return np.clip(np.floor(np.nan_to_num(v * f(N_SLABS), nan=0.0)), 0, N_SLABS - 1).astype(np.int64)

        sx = tq * (x2 - x1) - f(1e-6) * (np.abs(x1) + np.abs(x2))
        sy = tq * (y2 - y1) - f(1e-6) * (np.abs(y1) + np.abs(y2))
        ax, ay = slab(x1 + sx), slab(y1 + sy)
        bx, by = np.maximum(slab(x2 - sx), ax), np.maximum(slab(y2 - sy), ay)
        tp = f(0.99) * f(thr) / (f(1) + f(0.001) * f(thr))
        inv_l = f(-1) / np.log2(tp) if tp < f(0.98) else f(0)

        def size_cls(ext):
            return np.clip(np.floor(np.nan_to_num(-np.log2(ext) * inv_l, nan=0.0)), 0, N_SIZE - 1).astype(np.int64)

        cw, ch = size_cls(x2 - x1), size_cls(y2 - y1)
    i, j = np.tril_indices(len(b), -1)
    sizes = ((np.abs(cw[i] - cw[j]) <= 1) & (np.abs(ch[i] - ch[j]) <= 1)) | ~exact[i] | ~exact[j]
    keep = (sane[i] & sane[j] & (ax[j] <= bx[i]) & (bx[j] >= ax[i]) & (ay[j] <= by[i]) & (by[j] >= ay[i]) & sizes)
    return i, j, keep, exact


def _boxes(rng, n, lo, hi, wlo, whi):
    c = rng.uniform(lo, hi, (n, 2))
    wh = np.exp(rng.uniform(np.log(wlo), np.log(whi), (n, 2)))
    b = np.concatenate([c, wh], 1).astype(f)
    dup = b[1::5][:len(b[::5])].copy()               # near duplicates: real suppression
    dup[:, 2:] *= f(1.01)
    b[::5] = dup
    return b


@pytest.mark.parametrize("thr", [0.05, 0.3, 0.45, 0.6, 0.9])
def test_fixed_domain_join_never_drops_a_suppressing_pair(thr):
    rng = np.random.default_rng(int(thr * 1000))
    sets = {
        "unit square": _boxes(rng, 200, 0.0, 1.0, 0.01, 0.9),
        "beyond [0, 1]": _boxes(rng, 200, -1.5, 2.5, 0.05, 3.0),    # clamped slabs, widths above the reference
        "tiny": _boxes(rng, 200, 0.4, 0.45, 1e-6, 1e-4),            # exact and inexact boxes side by side
    }
    mixed = 0
    for name, boxes in sets.items():
        i, j, keep, exact = join_candidates(boxes, thr)
        with np.errstate(all="ignore"):
            hot = O.iou(boxes[i], boxes[j]) > f(thr)
        assert hot.sum() > 0, name
        assert not np.any(hot & ~keep), name
        if name != "tiny":
            assert keep.sum() < 0.5 * len(i), name                     # and it does prune
        mixed += int(np.sum(hot & (exact[i] != exact[j])))
    assert mixed > 0 or thr > 0.6                                       # the per-box rule is exercised
