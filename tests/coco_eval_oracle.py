"""NumPy restatement of the detection evaluation spec (include/ssdgeom.h, A11): pycocotools COCOeval.evaluateImg /
accumulate / summarize for iouType "bbox", area range "all", no crowd and no ignore flags, written line by line
so that the device results can be compared bit for bit.  The checker only: product code never imports it."""
from __future__ import annotations

import numpy as np

# COCOeval.Params.setDetParams, exactly
COCO_IOU_THRESHOLDS = np.linspace(.5, 0.95, int(np.round((0.95 - .5) / .05)) + 1, endpoint=True)
COCO_RECALL_THRESHOLDS = np.linspace(.0, 1.00, int(np.round((1.00 - .0) / .01)) + 1, endpoint=True)


def box_iou(d, g) -> float:
    """IoU of two float32 cxcywh boxes in float64, in the spec's operation order."""
    cxd, cyd, wd, hd = (float(v) for v in np.asarray(d, np.float32))
    cxg, cyg, wg, hg = (float(v) for v in np.asarray(g, np.float32))
    x0d, x1d, y0d, y1d = cxd - 0.5 * wd, cxd + 0.5 * wd, cyd - 0.5 * hd, cyd + 0.5 * hd
    x0g, x1g, y0g, y1g = cxg - 0.5 * wg, cxg + 0.5 * wg, cyg - 0.5 * hg, cyg + 0.5 * hg
    iw = min(x1d, x1g) - max(x0d, x0g)
    ih = min(y1d, y1g) - max(y0d, y0g)
    if iw <= 0 or ih <= 0:
        return 0.0
    inter = iw * ih
    return inter / ((wd * hd + wg * hg) - inter)


def coco_evaluate_image(det_boxes, gt_boxes, iou_thresholds=COCO_IOU_THRESHOLDS, max_dets=100):
    """One (image, class): detections in visit order (score desc, already sorted), ground truth in row order.
    Returns bool tp[T, min(n_det, max_dets)] (evaluateImg's dtMatches > 0)."""
    det_boxes = np.asarray(det_boxes, np.float32).reshape(-1, 4)[:max_dets]
    gt_boxes = np.asarray(gt_boxes, np.float32).reshape(-1, 4)
    n_t = len(iou_thresholds)
    tp = np.zeros((n_t, det_boxes.shape[0]), bool)
    gtm = np.zeros((n_t, gt_boxes.shape[0]), bool)
    ious = [[box_iou(d, g) for g in gt_boxes] for d in det_boxes]
    for tind, t in enumerate(iou_thresholds):
        for dind in range(det_boxes.shape[0]):
            iou = min([float(t), 1 - 1e-10])
            m = -1
            for gind in range(gt_boxes.shape[0]):
                if gtm[tind, gind]:
                    continue
                if ious[dind][gind] < iou:
                    continue
                iou = ious[dind][gind]
                m = gind
            if m == -1:
                continue
            gtm[tind, m] = True
            tp[tind, dind] = True
    return tp


def evaluate_batch(kept, count, kept_score, boxes, gt_boxes, gt_cls, gt_off, image_base=0,
                   iou_thresholds=COCO_IOU_THRESHOLDS, max_dets=100):
    """Records of one batch of ssdg_detect outputs: {class: [(score f32, global image, rank, tp bool[T])]} and
    {class: {global image: ground-truth rows}} (classes are gt_cls truncated to int)."""
    kept, count, kept_score = np.asarray(kept), np.asarray(count), np.asarray(kept_score, np.float32)
    boxes, gt_boxes = np.asarray(boxes, np.float32), np.asarray(gt_boxes, np.float32)
    gcls = np.trunc(np.asarray(gt_cls, np.float32)).astype(np.int64)
    b, k = count.shape
    records = {c: [] for c in range(k)}
    n_gt = {c: {} for c in range(k)}
    for i in range(b):
        rows = np.arange(gt_off[i], gt_off[i + 1])
        img = image_base + i
        for c in range(k):
            g = gt_boxes[rows[gcls[rows] == c]]
            n_gt[c][img] = g.shape[0]
            nd = min(int(count[i, c]), max_dets)
            pri = kept[i, c, :nd]
            tp = coco_evaluate_image(boxes[i, pri], g, iou_thresholds, max_dets)
            for r in range(nd):
                records[c].append((np.float32(kept_score[i, c, r]), img, r, tp[:, r]))
    return records, n_gt


def merge(*parts):
    """Union of evaluate_batch results of distinct images."""
    records, n_gt = {}, {}
    for rec, ng in parts:
        for c, v in rec.items():
            records.setdefault(c, []).extend(v)
        for c, v in ng.items():
            n_gt.setdefault(c, {}).update(v)
    return records, n_gt


def slots(records, n_gt, n_classes, max_images, max_dets):
    """The device state's slot arrays: keys i64[K,M,D], flags i32[K,M,D], n_gt i32[K,M]."""
    k = n_classes - 1
    keys = np.zeros((k, max_images, max_dets), np.uint64)
    flags = np.zeros((k, max_images, max_dets), np.int64)
    ng = np.zeros((k, max_images), np.int32)
    for c in range(k):
        for img, n in n_gt.get(c, {}).items():
            ng[c, img] = n
        for score, img, r, tp in records.get(c, []):
            sbits = int(np.float32(score).view(np.uint32))
            keys[c, img, r] = (sbits << 32) | (0xFFFFFFFF - ((img << 10) | r))
            flags[c, img, r] = (1 << 16) | int(sum(1 << t for t in np.nonzero(tp)[0]))
    return keys.view(np.int64), flags.astype(np.int32), ng


def coco_accumulate(records, n_gt, n_classes, n_thresholds=len(COCO_IOU_THRESHOLDS),
                    recall_thresholds=COCO_RECALL_THRESHOLDS):
    """COCOeval.accumulate for one area range and max_dets: precision f64[T,R,K], recall f64[T,K],
    n_gt i64[K], n_det i64[K]."""
    k = n_classes - 1
    rec_thrs = np.asarray(recall_thresholds, np.float64)
    n_r = rec_thrs.size
    precision = -np.ones((n_thresholds, n_r, k))
    recall = -np.ones((n_thresholds, k))
    out_gt = np.zeros(k, np.int64)
    out_det = np.zeros(k, np.int64)
    for c in range(k):
        rec = records.get(c, [])
        npig = int(sum(n_gt.get(c, {}).values()))
        nd = len(rec)
        out_gt[c], out_det[c] = npig, nd
        if npig == 0:
            continue
        scores = np.array([r[0] for r in rec], np.float64)
        imgs = np.array([r[1] for r in rec], np.int64)
        ranks = np.array([r[2] for r in rec], np.int64)
        tpm = np.array([r[3] for r in rec], bool).reshape(nd, n_thresholds).T
        order = np.lexsort((ranks, imgs, -scores))          # score desc, global image asc, rank asc
        tps = tpm[:, order]
        fps = np.logical_not(tps)
        tp_sum = np.cumsum(tps, axis=1).astype(dtype=float)
        fp_sum = np.cumsum(fps, axis=1).astype(dtype=float)
        for t, (tp, fp) in enumerate(zip(tp_sum, fp_sum)):
            tp, fp = np.array(tp), np.array(fp)
            rc = tp / npig
            pr = tp / (fp + tp + np.spacing(1))
            q = np.zeros((n_r,))
            recall[t, c] = rc[-1] if nd else 0
            pr = pr.tolist()
            for i in range(nd - 1, 0, -1):
                if pr[i] > pr[i - 1]:
                    pr[i - 1] = pr[i]
            inds = np.searchsorted(rc, rec_thrs, side="left")
            for ri, pi in enumerate(inds):
                if pi < nd:
                    q[ri] = pr[pi]
            precision[t, :, c] = q
    return precision, recall, out_gt, out_det


def _mean_valid(s):
    s = np.asarray(s)
    return float(np.mean(s[s > -1])) if np.any(s > -1) else -1.0


def coco_summarize(precision, recall, iou_thresholds=COCO_IOU_THRESHOLDS):
    """COCOeval.summarize's rule mean(s[s > -1]) (-1 if empty): AP@[.5:.95], AP50, AP75, AR, per-class AP."""
    thr = np.asarray(iou_thresholds)
    t50, t75 = np.where(.5 == thr)[0], np.where(.75 == thr)[0]
    return {"AP": _mean_valid(precision), "AP50": _mean_valid(precision[t50]), "AP75": _mean_valid(precision[t75]),
            "AR": _mean_valid(recall),
            "per_class_AP": np.array([_mean_valid(precision[:, :, c]) for c in range(precision.shape[2])])}
