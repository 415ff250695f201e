"""Detection evaluation on the device: COCO-style AP (AP@[.5:.95], AP50, AP75, AR@max_dets, per-class AP) over the
kept lists of ``ops.detect``, accumulated across batches and data-parallel processes (include/ssdgeom.h, A11).
Only the finished precision / recall arrays cross to the host.

    ev = DetectionEvaluator(max_images=5000)
    for each batch:
        det = ops.detect(pred_cls, pred_box, priors, want_scores=True, want_boxes=True)
        ev.add(det, gt_boxes, gt_cls, gt_off)        # CSR ground truth, as ops.match_encode
    ev.exchange(comm)                                # data parallel only: sum the slots over the processes
    res = ev.summarize()                             # {"AP", "AP50", "AP75", "AR", "per_class_AP", ...}

The evaluator caps each (image, class) list at ``max_dets``.  For a detector that emits at most K detections per image,
feed it the per-image capped lists of ``ops.keep_top_k``: their survivors are a prefix of every list, so only the counts
change --

        top = ops.keep_top_k(det, 100)
        ev.add(dict(det, count=top["count"]), gt_boxes, gt_cls, gt_off)
"""
from __future__ import annotations

import numpy as np

from . import device as D
from . import ops

# COCOeval.Params.setDetParams, exactly (0.5 and 0.75 are found by equality, as COCOeval.summarize does)
COCO_IOU_THRESHOLDS = np.linspace(.5, 0.95, int(np.round((0.95 - .5) / .05)) + 1, endpoint=True)
COCO_RECALL_THRESHOLDS = np.linspace(.0, 1.00, int(np.round((1.00 - .0) / .01)) + 1, endpoint=True)

_STATUS_TEXT = ((ops.EVAL_STATUS_BAD_CLASS, "a ground-truth class id outside [0, n_classes - 1)"),
                (ops.EVAL_STATUS_TOO_MANY_GT, "an image with more ground-truth rows than max_gt"),
                (ops.EVAL_STATUS_DUPLICATE, "a global image index written by more than one process or batch slot"),
                (ops.EVAL_STATUS_BAD_PRIOR, "a kept prior index outside the prior set"))


def _mean_valid(s) -> float:
    """COCOeval.summarize: mean(s[s > -1]), -1 when nothing is valid."""
    s = np.asarray(s)
    v = s[s > -1]
    return float(np.mean(v)) if v.size else -1.0


class DetectionEvaluator:
    """Accumulates one evaluation.  ``max_images`` bounds the global image indices (image_base + i): one fixed slot
    per (class, image, rank), 12 bytes each, so 5 000 images x 80 classes x 100 detections take 480 MB."""

    def __init__(self, n_classes: int = 81, max_images: int = 5000, max_dets: int = 100, iou_thresholds=None,
                 recall_thresholds=None, max_gt: int = 100, stream=None):
        """max_gt: the bound on ground-truth rows per image used when ``add`` gets its offsets on the device."""
        self.iou_thresholds = np.array(COCO_IOU_THRESHOLDS if iou_thresholds is None else iou_thresholds, np.float64)
        self.recall_thresholds = np.array(COCO_RECALL_THRESHOLDS if recall_thresholds is None else recall_thresholds,
                                          np.float64)
        self.n_classes, self.max_images, self.max_dets = int(n_classes), int(max_images), int(max_dets)
        self.max_gt = int(max_gt)
        self.state = ops.eval_state(self.n_classes, self.max_images, self.max_dets, self.iou_thresholds.size, stream)
        self.pool = ops.WorkspacePool()
        self.next_image = 0

    def reset(self, stream=None):
        ops.eval_reset(self.state, stream)
        self.next_image = 0

    def add(self, detect_out: dict, gt_boxes, gt_cls, gt_off, image_base=None, stream=None, max_gt=None) -> int:
        """Enqueue the matching of one batch (``ops.detect`` outputs with ``kept_score`` and ``boxes``) on ``stream``.
        image_base None continues after the highest image added so far.  Returns the batch's image_base."""
        base = self.next_image if image_base is None else int(image_base)
        if max_gt is None:
            max_gt = self.max_gt if D.is_device(gt_off) else max(int(np.max(np.diff(np.asarray(gt_off)), initial=0)), 0)
        kept = ops.eval_accumulate(detect_out, gt_boxes, gt_cls, gt_off, self.state, self.iou_thresholds, base, max_gt,
                                   stream)[0]     # the kept lists as a device array [B,C-1,top_k]
        self.next_image = max(self.next_image, base + kept.shape[0])
        return base

    def exchange_buffers(self) -> list:
        """[int64, int32] device buffers whose element-wise sum over the processes is the all-gathered state."""
        return ops.eval_exchange(self.state)

    def exchange(self, comm_or_allreduce, stream=None):
        """Sum the state over the data-parallel processes, in place on ``stream``: ``comm`` (ssdgeom.comm.Comm) or
        an ``allreduce(buf, stream)`` callable.  Every process then holds every image's slots."""
        bufs = self.exchange_buffers()
        if hasattr(comm_or_allreduce, "allreduce_multi"):
            comm_or_allreduce.allreduce_multi(bufs, stream)
        else:
            for buf in bufs:
                comm_or_allreduce(buf, stream)

    def finalize(self, stream=None) -> dict:
        """Host precision f64[T,R,K], recall f64[T,K], n_gt i64[K], n_det i64[K] (synchronises); raises when the
        device reported an error."""
        out = ops.eval_finalize(self.state, self.recall_thresholds, stream, self.pool)
        res = {k: out[k].to_host(stream) for k in ("precision", "recall", "n_gt", "n_det")}
        status = ops.eval_status(self.state, stream)
        if status:
            raise ValueError("detection evaluation: " + "; ".join(t for bit, t in _STATUS_TEXT if status & bit))
        return res

    def summarize(self, stream=None) -> dict:
        res = self.finalize(stream)
        p, r = res["precision"], res["recall"]
        thr = self.iou_thresholds
        res.update(AP=_mean_valid(p), AP50=_mean_valid(p[np.where(.5 == thr)[0]]),
                   AP75=_mean_valid(p[np.where(.75 == thr)[0]]), AR=_mean_valid(r),
                   per_class_AP=np.array([_mean_valid(p[:, :, c]) for c in range(p.shape[2])]))
        return res
