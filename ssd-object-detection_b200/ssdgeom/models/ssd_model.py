"""Drop-in for the box-geometry methods of the reference's ``SSDObjectDetectionModel``
(models/ssd_model.py): ``_build_prior_box`` (:173-194), the target assigner inside
``get_train_set`` (:209-227), ``_ssd_loss`` (:341-396), the score head of ``visualize``
(:477-490) with the inline decode of ``visualize_dataset`` (:466-467), plus the per-class NMS
the north star adds.  The network, training loop, TensorBoard and OpenCV parts are out of scope."""
from __future__ import annotations

import numpy as np

from .. import device as D
from .. import ops
from ..utils.bbox import match_encode_batch

# the tables hard-coded at models/ssd_model.py:153,176-177 (SSD300) and the SSD512 extension
SSD300 = dict(input_size=300, sizes=[(38, 38), (19, 19), (10, 10), (5, 5), (3, 3), (1, 1)],
              s_k_refer=[21, 45, 99, 153, 207, 261, 315], aspect_ratio=[[2], [2, 3], [2, 3], [2, 3], [2], [2]])
SSD512 = dict(input_size=512, sizes=[(64, 64), (32, 32), (16, 16), (8, 8), (4, 4), (2, 2), (1, 1)],
              s_k_refer=[20.48, 51.2, 133.12, 215.04, 296.96, 378.88, 460.8, 542.72],
              aspect_ratio=[[2], [2, 3], [2, 3], [2, 3], [2, 3], [2], [2]])


def build_prior_box(size_list, s_k_refer=None, aspect_ratio=None, input_size=300, device_out=False, clip=False):
    """``_build_prior_box(size_list)`` (models/ssd_model.py:173-194): float64 [A,4] cxcywh.  ``clip`` (an option
    the reference does not have) clamps every component to [0,1]."""
    size_list = [tuple(int(v) for v in s) for s in size_list]
    s_k_refer = SSD300["s_k_refer"] if s_k_refer is None else s_k_refer
    aspect_ratio = SSD300["aspect_ratio"] if aspect_ratio is None else aspect_ratio
    out = ops.prior_boxes(size_list, s_k_refer[:len(size_list) + 1], aspect_ratio[:len(size_list)], input_size, clip=clip)
    return out if device_out else out.to_host()


def _loss(y_true, y_pred, neg_ratio, **want):
    """The device loss of host or device arrays: (host result dict, info, device outputs)."""
    gt_cls, gt_box, gt_mask = y_true
    pred_box, pred_cls = y_pred
    if not D.is_device(gt_mask):
        gt_mask = np.ascontiguousarray(np.asarray(gt_mask).astype(np.uint8))
    out = ops.multibox_loss(gt_cls, gt_box, gt_mask, pred_box, pred_cls, neg_ratio, **want)
    r = ops.loss_result_to_host(out["result"])
    return r, {k: r[k] for k in ("cls loss pos", "cls loss neg", "loc loss")}, out


def ssd_loss(y_true, y_pred, neg_ratio=3, return_aux=False):
    """``_ssd_loss(y_true, y_pred)`` (models/ssd_model.py:341-396):
    y_true = (gt_cls int32[b,A], gt_box f32[b,A,4], gt_mask bool[b,A]); y_pred = (pred_box, pred_cls).
    Returns (total, {"cls loss pos", "cls loss neg", "loc loss"})."""
    shapes = [tuple(np.shape(v)) if not D.is_device(v) else tuple(v.shape) for v in (*y_true, *y_pred)]
    assert shapes[0][0] == shapes[1][0] == shapes[2][0] == shapes[3][0] == shapes[4][0]   # :347-348
    assert shapes[0][:2] == shapes[4][:2]                                                   # :350-351
    r, info, out = _loss(y_true, y_pred, neg_ratio, want_neg_mask=return_aux, want_neg_ce=return_aux)
    if return_aux:
        aux = dict(r, neg_mask=out["neg_mask"].to_host().astype(bool), neg_ce=out["neg_ce"].to_host())
        return r["total"], info, aux
    return r["total"], info


def ssd_loss_grad(y_true, y_pred, neg_ratio=3):
    """Loss plus what ``tape.gradient`` (models/ssd_model.py:248) propagates to the predictions:
    returns (total, info, grad_pred_box f32[b,A,4], grad_pred_cls f32[b,A,C])."""
    r, info, out = _loss(y_true, y_pred, neg_ratio, want_grad=True)
    return r["total"], info, out["grad_box"].to_host(), out["grad_cls"].to_host()


def score_head(pred_conf, thresh=0.5):
    """The head of ``visualize`` with ``mask=None`` (models/ssd_model.py:479-488):
    returns (pred_score f32[b,A], pred_cls int64[b,A], mask bool[b,A])."""
    pc = np.ascontiguousarray(np.asarray(pred_conf, dtype=np.float32)) if not D.is_device(pred_conf) else pred_conf
    b, a, c = pc.shape
    dummy_box = D.empty((b, a, 4), np.float32).zero_()
    dummy_pri = D.to_device(np.tile(np.array([[0.5, 0.5, 1.0, 1.0]]), (a, 1)))
    out = ops.detect(pc, dummy_box, dummy_pri, score_thresh=2.0, top_k=1, head_thresh=float(thresh))
    return (out["head_score"].to_host(), out["head_cls"].to_host().astype(np.int64),
            out["head_mask"].to_host().astype(bool))


def detect(pred_conf, pred_bbox, prior_box, score_thresh=0.01, top_k=200, iou_thresh=0.45, return_aux=False):
    """Decode (models/ssd_model.py:466-467, relative units) + softmax + per-class NMS.
    Returns (kept int32[b,C-1,top_k] padded with -1, counts int32[b,C-1])."""
    out = ops.detect(pred_conf, pred_bbox, prior_box, score_thresh, top_k, iou_thresh,
                     want_scores=return_aux, want_boxes=return_aux, want_probs=return_aux)
    kept, count = out["kept"].to_host(), out["count"].to_host()
    if return_aux:
        return kept, count, dict(kept_score=out["kept_score"].to_host(), boxes=out["boxes"].to_host(),
                                 probs=out["probs"].to_host())
    return kept, count


def detections(pred_conf, pred_bbox, prior_box, score_thresh=0.01, top_k=200, iou_thresh=0.45, keep_top_k=200):
    """The final detections of every image: decode + softmax + per-class NMS, then the lists ranked across classes
    (score desc, class asc) and capped at ``keep_top_k`` on the device -- what ``visualize`` (models/ssd_model.py:477-490)
    draws, with NMS and a per-image cap.  Returns host arrays {"boxes": f32[b,K,4] decoded cxcywh (relative units),
    "scores": f32[b,K], "labels": i32[b,K], "priors": i32[b,K], "n": i32[b]}; slots past n are -1 / 0."""
    det = ops.detect(pred_conf, pred_bbox, prior_box, score_thresh, top_k, iou_thresh, want_scores=True,
                     want_boxes=True)
    top = ops.keep_top_k(det, keep_top_k)
    return {"boxes": top["box"].to_host(), "scores": top["score"].to_host(), "labels": top["class"].to_host(),
            "priors": top["prior"].to_host(), "n": top["n"].to_host()}


def nms(probs, boxes, score_thresh=0.01, top_k=200, iou_thresh=0.45):
    """Per-class NMS on given probabilities f32[b,A,C] and decoded boxes f32[b,A,4]."""
    out = ops.nms(np.ascontiguousarray(np.asarray(probs, dtype=np.float32)) if not D.is_device(probs) else probs,
                  np.ascontiguousarray(np.asarray(boxes, dtype=np.float32)) if not D.is_device(boxes) else boxes,
                  score_thresh, top_k, iou_thresh)
    return out["kept"].to_host(), out["count"].to_host()


class SSDBoxGeometry:
    """The box-geometry state and methods of ``SSDObjectDetectionModel``: priors built once
    (``__init__`` -> ``_build`` -> ``_build_prior_box``, models/ssd_model.py:60,164), then the
    per-batch target assigner, loss and post-processing against them."""

    def __init__(self, classes=80, table=None, thresh=0.5):
        table = SSD300 if table is None else table
        self.classes = classes + 1                      # Config.classes, models/ssd_model.py:47
        self.thresh = thresh                            # Config.thresh, :48
        self.input_size = table["input_size"]
        self._prior_dev = ops.prior_boxes(table["sizes"], table["s_k_refer"], table["aspect_ratio"], table["input_size"])
        ops.prior_index(self._prior_dev)                # matcher acceleration index, built once
        self._prior_box = None

    def _build_prior_box(self, size_list):
        return build_prior_box(size_list, input_size=self.input_size)

    def get_prior_box(self):
        if self._prior_box is None:
            self._prior_box = self._prior_dev.to_host()
        return self._prior_box

    def assign(self, gt_boxes, gt_cls, gt_offsets, device_out=False, stream=None):
        """The generator body of ``get_train_set`` (:211-215) for one batch of CSR ground truth."""
        return match_encode_batch(gt_boxes, gt_cls, gt_offsets, self._prior_dev, self.thresh, device_out, stream)

    @staticmethod
    def _ssd_loss(y_true, y_pred):
        return ssd_loss(y_true, y_pred)

    def detect(self, pred_conf, pred_bbox, score_thresh=0.01, top_k=200, iou_thresh=0.45):
        return detect(pred_conf, pred_bbox, self._prior_dev, score_thresh, top_k, iou_thresh)

    def detections(self, pred_conf, pred_bbox, score_thresh=0.01, top_k=200, iou_thresh=0.45, keep_top_k=200):
        return detections(pred_conf, pred_bbox, self._prior_dev, score_thresh, top_k, iou_thresh, keep_top_k)

    def visualize_scores(self, pred_conf, thresh=0.5):
        return score_head(pred_conf, thresh)


def evaluate_detections(kept, count, kept_score, boxes, gt_boxes, gt_cls, gt_offsets, max_dets=100,
                        iou_thresholds=None, recall_thresholds=None) -> dict:
    """COCO-style AP of one set of host detections (``detect(..., return_aux=True)``: kept, count, kept_score and
    the decoded boxes) against CSR ground truth (relative cxcywh, class ids as float32), evaluated on the device.
    Returns {"AP", "AP50", "AP75", "AR", "per_class_AP", "precision", "recall", "n_gt", "n_det"}."""
    from ..evaluate import DetectionEvaluator
    kept = np.ascontiguousarray(kept, np.int32)
    b, k, _ = kept.shape
    ev = DetectionEvaluator(n_classes=k + 1, max_images=b, max_dets=max_dets, iou_thresholds=iou_thresholds,
                            recall_thresholds=recall_thresholds)
    det = {"kept": kept, "count": np.ascontiguousarray(count, np.int32),
           "kept_score": np.ascontiguousarray(kept_score, np.float32), "boxes": np.ascontiguousarray(boxes, np.float32)}
    ev.add(det, np.ascontiguousarray(gt_boxes, np.float32), np.ascontiguousarray(gt_cls, np.float32),
           np.ascontiguousarray(gt_offsets, np.int32), image_base=0)
    return ev.summarize()
