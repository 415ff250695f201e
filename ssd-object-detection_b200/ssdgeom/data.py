"""Batched input glue between the reference's loaders and the device matcher (SURVEY.md section 8f, row 3).

The reference prepares ONE image at a time on a Python generator thread: COCO annotations
``[x, y, w, h]`` -> centre form (data_loaders/coco/make_dataset.py:132), relative coordinates
(data_loaders/ssd/make_dataset.py:43-44), then ``match_bbox`` + ``apply_anchor_box`` + ``(image - 0.5) * 2``
per image (models/ssd_model.py:211-215) and ``.batch(B, drop_remainder=True)`` (:225).  Here the same
arithmetic runs once per BATCH on the device; only ragged packing (lists -> CSR) stays on the host."""
from __future__ import annotations

import queue
import threading

import numpy as np

from . import device as D
from . import ops


def pack_gt(cls_list, box_list):
    """Per-image label / box arrays -> (cls float32 [sum T], boxes [sum T,4] in the boxes' dtype, offsets int32 [B+1]).
    Labels are float32 on input like the loaders' TensorSpecs (data_loaders/ssd/make_dataset.py:57)."""
    if len(cls_list) != len(box_list):
        raise AssertionError("one label array per box array")
    counts = []
    for c, b in zip(cls_list, box_list):
        b = np.asarray(b)
        n = 0 if b.size == 0 else b.reshape(-1, 4).shape[0]
        if np.asarray(c).size != n:
            raise AssertionError("labels and boxes disagree")      # utils/bbox.py:49-style shape contract
        counts.append(n)
    off = np.zeros(len(counts) + 1, np.int32)
    np.cumsum(counts, out=off[1:])
    dt = np.result_type(*[np.asarray(b).dtype for b in box_list]) if box_list else np.float32
    dt = np.float64 if dt == np.float64 else np.float32
    boxes = np.zeros((int(off[-1]), 4), dt)
    cls = np.zeros((int(off[-1]),), np.float32)
    for i, (c, b) in enumerate(zip(cls_list, box_list)):
        if counts[i]:
            boxes[off[i]:off[i + 1]] = np.asarray(b).reshape(-1, 4)
            cls[off[i]:off[i + 1]] = np.asarray(c).reshape(-1)
    return cls, boxes, off


def coco_to_ssd_boxes(xywh, img_wh, gt_offsets, stream=None) -> D.DeviceArray:
    """Pixel [x,y,w,h] rows -> relative cxcywh float32 on the device (ops.gt_prepare)."""
    return ops.gt_prepare(xywh, img_wh, gt_offsets, stream=stream)


class TrainBatches:
    """``get_train_set(dataset, batch_size)`` (models/ssd_model.py:209-227) with the per-image generator body
    replaced by one device call per batch.  ``source`` yields ``(image float32 [H,W,3] in [0,1], cls, box)``
    per image -- what SSDDataLoader / COCODataLoader yield; boxes are relative cxcywh unless
    ``coco_pixels=True``, in which case they are COCO pixel [x,y,w,h] and ``image_wh`` is taken from a
    fourth element of the tuple (w, h) or from the image itself.  Iterating yields
    ``(images [B,H,W,3], (cls int32 [B,A], loc float32 [B,A,4], mask bool [B,A]))`` as host arrays
    (``device=True``: DeviceArrays, mask uint8).  The trailing partial batch is dropped (:225).

    ``prefetch`` mirrors ``.prefetch(10)`` (:225): a producer thread packs, assigns and downloads up to that many
    batches ahead of the consumer on a stream of its own (the library releases the GIL inside its calls), so the
    assignment of batch k+1 overlaps whatever the training step does with batch k.  ``prefetch=0`` is synchronous.

    ``augment``: None, or a dict of ``ops.augment`` options (``seed`` among them, default 0) to apply the SSD training
    augmentation (zoom-out, min-IoU crop, flip) to every batch on the device: images and boxes are uploaded,
    (``gt_prepare``), augmented, normalised and matched.  Image ``k`` emitted by this iterator draws its random numbers
    at global index ``image_base + k``; give each data-parallel rank its own ``image_base`` range."""

    def __init__(self, source, priors, batch_size=1, thresh=0.5, coco_pixels=False, device=False, stream=None,
                 prefetch=10, augment=None, image_base=0):
        self.source, self.batch_size, self.thresh = source, int(batch_size), float(thresh)
        self.priors = D.as_device(priors)
        ops.prior_index(self.priors)
        self.coco_pixels, self.device, self.stream = bool(coco_pixels), bool(device), stream
        self.prefetch = int(prefetch)
        self.pool = ops.WorkspacePool()      # this iterator's own matcher scratch (its calls are in stream order)
        self.augment = None if augment is None else dict(augment)
        self.seed = self.augment.pop("seed", 0) if augment is not None else None
        self.image_base = int(image_base)

    def _emit(self, images, cls_list, box_list, wh):
        cls, boxes, off = pack_gt(cls_list, box_list)
        b = len(images)
        if self.coco_pixels:
            d_boxes = ops.gt_prepare(boxes, np.asarray(wh, np.int32).reshape(b, 2), off, stream=self.stream)
        else:
            d_boxes = D.as_device(boxes.astype(np.float32, copy=False), np.float32)
        max_gt = int(np.diff(off).max()) if b else 0
        img = np.stack(images).astype(np.float32, copy=False)
        if self.augment is not None:
            # rows are only dropped, so max_gt still bounds every image of the augmented batch
            aug = ops.augment(img, d_boxes, cls, off, self.seed, self.image_base, max_gt=max_gt, stream=self.stream,
                              **self.augment)
            self.image_base += b
            img = ops.image_normalize(aug["images"], stream=self.stream)
            d_boxes, cls, off = aug["boxes"], aug["cls"], aug["offsets"]
        tgt = ops.match_encode(d_boxes, cls, off, self.priors, b, max(max_gt, 1), self.thresh, stream=self.stream,
                               pool=self.pool)
        if self.augment is None:
            img = ops.image_normalize(img, stream=self.stream)
        if self.device:
            ops.raise_for_match_status(ops.match_status(tgt, self.stream))      # synchronises: the batch is ready
            return img, (tgt["cls"], tgt["loc"], tgt["mask"])
        return img.to_host(self.stream), (tgt["cls"].to_host(self.stream), tgt["loc"].to_host(self.stream),
                                          tgt["mask"].to_host(self.stream).astype(bool))

    def __iter__(self):
        if self.prefetch <= 0:
            yield from self._batches()
            return
        if self.stream is None:
            self.stream = D.Stream()         # not the legacy default stream: it would serialise with the consumer
        q, stop, done = queue.Queue(maxsize=self.prefetch), threading.Event(), object()

        def put(item):                       # never blocks forever: an abandoned consumer sets `stop`
            while not stop.is_set():
                try:
                    q.put(item, timeout=0.1)
                    return True
                except queue.Full:
                    continue
            return False

        def produce():
            try:
                for batch in self._batches():
                    if not put(batch):
                        return
                put(done)
            except BaseException as e:       # surfaces in the consumer, like an error inside the tf.data generator
                put(e)

        t = threading.Thread(target=produce, name="ssdgeom-train-batches", daemon=True)
        t.start()
        try:
            while True:
                item = q.get()
                if item is done:
                    return
                if isinstance(item, BaseException):
                    raise item
                yield item
        finally:
            stop.set()

    def _batches(self):
        images, cls_list, box_list, wh = [], [], [], []
        for item in self.source:
            image, cls, box = item[0], item[1], item[2]
            image = np.asarray(image)
            images.append(image); cls_list.append(np.asarray(cls)); box_list.append(np.asarray(box))
            wh.append(tuple(item[3]) if len(item) > 3 else (image.shape[1], image.shape[0]))
            if len(images) == self.batch_size:
                yield self._emit(images, cls_list, box_list, wh)
                images, cls_list, box_list, wh = [], [], [], []
