"""Thin, allocation-explicit Python wrappers over the C ABI (include/ssdgeom.h).  Everything
here works on device memory (``device.DeviceArray`` or any ``__cuda_array_interface__`` object)
and is asynchronous on the given stream.  The reference-named drop-ins live in
``ssdgeom.utils.bbox`` and ``ssdgeom.models.ssd_model``."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as N
from . import device as D
from .parallel import loss_from_sums

_DT = {np.dtype(np.float32): N.F32, np.dtype(np.float64): N.F64}


def _code(dtype) -> int:
    try:
        return _DT[np.dtype(dtype)]
    except KeyError:
        raise TypeError("boxes must be float32 or float64, got %s" % dtype)


class WorkspacePool:
    """Grow-only device scratch, one buffer per kernel family so families can overlap on different streams.
    A pool belongs to ONE owner that enqueues its calls of a family in stream order: every ``HotPath`` and every
    ``StagedLoss`` has its own (pass ``pool=``); the module-level default ``POOL`` serves the stand-alone,
    one-call-at-a-time drop-ins and keeps a separate buffer per CUDA device."""

    def __init__(self):
        self._buf = {}

    def get(self, kind: str, nbytes: int) -> D.DeviceArray:
        key = (D.current_device(), kind)
        cur = self._buf.get(key)
        if cur is None or cur.nbytes < nbytes:
            cur = D.empty((int(nbytes) + 255) // 256 * 256, np.uint8)
            self._buf[key] = cur
        return cur

    def peek(self, kind: str):
        return self._buf.get((D.current_device(), kind))


POOL = WorkspacePool()


def _p(x):
    return None if x is None else x.ptr


# ---- A1 ------------------------------------------------------------------------------------------
def prior_boxes(size_list, s_k_refer, aspect_ratio, input_size=300, stream=None, clip=False) -> D.DeviceArray:
    """models/ssd_model.py:173-194 with the tables lifted to arguments; float64 [A,4] on the device.
    clip=True clamps every component to [0,1] (not in the reference; SURVEY.md section 8f row 4)."""
    n = len(size_list)
    if len(s_k_refer) != n + 1 or len(aspect_ratio) != n:
        raise ValueError("need len(s_k_refer) == len(size_list)+1 and one ratio list per level")
    fh = (C.c_int32 * n)(*[int(s[0]) for s in size_list])
    fw = (C.c_int32 * n)(*[int(s[1]) for s in size_list])
    sk = (C.c_double * (n + 1))(*[float(v) for v in s_k_refer])
    offs = [0]
    flat = []
    for r in aspect_ratio:
        flat += [float(v) for v in r]
        offs.append(len(flat))
    ro = (C.c_int32 * (n + 1))(*offs)
    rr = (C.c_double * max(len(flat), 1))(*flat)
    lib = N.lib()
    count = lib.ssdg_prior_count(fh, fw, ro, n)
    if count <= 0:
        N.check(int(count) if count < 0 else N.ERR_ARG, "prior_count")
    out = D.empty((count, 4), np.float64)
    N.check(lib.ssdg_prior_boxes(fh, fw, sk, ro, rr, n, float(input_size), out.ptr, count, D.stream_handle(stream)),
            "prior_boxes")
    if clip:
        N.check(lib.ssdg_priors_clip(out.ptr, _code(out.dtype), count, D.stream_handle(stream)), "priors_clip")
    return out


def loc_scale(loc, scale_xy, scale_wh, out=None, stream=None) -> D.DeviceArray:
    """Encoded offsets times (sxy, sxy, swh, swh): 1/variance after encoding, variance before decoding."""
    loc = D.as_device(loc, np.float32)
    out = D.empty(loc.shape, np.float32) if out is None else out
    N.check(N.lib().ssdg_loc_scale(loc.ptr, out.ptr, loc.size // 4, float(scale_xy), float(scale_wh),
                                   D.stream_handle(stream)), "loc_scale")
    out._keep = (loc,)
    return out


# ---- A3 + A4 + A5 ----------------------------------------------------------------------------------
def prior_index(priors, stream=None) -> D.DeviceArray:
    """Build (once per prior set; synchronises) the matcher's acceleration index for device priors and
    cache it on the array object.  It changes no result."""
    priors = D.as_device(priors)
    cached = getattr(priors, "_ssdg_index", None)
    if cached is not None:
        return cached
    lib = N.lib()
    a = int(priors.shape[0])
    idx = PriorIndex((int(lib.ssdg_prior_index_bytes(a)) + 255) // 256 * 256, np.uint8)
    N.check(lib.ssdg_prior_index_build(priors.ptr, _code(priors.dtype), a, idx.ptr, idx.nbytes, D.stream_handle(stream)),
            "prior_index_build")
    idx._built = True
    priors._ssdg_index = idx          # (the index does not keep the priors alive: the priors own the index)
    return idx


class PriorIndex(D.DeviceArray):
    """Device memory of a matcher index; unregisters itself from the library before the memory is freed."""
    _built = False

    def __del__(self):
        try:
            if self._built and self.ptr:
                N.lib().ssdg_prior_index_destroy(self.ptr)
        except Exception:
            pass
        D.DeviceArray.__del__(self)


def match_encode(gt_boxes, gt_cls, gt_offsets, priors, batch: int, max_gt: int, thresh: float = 0.5,
                 want=("cls", "loc", "mask"), out=None, stream=None, index=None, pool=None) -> dict:
    """Batched match_bbox + apply_anchor_box (utils/bbox.py:44-101, models/ssd_model.py:211-224).
    ``want`` selects outputs among cls, box, loc, mask, match; ``out`` may carry preallocated arrays."""
    gt_boxes, priors = D.as_device(gt_boxes), D.as_device(priors)
    gt_cls = D.as_device(gt_cls, np.float32)
    gt_offsets = D.as_device(gt_offsets, np.int32)
    a = int(priors.shape[0])
    out = dict(out or {})
    spec = {"cls": ((batch, a), np.int32), "box": ((batch, a, 4), np.float32), "loc": ((batch, a, 4), np.float32),
            "mask": ((batch, a), np.uint8), "match": ((batch, a), np.int32)}
    for k in want:
        if k not in out:
            out[k] = D.empty(*spec[k])
    lib = N.lib()
    nbytes = lib.ssdg_match_workspace_bytes(batch, a, max_gt)
    ws = (pool or POOL).get("match", nbytes)
    if index is None:
        index = getattr(priors, "_ssdg_index", None)     # built by prior_index() for long-lived prior sets
    N.check(lib.ssdg_match_encode(gt_boxes.ptr, _code(gt_boxes.dtype), gt_cls.ptr, gt_offsets.ptr, priors.ptr,
                                  _code(priors.dtype), _p(index), batch, a, int(max_gt), float(thresh),
                                  _p(out.get("cls")), _p(out.get("box")), _p(out.get("loc")), _p(out.get("mask")),
                                  _p(out.get("match")), ws.ptr, ws.nbytes, D.stream_handle(stream)), "match_encode")
    out["_keep"] = (gt_boxes, gt_cls, gt_offsets, priors, ws)
    out["_match_ws"] = ws
    return out


MATCH_STATUS_TOO_MANY_GT, MATCH_STATUS_MORE_GT_THAN_PRIORS, MATCH_STATUS_RESCAN, MATCH_STATUS_STALE_INDEX = 1, 2, 4, 8


def match_status(out, stream=None) -> int:
    """Status bits of the ``match_encode`` call that returned ``out`` (synchronises): see ssdg_match_status."""
    st = C.c_int32(0)
    ws = out["_match_ws"] if isinstance(out, dict) else out
    N.check(N.lib().ssdg_match_status(ws.ptr, C.byref(st), D.stream_handle(stream)), "match_status")
    return st.value


def raise_for_match_status(status: int):
    """The reference matches every ground-truth box or asserts (utils/bbox.py:50): images the device had to skip
    are an error, not a silent all-unmatched result."""
    status = int(status)
    if status & MATCH_STATUS_MORE_GT_THAN_PRIORS:
        raise AssertionError("number of default boxes should greater than the number of targets")   # utils/bbox.py:50
    if status & MATCH_STATUS_TOO_MANY_GT:
        raise ValueError("an image has more ground-truth boxes than max_gt: its targets were not assigned")
    if status & MATCH_STATUS_STALE_INDEX:
        raise N.SsdgeomError("the prior index was not built from these priors (modified after prior_index()?)")


def gt_prepare(xywh, img_wh, gt_offsets, out=None, stream=None) -> D.DeviceArray:
    """COCO pixel [x,y,w,h] rows of a batch -> relative cxcywh float32 (data_loaders/coco/make_dataset.py:132,
    data_loaders/ssd/make_dataset.py:43-44)."""
    xywh = D.as_device(xywh)
    if xywh.dtype not in (np.float32, np.float64):
        raise AssertionError("annotation boxes must be float32 or float64")
    img_wh, gt_offsets = D.as_device(img_wh, np.int32), D.as_device(gt_offsets, np.int32)
    rows = xywh.size // 4
    b = gt_offsets.size - 1
    if img_wh.size != 2 * b:
        raise AssertionError("img_wh must be [B,2]")
    out = D.empty((rows, 4), np.float32) if out is None else out
    N.check(N.lib().ssdg_gt_prepare(xywh.ptr, _code(xywh.dtype), img_wh.ptr, gt_offsets.ptr, b, rows, out.ptr,
                                    D.stream_handle(stream)), "gt_prepare")
    out._keep = (xywh, img_wh, gt_offsets)
    return out


def image_normalize(images, out=None, stream=None) -> D.DeviceArray:
    """(image - 0.5) * 2, float32 (models/ssd_model.py:214)."""
    images = D.as_device(images, np.float32)
    out = D.empty(images.shape, np.float32) if out is None else out
    N.check(N.lib().ssdg_image_normalize(images.ptr, out.ptr, images.size, D.stream_handle(stream)), "image_normalize")
    out._keep = (images,)
    return out


def encode(boxes, priors, out_dtype=np.float32, stream=None) -> D.DeviceArray:
    boxes, priors = D.as_device(boxes), D.as_device(priors)
    a = int(priors.shape[0])
    n = boxes.size // 4
    if n % a:
        raise AssertionError("boxes and priors disagree in shape")  # utils/bbox.py:95
    out = D.empty(boxes.shape, out_dtype)
    N.check(N.lib().ssdg_encode(boxes.ptr, _code(boxes.dtype), priors.ptr, _code(priors.dtype), n // a, a, out.ptr,
                                _code(out_dtype), D.stream_handle(stream)), "encode")
    out._keep = (boxes, priors)
    return out


def decode(loc, priors, scale=300.0, stream=None) -> D.DeviceArray:
    loc, priors = D.as_device(loc, np.float32), D.as_device(priors)
    a = int(priors.shape[0])
    n = loc.size // 4
    if n % a:
        raise AssertionError("loc and priors disagree in shape")
    out = D.empty(loc.shape, np.float32)
    N.check(N.lib().ssdg_decode(loc.ptr, priors.ptr, _code(priors.dtype), n // a, a, float(scale), out.ptr,
                                D.stream_handle(stream)), "decode")
    out._keep = (loc, priors)
    return out


def iou_pairs(boxes_1, boxes_2, use_eps_clamp: bool, stream=None) -> D.DeviceArray:
    b1, b2 = D.as_device(boxes_1), D.as_device(boxes_2)
    n = b1.size // 4
    if b2.size // 4 != n:
        raise ValueError("paired IoU needs equally many rows")
    odt = np.float32 if (b1.dtype == np.float32 and b2.dtype == np.float32) else np.float64
    out = D.empty((n,), odt)
    N.check(N.lib().ssdg_iou_pairs(b1.ptr, _code(b1.dtype), b2.ptr, _code(b2.dtype), n, int(bool(use_eps_clamp)),
                                   out.ptr, D.stream_handle(stream)), "iou_pairs")
    out._keep = (b1, b2)
    return out


# ---- A6 ----------------------------------------------------------------------------------------------
def _loss_operands(gt_cls, gt_box, gt_mask, pred_box, pred_cls, want_neg_mask, want_neg_ce, want_grad, out, pool,
                   ws_kind):
    """The five operands as device arrays, the output dict (caller-supplied arrays, torch tensors included, are
    used as they are; missing wanted ones are allocated) and the workspace."""
    gt_cls = D.as_device(gt_cls, np.int32)
    gt_box = D.as_device(gt_box, np.float32)
    gt_mask = D.as_device(gt_mask, np.uint8)
    pred_box = D.as_device(pred_box, np.float32)
    pred_cls = D.as_device(pred_cls, np.float32)
    if len(pred_cls.shape) != 3:
        raise AssertionError("pred_cls must be [B,A,C]")
    b, a, c = pred_cls.shape
    # models/ssd_model.py:347-351
    if not (gt_cls.size == b * a and gt_mask.size == b * a and gt_box.size == b * a * 4 and pred_box.size == b * a * 4):
        raise AssertionError("y_true / y_pred disagree in shape")
    out = {k: (D.as_device(v) if D.is_device(v) else v) for k, v in (out or {}).items()}   # torch tensors etc.: zero-copy views
    if "result" not in out:
        out["result"] = D.empty((N.LOSS_RESULT_LEN,), np.float64)
    if want_neg_mask and "neg_mask" not in out:
        out["neg_mask"] = D.empty((b, a), np.uint8)
    if want_neg_ce and "neg_ce" not in out:
        out["neg_ce"] = D.empty((b, a), np.float32)
    if want_grad:
        if "grad_box" not in out:
            out["grad_box"] = D.empty((b, a, 4), np.float32)
        if "grad_cls" not in out:
            out["grad_cls"] = D.empty((b, a, c), np.float32)
    ws = pool.get(ws_kind, N.lib().ssdg_loss_workspace_bytes(b, a, c))
    return (gt_cls, gt_box, gt_mask, pred_box, pred_cls), out, ws


def _loss_args(x, neg_ratio, out, ws, stream) -> tuple:
    """The arguments every loss entry point ends with (ssdg_multibox_loss's)."""
    gt_cls, gt_box, gt_mask, pred_box, pred_cls = x
    b, a, c = pred_cls.shape
    return (gt_cls.ptr, gt_box.ptr, gt_mask.ptr, pred_box.ptr, pred_cls.ptr, b, a, c, int(neg_ratio),
            out["result"].ptr, _p(out.get("neg_mask")), _p(out.get("neg_ce")), _p(out.get("grad_box")),
            _p(out.get("grad_cls")), ws.ptr, ws.nbytes, D.stream_handle(stream))


def multibox_loss(gt_cls, gt_box, gt_mask, pred_box, pred_cls, neg_ratio: int = 3, want_neg_mask=False,
                  want_neg_ce=False, want_grad=False, out=None, stream=None, ws_kind="loss", row_stats=None,
                  pool=None) -> dict:
    """models/ssd_model.py:341-396.  Returns {'result': float64[16] device block, ...}; see
    include/ssdgeom.h for the block layout.  row_stats = (row_ml, row_negbg) from ``detect(..., want_row_stats=True)``
    on the same pred_cls: the loss then skips its own pass over the logits (ssdg_multibox_loss_fused)."""
    x, out, ws = _loss_operands(gt_cls, gt_box, gt_mask, pred_box, pred_cls, want_neg_mask, want_neg_ce, want_grad,
                                out, pool or POOL, ws_kind)
    args = _loss_args(x, neg_ratio, out, ws, stream)
    if row_stats is None:
        N.check(N.lib().ssdg_multibox_loss(*args), "multibox_loss")
    else:
        b, a, _ = x[4].shape
        row_ml, row_negbg = row_stats
        if row_ml.size != 2 * b * a or row_negbg.size != b * a:
            raise AssertionError("row statistics disagree with pred_cls in shape")
        N.check(N.lib().ssdg_multibox_loss_fused(row_ml.ptr, row_negbg.ptr, *args), "multibox_loss_fused")
    out["_keep"] = (*x, ws)
    return out


def loss_result_words(result, words: slice) -> D.DeviceArray:
    """Device view of the words ``words`` (N.LOSS_*) of a loss result block, e.g. to sum them over the shards."""
    return D.DeviceArray((words.stop - words.start,), np.float64, ptr=result.ptr + words.start * 8, owner=result)


class StagedLoss:
    """The multibox loss of one shard of a batch whose hard-negative threshold is mined over ALL shards
    (include/ssdgeom.h, ssdg_multibox_loss_stage).  Usage, on every shard:

        sl = StagedLoss(gt_cls, gt_box, gt_mask, pred_box, pred_cls, global_priors=sum of b*A over shards)
        for stage in range(sl.n_stages):        # 4, or 5 with want_grad (the gradient runs AFTER the last exchange)
            sl.run(stage)
            for buf in sl.exchange(stage):      # device buffers (int32 / int64 / float64)
                <sum buf over the shards, in place>
        total, info = sl.finish()

    The buffers are DeviceArrays over the workspace / result block, so a torch.distributed all_reduce on
    torch.as_tensor(buf) works in place without a copy.  Arrays passed in ``out`` are written in place."""

    def __init__(self, gt_cls, gt_box, gt_mask, pred_box, pred_cls, global_priors: int, neg_ratio: int = 3,
                 want_neg_mask=False, want_neg_ce=False, want_grad=False, stream=None, ws_kind="loss_staged", out=None,
                 row_stats=None, pool=None):
        self.pool = pool or WorkspacePool()        # never shared: the stages keep state in the workspace
        x, self.out, self.ws = _loss_operands(gt_cls, gt_box, gt_mask, pred_box, pred_cls, want_neg_mask,
                                              want_neg_ce, want_grad, out, self.pool, ws_kind)
        self.gt_cls, self.gt_box, self.gt_mask, self.pred_box, self.pred_cls = x
        self.shape = self.pred_cls.shape
        self.global_priors = int(global_priors)
        self.row_stats = row_stats          # (row_ml, row_negbg) of detect(..., want_row_stats=True), or None
        self.neg_ratio = int(neg_ratio)
        self.stream = stream
        self._xb = {}
        self.n_stages = 5 if want_grad else 4

    def run(self, stage: int):
        rs = self.row_stats or (None, None)
        x = (self.gt_cls, self.gt_box, self.gt_mask, self.pred_box, self.pred_cls)
        N.check(N.lib().ssdg_multibox_loss_stage(int(stage), self.global_priors, _p(rs[0]), _p(rs[1]),
                                                 *_loss_args(x, self.neg_ratio, self.out, self.ws, self.stream)),
                "multibox_loss_stage")

    def _xbuf(self, which: int, dtype):
        ptr, cnt = C.c_void_p(), C.c_int64()
        N.check(N.lib().ssdg_loss_exchange(self.ws.ptr, which, C.byref(ptr), C.byref(cnt)), "loss_exchange")
        return D.DeviceArray((int(cnt.value),), dtype, ptr=ptr.value, owner=self.ws)

    def exchange(self, stage: int):
        """Buffers to sum over the shards after `stage` (in place)."""
        if stage not in self._xb:
            self._xb[stage] = self._exchange(stage)
        return self._xb[stage]

    def _exchange(self, stage: int):
        if stage == 0:
            return [self._xbuf(3, np.int64), self._xbuf(0, np.int32)]
        if stage in (1, 2):
            return [self._xbuf(stage, np.int32)]
        if stage == 4:
            return []
        r = self.out["result"]
        # the separable sums, the shard's own positives, its data-dependent error count and its mined negatives
        return [loss_result_words(r, slice(N.LOSS_SUM_POS_CE, N.LOSS_ERRORS + 1)),
                loss_result_words(r, slice(N.LOSS_NUM_NEG, N.LOSS_NUM_NEG + 1))]

    def finish(self) -> tuple:
        """After the stage-3 exchange: (total, info) of the whole batch, identical on every shard."""
        r = self.out["result"].to_host(self.stream)
        d = decode_loss_result(r, "multibox_loss_stage")
        # some shard mined a positive (models/ssd_model.py:375) or saw a class id out of range
        if r[N.LOSS_ERRORS] != 0:
            raise AssertionError("a shard of the batch reported %d positives mined as negatives / class ids out of "
                                 "range" % int(r[N.LOSS_ERRORS]))
        n_pos = r[N.LOSS_OWN_POS]      # summed over the shards: the positives of the batch
        total, info = loss_from_sums(d["sum_pos_ce"], d["sum_neg_ce"], d["sum_l1"], n_pos, r[N.LOSS_NUM_NEG])
        info.update(num_pos=int(n_pos), num_neg=d["num_neg"], kth=d["kth"])
        return total, info


def decode_loss_result(r, what: str = "multibox_loss") -> dict:
    """A loss result block on the host as a dict; raises like the reference on the device-side guards
    (num_pos == 0 -> IndexError at models/ssd_model.py:369; k out of range -> top_k error)."""
    status = int(r[N.LOSS_STATUS])
    if status == N.ERR_NO_POSITIVE:
        raise IndexError("no positive prior in the batch: hard-negative top-k is empty (models/ssd_model.py:369)")
    if status == N.ERR_TOPK_RANGE:
        raise ValueError("3*num_pos exceeds the number of priors in the batch (tf.math.top_k, models/ssd_model.py:368)")
    N.check(status, what)
    return {"total": r[N.LOSS_TOTAL], "cls loss pos": r[N.LOSS_POS], "cls loss neg": r[N.LOSS_NEG],
            "loc loss": r[N.LOSS_LOC], "num_pos": int(r[N.LOSS_NUM_POS]), "num_neg": int(r[N.LOSS_NUM_NEG]),
            "kth": r[N.LOSS_KTH], "sum_pos_ce": r[N.LOSS_SUM_POS_CE], "sum_neg_ce": r[N.LOSS_SUM_NEG_CE],
            "sum_l1": r[N.LOSS_SUM_L1]}


def loss_result_to_host(result: D.DeviceArray, stream=None) -> dict:
    """One synchronising read of the result block, decoded by ``decode_loss_result``."""
    return decode_loss_result(result.to_host(stream))


# ---- A7 + A8 + A9 ---------------------------------------------------------------------------------------
def detect(pred_cls, pred_box, priors, score_thresh=0.01, top_k=200, iou_thresh=0.45, want_scores=False,
           want_boxes=False, want_probs=False, head_thresh=None, out=None, stream=None, stage=None,
           want_row_stats=False, pool=None) -> dict:
    """stage: None = the whole post-processing; 0 = filter + decode + candidate lists only; 1 = the NMS of a previous
    stage-0 call with the same arguments (include/ssdgeom.h, ssdg_detect_stage)."""
    pred_cls = D.as_device(pred_cls, np.float32)
    pred_box = D.as_device(pred_box, np.float32)
    priors = D.as_device(priors)
    b, a, c = pred_cls.shape
    if pred_box.size != b * a * 4 or priors.shape[0] != a:
        raise AssertionError("pred_cls / pred_box / priors disagree in shape")
    out = dict(out or {})

    def need(key, shape, dtype):
        if key not in out:            # never dict.setdefault here: it would allocate (and free) eagerly
            out[key] = D.empty(shape, dtype)

    need("kept", (b, c - 1, top_k), np.int32)
    need("count", (b, c - 1), np.int32)
    if want_scores:
        need("kept_score", (b, c - 1, top_k), np.float32)
    if want_boxes:
        need("boxes", (b, a, 4), np.float32)
    if want_probs:
        need("probs", (b, a, c), np.float32)
    if want_row_stats:           # per-prior softmax statistics for multibox_loss(row_stats=...)
        need("row_ml", (b, a, 2), np.float32)
        need("row_negbg", (b, a), np.float32)
    if head_thresh is not None:
        need("head_score", (b, a), np.float32)
        need("head_cls", (b, a), np.int32)
        need("head_mask", (b, a), np.uint8)
    lib = N.lib()
    ws = (pool or POOL).get("detect", lib.ssdg_detect_workspace_bytes(b, a, c, top_k))
    args = (pred_cls.ptr, pred_box.ptr, priors.ptr, _code(priors.dtype), b, a, c, float(score_thresh),
            int(top_k), float(iou_thresh), out["kept"].ptr, out["count"].ptr, _p(out.get("kept_score")),
            _p(out.get("boxes")), _p(out.get("probs")),
            float(head_thresh if head_thresh is not None else 0.0), _p(out.get("head_score")),
            _p(out.get("head_cls")), _p(out.get("head_mask")))
    tail = (ws.ptr, ws.nbytes, D.stream_handle(stream))
    if stage is None and not want_row_stats:
        N.check(lib.ssdg_detect(*args, *tail), "detect")
    else:
        stats = (_p(out.get("row_ml")), _p(out.get("row_negbg"))) if want_row_stats else (None, None)
        for st in ((0, 1) if stage is None else (int(stage),)):
            N.check(lib.ssdg_detect_stage(st, *args, *stats, *tail), "detect_stage")
    out["_keep"] = (pred_cls, pred_box, priors, ws)
    return out


def nms(probs, boxes, score_thresh=0.01, top_k=200, iou_thresh=0.45, want_scores=False, stream=None) -> dict:
    probs = D.as_device(probs, np.float32)
    boxes = D.as_device(boxes, np.float32)
    b, a, c = probs.shape
    if boxes.size != b * a * 4:
        raise AssertionError("probs / boxes disagree in shape")
    out = {"kept": D.empty((b, c - 1, top_k), np.int32), "count": D.empty((b, c - 1), np.int32)}
    if want_scores:
        out["kept_score"] = D.empty((b, c - 1, top_k), np.float32)
    lib = N.lib()
    ws = POOL.get("detect", lib.ssdg_detect_workspace_bytes(b, a, c, top_k))
    N.check(lib.ssdg_nms(probs.ptr, boxes.ptr, b, a, c, float(score_thresh), int(top_k), float(iou_thresh),
                         out["kept"].ptr, out["count"].ptr, _p(out.get("kept_score")), ws.ptr, ws.nbytes,
                         D.stream_handle(stream)), "nms")
    out["_keep"] = (probs, boxes, ws)
    return out


# ---- A12 ------------------------------------------------------------------------------------------------
def keep_top_k(det: dict, keep_top_k: int, out=None, stream=None) -> dict:
    """The final detections of every image (include/ssdgeom.h, ssdg_detect_keep_top_k): the kept lists of a ``detect``
    / ``nms`` output with ``kept_score`` ranked across classes (score desc, class asc, position asc) and capped at
    ``keep_top_k``.  Returns device arrays prior i32[B,K], class i32[B,K], score f32[B,K], n i32[B] and count
    i32[B,C-1] (the survivors per class list, a prefix of each: ``dict(det, count=top["count"])`` is a capped
    detection output), plus box f32[B,K,4] when ``det`` has ``boxes``.  ``out`` may carry preallocated arrays."""
    if "kept_score" not in det:
        raise ValueError("detect output lacks 'kept_score': call ops.detect(..., want_scores=True)")
    kept, count = D.as_device(det["kept"], np.int32, stream), D.as_device(det["count"], np.int32, stream)
    kept_score = D.as_device(det["kept_score"], np.float32, stream)
    boxes = D.as_device(det["boxes"], np.float32, stream) if det.get("boxes") is not None else None
    if len(kept.shape) != 3:
        raise AssertionError("kept must be [B,C-1,top_k]")
    b, k, top_k = kept.shape
    if count.size != b * k or kept_score.size != kept.size or (boxes is not None and
                                                               (len(boxes.shape) != 3 or boxes.shape[0] != b)):
        raise AssertionError("kept, count, kept_score and boxes disagree in shape")
    kk = int(keep_top_k)
    out = dict(out or {})
    spec = {"prior": ((b, kk), np.int32), "class": ((b, kk), np.int32), "score": ((b, kk), np.float32),
            "n": ((b,), np.int32), "count": ((b, k), np.int32)}
    if boxes is not None:
        spec["box"] = ((b, kk, 4), np.float32)
    for key, (shape, dt) in spec.items():
        if key not in out:
            out[key] = D.empty(shape, dt)
    a = int(boxes.shape[1]) if boxes is not None else 0
    N.check(N.lib().ssdg_detect_keep_top_k(kept.ptr, count.ptr, kept_score.ptr, top_k, _p(boxes), b, a, k + 1, kk,
                                           out["prior"].ptr, out["class"].ptr, out["score"].ptr, _p(out.get("box")),
                                           out["n"].ptr, out["count"].ptr, D.stream_handle(stream)), "keep_top_k")
    out["_keep"] = (kept, count, kept_score, boxes)
    return out


# ---- A11 ------------------------------------------------------------------------------------------------
EVAL_STATUS_BAD_CLASS, EVAL_STATUS_TOO_MANY_GT, EVAL_STATUS_DUPLICATE, EVAL_STATUS_BAD_PRIOR = 1, 2, 4, 8


class EvalState(D.DeviceArray):
    """The device accumulator of the detection evaluation (include/ssdgeom.h, A11) with the sizes it was made for."""

    def __init__(self, n_classes: int, max_images: int, max_dets: int, n_thresholds: int):
        nbytes = int(N.lib().ssdg_eval_state_bytes(int(n_classes), int(max_images), int(max_dets), int(n_thresholds)))
        if nbytes == 0:
            raise ValueError("evaluation state out of range: n_classes >= 2, 0 < max_images < 2^22, "
                             "0 < max_dets <= 1024, 0 < n_thresholds <= 16, (n_classes-1)*max_images*max_dets < 2^31")
        super().__init__((nbytes,), np.uint8)
        self.n_classes, self.max_images = int(n_classes), int(max_images)
        self.max_dets, self.n_thresholds = int(max_dets), int(n_thresholds)


def eval_state(n_classes: int, max_images: int, max_dets: int = 100, n_thresholds: int = 10, stream=None) -> EvalState:
    st = EvalState(n_classes, max_images, max_dets, n_thresholds)
    eval_reset(st, stream)
    return st


def eval_reset(state: EvalState, stream=None):
    N.check(N.lib().ssdg_eval_reset(state.ptr, state.nbytes, D.stream_handle(stream)), "eval_reset")


def eval_accumulate(det: dict, gt_boxes, gt_cls, gt_offsets, state: EvalState, iou_thresholds, image_base: int,
                    max_gt: int, stream=None):
    """Match one batch of ``detect`` outputs (``kept``, ``count``, ``kept_score``, ``boxes``) to its ground truth
    (CSR, as ``match_encode``) and write the slots of global images ``image_base ..`` (ssdg_eval_accumulate)."""
    kept, count = D.as_device(det["kept"], np.int32, stream), D.as_device(det["count"], np.int32, stream)
    kept_score = D.as_device(det["kept_score"], np.float32, stream)
    boxes = D.as_device(det["boxes"], np.float32, stream)
    gt_boxes, gt_cls = D.as_device(gt_boxes, np.float32, stream), D.as_device(gt_cls, np.float32, stream)
    gt_offsets = D.as_device(gt_offsets, np.int32, stream)
    if len(kept.shape) != 3 or len(boxes.shape) != 3:
        raise AssertionError("kept must be [B,C-1,top_k] and boxes [B,A,4]")
    b, k, top_k = kept.shape
    if k + 1 != state.n_classes or count.size != b * k or kept_score.size != kept.size or boxes.shape[0] != b \
            or gt_offsets.size != b + 1:
        raise AssertionError("detections, ground truth and evaluation state disagree in shape")
    thr = np.ascontiguousarray(iou_thresholds, np.float64)
    if thr.size != state.n_thresholds:
        raise ValueError("the state was made for %d IoU thresholds" % state.n_thresholds)
    N.check(N.lib().ssdg_eval_accumulate(
        kept.ptr, count.ptr, kept_score.ptr, top_k, boxes.ptr, b, boxes.shape[1], state.n_classes, gt_boxes.ptr,
        gt_cls.ptr, gt_offsets.ptr, int(max_gt), thr.ctypes.data_as(C.POINTER(C.c_double)), thr.size, state.max_dets,
        int(image_base), state.max_images, state.ptr, state.nbytes, D.stream_handle(stream)), "eval_accumulate")
    return (kept, count, kept_score, boxes, gt_boxes, gt_cls, gt_offsets)     # keep-alives until the stream passes


def eval_exchange(state: EvalState) -> list:
    """The buffers a data-parallel caller sums over the ranks, in place: [int64 keys, int32 header/flags/GT counts]."""
    out = []
    for which, dt in ((0, np.int64), (1, np.int32)):
        ptr, cnt = C.c_void_p(), C.c_int64()
        N.check(N.lib().ssdg_eval_exchange(state.ptr, state.n_classes, state.max_images, state.max_dets, which,
                                           C.byref(ptr), C.byref(cnt)), "eval_exchange")
        out.append(D.DeviceArray((int(cnt.value),), dt, ptr=ptr.value, owner=state))
    return out


def eval_status(state: EvalState, stream=None) -> int:
    """Status bits of the state (synchronises): EVAL_STATUS_*."""
    st = C.c_int32(0)
    N.check(N.lib().ssdg_eval_status(state.ptr, C.byref(st), D.stream_handle(stream)), "eval_status")
    return st.value


def eval_finalize(state: EvalState, recall_thresholds, stream=None, pool=None) -> dict:
    """COCOeval.accumulate over everything accumulated: device precision f64[T,R,K], recall f64[T,K],
    n_gt i64[K], n_det i64[K].  The state is left unchanged."""
    rec = np.ascontiguousarray(recall_thresholds, np.float64)
    k, t, r = state.n_classes - 1, state.n_thresholds, rec.size
    out = {"precision": D.empty((t, r, k), np.float64), "recall": D.empty((t, k), np.float64),
           "n_gt": D.empty((k,), np.int64), "n_det": D.empty((k,), np.int64)}
    lib = N.lib()
    nbytes = int(lib.ssdg_eval_finalize_workspace_bytes(state.n_classes, state.max_images, state.max_dets))
    if nbytes == 0:
        raise N.SsdgeomError("eval_finalize: the workspace size query failed (no CUDA device?)")
    ws = (pool or POOL).get("eval_finalize", nbytes)
    N.check(lib.ssdg_eval_finalize(state.ptr, state.nbytes, state.n_classes, state.max_images, state.max_dets, t,
                                   rec.ctypes.data_as(C.POINTER(C.c_double)), r, out["precision"].ptr,
                                   out["recall"].ptr, out["n_gt"].ptr, out["n_det"].ptr, ws.ptr, ws.nbytes,
                                   D.stream_handle(stream)), "eval_finalize")
    out["_keep"] = (state, ws)
    return out
