"""The chained hot path (target assignment -> multibox loss, and decode -> per-class NMS) with
preallocated buffers and explicit streams: the call a data-parallel trainer/evaluator makes per
batch.  The two branches only share the predictions, so they run on separate streams: the
matcher is latency-bound and the loss/filter passes are HBM-bound, so they overlap."""
from __future__ import annotations

import numpy as np

from . import _native as N
from . import device as D
from . import ops
from .models.ssd_model import SSD300

INPUT_NAMES = ("gt_boxes", "gt_cls", "gt_off", "pred_cls", "pred_box")


class HotPath:
    def __init__(self, table=None, batch=256, max_gt=100, classes=81, thresh=0.5, neg_ratio=3,
                 score_thresh=0.01, top_k=200, iou_thresh=0.45, total_gt=None, mining="shard", global_priors=None,
                 allreduce=None, comm=None, depth=1, evaluator=None, keep_top_k=None):
        """depth: steps in flight.  1 -- ``step()`` joins both branches on ``s_main`` before it returns the stream to
        the caller (a step is a closed unit).  2 -- every per-step buffer (targets, row statistics, candidate lists,
        workspaces, results) exists twice and consecutive steps use them in turn: step k+1 starts as soon as its
        inputs are there and the buffers of step k-1 are free, so its filter pass and row search run under the NMS
        and the loss tail of step k (independent batches: an evaluator, or a trainer's target / loss path);
        ``join()`` / ``download()`` wait for what they need.  Not with mining='global' or a caller-supplied
        ``loss_exchange``.

        mining: "shard" -- the hard-negative threshold is mined over this process's batch (what the reference
        does per slice under split_batch, models/ssd_model.py:235-256); "global" -- over the batches of all
        data-parallel processes (ops.StagedLoss; ``global_priors`` is the total number of priors over all of them).

        Data-parallel exchange: ``comm`` (ssdgeom.comm.Comm, the library's own NCCL entry points) sums the additive
        loss words -- or the mining histograms -- over the processes; alternatively ``allreduce(buf, stream)`` /
        ``loss_exchange(stream)`` callables (a torch.distributed or gloo stand-in) do.

        evaluator: an ``evaluate.DetectionEvaluator``; every step then also matches its kept lists to its ground truth
        (``step(image_base)``) after the NMS, on the NMS stream.  None (the default) changes nothing.

        keep_top_k: an int K in [1, 1024]; every step then also ranks the kept lists of each image across classes and
        keeps the first K (ops.keep_top_k) on the NMS stream, right after the NMS; ``download_detections`` copies them
        out.  An evaluator then matches the capped lists.  None (the default) changes nothing."""
        table = SSD300 if table is None else table
        self.batch, self.max_gt, self.classes = int(batch), int(max_gt), int(classes)
        self.thresh, self.neg_ratio = float(thresh), int(neg_ratio)
        self.score_thresh, self.top_k, self.iou_thresh = float(score_thresh), int(top_k), float(iou_thresh)
        self.priors = ops.prior_boxes(table["sizes"], table["s_k_refer"], table["aspect_ratio"], table["input_size"])
        self.A = a = int(self.priors.shape[0])
        ops.prior_index(self.priors)                     # one-off, like the priors themselves
        b, c = self.batch, self.classes
        n_gt = int(total_gt if total_gt is not None else b * self.max_gt)
        self.total_gt = n_gt
        self._sets = [self._alloc_inputs()]
        self._bind(self._sets[0])
        self.depth = 1 if mining == "global" else max(1, int(depth))
        self._n_steps = 0
        self.evaluator = evaluator
        if evaluator is not None and (evaluator.n_classes != c or evaluator.max_dets > self.top_k):
            raise ValueError("the evaluator needs n_classes == classes and max_dets <= top_k")
        if keep_top_k is not None and not 1 <= int(keep_top_k) <= 1024:
            raise ValueError("keep_top_k must be None or in [1, 1024]")
        self.keep_top_k = None if keep_top_k is None else int(keep_top_k)

        def make_slot():   # everything a step writes
            det = {"kept": D.empty((b, c - 1, self.top_k), np.int32), "count": D.empty((b, c - 1), np.int32)}
            if evaluator is not None or self.keep_top_k is not None:   # the filter then writes the decoded boxes here
                det.update(kept_score=D.empty((b, c - 1, self.top_k), np.float32), boxes=D.empty((b, a, 4), np.float32))
            top = None
            if self.keep_top_k is not None:
                kk = self.keep_top_k
                top = {"prior": D.empty((b, kk), np.int32), "class": D.empty((b, kk), np.int32),
                       "score": D.empty((b, kk), np.float32), "box": D.empty((b, kk, 4), np.float32),
                       "n": D.empty((b,), np.int32), "count": D.empty((b, c - 1), np.int32)}
            return {"tgt": {"cls": D.empty((b, a), np.int32), "loc": D.empty((b, a, 4), np.float32),
                            "mask": D.empty((b, a), np.uint8)},
                    "loss": {"result": D.empty((N.LOSS_RESULT_LEN,), np.float64)},
                    "det": det, "top": top,
                    "det_stats": {"row_ml": D.empty((b, a, 2), np.float32), "row_negbg": D.empty((b, a), np.float32)},
                    "pool": ops.WorkspacePool(), "ev_a": D.Event(), "ev_d": D.Event(), "ev_x": D.Event(),
                    "x_pending": False, "used": False, "loss_exchange": None}
        self._slots = [make_slot() for _ in range(self.depth)]
        self._bind_slot(0)
        # the filter pass, the matcher and the loss at high priority, the NMS (20 480 small CTAs that would otherwise
        # occupy every SM ahead of everything else) at low.  With the matcher at low priority a step of 128 images per
        # GPU -- where the assignment chain is the longer one -- took 0.370 instead of 0.347 ms; at 256 images there is
        # no difference (profiles/r15_stream_priorities.txt).
        self.s_main, self.s_a, self.s_d = D.Stream(), D.Stream("high"), D.Stream("high")
        self.s_n, self.s_l = D.Stream("low"), D.Stream("high")
        self.s_x = D.Stream("high")                      # loss exchange (data parallel)
        self.ev_begin, self.ev_mid, self.ev_m = (D.Event() for _ in range(3))
        self.split = True
        # Who takes the SMs first.  Both branches become ready at the same moment (ev_begin); the filter's 148 CTAs of
        # 171 KB shared memory and the search's 1184 small CTAs then compete for every SM.  Below ~240 images per GPU the
        # assignment chain (search -> per-image matching -> loss, all latency-bound) is the longer one, and the step is
        # shorter when the search gets its CTAs placed first and the filter's fill in as they drain: a small zeroing
        # node in front of the filter pass (a few microseconds) decides that race (128 images: 0.34 -> 0.31 ms per
        # step; 256 images: 0.530 -> 0.539, so not there).  Ordering the filter behind the search with an event costs
        # the kernel boundary and is slower than either (0.35 ms).
        self.lead_assign = self.batch < 240
        self._lead_pad = D.empty((64 * 1024,), np.uint8)
        # one pass over the logits serves both branches: the filter leaves per-prior softmax statistics and the
        # loss gathers from them instead of streaming the 724 MB again (only in the chained step)
        self.fused = True
        if mining not in ("shard", "global"):
            raise ValueError("mining must be 'shard' or 'global'")
        self.mining, self.comm = mining, comm
        if comm is not None and allreduce is None:
            allreduce = comm.allreduce
        self.allreduce = allreduce
        # optional callable(stream): the data-parallel exchange of the additive loss sums (per-shard mining),
        # enqueued on a stream of its own right behind the loss so that it hides under the NMS of the other branch
        self.loss_exchange = None                        # a caller's own exchange (depth 1 only)
        if comm is not None and mining == "shard" and comm.world > 1:
            for sl in self._slots:
                sums = ops.loss_result_words(sl["loss"]["result"], N.LOSS_ADDITIVE)
                sl["loss_exchange"] = (lambda stream, sums=sums: comm.allreduce(sums, stream))
        self.staged = None
        if mining == "global":
            if allreduce is None or not global_priors:
                raise ValueError("global mining needs comm / allreduce and global_priors")
            self.staged = ops.StagedLoss(self.tgt["cls"], self.tgt["loc"], self.tgt["mask"], self.pred_box, self.pred_cls,
                                         int(global_priors), self.neg_ratio, out=self.loss)
        # search, match | lossprep (or ce), select x2, final | filter, nms
        self.kernel_launches_per_step = 8 + (1 if evaluator is not None else 0) + (1 if self.keep_top_k is not None else 0)
        # matcher head + loss histograms (cudaMemsetAsync), + the lead node of small batches
        self.memsets_per_step = 2 + (1 if self.lead_assign else 0)
        self.h2d_bytes = sum(self._sets[0][k].nbytes for k in INPUT_NAMES)
        # results + the matcher's status word
        self.d2h_bytes = self.loss["result"].nbytes + self.det["kept"].nbytes + self.det["count"].nbytes + 4
        self._status_host = D.PinnedArray((2,), np.uint32)
        self._status_host.array[...] = 0
        self._match_out = None

    # ---- per-step buffers -----------------------------------------------------------------------------------
    def _bind_slot(self, k: int):
        sl = self._slots[k]
        self._cur = sl
        self.tgt, self.loss, self.det, self.det_stats, self.pool = sl["tgt"], sl["loss"], sl["det"], sl["det_stats"], sl["pool"]
        self.top = sl["top"]
        self.ev_a, self.ev_d, self.ev_x = sl["ev_a"], sl["ev_d"], sl["ev_x"]

    @property
    def _x_pending(self):
        return self._cur["x_pending"]

    @_x_pending.setter
    def _x_pending(self, v):
        self._cur["x_pending"] = v

    # ---- input buffers --------------------------------------------------------------------------------------
    def _alloc_inputs(self):
        b, a, c = self.batch, self.A, self.classes
        return {"gt_boxes": D.empty((self.total_gt, 4), np.float32), "gt_cls": D.empty((self.total_gt,), np.float32),
                "gt_off": D.empty((b + 1,), np.int32), "pred_cls": D.empty((b, a, c), np.float32),
                "pred_box": D.empty((b, a, 4), np.float32)}

    def _bind(self, s):
        for k in INPUT_NAMES:
            setattr(self, k, s[k])
        if getattr(self, "staged", None) is not None:
            self.staged.pred_box, self.staged.pred_cls = self.pred_box, self.pred_cls

    def add_input_set(self) -> int:
        """Another resident copy of the input buffers (distinct batches to rotate over); returns its index."""
        self._sets.append(self._alloc_inputs())
        return len(self._sets) - 1

    def use_set(self, k: int):
        """Make input set ``k`` the one the next step / upload works on (host-side pointer swap)."""
        self._bind(self._sets[k])

    # ---- stages (asynchronous on the given stream) ---------------------------------------------------
    def assign(self, stream):
        self._match_out = ops.match_encode(self.gt_boxes, self.gt_cls, self.gt_off, self.priors, self.batch, self.max_gt,
                                           self.thresh, want=(), out=self.tgt, stream=stream, pool=self.pool)

    def loss_stage(self, stream, stats=False):
        row_stats = (self.det_stats["row_ml"], self.det_stats["row_negbg"]) if stats else None
        if self.staged is None:
            ops.multibox_loss(self.tgt["cls"], self.tgt["loc"], self.tgt["mask"], self.pred_box, self.pred_cls,
                              self.neg_ratio, out=self.loss, stream=stream, pool=self.pool, row_stats=row_stats)
            return
        self.staged.stream, self.staged.row_stats = stream, row_stats
        for stage in range(self.staged.n_stages):
            self.staged.run(stage)
            bufs = self.staged.exchange(stage)
            if not bufs:
                continue
            if self.comm is not None:
                self.comm.allreduce_multi(bufs, stream)       # one NCCL group per stage
            else:
                for buf in bufs:
                    self.allreduce(buf, stream)

    def detect_stage(self, stream, stage=None, stats=False):
        out = dict(self.det, **self.det_stats) if stats else self.det
        ops.detect(self.pred_cls, self.pred_box, self.priors, self.score_thresh, self.top_k, self.iou_thresh,
                   out=out, stream=stream, stage=stage, want_row_stats=stats, pool=self.pool)

    def keep_top_k_stage(self, stream):
        ops.keep_top_k(self.det, self.keep_top_k, out=self.top, stream=stream)

    def evaluate_stage(self, stream, image_base=None):
        det = self.det if self.top is None else dict(self.det, count=self.top["count"])   # the capped lists
        self.evaluator.add(det, self.gt_boxes, self.gt_cls, self.gt_off, image_base, stream, max_gt=self.max_gt)

    def step(self, image_base=None):
        """One pass of the chain over the resident batch; work is ordered on ``s_main``.  With an evaluator the batch's
        images get the global indices ``image_base ..`` (None: after the highest added so far).

        Four streams so that kernels bound by different resources share the SMs:
          phase A   the filter pass (HBM-bound, s_d, high priority)     with  the matcher (latency-bound, s_a, high)
          phase B   NMS (instruction-bound, s_n, low)                   with  the loss (HBM-bound, s_l, high)
        The loss must outrank the NMS or its 148 large-shared-memory CTAs starve behind 20 480 small NMS CTAs."""
        if self.depth > 1:
            if self.loss_exchange is not None:
                raise RuntimeError("a caller-supplied loss_exchange needs depth=1")
            self._bind_slot(self._n_steps % self.depth)
        self._n_steps += 1
        self.ev_begin.record(self.s_main)
        D.stream_wait_event(self.s_a, self.ev_begin)
        D.stream_wait_event(self.s_d, self.ev_begin)
        if self.depth > 1 and self._cur["used"]:
            # the step that used these buffers last must be through with them (its NMS reads the lists and boxes, its
            # loss the targets and row statistics); everything else of that step is ordered before these two events
            for st in (self.s_a, self.s_d):
                D.stream_wait_event(st, self.ev_a)
                D.stream_wait_event(st, self.ev_d)
        self._cur["used"] = True
        loss_exchange = self._cur["loss_exchange"] or self.loss_exchange
        fused = self.fused
        if self.split:
            if self.lead_assign:
                self._lead_pad.zero_(self.s_d)
            self.detect_stage(self.s_d, stage=0, stats=fused)
            self.assign(self.s_a)
            self.ev_m.record(self.s_a)
            self.ev_mid.record(self.s_d)
            D.stream_wait_event(self.s_n, self.ev_mid)
            self.detect_stage(self.s_n, stage=1, stats=fused)
            if self.top is not None:
                self.keep_top_k_stage(self.s_n)
            if self.evaluator is not None:      # before ev_d: the waits on ev_d cover its reads of GT and lists
                self.evaluate_stage(self.s_n, image_base)
            D.stream_wait_event(self.s_l, self.ev_m)
            if fused:
                D.stream_wait_event(self.s_l, self.ev_mid)
            if self._x_pending:      # the previous step's exchange still owns the result block
                D.stream_wait_event(self.s_l, self.ev_x)
            self.loss_stage(self.s_l, stats=fused)
            self.ev_a.record(self.s_l)
            if loss_exchange is not None:
                # The data-parallel exchange of the additive loss sums runs on a stream of its own and nobody in
                # THIS step waits for it (finish_exchange() / download() do): the processes need not meet inside
                # every step -- a rendezvous there costs the slowest process's skew plus the collective's latency
                # on the critical path once the loss ends less than that before the NMS (8 GPUs: 0.71 ms per step).
                D.stream_wait_event(self.s_x, self.ev_a)
                loss_exchange(self.s_x)
                self.ev_x.record(self.s_x)
                self._x_pending = True
            self.ev_d.record(self.s_n)
        else:
            self.detect_stage(self.s_d)
            if self.top is not None:
                self.keep_top_k_stage(self.s_d)
            if self.evaluator is not None:
                self.evaluate_stage(self.s_d, image_base)
            self.assign(self.s_a)
            self.loss_stage(self.s_a)
            if loss_exchange is not None:
                loss_exchange(self.s_a)
            self.ev_a.record(self.s_a)
            self.ev_d.record(self.s_d)
        if self.depth == 1:
            self.join()

    def join(self, stream=None):
        """Make ``stream`` (s_main) wait for every step enqueued so far (both branches)."""
        st = self.s_main if stream is None else stream
        for sl in self._slots:
            if sl["used"]:
                D.stream_wait_event(st, sl["ev_a"])
                D.stream_wait_event(st, sl["ev_d"])

    # ---- host-facing -------------------------------------------------------------------------------------
    def _check_gt(self, gt_off):
        """The reference matches every ground-truth box of every image (utils/bbox.py:44-91) and asserts T <= A
        (:50): a batch this pipeline was not sized for is an error here, not a silent all-unmatched image."""
        counts = np.diff(np.asarray(gt_off))
        if counts.size != self.batch:
            raise AssertionError("gt_off must have batch + 1 entries")
        if counts.size and int(counts.min()) < 0:
            raise ValueError("gt_off must be non-decreasing")
        if counts.size and int(counts.max()) > self.A:
            raise AssertionError("number of default boxes should greater than the number of targets")   # utils/bbox.py:50
        if counts.size and int(counts.max()) > self.max_gt:
            raise ValueError("an image has %d ground-truth boxes; this HotPath was built with max_gt=%d" %
                             (int(counts.max()), self.max_gt))

    def upload(self, gt_boxes, gt_cls, gt_off, pred_cls, pred_box, stream=None):
        """Host (ideally pinned) -> device copies of one batch, asynchronous on ``stream`` (s_main)."""
        self._check_gt(gt_off)
        st = self.s_main if stream is None else stream
        lib = N.lib()
        for dst, src in ((self.gt_boxes, gt_boxes), (self.gt_cls, gt_cls), (self.gt_off, gt_off),
                         (self.pred_box, pred_box), (self.pred_cls, pred_cls)):
            assert src.nbytes == dst.nbytes and src.dtype == dst.dtype and src.flags["C_CONTIGUOUS"]
            N.check(lib.ssdg_memcpy_h2d(dst.ptr, src.ctypes.data, dst.nbytes, D.stream_handle(st)), "h2d")

    def finish_exchange(self, stream=None):
        """Make ``stream`` (s_main) wait for the data-parallel exchange of the last step's loss sums."""
        for sl in self._slots:
            if sl["x_pending"]:
                D.stream_wait_event(self.s_main if stream is None else stream, sl["ev_x"])

    def download(self, out_result, out_kept, out_count, stream=None):
        st = self.s_main if stream is None else stream
        if self.depth > 1:
            self.join(st)             # the results of the LAST step (the slot bound now)
        self.finish_exchange(st)
        lib = N.lib()
        for src, dst in ((self.loss["result"], out_result), (self.det["kept"], out_kept), (self.det["count"], out_count)):
            N.check(lib.ssdg_memcpy_d2h(dst.ctypes.data, src.ptr, src.nbytes, D.stream_handle(st)), "d2h")
        if self._match_out is not None:      # the matcher's status word travels with the results (include/ssdgeom.h)
            ws = self._match_out["_match_ws"]
            N.check(lib.ssdg_memcpy_d2h(self._status_host.ptr, ws.ptr, 8, D.stream_handle(st)), "d2h")

    def download_detections(self, out: dict, stream=None):
        """Copy the last step's final detections (``keep_top_k``) into host arrays: ``out`` maps any of "prior",
        "class", "score", "box", "n", "count" to a host array of that shape and dtype.  Waits for the last step as
        ``download`` does; the copies are asynchronous on ``stream`` (s_main)."""
        if self.top is None:
            raise RuntimeError("this HotPath was built without keep_top_k")
        st = self.s_main if stream is None else stream
        if self.depth > 1:
            self.join(st)
        lib = N.lib()
        for key, dst in out.items():
            src = self.top[key]
            assert dst.nbytes == src.nbytes and dst.dtype == src.dtype and dst.flags["C_CONTIGUOUS"]
            N.check(lib.ssdg_memcpy_d2h(dst.ctypes.data, src.ptr, src.nbytes, D.stream_handle(st)), "d2h")

    def check_status(self, sync=False):
        """Raise if the device had to skip an image or saw a stale prior index: from the status word the last
        ``download`` brought back (after a synchronisation), or -- ``sync=True`` -- read now (synchronises)."""
        if sync:
            if self._match_out is not None:
                ops.raise_for_match_status(ops.match_status(self._match_out, self.s_main))
            return
        ops.raise_for_match_status(int(self._status_host.array[1]))

    # Pipelined end to end: two device copies of the inputs, the H2D copy of batch k+1 (PCIe-bound, ~14 ms) runs on
    # its own stream under the compute and D2H of batch k.
    def _submit_state(self):
        if getattr(self, "_sub", None) is None:
            while len(self._sets) < 2:
                self.add_input_set()
            self._n_sub = 0
            self.s_copy = D.Stream()
            self.ev_up, self.ev_done, self._done_valid = [D.Event(), D.Event()], [D.Event(), D.Event()], [False, False]
            self._sub = True

    def submit(self, host_in, host_out):
        """Enqueue one end-to-end step (host inputs -> host results) and return without waiting; call ``drain()``
        before reading ``host_out``.  Results of consecutive submits must go to different host buffers if they are
        to be kept.  Not available with cross-process mining (the staged loss holds its input buffers)."""
        if self.staged is not None:
            raise RuntimeError("submit() is not available with mining='global'; use step_host()")
        self._submit_state()
        slot = self._n_sub % 2
        if self._done_valid[slot]:      # the slot's inputs were read by the step two submits ago
            D.stream_wait_event(self.s_copy, self.ev_done[slot])
        self.use_set(slot)
        self.upload(*host_in, stream=self.s_copy)
        self.ev_up[slot].record(self.s_copy)
        D.stream_wait_event(self.s_main, self.ev_up[slot])
        self.step()
        self.download(*host_out)
        self.ev_done[slot].record(self.s_main)
        self._done_valid[slot] = True
        self._n_sub += 1

    def drain(self):
        self.s_main.sync()
        self.check_status()

    def step_host(self, gt_boxes, gt_cls, gt_off, pred_cls, pred_box, out_result, out_kept, out_count):
        """End to end: host inputs in, host results out (synchronises)."""
        self.upload(gt_boxes, gt_cls, gt_off, pred_cls, pred_box)
        self.step()
        self.download(out_result, out_kept, out_count)
        self.s_main.sync()
        self.check_status()
