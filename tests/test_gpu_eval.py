"""GPU (B200): the detection evaluation (ssdg_eval_*, ssdgeom.evaluate) against its NumPy restatement
(tests/coco_eval_oracle.py): the slots bit for bit, the precision / recall arrays bit for bit, independence of the
batching, the detect -> evaluate chain, the evaluator inside HotPath, and data-parallel accumulation."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import coco_eval_oracle as E                 # noqa: E402  (the checker)
from ssdgeom import _native as N, ops, synth   # noqa: E402
from ssdgeom.evaluate import DetectionEvaluator   # noqa: E402
from ssdgeom.models import ssd_model as M    # noqa: E402
from ssdgeom.pipeline import HotPath         # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
THR = E.COCO_IOU_THRESHOLDS


def rand_case(seed, b, n_classes=6, top_k=12, a=40, max_t=9):
    """Detections and ground truth on a 1/16 grid (equal IoUs and equal scores are common), counts beyond max_dets,
    images without ground truth and lists without detections."""
    rng = np.random.default_rng(seed)
    k = n_classes - 1
    g = lambda n, lo, hi: rng.integers(lo, hi, n) / 16.0
    boxes = np.stack([g((b, a), 3, 13), g((b, a), 3, 13), g((b, a), 2, 9), g((b, a), 2, 9)], -1).astype(np.float32)
    t = rng.integers(0, max_t + 1, b)
    t[rng.uniform(size=b) < 0.2] = 0
    off = np.concatenate([[0], np.cumsum(t)]).astype(np.int32)
    n = int(off[-1])
    src = boxes[np.repeat(np.arange(b), t), rng.integers(0, a, n)]
    gt = (src + rng.integers(-1, 2, (n, 4)) / 16.0 * np.array([1, 1, 0, 0])).astype(np.float32)
    gcls = rng.integers(0, k, n).astype(np.float32)
    kept = np.full((b, k, top_k), -1, np.int32)
    count = rng.integers(0, top_k + 1, (b, k)).astype(np.int32)
    count[rng.uniform(size=(b, k)) < 0.2] = 0
    score = np.zeros((b, k, top_k), np.float32)
    levels = np.array([0.95, 0.9, 0.7, 0.5, 0.3, 0.2, 0.05], np.float32)
    for i in range(b):
        for c in range(k):
            m = count[i, c]
            kept[i, c, :m] = rng.choice(a, m, replace=False)
            score[i, c, :m] = np.sort(rng.choice(levels, m))[::-1]
    return {"kept": kept, "count": count, "kept_score": score, "boxes": boxes}, gt, gcls, off


def sub(det, gt, gcls, off, lo, hi):
    d = {k: v[lo:hi] for k, v in det.items()}
    return d, gt[off[lo]:off[hi]], gcls[off[lo]:off[hi]], (off[lo:hi + 1] - off[lo]).astype(np.int32)


def device_slots(ev):
    keys, words = (x.to_host() for x in ev.exchange_buffers())
    k, m, d = ev.n_classes - 1, ev.max_images, ev.max_dets
    return (keys.reshape(k, m, d), words[64:64 + k * m * d].reshape(k, m, d), words[64 + k * m * d:].reshape(k, m),
            words[:64])


def oracle_of(det, gt, gcls, off, base=0, max_dets=100, thr=THR):
    return E.evaluate_batch(det["kept"], det["count"], det["kept_score"], det["boxes"], gt, gcls, off, base, thr,
                            max_dets)


def assert_same_result(res, want, n_classes, thr=THR):
    p, r, n_gt, n_det = E.coco_accumulate(*want, n_classes, len(thr))
    assert np.array_equal(res["precision"], p) and np.array_equal(res["recall"], r)
    assert np.array_equal(res["n_gt"], n_gt) and np.array_equal(res["n_det"], n_det)
    s = E.coco_summarize(p, r, thr)
    for key in ("AP", "AP50", "AP75", "AR"):
        assert abs(res[key] - s[key]) <= 1e-12, key
    np.testing.assert_allclose(res["per_class_AP"], s["per_class_AP"], rtol=0, atol=1e-12)


# ---- 1. the slots ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed,max_dets", [(1, 12), (2, 5), (3, 1)])
def test_accumulate_slots_equal_the_oracle(seed, max_dets):
    det, gt, gcls, off = rand_case(seed, 10)
    ev = DetectionEvaluator(n_classes=6, max_images=13, max_dets=max_dets)
    ev.add(det, gt, gcls, off, image_base=3)
    keys, flags, ngt, hdr = device_slots(ev)
    wk, wf, wg = E.slots(*oracle_of(det, gt, gcls, off, 3, max_dets), 6, 13, max_dets)
    assert np.array_equal(keys, wk) and np.array_equal(flags, wf) and np.array_equal(ngt, wg)
    assert not hdr.any()
    assert (np.diff(off) == 0).any() and (det["count"] == 0).any()
    assert max_dets == 12 or (det["count"] > max_dets).any()
    assert set(np.unique(gcls).astype(int)) == set(range(5))


def test_equal_iou_tie_goes_to_the_last_ground_truth():
    g0, g1, d0 = [0.375, 0.5, 0.5, 0.5], [0.625, 0.5, 0.5, 0.5], [0.5, 0.5, 0.5, 0.5]
    det = {"kept": np.array([[[0, 1]]], np.int32), "count": np.array([[2]], np.int32),
           "kept_score": np.array([[[0.9, 0.8]]], np.float32), "boxes": np.array([[d0, g1]], np.float32)}
    d0_bits = sum(1 << j for j in range(len(THR)) if 0.6 >= THR[j])        # d0: IoU 0.6 with both
    # d0 takes the last row where it matches; the exact copy of g1 is then a FP there (g1 taken, IoU 1/3 with g0) and
    # a TP at the stricter thresholds -- or, with the rows swapped, a TP everywhere
    for order, want in (([g0, g1], 0x10000 | (0x3FF & ~d0_bits)), ([g1, g0], 0x10000 | 0x3FF)):
        gt = np.array(order, np.float32)
        ev = DetectionEvaluator(n_classes=2, max_images=1, max_dets=2)
        ev.add(det, gt, np.zeros(2, np.float32), np.array([0, 2], np.int32))
        _, flags, _, _ = device_slots(ev)
        assert flags[0, 0, 0] == 0x10000 | d0_bits and flags[0, 0, 1] == want
        assert np.array_equal(flags, E.slots(*oracle_of(det, gt, np.zeros(2, np.float32), [0, 2], 0, 2), 2, 1, 2)[1])


def test_ground_truth_class_out_of_range_raises():
    det, gt, gcls, off = rand_case(4, 3)
    gcls = gcls.copy()
    gcls[0] = 5.0                                 # n_classes - 1
    ev = DetectionEvaluator(n_classes=6, max_images=3, max_dets=12)
    ev.add(det, gt, gcls, off)
    with pytest.raises(ValueError, match="class id"):
        ev.summarize()


# ---- 2. finalize ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [5, 6])
def test_finalize_equals_the_oracle(seed):
    det, gt, gcls, off = rand_case(seed, 60, n_classes=8, top_k=20, a=64, max_t=12)
    ev = DetectionEvaluator(n_classes=8, max_images=60, max_dets=15)
    ev.add(det, gt, gcls, off)
    assert_same_result(ev.summarize(), oracle_of(det, gt, gcls, off, 0, 15), 8)


def test_custom_thresholds():
    det, gt, gcls, off = rand_case(7, 20)
    thr, rec = np.array([0.3, 0.5, 0.62]), np.linspace(0, 1, 11)
    ev = DetectionEvaluator(n_classes=6, max_images=20, max_dets=12, iou_thresholds=thr, recall_thresholds=rec)
    ev.add(det, gt, gcls, off)
    res = ev.finalize()
    p, r, _, _ = E.coco_accumulate(*oracle_of(det, gt, gcls, off, 0, 12, thr), 6, 3, rec)
    assert np.array_equal(res["precision"], p) and np.array_equal(res["recall"], r)


# ---- 3. batching invariance --------------------------------------------------------------------------------
def test_result_is_independent_of_batching_and_order():
    det, gt, gcls, off = rand_case(8, 30)
    want = oracle_of(det, gt, gcls, off, 0, 12)
    one = DetectionEvaluator(n_classes=6, max_images=30, max_dets=12)
    one.add(det, gt, gcls, off)
    assert_same_result(one.summarize(), want, 6)
    ref = one.finalize()
    cuts = [(0, 7), (7, 25), (25, 30)]
    for order in (cuts, cuts[::-1], [cuts[1], cuts[0], cuts[2]]):
        ev = DetectionEvaluator(n_classes=6, max_images=30, max_dets=12)
        for lo, hi in order:
            ev.add(*sub(det, gt, gcls, off, lo, hi), image_base=lo)
        ev.add(*sub(det, gt, gcls, off, 7, 25), image_base=7)        # re-adding a batch overwrites it
        res = ev.finalize()
        assert all(np.array_equal(res[k], ref[k]) for k in ref)
        assert np.array_equal(device_slots(ev)[0], device_slots(one)[0])


# ---- 4. detect -> evaluate ------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["coco", "max"])
def test_detect_then_evaluate_on_trained_like_predictions(mode):
    b = 64
    priors = M.build_prior_box(synth.SSD300["sizes"])
    gt, gcls, off = synth.make_gt(21, b, 100, mode)
    t = ops.match_encode(gt, gcls, off, priors, b, int(np.diff(off).max()), 0.5)
    pc, pb = synth.make_trained_predictions(21, t["cls"].to_host(), t["loc"].to_host(), t["mask"].to_host())
    out = ops.detect(pc, pb, priors, want_scores=True, want_boxes=True)
    ev = DetectionEvaluator(max_images=b, max_gt=int(np.diff(off).max()))
    ev.add(out, gt, gcls, ops.D.to_device(off))          # offsets on the device: bounded by max_gt
    res = ev.summarize()
    host = {k: out[k].to_host() for k in ("kept", "count", "kept_score", "boxes")}
    assert_same_result(res, oracle_of(host, gt, gcls, off), 81)
    ap_t = [p[p > -1].mean() for p in res["precision"]]           # every threshold has TPs, and fewer at stricter ones
    assert 0.05 < res["AP"] < 0.95 and ap_t[0] > ap_t[5] > ap_t[-1] > 0


# ---- 5. inside HotPath -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("depth", [1, 2])
def test_hotpath_evaluator_equals_stand_alone(depth):
    b, n_batches = 32, 3
    priors = M.build_prior_box(synth.SSD300["sizes"])
    batches = []
    for k in range(n_batches):
        gt, gcls, off = synth.make_gt(40 + k, b, 30, "coco")
        t = ops.match_encode(gt, gcls, off, priors, b, 30, 0.5)
        pc, pb = synth.make_trained_predictions(40 + k, t["cls"].to_host(), t["loc"].to_host(), t["mask"].to_host())
        batches.append((gt, gcls, off, pc, pb))
    total = max(x[0].shape[0] for x in batches)
    pad = [(np.concatenate([gt, np.zeros((total - gt.shape[0], 4), np.float32)]),
            np.concatenate([gcls, np.zeros(total - gcls.shape[0], np.float32)]), off, pc, pb)
           for gt, gcls, off, pc, pb in batches]

    def run(evaluator):
        hp = HotPath(synth.SSD300, batch=b, max_gt=30, total_gt=total, depth=depth, evaluator=evaluator)
        outs = []
        for k in range(n_batches):
            if k:
                hp.add_input_set()
            hp.use_set(k)
            hp.upload(*pad[k])
        for k in range(n_batches):
            hp.use_set(k)
            hp.step(image_base=(2 - k) * b)                              # out of order on purpose
            o = (np.zeros(16), np.zeros((b, 80, 200), np.int32), np.zeros((b, 80), np.int32))
            hp.download(*o)
            outs.append(o)
        hp.s_main.sync()
        hp.check_status()
        return outs

    ev = DetectionEvaluator(max_images=n_batches * b, max_gt=30)
    with_ev, without = run(ev), run(None)
    for x, y in zip(with_ev, without):
        assert all(np.array_equal(u, v) for u, v in zip(x, y))
    got = ev.summarize()
    alone = DetectionEvaluator(max_images=n_batches * b)
    for k, (gt, gcls, off, pc, pb) in enumerate(batches):
        out = ops.detect(pc, pb, priors, want_scores=True, want_boxes=True)
        assert np.array_equal(out["kept"].to_host(), with_ev[k][1])
        alone.add(out, gt, gcls, off, image_base=(2 - k) * b)
    want = alone.finalize()
    assert all(np.array_equal(got[k], want[k]) for k in want)


# ---- 6. data parallel ---------------------------------------------------------------------------------------
def _host_sum(evs):
    """The all-reduce of the exchange buffers, done on the host; the result lands in evs[0]."""
    bufs = [ev.exchange_buffers() for ev in evs]
    for j in range(2):
        total = sum(b[j].to_host() for b in bufs)
        bufs[0][j].copy_from_host(total.astype(bufs[0][j].dtype))


@pytest.mark.parametrize("shards", [2, 3])
def test_emulated_shards_equal_one_device(shards):
    det, gt, gcls, off = rand_case(9, 24)
    one = DetectionEvaluator(n_classes=6, max_images=24, max_dets=12)
    one.add(det, gt, gcls, off)
    evs = [DetectionEvaluator(n_classes=6, max_images=24, max_dets=12) for _ in range(shards)]
    for r, ev in enumerate(evs):
        lo, hi = 24 * r // shards, 24 * (r + 1) // shards
        ev.add(*sub(det, gt, gcls, off, lo, hi), image_base=lo)
    _host_sum(evs)
    got, want = evs[0].summarize(), one.summarize()
    assert all(np.array_equal(got[k], want[k]) for k in ("precision", "recall", "n_gt", "n_det"))


def test_two_shards_writing_the_same_image_are_reported():
    det, gt, gcls, off = rand_case(10, 4)
    evs = [DetectionEvaluator(n_classes=6, max_images=8, max_dets=12) for _ in range(2)]
    evs[0].add(det, gt, gcls, off, image_base=0)
    evs[1].add(*sub(det, gt, gcls, off, 1, 3), image_base=3)          # image 3 is shard 0's too
    _host_sum(evs)
    with pytest.raises(ValueError, match="more than one"):
        evs[0].summarize()


_TWO_RANK = r"""
import os, sys, numpy as np
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, os.path.join(sys.argv[1], "ssd-object-detection_b200"))
sys.path.insert(0, os.path.join(sys.argv[1], "tests"))
rank, world, port = int(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4])
from ssdgeom import _native as N, device as D, comm
from ssdgeom.evaluate import DetectionEvaluator
from test_gpu_eval import rand_case, sub
N.check(N.lib().ssdg_set_device(rank), "set_device")
uid = comm.tcp_broadcast(comm.unique_id() if rank == 0 else None, world, rank, "127.0.0.1", port)
cm = comm.Comm(uid, world, rank)
st = D.Stream()
det, gt, gcls, off = rand_case(11, 20)
one = DetectionEvaluator(n_classes=6, max_images=20, max_dets=12)
one.add(det, gt, gcls, off)
ev = DetectionEvaluator(n_classes=6, max_images=20, max_dets=12)
lo, hi = (0, 9) if rank == 0 else (9, 20)
ev.add(*sub(det, gt, gcls, off, lo, hi), image_base=lo, stream=st)
ev.exchange(cm, st)
got, want = ev.summarize(st), one.summarize()
assert all(np.array_equal(got[k], want[k]) for k in ("precision", "recall", "n_gt", "n_det"))
cm.close()
print("rank", rank, "ok")
"""


def test_comm_two_ranks_evaluation():
    if N.device_count() < 2:
        pytest.skip("needs two GPUs")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    procs = [subprocess.Popen([sys.executable, "-c", _TWO_RANK, ROOT, str(r), "2", str(port)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=600)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and "rank %d ok" % r in o, o[-3000:]
