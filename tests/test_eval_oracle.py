"""CPU: the detection evaluation's NumPy restatement (tests/coco_eval_oracle.py) on hand-computed cases, against
pycocotools where it is installed, and the argument checks / state size of the ssdg_eval_* entry points."""
import ctypes as C
import os

import numpy as np
import pytest

import coco_eval_oracle as E

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
THR = E.COCO_IOU_THRESHOLDS
BOX = [0.5, 0.5, 0.25, 0.25]
ONE = pytest.approx(1.0, rel=1e-15, abs=0)     # a single TP has precision 1 / (1 + 2^-52), as in COCOeval


def one_image(dets, scores, gts, gt_cls=None, n_classes=3, max_dets=100, image=0):
    """Records of one image whose detections all belong to class 0."""
    dets = np.asarray(dets, np.float32).reshape(-1, 4)
    gts = np.asarray(gts, np.float32).reshape(-1, 4)
    k = n_classes - 1
    kept = np.full((1, k, max(len(dets), 1)), -1, np.int32)
    kept[0, 0, :len(dets)] = np.arange(len(dets))
    count = np.zeros((1, k), np.int32)
    count[0, 0] = len(dets)
    ks = np.zeros(kept.shape, np.float32)
    ks[0, 0, :len(dets)] = scores
    cls = np.zeros(len(gts), np.float32) if gt_cls is None else np.asarray(gt_cls, np.float32)
    return E.evaluate_batch(kept, count, ks, dets[None], gts, cls, np.array([0, len(gts)], np.int32), image,
                            THR, max_dets)


def ap(parts, n_classes=3):
    rec, ng = E.merge(*parts) if isinstance(parts, list) else parts
    p, r, _, _ = E.coco_accumulate(rec, ng, n_classes, len(THR))
    return E.coco_summarize(p, r, THR)


def test_perfect_detections_give_ap_one():
    s = ap(one_image([BOX, [0.2, 0.2, 0.1, 0.1]], [0.9, 0.7], [BOX, [0.2, 0.2, 0.1, 0.1]]))
    assert s["AP"] == 1.0 and s["AP50"] == 1.0 and s["AP75"] == 1.0 and s["AR"] == 1.0


def test_only_false_positives_give_ap_zero():
    s = ap(one_image([[0.1, 0.1, 0.05, 0.05]], [0.9], [[0.8, 0.8, 0.1, 0.1]]))
    assert s["AP"] == 0.0 and s["AR"] == 0.0


def test_fp_then_tp_gives_half():
    s = ap(one_image([[0.1, 0.1, 0.05, 0.05], BOX], [0.9, 0.8], [BOX]))
    assert s["AP"] == 0.5 and s["AR"] == 1.0


def test_duplicate_detection_is_a_false_positive():
    tp = E.coco_evaluate_image([BOX, BOX], [BOX], THR)
    assert tp[:, 0].all() and not tp[:, 1].any()
    s = ap(one_image([BOX, BOX], [0.9, 0.8], [BOX]))
    assert s["AP"] == ONE          # the envelope carries precision 1 at recall 1 from the first record


def test_last_ground_truth_among_equal_ious_wins():
    g0, g1 = [0.375, 0.5, 0.5, 0.5], [0.625, 0.5, 0.5, 0.5]
    d0 = [0.5, 0.5, 0.5, 0.5]                     # IoU 0.6 with both, exactly
    assert E.box_iou(d0, g0) == E.box_iou(d0, g1) == 0.6
    tp = E.coco_evaluate_image([d0, g1], [g0, g1], [0.5])
    assert tp[0].tolist() == [True, False]        # d0 takes g1; g1's exact copy finds g0 below 0.5
    tp = E.coco_evaluate_image([d0, g1], [g1, g0], [0.5])
    assert tp[0].tolist() == [True, True]         # with the rows swapped d0 takes g0 and the copy gets g1


def test_equal_scores_order_by_global_image_index():
    far = [0.1, 0.1, 0.05, 0.05]
    fp_img = one_image([far], [0.5], [], image=0)
    tp_img = one_image([BOX], [0.5], [BOX], image=1)
    assert ap([fp_img, tp_img])["AP"] == 0.5      # image 0 (FP) first
    fp_img = one_image([far], [0.5], [], image=1)
    tp_img = one_image([BOX], [0.5], [BOX], image=0)
    assert ap([fp_img, tp_img])["AP"] == ONE


def test_max_dets_truncates_each_list():
    far = [0.1, 0.1, 0.05, 0.05]
    assert ap(one_image([far, far, BOX], [0.9, 0.8, 0.7], [BOX], max_dets=3))["AR"] == 1.0
    s = ap(one_image([far, far, BOX], [0.9, 0.8, 0.7], [BOX], max_dets=2))
    assert s["AR"] == 0.0 and s["AP"] == 0.0


def test_classes_without_ground_truth_are_minus_one_and_excluded():
    rec, ng = one_image([BOX], [0.9], [BOX], n_classes=4)
    p, r, n_gt, n_det = E.coco_accumulate(rec, ng, 4, len(THR))
    assert (p[:, :, 1:] == -1).all() and (r[:, 1:] == -1).all()
    assert n_gt.tolist() == [1, 0, 0] and n_det.tolist() == [1, 0, 0]
    s = E.coco_summarize(p, r, THR)
    assert s["AP"] == ONE and s["per_class_AP"][0] == ONE and s["per_class_AP"][1:].tolist() == [-1.0, -1.0]


def test_thresholds_half_and_three_quarters_are_found_by_equality():
    assert np.where(THR == .5)[0].tolist() == [0] and np.where(THR == .75)[0].tolist() == [5]
    # a detection with IoU in [0.75, 0.8): TP up to 0.75, FP above
    g = [0.5, 0.5, 0.4, 0.4]
    d = [0.5, 0.5, 0.4, 0.4 * 0.77]
    iou = E.box_iou(d, g)
    assert 0.75 <= iou < 0.8
    s = ap(one_image([d], [0.9], [g]))
    assert s["AP50"] == ONE and s["AP75"] == ONE and s["AP"] == pytest.approx(0.6, rel=1e-15)


def test_oracle_matches_pycocotools():
    pytest.importorskip("pycocotools")
    from pycocotools.coco import COCO
    from pycocotools.cocoeval import COCOeval
    rng = np.random.default_rng(5)
    n_img, k, size = 12, 4, 300.0
    gt, dt, parts, gid = [], [], [], 1
    for i in range(n_img):
        t = int(rng.integers(0, 6))
        gb = np.concatenate([rng.uniform(0.2, 0.8, (t, 2)), rng.uniform(0.05, 0.4, (t, 2))], 1).astype(np.float32)
        gc = rng.integers(0, k, t).astype(np.float32)
        n = 3 * t + 2
        src = rng.integers(0, max(t, 1), n)
        db = (gb[src] if t else np.full((n, 4), 0.5, np.float32)) + rng.normal(0, 0.03, (n, 4)).astype(np.float32)
        db[:, 2:] = np.abs(db[:, 2:]) + 0.01
        dc = np.where(rng.uniform(size=n) < 0.8, gc[src] if t else 0, rng.integers(0, k, n)).astype(np.int64)
        sc = rng.uniform(0.05, 1.0, n).astype(np.float32)
        kept = np.full((1, k, n), -1, np.int32)
        count = np.zeros((1, k), np.int32)
        ks = np.zeros((1, k, n), np.float32)
        for c in range(k):
            idx = np.nonzero(dc == c)[0]
            idx = idx[np.lexsort((idx, -sc[idx].astype(np.float64)))]
            kept[0, c, :idx.size], count[0, c], ks[0, c, :idx.size] = idx, idx.size, sc[idx]
            for j in idx:
                x, y, w, h = (float(v) * size for v in db[j])
                dt.append({"image_id": i + 1, "category_id": c + 1, "bbox": [x - w / 2, y - h / 2, w, h],
                           "score": float(sc[j])})
        for j in range(t):
            x, y, w, h = (float(v) * size for v in gb[j])
            gt.append({"id": gid, "image_id": i + 1, "category_id": int(gc[j]) + 1, "bbox": [x - w / 2, y - h / 2, w, h],
                       "area": w * h, "iscrowd": 0})
            gid += 1
        parts.append(E.evaluate_batch(kept, count, ks, db[None], gb, gc, np.array([0, t], np.int32), i, THR, 100))
    cg = COCO()
    cg.dataset = {"images": [{"id": i + 1} for i in range(n_img)], "annotations": gt,
                  "categories": [{"id": c + 1} for c in range(k)]}
    cg.createIndex()
    ev = COCOeval(cg, cg.loadRes(dt), "bbox")
    ev.evaluate()
    ev.accumulate()
    p, r, _, _ = E.coco_accumulate(*E.merge(*parts), k + 1, len(THR))
    np.testing.assert_allclose(p, ev.eval["precision"][:, :, :, 0, 2], atol=1e-12)
    np.testing.assert_allclose(r, ev.eval["recall"][:, :, 0, 2], atol=1e-12)


# ---- the C ABI without a GPU -----------------------------------------------------------------------------
@pytest.fixture(scope="module")
def native():
    import build_native
    build_native.build()
    from ssdgeom import _native
    return _native


def test_state_size_formula(native):
    lib = native.lib()
    k, m, d = 80, 5000, 100
    slots = k * m * d
    keys_off = (64 * 4 + slots * 4 + k * m * 4 + 255) // 256 * 256
    assert lib.ssdg_eval_state_bytes(81, m, d, 10) == (keys_off + slots * 8 + 255) // 256 * 256
    assert abs(lib.ssdg_eval_state_bytes(81, m, d, 10) / 1e6 - 481.6) < 0.1       # ~12 B per slot
    for args in ((81, 1 << 22, 100, 10), (81, 5000, 1025, 10), (81, 5000, 100, 17), (1, 5000, 100, 10),
                 (81, 0, 100, 10), (81, 5000, 100, 0), (1025, 30000, 100, 10)):
        assert lib.ssdg_eval_state_bytes(*args) == 0, args


def test_exchange_buffers_cover_the_state(native):
    lib = native.lib()
    state = 1 << 20                 # never dereferenced: pointer arithmetic only
    ptr, cnt = C.c_void_p(), C.c_int64()
    assert lib.ssdg_eval_exchange(state, 81, 7, 3, 0, C.byref(ptr), C.byref(cnt)) == 0
    keys_off = (64 * 4 + 80 * 7 * 3 * 4 + 80 * 7 * 4 + 255) // 256 * 256
    assert ptr.value == state + keys_off and cnt.value == 80 * 7 * 3
    assert lib.ssdg_eval_exchange(state, 81, 7, 3, 1, C.byref(ptr), C.byref(cnt)) == 0
    assert ptr.value == state and cnt.value == 64 + 80 * 7 * 3 + 80 * 7
    assert lib.ssdg_eval_exchange(state, 81, 7, 3, 2, C.byref(ptr), C.byref(cnt)) == native.ERR_ARG
    assert lib.ssdg_eval_exchange(state, 81, 1 << 22, 3, 0, C.byref(ptr), C.byref(cnt)) == native.ERR_LIMIT


def test_entry_points_reject_bad_arguments(native):
    lib = native.lib()
    f = 1 << 20                      # fake, aligned device pointers: every call below fails before any CUDA call
    thr = (C.c_double * 17)(*([0.5] * 17))

    def acc(top_k=200, batch=4, max_gt=100, n_thr=10, max_dets=100, image_base=0, max_images=5000, n_classes=81,
            state_bytes=1 << 40, boxes=f):
        return lib.ssdg_eval_accumulate(f, f, f, top_k, boxes, batch, 8732, n_classes, f, f, f, max_gt, thr, n_thr,
                                        max_dets, image_base, max_images, f, state_bytes, None)
    assert acc(max_dets=201) == native.ERR_ARG                       # max_dets > top_k
    assert acc(n_thr=17) == native.ERR_LIMIT
    assert acc(n_thr=0) == native.ERR_ARG
    assert acc(image_base=4998) == native.ERR_ARG                    # image_base + batch > max_images
    assert acc(image_base=-1) == native.ERR_ARG
    assert acc(max_images=1 << 22) == native.ERR_LIMIT
    assert acc(max_dets=1025, top_k=2000) == native.ERR_LIMIT
    assert acc(max_gt=2049) == native.ERR_LIMIT
    assert acc(n_classes=1) == native.ERR_ARG
    assert acc(state_bytes=1000) == native.ERR_WORKSPACE
    assert acc(boxes=f + 4) == native.ERR_ALIGN
    assert lib.ssdg_eval_accumulate(None, f, f, 200, f, 4, 8732, 81, f, f, f, 100, thr, 10, 100, 0, 5000, f,
                                    1 << 40, None) == native.ERR_ARG
    rec = (C.c_double * 300)()
    fin = lib.ssdg_eval_finalize
    assert fin(f, 1 << 40, 81, 5000, 100, 17, rec, 101, f, f, f, f, f, 1 << 40, None) == native.ERR_LIMIT
    assert fin(f, 1 << 40, 81, 5000, 100, 10, rec, 257, f, f, f, f, f, 1 << 40, None) == native.ERR_LIMIT
    assert fin(f, 1 << 40, 81, 5000, 100, 10, None, 101, f, f, f, f, f, 1 << 40, None) == native.ERR_ARG
    assert fin(f, 1000, 81, 5000, 100, 10, rec, 101, f, f, f, f, f, 1 << 40, None) == native.ERR_WORKSPACE
    assert lib.ssdg_eval_reset(None, 10, None) == native.ERR_ARG
    assert lib.ssdg_eval_status(None, None, None) == native.ERR_ARG
