"""CPU: the per-image keep_top_k restatement (tests/keep_top_k_oracle.py) against an independent formulation,
the prefix property its per-class counts rely on, and the argument errors of ssdg_detect_keep_top_k (no GPU needed:
they are returned before any CUDA call)."""
import ctypes as C
import os

import numpy as np
import pytest

import keep_top_k_oracle as O    # the checker

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LEVELS = np.array([0.95, 0.9, 0.7, 0.5, 0.3, 0.2, 0.05], np.float32)   # test_gpu_eval.rand_case: ties across classes


def rand_lists(seed, b, n_classes, top_k, a=40):
    """Score-sorted class lists on discrete levels; counts beyond top_k, negative counts and empty images."""
    rng = np.random.default_rng(seed)
    k = n_classes - 1
    kept = rng.integers(-2, a + 2, (b, k, top_k)).astype(np.int32)     # indices outside [0, A) included
    count = rng.integers(-3, top_k + 4, (b, k)).astype(np.int32)
    count[rng.uniform(size=(b, k)) < 0.3] = 0
    count[0] = 0
    count[1, 0], count[-1, -1] = -1, top_k + 1
    score = np.sort(rng.choice(LEVELS, (b, k, top_k)), axis=-1)[..., ::-1].copy()
    boxes = rng.uniform(0, 1, (b, a, 4)).astype(np.float32)
    return kept, count, score, boxes


def by_sorted(kept, count, score, boxes, K):
    """The contract with Python's sorted over (-score, class, position) tuples."""
    b, k, top_k = kept.shape
    a = boxes.shape[1]
    res = []
    for i in range(b):
        cand = [(-float(score[i, c, j]), c, j) for c in range(k) for j in range(min(max(int(count[i, c]), 0), top_k))]
        sel = sorted(cand)[:K]
        prior = [int(kept[i, c, j]) for _, c, j in sel]
        box = [boxes[i, p] if 0 <= p < a else np.zeros(4, np.float32) for p in prior]
        res.append((prior, [c for _, c, _ in sel], [score[i, c, j] for _, c, j in sel], box,
                    np.bincount([c for _, c, _ in sel], minlength=k)))
    return res


@pytest.mark.parametrize("seed,n_classes,top_k,K", [(1, 2, 5, 3), (2, 6, 12, 1), (3, 6, 12, 5), (4, 6, 12, 40),
                                                      (5, 21, 8, 17), (6, 6, 12, 100)])
def test_oracle_equals_sorted_tuples(seed, n_classes, top_k, K):
    kept, count, score, boxes = rand_lists(seed, 7, n_classes, top_k)
    prior, cls, sc, box, n, cnt = O.keep_top_k(kept, count, score, boxes, K)
    want = by_sorted(kept, count, score, boxes, K)
    for i, (wp, wc, ws, wb, wcnt) in enumerate(want):
        m = len(wp)
        assert n[i] == m
        assert np.array_equal(prior[i, :m], wp) and np.all(prior[i, m:] == -1)
        assert np.array_equal(cls[i, :m], wc) and np.all(cls[i, m:] == -1)
        assert np.array_equal(sc[i, :m].view(np.uint32), np.array(ws, np.float32).view(np.uint32))
        assert np.all(sc[i, m:] == 0)
        assert np.array_equal(box[i, :m], np.array(wb, np.float32).reshape(m, 4)) and np.all(box[i, m:] == 0)
        assert np.array_equal(cnt[i], wcnt)
    assert n[0] == 0                              # an image without detections


def test_survivors_are_a_prefix_of_every_list():
    kept, count, score, boxes = rand_lists(7, 9, 11, 16)
    for K in (1, 4, 30, 200):
        prior, cls, _, box, n, cnt = O.keep_top_k(kept, count, score, None, K)
        assert box is None
        assert np.array_equal(cnt.sum(axis=1), n)
        assert np.all(cnt <= np.clip(count, 0, 16))
        for i in range(kept.shape[0]):
            for c in range(kept.shape[1]):
                m = cnt[i, c]
                # the class's survivors, in rank order, are exactly its first m entries in list order
                assert np.array_equal(prior[i, :n[i]][cls[i, :n[i]] == c], kept[i, c, :m])


def test_negative_zero_equals_positive_zero():
    kept = np.array([[[5, 6], [7, 8]]], np.int32)
    score = np.array([[[0.0, -0.0], [-0.0, 0.0]]], np.float32)
    prior, cls, sc, _, n, cnt = O.keep_top_k(kept, np.array([[2, 2]]), score, None, 3)
    assert list(prior[0]) == [5, 6, 7] and list(cls[0]) == [0, 0, 1] and n[0] == 3 and list(cnt[0]) == [2, 1]
    assert list(np.signbit(sc[0])) == [False, True, True]


@pytest.fixture(scope="module")
def native():
    import build_native
    build_native.build()
    from ssdgeom import _native
    return _native


def test_argument_errors_need_no_gpu(native):
    lib = native.lib()
    buf = (C.c_float * 64)()
    p = C.addressof(buf)
    al = (p + 15) // 16 * 16                      # 16-byte aligned inside the buffer

    def call(kept=al, count=al, score=al, top_k=200, boxes=None, batch=2, a=8732, n_classes=81, K=200, out=al,
             out_box=None, out_count=al):
        return lib.ssdg_detect_keep_top_k(kept, count, score, top_k, boxes, batch, a, n_classes, K, out, out, out,
                                          out_box, out, out_count, None)

    assert call(K=0) == native.ERR_ARG
    assert call(K=1025) == native.ERR_LIMIT
    assert call(score=None) == native.ERR_ARG
    assert call(kept=None) == native.ERR_ARG
    assert call(boxes=al + 4, out_box=al) == native.ERR_ALIGN
    assert call(boxes=al, out_box=al + 4) == native.ERR_ALIGN
    assert call(out_box=al) == native.ERR_ARG            # a box output needs the boxes
    assert call(n_classes=1) == native.ERR_ARG
    assert call(n_classes=2049) == native.ERR_LIMIT
    assert call(top_k=1025) == native.ERR_LIMIT
    assert call(batch=0) == native.ERR_ARG
