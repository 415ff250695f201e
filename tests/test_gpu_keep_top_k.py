"""GPU (B200): the per-image keep_top_k (ssdg_detect_keep_top_k, ops.keep_top_k) bit for bit against its NumPy
restatement (tests/keep_top_k_oracle.py) fed the same inputs -- random lists, exact ties, the size limits, prior
indices outside the prior set -- and the layers above it: ssd_model.detections, the evaluator fed the capped counts,
and HotPath(keep_top_k=K)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import keep_top_k_oracle as O                         # noqa: E402  (the checker)
from ssdgeom import ops, synth                        # noqa: E402
from ssdgeom.evaluate import DetectionEvaluator       # noqa: E402
from ssdgeom.models import ssd_model as M             # noqa: E402
from ssdgeom.pipeline import HotPath                  # noqa: E402
from test_gpu_eval import assert_same_result, oracle_of   # noqa: E402
from test_keep_top_k_oracle import rand_lists         # noqa: E402

CACHE = 16384          # candidate slots per image the kernel can keep in shared memory (csrc/detect.cu kTopkCache)
KEYS = ("prior", "class", "score", "box", "n", "count")


def device_top(kept, count, score, boxes, K):
    det = {"kept": kept, "count": count, "kept_score": score}
    if boxes is not None:
        det["boxes"] = boxes
    out = ops.keep_top_k(det, K)
    return {k: out[k].to_host() for k in KEYS if k in out}


def assert_bit_equal(got, want):
    for key, w in zip(KEYS, want):
        if w is None:
            assert key not in got
            continue
        g = got[key]
        assert g.dtype == w.dtype and g.shape == w.shape, key
        assert np.array_equal(g.view(np.uint32) if g.dtype == np.float32 else g,
                              w.view(np.uint32) if w.dtype == np.float32 else w), key


def totals(count, top_k):
    return np.clip(count, 0, top_k).sum(axis=1)


# ---- random lists -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_classes", [2, 6, 81])
@pytest.mark.parametrize("top_k", [1, 12, 200, 1024])
def test_random_lists_equal_the_oracle(n_classes, top_k):
    kept, count, score, boxes = rand_lists(100 + n_classes + top_k, 5, n_classes, top_k)
    score = score * np.random.default_rng(top_k).choice(np.float32([1, 1, 1, 0.999]), score.shape[:2])[..., None]
    score = np.sort(score, axis=-1)[..., ::-1].astype(np.float32).copy()   # levels and their scaled copies
    tot = int(totals(count, top_k).max())
    assert totals(count, top_k)[0] == 0 and (count > top_k).any() and (count < 0).any()
    paths = set()
    for K in sorted({1, 5, tot - 1, tot, tot + 1, 1024}):
        if not 1 <= K <= 1024:
            continue
        assert_bit_equal(device_top(kept, count, score, boxes, K), O.keep_top_k(kept, count, score, boxes, K))
        t = totals(count, min(top_k, K))         # what the kernel reads: no list contributes more than K
        paths |= {"select" if x > K else "all" for x in t}
        paths |= {"global" for x in t if x > K and (n_classes - 1) * min(top_k, K) > CACHE}
    assert "all" in paths and ("select" in paths or n_classes == 2)   # one list never holds more than K candidates
    if n_classes == 81 and top_k == 1024:
        assert "global" in paths                    # the select that reads global memory on every pass
    # without boxes: no box output
    got = device_top(kept, count, score, None, 5)
    assert_bit_equal(got, O.keep_top_k(kept, count, score, None, 5))


# ---- exact ties ----------------------------------------------------------------------------------------------
def test_all_scores_equal_cut_inside_the_run():
    b, k, top_k = 3, 9, 20
    rng = np.random.default_rng(3)
    kept = rng.integers(0, 50, (b, k, top_k)).astype(np.int32)
    count = rng.integers(0, top_k + 1, (b, k)).astype(np.int32)
    score = np.full((b, k, top_k), 0.5, np.float32)
    boxes = rng.uniform(0, 1, (b, 50, 4)).astype(np.float32)
    for K in (1, 7, 33, max(1, int(totals(count, top_k).min()) - 1), 150):
        got = device_top(kept, count, score, boxes, K)
        assert_bit_equal(got, O.keep_top_k(kept, count, score, boxes, K))
        c = got["count"]
        # the run of equal scores is cut in class order: full classes, one partial one, then empty ones
        for i in range(b):
            part = np.nonzero(c[i] != np.minimum(count[i], top_k))[0]
            assert part.size == 0 or np.all(c[i, part[1:]] == 0)


def test_levels_one_ulp_apart_at_the_cut():
    b, k, top_k = 4, 7, 30
    rng = np.random.default_rng(4)
    hi = np.float32(0.25)
    lo = np.nextafter(hi, np.float32(0))
    kept = rng.integers(0, 64, (b, k, top_k)).astype(np.int32)
    count = np.full((b, k), top_k, np.int32)
    n_hi = rng.integers(0, top_k + 1, (b, k))
    score = np.where(np.arange(top_k)[None, None, :] < n_hi[..., None], hi, lo).astype(np.float32)
    boxes = rng.uniform(0, 1, (b, 64, 4)).astype(np.float32)
    for i in range(b):
        K = int(n_hi[i].sum())          # the cut exactly between the two levels for image i, inside a run elsewhere
        for kk in (K - 1, K, K + 1):
            if 1 <= kk <= 1024:
                assert_bit_equal(device_top(kept, count, score, boxes, kk), O.keep_top_k(kept, count, score, boxes, kk))


def test_negative_zero_next_to_positive_zero():
    b, k, top_k = 2, 5, 8
    rng = np.random.default_rng(5)
    kept = rng.integers(0, 20, (b, k, top_k)).astype(np.int32)
    count = np.full((b, k), top_k, np.int32)
    score = np.zeros((b, k, top_k), np.float32)
    score[..., :2] = 0.75
    score[..., 2:] = np.where(rng.uniform(size=(b, k, top_k - 2)) < 0.5, np.float32(0.0), np.float32(-0.0))
    boxes = rng.uniform(0, 1, (b, 20, 4)).astype(np.float32)
    for K in (3, 10, 17, 40):
        got = device_top(kept, count, score, boxes, K)
        assert_bit_equal(got, O.keep_top_k(kept, count, score, boxes, K))
    assert np.signbit(got["score"][got["score"] == 0]).any()     # the -0 scores are carried through unchanged


# ---- the sizes the limits allow ----------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [100, 200])
def test_every_list_full_ssd300(K):
    b, k, top_k = 8, 80, 200
    rng = np.random.default_rng(K)
    kept = rng.integers(0, 8732, (b, k, top_k)).astype(np.int32)
    count = np.full((b, k), top_k, np.int32)
    score = np.sort(rng.integers(1, 400, (b, k, top_k)) / np.float32(400), axis=-1)[..., ::-1].astype(np.float32).copy()
    boxes = rng.uniform(0, 1, (b, 8732, 4)).astype(np.float32)
    assert_bit_equal(device_top(kept, count, score, boxes, K), O.keep_top_k(kept, count, score, boxes, K))


def test_largest_shape():
    b, k, top_k = 2, 2047, 1024
    rng = np.random.default_rng(6)
    kept = rng.integers(0, 30000, (b, k, top_k)).astype(np.int32)
    count = np.full((b, k), top_k, np.int32)
    count[1, ::3] = rng.integers(0, top_k, count[1, ::3].size)
    score = np.sort(rng.integers(1, 5000, (b, k, top_k)) / np.float32(5000), axis=-1)[..., ::-1].astype(np.float32).copy()
    boxes = rng.uniform(0, 1, (b, 30000, 4)).astype(np.float32)
    for K in (1, 1000, 1024):
        assert_bit_equal(device_top(kept, count, score, boxes, K), O.keep_top_k(kept, count, score, boxes, K))


def test_prior_outside_the_prior_set_gets_a_zero_box():
    b, k, top_k, a = 2, 4, 6, 10
    kept = np.array([-5, a, a + 100, 3, -1, 2], np.int32)[None, None].repeat(b, 0).repeat(k, 1)
    count = np.full((b, k), top_k, np.int32)
    score = np.linspace(0.9, 0.4, top_k, dtype=np.float32)[None, None].repeat(b, 0).repeat(k, 1).copy()
    boxes = np.random.default_rng(7).uniform(0.1, 1, (b, a, 4)).astype(np.float32)
    got = device_top(kept, count, score, boxes, 24)
    assert_bit_equal(got, O.keep_top_k(kept, count, score, boxes, 24))
    bad = (got["prior"] < 0) | (got["prior"] >= a)
    assert bad.sum() == b * k * 4 and np.all(got["box"][bad] == 0) and np.all(got["box"][~bad] != 0)


# ---- end to end ----------------------------------------------------------------------------------------------------
def trained_case(seed, b):
    priors = M.build_prior_box(synth.SSD300["sizes"])
    gt, gcls, off = synth.make_gt(seed, b, 100, "coco")
    t = ops.match_encode(gt, gcls, off, priors, b, int(np.diff(off).max()), 0.5)
    pc, pb = synth.make_trained_predictions(seed, t["cls"].to_host(), t["loc"].to_host(), t["mask"].to_host())
    return priors, gt, gcls, off, pc, pb


def test_detect_then_keep_top_k_and_ssd_model_detections():
    priors, _, _, _, pc, pb = trained_case(31, 64)
    det = ops.detect(pc, pb, priors, want_scores=True, want_boxes=True)
    host = {k: det[k].to_host() for k in ("kept", "count", "kept_score", "boxes")}
    tot = totals(host["count"], 200)
    assert tot.max() > 1
    for K in sorted({1, 20, 200, min(max(1, int(np.median(tot)) // 2), 1024), min(int(tot.max()) + 1, 1024)}):
        top = ops.keep_top_k(det, K)
        want = O.keep_top_k(host["kept"], host["count"], host["kept_score"], host["boxes"], K)
        assert_bit_equal({k: top[k].to_host() for k in KEYS}, want)
    res = M.detections(pc, pb, priors, keep_top_k=20)
    want = O.keep_top_k(host["kept"], host["count"], host["kept_score"], host["boxes"], 20)
    for key, w in (("priors", want[0]), ("labels", want[1]), ("scores", want[2]), ("boxes", want[3]), ("n", want[4])):
        assert np.array_equal(res[key], w), key
    geo = M.SSDBoxGeometry()
    assert all(np.array_equal(v, res[k]) for k, v in geo.detections(pc, pb, keep_top_k=20).items())


@pytest.mark.parametrize("K", [5, 100, 1024])
def test_evaluator_on_capped_counts(K):
    b = 32
    priors, gt, gcls, off, pc, pb = trained_case(32, b)
    det = ops.detect(pc, pb, priors, want_scores=True, want_boxes=True)
    host = {k: det[k].to_host() for k in ("kept", "count", "kept_score", "boxes")}
    top = ops.keep_top_k(det, K)
    capped = top["count"].to_host()
    ev = DetectionEvaluator(max_images=b)
    ev.add(dict(det, count=top["count"]), gt, gcls, off)
    res = ev.summarize()
    assert_same_result(res, oracle_of(dict(host, count=capped), gt, gcls, off), 81)
    if K >= totals(host["count"], 200).max():
        assert np.array_equal(capped, host["count"])
        alone = DetectionEvaluator(max_images=b)
        alone.add(det, gt, gcls, off)
        want = alone.finalize()
        assert all(np.array_equal(res[k], want[k]) for k in want)
    else:
        assert (capped < host["count"]).any()


@pytest.mark.parametrize("depth", [1, 2])
@pytest.mark.parametrize("with_evaluator", [False, True])
def test_hotpath_keep_top_k(depth, with_evaluator):
    b, n_batches, K = 32, 3, 50
    batches = [trained_case(60 + k, b) for k in range(n_batches)]
    priors = batches[0][0]
    total = max(x[1].shape[0] for x in batches)
    pad = [(np.concatenate([gt, np.zeros((total - gt.shape[0], 4), np.float32)]),
            np.concatenate([gcls, np.zeros(total - gcls.shape[0], np.float32)]), off, pc, pb)
           for _, gt, gcls, off, pc, pb in batches]

    def run(keep, evaluator):
        hp = HotPath(synth.SSD300, batch=b, max_gt=100, total_gt=total, depth=depth, evaluator=evaluator,
                     keep_top_k=keep)
        outs = []
        for k in range(n_batches):
            if k:
                hp.add_input_set()
            hp.use_set(k)
            hp.upload(*pad[k])
        for k in range(n_batches):
            hp.use_set(k)
            hp.step(image_base=k * b)
            o = (np.zeros(16), np.zeros((b, 80, 200), np.int32), np.zeros((b, 80), np.int32))
            hp.download(*o)
            top = None
            if keep is not None:
                top = {"prior": np.zeros((b, K), np.int32), "class": np.zeros((b, K), np.int32),
                       "score": np.zeros((b, K), np.float32), "box": np.zeros((b, K, 4), np.float32),
                       "n": np.zeros(b, np.int32), "count": np.zeros((b, 80), np.int32)}
                hp.download_detections(top)
            outs.append((o, top))
        hp.s_main.sync()
        hp.check_status()
        return hp, outs

    ev = DetectionEvaluator(max_images=n_batches * b) if with_evaluator else None
    hp, with_top = run(K, ev)
    hp0, without = run(None, None)
    assert hp.kernel_launches_per_step == hp0.kernel_launches_per_step + 1 + (1 if with_evaluator else 0)
    assert hp0.top is None and "kept_score" not in hp0.det
    alone = DetectionEvaluator(max_images=n_batches * b)
    for k, ((o, top), (o0, _)) in enumerate(zip(with_top, without)):
        assert all(np.array_equal(u, v) for u, v in zip(o, o0))          # loss block, kept, count unchanged
        _, gt, gcls, off, pc, pb = batches[k]
        det = ops.detect(pc, pb, priors, want_scores=True, want_boxes=True)
        t = ops.keep_top_k(det, K)
        assert np.array_equal(det["kept"].to_host(), o[1])
        for key in top:
            assert np.array_equal(top[key], t[key].to_host()), key
        alone.add(dict(det, count=t["count"]), gt, gcls, off, image_base=k * b)
    if with_evaluator:
        got, want = ev.finalize(), alone.finalize()
        assert all(np.array_equal(got[k], want[k]) for k in want)
