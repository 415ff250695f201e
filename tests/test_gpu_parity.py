"""GPU (B200): parity of the CUDA path -- called through the C ABI via ssdgeom's ctypes layer --
against the CPU oracle (oracle/ssd_oracle.py) and the fixtures the unmodified reference produced
(tests/golden, oracle/make_golden.py).

Contract (SURVEY.md section 8c):
  bit-exact      labeled_cls, labeled_boxes, mask, matched index, priors, NMS kept indices
  <= 1e-5 rel    encoded offsets, decoded boxes, loss terms, per-prior CE, softmax scores
"""
import hashlib
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import ssd_oracle as O          # noqa: E402  (the checker)
from ssdgeom import synth                   # noqa: E402
from ssdgeom import ops, device as D        # noqa: E402
from ssdgeom.utils import bbox              # noqa: E402
from ssdgeom.models import ssd_model as M   # noqa: E402

RTOL = 1e-5


def sha(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(str(a.dtype).encode() + str(a.shape).encode() + a.tobytes())
    return h.hexdigest()


def close(got, want, rtol=RTOL, atol=0.0):
    np.testing.assert_allclose(np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64), rtol=rtol, atol=atol)


@pytest.fixture(scope="module")
def priors300():
    return O.build_prior_box()


@pytest.fixture(scope="module")
def priors512():
    t = synth.SSD512
    return O.build_prior_box(t["sizes"], t["s_k_refer"], t["aspect_ratio"], t["input_size"])


@pytest.fixture(scope="module")
def priors_large():
    """SSD512's table with a 96 x 96 first feature map: 45 044 priors, 1 408 tiles of 32."""
    t = synth.SSD512
    return O.build_prior_box([(96, 96)] + t["sizes"][1:], t["s_k_refer"], t["aspect_ratio"], t["input_size"])


def _check_large_prior_path(priors, out):
    # more than kTileSmemMax (csrc/match.cu) tiles of 32 priors: the single-level row search, and match_kernel
    # reads the tile statistics from global memory
    assert priors.shape[0] > 32 * 1024
    assert ops.match_status(out) & 4 == 0     # every pair fit the pair list: no exhaustive rescan


# ---- A1 ----------------------------------------------------------------------------------------------
def test_priors_ssd300_bit_exact(golden_dir, priors300):
    got = M.build_prior_box(synth.SSD300["sizes"])
    want = np.load(os.path.join(golden_dir, "priors_ssd300.npz"))["priors"]
    assert got.dtype == np.float64 and got.shape == (8732, 4)
    assert np.array_equal(got, want)          # the reference's own output, bit for bit
    assert np.array_equal(M.SSDBoxGeometry().get_prior_box(), want)


def test_priors_ssd512_bit_exact(priors512):
    t = synth.SSD512
    got = M.build_prior_box(t["sizes"], t["s_k_refer"], t["aspect_ratio"], t["input_size"])
    assert got.shape == (24564, 4)
    assert np.array_equal(got, priors512)


# ---- input glue (section 8f row 3) --------------------------------------------------------------------
def test_gt_prepare_and_image_normalize_bit_exact():
    rng = np.random.default_rng(5)
    sizes = [(640, 427), (500, 375), (333, 500), (1, 1), (4000, 3000)]
    counts = [9, 1, 40, 3, 0]
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    rows = [np.concatenate([rng.uniform(0, [w, h], (t, 2)), rng.uniform(0.5, [w, h], (t, 2))], 1)
            for (w, h), t in zip(sizes, counts)]
    xywh = np.concatenate(rows)
    want = np.concatenate([O.coco_to_ssd_boxes(r, w, h) for r, (w, h) in zip(rows, sizes)])
    got = ops.gt_prepare(xywh, np.array(sizes, np.int32), off).to_host()
    assert got.dtype == np.float32 and np.array_equal(got, want)
    want32 = np.concatenate([O.coco_to_ssd_boxes(r.astype(np.float32), w, h) for r, (w, h) in zip(rows, sizes)])
    assert np.array_equal(ops.gt_prepare(xywh.astype(np.float32), np.array(sizes, np.int32), off).to_host(), want32)
    for n in (1, 7, 300 * 300 * 3 * 2 + 1):
        x = rng.uniform(-0.2, 1.2, n).astype(np.float32)
        assert np.array_equal(ops.image_normalize(x).to_host(), O.normalize_image(x))


def test_gt_prepare_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "glue_small.npz"))      # outputs of the unmodified reference
    got = ops.gt_prepare(g["xywh"], g["img_wh"], g["offsets"]).to_host()
    assert np.array_equal(got, g["rel"])


def test_train_batches_iterator_matches_per_image_oracle(priors300):
    """get_train_set semantics (models/ssd_model.py:209-227): per-image match + encode + image scaling, batched,
    trailing partial batch dropped."""
    from ssdgeom import data
    rng = np.random.default_rng(6)
    items = []
    for i in range(7):
        w, h, t = int(rng.integers(200, 700)), int(rng.integers(200, 700)), int(rng.integers(1, 12))
        xywh = np.concatenate([rng.uniform(0, [w * 0.7, h * 0.7], (t, 2)), rng.uniform(8, [w * 0.3, h * 0.3], (t, 2))], 1)
        items.append((rng.uniform(0, 1, (30, 30, 3)).astype(np.float32), rng.integers(0, 80, t).astype(np.float32), xywh, (w, h)))
    batches = list(data.TrainBatches(items, priors300, batch_size=3, coco_pixels=True))
    assert len(batches) == 2                                    # 7 images, batch 3, remainder dropped (:225)
    k = 0
    for images, (cls, loc, mask) in batches:
        assert images.shape == (3, 30, 30, 3) and cls.shape == (3, 8732) and loc.shape == (3, 8732, 4)
        assert cls.dtype == np.int32 and loc.dtype == np.float32 and mask.dtype == bool
        for i in range(3):
            image, c, xywh, (w, h) = items[k]
            box = O.coco_to_ssd_boxes(xywh, w, h)
            w_cls, w_loc, w_mask = O.assign_encode(c, box, priors300, sweeps=False)
            assert np.array_equal(cls[i], w_cls) and np.array_equal(mask[i], w_mask)
            close(loc[i], w_loc)
            assert np.array_equal(images[i], O.normalize_image(image))
            k += 1


# ---- A10 / A2 ---------------------------------------------------------------------------------------
IOU_KAT = [([10, 10, 2, 2], [10, 10, 2, 2], 1.0), ([10, 10, 1, 1], [20, 20, 1, 1], 0.0),
           ([10, 10, 2, 2], [10, 10, 4, 4], 0.25), ([10, 10, 0, 0], [20, 20, 0, 0], 0.0),
           ([10, 10, -1, -1], [10, 10, -1, -1], 0.0), ([10, 10, 2, 2], [11, 11, 2, 2], 1 / 7),
           ([10, 10, 6, 6], [13, 13, 2, 2], 1 / 39), ([10, -10, 1, 1], [10, -10, 1, 1], 1.0)]


@pytest.mark.parametrize("a,b,want", IOU_KAT)
def test_iou_known_answers(a, b, want):
    assert abs(float(bbox.iou(a, b)) - want) < 5e-5          # reference tests/utils/test_bbox.py:10-17


def test_iou_n_bit_exact_all_dtype_mixes():
    rng = np.random.default_rng(0)
    n = 5000
    b1 = np.concatenate([rng.uniform(0, 1, (n, 2)), rng.uniform(0.01, 0.6, (n, 2))], 1)
    b2 = np.concatenate([b1[:, :2] + rng.normal(0, 0.1, (n, 2)), rng.uniform(0.01, 0.6, (n, 2))], 1)
    for d1 in (np.float32, np.float64):
        for d2 in (np.float32, np.float64):
            got = bbox.iou_n(b1.astype(d1), b2.astype(d2))
            want = O.iou_n(b1.astype(d1), b2.astype(d2))
            assert got.dtype == want.dtype
            assert np.array_equal(got, want), (d1, d2)
    a = np.array([[10, 10, 2, 2], [10, 10, 1, 1], [10, 10, 2, 2]], dtype=np.float32)
    b = np.array([[10, 10, 2, 2], [20, 20, 1, 1], [10, 10, 4, 4]], dtype=np.float32)
    np.testing.assert_allclose(bbox.iou_n(a, b), [1.0, 5.0000002e-21, 0.25], rtol=1e-6)


# ---- A3 / A4 ----------------------------------------------------------------------------------------
def test_match_small_golden_bit_exact(golden_dir):
    """Small and degenerate inputs in every dtype mix, outputs of the unmodified reference."""
    g = np.load(os.path.join(golden_dir, "match_small.npz"))
    for name in g["names"]:
        cls, box, mask, match = bbox.match_bbox(g[name + "_cls_in"], g[name + "_box_in"], g[name + "_pri_in"],
                                                float(g[name + "_thresh"]), return_match=True)
        assert np.array_equal(cls, g[name + "_cls"]), name
        assert np.array_equal(box, g[name + "_box"]), name
        assert np.array_equal(mask, g[name + "_mask"]), name
        assert cls.dtype == np.int32 and box.dtype == np.float32 and mask.dtype == bool
        assert np.array_equal(match >= 0, mask), name
        with np.errstate(all="ignore"):
            enc = bbox.apply_anchor_box(box, g[name + "_pri_in"])
        want = g[name + "_enc"]
        ok = np.isfinite(want)
        close(enc[ok], want[ok], rtol=1e-5, atol=1e-12)


def test_match_reference_known_answers():
    d = np.array([[10, 10, 1, 1], [20, 20, 1, 1], [20, 20, 0.5, 0.5]])
    t = np.array([[0, 10, 10, 0.5, 0.5], [1, 20, 20, 1, 1], [2, 20, 20, 0.5, 0.5]])
    cls, loc, mask = bbox.match_bbox(t[:, 0], t[:, 1:], d)
    np.testing.assert_almost_equal(loc, t[:, 1:])                     # tests/utils/test_bbox.py:35-39
    d = np.array([[10, 10, 1, 1], [20, 20, 1.1, 1.1], [20, 20, 0.5, 0.5]])
    t = np.array([[0, 15, 15, 13, 13], [1, 15, 15, 14, 14]])
    cls, loc, mask = bbox.match_bbox(t[:, 0], t[:, 1:], d)
    np.testing.assert_almost_equal(loc, np.array([[15, 15, 14, 14], [15, 15, 13, 13], [0, 0, 0, 0]]))  # :40-44
    assert cls.tolist() == [1, 0, 0] and mask.tolist() == [True, True, False]


def _config1_inputs():
    b_max, c_max, o_max = synth.make_gt(0, 4, 100, "max")
    b_coco, c_coco, o_coco = synth.make_gt(1, 4, 100, "coco")
    return (np.concatenate([b_max, b_coco]), np.concatenate([c_max, c_coco]),
            np.concatenate([o_max, o_coco[1:] + o_max[-1]]).astype(np.int32))


def test_assign_config1_golden(golden_dir, priors300):
    """BASELINE config 1 (8 SSD300 images, <= 100 GT) against the reference's recorded outputs."""
    g = np.load(os.path.join(golden_dir, "assign_ssd300.npz"))
    boxes, cls, offsets = _config1_inputs()
    assert sha(boxes, cls, offsets, priors300) == str(g["input_sha"])
    out = ops.match_encode(boxes, cls, offsets, priors300, 8, 100, 0.5, want=("cls", "box", "loc", "mask", "match"))
    assert ops.match_status(out) & 11 == 0
    o_cls, o_box, o_loc = out["cls"].to_host(), out["box"].to_host(), out["loc"].to_host()
    o_mask = out["mask"].to_host().astype(bool)
    for i in range(8):
        assert sha(o_cls[i]) == str(g["sha_cls"][i]), i
        assert sha(o_box[i]) == str(g["sha_box"][i]), i
        assert sha(o_mask[i]) == str(g["sha_mask"][i]), i
        ps, pe = g["pos_offsets"][i], g["pos_offsets"][i + 1]
        assert np.array_equal(np.nonzero(o_mask[i])[0], g["pos_index"][ps:pe])
        close(o_loc[i][o_mask[i]], g["pos_loc"][ps:pe])
        want_loc = O.apply_anchor_box(o_box[i], priors300).astype(np.float32)
        close(o_loc[i], want_loc)
        exact = np.mean(o_loc[i] == want_loc)
        assert exact > 0.999, exact        # float64 evaluation on both sides: expected identical


@pytest.mark.parametrize("table,batch,max_t,mode,seed", [
    ("ssd300", 16, 100, "max", 3), ("ssd300", 32, 100, "coco", 4), ("ssd300", 8, 37, "max", 5),
    ("ssd512", 4, 100, "max", 6), ("ssd512", 2, 500, "max", 7), ("large", 3, 100, "max", 8)])
def test_assign_random_bit_exact(table, batch, max_t, mode, seed, priors300, priors512, priors_large):
    priors = {"ssd300": priors300, "ssd512": priors512, "large": priors_large}[table]
    boxes, cls, off = synth.make_gt(seed, batch, max_t, mode)
    o_cls, o_loc, o_mask = bbox.match_encode_batch(boxes, cls, off, priors, 0.5)
    out = ops.match_encode(boxes, cls, off, priors, batch, int(np.diff(off).max()), 0.5, want=("box", "match"))
    if table == "large":
        _check_large_prior_path(priors, out)
    o_box, o_match = out["box"].to_host(), out["match"].to_host()
    for i in range(batch):
        s, e = off[i], off[i + 1]
        w_cls, w_box, w_mask, pairs = O.match_bbox(cls[s:e], boxes[s:e], priors, 0.5, sweeps=False, return_pairs=True)
        assert np.array_equal(o_cls[i], w_cls), i
        assert np.array_equal(o_box[i], w_box), i
        assert np.array_equal(o_mask[i], w_mask), i
        w_match = np.full(priors.shape[0], -1, np.int32)
        for t, a in pairs:
            w_match[a] = t
        assert np.array_equal(o_match[i], w_match), i
        close(o_loc[i], O.apply_anchor_box(w_box, priors).astype(np.float32))


@pytest.mark.parametrize("table,batch,max_t,mode", [("ssd300", 12, 100, "max"), ("ssd300", 16, 100, "coco"),
                                                   ("ssd512", 3, 100, "max"), ("ssd512", 2, 500, "max"),
                                                   ("large", 3, 100, "max")])
def test_assign_with_prior_index(table, batch, max_t, mode, priors300, priors512, priors_large):
    """The shape-sorted prior index is an acceleration structure only: identical outputs with and
    without it, and equal to the oracle."""
    priors = {"ssd300": priors300, "ssd512": priors512, "large": priors_large}[table]
    boxes, cls, off = synth.make_gt(41, batch, max_t, mode)
    want = ("cls", "box", "loc", "mask", "match")
    plain = ops.match_encode(boxes, cls, off, priors, batch, int(np.diff(off).max()), 0.5, want=want)
    if table == "large":
        _check_large_prior_path(priors, plain)
    d_pri = D.to_device(priors)
    idx = ops.prior_index(d_pri)
    assert ops.prior_index(d_pri) is idx                      # cached on the array
    fast = ops.match_encode(boxes, cls, off, d_pri, batch, int(np.diff(off).max()), 0.5, want=want)
    if table == "large":
        _check_large_prior_path(priors, fast)
    for k in want:
        assert np.array_equal(plain[k].to_host(), fast[k].to_host()), k
    for i in (0, batch - 1):
        w = O.match_bbox(cls[off[i]:off[i + 1]], boxes[off[i]:off[i + 1]], priors, 0.5, sweeps=False)
        assert np.array_equal(fast["cls"].to_host()[i], w[0]) and np.array_equal(fast["mask"].to_host()[i].astype(bool), w[2])
    # irregular priors (many distinct shapes -> single class, spatial blocking only) and float32 priors
    rng = np.random.default_rng(3)
    odd = np.concatenate([rng.uniform(0, 1, (1500, 2)), rng.uniform(0.03, 0.6, (1500, 2))], 1)
    for pri in (odd, odd.astype(np.float32), priors[::5].astype(np.float32)):
        d = D.to_device(pri)
        ops.prior_index(d)
        b2, c2, o2 = synth.make_gt(42, 4, 30, "max")
        a = ops.match_encode(b2, c2, o2, pri, 4, 30, 0.5, want=want)
        f = ops.match_encode(b2, c2, o2, d, 4, 30, 0.5, want=want)
        for k in want:
            assert np.array_equal(a[k].to_host(), f[k].to_host()), k
        w = O.match_bbox(c2[o2[1]:o2[2]], b2[o2[1]:o2[2]], pri, 0.5, sweeps=False)
        assert np.array_equal(f["cls"].to_host()[1], w[0]) and np.array_equal(f["mask"].to_host()[1].astype(bool), w[2])


def test_assign_edge_cases(priors300):
    pri = priors300[::7].copy()
    # duplicates, GT outside the image, tiny GT, T == 1, ragged offsets incl. an empty image
    boxes = np.array([[0.5, 0.5, 0.3, 0.3], [0.5, 0.5, 0.3, 0.3], [3.0, 3.0, 0.1, 0.1], [0.2, 0.7, 1e-4, 1e-4],
                      [0.31, 0.62, 0.25, 0.4]], dtype=np.float32)
    cls = np.array([1, 2, 3, 4, 5], dtype=np.float32)
    off = np.array([0, 4, 4, 5], dtype=np.int32)
    out = ops.match_encode(boxes, cls, off, pri, 3, 4, 0.5, want=("cls", "box", "mask"))
    o_cls, o_box, o_mask = out["cls"].to_host(), out["box"].to_host(), out["mask"].to_host().astype(bool)
    for i in (0, 2):
        s, e = off[i], off[i + 1]
        for sweeps in (True, False):
            w = O.match_bbox(cls[s:e], boxes[s:e], pri, 0.5, sweeps=sweeps)
            assert np.array_equal(o_cls[i], w[0]) and np.array_equal(o_box[i], w[1]) and np.array_equal(o_mask[i], w[2])
    assert not o_mask[1].any() and not o_cls[1].any() and not o_box[1].any()     # empty image: all unmatched
    # thresholds other than 0.5, float32 priors (all-float32 arithmetic path)
    b, c, o = synth.make_gt(9, 2, 20, "max")
    for thr in (0.3, 0.7, 1e-9, 2.0):
        for p in (pri, pri.astype(np.float32)):
            got = bbox.match_encode_batch(b, c, o, p, thr)
            for i in range(2):
                w = O.match_bbox(c[o[i]:o[i + 1]], b[o[i]:o[i + 1]], p, thr, sweeps=False)
                assert np.array_equal(got[0][i], w[0]) and np.array_equal(got[2][i], w[2]), (thr, p.dtype)


def test_assign_full_size_properties(priors300):
    """BASELINE batch size (256 x SSD300 x 100 GT): size-independent properties + a sampled exact check."""
    batch = 256
    boxes, cls, off = synth.make_gt(11, batch, 100, "max")
    out = ops.match_encode(boxes, cls, off, priors300, batch, 100, 0.5, want=("cls", "box", "loc", "mask", "match"))
    o_match, o_mask = out["match"].to_host(), out["mask"].to_host()
    o_box, o_cls = out["box"].to_host(), out["cls"].to_host()
    assert ops.match_status(out) & 11 == 0
    # forced assignment: every ground truth owns at least one prior; mask <=> match >= 0
    assert np.array_equal(o_mask.astype(bool), o_match >= 0)
    for i in range(batch):
        assert np.unique(o_match[i][o_match[i] >= 0]).size == 100
    # labeled boxes / classes are pure gathers of the inputs
    gt_b = boxes.reshape(batch, 100, 4)
    gt_c = cls.reshape(batch, 100).astype(np.int32)
    idx = np.maximum(o_match, 0)
    gathered = np.take_along_axis(gt_b, idx[..., None], axis=1) * o_mask[..., None]
    assert np.array_equal(o_box, gathered.astype(np.float32))
    assert np.array_equal(o_cls, np.take_along_axis(gt_c, idx, axis=1) * o_mask)
    # idempotence / determinism
    again = ops.match_encode(boxes, cls, off, priors300, batch, 100, 0.5, want=("match",))["match"].to_host()
    assert np.array_equal(again, o_match)
    # decode(encode) round trip on the positives
    dec = bbox.decode_bbox(out["loc"].to_host(), priors300, scale=1.0)
    close(dec[o_mask.astype(bool)], o_box[o_mask.astype(bool)], rtol=2e-5, atol=1e-6)
    for i in (0, 97, 255):
        w = O.match_bbox(cls[off[i]:off[i + 1]], boxes[off[i]:off[i + 1]], priors300, 0.5, sweeps=False)
        assert np.array_equal(o_cls[i], w[0]) and np.array_equal(o_box[i], w[1]) and np.array_equal(o_mask[i].astype(bool), w[2])


def test_encode_decode_against_oracle(priors300):
    rng = np.random.default_rng(2)
    g = np.concatenate([rng.uniform(0, 1, (3, 8732, 2)), np.exp(rng.uniform(np.log(0.02), np.log(0.9), (3, 8732, 2)))],
                       2).astype(np.float32)
    g[0, :5] = 0.0          # unmatched rows are all-zero boxes (utils/bbox.py:85)
    for i in range(3):
        enc = bbox.apply_anchor_box(g[i], priors300)
        want = O.apply_anchor_box(g[i], priors300)
        assert enc.dtype == want.dtype == np.float64
        close(enc, want, rtol=1e-12, atol=1e-15)
    loc = ops.encode(g, priors300).to_host()
    dec = bbox.decode_bbox(loc, priors300, scale=300.0)
    close(dec, O.decode_bbox(loc, priors300, scale=300.0), rtol=RTOL, atol=1e-7)
    assert np.array_equal(dec, O.decode_bbox(loc, priors300, scale=300.0, exp_dtype=np.float64)) or \
        np.mean(dec == O.decode_bbox(loc, priors300, scale=300.0, exp_dtype=np.float64)) > 0.9999


# ---- A6 ------------------------------------------------------------------------------------------------
def _targets(boxes, cls, off, priors, n):
    tgt = [O.assign_encode(cls[off[i]:off[i + 1]], boxes[off[i]:off[i + 1]], priors, sweeps=False) for i in range(n)]
    return tuple(np.stack([t[k] for t in tgt]) for k in range(3))


def _check_loss(y_true, y_pred, ratio=3):
    total, info, aux = M.ssd_loss(y_true, y_pred, neg_ratio=ratio, return_aux=True)
    w_total, w_info, w_aux = O.ssd_loss(y_true, y_pred, ratio=ratio, return_masks=True)
    close(total, w_total)
    for k in ("cls loss pos", "cls loss neg", "loc loss"):
        close(info[k], w_info[k])
    assert aux["num_pos"] == w_aux["num_pos"]
    # stage 1: per-prior mining input within tolerance of the float64 oracle
    close(aux["neg_ce"], w_aux["neg_ce"], rtol=RTOL, atol=1e-6)
    # stage 2: the mask is bit-exact given the kernel's own float32 CE vector
    kth, want_mask = O.hard_negative_select(aux["neg_ce"], aux["num_pos"], ratio)
    assert np.array_equal(aux["neg_mask"], want_mask)
    assert np.float32(aux["kth"]) == kth and aux["num_neg"] == int(want_mask.sum())
    # end to end (reported, expected equal: the top-k tail is sparse)
    flips = int(np.sum(aux["neg_mask"] != w_aux["neg_mask"]))
    return flips


def test_loss_golden(golden_dir, priors300):
    g = np.load(os.path.join(golden_dir, "loss_ssd300.npz"))
    boxes, cls, off = _config1_inputs()
    y_true = _targets(boxes, cls, off, priors300, 4)
    pred_cls, pred_box = synth.make_predictions(0, 4, 8732)
    assert sha(pred_cls, pred_box, *y_true) == str(g["input_sha"])
    total, info, aux = M.ssd_loss(y_true, (pred_box, pred_cls), return_aux=True)
    close(total, float(g["total"]))
    close(info["cls loss pos"], float(g["loss_pos"]))
    close(info["cls loss neg"], float(g["loss_neg"]))
    close(info["loc loss"], float(g["loss_loc"]))
    assert aux["num_pos"] == int(g["num_pos"])
    assert aux["num_neg"] == int(g["num_neg"])
    assert np.array_equal(np.packbits(aux["neg_mask"], axis=1), g["neg_mask_bits"])   # the reference's own mask


@pytest.mark.parametrize("batch,bias,seed", [(4, 7.0, 1), (16, 7.0, 2), (3, 0.0, 3), (1, 7.0, 4)])
def test_loss_random(batch, bias, seed, priors300):
    boxes, cls, off = synth.make_gt(seed, batch, 100, "coco" if seed % 2 else "max")
    y_true = _targets(boxes, cls, off, priors300, batch)
    pred_cls, pred_box = synth.make_predictions(seed, batch, 8732, bg_bias=bias)
    flips = _check_loss(y_true, (pred_box, pred_cls))
    assert flips == 0, "negative-mask flips vs the float64 oracle: %d" % flips


def test_loss_odd_sizes_and_ratios():
    rng = np.random.default_rng(8)
    for (b, a, c) in [(1, 37, 5), (3, 1000, 21), (2, 333, 81), (5, 64, 4)]:
        gt_cls = rng.integers(0, c - 1, (b, a)).astype(np.int32)
        gt_mask = rng.uniform(size=(b, a)) < 0.08
        gt_mask[0, 0] = True
        gt_box = rng.normal(size=(b, a, 4)).astype(np.float32)
        pred_box = rng.normal(size=(b, a, 4)).astype(np.float32)
        pred_cls = (rng.normal(size=(b, a, c)) * 3).astype(np.float32)
        for ratio in (1, 3):
            _check_loss((gt_cls, gt_box, gt_mask), (pred_box, pred_cls), ratio)


def test_loss_guards():
    y_true = (np.zeros((1, 64), np.int32), np.zeros((1, 64, 4), np.float32), np.zeros((1, 64), bool))
    y_pred = (np.zeros((1, 64, 4), np.float32), np.random.default_rng(0).normal(size=(1, 64, 5)).astype(np.float32))
    with pytest.raises(IndexError):
        M.ssd_loss(y_true, y_pred)                  # num_pos == 0 (models/ssd_model.py:369)
    y_true[2][0, :32] = True
    with pytest.raises(ValueError):
        M.ssd_loss(y_true, y_pred)                  # 3*32 > 64 (tf.math.top_k, :368)
    with pytest.raises(AssertionError):
        M.ssd_loss((y_true[0], y_true[1], y_true[2]), (y_pred[0], np.zeros((2, 64, 5), np.float32)))   # :347


def test_loss_grad(priors300):
    boxes, cls, off = synth.make_gt(5, 2, 100, "coco")
    y_true = _targets(boxes, cls, off, priors300, 2)
    pred_cls, pred_box = synth.make_predictions(5, 2, 8732)
    total, info, g_box, g_cls = M.ssd_loss_grad(y_true, (pred_box, pred_cls))
    w_box, w_cls = O.ssd_loss_grad(y_true, (pred_box, pred_cls))
    close(total, O.ssd_loss(y_true, (pred_box, pred_cls))[0])
    close(g_box, w_box, rtol=1e-5, atol=1e-12)
    close(g_cls, w_cls, rtol=2e-5, atol=1e-9)


def test_loss_full_size_properties(priors300):
    """B=256 (BASELINE config 2): batch-global mining is invariant under a permutation of the images,
    and the separable sums add up across shards when the threshold is shared."""
    batch = 256
    boxes, cls, off = synth.make_gt(21, batch, 100, "coco")
    tgt = ops.match_encode(boxes, cls, off, priors300, batch, 100, 0.5)
    pred_cls, pred_box = synth.make_predictions(21, batch, 8732)
    d_cls, d_box = D.to_device(pred_cls), D.to_device(pred_box)
    r = ops.loss_result_to_host(ops.multibox_loss(tgt["cls"], tgt["loc"], tgt["mask"], d_box, d_cls)["result"])
    assert 2.9 < r["num_neg"] / r["num_pos"] < 3.1
    perm = np.random.default_rng(0).permutation(batch)
    g = [tgt[k].to_host()[perm] for k in ("cls", "loc", "mask")]
    r2 = ops.loss_result_to_host(ops.multibox_loss(g[0], g[1], g[2], pred_box[perm], pred_cls[perm])["result"])
    assert r2["num_pos"] == r["num_pos"] and r2["num_neg"] == r["num_neg"] and r2["kth"] == r["kth"]
    close(r2["total"], r["total"], rtol=1e-9)
    # sampled oracle check on the first 8 images
    y_true = tuple(tgt[k].to_host()[:8] for k in ("cls", "loc", "mask"))
    _check_loss((y_true[0], y_true[1], y_true[2].astype(bool)), (pred_box[:8], pred_cls[:8]))


@pytest.mark.parametrize("shards", [2, 3])
def test_loss_cross_shard_global_mining(shards, priors300):
    """SURVEY.md section 8e, exact-global option: the batch split over `shards` workspaces (emulated on one
    device, the all-reduce is a host-side sum of the exchange buffers), staged through
    ssdg_multibox_loss_stage.  The mined masks must equal the slices of the single-device mask bit for bit,
    the threshold must be identical, and the combined loss must agree to rounding of the final sums."""
    from ssdgeom import parallel
    batch = 6
    boxes, cls, off = synth.make_gt(31, batch, 100, "coco")
    y_true = _targets(boxes, cls, off, priors300, batch)
    pred_cls, pred_box = synth.make_predictions(31, batch, 8732)
    full = ops.multibox_loss(y_true[0], y_true[1], y_true[2], pred_box, pred_cls, want_neg_mask=True)
    want = ops.loss_result_to_host(full["result"])
    want_mask = full["neg_mask"].to_host()
    spans = [parallel.shard_range(batch, shards, r) for r in range(shards)]
    staged = [ops.StagedLoss(*(v[lo:hi] for v in y_true), pred_box[lo:hi], pred_cls[lo:hi],
                             global_priors=batch * 8732, want_neg_mask=True, ws_kind="loss_staged_%d" % r)
              for r, (lo, hi) in enumerate(spans)]
    for stage in range(4):
        for s in staged:
            s.run(stage)
        for bufs in zip(*(s.exchange(stage) for s in staged)):
            tot = sum(b.to_host().astype(np.float64 if b.dtype == np.float64 else np.int64) for b in bufs)
            for b in bufs:
                b.copy_from_host(tot.astype(b.dtype))
            D.sync()
    results = [s.finish() for s in staged]
    masks = np.concatenate([s.out["neg_mask"].to_host() for s in staged])
    assert np.array_equal(masks, want_mask)
    for total, info in results:
        assert info["num_pos"] == want["num_pos"] and info["num_neg"] == want["num_neg"]
        assert info["kth"] == want["kth"]
        close(total, want["total"], rtol=1e-9)      # float partial sums depend on how priors fall into tiles
        for k in ("cls loss pos", "cls loss neg", "loc loss"):
            close(info[k], want[k], rtol=1e-9)
    # per-shard mining (the default data-parallel mode) gives a different mask here: the check is not vacuous
    local = ops.multibox_loss(*(v[spans[0][0]:spans[0][1]] for v in y_true), pred_box[spans[0][0]:spans[0][1]],
                              pred_cls[spans[0][0]:spans[0][1]], want_neg_mask=True)["neg_mask"].to_host()
    assert not np.array_equal(local, want_mask[spans[0][0]:spans[0][1]])


def test_staged_loss_writes_caller_outputs(priors300):
    """Arrays passed in ``out`` receive the staged loss's mask and gradient, as they do for multibox_loss."""
    batch = 2
    boxes, cls, off = synth.make_gt(33, batch, 100, "coco")
    y_true = _targets(boxes, cls, off, priors300, batch)
    pred_cls, pred_box = synth.make_predictions(33, batch, 8732)
    full = ops.multibox_loss(*y_true, pred_box, pred_cls, want_neg_mask=True, want_grad=True)
    mine = {"neg_mask": D.empty((batch, 8732), np.uint8), "grad_box": D.empty(pred_box.shape, np.float32),
            "grad_cls": D.empty(pred_cls.shape, np.float32)}
    for v in mine.values():
        v.zero_()
    sl = ops.StagedLoss(*y_true, pred_box, pred_cls, global_priors=batch * 8732, want_neg_mask=True, want_grad=True,
                        out=mine)
    for stage in range(sl.n_stages):       # one shard: the exchanges have nothing to sum
        sl.run(stage)
    assert sl.finish()[1]["num_neg"] == ops.loss_result_to_host(full["result"])["num_neg"]
    for k, v in mine.items():
        assert sl.out[k] is v
        assert np.array_equal(v.to_host(), full[k].to_host()), k


# ---- A7 / A8 / A9 -----------------------------------------------------------------------------------------
def _check_detect(pred_cls, pred_box, priors, **kw):
    kept, count, aux = M.detect(pred_cls, pred_box, priors, return_aux=True, **kw)
    b = pred_cls.shape[0]
    e2e_equal, lists = 0, 0
    for i in range(b):
        w_kept, w_count, w_probs, w_boxes = O.detect(pred_cls[i], pred_box[i], priors, **kw)
        # stage 1: scores and boxes within tolerance of the float64 oracle
        close(aux["probs"][i], w_probs, rtol=RTOL, atol=1e-9)
        close(aux["boxes"][i], w_boxes, rtol=RTOL, atol=1e-9)
        # stage 2: selection + suppression bit-exact on the kernel's own scores and boxes
        s_kept, s_count = O.nms_per_class(aux["probs"][i], aux["boxes"][i], **kw)
        assert np.array_equal(count[i], s_count), i
        assert np.array_equal(kept[i], s_kept), i
        for c in range(kept.shape[1]):
            k = kept[i, c, :count[i, c]]
            assert np.array_equal(aux["kept_score"][i, c, :count[i, c]], aux["probs"][i][k, c])
        lists += kept.shape[1]
        e2e_equal += int(np.sum(np.all(kept[i] == w_kept, axis=1)))
    return e2e_equal, lists


def test_detect_trained_like(priors300):
    pred_cls, pred_box = synth.make_predictions(31, 2, 8732, bg_bias=7.0)
    eq, lists = _check_detect(pred_cls, pred_box, priors300, score_thresh=0.01, top_k=200, iou_thresh=0.45)
    assert eq >= lists - 2, "end-to-end kept lists equal to the float64 oracle: %d of %d" % (eq, lists)


def test_detect_adversarial_no_bias(priors300):
    """bias 0: ~3400 candidates per class, the radix-select path before the sort."""
    pred_cls, pred_box = synth.make_predictions(32, 1, 8732, bg_bias=0.0)
    eq, lists = _check_detect(pred_cls, pred_box, priors300, score_thresh=0.01, top_k=200, iou_thresh=0.45)
    assert eq >= lists - 2


def test_detect_other_parameters(priors300):
    pred_cls, pred_box = synth.make_predictions(33, 1, 8732, bg_bias=5.0)
    pred_box *= 0.2                        # tighter boxes: more suppression
    for kw in (dict(score_thresh=0.02, top_k=50, iou_thresh=0.3), dict(score_thresh=0.005, top_k=400, iou_thresh=0.6)):
        _check_detect(pred_cls, pred_box, priors300, **kw)


# Foreground class counts at every boundary of the filter's class words: <= 32, <= 64, (64, 80] (two lanes share a
# class of the third word), (80, 96), exactly 96 (the last streaming case) and 97 (the two-pass variant), with prior
# counts that are not multiples of 4 or 32 (the non-TMA tile path).
FILTER_WORD_CASES = [(2, 203, nfg + 1, 2.0) for nfg in (1, 16, 31, 32, 33, 63, 64, 65, 79, 80, 81, 90, 95, 96, 97)]
# SSD300-sized rows (8 732 priors): the COCO label space of torchvision's SSD (91) and each side of the two-pass switch
FILTER_SSD300_CLASSES = (91, 97, 98)


def _rand_detect_inputs(rng, b, a, c, bias):
    pri = np.concatenate([rng.uniform(0.1, 0.9, (a, 2)), rng.uniform(0.05, 0.4, (a, 2))], 1)
    pred_cls = rng.normal(size=(b, a, c)).astype(np.float32)
    pred_cls[..., -1] += bias
    pred_box = (rng.normal(size=(b, a, 4)) * 0.3).astype(np.float32)
    return pred_cls, pred_box, pri


def test_detect_many_classes_and_odd_shapes(priors300):
    """C > 97 (classes beyond the register bit-sets), every class-word boundary of the filter, prior counts that are
    not multiples of 4 or 32 (the non-TMA tile path), tiny images."""
    rng = np.random.default_rng(12)
    for (b, a, c, bias) in [(2, 333, 130, 3.0), (3, 64, 21, 2.0), (1, 37, 5, 0.0), (2, 1000, 200, 4.0)] + FILTER_WORD_CASES:
        pred_cls, pred_box, pri = _rand_detect_inputs(rng, b, a, c, bias)
        _check_detect(pred_cls, pred_box, pri, score_thresh=0.01, top_k=100, iou_thresh=0.45)
    for c in FILTER_SSD300_CLASSES:
        pred_cls, pred_box = synth.make_predictions(90 + c, 1, 8732, c, bg_bias=4.0)
        _check_detect(pred_cls, pred_box, priors300, score_thresh=0.01, top_k=100, iou_thresh=0.45)


@pytest.mark.parametrize("b,a,c,bias", FILTER_WORD_CASES + [(1, 8732, c, 4.0) for c in FILTER_SSD300_CLASSES])
def test_detect_streaming_filter_word_boundaries(b, a, c, bias, priors300):
    """The streaming variant (background logit as the exponent reference, row statistics for the loss) at the same
    class counts: kept scores, row_ml and row_negbg against the float64 oracle, the lists end to end."""
    rng = np.random.default_rng(1000 + c)
    pred_cls, pred_box, pri = _rand_detect_inputs(rng, b, a, c, bias)
    if a == 8732:
        pri = priors300
    eq, lists = _check_detect_streaming(pred_cls, pred_box, pri, score_thresh=0.01, top_k=100, iou_thresh=0.45)
    assert eq >= lists - 2, "end-to-end kept lists equal to the float64 oracle: %d of %d" % (eq, lists)


def test_nms_on_oracle_inputs_bit_exact(priors300):
    """The second stage alone, fed the oracle's own float32 scores and boxes: no tolerance anywhere."""
    pred_cls, pred_box = synth.make_predictions(34, 2, 8732, bg_bias=6.0)
    pred_box *= 0.3
    probs = np.stack([O.softmax(pred_cls[i]) for i in range(2)])
    boxes = np.stack([O.decode_bbox(pred_box[i], priors300, 1.0, np.float64) for i in range(2)])
    kept, count = M.nms(probs, boxes)
    for i in range(2):
        w_kept, w_count = O.nms_per_class(probs[i], boxes[i])
        assert np.array_equal(count[i], w_count)
        assert np.array_equal(kept[i], w_kept)
    assert (count < 200).any() and count.max() > 20        # suppression actually happened


def test_nms_heavy_overlap_chain():
    """Long suppression chains (the fixed-point resolution must equal the sequential greedy)."""
    rng = np.random.default_rng(1)
    a, c = 600, 3
    boxes = np.zeros((1, a, 4), np.float32)
    boxes[0, :, 0] = 0.2 + 0.001 * np.arange(a)            # sliding boxes: each overlaps many neighbours
    boxes[0, :, 1] = 0.5
    boxes[0, :, 2:] = 0.1
    probs = rng.uniform(0.02, 0.9, (1, a, c)).astype(np.float32)
    probs[0, :, 1] = np.linspace(0.9, 0.02, a)             # monotone scores: chain of length ~a
    for thr in (0.45, 0.9, 0.05):
        kept, count = M.nms(probs, boxes, top_k=512, iou_thresh=thr)
        w_kept, w_count = O.nms_per_class(probs[0], boxes[0], top_k=512, iou_thresh=thr)
        assert np.array_equal(count[0], w_count) and np.array_equal(kept[0], w_kept), thr


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_nms_random_geometry_all_thresholds(seed):
    """Random box clouds -- clusters of near-duplicates, boxes a few ulps wide, zero / negative sizes, boxes far
    outside the unit square -- at thresholds on both sides of 0.5 and at the values that switch the kernel to its
    all-pairs path (<= 0, huge).  Kept sets must equal the sequential greedy of the oracle, bit for bit."""
    rng = np.random.default_rng(100 + seed)
    a, c = 700, 4
    centres = rng.uniform(0.1, 0.9, (12, 2))
    pick = rng.integers(0, 12, a)
    boxes = np.empty((1, a, 4), np.float32)
    boxes[0, :, :2] = centres[pick] + rng.normal(0, 0.02, (a, 2))
    boxes[0, :, 2:] = rng.uniform(0.05, 0.3, (a, 2)) * rng.choice([1.0, 1.0, 1.0, 0.1, 3.0], (a, 1))
    boxes[0, 0:40, 2:] = rng.uniform(1e-7, 3e-7, (40, 2))              # a few ulps wide at these centres
    boxes[0, 40:60, 2] = 0.0
    boxes[0, 60:70, 3] = -0.1
    boxes[0, 70:90, :2] += 50.0                                        # far away, coarse float grid
    boxes[0, 90:100] = boxes[0, 100:110]                               # exact duplicates
    if seed == 2:
        boxes[0, :, 2:] = rng.uniform(1e-7, 1e-6, (a, 2))              # every box tiny: extents unreliable
        boxes[0, :, :2] = 0.5 + rng.integers(0, 8, (a, 2)) * 1.2e-7
    probs = rng.uniform(0.0, 1.0, (1, a, c)).astype(np.float32)
    for thr in (0.45, 0.5, 0.3, 0.7, 0.95, 0.02, 0.0, -1.0, 2e6):
        kept, count = M.nms(probs, boxes, top_k=200, iou_thresh=thr)
        w_kept, w_count = O.nms_per_class(probs[0], boxes[0], top_k=200, iou_thresh=thr)
        assert np.array_equal(count[0], w_count), (seed, thr)
        assert np.array_equal(kept[0], w_kept), (seed, thr)


def test_score_head(priors300):
    pred_cls, _ = synth.make_predictions(35, 2, 8732, bg_bias=2.0)
    score, cls, mask = M.score_head(pred_cls, thresh=0.3)
    w_score, w_cls, w_mask = O.score_head(pred_cls, thresh=0.3)
    close(score, w_score, rtol=RTOL, atol=1e-9)
    p = np.sort(O.softmax(pred_cls), axis=-1)
    clear = (p[..., -1] - p[..., -2]) > 1e-6
    assert np.array_equal(cls[clear], w_cls[clear])
    far = (np.abs(w_score - 0.3) > 1e-5) & (np.abs(O.softmax(pred_cls)[..., -1] - 0.3) > 1e-5)
    assert np.array_equal(mask[far], w_mask[far])


def test_detect_full_batch_properties(priors300):
    """B=64 SSD300: kept indices are valid, unique per list, scores descending, counts <= top_k, and the
    result is identical when the batch is processed in two halves (images are independent)."""
    batch = 64
    pred_cls, pred_box = synth.make_predictions(36, batch, 8732)
    out = ops.detect(pred_cls, pred_box, priors300, want_scores=True)
    kept, count, score = out["kept"].to_host(), out["count"].to_host(), out["kept_score"].to_host()
    assert count.max() <= 200 and count.min() >= 0
    valid = np.arange(200)[None, None, :] < count[..., None]
    assert np.all(kept[valid] >= 0) and np.all(kept[valid] < 8732) and np.all(kept[~valid] == -1)
    d = np.diff(score, axis=-1)
    assert np.all(d[valid[..., 1:]] <= 0)
    for i in (0, 33):
        for c in (0, 41, 79):
            k = kept[i, c, :count[i, c]]
            assert np.unique(k).size == k.size
    h1 = ops.detect(pred_cls[:32], pred_box[:32], priors300)
    k1 = h1["kept"].to_host()
    h2 = ops.detect(pred_cls[32:], pred_box[32:], priors300)
    assert np.array_equal(np.concatenate([k1, h2["kept"].to_host()]), kept)


def _check_detect_streaming(pred_cls, pred_box, priors, **kw):
    """The streaming variant of the filter (no probabilities output: the rows are not overwritten, the exponent
    reference is the background logit with an exact fallback) against the float64 oracle: kept scores within
    tolerance, the lists equal wherever no score sits within rounding of the threshold / of a neighbour."""
    out = ops.detect(pred_cls, pred_box, priors, want_scores=True, want_row_stats=True, **kw)
    kept, count, score = out["kept"].to_host(), out["count"].to_host(), out["kept_score"].to_host()
    row_ml, negbg = out["row_ml"].to_host().astype(np.float64), out["row_negbg"].to_host().astype(np.float64)
    equal = lists = 0
    for i in range(pred_cls.shape[0]):
        w_kept, w_count, w_probs, _ = O.detect(pred_cls[i], pred_box[i], priors, **kw)
        for c in range(kept.shape[1]):
            k = kept[i, c, :count[i, c]]
            close(score[i, c, :count[i, c]], w_probs[k, c], rtol=RTOL, atol=1e-9)
            assert np.all(score[i, c, :count[i, c]] > kw["score_thresh"]) and np.all(np.diff(score[i, c, :count[i, c]]) <= 0)
        lists += kept.shape[1]
        equal += int(np.sum(np.all(kept[i] == w_kept, axis=1)))
        # the loss's by-product: log-sum-exp = reference + log sum, background CE
        x = pred_cls[i].astype(np.float64)
        lse = np.log(np.sum(np.exp(x - x.max(axis=1, keepdims=True)), axis=1)) + x.max(axis=1)
        close(row_ml[i, :, 0] + row_ml[i, :, 1], lse, rtol=RTOL, atol=2e-6)
        close(negbg[i], lse - x[:, -1], rtol=RTOL, atol=2e-6)
    return equal, lists


def test_detect_streaming_background_reference_and_fallback(priors300):
    kw = dict(score_thresh=0.01, top_k=200, iou_thresh=0.45)
    # trained-like rows: the background logit is the reference of nearly every row (one pass)
    pred_cls, pred_box = synth.make_predictions(51, 2, 8732, bg_bias=7.0)
    eq, lists = _check_detect_streaming(pred_cls, pred_box, priors300, **kw)
    assert eq >= lists - 2
    # wide logits: foreground far above the background (sum > 2^16, overflow of the float exponent) -> the rows
    # are redone with their maximum; background far above everything -> sums of exactly 1
    rng = np.random.default_rng(52)
    wide = (rng.standard_normal((2, 8732, 81)) * 12.0).astype(np.float32)
    wide[0, ::7, 3] += 90.0
    wide[1, ::5, -1] += 120.0
    wide[1, 1::5, -1] -= 150.0
    # (saturated scores tie within rounding by the hundred here: the kept scores and the row statistics are
    # checked against the oracle, list equality is not meaningful)
    _check_detect_streaming(wide, pred_box, priors300, **kw)
    # both filter variants agree on what they keep
    plain = ops.detect(pred_cls, pred_box, priors300, **kw)
    full = ops.detect(pred_cls, pred_box, priors300, want_probs=True, **kw)
    same = np.all(plain["kept"].to_host() == full["kept"].to_host(), axis=2)
    assert same.sum() >= same.size - 2


def test_loss_from_filter_row_statistics(priors300):
    """The chained step's single pass over the logits: the softmax filter leaves per-prior (max, log-sum) and the
    background CE, and ssdg_multibox_loss_fused must give the loss of the standalone path -- per-prior CE within
    tolerance of the float64 oracle, the mask bit-exact on its own CE vector (two-stage contract), same counts."""
    batch = 5
    boxes, cls, off = synth.make_gt(41, batch, 100, "coco")
    y_true = _targets(boxes, cls, off, priors300, batch)
    for bias in (7.0, 0.0):
        pred_cls, pred_box = synth.make_predictions(41, batch, 8732, bg_bias=bias)
        d_cls = D.to_device(pred_cls)
        det = ops.detect(d_cls, pred_box, priors300, want_row_stats=True)
        plain = ops.detect(d_cls, pred_box, priors300)
        assert np.array_equal(det["kept"].to_host(), plain["kept"].to_host())          # the statistics are a by-product
        assert np.array_equal(det["count"].to_host(), plain["count"].to_host())
        fused = ops.multibox_loss(y_true[0], y_true[1], y_true[2], pred_box, d_cls, want_neg_mask=True, want_neg_ce=True,
                                  row_stats=(det["row_ml"], det["row_negbg"]), ws_kind="loss_fused")
        r = ops.loss_result_to_host(fused["result"])
        w_total, w_info, w_aux = O.ssd_loss(y_true, (pred_box, pred_cls), return_masks=True)
        close(r["total"], w_total)
        for k in ("cls loss pos", "cls loss neg", "loc loss"):
            close(r[k], w_info[k])
        neg_ce, neg_mask = fused["neg_ce"].to_host(), fused["neg_mask"].to_host().astype(bool)
        close(neg_ce, w_aux["neg_ce"], rtol=RTOL, atol=1e-6)
        kth, want_mask = O.hard_negative_select(neg_ce, r["num_pos"], 3)
        assert np.array_equal(neg_mask, want_mask) and np.float32(r["kth"]) == kth
        assert r["num_pos"] == w_aux["num_pos"] and r["num_neg"] == int(want_mask.sum())
        assert int(np.sum(neg_mask != w_aux["neg_mask"])) <= 2      # end to end vs the float64 oracle (reported)


def test_pipelined_host_steps_match_serial(priors300):
    """HotPath.submit (double-buffered inputs, copies overlapped with compute) returns exactly what step_host returns,
    batch after batch, including when consecutive batches differ."""
    from ssdgeom.pipeline import HotPath
    b = 4
    hp = HotPath(synth.TABLES["ssd300"], batch=b, max_gt=100, total_gt=b * 100)
    batches = []
    for seed in (51, 52, 53):
        boxes, cls, off = synth.make_gt(seed, b, 100, "max")
        pc, pb = synth.make_predictions(seed, b, 8732)
        batches.append((boxes, cls, off, pc, pb))
    def outs():
        return (np.zeros(16), np.zeros((b, 80, 200), np.int32), np.zeros((b, 80), np.int32))
    serial = []
    for inp in batches:
        o = outs()
        hp.step_host(*inp, *o)
        serial.append(o)
    piped = [outs() for _ in batches]
    for inp, o in zip(batches, piped):
        hp.submit(inp, o)
    hp.drain()
    for s, p in zip(serial, piped):
        assert np.array_equal(s[1], p[1]) and np.array_equal(s[2], p[2])
        close(p[0][:11], s[0][:11], rtol=1e-12)
    assert not np.array_equal(serial[0][1], serial[1][1])


def test_generalised_anchor_options(priors300):
    """Section 8f row 4: clipping and variances (options the reference lacks) against the oracle's restatement;
    clip=False / variances=None are the reference's behaviour (covered by every other test)."""
    t = synth.SSD300
    got = M.build_prior_box(t["sizes"], clip=True)
    assert np.array_equal(got, O.clip_priors(priors300)) and got.max() <= 1.0 and (priors300.max() > 1.0)
    boxes, cls, off = synth.make_gt(61, 3, 20, "max")
    var = (0.1, 0.2)
    c0, l0, m0 = bbox.match_encode_batch(boxes, cls, off, priors300, 0.5)
    c1, l1, m1 = bbox.match_encode_batch(boxes, cls, off, priors300, 0.5, variances=var)
    assert np.array_equal(c0, c1) and np.array_equal(m0, m1)
    for i in range(3):
        w_cls, w_box, w_mask = O.match_bbox(cls[off[i]:off[i + 1]], boxes[off[i]:off[i + 1]], priors300)
        close(l1[i], O.apply_anchor_box_var(w_box, priors300, var), rtol=RTOL)      # float32 product vs float64 division
    dec = bbox.decode_bbox(l1[0], priors300, scale=300.0, variances=var)
    close(dec, O.decode_bbox_var(l1[0], priors300, 300.0, var), rtol=RTOL, atol=1e-6)
    close(dec[m1[0]], bbox.decode_bbox(l0[0], priors300, scale=300.0)[m0[0]], rtol=1e-4, atol=1e-4)   # round trip


def test_ssd512_loss_and_detect(priors512):
    """BASELINE config 4's table (SSD512, 24 564 priors, 768 tiles -- more than the SSD300 index): the loss and the
    post-processing against the oracle on a small batch (the assignment is covered by test_assign_random_bit_exact)."""
    batch = 2
    boxes, cls, off = synth.make_gt(81, batch, 100, "coco")
    y_true = _targets(boxes, cls, off, priors512, batch)
    pred_cls, pred_box = synth.make_predictions(81, batch, priors512.shape[0], bg_bias=7.0)
    _check_loss(y_true, (pred_box, pred_cls))
    eq, lists = _check_detect(pred_cls[:1], pred_box[:1], priors512, score_thresh=0.01, top_k=200, iou_thresh=0.45)
    assert eq >= lists - 2
    eq, lists = _check_detect_streaming(pred_cls[:1], pred_box[:1], priors512, score_thresh=0.01, top_k=200, iou_thresh=0.45)
    assert eq >= lists - 2


def test_chained_step_full_batch_equals_standalone_calls(priors300):
    """BASELINE size (SSD300, B=256): the chained HotPath.step -- four streams, one pass over the logits shared by
    the loss and the post-processing -- against the three standalone entry points on the same device buffers:
    targets and detections identical, loss within tolerance (the two CE passes round differently), and the result
    is reproducible run to run (no race between the streams)."""
    from ssdgeom.pipeline import HotPath
    b = 256
    boxes, cls, off = synth.make_gt(71, b, 100, "coco")
    hp = HotPath(synth.TABLES["ssd300"], batch=b, max_gt=int(np.diff(off).max()), total_gt=boxes.shape[0])
    pc = np.empty((b, hp.A, hp.classes), np.float32)
    pb = np.empty((b, hp.A, 4), np.float32)
    for i in range(0, b, 32):
        pc[i:i + 32], pb[i:i + 32] = synth.make_predictions(700 + i, 32, hp.A, hp.classes)
    hp.upload(boxes, cls, off, pc, pb)
    runs = []
    for _ in range(3):
        hp.step()
        hp.s_main.sync()
        runs.append((hp.loss["result"].to_host(), hp.det["kept"].to_host(), hp.det["count"].to_host(),
                     hp.tgt["cls"].to_host(), hp.tgt["mask"].to_host(), hp.tgt["loc"].to_host()))
    for r in runs[1:]:
        assert all(np.array_equal(x, y) for x, y in zip(r[1:], runs[0][1:]))
        close(r[0][:11], runs[0][0][:11], rtol=1e-12)
    tgt = ops.match_encode(hp.gt_boxes, hp.gt_cls, hp.gt_off, hp.priors, b, hp.max_gt, 0.5)
    assert np.array_equal(tgt["cls"].to_host(), runs[0][3]) and np.array_equal(tgt["mask"].to_host(), runs[0][4])
    assert np.array_equal(tgt["loc"].to_host(), runs[0][5])
    det = ops.detect(hp.pred_cls, hp.pred_box, hp.priors)
    assert np.array_equal(det["kept"].to_host(), runs[0][1]) and np.array_equal(det["count"].to_host(), runs[0][2])
    alone = ops.loss_result_to_host(ops.multibox_loss(tgt["cls"], tgt["loc"], tgt["mask"], hp.pred_box, hp.pred_cls)["result"])
    r = runs[0][0]
    assert int(r[4]) == alone["num_pos"] and abs(int(r[5]) - alone["num_neg"]) <= 2
    close(r[0], alone["total"], rtol=1e-6)
    # sampled oracle check of the chained outputs: first 4 images
    for i in range(4):
        w_cls, w_loc, w_mask = O.assign_encode(cls[off[i]:off[i + 1]], boxes[off[i]:off[i + 1]], priors300, sweeps=False)
        assert np.array_equal(runs[0][3][i], w_cls) and np.array_equal(runs[0][4][i].astype(bool), w_mask)
