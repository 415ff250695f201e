"""GPU (B200): the SSD training augmentation (ssdg_augment_boxes / ssdg_augment_images, ops.augment) bit for bit against
its NumPy restatement (tests/augment_oracle.py) -- records, offsets, boxes, labels and source rows; images within 1e-4
-- over batch sizes, ground-truth counts from 0 to 2048, degenerate boxes, option sets, trial counts and gate
probabilities; independence of the batch an image runs in; and TrainBatches(augment=...) end to end."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import augment_oracle as O                             # noqa: E402  (the checker)
from ssdgeom import ops, synth                         # noqa: E402
from ssdgeom.data import TrainBatches, pack_gt         # noqa: E402
from ssdgeom.models import ssd_model as M              # noqa: E402

KEYS = ("transform", "offsets", "boxes", "cls", "src_row")


def device_aug(images, boxes, cls, off, seed, base=0, **cfg):
    out = ops.augment(images, boxes, cls, off, seed, base, **cfg)
    return {k: out[k].to_host() for k in KEYS + ("images",)}


def same_bits(a, b):
    """Equal bit for bit, except that any NaN equals any NaN."""
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    if a.dtype == np.float32:
        both_nan = np.isnan(a) & np.isnan(b)
        return bool(np.all(both_nan | (a.view(np.uint32) == b.view(np.uint32))))
    return np.array_equal(a, b)


def check(images, boxes, cls, off, seed, base=0, **cfg):
    got = device_aug(images, boxes, cls, off, seed, base, **cfg)
    want = O.augment(images, boxes, cls, off, seed, base, **cfg)
    for k in KEYS:
        assert same_bits(got[k], want[k]), k
    np.testing.assert_allclose(got["images"], want["images"], atol=1e-4, rtol=0)
    return got


def rand_images(seed, b, h, w):
    return np.random.default_rng(seed).random((b, h, w, 3), dtype=np.float32)


@pytest.mark.parametrize("b", [1, 7, 256])
@pytest.mark.parametrize("mode", ["max", "coco"])
def test_random_batches_equal_the_oracle(b, mode):
    boxes, cls, off = synth.make_gt(b + len(mode), b, 100, mode)
    h, w = (300, 300) if b < 256 else (48, 64)
    got = check(rand_images(b, b, h, w), boxes, cls, off, 11 + b)
    rec = got["transform"]
    if b == 256:        # every branch of the recipe occurs
        assert (rec[:, 0] > w).any() and (rec[:, 0] == w).any() and rec[:, 8].any() and not rec[:, 8].all()
        assert (rec[:, 6] < rec[:, 0]).any() and (rec[:, 9] > 1).any()


def test_no_ground_truth_and_the_round_cap():
    b = 24
    boxes, cls, off = synth.make_gt(5, b, 20, "max")
    counts = np.diff(off)
    counts[::3] = 0                       # some images without rows
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    boxes, cls = boxes[:off[-1]], cls[:off[-1]]
    got = check(rand_images(1, b, 40, 30), boxes, cls, off, 3, min_ious=(0.1, 0.5), max_rounds=4)
    assert (got["transform"][counts == 0, 9] == -1).all()        # never terminates in torchvision: capped here
    empty = np.zeros((0, 4), np.float32)
    got = check(rand_images(2, 9, 40, 30), empty, np.zeros(0, np.float32), np.zeros(10, np.int32), 4)
    assert got["offsets"][-1] == 0 and set(got["transform"][:, 9]) <= {-1} | set(range(1, 51))


def test_2048_rows():
    rng = np.random.default_rng(8)
    boxes = np.concatenate([rng.uniform(0, 1, (4096, 2)), rng.uniform(0.02, 0.5, (4096, 2))], 1).astype(np.float32)
    off = np.int32([0, 2048, 2048, 4096])
    cls = np.arange(4096, dtype=np.float32)
    check(rand_images(3, 3, 32, 32), boxes, cls, off, 5)
    # rows beyond max_gt are read from global memory: same result
    got = device_aug(rand_images(3, 3, 32, 32), boxes, cls, off, 5, max_gt=100)
    want = O.augment(rand_images(3, 3, 32, 32), boxes, cls, off, 5)
    for k in KEYS:
        assert same_bits(got[k], want[k]), k


def test_degenerate_boxes():
    rng = np.random.default_rng(6)
    n = 40
    boxes = rng.uniform(0, 1, (n, 4)).astype(np.float32)
    boxes[0:5, 2] = 0                           # zero width
    boxes[5:10, 3] = 0
    boxes[10:15, :2] += 1.5                     # centres outside the image
    boxes[15:18, 0] = np.nan
    boxes[18:21, 2] = np.nan
    boxes[21:23, 2:] = -boxes[21:23, 2:]        # negative sizes
    boxes[23, 2] = np.inf
    off = np.int32([0, 8, 16, 24, 32, 40])
    cls = np.arange(n, dtype=np.float32)
    for seed in range(6):
        check(rand_images(seed, 5, 30, 50), boxes, cls, off, seed)


@pytest.mark.parametrize("cfg", [dict(min_ious=(1.0,)), dict(min_ious=(0.9,), min_scale=0.05), dict(min_ious=()),
                                 dict(trials=1), dict(trials=40, zoom_p=0.0, flip_p=1.0),
                                 dict(zoom_p=1.0, flip_p=0.0), dict(side_range=(1.0, 1.0), min_ious=(0.0,))])
def test_configurations(cfg):
    boxes, cls, off = synth.make_gt(21, 40, 30, "coco")
    if cfg.get("min_scale") == 0.05:
        boxes[:, 2:] = np.float32(0.01)         # tiny boxes: a 0.9 overlap needs a tiny crop
    got = check(rand_images(4, 40, 60, 80), boxes, cls, off, 8, **cfg)
    rec = got["transform"]
    if cfg.get("min_ious") == (1.0,):
        assert (rec[:, 9] == 1).all() and (rec[:, 6] == rec[:, 0]).all()
    if cfg.get("min_ious") == ():
        assert (rec[:, 9] == 0).all() and np.array_equal(got["offsets"], off)
    if cfg.get("zoom_p") == 0.0:
        assert (rec[:, 0] == 80).all() and rec[:, 8].all()
    if cfg.get("zoom_p") == 1.0:
        assert (rec[:, 0] > 80).sum() > 30 and not rec[:, 8].any()


def test_an_image_does_not_depend_on_its_batch():
    boxes, cls, off = synth.make_gt(30, 64, 50, "coco")
    imgs = rand_images(5, 64, 36, 36)
    full = device_aug(imgs, boxes, cls, off, 77, 1000)
    for lo, hi in ((0, 1), (5, 12), (40, 64)):
        part = device_aug(imgs[lo:hi], boxes[off[lo]:off[hi]], cls[off[lo]:off[hi]], off[lo:hi + 1] - off[lo], 77,
                          1000 + lo)
        assert np.array_equal(part["transform"], full["transform"][lo:hi])
        assert np.array_equal(part["images"], full["images"][lo:hi])
        n0, n1 = full["offsets"][lo], full["offsets"][hi]
        assert np.array_equal(part["offsets"], full["offsets"][lo:hi + 1] - n0)
        assert same_bits(part["boxes"][:n1 - n0], full["boxes"][n0:n1])
        assert np.array_equal(part["src_row"][:n1 - n0] + off[lo], full["src_row"][n0:n1])


def test_augmented_targets_match_cleanly():
    priors = M.build_prior_box(synth.SSD300["sizes"])
    boxes, cls, off = synth.make_gt(31, 32, 100, "max")
    max_gt = int(np.diff(off).max())
    aug = ops.augment(rand_images(6, 32, 30, 30), boxes, cls, off, 9, max_gt=max_gt)
    tgt = ops.match_encode(aug["boxes"], aug["cls"], aug["offsets"], priors, 32, max_gt)
    assert ops.match_status(tgt) == 0


class Source:
    def __init__(self, n, h, w, coco):
        self.n, self.h, self.w, self.coco = n, h, w, coco

    def __iter__(self):
        self.rng = np.random.default_rng(40)
        boxes, cls, off = synth.make_gt(41, self.n, 30, "coco")
        for i in range(self.n):
            img = self.rng.random((self.h, self.w, 3), dtype=np.float32)
            b = boxes[off[i]:off[i + 1]]
            if self.coco:       # COCO pixel [x, y, w, h]
                b = np.concatenate([(b[:, :2] - b[:, 2:] / 2) * [self.w, self.h], b[:, 2:] * [self.w, self.h]], 1)
            yield img, cls[off[i]:off[i + 1]], b


@pytest.mark.parametrize("coco", [False, True])
@pytest.mark.parametrize("prefetch", [0, 3])
def test_train_batches_with_augmentation(coco, prefetch):
    priors = M.build_prior_box(synth.SSD300["sizes"])
    src = Source(20, 30, 40, coco)
    cfg = dict(seed=5, min_ious=(0.0, 0.3, 0.7, 1.0), flip_p=0.5)
    it = TrainBatches(src, priors, batch_size=4, coco_pixels=coco, prefetch=prefetch, augment=cfg, image_base=100)
    got = list(it)
    assert len(got) == 5
    items = list(src)
    for k, (img, (g_cls, g_loc, g_mask)) in enumerate(got):
        part = items[4 * k:4 * k + 4]
        c, b, off = pack_gt([p[1] for p in part], [p[2] for p in part])
        imgs = np.stack([p[0] for p in part])
        d_boxes = ops.gt_prepare(b, np.int32([[40, 30]] * 4), off) if coco else b.astype(np.float32)
        aug = ops.augment(imgs, d_boxes, c, off, 5, 100 + 4 * k, min_ious=(0.0, 0.3, 0.7, 1.0), flip_p=0.5)
        want_img = ops.image_normalize(aug["images"]).to_host()
        tgt = ops.match_encode(aug["boxes"], aug["cls"], aug["offsets"], priors, 4, max(int(np.diff(off).max()), 1))
        assert np.array_equal(img, want_img)
        assert np.array_equal(g_cls, tgt["cls"].to_host()) and np.array_equal(g_loc, tgt["loc"].to_host())
        assert np.array_equal(g_mask, tgt["mask"].to_host().astype(bool))
    # without augment the iterator is unchanged: the plain path
    plain = list(TrainBatches(src, priors, batch_size=4, coco_pixels=coco, prefetch=prefetch))
    assert not np.array_equal(plain[0][0], got[0][0])
