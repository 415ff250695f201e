"""CPU: the NumPy restatement of the SSD training augmentation (tests/augment_oracle.py) against independent references
-- Random123's Philox known answers, torchvision's own RandomZoomOut / RandomIoUCrop make_params fed the same uniforms,
F.interpolate of an explicitly built canvas crop -- and the argument checks of ssdg_augment_boxes /
ssdg_augment_images, one invalid argument per call, each answered with its exact status before any CUDA call."""
import numpy as np
import pytest

import augment_oracle as O

F = 1 << 20              # a fake device pointer, 256-byte aligned


def test_philox_known_answers():
    # Random123 kat_vectors, philox4x32 with 10 rounds: (counter, key) -> output
    assert O.philox4x32((0, 0, 0, 0), 0) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    ones = 0xFFFFFFFF
    assert O.philox4x32((ones,) * 4, (ones << 32) | ones) == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert O.philox4x32((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0x299f31d0 << 32) | 0xa4093822) == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]
    assert O.unif(0xFFFFFFFF) == np.float32(1 - 2.0 ** -24) and O.unif(0xFF) == 0.0


def rand_gt(seed, b, max_t, empty_every=5):
    """Relative cxcywh rows of b images (some without rows), CSR."""
    rng = np.random.default_rng(seed)
    counts = rng.integers(0, max_t + 1, b)
    counts[::empty_every] = 0
    off = np.zeros(b + 1, np.int32)
    np.cumsum(counts, out=off[1:])
    n = int(off[-1])
    wh = rng.uniform(0.02, 0.9, (n, 2))
    cxy = rng.uniform(0.0, 1.0, (n, 2))
    boxes = np.concatenate([cxy, wh], 1).astype(np.float32)
    cls = rng.integers(0, 80, n).astype(np.float32)
    return boxes, cls, off


class CapHit(Exception):
    pass


class Feeder:
    """torch.rand / torch.randint in torchvision's call order for one image, served from the image's fixed draw
    addresses.  To route a trial's second torch.rand(2) (left, top) it repeats torchvision's aspect test on the first."""

    def __init__(self, u, cw, ch, cfg):
        import torch
        self.torch, self.u, self.cw, self.ch, self.cfg = torch, u, cw, ch, cfg
        self.q, self.t, self.pos = -1, 0, False

    def randint(self, low=0, high=None, size=None, **kw):
        self.q += 1
        if self.q >= self.cfg["max_rounds"]:
            raise CapHit
        self.t, self.pos = 0, False
        return self.torch.tensor([self.u.option(self.q, high)])

    def rand(self, *size, **kw):
        torch, cfg = self.torch, self.cfg
        uu = self.u.trial(self.q, self.t)
        if self.pos:
            self.pos, self.t = False, self.t + 1
            return torch.tensor(uu[2:], dtype=torch.float32)
        r = cfg["min_scale"] + (cfg["max_scale"] - cfg["min_scale"]) * torch.tensor(uu[:2], dtype=torch.float32)
        nw, nh = int(self.cw * r[0]), int(self.ch * r[1])
        if nh != 0 and cfg["min_aspect"] <= nw / nh <= cfg["max_aspect"]:
            self.pos = True
        else:
            self.t += 1
        return torch.tensor(uu[:2], dtype=torch.float32)


@pytest.mark.parametrize("config", [{}, dict(min_ious=(0.9,), max_rounds=3), dict(min_ious=(0.0, 0.5), trials=1),
                                    dict(side_range=(1.5, 2.5), min_scale=0.1, max_aspect=3.0)])
def test_decisions_equal_torchvision_make_params(monkeypatch, config):
    torch = pytest.importorskip("torch")
    tv = pytest.importorskip("torchvision")
    from torchvision import tv_tensors
    from torchvision.transforms import v2
    cfg = dict(O.DEFAULTS, **config)
    boxes, _, off = rand_gt(len(config), 60, 12)
    H, W, seed = 300, 200, 1234 + len(config)
    zoom = v2.RandomZoomOut(side_range=cfg["side_range"], p=cfg["zoom_p"])
    crop = v2.RandomIoUCrop(cfg["min_scale"], cfg["max_scale"], cfg["min_aspect"], cfg["max_aspect"],
                            list(cfg["min_ious"]), cfg["trials"])
    n_crop = n_cap = 0
    for i in range(off.size - 1):
        rows = boxes[off[i]:off[i + 1]]
        rec, mask = O.sample(rows, seed, i, H, W, cfg)
        u = O.Uniforms(seed, i)
        z = u.zoom()
        # gates: _RandomApplyTransform skips when torch.rand(1) >= p
        zoomed = not bool(torch.tensor([z[0]]) >= cfg["zoom_p"])
        assert not bool(torch.tensor([u.flip()]) >= cfg["flip_p"]) == bool(rec[8])
        if zoomed:
            draws = iter([torch.tensor([z[1]]), torch.tensor([z[2], z[3]])])
            monkeypatch.setattr(torch, "rand", lambda *a, **k: next(draws))
            pad = zoom.make_params([tv_tensors.Image(torch.zeros(3, H, W))])["padding"]
            monkeypatch.undo()
            assert pad == [rec[2], rec[3], rec[0] - rec[2] - W, rec[1] - rec[3] - H], i
        else:
            assert tuple(rec[:4]) == (W, H, 0, 0)
        cw, ch = int(rec[0]), int(rec[1])
        k = O.canvas_corners(rows, W, H, rec[2], rec[3])
        flat = [tv_tensors.Image(torch.zeros(3, ch, cw)),
                tv_tensors.BoundingBoxes(torch.from_numpy(k), format="XYXY", canvas_size=(ch, cw))]
        feed = Feeder(u, cw, ch, cfg)
        monkeypatch.setattr(torch, "rand", feed.rand)
        monkeypatch.setattr(torch, "randint", feed.randint)
        try:
            p = crop.make_params(flat)
        except CapHit:
            p = None
        monkeypatch.undo()
        if p is None:
            assert rec[9] == -1 and mask is None, i
            n_cap += 1
            continue
        assert rec[9] == feed.q + 1, i
        if not p:
            assert mask is None and tuple(rec[4:8]) == (0, 0, cw, ch), i
            continue
        n_crop += 1
        assert (p["left"], p["top"], p["width"], p["height"]) == tuple(rec[4:8]), i
        assert np.array_equal(p["is_within_crop_area"].numpy(), mask), i
    # torchvision was given the same float64 corners, so its centre / IoU tests are the restatement's: no image may
    # disagree (with its default float32 boxes a centre or IoU within rounding of a threshold could)
    print("images %d, cropped %d, round cap %d, disagreements 0" % (off.size - 1, n_crop, n_cap))
    assert n_crop > 0 or n_cap > 0


def test_image_equals_interpolate_of_the_canvas_crop():
    torch = pytest.importorskip("torch")
    import torch.nn.functional as Fn
    rng = np.random.default_rng(3)
    H, W = 37, 53
    fill = O.DEFAULTS["fill"]
    seen = set()
    for g in range(40):
        img = rng.random((H, W, 3), dtype=np.float32)
        rows = np.float32([[0.5, 0.5, 0.3, 0.4], [0.2, 0.7, 0.1, 0.1]])
        rec, _ = O.sample(rows, 99, g, H, W, O.DEFAULTS)
        cw, ch, pl, pt, l, t, w, h, flip, _ = (int(v) for v in rec)
        canvas = np.empty((ch, cw, 3), np.float32)
        canvas[:] = np.float32(fill)
        canvas[pt:pt + H, pl:pl + W] = img
        crop = torch.from_numpy(canvas[t:t + h, l:l + w].copy()).permute(2, 0, 1)[None]
        want = Fn.interpolate(crop, size=(H, W), mode="bilinear", align_corners=False, antialias=False)[0]
        want = want.permute(1, 2, 0).numpy()
        if flip:
            want = want[:, ::-1]
        np.testing.assert_allclose(O.resample(img, rec, fill), want, atol=1e-5, rtol=0)
        seen.add((cw != W, (w, h) != (cw, ch), flip))
    assert len(seen) >= 4


# ---- argument checks ----------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def native():
    import build_native
    build_native.build()
    from ssdgeom import _native
    return _native


def _boxes(lib, **kw):
    import ctypes as C
    a = dict(gt_boxes=F, gt_cls=F, gt_offsets=F, batch=4, max_gt=100, height=300, width=300, seed=1, image_base=0,
             zoom_p=0.5, side_lo=1.0, side_hi=4.0, min_ious=[0.0, 0.1, 0.3, 0.5, 0.7, 0.9, 1.0], n_options=None,
             min_scale=0.3, max_scale=1.0, min_aspect=0.5, max_aspect=2.0, trials=40, max_rounds=50, flip_p=0.5,
             out_boxes=F, out_cls=F, out_offsets=F, out_src_row=F, out_transform=F)
    a.update(kw)
    opts = None if a["min_ious"] is None else (C.c_double * max(len(a["min_ious"]), 1))(*a["min_ious"])
    n = len(a["min_ious"] or []) if a["n_options"] is None else a["n_options"]
    return lib.ssdg_augment_boxes(a["gt_boxes"], a["gt_cls"], a["gt_offsets"], a["batch"], a["max_gt"], a["height"],
                                  a["width"], a["seed"], a["image_base"], a["zoom_p"], a["side_lo"], a["side_hi"], opts,
                                  n, a["min_scale"], a["max_scale"], a["min_aspect"], a["max_aspect"], a["trials"],
                                  a["max_rounds"], a["flip_p"], a["out_boxes"], a["out_cls"], a["out_offsets"],
                                  a["out_src_row"], a["out_transform"], None)


def test_augment_boxes_rejects_each_bad_argument(native):
    N, lib, nan = native, native.lib(), float("nan")
    cases = [({k: None}, N.ERR_ARG) for k in ("gt_boxes", "gt_cls", "gt_offsets", "out_boxes", "out_cls",
                                              "out_offsets", "out_src_row", "out_transform")]
    cases += [({"min_ious": None, "n_options": 3}, N.ERR_ARG), ({"n_options": -1}, N.ERR_ARG)]
    cases += [({"batch": 0}, N.ERR_ARG), ({"batch": -2}, N.ERR_ARG), ({"max_gt": -1}, N.ERR_ARG),
              ({"height": 0}, N.ERR_ARG), ({"width": -1}, N.ERR_ARG), ({"trials": 0}, N.ERR_ARG),
              ({"max_rounds": 0}, N.ERR_ARG)]
    cases += [({"zoom_p": -0.1}, N.ERR_ARG), ({"zoom_p": 1.5}, N.ERR_ARG), ({"zoom_p": nan}, N.ERR_ARG),
              ({"flip_p": 2.0}, N.ERR_ARG), ({"flip_p": nan}, N.ERR_ARG), ({"side_lo": 0.5}, N.ERR_ARG),
              ({"side_lo": 3.0, "side_hi": 2.0}, N.ERR_ARG), ({"side_hi": nan}, N.ERR_ARG),
              ({"min_scale": -0.1}, N.ERR_ARG), ({"min_scale": 0.8, "max_scale": 0.5}, N.ERR_ARG),
              ({"max_scale": 1.5}, N.ERR_ARG), ({"min_aspect": 0.0}, N.ERR_ARG),
              ({"min_aspect": 2.0, "max_aspect": 1.0}, N.ERR_ARG), ({"max_aspect": nan}, N.ERR_ARG),
              ({"min_ious": [0.1, nan]}, N.ERR_ARG)]
    cases += [({"min_ious": [0.5] * 17}, N.ERR_LIMIT), ({"max_gt": 2049}, N.ERR_LIMIT),
              ({"height": 16385}, N.ERR_LIMIT), ({"width": 16385}, N.ERR_LIMIT), ({"side_hi": 65.0}, N.ERR_LIMIT)]
    cases += [({"gt_boxes": F + 4}, N.ERR_ALIGN), ({"out_boxes": F + 8}, N.ERR_ALIGN), ({"gt_cls": F + 2}, N.ERR_ALIGN),
              ({"gt_offsets": F + 1}, N.ERR_ALIGN), ({"out_cls": F + 2}, N.ERR_ALIGN),
              ({"out_offsets": F + 2}, N.ERR_ALIGN), ({"out_src_row": F + 1}, N.ERR_ALIGN),
              ({"out_transform": F + 2}, N.ERR_ALIGN)]
    for kw, status in cases:
        assert _boxes(lib, **kw) == status, kw


def test_augment_images_rejects_each_bad_argument(native):
    import ctypes as C
    N, lib = native, native.lib()
    fill = (C.c_float * 3)(0.5, 0.5, 0.5)
    n = 4 * 300 * 300 * 3 * 4

    def call(images=F, transform=F, batch=4, height=300, width=300, fill=fill, out=F + n):
        return lib.ssdg_augment_images(images, transform, batch, height, width, fill, out, None)

    cases = [(dict(images=None), N.ERR_ARG), (dict(transform=None), N.ERR_ARG), (dict(fill=None), N.ERR_ARG),
             (dict(out=None), N.ERR_ARG), (dict(batch=0), N.ERR_ARG), (dict(height=0), N.ERR_ARG),
             (dict(width=-3), N.ERR_ARG), (dict(out=F), N.ERR_ARG), (dict(out=F + n - 4), N.ERR_ARG),
             (dict(images=F + n, out=F + 4), N.ERR_ARG), (dict(height=16385), N.ERR_LIMIT),
             (dict(width=16385), N.ERR_LIMIT), (dict(images=F + 2), N.ERR_ALIGN), (dict(transform=F + 1), N.ERR_ALIGN),
             (dict(out=F + n + 2), N.ERR_ALIGN)]
    for kw, status in cases:
        assert call(**kw) == status, kw
