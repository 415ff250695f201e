"""GPU (B200): the discrete decisions of the hot path at exact ties, saturated rows and code-path boundaries, against
the CPU oracle (oracle/ssd_oracle.py).  The logits of the parity suite are continuous, so a cut there never falls
inside a run of equal values; here every input is built so that it does, and every test asserts that the path it
aims at was taken.

  A  NMS top-k (nms_kernel): all-equal scores (the prior-word buckets of the rank sort), the top_k cut inside a run of
     equal scores, levels one ulp apart, list lengths at top_k +- 1 and at the sort width +- 1 (radix select),
     duplicate boxes of equal score
  B  the all-candidates worst case the detection workspace is sized for: identical rows everywhere
  C  hard-negative mining with CE values that tie by the hundred, the k-th position inside a tie group
  D  saturated background rows (float32 CE exactly 0) on the standalone, fused, staged and chained loss paths
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import ssd_oracle as O          # noqa: E402  (the checker)
from ssdgeom import synth                   # noqa: E402
from ssdgeom import ops, device as D        # noqa: E402
from ssdgeom import parallel                # noqa: E402

A300 = 8732


@pytest.fixture(scope="module")
def priors300():
    return O.build_prior_box()


def close(got, want, rtol=1e-5, atol=0.0):
    np.testing.assert_allclose(np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64), rtol=rtol, atol=atol)


def sort_width(top_k):
    """The NMS sort width: lists longer than this go through the radix select first."""
    p = 32
    while p < top_k:
        p <<= 1
    return p


def ulps(hi, lo):
    """Distance in float32 units in the last place of two positive floats."""
    return int(np.float32(hi).view(np.int32)) - int(np.float32(lo).view(np.int32))


# ---- A: NMS top-k at ties and size boundaries -------------------------------------------------------------------
def ranked_scores(pattern, n, top_k):
    """The n candidate scores in visit order (descending).  'levels' and 'ulp' have three levels; the middle one
    covers [top_k - r, top_k + r), so positions top_k - 1 and top_k tie whenever the list is longer than top_k."""
    mid = np.float32(0.5)
    if pattern == "equal":
        return np.full(n, mid, np.float32)
    if pattern == "levels":
        hi, lo = np.float32(0.75), np.float32(0.25)
    else:                                                  # one ulp apart
        hi, lo = np.nextafter(mid, np.float32(1)), np.nextafter(mid, np.float32(0))
    r = max(1, top_k // 2)
    out = np.full(n, lo, np.float32)
    out[:max(0, top_k - r)] = hi
    out[max(0, top_k - r):top_k + r] = mid
    return out


def nms_case(rng, n, pattern, geometry, top_k, a):
    """One image: class 1 holds exactly n candidates (scattered over the priors, the scores dealt at random so that
    tie runs interleave in prior order), class 0 and the background are 0.  'disjoint': every prior has its own cell
    of a grid, nothing overlaps, the kept list is the visit order.  'dup': candidates of equal score come in clusters
    of up to three exact duplicates, of which only the lowest prior may survive."""
    probs = np.zeros((a, 3), np.float32)
    cand = rng.choice(a, n, replace=False)
    probs[cand, 1] = ranked_scores(pattern, n, top_k)
    g = int(np.ceil(np.sqrt(a)))
    cell = np.arange(a)
    boxes = np.stack([(cell % g + 0.5) / g, (cell // g + 0.5) / g, np.full(a, 0.4 / g), np.full(a, 0.4 / g)], 1)
    boxes = boxes.astype(np.float32)
    if geometry == "dup":
        for s in np.unique(probs[cand, 1]):
            members = np.sort(cand[probs[cand, 1] == s])       # consecutive in the visit order
            for i in range(0, members.size, 3):
                boxes[members[i:i + 3]] = boxes[members[i]]
    return probs, boxes


@pytest.mark.parametrize("top_k", [1, 31, 32, 33, 200, 256, 1000, 1024])
def test_nms_topk_ties_and_boundaries(top_k):
    """Kept lists and counts bit-equal to O.nms_per_class at exact ties, for list lengths at top_k +- 1, at the sort
    width and one beyond it (radix select), and at more than four times the sort width.  top_k = 1024 is the
    documented limit of ssdg_nms."""
    rng = np.random.default_rng(top_k)
    sortn = sort_width(top_k)
    sizes = sorted({v for v in (top_k - 1, top_k, top_k + 1, sortn, sortn + 1, 4 * sortn + 3) if v >= 1})
    a = 4 * sortn + 37                                    # not a multiple of 32: the last tile is partial
    cases = [(n, p, g) for n in sizes for p in ("equal", "levels", "ulp") for g in ("disjoint", "dup")]
    built = [nms_case(rng, n, p, g, top_k, a) for n, p, g in cases]
    probs = np.stack([b[0] for b in built])
    boxes = np.stack([b[1] for b in built])
    out = ops.nms(probs, boxes, score_thresh=0.01, top_k=top_k, iou_thresh=0.45, want_scores=True)
    kept, count, score = out["kept"].to_host(), out["count"].to_host(), out["kept_score"].to_host()
    selected = tie_cuts = suppressed = 0
    for i, (n, pattern, geometry) in enumerate(cases):
        what = (n, pattern, geometry)
        w_kept, w_count = O.nms_per_class(probs[i], boxes[i], 0.01, top_k, 0.45)
        assert np.array_equal(count[i], w_count), what
        assert np.array_equal(kept[i], w_kept), what
        k = kept[i, 1, :count[i, 1]]
        assert np.array_equal(score[i, 1, :count[i, 1]], probs[i, k, 1]), what
        assert count[i, 0] == 0 and np.all(kept[i, 0] == -1)
        # not vacuous: the list really had n entries, the cut really fell inside a run of equal scores
        s = probs[i, :, 1]
        cand = np.nonzero(s > np.float32(0.01))[0]
        assert cand.size == n
        selected += n > sortn
        if n > top_k:
            visit = s[cand[np.lexsort((cand, -s[cand].astype(np.float64)))]]
            assert visit[top_k - 1] == visit[top_k], what
            tie_cuts += 1
        if geometry == "dup" and min(n, top_k) >= 3:
            assert count[i, 1] < min(n, top_k), what      # duplicates were suppressed
            suppressed += 1
        if geometry == "disjoint":
            assert count[i, 1] == min(n, top_k), what     # nothing overlaps: the kept list is the visit order
    assert selected == 12 and tie_cuts > 0 and (suppressed > 0 or top_k < 3)


# ---- B: identical rows everywhere --------------------------------------------------------------------------------
def constant_case(priors, top_k=200):
    """Logits 0 everywhere: every class list of every image holds all A priors at the same score 1/81, and the
    decoded boxes are the priors themselves.  One oracle list stands for every (image, class)."""
    boxes = O.decode_bbox(np.zeros((A300, 4), np.float32), priors, 1.0, np.float64)
    score = np.full(A300, np.float32(1.0 / 81.0), np.float32)
    want = O.nms_single_class(score, boxes, 0.01, top_k, 0.45)
    return want


def assert_all_lists(kept, count, want, top_k=200):
    row = np.full(top_k, -1, np.int32)
    row[:want.size] = want
    assert np.all(count == want.size)
    assert np.all(kept == row[None, None, :])


def test_detect_all_candidates_constant_logits(priors300):
    """ops.detect on both filter variants (the probabilities variant and the streaming one) with every row
    identical: all 3 x 80 lists must equal the one oracle list."""
    b = 3
    pc = np.zeros((b, A300, 81), np.float32)
    pb = np.zeros((b, A300, 4), np.float32)
    want = constant_case(priors300)
    assert A300 > sort_width(200) and 0 < want.size < 200
    probs_v = ops.detect(pc, pb, priors300, want_probs=True, want_scores=True)
    stream_v = ops.detect(pc, pb, priors300, want_row_stats=True, want_scores=True)
    for out in (probs_v, stream_v):
        kept, count = out["kept"].to_host(), out["count"].to_host()
        assert_all_lists(kept, count, want)
        score = out["kept_score"].to_host()
        assert np.all(score[:, :, :want.size] == score[0, 0, 0]) and score[0, 0, 0] > np.float32(0.01)
    p = probs_v["probs"].to_host()
    close(p, 1.0 / 81.0, rtol=1e-6)
    assert np.all(p[..., :-1] > np.float32(0.01))        # every prior is a candidate of every class
    close(stream_v["row_negbg"].to_host(), np.log(81.0), rtol=1e-6)


def test_chained_step_all_candidates_full_batch(priors300):
    """One HotPath step (depth 2) at B = 256 with identical rows: every one of the 256 x 80 lists holds all 8 732
    priors and must equal the one oracle list; in the loss every negative ties, so all of them are mined and the
    threshold is the common CE log(81)."""
    from ssdgeom.pipeline import HotPath
    b = 256
    boxes, cls, off = synth.make_gt(91, b, 100, "coco")
    hp = HotPath(synth.SSD300, batch=b, max_gt=int(np.diff(off).max()), total_gt=boxes.shape[0], depth=2)
    pc = np.zeros((b, A300, 81), np.float32)
    pb = np.zeros((b, A300, 4), np.float32)
    hp.upload(boxes, cls, off, pc, pb)
    hp.step()
    hp.join()
    hp.s_main.sync()
    want = constant_case(priors300)
    assert_all_lists(hp.det["kept"].to_host(), hp.det["count"].to_host(), want)
    r = ops.loss_result_to_host(hp.loss["result"])
    num_pos = int(hp.tgt["mask"].to_host().astype(bool).sum())
    assert r["num_pos"] == num_pos > 0
    assert r["num_neg"] == b * A300 - num_pos > 3 * num_pos
    close(r["kth"], np.log(81.0), rtol=1e-6)
    close(r["cls loss neg"], r["kth"], rtol=1e-12)      # every mined value is the same float


# ---- C / D: hard-negative mining at exact ties -------------------------------------------------------------------
def targets(seed, b, priors):
    boxes, cls, off = synth.make_gt(seed, b, 100, "coco")
    t = ops.match_encode(boxes, cls, off, priors, b, int(np.diff(off).max()), 0.5)
    y_true = (t["cls"].to_host(), t["loc"].to_host(), t["mask"].to_host().astype(bool))
    return y_true, (boxes, cls, off)


def ce64(rows):
    x = np.asarray(rows, np.float64)
    m = x.max(axis=-1, keepdims=True)
    return np.log(np.exp(x - m).sum(axis=-1)) - (x[..., -1] - m[..., 0])


def pool_rows(rng, n, fg_shift, bg):
    """n rows sharing one foreground vector, background logits `bg` (one per row): CE values far apart."""
    v = (rng.standard_normal(80) * 0.5 + fg_shift).astype(np.float32)
    rows = np.empty((n, 81), np.float32)
    rows[:, :80] = v
    rows[:, 80] = np.asarray(bg, np.float32)
    return rows


def ulp_pair(row):
    """A copy of `row` with one foreground logit raised until the float32 CE is exactly two ulps above the row's,
    both CE values sharing their top 22 key bits (so the select resolves them at its last radix level only)."""
    lo = np.float32(ce64(row))

    def raised(delta):
        r = row.copy()
        r[0] = np.float32(row[0] + delta)
        return r, ulps(np.float32(ce64(r)), lo)

    below, above = 0.0, 1e-7
    while raised(above)[1] < 2:
        above *= 2
    for _ in range(60):             # the smallest raise that moves the CE by two ulps
        mid = (below + above) / 2
        if raised(mid)[1] >= 2:
            above = mid
        else:
            below = mid
    hi_row, d = raised(above)
    assert d == 2 and (int(lo.view(np.int32)) & 1023) < 1000, (d, lo)
    return hi_row


def deal(rng, y_true, groups, rest, pool):
    """Logits [B,A,81]: negatives take the pool rows of `groups` (list of (pool index, count), in that order of the
    dealing) and then, at random, the rows of `rest`; positives take random rows of `rest`.  Returns the logits and
    the pool index of every prior."""
    mask = y_true[2]
    b, a = mask.shape
    which = np.empty(b * a, np.int64)
    neg = rng.permutation(np.nonzero(~mask.reshape(-1))[0])
    pos = np.nonzero(mask.reshape(-1))[0]
    at = 0
    for g, cnt in groups:
        which[neg[at:at + cnt]] = g
        at += cnt
    which[neg[at:]] = rng.choice(rest, neg.size - at)
    which[pos] = rng.choice(rest, pos.size)
    return pool[which].reshape(b, a, 81), which.reshape(b, a)


def outcome(out):
    """(result dict, mask, neg_ce) of a loss call, or the AssertionError its result block raises."""
    try:
        r = ops.loss_result_to_host(out["result"])
    except AssertionError as e:
        return e
    return r, out["neg_mask"].to_host().astype(bool), out["neg_ce"].to_host()


def run_paths(y_true, pred_box, pred_cls, priors, shards=(2, 3)):
    """The outcome of every loss path on one batch: standalone, fused (the filter's row statistics), and the staged
    cross-shard mining over `shards` emulated shards without and with row statistics (then also the shard spans)."""
    gt_cls, gt_box, gt_mask = y_true
    b = pred_cls.shape[0]
    d_cls = D.to_device(pred_cls)
    res = {}
    res["standalone"] = outcome(ops.multibox_loss(gt_cls, gt_box, gt_mask, pred_box, d_cls, want_neg_mask=True,
                                                  want_neg_ce=True))
    det = ops.detect(d_cls, pred_box, priors, want_row_stats=True)
    res["fused"] = outcome(ops.multibox_loss(gt_cls, gt_box, gt_mask, pred_box, d_cls, want_neg_mask=True,
                                             want_neg_ce=True, row_stats=(det["row_ml"], det["row_negbg"]),
                                             ws_kind="loss_fused"))
    row_ml, row_negbg = det["row_ml"].to_host(), det["row_negbg"].to_host()
    for n in shards:
        for stats in (False, True):
            name = "staged%d%s" % (n, "_fused" if stats else "")
            spans = [parallel.shard_range(b, n, r) for r in range(n)]
            staged = [ops.StagedLoss(*(v[lo:hi] for v in y_true), pred_box[lo:hi], pred_cls[lo:hi],
                                     global_priors=b * A300, want_neg_mask=True, want_neg_ce=True,
                                     ws_kind="loss_staged_%d" % r,
                                     row_stats=(D.to_device(row_ml[lo:hi]), D.to_device(row_negbg[lo:hi])) if stats else None)
                      for r, (lo, hi) in enumerate(spans)]
            for stage in range(4):
                for s in staged:
                    s.run(stage)
                for bufs in zip(*(s.exchange(stage) for s in staged)):     # the all-reduce: a host-side sum
                    tot = sum(x.to_host().astype(np.float64 if x.dtype == np.float64 else np.int64) for x in bufs)
                    for x in bufs:
                        x.copy_from_host(tot.astype(x.dtype))
                    D.sync()
            try:
                info = [s.finish()[1] for s in staged]
            except AssertionError as e:
                res[name] = e
                continue
            assert all(i["kth"] == info[0]["kth"] and i["num_neg"] == info[0]["num_neg"] for i in info)
            res[name] = (dict(info[0]), np.concatenate([s.out["neg_mask"].to_host() for s in staged]).astype(bool),
                         np.concatenate([s.out["neg_ce"].to_host() for s in staged]), spans)
    return res


def cut_plan(k, order, lead):
    """Negatives dealt to the pool rows `order` (CE descending), `lead` of them in counts of ~0.23 k each: the k-th
    largest value then falls strictly inside the group at index `lead - 1`."""
    s = int(np.ceil(0.23 * k))
    assert (lead - 1) * s < k - 1 and lead * s > k + 1
    return [(g, s) for g in order[:lead]]


@pytest.mark.parametrize("case", ["separated", "ulp_pair"])
def test_mining_exact_ties(case, priors300):
    """CE values tie in groups of hundreds (every prior takes one of ~30 pool rows) and k = 3 num_pos falls inside
    a group.

    separated: neighbouring groups differ by far more than rounding, so the ties are exact in the kernels and in the
    float64 oracle alike: the mask must equal the oracle's end to end on every path, and the gradient the oracle's.
    ulp_pair: the cut group and the one above it are two float32 ulps apart -- the select must resolve them at its
    last radix level; at that spacing the kernels' and the oracle's roundings may order the pair differently, so the
    mask is checked on each path's own CE vector (two-stage contract).

    kth is the cut group's own CE value on every path and identical between the paths that share a CE formula
    (standalone / staged / gradient, and fused / staged with row statistics); the two formulas round differently,
    so across them it agrees to rounding (and the masks are identical: the groups are far apart or exactly tied)."""
    rng = np.random.default_rng(17 if case == "separated" else 18)
    b = 4
    y_true, _ = targets(61, b, priors300)
    num_pos = int(y_true[2].sum())
    k = 3 * num_pos
    pool = pool_rows(rng, 30, 0.0, np.linspace(-2.0, 6.0, 30))   # CE descending with the index
    order = list(range(30))
    if case == "ulp_pair":
        lo = pool_rows(np.random.default_rng(5), 1, 0.0, [(pool[2, 80] + pool[3, 80]) / 2])[0]
        lo[:80] = pool[0, :80]
        pool = np.concatenate([pool, ulp_pair(lo)[None], lo[None]])      # 30: two ulps above 31
        order = [0, 1, 2, 30, 31] + list(range(3, 30))
    gaps = -np.diff(ce64(pool)[order])
    if case == "ulp_pair":
        assert ulps(np.float32(ce64(pool[30])), np.float32(ce64(pool[31]))) == 2
        gaps = np.delete(gaps, 3)
    assert np.all(gaps > 1e-3)                                           # far more than rounding
    groups = cut_plan(k, order, 5)
    cut = groups[-1][0]
    pred_cls, which = deal(rng, y_true, groups, order[5:], pool)
    pred_box = (rng.standard_normal((b, A300, 4)) * 0.5).astype(np.float32)
    res = run_paths(y_true, pred_box, pred_cls, priors300)

    w_total, w_info, w_aux = O.ssd_loss(y_true, (pred_box, pred_cls), return_masks=True)
    cut_rows = (which == cut) & ~y_true[2]
    kths = {}
    for name, v in res.items():
        assert not isinstance(v, Exception), (name, v)
        r, mask, neg_ce = v[:3]
        assert r["num_pos"] == num_pos
        # the two-stage contract: the mask is the hard-negative select of the path's own CE vector
        kth, want = O.hard_negative_select(neg_ce, num_pos, 3)
        assert np.array_equal(mask, want), name
        assert np.float32(r["kth"]) == kth and r["num_neg"] == int(mask.sum()), name
        # not vacuous: the k-th value is the cut group's (exact ties), so more than k negatives are mined
        assert np.all(neg_ce[cut_rows] == kth), name
        assert r["num_neg"] > k, name
        close(neg_ce, w_aux["neg_ce"], rtol=1e-5, atol=1e-6)
        kths[name] = kth
        if case == "separated":
            assert np.array_equal(mask, w_aux["neg_mask"]), name       # end to end
        if name.startswith("staged"):
            spans = v[3]
            for lo_, hi_ in spans:      # the cut group spans the shards; each shard's mask is its slice
                assert cut_rows[lo_:hi_].any()
                single = res["fused" if name.endswith("_fused") else "standalone"][1]
                assert np.array_equal(mask[lo_:hi_], single[lo_:hi_]), name
    assert np.array_equal(res["standalone"][1], res["fused"][1])
    plain = [v for n, v in kths.items() if not n.endswith("fused")]
    fusedk = [v for n, v in kths.items() if n.endswith("fused")]
    assert len(set(plain)) == 1 and len(set(fusedk)) == 1
    close(fusedk[0], plain[0], rtol=1e-6)
    if case == "ulp_pair":
        hi_rows = (which == 30) & ~y_true[2]
        for name in ("standalone", "fused"):
            neg_ce = res[name][2]
            hi_v, lo_v = np.float32(neg_ce[hi_rows][0]), np.float32(neg_ce[cut_rows][0])
            assert np.all(neg_ce[hi_rows] == hi_v)
            assert 0 < ulps(hi_v, lo_v) <= 8, (name, hi_v, lo_v)   # distinct and adjacent on the device too
            assert (int(hi_v.view(np.int32)) >> 10) == (int(lo_v.view(np.int32)) >> 10)
    else:
        from ssdgeom.models import ssd_model as M
        total, _, g_box, g_cls = M.ssd_loss_grad(y_true, (pred_box, pred_cls))
        w_box, w_cls = O.ssd_loss_grad(y_true, (pred_box, pred_cls))
        close(total, w_total, rtol=1e-5)
        close(g_box, w_box, rtol=1e-5, atol=1e-12)
        close(g_cls, w_cls, rtol=2e-5, atol=1e-9)
        grad_neg = np.any(g_cls != 0, axis=-1) & ~y_true[2]
        assert np.array_equal(grad_neg, res["standalone"][1])           # the gradient reuses the threshold


@pytest.mark.parametrize("case", ["k_in_unsaturated", "k_in_saturated"])
def test_mining_saturated_background(case, priors300):
    """Negative rows whose background logit is 40 above the rest: their float32 CE is exactly 0 on every kernel
    path (the sum of the max-shifted exponentials rounds to 1, as in TensorFlow's float32 evaluation of the
    formula).  The float64 oracle keeps a tiny value there (0 or a few 1e-16,
    its own resolution), so its k-th value stays positive and it does not raise; on rows below the formula's float32
    resolution the kernels follow the float32 evaluation.

    k_in_unsaturated: k = 3 num_pos falls among the other negatives (background 1.5 + 0.1 j, CE ~0.1-1): every path
    mines the same mask with the same count and threshold.
    k_in_saturated: fewer than k negatives are unsaturated, the k-th value is 0, the positives (0 in the mining
    vector) tie with it and are mined: every path raises the reference's AssertionError (models/ssd_model.py:375)."""
    from ssdgeom.pipeline import HotPath
    rng = np.random.default_rng(23)
    b = 4
    y_true, (boxes, cls, off) = targets(62, b, priors300)
    num_pos = int(y_true[2].sum())
    k = 3 * num_pos
    unsat = pool_rows(rng, 20, -3.0, 1.5 + 0.1 * np.arange(20))          # CE descending with the index
    sat = pool_rows(rng, 8, 0.0, 40.0 + 0.25 * np.arange(8))
    pool = np.concatenate([unsat, sat])
    ce = ce64(pool)
    assert np.all((ce[:20] > 0.1) & (ce[:20] < 1.0)) and np.all(ce[20:] < 1e-12)
    n_neg = b * A300 - num_pos
    if case == "k_in_unsaturated":
        groups = cut_plan(k, list(range(20)), 5)
        groups += [(g, k // 10) for g in range(5, 20)]                   # more unsaturated ones below the cut
    else:
        s = int(0.23 * k)
        groups = [(0, s), (1, s)]                                         # 0.46 k unsaturated negatives
    n_unsat = sum(c for _, c in groups)
    assert n_unsat < n_neg - 1000
    pred_cls, which = deal(rng, y_true, groups, list(range(20, 28)), pool)
    # the positives and the dealt negatives keep their rows; only negatives beyond the groups are saturated
    pos = y_true[2]
    pred_cls[pos] = unsat[rng.integers(0, 20, int(pos.sum()))]
    which[pos] = -1
    pred_box = (rng.standard_normal((b, A300, 4)) * 0.5).astype(np.float32)
    sat_rows = (which >= 20) & ~pos
    assert sat_rows.sum() == n_neg - n_unsat

    gt_cls, gt_box, gt_mask = y_true
    d_cls = D.to_device(pred_cls)
    hp = HotPath(synth.SSD300, batch=b, max_gt=int(np.diff(off).max()), total_gt=boxes.shape[0])
    hp.upload(boxes, cls, off, pred_cls, pred_box)
    hp.step()
    hp.s_main.sync()
    assert np.array_equal(hp.tgt["mask"].to_host().astype(bool), gt_mask)

    if case == "k_in_saturated":
        # the oracle does not raise: its CE of the saturated rows is a tiny positive float32
        _, _, w_aux = O.ssd_loss(y_true, (pred_box, pred_cls), return_masks=True)
        assert w_aux["kth"] > 0 and w_aux["neg_ce"][sat_rows].max() > 0
        alone = ops.multibox_loss(gt_cls, gt_box, gt_mask, pred_box, d_cls, want_neg_ce=True)
        assert np.all(alone["neg_ce"].to_host()[sat_rows] == 0)           # not vacuous: the zero run is there
        res = run_paths(y_true, pred_box, pred_cls, priors300, shards=(2,))
        for name in ("standalone", "fused", "staged2", "staged2_fused"):
            assert isinstance(res[name], AssertionError), name
        with pytest.raises(AssertionError):
            ops.loss_result_to_host(hp.loss["result"])
        return

    res = run_paths(y_true, pred_box, pred_cls, priors300, shards=(2,))
    cut_rows = (which == groups[4][0]) & ~pos
    ref = res["standalone"]
    for name, v in res.items():
        assert not isinstance(v, Exception), (name, v)
        r, mask, neg_ce = v[:3]
        assert np.array_equal(mask, ref[1]), name
        assert r["num_neg"] == ref[0]["num_neg"] == int(mask.sum()) > k, name
        assert np.all(neg_ce[cut_rows] == np.float32(r["kth"])), name
        close(r["kth"], ref[0]["kth"], rtol=1e-6)
        assert not np.any(mask[sat_rows]), name
        # the CE of a saturated row is +0 on every path, never negative anywhere
        assert np.all(neg_ce[sat_rows] == 0) and not np.any(np.signbit(neg_ce)), name
    r = ops.loss_result_to_host(hp.loss["result"])
    assert r["num_neg"] == res["fused"][0]["num_neg"] and r["kth"] == res["fused"][0]["kth"]
    w_total, _, w_aux = O.ssd_loss(y_true, (pred_box, pred_cls), return_masks=True)
    assert np.array_equal(ref[1], w_aux["neg_mask"])
    close(ref[0]["total"], w_total)
