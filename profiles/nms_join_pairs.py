"""Candidate pairs per class list that nms_kernel's interval join passes to the pair test, for the join over the list's
own box extents (tests/test_oracle.py, _nms_join_candidates) and over the fixed domain [0, 1]
(tests/test_nms_join_fixed_domain.py), on bench.py's SSD300 inputs: synthetic logits, top 200 of each (image, class)
list with score > 0.01, IoU threshold 0.45.  Both restatements use the kernel's float32 arithmetic; the counts are
computed on the CPU.  Also the rank sort's count-loop steps per list (the sum over buckets of their squared sizes)
with the buckets fitted to the list's score range and fixed over (0.01, 1].
usage: python profiles/nms_join_pairs.py [images]"""
import os
import sys

import numpy as np

root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [root, os.path.join(root, "tests"), os.path.join(root, "ssd-object-detection_b200")]
from oracle import ssd_oracle as O                                   # noqa: E402
from ssdgeom import synth                                            # noqa: E402
from test_oracle import _nms_join_candidates as join_list_extents    # noqa: E402
from test_nms_join_fixed_domain import join_candidates as join_fixed  # noqa: E402

images = int(sys.argv[1]) if len(sys.argv) > 1 else 8
priors = O.build_prior_box()
a = priors.shape[0]
pred_cls, pred_box = synth.make_predictions(100, images, a)
probs = O.softmax(pred_cls)
boxes = O.decode_bbox(pred_box, priors, scale=1.0)
old, new, hot, sizes, steps_fit, steps_fixed = [], [], [], [], [], []
key_thr, key_one = (np.array([0.01, 1.0], np.float32).view(np.uint32) | np.uint32(0x80000000)).astype(np.int64)
for b in range(images):
    for c in range(probs.shape[2] - 1):
        s = probs[b, :, c]
        cand = np.nonzero(s > np.float32(0.01))[0]
        cand = cand[np.lexsort((cand, -s[cand].astype(np.float64)))][:200]
        bx = boxes[b, cand]
        k = (s[cand].view(np.uint32) | np.uint32(0x80000000)).astype(np.int64)   # score words of the keys
        fit = np.minimum(255, ((k - k.min()) * np.float32(256.0 / (k.max() - k.min() + 1) * 0.999)).astype(np.int64))
        fixed = np.minimum(255, ((k - key_thr) * np.float32(256.0 / (key_one - key_thr))).astype(np.int64))
        steps_fit.append(int((np.bincount(fit) ** 2).sum())); steps_fixed.append(int((np.bincount(fixed) ** 2).sum()))
        _, _, k_old = join_list_extents(bx, 0.45)
        i, j, k_new, _ = join_fixed(bx, 0.45)
        with np.errstate(all="ignore"):
            h = O.iou(bx[i], bx[j]) > np.float32(0.45)
        assert not np.any(h & ~k_new)
        old.append(int(k_old.sum())); new.append(int(k_new.sum())); hot.append(int(h.sum())); sizes.append(len(cand))
print("SSD300, %d images x 80 lists, %.1f boxes per list (%.0f pairs), IoU 0.45" %
      (images, np.mean(sizes), np.mean([n * (n - 1) / 2 for n in sizes])))
print("candidate pairs per list: list extents %.1f, fixed [0, 1] domain %.1f; pairs above the threshold %.1f" %
      (np.mean(old), np.mean(new), np.mean(hot)))
print("rank-sort count-loop steps per list: fitted buckets %.1f, fixed buckets %.1f" %
      (np.mean(steps_fit), np.mean(steps_fixed)))
