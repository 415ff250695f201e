"""CPU: the argument checks of the detection entry points (ssdg_detect, ssdg_detect_stage, ssdg_nms), one invalid
argument per call, each answered with its exact status code.  Every call below fails validation, so none reaches a
CUDA launch: the pointers are fake (aligned where they are not under test) and the workspace is declared large."""
import pytest

F = 1 << 20              # a fake device pointer, 256-byte aligned
BIG_WS = 1 << 40         # workspace bytes that pass the size check


@pytest.fixture(scope="module")
def native():
    import build_native
    build_native.build()
    from ssdgeom import _native
    return _native


def _logits_args(**kw):
    """The arguments ssdg_detect and ssdg_detect_stage share, as a valid SSD300-sized call, with overrides."""
    a = dict(pred_cls=F, pred_box=F, priors=F, prior_dtype=1, batch=4, n_priors=8732, n_classes=81, score_thresh=0.01,
             top_k=200, iou_thresh=0.45, out_kept=F, out_count=F, out_kept_score=F, out_boxes=F, out_probs=F,
             head_thresh=0.5, head_score=F, head_cls=F, head_mask=F, out_row_ml=F, out_row_negbg=F, workspace=F,
             workspace_bytes=BIG_WS)
    a.update(kw)
    return a


def _detect(lib, **kw):
    a = _logits_args(**kw)
    return lib.ssdg_detect(a["pred_cls"], a["pred_box"], a["priors"], a["prior_dtype"], a["batch"], a["n_priors"],
                           a["n_classes"], a["score_thresh"], a["top_k"], a["iou_thresh"], a["out_kept"],
                           a["out_count"], a["out_kept_score"], a["out_boxes"], a["out_probs"], a["head_thresh"],
                           a["head_score"], a["head_cls"], a["head_mask"], a["workspace"], a["workspace_bytes"], None)


def _stage(lib, stage, **kw):
    a = _logits_args(**kw)
    return lib.ssdg_detect_stage(stage, a["pred_cls"], a["pred_box"], a["priors"], a["prior_dtype"], a["batch"],
                                 a["n_priors"], a["n_classes"], a["score_thresh"], a["top_k"], a["iou_thresh"],
                                 a["out_kept"], a["out_count"], a["out_kept_score"], a["out_boxes"], a["out_probs"],
                                 a["head_thresh"], a["head_score"], a["head_cls"], a["head_mask"], a["out_row_ml"],
                                 a["out_row_negbg"], a["workspace"], a["workspace_bytes"], None)


def _nms(lib, **kw):
    a = dict(probs=F, boxes=F, batch=4, n_priors=8732, n_classes=81, score_thresh=0.01, top_k=200, iou_thresh=0.45,
             out_kept=F, out_count=F, out_kept_score=F, workspace=F, workspace_bytes=BIG_WS)
    a.update(kw)
    return lib.ssdg_nms(a["probs"], a["boxes"], a["batch"], a["n_priors"], a["n_classes"], a["score_thresh"],
                        a["top_k"], a["iou_thresh"], a["out_kept"], a["out_count"], a["out_kept_score"], a["workspace"],
                        a["workspace_bytes"], None)


def _common_cases(N, inputs):
    """(override, status) for the checks every entry point makes; ``inputs``: its non-null input pointers."""
    cases = [({k: None}, N.ERR_ARG) for k in inputs + ("out_kept", "out_count")]
    cases += [({"batch": 0}, N.ERR_ARG), ({"batch": -1}, N.ERR_ARG), ({"n_priors": 0}, N.ERR_ARG),
              ({"n_priors": -5}, N.ERR_ARG), ({"n_classes": 1}, N.ERR_ARG), ({"n_classes": 0}, N.ERR_ARG),
              ({"top_k": 0}, N.ERR_ARG), ({"top_k": -1}, N.ERR_ARG)]
    cases += [({"top_k": 1025}, N.ERR_LIMIT), ({"n_classes": 2049}, N.ERR_LIMIT), ({"n_priors": 1 << 21}, N.ERR_LIMIT),
              ({"batch": 0x7fffffff // 64 + 1}, N.ERR_LIMIT)]
    cases += [({"workspace": None}, N.ERR_WORKSPACE), ({"workspace": F + 16}, N.ERR_WORKSPACE),
              ({"workspace_bytes": 1000}, N.ERR_WORKSPACE), ({"workspace_bytes": 0}, N.ERR_WORKSPACE)]
    return cases


def _logits_cases(N):
    cases = _common_cases(N, ("pred_cls", "pred_box", "priors"))
    cases += [({"prior_dtype": 2}, N.ERR_ARG), ({"prior_dtype": -1}, N.ERR_ARG)]
    cases += [({"pred_cls": F + 2}, N.ERR_ALIGN), ({"out_probs": F + 2}, N.ERR_ALIGN), ({"pred_box": F + 4}, N.ERR_ALIGN),
              ({"priors": F + 8}, N.ERR_ALIGN), ({"out_boxes": F + 4}, N.ERR_ALIGN)]
    return cases


def test_detect_rejects_each_bad_argument(native):
    lib = native.lib()
    for kw, status in _logits_cases(native):
        assert _detect(lib, **kw) == status, kw


@pytest.mark.parametrize("stage", [0, 1])
def test_detect_stage_rejects_each_bad_argument(native, stage):
    lib = native.lib()
    cases = _logits_cases(native)
    cases += [({"out_row_ml": None}, native.ERR_ARG), ({"out_row_negbg": None}, native.ERR_ARG),
              ({"out_row_ml": F + 4}, native.ERR_ALIGN), ({"out_row_negbg": F + 2}, native.ERR_ALIGN)]
    for kw, status in cases:
        assert _stage(lib, stage, **kw) == status, (stage, kw)
    for bad in (-1, 2):
        assert _stage(lib, bad) == native.ERR_ARG, bad


def test_nms_rejects_each_bad_argument(native):
    lib = native.lib()
    cases = _common_cases(native, ("probs", "boxes"))
    cases += [({"probs": F + 2}, native.ERR_ALIGN), ({"boxes": F + 4}, native.ERR_ALIGN),
              ({"boxes": F + 8}, native.ERR_ALIGN)]
    for kw, status in cases:
        assert _nms(lib, **kw) == status, kw
