"""GPU (B200): torch CUDA tensors passed in ``out=`` to ops.detect, ops.nms, ops.keep_top_k and ops.match_encode are
written in place, bit for bit what the same calls write into library-allocated outputs."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
from ssdgeom import ops, synth                  # noqa: E402
from ssdgeom.models import ssd_model as M       # noqa: E402

B = 2


@pytest.fixture(scope="module")
def inputs():
    priors = M.build_prior_box(synth.SSD300["sizes"])
    pc, pb = synth.make_predictions(11, B, priors.shape[0])
    return pc, pb, priors


def _tensors_like(ref, keys):
    """A torch CUDA tensor per key, shaped and typed like the library's output, filled with a value no output has."""
    dt = {np.dtype(np.int32): torch.int32, np.dtype(np.float32): torch.float32, np.dtype(np.uint8): torch.uint8}
    return {k: torch.full(ref[k].shape, 77, dtype=dt[ref[k].dtype], device="cuda") for k in keys}


def _assert_written_in_place(ref, out, tensors):
    torch.cuda.synchronize()
    for k, t in tensors.items():
        assert out[k].ptr == t.data_ptr(), k           # the output is a view of the caller's tensor
        got, want = t.cpu().numpy(), ref[k].to_host()
        assert got.dtype == want.dtype and got.shape == want.shape, k
        assert np.array_equal(got.view(np.uint8), want.view(np.uint8)), k


def test_detect_writes_torch_outputs(inputs):
    pc, pb, priors = inputs
    keys = ("kept", "count", "kept_score", "boxes")
    ref = ops.detect(pc, pb, priors, want_scores=True, want_boxes=True)
    tensors = _tensors_like(ref, keys)
    out = ops.detect(pc, pb, priors, want_scores=True, want_boxes=True, out=dict(tensors))
    _assert_written_in_place(ref, out, tensors)
    assert int(ref["count"].to_host().sum()) > 0


def test_nms_writes_torch_outputs(inputs):
    pc, pb, priors = inputs
    det = ops.detect(pc, pb, priors, want_boxes=True, want_probs=True)
    ref = ops.nms(det["probs"], det["boxes"], want_scores=True)
    tensors = _tensors_like(ref, ("kept", "count", "kept_score"))
    out = ops.nms(det["probs"], det["boxes"], want_scores=True, out=dict(tensors))
    _assert_written_in_place(ref, out, tensors)


def test_keep_top_k_writes_torch_outputs(inputs):
    pc, pb, priors = inputs
    det = ops.detect(pc, pb, priors, want_scores=True, want_boxes=True)
    ref = ops.keep_top_k(det, 100)
    tensors = _tensors_like(ref, ("prior", "class", "score", "box", "n", "count"))
    out = ops.keep_top_k(det, 100, out=dict(tensors))
    _assert_written_in_place(ref, out, tensors)


def test_match_encode_writes_torch_outputs(inputs):
    priors = inputs[2]
    boxes, cls, off = synth.make_gt(12, B, 20, "max")
    ref = ops.match_encode(boxes, cls, off, priors, B, 20, 0.5)
    tensors = _tensors_like(ref, ("cls", "loc", "mask"))
    out = ops.match_encode(boxes, cls, off, priors, B, 20, 0.5, out=dict(tensors))
    _assert_written_in_place(ref, out, tensors)
