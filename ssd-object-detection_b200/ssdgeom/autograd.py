"""Autograd bridge for the multibox loss: what ``tape.gradient`` does through ``_ssd_loss`` in the reference's
training step (models/ssd_model.py:240-248), for a PyTorch host.  The reference is TensorFlow (absent here); the
same three lines would sit in a ``tf.custom_gradient`` (INTEGRATION.md).  torch is used for device memory and the
autograd tape only: forward and backward are the library's kernels, called through the C ABI on torch's current
stream with zero-copy views (``__cuda_array_interface__``) -- no host round trip, no synchronisation.

    total, info = ssdgeom.autograd.ssd_loss((gt_cls, gt_box, gt_mask), (pred_box, pred_cls))
    total.backward()            # pred_box.grad, pred_cls.grad

``total`` is a float64 CUDA scalar.  Data-dependent errors (no positive prior, k out of range: models/ssd_model.py:369,
:368) make it NaN -- ``check=True`` reads the status word (one synchronisation) and raises like the reference."""
from __future__ import annotations

import numpy as np
import torch

from . import _native as N
from . import ops

_POOL = ops.WorkspacePool()


def _u8(mask: torch.Tensor) -> torch.Tensor:
    return mask.view(torch.uint8) if mask.dtype == torch.bool else mask


class _MultiboxLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred_box, pred_cls, gt_cls, gt_box, gt_mask, neg_ratio):
        if not (pred_box.is_cuda and pred_cls.is_cuda):
            raise N.SsdgeomError("ssdgeom.autograd.ssd_loss needs CUDA tensors (there is no CPU fallback)")
        pb, pc = pred_box.detach().contiguous().float(), pred_cls.detach().contiguous().float()
        result = torch.empty(N.LOSS_RESULT_LEN, dtype=torch.float64, device=pc.device)
        need_grad = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        out = {"result": result}
        if need_grad:       # the backward kernel runs right behind the forward: one enqueue, no tape-time launch
            out["grad_box"], out["grad_cls"] = torch.empty_like(pb), torch.empty_like(pc)
        stream = torch.cuda.current_stream(pc.device).cuda_stream
        ops.multibox_loss(gt_cls.contiguous().int(), gt_box.contiguous().float(), _u8(gt_mask.contiguous()), pb, pc,
                          int(neg_ratio), want_grad=need_grad, out=out, stream=stream, pool=_POOL)
        if need_grad:
            ctx.save_for_backward(out["grad_box"], out["grad_cls"])
        ctx.mark_non_differentiable(result)
        return result[N.LOSS_TOTAL].clone(), result

    @staticmethod
    def backward(ctx, g_total, _g_result):
        g_box, g_cls = ctx.saved_tensors
        g = g_total.to(torch.float32)
        return (g_box * g if ctx.needs_input_grad[0] else None, g_cls * g if ctx.needs_input_grad[1] else None,
                None, None, None, None)


def ssd_loss(y_true, y_pred, neg_ratio: int = 3, check: bool = False):
    """``_ssd_loss(y_true, y_pred)`` (models/ssd_model.py:341-396) on CUDA tensors, differentiable w.r.t. the
    predictions.  y_true = (gt_cls int32 [b,A], gt_box f32 [b,A,4], gt_mask bool/uint8 [b,A]); y_pred = (pred_box,
    pred_cls).  Returns (total, {"cls loss pos", "cls loss neg", "loc loss"}) as CUDA scalars (info is detached)."""
    gt_cls, gt_box, gt_mask = y_true
    pred_box, pred_cls = y_pred
    # models/ssd_model.py:347-351
    assert gt_cls.shape[0] == gt_box.shape[0] == gt_mask.shape[0] == pred_box.shape[0] == pred_cls.shape[0]
    assert tuple(gt_cls.shape[:2]) == tuple(pred_cls.shape[:2])
    total, result = _MultiboxLoss.apply(pred_box, pred_cls, gt_cls, gt_box, gt_mask, neg_ratio)
    if check:
        ops.loss_result_to_host(result)       # raises IndexError / ValueError / AssertionError like the reference
    info = {"cls loss pos": result[N.LOSS_POS], "cls loss neg": result[N.LOSS_NEG], "loc loss": result[N.LOSS_LOC],
            "num_pos": result[N.LOSS_NUM_POS], "num_neg": result[N.LOSS_NUM_NEG]}
    return total, info
