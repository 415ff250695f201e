"""Data-parallel host logic: the hot path shards by image (the reference's generator body is a
per-image loop, models/ssd_model.py:211-215, and NMS is per image and class), so the only exchange
step is the loss: the separable sums {sum positive CE, sum mined-negative CE, sum L1, num_pos,
num_neg} are all-reduced once (a 56-byte payload, latency-bound; NCCL over NVLink on GPUs, gloo in
the CPU tests).

Mining is per shard by default -- exactly what the reference does when ``split_batch`` slices a batch
and calls ``_ssd_loss`` per slice (models/ssd_model.py:235-256).  ``combine_loss`` offers the two
normalisations: ``pooled`` (sums and counts pooled over all shards) and ``mean_of_shards`` (the
reference's accumulate-and-average of per-slice losses, :251-256).

``global_mining_loss`` is the exact alternative (SURVEY.md section 8e): the threshold of :368-372 is the
k-th largest background CE of the WHOLE batch, found by a radix select whose three 2048-bin histograms are
summed over the shards between the stages of ``ops.StagedLoss`` -- five small all-reduces, after which the
mined mask of every shard equals the corresponding slice of the single-device mask, bit for bit.

torch is imported lazily: only callers that use torch.distributed need it."""
from __future__ import annotations

import numpy as np

from . import _native as N

SUM_SLICE = N.LOSS_ADDITIVE   # result-block words that are additive across shards: see include/ssdgeom.h


def shard_range(n_items: int, world: int, rank: int):
    """Contiguous, balanced slice [start, stop) of ``n_items`` for ``rank`` (first ranks get the remainder)."""
    if not (0 <= rank < world):
        raise ValueError("rank %d outside world of %d" % (rank, world))
    base, rem = divmod(int(n_items), int(world))
    start = rank * base + min(rank, rem)
    return start, start + base + (1 if rank < rem else 0)


def shard_csr(gt_offsets, world: int, rank: int):
    """Slice CSR ground truth by image: returns (image range, row range, rebased offsets)."""
    off = np.asarray(gt_offsets, dtype=np.int64)
    lo, hi = shard_range(off.size - 1, world, rank)
    return (lo, hi), (int(off[lo]), int(off[hi])), (off[lo:hi + 1] - off[lo]).astype(np.int32)


def loss_from_sums(sum_pos_ce, sum_neg_ce, sum_l1, num_pos, num_neg):
    """models/ssd_model.py:356-396 from the additive pieces: each term is normalised by its own count."""
    if num_pos <= 0:
        raise IndexError("no positive prior: hard-negative top-k is empty (models/ssd_model.py:369)")
    info = {"cls loss pos": sum_pos_ce / num_pos, "cls loss neg": sum_neg_ce / num_neg, "loc loss": sum_l1 / num_pos}
    return (info["loc loss"] + info["cls loss pos"]) + info["cls loss neg"], info


def _loss_of(s):
    return loss_from_sums(s["sum_pos_ce"], s["sum_neg_ce"], s["sum_l1"], s["num_pos"], s["num_neg"])


def block_sums(result_block):
    """The additive entries of a loss result block (host array) -> dict."""
    r = np.asarray(result_block, dtype=np.float64)
    return {"num_pos": r[N.LOSS_NUM_POS], "num_neg": r[N.LOSS_NUM_NEG], "sum_pos_ce": r[N.LOSS_SUM_POS_CE],
            "sum_neg_ce": r[N.LOSS_SUM_NEG_CE], "sum_l1": r[N.LOSS_SUM_L1]}


def combine_loss(shard_sums, mode="pooled"):
    """Combine per-shard additive sums (list of dicts as from ``block_sums``)."""
    if mode == "pooled":
        tot = {k: float(sum(s[k] for s in shard_sums)) for k in ("num_pos", "num_neg", "sum_pos_ce", "sum_neg_ce", "sum_l1")}
        return _loss_of(tot)
    if mode == "mean_of_shards":
        parts = [_loss_of(s) for s in shard_sums]
        n = len(parts)
        info = {k: sum(p[1][k] for p in parts) / n for k in parts[0][1]}
        return sum(p[0] for p in parts) / n, info
    raise ValueError("mode must be 'pooled' or 'mean_of_shards'")


def allreduce_sums(vec, group=None):
    """Sum a small float64 vector (torch tensor, CPU for gloo or CUDA for NCCL) over the ranks, in place."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(vec, op=dist.ReduceOp.SUM, group=group)
    return vec


def distributed_loss(result_block_tensor, group=None, mode="pooled"):
    """result_block_tensor: torch float64[16] view of one rank's loss result block (include/ssdgeom.h).
    Returns (total, info) identical on every rank."""
    import torch.distributed as dist
    r = result_block_tensor
    world = dist.get_world_size(group) if (dist.is_available() and dist.is_initialized()) else 1
    if mode == "pooled":
        v = np.zeros(N.LOSS_RESULT_LEN)
        v[SUM_SLICE] = allreduce_sums(r[SUM_SLICE].clone(), group).double().cpu().numpy()
        return _loss_of(block_sums(v))
    if mode == "mean_of_shards":
        vec = r[N.LOSS_TOTAL:N.LOSS_LOC + 1].clone()
        allreduce_sums(vec, group)
        v = (vec.double().cpu().numpy()) / world
        return float(v[0]), {"cls loss pos": float(v[1]), "cls loss neg": float(v[2]), "loc loss": float(v[3])}
    raise ValueError("mode must be 'pooled' or 'mean_of_shards'")


def global_mining_loss(staged, allreduce):
    """Drive a staged loss (``ops.StagedLoss`` or anything with run / exchange / finish) through the
    stages of the cross-shard mining protocol.  ``allreduce(buf)`` sums one exchange buffer over the shards
    in place; every shard must call this function collectively.  Returns (total, info) of the whole batch."""
    for stage in range(getattr(staged, "n_stages", 4)):     # 5 with gradients: they run after the last exchange
        staged.run(stage)
        for buf in staged.exchange(stage):
            allreduce(buf)
    return staged.finish()


def torch_allreduce(group=None, device="cuda"):
    """allreduce callable for ``global_mining_loss``: zero-copy torch view of a device buffer (anything with
    __cuda_array_interface__) or of a NumPy array (gloo), summed over ``group``."""
    import torch
    import torch.distributed as dist

    def run(buf):
        if not (dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1):
            return buf
        if isinstance(buf, np.ndarray):
            t = torch.from_numpy(buf)
        else:
            t = torch.as_tensor(buf, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
        return buf

    return run
