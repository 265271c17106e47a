"""Multi-GPU plumbing for the path: scenes are sharded by batch across ranks (one process per GPU).

Inference needs no collective.  Training needs exactly one gradient all-reduce per step: the
reference does it implicitly through torch.nn.DataParallel (scripts/train.py:198-200); the
one-process-per-GPU equivalent is a single flat bucket (0.95 M detector parameters = 3.8 MB, one
latency-bound NCCL call over NVLink) -- `allreduce_gradients`.  BatchNorm statistics stay per rank by
default, which is what DataParallel does as well.  `nn.SyncBatchNorm.convert_sync_batchnorm(model)` makes every
BatchNorm take its statistics over all ranks: the fused BatchNorm + ReLU blocks of the SA, FP and vote-aggregation
MLPs then exchange one small fp64 buffer per block in the forward and one in the backward (pytorch_utils.py), the
other BatchNorm layers run torch's SyncBatchNorm.  Their dgamma / dbeta stay per rank and are summed by the same
gradient all-reduce.
"""
import torch
import torch.distributed as dist


def shard_range(total, rank, world):
    """[begin, end) of the `total` scenes owned by `rank` (contiguous, sizes differ by at most 1)."""
    base, rem = divmod(total, world)
    begin = rank * base + min(rank, rem)
    return begin, begin + base + (1 if rank < rem else 0)


def max_over_ranks(value, device=None):
    """Max of a python float over all ranks (used for device-time reporting)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return float(value)
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t[0])


def allreduce_gradients(module, average=True):
    """One flat all-reduce of every parameter gradient of `module` (sum, then / world)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return 0
    grads = [p.grad for p in module.parameters() if p.grad is not None]
    if not grads:
        return 0
    flat = torch.cat([g.reshape(-1) for g in grads])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM)
    if average:
        flat /= dist.get_world_size()
    views, off = [], 0
    for g in grads:
        n = g.numel()
        views.append(flat[off:off + n].view_as(g))
        off += n
    torch._foreach_copy_(grads, views)        # one multi-tensor kernel instead of ~100 small copies
    return flat.numel()
