"""Data-parallel training, one process per GPU (SURVEY.md §8e): every rank holds a full replica and its own shard of
the batch (independent CMAQ time steps); the gradient all-reduce is started per finished gradient section from inside
backward on a side stream so that it overlaps the remaining backward kernels (train.GradSync).
BatchNorm uses per-rank batch statistics (the DistributedDataParallel default) unless the module was converted with
``nn.SyncBatchNorm.convert_sync_batchnorm``: a converted BatchNorm takes its train-mode statistics over the rows of every rank
of its process group (DESIGN.md §5).  Inference needs no collective."""
from __future__ import annotations

import torch
import torch.distributed as dist
import torch.nn as nn

from .train import GradSync


class DataParallel(nn.Module):
    def __init__(self, module: nn.Module, process_group=None, broadcast: bool = True):
        super().__init__()
        if not (dist.is_available() and dist.is_initialized()):
            raise RuntimeError("DataParallel needs an initialised torch.distributed process group (one process per GPU)")
        self.module = module                            # state_dict keys carry the 'module.' prefix of the reference's nn.DataParallel checkpoints (evaluation_vit.py:107-109)
        self.process_group = process_group
        if broadcast:                                   # replicas start from rank 0's weights and buffers
            with torch.no_grad():
                for t in list(module.parameters()) + list(module.buffers()):
                    dist.broadcast(t, src=0, group=process_group)
            if hasattr(module, "invalidate_packed"):    # kernel-layout weight copies made before wrapping are stale now
                module.invalidate_packed()
        # A NCCL process group runs its collectives in issue order, and GradSync issues the all-reduces of the head, decoder and
        # ConvTranspose gradients before the MaxViT backward: a statistics exchange in that group would queue behind them and
        # stall the compute stream.  SyncBatchNorms without a group of their own get a dedicated one over the same ranks
        # (dist.new_group is collective: every rank constructs DataParallel).
        unset = [m for m in module.modules() if isinstance(m, nn.SyncBatchNorm) and m.process_group is None]
        self.stats_group = None
        if unset:
            ranks = None if process_group is None else dist.get_process_group_ranks(process_group)
            self.stats_group = dist.new_group(ranks=ranks)
            for m in unset:
                m.process_group = self.stats_group
        module._grad_sync = GradSync(process_group)

    def forward(self, *args, **kwargs):
        return self.module(*args, **kwargs)


def shard_batch(B: int, rank: int, world: int):
    """contiguous [lo, hi) slice of the B samples owned by `rank` (sizes differ by at most one)"""
    base, rem = divmod(B, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)
