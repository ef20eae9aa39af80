"""Data-parallel training plumbing (BASELINE configs[4], SURVEY §8e): one process per GPU, per-GPU BatchNorm statistics (like the
reference's nn.DataParallel replicas, main.py:117), ONE bucketed gradient all-reduce per step instead of DataParallel's per-step parameter
broadcast + reduce_add to GPU 0, and an all-reduce(max) of the per-example "close" table so that every rank's AdjustableDataSampler
(dl4vc/dataset.py:697-746) draws the same epoch list, which is then strided by rank.

The native backward produces the FC-trunk gradients first (97 % of the bytes: conv2hidden.1 is 302 MB), then, with pool_combine_dimension > 0,
the post-pool Linear's (105 M parameters at D = 2048, more than PROD's whole FC trunk): `allreduce_gradients` sends that bucket off on a side
stream as soon as the backward call has been enqueued, the small conv-stack bucket afterwards; torch.distributed (NCCL over NVLink on the GPU
box, gloo in the CPU tests) is plumbing only."""
from __future__ import annotations

import torch
import torch.distributed as dist


def shard_epoch_indices(indices, rank: int, world: int):
    """Every rank holds the same sampler list (same seed, same close table after sync_close_table): rank r trains on indices[r::world],
    truncated so that all ranks run the same number of steps."""
    n = len(indices) // world * world
    return indices[:n][rank::world]


def sync_close_table(table: torch.Tensor, group=None):
    """all-reduce(max) of the uint8 close / blacklist tables (dataset.py:442,445), once per epoch."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        t = table if table.dtype != torch.bool else table.to(torch.uint8)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
        if t is not table:
            table.copy_(t.bool())
    return table


class GradientAllReducer:
    """Averages .grad over the ranks in two flat buckets: [FC trunk + heads + post-pool Linear] and [everything else]."""

    def __init__(self, model, group=None):
        self.group = group
        m = model.module if hasattr(model, "module") else model
        big, small = [], []
        for name, p in m.named_parameters():
            if not p.requires_grad:
                continue
            (big if name.startswith(("conv2hidden", "fcHidden2", "post_pool_conv1D")) else small).append(p)
        self.buckets = [big, small]
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.side = torch.cuda.Stream() if torch.cuda.is_available() and any(p.is_cuda for p in big + small) else None

    def __call__(self):
        if self.world == 1:
            return
        handles = []
        for params in self.buckets:
            grads = [p.grad for p in params if p.grad is not None]
            if not grads:
                continue
            flat = torch.cat([g.reshape(-1) for g in grads])
            if self.side is not None:
                self.side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(self.side):
                    h = dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group, async_op=True)
            else:
                h = dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group, async_op=True)
            handles.append((h, flat, grads))
        for h, flat, grads in handles:
            h.wait()
            if self.side is not None:
                torch.cuda.current_stream().wait_stream(self.side)
            flat.div_(self.world)
            off = 0
            for g in grads:
                n = g.numel()
                g.copy_(flat[off:off + n].view_as(g))
                off += n
