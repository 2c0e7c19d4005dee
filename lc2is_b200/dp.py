"""Data-parallel glue for the head (north_star stage 4; absent from the reference, which is single
process / single device: engine.py:17,29-31).

One process per GPU (torchrun), batch-dimension sharding, replicas of the head parameters.
Exchange steps - the only cross-image reductions of the path are sums (SURVEY 8e):
  * eval : ONE int64 all-reduce of the [C,C] confusion matrix (integer => order independent =>
           bit-identical to the single-GPU matrix), optionally an all-gather of per-image stats.
  * train: all-reduce of the valid-pixel count BEFORE the loss kernel (the reference's CE is a mean
           over the valid pixels of the whole batch, so every rank scales its gradients by
           1/N_valid_global, not 1/world), then ONE fp32 all-reduce of a flat gradient bucket
           (d prototypes + TextToPatch grads, 2.93 MB) and a scalar loss-sum all-reduce for logging.
dV stays local (it flows into the local upstream decoder).
Everything is enqueued on the current stream through torch.distributed (NCCL over NVLink on the
GPU box, gloo in the CPU tests); no host synchronisation.
"""
from __future__ import annotations

import os
from typing import Iterable, List, Optional, Sequence, Tuple

import torch
import torch.distributed as dist
from torch import Tensor


def init_distributed(backend: Optional[str] = None) -> Tuple[int, int, int]:
    """Initialise the default process group from the torchrun environment.  Returns
    (rank, world_size, local_rank).  A plain single-process run returns (0, 1, 0) without a group."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1:
        return 0, 1, local_rank
    if not dist.is_initialized():
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(local_rank)
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        kwargs = {}
        if backend == "nccl":
            kwargs["device_id"] = torch.device("cuda", local_rank)
        dist.init_process_group(backend=backend, rank=rank, world_size=world, **kwargs)
    return rank, world, local_rank


def is_dist() -> bool:
    return dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1


def shard_range(n: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous image range of `rank` (2000 images / 8 ranks = 250 each; remainders go to the
    first ranks)."""
    base, rem = divmod(n, world)
    start = rank * base + min(rank, rem)
    return start, start + base + (1 if rank < rem else 0)


def allreduce_sum_(t: Tensor) -> Tensor:
    if is_dist():
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t


class _Done:
    def wait(self):
        return None


def allreduce_sum_async(t: Tensor):
    """SUM all-reduce issued asynchronously (NCCL: on its own stream after the current one; `wait()` makes
    the current stream wait, never the host).  Returns an object with .wait()."""
    if is_dist():
        return dist.all_reduce(t, op=dist.ReduceOp.SUM, async_op=True)
    return _Done()


def allreduce_confmat_(confmat: Tensor) -> Tensor:
    """int64 [C,C] SUM all-reduce (180 kB at C=150, 5.7 MB at C=847)."""
    assert confmat.dtype == torch.int64
    return allreduce_sum_(confmat)


def gather_per_image(per_image: Tensor, counts: Sequence[int]) -> Tensor:
    """All-gather ragged per-image stats [n_local,3,C] -> [N,3,C] in rank order (any tensor ragged in dim 0;
    `counts` are every rank's first dimensions)."""
    if not is_dist():
        return per_image
    world = dist.get_world_size()
    mx = max(counts)
    pad = torch.zeros((mx,) + tuple(per_image.shape[1:]), dtype=per_image.dtype, device=per_image.device)
    pad[: per_image.shape[0]] = per_image
    out = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(out, pad)
    return torch.cat([o[:c] for o, c in zip(out, counts)], dim=0)


def gather_ragged(t: Optional[Tensor], device) -> Optional[Tensor]:
    """All-gather tensors that differ in their first dimension -> their concatenation in rank order, on every rank.
    A rank may hold nothing (`t=None`, e.g. an empty evaluation shard): it still enters every collective, learning the
    trailing shape and dtype from the others.  Returns None when no rank holds a tensor.  `device` is where the
    collective runs (CUDA for NCCL)."""
    world = dist.get_world_size()
    metas = [None] * world
    dist.all_gather_object(metas, None if t is None else (t.shape[0], tuple(t.shape[1:]), t.dtype))
    known = [m for m in metas if m is not None]
    if not known:
        return None
    _, tail, dtype = known[0]
    local = t.to(device) if t is not None else torch.empty((0,) + tail, dtype=dtype, device=device)
    return gather_per_image(local, [m[0] if m is not None else 0 for m in metas])


class GradBucket:
    """One flat buffer (fp32 unless `dtype` says otherwise) holding views of every head gradient, all-reduced with a
    single call."""

    def __init__(self, shapes: Iterable[Sequence[int]], device, flat: Optional[Tensor] = None,
                 dtype: torch.dtype = torch.float32) -> None:
        self.shapes = [tuple(s) for s in shapes]
        self.sizes = [int(torch.Size(s).numel()) for s in self.shapes]
        # `flat`: optional caller-owned storage of exactly the bucket's size (e.g. a slice of a larger
        # buffer that is zeroed in one go)
        if flat is not None:
            assert flat.dtype == dtype and flat.numel() == sum(self.sizes) and flat.is_contiguous()
        self.flat = flat if flat is not None else torch.zeros(sum(self.sizes), dtype=dtype, device=device)
        self.views: List[Tensor] = []
        o = 0
        for s, n in zip(self.shapes, self.sizes):
            self.views.append(self.flat[o:o + n].view(s))
            o += n

    def zero_(self) -> None:
        self.flat.zero_()

    def allreduce_(self) -> Tensor:
        return allreduce_sum_(self.flat)


def global_valid_count_(n_valid_local: Tensor) -> Tensor:
    """All-reduce the per-rank valid-pixel count (1 x int64) so each rank can scale by 1/N_global."""
    return allreduce_sum_(n_valid_local)
