"""One-process-per-GPU plumbing (torch.distributed; NCCL over NVLink on the GPU box, gloo in
CPU tests).  The reference has no distributed code at all (SURVEY 2.2); the only collective the
path needs is one sum all-reduce of the flat gradient buffer per step (SURVEY 8e)."""
from __future__ import annotations

import os

import torch
import torch.distributed as dist


def env_world():
    return int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))


def init(backend=None):
    """Initialise the default process group from the torchrun environment.  Returns
    (world_size, rank, local_rank)."""
    world, rank, local = env_world()
    if world > 1 and not dist.is_initialized():
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29500")
        if backend == "nccl":
            torch.cuda.set_device(local)
            dist.init_process_group(backend, device_id=torch.device("cuda", local))
        else:
            dist.init_process_group(backend)
    return world, rank, local


def allreduce_sum(t):
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t


def barrier():
    if dist.is_initialized():
        dist.barrier()


def max_over_ranks(value, device):
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    if dist.is_initialized():
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def gather_rows(vec, device):
    """Every rank's 1-D float vector (equal lengths) as a [world, len] float64 tensor on all ranks."""
    t = torch.as_tensor(vec, dtype=torch.float64, device=device).reshape(-1).contiguous()
    if not dist.is_initialized():
        return t[None, :].cpu()
    out = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(out, t)
    return torch.stack(out).cpu()


def gather_shards(t, total):
    """The contiguous shards of a ``total``-entry 1-D device tensor (rank r holds entries [r*per, (r+1)*per) of it,
    per = ceil(total / world), trailing shards short or empty) put back together in order on every rank: each shard
    is padded to ``per`` entries for one all_gather_into_tensor and the padding is cut away."""
    world = dist.get_world_size()
    per = (total + world - 1) // world
    buf = torch.zeros(per, dtype=t.dtype, device=t.device)
    buf[:t.numel()].copy_(t)
    out = torch.empty(per * world, dtype=t.dtype, device=t.device)
    dist.all_gather_into_tensor(out, buf)
    return out[:total]


def sum_over_ranks(value, device):
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    if dist.is_initialized():
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())
