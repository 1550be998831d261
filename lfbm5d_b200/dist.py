"""Host-side multi-GPU plumbing (one process per GPU, torch.distributed): SAI sharding for the per-SAI BM3D path
(config 4: SAIs are independent, no data-path collective), the NCCL team that runs one LFBM5D light field on all ranks,
and the max-over-ranks timing reduction the bench reports. Works with the gloo backend on CPU (tests) and nccl on GPUs."""
import numpy as np


def shard_sais(asize, world, rank):
    """Contiguous, balanced [lo, hi) slice of the SAI index range for this rank."""
    base, rem = divmod(asize, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def shard_mask(mask, world, rank):
    """SAI mask restricted to this rank's shard (other SAIs are skipped by the C ABI like empty ones)."""
    m = np.zeros_like(np.asarray(mask, np.uint32))
    lo, hi = shard_sais(len(m), world, rank)
    m[lo:hi] = np.asarray(mask, np.uint32)[lo:hi]
    return m


def gather_shards(local, asize, dist, device="cpu"):
    """All ranks contribute their [hi-lo, ...] block; returns the full [asize, ...] array on every rank."""
    import torch
    world, rank = dist.get_world_size(), dist.get_rank()
    sizes = [shard_sais(asize, world, r) for r in range(world)]
    maxn = max(hi - lo for lo, hi in sizes)
    t = torch.zeros((maxn,) + tuple(local.shape[1:]), dtype=torch.float32, device=device)
    t[: local.shape[0]] = torch.as_tensor(local, dtype=torch.float32, device=device)
    out = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(out, t)
    return torch.cat([o[: hi - lo] for o, (lo, hi) in zip(out, sizes)], 0)


def max_over_ranks(value, dist, device="cpu"):
    import torch
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


# ---- one light field on several GPUs: parallelism inside a window (csrc/team.cuh) -------------------------------------------
def make_team(eng, dist, device):
    """NCCL team over the ranks of the default process group: rank 0 draws the NCCL unique id, torch.distributed ships it."""
    import torch
    from . import Team
    rank, world = dist.get_rank(), dist.get_world_size()
    uid = torch.zeros(128, dtype=torch.uint8, device=device)
    if rank == 0:
        uid = torch.frombuffer(bytearray(Team.unique_id()), dtype=torch.uint8).to(device)
    dist.broadcast(uid, src=0)
    return Team.nccl(eng, rank, world, bytes(uid.cpu().numpy().tobytes()))
