"""Chain sharding and end-of-run gathers (replaces the reference's mpi4py usage:
comm.bcast(dobs), comm.bcast(x) at main_base.py:59-60 and comm.Gather(misfit) at :90).

One process per GPU; chains are independent, so nothing on the data path communicates.  The only
collectives are a broadcast of the observations at start and all-gathers of per-chain results at
the end (NCCL over NVLink on GPUs; the same code runs on `gloo` for the CPU tests)."""
import numpy as np
import torch
import torch.distributed as dist


def world():
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_chains(nchains, rank=None, world_size=None):
    """Contiguous block of chain ids owned by `rank` (chain i is the reference's MPI rank i and is
    seeded with seed + i, pyhmc/hmc.py:43).  Blocks differ by at most one chain."""
    if rank is None:
        rank, world_size = world()
    base, rem = divmod(int(nchains), int(world_size))
    lo = rank * base + min(rank, rem)
    hi = lo + base + (1 if rank < rem else 0)
    return np.arange(lo, hi, dtype=np.int64)


def shard_station_chains(nstations, nchains, rank=None, world_size=None):
    """(station [m], chain id [m]) of the (station, chain) pairs owned by `rank`: the S*K pairs are
    sharded as S*K chains by shard_chains; global index g is chain g % K of station g // K, so
    gather_chains(..., S*K) returns them station-major.  Chain ids repeat across stations: station s's
    chain k is seeded seed + k, as in a one-station run."""
    g = shard_chains(int(nstations) * int(nchains), rank, world_size)
    return g // int(nchains), g % int(nchains)


def _dev():
    if dist.is_initialized() and dist.get_backend() == "nccl":
        return torch.device("cuda", torch.cuda.current_device())
    return torch.device("cpu")


def bcast_array(a, src=0):
    """Broadcast a float64 array (dobs / true model) from `src`; shape must be known on all ranks."""
    rank, ws = world()
    t = torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).to(_dev())
    if ws > 1:
        dist.broadcast(t, src=src)
    return t.cpu().numpy()


def gather_chains(local, nchains):
    """All-gather a per-chain array whose first axis is this rank's chain block -> [nchains, ...] on
    every rank (ragged blocks are padded to the largest block)."""
    rank, ws = world()
    local = np.ascontiguousarray(local)
    if ws == 1:
        return local
    counts = [len(shard_chains(nchains, r, ws)) for r in range(ws)]
    mx = max(counts)
    pad = np.zeros((mx,) + local.shape[1:], dtype=local.dtype)
    pad[:local.shape[0]] = local
    t = torch.as_tensor(pad).to(_dev())
    outs = [torch.empty_like(t) for _ in range(ws)]
    dist.all_gather(outs, t)
    return np.concatenate([o.cpu().numpy()[:c] for o, c in zip(outs, counts)], axis=0)


def max_over_ranks(v):
    rank, ws = world()
    t = torch.tensor([float(v)], dtype=torch.float64, device=_dev())
    if ws > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())
