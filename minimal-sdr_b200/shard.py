"""Multi-GPU plumbing: the receive chain shards by channel and nothing else.

Every channel owns its FIR history, biquad state, mode and tables (no cross-channel term anywhere in
Minimal-SDR.ino:518-775 or filter_biquad.cpp:33-82), so rank r of W simply owns a contiguous channel range and runs its own
chain object; there is NO collective on the data path.  torch.distributed is only used to agree on timing (max over ranks)
and, if asked, to gather results or checksums.
"""
from dataclasses import dataclass
from typing import NamedTuple


@dataclass(frozen=True)
class Shard:
    rank: int
    world: int
    ch0: int      # first global channel owned by this rank
    n: int        # number of channels owned


def plan(total_channels, world, rank=None, granule=32):
    """Contiguous ranges, sizes differing by at most one `granule` (32 = the kernel's channel group), every channel owned
    exactly once.  Returns the list of all shards, or this rank's shard when `rank` is given."""
    if total_channels < 0 or world < 1:
        raise ValueError("bad arguments")
    groups = (total_channels + granule - 1) // granule
    base, extra = divmod(groups, world)
    shards, g0 = [], 0
    for r in range(world):
        g = base + (1 if r < extra else 0)
        ch0 = min(g0 * granule, total_channels)
        ch1 = min((g0 + g) * granule, total_channels)
        shards.append(Shard(r, world, ch0, ch1 - ch0))
        g0 += g
    return shards if rank is None else shards[rank]


class Piece(NamedTuple):
    old_rank: int
    first: int     # first channel of the piece inside old_rank's chain (and snapshot of its whole range)
    n: int
    new_rank: int
    dst_ch0: int   # where the piece goes inside new_rank's chain


def reshard(total_channels, old_world, new_world, granule=32):
    """The pieces that move a plan(total, old_world) layout to plan(total, new_world): every channel in exactly one piece, in global
    channel order.  Rank r of the new layout restores each piece with new_rank == r from old_rank's snapshot:
    chain.restore(snapshots[p.old_rank], ch0=p.dst_ch0, first=p.first, n=p.n)."""
    old, new = plan(total_channels, old_world, granule=granule), plan(total_channels, new_world, granule=granule)
    pieces = []
    for o in old:
        for s in new:
            lo, hi = max(o.ch0, s.ch0), min(o.ch0 + o.n, s.ch0 + s.n)
            if hi > lo:
                pieces.append(Piece(o.rank, lo - o.ch0, hi - lo, s.rank, lo - s.ch0))
    return pieces


def weak_scaling_shard(channels_per_rank, world, rank):
    """Benchmark layout: per-GPU work fixed, rank r owns global channels [r*C, (r+1)*C)."""
    return Shard(rank, world, rank * channels_per_rank, channels_per_rank)


def max_over_ranks(value, device=None):
    """Timing rule: a multi-GPU number is the max over ranks.  Works on any backend (gloo on CPU, nccl on GPU)."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return float(value)
    t = torch.tensor([float(value)], dtype=torch.float64, device=device or "cpu")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(value, device=None):
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return float(value)
    t = torch.tensor([float(value)], dtype=torch.float64, device=device or "cpu")
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


def gather_rows(local_rows, shard, total_channels, device=None):
    """Optional, untimed: assemble [total_channels, n] on every rank from per-rank [shard.n, n] int16 tensors."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return local_rows
    shards = plan(total_channels, shard.world)
    nmax = max(s.n for s in shards)
    pad = torch.zeros((nmax, local_rows.shape[1]), dtype=local_rows.dtype, device=local_rows.device)
    pad[:shard.n] = local_rows
    raw = pad.view(torch.uint8)  # gloo has no int16 collectives; bytes travel on every backend
    parts = [torch.empty_like(raw) for _ in shards]
    dist.all_gather(parts, raw)
    return torch.cat([p.view(local_rows.dtype)[:s.n] for p, s in zip(parts, shards)], dim=0)


def _parse_cpulist(text):
    cpus = set()
    for part in text.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        cpus.update(range(int(a), int(b or a) + 1))
    return cpus


def bind_to_gpu_numa(local_rank):
    """Pin this process (and so its pinned-buffer pages, which are allocated on first touch, and its copy-issuing thread) to the
    CPUs of the NUMA node its GPU hangs off.  Eight ranks that all sit on node 0 push every host<->device byte of the other
    socket's GPUs through the inter-socket link; this is the host-side half of "one process per GPU".  Returns what was done."""
    import os
    info = {"node": None, "cpus": None, "bound": False}
    try:
        import torch
        p = torch.cuda.get_device_properties(local_rank)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read().strip())
        info["pci"] = bdf
        info["node"] = node
        if node < 0:
            return info
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = _parse_cpulist(f.read())
        allowed = os.sched_getaffinity(0)
        use = (cpus & allowed) or None
        if use:
            os.sched_setaffinity(0, use)
            info.update(cpus=len(use), bound=True, allowed_before=len(allowed))
    except Exception as e:  # no sysfs / not permitted: run unbound and say so
        info["error"] = f"{type(e).__name__}: {e}"
    return info
