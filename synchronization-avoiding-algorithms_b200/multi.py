"""One process per GPU (torchrun): attach a halo transport to this rank's StepPlan.

`peer`  — the default on one NVLink/NVSwitch node: receive areas are exchanged as CUDA IPC handles through
          `torch.distributed` object collectives and mapped into the neighbours; per step the pack kernel
          stores the shared-node partial forces straight into the neighbours' HBM and raises their arrival
          flags (no NCCL / host call inside the time loop; the loop is a replayed CUDA graph).
`nccl`  — grouped ncclSend/ncclRecv per neighbour per step on the plan's stream (multi-node capable).
`host`  — messages staged through host memory and carried by the caller's communicator (`saa_b200.comm`).
"""
from __future__ import annotations

from . import plan as _plan


def peer_access_everywhere(pl):
    """True when every rank can map the receive areas of all its neighbours (same node, P2P-capable GPUs).
    Collective; all ranks get the same answer."""
    import socket
    import torch
    import torch.distributed as dist
    me = dict(rank=pl.rank, host=socket.gethostname(), dev=pl.device, nb=[int(r) for r in pl.halo_layout()[0]])
    infos = [None] * dist.get_world_size()
    dist.all_gather_object(infos, me)
    by_rank = {i["rank"]: i for i in infos}
    ok = True
    for r in me["nb"]:
        o = by_rank[r]
        if o["host"] != me["host"]:
            ok = False
        elif o["dev"] != me["dev"] and not torch.cuda.can_device_access_peer(me["dev"], o["dev"]):
            ok = False
    flags = [None] * dist.get_world_size()
    dist.all_gather_object(flags, ok)
    return all(flags)


def attach_transport(pl, transport="peer"):
    import torch.distributed as dist
    if pl.size == 1:
        return "none"
    if transport == "peer" and not peer_access_everywhere(pl):
        transport = "nccl"                      # several nodes, or GPUs without peer access: NCCL carries the messages
    if transport == "peer":
        exports = [None] * dist.get_world_size()
        dist.all_gather_object(exports, pl.peer_export())
        pl.peer_attach(exports)
        dist.barrier()
    elif transport == "nccl":
        ids = [_plan.nccl_unique_id() if dist.get_rank() == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        pl.init_nccl(ids[0])
    elif transport != "host":
        raise ValueError(f"unknown transport {transport!r}")
    return transport


def gather_energy(pl, first=0, count=None):
    """Global energy balance of a partition stepped one process per rank: every rank's energy records
    (StepPlan.read_energy) all-gathered through `torch.distributed` and combined by plan.energy_balance.
    Collective; all ranks get the same array."""
    import torch.distributed as dist
    recs = [None] * dist.get_world_size()
    dist.all_gather_object(recs, (pl.rank, pl.read_energy(first, count)))
    return _plan.energy_balance([r for _, r in sorted(recs, key=lambda t: t[0])])
