"""Averaged nodal stresses from the per-rank partial sums of StepPlan.nodal_stress_partial (DESIGN.md §7b).

A node's stress is the volume-weighted mean of the constant stresses of its elements,
    sigma_node = sum_e V_e sigma_e / sum_e V_e,
over ALL elements around it, so at a shared node the partial sums of its holders are added first, in ascending rank
order (device_setup.holders_sum, the association of syn_cpus).  Works on torch tensors on the CPU or a GPU.
"""
from __future__ import annotations

from . import device_setup
from .plan import SaaError


def von_mises(sigma):
    """von Mises stress of (..., 6) Voigt stresses (xx yy zz yz xz xy), the kernel's formula and association."""
    s = sigma
    a, b, c = s[..., 0] - s[..., 1], s[..., 1] - s[..., 2], s[..., 2] - s[..., 0]
    return (0.5 * (a * a + b * b + c * c) + 3.0 * (s[..., 3] * s[..., 3] + s[..., 4] * s[..., 4] + s[..., 5] * s[..., 5])).sqrt()


def nodal_stress(partial, halo=None, rank=0, recv=None, size=1):
    """(n_nodes, 7): averaged sigma (6) and its von Mises stress, from this rank's partial sums (n_nodes, 7).

    With a `halo` (the rank's maps.halo_plan) the shared rows are replaced by their sums over the holders; `recv` is
    {neighbour: its device_setup.holders_send message of partial[halo['shared_pos']] for this rank}.  Without one the
    rank is taken to be the whole partition: `size` > 1 and no halo is refused.  A node whose summed weight is not
    positive (no local element touches it) is refused too, instead of being returned as NaN."""
    import torch
    if partial.ndim != 2 or partial.shape[1] != 7:
        raise SaaError(f"nodal_stress: partial must be (n_nodes, 7), got {tuple(partial.shape)}")
    out = partial.clone()
    if halo is None and size > 1:
        raise SaaError("nodal_stress: a partition of size > 1 needs this rank's halo (maps.halo_plan) and the neighbours' messages")
    if halo is not None:
        missing = [nb for nb in halo["neighbours"] if recv is None or nb not in recv]
        if missing:
            raise SaaError(f"nodal_stress: no message from neighbour(s) {missing}")
        if len(halo["shared_pos"]):
            sp = torch.as_tensor(halo["shared_pos"], device=partial.device)
            out[sp] = device_setup.holders_sum(halo, rank, partial[sp], recv)
    bad = torch.nonzero(~(out[:, 6] > 0)).reshape(-1)
    if bad.numel():
        raise SaaError(f"nodal_stress: {bad.numel()} node(s) have no element weight (no element touches them), "
                       f"first at position {int(bad[0])}")
    sig = out[:, :6] / out[:, 6:7]
    return torch.cat([sig, von_mises(sig)[:, None]], dim=1)


def shared_message(partial, halo):
    """{neighbour: rows of `partial` at the nodes shared with it} — what this rank sends for nodal_stress."""
    import torch
    sp = torch.as_tensor(halo["shared_pos"], device=partial.device)
    return device_setup.holders_send(halo, partial[sp])


def nodal_stress_in_process(plans, halos=None):
    """Averaged nodal stresses of P plans of ONE process (a PlanGroup's plans, in rank order): list of (n_nodes_r, 7)
    tensors.  halos: the ranks' maps.halo_plan (None for a single partition)."""
    parts = [pl.nodal_stress_partial() for pl in plans]
    size = len(plans)
    if size == 1:
        return [nodal_stress(parts[0])]
    if halos is None or len(halos) != size:
        raise SaaError("nodal_stress_in_process: a partition of size > 1 needs the halo of every rank")
    sends = [shared_message(parts[r], halos[r]) for r in range(size)]
    return [nodal_stress(parts[r], halos[r], r, {nb: sends[nb][r] for nb in halos[r]["neighbours"]}) for r in range(size)]
