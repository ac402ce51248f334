"""Geometric multigrid V-cycle preconditioner for the static solve on the structured cantilever (DESIGN.md §7d).

The Kuhn triangulation of mesh.structured_beam(m) refines that of structured_beam(m / 2): every coarse P1 function is
a P1 function of the fine mesh, so the prolongation is the nodal interpolation (a fine node at grid index i takes the
average of the coarse nodes at floor(i / 2) and ceil(i / 2), per axis) and the stiffness the device set-up assembles on
the coarse mesh is the Galerkin operator P^T K P.  No triple product is formed: every coarse level is a plan built by
device_setup.build_structured_rank, and the kernels (csrc/saa_multigrid.cuh) only know node CSR tables.

    mg = StructuredMultigrid(plan, m, info["local_nodes"])
    res = plan.solve_static(rtol=1e-8, precond=mg)
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import device_setup, mesh
from .plan import SaaError, _check, _dev_vector, lib

COARSEST_MAX_DOF = 16384      # the coarsest level's dense inverse takes 8 n^2 bytes: 2 GB at this size


def structured_dof(m, length=25):
    nx, ny, nz = mesh.structured_beam_dims(m, length)
    return 3 * (nx + 1) * (ny + 1) * (nz + 1)


def _halvings(m):
    ms = [int(m)]
    while ms[-1] % 2 == 0 and ms[-1] // 2 >= 2:      # a beam one element thick locks in bending: coarsest m >= 2
        ms.append(ms[-1] // 2)
    return ms


def _supported(m, length, coarsest_max_dof):
    ms = _halvings(m)
    return len(ms) >= 2 and structured_dof(ms[-1], length) <= coarsest_max_dof


def structured_levels(m, length=25, coarsest_max_dof=COARSEST_MAX_DOF):
    """The mesh parameters m, m/2, ... of the hierarchy: halved while even and the half is >= 2.  Raises ValueError when
    that gives fewer than two levels or a coarsest level above coarsest_max_dof DOF, naming the nearest supported m."""
    m = int(m)
    ms = _halvings(m)
    if _supported(m, length, coarsest_max_dof):
        return ms
    lo = next((k for k in range(m - 1, 1, -1) if _supported(k, length, coarsest_max_dof)), None)
    hi = next(k for k in range(m + 1, 4 * m + 8) if _supported(k, length, coarsest_max_dof))
    why = (f"it cannot be halved (m/2 would be {m / 2:g})" if len(ms) < 2 else
           f"halving stops at the odd m = {ms[-1]} with {structured_dof(ms[-1], length)} DOF, above coarsest_max_dof = "
           f"{coarsest_max_dof}")
    near = f"{lo} and {hi}" if lo is not None else f"{hi}"
    raise ValueError(f"StructuredMultigrid: m = {m} is not supported: {why}; the nearest supported values are {near}")


def prolongation_table(m_f, nodes_f, nodes_c, length=25):
    """Node CSR (ptr int64, col int32, weight float64; device tensors) of the prolongation from structured_beam(m_f / 2)
    to structured_beam(m_f): row e is the fine local node e (global id nodes_f[e]), columns the coarse local nodes
    (positions in nodes_c) of its parents, weight 1/2 each, or one parent with weight 1 where both coincide."""
    import torch
    nx, ny, nz = mesh.structured_beam_dims(m_f, length)
    cx, cy, cz = mesh.structured_beam_dims(m_f // 2, length)
    g = nodes_f.long()
    iz, iy, ix = g % (nz + 1), (g // (nz + 1)) % (ny + 1), g // ((nz + 1) * (ny + 1))
    cid = lambda a, b, c: (a * (cy + 1) + b) * (cz + 1) + c
    a, b = cid(ix // 2, iy // 2, iz // 2), cid((ix + 1) // 2, (iy + 1) // 2, (iz + 1) // 2)
    inv = torch.full(((cx + 1) * (cy + 1) * (cz + 1),), -1, dtype=torch.int64, device=g.device)
    inv[nodes_c.long()] = torch.arange(nodes_c.numel(), device=g.device)
    la, lb = inv[a], inv[b]
    if bool((la < 0).any()) or bool((lb < 0).any()):
        raise SaaError("StructuredMultigrid: a parent node is missing from the coarse level's local node list")
    same = a == b
    ptr = torch.zeros(g.numel() + 1, dtype=torch.int64, device=g.device)
    ptr[1:] = torch.cumsum(2 - same.long(), 0)
    keep = torch.stack([torch.ones_like(same), ~same], 1).reshape(-1)
    col = torch.stack([la, lb], 1).reshape(-1)[keep].to(torch.int32).contiguous()
    w = torch.where(same, 1.0, 0.5).double()
    wt = torch.stack([w, w], 1).reshape(-1)[keep].contiguous()
    return ptr, col, wt


def _coarse_inverse(info, device):
    """(S K S + I - S)^-1 of a level kept with keep_csr, dense, in its local DOF order (one-off Cholesky by torch)"""
    import torch
    K = info["K"]
    dev = torch.device("cuda", device)
    ip = torch.empty(K.n_rows + 1, dtype=torch.int64, device=dev)
    ix = torch.empty(K.nnz, dtype=torch.int32, device=dev)
    dv = torch.empty(K.nnz, dtype=torch.float64, device=dev)
    torch.cuda.synchronize(dev)
    for dst, src in ((ip, K.indptr), (ix, K.indices), (dv, K.data)):
        _check(lib().saa_device_copy(dst.data_ptr(), src, dst.numel() * dst.element_size()), "saa_device_copy")
    K.free()
    A = torch.zeros((K.n_rows, K.n_rows), dtype=torch.float64, device=dev)
    A[torch.repeat_interleave(torch.arange(K.n_rows, device=dev), ip.diff()), ix.long()] = dv
    clamped = torch.as_tensor(np.asarray(info["dirichlet"], dtype=np.int64), device=dev)
    keep = torch.ones(K.n_rows, dtype=torch.float64, device=dev)
    keep[clamped] = 0.0
    A = A * keep[:, None] * keep[None, :]
    A[clamped, clamped] = 1.0
    L, err = torch.linalg.cholesky_ex(A)
    if int(err) != 0:
        raise SaaError("StructuredMultigrid: the coarsest level's matrix is not positive definite")
    inv = torch.cholesky_inverse(L)
    return (0.5 * (inv + inv.T)).contiguous()


class StructuredMultigrid:
    """V-cycle hierarchy over `plan` (a size-1 plan of mesh.structured_beam(m, length)) and coarse plans of m/2, m/4, ...
    built by the device set-up.  local_nodes: the global structured node id of every local node of `plan`
    (info["local_nodes"] of device_setup, or arange(n) for a plan of structured_beam(m) built on the host).
    degree: Chebyshev smoothing steps before and after the coarse correction; power_iters: power steps of the
    lambda_max estimate.  Use as a context manager or call close(); StepPlan.solve_static(precond=...) runs it."""

    def __init__(self, plan, m, local_nodes, length=25, degree=2, power_iters=20, coarsest_max_dof=COARSEST_MAX_DOF):
        import torch
        self.h = None
        self._plans = []
        if plan.size != 1:
            raise SaaError(f"StructuredMultigrid: the plan is rank {plan.rank} of a partition of size {plan.size}; the multigrid "
                           "preconditioner needs a single-partition plan")
        ms = structured_levels(m, length, coarsest_max_dof)
        if plan.n_dof != structured_dof(m, length):
            raise SaaError(f"StructuredMultigrid: the plan has {plan.n_dof} DOF, structured_beam({m}) has {structured_dof(m, length)}")
        dev = torch.device("cuda", plan.device)
        nodes = torch.as_tensor(np.asarray(local_nodes.cpu() if isinstance(local_nodes, torch.Tensor) else local_nodes),
                                dtype=torch.int64).to(dev)
        if nodes.numel() != plan.n_dof // 3 or not torch.equal(torch.sort(nodes).values, torch.arange(nodes.numel(), device=dev)):
            raise SaaError("StructuredMultigrid: local_nodes must list every global node of the beam once")
        self.plan, self.m, self.length = plan, int(m), int(length)
        node_lists, infos = [nodes], []
        for k, ml in enumerate(ms[1:]):
            pl, info = device_setup.build_structured_rank(ml, 0, 1, device_index=plan.device, length=length,
                                                          keep_csr=(k == len(ms) - 2))
            self._plans.append(pl)
            node_lists.append(info["local_nodes"])
            infos.append(info)
        tables = [prolongation_table(ms[l], node_lists[l], node_lists[l + 1], length) for l in range(len(ms) - 1)]
        cinv = _coarse_inverse(infos[-1], plan.device)
        levels = [plan] + self._plans
        arr = lambda xs: (ctypes.c_void_p * len(xs))(*xs)
        torch.cuda.synchronize(dev)
        h = ctypes.c_void_p()
        _check(lib().saa_mg_create(ctypes.byref(h), arr([p.h for p in levels]), len(levels), arr([t[0].data_ptr() for t in tables]),
                                   arr([t[1].data_ptr() for t in tables]), arr([t[2].data_ptr() for t in tables]), cinv.data_ptr(),
                                   int(degree), int(power_iters), int(coarsest_max_dof)), "saa_mg_create")
        self.h = h
        self.levels = [(ml, p.n_dof) for ml, p in zip(ms, levels)]
        self.plans, self.local_nodes = levels, node_lists
        lam = np.zeros(len(levels))
        own = ctypes.c_int64(0)
        _check(lib().saa_mg_info(self.h, lam.ctypes.data_as(ctypes.c_void_p), ctypes.byref(own)), "saa_mg_info")
        self.lambda_max = [float(v) for v in lam]
        # the hierarchy's own vectors, tables and coarsest inverse, plus the coarse plans' matrices and vectors
        self.bytes = int(own.value) + sum(p.streamed_matrix_bytes + p.vector_bytes for p in self._plans)

    def handle(self):
        if not self.h:
            raise SaaError("StructuredMultigrid: used after close()")
        return self.h

    def vcycle(self, r):
        """z = V r (float64 CUDA tensors of the fine plan's n_dof, local DOF order; r is taken as 0 on clamped DOFs)"""
        import torch
        h, n = self.handle(), self.levels[0][1]
        r = _dev_vector(r, n, self.plan.device, "vcycle: r")
        z = torch.empty_like(r)
        torch.cuda.current_stream(r.device).synchronize()
        _check(lib().saa_mg_vcycle_dev(h, r.data_ptr(), z.data_ptr()), "saa_mg_vcycle_dev")
        return z

    def _transfer(self, level, v, prolong):
        import torch
        h = self.handle()
        what = "saa_mg_prolong_dev" if prolong else "saa_mg_restrict_dev"
        if not 0 <= int(level) < len(self.levels) - 1:
            raise SaaError(f"{what}: level {level} is not in [0, {len(self.levels) - 1})")
        n_f, n_c = self.levels[level][1], self.levels[level + 1][1]
        v = _dev_vector(v, n_c if prolong else n_f, self.plan.device, f"{what}: input")
        out = torch.empty(n_f if prolong else n_c, dtype=torch.float64, device=v.device)
        torch.cuda.current_stream(v.device).synchronize()
        fn = lib().saa_mg_prolong_dev if prolong else lib().saa_mg_restrict_dev
        _check(fn(h, int(level), v.data_ptr(), out.data_ptr()), what)
        return out

    def prolong(self, level, xc):
        """S_f P x_c from level + 1 to `level` (0: the fine plan), local DOF order"""
        return self._transfer(level, xc, True)

    def restrict(self, level, rf):
        """S_c P^T r_f from `level` to level + 1, local DOF order"""
        return self._transfer(level, rf, False)

    def close(self):
        if getattr(self, "h", None):
            lib().saa_mg_destroy(self.h)
            self.h = None
        for p in getattr(self, "_plans", []):
            p.close()
        self._plans, self.plans = [], []

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
