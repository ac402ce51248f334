"""ctypes binding of the C ABI in include/saa_fem.h (csrc/libsaa_fem.so) — the device plan of one partition.

`StepPlan` owns what one MPI rank of the reference hands to
`parallel_explicit_solver_dis_pre` every step (/root/reference/Tools/Dynamic_solver.py:9-10):
LocalK, F_rankwise, l_M, Local_Dirichlet, dt, alpha — uploaded once — plus the state
(d0, dn, tn) of `Time_integration_displacement` (Tools/commons.py:47-52), resident in HBM.

There is no CPU fallback: if the shared library is missing, or no CUDA device is visible, every
constructor / compute call raises.
"""
from __future__ import annotations

import ctypes
import os
import sys
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "csrc")
_SO = os.path.join(_CSRC, "libsaa_fem.so")
_lib = None

MODE_LOCAL, MODE_SYNC, MODE_PREDICT = 0, 1, 2
LAUNCH_AUTO, LAUNCH_PER_STEP, LAUNCH_GRAPH, LAUNCH_PERSISTENT = 0, 1, 2, 3
HOST_DN_IS_PREVIOUS_D0 = 1
OPT_PEER_FUSED, OPT_PREFER_NCCL, OPT_MATFREE = 1, 2, 3

# every symbol include/saa_fem.h declares: name -> (restype, argtypes)
_vp, _i64, _i32, _f64, _int = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_double, ctypes.c_int
_PP = ctypes.POINTER(ctypes.c_void_p)
ABI = {
    "saa_version": (_int, []),
    "saa_last_error": (ctypes.c_char_p, []),
    "saa_device_count": (_int, []),
    "saa_plan_create": (_int, [_PP, _int, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _f64, _f64, _f64, _f64, _f64]),
    "saa_plan_create_dev": (_int, [_PP, _int, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _f64, _f64, _f64, _f64, _f64]),
    "saa_assemble_stiffness_dev": (_int, [_int, _i64, _i64, _vp, _vp, _f64, _f64, _PP, _PP, _PP, _vp]),
    "saa_assemble_mass_load_dev": (_int, [_int, _i64, _i64, _vp, _vp, _f64, _f64, _vp, _vp]),
    "saa_device_free": (_int, [_vp]),
    "saa_device_copy": (_int, [_vp, _vp, _i64]),
    "saa_plan_set_halo": (_int, [_vp, _int, _int, _i64, _vp, _int, _vp, _vp, _vp, _vp, _vp, _vp]),
    "saa_plan_set_node_order": (_int, [_vp, _vp, _i64]),
    "saa_plan_finalize": (_int, [_vp]),
    "saa_plan_destroy": (_int, [_vp]),
    "saa_plan_n_dof": (_i64, [_vp]),
    "saa_plan_nnz": (_i64, [_vp]),
    "saa_plan_padded_entries": (_i64, [_vp]),
    "saa_plan_value_planes": (_i64, [_vp]),
    "saa_plan_coded_planes": (_i64, [_vp]),
    "saa_plan_kernel_launches": (_i64, [_vp]),
    "saa_plan_matrix_bytes": (_i64, [_vp]),
    "saa_plan_streamed_matrix_bytes": (_i64, [_vp]),
    "saa_plan_vector_bytes": (_i64, [_vp]),
    "saa_plan_set_state": (_int, [_vp, _vp, _vp, _f64]),
    "saa_plan_get_state": (_int, [_vp, _vp, _vp, _vp]),
    "saa_plan_set_state_dev": (_int, [_vp, _vp, _vp, _f64]),
    "saa_plan_get_state_dev": (_int, [_vp, _vp, _vp, _vp]),
    "saa_plan_step": (_int, [_vp, _i64, _int, _int]),
    "saa_plan_synchronize": (_int, [_vp]),
    "saa_plan_set_option": (_int, [_vp, _int, _int]),
    "saa_plan_set_matfree_dev": (_int, [_vp, _i64, _vp, _vp, _f64, _f64]),
    "saa_plan_matfree_bytes": (_i64, [_vp]),
    "saa_plan_element_stress_dev": (_int, [_vp, _vp]),
    "saa_plan_nodal_stress_dev": (_int, [_vp, _vp, _vp]),
    "saa_plan_apply_stiffness_dev": (_int, [_vp, _vp, _vp]),
    "saa_group_apply_stiffness_dev": (_int, [_vp, _vp, _vp]),
    "saa_plan_solve_static_dev": (_int, [_vp, _vp, _vp, _f64, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "saa_group_solve_static_dev": (_int, [_vp, _vp, _vp, _f64, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "saa_mg_create": (_int, [_PP, _vp, _int, _vp, _vp, _vp, _vp, _int, _int, _i64]),
    "saa_mg_destroy": (_int, [_vp]),
    "saa_mg_info": (_int, [_vp, _vp, _vp]),
    "saa_plan_solve_static_mg_dev": (_int, [_vp, _vp, _vp, _f64, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "saa_mg_vcycle_dev": (_int, [_vp, _vp, _vp]),
    "saa_mg_prolong_dev": (_int, [_vp, _int, _vp, _vp]),
    "saa_mg_restrict_dev": (_int, [_vp, _int, _vp, _vp]),
    "saa_plan_stream": (_vp, [_vp]),
    "saa_step_host": (_int, [_vp, _vp, _vp, _f64, _int, _vp]),
    "saa_step_host_ex": (_int, [_vp, _vp, _vp, _f64, _int, _vp, _int]),
    "saa_plan_host_pipe_info": (_int, [_vp, _int, _vp, _vp, _vp, _int]),
    "saa_host_alloc": (_vp, [_i64]),
    "saa_host_free": (_int, [_vp]),
    "saa_plan_set_history": (_int, [_vp, _vp, _i64, _i64, _i64]),
    "saa_plan_history_count": (_i64, [_vp]),
    "saa_plan_read_history": (_int, [_vp, _i64, _i64, _vp]),
    "saa_plan_read_history_dev": (_int, [_vp, _i64, _i64, _vp]),
    "saa_plan_set_prediction": (_int, [_vp, _vp, _i64, _vp, _i64]),
    "saa_plan_set_energy": (_int, [_vp, _i64, _i64]),
    "saa_plan_energy_count": (_i64, [_vp]),
    "saa_plan_read_energy": (_int, [_vp, _i64, _i64, _vp]),
    "saa_plan_halo_layout": (_int, [_vp, _vp, _vp, _vp, _int]),
    "saa_plan_step_begin_host": (_int, [_vp, _vp]),
    "saa_plan_step_end_host": (_int, [_vp, _vp]),
    "saa_plan_forces_begin_host": (_int, [_vp, _vp, _vp]),
    "saa_plan_forces_end_host": (_int, [_vp, _vp, _vp]),
    "saa_group_create": (_int, [_PP, _PP, _int]),
    "saa_group_step": (_int, [_vp, _i64, _int, _int]),
    "saa_group_synchronize": (_int, [_vp]),
    "saa_group_destroy": (_int, [_vp]),
    "saa_plan_peer_export": (_int, [_vp, _vp, _vp]),
    "saa_plan_peer_attach": (_int, [_vp, _int, _vp, _vp, _vp, _vp, _vp]),
    "saa_nccl_unique_id": (_int, [_vp]),
    "saa_plan_init_nccl": (_int, [_vp, _vp]),
}


class SaaError(RuntimeError):
    pass


# one energy record (include/saa_fem.h, SAA_ENERGY_FIELDS): fields 2-8 are additive over the ranks of a partition
ENERGY_FIELDS = ("step", "tn", "kinetic_half", "coupling", "strain", "kinetic", "work_external", "work_damping",
                 "energy_at_arm")
ENERGY_DTYPE = np.dtype([("step", np.int64)] + [(f, np.float64) for f in ENERGY_FIELDS[1:]])
BALANCE_DTYPE = np.dtype(ENERGY_DTYPE.descr + [("total", np.float64), ("residual", np.float64)])

# one element row of StepPlan.element_stress (include/saa_fem.h, SAA_STRESS_FIELDS)
STRESS_FIELDS = ("sxx", "syy", "szz", "syz", "sxz", "sxy", "von_mises", "weight")


def energy_balance(records_per_rank):
    """Global energy balance of a partition from the per-rank records of the same steps (read_energy of every rank,
    in rank order): the additive fields summed in ascending rank order, plus
      total    = kinetic_half + coupling                      (E_{n-1/2} = T_{n-1/2} + S_{n-1/2})
      residual = total - energy_at_arm - work_external + work_damping   (0 in exact arithmetic).
    Raises ValueError when the ranks' records are not of the same steps."""
    recs = [np.asarray(r) for r in records_per_rank]
    if not recs:
        raise ValueError("energy_balance: no records")
    out = np.zeros(recs[0].shape, dtype=BALANCE_DTYPE)
    out["step"], out["tn"] = recs[0]["step"], recs[0]["tn"]
    for q, r in enumerate(recs):
        if r.shape != out.shape or not np.array_equal(r["step"], out["step"]) or not np.array_equal(r["tn"], out["tn"]):
            raise ValueError(f"energy_balance: the records of rank {q} are not of the same steps as rank 0's (step / tn differ)")
        for f in ENERGY_FIELDS[2:]:
            out[f] += r[f]
    out["total"] = out["kinetic_half"] + out["coupling"]
    out["residual"] = out["total"] - out["energy_at_arm"] - out["work_external"] + out["work_damping"]
    return out


class StaticResult:
    """Result of StepPlan.solve_static / PlanGroup.solve_static.
    x                  solution in local DOF order: a float64 CUDA tensor, or a list of them (one per plan of a group)
    iterations         CG iterations run
    rel_residual       ||r|| / ||b|| of the CG recurrence at the returned iterate
    rel_residual_true  ||b - A x|| / ||b|| from one more stiffness apply
    converged          rel_residual <= rtol was reached within max_iter
    history            float64 CUDA tensor (iterations,): ||r_k|| after iteration k = 1, 2, ..."""

    def __init__(self, x, iterations, rel_residual, rel_residual_true, converged, history):
        self.x, self.iterations, self.history = x, iterations, history
        self.rel_residual, self.rel_residual_true, self.converged = rel_residual, rel_residual_true, converged

    def __repr__(self):
        return (f"StaticResult(iterations={self.iterations}, rel_residual={self.rel_residual:.3e}, "
                f"rel_residual_true={self.rel_residual_true:.3e}, converged={self.converged})")


def _dev_vector(t, n, device, what):
    """t checked as a contiguous float64 CUDA tensor of n entries on `device`"""
    import torch
    dev = torch.device("cuda", device)
    if not isinstance(t, torch.Tensor) or t.dtype != torch.float64 or t.device != dev or t.numel() != n or not t.is_contiguous():
        raise SaaError(f"{what}: need a contiguous float64 tensor of {n} entries on {dev}")
    return t


# default iteration cap of solve_static: the history takes max_iter doubles on the device during the call (8 MB here)
MAX_ITER_DEFAULT = 1_000_000


# default iteration cap of the multigrid-preconditioned solve (its iteration count does not grow with the mesh)
MG_MAX_ITER_DEFAULT = 1000


def _solve_static(fn, handle, plans, rtol, max_iter, x0, check_every, single=False):
    import torch
    dev = torch.device("cuda", plans[0].device)
    max_iter = min(10 * sum(pl.n_dof for pl in plans), MAX_ITER_DEFAULT) if max_iter is None else int(max_iter)
    x0 = [None] * len(plans) if x0 is None else list(x0)
    if len(x0) != len(plans):
        raise SaaError(f"solve_static: x0 needs one vector per plan ({len(plans)})")
    x0 = [None if v is None else _dev_vector(v, pl.n_dof, pl.device, "solve_static: x0") for v, pl in zip(x0, plans)]
    xs = [torch.empty(pl.n_dof, dtype=torch.float64, device=dev) for pl in plans]
    hist = torch.empty(max(max_iter, 1), dtype=torch.float64, device=dev)
    ptrs = lambda ts: (ctypes.c_void_p * len(ts))(*[None if t is None else t.data_ptr() for t in ts])
    it, rel, rel_true, conv = ctypes.c_int64(0), ctypes.c_double(0), ctypes.c_double(0), ctypes.c_int(0)
    torch.cuda.current_stream(dev).synchronize()              # torch's pending work on x0 precedes the plans' stream
    args = (float(rtol), max_iter, int(check_every), hist.data_ptr(), ctypes.byref(it), ctypes.byref(rel),
            ctypes.byref(rel_true), ctypes.byref(conv))
    if handle is None or single:
        _check(fn(plans[0].h if handle is None else handle, None if x0[0] is None else x0[0].data_ptr(), xs[0].data_ptr(), *args),
               "saa_plan_solve_static_dev" if handle is None else "saa_plan_solve_static_mg_dev")
    else:
        _check(fn(handle, ptrs(x0), ptrs(xs), *args), "saa_group_solve_static_dev")
    return StaticResult(xs[0] if handle is None or single else xs, int(it.value), rel.value, rel_true.value, bool(conv.value),
                        hist[:int(it.value)].clone())        # the max_iter-long buffer is released


PINNED_POOL = 4


class _PinnedVector:
    """n float64 of page-locked host memory (saa_host_alloc); numpy arrays made from it keep it alive through
    their .base and it returns the memory when the last one is gone."""

    def __init__(self, n):
        self.ptr = lib().saa_host_alloc(8 * int(n))
        if not self.ptr:
            raise SaaError("saa_host_alloc: " + lib().saa_last_error().decode())
        self.__array_interface__ = {"shape": (int(n),), "typestr": "<f8", "data": (self.ptr, False), "version": 3}

    def __del__(self):
        try:
            if self.ptr:
                lib().saa_host_free(self.ptr)
                self.ptr = None
        except Exception:
            pass


def library_path():
    return _SO


def build(force=False, verbose=False):
    """Compile csrc/libsaa_fem.so for sm_100a with nvcc (cross-compiles without a GPU)."""
    srcs = [os.path.join(_CSRC, f) for f in os.listdir(_CSRC) if f.endswith((".cu", ".cuh"))]
    srcs.append(os.path.join(os.path.dirname(_HERE), "include", "saa_fem.h"))
    stale = (not os.path.isfile(_SO)) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs)
    if force or stale:
        r = subprocess.run(["make", "-C", _CSRC] + (["-B"] if force else []), capture_output=True, text=True)
        if verbose or r.returncode:
            print(r.stdout, r.stderr)
        if r.returncode:
            raise SaaError("building libsaa_fem.so failed")
    return _SO


def lib():
    """Load libsaa_fem.so and declare every prototype of include/saa_fem.h.  Fails loudly when absent."""
    global _lib
    if _lib is None:
        if not os.path.isfile(_SO):
            raise SaaError(f"{_SO} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback for the time-step path)")
        L = ctypes.CDLL(_SO, mode=ctypes.RTLD_GLOBAL)
        for name, (res, args) in ABI.items():
            f = getattr(L, name)
            f.restype, f.argtypes = res, args
        _lib = L
    return _lib


def _check(rc, what=""):
    if rc != 0:
        raise SaaError(f"{what}: {lib().saa_last_error().decode(errors='replace')}")


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def rcm_node_order(K):
    """Reverse Cuthill-McKee order of the node graph of a 3-DOF-per-node CSR matrix (memory-layout hint)."""
    from scipy.sparse import csr_matrix
    from scipy.sparse.csgraph import reverse_cuthill_mckee
    n = K.shape[0] // 3
    rows = np.repeat(np.arange(K.shape[0]), np.diff(K.indptr)) // 3
    G = csr_matrix((np.ones(K.indices.size, dtype=np.int8), (rows, K.indices // 3)), shape=(n, n))
    return reverse_cuthill_mckee(G.tocsr(), symmetric_mode=True).astype(np.int32)


def step_scalars(dt, alpha):
    """Scalar sub-expressions of Dynamic_solver.py:17 with the reference's own Python expressions on the
    reference's own types (dt: np.float64, so `dt**2` is numpy's power; alpha: Python float)."""
    dt = np.float64(dt)
    return float(dt), float(dt ** 2), float(dt / 2), float(0.5 * alpha), float(alpha)


class StepPlan:
    """Device-resident problem + state of one partition (one reference MPI rank)."""

    def __init__(self, LocalK, F_rankwise, l_M, Local_Dirichlet, dt, alpha, device=0, halo=None, rank=0, size=1, node_order=None):
        """LocalK: scipy CSR (sorted indices; its stored order is the summation order).
        halo: dict from maps.halo_plan(rank, size, rank_nodal_list) when size > 1.
        node_order: optional permutation of the local nodes (memory layout only, see saa_plan_set_node_order);
        "rcm" computes a reverse Cuthill-McKee order of the node graph here."""
        L = lib()
        K = LocalK.tocsr() if not hasattr(LocalK, "indptr") else LocalK
        n = K.shape[0]
        if int(K.indptr[-1]) >= 2 ** 31:
            raise SaaError("LocalK has more than 2^31 stored entries; use the 64-bit device assembly path")
        self._indptr = np.ascontiguousarray(K.indptr, dtype=np.int32)
        self._indices = np.ascontiguousarray(K.indices, dtype=np.int32)
        self._data = np.ascontiguousarray(K.data, dtype=np.float64)
        F = np.ascontiguousarray(F_rankwise, dtype=np.float64).reshape(-1)
        M = np.ascontiguousarray(l_M, dtype=np.float64).reshape(-1)
        D = np.ascontiguousarray(Local_Dirichlet, dtype=np.int64).reshape(-1)
        if F.size != n or M.size != n:
            raise SaaError(f"F_rankwise/l_M have {F.size}/{M.size} entries, LocalK has {n} rows")
        self.n_dof, self.rank, self.size, self.device = n, int(rank), int(size), int(device)
        self.dt, self.dt2, self.dt_half, self.half_alpha, self.alpha = step_scalars(dt, alpha)
        h = ctypes.c_void_p()
        _check(L.saa_plan_create(ctypes.byref(h), device, n, _p(self._indptr), _p(self._indices), _p(self._data),
                                 _p(F), _p(M), _p(D), D.size, self.dt, self.dt2, self.dt_half, self.half_alpha,
                                 self.alpha), "saa_plan_create")
        self.h = h
        if isinstance(node_order, str) and node_order == "rcm":
            node_order = rcm_node_order(K)
        self._set_halo_and_finalize(halo, node_order)
        del self._indptr, self._indices, self._data

    @classmethod
    def from_device(cls, n_dof, indptr_ptr, indices_ptr, data_ptr, F_ptr, lM_ptr, Local_Dirichlet, dt, alpha, device=0,
                    halo=None, rank=0, size=1, node_order=None):
        """Plan from a CSR that already lives on the GPU (raw device pointers; int64 indptr, int32 indices)."""
        self = cls.__new__(cls)
        D = np.ascontiguousarray(Local_Dirichlet, dtype=np.int64).reshape(-1)
        self.n_dof, self.rank, self.size, self.device = int(n_dof), int(rank), int(size), int(device)
        self.dt, self.dt2, self.dt_half, self.half_alpha, self.alpha = step_scalars(dt, alpha)
        h = ctypes.c_void_p()
        _check(lib().saa_plan_create_dev(ctypes.byref(h), device, int(n_dof), indptr_ptr, indices_ptr, data_ptr, F_ptr, lM_ptr,
                                         _p(D), D.size, self.dt, self.dt2, self.dt_half, self.half_alpha, self.alpha),
               "saa_plan_create_dev")
        self.h = h
        self._set_halo_and_finalize(halo, node_order)
        return self

    def _set_halo_and_finalize(self, halo, node_order=None):
        L, h, rank, size = lib(), self.h, self.rank, self.size
        self._halo_desc = halo
        if node_order is not None:
            o = np.ascontiguousarray(node_order, dtype=np.int32).reshape(-1)
            _check(L.saa_plan_set_node_order(h, _p(o), o.size), "saa_plan_set_node_order")
        if size > 1:
            if halo is None:
                raise SaaError("size > 1 needs the halo description (maps.halo_plan)")
            nb = np.ascontiguousarray(halo["neighbours"], dtype=np.int32)
            ptr = np.zeros(nb.size + 1, dtype=np.int64)
            for k, r in enumerate(halo["neighbours"]):
                ptr[k + 1] = ptr[k] + halo["send_idx"][r].size
            send = (np.concatenate([halo["send_idx"][r] for r in halo["neighbours"]]) if nb.size
                    else np.zeros(0, dtype=np.int64)).astype(np.int64)
            sp = np.ascontiguousarray(halo["shared_pos"], dtype=np.int64)
            hp = np.ascontiguousarray(halo["holders_ptr"], dtype=np.int64)
            hr = np.ascontiguousarray(halo["holders_rank"], dtype=np.int32)
            hs = np.ascontiguousarray(halo["holders_slot"], dtype=np.int64)
            _check(L.saa_plan_set_halo(h, rank, size, sp.size, _p(sp), nb.size, _p(nb), _p(ptr), _p(send), _p(hp),
                                       _p(hr), _p(hs)), "saa_plan_set_halo")
        _check(L.saa_plan_finalize(h), "saa_plan_finalize")

    # ---- facts -------------------------------------------------------------------------------------
    @property
    def nnz(self):
        return int(lib().saa_plan_nnz(self.h))

    @property
    def padded_entries(self):
        return int(lib().saa_plan_padded_entries(self.h))

    @property
    def value_planes(self):
        """value planes the step kernel streams, raw or coded; padded_entries / 32 when every plane is stored"""
        return int(lib().saa_plan_value_planes(self.h))

    @property
    def coded_planes(self):
        """value planes stored as an int64 base + 32 16-bit lane offsets (64 B instead of 256 B)"""
        return int(lib().saa_plan_coded_planes(self.h))

    @property
    def matrix_bytes(self):
        """bytes of the plane-masked matrix layout without value coding (256 B per value plane)"""
        return int(lib().saa_plan_matrix_bytes(self.h))

    @property
    def streamed_matrix_bytes(self):
        """bytes of matrix storage the step kernel streams per time step (coded planes at their coded size)"""
        return int(lib().saa_plan_streamed_matrix_bytes(self.h))

    @property
    def vector_bytes(self):
        """bytes of the fp64 vector streams of one time step (d0, dn read; d1 written; F; lumped mass per DOF or per node)"""
        return int(lib().saa_plan_vector_bytes(self.h))

    @property
    def kernel_launches(self):
        return int(lib().saa_plan_kernel_launches(self.h))

    @property
    def stream(self):
        """raw cudaStream_t of the plan (int) — wrap with torch.cuda.ExternalStream to time on it"""
        return int(lib().saa_plan_stream(self.h) or 0)

    # ---- state -------------------------------------------------------------------------------------
    def set_state(self, d0, dn, tn):
        d0 = np.ascontiguousarray(d0, dtype=np.float64).reshape(-1)
        dn = np.ascontiguousarray(dn, dtype=np.float64).reshape(-1)
        if d0.size != self.n_dof or dn.size != self.n_dof:
            raise SaaError("set_state: wrong vector length")
        _check(lib().saa_plan_set_state(self.h, _p(d0), _p(dn), float(tn)), "saa_plan_set_state")

    def get_state(self):
        d0, dn = np.empty(self.n_dof), np.empty(self.n_dof)
        tn = ctypes.c_double(0)
        _check(lib().saa_plan_get_state(self.h, _p(d0), _p(dn), ctypes.byref(tn)), "saa_plan_get_state")
        return d0, dn, tn.value

    def d0(self):
        d0 = np.empty(self.n_dof)
        _check(lib().saa_plan_get_state(self.h, _p(d0), None, None), "saa_plan_get_state")
        return d0

    def set_state_dev(self, d0_ptr, dn_ptr, tn):
        _check(lib().saa_plan_set_state_dev(self.h, d0_ptr, dn_ptr, float(tn)), "saa_plan_set_state_dev")

    def get_state_dev(self, d0_ptr, dn_ptr):
        tn = ctypes.c_double(0)
        _check(lib().saa_plan_get_state_dev(self.h, d0_ptr, dn_ptr, ctypes.byref(tn)), "saa_plan_get_state_dev")
        return tn.value

    # ---- stepping ----------------------------------------------------------------------------------
    def step(self, n_steps=1, mode=MODE_LOCAL, launch=LAUNCH_AUTO):
        _check(lib().saa_plan_step(self.h, int(n_steps), int(mode), int(launch)), "saa_plan_step")

    def synchronize(self):
        _check(lib().saa_plan_synchronize(self.h), "saa_plan_synchronize")

    def set_option(self, option, value):
        _check(lib().saa_plan_set_option(self.h, int(option), int(value)), "saa_plan_set_option")

    def set_matfree(self, cells_local, coords_local, lmd, mu):
        """Hand the element connectivity (nE,4; local node ids) and the local node coordinates (n,3) to the plan for the
        matrix-free kernel K5 (torch CUDA tensors, or host arrays which are uploaded through torch); enable it with
        set_option(OPT_MATFREE, 1).  Refused (SaaError, the plan unchanged): a node id outside [0, n_dof/3), an element with
        a repeated corner or detJ == 0; negative detJ is accepted (the reference's volume is signed)."""
        import torch
        dev = torch.device("cuda", self.device)
        nn = self.n_dof // 3
        # node ids are checked in their own type: the int32 cast below would wrap an id >= 2^31 into range
        if isinstance(cells_local, torch.Tensor):
            c = cells_local
            if c.is_floating_point() or c.is_complex() or c.dtype == torch.bool:
                raise SaaError(f"set_matfree: cells must hold integer node ids, not {c.dtype}")
            lo, hi = (int(c.min()), int(c.max())) if c.numel() else (0, 0)
        else:
            a = np.asarray(cells_local)
            if not np.issubdtype(a.dtype, np.integer):
                raise SaaError(f"set_matfree: cells must hold integer node ids, not {a.dtype}")
            lo, hi = (int(a.min()), int(a.max())) if a.size else (0, 0)
            c = torch.from_numpy(np.ascontiguousarray(a.astype(np.int64)))
        if lo < 0 or hi >= nn:
            raise SaaError(f"set_matfree: node id {lo if lo < 0 else hi} outside [0, {nn})")
        x = coords_local if isinstance(coords_local, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(coords_local, dtype=np.float64))
        c = c.to(device=dev, dtype=torch.int32).contiguous()
        x = x.to(device=dev, dtype=torch.float64).contiguous()
        if c.ndim != 2 or c.shape[1] != 4 or x.shape != (self.n_dof // 3, 3):
            raise SaaError("set_matfree: cells must be (nE,4) and coords (n_dof/3, 3)")
        torch.cuda.synchronize(dev)
        _check(lib().saa_plan_set_matfree_dev(self.h, c.shape[0], c.data_ptr(), x.data_ptr(), float(lmd), float(mu)),
               "saa_plan_set_matfree_dev")
        self.n_elem = int(c.shape[0])

    @property
    def matfree_bytes(self):
        return int(lib().saa_plan_matfree_bytes(self.h))

    # ---- stress recovery ---------------------------------------------------------------------------
    def element_stress(self, out=None):
        """(n_elem, 8) float64 CUDA tensor of the current d0, one row per element in the order of the cells given to
        set_matfree: sigma in Voigt order (xx yy zz yz xz xy), von Mises, weight V = detJ/6 (STRESS_FIELDS).  Needs
        the geometry of set_matfree (the matrix-free step need not be enabled).  Raises SaaError for an element with
        detJ <= 0.  The values are complete when it returns."""
        import torch
        if not hasattr(self, "n_elem"):
            _check(lib().saa_plan_element_stress_dev(self.h, None), "saa_plan_element_stress_dev")
        dev = torch.device("cuda", self.device)
        if out is None:
            out = torch.empty((self.n_elem, 8), dtype=torch.float64, device=dev)
        elif out.shape != (self.n_elem, 8) or out.dtype != torch.float64 or out.device != dev or not out.is_contiguous():
            raise SaaError(f"element_stress: out must be a contiguous float64 ({self.n_elem}, 8) tensor on {dev}")
        torch.cuda.current_stream(dev).synchronize()          # torch's pending work on `out` precedes the plan's stream
        _check(lib().saa_plan_element_stress_dev(self.h, out.data_ptr()), "saa_plan_element_stress_dev")
        return out

    def nodal_stress_partial(self, elem=None):
        """(n_nodes, 7) float64 CUDA tensor, Local_nodal_list order: this rank's sums of V_e sigma_e (6) and V_e (1)
        over its elements incident to each node, added in ascending element order.  `elem` is an element_stress
        result (computed here when not given).  stress.nodal_stress turns it into averaged nodal stresses."""
        import torch
        if not hasattr(self, "n_elem"):
            _check(lib().saa_plan_nodal_stress_dev(self.h, None, None), "saa_plan_nodal_stress_dev")
        dev = torch.device("cuda", self.device)
        if elem is None:
            elem = self.element_stress()
        elif elem.shape != (self.n_elem, 8) or elem.dtype != torch.float64 or elem.device != dev or not elem.is_contiguous():
            raise SaaError(f"nodal_stress_partial: elem must be a contiguous float64 ({self.n_elem}, 8) tensor on {dev}")
        out = torch.empty((self.n_dof // 3, 7), dtype=torch.float64, device=dev)
        torch.cuda.current_stream(dev).synchronize()
        _check(lib().saa_plan_nodal_stress_dev(self.h, elem.data_ptr(), out.data_ptr()), "saa_plan_nodal_stress_dev")
        self.synchronize()
        return out

    # ---- static solve ------------------------------------------------------------------------------
    def apply_stiffness(self, x):
        """y = LocalK x (float64 CUDA tensors of n_dof, local DOF order), bit for bit scipy's LocalK @ x on a host-built
        plan.  Shared rows of a partition hold this rank's partial (PlanGroup.apply_stiffness sums them)."""
        import torch
        x = _dev_vector(x, self.n_dof, self.device, "apply_stiffness: x")
        y = torch.empty_like(x)
        torch.cuda.current_stream(x.device).synchronize()
        _check(lib().saa_plan_apply_stiffness_dev(self.h, x.data_ptr(), y.data_ptr()), "saa_plan_apply_stiffness_dev")
        return y

    def solve_static(self, rtol=1e-10, max_iter=None, x0=None, check_every=None, precond=None):
        """Solve the steady system of Steady_Elasticity_solver, (S K S + I - S) x = S F, on the device by block-Jacobi
        preconditioned CG (DESIGN.md §7c).  max_iter defaults to 10 n_dof, at most MAX_ITER_DEFAULT (CG in floating
        point needs more than n_dof iterations on an ill-conditioned system); x0: start tensor (None: 0).  Returns a
        StaticResult; not converging within max_iter is not an error (converged=False).  A plan of a partition with
        size > 1 is solved through PlanGroup.solve_static.
        precond: a multigrid.StructuredMultigrid built for this plan: one V-cycle per iteration instead of the
        block-Jacobi step (DESIGN.md §7d); max_iter then defaults to 1000 and check_every to 10 (50 without)."""
        if precond is None:
            return _solve_static(lib().saa_plan_solve_static_dev, None, [self], rtol, max_iter, None if x0 is None else [x0],
                                 50 if check_every is None else check_every)
        if getattr(precond, "plan", None) is not self:
            raise SaaError("solve_static: the multigrid hierarchy was built for another plan")
        return _solve_static(lib().saa_plan_solve_static_mg_dev, precond.handle(), [self], rtol,
                             MG_MAX_ITER_DEFAULT if max_iter is None else max_iter, None if x0 is None else [x0],
                             10 if check_every is None else check_every, single=True)

    def _host_out(self):
        """The array a host call returns d1 in.  From 1 MiB per vector on it is a view of page-locked memory
        (saa_host_alloc), so that this download and — once the caller has rotated it into d_0 / d_n
        (Data_prepare.py:233-234) — the next uploads are asynchronous full-rate PCIe copies that the pipelined call
        can overlap.  A buffer is handed out again only when no array refers to it any more (the views hold a
        reference to their owner); at most PINNED_POOL buffers exist per plan, beyond that (a caller that keeps every
        d1) plain numpy memory is returned.  SAA_STEP_HOST_PINNED=0 switches it off."""
        n = self.n_dof
        if 8 * n < (1 << 20) or os.environ.get("SAA_STEP_HOST_PINNED", "1") == "0":
            return np.empty(n)
        pool = self.__dict__.setdefault("_pinned_pool", [])
        for i in range(len(pool)):
            if sys.getrefcount(pool[i]) == 2:            # the list's reference + getrefcount's argument: no array left
                return np.asarray(pool[i])
        if len(pool) < PINNED_POOL:
            pool.append(_PinnedVector(n))
            return np.asarray(pool[-1])
        return np.empty(n)

    def host_pipe_info(self, mode=MODE_LOCAL):
        """(K, slice_end[K], need_upload[K]) of the pipelined host call for `mode`; K = 0: plain sequence."""
        k = ctypes.c_int(0)
        se, nu = np.zeros(64, dtype=np.int64), np.zeros(64, dtype=np.int32)
        _check(lib().saa_plan_host_pipe_info(self.h, int(mode), ctypes.byref(k), _p(se), _p(nu), 64), "saa_plan_host_pipe_info")
        return k.value, se[:k.value].copy(), nu[:k.value].copy()

    def step_host(self, d0, dn, tn, mode=MODE_LOCAL, out=None):
        """One parallel_explicit_solver_dis_pre evaluation with host buffers -> d1 (n_dof,).

        The reference's loop rotates `d_n = d_0; d_0 = d1` (Data_prepare.py:233-234), so the `dn` of a call is
        normally the very array passed as `d0` to the previous call; its values are still on the device and are not
        uploaded again (saa_step_host_ex, SAA_HOST_DN_IS_PREVIOUS_D0).  "The very array" = same memory, kept alive
        by this plan since the previous call.  Writing INTO that array between the two calls is not detected — the
        reference never does (it only writes into the returned d1, Online_predictor.py:298, which is always
        uploaded); set SAA_STEP_HOST_FULL_UPLOAD=1 to upload both vectors on every call."""
        d0 = np.ascontiguousarray(d0, dtype=np.float64).reshape(-1)
        dn = np.ascontiguousarray(dn, dtype=np.float64).reshape(-1)
        if d0.size != self.n_dof or dn.size != self.n_dof:
            raise SaaError("step_host: wrong vector length")
        d1 = self._host_out() if out is None else out
        prev = getattr(self, "_host_prev_d0", None)
        flags = 0
        if prev is not None and prev.ctypes.data == dn.ctypes.data and not os.environ.get("SAA_STEP_HOST_FULL_UPLOAD"):
            flags = HOST_DN_IS_PREVIOUS_D0
        rc = lib().saa_step_host_ex(self.h, _p(d0), _p(dn), float(tn), int(mode), _p(d1), flags)
        if rc < 0:
            _check(rc, "saa_step_host_ex")
        self._host_prev_d0 = d0                      # keeps the memory alive: the same address next time is the same array
        self.host_uploads_skipped = getattr(self, "host_uploads_skipped", 0) + (1 if rc == 1 else 0)
        return d1

    # ---- history / prediction ----------------------------------------------------------------------
    def set_history(self, dofs, capacity, save_every=1):
        d = None if dofs is None else np.ascontiguousarray(dofs, dtype=np.int64).reshape(-1)
        self._hist_n = self.n_dof if d is None else d.size
        _check(lib().saa_plan_set_history(self.h, _p(d), self._hist_n, int(capacity), int(save_every)),
               "saa_plan_set_history")

    @property
    def history_count(self):
        return int(lib().saa_plan_history_count(self.h))

    def read_history(self, first=0, count=None):
        count = self.history_count - first if count is None else count
        out = np.empty((count, self._hist_n))
        _check(lib().saa_plan_read_history(self.h, int(first), int(count), _p(out)), "saa_plan_read_history")
        return out

    def read_history_dev(self, first, count, dev_ptr):
        _check(lib().saa_plan_read_history_dev(self.h, int(first), int(count), dev_ptr), "saa_plan_read_history_dev")

    def set_prediction(self, dofs, table_dev_ptr, n_rows):
        d = None if dofs is None else np.ascontiguousarray(dofs, dtype=np.int64).reshape(-1)
        n = self._pred_n if d is None else d.size
        self._pred_n = n
        _check(lib().saa_plan_set_prediction(self.h, _p(d), n, table_dev_ptr, int(n_rows)), "saa_plan_set_prediction")

    # ---- energy monitor ----------------------------------------------------------------------------
    def set_energy(self, capacity, every=1):
        """Arm the on-device energy monitor with a ring of `capacity` records, one every `every` steps (capacity 0
        disarms).  Every rank of a partition must arm at the same step with the same `every`."""
        _check(lib().saa_plan_set_energy(self.h, int(capacity), int(every)), "saa_plan_set_energy")

    @property
    def energy_count(self):
        return int(lib().saa_plan_energy_count(self.h))

    def read_energy(self, first=0, count=None):
        """Records [first, first + count) as a structured array of ENERGY_DTYPE (this rank's share; energy_balance
        combines the ranks)."""
        count = self.energy_count - first if count is None else count
        raw = np.empty((max(int(count), 0), len(ENERGY_FIELDS)))
        _check(lib().saa_plan_read_energy(self.h, int(first), int(count), _p(raw)), "saa_plan_read_energy")
        out = np.empty(raw.shape[0], dtype=ENERGY_DTYPE)
        for k, f in enumerate(ENERGY_FIELDS):
            out[f] = raw[:, k]
        return out

    # ---- caller-provided transport (messages through host memory) -----------------------------------
    def halo_layout(self):
        """(neighbour ranks ascending, message offsets in doubles) of the send / receive buffers."""
        n = ctypes.c_int(0)
        _check(lib().saa_plan_halo_layout(self.h, ctypes.byref(n), None, None, 0), "saa_plan_halo_layout")
        nb = np.zeros(n.value, dtype=np.int32)
        off = np.zeros(n.value + 1, dtype=np.int64)
        _check(lib().saa_plan_halo_layout(self.h, ctypes.byref(n), _p(nb), _p(off), n.value), "saa_plan_halo_layout")
        return nb, off

    def step_exchange(self, exchange):
        """One synchronised step with the caller's transport: `exchange(send, nb, off) -> recv` moves
        send[off[k]:off[k+1]] to rank nb[k] and returns the buffer received from the neighbours (same layout)."""
        if not hasattr(self, "_nb"):
            self._nb, self._off = self.halo_layout()
            self._send = np.zeros(max(int(self._off[-1]), 1))
        _check(lib().saa_plan_step_begin_host(self.h, _p(self._send)), "saa_plan_step_begin_host")
        recv = np.ascontiguousarray(exchange(self._send[:int(self._off[-1])], self._nb, self._off), dtype=np.float64)
        _check(lib().saa_plan_step_end_host(self.h, _p(recv)), "saa_plan_step_end_host")

    def sync_forces(self, f, exchange):
        """syn_cpus on a host force vector: returns f_global[dofs_local] (n_dof,)."""
        if not hasattr(self, "_nb"):
            self._nb, self._off = self.halo_layout()
            self._send = np.zeros(max(int(self._off[-1]), 1))
        f = np.ascontiguousarray(f, dtype=np.float64).reshape(-1)
        if f.size != self.n_dof:
            raise SaaError("sync_forces: wrong vector length")
        _check(lib().saa_plan_forces_begin_host(self.h, _p(f), _p(self._send)), "saa_plan_forces_begin_host")
        recv = np.ascontiguousarray(exchange(self._send[:int(self._off[-1])], self._nb, self._off), dtype=np.float64)
        out = np.empty(self.n_dof)
        _check(lib().saa_plan_forces_end_host(self.h, _p(recv), _p(out)), "saa_plan_forces_end_host")
        return out

    # ---- peer-memory transport (NVLink, one process per GPU) ----------------------------------------
    def peer_export(self):
        """(64-byte CUDA IPC handle of the receive area, neighbour ranks, message offsets)."""
        buf = ctypes.create_string_buffer(64)
        tot = ctypes.c_int64(0)
        _check(lib().saa_plan_peer_export(self.h, buf, ctypes.byref(tot)), "saa_plan_peer_export")
        nb, off = self.halo_layout()
        return dict(rank=self.rank, handle=buf.raw, nb=nb.tolist(), off=off.tolist())

    def peer_attach(self, exports):
        """exports: list over ALL ranks of peer_export() dicts (e.g. from all_gather_object)."""
        nb, off = self.halo_layout()
        by_rank = {e["rank"]: e for e in exports if e is not None}
        handles = b""
        r_off, r_tot, r_slot, r_nnb = [], [], [], []
        for r in nb.tolist():
            e = by_rank[r]
            slot = e["nb"].index(self.rank)
            handles += e["handle"]
            r_off.append(e["off"][slot]); r_tot.append(e["off"][-1]); r_slot.append(slot); r_nnb.append(len(e["nb"]))
        hb = ctypes.create_string_buffer(handles, max(len(handles), 1))
        a = lambda v, t: np.ascontiguousarray(v, dtype=t)
        ro, rt, rs, rn = a(r_off, np.int64), a(r_tot, np.int64), a(r_slot, np.int32), a(r_nnb, np.int32)
        _check(lib().saa_plan_peer_attach(self.h, nb.size, hb, _p(ro), _p(rt), _p(rs), _p(rn)), "saa_plan_peer_attach")

    # ---- NCCL transport ----------------------------------------------------------------------------
    def init_nccl(self, unique_id: bytes):
        buf = ctypes.create_string_buffer(bytes(unique_id), 128)
        _check(lib().saa_plan_init_nccl(self.h, buf), "saa_plan_init_nccl")

    def close(self):
        if getattr(self, "h", None):
            lib().saa_plan_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def nccl_unique_id() -> bytes:
    buf = ctypes.create_string_buffer(128)
    _check(lib().saa_nccl_unique_id(buf), "saa_nccl_unique_id")
    return buf.raw


class PlanGroup:
    """All P partitions in ONE process on one GPU, stepped together; the halo exchange is a set of
    device-to-device copies.  Used to run a P-way partition when fewer than P GPUs are available
    (and by the parity tests, which need every P on a single B200)."""

    def __init__(self, plans):
        self.plans = list(plans)
        arr = (ctypes.c_void_p * len(self.plans))(*[p.h for p in self.plans])
        h = ctypes.c_void_p()
        _check(lib().saa_group_create(ctypes.byref(h), arr, len(self.plans)), "saa_group_create")
        self.h = h

    def step(self, n_steps=1, mode=MODE_SYNC, launch=LAUNCH_AUTO):
        _check(lib().saa_group_step(self.h, int(n_steps), int(mode), int(launch)), "saa_group_step")

    def synchronize(self):
        _check(lib().saa_group_synchronize(self.h), "saa_group_synchronize")

    def apply_stiffness(self, xs):
        """[LocalK_r x_r] of every plan with the shared rows summed over their holders in ascending rank order
        (f_global[dofs_local] of syn_cpus): list of float64 CUDA tensors, local DOF order."""
        import torch
        if len(xs) != len(self.plans):
            raise SaaError(f"apply_stiffness: need one vector per plan ({len(self.plans)})")
        xs = [_dev_vector(x, pl.n_dof, pl.device, "apply_stiffness: x") for x, pl in zip(xs, self.plans)]
        ys = [torch.empty_like(x) for x in xs]
        ptrs = lambda ts: (ctypes.c_void_p * len(ts))(*[t.data_ptr() for t in ts])
        torch.cuda.current_stream(xs[0].device).synchronize()
        _check(lib().saa_group_apply_stiffness_dev(self.h, ptrs(xs), ptrs(ys)), "saa_group_apply_stiffness_dev")
        return ys

    def solve_static(self, rtol=1e-10, max_iter=None, x0=None, check_every=50, precond=None):
        """StepPlan.solve_static over all partitions of the group; x0 and the result's x are lists, one per plan.
        max_iter defaults to 10 times the sum of the plans' n_dof, at most MAX_ITER_DEFAULT.  The multigrid
        preconditioner is not available for a partitioned problem (precond must be None)."""
        if precond is not None:
            raise SaaError("PlanGroup.solve_static: the multigrid preconditioner (precond) works on a single-partition plan "
                           "only; a partitioned problem is solved with block-Jacobi CG (precond=None)")
        return _solve_static(lib().saa_group_solve_static_dev, self.h, self.plans, rtol, max_iter, x0, check_every)

    def close(self):
        if getattr(self, "h", None):
            lib().saa_group_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def device_count():
    return int(lib().saa_device_count())
