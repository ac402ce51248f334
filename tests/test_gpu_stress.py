"""Stress recovery on the device (StepPlan.element_stress / nodal_stress_partial, saa_b200.stress, multi.gather_nodal_stress).

  * patch test: a linear displacement gives D voigt(sym G) in every element and node, a rigid motion gives ~0;
  * element sigma, von Mises and V equal a numpy evaluation through assembly._B_stack / elasticity_D;
  * sum_e V_e B_e^T sigma_e equals LocalK d0 (the stiffness the parity path streams);
  * an element's fields are the same bits on one partition, on three, and in another node order; averaged nodal
    stresses too, except for the association of the holder sum at shared nodes;
  * evaluations change no state bit and no energy record, and work after the matrix is released;
  * the device set-up path at 1.13 M DOF; refusals; the one-process-per-rank form.
"""
import ctypes
import os
import sys

import numpy as np
import pytest
import scipy.sparse as sp

import saa_b200  # noqa: F401
from saa_b200 import assembly, device_setup, maps, plan as splan, problem, stress
from util import ROOT, bits_equal, load_golden, make_oracle

pytestmark = pytest.mark.gpu
PATCH_REL = 1e-13
NUMPY_REL = 1e-12


def _K(r):
    n = r["F"].size
    return sp.csr_matrix((r["K_data"], r["K_indices"], r["K_indptr"]), shape=(n, n))


def _lame(g):
    return problem.lame(float(g["E"]), float(g["nu"]))


def local_mesh(g, q):
    """(cells in local node ids, local coordinates) of rank q of a golden case, elements in r['ele'] order"""
    r = g["ranks"][q]
    nodes = np.asarray(r["nodes"], dtype=np.int64)
    pos = np.full(len(g["points"]), -1, dtype=np.int64)
    pos[nodes] = np.arange(nodes.size)
    cells = pos[np.asarray(g["cells"], dtype=np.int64)[np.asarray(r["ele"], dtype=np.int64)]]
    return cells, np.asarray(g["points"], dtype=np.float64)[nodes]


def make_plans(g, node_order=None, group=True):
    """every rank of a golden case with its mesh attached; a PlanGroup for P > 1"""
    P = g["P"]
    lists = [r["nodes"] for r in g["ranks"]]
    halos = [maps.halo_plan(q, P, lists) if P > 1 else None for q in range(P)]
    plans = []
    for q, r in enumerate(g["ranks"]):
        pl = splan.StepPlan(_K(r), r["F"], r["lM"], r["dirichlet"], g["dt"], float(g["alpha"]), halo=halos[q], rank=q, size=P,
                            node_order=node_order)
        pl.set_matfree(*local_mesh(g, q), *_lame(g))
        plans.append(pl)
    grp = splan.PlanGroup(plans) if (P > 1 and group) else None
    return plans, grp, halos


def numpy_elements(pts, cells, d0, lmd, mu):
    """(sigma (nE,6), von Mises (nE,), V (nE,)) through the reference's B and D"""
    P = pts[cells]
    Jac = assembly._jacobians(P)
    detJ = np.linalg.det(Jac)
    N_xyz = assembly._D_XI @ np.linalg.inv(Jac)
    B = assembly._B_stack(N_xyz)                                   # (nE,4,6,3)
    U = np.asarray(d0, dtype=np.float64).reshape(-1, 3)[cells]      # (nE,4,3)
    eps = np.einsum("eaij,eaj->ei", B, U)
    sig = eps @ assembly.elasticity_D(lmd, mu).T
    return sig, vm_np(sig), detJ / 6.0


def vm_np(s):
    s = np.asarray(s)
    return np.sqrt(0.5 * ((s[..., 0] - s[..., 1]) ** 2 + (s[..., 1] - s[..., 2]) ** 2 + (s[..., 2] - s[..., 0]) ** 2)
                   + 3.0 * (s[..., 3] ** 2 + s[..., 4] ** 2 + s[..., 5] ** 2))


def voigt_sigma(G, lmd, mu):
    eps = np.array([G[0, 0], G[1, 1], G[2, 2], G[1, 2] + G[2, 1], G[0, 2] + G[2, 0], G[0, 1] + G[1, 0]])
    return assembly.elasticity_D(lmd, mu) @ eps


def max_err(a, b):
    return float(np.abs(np.asarray(a) - np.asarray(b)).max())


def elem_np(pl):
    return pl.element_stress().cpu().numpy()


# ---- 1. patch test ----------------------------------------------------------------------------------------------------
def _patch_cases():
    return ["beam_coarse_P1", "struct_m3_P1", "device_m8"]


def _patch_plan(name):
    if name == "device_m8":
        pl, info = device_setup.build_structured_rank(8, 0, 1, keep_mesh=True)
        pl.set_matfree(info["cells_loc"], info["pts"], *info["lame"])
        return pl, info["pts"].cpu().numpy(), info["lame"]
    g = load_golden(name)
    (pl,), _, _ = make_plans(g)
    return pl, local_mesh(g, 0)[1], _lame(g)


@pytest.mark.parametrize("name", _patch_cases())
def test_patch_test_linear_field_and_rigid_motion(name):
    pl, X, (lmd, mu) = _patch_plan(name)
    rng = np.random.default_rng(7)
    G, c = 1e-3 * rng.standard_normal((3, 3)), 1e-3 * rng.standard_normal(3)
    u = (X @ G.T + c).reshape(-1)
    pl.set_state(u, u, 0.0)
    want = voigt_sigma(G, lmd, mu)
    scale = np.abs(want).max()
    e = elem_np(pl)
    assert max_err(e[:, :6], want[None, :]) <= PATCH_REL * scale
    vm = float(vm_np(want))
    assert max_err(e[:, 6], vm) <= PATCH_REL * scale
    nod = stress.nodal_stress(pl.nodal_stress_partial()).cpu().numpy()
    assert nod.shape == (pl.n_dof // 3, 7)
    assert max_err(nod[:, :6], want[None, :]) <= PATCH_REL * scale
    assert max_err(nod[:, 6], vm) <= PATCH_REL * scale
    # rigid motion u = c + W x, W skew
    w = 1e-3 * rng.standard_normal(3)
    W = np.array([[0.0, -w[2], w[1]], [w[2], 0.0, -w[0]], [-w[1], w[0], 0.0]])
    u = (X @ W.T + c).reshape(-1)
    pl.set_state(u, u, 0.0)
    bound = PATCH_REL * (lmd + 2 * mu) * np.linalg.norm(W)
    e = elem_np(pl)
    assert np.abs(e[:, :7]).max() <= bound
    nod = stress.nodal_stress(pl.nodal_stress_partial()).cpu().numpy()
    assert np.abs(nod).max() <= bound


# ---- 2./3. against numpy and against LocalK d0 ------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["beam_coarse_P1", "struct_m3_P1"])
def test_element_stress_equals_numpy_and_ties_to_local_K(name):
    g = load_golden(name)
    (pl,), _, _ = make_plans(g)
    o = make_oracle(g)
    o.run(400)
    d0, dn, tn = o.state(0)
    pl.set_state(d0, dn, tn)
    e = elem_np(pl)
    cells, X = local_mesh(g, 0)
    lmd, mu = _lame(g)
    sig, vm, V = numpy_elements(X, cells, d0, lmd, mu)
    scale = np.abs(sig).max()
    assert scale > 0
    assert max_err(e[:, :6], sig) <= NUMPY_REL * scale
    assert max_err(e[:, 6], vm) <= NUMPY_REL * scale
    assert max_err(e[:, 7], V) <= NUMPY_REL * np.abs(V).max()
    # sum_e V_e B_e^T sigma_e == LocalK d0
    P = X[cells]
    B = assembly._B_stack(assembly._D_XI @ np.linalg.inv(assembly._jacobians(P)))
    fe = np.einsum("e,eaij,ei->eaj", e[:, 7], B, e[:, :6])          # (nE,4,3)
    f = np.zeros((X.shape[0], 3))
    np.add.at(f, cells, fe)
    K = _K(g["ranks"][0])
    ref = K @ d0
    scale_f = (abs(K) @ np.abs(d0)).max()
    assert max_err(f.reshape(-1), ref) <= NUMPY_REL * scale_f
    # the state is still the oracle's
    got0, gotn, gott = pl.get_state()
    assert bits_equal(got0, d0) and bits_equal(gotn, dn) and gott == tn


def volume_weighted_mean(X, cells, d0, lmd, mu):
    """numpy nodal stresses: sum_e V_e sigma_e / sum_e V_e over the elements at each node"""
    sig, _, V = numpy_elements(X, cells, d0, lmd, mu)
    acc = np.zeros((X.shape[0], 7))
    for a in range(4):
        np.add.at(acc, cells[:, a], np.hstack([V[:, None] * sig, V[:, None]]))
    return acc[:, :6] / acc[:, 6:7], V


@pytest.mark.parametrize("name", ["beam_coarse_P1", "beam_coarse_P3"])
def test_nodal_stress_equals_numpy_volume_weighted_mean(name):
    """element volumes of this mesh differ, so the weighting of the nodal mean is seen"""
    g = load_golden(name)
    plans, _, halos = make_plans(g)
    o = make_oracle(g)
    o.run(400)
    X, cells = np.asarray(g["points"], dtype=np.float64), np.asarray(g["cells"], dtype=np.int64)
    U = np.zeros_like(X)
    for q, pl in enumerate(plans):
        d0, dn, tn = o.state(q)
        pl.set_state(d0, dn, tn)
        U[np.asarray(g["ranks"][q]["nodes"])] = d0.reshape(-1, 3)
    want, V = volume_weighted_mean(X, cells, U.reshape(-1), *_lame(g))
    assert V.min() < 0.9 * V.max()
    plain = np.zeros((X.shape[0], 6))
    cnt = np.zeros(X.shape[0])
    sig, _, _ = numpy_elements(X, cells, U.reshape(-1), *_lame(g))
    for a in range(4):
        np.add.at(plain, cells[:, a], sig)
        np.add.at(cnt, cells[:, a], 1.0)
    scale = np.abs(want).max()
    assert max_err(plain / cnt[:, None], want) > 1e-6 * scale        # an unweighted mean would fail below
    out = stress.nodal_stress_in_process(plans, halos)
    for q in range(g["P"]):
        nodes = np.asarray(g["ranks"][q]["nodes"])
        got = out[q].cpu().numpy()
        assert max_err(got[:, :6], want[nodes]) <= NUMPY_REL * scale, q
        assert max_err(got[:, 6], vm_np(want[nodes])) <= NUMPY_REL * scale, q


# ---- 4. partition and layout invariance --------------------------------------------------------------------------------
@pytest.mark.parametrize("name,step", [("beam_coarse", 1000), ("struct_m3", 500)])
def test_element_and_nodal_stress_partition_and_layout_invariant(name, step):
    g1, g3 = load_golden(name + "_P1"), load_golden(name + "_P3")
    assert np.array_equal(g1["cells"], g3["cells"]) and np.array_equal(g1["points"], g3["points"])
    for r in g1["ranks"] + g3["ranks"]:
        assert np.all(np.diff(np.asarray(r["ele"])) > 0), "each rank's elements in ascending global order"
    n_glob = len(g1["points"])
    U = np.zeros((n_glob, 3))
    U[np.asarray(g1["ranks"][0]["nodes"])] = np.asarray(g1[f"hist_{step}_r0"]).reshape(-1, 3)

    def put(plans, g):
        for q, pl in enumerate(plans):
            u = U[np.asarray(g["ranks"][q]["nodes"])].reshape(-1)
            pl.set_state(u, np.zeros_like(u), 0.5)

    (p1,), _, _ = make_plans(g1)
    put([p1], g1)
    e1 = elem_np(p1)
    n1 = stress.nodal_stress(p1.nodal_stress_partial()).cpu().numpy()
    ele1 = np.asarray(g1["ranks"][0]["ele"])
    by_elem = np.empty_like(e1)
    by_elem[ele1] = e1
    nodes1 = np.asarray(g1["ranks"][0]["nodes"])
    by_node = np.empty_like(n1)
    by_node[nodes1] = n1

    # Morton order of the same single partition
    import torch
    order = device_setup.morton_node_order(torch.from_numpy(local_mesh(g1, 0)[1]))
    assert not np.array_equal(order, np.arange(order.size))
    (pm,), _, _ = make_plans(g1, node_order=order)
    put([pm], g1)
    assert bits_equal(elem_np(pm), e1)
    assert bits_equal(stress.nodal_stress(pm.nodal_stress_partial()).cpu().numpy(), n1)

    # three partitions, stepped as a group
    plans, grp, halos = make_plans(g3)
    put(plans, g3)
    out3 = stress.nodal_stress_in_process(plans, halos)
    scale = np.abs(n1[:, :6]).max()
    for q, pl in enumerate(plans):
        assert bits_equal(elem_np(pl), by_elem[np.asarray(g3["ranks"][q]["ele"])]), (name, q)
        nodes = np.asarray(g3["ranks"][q]["nodes"])
        got, want = out3[q].cpu().numpy(), by_node[nodes]
        shared = np.zeros(nodes.size, dtype=bool)
        shared[halos[q]["shared_pos"]] = True
        assert shared.any() and not shared.all()
        assert bits_equal(got[~shared], want[~shared]), (name, q)
        assert max_err(got[shared], want[shared]) <= 1e-14 * scale, (name, q)
    # the group still steps on: stress calls left the state and the group usable
    grp.step(3, splan.MODE_SYNC)
    grp.synchronize()


# ---- 5. nothing else changes -------------------------------------------------------------------------------------------
def _run_interleaved(g, with_stress, launches, energy):
    plans, grp, _ = make_plans(g)
    if energy:
        for pl in plans:
            pl.set_energy(200, 1)
    evals = []
    for n, launch in launches:
        if grp is None:
            plans[0].step(n, splan.MODE_LOCAL, launch)
        else:
            grp.step(n, splan.MODE_SYNC, launch)
        if with_stress:
            for pl in plans:
                e = pl.element_stress()
                evals.append((e.cpu().numpy(), pl.nodal_stress_partial(e).cpu().numpy()))
    for pl in plans:
        pl.synchronize()
    states = [pl.get_state() for pl in plans]
    recs = [pl.read_energy() for pl in plans] if energy else None
    return states, recs, evals


@pytest.mark.parametrize("name", ["beam_coarse_P1", "beam_coarse_P3"])
def test_stress_calls_change_no_state_bit_and_no_energy_record(name):
    g = load_golden(name)
    L = splan
    configs = [(True, [(5, L.LAUNCH_PER_STEP), (8, L.LAUNCH_GRAPH), (1, L.LAUNCH_PER_STEP), (6, L.LAUNCH_GRAPH)])]
    if g["P"] == 1:
        configs.append((False, [(5, L.LAUNCH_PERSISTENT), (8, L.LAUNCH_GRAPH), (7, L.LAUNCH_PERSISTENT)]))
    for energy, launches in configs:
        a_states, a_recs, evals = _run_interleaved(g, True, launches, energy)
        b_states, b_recs, _ = _run_interleaved(g, False, launches, energy)
        assert len(evals) == len(launches) * g["P"]
        for (a0, an, at), (b0, bn, bt) in zip(a_states, b_states):
            assert bits_equal(a0, b0) and bits_equal(an, bn) and at == bt, (name, energy)
        if energy:
            for ra, rb in zip(a_recs, b_recs):
                for f in splan.ENERGY_FIELDS:
                    assert np.array_equal(ra[f], rb[f]), (name, f)


def test_repeated_evaluation_bit_identical_and_after_matrix_release():
    g = load_golden("struct_m3_P1")
    (pl,), _, _ = make_plans(g)
    pl.step(150, splan.MODE_LOCAL)
    pl.synchronize()
    e1, e2 = elem_np(pl), elem_np(pl)
    assert bits_equal(e1, e2)
    n1, n2 = pl.nodal_stress_partial().cpu().numpy(), pl.nodal_stress_partial().cpu().numpy()
    assert bits_equal(n1, n2)
    import torch
    out = torch.empty((pl.n_elem, 8), dtype=torch.float64, device="cuda")
    assert pl.element_stress(out=out) is out and bits_equal(out.cpu().numpy(), e1)
    pl.set_option(splan.OPT_MATFREE, 2)
    assert bits_equal(elem_np(pl), e1)
    assert bits_equal(pl.nodal_stress_partial().cpu().numpy(), n1)
    d0 = pl.d0()
    pl.step(10, splan.MODE_LOCAL)                    # the matrix-free step runs on, and stress follows the new d0
    pl.synchronize()
    assert not bits_equal(pl.d0(), d0)
    cells, X = local_mesh(g, 0)
    sig, _, _ = numpy_elements(X, cells, pl.d0(), *_lame(g))
    assert max_err(elem_np(pl)[:, :6], sig) <= NUMPY_REL * np.abs(sig).max()


# ---- 6. device set-up path --------------------------------------------------------------------------------------------
def test_device_setup_m24_against_numpy_sample():
    pl, info = device_setup.build_structured_rank(24, 0, 1, keep_mesh=True)
    pl.set_matfree(info["cells_loc"], info["pts"], *info["lame"])
    pl.step(200, splan.MODE_LOCAL)
    pl.synchronize()
    e = pl.element_stress()
    nod = stress.nodal_stress(pl.nodal_stress_partial(e)).cpu().numpy()
    e = e.cpu().numpy()
    d0 = pl.d0()
    cells = info["cells_loc"].cpu().numpy().astype(np.int64)
    X = info["pts"].cpu().numpy()
    lmd, mu = info["lame"]
    rng = np.random.default_rng(11)
    sel = np.sort(rng.choice(cells.shape[0], 10_000, replace=False))
    sig, vm, V = numpy_elements(X, cells[sel], d0, lmd, mu)
    scale = np.abs(sig).max()
    assert scale > 0
    assert max_err(e[sel, :6], sig) <= NUMPY_REL * scale
    assert max_err(e[sel, 6], vm) <= NUMPY_REL * scale
    assert max_err(e[sel, 7], V) <= NUMPY_REL * np.abs(V).max()
    # nodes of the sampled elements: volume-weighted mean over all their elements, in numpy
    nodes = rng.choice(np.unique(cells[sel]), 2000, replace=False)
    mask = np.zeros(X.shape[0], dtype=bool)
    mask[nodes] = True
    inc = np.nonzero(mask[cells].any(1))[0]
    s_i, _, V_i = numpy_elements(X, cells[inc], d0, lmd, mu)
    acc = np.zeros((X.shape[0], 7))
    for a in range(4):
        np.add.at(acc, cells[inc, a], np.hstack([V_i[:, None] * s_i, V_i[:, None]]))
    want = acc[nodes, :6] / acc[nodes, 6:7]
    assert max_err(nod[nodes, :6], want) <= NUMPY_REL * scale
    assert max_err(nod[nodes, 6], vm_np(want)) <= NUMPY_REL * scale


# ---- 7. refusals -------------------------------------------------------------------------------------------------------
def test_refusals():
    g = load_golden("beam_coarse_P1")
    r = g["ranks"][0]
    pl = splan.StepPlan(_K(r), r["F"], r["lM"], r["dirichlet"], g["dt"], float(g["alpha"]))
    with pytest.raises(splan.SaaError, match="saa_plan_set_matfree_dev"):
        pl.element_stress()
    with pytest.raises(splan.SaaError, match="saa_plan_set_matfree_dev"):
        pl.nodal_stress_partial()
    # a plan that is not finalised
    L = splan.lib()
    K = _K(r)
    ip, ix, dv = (np.ascontiguousarray(a) for a in (K.indptr.astype(np.int32), K.indices.astype(np.int32), K.data))
    F, M, D = (np.ascontiguousarray(a, dtype=t) for a, t in ((r["F"], np.float64), (r["lM"], np.float64), (r["dirichlet"], np.int64)))
    h = ctypes.c_void_p()
    splan._check(L.saa_plan_create(ctypes.byref(h), 0, F.size, splan._p(ip), splan._p(ix), splan._p(dv), splan._p(F), splan._p(M),
                                   splan._p(D), D.size, *splan.step_scalars(g["dt"], float(g["alpha"]))), "saa_plan_create")
    import torch
    buf = torch.empty((len(r["ele"]), 8), dtype=torch.float64, device="cuda")
    try:
        with pytest.raises(splan.SaaError, match="not finalized"):
            splan._check(L.saa_plan_element_stress_dev(h, buf.data_ptr()), "saa_plan_element_stress_dev")
        with pytest.raises(splan.SaaError, match="not finalized"):
            splan._check(L.saa_plan_nodal_stress_dev(h, buf.data_ptr(), buf.data_ptr()), "saa_plan_nodal_stress_dev")
    finally:
        L.saa_plan_destroy(h)
    # one inverted element (two corners swapped): reported by index, no NaN handed out
    cells, X = local_mesh(g, 0)
    bad = cells.copy()
    bad[37, [1, 2]] = bad[37, [2, 1]]
    pl.set_matfree(bad, X, *_lame(g))
    with pytest.raises(splan.SaaError, match=r"element 37 .*detJ <= 0"):
        pl.element_stress()
    # a valid plan evaluates normally afterwards, and the steps are unaffected
    (ok,), _, _ = make_plans(g)
    ok.step(20, splan.MODE_LOCAL)
    assert np.isfinite(elem_np(ok)).all()
    # size > 1 without a halo
    part = ok.nodal_stress_partial()
    with pytest.raises(splan.SaaError, match="halo"):
        stress.nodal_stress(part, size=3)
    with pytest.raises(splan.SaaError, match="halo"):
        stress.nodal_stress_in_process([ok, ok])


# ---- 8. one process per rank -------------------------------------------------------------------------------------------
def test_gather_nodal_stress_two_processes_equals_in_process():
    import subprocess
    port = 29550 + os.getpid() % 150
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "stress_dist_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count("stress ok") == 2
