"""Plane-masked matrix layout: value planes that are zero in every lane of a slice are not stored, and the step kernels
put 0.0 in their registers instead.  Every case builds the same plan twice, once with all nine planes of every block
(SAA_PLANE_MASK=0) and once with the default masked layout, runs the same steps and compares the states bit for bit."""
import numpy as np
import pytest
import scipy.sparse as sp

import saa_b200  # noqa: F401
from saa_b200 import device_setup as ds, maps, mesh, plan as splan
from util import bits_equal, load_golden

pytestmark = pytest.mark.gpu


def _both(monkeypatch, build):
    """build() under the full-plane layout and under the masked one"""
    monkeypatch.setenv("SAA_PLANE_MASK", "0")
    full = build()
    monkeypatch.delenv("SAA_PLANE_MASK")
    return full, build()


def _state(pl):
    d0, dn, tn = pl.get_state()
    return d0, dn, tn


def _same_states(plans_a, plans_b):
    for a, b in zip(plans_a, plans_b):
        a0, an, atn = _state(a)
        b0, bn, btn = _state(b)
        assert bits_equal(a0, b0) and bits_equal(an, bn) and atn == btn
        assert np.abs(a0).max() > 0


def _golden_plans(name):
    g = load_golden(name)
    P = g["P"]
    lists = [r["nodes"] for r in g["ranks"]]
    plans = []
    for q, r in enumerate(g["ranks"]):
        n = r["F"].size
        K = sp.csr_matrix((r["K_data"], r["K_indices"], r["K_indptr"]), shape=(n, n))
        plans.append(splan.StepPlan(K, r["F"], r["lM"], r["dirichlet"], g["dt"], float(g["alpha"]), rank=q, size=P,
                                    halo=maps.halo_plan(q, P, lists) if P > 1 else None))
    return plans


def _run(plans, n, mode=splan.MODE_SYNC, launch=splan.LAUNCH_AUTO):
    if len(plans) > 1:
        grp = splan.PlanGroup(plans)
        grp.step(n, mode, launch)
        grp.synchronize()
    else:
        plans[0].step(n, splan.MODE_LOCAL, launch)
        plans[0].synchronize()


def test_structured_device_plan_same_bits_fewer_bytes(monkeypatch):
    """m = 24 through the device set-up, 200 local steps; the masked plan streams 256 B less per plane it drops."""
    (full, _), (masked, _) = _both(monkeypatch, lambda: ds.build_structured_in_process(24, 1))
    full, masked = full[0], masked[0]
    assert full.padded_entries == masked.padded_entries
    assert full.value_planes == full.padded_entries // 32
    assert 0 < masked.value_planes < full.value_planes
    dropped = full.value_planes - masked.value_planes
    assert full.matrix_bytes - masked.matrix_bytes == 256 * dropped
    # the stencil of the axis-aligned beam leaves whole planes zero in every lane of a slice
    assert masked.value_planes / full.value_planes < 0.95
    for pl in (full, masked):
        pl.step(200, splan.MODE_LOCAL)
        pl.synchronize()
    _same_states([full], [masked])


@pytest.mark.parametrize("name", ["beam_coarse_P1", "beam_coarse_P3"])
def test_host_assembled_fixtures_same_bits(monkeypatch, name):
    """The reference's matrices (host finalisation; BLAS residues leave few exact zeros) under the group transport:
    boundary slices (K2), shared-row update (K3) and interior; both layouts equal the golden history."""
    g = load_golden(name)
    full, masked = _both(monkeypatch, lambda: _golden_plans(name))
    for plans in (full, masked):
        done = 0
        for n in [int(s) for s in g["steps"]][:5]:
            _run(plans, n - done)
            done = n
            for q, pl in enumerate(plans):
                assert bits_equal(pl.d0(), g[f"hist_{n}_r{q}"])
    _same_states(full, masked)


def test_morton_ordered_mesh_plan_same_bits(monkeypatch):
    pts, cells, fac = mesh.structured_beam(5, length=6)
    epart = np.zeros(len(cells), dtype=np.int64)
    (full, _), (masked, _) = _both(monkeypatch, lambda: ds.build_mesh_rank(pts, cells, fac, epart, 0, 1))
    for pl in (full, masked):
        pl.step(150, splan.MODE_LOCAL)
        pl.synchronize()
    _same_states([full], [masked])


def test_three_partitions_synchronised_same_bits(monkeypatch):
    (full, _), (masked, _) = _both(monkeypatch, lambda: ds.build_structured_in_process(6, 3))
    assert sum(a.value_planes for a in full) > sum(b.value_planes for b in masked)
    for plans in (full, masked):
        _run(plans, 120)
    _same_states(full, masked)


def test_persistent_loop_same_bits(monkeypatch):
    (full, _), (masked, _) = _both(monkeypatch, lambda: ds.build_structured_in_process(8, 1))
    for pl in (full[0], masked[0]):
        pl.step(301, splan.MODE_LOCAL, splan.LAUNCH_PERSISTENT)
        pl.synchronize()
    _same_states(full, masked)
    ref = ds.build_structured_in_process(8, 1)[0][0]            # masked, graph launches
    ref.step(301, splan.MODE_LOCAL)
    ref.synchronize()
    _same_states([ref], masked)


def test_pipelined_host_call_same_bits(monkeypatch):
    monkeypatch.setenv("SAA_STEP_HOST_PIPELINE", "5")
    (full, info), (masked, _) = _both(monkeypatch, lambda: ds.build_structured_in_process(10, 1))
    full, masked, dt = full[0], masked[0], info[0]["dt"]
    out = []
    for pl in (full, masked):
        d_0, d_n, tn = np.zeros(pl.n_dof), np.zeros(pl.n_dof), 0.0
        for _ in range(40):
            d1 = pl.step_host(d_0, d_n, tn, splan.MODE_LOCAL)
            d_n, d_0, tn = d_0, d1, tn + dt
        out.append((d_0.copy(), d_n.copy()))
    assert pl.host_pipe_info(splan.MODE_LOCAL)[0] == 5
    assert bits_equal(out[0][0], out[1][0]) and bits_equal(out[0][1], out[1][1]) and np.abs(out[0][0]).max() > 0


def _with_full_blocks(K):
    """K with every 3x3 node block that holds an entry completed by explicitly stored zeros"""
    c = K.tocoo()
    pairs = np.unique(np.stack([c.row // 3, c.col // 3], 1), axis=0)
    a, b = np.meshgrid(np.arange(3), np.arange(3), indexing="ij")
    rows = (3 * pairs[:, :1] + a.reshape(1, -1)).reshape(-1)
    cols = (3 * pairs[:, 1:] + b.reshape(1, -1)).reshape(-1)
    order = np.lexsort((cols, rows))
    rows, cols = rows[order], cols[order]
    data = np.asarray(K[rows, cols]).reshape(-1)
    indptr = np.searchsorted(rows, np.arange(K.shape[0] + 1))
    Kf = sp.csr_matrix((data, cols, indptr), shape=K.shape)
    assert Kf.nnz == 9 * len(pairs) and Kf.nnz > K.nnz and np.count_nonzero(Kf.data) == K.nnz
    return Kf


def test_explicitly_stored_zeros_keep_their_planes():
    """The mask follows the stored pattern, not the value bits: a matrix whose blocks are completed by stored zeros
    keeps every plane, and gives the bits of the matrix without them (adding 0.0*x leaves the row sums unchanged)."""
    g = load_golden("beam_coarse_P1")
    r = g["ranks"][0]
    n = r["F"].size
    K = sp.csr_matrix((r["K_data"], r["K_indices"], r["K_indptr"]), shape=(n, n))
    plans = [splan.StepPlan(M, r["F"], r["lM"], r["dirichlet"], g["dt"], float(g["alpha"])) for M in (K, _with_full_blocks(K))]
    assert plans[1].value_planes == plans[1].padded_entries // 32
    assert plans[0].value_planes <= plans[1].value_planes
    for pl in plans:
        pl.step(300, splan.MODE_LOCAL)
        pl.synchronize()
    _same_states(plans[:1], plans[1:])
