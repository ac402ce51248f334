"""Value coding of the plane-masked layout (DESIGN.md §3): a block-row whose stored planes each span at most 65535
between the smallest and the largest bit pattern of their 32 lanes (read as int64) is stored as one int64 base per
plane plus 32 16-bit lane offsets, and the readers decode base + offset with integer arithmetic.  The coding is
lossless on the bits, so every case compares the coded layout with SAA_VALUE_CODE=0 (all block-rows raw) or with the
reference's arithmetic, bit for bit, and the byte counters with a Python model of the layout."""
import numpy as np
import pytest
import scipy.sparse as sp

import saa_b200  # noqa: F401
from saa_b200 import device_setup as ds, maps, plan as splan
from util import bits_equal, load_golden
from test_gpu_format_conformance import SIGMA, check_plan, device_plan, host_plan, make_problem, references

pytestmark = pytest.mark.gpu

SPAN = 65535


def _both(monkeypatch, build):
    """build() with every block-row raw and with the default coded layout"""
    monkeypatch.setenv("SAA_VALUE_CODE", "0")
    raw = build()
    monkeypatch.delenv("SAA_VALUE_CODE")
    return raw, build()


def _same_states(plans_a, plans_b):
    for a, b in zip(plans_a, plans_b):
        a0, an, atn = a.get_state()
        b0, bn, btn = b.get_state()
        assert bits_equal(a0, b0) and bits_equal(an, bn) and atn == btn
        assert np.abs(a0).max() > 0


def _run(plans, n, launch=splan.LAUNCH_AUTO):
    if len(plans) > 1:
        grp = splan.PlanGroup(plans)
        grp.step(n, splan.MODE_SYNC, launch)
        grp.synchronize()
    else:
        plans[0].step(n, splan.MODE_LOCAL, launch)
        plans[0].synchronize()


# ---- the coded layout, from DESIGN.md §3 ---------------------------------------------------------------------------
def coded_model(K):
    """value_planes, coded_planes and streamed_matrix_bytes of the coded layout of K (single partition, no node order)"""
    n = K.shape[0]
    nn = n // 3
    r = np.repeat(np.arange(n), np.diff(K.indptr))
    c = K.indices.astype(np.int64)
    key, inv = np.unique((r // 3) * nn + c // 3, return_inverse=True)          # node blocks, ascending per node
    vals = np.zeros((key.size, 9))
    vals[inv, 3 * (r % 3) + c % 3] = K.data
    bits = np.zeros(key.size, dtype=np.int64)
    np.bitwise_or.at(bits, inv, 1 << (3 * (r % 3) + c % 3))
    nblk = np.bincount(key // nn, minlength=nn)
    first = np.concatenate([[0], np.cumsum(nblk)])
    # windows of SIGMA nodes sorted by decreasing block count (stable), padded to 32
    order = np.lexsort((-nblk, np.arange(nn) // SIGMA))
    slots = np.concatenate([order, -np.ones(-nn % 32, dtype=np.int64)])
    lane_node = slots.reshape(-1, 32)
    lane_nblk = np.where(lane_node >= 0, nblk[np.maximum(lane_node, 0)], 0)
    L = lane_nblk.max(axis=1)
    s_of = np.repeat(np.arange(L.size), L)                                      # block-row -> slice
    j_of = np.arange(s_of.size) - np.repeat(np.cumsum(L) - L, L)                # block-row -> block index j
    valid = j_of[:, None] < lane_nblk[s_of]
    bid = np.where(valid, first[np.maximum(lane_node[s_of], 0)] + j_of[:, None], -1)
    mask = np.bitwise_or.reduce(np.where(valid, bits[np.maximum(bid, 0)], 0), axis=1)
    lv = np.where(valid[:, :, None], vals[np.maximum(bid, 0)], 0.0).view(np.int64)   # (block-rows, 32 lanes, 9)
    span = lv.max(axis=1).astype(np.uint64) - lv.min(axis=1).astype(np.uint64)
    stored = (mask[:, None] >> np.arange(9)) & 1 == 1
    code = (mask != 0) & np.all(~stored | (span <= SPAN), axis=1)
    planes = stored.sum(axis=1)
    value_planes, coded = int(planes.sum()), int(planes[code].sum())
    lanes, n_slices, n_rows = 32 * int(L.sum()), L.size, 3 * slots.size
    streamed = 256 * (value_planes - coded) + 72 * coded + 4 * lanes + 2 * (lanes // 32) + 24 * (n_slices + 1) + 4 * (n_rows // 32)
    return dict(value_planes=value_planes, coded_planes=coded, streamed_matrix_bytes=streamed)


def _counters(pl):
    return dict(value_planes=pl.value_planes, coded_planes=pl.coded_planes, streamed_matrix_bytes=pl.streamed_matrix_bytes)


def test_structured_device_plan_same_bits_fewer_bytes(monkeypatch):
    """m = 24 through the device set-up, 200 local steps; counters equal the model of the same CSR"""
    (raw, _), (coded, info) = _both(monkeypatch, lambda: ds.build_structured_in_process(24, 1, keep_csr=True))
    raw, coded, K = raw[0], coded[0], info[0]["K"].to_scipy()
    assert raw.coded_planes == 0 and raw.value_planes == coded.value_planes and raw.matrix_bytes == coded.matrix_bytes
    assert raw.streamed_matrix_bytes > raw.matrix_bytes            # only the per-slice base offsets on top
    assert _counters(coded) == coded_model(K)
    assert coded.coded_planes > 0.7 * coded.value_planes
    assert coded.streamed_matrix_bytes < 0.6 * coded.matrix_bytes
    for pl in (raw, coded):
        pl.step(200, splan.MODE_LOCAL)
        pl.synchronize()
    _same_states([raw], [coded])


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


@pytest.mark.parametrize("name", ["beam_coarse_P1", "beam_coarse_P3"])
def test_host_assembled_fixtures_same_bits(monkeypatch, name):
    """host finalisation, group transport (boundary slices, shared rows, interior): both layouts equal the golden history
    (the reference's unstructured matrices leave few block-rows within the coding span)"""
    g = load_golden(name)
    raw, coded = _both(monkeypatch, lambda: _golden_plans(name))
    for plans in (raw, coded):
        done = 0
        for n in [int(s) for s in g["steps"]][:5]:
            _run(plans, n - done)
            done = n
            for q, pl in enumerate(plans):
                assert bits_equal(pl.d0(), g[f"hist_{n}_r{q}"])
    _same_states(raw, coded)


def test_three_partitions_synchronised_same_bits(monkeypatch):
    raw, coded = _both(monkeypatch, lambda: ds.build_structured_in_process(6, 3)[0])
    assert all(p.coded_planes > 0 for p in coded)
    for plans in (raw, coded):
        _run(plans, 120)
    _same_states(raw, coded)


def test_persistent_loop_same_bits(monkeypatch):
    raw, coded = _both(monkeypatch, lambda: ds.build_structured_in_process(8, 1)[0][0])
    for pl in (raw, coded):
        pl.step(301, splan.MODE_LOCAL, splan.LAUNCH_PERSISTENT)
        pl.synchronize()
    _same_states([raw], [coded])


def test_pipelined_host_call_same_bits(monkeypatch):
    monkeypatch.setenv("SAA_STEP_HOST_PIPELINE", "5")
    (raw, info), (coded, _) = _both(monkeypatch, lambda: ds.build_structured_in_process(10, 1))
    raw, coded, dt = raw[0], coded[0], info[0]["dt"]
    out = []
    for pl in (raw, coded):
        d_0, d_n, tn = np.zeros(pl.n_dof), np.zeros(pl.n_dof), 0.0
        for _ in range(40):
            d1 = pl.step_host(d_0, d_n, tn, splan.MODE_LOCAL)
            d_n, d_0, tn = d_0, d1, tn + dt
        out.append((d_0.copy(), d_n.copy()))
    assert coded.host_pipe_info(splan.MODE_LOCAL)[0] == 5
    assert bits_equal(out[0][0], out[1][0]) and bits_equal(out[0][1], out[1][1]) and np.abs(out[0][0]).max() > 0


def test_static_solve_and_energy_same_bits(monkeypatch):
    """block-Jacobi CG (the diagonal blocks come from the coded planes) and the energy records of the armed step"""
    import torch
    raw, coded = _both(monkeypatch, lambda: ds.build_structured_in_process(8, 1)[0][0])
    assert coded.coded_planes > 0
    res = [pl.solve_static(rtol=1e-9) for pl in (raw, coded)]
    assert res[0].converged and res[0].iterations == res[1].iterations
    assert bits_equal(res[0].x.cpu().numpy(), res[1].x.cpu().numpy())
    x = torch.randn(raw.n_dof, dtype=torch.float64, device="cuda:0")
    assert bits_equal(raw.apply_stiffness(x).cpu().numpy(), coded.apply_stiffness(x).cpu().numpy())
    recs = []
    for pl in (raw, coded):
        pl.set_energy(60, 1)
        pl.step(60, splan.MODE_LOCAL)
        pl.synchronize()
        recs.append(pl.read_energy())
    assert recs[0].tobytes() == recs[1].tobytes() and len(recs[0]) == 60
    _same_states([raw], [coded])


# ---- the decision boundary on hand-built block-rows ------------------------------------------------------------------
def _from_bits(b):
    return np.asarray(b, dtype=np.int64).view(np.float64)


def _bits(x):
    return np.asarray(x, dtype=np.float64).view(np.int64)


def boundary_problem():
    """7 slices of one 3x3 block per node (the node's own); plane (0,1) of slice s is the case under test, the other
    planes span at most 31.  Coded: slices 0 (span exactly 65535), 4 (+0.0 and subnormals), 5 (-0.0 and negative
    subnormals).  Raw: 1 (span 65536), 2 (+0.0 and -0.0), 3 (sign change), 6 (28 nodes: padding lanes hold +0.0)."""
    nn = 6 * 32 + 28
    lane = np.arange(32)
    lo = _bits(1.0e3)
    cases = [lo + (lane * SPAN) // 31, lo + (lane * (SPAN + 1)) // 31,
             _bits(np.where(lane % 2 == 0, 0.0, -0.0)), _bits(np.where(lane % 2 == 0, 1e-3, -1e-3) * (1 + lane)),
             np.where(lane % 3 == 0, 0, lane), np.where(lane % 3 == 0, _bits(-0.0), _bits(-0.0) + lane)]
    rows, cols, data = [], [], []
    for e in range(nn):
        s, l = divmod(e, 32)
        for A in range(3):
            for B in range(3):
                if (A, B) == (0, 1):
                    v = _from_bits(cases[s][l] if s < 6 else _bits(1.0) + l)
                elif A == B:
                    v = _from_bits(_bits(2.0e3) + l)
                else:
                    v = _from_bits(_bits(-3.0e2) + (l % 7))
                rows.append(3 * e + A), cols.append(3 * e + B), data.append(v)
    n = 3 * nn
    K = sp.csr_matrix((np.array(data), (np.array(rows), np.array(cols))), shape=(n, n))
    K.sort_indices()
    assert K.nnz == 9 * nn                        # the stored zeros are kept
    rng = np.random.default_rng(11)
    return dict(K=K, F=rng.standard_normal(n), lM=1.0 + rng.random(n), dirichlet=np.array([4, 100], dtype=np.int64),
                dt=1e-3, alpha=0.3, d0=1e-3 * rng.standard_normal(n), dn=1e-3 * rng.standard_normal(n), tn0=0.5,
                rows=np.repeat(np.arange(n), np.diff(K.indptr)), cols=K.indices.astype(np.int64), vals=K.data,
                n_nodes=nn, family="value_coding_boundary")


@pytest.mark.parametrize("variant", [0, 1, 2, 3, 4, 5])
def test_decision_boundary_equals_reference(monkeypatch, variant):
    prob = boundary_problem()
    refs = references(prob)
    monkeypatch.setenv("SAA_KVARIANT", str(variant))
    monkeypatch.setenv("SAA_STEP_HOST_PIPELINE", "5")
    for setup in (host_plan, device_plan):
        pl = setup(prob)
        assert pl.value_planes == 7 * 9 and pl.coded_planes == 3 * 9, (setup.__name__, pl.coded_planes)
        assert _counters(pl) == coded_model(prob["K"])
        check_plan(pl, prob, refs, variant, (variant, setup.__name__))


@pytest.mark.parametrize("family", ["random", "planes", "zeros", "wide", "heavy"])
def test_host_and_device_set_up_same_layout(family):
    """the same CSR through both finalisation paths gives the same coding decision and counters"""
    prob = make_problem(1025, family)
    plans = [host_plan(prob), device_plan(prob)]
    assert _counters(plans[0]) == _counters(plans[1]) == coded_model(prob["K"])
    refs = references(prob)
    for pl in plans:
        pl.set_state(prob["d0"], prob["dn"], prob["tn0"])
        pl.step(1, splan.MODE_LOCAL, splan.LAUNCH_PER_STEP)
        pl.synchronize()
        st = pl.get_state()
        assert bits_equal(st[0], refs[1][0]) and bits_equal(st[1], refs[1][1])
