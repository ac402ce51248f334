"""Conformance of the plane-masked node-block sliced-ELL format (DESIGN.md §3) and of every kernel that reads it, on
synthetic matrices built to reach the format's edge cases rather than on FE stiffness matrices.

The FE matrices of the other tests have nearly full 3x3 blocks, a stored diagonal and one stencil per slice.  The
generator below makes single-partition problems whose slices mix lanes of very different block counts, with empty
node rows and empty slices, rows of one or two blocks (odd-length tails of the two-block pipelines), plane masks that
change from block-row to block-row with non-contiguous bits, a node whose three rows have disjoint column nodes, nodes
with hundreds of blocks, stored +0.0 / -0.0, unsymmetric values and values from 1e-200 to 1e+200 with subnormals.

Every schedule variant (SAA_KVARIANT 0-5 of saa_k_step, 6 = the cp.async kernel saa_k_step_stream), both layouts
(plane-masked, SAA_PLANE_MASK=0), both set-up paths (host StepPlan, StepPlan.from_device), every launch strategy,
with and without a node order, with the energy monitor armed and through the pipelined host call must give the
bits of the reference's arithmetic (DESIGN.md §2): scipy's csr_matvec plus the update of Dynamic_solver.py:17 in
Python's association (oracle/numpy_step.py), and independently the C oracle (oracle/fem_oracle.c).

Scope: finite states only.  With an inf in d0, a padding block or a plane that is not stored computes
0.0 * inf = NaN where csr_matvec skips the entry; the parity contract covers finite values, and so do these tests.
"""
import math
import os

import numpy as np
import pytest
import scipy.sparse as sp

import saa_b200  # noqa: F401
from saa_b200 import device_setup as ds, maps, mesh, plan as splan
from util import GOLDEN, bits_equal, load_golden, oracle_module

pytestmark = pytest.mark.gpu

FAMILIES = ("random", "heavy", "empty", "planes", "zeros", "unsym", "wide")
LADDER = (1, 31, 32, 33, 1023, 1024, 1025, 2049)      # around the 32-node slice and the 1024-node sorting window
VARIANTS = (0, 1, 2, 3, 4, 5, 6)
NSTEPS = 50
SIGMA = 1024
# per family: (one mass value per node, alpha, tn of the initial state) — every family crosses some other combination;
# tn = 0.99 crosses the end of the ramp (tn = 1) inside the 50 steps
KNOBS = {"random": (True, 0.0, 0.25), "heavy": (False, 0.5, 3.0), "empty": (True, 0.7, 0.99), "planes": (False, 0.0, 1.5),
         "zeros": (True, 0.3, 0.0), "unsym": (False, 0.0, 0.5), "wide": (False, 0.5, 2.0)}
DT = 1e-3


# ---- synthetic problems ---------------------------------------------------------------------------------------
def _block_counts(rng, nn, family):
    if family == "heavy":                             # most nodes 0-3 blocks, a few 100-300
        cnt = rng.integers(0, 4, nn)
        few = rng.choice(nn, size=max(1, nn // 150), replace=False)
        cnt[few] = rng.integers(100, 301, few.size)
    elif family == "empty":                           # empty node rows (whole empty slices), rows of 1 or 2 blocks
        cnt = rng.choice([0, 0, 0, 1, 2, 2, 3, 7], nn)
    else:
        cnt = rng.integers(1, 14, nn)
    return np.minimum(cnt, nn)


def _block_masks(rng, nb, family):
    """3x3 stored pattern of nb blocks as 9-bit masks (bit 3A+B = entry (A,B))"""
    if family == "planes":                            # one stored plane, alternating patterns, or full
        choice = rng.integers(0, 4, nb)
        single = 1 << rng.integers(0, 9, nb)
        return np.where(choice == 0, single, np.where(choice == 1, 0b101010101, np.where(choice == 2, 0b010101010, 0x1FF)))
    keep = rng.random((nb, 9)) < 0.6                  # every entry dropped independently
    return (keep * (1 << np.arange(9))).sum(1)


def make_problem(n_nodes, family, seed=0):
    """Seeded single-partition problem: scipy CSR (sorted, duplicate-free indices) K, load F, lumped mass lM, Dirichlet
    DOFs, dt, alpha, initial state (d0, dn, tn0) and the generator's own entry list (rows, cols, vals)."""
    rng = np.random.default_rng([seed, n_nodes, FAMILIES.index(family)])
    nn, n = n_nodes, 3 * n_nodes
    cnt = _block_counts(rng, nn, family)
    rows, cols = [], []
    disjoint = int(rng.integers(0, nn)) if family == "empty" else -1
    for e in range(nn):
        cn = np.sort(rng.choice(nn, size=int(cnt[e]), replace=False))
        m = _block_masks(rng, cn.size, family)
        if e == disjoint:                             # the three rows of this node reach disjoint column nodes
            m = np.array([0b111 << (3 * (j % 3)) for j in range(cn.size)], dtype=np.int64)
        for c, mk in zip(cn, m):
            for k in range(9):
                if (int(mk) >> k) & 1:
                    rows.append(3 * e + k // 3)
                    cols.append(3 * c + k % 3)
    if not rows:                                      # keep nnz >= 1 (the device path takes raw pointers)
        rows, cols = [0], [0]
    r, c = np.asarray(rows, dtype=np.int64), np.asarray(cols, dtype=np.int64)
    v = rng.uniform(-1.0, 1.0, r.size)
    if family == "random":                            # symmetric pattern and values
        up = r <= c
        r, c, v = np.concatenate([r[up], c[up & (r != c)]]), np.concatenate([c[up], r[up & (r != c)]]), \
            np.concatenate([v[up], v[up & (r != c)]])
    if family == "zeros":                             # explicitly stored +0.0 and -0.0
        z = rng.random(r.size)
        v[z < 0.2] = 0.0
        v[(z >= 0.2) & (z < 0.4)] = -0.0
    row_scale = np.ones(n)
    if family == "wide":                              # rows scaled over 1e-200 .. 1e+200, entries over 20 decades, subnormals
        row_scale = 10.0 ** rng.uniform(-200, 200, n)
        v = np.sign(v) * 10.0 ** rng.uniform(-20, 0, r.size) * row_scale[r]
        sub = rng.random(r.size) < 0.05
        v[sub] = rng.integers(1, 1 << 40, int(sub.sum())) * 5e-324 * np.sign(rng.uniform(-1, 1, int(sub.sum())))
    key, first = np.unique(r * n + c, return_index=True)
    r, c, v = key // n, key % n, v[first]
    indptr = np.concatenate([[0], np.cumsum(np.bincount(r, minlength=n))]).astype(np.int32)
    K = sp.csr_matrix((v, c.astype(np.int32), indptr), shape=(n, n))
    assert K.nnz == v.size and K.has_sorted_indices

    mass_node, alpha, tn0 = KNOBS[family]
    # lumped mass large enough against dt^2 |K| that 50 steps stay finite and bounded
    rowsum = np.bincount(r, weights=np.abs(v), minlength=n)
    lM = rowsum * DT ** 2 * 50.0 + row_scale * rng.uniform(0.5, 1.5, n)
    if mass_node:                                     # identical bits on the three DOFs of a node: the node-mass stream
        lM = np.repeat(lM.reshape(-1, 3).max(1), 3)
    F = rng.uniform(-1.0, 1.0, n) * row_scale
    F[rng.random(n) < 0.1] = 0.0
    dnodes = rng.choice(nn, size=nn // 30, replace=False)
    dirichlet = np.unique(np.concatenate([rng.choice(n, size=n // 20, replace=False),
                                          (3 * dnodes[:, None] + np.arange(3)).reshape(-1)])).astype(np.int64)
    d0, dn = rng.uniform(-1.0, 1.0, n), rng.uniform(-1.0, 1.0, n)
    for d in (d0, dn):
        z = rng.random(n)
        d[z < 0.03] = 0.0
        d[(z >= 0.03) & (z < 0.05)] = -0.0
    return dict(K=K, F=F, lM=lM, dirichlet=dirichlet, dt=DT, alpha=alpha, d0=d0, dn=dn, tn0=tn0,
                rows=r, cols=c, vals=v, n_nodes=nn, family=family)


# ---- the reference ----------------------------------------------------------------------------------------------
def _numpy_step():
    oracle_module()                                   # puts oracle/ on sys.path
    import numpy_step
    return numpy_step


def reference(prob, n_steps, d0=None, dn=None, tn=None):
    """(d0, dn, tn) after n_steps of the reference's statement sequence (oracle/numpy_step.py, size 1)"""
    ns = _numpy_step()
    d0 = prob["d0"] if d0 is None else d0
    dn = prob["dn"] if dn is None else dn
    tn = prob["tn0"] if tn is None else tn
    dt = np.float64(prob["dt"])
    for _ in range(n_steps):
        d1 = ns.step(None, prob["K"], prob["F"], None, None, prob["dirichlet"], tn, dt, d0, dn, prob["lM"],
                     prob["alpha"], 1, 0)
        dn, d0, tn = d0, d1, tn + dt
    return d0, dn, tn


def oracle_c(prob, n_steps):
    """the same steps through oracle/fem_oracle.c with the identity node list"""
    K = prob["K"]
    o = oracle_module().OracleProblem(prob["n_nodes"], [dict(K_indptr=K.indptr, K_indices=K.indices, K_data=K.data,
                                                             F=prob["F"], lM=prob["lM"], dirichlet=prob["dirichlet"],
                                                             nodes=np.arange(prob["n_nodes"]))], prob["dt"], prob["alpha"])
    o.set_state(0, prob["d0"], prob["dn"], prob["tn0"])
    o.run(n_steps)
    return o.state(0)


_REF = {}


def references(prob):
    """{1: state, NSTEPS: state}, each checked against the C oracle, and the row sums against math.fsum"""
    key = (prob["family"], prob["n_nodes"])
    if key not in _REF:
        x = prob["d0"]
        y = prob["K"].dot(x)
        prods = prob["vals"] * x[prob["cols"]]
        bounds = np.concatenate([[0], np.cumsum(np.bincount(prob["rows"], minlength=x.size))])
        for i in range(x.size):
            p = prods[bounds[i]:bounds[i + 1]]
            exact = math.fsum(p)
            assert abs(y[i] - exact) <= p.size * np.finfo(float).eps * np.abs(p).sum(), (key, i)
        out = {}
        for k in (1, NSTEPS):
            st = reference(prob, k)
            assert np.all(np.isfinite(st[0])) and np.all(np.isfinite(st[1])), key
            oc = oracle_c(prob, k)
            assert bits_equal(st[0], oc[0]) and bits_equal(st[1], oc[1]) and st[2] == oc[2], (key, k)
            out[k] = st
        _REF[key] = out
    return _REF[key]


# ---- the layout, from DESIGN.md §3 -----------------------------------------------------------------------------
def layout_model(K, shared=(), node_order=None, full=False):
    """padded_entries, value_planes and matrix_bytes of the plane-masked node-block sliced ELL of K: shared nodes
    first (in the given order), then the others in node_order; inside windows of 1024 nodes a stable sort by
    decreasing block count; each region padded to 32 nodes.  A slice is as long as its longest lane; the plane
    mask of a block-row is the union of the stored patterns of its 32 lanes (all nine planes when full)."""
    n = K.shape[0]
    nn = n // 3
    r = np.repeat(np.arange(n), np.diff(K.indptr))
    c = K.indices.astype(np.int64)
    key, inv = np.unique((r // 3) * nn + c // 3, return_inverse=True)          # node blocks, ascending per node
    bits = np.zeros(key.size, dtype=np.int64)
    np.bitwise_or.at(bits, inv, 1 << (3 * (r % 3) + c % 3))
    owner = key // nn
    nblk = np.bincount(owner, minlength=nn)
    first = np.concatenate([[0], np.cumsum(nblk)])

    def region(nodes):
        nodes = list(nodes)
        for w in range(0, len(nodes), SIGMA):
            nodes[w:w + SIGMA] = sorted(nodes[w:w + SIGMA], key=lambda e: -nblk[e])    # sorted() is stable
        return nodes + [-1] * (-len(nodes) % 32)

    shared = [int(e) for e in shared]
    is_sh = np.zeros(nn, dtype=bool)
    is_sh[shared] = True
    rest = [int(e) for e in (range(nn) if node_order is None else node_order) if not is_sh[e]]
    slots = region(shared) + region(rest)
    lanes = planes = 0
    for s in range(len(slots) // 32):
        lane_nodes = [e for e in slots[32 * s:32 * s + 32] if e >= 0]
        L = max([nblk[e] for e in lane_nodes], default=0)
        lanes += 32 * L
        for j in range(L):
            m = 0x1FF if full else 0
            for e in lane_nodes:
                if j < nblk[e]:
                    m |= int(bits[first[e] + j])
            planes += bin(m).count("1")
    n_slices = len(slots) // 32
    n_rows = 3 * len(slots)
    return dict(padded_entries=9 * lanes, value_planes=planes,
                matrix_bytes=256 * planes + 4 * lanes + 2 * (lanes // 32) + 16 * (n_slices + 1) + 4 * (n_rows // 32))


def assert_layout(pl, K, variant, plane_mask, node_order=None, shared=()):
    full = plane_mask == "0" or variant == 6         # the cp.async kernel always gets all nine planes
    want = layout_model(K, shared, node_order, full)
    got = dict(padded_entries=pl.padded_entries, value_planes=pl.value_planes, matrix_bytes=pl.matrix_bytes)
    assert got == want, (variant, plane_mask, got, want)


# ---- plans ------------------------------------------------------------------------------------------------------
def host_plan(prob, node_order=None):
    return splan.StepPlan(prob["K"], prob["F"], prob["lM"], prob["dirichlet"], prob["dt"], prob["alpha"],
                          node_order=node_order)


def device_plan(prob, node_order=None, indptr=None, indices=None):
    """StepPlan.from_device on the same CSR uploaded with torch (int64 indptr, int32 indices)"""
    import torch
    K = prob["K"]
    dev = torch.device("cuda", 0)
    t = [torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(dev) for a, dt in
         ((K.indptr if indptr is None else indptr, np.int64), (K.indices if indices is None else indices, np.int32),
          (K.data, np.float64), (prob["F"], np.float64), (prob["lM"], np.float64))]
    torch.cuda.synchronize(dev)
    return splan.StepPlan.from_device(K.shape[0], *[x.data_ptr() for x in t], prob["dirichlet"], prob["dt"],
                                      prob["alpha"], node_order=node_order)


def _same_state(got, want, what):
    assert bits_equal(got[0], want[0]) and bits_equal(got[1], want[1]) and got[2] == want[2], what


def check_plan(pl, prob, refs, variant, what):
    """every launch strategy, the energy monitor and the pipelined host call against the reference"""
    start = (prob["d0"], prob["dn"], prob["tn0"])
    for launch, k in ((splan.LAUNCH_PER_STEP, 1), (splan.LAUNCH_PER_STEP, NSTEPS), (splan.LAUNCH_GRAPH, NSTEPS),
                      (splan.LAUNCH_PERSISTENT, NSTEPS)):
        pl.set_state(*start)
        pl.step(k, splan.MODE_LOCAL, launch)
        pl.synchronize()
        _same_state(pl.get_state(), refs[k], (what, "launch", launch, k))
    # energy monitor armed: the step runs as K1E, same d bits
    pl.set_state(*start)
    pl.set_energy(NSTEPS, 1)
    pl.step(NSTEPS, splan.MODE_LOCAL, splan.LAUNCH_GRAPH)
    pl.synchronize()
    _same_state(pl.get_state(), refs[NSTEPS], (what, "energy"))
    assert pl.energy_count == NSTEPS
    rec = pl.read_energy()
    pl.set_energy(0)
    # the reference's loop over the host call, pipelined in 5 chunks (the cp.async variant has no pipelined form)
    if variant < 6:
        d_0, d_n, tn = prob["d0"].copy(), prob["dn"].copy(), prob["tn0"]
        for _ in range(NSTEPS):
            d1 = pl.step_host(d_0, d_n, tn, splan.MODE_LOCAL)
            d_n, d_0, tn = d_0, d1, tn + np.float64(prob["dt"])
        _same_state((d_0, d_n, tn), refs[NSTEPS], (what, "step_host"))
        if prob["n_nodes"] >= 5:
            assert pl.host_pipe_info(splan.MODE_LOCAL)[0] == 5
    return rec


PATHS = [(v, f, s) for v in VARIANTS for f in FAMILIES for s in (33, 1025)] + \
        [(v, f, s) for v in (5, 6) for f in ("empty", "heavy") for s in LADDER if s not in (33, 1025)]


@pytest.mark.parametrize("variant,family,n_nodes", PATHS)
def test_path_matrix(monkeypatch, variant, family, n_nodes):
    prob = make_problem(n_nodes, family)
    refs = references(prob)
    monkeypatch.setenv("SAA_KVARIANT", str(variant))
    monkeypatch.setenv("SAA_STEP_HOST_PIPELINE", "5")
    order = np.random.default_rng(n_nodes).permutation(n_nodes)
    for plane_mask in (None, "0"):
        if plane_mask is None:
            monkeypatch.delenv("SAA_PLANE_MASK", raising=False)
        else:
            monkeypatch.setenv("SAA_PLANE_MASK", plane_mask)
        for setup in (host_plan, device_plan):
            for no in (None, order):
                pl = setup(prob, node_order=no)
                what = (variant, family, n_nodes, plane_mask, setup.__name__, no is not None)
                assert pl.nnz == prob["K"].nnz
                assert_layout(pl, prob["K"], variant, plane_mask, no)
                check_plan(pl, prob, refs, variant, what)
                pl.close()


@pytest.mark.parametrize("family", FAMILIES)
def test_stream_variant_energy_records_equal_default_layout(monkeypatch, family):
    """K1E on the full-plane layout of the cp.async variant gives the records of the default (masked) layout"""
    prob = make_problem(1025, family)
    refs = references(prob)
    recs = []
    for variant in (None, "6"):
        if variant is None:
            monkeypatch.delenv("SAA_KVARIANT", raising=False)
        else:
            monkeypatch.setenv("SAA_KVARIANT", variant)
        for setup in (host_plan, device_plan):
            pl = setup(prob)
            recs.append(check_plan(pl, prob, refs, 6, (family, variant, setup.__name__)))
            pl.close()
    for r in recs[1:]:
        for f in splan.ENERGY_FIELDS:
            assert np.array_equal(np.asarray(recs[0][f]).view(np.uint64), np.asarray(r[f]).view(np.uint64)), (family, f)


# ---- several partitions -----------------------------------------------------------------------------------------
def _golden_group(name):
    g = load_golden(name)
    P = g["P"]
    lists = [r["nodes"] for r in g["ranks"]]
    plans = []
    for q, r in enumerate(g["ranks"]):
        n = r["F"].size
        K = sp.csr_matrix((r["K_data"], r["K_indices"], r["K_indptr"]), shape=(n, n))
        plans.append(splan.StepPlan(K, r["F"], r["lM"], r["dirichlet"], g["dt"], float(g["alpha"]), rank=q, size=P,
                                    halo=maps.halo_plan(q, P, lists)))
    return g, plans


def _mid_group(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    pts, cells, fac = mesh.structured_beam(int(z["m"]), length=int(z["length"]))
    plans, _ = ds.build_mesh_in_process(pts, cells, fac, z["epart"].astype(np.int64), int(z["size"]))
    return z, plans


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("name", ["beam_coarse_P3", "beam_coarse_P4", "mid_np4"])
def test_fixture_partitions_per_variant(monkeypatch, variant, name):
    """Synchronised steps through the group transport: K1 runs the interior phase with slice_begin = sh_slices > 0"""
    monkeypatch.setenv("SAA_KVARIANT", str(variant))
    g, plans = _mid_group(name) if name.startswith("mid") else _golden_group(name)
    grp = splan.PlanGroup(plans)
    done = 0
    for n in [int(s) for s in g["steps"]]:
        grp.step(n - done, splan.MODE_SYNC)
        grp.synchronize()
        done = n
        for q, pl in enumerate(plans):
            assert bits_equal(pl.d0(), g[f"hist_{n}_r{q}"]), (name, variant, n, q)


def _synthetic_partition(family):
    """Three ranks over 700 global nodes: rank 0 holds 0..399, rank 1 300..699, rank 2 only 300..399, which ranks 0
    and 1 hold too — so rank 2 has no interior (sh_slices == n_slices) and ranks 0 and 1 start their interior at
    slice 4.  Each rank has its own synthetic matrix; load and mass are global, as the reference assembles them."""
    G = 700
    lists = [np.arange(0, 400), np.arange(300, 700), np.arange(300, 400)[::-1].copy()]
    probs = [make_problem(l.size, family, seed=10 + q) for q, l in enumerate(lists)]
    rng = np.random.default_rng(7)
    lM_g = 1.0 + np.zeros(3 * G)
    for l, p in zip(lists, probs):
        dof = (3 * l[:, None] + np.arange(3)).reshape(-1)
        lM_g[dof] = np.maximum(lM_g[dof], p["lM"])
    F_g = rng.uniform(-1, 1, 3 * G)
    dir_g = rng.choice(3 * G, size=60, replace=False)
    d0_g, dn_g = rng.uniform(-1, 1, 3 * G), rng.uniform(-1, 1, 3 * G)
    ranks = []
    for l, p in zip(lists, probs):
        dof = (3 * l[:, None] + np.arange(3)).reshape(-1)
        loc = np.full(3 * G, -1)
        loc[dof] = np.arange(dof.size)
        K = p["K"]
        ranks.append(dict(K_indptr=K.indptr, K_indices=K.indices, K_data=K.data, F=F_g[dof], lM=lM_g[dof],
                          dirichlet=np.sort(loc[dir_g][loc[dir_g] >= 0]).astype(np.int64), nodes=l,
                          d0=d0_g[dof], dn=dn_g[dof]))
    return G, lists, ranks


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("family", ["empty", "heavy"])
def test_synthetic_partition_with_empty_interior_per_variant(monkeypatch, variant, family):
    monkeypatch.setenv("SAA_KVARIANT", str(variant))
    G, lists, ranks = _synthetic_partition(family)
    P, alpha, tn0 = len(ranks), 0.5, 0.98
    o = oracle_module().OracleProblem(G, ranks, DT, alpha)
    plans = []
    for q, r in enumerate(ranks):
        n = r["F"].size
        K = sp.csr_matrix((r["K_data"], r["K_indices"], r["K_indptr"]), shape=(n, n))
        plans.append(splan.StepPlan(K, r["F"], r["lM"], r["dirichlet"], DT, alpha, rank=q, size=P,
                                    halo=maps.halo_plan(q, P, lists)))
        assert_layout(plans[-1], K, variant, None, shared=maps.halo_plan(q, P, lists)["shared_pos"])
    grp = splan.PlanGroup(plans)
    for q, (pl, r) in enumerate(zip(plans, ranks)):
        pl.set_state(r["d0"], r["dn"], tn0)
        o.set_state(q, r["d0"], r["dn"], tn0)
    done = 0
    for n in (1, NSTEPS):
        grp.step(n - done, splan.MODE_SYNC)
        grp.synchronize()
        o.run(n - done)
        done = n
        for q, pl in enumerate(plans):
            want = o.state(q)
            _same_state(pl.get_state(), want, (family, variant, n, q))
            assert np.all(np.isfinite(want[0])) and np.abs(want[0]).max() > 0


# ---- validation of a device-resident CSR ------------------------------------------------------------------------
def test_device_setup_rejects_malformed_csr():
    """from_device applies the host path's checks before any set-up kernel indexes by a column id"""
    prob = make_problem(40, "random")
    K = prob["K"]
    n = K.shape[0]
    row = int(np.argmax(np.diff(K.indptr)))
    a, b = int(K.indptr[row]), int(K.indptr[row + 1])
    assert b - a >= 2
    rev = K.indices.copy()
    rev[a:b] = rev[a:b][::-1]
    dup = K.indices.copy()
    dup[a + 1] = dup[a]
    out = K.indices.copy()
    out[b - 1] = n                                    # one past the last column
    neg = K.indices.copy()
    neg[a] = -1
    for bad, match in ((rev, "sorted"), (dup, "sorted"), (out, "out of range"), (neg, "out of range")):
        with pytest.raises(splan.SaaError, match=match):
            device_plan(prob, indices=bad)
        Kbad = sp.csr_matrix((K.data, bad, K.indptr), shape=K.shape)
        Kbad.has_sorted_indices = True                # keep scipy from repairing it
        with pytest.raises(splan.SaaError, match=match):
            splan.StepPlan(Kbad, prob["F"], prob["lM"], prob["dirichlet"], prob["dt"], prob["alpha"])
    ip = K.indptr.astype(np.int64)
    mono = ip.copy()
    mono[row + 1] = mono[row] - 1                     # indptr decreases
    start = ip.copy()
    start[0] = 1
    for bad, match in ((mono, "monotone"), (start, "indptr")):
        with pytest.raises(splan.SaaError, match=match):
            device_plan(prob, indptr=bad)
    # the failed set-ups leave nothing behind: a valid plan still gives the reference's bits
    pl = device_plan(prob)
    pl.set_state(prob["d0"], prob["dn"], prob["tn0"])
    pl.step(1, splan.MODE_LOCAL)
    pl.synchronize()
    _same_state(pl.get_state(), reference(prob, 1), "after rejections")
