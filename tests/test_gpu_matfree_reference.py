"""Kernel K5 (the matrix-free step, saa_matfree.cuh) against an exact reference of its own operation.

K5's internal force f = sum_e V sigma(u_e) grad N_a is recovered from ONE shipped step with alpha = 0, tn = 0 (ramp 0,
no external load) and dn = d0 = u:  d1 = d0 - dt^2 f / M, so f = M (d0 - d1) / dt^2 up to a rounding bounded from the
update's own operations.  Every row must then satisfy
    |f_K5 - f_exact| <= force_bound + recovery bound        (oracle/matfree_ref.py derives both; no fitted constant)
where f_exact is the formula in rational arithmetic on the exact double inputs.  On the loaded beam a whole-step
comparison admits a force error of ~5e-8 relative; this admits about 1e-14 relative, and planted errors of 1e-12 in
the element force are caught (tests/test_matfree_reference_cpu.py).

Random (rough) fields with dt chosen so that |dt^2 K u / M| / |u| = 0.6: the force is a large part of the increment.
Meshes: the golden beam_coarse / struct_m3 and the adversarial meshes of matfree_ref.adversarial_meshes (jittered,
inverted elements, translated by 1e3, slivers, a hub node in 136 tets, nodes in no element, 31 / 33 / 257 nodes).
"""
import numpy as np
import pytest

import saa_b200  # noqa: F401
from saa_b200 import assembly, device_setup as ds, maps, plan as splan, problem
from test_gpu_format_conformance import device_plan, host_plan
from util import bits_equal, load_golden, oracle_module

pytestmark = pytest.mark.gpu

oracle_module()                                   # puts oracle/ on sys.path
import matfree_ref as mr  # noqa: E402

LMD, MU = problem.lame(problem.E_DEFAULT, problem.NU_DEFAULT)
RATIO = 0.6
GOLDEN = ("beam_coarse_P1", "struct_m3_P1")
ADVERSARIAL = ("jittered", "inverted", "translated", "slivers", "fan", "orphans", "delaunay31", "delaunay33", "delaunay257")
MESHES = GOLDEN + ADVERSARIAL
_cache = {}


def _mesh(name):
    if name in GOLDEN:
        return mr.golden_mesh(load_golden(name))
    return mr.adversarial_meshes()[name]


def _problem(name, seed=0):
    """one mesh with a rough field, its exact force and bound, and the single-partition problem of its
    reference-assembled LocalK (unit lumped mass, no Dirichlet rows, no load)"""
    key = (name, seed)
    if key not in _cache:
        pts, cells = _mesh(name)
        n = len(pts)
        u = np.random.default_rng(seed).standard_normal(3 * n)
        exact = mr.internal_force_exact(pts, cells, u, LMD, MU).reshape(-1)
        fl = mr.to_float(exact)
        dt = float(np.sqrt(RATIO * np.linalg.norm(u) / np.linalg.norm(fl)))
        K = assembly.local_stiffness_csr(np.arange(n), cells, pts, LMD, MU)
        _cache[key] = dict(pts=pts, cells=cells, u=u, exact=exact, bound=mr.force_bound(pts, cells, u, LMD, MU).reshape(-1),
                           K=K, F=np.zeros(3 * n), lM=np.ones(3 * n), dirichlet=np.zeros(0, dtype=np.int64), dt=dt, alpha=0.0)
    return _cache[key]


def _k5_plan(prob, setup="host", node_order=None):
    pl = (host_plan if setup == "host" else device_plan)(prob, node_order=node_order)
    pl.set_matfree(prob["cells"], prob["pts"], LMD, MU)
    pl.set_option(splan.OPT_MATFREE, 1)
    return pl


def _k5_step(pl, u, launch=splan.LAUNCH_PER_STEP):
    pl.set_state(u, u, 0.0)
    pl.step(1, splan.MODE_LOCAL, launch)
    pl.synchronize()
    return pl.d0()


def _ratio(err, bound):
    """largest err / bound; a row with bound 0 (a node in no element) must be exact"""
    assert np.all(err[bound == 0] == 0), "a row without incident elements has a non-zero force"
    return float(np.max(err[bound > 0] / bound[bound > 0], initial=0.0))


def _check_force(d1, u, M, dt2, exact, bound, what):
    """the force recovered from d1 within force_bound + the recovery bound; rows of nodes in no element (force_bound
    0) must come back exactly 0: there the update computes 2 d0 - d0 = d0 without rounding"""
    R, rb = mr.recover_force(u, d1, M, dt2)
    err = mr.abs_error(R, exact)
    assert np.all(err[bound == 0] == 0), f"{what}: a row without incident elements has a non-zero force"
    r = _ratio(np.where(bound == 0, 0.0, err), np.where(bound == 0, 1.0, bound + rb))
    print(f"{what}: max |f_K5 - f_exact| / bound = {r:.3f}")
    assert r <= 1.0, what
    return r


@pytest.mark.parametrize("name", MESHES)
def test_k5_force_within_exact_bound(monkeypatch, name):
    """every row, SAA_MF_MINB 3-6, both set-up paths, per-step and graph launches; for one MINB the launch strategies,
    set-up paths and repeats agree bit for bit.  Across MINB values only the bound is asserted (the register cap may
    change the instruction schedule); whether the bits agree is reported."""
    prob = _problem(name)
    per_minb = {}
    for minb in (3, 4, 5, 6):
        monkeypatch.setenv("SAA_MF_MINB", str(minb))
        outs = []
        for setup in ("host", "device"):
            pl = _k5_plan(prob, setup)
            for launch in (splan.LAUNCH_PER_STEP, splan.LAUNCH_GRAPH, splan.LAUNCH_PER_STEP):
                outs.append(_k5_step(pl, prob["u"], launch))
            _check_force(outs[-1], prob["u"], 1.0, pl.dt2, prob["exact"], prob["bound"], f"{name} MINB={minb} {setup}")
        assert all(bits_equal(o, outs[0]) for o in outs[1:]), f"MINB={minb}: launch, set-up path or a repeat changed the bits"
        per_minb[minb] = outs[0]
    same = [m for m in (4, 5, 6) if bits_equal(per_minb[m], per_minb[3])]
    print(f"{name}: MINB 4/5/6 give the bits of MINB 3: {same == [4, 5, 6]} (equal for {same})")


@pytest.mark.parametrize("name", MESHES)
def test_assembled_path_within_the_same_bound(name):
    """apply_stiffness of the reference-assembled LocalK (scipy's LocalK @ u, bit for bit) against the same exact
    force.  Its operation sequence is not K5's, so K5's bound is an acceptance bound here, not a derived one; both
    paths are pinned to the exact value rather than to each other."""
    import torch
    prob = _problem(name)
    pl = host_plan(prob)
    y = pl.apply_stiffness(torch.from_numpy(prob["u"]).cuda()).cpu().numpy()
    assert bits_equal(y, prob["K"] @ prob["u"])
    r = _ratio(mr.abs_error(y, prob["exact"]), prob["bound"])
    print(f"{name}: assembled max |K u - f_exact| / bound = {r:.3f}")
    assert r <= 1.0


@pytest.mark.parametrize("name", ["struct_m3_P1", "jittered", "orphans", "fan", "delaunay257"])
def test_k5_bits_do_not_depend_on_node_order_or_setup(name):
    """a node's force does not depend on the internal numbering: no order, RCM, Morton and reversed orders, host and
    device finalisation give the same bits"""
    import torch
    prob = _problem(name)
    n = len(prob["pts"])
    orders = {"none": None, "rcm": splan.rcm_node_order(prob["K"]),
              "morton": ds.morton_node_order(torch.from_numpy(prob["pts"]).cuda()),
              "reversed": np.arange(n - 1, -1, -1, dtype=np.int32)}
    ref = None
    for setup in ("host", "device"):
        for oname, order in orders.items():
            d1 = _k5_step(_k5_plan(prob, setup, order), prob["u"], splan.LAUNCH_GRAPH)
            ref = d1 if ref is None else ref
            assert bits_equal(d1, ref), (setup, oname)


def _partition(name):
    """(whole-mesh problem of _problem, its global node ids, ranks as (node list, element list) in the reference's
    local orders): a golden P = 3 fixture, or x-slabs of the jittered mesh"""
    if name.startswith("jittered"):
        from saa_b200 import partition
        whole = _problem("jittered")
        pts, cells = whole["pts"], whole["cells"]
        ep = partition.slab_partition(pts, cells, 3)
        ranks = []
        for q in range(3):
            ele = np.nonzero(ep == q)[0]
            flat = cells[ele].reshape(-1)
            _, first = np.unique(flat, return_index=True)
            ranks.append((flat[np.sort(first)], ele))                   # Local_nodal_list: first-appearance order
        return whole, np.arange(len(pts)), pts, cells, ranks
    g = load_golden(name)
    whole = _problem(name.replace("_P3", "_P1"))
    nodes1 = np.asarray(load_golden(name.replace("_P3", "_P1"))["ranks"][0]["nodes"], dtype=np.int64)
    ranks = [(np.asarray(r["nodes"], dtype=np.int64), np.asarray(r["ele"], dtype=np.int64)) for r in g["ranks"]]
    return whole, nodes1, np.asarray(g["points"], dtype=np.float64), np.asarray(g["cells"], dtype=np.int64)[:, :4], ranks


@pytest.mark.parametrize("name", ["beam_coarse_P3", "struct_m3_P3", "jittered_slabs3"])
def test_k5_partitions(name):
    """each rank of a P = 3 partition: its partial force over its own elements against the exact reference of those
    elements; at nodes no other rank holds, the same bits as the single-partition plan"""
    whole, nodes1, pts_all, cells_all, ranks = _partition(name)
    P = len(ranks)
    u_all = np.random.default_rng(7).standard_normal(3 * len(pts_all))
    u1 = u_all.reshape(-1, 3)[nodes1].reshape(-1)
    p1 = _k5_plan(dict(whole, u=u1))
    d1_whole = _k5_step(p1, u1).reshape(-1, 3)
    dt2 = p1.dt2
    at = np.full(len(pts_all), -1)
    at[nodes1] = np.arange(nodes1.size)
    lists = [nodes for nodes, _ in ranks]
    count = np.zeros(len(pts_all), dtype=np.int64)
    for nodes in lists:
        count[nodes] += 1
    for q, (nodes, ele) in enumerate(ranks):
        n = nodes.size
        pos = np.full(len(pts_all), -1)
        pos[nodes] = np.arange(n)
        pts, cells = pts_all[nodes], pos[cells_all[ele]]
        u = u_all.reshape(-1, 3)[nodes].reshape(-1)
        K = assembly.local_stiffness_csr(np.arange(n), cells, pts, LMD, MU)
        pl = splan.StepPlan(K, np.zeros(3 * n), np.ones(3 * n), np.zeros(0, dtype=np.int64), whole["dt"], 0.0, rank=q, size=P,
                            halo=maps.halo_plan(q, P, lists))
        pl.set_matfree(cells, pts, LMD, MU)
        pl.set_option(splan.OPT_MATFREE, 1)
        d1 = _k5_step(pl, u)
        assert pl.dt2 == dt2
        exact = mr.internal_force_exact(pts, cells, u, LMD, MU).reshape(-1)
        _check_force(d1, u, 1.0, dt2, exact, mr.force_bound(pts, cells, u, LMD, MU).reshape(-1), f"{name} rank {q}")
        own = count[nodes] == 1
        assert own.any() and not own.all()
        assert bits_equal(d1.reshape(-1, 3)[own], d1_whole[at[nodes[own]]]), f"rank {q}: non-shared rows differ from P = 1"


def _golden_k5_plan(g, q, **kw):
    """the golden rank's plan (its LocalK, load, mass, Dirichlet rows, dt, alpha) with K5 attached and enabled"""
    import scipy.sparse as sp
    r = g["ranks"][q]
    n = r["F"].size
    K = sp.csr_matrix((r["K_data"], r["K_indices"], r["K_indptr"]), shape=(n, n))
    pl = splan.StepPlan(K, r["F"], r["lM"], r["dirichlet"], g["dt"], float(g["alpha"]), **kw)
    pts, cells = mr.golden_mesh(g, q)
    pl.set_matfree(cells, pts, LMD, MU)
    pl.set_option(splan.OPT_MATFREE, 1)
    return pl


def test_k5_in_the_sync_avoiding_schedule():
    """A PlanGroup with K5 enabled, 3 local steps then 1 synchronised step, five times, on the loaded golden P = 3
    beam.  Local steps are K5 and equal, bit for bit, the same step of an ungrouped plan of the rank started from the
    same state; synchronised steps stream the assembled matrix and equal the C oracle's synchronised step started
    from the device state; tn and the step counters advance as in the assembled schedule."""
    g = load_golden("beam_coarse_P3")
    P = g["P"]
    lists = [r["nodes"] for r in g["ranks"]]
    plans = [_golden_k5_plan(g, q, rank=q, size=P, halo=maps.halo_plan(q, P, lists)) for q in range(P)]
    grp = splan.PlanGroup(plans)
    alone = [_golden_k5_plan(g, q) for q in range(P)]
    asm_plans = [_golden_k5_plan(g, q, rank=q, size=P, halo=maps.halo_plan(q, P, lists)) for q in range(P)]
    for pl in asm_plans:
        pl.set_option(splan.OPT_MATFREE, 0)
    asm = splan.PlanGroup(asm_plans)
    o = oracle_module().OracleProblem(len(g["points"]), g["ranks"], g["dt"], float(g["alpha"]))
    grp.step(40, splan.MODE_SYNC)                                          # a loaded, moving beam
    asm.step(40, splan.MODE_SYNC)
    grp.synchronize()
    asm.synchronize()
    for cycle in range(5):
        for k in range(3):
            before = [pl.get_state() for pl in plans]
            grp.step(1, splan.MODE_LOCAL)
            asm.step(1, splan.MODE_LOCAL)
            grp.synchronize()
            asm.synchronize()
            for q in range(P):
                alone[q].set_state(*before[q])
                alone[q].step(1, splan.MODE_LOCAL)
                alone[q].synchronize()
                got, want = plans[q].get_state(), alone[q].get_state()
                assert bits_equal(got[0], want[0]) and bits_equal(got[1], want[1]), (cycle, k, q)
                assert got[2] == want[2] == asm_plans[q].get_state()[2], (cycle, k, q)
        for q in range(P):
            o.set_state(q, *plans[q].get_state())
        grp.step(1, splan.MODE_SYNC)
        asm.step(1, splan.MODE_SYNC)
        grp.synchronize()
        asm.synchronize()
        o.run(1)
        for q in range(P):
            got, want = plans[q].get_state(), o.state(q)
            assert bits_equal(got[0], want[0]) and bits_equal(got[1], want[1]), (cycle, "sync", q)
            assert got[2] == want[2] == asm_plans[q].get_state()[2], (cycle, "sync", q)
    # the step counters: a history ring armed now records at the same steps in both schedules
    for pls, gr in ((plans, grp), (asm_plans, asm)):
        for pl in pls:
            pl.set_history(None, capacity=8, save_every=3)
        gr.step(7, splan.MODE_LOCAL)
        gr.synchronize()
    assert [pl.history_count for pl in plans] == [pl.history_count for pl in asm_plans]
    assert plans[0].history_count == len([s for s in range(60, 67) if s % 3 == 0])


def test_k5_with_history_and_prediction_hooks_from_a_graph():
    """MODE_PREDICT with a history ring, replayed from a CUDA graph with K5 enabled, against unhooked K5 steps
    followed by the prediction overwrite on the host: the same bits, and the ring holds exactly the d0s read back"""
    import torch
    g = load_golden("beam_coarse_P2")
    r = g["ranks"][0]
    dofs = np.asarray(r["loc_dof_shared"], dtype=np.int64)
    N = 12
    table = np.random.default_rng(5).standard_normal((N, dofs.size)) * 1e-4
    tdev = torch.from_numpy(table).cuda()
    hooked, plain = _golden_k5_plan(g, 0), _golden_k5_plan(g, 0)
    for pl in (hooked, plain):
        pl.step(5, splan.MODE_LOCAL)                                       # hooks armed mid-run, at an odd step
    hooked.set_history(None, capacity=N, save_every=1)
    hooked.set_prediction(dofs, tdev.data_ptr(), N)
    hooked.step(N, splan.MODE_PREDICT, splan.LAUNCH_GRAPH)
    hooked.synchronize()
    want = []
    for k in range(N):
        plain.step(1, splan.MODE_LOCAL, splan.LAUNCH_PER_STEP)
        d0, dn, tn = plain.get_state()
        d0[dofs] = table[k]
        plain.set_state(d0, dn, tn)
        want.append(d0)
    got = hooked.get_state()
    assert bits_equal(got[0], want[-1]) and bits_equal(got[1], want[-2]) and got[2] == plain.get_state()[2]
    assert hooked.history_count == N
    assert bits_equal(hooked.read_history(0, N), np.stack(want))


def test_step_host_takes_the_plain_path_and_equals_resident_k5():
    prob = _problem("jittered")
    pl = _k5_plan(prob)
    assert pl.host_pipe_info(splan.MODE_LOCAL)[0] == 0                      # K5 has no pipelined host call
    d1 = np.array(pl.step_host(prob["u"], prob["u"], 0.0))
    assert bits_equal(d1, _k5_step(_k5_plan(prob), prob["u"]))


def test_k5_at_scale_against_extended_precision():
    """m = 24 device set-up (1.13 M DOF), alpha = 0, random d0: every non-Dirichlet row within the bound of the
    long-double reference"""
    if np.finfo(np.longdouble).nmant < 63:
        pytest.skip("np.longdouble has no 64-bit mantissa on this host: no extended-precision reference")
    pl, info = ds.build_structured_rank(24, 0, 1, alpha=0.0, keep_csr=True, keep_mesh=True)
    cells = info["cells_loc"].cpu().numpy()
    pts = info["pts"].cpu().numpy()
    lM = info["lM"].cpu().numpy()
    pl.set_matfree(info["cells_loc"], info["pts"], *info["lame"])
    pl.set_option(splan.OPT_MATFREE, 1)
    u = np.random.default_rng(11).standard_normal(pl.n_dof)
    d1 = _k5_step(pl, u)
    keep = np.ones(pl.n_dof, dtype=bool)
    keep[np.asarray(info["dirichlet"], dtype=np.int64)] = False
    R, rb = mr.recover_force(u, d1, lM, pl.dt2)
    ref = mr.internal_force_ld(pts, cells, u, *info["lame"]).reshape(-1)
    b = mr.force_bound(pts, cells, u, *info["lame"]).reshape(-1) + rb
    err = np.abs(R - ref).astype(np.float64)
    r = _ratio(err[keep], b[keep])
    print(f"m = 24 ({pl.n_dof} DOF): max |f_K5 - f_ld| / bound = {r:.3f}")
    assert r <= 1.0


# ---- refused cells -------------------------------------------------------------------------------------------------
def test_set_matfree_refuses_bad_cells_and_stays_usable():
    import torch
    prob = _problem("jittered")
    pts, cells = prob["pts"], prob["cells"]
    n = len(pts)
    pl = host_plan(prob)
    bad_ids = []
    for v in (-1, n, 2 ** 31 + 5):
        c = cells.astype(np.int64)
        c[17, 2] = v
        bad_ids.append(c)
    for c in bad_ids:                                                      # numpy and torch, checked before the int32 cast
        for arg in (c, torch.from_numpy(c)):
            with pytest.raises(splan.SaaError, match="outside"):
                pl.set_matfree(arg, pts, LMD, MU)
    with pytest.raises(splan.SaaError, match="integer"):
        pl.set_matfree(cells.astype(np.float64), pts, LMD, MU)
    rep = cells.copy()
    rep[29, 3] = rep[29, 1]                                                # a repeated corner
    with pytest.raises(splan.SaaError, match="element 29 has zero volume"):
        pl.set_matfree(rep, pts, LMD, MU)
    flat = pts.copy()
    flat[cells[41], 2] = 0.25                                              # four corners in one plane: detJ == 0 exactly
    with pytest.raises(splan.SaaError, match="element 41 has zero volume"):
        pl.set_matfree(cells, flat, LMD, MU)
    with pytest.raises(splan.SaaError):
        pl.set_option(splan.OPT_MATFREE, 1)                                # nothing was attached
    pl.set_matfree(cells, pts, LMD, MU)                                    # a valid call after the refusals
    pl.set_option(splan.OPT_MATFREE, 1)
    _check_force(_k5_step(pl, prob["u"]), prob["u"], 1.0, pl.dt2, prob["exact"], prob["bound"], "after refusals")


def test_set_matfree_device_check_refuses_ids_the_python_check_never_sees():
    """the C entry point checks its cells itself: ids outside the node range reach it through a caller that skips
    StepPlan.set_matfree"""
    import torch
    from saa_b200.plan import lib
    prob = _problem("jittered")
    pl = host_plan(prob)
    c = torch.from_numpy(prob["cells"].astype(np.int32)).cuda()
    c[5, 0] = len(prob["pts"])
    x = torch.from_numpy(prob["pts"]).cuda()
    torch.cuda.synchronize()
    assert lib().saa_plan_set_matfree_dev(pl.h, c.shape[0], c.data_ptr(), x.data_ptr(), LMD, MU) != 0
    c[5, 0] = -3
    assert lib().saa_plan_set_matfree_dev(pl.h, c.shape[0], c.data_ptr(), x.data_ptr(), LMD, MU) != 0
    c[5, 0] = int(prob["cells"][5, 0])
    assert lib().saa_plan_set_matfree_dev(pl.h, c.shape[0], c.data_ptr(), x.data_ptr(), LMD, MU) == 0
