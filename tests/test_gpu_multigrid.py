"""Multigrid-preconditioned static solve (multigrid.StructuredMultigrid, StepPlan.solve_static(precond=...),
csrc/saa_multigrid.cuh; DESIGN.md §7d).

  * nesting: prolonged coarse coordinates are the fine coordinates, and restriction is the transpose of prolongation;
  * the coarse plans' stiffness is the Galerkin operator S P^T S K S P S of the level above, on the device;
  * the V-cycle is symmetric positive definite, and lambda_max(B^-1 A) is estimated from below within 10 %;
  * the solution matches spsolve and the block-Jacobi solve, recovers a manufactured solution, and a host-built plan
    gives the device-built plan's result;
  * iteration counts do not grow with the mesh; bits are repeatable; no plan state changes; refusals.
"""
import numpy as np
import pytest
import scipy.sparse as sp
from scipy.sparse.linalg import eigsh, spsolve

import saa_b200  # noqa: F401
from saa_b200 import device_setup, multigrid, plan as splan
from util import bits_equal

pytestmark = pytest.mark.gpu


def _cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to("cuda")


def _np(t):
    return t.cpu().numpy()


def rel(a, b):
    return float(np.linalg.norm(np.asarray(a) - np.asarray(b)) / np.linalg.norm(np.asarray(b)))


def free_dofs(m, nodes):
    """free-DOF mask of a structured level from its global node ids (clamped: the x = 0 face)"""
    nodes = np.asarray(nodes.cpu() if hasattr(nodes, "cpu") else nodes)
    return np.repeat(nodes >= (m + 1) ** 2, 3)


def build(m):
    """device plan of structured_beam(m) with its host CSR, steady system A, b and node list"""
    pl, info = device_setup.build_structured_rank(m, 0, 1, keep_csr=True)
    K = info["K"].to_scipy()
    info["K"].free()
    keep = np.ones(K.shape[0])
    keep[np.asarray(info["dirichlet"], dtype=np.int64)] = 0.0
    S = sp.diags(keep)
    A = (S @ K @ S + sp.diags(1.0 - keep)).tocsr()
    b = keep * info["F"].cpu().numpy()
    return dict(plan=pl, info=info, K=K, A=A, b=b, keep=keep, m=m, nodes=info["local_nodes"])


def host_plan(c, K=None, F=None, dirichlet=None):
    i = c["info"]
    return splan.StepPlan(c["K"] if K is None else K, i["F"].cpu().numpy() if F is None else F, i["lM"].cpu().numpy(),
                          i["dirichlet"] if dirichlet is None else dirichlet, i["dt"], 0.5)


@pytest.fixture(scope="module")
def m4():
    c = build(4)
    c["mg"] = multigrid.StructuredMultigrid(c["plan"], 4, c["nodes"])
    yield c
    c["mg"].close()


@pytest.fixture(scope="module")
def m6():
    c = build(6)
    c["mg"] = multigrid.StructuredMultigrid(c["plan"], 6, c["nodes"])
    yield c
    c["mg"].close()


# ---- 1. nesting --------------------------------------------------------------------------------------------------------
def test_prolongation_reproduces_coordinates_and_restriction_is_its_transpose():
    c = build(8)
    rng = np.random.default_rng(1)
    with multigrid.StructuredMultigrid(c["plan"], 8, c["nodes"]) as mg:
        assert [lv[0] for lv in mg.levels] == [8, 4, 2]
        for l in range(2):
            mf, mc = mg.levels[l][0], mg.levels[l + 1][0]
            Xf = device_setup.structured_points(mf, mg.local_nodes[l].cuda()).reshape(-1)
            Xc = device_setup.structured_points(mc, mg.local_nodes[l + 1].cuda()).reshape(-1)
            ff, fc = free_dofs(mf, mg.local_nodes[l]), free_dofs(mc, mg.local_nodes[l + 1])
            Px = _np(mg.prolong(l, Xc))
            err = np.abs(Px[ff] - _np(Xf)[ff]).max() / np.abs(_np(Xf)).max()
            assert err <= 1e-15 and np.all(Px[~ff] == 0.0), (l, err)
            x = rng.standard_normal(fc.size) * fc
            y = rng.standard_normal(ff.size) * ff
            lhs, rhs = float(_np(mg.restrict(l, _cuda(y))) @ x), float(y @ _np(mg.prolong(l, _cuda(x))))
            assert abs(lhs - rhs) <= 1e-14 * abs(rhs), (l, lhs, rhs)


# ---- 2. Galerkin identity on the device ---------------------------------------------------------------------------------
@pytest.mark.parametrize("m", [4, 24])
def test_coarse_stiffness_is_the_galerkin_operator(m):
    pl, info = device_setup.build_structured_rank(m, 0, 1)
    rng = np.random.default_rng(m)
    with multigrid.StructuredMultigrid(pl, m, info["local_nodes"]) as mg:
        for l in range(len(mg.levels) - 1):
            ff, fc = free_dofs(mg.levels[l][0], mg.local_nodes[l]), free_dofs(mg.levels[l + 1][0], mg.local_nodes[l + 1])
            x = rng.standard_normal(fc.size) * fc
            Px = mg.prolong(l, _cuda(x))
            lhs = _np(mg.restrict(l, _cuda(ff * _np(mg.plans[l].apply_stiffness(Px)))))
            rhs = fc * _np(mg.plans[l + 1].apply_stiffness(_cuda(x)))
            err = np.abs(lhs - rhs).max() / np.abs(rhs).max()
            print(f"m={m}: {mg.levels[l][0]} -> {mg.levels[l + 1][0]}: {err:.2e}")
            assert err <= 1e-12


# ---- 3. V-cycle SPD, 4. lambda estimate ---------------------------------------------------------------------------------
def test_vcycle_is_symmetric_positive_definite(m6):
    mg, keep = m6["mg"], m6["keep"]
    rng = np.random.default_rng(3)
    for _ in range(3):
        a, b = rng.standard_normal(keep.size) * keep, rng.standard_normal(keep.size) * keep
        Va, Vb = _np(mg.vcycle(_cuda(a))), _np(mg.vcycle(_cuda(b)))
        assert abs(Va @ b - a @ Vb) <= 1e-12 * np.linalg.norm(Va) * np.linalg.norm(b)
        assert Va @ a > 0 and np.all(Va[keep == 0] == 0.0)


def block_jacobi(A):
    n = A.shape[0] // 3
    C = A.tocoo()
    on = (C.row // 3) == (C.col // 3)
    D = np.zeros((n, 3, 3))
    D[C.row[on] // 3, C.row[on] % 3, C.col[on] % 3] = C.data[on]
    return sp.block_diag([sp.csr_matrix(d) for d in D], format="csr")


@pytest.mark.parametrize("m", [4, 8])
def test_lambda_estimate_is_within_ten_percent_below_eigsh(m):
    c = build(m)
    true = float(eigsh(c["A"], k=1, M=block_jacobi(c["A"]), which="LA", return_eigenvectors=False)[0])
    with multigrid.StructuredMultigrid(c["plan"], m, c["nodes"]) as mg:
        ratio = mg.lambda_max[0] / true
        print(f"m={m}: lambda estimates {mg.lambda_max}, eigsh {true:.4f}, ratio {ratio:.4f}")
        assert 0.9 <= ratio <= 1.0 + 1e-12


# ---- 5. accuracy --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fixture", ["m4", "m6"])
def test_solution_matches_spsolve_and_block_jacobi(fixture, request):
    c = request.getfixturevalue(fixture)
    u = spsolve(c["A"].tocsc(), c["b"])
    res = c["plan"].solve_static(rtol=1e-12, max_iter=200, precond=c["mg"])
    bj = c["plan"].solve_static(rtol=1e-12)
    e1, e2 = rel(_np(res.x), u), rel(_np(res.x), _np(bj.x))
    print(f"m={c['m']}: {res}, vs spsolve {e1:.2e}, vs block-Jacobi ({bj.iterations} its) {e2:.2e}")
    assert res.converged and e1 <= 1e-8 and e2 <= 1e-8


def test_manufactured_solution_and_host_plan(m4):
    c = m4
    rng = np.random.default_rng(5)
    xs = rng.standard_normal(c["keep"].size) * c["keep"]
    F = c["A"] @ xs
    hp = host_plan(c, F=F)
    with multigrid.StructuredMultigrid(hp, 4, c["nodes"].cpu().numpy()) as mg:
        res = hp.solve_static(rtol=1e-12, max_iter=200, precond=mg)
        print(f"manufactured: {res}, error {rel(_np(res.x), xs):.2e}")
        assert res.converged and rel(_np(res.x), xs) <= 1e-8
    # the same system on a host-built plan and on the device-built plan
    hp2 = host_plan(c)
    with multigrid.StructuredMultigrid(hp2, 4, c["nodes"]) as mg:
        a = hp2.solve_static(rtol=1e-12, max_iter=200, precond=mg)
    d = c["plan"].solve_static(rtol=1e-12, max_iter=200, precond=c["mg"])
    print(f"host plan vs device plan: {rel(_np(a.x), _np(d.x)):.2e}")
    assert rel(_np(a.x), _np(d.x)) <= 1e-12


# ---- 6. mesh-independent iteration counts -------------------------------------------------------------------------------
def test_iteration_counts_do_not_grow_with_the_mesh():
    its = {}
    for m in (4, 6, 12, 24):
        c = build(m)
        with multigrid.StructuredMultigrid(c["plan"], m, c["nodes"]) as mg:
            res = c["plan"].solve_static(rtol=1e-8, precond=mg)
        its[m] = res.iterations
        x = _np(res.x)
        floor = float(np.finfo(np.float64).eps / 2 * np.linalg.norm(c["keep"] * (abs(c["K"]) @ np.abs(x))) / np.linalg.norm(c["b"]))
        bound = max(10 * 1e-8, np.sqrt(res.iterations) * floor)
        print(f"m={m} ({c['plan'].n_dof} DOF, levels {mg.levels}): {res}, floor {floor:.2e}")
        assert res.converged and res.iterations <= 40 and res.rel_residual_true <= bound
        c["plan"].close()
    assert its[24] <= 1.5 * its[6], its


# ---- 7. determinism -----------------------------------------------------------------------------------------------------
def test_bits_repeatable_across_calls_check_intervals_launches_and_hierarchies(m6, monkeypatch):
    pl, mg = m6["plan"], m6["mg"]
    a = pl.solve_static(rtol=1e-10, precond=mg)
    b = pl.solve_static(rtol=1e-10, precond=mg)
    c = pl.solve_static(rtol=1e-10, precond=mg, check_every=1)
    with multigrid.StructuredMultigrid(pl, 6, m6["nodes"]) as mg2:
        e = pl.solve_static(rtol=1e-10, precond=mg2)
        assert mg2.lambda_max == mg.lambda_max
    monkeypatch.setenv("SAA_STATIC_GRAPH", "0")
    d = pl.solve_static(rtol=1e-10, precond=mg)
    for r in (b, c, d, e):
        assert r.iterations == a.iterations and bits_equal(_np(r.x), _np(a.x)) and bits_equal(_np(r.history), _np(a.history))


# ---- 8. no side effects -------------------------------------------------------------------------------------------------
def _run(with_mg, monitors, launches):
    pl, info = device_setup.build_structured_rank(4, 0, 1)
    if monitors:
        pl.set_energy(200, 1)
        pl.set_history(None, 64, 3)
    mg = multigrid.StructuredMultigrid(pl, 4, info["local_nodes"]) if with_mg else None
    coarse0 = [p.get_state() for p in mg.plans[1:]] if with_mg else None
    for n, launch in launches:
        pl.step(n, splan.MODE_LOCAL, launch)
        if with_mg:
            pl.solve_static(rtol=1e-6, max_iter=15, check_every=4, precond=mg)
            mg.vcycle(_cuda(np.ones(pl.n_dof)))
    pl.synchronize()
    out = (pl.get_state(), pl.read_energy() if monitors else None, pl.read_history() if monitors else None)
    if with_mg:
        for s0, p in zip(coarse0, mg.plans[1:]):
            s1 = p.get_state()
            assert bits_equal(s0[0], s1[0]) and bits_equal(s0[1], s1[1]) and s0[2] == s1[2]
        mg.close()
    pl.close()
    return out


def test_solves_change_no_state_energy_record_or_history():
    L = splan
    for monitors, launches in ((True, [(5, L.LAUNCH_PER_STEP), (8, L.LAUNCH_GRAPH), (1, L.LAUNCH_PER_STEP), (6, L.LAUNCH_GRAPH)]),
                               (False, [(5, L.LAUNCH_PERSISTENT), (8, L.LAUNCH_GRAPH), (7, L.LAUNCH_PERSISTENT)])):
        (a0, an, at), ea, ha = _run(True, monitors, launches)
        (b0, bn, bt), eb, hb = _run(False, monitors, launches)
        assert bits_equal(a0, b0) and bits_equal(an, bn) and at == bt
        if monitors:
            for f in splan.ENERGY_FIELDS:
                assert np.array_equal(ea[f], eb[f]), f
            assert ha.shape == hb.shape and bits_equal(ha, hb)


def test_block_jacobi_solve_unchanged_by_a_hierarchy():
    pl, info = device_setup.build_structured_rank(4, 0, 1)
    a = pl.solve_static(rtol=1e-10)
    with multigrid.StructuredMultigrid(pl, 4, info["local_nodes"]) as mg:
        b = pl.solve_static(rtol=1e-10)
        pl.solve_static(rtol=1e-10, precond=mg)
        c = pl.solve_static(rtol=1e-10)
    for r in (b, c):
        assert r.iterations == a.iterations and bits_equal(_np(r.x), _np(a.x))


# ---- 9. refusals --------------------------------------------------------------------------------------------------------
def test_refusals(m4):
    import torch
    pl, mg = m4["plan"], m4["mg"]
    with pytest.raises(ValueError, match=r"m = 111 .*cannot be halved.*96 and 128"):
        multigrid.StructuredMultigrid(pl, 111, m4["nodes"])
    with pytest.raises(ValueError, match=r"m = 112 .*odd m = 7 with 33792 DOF"):
        multigrid.StructuredMultigrid(pl, 112, m4["nodes"])
    # a partition: the group refuses precond, a rank plan refuses the hierarchy
    plans, infos = device_setup.build_structured_in_process(4, 2)
    grp = splan.PlanGroup(plans)
    with pytest.raises(splan.SaaError, match="single-partition plan only"):
        grp.solve_static(precond=mg)
    with pytest.raises(splan.SaaError, match="size 2"):
        multigrid.StructuredMultigrid(plans[0], 4, infos[0]["local_nodes"])
    grp.close()
    # another plan's hierarchy; use after close
    other, info = device_setup.build_structured_rank(4, 0, 1, keep_mesh=True)
    with pytest.raises(splan.SaaError, match="another plan"):
        other.solve_static(precond=mg)
    mg2 = multigrid.StructuredMultigrid(other, 4, info["local_nodes"])
    mg2.close()
    with pytest.raises(splan.SaaError, match="after close"):
        other.solve_static(precond=mg2)
    with pytest.raises(splan.SaaError, match="after close"):
        mg2.vcycle(_cuda(np.zeros(other.n_dof)))
    # the assembled matrix released, before and after the hierarchy exists
    mg3 = multigrid.StructuredMultigrid(other, 4, info["local_nodes"])
    other.set_matfree(info["cells_loc"], info["pts"], *info["lame"])
    other.set_option(splan.OPT_MATFREE, 2)
    with pytest.raises(splan.SaaError, match="SAA_OPT_MATFREE = 2"):
        other.solve_static(precond=mg3)
    with pytest.raises(splan.SaaError, match="SAA_OPT_MATFREE = 2"):
        multigrid.StructuredMultigrid(other, 4, info["local_nodes"])
    mg3.close()
    # -K on the fine level: no diagonal block is positive definite
    neg = host_plan(m4, K=-m4["K"])
    with pytest.raises(splan.SaaError, match=r"level 0, local node \d+: .*not positive definite"):
        multigrid.StructuredMultigrid(neg, 4, m4["nodes"])
    # a floating model with a net load: no convergence, finite values
    fl = host_plan(m4, dirichlet=np.zeros(0, dtype=np.int64))
    with multigrid.StructuredMultigrid(fl, 4, m4["nodes"]) as mgf:
        res = fl.solve_static(rtol=1e-10, max_iter=30, check_every=8, precond=mgf)
    assert not res.converged and res.iterations == 30
    assert torch.isfinite(res.x).all() and torch.isfinite(res.history).all()
    assert np.isfinite(res.rel_residual) and np.isfinite(res.rel_residual_true)
