"""On-device energy monitor (saa_plan_set_energy / StepPlan.set_energy / plan.energy_balance).

  * arming the monitor changes no state bit (golden histories, monitor-off runs, PREDICT steps);
  * every record field equals a numpy evaluation from the all-DOF history, the scipy matrices and the owner rule;
  * the discrete balance closes (|residual| tiny against the energies) and E is conserved without load and damping;
  * records are bit-identical across launch strategies, transports and repeats; ring semantics;
  * PREDICT: the balance residual measures the energy a prediction table injects;
  * refusals: persistent loop, SAA_OPT_MATFREE, every < 1.
"""
import os
import sys

import numpy as np
import pytest
import scipy.sparse as sp

import saa_b200  # noqa: F401
from saa_b200 import maps, plan as splan
from util import ROOT, bits_equal, load_golden

pytestmark = pytest.mark.gpu
F_REL = 1e-12          # per-field agreement with the numpy evaluation, relative to the field's largest magnitude


def _K(r):
    n = r["F"].size
    return sp.csr_matrix((r["K_data"], r["K_indices"], r["K_indptr"]), shape=(n, n))


def make_plans(g, group=True, alpha=None, zero_load=False):
    P = g["P"]
    lists = [r["nodes"] for r in g["ranks"]]
    a = float(g["alpha"]) if alpha is None else alpha
    plans = []
    for q, r in enumerate(g["ranks"]):
        F = np.zeros_like(r["F"]) if zero_load else r["F"]
        plans.append(splan.StepPlan(_K(r), F, r["lM"], r["dirichlet"], g["dt"], a, halo=maps.halo_plan(q, P, lists) if P > 1 else None,
                                    rank=q, size=P))
    grp = splan.PlanGroup(plans) if (P > 1 and group) else None
    return plans, grp


def step(plans, grp, n, mode=splan.MODE_SYNC, launch=splan.LAUNCH_AUTO):
    if grp is None:
        for pl in plans:
            pl.step(n, splan.MODE_LOCAL if mode == splan.MODE_SYNC else mode, launch)
            pl.synchronize()
    else:
        grp.step(n, mode)
        grp.synchronize()


def balance(plans):
    return splan.energy_balance([pl.read_energy() for pl in plans])


def scale(b):
    return max(np.abs(b["total"]).max(), np.abs(b["work_external"]).max(), np.abs(b["work_damping"]).max())


def owned_dofs(g):
    """per rank: DOF mask of the rows whose mass / load it counts (non-shared, or shared and lowest holder)"""
    lists = [np.asarray(r["nodes"]) for r in g["ranks"]]
    low = {}
    for q, l in enumerate(lists):
        for e in l.tolist():
            low.setdefault(e, q)
    return [np.repeat(np.array([low[e] == q for e in l.tolist()]), 3) for q, l in enumerate(lists)]


def numpy_records(g, q, H, dt, alpha, own, F=None):
    """records of rank q from its all-DOF history H[k] = d_{k+1} (H[-1] = d_0 = d_{-1} = 0 start), every step"""
    r = g["ranks"][q]
    K, m = _K(r), np.asarray(r["lM"], dtype=np.float64).reshape(-1)
    F = np.asarray(r["F"] if F is None else F, dtype=np.float64).reshape(-1)
    n_dof = m.size
    d = np.vstack([np.zeros((2, n_dof)), H])                      # d[k + 1] = d_k, k = -1, 0, 1, ...
    dt2 = float(np.float64(dt) ** 2)
    N = H.shape[0] - 1
    out = np.zeros(N, dtype=splan.ENERGY_DTYPE)
    t, W, D = 0.0, 0.0, 0.0
    E_arm = None
    for n in range(N):
        dm, d0, dp = d[n], d[n + 1], d[n + 2]
        f = K @ d0
        kh = 0.5 * np.sum((m * (d0 - dm) ** 2)[own]) / dt2
        cp, st = 0.5 * np.dot(dm, f), 0.5 * np.dot(d0, f)
        kin = 0.5 * np.sum((m * (dp - dm) ** 2)[own]) / (4 * dt2)
        dW = 0.5 * np.sum((F * min(t, 1.0) * (dp - dm))[own])
        if E_arm is None:
            E_arm = kh + cp
        out[n] = (n, t, kh, cp, st, kin, W, D, E_arm)
        W, D = W + dW, D + alpha * dt * 2 * kin
        t = t + dt
    return out


def assert_records_close(got, want, what):
    assert np.array_equal(got["step"], want["step"]), what
    assert np.array_equal(got["tn"], want["tn"]), what
    for f in splan.ENERGY_FIELDS[2:]:
        s = max(np.abs(want[f]).max(), 1e-300)
        err = np.abs(got[f] - want[f]).max() / s
        assert err <= F_REL, (what, f, err)


def records_equal(a, b):
    return all(bits_equal(a[f].astype(np.float64), b[f].astype(np.float64)) for f in splan.ENERGY_FIELDS)


# ---- 1. no behaviour change --------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["beam_coarse_P1", "beam_coarse_P3"])
def test_monitor_changes_no_state_bit(name):
    g = load_golden(name)
    runs = []
    for every in (None, 1, 7):
        plans, grp = make_plans(g)
        if every:
            for pl in plans:
                pl.set_energy(400, every)
        done = 0
        for s in [int(x) for x in g["steps"] if x <= 2000] + [2000]:
            if s > done:
                step(plans, grp, s - done)
                done = s
            if f"hist_{s}_r0" in g:
                for q, pl in enumerate(plans):
                    assert bits_equal(pl.d0(), g[f"hist_{s}_r{q}"]), (name, every, s, q)
        runs.append([pl.get_state() for pl in plans])
        if every:
            assert plans[0].energy_count == (2000 + every - 1) // every
    for r in runs[1:]:
        for (a0, an, at), (b0, bn, bt) in zip(runs[0], r):
            assert bits_equal(a0, b0) and bits_equal(an, bn) and at == bt


def test_monitor_changes_no_bit_of_a_predict_run():
    import torch
    g = load_golden("beam_coarse_P2")
    r = g["ranks"][1]
    dofs = r["loc_dof_shared"]
    table = torch.from_numpy(np.random.default_rng(3).standard_normal((40, dofs.size)) * 1e-5).cuda()
    out = []
    for every in (None, 1, 7):
        pl = splan.StepPlan(_K(r), r["F"], r["lM"], r["dirichlet"], g["dt"], float(g["alpha"]))
        pl.step(30, splan.MODE_LOCAL)
        if every:
            pl.set_energy(64, every)
        pl.set_prediction(dofs, table.data_ptr(), 40)
        pl.step(40, splan.MODE_PREDICT)
        pl.synchronize()
        out.append(pl.get_state())
    for o in out[1:]:
        assert bits_equal(o[0], out[0][0]) and bits_equal(o[1], out[0][1])


# ---- 2. against a numpy evaluation ----------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["beam_coarse_P1", "beam_coarse_P3"])
def test_records_equal_numpy_evaluation(name):
    g = load_golden(name)
    N = 300
    plans, grp = make_plans(g)
    for pl in plans:
        pl.set_history(None, N + 1, 1)
        pl.set_energy(N + 1, 1)
    step(plans, grp, N + 1)
    own = owned_dofs(g)
    for q, pl in enumerate(plans):
        want = numpy_records(g, q, pl.read_history(), float(g["dt"]), float(g["alpha"]), own[q])
        assert_records_close(pl.read_energy(0, N), want, (name, q))


# ---- 3. the balance closes ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["beam_coarse_P1", "beam_coarse_P3"])
def test_balance_closes_over_10000_steps(name):
    g = load_golden(name)
    plans, grp = make_plans(g)
    for pl in plans:
        pl.set_energy(200, 50)
    step(plans, grp, 10000)
    b = balance(plans)
    assert b.size == 200 and b["step"][-1] == 9950
    rel = np.abs(b["residual"]).max() / scale(b)
    print(f"\n{name}: max |residual| / max(|E|, W, D) over 10000 steps = {rel:.3e}")
    assert rel <= 1e-10
    assert b["work_external"][-1] > 0 and b["work_damping"][-1] > 0


def test_energy_is_conserved_without_load_and_damping():
    g = load_golden("beam_coarse_P1")
    r = g["ranks"][0]
    (pl,), _ = make_plans(g, alpha=0.0, zero_load=True)
    rng = np.random.default_rng(5)
    d0, dn = rng.standard_normal(r["F"].size) * 1e-4, rng.standard_normal(r["F"].size) * 1e-4
    d0[r["dirichlet"]] = 0.0
    dn[r["dirichlet"]] = 0.0
    pl.set_state(d0, dn, 0.0)
    pl.set_energy(100, 20)
    pl.step(2000, splan.MODE_LOCAL)
    b = balance([pl])
    E = b["kinetic_half"] + b["coupling"]
    drift = np.abs(E - E[0]).max() / abs(E[0])
    print(f"\nalpha = 0, F = 0: max relative drift of T + S over 2000 steps = {drift:.3e}")
    assert drift <= 1e-12
    assert np.all(b["work_external"] == 0.0) and np.all(b["work_damping"] == 0.0)


# ---- 4. determinism and the ring ----------------------------------------------------------------------------------
def test_records_bit_identical_across_launch_strategies_and_repeats():
    g = load_golden("beam_coarse_P1")
    N = 61
    recs = []
    for how in ("per_step", "graph", "graph", "host"):
        (pl,), _ = make_plans(g)
        pl.set_energy(N, 1)
        if how == "host":                                   # the reference's loop: state uploaded every call
            n = pl.n_dof
            d0, dn, t = np.zeros(n), np.zeros(n), 0.0
            for _ in range(N):
                d1 = pl.step_host(d0, dn, t, splan.MODE_LOCAL)
                dn, d0, t = d0, d1.copy(), t + float(g["dt"])
        else:
            pl.step(N, splan.MODE_LOCAL, splan.LAUNCH_PER_STEP if how == "per_step" else splan.LAUNCH_GRAPH)
            pl.synchronize()
        recs.append(pl.read_energy())
    assert recs[0].size == N
    for r in recs[1:]:
        assert records_equal(r, recs[0])


def _host_staged_step(plans):
    """one synchronised step of all plans, messages through host memory (saa_plan_step_begin_host / _end_host)"""
    L = splan.lib()
    staged = []
    for pl in plans:
        nb, off = pl.halo_layout()
        send = np.zeros(max(int(off[-1]), 1))
        splan._check(L.saa_plan_step_begin_host(pl.h, splan._p(send)), "begin_host")
        staged.append((nb.tolist(), off, send))
    for q, pl in enumerate(plans):
        nb, off, _ = staged[q]
        recv = np.zeros(max(int(off[-1]), 1))
        for k, b in enumerate(nb):
            nbb, offb, sendb = staged[b]
            kk = nbb.index(q)
            recv[off[k]:off[k + 1]] = sendb[offb[kk]:offb[kk + 1]]
        splan._check(L.saa_plan_step_end_host(pl.h, splan._p(recv)), "end_host")


def test_records_bit_identical_between_group_and_host_staged_transport():
    g = load_golden("beam_coarse_P3")
    N = 40
    plans, grp = make_plans(g)
    hplans, _ = make_plans(g, group=False)
    for pl in plans + hplans:
        pl.set_energy(N, 1)
    step(plans, grp, N)
    for _ in range(N):
        _host_staged_step(hplans)
    for a, b in zip(plans, hplans):
        b.synchronize()
        assert bits_equal(a.d0(), b.d0())
        assert records_equal(a.read_energy(), b.read_energy())


def test_ring_and_every_semantics():
    g = load_golden("beam_coarse_P1")
    (pl,), _ = make_plans(g)
    pl.step(5, splan.MODE_LOCAL)
    pl.set_energy(4, 3)                                    # step 5 arms; records at steps 6, 9, 12, ...
    pl.step(20, splan.MODE_LOCAL)                          # steps 5..24
    pl.synchronize()
    assert pl.energy_count == 7
    with pytest.raises(splan.SaaError, match="overwritten"):
        pl.read_energy(0, 7)
    with pytest.raises(splan.SaaError, match="out of bounds"):
        pl.read_energy(3, 5)
    r = pl.read_energy(3, 4)
    assert r["step"].tolist() == [15, 18, 21, 24]
    assert np.all(r["energy_at_arm"] == r["energy_at_arm"][0])
    # set_state keeps the work sums; re-arming resets them
    W = r["work_external"][-1]
    d0, dn, tn = pl.get_state()
    pl.set_state(d0, dn, tn)
    pl.step(3, splan.MODE_LOCAL)
    assert pl.read_energy(pl.energy_count - 1, 1)["work_external"][0] > W
    pl.set_energy(4, 1)
    pl.step(2, splan.MODE_LOCAL)
    r = pl.read_energy()
    assert r.size == 2 and r["work_external"][0] == 0.0 and r["step"][0] == 28


# ---- 5. PREDICT -----------------------------------------------------------------------------------------------------
def test_predict_with_the_exact_table_reproduces_sync_and_a_perturbed_one_injects_energy():
    import torch
    g = load_golden("beam_coarse_P2")
    N = 400
    plans, grp = make_plans(g)
    for q, pl in enumerate(plans):
        pl.set_history(g["ranks"][q]["loc_dof_shared"], N, 1)
        pl.set_energy(N, 1)
    step(plans, grp, N, splan.MODE_SYNC)
    tables = [pl.read_history() for pl in plans]
    b_sync = balance(plans)
    own = owned_dofs(g)
    for perturb in (0.0, 1e-3):
        pplans, pgrp = make_plans(g)
        keep = []
        rng = np.random.default_rng(17)
        for q, pl in enumerate(pplans):
            t = tables[q] * (1.0 + perturb * rng.standard_normal(tables[q].shape))
            keep.append(torch.from_numpy(t).cuda())
            pl.set_history(None, N, 1)
            pl.set_energy(N, 1)
            pl.set_prediction(g["ranks"][q]["loc_dof_shared"], keep[-1].data_ptr(), N)
        step(pplans, pgrp, N, splan.MODE_PREDICT)
        b = balance(pplans)
        if perturb == 0.0:
            for pl, ref in zip(pplans, plans):
                assert bits_equal(pl.d0(), ref.d0())
            s = scale(b_sync)
            for f in splan.ENERGY_FIELDS[2:] + ("residual",):
                assert np.abs(b[f] - b_sync[f]).max() <= F_REL * s, f
        else:
            H = [pl.read_history() for pl in pplans]
            want = splan.energy_balance([numpy_records(g, q, np.vstack([H[q], H[q][-1:]]), float(g["dt"]), float(g["alpha"]), own[q])
                                         for q in range(2)])
            s = scale(want)
            got_res, want_res = b["residual"][:N - 1], want["residual"][:N - 1]
            print(f"\nperturbed prediction table: residual grows to {np.abs(want_res).max() / s:.3e} of max(|E|, W, D)")
            assert np.abs(got_res - want_res).max() <= F_REL * s
            assert np.abs(want_res[-50:]).max() > 1e3 * np.abs(b_sync["residual"]).max()


# ---- 6. scale: device set-up ----------------------------------------------------------------------------------------
def test_structured_m24_balance_and_graph_determinism():
    from saa_b200 import device_setup as ds
    recs = []
    for launch in (splan.LAUNCH_PER_STEP, splan.LAUNCH_GRAPH):
        plans, _ = ds.build_structured_in_process(24, 1)
        pl = plans[0]
        pl.set_energy(50, 10)
        pl.step(500, splan.MODE_LOCAL, launch)
        pl.synchronize()
        recs.append(pl.read_energy())
        pl.close()
    assert recs[0].size == 50 and records_equal(recs[0], recs[1])
    b = splan.energy_balance([recs[0]])
    rel = np.abs(b["residual"]).max() / scale(b)
    print(f"\nm = 24 (1.13 M DOF), 500 steps: max |residual| / max(|E|, W, D) = {rel:.3e}")
    assert rel <= 1e-10


# ---- 7. refusals ----------------------------------------------------------------------------------------------------
def test_refusals_and_launch_count_after_disarm():
    g = load_golden("beam_coarse_P1")
    (pl,), _ = make_plans(g)

    def launches_per_step():
        a = pl.kernel_launches
        pl.step(1, splan.MODE_LOCAL, splan.LAUNCH_PER_STEP)
        return pl.kernel_launches - a

    base = launches_per_step()
    with pytest.raises(splan.SaaError, match="every"):
        pl.set_energy(8, 0)
    pl.set_energy(8, 1)
    assert launches_per_step() == base + 1
    with pytest.raises(splan.SaaError, match="persistent"):
        pl.step(4, splan.MODE_LOCAL, splan.LAUNCH_PERSISTENT)
    with pytest.raises(splan.SaaError, match="MATFREE"):
        pl.set_option(splan.OPT_MATFREE, 1)
    pl.set_energy(0)
    assert launches_per_step() == base
    pl.step(4, splan.MODE_LOCAL, splan.LAUNCH_PERSISTENT)   # available again
    pl.synchronize()


# ---- 8. peer transport ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("transport", ["peer", "nccl"])
@pytest.mark.parametrize("name", ["beam_coarse_P2", "mid_np2"])
def test_peer_and_nccl_records_equal_group_records(transport, name):
    """two processes (sharing this GPU when the box has one): the records of the synchronised steps over the peer
    (three-kernel form) / NCCL transport equal those of the in-process group transport bit for bit"""
    import subprocess
    if transport == "nccl" and splan.device_count() < 2:
        pytest.skip("NCCL needs one GPU per process")
    if name.startswith("mid_") and not os.path.isfile(os.path.join(ROOT, "tests", "golden", name + ".npz")):
        pytest.skip("mid-size fixture not generated")
    port = 29400 + (os.getpid() + len(name) + len(transport)) % 150
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "energy_dist_worker.py"), transport, name]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count(f"energy ok ({transport})") == 2
