#!/usr/bin/env python
"""bench.py — DOF-steps/s of the explicit FE time step on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--refine M] [--partition slabs|blocks|metis] [--impl native|reference]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is ONE explicit time step (one pass of Dynamic_solver.py:9-34 over the whole mesh): force K.u,
central-difference update, Dirichlet clamp and — for N > 1 — the shared-node force exchange.

Workload (config.workload): the 25 x 1 x 1 cantilever of Mesh_info/beam_US.geo as a structured tet mesh with m cells
per unit length.  ONE mesh for every N (strong scaling): m = 111, 104 M DOF — BASELINE.json configs[3], the mesh the
north star's ">= 80 % at 8 GPUs" is quoted on; it fits one B200 (38 GB).  configs[1] (m = 24, ~1 M DOF, one GPU) and
configs[2] (m = 65, ~20 M DOF) are measured in the same run and reported under `also`; configs[4] (m = 65,
synchronization-avoiding mode) under `sync_avoiding` for N > 1.

Timing protocol: set-up, graph instantiation (done inside the library at plan finalisation), --warmup steps from rest
and an untimed spin-up of >= --spin-ms of steps come first; the spin-up's steps are then undone (the warm-up's state
is put back), and EXACTLY --steps steps are timed, as --repeats back-to-back parts (default 5), each bracketed by
barrier + synchronize and timed with CUDA events on the plan's stream, max over ranks per part; `value` is the MEDIAN
part's rate (min / max reported).  The timed steps thus end in the state --warmup + --steps steps from rest reach,
which --dump-outputs DIR writes out.  Inputs are larger than L2 (see config.l2).

`value`   whole-job DOF-steps/s with the state resident in HBM.
`e2e`     the same metric through the reference-facing call saa_step_host_ex — one parallel_explicit_solver_dis_pre
          evaluation per call with (d0, dn) in pinned HOST memory and d1 returned to HOST memory every step.
`roofline` algorithmic bytes of the fused force+update kernel in the format it streams / median step time, vs the
          measured HBM copy bandwidth.
`cpu_baseline` CPU baselines on a bounded sample (an x-slab of the same mesh): the OpenMP C port of the oracle on all
          cores, and the reference's own numpy/scipy statement sequence on P single-threaded processes.
`parity`  (N > 1) golden histories of the unmodified reference reproduced bit for bit through the attached transport
          before anything is timed, and a cross-path check (fused peer kernel == three-kernel form == NCCL transport,
          bitwise) on the timed mesh afterwards.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=0, help="timed time steps (0: 2000 for m <= 32, 500 for m <= 80, else 100)")
    ap.add_argument("--warmup", type=int, default=10, help="untimed steps from rest before the timed steps")
    ap.add_argument("--refine", "--m", dest="m", type=int, default=0,
                    help="cells per unit length of the 25x1x1 beam (0: 111 = the 104 M-DOF mesh); spell it --refine under torchrun")
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--repeats", type=int, default=0, help="back-to-back parts the timed steps run in, each timed on its own (0: min(5, steps))")
    ap.add_argument("--spin-ms", type=float, default=300.0, help="untimed spin-up of steps after the warm-up; the state is put back afterwards")
    ap.add_argument("--e2e-steps", type=int, default=0, help="timed host-call steps (0: 200 for m <= 32, 60 for m <= 80, else 20)")
    ap.add_argument("--launch", default="auto", choices=["auto", "per_step", "graph", "persistent"])
    ap.add_argument("--setup", default="device", choices=["device", "host"], help="where the problem is assembled")
    ap.add_argument("--partition", default="slabs", choices=["slabs", "blocks", "metis"],
                    help="N > 1: x-slabs of whole hexahedron layers, a px x py x pz block grid (8 -> 2x2x2), or METIS_PartMeshDual "
                         "(host mesh, m <= 27)")
    ap.add_argument("--blocks", default="", help="--partition blocks: the process grid PXxPYxPZ (default: cuts along x, then y, then z)")
    ap.add_argument("--kernel", default="assembled", choices=["assembled", "matfree"],
                    help="matfree (one GPU): kernel K5, f_int = sum_e B^T D B u_e evaluated element by element, node-owned accumulation — a "
                         "throughput / low-memory mode reported with its own roofline and its measured difference from the assembled path")
    ap.add_argument("--cpu-seconds", type=float, default=0.0, help="CPU time budget per baseline (0: 10 s native arm, 15 s reference arm)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the extra measurements of the other BASELINE configs")
    ap.add_argument("--no-parity", action="store_true", help="N > 1: skip the parity pre-check and the cross-path check")
    ap.add_argument("--transport", default="peer", choices=["peer", "nccl"], help="halo transport for N > 1")
    ap.add_argument("--sync-avoid", default="auto", help="N > 1: time the synchronization-avoiding loop (BASELINE config 5) on the "
                    "m = 65 mesh; comma list of re-sync periods k, 0 = never re-synchronise (the reference's behaviour); "
                    "auto = 0,10,50; off = skip")
    ap.add_argument("--balance", action="store_true", help="N > 1: size the x-slabs by each GPU's measured speed")
    ap.add_argument("--filter-size", type=int, default=25, help="n_s of the LSTM refill (Online_predictor.py:57 uses 150; shortened so "
                    "that warm-up + three refill blocks fit the bench)")
    ap.add_argument("--train-epochs", type=int, default=20)
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the state they computed (d0, dn, tn of StepPlan.get_state) to DIR/<name>.npy; "
                         "vectors longer than 2**21 / N values are a fixed, seeded sample")
    return ap.parse_args()


M_DEFAULT = 111


def default_steps(m):
    return 2000 if m <= 32 else (500 if m <= 80 else 100)


def workload_name(m, n_dof, n_el):
    cfg = {24: "BASELINE config 2 (~1M DOF, single B200, fp64)", 65: "BASELINE config 3 (~20M DOF over 2/4/8 B200)",
           111: "BASELINE config 4 (~100M DOF strong-scaling sweep 1/2/4/8)"}.get(m, "custom refinement")
    return f"structured 25x1x1 cantilever (Mesh_info/beam_US.geo box) m={m}: {n_dof} DOF, {n_el} tets; {cfg}"


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "50"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            t = [x.strip() for x in line.split(",")]
            if len(t) < 7:
                continue
            try:
                sm.append(float(t[0])); mx.append(float(t[1])); pw.append(float(t[2]))
            except ValueError:
                continue
            for nm, v in zip(names, t[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            # median over the samples taken under load (power above half of the maximum seen)
            busy = [s for s, p in zip(sm, pw) if p > 0.5 * max(pw)] or sm
            out.update(sm_mhz=float(np.median(busy)), sm_max_mhz=float(max(mx)), power_w_max=float(max(pw)),
                       reasons=sorted(reasons), samples=len(sm), samples_under_load=len(busy))
        return out


# ---- problem set-up -------------------------------------------------------------------------------------------
def setup_host(m, size, rank, local, make_plan=True, nx=None, all_ranks=False, exact_rowsum=None):
    """Host set-up (numpy/scipy, the reference's own arithmetic): METIS partition for N > 1 (x-slabs for a sample slab)."""
    import saa_b200  # noqa: F401
    from saa_b200 import device_setup, mesh, partition, problem
    pts, cells, fac = mesh.structured_beam(m, nx=nx)
    if size == 1:
        ep, part = np.zeros(len(cells), dtype=np.int64), "none"
    elif nx is not None:
        layer = np.arange(len(cells), dtype=np.int64) // (6 * m * m)
        ep, part = (layer * size) // nx, f"{size} x-slabs"
    else:
        ep, part = partition.metis_part_mesh(cells, len(pts), size), "METIS_PartMeshDual(ncommon=3)"
    pb = problem.build_problem(pts, cells, fac, ep, size, ranks=None if all_ranks else [rank], exact_rowsum=exact_rowsum)
    q = pb["ranks"][rank]
    pl = problem.make_plan(q, pb["dt"], problem.DAMP_DEFAULT, size, device=local) if make_plan else None
    csr = dict(K=q["K"], F=q["F"], lM=q["lM"], dirichlet=q["dirichlet"], nodes=q["nodes"])
    return pl, dict(dt=float(pb["dt"]), n_nodes=len(pts), n_elem=len(cells), part=part, csr=csr, problem=pb,
                    assembly="host (numpy/scipy, bit-exact with the reference's assembly)")


def setup_device(m, size, rank, local, partition="slabs", grid=None, keep_mesh=False):
    """Device set-up (saa_b200.device_setup): mesh part, numbering, K6 assembly and the plan, all on the GPU."""
    import saa_b200  # noqa: F401
    from saa_b200 import device_setup
    if partition == "metis" and size > 1:
        from saa_b200 import mesh, partition as part_mod
        if m > 27:
            raise SystemExit("--partition metis: serial METIS on the host mesh is practical up to m = 27 (3 M elements); use blocks")
        pts, cells, fac = mesh.structured_beam(m)
        ep = part_mod.metis_part_mesh(cells, len(pts), size)
        pl, info = device_setup.build_mesh_rank(pts, cells, fac, ep, rank, size, device_index=local)
        pname = "METIS_PartMeshDual(ncommon=3) on the host mesh"
    else:
        kind = "blocks" if (partition == "blocks" and size > 1) else "slabs"
        pl, info = device_setup.build_structured_rank(m, rank, size, device_index=local, partition=kind, grid=grid, keep_mesh=keep_mesh)
        g = (grid or device_setup.block_grid(size)) if kind == "blocks" else None
        pname = ("none" if size == 1 else
                 f"{size} x-slabs of whole hexahedron layers (what a k-way cut of a 25:1:1 beam gives)" if kind == "slabs" else
                 f"{g[0]}x{g[1]}x{g[2]} blocks of hexahedra (up to {min(size - 1, 7)} neighbours per rank, nodes held by up to {size} ranks)")
    halo = info.get("halo")
    return pl, dict(mesh=({k: info[k] for k in ("cells_loc", "pts", "lame")} if keep_mesh else None),
                    dt=float(info["dt"]), n_nodes=info["n_global_nodes"], n_elem=info["n_global_elem"], part=pname,
                    neighbours=(len(halo["neighbours"]) if halo else 0), shared_nodes=(len(halo["shared_pos"]) if halo else 0),
                    assembly="device (saa_assemble_stiffness_dev, closed-form element matrices)")


# ---- CPU baselines (the ONLY legs that touch oracle/) ------------------------------------------------------------
def cpu_sample(m, size):
    """Bounded sample of the m-mesh for the CPU runs: an x-slab of the same cross-section (same element shapes, same
    stencil) with about a million tetrahedra, or the whole mesh when it is smaller."""
    nx_full = 25 * m
    nx = min(nx_full, max(2 * size, int(round(1.0e6 / (6 * m * m)))))
    return nx, nx_full


def cpu_baselines(m, size, seconds, steps, warmup):
    """(C-port record, numpy/scipy record) on the sample slab, `size` partitions for the numpy/scipy processes."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import fem_oracle
    import numpy_step
    nx, nx_full = cpu_sample(m, size)
    _, info = setup_host(m, size, 0, 0, make_plan=False, nx=nx, all_ranks=True, exact_rowsum=False)
    pb = info["problem"]
    n_dof = 3 * info["n_nodes"]
    what = (f"an x-slab of {nx} of the {nx_full} hexahedron layers of the m={m} mesh ({n_dof} DOF, {info['n_elem']} tets)"
            if nx < nx_full else f"the whole m={m} mesh ({n_dof} DOF)")
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    # (1) C port of the oracle, serial problem, all OpenMP threads: R repeats of `steps` steps, median
    if size == 1:
        serial = pb["ranks"][0]
    else:
        _, i1 = setup_host(m, 1, 0, 0, make_plan=False, nx=nx, exact_rowsum=False)
        serial = i1["problem"]["ranks"][0]
    K = serial["K"]
    o = fem_oracle.OracleProblem(info["n_nodes"], [dict(K_indptr=K.indptr, K_indices=K.indices, K_data=K.data, F=serial["F"],
                                                        lM=serial["lM"], dirichlet=serial["dirichlet"], nodes=serial["nodes"])],
                                 info["dt"], 0.5)
    o.run(max(3, warmup))
    t0 = time.perf_counter(); o.run(steps); t1 = time.perf_counter() - t0
    reps = int(max(3, min(50, seconds / max(t1, 1e-6))))
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter(); o.run(steps); ts.append(time.perf_counter() - t0)
    o.close()
    threads = int(os.environ.get("OMP_NUM_THREADS", cores))
    port = dict(value=n_dof * steps / float(np.median(ts)), unit="DOF-steps/s", cores=threads, kind="port",
                sample=f"{reps} repeats of {steps} time steps (median) on {what} with oracle/fem_oracle.c (OpenMP over rows, "
                       f"{threads} threads, serial problem)")
    # (2) the reference's own statement sequence: scipy csr.dot + numpy update (+ syn_cpus), one thread per rank
    ranks = [dict(K_indptr=pb["ranks"][r]["K"].indptr, K_indices=pb["ranks"][r]["K"].indices, K_data=pb["ranks"][r]["K"].data,
                  F=pb["ranks"][r]["F"], lM=pb["ranks"][r]["lM"], dirichlet=pb["ranks"][r]["dirichlet"], nodes=pb["ranks"][r]["nodes"])
             for r in range(size)]
    ns = max(20, steps) if size == 1 else 20
    secs, _ = numpy_step.run_ranks(ranks, info["n_nodes"], info["dt"], 0.5, ns, warmup=2)
    nps = dict(value=n_dof * ns / secs, unit="DOF-steps/s", cores=size, kind="numpy-scipy", ms_per_step=1e3 * secs / ns,
               sample=f"{ns} time steps on {what} in {size} x-slab partition(s): {size} single-threaded process(es) running the "
                      f"statement sequence of Dynamic_solver.py:12-32 (scipy csr.dot + numpy update"
                      + (", evaluated twice, with syn_cpus of Distributed_tools.py:77-92: pickled gather to rank 0, Python-list "
                         "node_to_dof, broadcast of the global vector)" if size > 1 else ")"))
    if size > 1:
        secs2, _ = numpy_step.run_ranks(ranks, info["n_nodes"], info["dt"], 0.5, ns, warmup=2, model=True)
        nps["value_without_syn_cpus"] = n_dof * ns / secs2
    return port, nps, dict(n_dof=n_dof, n_elem=info["n_elem"], nx=nx, nx_full=nx_full, what=what, dt=info["dt"])


def run_reference(args, emit):
    """--impl reference: the reference's CPU path on the host cores, same workload (a bounded sample of it), no GPU, none
    of the repo's native code except oracle/ (the reference is pure Python and does not exist on the GPU box;
    oracle/fem_oracle.c is its pinned bit-exact port, oracle/numpy_step.py its numpy/scipy statement sequence).
    Rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    os.environ.pop("OMP_NUM_THREADS", None)   # torchrun pins it to 1; the baseline may use every core
    m = args.m or M_DEFAULT
    steps = args.steps or 20
    warmup = max(3, args.warmup)
    port, nps, smp = cpu_baselines(m, args.gpus, args.cpu_seconds or 15.0, steps, warmup)
    nxf, ny = 25 * m, m
    n_dof_full, n_el_full = 3 * (nxf + 1) * (ny + 1) * (ny + 1), 6 * nxf * ny * ny
    line = {"impl": "reference", "metric": "DOF-steps/sec", "value": port["value"], "unit": "DOF-steps/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": 1e3 * smp["n_dof"] / port["value"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(m, n_dof_full, n_el_full), "sample": smp["what"],
                       "note": "value = the faster of the two CPU baselines (OpenMP C port on all cores); cpu_baseline_numpy_scipy is "
                               "the reference's own numpy/scipy path on --gpus single-threaded processes; ms_per_step is per step of the sample"},
            "cpu_baseline": port, "cpu_baseline_numpy_scipy": nps,
            "e2e": {"value": port["value"], "unit": "DOF-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ---- timing ------------------------------------------------------------------------------------------------------
def time_repeats(pl, torch, stream, steps, mode, launch, barrier, max_over_ranks, repeats, spin_ms, warmup):
    """`warmup` steps, a spin-up of >= spin_ms, the state put back to where the warm-up left it, then exactly `steps`
    timed steps in `repeats` (0: min(5, steps)) back-to-back parts -> (ms per step of each part [max over ranks],
    kernel launches of all parts).  The timed steps thus always continue from the warm-up's state, whatever the
    spin-up did, and the state they leave depends on the arguments alone."""
    if warmup > 0:
        pl.step(warmup, mode, launch)
    repeats = min(repeats or 5, steps)
    parts = [steps // repeats + (i < steps % repeats) for i in range(repeats)]
    d0 = torch.empty(pl.n_dof, dtype=torch.float64, device="cuda")
    dn = torch.empty_like(d0)
    tn = pl.get_state_dev(d0.data_ptr(), dn.data_ptr())
    pl.synchronize()
    barrier()
    t0 = time.perf_counter()
    n_spin = 0
    while True:                                   # the same call pattern as the timed parts
        pl.step(parts[0], mode, launch)
        pl.synchronize()
        n_spin += 1
        if max_over_ranks(1.0 if (time.perf_counter() - t0) * 1e3 >= spin_ms else 0.0) >= 1.0 or n_spin >= 10000:
            break
    pl.set_state_dev(d0.data_ptr(), dn.data_ptr(), tn)
    del d0, dn
    out, l0 = [], pl.kernel_launches
    for k in parts:
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        pl.step(k, mode, launch)
        e1.record(stream)
        pl.synchronize()
        barrier()
        out.append(max_over_ranks(e0.elapsed_time(e1)) / k)
    return out, pl.kernel_launches - l0


DUMP_SAMPLE = 2 ** 21   # values per vector over all ranks: d0 + dn stay at 32 MB


def dump_outputs(pl, torch, out_dir, rank, world):
    """What a caller of the timed steps receives (StepPlan.get_state: d0, dn, tn) as float64 .npy files in out_dir,
    suffixed _rank<r> for N > 1.  A vector longer than DUMP_SAMPLE / N is sampled at sorted indices drawn from a
    generator seeded with its length, so that two builds of the project write the same entries."""
    n = pl.n_dof
    d0 = torch.empty(n, dtype=torch.float64, device="cuda")
    dn = torch.empty_like(d0)
    tn = pl.get_state_dev(d0.data_ptr(), dn.data_ptr())
    k = DUMP_SAMPLE // world
    idx = None if n <= k else np.unique(np.random.default_rng(n).integers(0, n, k))
    os.makedirs(out_dir, exist_ok=True)
    sfx = f"_rank{rank}" if world > 1 else ""
    sel = (lambda v: v) if idx is None else (lambda v: v[torch.from_numpy(idx).to(v.device)])
    for name, v in (("d0", sel(d0)), ("dn", sel(dn))):
        np.save(os.path.join(out_dir, f"{name}{sfx}.npy"), v.cpu().numpy())
    np.save(os.path.join(out_dir, f"tn{sfx}.npy"), np.float64(tn))
    return {"dir": out_dir, "files": [f"{x}{sfx}.npy" for x in ("d0", "dn", "tn")], "n_dof_rank0": n,
            "sampled_entries": n if idx is None else int(idx.size), "sample_seed": None if idx is None else n}


def time_host_calls(pl, torch, dist, world, mode, dt, e2e_steps, barrier, max_over_ranks, n_dof_global):
    """The loop of Data_prepare.py:223-235 with host arrays through StepPlan.step_host (saa_step_host_ex): d1 comes back
    in page-locked memory owned by the plan's pool and is rotated into d_0 / d_n, so from the second call on every vector
    that crosses PCIe is pinned.  The call is synchronous: wall clock covers copies + kernels.  Afterwards the result is
    compared bit for bit with the same number of device-resident steps from the same state."""
    from saa_b200 import plan as splan  # noqa: F401
    n_dof_local = pl.n_dof
    s0, sn, tn0 = pl.get_state()
    h0, hn, tn = s0, sn, tn0
    for _ in range(3):
        h1 = pl.step_host(h0, hn, tn, mode)
        hn, h0 = h0, h1
        tn = tn + dt
    barrier()
    skipped0 = getattr(pl, "host_uploads_skipped", 0)
    w0 = time.perf_counter()
    for _ in range(e2e_steps):
        h1 = pl.step_host(h0, hn, tn, mode)          # d1 lands in host memory every call
        hn, h0 = h0, h1                              # d_n = d_0; d_0 = d1 (Data_prepare.py:233-234)
        tn = tn + dt
    pl.synchronize()
    barrier()
    ms_e2e = max_over_ranks((time.perf_counter() - w0) * 1e3)
    dn_skipped = getattr(pl, "host_uploads_skipped", 0) - skipped0
    h2d = (8 * n_dof_local * (2 * e2e_steps - dn_skipped)) / e2e_steps
    pipe_k, _, pipe_need = pl.host_pipe_info(mode)
    pipe = {"chunks": int(pipe_k), "max_lag_chunks": int(max(pipe_need - np.arange(pipe_k))) if pipe_k else None,
            "pinned_result_buffers": len(getattr(pl, "_pinned_pool", []))}
    pl.set_state(s0, sn, tn0)
    pl.step(3 + e2e_steps, mode)
    pl.synchronize()
    same = bool(np.array_equal(pl.d0().view(np.uint64), h0.view(np.uint64)))
    if world > 1:
        tt = torch.tensor([1.0 if same else 0.0], device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MIN)
        same = bool(tt.item() == 1.0)
    return {"value": n_dof_global * e2e_steps / (ms_e2e * 1e-3), "unit": "DOF-steps/s",
            "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 8 * n_dof_local,
            "steps": e2e_steps, "ms_per_step": ms_e2e / e2e_steps, "dn_uploads_skipped": dn_skipped,
            "pipeline": pipe, "bit_identical_to_resident_steps": same}


def bits_equal_dev(torch, a, b):
    return bool(torch.equal(a.view(torch.int64), b.view(torch.int64)))


def parity_fixture(world, rank, local, transport, torch, dist):
    """Golden histories of the UNMODIFIED reference (tests/golden/beam_coarse_P{N}.npz, oracle/gen_golden.py) through the
    attached transport of this very launch: N partitions on N GPUs, compared as uint64."""
    import scipy.sparse as sp
    from saa_b200 import maps, multi, plan as splan
    name = f"beam_coarse_P{world}"
    path = os.path.join(ROOT, "tests", "golden", name + ".npz")
    if not os.path.isfile(path):
        return {"fixture": None, "bit_identical": None, "note": f"no fixture for {world} partitions"}
    z = np.load(path)
    n = z[f"r{rank}_F"].size
    K = sp.csr_matrix((z[f"r{rank}_K_data"], z[f"r{rank}_K_indices"], z[f"r{rank}_K_indptr"]), shape=(n, n))
    lists = [z[f"r{q}_nodes"] for q in range(world)]
    pl = splan.StepPlan(K, z[f"r{rank}_F"], z[f"r{rank}_lM"], z[f"r{rank}_dirichlet"], z["dt"], float(z["alpha"]), device=local,
                        halo=maps.halo_plan(rank, world, lists), rank=rank, size=world)
    tr = multi.attach_transport(pl, transport)
    ok, done, checked = True, 0, []
    for s in [int(x) for x in z["steps"]]:
        pl.step(s - done, splan.MODE_SYNC)
        pl.synchronize()
        done = s
        ok = ok and np.array_equal(pl.d0().view(np.uint64), z[f"hist_{s}_r{rank}"].view(np.uint64))
        checked.append(s)
    flag = torch.tensor([1.0 if ok else 0.0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    pl.close()
    return {"fixture": f"tests/golden/{name}.npz (unmodified reference, {world} METIS partitions)", "transport": tr,
            "steps_compared": checked, "bit_identical": bool(flag.item() >= 1.0)}


def parity_mid(world, rank, local, transport, torch, dist):
    """Mid-size case (3 x 1 x 1 beam, m = 14, METIS partition stored in the fixture: several boundary slices and shared-row units
    per rank, nodes held by >= 3 ranks): device set-up + fused peer step vs histories the CPU oracle produced from the
    same device-assembled matrices (tests/golden/mid_np{N}.npz, oracle/gen_golden_mid.py)."""
    from saa_b200 import device_setup, mesh, multi, plan as splan
    path = os.path.join(ROOT, "tests", "golden", f"mid_np{world}.npz")
    if not os.path.isfile(path):
        return None
    z = np.load(path)
    m = int(z["m"])
    pts, cells, fac = mesh.structured_beam(m, length=int(z["length"]))
    pl, info = device_setup.build_mesh_rank(pts, cells, fac, z["epart"].astype(np.int64), rank, world, device_index=local)
    tr = multi.attach_transport(pl, transport)
    ok, done = True, 0
    for s in [int(x) for x in z["steps"]]:
        pl.step(s - done, splan.MODE_SYNC)
        pl.synchronize()
        done = s
        ok = ok and np.array_equal(pl.d0().view(np.uint64), z[f"hist_{s}_r{rank}"].view(np.uint64))
    flag = torch.tensor([1.0 if ok else 0.0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    halo = info["halo"]
    out = {"fixture": f"tests/golden/mid_np{world}.npz (CPU oracle on the device-assembled matrices, METIS)", "transport": tr,
           "n_dof": 3 * len(pts), "steps_compared": [int(x) for x in z["steps"]], "neighbours_rank0": len(halo["neighbours"]),
           "shared_nodes_rank0": len(halo["shared_pos"]), "bit_identical": bool(flag.item() >= 1.0)}
    pl.close()
    return out


def cross_path_check(pl, torch, dist, k=24):
    """On the timed mesh, from the state the timed run left: k more synchronised steps with (a) the fused peer kernel,
    (b) its three-kernel form, (c) the NCCL transport — all three must agree bit for bit on every rank."""
    from saa_b200 import plan as splan
    n = pl.n_dof
    d0 = torch.empty(n, dtype=torch.float64, device="cuda")
    dn = torch.empty(n, dtype=torch.float64, device="cuda")
    tn = pl.get_state_dev(d0.data_ptr(), dn.data_ptr())
    res = {}

    def run(tag):
        pl.set_state_dev(d0.data_ptr(), dn.data_ptr(), tn)
        pl.step(k, splan.MODE_SYNC)
        pl.synchronize()
        out = torch.empty(n, dtype=torch.float64, device="cuda")
        pl.get_state_dev(out.data_ptr(), None)
        res[tag] = out

    run("fused")
    pl.set_option(splan.OPT_PEER_FUSED, 0)
    run("three_kernel")
    pl.set_option(splan.OPT_PEER_FUSED, 1)
    ids = [splan.nccl_unique_id() if dist.get_rank() == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    pl.init_nccl(ids[0])
    pl.set_option(splan.OPT_PREFER_NCCL, 1)
    run("nccl")
    pl.set_option(splan.OPT_PREFER_NCCL, 0)
    pl.set_state_dev(d0.data_ptr(), dn.data_ptr(), tn)
    ok = bits_equal_dev(torch, res["fused"], res["three_kernel"]) and bits_equal_dev(torch, res["fused"], res["nccl"])
    moved = not bits_equal_dev(torch, res["fused"], d0)
    flag = torch.tensor([1.0 if (ok and moved) else 0.0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    return {"steps": k, "paths": ["peer fused (1 launch/step)", "peer three-kernel", "nccl send/recv three-kernel"],
            "bit_identical": bool(flag.item() >= 1.0)}


def train_surrogate(torch, hist, input_size, n_s, n_p, n_f, epochs, device, seed):
    """The Model_training.py flow (:19-24, 65-71, 100-139) on a short synchronised history of this rank's shared DOFs:
    windows from the first `cut_off` fraction strided by n_s, joint [-1, 0] scaling, Adam(5e-4), MSE, recursive decoding.
    Returns (model, scale_max, scale_min, first / last epoch loss)."""
    sys.path.insert(0, os.path.join(ROOT, "synchronization-avoiding-algorithms_b200"))
    from Tools.DNN_tools import LSTM_encoder_decoder, MyDataset, Scale_to_zero_one, model_train, windows_from_history
    torch.manual_seed(seed)
    np.random.seed(seed)
    # training windows start anywhere in the history (the reference strides a single comb; all n_s combs are used here so that
    # a short history yields enough samples)
    Xs, Ys = [], []
    H = hist.float()
    for off in range(n_s):
        T = H[off::n_s]
        if T.shape[0] < n_p + n_f:
            continue
        W = T.unfold(0, n_p + n_f, 1).permute(0, 2, 1)
        Xs.append(W[:, :n_p]); Ys.append(W[:, n_p:])
    X, Y = torch.cat(Xs).contiguous(), torch.cat(Ys).contiguous()
    X, Y, smax, smin = Scale_to_zero_one(X, Y)
    model = LSTM_encoder_decoder(input_size, 50, 2, True, 0.0, 0.0).to(device)
    crit = torch.nn.MSELoss()
    opt = torch.optim.Adam(model.parameters(), lr=5e-4)
    loader = torch.utils.data.DataLoader(MyDataset(X, Y), batch_size=32, shuffle=True)
    first = last = None
    for ep in range(epochs):
        tot = model_train(device, model, loader, crit, opt, n_f)[0] / max(1, len(loader))
        first = tot if first is None else first
        last = tot
    return model.eval(), float(smax), float(smin), first, last, int(X.shape[0])


def time_sync_avoiding(args, torch, dist, world, rank, local, barrier, max_over_ranks, transport):
    """BASELINE config 5 on the m = 65 mesh: the loop of Online_predictor.py:251-318 on the device.  The surrogate is the
    reference's LSTM encoder-decoder (2-layer bidirectional encoder, hidden 50, n_past = n_future = 20), TRAINED here the
    way Model_training.py does on a short synchronised history; a true exchange runs every k steps (k = 0: never again
    after the warm-up, the reference's behaviour).  Reports throughput and the relative L2 error of the modelled
    displacement against the fully synchronised run at the end of every refill block."""
    from saa_b200 import multi, plan as splan, sync_avoiding
    m = 65
    pl, info = setup_device(m, world, rank, local, "slabs")
    multi.attach_transport(pl, transport)
    stream = torch.cuda.ExternalStream(pl.stream, device=torch.device("cuda", local))
    n_dof_global = 3 * info["n_nodes"]
    hp = pl._halo_desc
    dofs = (3 * np.asarray(hp["shared_pos"], dtype=np.int64)[:, None] + np.arange(3)[None, :]).ravel()
    n_p = n_f = 20
    n_s = args.filter_size
    warm, block, n_blocks = n_p * n_s, n_f * n_s, 3
    total = warm + n_blocks * block
    dev = f"cuda:{local}"
    # (1) fully synchronised run: history of the shared DOFs (training data + the truth for the error), state at block ends
    pl.set_history(dofs, capacity=total, save_every=1)
    truth_norm, truth = [], []
    pl.step(warm, splan.MODE_SYNC)
    for b in range(n_blocks):
        pl.step(block, splan.MODE_SYNC)
        pl.synchronize()
        d = torch.empty(pl.n_dof, dtype=torch.float64, device=dev)
        pl.get_state_dev(d.data_ptr(), None)
        truth.append(d)
    hist = torch.empty((total, dofs.size), dtype=torch.float64, device=dev)
    pl.read_history_dev(0, total, hist.data_ptr())
    pl.synchronize()
    t0 = time.perf_counter()
    # Model_training.py:65-71 trains on the first cut_off fraction of a fully synchronised run, which in the reference's flow
    # (1e5 synchronised steps, cut_off 0.5, online run from t = 0) covers the steps the online run later predicts; same here:
    # the synchronised history of exactly the range the online runs below cover, windows strided by n_s
    model, smax, smin, l0, l1, n_win = train_surrogate(torch, hist, int(dofs.size), n_s=n_s, n_p=n_p, n_f=n_f,
                                                     epochs=args.train_epochs, device=dev, seed=1234 + rank)
    torch.cuda.synchronize()
    t_train = time.perf_counter() - t0
    out = {"workload": workload_name(m, n_dof_global, info["n_elem"]), "n_past": n_p, "n_future": n_f, "filter_size": n_s,
           "input_size_rank0": int(dofs.size), "hidden": 50,
           "model": "LSTM_encoder_decoder(input, 50, 2, bidirectional), fp32, trained on-device (Adam 5e-4, MSE, recursive decoding) on the "
                    "synchronised warm-up history of this rank's shared DOFs; scale_max/min from the training windows",
           "training": {"epochs": args.train_epochs, "windows_rank0": n_win, "history_steps": total, "loss_first_epoch": l0,
                        "loss_last_epoch": l1, "seconds_rank0": t_train},
           "runs": []}
    zeros = np.zeros(pl.n_dof)
    for k in [int(x) for x in (("0,10,50" if args.sync_avoid == "auto" else args.sync_avoid).split(","))]:
        pl.set_history(None, 0, 1)
        pl.set_state(zeros, zeros, 0.0)
        run = sync_avoiding.SyncAvoidingRun([pl], pl, [dofs], [model], [(smax, smin)], n_p, n_f, n_s, device=dev, resync_every=(k or None))
        run.i = 0
        run.run(warm)
        pl.synchronize()
        errs = []
        barrier()
        ms_tot = 0.0
        for b in range(n_blocks):
            barrier()
            w0 = time.perf_counter()
            run.run(warm + (b + 1) * block)
            pl.synchronize()
            barrier()
            ms_tot += max_over_ranks((time.perf_counter() - w0) * 1e3)     # wall clock: includes the LSTM inference of the block
            d = torch.empty(pl.n_dof, dtype=torch.float64, device=dev)
            pl.get_state_dev(d.data_ptr(), None)
            num = torch.tensor([float(((d - truth[b]) ** 2).sum()), float((truth[b] ** 2).sum())], dtype=torch.float64, device=dev)
            dist.all_reduce(num)
            errs.append(float(torch.sqrt(num[0] / num[1]).item()))
        nst = n_blocks * block
        out["runs"].append({"resync_every": k, "steps": nst, "ms_per_step": ms_tot / nst, "value": n_dof_global * nst / (ms_tot * 1e-3),
                            "unit": "DOF-steps/s", "lstm_ms_per_block_rank0": 1e3 * run.t_predict / max(1, run.n_predict),
                            "error_vs_sync": {"rel_l2_displacement_at_block_ends": errs,
                                              "note": "all DOFs of all ranks (shared nodes counted once per holder) vs the fully synchronised run"}})
    # fully synchronised reference speed of the same mesh in the same run
    ms, _ = time_repeats(pl, torch, stream, 2500, splan.MODE_SYNC, splan.LAUNCH_AUTO, barrier, max_over_ranks, 5, 100.0, 10)
    out["synchronised_every_step"] = {"value": n_dof_global / (float(np.median(ms)) * 1e-3), "ms_per_step": float(np.median(ms))}
    pl.close()
    return out


def main():
    args = parse()
    # keep stdout clean for the single JSON line: libraries (NCCL's version banner, torchrun notices) write to it
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)

    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs: the native implementation's timed steps only")
        run_reference(args, emit)
        return
    import torch
    import torch.distributed as dist
    import saa_b200  # noqa: F401
    from saa_b200 import multi, plan as splan

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1 and args.gpus > 1:
        raise SystemExit("bench.py --gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the time-step path has no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    m = args.m or M_DEFAULT
    steps = args.steps or default_steps(m)
    e2e_steps = args.e2e_steps or (200 if m <= 32 else (60 if m <= 80 else 20))
    want_cpu = (not args.no_cpu_baseline) and world == 1
    launch = {"auto": splan.LAUNCH_AUTO, "per_step": splan.LAUNCH_PER_STEP, "graph": splan.LAUNCH_GRAPH,
              "persistent": splan.LAUNCH_PERSISTENT}[args.launch]

    # ---- parity before anything is timed (N > 1): the reference's golden histories through this launch's transport ----
    parity = None
    if world > 1 and not args.no_parity:
        parity = {"golden": parity_fixture(world, rank, local, args.transport, torch, dist)}
        mid = parity_mid(world, rank, local, args.transport, torch, dist)
        if mid is not None:
            parity["mid_size"] = mid
        bad = [k for k, v in parity.items() if v.get("bit_identical") is False]
        if bad:
            if rank == 0:
                emit({"error": "parity pre-check failed; nothing was timed", "parity": parity})
            dist.barrier()
            dist.destroy_process_group()
            raise SystemExit(3)

    t_setup = time.time()
    balance = None
    if args.setup == "host":
        pl, info = setup_host(m, world, rank, local)
        info.update(neighbours=None, shared_nodes=None)
    else:
        grid = tuple(int(x) for x in args.blocks.lower().split("x")) if args.blocks else None
        pl, info = setup_device(m, world, rank, local, args.partition, grid=grid, keep_mesh=(args.kernel == "matfree"))
        if world > 1 and args.balance and args.partition == "slabs":
            from saa_b200 import device_setup
            st0 = torch.cuda.ExternalStream(pl.stream, device=torch.device("cuda", local))
            ms0, _ = time_repeats(pl, torch, st0, 300, splan.MODE_LOCAL, splan.LAUNCH_AUTO, lambda: torch.cuda.synchronize(),
                                  lambda x: float(x), 3, 50.0, 10)
            speed = torch.tensor([pl.n_dof / float(np.median(ms0))], dtype=torch.float64, device="cuda")
            allv = [torch.zeros_like(speed) for _ in range(world)]
            dist.all_gather(allv, speed)
            balance = [float(v.item()) for v in allv]
            pl.close()
            del pl
            torch.cuda.empty_cache()
            device_setup.set_layer_weights(balance)
            pl, info = setup_device(m, world, rank, local, args.partition)
            balance = [b / max(balance) for b in balance]
    transport = multi.attach_transport(pl, args.transport) if world > 1 else "none"
    t_setup = time.time() - t_setup
    n_dof_global = 3 * info["n_nodes"]
    n_dof_local = pl.n_dof
    dtv = info["dt"]
    mode = splan.MODE_SYNC if world > 1 else splan.MODE_LOCAL
    stream = torch.cuda.ExternalStream(pl.stream, device=torch.device("cuda", local))

    matfree = None
    if args.kernel == "matfree":
        if world > 1 or args.setup != "device":
            raise SystemExit("--kernel matfree: one GPU, device set-up (synchronised multi-partition steps stream the assembled matrix)")
        # measured difference from the assembled (parity) path first: the same 1000 steps from rest with both kernels
        msh = info["mesh"]
        pl.set_matfree(msh["cells_loc"], msh["pts"], *msh["lame"])
        k_cmp = 1000 if m <= 32 else 200
        pl.step(k_cmp, splan.MODE_LOCAL)
        pl.synchronize()
        a = torch.empty(n_dof_local, dtype=torch.float64, device="cuda")
        pl.get_state_dev(a.data_ptr(), None)
        z = torch.zeros(n_dof_local, dtype=torch.float64, device="cuda")
        pl.set_state_dev(z.data_ptr(), z.data_ptr(), 0.0)
        mat_bytes = pl.matrix_bytes
        pl.set_option(splan.OPT_MATFREE, 2)          # matrix-free from here on; the assembled matrix is released
        pl.step(k_cmp, splan.MODE_LOCAL)
        pl.synchronize()
        b = torch.empty(n_dof_local, dtype=torch.float64, device="cuda")
        pl.get_state_dev(b.data_ptr(), None)
        matfree = {"rel_l2_vs_assembled": float(((a - b).norm() / a.norm()).item()), "after_steps": k_cmp,
                   "bytes_streamed_besides_vectors": pl.matfree_bytes, "assembled_matrix_bytes": mat_bytes,
                   "hbm_in_use_gb_after_release": (torch.cuda.mem_get_info()[1] - torch.cuda.mem_get_info()[0]) / 1e9}
        del a, b, z, msh
        info["mesh"] = None
        torch.cuda.empty_cache()

    # ---- device-resident timing --------------------------------------------------------------------
    sampler = ClockSampler(local) if rank == 0 else None
    reps, launches = time_repeats(pl, torch, stream, steps, mode, launch, barrier, max_over_ranks, args.repeats, args.spin_ms, args.warmup)
    ms = float(np.median(reps))
    dumped = dump_outputs(pl, torch, args.dump_outputs, rank, world) if args.dump_outputs else None
    ms_local = None
    if world > 1:   # the same shards stepped WITHOUT the exchange (MODEL=True arithmetic): what the halo costs per step
        rl, _ = time_repeats(pl, torch, stream, 5 * steps, splan.MODE_LOCAL, launch, barrier, max_over_ranks, 5, 50.0, 0)
        ms_local = float(np.median(rl))

    # ---- end to end through the reference-facing host call -----------------------------------------
    e2e = time_host_calls(pl, torch, dist, world, mode, dtv, e2e_steps, barrier, max_over_ranks, n_dof_global)
    clocks = sampler.stop() if sampler else None

    # ---- cross-path check on the timed mesh (N > 1, peer transport) ----------------------------------
    if parity is not None and transport == "peer":
        parity["cross_path"] = cross_path_check(pl, torch, dist)

    # ---- roofline of the fused force+update kernel (largest shard bounds the step) ------------------
    # algorithmic bytes of the format actually streamed (node-block sliced ELL): 76 B per stored 3x3 block (nine
    # fp64 values + one int32 column-node id) + slice offsets + Dirichlet mask words + five fp64 vector streams.
    # The scalar-CSR figure of SURVEY.md §8d (12 B per stored entry + 4 B per row pointer + 40 B per row) is given
    # beside it as csr_equivalent.
    nnz = pl.nnz
    alg_bytes = max_over_ranks(float((pl.matfree_bytes if matfree else pl.matrix_bytes) + pl.vector_bytes))
    csr_bytes = max_over_ranks(float(nnz * 12 + (n_dof_local + 1) * 4 + 5 * 8 * n_dof_local))
    step_s = ms * 1e-3
    peak, peak_src = measured_peak()
    achieved = alg_bytes / step_s / 1e9
    traffic, traffic_src = None, None
    tf = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.isfile(tf):
        try:
            t = json.load(open(tf)).get(f"m{m}_n{world}")
            if t:
                traffic, traffic_src = t["dram_bytes_per_launch"], t["source"]
        except Exception:
            pass
    mat_mb = pl.matrix_bytes / 1e6
    nb_cnt, sh_cnt = info.get("neighbours"), info.get("shared_nodes")
    blocks_per_node = (pl.padded_entries / 9) / (n_dof_local / 3)
    pl.close()
    del pl
    torch.cuda.empty_cache()

    also = None
    if not args.no_also and args.setup == "device" and m == M_DEFAULT and not matfree:
        also = []
        # N > 1: config 3 is timed inside time_sync_avoiding (synchronised_every_step) unless that leg is off
        todo = [(24, 1, 2000), (65, 1, 500)] if world == 1 else ([(65, world, 500)] if args.sync_avoid in ("off", "", "none") else [])
        for (m2, w2, k2) in todo:
            try:
                pl2, info2 = setup_device(m2, w2, rank, local, "slabs")
                if w2 > 1:
                    multi.attach_transport(pl2, args.transport)
                st2 = torch.cuda.ExternalStream(pl2.stream, device=torch.device("cuda", local))
                md2 = splan.MODE_SYNC if w2 > 1 else splan.MODE_LOCAL
                r2, _ = time_repeats(pl2, torch, st2, 5 * k2, md2, launch, barrier, max_over_ranks, 5, 200.0, 10)
                ms2 = float(np.median(r2))
                b2 = max_over_ranks(float(pl2.matrix_bytes + pl2.vector_bytes))
                e2 = time_host_calls(pl2, torch, dist, w2, md2, info2["dt"], 200 if m2 <= 32 else 60, barrier, max_over_ranks, 3 * info2["n_nodes"])
                also.append({"workload": workload_name(m2, 3 * info2["n_nodes"], info2["n_elem"]), "n_gpus": w2, "steps": k2, "repeats": len(r2),
                             "value": 3 * info2["n_nodes"] / (ms2 * 1e-3), "ms_per_step": ms2,
                             "ms_per_step_min": min(r2), "ms_per_step_max": max(r2),
                             "roofline_frac": b2 / (ms2 * 1e-3) / 1e9 / peak, "nnz_per_row": pl2.nnz / pl2.n_dof, "e2e": e2})
                pl2.close()
                del pl2
                torch.cuda.empty_cache()
            except Exception as e:
                also.append({"m": m2, "error": str(e)[:300]})

    sync_avoid = None
    if world > 1 and args.sync_avoid not in ("off", "", "none"):
        try:
            sync_avoid = time_sync_avoiding(args, torch, dist, world, rank, local, barrier, max_over_ranks, args.transport)
        except Exception as e:
            import traceback
            traceback.print_exc(file=sys.stderr)
            sync_avoid = {"error": str(e)[:300]}

    if rank == 0:
        line = {
            "metric": "DOF-steps/sec", "value": n_dof_global / (ms * 1e-3), "unit": "DOF-steps/s",
            "n_gpus": world, "steps": steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "timing": {"repeats": len(reps), "statistic": "median over the `repeats` back-to-back parts of the `steps` timed steps of ms per "
                                                          "step, each part = max over ranks of CUDA-event time",
                       "ms_per_step_min": min(reps), "ms_per_step_max": max(reps),
                       "spin_up_ms": args.spin_ms, "graphs": "instantiated at plan finalisation / transport attach, before any timing"},
            "config": {"workload": workload_name(m, n_dof_global, info["n_elem"]),
                       "partition": info["part"], "neighbours_rank0": nb_cnt, "shared_nodes_rank0": sh_cnt,
                       "balance": balance, "transport": transport, "assembly": info["assembly"],
                       "nnz_per_row": nnz / n_dof_local, "local_dof_rank0": n_dof_local,
                       "launch": args.launch, "dt": dtv, "setup_s": round(t_setup, 1), "ms_per_step_without_exchange": ms_local,
                       "l2": "inputs larger than L2: matrix stream per step per GPU = %.0f MB vs 126 MB L2" % mat_mb},
            "e2e": dict(e2e, call="saa_step_host_ex (one parallel_explicit_solver_dis_pre evaluation per call, host d0/dn in, d1 out in page-locked "
                                   "memory that the caller rotates into d0/dn; dn = the previous call's d0 array is recognised and not uploaded "
                                   "again; upload, step and download of the row chunks overlap on three streams)"),
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "bytes_per_launch": alg_bytes,
                         "bytes_formula": ("16*elements + 4*incidence lanes + 24*nodes + 8*(slices+1) + 4*rows/32 + 32*rows + 8*nodes" if matfree else
                                           "76*blocks + 8*(slices+1) + 4*rows/32 + 32*rows + 8*nodes (largest shard; lumped mass streamed per node)"),
                         "csr_equivalent": {"bytes_per_launch": csr_bytes, "formula": "12*nnz + 4*(rows+1) + 40*rows",
                                            "achieved": csr_bytes / step_s / 1e9, "frac": csr_bytes / step_s / 1e9 / peak},
                         "blocks_per_node": blocks_per_node,
                         "kernel": ("saa_k_step_matfree (K5: element-wise B^T D B u_e, node-owned, fused with the update) — fp64/L1-bound, "
                                    "see profiles/" if matfree else "saa_k_step (fused K.u + central-difference update + Dirichlet mask)")},
            "clocks": clocks,
        }
        if matfree:
            line["matfree"] = matfree
            line["config"]["kernel"] = "matfree (K5) — NOT the parity path; see line['matfree'].rel_l2_vs_assembled"
        if dumped is not None:
            line["dumped_outputs"] = dumped
        if parity is not None:
            line["parity"] = parity
        if also is not None:
            line["also"] = also
        if sync_avoid is not None:
            line["sync_avoiding"] = sync_avoid
        if want_cpu:
            os.environ.pop("OMP_NUM_THREADS", None)
            port, nps, smp = cpu_baselines(m, 1, args.cpu_seconds or 10.0, 20, 3)
            line["cpu_baseline"] = port
            line["cpu_baseline_numpy_scipy"] = nps
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
