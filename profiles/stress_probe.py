"""Cost of stress recovery (StepPlan.element_stress / nodal_stress_partial) on one GPU.

For the structured cantilever at m = 24 (1.13 M DOF) and m = 111 (104 M DOF), device set-up with keep_mesh=True, one
partition, from a state 40 steps away from rest:
  * element kernel: CUDA events on the plan's stream around each of --evals calls of saa_plan_element_stress_dev after
    --warmup untimed ones.  A call also resets the detJ flag, reads it back and waits for the stream, so the per-call
    time includes that round trip; the kernel alone is taken from a torch.profiler pass run afterwards;
  * nodal kernel: the same around saa_plan_nodal_stress_dev (enqueued only: the events time the kernel);
  * the graph-launched step (--steps steps per event pair, --evals // 4 repeats), for scale.
Rates are algorithmic bytes over time, counted from the shapes:
  element  16 B connectivity read + 64 B written per element, 48 B of coordinates and displacement per node
  nodal    4 B per incidence (4 per element, slice padding not counted), 64 B per element row, 56 B written per node
Each node's and each element row's bytes are counted once; the repeated gathers of corner data and element rows are
not.  This is no DRAM measurement: neither DRAM traffic nor cache hit rates are read, so how many of those repeats
L1/L2 serve is not known.  The free device memory before and after the evaluations is recorded.  The card's name and
power limit are read in the same run.

    python profiles/stress_probe.py [--meshes 24 111] [--evals 20] [--warmup 3] [--steps 20] [--out profiles/stress]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "profiles")]
from energy_probe import card  # noqa: E402


def timed(stream, n, fn):
    """per-call milliseconds of n calls of fn, CUDA events on `stream`"""
    import torch
    out = []
    for _ in range(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        e1.record(stream)
        e1.synchronize()
        out.append(e0.elapsed_time(e1))
    return out


def profiled_kernel_us(pl, elem, nodal, n=5):
    """mean device time (us) of the two stress kernels from a torch.profiler pass"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            elem()
            nodal()
        pl.synchronize()
    res = {}
    for ev in prof.key_averages():
        for k in ("saa_k_stress_elem", "saa_k_stress_node"):
            if k in ev.key:
                tot = getattr(ev, "device_time_total", None)
                if tot is None:
                    tot = ev.cuda_time_total
                res[k] = dict(us=tot / max(ev.count, 1), count=ev.count)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--meshes", type=int, nargs="+", default=[24, 111])
    ap.add_argument("--evals", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "stress"))
    a = ap.parse_args()
    import torch
    import saa_b200  # noqa: F401
    from saa_b200 import device_setup, plan as splan
    if not torch.cuda.is_available():
        raise SystemExit("stress_probe: no CUDA device")
    os.makedirs(a.out, exist_ok=True)
    L = splan.lib()
    result = dict(card(), evals=a.evals, warmup=a.warmup, steps=a.steps, meshes={})
    for m in a.meshes:
        pl, info = device_setup.build_structured_rank(m, 0, 1, device_index=0, keep_mesh=True)
        pl.set_matfree(info["cells_loc"], info["pts"], *info["lame"])
        del info["cells_loc"], info["pts"]
        torch.cuda.empty_cache()
        stream = torch.cuda.ExternalStream(pl.stream, device=torch.device("cuda", 0))
        pl.step(40, splan.MODE_LOCAL)
        pl.synchronize()
        nE, nN = pl.n_elem, pl.n_dof // 3
        free_before = torch.cuda.mem_get_info()[0]
        elem = torch.empty((nE, 8), dtype=torch.float64, device="cuda")
        nod = torch.empty((nN, 7), dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        run_elem = lambda: splan._check(L.saa_plan_element_stress_dev(pl.h, elem.data_ptr()), "saa_plan_element_stress_dev")
        run_nod = lambda: splan._check(L.saa_plan_nodal_stress_dev(pl.h, elem.data_ptr(), nod.data_ptr()), "saa_plan_nodal_stress_dev")
        for _ in range(a.warmup):
            run_elem()
            run_nod()
        pl.synchronize()
        t_elem = timed(stream, a.evals, run_elem)
        t_nod = timed(stream, a.evals, run_nod)
        free_after = torch.cuda.mem_get_info()[0]
        kern = profiled_kernel_us(pl, run_elem, run_nod)
        t_step = timed(stream, max(a.evals // 4, 3), lambda: pl.step(a.steps, splan.MODE_LOCAL, splan.LAUNCH_GRAPH))
        t_step = [t / a.steps for t in t_step]
        vm = elem[:, 6]
        b_elem = 16 * nE + 64 * nE + 48 * nN
        b_nod = 4 * 4 * nE + 64 * nE + 56 * nN
        me, mn, ms = float(np.median(t_elem)), float(np.median(t_nod)), float(np.median(t_step))
        r = dict(n_dof=3 * nN, n_elem=nE, n_nodes=nN,
                 element=dict(ms_per_call=t_elem, median_ms_per_call=me, algorithmic_bytes=b_elem,
                              GBps_per_call=b_elem / me / 1e6),
                 nodal=dict(ms_per_call=t_nod, median_ms_per_call=mn, algorithmic_bytes=b_nod, GBps=b_nod / mn / 1e6),
                 profiler_kernel_us=kern, graph_step_ms=t_step, median_graph_step_ms=ms,
                 free_bytes_before=int(free_before), free_bytes_after=int(free_after),
                 output_bytes=int(elem.numel() * 8 + nod.numel() * 8),
                 max_von_mises=float(vm.max()), finite=bool(torch.isfinite(elem).all() and torch.isfinite(nod).all()))
        for k, b in (("saa_k_stress_elem", b_elem), ("saa_k_stress_node", b_nod)):
            if k in kern:
                kern[k]["GBps"] = b / kern[k]["us"] / 1e3
        result["meshes"][str(m)] = r
        print(json.dumps({m: {k: v for k, v in r.items() if not isinstance(v, list)}}), flush=True)
        pl.close()
        del elem, nod
        torch.cuda.empty_cache()
    path = os.path.join(a.out, "stress_probe.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print(f"[stress_probe] {result['gpu']} at {result['power_limit']}: wrote {path}")


if __name__ == "__main__":
    main()
