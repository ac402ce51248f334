"""Cost of the static solve (StepPlan.solve_static, csrc/saa_static.cuh) on one GPU.

For the structured cantilever at m = 24 (1.13 M DOF) and m = 111 (104 M DOF), device set-up, one partition:
  * time per CG iteration: CUDA events on the plan's stream around solves with rtol = 0 (never met) and max_iter =
    --base and --base + --iters, after --warmup untimed solves; the difference over --iters iterations (>= 200) takes
    out the set-up of a call (preconditioner, work vectors, final residual apply).  check_every = 50, graph launches;
  * the algorithmic bytes of one iteration from the plan's shapes (matrix_bytes of the step layout, and per row
    x, r, p, q read and x, r, z written in the update, p gathered and q written in the apply, z and p read and p
    written in the direction update, 16 B of block inverse, two free-row mask reads; the p gathers counted once; the
    few slice-padding rows not counted) over that time, as a
    fraction of the device-to-device copy rate measured in the same run (a --copy-gb buffer copied with torch);
  * the graph-launched time step measured in the same run, for scale;
  * a full solve to --rtol: iterations and wall time (host clock around the call, which ends synchronised).  At the
    largest mesh it runs at most --full-seconds worth of iterations (from the measured time per iteration); when that
    is not enough it is recorded as not converged, with the residual reached.
The card's name and power limit are read in the same run.

    python profiles/static_probe.py [--meshes 24 111] [--iters 200] [--out profiles/static]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "profiles")]
from energy_probe import card  # noqa: E402
from stress_probe import timed  # noqa: E402


def copy_rate_GBps(gb, reps=10):
    """device-to-device copy rate (read + write bytes per second) of a buffer of `gb` GB"""
    import torch
    n = int(gb * 1e9) // 8
    a = torch.ones(n, dtype=torch.float64, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    torch.cuda.synchronize()
    t = timed(torch.cuda.current_stream(), reps, lambda: b.copy_(a))
    del a, b
    torch.cuda.empty_cache()
    return 2 * 8 * n / (float(np.median(t)) * 1e-3) / 1e9


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--meshes", type=int, nargs="+", default=[24, 111])
    ap.add_argument("--base", type=int, default=50)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rtol", type=float, default=1e-8)
    ap.add_argument("--full-seconds", type=float, default=300.0)
    ap.add_argument("--copy-gb", type=float, default=8.0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "static"))
    a = ap.parse_args()
    import torch
    import saa_b200  # noqa: F401
    from saa_b200 import device_setup, plan as splan
    if not torch.cuda.is_available():
        raise SystemExit("static_probe: no CUDA device")
    os.makedirs(a.out, exist_ok=True)
    result = dict(card(), base=a.base, iters=a.iters, repeats=a.repeats, rtol=a.rtol, copy_GBps=copy_rate_GBps(a.copy_gb), meshes={})
    print(f"[static_probe] {result['gpu']} at {result['power_limit']}: copy rate {result['copy_GBps']:.0f} GB/s", flush=True)
    for m in a.meshes:
        pl, info = device_setup.build_structured_rank(m, 0, 1, device_index=0)
        torch.cuda.empty_cache()
        stream = torch.cuda.ExternalStream(pl.stream, device=torch.device("cuda", 0))
        solve = lambda k: pl.solve_static(rtol=0.0, max_iter=k, check_every=50)
        for _ in range(a.warmup):
            solve(a.base + a.iters)
        t_lo = timed(stream, a.repeats, lambda: solve(a.base))
        t_hi = timed(stream, a.repeats, lambda: solve(a.base + a.iters))
        ms_it = (float(np.median(t_hi)) - float(np.median(t_lo))) / a.iters
        pl.step(10, splan.MODE_LOCAL, splan.LAUNCH_GRAPH)
        pl.synchronize()
        t_step = [t / a.steps for t in timed(stream, 5, lambda: pl.step(a.steps, splan.MODE_LOCAL, splan.LAUNCH_GRAPH))]
        b_it = pl.matrix_bytes + 112 * pl.n_dof + 2 * (pl.n_dof // 8)
        free_before = torch.cuda.mem_get_info()[0]
        budget = 200_000 if m <= 32 else max(1000, int(a.full_seconds * 1e3 / ms_it))
        t0 = time.perf_counter()
        full = pl.solve_static(rtol=a.rtol, max_iter=budget, check_every=200)
        wall = time.perf_counter() - t0
        x = full.x
        r = dict(n_dof=pl.n_dof, matrix_bytes=pl.matrix_bytes, iteration_bytes=int(b_it),
                 solve_ms_base=t_lo, solve_ms_base_plus_iters=t_hi, ms_per_iteration=ms_it,
                 GBps_per_iteration=b_it / ms_it / 1e6, fraction_of_copy_rate=b_it / ms_it / 1e6 / result["copy_GBps"],
                 graph_step_ms=t_step, median_graph_step_ms=float(np.median(t_step)),
                 step_bytes=pl.matrix_bytes + pl.vector_bytes,
                 full_solve=dict(rtol=a.rtol, max_iter=budget, iterations=full.iterations, converged=full.converged,
                                 rel_residual=full.rel_residual, rel_residual_true=full.rel_residual_true, wall_s=wall,
                                 max_abs_uz=float(x[2::3].abs().max()), finite=bool(torch.isfinite(x).all())),
                 free_bytes_before_full_solve=int(free_before), free_bytes_after=int(torch.cuda.mem_get_info()[0]))
        result["meshes"][str(m)] = r
        print(json.dumps({m: {k: v for k, v in r.items() if not isinstance(v, list)}}), flush=True)
        pl.close()
        del x, full
        torch.cuda.empty_cache()
    path = os.path.join(a.out, "static_probe.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print(f"[static_probe] {result['gpu']} at {result['power_limit']}: wrote {path}")


if __name__ == "__main__":
    main()
