"""Cost of the multigrid-preconditioned static solve (StepPlan.solve_static(precond=StructuredMultigrid), DESIGN.md §7d).

For the structured cantilever at m = 24, 48 and 96 (1.13 M, 8.8 M and 67.8 M DOF), device set-up, one partition:
  * set-up time of the hierarchy (host clock around StructuredMultigrid(...), which ends synchronised: coarse plans,
    tables, coarsest Cholesky inverse, block inverses, lambda estimates), lambda per level and the bytes it holds;
  * a full solve to --rtol: iterations, recurrence and true residual, wall time (host clock around the call; median
    of --repeats solves after one untimed);
  * ms per outer iteration: CUDA events around solves with rtol = 0 (never met) and max_iter = --base and --base +
    --iters, the difference over --iters iterations, check_every = 10, graph launches;
  * how one iteration splits across the levels: one solve under torch.profiler (a run of its own), kernel time summed
    per level (a level's kernels are told apart by their grid size) and for the outer CG kernels;
  * the block-Jacobi solve at m = 24 (--bj-meshes) for comparison, and the device-to-device copy rate of the same run.
The card's name and power limit are read in the same run.

    python profiles/multigrid_probe.py [--meshes 24 48 96] [--out profiles/multigrid]
"""
import argparse
import json
import os
import sys
import tempfile
import time
from collections import defaultdict

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "profiles")]
from energy_probe import card  # noqa: E402
from static_probe import copy_rate_GBps  # noqa: E402
from stress_probe import timed  # noqa: E402

LEVEL_KERNELS = ("saa_k_mg_residual", "saa_k_mg_cheb", "saa_k_mg_prolong", "saa_k_mg_restrict", "saa_k_mg_coarse")


def level_split(pl, mg, rtol):
    """kernel microseconds of one solve per level (by the grid of the level kernels) and for the outer iteration"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = pl.solve_static(rtol=rtol, precond=mg)
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        ev = [e for e in json.load(open(path))["traceEvents"] if e.get("cat") == "kernel"]
    grids = sorted({e["args"]["grid"][0] for e in ev if "saa_k_mg_residual" in e["name"]}, reverse=True)
    coarse = {e["args"]["grid"][0] for e in ev if "saa_k_mg_restrict" in e["name"]} - set(grids)
    level_of = {g: l for l, g in enumerate(grids + sorted(coarse, reverse=True))}
    us = defaultdict(float)
    for e in ev:
        if any(k in e["name"] for k in LEVEL_KERNELS):
            l = len(mg.levels) - 1 if "saa_k_mg_coarse" in e["name"] else level_of.get(e["args"]["grid"][0], -1)
            us[f"level_{l}_m{mg.levels[l][0]}" if l >= 0 else "unassigned"] += e["dur"]
        elif "saa_k_" in e["name"]:
            us["outer_cg"] += e["dur"]
        else:
            us["other"] += e["dur"]
    return res.iterations, {k: v / 1e3 for k, v in us.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--meshes", type=int, nargs="+", default=[24, 48, 96])
    ap.add_argument("--bj-meshes", type=int, nargs="*", default=[24])
    ap.add_argument("--base", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--rtol", type=float, default=1e-8)
    ap.add_argument("--copy-gb", type=float, default=8.0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "multigrid"))
    a = ap.parse_args()
    import torch
    import saa_b200  # noqa: F401
    from saa_b200 import device_setup, multigrid
    if not torch.cuda.is_available():
        raise SystemExit("multigrid_probe: no CUDA device")
    os.makedirs(a.out, exist_ok=True)
    result = dict(card(), rtol=a.rtol, base=a.base, iters=a.iters, repeats=a.repeats, copy_GBps=copy_rate_GBps(a.copy_gb),
                  meshes={}, block_jacobi={})
    print(f"[multigrid_probe] {result['gpu']} at {result['power_limit']}: copy rate {result['copy_GBps']:.0f} GB/s", flush=True)
    for m in a.meshes:
        t0 = time.perf_counter()
        pl, info = device_setup.build_structured_rank(m, 0, 1, device_index=0)
        t_plan = time.perf_counter() - t0
        torch.cuda.empty_cache()
        t0 = time.perf_counter()
        mg = multigrid.StructuredMultigrid(pl, m, info["local_nodes"])
        torch.cuda.synchronize()
        t_setup = time.perf_counter() - t0
        stream = torch.cuda.ExternalStream(pl.stream, device=torch.device("cuda", 0))
        pl.solve_static(rtol=a.rtol, precond=mg)
        walls, full = [], None
        for _ in range(a.repeats):
            t0 = time.perf_counter()
            full = pl.solve_static(rtol=a.rtol, precond=mg)
            walls.append(time.perf_counter() - t0)
        solve = lambda k: pl.solve_static(rtol=0.0, max_iter=k, check_every=10, precond=mg)
        solve(a.base + a.iters)
        t_lo = timed(stream, a.repeats, lambda: solve(a.base))
        t_hi = timed(stream, a.repeats, lambda: solve(a.base + a.iters))
        ms_it = (float(np.median(t_hi)) - float(np.median(t_lo))) / a.iters
        its_prof, split = level_split(pl, mg, a.rtol)
        r = dict(n_dof=pl.n_dof, levels=mg.levels, lambda_max=mg.lambda_max, hierarchy_bytes=mg.bytes,
                 fine_matrix_bytes=pl.matrix_bytes, plan_setup_s=t_plan, hierarchy_setup_s=t_setup,
                 iterations=full.iterations, converged=full.converged, rel_residual=full.rel_residual,
                 rel_residual_true=full.rel_residual_true, solve_wall_s=walls, median_solve_wall_s=float(np.median(walls)),
                 solve_ms_base=t_lo, solve_ms_base_plus_iters=t_hi, ms_per_iteration=ms_it,
                 profiled_solve_iterations=its_prof, profiled_kernel_ms=split,
                 profiled_kernel_ms_per_iteration={k: v / max(its_prof, 1) for k, v in split.items()},
                 max_abs_uz=float(full.x[2::3].abs().max()), finite=bool(torch.isfinite(full.x).all()))
        result["meshes"][str(m)] = r
        print(json.dumps({m: {k: v for k, v in r.items() if not isinstance(v, (list, dict))}}), flush=True)
        print(json.dumps({m: split}), flush=True)
        if m in a.bj_meshes:
            pl.solve_static(rtol=a.rtol, max_iter=200_000, check_every=200)
            t0 = time.perf_counter()
            bj = pl.solve_static(rtol=a.rtol, max_iter=200_000, check_every=200)
            wall = time.perf_counter() - t0
            result["block_jacobi"][str(m)] = dict(iterations=bj.iterations, converged=bj.converged, rel_residual_true=bj.rel_residual_true,
                                                  wall_s=wall, rel_diff_to_mg=float((bj.x - full.x).norm() / full.x.norm()))
            print(json.dumps({f"block_jacobi_{m}": result["block_jacobi"][str(m)]}), flush=True)
        mg.close()
        pl.close()
        del full
        torch.cuda.empty_cache()
    path = os.path.join(a.out, "multigrid_probe.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print(f"[multigrid_probe] {result['gpu']} at {result['power_limit']}: wrote {path}")


if __name__ == "__main__":
    main()
