"""Cost of the on-device energy monitor (StepPlan.set_energy) on one GPU.

For the structured cantilever at m = 24 (1.13 M DOF) and m = 111 (104 M DOF), device set-up, one partition:
monitor off, every = 1 and every = 100 are timed alternately in one run (CUDA events on the plan's stream around
--steps graph-launched steps, after 3 untimed steps, --repeats rounds).  Every timed run starts from the same state,
so the final states of the three configurations must be bit-identical; the probe checks that, and reports the
largest |balance residual| / max(|E|, W, D) of the every = 1 records.  The card's name and power limit are read in
the same run.

    python profiles/energy_probe.py [--meshes 24 111] [--steps 20] [--repeats 5] [--out profiles/energy]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clk = [s.strip() for s in q.split(",")]
        return dict(gpu=name, power_limit=power, sm_clock_max=clk)
    except Exception as e:                          # the timings stand without it, but say so
        return dict(gpu="unknown", power_limit="unknown", error=str(e))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--meshes", type=int, nargs="+", default=[24, 111])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "energy"))
    a = ap.parse_args()
    import torch
    import saa_b200  # noqa: F401
    from saa_b200 import device_setup, plan as splan
    if not torch.cuda.is_available():
        raise SystemExit("energy_probe: no CUDA device")
    os.makedirs(a.out, exist_ok=True)
    configs = [("off", 0), ("every_1", 1), ("every_100", 100)]
    result = dict(card(), steps=a.steps, repeats=a.repeats, launch="graph", meshes={})
    for m in a.meshes:
        pl, info = device_setup.build_structured_rank(m, 0, 1, device_index=0)
        stream = torch.cuda.ExternalStream(pl.stream, device=torch.device("cuda", 0))
        pl.step(40, splan.MODE_LOCAL)                # a start state away from rest
        d0 = torch.empty(pl.n_dof, dtype=torch.float64, device="cuda")
        dn = torch.empty_like(d0)
        tn = pl.get_state_dev(d0.data_ptr(), dn.data_ptr())
        fin = torch.empty_like(d0)
        ref_bits, same, times, residual = None, True, {c: [] for c, _ in configs}, None
        for r in range(a.repeats):
            for cfg, every in configs:
                pl.set_state_dev(d0.data_ptr(), dn.data_ptr(), tn)
                pl.set_energy(a.steps + 3 if every else 0, max(every, 1))
                pl.step(3, splan.MODE_LOCAL)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                pl.step(a.steps, splan.MODE_LOCAL)
                e1.record(stream)
                pl.synchronize()
                times[cfg].append(e0.elapsed_time(e1) / a.steps)
                pl.get_state_dev(fin.data_ptr(), None)
                bits = fin.view(torch.int64).clone()
                if ref_bits is None:
                    ref_bits = bits
                else:
                    same = same and bool(torch.equal(bits, ref_bits))
                if every == 1 and r == 0:
                    b = splan.energy_balance([pl.read_energy()])
                    s = max(np.abs(b["total"]).max(), np.abs(b["work_external"]).max(), np.abs(b["work_damping"]).max())
                    residual = float(np.abs(b["residual"]).max() / s)
        pl.set_energy(0, 1)
        med = {c: float(np.median(v)) for c, v in times.items()}
        result["meshes"][str(m)] = dict(
            n_dof=int(info["n_global_nodes"]) * 3, ms_per_step=times, median_ms_per_step=med,
            overhead_every_1=med["every_1"] / med["off"] - 1.0, overhead_every_100=med["every_100"] / med["off"] - 1.0,
            states_bit_identical=same, max_rel_residual_every_1=residual)
        print(json.dumps({m: result["meshes"][str(m)]}), flush=True)
        pl.close()
        del d0, dn, fin
        torch.cuda.empty_cache()
    path = os.path.join(a.out, "energy_probe.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print(f"[energy_probe] {result['gpu']} at {result['power_limit']}: wrote {path}")


if __name__ == "__main__":
    main()
