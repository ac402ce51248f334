"""Value coding of the stiffness planes (DESIGN.md §3) on one GPU: layout counters and the step kernel's variant table
with the coded layout and with every block-row raw (SAA_VALUE_CODE=0).

For the structured cantilever (device set-up, one partition) at each of --meshes: coded and raw plane counts,
streamed_matrix_bytes and matrix_bytes (the plane-masked layout without coding).  At each of --time-meshes, for every
schedule variant of --variants, a coded and a raw plan are built and timed alternately in one process (CUDA events on
the plan's stream around --steps graph-launched local steps, after 3 untimed steps, --repeats rounds, every round from
the same state); the final states of both layouts must be bit-identical.  Achieved bandwidth is computed from the
bytes each layout streams (streamed_matrix_bytes + vector_bytes).  The card's name and power limit are read in the
same run.

    python profiles/value_coding_probe.py [--meshes 24 65 111] [--time-meshes 24 111] [--variants 0 1 2 3 4 5]
                                          [--steps 20] [--repeats 5] [--out profiles/value_coding]
"""
import argparse
import gc
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


def build(m, code, variant=None):
    from saa_b200 import device_setup
    os.environ["SAA_VALUE_CODE"] = "1" if code else "0"
    if variant is None:
        os.environ.pop("SAA_KVARIANT", None)
    else:
        os.environ["SAA_KVARIANT"] = str(variant)
    try:
        return device_setup.build_structured_rank(m, 0, 1, device_index=0)
    finally:
        os.environ.pop("SAA_VALUE_CODE", None)
        os.environ.pop("SAA_KVARIANT", None)


def counters(pl):
    return dict(n_dof=pl.n_dof, value_planes=pl.value_planes, coded_planes=pl.coded_planes, raw_planes=pl.value_planes - pl.coded_planes,
                streamed_matrix_bytes=pl.streamed_matrix_bytes, matrix_bytes=pl.matrix_bytes, vector_bytes=pl.vector_bytes)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--meshes", type=int, nargs="+", default=[24, 65, 111])
    ap.add_argument("--time-meshes", type=int, nargs="+", default=[24, 111])
    ap.add_argument("--variants", type=int, nargs="+", default=[0, 1, 2, 3, 4, 5])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "value_coding"))
    a = ap.parse_args()
    import torch
    import saa_b200  # noqa: F401
    from saa_b200 import plan as splan
    if not torch.cuda.is_available():
        raise SystemExit("value_coding_probe: no CUDA device")
    os.makedirs(a.out, exist_ok=True)
    result = dict(card(), steps=a.steps, repeats=a.repeats, launch="graph", layouts={}, variants={})
    for m in a.meshes:
        pl, _ = build(m, True)
        c = counters(pl)
        c["streamed_over_matrix_bytes"] = c["streamed_matrix_bytes"] / c["matrix_bytes"]
        c["bytes_per_node_step"] = dict(coded=(c["streamed_matrix_bytes"] + c["vector_bytes"]) / (c["n_dof"] / 3),
                                        uncoded=(c["matrix_bytes"] + c["vector_bytes"]) / (c["n_dof"] / 3))
        result["layouts"][str(m)] = c
        print(json.dumps({m: c}), flush=True)
        pl.close()
        gc.collect()
        torch.cuda.empty_cache()
    for m in a.time_meshes:
        table = {}
        for v in a.variants:
            plans = {}
            for code in (True, False):
                plans["coded" if code else "raw"] = build(m, code, v)[0]
            start = None
            times = {k: [] for k in plans}
            ref_bits, same = None, True
            for r in range(a.repeats):
                for k, pl in plans.items():
                    stream = torch.cuda.ExternalStream(pl.stream, device=torch.device("cuda", 0))
                    if start is None:                  # a start state away from rest, shared by every run
                        pl.step(40, splan.MODE_LOCAL)
                        d0 = torch.empty(pl.n_dof, dtype=torch.float64, device="cuda")
                        dn = torch.empty_like(d0)
                        start = (d0, dn, pl.get_state_dev(d0.data_ptr(), dn.data_ptr()))
                    pl.set_state_dev(start[0].data_ptr(), start[1].data_ptr(), start[2])
                    pl.step(3, splan.MODE_LOCAL)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    pl.step(a.steps, splan.MODE_LOCAL)
                    e1.record(stream)
                    pl.synchronize()
                    times[k].append(e0.elapsed_time(e1) / a.steps)
                    fin = torch.empty_like(start[0])
                    pl.get_state_dev(fin.data_ptr(), None)
                    bits = fin.view(torch.int64)
                    if ref_bits is None:
                        ref_bits = bits
                    else:
                        same = same and bool(torch.equal(bits, ref_bits))
            row = {}
            for k, pl in plans.items():
                med = float(np.median(times[k]))
                streamed = (pl.streamed_matrix_bytes if k == "coded" else pl.matrix_bytes) + pl.vector_bytes
                row[k] = dict(ms_per_step=times[k], median_ms_per_step=med, streamed_bytes=streamed,
                              achieved_TB_per_s=streamed / (med * 1e-3) / 1e12)
            row["speedup_coded"] = row["raw"]["median_ms_per_step"] / row["coded"]["median_ms_per_step"]
            row["states_bit_identical"] = same
            table[str(v)] = row
            print(json.dumps({"m": m, "variant": v, "coded_ms": row["coded"]["median_ms_per_step"],
                              "raw_ms": row["raw"]["median_ms_per_step"], "coded_TBs": row["coded"]["achieved_TB_per_s"],
                              "raw_TBs": row["raw"]["achieved_TB_per_s"], "same": same}), flush=True)
            for pl in plans.values():
                pl.close()
            del plans, start, ref_bits
            gc.collect()
            torch.cuda.empty_cache()
        result["variants"][str(m)] = table
    path = os.path.join(a.out, "value_coding_probe.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print(f"[value_coding_probe] {result['gpu']} at {result['power_limit']}: wrote {path}")


if __name__ == "__main__":
    main()
