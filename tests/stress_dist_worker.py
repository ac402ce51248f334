"""Worker of test_gpu_stress.py (one process per rank, torchrun): averaged nodal stresses of a two-rank partition from
multi.gather_nodal_stress (partial sums exchanged between the processes) must equal, bit for bit, those of
stress.nodal_stress_in_process on the same partition built in one process, which every process also builds.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import torch
import torch.distributed as dist

import saa_b200  # noqa: F401
from saa_b200 import multi, plan as splan, stress
from test_gpu_stress import _K, _lame, local_mesh, make_plans
from util import bits_equal, load_golden

world = int(os.environ["WORLD_SIZE"])
ndev = torch.cuda.device_count()
local = int(os.environ["LOCAL_RANK"]) % ndev
torch.cuda.set_device(local)
if ndev < world:
    dist.init_process_group("gloo")
else:
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
rank, size = dist.get_rank(), dist.get_world_size()

g = load_golden("beam_coarse_P2")
assert g["P"] == size
gplans, grp, halos = make_plans(g)                      # the in-process reference: all ranks, stepped as a group
grp.step(300, splan.MODE_SYNC)
grp.synchronize()
ref = stress.nodal_stress_in_process(gplans, halos)[rank].cpu().numpy()

r = g["ranks"][rank]
mine = splan.StepPlan(_K(r), r["F"], r["lM"], r["dirichlet"], g["dt"], float(g["alpha"]), device=local, halo=halos[rank], rank=rank,
                      size=size)
mine.set_matfree(*local_mesh(g, rank), *_lame(g))
mine.set_state(*gplans[rank].get_state())
got = multi.gather_nodal_stress(mine, halos[rank]).cpu().numpy()
assert bits_equal(got, ref), (rank, float(np.abs(got - ref).max()))
dist.barrier()
print(f"rank {rank}/{size} stress ok")
dist.destroy_process_group()
