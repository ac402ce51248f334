"""Worker of test_gpu_energy.py (one process per rank, torchrun): the energy records of synchronised steps over the
peer-memory (three-kernel form while the monitor is armed) or NCCL transport must equal, bit for bit, those of the
same partition stepped with the in-process group transport, which every process also builds.

    energy_dist_worker.py <peer|nccl> <beam_coarse_P2|mid_np2>
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import scipy.sparse as sp
import torch
import torch.distributed as dist

import saa_b200  # noqa: F401
from saa_b200 import device_setup, maps, mesh, multi, plan as splan
from util import GOLDEN, bits_equal, load_golden

transport, golden = sys.argv[1], sys.argv[2]
world = int(os.environ["WORLD_SIZE"])
ndev = torch.cuda.device_count()
local = int(os.environ["LOCAL_RANK"]) % ndev
torch.cuda.set_device(local)
if ndev < world:
    dist.init_process_group("gloo")
else:
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
rank, size = dist.get_rank(), dist.get_world_size()
N = 40 if ndev < world else 200                           # time-sliced ranks: a context switch per step

if golden.startswith("mid_"):
    z = np.load(os.path.join(GOLDEN, golden + ".npz"))
    assert int(z["size"]) == size
    pts, cells, fac = mesh.structured_beam(int(z["m"]), length=int(z["length"]))
    epart = z["epart"].astype(np.int64)
    pl, _ = device_setup.build_mesh_rank(pts, cells, fac, epart, rank, size, device_index=local)
    gplans, _ = device_setup.build_mesh_in_process(pts, cells, fac, epart, size, device_index=local)
else:
    g = load_golden(golden)
    assert g["P"] == size
    lists = [q["nodes"] for q in g["ranks"]]

    def rank_plan(q):
        r = g["ranks"][q]
        n = r["F"].size
        K = sp.csr_matrix((r["K_data"], r["K_indices"], r["K_indptr"]), shape=(n, n))
        return splan.StepPlan(K, r["F"], r["lM"], r["dirichlet"], g["dt"], float(g["alpha"]), device=local,
                              halo=maps.halo_plan(q, size, lists), rank=q, size=size)

    pl = rank_plan(rank)
    gplans = [rank_plan(q) for q in range(size)]

assert multi.attach_transport(pl, transport) == transport
pl.set_energy(N, 1)
pl.step(N // 2, splan.MODE_SYNC, splan.LAUNCH_GRAPH)
pl.step(N - N // 2, splan.MODE_SYNC, splan.LAUNCH_PER_STEP)
pl.synchronize()
mine = pl.read_energy()
glob = multi.gather_energy(pl)

grp = splan.PlanGroup(gplans)
for q in gplans:
    q.set_energy(N, 1)
grp.step(N, splan.MODE_SYNC)
grp.synchronize()
ref = gplans[rank].read_energy()
assert bits_equal(pl.d0(), gplans[rank].d0()), (golden, transport, rank, "state")
for f in splan.ENERGY_FIELDS:
    assert np.array_equal(mine[f], ref[f]), (golden, transport, rank, f)
gref = splan.energy_balance([q.read_energy() for q in gplans])
for f in gref.dtype.names:
    assert np.array_equal(glob[f], gref[f]), (golden, transport, rank, f)
dist.barrier()
print(f"rank {rank}/{size} energy ok ({transport})")
dist.destroy_process_group()
