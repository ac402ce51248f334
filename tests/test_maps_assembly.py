"""Host-side restatements (mesh / maps / sparse assembly) against the golden fixtures the reference's own functions
produced."""
import numpy as np
import pytest

import saa_b200  # noqa: F401
from saa_b200 import assembly, maps, mesh, partition
from util import bits_equal, golden_names, load_golden

LAM = 1e6 * 0.3 / ((1 + 0.3) * (1 - 2 * 0.3))
MU = 1e6 / (2 * (1 + 0.3))


@pytest.mark.parametrize("name", golden_names())
def test_maps_are_sequence_exact(name):
    g = load_golden(name)
    D = mesh.dirichlet_nodes(g["points"], g["facets"])
    assert np.array_equal(D, g["Dirichlet_node"])
    per, gshared = maps.partition_maps(g["epart"], g["cells"], g["P"], D)
    assert np.array_equal(gshared, g["Global_shared"])
    for q, (m, r) in enumerate(zip(per, g["ranks"])):
        assert np.array_equal(m["Local_ele_list"], r["ele"])
        assert np.array_equal(m["Local_nodal_list"], r["nodes"])
        assert np.array_equal(m["shared_nodes"], r["shared"])
        assert np.array_equal(m["Local_Dirichlet"], r["dirichlet"])
        assert np.array_equal(m["loc_dof_shared"], r["loc_dof_shared"])


@pytest.mark.parametrize("name", golden_names())
def test_dt_matches_reference(name):
    g = load_golden(name)
    dts = [mesh.stable_dt(g["cells"][r["ele"]], g["points"]) for r in g["ranks"]]
    assert min(dts) == float(g["dt"])


@pytest.mark.parametrize("name", golden_names())
def test_sparse_stiffness_assembly_matches_reference(name):
    """Bit-equal in the authoring container (same BLAS/LAPACK kernels as the fixture run); elsewhere the
    structure must be identical and values within 4 ulp-ish (1e-15 relative to the row scale)."""
    g = load_golden(name)
    for r in g["ranks"]:
        K = assembly.local_stiffness_csr(r["nodes"], g["cells"][r["ele"]], g["points"], LAM, MU)
        assert K.indices.dtype == np.int32
        assert np.array_equal(K.indptr, r["K_indptr"])
        assert np.array_equal(K.indices, r["K_indices"])
        scale = np.abs(r["K_data"]).max()
        assert np.abs(K.data - r["K_data"]).max() <= 1e-15 * scale


@pytest.mark.parametrize("name", golden_names())
def test_sparse_assembly_bit_exact_here(name):
    g = load_golden(name)
    for r in g["ranks"]:
        K = assembly.local_stiffness_csr(r["nodes"], g["cells"][r["ele"]], g["points"], LAM, MU)
        assert bits_equal(K.data, r["K_data"])
    lM, F = assembly.lumped_mass_and_load(g["points"], g["cells"], 1, 0.5)
    assert bits_equal(lM, g["lumped_M"])
    assert bits_equal(F, g["F_pre"])


@pytest.mark.parametrize("name", ["beam_coarse_P1", "struct_m2_P1"])
def test_lumped_mass_and_load(name):
    g = load_golden(name)
    lM, F = assembly.lumped_mass_and_load(g["points"], g["cells"], 1, 0.5)
    assert np.abs(lM - g["lumped_M"]).max() <= 4e-16 * np.abs(g["lumped_M"]).max()
    assert np.abs(F - g["F_pre"]).max() <= 4e-16 * np.abs(g["F_pre"]).max()
    # invariants measured on the reference (SURVEY.md §4): total mass = rho*volume, total load
    assert abs(lM.sum() / 3 - 25.0) < 1e-12
    assert np.allclose(F.reshape(-1, 3).sum(0), [0, -12.5, -12.5], atol=1e-12)
    lM2, _ = assembly.lumped_mass_and_load(g["points"], g["cells"], 1, 0.5, exact_rowsum=False)
    assert np.abs(lM2 - g["lumped_M"]).max() <= 4e-16 * np.abs(g["lumped_M"]).max()


def test_structured_beam_matches_fixture_inputs():
    g = load_golden("struct_m2_P1")
    p, c, f = mesh.structured_beam(2)
    assert bits_equal(p, g["points"]) and np.array_equal(c, g["cells"]) and np.array_equal(f, g["facets"])
    # positive orientation everywhere (reference integrates with the signed det J)
    P = p[c]
    J = np.transpose(P[:, 1:4, :] - P[:, 0:1, :], (0, 2, 1))
    assert (np.linalg.det(J) > 0).all()
    # conforming: every interior face is shared by exactly two tets
    faces = np.sort(np.concatenate([c[:, [0, 1, 2]], c[:, [0, 1, 3]], c[:, [0, 2, 3]], c[:, [1, 2, 3]]]), axis=1)
    _, cnt = np.unique(faces, axis=0, return_counts=True)
    assert set(cnt.tolist()) <= {1, 2}
    assert (cnt == 1).sum() == 2 * 2 * (50 * 2 * 2 + 2 * 2)  # boundary triangles of a 50x2x2 box


def test_vtk_roundtrip(tmp_path):
    p, c, f = mesh.structured_beam(1, length=3, with_facets="all")
    path = tmp_path / "m.vtk"
    mesh.write_vtk(str(path), p, c, f)
    p2, c2, f2 = mesh.read_vtk(str(path))
    assert bits_equal(p, p2) and np.array_equal(c, c2) and np.array_equal(f, f2)


def test_metis_partition_reproduces_fixture_epart():
    g = load_golden("beam_coarse_P2")
    ep = partition.metis_part_mesh(g["cells"], len(g["points"]), 2)
    assert np.array_equal(ep, g["epart"])
    assert np.bincount(partition.slab_partition(g["points"], g["cells"], 3)).tolist() == [86, 85, 85]


@pytest.mark.parametrize("name", ["beam_coarse_P3", "beam_coarse_P8", "struct_m2_P4"])
def test_halo_plan_reproduces_syn_cpus_sum(name):
    """The per-neighbour exchange + ascending-rank holder lists of maps.halo_plan give exactly the
    numbers of gather -> root sum in rank order -> bcast (Distributed_tools.py:77-92)."""
    g = load_golden(name)
    P = g["P"]
    lists = [r["nodes"] for r in g["ranks"]]
    rng = np.random.default_rng(1)
    f = [rng.standard_normal(3 * len(l)) * 10.0 ** rng.integers(-3, 3, 3 * len(l)) for l in lists]
    # literal syn_cpus
    fg = np.zeros(3 * len(g["points"]))
    for r in range(P):
        fg[maps.node_to_dof(3, [0, 1, 2], lists[r])] += f[r]
    plans = [maps.halo_plan(r, P, lists) for r in range(P)]
    multi = 0
    for r in range(P):
        hp = plans[r]
        want = fg[maps.node_to_dof(3, [0, 1, 2], lists[r])]
        got = 0.0 + f[r]                                   # non-shared DOFs: 0.0 + own
        own = f[r].reshape(-1, 3)
        # messages: rank nb sends its partial forces at the common nodes in ascending global id
        recv = {}
        for nb in hp["neighbours"]:
            hpn = plans[nb]
            recv[nb] = f[nb].reshape(-1, 3)[hpn["shared_pos"][hpn["send_idx"][r]]]
            assert np.array_equal(np.asarray(lists[nb])[hpn["shared_pos"][hpn["send_idx"][r]]],
                                  np.asarray(lists[r])[hp["shared_pos"][hp["send_idx"][nb]]])
        out = got.reshape(-1, 3)
        for j, pos in enumerate(hp["shared_pos"]):
            acc = np.zeros(3)
            lo, hi = hp["holders_ptr"][j], hp["holders_ptr"][j + 1]
            multi += (hi - lo) > 2
            for k in range(lo, hi):
                hr, slot = hp["holders_rank"][k], hp["holders_slot"][k]
                acc = acc + (own[pos] if slot < 0 else recv[hr][slot])
            out[pos] = acc
        assert bits_equal(out, want)
    if name == "beam_coarse_P8":
        assert multi > 0   # nodes held by >= 3 ranks exist: the ascending-rank order is exercised
