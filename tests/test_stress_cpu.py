"""saa_b200.stress on CPU tensors (no GPU): von Mises, and the averaged nodal stresses of a three-rank partition against
a direct numpy sum over the holders of every node in ascending rank order."""
import numpy as np
import pytest

import saa_b200  # noqa: F401
from saa_b200 import maps, plan as splan, stress

torch = pytest.importorskip("torch")


def test_von_mises_matches_the_formula_and_simple_states():
    rng = np.random.default_rng(3)
    s = rng.standard_normal((50, 6))
    want = np.sqrt(0.5 * ((s[:, 0] - s[:, 1]) ** 2 + (s[:, 1] - s[:, 2]) ** 2 + (s[:, 2] - s[:, 0]) ** 2)
                   + 3.0 * (s[:, 3] ** 2 + s[:, 4] ** 2 + s[:, 5] ** 2))
    got = stress.von_mises(torch.from_numpy(s)).numpy()
    assert np.allclose(got, want, rtol=1e-15, atol=0)
    uni = torch.tensor([[2.0, 0, 0, 0, 0, 0], [0, 0, 0, 0, 0, 3.0], [5.0, 5.0, 5.0, 0, 0, 0]], dtype=torch.float64)
    assert stress.von_mises(uni).tolist() == [2.0, 3.0 * np.sqrt(3.0), 0.0]     # uniaxial, pure shear, hydrostatic
    assert stress.von_mises(torch.from_numpy(s.reshape(5, 10, 6))).shape == (5, 10)


def _three_ranks():
    # global nodes 0..11; ranks overlap at 3, 4 (ranks 0, 1), 7 (ranks 1, 2) and 5 (all three)
    return [np.array([0, 1, 2, 3, 4, 5]), np.array([4, 3, 5, 6, 7]), np.array([8, 7, 9, 5, 10, 11])]


def test_nodal_stress_three_ranks_equals_direct_sum():
    lists = _three_ranks()
    P = len(lists)
    halos = [maps.halo_plan(q, P, lists) for q in range(P)]
    rng = np.random.default_rng(5)
    parts = []
    for l in lists:
        p = rng.standard_normal((l.size, 7))
        p[:, 6] = rng.uniform(0.5, 2.0, l.size)                  # summed weights are positive
        parts.append(p)
    # direct numpy: per global node, 0.0 + the holders' partials in ascending rank order
    acc, seen = np.zeros((12, 7)), np.zeros(12, dtype=int)
    for q in range(P):
        for i, n in enumerate(lists[q]):
            acc[n] = acc[n] + parts[q][i]
            seen[n] += 1
    sig = acc[:, :6] / acc[:, 6:7]
    vm = np.sqrt(0.5 * ((sig[:, 0] - sig[:, 1]) ** 2 + (sig[:, 1] - sig[:, 2]) ** 2 + (sig[:, 2] - sig[:, 0]) ** 2)
                 + 3.0 * (sig[:, 3] * sig[:, 3] + sig[:, 4] * sig[:, 4] + sig[:, 5] * sig[:, 5]))
    tparts = [torch.from_numpy(p) for p in parts]
    sends = [stress.shared_message(tparts[q], halos[q]) for q in range(P)]
    for q in range(P):
        recv = {nb: sends[nb][q] for nb in halos[q]["neighbours"]}
        got = stress.nodal_stress(tparts[q], halos[q], q, recv).numpy()           # a halo alone turns the holder sum on
        assert got.shape == (lists[q].size, 7)
        assert np.array_equal(got, stress.nodal_stress(tparts[q], halos[q], q, recv, size=P).numpy()), q
        assert np.array_equal(got[:, :6], sig[lists[q]]), q
        assert np.allclose(got[:, 6], vm[lists[q]], rtol=1e-15, atol=0), q
    assert seen[5] == 3 and seen[7] == 2


def test_nodal_stress_single_partition_and_refusals():
    p = torch.tensor([[2.0, 4.0, 6.0, 0.0, 0.0, 1.0, 2.0]], dtype=torch.float64)
    out = stress.nodal_stress(p)
    assert out[0, :6].tolist() == [1.0, 2.0, 3.0, 0.0, 0.0, 0.5]
    with pytest.raises(splan.SaaError, match="halo"):
        stress.nodal_stress(p, size=2)
    lists = _three_ranks()
    halo = maps.halo_plan(1, 3, lists)
    with pytest.raises(splan.SaaError, match="neighbour"):
        stress.nodal_stress(torch.zeros((5, 7), dtype=torch.float64), halo, 1, {0: torch.zeros((3, 7), dtype=torch.float64)}, size=3)
    orphan = torch.tensor([[1.0, 1, 1, 0, 0, 0, 1.0], [0.0, 0, 0, 0, 0, 0, 0.0]], dtype=torch.float64)
    with pytest.raises(splan.SaaError, match="no element weight.*position 1"):
        stress.nodal_stress(orphan)
    with pytest.raises(splan.SaaError, match=r"\(n_nodes, 7\)"):
        stress.nodal_stress(torch.zeros((5, 6), dtype=torch.float64))
