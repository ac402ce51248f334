"""oracle/matfree_ref.py without a GPU: the exact internal force against the golden assembled stiffness, the
extended-precision version against the exact one, and planted errors against force_bound (how sensitive the K5
tolerance of tests/test_gpu_matfree_reference.py is)."""
import numpy as np
import pytest
import scipy.sparse as sp

import saa_b200  # noqa: F401
from saa_b200 import problem
from util import golden_names, load_golden, oracle_module

oracle_module()
import matfree_ref as mr  # noqa: E402

LMD, MU = problem.lame(problem.E_DEFAULT, problem.NU_DEFAULT)
ADVERSARIAL = ("jittered", "inverted", "translated", "slivers", "fan", "orphans", "delaunay31", "delaunay33", "delaunay257")


def _ratio(err, bound):
    assert np.all(err[bound == 0] == 0)
    return float(np.max(err[bound > 0] / bound[bound > 0], initial=0.0))


@pytest.mark.parametrize("name", golden_names())
def test_exact_force_equals_golden_stiffness_times_u(name):
    """every rank of every fixture: golden LocalK @ u (the reference's own assembly) against the exact force, within
    force_bound; and within a few eps |K| |u| per row"""
    g = load_golden(name)
    for q, r in enumerate(g["ranks"]):
        pts, cells = mr.golden_mesh(g, q)
        n = r["F"].size
        K = sp.csr_matrix((r["K_data"], r["K_indices"], r["K_indptr"]), shape=(n, n))
        u = np.random.default_rng(q).standard_normal(n)
        exact = mr.internal_force_exact(pts, cells, u, LMD, MU).reshape(-1)
        err = mr.abs_error(K @ u, exact)
        assert _ratio(err, mr.force_bound(pts, cells, u, LMD, MU).reshape(-1)) <= 1.0
        assert np.all(err <= 8 * 2.0 ** -52 * (abs(K) @ np.abs(u)))


@pytest.mark.skipif(np.finfo(np.longdouble).nmant < 63, reason="np.longdouble has no 64-bit mantissa on this host")
@pytest.mark.parametrize("name", ADVERSARIAL)
def test_long_double_force_far_inside_the_bound(name):
    pts, cells = mr.adversarial_meshes()[name]
    u = np.random.default_rng(1).standard_normal(3 * len(pts))
    exact = mr.internal_force_exact(pts, cells, u, LMD, MU).reshape(-1)
    ld = mr.internal_force_ld(pts, cells, u, LMD, MU).reshape(-1)
    assert _ratio(mr.abs_error(ld, exact), mr.force_bound(pts, cells, u, LMD, MU).reshape(-1)) <= 1e-3


def test_adversarial_meshes_are_what_they_claim():
    m = mr.adversarial_meshes()

    def det(p, c):
        e = p[c][:, 1:] - p[c][:, :1]
        return np.linalg.det(e)
    assert np.all(det(*m["jittered"]) > 0)
    assert np.all((det(*m["inverted"]) < 0) == (np.arange(len(m["inverted"][1])) % 3 == 0))
    assert np.bincount(m["fan"][1].ravel()).max() >= 128
    p, c = m["orphans"]
    assert np.setdiff1d(np.arange(len(p)), c).size > 0
    assert mr.element_kappa(*m["slivers"]).max() > 1e3
    assert [len(m[f"delaunay{n}"][0]) for n in (31, 33, 257)] == [31, 33, 257]


@pytest.mark.parametrize("name", ADVERSARIAL)
def test_planted_errors_violate_the_bound(name):
    """a 1e-12 relative bias of -1/(6 detJ), lmd and mu swapped, one element dropped: each breaks the bound on some row"""
    pts, cells = mr.adversarial_meshes()[name]
    u = np.random.default_rng(2).standard_normal(3 * len(pts))
    exact = mr.internal_force_exact(pts, cells, u, LMD, MU).reshape(-1)
    bound = mr.force_bound(pts, cells, u, LMD, MU).reshape(-1)
    biased = exact * mr.Fraction(1 + 10 ** 12, 10 ** 12)                  # every element force scaled by 1 + 1e-12
    swapped = mr.internal_force_exact(pts, cells, u, MU, LMD).reshape(-1)
    dropped = mr.internal_force_exact(pts, cells[np.arange(len(cells)) != len(cells) // 2], u, LMD, MU).reshape(-1)
    for what, planted in (("bias", biased), ("lmd<->mu", swapped), ("dropped element", dropped)):
        err = np.array([float(abs(a - b)) for a, b in zip(planted.tolist(), exact.tolist())])
        assert np.max(err / np.where(bound > 0, bound, np.inf)) > 1.0, what


def test_recovery_bound_covers_the_update_rounding():
    """the update of one step with alpha = 0, tn = 0, dn = d0 (saa_cd_update in Python's association) against the
    exact force it was given: recover_force gets it back within its bound"""
    rng = np.random.default_rng(4)
    n = 3000
    f = rng.standard_normal(n) * 10.0 ** rng.uniform(-3, 3, n)
    d0 = rng.standard_normal(n)
    M = rng.uniform(0.5, 2.0, n)
    dt2 = 0.37
    num = (dt2 * (0.0 - f) + (2.0 * M) * d0) - M * d0
    d1 = num / M
    R, b = mr.recover_force(d0, d1, M, dt2)
    assert np.all(np.abs(R - f).astype(np.float64) <= b)


def test_exact_force_with_zero_and_integer_inputs():
    """the unit tetrahedron: every coordinate 0 or 1, so every non-zero input is >= 0.5 (the power-of-two scaling of
    zero entries), against the long-double version and the reference assembly"""
    from saa_b200 import assembly
    pts = np.array([[0.0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1]])
    cells = np.array([[0, 1, 2, 3]])
    u = np.array([0.0, 1, 2, 3, 0, 5, 6, 7, 0, 9, 10, 11])
    exact = mr.internal_force_exact(pts, cells, u, LMD, MU).reshape(-1)
    bound = mr.force_bound(pts, cells, u, LMD, MU).reshape(-1)
    assert _ratio(mr.abs_error(mr.internal_force_ld(pts, cells, u, LMD, MU).reshape(-1), exact), bound) <= 1e-3
    K = assembly.local_stiffness_csr(np.arange(4), cells, pts, LMD, MU)
    assert _ratio(mr.abs_error(K @ u, exact), bound) <= 1.0
