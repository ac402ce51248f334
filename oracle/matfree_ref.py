"""oracle/matfree_ref.py — exact reference of the matrix-free internal force of kernel K5 (TEST INFRASTRUCTURE ONLY).

K5 (saa_matfree.cuh) evaluates, per node a and per incident tetrahedron e,
    f_a = V sigma(u_e) grad N_a = sigma' c_a / (6 detJ),   sigma' = lmd tr(H) I + mu (H + H^T),   H = sum_b du_b (x) c_b
with c_b = detJ grad N_b formed from edge vectors of the corner a (c1 = e2 x e3, c2 = e3 x e1, c3 = e1 x e2,
c_a = -(c1 + c2 + c3)) and the SIGNED detJ = e1 . c1 (assembly.py:78-90: the reference's V = detJ * w is signed too).

  internal_force_exact   the formula in exact rational arithmetic on the exact double inputs (Python integers with
                         one power-of-two scale per input array; a Fraction per incidence).  Small meshes.
  internal_force_ld      the same formula vectorised in np.longdouble (64-bit mantissa on x86: the caller skips
                         unless np.finfo(np.longdouble).nmant >= 63).  Large meshes.
  force_bound            a per-row bound of |f_K5 - f_exact| for K5's own operation sequence.
  recover_force          f from one shipped step (alpha = 0, tn = 0, dn = d0), and the bound of that recovery.

Derivation of force_bound (u = 2^-53, the unit roundoff; gamma_k = k u / (1 - k u)).  Leaves are the exact differences
x_b - x_a and u_b - u_a, each rounded once.  For an expression without division, the computed value differs from
the exact one by at most gamma_k times the expression evaluated with absolute values of every leaf and exact
operations, where k is the largest number of roundings on a path from a leaf to the result.  An FMA merges a product
rounding into an addition rounding, so it never lengthens a path: the count below (no FMA) bounds both.  In
saa_mf_corner_force:
    e_b, du_b                 1
    c_b   (p1 q2 - p2 q1)     1 + 2 = 3
    H_ij  (3 products, 2 adds) max(3, 1) + 1 + 2 = 6
    tr    lmd (H00+H11+H22)   6 + 2 + 1 = 9
    g0    c1 + c2 + c3        3 + 2 = 5
    mu (H_ij + H_ji) g0_j     6 + 1 + 1 + 1 = 9
    t_i   tr g0_i + 3 terms   10 + 3 = 13
    detJ  e1 . c1             1 + 3 = 4 -> + 2 adds = 6: |detJ~ - detJ| <= gamma_6 D, D = sum_i |e1_i| |c1|_i
The factor s = -1/(6 detJ~) adds two roundings and the relative error of detJ~, gamma_6 kappa_e with
kappa_e = D / |detJ| >= 1 (the cancellation in detJ; large for slivers).  f = t s adds one.  With A_{e,a} = the
force of corner a of element e evaluated with absolute values (|lmd|, |mu|, abs cross products, exact 1/(6 |detJ|)):
    |f~_{e,a} - f_{e,a}| <= (13 + 3 + 6 kappa_e) u A_{e,a}   (first order)
The kernel adds the k_a incident forces of node a in ascending element order starting from the first: (k_a - 1)
more roundings on the sum of |f| <= A.  So per row of node a
    bound = u sum_e [16 + 6 kappa_e + (k_a - 1)] A_{e,a} * (1 + 1e-6),
i.e. C eps sum_e kappa_e A_{e,a} with eps = 2u and C = 11 plus the summation term.  The factor 1 + 1e-6 covers the
second-order terms (gamma_k against k u) and the float64 evaluation of the bound itself; force_bound refuses an
element with u (22 kappa_e + k_a) > 1e-8, where that would not hold.  C is counted, not fitted.

Derivation of the recovery bound.  saa_cd_update with alpha = 0, ramp(0) = 0 and dn = d0 computes
    t1 = dt2 (0 - Fi) (1 + d1),  t2 = 2M d0 (1 + d2),  t3 = M d0 (1 + d3),  t4 = +-0,  den = M exactly,
    n = ((t1 + t2)(1 + d4) - t3)(1 + d5),  d1 = n / M (1 + d6).
With R = M (d0 - d1) / dt2 evaluated exactly, solving for t1 gives
    |Fi - R| <= u |R| + (M / dt2) u (3 |d1| + 4 |d0|)   (first order; times 1 + 1e-6 again).
Rows the kernel clamps (Dirichlet) carry no force and are excluded by the caller.
"""
from __future__ import annotations

from fractions import Fraction

import numpy as np

U = 2.0 ** -53
# K5's corner rotation (saa_matfree.cuh: own corner first, an even permutation keeps the orientation)
ROT = ((0, 1, 2, 3), (1, 0, 3, 2), (2, 3, 0, 1), (3, 2, 1, 0))
SLACK = 1.0 + 1e-6


# ---- exact ------------------------------------------------------------------------------------------------------
def _scaled_ints(a):
    """(object array of Python ints, k) with a == ints * 2^-k exactly"""
    a = np.ascontiguousarray(a, dtype=np.float64)
    m, e = np.frexp(a)
    nz = a != 0
    k = int(np.max(53 - e[nz])) if nz.any() else 0
    mant = np.ldexp(m, 53).astype(np.int64)                       # exact: |m| < 1
    sh = (e - 53 + k).astype(np.int64)
    out = np.empty(a.shape, dtype=object)
    flat = out.reshape(-1)
    for i, (v, s) in enumerate(zip(mant.reshape(-1).tolist(), sh.reshape(-1).tolist())):
        flat[i] = v << s if v else 0                              # s >= 0 for every non-zero entry by the choice of k
    return out, k


def _cross(p, q):
    return np.stack([p[..., 1] * q[..., 2] - p[..., 2] * q[..., 1], p[..., 2] * q[..., 0] - p[..., 0] * q[..., 2],
                     p[..., 0] * q[..., 1] - p[..., 1] * q[..., 0]], axis=-1)


def _element_forces(X, Uu, cells, lmd, mu):
    """(nE,4,3) numerators N and (nE,) denominators 6 detJ of sigma' c_a / (6 detJ) in the arithmetic of the arrays
    (object arrays of ints: exact; longdouble: vectorised)."""
    P = X[cells]                                                  # (nE,4,3)
    D = Uu[cells]
    e = P[:, 1:] - P[:, :1]                                       # e_b = x_b - x_0, b = 1..3
    du = D[:, 1:] - D[:, :1]
    c = np.stack([_cross(e[:, 1], e[:, 2]), _cross(e[:, 2], e[:, 0]), _cross(e[:, 0], e[:, 1])], axis=1)
    detJ = (e[:, 0] * c[:, 0]).sum(axis=-1)
    H = np.einsum("nbi,nbj->nij", du, c) if du.dtype != object else \
        sum(du[:, b, :, None] * c[:, b, None, :] for b in range(3))
    tr = H[:, 0, 0] + H[:, 1, 1] + H[:, 2, 2]
    S = mu * (H + np.transpose(H, (0, 2, 1)))
    for i in range(3):
        S[:, i, i] = S[:, i, i] + lmd * tr
    c0 = -(c[:, 0] + c[:, 1] + c[:, 2])
    ca = np.concatenate([c0[:, None], c], axis=1)                 # (nE,4,3): detJ grad N_a
    N = sum(S[:, None, :, j] * ca[:, :, None, j] for j in range(3))    # (nE,4,3): sigma' c_a
    return N, 6 * detJ


def internal_force_exact(points, cells, u, lmd, mu):
    """(n_nodes, 3) object array of Fractions: sum over the elements of each node of V sigma(u_e) grad N_a, exact."""
    points = np.asarray(points, dtype=np.float64)
    cells = np.asarray(cells, dtype=np.int64)
    u = np.asarray(u, dtype=np.float64).reshape(-1, 3)
    Xi, kx = _scaled_ints(points)
    Ui, ku = _scaled_ints(u)
    (L, M), kl = _scaled_ints(np.array([lmd, mu]))
    N, den = _element_forces(Xi, Ui, cells, L, M)
    # N carries the scale 2^-(kl + ku + 4 kx), den 2^-(3 kx)
    scale = Fraction(1, 2 ** (kl + ku + kx))
    out = np.empty((points.shape[0], 3), dtype=object)
    out.fill(Fraction(0))
    for el in range(cells.shape[0]):
        d = den[el]
        if d == 0:
            raise ZeroDivisionError(f"element {el} has zero volume")
        for a in range(4):
            n = cells[el, a]
            for i in range(3):
                out[n, i] += Fraction(N[el, a, i], d)
    return out * scale


def internal_force_ld(points, cells, u, lmd, mu):
    """(n_nodes, 3) np.longdouble: the same sum, vectorised in extended precision."""
    ld = np.longdouble
    X = np.asarray(points, dtype=np.float64).astype(ld)
    Uu = np.asarray(u, dtype=np.float64).reshape(-1, 3).astype(ld)
    cells = np.asarray(cells, dtype=np.int64)
    N, den = _element_forces(X, Uu, cells, ld(lmd), ld(mu))
    f = N / den[:, None, None]
    out = np.zeros((X.shape[0], 3), dtype=ld)
    np.add.at(out, cells.reshape(-1), f.reshape(-1, 3))
    return out


def to_float(exact):
    return np.vectorize(float, otypes=[np.float64])(exact)


# ---- bound -----------------------------------------------------------------------------------------------------
def element_kappa(points, cells):
    """kappa_e = D_e / |detJ_e| >= 1 of corner 0 (the cancellation in detJ)"""
    return _corner_terms(points, cells, np.zeros((len(points), 3)), 1.0, 1.0, 0)[1]


def _corner_terms(points, cells, u, lmd, mu, a):
    """(A, kappa) of corner a of every element, with K5's rotation of the corners"""
    X = np.asarray(points, dtype=np.float64)
    Uu = np.asarray(u, dtype=np.float64).reshape(-1, 3)
    cells = np.asarray(cells, dtype=np.int64)
    r = ROT[a]
    own, nb = cells[:, r[0]], cells[:, list(r[1:])]
    E = np.abs(X[nb] - X[own][:, None])                                      # (nE,3,3) |e_b|
    DU = np.abs(Uu[nb] - Uu[own][:, None])
    eld = X[nb].astype(np.longdouble) - X[own][:, None].astype(np.longdouble)
    detJ = np.abs((eld[:, 0] * _cross(eld[:, 1], eld[:, 2])).sum(-1)).astype(np.float64)

    def across(p, q):
        return np.stack([p[:, 1] * q[:, 2] + p[:, 2] * q[:, 1], p[:, 2] * q[:, 0] + p[:, 0] * q[:, 2],
                         p[:, 0] * q[:, 1] + p[:, 1] * q[:, 0]], axis=-1)
    C = np.stack([across(E[:, 1], E[:, 2]), across(E[:, 2], E[:, 0]), across(E[:, 0], E[:, 1])], axis=1)
    Dabs = (E[:, 0] * C[:, 0]).sum(-1)
    with np.errstate(divide="ignore", invalid="ignore"):
        kappa = Dabs / detJ
    HA = np.einsum("nbi,nbj->nij", DU, C)
    G = C.sum(axis=1)
    T = abs(lmd) * np.einsum("nii->n", HA)[:, None] * G + abs(mu) * np.einsum("nij,nj->ni", HA + np.transpose(HA, (0, 2, 1)), G)
    with np.errstate(divide="ignore", invalid="ignore"):
        A = T / (6.0 * detJ)[:, None]
    return A, kappa


def force_bound(points, cells, u, lmd, mu):
    """(n_nodes, 3) float64: bound of |f_K5 - f_exact| per row (module docstring)."""
    cells = np.asarray(cells, dtype=np.int64)
    n = len(points)
    k = np.bincount(cells.reshape(-1), minlength=n).astype(np.float64)       # incident elements per node
    out = np.zeros((n, 3))
    for a in range(4):
        A, kappa = _corner_terms(points, cells, u, lmd, mu, a)
        own = cells[:, ROT[a][0]]
        if not np.all(np.isfinite(kappa)) or np.any(U * (22.0 * kappa + k[own]) > 1e-8):
            bad = int(np.nonzero(~np.isfinite(kappa) | (U * (22.0 * kappa + k[own]) > 1e-8))[0][0])
            raise ValueError(f"force_bound: element {bad} is too close to degenerate for a first-order bound")
        w = (16.0 + 6.0 * kappa + (k[own] - 1.0))[:, None] * A
        np.add.at(out, own, w)
    return U * out * SLACK


def recover_force(d0, d1, M, dt2):
    """(R, bound): the force one step with alpha = 0, tn = 0, dn = d0 applied, R = M (d0 - d1) / dt2 in extended
    precision, and the rounding of that recovery (module docstring).  Vectors of n_dof."""
    ld = np.longdouble
    d0 = np.asarray(d0, dtype=np.float64).reshape(-1)
    d1 = np.asarray(d1, dtype=np.float64).reshape(-1)
    M = np.broadcast_to(np.asarray(M, dtype=np.float64).reshape(-1), d0.shape)
    R = M.astype(ld) * (d0.astype(ld) - d1.astype(ld)) / ld(dt2)
    b = (U * np.abs(R).astype(np.float64) + (M / dt2) * U * (3.0 * np.abs(d1) + 4.0 * np.abs(d0))) * SLACK
    return R, b


def abs_error(got, exact):
    """|got - exact| per entry, got float64 / longdouble, exact Fractions (object) or longdouble"""
    got = np.asarray(got).reshape(-1)
    exact = np.asarray(exact).reshape(-1)
    if exact.dtype == object:
        vals = got if got.dtype == object else [Fraction(*v.as_integer_ratio()) for v in got]
        return np.array([float(abs(g - e)) for g, e in zip(vals, exact.tolist())])
    return np.abs(got.astype(np.longdouble) - exact.astype(np.longdouble)).astype(np.float64)


# ---- adversarial meshes -----------------------------------------------------------------------------------------
def _structured(m, length, seed=None, jitter=0.0):
    import saa_b200  # noqa: F401
    from saa_b200 import mesh
    pts, cells, _ = mesh.structured_beam(m, length=length, with_facets=None)
    if jitter:
        rng = np.random.default_rng(seed)
        pts = pts + rng.uniform(-jitter, jitter, pts.shape) / m
    return pts, cells


def _delaunay(n, seed):
    from scipy.spatial import Delaunay
    rng = np.random.default_rng(seed)
    pts = rng.uniform(0.0, 1.0, (n, 3)) * np.array([3.0, 1.0, 0.7])
    cells = Delaunay(pts).simplices.astype(np.int64)
    assert np.unique(cells).size == n
    return pts, cells


def _fan(n_sphere):
    """a hub node (id 0) in every tetrahedron of the convex hull of points on a sphere"""
    from scipy.spatial import ConvexHull
    i = np.arange(n_sphere) + 0.5
    phi, th = np.arccos(1 - 2 * i / n_sphere), np.pi * (1 + 5 ** 0.5) * i
    s = np.stack([np.cos(th) * np.sin(phi), np.sin(th) * np.sin(phi), np.cos(phi)], axis=1)
    pts = np.concatenate([np.zeros((1, 3)), s])
    tri = ConvexHull(s).simplices + 1
    cells = np.concatenate([np.zeros((tri.shape[0], 1), dtype=np.int64), tri], axis=1)
    return pts, cells


def adversarial_meshes():
    """name -> (points, cells): the meshes K5 is checked on besides the golden fixtures (deterministic)."""
    out = {}
    pj, cj = _structured(2, 4, seed=1, jitter=0.3)                # 9 x 3 x 3 nodes, all detJ > 0
    out["jittered"] = (pj, cj)
    cf = cj.copy()
    cf[::3, [1, 2]] = cf[::3, [2, 1]]                             # every third element inverted: detJ < 0
    out["inverted"] = (pj, cf)
    out["translated"] = (pj + 1e3, cj)
    # slivers: a new node just off the centroid of a face of a few elements (height 1e-4 h)
    ps, cs = [pj], [cj]
    nxt = len(pj)
    for el in (3, 40, 100):
        a, b, c = cj[el, 1], cj[el, 2], cj[el, 3]
        nrm = np.cross(pj[b] - pj[a], pj[c] - pj[a])
        ps.append(((pj[a] + pj[b] + pj[c]) / 3 + 1e-4 * 0.5 * nrm / np.linalg.norm(nrm))[None])
        cs.append(np.array([[a, b, c, nxt]]))
        nxt += 1
    out["slivers"] = (np.concatenate(ps), np.concatenate(cs))
    out["fan"] = _fan(70)                                         # hub valence 136
    # nodes in no element, interleaved with the used ones
    rng = np.random.default_rng(5)
    n_used, n_free = len(pj), 11
    perm = rng.permutation(n_used + n_free)
    pts = np.empty((n_used + n_free, 3))
    pts[perm[:n_used]] = pj
    pts[perm[n_used:]] = rng.uniform(0, 1, (n_free, 3))
    out["orphans"] = (pts, perm[:n_used][cj])
    for n in (31, 33, 257):
        out[f"delaunay{n}"] = _delaunay(n, n)
    return out


def golden_mesh(g, rank=0):
    """(points, cells) of one rank of a golden fixture in its local node numbering"""
    r = g["ranks"][rank]
    nodes = np.asarray(r["nodes"], dtype=np.int64)
    pos = np.empty(len(g["points"]), dtype=np.int64)
    pos[nodes] = np.arange(nodes.size)
    cells = pos[np.asarray(g["cells"], dtype=np.int64)[np.asarray(r["ele"], dtype=np.int64)][:, :4]]
    return np.asarray(g["points"], dtype=np.float64)[nodes], cells
