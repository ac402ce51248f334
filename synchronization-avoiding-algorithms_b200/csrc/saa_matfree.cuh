// saa_matfree.cuh — kernel K5: matrix-free internal force  f_int = sum_e B_e^T D B_e u_e  fused with the
// central-difference update, node-owned ("row ownership") — a THROUGHPUT / LOW-MEMORY mode, not the parity path.
//
// What it restates: the element stiffness of /root/reference/Tools/Mat_construction.py:79-119 (Local_K_coronary:
// linear tetrahedron, B of :99-104, D of commons.py:25-31, four equal quadrature addends detJ*w, w = 0.25/6) applied to
// the element displacement instead of being assembled (:122-150), followed by Dynamic_solver.py:13-20.  No stiffness
// matrix exists: per time step the kernel reads the connectivity (16 B per element), the node -> element incidence
// (4 x 4 B per element), the node coordinates (24 B per node) and the five vector streams — about 107 B per DOF-step
// against 400 B for the node-block matrix, and 11 GB instead of 44 GB of HBM for the 104 M-DOF mesh.  It is bound by the
// fp64 pipe and by gather latency instead (every element is evaluated once per corner): see DESIGN.md section 4a.
//
// Scatter-add is made deterministic by ROW OWNERSHIP: one thread owns one node (its three rows) and walks the
// incident tetrahedra in ascending element order, evaluating for each only the force on its own node
//     f_a = V * sigma(u_e) * grad N_a,   sigma = lmd*tr(eps)*I + 2*mu*eps,   eps = sym(sum_b u_b (x) grad N_b)
// — no atomics, no colouring, every output has exactly one writer, results are run-to-run reproducible.  Each element
// is therefore evaluated four times (once per corner); the gathers of the other three corners (coordinates and
// displacements, 2 x 24 B each) are served by L1/L2.
//
// Arithmetic differs from the assembled path by association (K u is summed per element here, per matrix entry there;
// the library is built with -fmad=false): results agree with the parity path to ~1e-13 relative per step and drift apart as SURVEY.md §0.5
// describes (measured: tests/test_gpu_matfree.py, bench.py --kernel matfree).  It can therefore not meet the 1e-12
// history criterion over 10^4 steps and is never used by the parity tests or the default bench line.
// Accuracy: every row of the force is within a bound counted from the operation sequence below of the exact rational
// value (oracle/matfree_ref.py, tests/test_gpu_matfree_reference.py); keep a rewrite of this arithmetic inside it.
#pragma once

struct SaaMatFreeDev {
    const int64_t *slice_ptr;   // [n_slices + 1] offsets in incidence-lanes (multiples of 32), sliced like the matrix
    const int32_t *inc;         // 4*element + corner of the j-th incident element of lane l: inc[slice_ptr[s] + 32*j + l], -1 = none
    const int4 *cells;          // element connectivity in INTERNAL node ids
    const double *X;            // node coordinates, internal node order (3 per node)
    double lmd, mu;
};

// force on corner 0 of the tetrahedron (x0; x1, x2, x3) with displacements (u0; u1, u2, u3), times -1/(6 detJ) pulled out:
// the caller passes the corners rotated by an EVEN permutation so that its own node comes first (orientation kept).
__device__ __forceinline__ void saa_mf_corner_force(const double (&x0)[3], const double (&u0)[3], const double *__restrict__ X,
                                                    const double *__restrict__ d0, int32_t n1, int32_t n2, int32_t n3, double lmd,
                                                    double mu, double (&f)[3])
{
    double e[3][3], du[3][3];
    const int32_t nb[3] = {n1, n2, n3};
#pragma unroll
    for (int b = 0; b < 3; ++b) {
        const double *xp = X + 3 * (int64_t)nb[b];
        const double *up = d0 + 3 * (int64_t)nb[b];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            e[b][i] = __ldg(xp + i) - x0[i];
            du[b][i] = __ldg(up + i) - u0[i];
        }
    }
    // c_b = detJ * grad N_b  (b = 1, 2, 3):  c1 = e2 x e3, c2 = e3 x e1, c3 = e1 x e2;  detJ = e1 . c1 (signed, :93/:112)
    double c[3][3];
#pragma unroll
    for (int b = 0; b < 3; ++b) {
        const double(&p)[3] = e[(b + 1) % 3];
        const double(&q)[3] = e[(b + 2) % 3];
        c[b][0] = p[1] * q[2] - p[2] * q[1];
        c[b][1] = p[2] * q[0] - p[0] * q[2];
        c[b][2] = p[0] * q[1] - p[1] * q[0];
    }
    const double detJ = e[0][0] * c[0][0] + e[0][1] * c[0][1] + e[0][2] * c[0][2];
    // H' = detJ * grad u = sum_b (u_b - u_0) (x) c_b   (sum_b grad N_b = 0 eliminates corner 0)
    double H[3][3];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) H[i][j] = du[0][i] * c[0][j] + du[1][i] * c[1][j] + du[2][i] * c[2][j];
    const double tr = lmd * (H[0][0] + H[1][1] + H[2][2]);
    // detJ * grad N_0 = -(c1 + c2 + c3)
    const double g0[3] = {c[0][0] + c[1][0] + c[2][0], c[0][1] + c[1][1] + c[2][1], c[0][2] + c[1][2] + c[2][2]};
    // f_0 = V * sigma * grad N_0 = (detJ/6) * (sigma'/detJ) * (-g0/detJ) = -(sigma' g0) / (6 detJ)
    const double s = -1.0 / (6.0 * detJ);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        double t = tr * g0[i];
#pragma unroll
        for (int j = 0; j < 3; ++j) t += mu * (H[i][j] + H[j][i]) * g0[j];
        f[i] = t * s;
    }
}

template <int MINB>
__global__ void __launch_bounds__(256, MINB) saa_k_step_matfree(SaaDev P, SaaMatFreeDev Q, const double *__restrict__ d0,
                                                                double *__restrict__ dn_d1, const SaaClock *clk_in, SaaClock *clk_out)
{
    const double tn = clk_in->tn;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        clk_out->tn = __dadd_rn(tn, P.dt);
        clk_out->sync_step = clk_in->sync_step;
        clk_out->step_idx = clk_in->step_idx + 1ull;
    }
    const int lane = threadIdx.x & 31;
    const int64_t slice = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (slice >= P.n_slices) return;
    const int64_t node = slice * 32 + lane;
    const int64_t beg = Q.slice_ptr[slice];
    const int len = (int)((Q.slice_ptr[slice + 1] - beg) >> 5);
    const int32_t *inc = Q.inc + beg + lane;
    double x0[3], u0[3], s[3] = {0.0, 0.0, 0.0};
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        x0[i] = Q.X[3 * node + i];
        u0[i] = d0[3 * node + i];
    }
    int32_t code = (len > 0) ? ld_stream_s32(inc) : -1;
    for (int j = 0; j < len; ++j) {
        const int32_t cur = code;
        if (j + 1 < len) code = ld_stream_s32(inc + 32 * (j + 1));     // next incidence one iteration ahead
        if (cur < 0) continue;                                         // padding lane of this slice
        const int4 cn = __ldg(Q.cells + (cur >> 2));
        const int a = cur & 3;
        // own corner first, by an even permutation: (0123) (1032) (2301) (3210)
        const int32_t n1 = (a == 0) ? cn.y : (a == 1) ? cn.x : (a == 2) ? cn.w : cn.z;
        const int32_t n2 = (a == 0) ? cn.z : (a == 1) ? cn.w : (a == 2) ? cn.x : cn.y;
        const int32_t n3 = (a == 0) ? cn.w : (a == 1) ? cn.z : (a == 2) ? cn.y : cn.x;
        double f[3];
        saa_mf_corner_force(x0, u0, Q.X, d0, n1, n2, n3, Q.lmd, Q.mu, f);
#pragma unroll
        for (int i = 0; i < 3; ++i) s[i] += f[i];                      // ascending element order: deterministic
    }
    saa_finish_node<false>(P, slice, lane, s, d0, dn_d1, saa_ramp(tn));
}

// ---- set-up kernels -----------------------------------------------------------------------------------------------
// 6 detJ of the tetrahedron (x0; x1, x2, x3) in the operations of saa_mf_corner_force (the library is built with
// -fmad=false, so neither side contracts to FMA)
__device__ __forceinline__ double saa_mf_six_detJ(const double *__restrict__ X, int32_t n0, int32_t n1, int32_t n2, int32_t n3)
{
    const int32_t nb[3] = {n1, n2, n3};
    double e[3][3];
#pragma unroll
    for (int b = 0; b < 3; ++b)
#pragma unroll
        for (int i = 0; i < 3; ++i) e[b][i] = __dsub_rn(X[3 * (int64_t)nb[b] + i], X[3 * (int64_t)n0 + i]);
    const double c0 = __dsub_rn(__dmul_rn(e[1][1], e[2][2]), __dmul_rn(e[1][2], e[2][1]));
    const double c1 = __dsub_rn(__dmul_rn(e[1][2], e[2][0]), __dmul_rn(e[1][0], e[2][2]));
    const double c2 = __dsub_rn(__dmul_rn(e[1][0], e[2][1]), __dmul_rn(e[1][1], e[2][0]));
    return __dmul_rn(6.0, __dadd_rn(__dadd_rn(__dmul_rn(e[0][0], c0), __dmul_rn(e[0][1], c1)), __dmul_rn(e[0][2], c2)));
}
// the check saa_plan_set_matfree_dev makes before it allocates or indexes anything, one thread per element; keeps the
// lowest offending element per kind:  first[0] a node id outside [0, n_nodes) (nothing else of that element is read),
// first[1] zero volume: a repeated corner, or a corner whose factor -1/(6 detJ) in K5 (the four even rotations of
// saa_k_step_matfree, each with its own rounding of detJ) is not finite.  Negative detJ is accepted: V = detJ/6 is
// signed in the reference.
__global__ void saa_k_mf_check_cells(int64_t n_elem, int64_t n_nodes, const int32_t *__restrict__ cells, const double *__restrict__ X,
                                     unsigned long long *__restrict__ first)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_elem) return;
    int32_t n[4];
    bool bad_id = false;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        n[a] = cells[4 * e + a];
        if (n[a] < 0 || n[a] >= n_nodes) bad_id = true;
    }
    if (bad_id) {
        atomicMin(first, (unsigned long long)e);
        return;
    }
    bool zero = n[0] == n[1] || n[0] == n[2] || n[0] == n[3] || n[1] == n[2] || n[1] == n[3] || n[2] == n[3];
    // own corner first, by an even permutation: (0123) (1032) (2301) (3210), as saa_k_step_matfree rotates them
    const double d[4] = {saa_mf_six_detJ(X, n[0], n[1], n[2], n[3]), saa_mf_six_detJ(X, n[1], n[0], n[3], n[2]),
                         saa_mf_six_detJ(X, n[2], n[3], n[0], n[1]), saa_mf_six_detJ(X, n[3], n[2], n[1], n[0])};
#pragma unroll
    for (int a = 0; a < 4; ++a) zero = zero || !isfinite(__ddiv_rn(-1.0, d[a]));
    if (zero) atomicMin(first + 1, (unsigned long long)e);
}
__global__ void saa_k_mf_cells_to_internal(int64_t n4, const int32_t *__restrict__ cells_ext, const int32_t *__restrict__ iperm,
                                           int32_t *__restrict__ cells_int)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n4) cells_int[i] = iperm[3 * (int64_t)cells_ext[i]] / 3;
}
__global__ void saa_k_mf_coords_to_internal(int64_t n_ext_nodes, const double *__restrict__ X_ext, const int32_t *__restrict__ iperm,
                                            double *__restrict__ X_int)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_ext_nodes) return;
    const int64_t q = iperm[3 * i] / 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) X_int[3 * q + c] = X_ext[3 * i + c];
}
__global__ void saa_k_mf_slice_width(int64_t n_slices, const int64_t *__restrict__ inc_ptr, int64_t *__restrict__ width32)
{
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s > n_slices) return;
    int64_t w = 0;
    if (s < n_slices)
        for (int l = 0; l < 32; ++l) w = max(w, inc_ptr[s * 32 + l + 1] - inc_ptr[s * 32 + l]);
    width32[s] = 32 * w;
}
__global__ void saa_k_mf_fill(int64_t n_nodes, const int64_t *__restrict__ inc_ptr, const int32_t *__restrict__ inc_slot,
                              const int64_t *__restrict__ slice_ptr, int32_t *__restrict__ inc)
{
    const int64_t node = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (node >= n_nodes) return;
    const int64_t s = node >> 5;
    const int l = (int)(node & 31);
    const int64_t w = (slice_ptr[s + 1] - slice_ptr[s]) >> 5, cnt = inc_ptr[node + 1] - inc_ptr[node];
    for (int64_t j = 0; j < w; ++j) inc[slice_ptr[s] + 32 * j + l] = (j < cnt) ? inc_slot[inc_ptr[node] + j] : -1;
}
