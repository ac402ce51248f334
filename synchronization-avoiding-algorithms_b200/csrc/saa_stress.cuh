// saa_stress.cuh — stress recovery from the resident displacement d0 (DESIGN.md §7b).  Output only: nothing here
// touches the state, the clock, the hooks or the energy sums, and no step kernel calls it.
//
// Element kernel: for a linear tetrahedron eps = B u_e and sigma = D eps are constant over the element (B of
// the reference's Tools/Mat_construction.py:99-104, Voigt order xx yy zz yz xz xy with engineering shear; D of
// commons.py:25-31).  detJ * grad N_b is formed as K5 forms it (saa_mf_corner_force): edge vectors from corner 0,
// cross products, corner 0 eliminated by sum_b grad N_b = 0.  The arithmetic reads only the element's four corners in
// connectivity order (coordinates and d0), so one element gives the same bits whatever the internal node order, the
// partition or the set-up path.
//
// Nodal kernel: node-owned like K5 — one thread per node, one warp per slice, walking the sliced incidence list in
// ascending element order and summing V_e sigma_e and V_e (no atomics, one writer per output).  The output is this
// rank's partial sums; shared nodes still need the sum over their holders (stress.nodal_stress).
#pragma once

#define SAA_STRESS_NODE_FIELDS 7   // sum V sigma (6), sum V

__global__ void __launch_bounds__(256) saa_k_stress_elem(int64_t n_elem, const int4 *__restrict__ cells, const double *__restrict__ X,
                                                         const double *__restrict__ d0, double lmd, double mu, double *__restrict__ out,
                                                         unsigned long long *__restrict__ bad)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_elem) return;
    const int4 cn = __ldg(cells + e);
    const int32_t nb[4] = {cn.x, cn.y, cn.z, cn.w};
    double x0[3], u0[3], ed[3][3], du[3][3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        x0[i] = __ldg(X + 3 * (int64_t)nb[0] + i);
        u0[i] = __ldg(d0 + 3 * (int64_t)nb[0] + i);
    }
#pragma unroll
    for (int b = 0; b < 3; ++b)
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            ed[b][i] = __ldg(X + 3 * (int64_t)nb[b + 1] + i) - x0[i];
            du[b][i] = __ldg(d0 + 3 * (int64_t)nb[b + 1] + i) - u0[i];
        }
    // c_b = detJ * grad N_b  (b = 1, 2, 3):  c1 = e2 x e3, c2 = e3 x e1, c3 = e1 x e2;  detJ = e1 . c1
    double c[3][3];
#pragma unroll
    for (int b = 0; b < 3; ++b) {
        const double(&p)[3] = ed[(b + 1) % 3];
        const double(&q)[3] = ed[(b + 2) % 3];
        c[b][0] = p[1] * q[2] - p[2] * q[1];
        c[b][1] = p[2] * q[0] - p[0] * q[2];
        c[b][2] = p[0] * q[1] - p[1] * q[0];
    }
    const double detJ = ed[0][0] * c[0][0] + ed[0][1] * c[0][1] + ed[0][2] * c[0][2];
    double2 *o = reinterpret_cast<double2 *>(out + 8 * e);    // rows are 64 B; out is 16-B aligned (checked by the caller)
    if (!(detJ > 0.0)) {                     // inverted or degenerate element (NaN included): report the lowest index
        atomicMin(bad, (unsigned long long)e);
#pragma unroll
        for (int k = 0; k < 4; ++k) o[k] = make_double2(0.0, 0.0);
        return;
    }
    // H = detJ * grad u = sum_b (u_b - u_0) (x) c_b
    double H[3][3];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) H[i][j] = du[0][i] * c[0][j] + du[1][i] * c[1][j] + du[2][i] * c[2][j];
    const double tr = lmd * (H[0][0] + H[1][1] + H[2][2]);
    const double s[6] = {(tr + 2.0 * mu * H[0][0]) / detJ, (tr + 2.0 * mu * H[1][1]) / detJ, (tr + 2.0 * mu * H[2][2]) / detJ,
                         mu * (H[1][2] + H[2][1]) / detJ, mu * (H[0][2] + H[2][0]) / detJ, mu * (H[0][1] + H[1][0]) / detJ};
    const double a = s[0] - s[1], b = s[1] - s[2], d = s[2] - s[0];
    const double vm = sqrt(0.5 * (a * a + b * b + d * d) + 3.0 * (s[3] * s[3] + s[4] * s[4] + s[5] * s[5]));
    o[0] = make_double2(s[0], s[1]);
    o[1] = make_double2(s[2], s[3]);
    o[2] = make_double2(s[4], s[5]);
    o[3] = make_double2(vm, detJ / 6.0);
}

// ext_of_int: external (Local_nodal_list) position of every internal node, -1 for slice padding
__global__ void __launch_bounds__(256) saa_k_stress_node(int64_t n_slices, const int64_t *__restrict__ slice_ptr,
                                                         const int32_t *__restrict__ inc, const int32_t *__restrict__ ext_of_int,
                                                         const double *__restrict__ elem, double *__restrict__ out)
{
    const int lane = threadIdx.x & 31;
    const int64_t slice = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (slice >= n_slices) return;
    const int32_t ext = ext_of_int[slice * 32 + lane];
    const int64_t beg = slice_ptr[slice];
    const int len = (int)((slice_ptr[slice + 1] - beg) >> 5);
    const int32_t *il = inc + beg + lane;
    double acc[SAA_STRESS_NODE_FIELDS] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    int32_t code = (len > 0) ? ld_stream_s32(il) : -1;
    for (int j = 0; j < len; ++j) {
        const int32_t cur = code;
        if (j + 1 < len) code = ld_stream_s32(il + 32 * (j + 1));      // next incidence one iteration ahead
        if (cur < 0) continue;                                          // padding lane of this slice
        const double2 *row = reinterpret_cast<const double2 *>(elem + 8 * (int64_t)(cur >> 2));   // 16-B aligned rows
        const double2 r0 = __ldg(row), r1 = __ldg(row + 1), r2 = __ldg(row + 2), r3 = __ldg(row + 3);
        const double v = r3.y, s[6] = {r0.x, r0.y, r1.x, r1.y, r2.x, r2.y};
#pragma unroll
        for (int k = 0; k < 6; ++k) acc[k] += v * s[k];                 // ascending element order: deterministic
        acc[6] += v;
    }
    if (ext < 0) return;
#pragma unroll
    for (int k = 0; k < SAA_STRESS_NODE_FIELDS; ++k) out[SAA_STRESS_NODE_FIELDS * (int64_t)ext + k] = acc[k];
}
