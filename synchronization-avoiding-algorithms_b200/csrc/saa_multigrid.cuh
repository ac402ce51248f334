// saa_multigrid.cuh — geometric multigrid V-cycle preconditioner for the static solve (include/saa_fem.h: saa_mg_create,
// saa_plan_solve_static_mg_dev; DESIGN.md §7d).
//
// Every level is a plan of its own (size 1) and every vector is in that plan's internal row order; S_l keeps the
// level's free rows (not Dirichlet, not slice padding), so A_l = S_l K_l S_l + (I - S_l) as in saa_static.cuh.  The
// prolongation P from level l+1 (coarse) to level l (fine) is a node CSR: fine node -> (coarse node, weight), the same
// weight on all three components.  Nothing here sums with atomics: every output element has one writer and a fixed
// summation order.  Every kernel first reads the solve's `done` word (gate; nullptr: always run) and leaves its outputs
// untouched once it is set, so a chunk of iterations replayed from a CUDA graph is a no-op after convergence.
#pragma once
#include "saa_static.cuh"

// r = b - S K x (b given by the caller and 0 on every non-free row; x is only read), one warp per slice as K1
__global__ void __launch_bounds__(256, 3) saa_k_mg_residual(SaaDev P, const double *__restrict__ x, const double *__restrict__ b,
                                                            double *__restrict__ r, const uint32_t *__restrict__ free_mask,
                                                            const long long *gate)
{
    if (gate != nullptr && *gate) return;
    const int lane = threadIdx.x & 31;
    const int64_t slice = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (slice >= P.n_slices) return;
    double s[3];
    saa_node_dot<1, true>(P, slice, lane, x, s);
#pragma unroll
    for (int A = 0; A < 3; ++A) {
        const int64_t row = 3 * (slice * 32 + lane) + A;
        r[row] = saa_cg_free(free_mask, row) ? __dsub_rn(b[row], s[A]) : 0.0;
    }
}

// One Chebyshev step on node blocks: d = c1 d + c2 B^-1 r, x += d (B^-1: the level's 3x3 inverse blocks).
//   FIRST_ZERO  first step from x = 0:   d = c2 B^-1 r, x = d  (d and x are not read)
//   FIRST       first step from any x:   d = c2 B^-1 r, x += d (d is not read)
//   NEXT        later steps:             d = c1 d + c2 B^-1 r, x += d
enum { SAA_MG_CHEB_FIRST_ZERO = 0, SAA_MG_CHEB_FIRST = 1, SAA_MG_CHEB_NEXT = 2 };
template <int MODE>
__global__ void __launch_bounds__(256) saa_k_mg_cheb(int64_t n_nodes, const double *__restrict__ r, double *__restrict__ d,
                                                     double *__restrict__ x, const double *__restrict__ binv,
                                                     const uint32_t *__restrict__ free_mask, double c1, double c2, const long long *gate)
{
    if (gate != nullptr && *gate) return;
    const int64_t node = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (node >= n_nodes) return;
    double rv[3], zv[3];
    bool fr[3];
#pragma unroll
    for (int A = 0; A < 3; ++A) {
        fr[A] = saa_cg_free(free_mask, 3 * node + A);
        rv[A] = fr[A] ? r[3 * node + A] : 0.0;
    }
    saa_cg_precond(binv, n_nodes, node, rv, zv);
#pragma unroll
    for (int A = 0; A < 3; ++A) {
        const int64_t row = 3 * node + A;
        double dv = 0.0;
        if (fr[A]) {
            dv = __dmul_rn(c2, zv[A]);
            if (MODE == SAA_MG_CHEB_NEXT) dv = __dadd_rn(__dmul_rn(c1, d[row]), dv);
        }
        d[row] = dv;
        if (MODE == SAA_MG_CHEB_FIRST_ZERO) x[row] = dv;
        else if (fr[A]) x[row] = __dadd_rn(x[row], dv);
    }
}

// x_f += S_f P x_c, one thread per fine node: its coarse parents in stored order, from 0.0 (ext_f: external node of
// every internal fine node, -1 for padding; ptr over external fine nodes, cnode: the parents' internal coarse nodes)
__global__ void __launch_bounds__(256) saa_k_mg_prolong(int64_t n_nodes_f, const int32_t *__restrict__ ext_f,
                                                        const int64_t *__restrict__ ptr, const int32_t *__restrict__ cnode,
                                                        const double *__restrict__ w, const double *__restrict__ xc,
                                                        double *__restrict__ xf, const uint32_t *__restrict__ free_f,
                                                        const long long *gate)
{
    if (gate != nullptr && *gate) return;
    const int64_t node = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (node >= n_nodes_f) return;
    const int32_t e = ext_f[node];
    if (e < 0) return;
    double s[3] = {0.0, 0.0, 0.0};
    for (int64_t k = ptr[e]; k < ptr[e + 1]; ++k) {
        const int64_t c = cnode[k];
        const double wk = w[k];
#pragma unroll
        for (int A = 0; A < 3; ++A) s[A] = __dadd_rn(s[A], __dmul_rn(wk, xc[3 * c + A]));
    }
#pragma unroll
    for (int A = 0; A < 3; ++A) {
        const int64_t row = 3 * node + A;
        if (saa_cg_free(free_f, row)) xf[row] = __dadd_rn(xf[row], s[A]);
    }
}

// b_c = S_c P^T r_f, one thread per coarse node: the transposed table of its external node lists its fine children in
// ascending external fine-node order (fnode: internal fine node, w: weight); padding and clamped rows get 0
__global__ void __launch_bounds__(256) saa_k_mg_restrict(int64_t n_nodes_c, const int32_t *__restrict__ ext_c,
                                                         const int64_t *__restrict__ tptr, const int32_t *__restrict__ fnode,
                                                         const double *__restrict__ w, const double *__restrict__ rf,
                                                         double *__restrict__ bc, const uint32_t *__restrict__ free_c,
                                                         const long long *gate)
{
    if (gate != nullptr && *gate) return;
    const int64_t node = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (node >= n_nodes_c) return;
    const int32_t e = ext_c[node];
    double s[3] = {0.0, 0.0, 0.0};
    if (e >= 0)
        for (int64_t k = tptr[e]; k < tptr[e + 1]; ++k) {
            const int64_t f = fnode[k];
            const double wk = w[k];
#pragma unroll
            for (int A = 0; A < 3; ++A) s[A] = __dadd_rn(s[A], __dmul_rn(wk, rf[3 * f + A]));
        }
#pragma unroll
    for (int A = 0; A < 3; ++A) {
        const int64_t row = 3 * node + A;
        bc[row] = saa_cg_free(free_c, row) ? s[A] : 0.0;
    }
}

// x = A_c^-1 b on the coarsest level (dense n x n, row-major, internal order), one warp per row: lane l adds columns
// l, l + 32, ... in ascending order, then the fixed warp tree
__global__ void __launch_bounds__(256) saa_k_mg_coarse(int64_t n, const double *__restrict__ inv, const double *__restrict__ b,
                                                       double *__restrict__ x, const uint32_t *__restrict__ free_mask,
                                                       const long long *gate)
{
    if (gate != nullptr && *gate) return;
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= n) return;
    const double *a = inv + row * n;
    double s = 0.0;
    for (int64_t j = lane; j < n; j += 32) s = __dadd_rn(s, __dmul_rn(a[j], b[j]));
    s = saa_warp_sum(s);
    if (lane == 0) x[row] = saa_cg_free(free_mask, row) ? s : 0.0;
}

// outer PCG, (b) without the block-Jacobi step: x += alpha p, r -= alpha q on free rows, r.r partial per block of 256
// nodes at field 1 of the update partials (part[n_parts + block]); saa_k_mg_rz adds field 0 after the V-cycle
__global__ void __launch_bounds__(256) saa_k_mg_update(int64_t n_nodes, const SaaCgState *__restrict__ S, double *__restrict__ x,
                                                       double *__restrict__ r, const double *__restrict__ p,
                                                       const double *__restrict__ q, const uint32_t *__restrict__ free_mask,
                                                       double *__restrict__ part, int64_t n_parts)
{
    if (S->done) return;
    const int64_t node = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double e[1] = {0.0};
    if (node < n_nodes) {
        const double alpha = S->alpha;
#pragma unroll
        for (int A = 0; A < 3; ++A) {
            const int64_t row = 3 * node + A;
            if (saa_cg_free(free_mask, row)) {
                x[row] = __dadd_rn(x[row], __dmul_rn(alpha, p[row]));
                const double rv = __dsub_rn(r[row], __dmul_rn(alpha, q[row]));
                r[row] = rv;
                e[0] = __dadd_rn(e[0], __dmul_rn(rv, rv));
            }
        }
    }
    saa_cg_block_partials<1>(e, part + n_parts, n_parts, blockIdx.x);
}

// after the V-cycle z = V r: the r.z partial per block of 256 nodes (field 0).  INIT (before the first iteration) also
// sets p = z and writes the r.r partial (field 1), as saa_k_cg_update<true> does.
template <bool INIT>
__global__ void __launch_bounds__(256) saa_k_mg_rz(int64_t n_nodes, const SaaCgState *__restrict__ S, const double *__restrict__ r,
                                                   const double *__restrict__ z, double *__restrict__ p, double *__restrict__ part,
                                                   int64_t n_parts)
{
    if (S->done) return;
    const int64_t node = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double e[2] = {0.0, 0.0};
    if (node < n_nodes) {
#pragma unroll
        for (int A = 0; A < 3; ++A) {
            const int64_t row = 3 * node + A;
            const double rv = r[row], zv = z[row];
            if (INIT) p[row] = zv;
            e[0] = __dadd_rn(e[0], __dmul_rn(rv, zv));
            e[1] = __dadd_rn(e[1], __dmul_rn(rv, rv));
        }
    }
    if (INIT) {
        saa_cg_block_partials<2>(e, part, n_parts, blockIdx.x);
    } else {
        double e0[1] = {e[0]};
        saa_cg_block_partials<1>(e0, part, n_parts, blockIdx.x);
    }
}

// ---- set-up --------------------------------------------------------------------------------------------------------
// start vector of the power iteration: a hash of the external DOF index in [-1, 1) on free rows, so that set-up is
// bit-reproducible and independent of the node order
__global__ void saa_k_mg_start(int64_t n_nodes, const int32_t *__restrict__ ext, const uint32_t *__restrict__ free_mask,
                               double *__restrict__ x)
{
    const int64_t node = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (node >= n_nodes) return;
    for (int A = 0; A < 3; ++A) {
        const int64_t row = 3 * node + A;
        double v = 0.0;
        if (ext[node] >= 0 && saa_cg_free(free_mask, row)) {
            unsigned long long h = (unsigned long long)(3 * (int64_t)ext[node] + A) + 0x9E3779B97F4A7C15ull;   // splitmix64
            h = (h ^ (h >> 30)) * 0xBF58476D1CE4E5B9ull;
            h = (h ^ (h >> 27)) * 0x94D049BB133111EBull;
            h ^= h >> 31;
            v = __dsub_rn(__dmul_rn((double)(h >> 11), 0x1.0p-52), 1.0);
        }
        x[row] = v;
    }
}

// one power step of B^-1 A: z = B^-1 q (q = A x), partial of q.z (field 0), x = z / sqrt(x.q) (xq: the reduced x.q)
__global__ void __launch_bounds__(256) saa_k_mg_power(int64_t n_nodes, const double *__restrict__ q, double *__restrict__ x,
                                                      const double *__restrict__ binv, const uint32_t *__restrict__ free_mask,
                                                      const double *__restrict__ xq, double *__restrict__ part, int64_t n_parts)
{
    const int64_t node = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double e[1] = {0.0};
    if (node < n_nodes) {
        const double scale = __drcp_rn(__dsqrt_rn(*xq));
        double qv[3], zv[3];
        bool fr[3];
#pragma unroll
        for (int A = 0; A < 3; ++A) {
            fr[A] = saa_cg_free(free_mask, 3 * node + A);
            qv[A] = fr[A] ? q[3 * node + A] : 0.0;
        }
        saa_cg_precond(binv, n_nodes, node, qv, zv);
#pragma unroll
        for (int A = 0; A < 3; ++A) {
            const double zz = fr[A] ? zv[A] : 0.0;
            e[0] = __dadd_rn(e[0], __dmul_rn(qv[A], zz));
            x[3 * node + A] = __dmul_rn(zz, scale);
        }
    }
    saa_cg_block_partials<1>(e, part, n_parts, blockIdx.x);
}

// prolongation table checks: ptr[0] == 0, ptr non-decreasing, columns in [0, n_c); *bad = lowest offending fine node
__global__ void saa_k_mg_check_table(int64_t n_f, int64_t n_c, const int64_t *__restrict__ ptr, const int32_t *__restrict__ col,
                                     unsigned long long *bad)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_f) return;
    bool ok = (e > 0 || ptr[0] == 0) && ptr[e] <= ptr[e + 1];
    if (ok)
        for (int64_t k = ptr[e]; k < ptr[e + 1]; ++k) ok = ok && col[k] >= 0 && col[k] < n_c;
    if (!ok) atomicMin(bad, (unsigned long long)e);
}

// row (external fine node) of every table entry, and the parents' internal coarse nodes
__global__ void saa_k_mg_table_rows(int64_t n_f, const int64_t *__restrict__ ptr, const int32_t *__restrict__ col,
                                    const int32_t *__restrict__ iperm_c, int32_t *__restrict__ row_of, int32_t *__restrict__ cnode)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_f) return;
    for (int64_t k = ptr[e]; k < ptr[e + 1]; ++k) {
        row_of[k] = (int32_t)e;
        cnode[k] = iperm_c[3 * (int64_t)col[k]] / 3;
    }
}

// transposed entries (sorted by coarse node, stably: ascending fine node within one) -> internal fine node, weight
__global__ void saa_k_mg_table_transpose(int64_t nnz, const int32_t *__restrict__ entry, const int32_t *__restrict__ row_of,
                                         const double *__restrict__ w, const int32_t *__restrict__ iperm_f,
                                         int32_t *__restrict__ fnode, double *__restrict__ tw)
{
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nnz) return;
    const int32_t k = entry[j];
    fnode[j] = iperm_f[3 * (int64_t)row_of[k]] / 3;
    tw[j] = w[k];
}

// the caller's dense A_c^-1 (external DOF order, n_ext x n_ext) into internal order (n_int x n_int, zero-filled before)
__global__ void saa_k_mg_coarse_permute(int64_t n_ext, int64_t n_int, const int32_t *__restrict__ iperm, const double *__restrict__ src,
                                        double *__restrict__ dst)
{
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_ext * n_ext) return;
    const int64_t i = k / n_ext, j = k % n_ext;
    dst[(int64_t)iperm[i] * n_int + iperm[j]] = src[k];
}
