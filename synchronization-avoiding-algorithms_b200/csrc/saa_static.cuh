// saa_static.cuh — static solve on the resident stiffness (include/saa_fem.h: saa_plan_apply_stiffness_dev,
// saa_plan_solve_static_dev and their group forms; DESIGN.md §7c).
//
// The system is the one Tools/Steady_solvers.py:13-22 builds: A = S K S + (I - S), b = S F, where S keeps the free
// DOFs (not Dirichlet, not slice padding) and F is the plan's un-ramped load.  It is solved by conjugate gradients with
// a 3x3 node-block Jacobi preconditioner B (the inverse of every node's diagonal block, clamped rows and columns
// replaced by the identity).  x, r, p, q and z are 0 on every clamped DOF, so q = A p is S (K p).
//
// Determinism (the energy monitor's rules, saa_energy.cuh): every dot product is formed from per-block partials with a
// fixed warp and block tree, saa_k_cg_reduce sums them with a fixed assignment of partials to threads and its last
// block (ticket counter, no atomics on values) adds the block sums in block order into the rank's slot.  The rank
// slots are added in ascending rank order by saa_k_cg_scalar, the only kernel that writes alpha, beta and the flags.
// A partial counts OWNED rows only: the non-shared rows, and a shared row on its lowest-rank holder.  Shared rows of
// q are the rank-ordered holder sums (the association of syn_cpus), so every holder updates its copy of a shared row
// with identical bits.  Every work kernel reads the `done` flag first and leaves its vectors untouched once the
// criterion has held (or max_iter was reached, or a breakdown was detected): a chunk of iterations replayed from a
// CUDA graph returns the iterate of the first iteration that met the criterion.
#pragma once
#include "saa_energy.cuh"

// device-resident scalars of one solve (one per group; every plan reads the same alpha and beta)
struct SaaCgState {
    double bb, rr, rz, alpha, beta, rtol, rr_true;
    long long it, max_iter;
    long long done;                 // converged, max_iter reached or breakdown: work kernels leave every vector unchanged
    long long converged;
    long long fail, fail_it;        // breakdown code (1: p.Ap <= 0, 2: r.z <= 0, 3: non-finite residual) and iteration
};

__device__ __forceinline__ bool saa_cg_free(const uint32_t *free_mask, int64_t row) { return (free_mask[row >> 5] >> (row & 31)) & 1u; }

// NF block sums of a 256-thread block by a fixed tree, stored at part[f * n_parts + idx]
template <int NF>
__device__ __forceinline__ void saa_cg_block_partials(double (&e)[NF], double *part, int64_t n_parts, int64_t idx)
{
    __shared__ double sh[NF][8];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int f = 0; f < NF; ++f) e[f] = saa_warp_sum(e[f]);
    if (lane == 0)
#pragma unroll
        for (int f = 0; f < NF; ++f) sh[f][w] = e[f];
    __syncthreads();
    if (threadIdx.x == 0)
#pragma unroll
        for (int f = 0; f < NF; ++f) {
            double t = 0.0;
            for (int k = 0; k < 8; ++k) t = __dadd_rn(t, sh[f][k]);
            part[f * n_parts + idx] = t;
        }
}

// Stiffness apply over the slices, one thread per node, one warp per slice (as K1): s = LocalK x in the stored CSR
// order from 0.0 (saa_node_dot), so a host-built plan gives scipy's LocalK @ x bit for bit.
//   RAW: y = s on every row.
//   DOT: y = S s, and one partial of x.y per block (q = A p with x = p).
//   RES: y = b - S s with b = S F (r = b - A x, x = 0 on clamped rows), partials of y.y and b.b.
// Shared slices (a plan of a group) store the raw partial s and contribute 0: saa_k_cg_shared finishes those rows after
// the holder exchange.  x is only read here.
enum { SAA_APPLY_RAW = 0, SAA_APPLY_DOT = 1, SAA_APPLY_RES = 2 };
template <int MODE>
__global__ void __launch_bounds__(256, 3) saa_k_cg_apply(SaaDev P, const double *__restrict__ x, double *__restrict__ y,
                                                         const uint32_t *__restrict__ free_mask, double *__restrict__ part,
                                                         int64_t n_parts, const long long *gate)
{
    if (gate != nullptr && *gate) return;                      // the same value for the whole grid
    const int lane = threadIdx.x & 31;
    const int64_t slice = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    double e[2] = {0.0, 0.0};
    if (slice < P.n_slices) {
        double s[3];
        saa_node_dot<1, true>(P, slice, lane, x, s);
#pragma unroll
        for (int A = 0; A < 3; ++A) {
            const int64_t row = 3 * (slice * 32 + lane) + A;
            if (MODE == SAA_APPLY_RAW || slice < P.sh_slices) {
                y[row] = s[A];
            } else if (MODE == SAA_APPLY_DOT) {
                const double q = saa_cg_free(free_mask, row) ? s[A] : 0.0;
                y[row] = q;
                e[0] = __dadd_rn(e[0], __dmul_rn(x[row], q));
            } else {
                const bool fr = saa_cg_free(free_mask, row);
                const double b = fr ? P.F[row] : 0.0;
                const double r = fr ? __dsub_rn(b, s[A]) : 0.0;
                y[row] = r;
                e[0] = __dadd_rn(e[0], __dmul_rn(r, r));
                e[1] = __dadd_rn(e[1], __dmul_rn(b, b));
            }
        }
    }
    if (MODE == SAA_APPLY_DOT) {
        double e1[1] = {e[0]};
        saa_cg_block_partials<1>(e1, part, n_parts, blockIdx.x);
    } else if (MODE == SAA_APPLY_RES) {
        saa_cg_block_partials<2>(e, part, n_parts, blockIdx.x);
    }
}

// The shared rows of a plan of a group after the exchange of the partials (H: the solve's own copies of the pack and
// receive buffers): F_int = ((0.0 + f_r0) + f_r1) + ... over the holders in ascending rank order, then the finish of
// saa_k_cg_apply; one partial per unit of 256 rows at part index part0 + unit, owned rows only.
template <int MODE>
__global__ void __launch_bounds__(256) saa_k_cg_shared(SaaDev P, SaaHaloDev H, const double *__restrict__ x, double *__restrict__ y,
                                                       const uint32_t *__restrict__ free_mask, double *__restrict__ part,
                                                       int64_t n_parts, int64_t part0, const long long *gate)
{
    if (gate != nullptr && *gate) return;
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double e[2] = {0.0, 0.0};
    if (row < H.sh_rows) {
        double Fi = 0.0;
        for (int64_t k = H.src_ptr[row]; k < H.src_ptr[row + 1]; ++k) {
            const int32_t s = H.src_pos[k];
            Fi = __dadd_rn(Fi, (s < H.sh_rows) ? H.xbuf[s] : H.recv[s - H.sh_rows]);
        }
        const bool fr = saa_cg_free(free_mask, row), own = saa_row_owned(H, row);
        if (MODE == SAA_APPLY_DOT) {
            const double q = fr ? Fi : 0.0;
            y[row] = q;
            if (own) e[0] = __dmul_rn(x[row], q);
        } else {
            const double b = fr ? P.F[row] : 0.0;
            const double r = fr ? __dsub_rn(b, Fi) : 0.0;
            y[row] = r;
            if (own) { e[0] = __dmul_rn(r, r); e[1] = __dmul_rn(b, b); }
        }
    }
    if (MODE == SAA_APPLY_DOT) {
        double e1[1] = {e[0]};
        saa_cg_block_partials<1>(e1, part, n_parts, part0 + blockIdx.x);
    } else {
        saa_cg_block_partials<2>(e, part, n_parts, part0 + blockIdx.x);
    }
}

// z = B^-1 r per node (B^-1 symmetric, six planes of n_nodes: 00 01 02 11 12 22), left-to-right sums
__device__ __forceinline__ void saa_cg_precond(const double *__restrict__ binv, int64_t n_nodes, int64_t node, const double (&r)[3],
                                               double (&z)[3])
{
    double b[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) b[k] = binv[k * n_nodes + node];
    z[0] = __dadd_rn(__dadd_rn(__dmul_rn(b[0], r[0]), __dmul_rn(b[1], r[1])), __dmul_rn(b[2], r[2]));
    z[1] = __dadd_rn(__dadd_rn(__dmul_rn(b[1], r[0]), __dmul_rn(b[3], r[1])), __dmul_rn(b[4], r[2]));
    z[2] = __dadd_rn(__dadd_rn(__dmul_rn(b[2], r[0]), __dmul_rn(b[4], r[1])), __dmul_rn(b[5], r[2]));
}

// (b) of an iteration, one thread per node: x += alpha p, r -= alpha q, z = B^-1 r, partials of r.z and r.r (owned
// rows) per block of 256 nodes.  INIT (before the first iteration): z = B^-1 r, p = z and the same partials.
template <bool INIT>
__global__ void __launch_bounds__(256) saa_k_cg_update(int64_t n_nodes, SaaHaloDev H, const SaaCgState *__restrict__ S,
                                                       double *__restrict__ x, double *__restrict__ r, double *__restrict__ p,
                                                       const double *__restrict__ q, double *__restrict__ z,
                                                       const double *__restrict__ binv, const uint32_t *__restrict__ free_mask,
                                                       double *__restrict__ part, int64_t n_parts)
{
    if (S->done) return;
    const int64_t node = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double e[2] = {0.0, 0.0};
    if (node < n_nodes) {
        const double alpha = S->alpha;
        double rv[3], zv[3];
        bool fr[3];
#pragma unroll
        for (int A = 0; A < 3; ++A) {
            const int64_t row = 3 * node + A;
            fr[A] = saa_cg_free(free_mask, row);
            if (INIT) {
                rv[A] = r[row];
            } else if (fr[A]) {
                x[row] = __dadd_rn(x[row], __dmul_rn(alpha, p[row]));
                rv[A] = __dsub_rn(r[row], __dmul_rn(alpha, q[row]));
                r[row] = rv[A];
            } else {
                rv[A] = 0.0;
            }
        }
        saa_cg_precond(binv, n_nodes, node, rv, zv);
#pragma unroll
        for (int A = 0; A < 3; ++A) {
            const int64_t row = 3 * node + A;
            const double zz = fr[A] ? zv[A] : 0.0;
            z[row] = zz;
            if (INIT) p[row] = zz;
            if (saa_row_owned(H, row)) {
                e[0] = __dadd_rn(e[0], __dmul_rn(rv[A], zz));
                e[1] = __dadd_rn(e[1], __dmul_rn(rv[A], rv[A]));
            }
        }
    }
    saa_cg_block_partials<2>(e, part, n_parts, blockIdx.x);
}

// (c) p = z + beta p
__global__ void __launch_bounds__(256) saa_k_cg_direction(int64_t n_rows, const SaaCgState *__restrict__ S, const double *__restrict__ z,
                                                          double *__restrict__ p)
{
    if (S->done) return;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_rows) p[i] = __dadd_rn(z[i], __dmul_rn(S->beta, p[i]));
}

// Sum of NF fields of partials [0, n) (stride n_parts) into this rank's slots out[f * out_stride]: thread t of block b
// adds the partials b*256 + t + k*256*gridDim.x (k ascending), each block reduces with the fixed tree into stage, and
// the last block to finish adds the block sums in block order.
template <int NF>
__global__ void __launch_bounds__(256) saa_k_cg_reduce(const double *__restrict__ part, int64_t n_parts, int64_t n, double *stage,
                                                       unsigned int *ticket, double *out, int64_t out_stride, const long long *gate)
{
    if (gate != nullptr && *gate) return;
    double e[NF];
#pragma unroll
    for (int f = 0; f < NF; ++f) e[f] = 0.0;
    const int64_t G = gridDim.x;
    for (int64_t v = (int64_t)blockIdx.x * 256 + threadIdx.x; v < n; v += 256 * G)
#pragma unroll
        for (int f = 0; f < NF; ++f) e[f] = __dadd_rn(e[f], part[f * n_parts + v]);
    saa_cg_block_partials<NF>(e, stage, G, blockIdx.x);
    __shared__ unsigned int s_last;
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = (atomicAdd(ticket, 1u) == (unsigned int)G - 1u) ? 1u : 0u;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
#pragma unroll
    for (int f = 0; f < NF; ++f) e[f] = 0.0;
    for (int64_t b = threadIdx.x; b < G; b += 256)
#pragma unroll
        for (int f = 0; f < NF; ++f) e[f] = __dadd_rn(e[f], __ldcg(stage + f * G + b));
    __syncthreads();                                           // the shared tree of the first call is reused
    saa_cg_block_partials<NF>(e, out, out_stride, 0);
    if (threadIdx.x == 0) *ticket = 0u;                         // re-armed for the next reduction (stream-ordered)
}

// The scalar step of the iteration, one thread: the P rank slots (rk[f * P + rank]) added in ascending rank order.
//   stage 0  after the residual apply: rr, bb
//   stage 1  after the INIT update: rz, rr; criterion at iteration 0
//   stage 2  after q = A p: alpha = rz / p.q
//   stage 3  after the update: history, criterion, beta, iteration count
//   stage 4  after the final residual apply: rr_true
enum { SAA_CG_RES0 = 0, SAA_CG_INIT = 1, SAA_CG_ALPHA = 2, SAA_CG_BETA = 3, SAA_CG_TRUE = 4 };
__global__ void saa_k_cg_scalar(SaaCgState *S, const double *__restrict__ rk, int P, int stage, double *hist)
{
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    if ((stage == SAA_CG_ALPHA || stage == SAA_CG_BETA) && S->done) return;
    double a = 0.0, b = 0.0;
    for (int q = 0; q < P; ++q) {
        a = __dadd_rn(a, rk[q]);
        b = __dadd_rn(b, rk[P + q]);
    }
    const auto met = [&](double rr) { return __dsqrt_rn(rr) <= __dmul_rn(S->rtol, __dsqrt_rn(S->bb)); };
    const auto breakdown = [&](long long code) { S->fail = code; S->fail_it = S->it; S->done = 1; };
    if (stage == SAA_CG_RES0) {
        S->rr = a;
        S->bb = b;
    } else if (stage == SAA_CG_INIT) {
        S->rz = a;
        S->rr = b;
        if (!isfinite(b)) breakdown(3);
        else if (met(b)) { S->converged = 1; S->done = 1; }
        else if (!(a > 0.0) || !isfinite(a)) breakdown(2);
        else if (S->max_iter <= 0) S->done = 1;
    } else if (stage == SAA_CG_ALPHA) {
        if (!(a > 0.0) || !isfinite(a)) breakdown(1);
        else S->alpha = __ddiv_rn(S->rz, a);
        if (!S->done && !isfinite(S->alpha)) breakdown(1);
    } else if (stage == SAA_CG_BETA) {
        if (hist != nullptr) hist[S->it] = __dsqrt_rn(b);
        S->rr = b;
        if (!isfinite(b)) { breakdown(3); return; }
        if (met(b)) { S->it += 1; S->converged = 1; S->done = 1; return; }
        if (!(a > 0.0) || !isfinite(a)) { breakdown(2); return; }
        S->it += 1;
        S->beta = __ddiv_rn(a, S->rz);
        S->rz = a;
        if (S->it >= S->max_iter) S->done = 1;
    } else {
        S->rr_true = a;
    }
}

// ---- preconditioner set-up ----------------------------------------------------------------------------------------
// free rows: not Dirichlet and not slice padding (ext_of_int: external node of every internal node, -1 for padding)
__global__ void saa_k_cg_free_mask(int64_t n_words, const uint32_t *__restrict__ dir, const int32_t *__restrict__ ext_of_int,
                                   uint32_t *__restrict__ free_mask)
{
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= n_words) return;
    uint32_t word = 0u;
    for (int bit = 0; bit < 32; ++bit) {
        const int64_t row = 32 * w + bit;
        if (ext_of_int[row / 3] >= 0 && !((dir[w] >> bit) & 1u)) word |= 1u << bit;
    }
    free_mask[w] = word;
}

__global__ void saa_k_cg_mask(int64_t n_rows, const uint32_t *__restrict__ free_mask, double *__restrict__ v)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_rows && !saa_cg_free(free_mask, i)) v[i] = 0.0;
}

// the node's diagonal block (the first block whose column node is the node itself; the padding blocks that follow
// also point at the node but hold zeros) as three column vectors c_b[3 node + A] = K(A, b)
__global__ void __launch_bounds__(256) saa_k_cg_diag(SaaDev P, double *__restrict__ c0, double *__restrict__ c1, double *__restrict__ c2)
{
    const int lane = threadIdx.x & 31;
    const int64_t slice = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (slice >= P.n_slices) return;
    const int64_t node = slice * 32 + lane, beg = P.slice_ptr[slice];
    const int len = (int)((P.slice_ptr[slice + 1] - beg) >> 5);
    const char *v = (const char *)(P.val + P.val_ptr[slice]);
    const long long *b = P.vbase + P.vb_ptr[slice];
    double a[9] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    for (int j = 0; j < len; ++j) {
        const unsigned m = P.pmask[(beg >> 5) + j];
        if (P.col[beg + 32 * j + lane] == (int32_t)node) {
            saa_load_block_lane(v, b, lane, m, a);
            break;
        }
        saa_next_block(v, b, m);
    }
#pragma unroll
    for (int A = 0; A < 3; ++A) {
        c0[3 * node + A] = a[3 * A];
        c1[3 * node + A] = a[3 * A + 1];
        c2[3 * node + A] = a[3 * A + 2];
    }
}

// B^-1 of every node from its (holder-summed) diagonal block, clamped rows and columns replaced by the identity:
// Cholesky L L^T of the lower triangle, B^-1 = L^-T L^-1.  A block that is not positive definite (or gives a
// non-finite inverse) lowers *bad to its external node.
__global__ void saa_k_cg_binv(int64_t n_nodes, const double *__restrict__ c0, const double *__restrict__ c1, const double *__restrict__ c2,
                              const uint32_t *__restrict__ free_mask, const int32_t *__restrict__ ext_of_int, double *__restrict__ binv,
                              unsigned long long *bad)
{
    const int64_t node = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (node >= n_nodes) return;
    const int64_t r0 = 3 * node;
    bool fr[3];
#pragma unroll
    for (int A = 0; A < 3; ++A) fr[A] = saa_cg_free(free_mask, r0 + A);
    const auto m = [&](int A, int b, const double *c) { return (fr[A] && fr[b]) ? c[r0 + A] : (A == b ? 1.0 : 0.0); };
    const double m00 = m(0, 0, c0), m10 = m(1, 0, c0), m20 = m(2, 0, c0), m11 = m(1, 1, c1), m21 = m(2, 1, c1), m22 = m(2, 2, c2);
    bool ok = m00 > 0.0;
    const double l00 = __dsqrt_rn(m00);
    const double l10 = __ddiv_rn(m10, l00), l20 = __ddiv_rn(m20, l00);
    const double d11 = __dsub_rn(m11, __dmul_rn(l10, l10));
    ok = ok && d11 > 0.0;
    const double l11 = __dsqrt_rn(d11);
    const double l21 = __ddiv_rn(__dsub_rn(m21, __dmul_rn(l20, l10)), l11);
    const double d22 = __dsub_rn(__dsub_rn(m22, __dmul_rn(l20, l20)), __dmul_rn(l21, l21));
    ok = ok && d22 > 0.0;
    const double l22 = __dsqrt_rn(d22);
    const double i00 = __drcp_rn(l00), i11 = __drcp_rn(l11), i22 = __drcp_rn(l22);
    const double i10 = -__dmul_rn(__dmul_rn(l10, i00), i11);
    const double i21 = -__dmul_rn(__dmul_rn(l21, i11), i22);
    const double i20 = -__dmul_rn(__dadd_rn(__dmul_rn(l20, i00), __dmul_rn(l21, i10)), i22);
    double b[6];
    b[0] = __dadd_rn(__dadd_rn(__dmul_rn(i00, i00), __dmul_rn(i10, i10)), __dmul_rn(i20, i20));
    b[1] = __dadd_rn(__dmul_rn(i10, i11), __dmul_rn(i20, i21));
    b[2] = __dmul_rn(i20, i22);
    b[3] = __dadd_rn(__dmul_rn(i11, i11), __dmul_rn(i21, i21));
    b[4] = __dmul_rn(i21, i22);
    b[5] = __dmul_rn(i22, i22);
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        ok = ok && isfinite(b[k]);
        binv[k * n_nodes + node] = b[k];
    }
    if (!ok) atomicMin(bad, (unsigned long long)ext_of_int[node]);
}
