// saa_energy.cuh — on-device energy monitor of the central-difference step (include/saa_fem.h, saa_plan_set_energy).
//
// The update of saa_cd_update is algebraically
//     M (d_{n+1} - 2 d_n + d_{n-1}) / dt^2 + alpha M (d_{n+1} - d_{n-1}) / (2 dt) + K d_n = F ramp(t_n).
// Multiplied by (d_{n+1} - d_{n-1}) / 2 and with K = K^T it gives the discrete balance
//     E_{n+1/2} = E_{n-1/2} + dW_n - dD_n,        E_{n-1/2} = T_{n-1/2} + S_{n-1/2},
//     T_{n-1/2} = 1/2 sum m (d_n - d_{n-1})^2 / dt^2,          S_{n-1/2} = 1/2 d_{n-1}^T K d_n,
//     dW_n = F_n . (d_{n+1} - d_{n-1}) / 2,                     dD_n = alpha dt 2 T_n,
//     T_n = 1/2 sum m (d_{n+1} - d_{n-1})^2 / (4 dt^2).
// Every term is formed from values the step already holds: d_n, d_{n-1}, the row force f = LocalK d_n, the mass, the
// load and the new d_{n+1}, so the monitor reads no extra matrix bytes.
//
// Weighting.  The stiffness terms use this rank's OWN row force (the value K2 puts in xbuf on shared rows) on every
// local row: summed over ranks, sum_p d^T K_p d = d^T K d, so they need no owner weighting.  l_M and F_rankwise are
// globally assembled, so mass and load terms are counted on OWNED rows only: the non-shared rows, and a shared row on
// its lowest-rank holder, i.e. where the first entry of the row's rank-ordered source list is the own xbuf.
//
// Determinism.  Sums are reordered against any serial evaluation, but never depend on timing: a slice is reduced by a
// fixed warp tree (K1E), a unit of 256 shared rows or predicted rows by a fixed block tree (K3E, prediction scatter),
// and saa_k_energy_reduce sums those partials with a fixed assignment of partials to threads and a fixed tree; the
// last of its blocks (a ticket counter, no atomics on values) adds the block sums in block order and is the one place
// where the work / dissipation accumulators advance.  Records are therefore bit-identical between runs, launch
// strategies and transports that execute the same step kernels on the same partition.
//
// Partials: field f (0 kinetic_half, 1 coupling, 2 strain, 3 kinetic, 4 work) of partial i lives at part[f*n_parts + i];
// the raw sums are sum m v^2, sum d f and sum F w, the constant factors are applied once, in the reduction.
#pragma once
#include "saa_kernels.cuh"
#include "../../include/saa_fem.h"

#define SAA_ENERGY_PARTS 5

// accumulators and ring parameters of the monitor (device memory; graph replays read everything from here)
struct SaaEnergyDev {
    double W, D, E_arm;             // external work and damping work since the arming step, T + S at the arming step
    long long arm;                  // 1: the next reduced step is the arming step
    long long every, first, cap;    // record when step_idx % every == 0, into slot (step_idx / every - first) % cap
    double *ring;                   // [cap][SAA_ENERGY_FIELDS]
};

// lowest-rank holder of a shared row (rows past the interface are not shared)
__device__ __forceinline__ bool saa_row_owned(const SaaHaloDev &H, int64_t row)
{
    if (row >= H.sh_rows) return true;
    const int64_t k = H.src_ptr[row];
    return k < H.src_ptr[row + 1] && H.src_pos[k] < H.sh_rows;
}

__device__ __forceinline__ double saa_warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = __dadd_rn(v, __shfl_down_sync(0xffffffffu, v, o));
    return v;   // lane 0
}

// fixed-order tree over the 256 threads of a block; the sums are valid in thread 0
__device__ __forceinline__ void saa_block_sum5(double (&e)[SAA_ENERGY_PARTS])
{
    __shared__ double sh[SAA_ENERGY_PARTS][8];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int f = 0; f < SAA_ENERGY_PARTS; ++f) e[f] = saa_warp_sum(e[f]);
    if (lane == 0)
#pragma unroll
        for (int f = 0; f < SAA_ENERGY_PARTS; ++f) sh[f][w] = e[f];
    __syncthreads();
    if (threadIdx.x == 0)
#pragma unroll
        for (int f = 0; f < SAA_ENERGY_PARTS; ++f) {
            double t = 0.0;
            for (int k = 0; k < 8; ++k) t = __dadd_rn(t, sh[f][k]);
            e[f] = t;
        }
    __syncthreads();   // sh is reused by a later call
}

// the energy terms of one row; x0 = d_n, xn = d_{n-1}, x1 = stored d_{n+1}, f = own row force, Fe = F ramp(t_n)
// skip_new: the row is overwritten after the step (PREDICT); its d_{n+1} terms are added by the prediction scatter
__device__ __forceinline__ void saa_energy_row(double (&e)[SAA_ENERGY_PARTS], bool own, bool skip_new, double M, double Fe,
                                               double f, double x0, double xn, double x1)
{
    const double v = __dsub_rn(x0, xn);
    e[1] = __dadd_rn(e[1], __dmul_rn(xn, f));
    e[2] = __dadd_rn(e[2], __dmul_rn(x0, f));
    if (own) {
        e[0] = __dadd_rn(e[0], __dmul_rn(__dmul_rn(M, v), v));
        if (!skip_new) {
            const double w = __dsub_rn(x1, xn);
            e[3] = __dadd_rn(e[3], __dmul_rn(__dmul_rn(M, w), w));
            e[4] = __dadd_rn(e[4], __dmul_rn(Fe, w));
        }
    }
}

// K1E: K1 (the interior path of saa_k_step) over slices [slice_begin, n_slices) plus the per-slice partials.  Same
// saa_node_dot, saa_cd_update and Dirichlet clamp as K1, so d1 is bit-identical.  H is the plan's halo (sh_rows of
// the real interface) for the owner test of shared rows stepped locally.  skip (PREDICT steps, else null): rows the
// prediction overwrites; their d_{n-1} goes to stash and their d_{n+1} terms are left to saa_k_hook_scatter_energy.
template <int MODE>
__global__ void __launch_bounds__(256, 3) saa_k_step_energy(SaaDev P, SaaHaloDev H, const double *__restrict__ d0,
                                                            double *__restrict__ dn_d1, const SaaClock *clk_in, SaaClock *clk_out,
                                                            int64_t slice_begin, unsigned int count_sync, double *__restrict__ part,
                                                            int64_t n_parts, const uint32_t *__restrict__ skip,
                                                            double *__restrict__ stash)
{
    const double tn = clk_in->tn;
    if (clk_out != nullptr && blockIdx.x == 0 && threadIdx.x == 0) {
        clk_out->tn = __dadd_rn(tn, P.dt);
        clk_out->sync_step = clk_in->sync_step + count_sync;
        clk_out->step_idx = clk_in->step_idx + 1ull;
    }
    const int lane = threadIdx.x & 31;
    const int64_t slice = slice_begin + (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (slice >= P.n_slices) return;
    double s[3];
    saa_node_dot<MODE, true>(P, slice, lane, d0, s);
    const double ramp = saa_ramp(tn);
    const int64_t node = slice * 32 + lane;
    double e[SAA_ENERGY_PARTS] = {0.0, 0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int A = 0; A < 3; ++A) {
        const int64_t row = 3 * node + A;
        const double M = P.M[P.node_mass ? node : row], F = P.F[row], x0 = d0[row], xn = dn_d1[row];
        const double d1 = saa_cd_update(P, __dadd_rn(0.0, s[A]), F, M, x0, xn, ramp);
        const bool clamp = (P.dir_mask[row >> 5] >> (row & 31)) & 1u;
        const double x1 = clamp ? 0.0 : d1;
        dn_d1[row] = x1;
        const bool skipped = skip != nullptr && ((skip[row >> 5] >> (row & 31)) & 1u);
        if (skipped) stash[row] = xn;
        saa_energy_row(e, saa_row_owned(H, row), skipped, M, __dmul_rn(F, ramp), s[A], x0, xn, x1);
    }
#pragma unroll
    for (int f = 0; f < SAA_ENERGY_PARTS; ++f) e[f] = saa_warp_sum(e[f]);
    if (lane == 0)
#pragma unroll
        for (int f = 0; f < SAA_ENERGY_PARTS; ++f) part[f * n_parts + slice] = e[f];
}

// K3E: K3 (saa_k_shared_update) plus one partial per unit of 256 shared rows, stored at part index part0 + unit.
// The coupling and strain terms use the own partial force xbuf[row], not the rank-ordered sum.
template <bool PEER>
__global__ void __launch_bounds__(256) saa_k_shared_update_energy(SaaDev P, SaaHaloDev H, const double *__restrict__ d0,
                                                                  double *__restrict__ dn_d1, const SaaClock *clk_in,
                                                                  double *__restrict__ part, int64_t n_parts, int64_t part0)
{
    const double *recv = H.recv;
    if (PEER) {
        const unsigned long long step = clk_in->sync_step;
        if (threadIdx.x < H.n_nb) saa_wait_ge<true>(H.flags + threadIdx.x, step + 1ull, H.err);
        __syncthreads();
        recv += (int64_t)(step & 1ull) * H.recv_stride;
    }
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double e[SAA_ENERGY_PARTS] = {0.0, 0.0, 0.0, 0.0, 0.0};
    if (row < H.sh_rows) {
        double Fi = 0.0;
        for (int64_t k = H.src_ptr[row]; k < H.src_ptr[row + 1]; ++k) {
            const int32_t s = H.src_pos[k];
            const double v = (s < H.sh_rows) ? H.xbuf[s] : *((const volatile double *)(recv + (s - H.sh_rows)));
            Fi = __dadd_rn(Fi, v);
        }
        const double ramp = saa_ramp(clk_in->tn);
        const double M = P.M[P.node_mass ? row / 3 : row], F = P.F[row], x0 = d0[row], xn = dn_d1[row];
        const double d1 = saa_cd_update(P, Fi, F, M, x0, xn, ramp);
        const bool clamp = (P.dir_mask[row >> 5] >> (row & 31)) & 1u;
        const double x1 = clamp ? 0.0 : d1;
        dn_d1[row] = x1;
        saa_energy_row(e, saa_row_owned(H, row), false, M, __dmul_rn(F, ramp), H.xbuf[row], x0, xn, x1);
    }
    saa_block_sum5(e);
    if (threadIdx.x == 0)
#pragma unroll
        for (int f = 0; f < SAA_ENERGY_PARTS; ++f) part[f * n_parts + part0 + blockIdx.x] = e[f];
}

// saa_k_hook_scatter plus the d_{n+1} terms (kinetic, work) of the rows it overwrites, computed from the stored value;
// d_{n-1} of those rows was stashed by K1E.  One partial per block of 256 predicted rows, at part index blockIdx.x.
__global__ void __launch_bounds__(256) saa_k_hook_scatter_energy(SaaDev P, SaaHaloDev H, int64_t n, const int32_t *__restrict__ rows,
                                                                 const SaaHookDev *__restrict__ hk, const SaaClock *__restrict__ clk_old,
                                                                 double *__restrict__ d1, const double *__restrict__ stash,
                                                                 double *__restrict__ part, int64_t n_parts)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const long long r = (long long)clk_old->step_idx - hk->pred_base_step;
    double e[SAA_ENERGY_PARTS] = {0.0, 0.0, 0.0, 0.0, 0.0};
    if (i < n) {
        const int64_t row = rows[i];
        double x1;
        if (r >= 0 && r < hk->pred_rows) {
            x1 = hk->pred_table[r * n + i];
            d1[row] = x1;
        } else {
            x1 = d1[row];
        }
        if (saa_row_owned(H, row)) {
            const double M = P.M[P.node_mass ? row / 3 : row];
            const double w = __dsub_rn(x1, stash[row]);
            e[3] = __dmul_rn(__dmul_rn(M, w), w);
            e[4] = __dmul_rn(__dmul_rn(P.F[row], saa_ramp(clk_old->tn)), w);
        }
    }
    saa_block_sum5(e);
    if (threadIdx.x == 0)
#pragma unroll
        for (int f = 0; f < SAA_ENERGY_PARTS; ++f) part[f * n_parts + blockIdx.x] = e[f];
}

// Reduction of one step: partials [a0, a0 + na) of part (stride n_parts) and [b0, b0 + nb) of part_b (stride nb_parts).
// Thread t of block b sums the partials b*256 + t + k*256*gridDim.x (k ascending), each block reduces with the fixed
// tree into stage, and the last block to finish adds the block sums in block order.  That block writes the record of
// step clk_old->step_idx (if it is a multiple of `every`) and then advances W and D by this step's dW_n and dD_n.
__global__ void __launch_bounds__(256) saa_k_energy_reduce(const double *__restrict__ part, int64_t n_parts, int64_t a0, int64_t na,
                                                           const double *__restrict__ part_b, int64_t nb_parts, int64_t b0, int64_t nb,
                                                           double *stage, unsigned int *ticket, SaaEnergyDev *E,
                                                           const SaaClock *__restrict__ clk_old, double dt, double dt2, double alpha)
{
    double e[SAA_ENERGY_PARTS] = {0.0, 0.0, 0.0, 0.0, 0.0};
    const int64_t n = na + nb, G = gridDim.x;
    for (int64_t v = (int64_t)blockIdx.x * 256 + threadIdx.x; v < n; v += 256 * G) {
        const double *q = (v < na) ? part + a0 + v : part_b + b0 + (v - na);
        const int64_t stride = (v < na) ? n_parts : nb_parts;
#pragma unroll
        for (int f = 0; f < SAA_ENERGY_PARTS; ++f) e[f] = __dadd_rn(e[f], q[f * stride]);
    }
    saa_block_sum5(e);
    __shared__ unsigned int s_last;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int f = 0; f < SAA_ENERGY_PARTS; ++f) stage[f * G + blockIdx.x] = e[f];
        __threadfence();
        s_last = (atomicAdd(ticket, 1u) == (unsigned int)G - 1u) ? 1u : 0u;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
#pragma unroll
    for (int f = 0; f < SAA_ENERGY_PARTS; ++f) e[f] = 0.0;
    for (int64_t b = threadIdx.x; b < G; b += 256)
#pragma unroll
        for (int f = 0; f < SAA_ENERGY_PARTS; ++f) e[f] = __dadd_rn(e[f], __ldcg(stage + f * G + b));
    saa_block_sum5(e);
    if (threadIdx.x != 0) return;
    *ticket = 0u;                                           // re-armed for the next step (stream-ordered)
    const long long step = (long long)clk_old->step_idx;
    const double kin_half = __dmul_rn(0.5, e[0]) / dt2;
    const double coupling = __dmul_rn(0.5, e[1]);
    const double strain = __dmul_rn(0.5, e[2]);
    const double kin = __dmul_rn(0.5, e[3]) / __dmul_rn(4.0, dt2);
    const double work = __dmul_rn(0.5, e[4]);
    if (E->arm) {
        E->E_arm = __dadd_rn(kin_half, coupling);
        E->W = 0.0;
        E->D = 0.0;
        E->arm = 0;
    }
    if (step % E->every == 0) {
        double *rec = E->ring + ((step / E->every - E->first) % E->cap) * SAA_ENERGY_FIELDS;
        rec[0] = (double)step;
        rec[1] = clk_old->tn;
        rec[2] = kin_half;
        rec[3] = coupling;
        rec[4] = strain;
        rec[5] = kin;
        rec[6] = E->W;
        rec[7] = E->D;
        rec[8] = E->E_arm;
    }
    E->W = __dadd_rn(E->W, work);
    E->D = __dadd_rn(E->D, __dmul_rn(__dmul_rn(__dmul_rn(alpha, dt), 2.0), kin));
}
