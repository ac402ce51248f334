// saa_kernels.cuh — sm_100a kernels of the explicit FE time step.
//
// One time step of /root/reference/Tools/Dynamic_solver.py:9-34 for one partition:
//   F_int = LocalK.dot(d0)                         (:12, scipy csr_matvec order)
//   F_ext = F_rankwise * linear_ramp(tn)           (:13, commons.py:7-11)
//   d1    = (dt**2*(F_ext-F_int) + 2*M*d0 - M*dn + dt/2*M*alpha*dn) / (M + 0.5*alpha*M*dt)   (:17/:29)
//   d1[Local_Dirichlet] = 0                        (:20/:32)
// fused into a single pass over the matrix.  Arithmetic contract: every multiply, add, subtract and
// divide below is an explicitly rounded binary64 intrinsic (__dmul_rn/__dadd_rn/__dsub_rn/__ddiv_rn),
// which nvcc never contracts into FMA, and the row sum runs over the stored entries in order starting
// from 0.0 — the same sequence of roundings scipy/numpy perform, hence bit-identical results.
//
// Storage (HBM): plane-masked node-block sliced ELL.  The stiffness of 3-D elasticity is made of 3x3 node blocks, so
// one thread owns one NODE (its three DOF rows) and one warp owns a slice of 32 nodes.  Block j of the node of lane l in
// slice s has one column-node id and up to nine value planes (plane (A,B) = entry (A,B) of block j in all 32 lanes);
// slice_ptr counts block-lanes, the block-row of block j is r = slice_ptr[s]/32 + j:
//     column node of block j  :  col[slice_ptr[s] + j*32 + l]
//     stored planes of block j:  bit 3A+B of pmask[r]
//     value (A,B) of block j  :  val[val_ptr[s] + 32*(off_j + popc(pmask[r] & ((1 << (3A+B)) - 1))) + l]  if that bit is set
// where off_j is the number of planes stored for blocks 0..j-1 of the slice.  A plane is stored iff at least one lane
// of the slice has a stored CSR entry there; a plane that is not stored is 0.0 in every lane, and the kernel puts 0.0
// in the register instead of loading it, so the arithmetic is the same as with all nine planes.  On structured meshes
// the 32 nodes of a slice share their stencil, so whole planes are zero in every lane (DESIGN.md §3).  Every warp-wide
// load stays a fully coalesced, aligned 256-B (values) or 128-B (ids) request, and the column id is shared by the
// entries of a block.  Entries the reference dropped as exact zeros (csr_matrix(dense), Mat_construction.py:150) in a
// stored plane are 0.0; adding 0.0*x leaves a finite row sum bit-identical (the sum starts at +0.0 and can never
// become -0.0).  Within a row the blocks are in ascending column order and inside a block B = 0,1,2, i.e. exactly the
// stored order of the CSR row, which is the summation order of csr_matvec.  SAA_PLANE_MASK=0 at finalisation stores
// all nine planes of every block (pmask = 0x1FF, val_ptr[s] = 9*slice_ptr[s]).
// Nodes are ordered boundary-first (nodes of the partition interface, then interior) and, inside windows of
// SIGMA nodes, by decreasing block count, so slices are almost padding-free; all vectors (d0, dn, M, F) live
// in that internal order (row = 3*node + component) and are streamed.  The only non-streaming access is the
// gather of the three d0 components of a column node (24 contiguous bytes).
#pragma once
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace cg = cooperative_groups;

#ifndef SAA_DOT_MODE
#define SAA_DOT_MODE 0
#endif
#ifndef SAA_UNROLL
#define SAA_UNROLL 2          // blocks whose loads are in flight together per thread (2 x at most 76 B x 32 lanes per warp)
#endif

struct SaaDev {
    int64_t n_rows;            // padded DOF rows = 3 * 32 * n_slices
    int64_t n_slices;          // slices of 32 nodes
    int64_t sh_slices;         // slices [0, sh_slices) hold the shared (interface) nodes
    const int64_t *slice_ptr;  // [n_slices + 1] offsets in block-lanes (multiples of 32)
    const int64_t *val_ptr;    // [n_slices + 1] offsets of the slices in val, in doubles
    const uint16_t *pmask;     // [block-rows] stored value planes of each block-row (see above)
    const double *val;         // stored value planes
    const int32_t *col;        // internal column NODE ids
    const uint32_t *dir_mask;  // bit (row & 31) of word (row >> 5) set: row is a Dirichlet DOF
    const double *M;           // lumped mass, internal row order — or one value per NODE when node_mass is set (all three
                               // DOFs of every node carry the same bits, checked at finalisation), which saves 16 B per
                               // node-step; the reference's pairwise row sums (commons.py:103-107) may differ in the last
                               // bit between the DOFs of a node and then keep the per-DOF stream
    int node_mass;
    const double *F;           // un-ramped load, internal row order
    double dt, dt2, dt_half, half_alpha, alpha;
};

// (tn, number of synchronised steps so far) live in device memory so that launches can be replayed from a
// CUDA graph; every step reads slot `cur` and writes slot `cur ^ 1`.
struct SaaClock {
    double tn;
    unsigned long long sync_step;   // synchronised steps so far (message / arrival-flag numbering of the peer transport)
    unsigned long long step_idx;    // all steps so far = the loop index i of Data_prepare.py:223 / Online_predictor.py:251
};

// History / prediction hooks read their indices from device memory, so that steps with hooks are graph-replayable too.
struct SaaHookDev {
    const double *pred_table;       // (pred_rows, pred_n) predictions of the shared DOFs (Online_predictor.py:280)
    long long pred_base_step;       // step index whose d1 takes row 0
    long long pred_rows;
    long long hist_every;           // record when step_idx % hist_every == 0 (Data_prepare.py:238)
    long long hist_first;           // step_idx / hist_every of snapshot 0
    long long hist_cap;             // ring capacity in snapshots
};

// halo description on the device
struct SaaHaloDev {
    int64_t sh_rows;            // 32 * sh_slices
    double *xbuf;               // [sh_rows] own partial forces of the shared rows
    double *sendbuf;            // packed messages to all neighbours, concatenated (NCCL / group / host transports)
    const double *recv;         // received partial forces of all neighbours, concatenated like sendbuf
    int64_t recv_stride;        // peer transport: the receive area is double-buffered, parity p lives at recv + p*stride
    const int64_t *dst_ptr;     // [sh_rows + 1] CSR: where the partial force of a shared row goes ...
    const int32_t *dst_pos;     //   position inside sendbuf (or, peer transport, inside the neighbour's receive area)
    const int32_t *dst_nb;      //   neighbour index k of that destination
    const int64_t *src_ptr;     // [sh_rows + 1] CSR: sources of a shared row, ASCENDING holder rank:
    const int32_t *src_pos;     //   < sh_rows: xbuf[src_pos]; otherwise recv[src_pos - sh_rows]
    // peer-memory transport over NVLink (one process per GPU, cudaIpc-mapped receive areas)
    int n_nb;
    double *const *peer_recv;               // [n_nb] base of neighbour k's receive area (mapped peer memory)
    const int64_t *peer_stride;             // [n_nb] its parity stride (the neighbour's total message length)
    unsigned long long *const *peer_flag;   // [n_nb] the neighbour's arrival flag for messages from this rank
    const unsigned long long *flags;        // [n_nb] local arrival flags, flag[k] = number of messages received from k
    unsigned int *done_ctr;                 // blocks of the pack kernel that have finished (last one raises the flags)
    unsigned long long *own_ready;          // fused step: number of steps whose own boundary forces are complete
    unsigned int *err;                      // set when a bounded wait expired (a peer never delivered)
    unsigned int *tail_ticket;              // fused step: [0..2], [8..10] two sets of (tail blocks gone, claimed shared-row units, waiting blocks); [16] fused-launch number
    int dbg;                                // -DSAA_DEBUG_PEER builds only (timing experiments): 1 no waits, 2 local stores,
                                            // 4 skip the shared rows, 8 treat boundary slices as interior
};

__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long *p)
{
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys_u64(unsigned long long *p, unsigned long long v)
{
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// relaxed system-scope store: together with the __threadfence_system() in front of it this is a release pattern
// (fence.acq_rel.sys ; st.relaxed.sys), which publishes to SEVERAL flags with ONE fence instead of one per st.release
__device__ __forceinline__ void st_relaxed_sys_u64(unsigned long long *p, unsigned long long v)
{
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_gpu_u64(const unsigned long long *p)
{
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu_u64(unsigned long long *p, unsigned long long v)
{
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// bounded spin (about 30 s at 1.9 GHz — ranks may legitimately be seconds apart, e.g. around file output or the first
// cuDNN call of the surrogate): a peer that never delivers must not hang the GPU for good
template <bool SYS>
__device__ __forceinline__ void saa_wait_ge(const unsigned long long *flag, unsigned long long target, unsigned int *err)
{
    const long long t0 = clock64();
    while ((SYS ? ld_acquire_sys_u64(flag) : ld_acquire_gpu_u64(flag)) < target) {
        __nanosleep(100);
        if (clock64() - t0 > 60000000000ll) { *err = 1u; break; }
    }
}


__device__ __forceinline__ double ld_stream_f64(const double *p)
{
    double v;
    asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ int32_t ld_stream_s32(const int32_t *p)
{
    int32_t v;
    asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}

// linear_ramp, commons.py:7-11
__device__ __forceinline__ double saa_ramp(double t) { return (t <= 1.0) ? t : 1.0; }

// Row sums of csr_matvec (Dynamic_solver.py:12) for the three rows of one node:
//   s_A = 0.0;  s_A = s_A + (a_j * x[c_j])  over the row's stored entries in order  (A = 0, 1, 2).
// The loads of UNROLL blocks (9 values + 1 id + 3 gathered components each) are issued ahead of the dependent
// add chains (memory-level parallelism); the arithmetic order is untouched.
//   NC_X: the gathered vector is constant for the whole launch (per-step kernels) -> read-only path;
//         the persistent kernel re-reads vectors other blocks wrote before the last grid barrier and
//         must use ordinary (coherent after the barrier's fence) loads.
// Scheduling fence: every value listed must be in its register before any instruction after this point issues,
// and nothing after it may be hoisted above it.  Used to make ALL loads of a batch issue back to back (the
// compiler otherwise interleaves each dependent multiply-add right behind its own load, which stalls the warp on
// the first outstanding load and leaves only 3-4 requests in flight).
#define SAA_FENCE9(a) asm volatile("" : "+d"(a[0]), "+d"(a[1]), "+d"(a[2]), "+d"(a[3]), "+d"(a[4]), "+d"(a[5]), "+d"(a[6]), "+d"(a[7]), "+d"(a[8]))
#define SAA_FENCE3(x) asm volatile("" : "+d"(x[0]), "+d"(x[1]), "+d"(x[2]))

template <bool NC_X>
__device__ __forceinline__ void saa_gather3(const double *x, int32_t k, double (&xv)[3])
{
    const double *xp = x + 3 * (int64_t)k;
#pragma unroll
    for (int b = 0; b < 3; ++b) xv[b] = NC_X ? __ldg(xp + b) : xp[b];
}
// s_A = s_A + a[A][b]*x[b], b = 0,1,2: separately rounded multiply and add, ascending column order
__device__ __forceinline__ void saa_block_madd(const double (&a)[9], const double (&xv)[3], double (&s)[3])
{
#pragma unroll
    for (int A = 0; A < 3; ++A)
#pragma unroll
        for (int b = 0; b < 3; ++b) s[A] = __dadd_rn(s[A], __dmul_rn(a[3 * A + b], xv[b]));
}

// Value planes of one block: plane e is loaded iff bit e of the block's plane mask m is set (m is warp-uniform, so the
// predicate is too); otherwise a[e] = 0.0, the value every lane would have loaded from a full-plane layout.  v points
// at the block's first stored plane (of this lane); the stored planes follow each other in bit order.
__device__ __forceinline__ double ld_stream_f64_if(const double *p, unsigned pred)
{
    double v;
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %2, 0;\n\tmov.b64 %0, 0d0000000000000000;\n\t"
                 "@q ld.global.nc.L1::no_allocate.f64 %0, [%1];\n\t}"
                 : "=&d"(v) : "l"(p), "r"(pred));
    return v;
}
__device__ __forceinline__ void saa_load_block(const double *v, unsigned m, double (&a)[9])
{
#pragma unroll
    for (int e = 0; e < 9; ++e) a[e] = ld_stream_f64_if(v + 32 * __popc(m & ((1u << e) - 1u)), m & (1u << e));
}

template <int UNROLL, bool NC_X>
__device__ __forceinline__ void saa_node_dot_pipe(const SaaDev &P, int64_t slice, int lane, const double *x, double (&s)[3])
{
    static_assert(UNROLL == 2, "the software pipeline below is written for two blocks per batch");
    const int64_t beg = P.slice_ptr[slice];
    const int len = (int)((P.slice_ptr[slice + 1] - beg) >> 5);
    const double *v = P.val + P.val_ptr[slice] + lane;
    const int32_t *c = P.col + beg + lane;
    const uint16_t *mk = P.pmask + (beg >> 5);
    s[0] = 0.0; s[1] = 0.0; s[2] = 0.0;
    // column ids and plane masks run one batch ahead of the values, so that the gathers of a batch are issued together
    // with its value loads instead of after a first round trip
    int32_t k0 = 0, k1 = 0;
    unsigned m0 = 0, m1 = 0;
    if (len > 0) { k0 = ld_stream_s32(c); m0 = __ldg(mk); }
    if (len > 1) { k1 = ld_stream_s32(c + 32); m1 = __ldg(mk + 1); }
    int j = 0;
    for (; j + 2 <= len; j += 2) {
        double a0[9], a1[9], x0[3], x1[3];
        saa_load_block(v, m0, a0);
        v += 32 * __popc(m0);
        saa_load_block(v, m1, a1);
        v += 32 * __popc(m1);
        saa_gather3<NC_X>(x, k0, x0);
        saa_gather3<NC_X>(x, k1, x1);
        if (j + 2 < len) { k0 = ld_stream_s32(c + 32 * (j + 2)); m0 = __ldg(mk + j + 2); }
        if (j + 3 < len) { k1 = ld_stream_s32(c + 32 * (j + 3)); m1 = __ldg(mk + j + 3); }
        SAA_FENCE9(a0); SAA_FENCE9(a1); SAA_FENCE3(x0); SAA_FENCE3(x1);
        saa_block_madd(a0, x0, s);              // blocks in ascending column order: the order of the CSR row
        saa_block_madd(a1, x1, s);
    }
    if (j < len) {
        double a0[9], x0[3];
        saa_load_block(v, m0, a0);
        saa_gather3<NC_X>(x, k0, x0);
        saa_block_madd(a0, x0, s);
    }
}

// plain form: the compiler schedules the loads of UNROLL blocks against the dependent add chains
template <int UNROLL, bool NC_X>
__device__ __forceinline__ void saa_node_dot_simple(const SaaDev &P, int64_t slice, int lane, const double *x, double (&s)[3])
{
    const int64_t beg = P.slice_ptr[slice];
    const int len = (int)((P.slice_ptr[slice + 1] - beg) >> 5);
    const double *v = P.val + P.val_ptr[slice] + lane;
    const int32_t *c = P.col + beg + lane;
    const uint16_t *mk = P.pmask + (beg >> 5);
    s[0] = 0.0; s[1] = 0.0; s[2] = 0.0;
    int j = 0;
    for (; j + UNROLL <= len; j += UNROLL) {
        double a[UNROLL][9];
        int32_t k[UNROLL];
        unsigned m[UNROLL];
        double xv[UNROLL][3];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            k[u] = ld_stream_s32(c + 32 * (j + u));
            m[u] = __ldg(mk + j + u);
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            saa_load_block(v, m[u], a[u]);
            v += 32 * __popc(m[u]);
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const double *xp = x + 3 * (int64_t)k[u];
#pragma unroll
            for (int b = 0; b < 3; ++b) xv[u][b] = NC_X ? __ldg(xp + b) : xp[b];
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u)
#pragma unroll
            for (int A = 0; A < 3; ++A)
#pragma unroll
                for (int b = 0; b < 3; ++b) s[A] = __dadd_rn(s[A], __dmul_rn(a[u][3 * A + b], xv[u][b]));
    }
    for (; j < len; ++j) {
        const int32_t k = ld_stream_s32(c + 32 * j);
        const unsigned m = __ldg(mk + j);
        double a[9];
        saa_load_block(v, m, a);
        v += 32 * __popc(m);
        const double *xp = x + 3 * (int64_t)k;
        double xv[3];
#pragma unroll
        for (int b = 0; b < 3; ++b) xv[b] = NC_X ? __ldg(xp + b) : xp[b];
#pragma unroll
        for (int A = 0; A < 3; ++A)
#pragma unroll
            for (int b = 0; b < 3; ++b) s[A] = __dadd_rn(s[A], __dmul_rn(a[3 * A + b], xv[b]));
    }
}

// MODE 0: plain loop, 1: column ids prefetched one batch ahead (both give the same bits; which one is faster is a
// matter of the instruction schedule ptxas picks, see profiles/)
template <int MODE, bool NC_X>
__device__ __forceinline__ void saa_node_dot(const SaaDev &P, int64_t slice, int lane, const double *x, double (&s)[3])
{
    if (MODE == 0) saa_node_dot_simple<SAA_UNROLL, NC_X>(P, slice, lane, x, s);
    else saa_node_dot_pipe<SAA_UNROLL, NC_X>(P, slice, lane, x, s);
}

// Dynamic_solver.py:17 / :29 with Python's left-to-right association
__device__ __forceinline__ double saa_cd_update(const SaaDev &P, double Fi, double F, double M, double d0, double dn,
                                                double ramp)
{
    const double Fe = __dmul_rn(F, ramp);                                        // :13
    const double t1 = __dmul_rn(P.dt2, __dsub_rn(Fe, Fi));                       // dt**2*(F_ext - F_int)
    const double t2 = __dmul_rn(__dmul_rn(2.0, M), d0);                          // 2*l_M*d0
    const double t3 = __dmul_rn(M, dn);                                          // l_M*dn
    const double t4 = __dmul_rn(__dmul_rn(__dmul_rn(P.dt_half, M), P.alpha), dn);// dt/2*l_M*alpha*dn
    const double num = __dadd_rn(__dsub_rn(__dadd_rn(t1, t2), t3), t4);
    const double den = __dadd_rn(M, __dmul_rn(__dmul_rn(P.half_alpha, M), P.dt)); // l_M + 0.5*alpha*l_M*dt
    return __ddiv_rn(num, den);
}

__device__ __forceinline__ void saa_finish_row_m(const SaaDev &P, int64_t row, double Fi, double M, const double *d0, double *dn_d1,
                                                 double ramp)
{
    const double d1 = saa_cd_update(P, Fi, P.F[row], M, d0[row], dn_d1[row], ramp);
    const bool clamp = (P.dir_mask[row >> 5] >> (row & 31)) & 1u;
    dn_d1[row] = clamp ? 0.0 : d1;                                               // :20 / :32
}
__device__ __forceinline__ void saa_finish_row(const SaaDev &P, int64_t row, double Fi, const double *d0, double *dn_d1,
                                               double ramp)
{
    saa_finish_row_m(P, row, Fi, P.M[P.node_mass ? row / 3 : row], d0, dn_d1, ramp);
}
// the three rows of the node of (slice, lane);  ADD_ZERO: f_global = 0; f_global += f (Distributed_tools.py:84-86)
template <bool ADD_ZERO>
__device__ __forceinline__ void saa_finish_node(const SaaDev &P, int64_t slice, int lane, const double (&s)[3], const double *d0,
                                                double *dn_d1, double ramp)
{
    const int64_t node = slice * 32 + lane, row0 = 3 * node;
    double M[3];
    if (P.node_mass) {
        M[0] = M[1] = M[2] = P.M[node];
    } else {
#pragma unroll
        for (int A = 0; A < 3; ++A) M[A] = P.M[row0 + A];
    }
#pragma unroll
    for (int A = 0; A < 3; ++A) saa_finish_row_m(P, row0 + A, ADD_ZERO ? __dadd_rn(0.0, s[A]) : s[A], M[A], d0, dn_d1, ramp);
}

// ---------------------------------------------------------------------------------------------------
// K1 is the interior path of saa_k_step (below): fused force + update, one warp per slice of 32 nodes.  d1
// overwrites dn in place (row i only needs its own dn[i]).  The clock is read from device memory so that the
// launch can be replayed from a CUDA graph; block 0 writes tn + dt for the next step (Data_prepare.py:235).
// On the synchronised path every force passes through f_global = 0; f_global += f (Distributed_tools.py:84-86),
// i.e. F_int = 0.0 + s; a row sum that starts at +0.0 can never be -0.0, so 0.0 + s == s bit for bit and the
// same code serves the local path.

// K2: partial internal force of the shared rows, stored for the own sum and packed into the messages
// of every neighbour holding the node (fused halo pack).
//   PEER: the message entries are stored straight into the neighbours' receive areas over NVLink (mapped peer
//   memory, parity = sync_step & 1); the last block to finish publishes "message sync_step+1 has arrived" to
//   every neighbour with a system-scope release store.
template <bool PEER>
__global__ void __launch_bounds__(256) saa_k_boundary(SaaDev P, SaaHaloDev H, const double *__restrict__ d0, const SaaClock *clk_in)
{
    const int lane = threadIdx.x & 31;
    const int64_t slice = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    unsigned long long step = 0;
    if (PEER) step = clk_in->sync_step;
    if (slice < P.sh_slices) {
        double s[3];
        saa_node_dot<SAA_DOT_MODE, true>(P, slice, lane, d0, s);
#pragma unroll
        for (int A = 0; A < 3; ++A) {
            const int64_t row = 3 * (slice * 32 + lane) + A;
            H.xbuf[row] = s[A];
            for (int64_t k = H.dst_ptr[row]; k < H.dst_ptr[row + 1]; ++k) {
                if (PEER) {
                    const int nb = H.dst_nb[k];
                    H.peer_recv[nb][(int64_t)(step & 1ull) * H.peer_stride[nb] + H.dst_pos[k]] = s[A];
                } else {
                    H.sendbuf[H.dst_pos[k]] = s[A];
                }
            }
        }
    }
    if (PEER) {
        __threadfence_system();                      // this thread's peer stores are visible system-wide ...
        __syncthreads();                             // ... before thread 0 counts the block as done
        if (threadIdx.x == 0) {
            const unsigned int t = atomicAdd(H.done_ctr, 1u);
            if (t == gridDim.x - 1) {
                *H.done_ctr = 0u;                    // re-arm for the next step (next launch is stream-ordered)
                __threadfence_system();              // one release fence for all flags below
                for (int k = 0; k < H.n_nb; ++k) st_relaxed_sys_u64(H.peer_flag[k], step + 1ull);
            }
        }
    }
}

// K3: fused halo unpack + rank-ordered sum + update of the shared rows:
//   F_int = ((0.0 + f_r0) + f_r1) + ...   holders r0 < r1 < ... (Distributed_tools.py:84-86)
//   PEER: first wait (acquire, system scope) until every neighbour's message of this step has arrived.
template <bool PEER>
__global__ void __launch_bounds__(256) saa_k_shared_update(SaaDev P, SaaHaloDev H, const double *__restrict__ d0,
                                                           double *__restrict__ dn_d1, const SaaClock *clk_in)
{
    const double *recv = H.recv;
    if (PEER) {
        const unsigned long long step = clk_in->sync_step;
        if (threadIdx.x < H.n_nb) {
            saa_wait_ge<true>(H.flags + threadIdx.x, step + 1ull, H.err);
        }
        __syncthreads();
        recv += (int64_t)(step & 1ull) * H.recv_stride;
    }
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= H.sh_rows) return;
    double Fi = 0.0;
    for (int64_t k = H.src_ptr[row]; k < H.src_ptr[row + 1]; ++k) {
        const int32_t s = H.src_pos[k];
        // received entries were written by another GPU during this launch sequence: plain (coherent) loads
        const double v = (s < H.sh_rows) ? H.xbuf[s] : *((const volatile double *)(recv + (s - H.sh_rows)));
        Fi = __dadd_rn(Fi, v);
    }
    saa_finish_row(P, row, Fi, d0, dn_d1, saa_ramp(clk_in->tn));
}

// syn_cpus as a stand-alone operation (Distributed_tools.py:77-92) on a caller-provided force vector:
// pack the shared rows of f (internal order) into the neighbour messages ...
__global__ void saa_k_pack_forces(SaaHaloDev H, const double *__restrict__ f)
{
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= H.sh_rows) return;
    const double s = f[row];
    H.xbuf[row] = s;
    for (int64_t k = H.dst_ptr[row]; k < H.dst_ptr[row + 1]; ++k) H.sendbuf[H.dst_pos[k]] = s;
}
// ... and, after the exchange, f_global[dofs_local]: rank-ordered sum on shared rows, 0.0 + f elsewhere (:84-86)
__global__ void saa_k_sum_forces(int64_t n_rows, SaaHaloDev H, const double *__restrict__ f, double *__restrict__ out)
{
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n_rows) return;
    double Fi = 0.0;
    if (row < H.sh_rows) {
        for (int64_t k = H.src_ptr[row]; k < H.src_ptr[row + 1]; ++k) {
            const int32_t s = H.src_pos[k];
            Fi = __dadd_rn(Fi, (s < H.sh_rows) ? H.xbuf[s] : H.recv[s - H.sh_rows]);
        }
    } else {
        Fi = __dadd_rn(Fi, f[row]);
    }
    out[row] = Fi;
}

// THE step kernel.  Local steps and the interior phase of the staged transports run it with sh_slices = 0 and
// max_waiters = 0 (pure K1 over slices [slice_begin, n_slices)).  With the peer transport it is K1+K2+K3 in ONE
// launch per synchronised step; the grid is n_main slice blocks followed by n_tail = ceil(shared rows / 256) tail blocks:
//   * the blocks owning the boundary slices (internal order is boundary-first, so these are the lowest block
//     indices): partial forces -> own buffer and straight into the neighbours' receive areas; the warp that
//     completes the last boundary slice raises the neighbours' arrival flags (system scope) and the local "own
//     forces ready" flag;
//   * the bulk of the grid streams the interior slices, overlapping the NVLink traffic;
//   * the tail blocks do the rank-ordered sum and the update of the shared rows, in units of 256 rows claimed from a
//     counter.  The hardware dispatches blocks in index order, so they normally start while the last interior
//     blocks are still streaming, find every message already there and finish in their shadow.
// Correctness does NOT depend on that order: a tail block that finds a message missing may wait for it (bounded)
// only while fewer than `max_waiters` (< resident capacity of the GPU) tail blocks are waiting; otherwise it leaves,
// and the waiting ones drain every unit that is left once the messages have arrived.  So blocks that have not run
// yet — the boundary blocks in particular — always find a free slot, whatever the dispatch order.
// The counters exist twice; a launch uses the set selected by the parity of a fused-launch sequence number kept in
// device memory, and the last tail block to leave clears the other set and advances the number.
// Same arithmetic, same order as the three-kernel sequence — one launch gap and no pipeline drain per step.
//   count_sync: 1 on synchronised steps (advances the exchange counter), 0 on local ones.
#ifdef SAA_DEBUG_PEER          // timing experiments only (profiling builds): results are WRONG when H.dbg != 0
#define SAA_DBG(H, bit) ((H).dbg & (bit))
#else
#define SAA_DBG(H, bit) 0
#endif
template <int MODE, int MINB>
__global__ void __launch_bounds__(256, MINB) saa_k_step(SaaDev P, SaaHaloDev H, const double *__restrict__ d0,
                                                        double *__restrict__ dn_d1, const SaaClock *clk_in, SaaClock *clk_out,
                                                        int64_t slice_begin, unsigned int max_waiters, unsigned int count_sync)
{
    const unsigned long long step = clk_in->sync_step;
    const double tn = clk_in->tn;
    if (clk_out != nullptr && blockIdx.x == 0 && threadIdx.x == 0) {
        clk_out->tn = __dadd_rn(tn, P.dt);
        clk_out->sync_step = step + count_sync;
        clk_out->step_idx = clk_in->step_idx + 1ull;
    }
    const unsigned int n_units = (max_waiters != 0u) ? (unsigned int)((H.sh_rows + 255) >> 8) : 0u;
    const unsigned int n_main = gridDim.x - n_units;
    if (blockIdx.x < n_main) {
        const int lane = threadIdx.x & 31;
        const int64_t slice = slice_begin + (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
        if (slice >= P.n_slices) return;
        double s[3];
        saa_node_dot<MODE, true>(P, slice, lane, d0, s);
        if (slice < P.sh_slices && !SAA_DBG(H, 8)) {
#pragma unroll
            for (int A = 0; A < 3; ++A) {
                const int64_t row = 3 * (slice * 32 + lane) + A;
                H.xbuf[row] = s[A];
                for (int64_t k = H.dst_ptr[row]; k < H.dst_ptr[row + 1]; ++k) {
                    const int nb = H.dst_nb[k];
                    if (SAA_DBG(H, 2)) H.sendbuf[H.dst_pos[k] % 3] = s[A];
                    else H.peer_recv[nb][(int64_t)(step & 1ull) * H.peer_stride[nb] + H.dst_pos[k]] = s[A];
                }
            }
            if (!SAA_DBG(H, 2)) __threadfence_system();
            __syncwarp();
            if (lane == 0) {
                const unsigned int t = atomicAdd(H.done_ctr, 1u);
                if (t == (unsigned int)P.sh_slices - 1u) {
                    *H.done_ctr = 0u;
                    __threadfence_system();          // one release fence for all flags below
                    for (int k = 0; k < H.n_nb; ++k) st_relaxed_sys_u64(H.peer_flag[k], step + 1ull);
                    st_relaxed_sys_u64(H.own_ready, step + 1ull);
                }
            }
        } else {
            saa_finish_node<true>(P, slice, lane, s, d0, dn_d1, saa_ramp(tn));
        }
        return;
    }
    // ---- tail blocks: shared rows
    __shared__ unsigned int s_go, s_unit;
    const unsigned int seq = *((volatile const unsigned int *)(H.tail_ticket + 16));
    unsigned int *cnt = H.tail_ticket + 8u * (seq & 1u);   // [0] tail blocks that have left, [1] claimed units, [2] waiting blocks
    if (threadIdx.x == 0) {
        bool ready = ld_acquire_gpu_u64(H.own_ready) >= step + 1ull;
        for (int k = 0; k < H.n_nb; ++k) ready = ready && (ld_acquire_sys_u64(H.flags + k) >= step + 1ull);
        s_go = SAA_DBG(H, 4) ? 0u : (ready || SAA_DBG(H, 1)) ? 1u : (atomicAdd(cnt + 2, 1u) < max_waiters) ? 2u : 0u;
    }
    __syncthreads();
    if (s_go == 2u) {
        if (threadIdx.x < H.n_nb) saa_wait_ge<true>(H.flags + threadIdx.x, step + 1ull, H.err);
        if (threadIdx.x == 255) saa_wait_ge<false>(H.own_ready, step + 1ull, H.err);
        __syncthreads();
    }
    if (s_go != 0u) {
        const double *recv = H.recv + (int64_t)(step & 1ull) * H.recv_stride;
        const double ramp = saa_ramp(tn);
        for (;;) {
            if (threadIdx.x == 0) s_unit = atomicAdd(cnt + 1, 1u);
            __syncthreads();
            const unsigned int u = s_unit;
            if (u >= n_units) break;
            const int64_t row = (int64_t)u * 256 + threadIdx.x;
            if (row < H.sh_rows) {
                double Fi = 0.0;
                for (int64_t k = H.src_ptr[row]; k < H.src_ptr[row + 1]; ++k) {
                    const int32_t q = H.src_pos[k];
                    const double v = (q < H.sh_rows) ? __ldcg(H.xbuf + q) : __ldcg(recv + (q - H.sh_rows));   // L2: written during this launch
                    Fi = __dadd_rn(Fi, v);
                }
                saa_finish_row(P, row, Fi, d0, dn_d1, ramp);
            }
            __syncthreads();                          // s_unit is rewritten in the next round
        }
    }
    if (threadIdx.x == 0) {
        const unsigned int t = atomicAdd(cnt, 1u);
        if (t == n_units - 1u) {                      // last tail block of this launch: every tail block has read `seq`
            unsigned int *nxt = H.tail_ticket + 8u * ((seq & 1u) ^ 1u);
            nxt[0] = 0u; nxt[1] = 0u; nxt[2] = 0u;
            __threadfence();
            *((volatile unsigned int *)(H.tail_ticket + 16)) = seq + 1u;
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// Streaming variant of K1 (schedule variant 6): the matrix reaches the SM through cp.async (L2 -> shared memory,
// no registers, no L1), so the number of bytes in flight no longer depends on how ptxas schedules the loads.
// The grid is persistent (one CTA per SM); every warp owns a CONTIGUOUS range of slices holding an equal share
// of the block-lanes, i.e. one contiguous stream of the value / id arrays, which it pulls through a ring of
// STAGES buffers of two block-rows (2 x (2304 B values + 128 B ids)) each.  The d0 gathers of a stage are issued
// one stage ahead.  Same arithmetic in the same order as saa_node_dot / saa_finish_node — same bits.
// It addresses val by block-row arithmetic, so it needs the full-plane layout (all nine planes of every block stored);
// finalisation builds that layout when this variant is selected.
#define SAA_STREAM_STAGE_BYTES(BR) ((BR) * (2304 + 128))
__device__ __forceinline__ void saa_cp_async16(void *smem_dst, const void *gmem_src)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}
template <int N>
__device__ __forceinline__ void saa_cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int STAGES, int WARPS, int BR>
__global__ void __launch_bounds__(32 * WARPS, 1) saa_k_step_stream(SaaDev P, const double *__restrict__ d0, double *__restrict__ dn_d1,
                                                                const SaaClock *clk_in, SaaClock *clk_out, int64_t slice_begin,
                                                                unsigned int count_sync)
{
    extern __shared__ __align__(16) unsigned char saa_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const double tn = clk_in->tn;
    if (clk_out != nullptr && blockIdx.x == 0 && threadIdx.x == 0) {
        clk_out->tn = __dadd_rn(tn, P.dt);
        clk_out->sync_step = clk_in->sync_step + count_sync;
        clk_out->step_idx = clk_in->step_idx + 1ull;
    }
    const double ramp = saa_ramp(tn);
    // ---- this warp's contiguous range of slices: equal shares of the block-rows (a block-row = 32 block-lanes)
    const int64_t gw = (int64_t)blockIdx.x * WARPS + warp, GW = (int64_t)gridDim.x * WARPS;
    const int64_t base = P.slice_ptr[slice_begin] >> 5, total = (P.slice_ptr[P.n_slices] >> 5) - base;
    auto first_slice_at = [&](int64_t brow) {          // first slice s >= slice_begin with slice_ptr[s]/32 >= brow
        int64_t lo = slice_begin, hi = P.n_slices;
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if ((P.slice_ptr[mid] >> 5) < brow) lo = mid + 1; else hi = mid;
        }
        return lo;
    };
    // slices are split where their first block-row crosses the share boundary; zero-length slices go with their successor's owner
    int64_t sa = (gw == 0) ? slice_begin : first_slice_at(base + (total * gw + GW - 1) / GW);
    int64_t sb = (gw == GW - 1) ? P.n_slices : first_slice_at(base + (total * (gw + 1) + GW - 1) / GW);
    if (gw != 0) { while (sa > slice_begin && P.slice_ptr[sa - 1] == P.slice_ptr[sa]) --sa; }       // leading empty slices belong here ...
    if (gw != GW - 1) { while (sb > sa && sb > slice_begin && P.slice_ptr[sb - 1] == P.slice_ptr[sb]) --sb; }   // ... so trailing ones do not
    if (sa >= sb) return;
    const int64_t br0 = P.slice_ptr[sa] >> 5, br1 = P.slice_ptr[sb] >> 5;
    const int64_t n_stage = (br1 - br0 + BR - 1) / BR;
    constexpr int SB = SAA_STREAM_STAGE_BYTES(BR);
    unsigned char *ring = saa_smem + (size_t)warp * STAGES * SB;

    auto issue = [&](int64_t k) {                      // stage k -> buffer k % STAGES (an empty group past the end)
        if (k < n_stage) {
            const int64_t br = br0 + BR * k;
            const int nbr = (int)((br1 - br) < BR ? (br1 - br) : BR);
            unsigned char *buf = ring + (size_t)(k % STAGES) * SB;
            const unsigned char *gv = (const unsigned char *)(P.val + 288 * br);       // 9 planes x 32 lanes per block-row
            const unsigned char *gc = (const unsigned char *)(P.col + 32 * br);
            for (int ch = lane; ch < 144 * nbr; ch += 32) saa_cp_async16(buf + 16 * ch, gv + 16 * ch);
            for (int ch = lane; ch < 8 * nbr; ch += 32) saa_cp_async16(buf + 2304 * BR + 16 * ch, gc + 16 * ch);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto gather = [&](int64_t k, double (&x)[BR][3]) {  // d0 components of the column nodes of stage k (already in shared memory)
        const unsigned char *buf = ring + (size_t)(k % STAGES) * SB;
        const int32_t *sc = (const int32_t *)(buf + 2304 * BR);
        const int64_t br = br0 + BR * k;
#pragma unroll
        for (int j = 0; j < BR; ++j)
            if (br + j < br1) {
                const double *xp = d0 + 3 * (int64_t)sc[32 * j + lane];
#pragma unroll
                for (int b = 0; b < 3; ++b) x[j][b] = __ldg(xp + b);
            }
    };

#pragma unroll
    for (int k = 0; k < STAGES - 1; ++k) issue(k);
    saa_cp_async_wait<STAGES - 2>();                   // stage 0 has landed
    __syncwarp();
    double xc[BR][3], xn[BR][3];
    gather(0, xc);
    int64_t cs = sa;                                   // current slice and the block-rows it still expects
    int64_t rem = (P.slice_ptr[cs + 1] - P.slice_ptr[cs]) >> 5;
    double s[3] = {0.0, 0.0, 0.0};
    auto close_finished_slices = [&]() {               // finish every slice whose rows are complete (also empty ones)
        while (rem == 0 && cs < sb) {
            saa_finish_node<true>(P, cs, lane, s, d0, dn_d1, ramp);
            s[0] = 0.0; s[1] = 0.0; s[2] = 0.0;
            ++cs;
            if (cs < sb) rem = (P.slice_ptr[cs + 1] - P.slice_ptr[cs]) >> 5;
        }
    };
    close_finished_slices();
    for (int64_t k = 0; k < n_stage; ++k) {
        issue(k + STAGES - 1);                         // refills the buffer consumed in the previous iteration
        saa_cp_async_wait<STAGES - 2>();               // stages <= k + 1 have landed
        __syncwarp();
        if (k + 1 < n_stage) gather(k + 1, xn);
        const unsigned char *buf = ring + (size_t)(k % STAGES) * SB;
        const double *sv = (const double *)buf;
        const int64_t br = br0 + BR * k;
#pragma unroll
        for (int j = 0; j < BR; ++j)
            if (br + j < br1) {
                double a[9];
#pragma unroll
                for (int e = 0; e < 9; ++e) a[e] = sv[(9 * j + e) * 32 + lane];
                saa_block_madd(a, xc[j], s);
                --rem;
                close_finished_slices();
            }
#pragma unroll
        for (int j = 0; j < BR; ++j)
#pragma unroll
            for (int b = 0; b < 3; ++b) xc[j][b] = xn[j][b];
        __syncwarp();                                  // every lane is done with this buffer before it is refilled
    }
    saa_cp_async_wait<0>();
}

// Persistent variant of K1 (local mode): one cooperative launch runs n_steps time steps; u stays in HBM/L2,
// the two displacement buffers swap roles after each grid-wide barrier.  tn advances in registers with the
// same sequence of additions as the host loop (Data_prepare.py:235).
__global__ void __launch_bounds__(256) saa_k_persistent(SaaDev P, double *bufA, double *bufB, SaaClock *clk_io,
                                                        int64_t n_steps)
{
    cg::grid_group grid = cg::this_grid();
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    double tn = clk_io->tn;
    double *d0 = bufA, *dn = bufB;
    for (int64_t step = 0; step < n_steps; ++step) {
        const double ramp = saa_ramp(tn);
        for (int64_t slice = warp0; slice < P.n_slices; slice += nwarps) {
            double s[3];
            saa_node_dot<SAA_DOT_MODE, false>(P, slice, lane, d0, s);
            saa_finish_node<false>(P, slice, lane, s, d0, dn, ramp);
        }
        tn = __dadd_rn(tn, P.dt);
        double *t = d0; d0 = dn; dn = t;
        grid.sync();
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        clk_io->tn = tn;
        clk_io->step_idx += (unsigned long long)n_steps;
    }
}

// Persistent SYNCHRONISED loop (peer transport): one cooperative launch runs n_steps synchronised time steps — for
// shards so small that a step is a few microseconds and the per-step launch is what limits it.  Every block is resident
// (cooperative launch), so waiting on a neighbour's arrival flag cannot starve anybody.  Per step:
//   * grid-stride over the slices; the boundary slices come first (lowest warp ids, first round): partial forces -> own
//     buffer and the neighbours' receive areas, last boundary warp raises the flags (exactly as in saa_k_step);
//   * interior slices: fused force + update;
//   * shared rows in units of 256, grid-strided over the blocks, after the flags have arrived: rank-ordered sum + update;
//   * one grid-wide barrier; buffers swap roles; tn and the exchange number advance in registers.
// Same arithmetic and order as the per-step kernels — same bits.
__global__ void __launch_bounds__(256) saa_k_persistent_sync(SaaDev P, SaaHaloDev H, double *bufA, double *bufB, SaaClock *clk_io,
                                                             int64_t n_steps)
{
    cg::grid_group grid = cg::this_grid();
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const int64_t n_units = (H.sh_rows + 255) >> 8;
    double tn = clk_io->tn;
    const unsigned long long sync0 = clk_io->sync_step;
    double *d0 = bufA, *dn = bufB;
    for (int64_t it = 0; it < n_steps; ++it) {
        const unsigned long long step = sync0 + (unsigned long long)it;
        const double ramp = saa_ramp(tn);
        for (int64_t slice = warp0; slice < P.n_slices; slice += nwarps) {
            double s[3];
            saa_node_dot<SAA_DOT_MODE, false>(P, slice, lane, d0, s);
            if (slice < P.sh_slices) {
#pragma unroll
                for (int A = 0; A < 3; ++A) {
                    const int64_t row = 3 * (slice * 32 + lane) + A;
                    H.xbuf[row] = s[A];
                    for (int64_t k = H.dst_ptr[row]; k < H.dst_ptr[row + 1]; ++k) {
                        const int nb = H.dst_nb[k];
                        H.peer_recv[nb][(int64_t)(step & 1ull) * H.peer_stride[nb] + H.dst_pos[k]] = s[A];
                    }
                }
                __threadfence_system();
                __syncwarp();
                if (lane == 0) {
                    const unsigned int t = atomicAdd(H.done_ctr, 1u);
                    if (t == (unsigned int)P.sh_slices - 1u) {
                        *H.done_ctr = 0u;
                        __threadfence_system();      // one release fence for all flags below
                        for (int k = 0; k < H.n_nb; ++k) st_relaxed_sys_u64(H.peer_flag[k], step + 1ull);
                        st_relaxed_sys_u64(H.own_ready, step + 1ull);
                    }
                }
            } else {
                saa_finish_node<true>(P, slice, lane, s, d0, dn, ramp);
            }
        }
        if ((int64_t)blockIdx.x < n_units) {                    // this block owns shared-row units of this step
            if (threadIdx.x < H.n_nb) saa_wait_ge<true>(H.flags + threadIdx.x, step + 1ull, H.err);
            if (threadIdx.x == 255) saa_wait_ge<false>(H.own_ready, step + 1ull, H.err);
            __syncthreads();
            const double *recv = H.recv + (int64_t)(step & 1ull) * H.recv_stride;
            for (int64_t u = blockIdx.x; u < n_units; u += gridDim.x) {
                const int64_t row = u * 256 + threadIdx.x;
                if (row < H.sh_rows) {
                    double Fi = 0.0;
                    for (int64_t k = H.src_ptr[row]; k < H.src_ptr[row + 1]; ++k) {
                        const int32_t q = H.src_pos[k];
                        const double v = (q < H.sh_rows) ? __ldcg(H.xbuf + q) : __ldcg(recv + (q - H.sh_rows));
                        Fi = __dadd_rn(Fi, v);
                    }
                    saa_finish_row(P, row, Fi, d0, dn, ramp);
                }
            }
        }
        tn = __dadd_rn(tn, P.dt);
        double *t = d0; d0 = dn; dn = t;
        grid.sync();
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        clk_io->tn = tn;
        clk_io->sync_step = sync0 + (unsigned long long)n_steps;
        clk_io->step_idx += (unsigned long long)n_steps;
    }
}

// ---- small data-movement kernels -----------------------------------------------------------------------
// lumped mass per node instead of per DOF when the three DOFs of every node carry identical bits
__global__ void saa_k_mass_check(int64_t n_nodes, const double *__restrict__ M, int *__restrict__ differs)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_nodes) return;
    const long long a = __double_as_longlong(M[3 * i]), b = __double_as_longlong(M[3 * i + 1]), c = __double_as_longlong(M[3 * i + 2]);
    if (a != b || a != c) *differs = 1;
}
__global__ void saa_k_mass_compact(int64_t n_nodes, const double *__restrict__ M, double *__restrict__ Mn)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_nodes) Mn[i] = M[3 * i];
}
// external (reference local DOF order) <-> internal (boundary-first, sigma-sorted) order
__global__ void saa_k_scatter_to_internal(int64_t n_ext, const int32_t *__restrict__ iperm, const double *__restrict__ src_ext,
                                          double *__restrict__ dst_int)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_ext) dst_int[iperm[i]] = src_ext[i];
}
__global__ void saa_k_gather_to_external(int64_t n_ext, const int32_t *__restrict__ iperm, const double *__restrict__ src_int,
                                         double *__restrict__ dst_ext)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_ext) dst_ext[i] = src_int[iperm[i]];
}
// Hooks after a step whose input clock was *clk_old (its step_idx is the loop index i of this step):
//   Online_predictor.py:298   d1[loc_dof_shared] = d_shared[i - first predicted step]
__global__ void saa_k_hook_scatter(int64_t n, const int32_t *__restrict__ rows, const SaaHookDev *__restrict__ hk,
                                   const SaaClock *__restrict__ clk_old, double *__restrict__ d1)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const long long r = (long long)clk_old->step_idx - hk->pred_base_step;
    if (i < n && r >= 0 && r < hk->pred_rows) d1[rows[i]] = hk->pred_table[r * n + i];
}
//   Data_prepare.py:238-240 / Online_predictor.py:260,301   d1_save[:, i / save_every] = d1  (device ring)
__global__ void saa_k_hook_gather(int64_t n, const int32_t *__restrict__ rows, const SaaHookDev *__restrict__ hk,
                                  const SaaClock *__restrict__ clk_old, const double *__restrict__ d1, double *__restrict__ hist)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const long long s = (long long)clk_old->step_idx;
    if (i >= n || (s % hk->hist_every) != 0) return;
    const long long slot = (s / hk->hist_every - hk->hist_first) % hk->hist_cap;
    hist[slot * n + i] = d1[rows[i]];
}
