// saa_device_setup.cuh — set-up at scale, entirely on the GPU (included at the end of saa_fem.cu):
//   * saa_assemble_*_dev : sparse stiffness / lumped mass / load assembly (kernels in saa_assembly.cuh)
//   * saa_plan_create_dev + finalize_device : plan from a device-resident CSR — row ordering (boundary first,
//     sigma-sorted), sliced-ELL conversion and all per-row tables are built by kernels / thrust, so that a
//     100 M-DOF partition never visits host memory.  Produces exactly the layout of the host path
//     (saa_plan_finalize) for the same matrix.
#pragma once
#include "saa_assembly.cuh"

#include <thrust/binary_search.h>
#include <thrust/copy.h>
#include <thrust/device_ptr.h>
#include <thrust/execution_policy.h>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/scan.h>
#include <thrust/sequence.h>
#include <thrust/sort.h>


// ---- kernels of the device finalize (node-block sliced ELL, same layout as the host path) ---------------------
// three-way merge over the (sorted) rows 3e, 3e+1, 3e+2 of node e: visits the distinct column nodes ascending
struct SaaRowTriple {
    int64_t q[3], qe[3];
    __device__ SaaRowTriple(const int64_t *indptr, int64_t e)
    {
        for (int A = 0; A < 3; ++A) { q[A] = indptr[3 * e + A]; qe[A] = indptr[3 * e + A + 1]; }
    }
    __device__ int32_t next_col_node(const int32_t *indices) const
    {
        int32_t cn = INT32_MAX;
        for (int A = 0; A < 3; ++A)
            if (q[A] < qe[A]) cn = min(cn, indices[q[A]] / 3);
        return cn;
    }
};
// the checks saa_plan_create / saa_plan_finalize make on a host CSR, one thread per row; sets bits of *bad:
//   1 indptr[0] != 0, 2 indptr decreases, 4 a column index outside [0, n_rows), 8 columns of a row not strictly increasing.
// A row reads indices only inside [0, nnz), so a malformed indptr cannot make the check itself read out of bounds.
#define SAA_CSR_BAD_START 1u
#define SAA_CSR_BAD_INDPTR 2u
#define SAA_CSR_BAD_COLUMN 4u
#define SAA_CSR_BAD_ORDER 8u
__global__ void saa_k_fin_check_csr(int64_t n_rows, int64_t nnz, const int64_t *__restrict__ indptr,
                                    const int32_t *__restrict__ indices, unsigned int *__restrict__ bad)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    const int64_t a = indptr[i], b = indptr[i + 1];
    unsigned int f = 0u;
    if (i == 0 && a != 0) f |= SAA_CSR_BAD_START;
    if (b < a) f |= SAA_CSR_BAD_INDPTR;
    if (a >= 0 && a <= b && b <= nnz)
        for (int64_t k = a; k < b; ++k) {
            const int32_t c = indices[k];
            if (c < 0 || c >= n_rows) f |= SAA_CSR_BAD_COLUMN;
            if (k > a && c <= indices[k - 1]) f |= SAA_CSR_BAD_ORDER;
        }
    if (f) atomicOr(bad, f);
}
__global__ void saa_k_fin_nblk(int64_t n_nodes, const int64_t *__restrict__ indptr, const int32_t *__restrict__ indices, int32_t *__restrict__ nblk)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_nodes) return;
    SaaRowTriple t(indptr, e);
    int32_t cnt = 0;
    for (;;) {
        const int32_t cn = t.next_col_node(indices);
        if (cn == INT32_MAX) break;
        for (int A = 0; A < 3; ++A)
            while (t.q[A] < t.qe[A] && indices[t.q[A]] / 3 == cn) ++t.q[A];
        ++cnt;
    }
    nblk[e] = cnt;
}
__global__ void saa_k_fin_flag(int64_t m, const int32_t *__restrict__ nodes, uint8_t *__restrict__ flag)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < m) flag[nodes[i]] = 1;
}
// key of the sigma sort: (window of SIGMA consecutive positions, decreasing block count)
__global__ void saa_k_fin_keys(int64_t m, const int32_t *__restrict__ nodes, const int32_t *__restrict__ nblk, uint64_t *__restrict__ key)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < m) key[i] = ((uint64_t)(i / SAA_SIGMA) << 32) | (uint32_t)(0x7fffffff - nblk[nodes[i]]);
}
// permn: internal node -> external node; iperm: external row -> internal row
__global__ void saa_k_fin_perm(int64_t m, const int32_t *__restrict__ nodes, int64_t offset, int32_t *__restrict__ permn, int32_t *__restrict__ iperm)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < m) {
        const int32_t e = nodes[i];
        permn[offset + i] = e;
        for (int c = 0; c < 3; ++c) iperm[3 * (int64_t)e + c] = (int32_t)(3 * (offset + i) + c);
    }
}
__global__ void saa_k_fin_slice_len(int64_t n_slices, const int32_t *__restrict__ permn, const int32_t *__restrict__ nblk, int64_t *__restrict__ cnt)
{
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_slices) return;
    int32_t mx = 0;
    for (int l = 0; l < 32; ++l) {
        const int32_t e = permn[s * 32 + l];
        if (e >= 0) mx = max(mx, nblk[e]);
    }
    cnt[s] = 32 * (int64_t)mx;
}
// one warp per slice: stored planes of every block-row = the union of the stored patterns of the 32 lanes (the pattern,
// not the value bits, so that an explicitly stored 0.0 is kept; full: all nine planes), and the doubles the slice
// takes in val
__global__ void saa_k_fin_pmask(int64_t n_slices, const int64_t *__restrict__ slice_ptr, const int32_t *__restrict__ permn,
                                const int64_t *__restrict__ indptr, const int32_t *__restrict__ indices, int full,
                                uint16_t *__restrict__ pmask, int64_t *__restrict__ slice_vals)
{
    const int lane = threadIdx.x & 31;
    const int64_t s = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (s >= n_slices) return;
    const int64_t beg = slice_ptr[s];
    const int L = (int)((slice_ptr[s + 1] - beg) >> 5);
    const int32_t e = permn[s * 32 + lane];
    SaaRowTriple t(indptr, e >= 0 ? e : 0);
    int64_t planes = 0;
    for (int j = 0; j < L; ++j) {
        unsigned bits = 0;
        if (e >= 0) {
            const int32_t cn = t.next_col_node(indices);
            if (cn != INT32_MAX)
                for (int A = 0; A < 3; ++A)
                    while (t.q[A] < t.qe[A] && indices[t.q[A]] / 3 == cn) {
                        bits |= 1u << (3 * A + indices[t.q[A]] % 3);
                        ++t.q[A];
                    }
        }
        bits = full ? 0x1FFu : __reduce_or_sync(0xffffffffu, bits);
        if (lane == 0) pmask[(beg >> 5) + j] = (uint16_t)bits;
        planes += __popc(bits);
    }
    if (lane == 0) slice_vals[s] = 32 * planes;
}
// one warp per slice: every lane writes the stored planes of its blocks (stored order of each row kept), then pads with
// blocks 0.0 * d0[own node]
__global__ void saa_k_fin_fill(int64_t n_slices, const int64_t *__restrict__ slice_ptr, const int64_t *__restrict__ val_ptr,
                               const uint16_t *__restrict__ pmask, const int32_t *__restrict__ permn,
                               const int32_t *__restrict__ iperm, const int64_t *__restrict__ indptr,
                               const int32_t *__restrict__ indices, const double *__restrict__ data, double *__restrict__ val,
                               int32_t *__restrict__ col)
{
    const int lane = threadIdx.x & 31;
    const int64_t s = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (s >= n_slices) return;
    const int64_t beg = slice_ptr[s];
    const int L = (int)((slice_ptr[s + 1] - beg) >> 5);
    double *vs = val + val_ptr[s] + lane;
    const uint16_t *ms = pmask + (beg >> 5);
    int32_t *cs = col + beg + lane;
    const int64_t inode = s * 32 + lane;
    const int32_t e = permn[inode];
    int64_t off = 0;                                   // planes stored for the blocks before j
    auto store = [&](int j, const double (&a)[9]) {
        const unsigned m = ms[j];
        for (int k = 0; k < 9; ++k)
            if (m & (1u << k)) vs[32 * (off + __popc(m & ((1u << k) - 1u)))] = a[k];
        off += __popc(m);
    };
    int j = 0;
    if (e >= 0) {
        SaaRowTriple t(indptr, e);
        for (;; ++j) {
            const int32_t cn = t.next_col_node(indices);
            if (cn == INT32_MAX) break;
            double a[9];
            for (int k = 0; k < 9; ++k) a[k] = 0.0;
            for (int A = 0; A < 3; ++A)
                while (t.q[A] < t.qe[A] && indices[t.q[A]] / 3 == cn) {
                    a[3 * A + indices[t.q[A]] % 3] = data[t.q[A]];
                    ++t.q[A];
                }
            store(j, a);
            cs[32 * (int64_t)j] = iperm[3 * (int64_t)cn] / 3;
        }
    }
    const double z[9] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    for (; j < L; ++j) {
        store(j, z);
        cs[32 * (int64_t)j] = (int32_t)inode;
    }
}
__global__ void saa_k_fin_vectors(int64_t n_rows, const int32_t *__restrict__ permn, const double *__restrict__ M_ext,
                                  const double *__restrict__ F_ext, double *__restrict__ M, double *__restrict__ F)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    const int32_t e = permn[i / 3];
    const int64_t r = 3 * (int64_t)e + (i % 3);
    M[i] = (e >= 0) ? M_ext[r] : 1.0;
    F[i] = (e >= 0) ? F_ext[r] : 0.0;
}
__global__ void saa_k_fin_dirichlet(int64_t m, const int64_t *__restrict__ dofs, const int32_t *__restrict__ iperm, uint32_t *__restrict__ mask)
{
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= m) return;
    const int32_t i = iperm[dofs[k]];
    atomicOr(mask + (i >> 5), 1u << (i & 31));       // bit set: commutative, result independent of order
}
struct SaaIsZeroFlag {
    const uint8_t *flag;
    __host__ __device__ bool operator()(int32_t i) const { return flag[i] == 0; }
};

extern "C" int saa_plan_create_dev(saa_plan **out, int device, int64_t n_dof, const int64_t *indptr_dev,
                                   const int32_t *indices_dev, const double *data_dev, const double *F_dev,
                                   const double *lM_dev, const int64_t *dirichlet, int64_t n_dirichlet, double dt,
                                   double dt2, double dt_half, double half_alpha, double alpha)
{
    if (!out || n_dof <= 0 || !indptr_dev || !indices_dev || !data_dev || !F_dev || !lM_dev)
        return fail("saa_plan_create_dev: null or empty argument");
    if (n_dof % 3 != 0) return fail("saa_plan_create_dev: n_dof=%lld is not a multiple of 3", (long long)n_dof);
    if (n_dof >= (int64_t)INT32_MAX - 64) return fail("saa_plan_create_dev: more than 2^31 rows per partition not supported");
    if (n_dirichlet > 0 && !dirichlet) return fail("saa_plan_create_dev: dirichlet is null");
    if (saa_device_count() <= device) return fail("saa_plan_create_dev: CUDA device %d not available (no CPU fallback)", device);
    for (int64_t k = 0; k < n_dirichlet; ++k)
        if (dirichlet[k] < 0 || dirichlet[k] >= n_dof) return fail("saa_plan_create_dev: Dirichlet DOF out of range");
    saa_plan *p = new saa_plan();
    p->device = device;
    p->n_dof = n_dof;
    p->dev_input = true;
    p->in_indptr = indptr_dev; p->in_indices = indices_dev; p->in_data = data_dev; p->in_F = F_dev; p->in_M = lM_dev;
    p->dirichlet.assign(dirichlet, dirichlet + n_dirichlet);
    p->dt = dt; p->dt2 = dt2; p->dt_half = dt_half; p->half_alpha = half_alpha; p->alpha = alpha;
    *out = p;
    return 0;
}

static int finalize_device(saa_plan *p)
{
    CK(cudaSetDevice(p->device));
    const int64_t n = p->n_dof, nn = n / 3;
    const int64_t n_sh = (int64_t)p->shared_pos.size();
    CK(cudaMemcpy(&p->nnz, p->in_indptr + n, sizeof(int64_t), cudaMemcpyDeviceToHost));
    auto pad32 = [](int64_t v) { return (v + 31) / 32 * 32; };

    // 0. the CSR must be what the host path accepts: every kernel below indexes by its column ids
    {
        DevBuf b_bad;
        if (b_bad.alloc(sizeof(unsigned int))) return -1;
        CK(cudaMemset(b_bad.p, 0, sizeof(unsigned int)));
        saa_k_fin_check_csr<<<nblk(n, 256), 256>>>(n, p->nnz, p->in_indptr, p->in_indices, b_bad.as<unsigned int>());
        CK(cudaGetLastError());
        unsigned int bad = 0;
        CK(cudaMemcpy(&bad, b_bad.p, sizeof(unsigned int), cudaMemcpyDeviceToHost));
        if (bad & SAA_CSR_BAD_START) return fail("saa_plan_finalize: indptr[0] is not 0");
        if (bad & SAA_CSR_BAD_INDPTR) return fail("saa_plan_finalize: indptr not monotone");
        if (bad & SAA_CSR_BAD_COLUMN) return fail("saa_plan_finalize: column index out of range");
        if (bad & SAA_CSR_BAD_ORDER) return fail("saa_plan_finalize: LocalK must have sorted, duplicate-free column indices");
    }

    // 1. block counts, shared flags, the two regions in their starting order
    DevBuf b_nblk, b_flag, b_sh, b_in, b_key;
    if (b_nblk.alloc(nn * sizeof(int32_t)) || b_flag.alloc(nn) || b_in.alloc(nn * sizeof(int32_t))) return -1;
    int32_t *nblk_d = b_nblk.as<int32_t>();
    uint8_t *flag = b_flag.as<uint8_t>();
    saa_k_fin_nblk<<<nblk(nn, 128), 128>>>(nn, p->in_indptr, p->in_indices, nblk_d);
    CK(cudaMemset(flag, 0, nn));
    std::vector<int32_t> sh_h(p->shared_pos.begin(), p->shared_pos.end());
    {   // duplicates would break the permutation
        std::vector<int32_t> chk(sh_h);
        std::sort(chk.begin(), chk.end());
        if (std::adjacent_find(chk.begin(), chk.end()) != chk.end()) return fail("saa_plan_finalize: duplicate shared node");
    }
    if (b_sh.alloc(std::max<int64_t>(n_sh, 1) * sizeof(int32_t))) return -1;
    int32_t *sh_nodes = b_sh.as<int32_t>();
    if (n_sh) {
        CK(cudaMemcpy(sh_nodes, sh_h.data(), n_sh * sizeof(int32_t), cudaMemcpyHostToDevice));
        saa_k_fin_flag<<<nblk(n_sh, 256), 256>>>(n_sh, sh_nodes, flag);
    }
    int32_t *in_nodes = b_in.as<int32_t>();
    int64_t n_in = 0;
    if (p->node_order.empty()) {
        n_in = thrust::copy_if(thrust::device, thrust::counting_iterator<int32_t>(0), thrust::counting_iterator<int32_t>((int32_t)nn),
                               in_nodes, SaaIsZeroFlag{flag}) - in_nodes;
    } else {                                           // caller's locality-preserving order, interface nodes filtered out
        DevBuf b_ord;
        if (b_ord.alloc(nn * sizeof(int32_t))) return -1;
        CK(cudaMemcpy(b_ord.p, p->node_order.data(), nn * sizeof(int32_t), cudaMemcpyHostToDevice));
        n_in = thrust::copy_if(thrust::device, b_ord.as<int32_t>(), b_ord.as<int32_t>() + nn, in_nodes, SaaIsZeroFlag{flag}) - in_nodes;
    }
    if (n_in != nn - n_sh) return fail("saa_plan_finalize: internal error (interior nodes %lld != %lld)", (long long)n_in, (long long)(nn - n_sh));

    // 2. sigma sort of both regions (stable: ties keep their order, like the host path)
    if (b_key.alloc(std::max<int64_t>(std::max(n_in, n_sh), 1) * sizeof(uint64_t))) return -1;
    uint64_t *key = b_key.as<uint64_t>();
    if (n_sh) {
        saa_k_fin_keys<<<nblk(n_sh, 256), 256>>>(n_sh, sh_nodes, nblk_d, key);
        thrust::stable_sort_by_key(thrust::device, key, key + n_sh, sh_nodes);
    }
    if (n_in) {
        saa_k_fin_keys<<<nblk(n_in, 256), 256>>>(n_in, in_nodes, nblk_d, key);
        thrust::stable_sort_by_key(thrust::device, key, key + n_in, in_nodes);
    }
    cudaFree(b_key.p); b_key.p = nullptr;

    // 3. node permutation (internal -> external, -1 = padding) and the row map external -> internal
    const int64_t sh_padn = pad32(n_sh), in_padn = pad32(n_in);
    const int64_t n_slots = sh_padn + in_padn;
    p->n_rows = 3 * n_slots;
    p->n_slices = n_slots / 32;
    p->sh_slices = sh_padn / 32;
    if (p->n_rows >= (int64_t)INT32_MAX) return fail("saa_plan_finalize: more than 2^31 rows per partition not supported");
    DevBuf b_perm, b_cnt;
    if (b_perm.alloc(n_slots * sizeof(int32_t))) return -1;
    int32_t *permn = b_perm.as<int32_t>();
    CK(cudaMemset(permn, 0xff, n_slots * sizeof(int32_t)));
    CK(cudaMalloc((void **)&p->d_iperm, n * sizeof(int32_t)));
    if (n_sh) saa_k_fin_perm<<<nblk(n_sh, 256), 256>>>(n_sh, sh_nodes, 0, permn, p->d_iperm);
    if (n_in) saa_k_fin_perm<<<nblk(n_in, 256), 256>>>(n_in, in_nodes, sh_padn, permn, p->d_iperm);
    cudaFree(b_in.p); b_in.p = nullptr;

    // 4. slice offsets (block-lanes)
    if (b_cnt.alloc((p->n_slices + 1) * sizeof(int64_t))) return -1;
    int64_t *cnt = b_cnt.as<int64_t>();
    CK(cudaMemset(cnt, 0, (p->n_slices + 1) * sizeof(int64_t)));
    saa_k_fin_slice_len<<<nblk(p->n_slices, 256), 256>>>(p->n_slices, permn, nblk_d, cnt);
    CK(cudaMalloc((void **)&p->d_slice_ptr, (p->n_slices + 1) * sizeof(int64_t)));
    thrust::exclusive_scan(thrust::device, cnt, cnt + p->n_slices + 1, p->d_slice_ptr);
    int64_t lanes = 0;
    CK(cudaMemcpy(&lanes, p->d_slice_ptr + p->n_slices, sizeof(int64_t), cudaMemcpyDeviceToHost));
    p->padded_entries = 9 * lanes;

    // 5. plane masks and value offsets; matrix in plane-masked node-block sliced-ELL order (val allocated at its exact
    //    size), vectors, Dirichlet mask
    CK(cudaMalloc((void **)&p->d_pmask, std::max<int64_t>(lanes / 32, 1) * sizeof(uint16_t)));
    saa_k_fin_pmask<<<nblk(p->n_slices, 8), 256>>>(p->n_slices, p->d_slice_ptr, permn, p->in_indptr, p->in_indices,
                                                   p->plane_mask ? 0 : 1, p->d_pmask, cnt);   // cnt[n_slices] is still 0
    CK(cudaMalloc((void **)&p->d_val_ptr, (p->n_slices + 1) * sizeof(int64_t)));
    thrust::exclusive_scan(thrust::device, cnt, cnt + p->n_slices + 1, p->d_val_ptr);
    int64_t n_val = 0;
    CK(cudaMemcpy(&n_val, p->d_val_ptr + p->n_slices, sizeof(int64_t), cudaMemcpyDeviceToHost));
    p->value_planes = n_val / 32;
    CK(cudaMalloc((void **)&p->d_val, std::max<int64_t>(n_val, 1) * sizeof(double)));
    CK(cudaMalloc((void **)&p->d_col, std::max<int64_t>(lanes, 1) * sizeof(int32_t)));
    saa_k_fin_fill<<<nblk(p->n_slices, 8), 256>>>(p->n_slices, p->d_slice_ptr, p->d_val_ptr, p->d_pmask, permn, p->d_iperm,
                                                  p->in_indptr, p->in_indices, p->in_data, p->d_val, p->d_col);
    CK(cudaMalloc((void **)&p->d_M, p->n_rows * sizeof(double)));
    CK(cudaMalloc((void **)&p->d_F, p->n_rows * sizeof(double)));
    saa_k_fin_vectors<<<nblk(p->n_rows, 256), 256>>>(p->n_rows, permn, p->in_M, p->in_F, p->d_M, p->d_F);
    CK(cudaMalloc((void **)&p->d_dir, (p->n_rows / 32) * sizeof(uint32_t)));
    CK(cudaMemset(p->d_dir, 0, (p->n_rows / 32) * sizeof(uint32_t)));
    if (!p->dirichlet.empty()) {
        DevBuf b_d;
        if (b_d.alloc(p->dirichlet.size() * sizeof(int64_t))) return -1;
        CK(cudaMemcpy(b_d.p, p->dirichlet.data(), p->dirichlet.size() * sizeof(int64_t), cudaMemcpyHostToDevice));
        saa_k_fin_dirichlet<<<nblk((int64_t)p->dirichlet.size(), 256), 256>>>((int64_t)p->dirichlet.size(), b_d.as<int64_t>(), p->d_iperm, p->d_dir);
        CK(cudaDeviceSynchronize());
    }
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    p->iperm_h.resize(n);
    CK(cudaMemcpy(p->iperm_h.data(), p->d_iperm, n * sizeof(int32_t), cudaMemcpyDeviceToHost));
    p->in_indptr = nullptr; p->in_indices = nullptr; p->in_data = nullptr; p->in_F = nullptr; p->in_M = nullptr;
    return finalize_tail(p, 3 * sh_padn);
}

// ---- K6: sparse assembly on the device ---------------------------------------------------------------------------
extern "C" int saa_device_free(void *ptr)
{
    if (ptr) CK(cudaFree(ptr));
    return 0;
}

extern "C" int saa_device_copy(void *dst, const void *src, int64_t bytes)
{
    if (bytes > 0) CK(cudaMemcpy(dst, src, (size_t)bytes, cudaMemcpyDefault));
    return 0;
}

// node -> (4*element + corner) incidence, ascending element order within a node
static int build_incidence(int64_t n_nodes, int64_t n_elem, const int32_t *cells, DevBuf &inc_ptr, DevBuf &inc_slot)
{
    const int64_t m = 4 * n_elem;
    if (m >= (int64_t)INT32_MAX) return fail("assembly: more than 2^29 elements per partition not supported");
    DevBuf keys;
    if (keys.alloc(m * sizeof(int32_t)) || inc_slot.alloc(m * sizeof(int32_t)) || inc_ptr.alloc((n_nodes + 1) * sizeof(int64_t))) return -1;
    CK(cudaMemcpy(keys.p, cells, m * sizeof(int32_t), cudaMemcpyDeviceToDevice));
    thrust::sequence(thrust::device, inc_slot.as<int32_t>(), inc_slot.as<int32_t>() + m);
    thrust::stable_sort_by_key(thrust::device, keys.as<int32_t>(), keys.as<int32_t>() + m, inc_slot.as<int32_t>());
    // inc_ptr[v] = first position with key >= v
    thrust::lower_bound(thrust::device, keys.as<int32_t>(), keys.as<int32_t>() + m, thrust::counting_iterator<int32_t>(0),
                        thrust::counting_iterator<int32_t>((int32_t)n_nodes + 1), inc_ptr.as<int64_t>());
    CK(cudaGetLastError());
    return 0;
}

extern "C" int saa_assemble_stiffness_dev(int device, int64_t n_nodes, int64_t n_elem, const int32_t *cells_dev,
                                          const double *coords_dev, double lmd, double mu, int64_t **indptr_out,
                                          int32_t **indices_out, double **data_out, int64_t *nnz_out)
{
    if (!cells_dev || !coords_dev || !indptr_out || !indices_out || !data_out || n_nodes <= 0 || n_elem <= 0)
        return fail("saa_assemble_stiffness_dev: null or empty argument");
    if (saa_device_count() <= device) return fail("saa_assemble_stiffness_dev: CUDA device %d not available", device);
    if (3 * n_nodes >= (int64_t)INT32_MAX) return fail("saa_assemble_stiffness_dev: too many nodes for int32 column ids");
    CK(cudaSetDevice(device));
    DevBuf inc_ptr, inc_slot, counts, blk_ptr, blk_col, bval, ovf;
    if (build_incidence(n_nodes, n_elem, cells_dev, inc_ptr, inc_slot)) return -1;
    if (counts.alloc((n_nodes + 1) * sizeof(int32_t)) || blk_ptr.alloc((n_nodes + 1) * sizeof(int64_t)) || ovf.alloc(sizeof(int))) return -1;
    CK(cudaMemset(ovf.p, 0, sizeof(int)));
    CK(cudaMemset(counts.p, 0, (n_nodes + 1) * sizeof(int32_t)));
    saa_k_asm_pattern<<<nblk(n_nodes, 128), 128>>>(n_nodes, inc_ptr.as<int64_t>(), inc_slot.as<int32_t>(), cells_dev, 0,
                                                   counts.as<int32_t>(), nullptr, nullptr, ovf.as<int>());
    int overflow = 0;
    CK(cudaMemcpy(&overflow, ovf.p, sizeof(int), cudaMemcpyDeviceToHost));
    if (overflow) return fail("saa_assemble_stiffness_dev: a node has more than %d neighbours", SAA_ASM_MAX_NB);
    thrust::exclusive_scan(thrust::device, counts.as<int32_t>(), counts.as<int32_t>() + n_nodes + 1, blk_ptr.as<int64_t>(), (int64_t)0);
    int64_t n_blk = 0;
    CK(cudaMemcpy(&n_blk, blk_ptr.as<int64_t>() + n_nodes, sizeof(int64_t), cudaMemcpyDeviceToHost));
    if (blk_col.alloc(n_blk * sizeof(int32_t)) || bval.alloc(n_blk * 9 * sizeof(double))) return -1;
    saa_k_asm_pattern<<<nblk(n_nodes, 128), 128>>>(n_nodes, inc_ptr.as<int64_t>(), inc_slot.as<int32_t>(), cells_dev, 1,
                                                   nullptr, blk_ptr.as<int64_t>(), blk_col.as<int32_t>(), ovf.as<int>());
    CK(cudaMemset(bval.p, 0, n_blk * 9 * sizeof(double)));
    saa_k_asm_values<<<nblk(n_nodes, 128), 128>>>(n_nodes, inc_ptr.as<int64_t>(), inc_slot.as<int32_t>(), cells_dev, coords_dev,
                                                  lmd, mu, blk_ptr.as<int64_t>(), blk_col.as<int32_t>(), bval.as<double>());
    CK(cudaGetLastError());
    cudaFree(inc_slot.p); inc_slot.p = nullptr;
    cudaFree(inc_ptr.p); inc_ptr.p = nullptr;
    // zero dropping + scalar CSR
    const int64_t n_rows = 3 * n_nodes;
    DevBuf row_nnz;
    if (row_nnz.alloc((n_rows + 1) * sizeof(int64_t))) return -1;
    CK(cudaMemset(row_nnz.p, 0, (n_rows + 1) * sizeof(int64_t)));
    saa_k_asm_row_nnz<<<nblk(n_rows, 256), 256>>>(n_nodes, blk_ptr.as<int64_t>(), bval.as<double>(), row_nnz.as<int64_t>());
    int64_t *indptr = nullptr;
    CK(cudaMalloc((void **)&indptr, (n_rows + 1) * sizeof(int64_t)));
    thrust::exclusive_scan(thrust::device, row_nnz.as<int64_t>(), row_nnz.as<int64_t>() + n_rows + 1, indptr);
    int64_t nnz = 0;
    CK(cudaMemcpy(&nnz, indptr + n_rows, sizeof(int64_t), cudaMemcpyDeviceToHost));
    int32_t *indices = nullptr;
    double *data = nullptr;
    CK(cudaMalloc((void **)&indices, std::max<int64_t>(nnz, 1) * sizeof(int32_t)));
    CK(cudaMalloc((void **)&data, std::max<int64_t>(nnz, 1) * sizeof(double)));
    saa_k_asm_compact<<<nblk(n_rows, 256), 256>>>(n_nodes, blk_ptr.as<int64_t>(), blk_col.as<int32_t>(), bval.as<double>(), indptr, indices, data);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    *indptr_out = indptr; *indices_out = indices; *data_out = data;
    if (nnz_out) *nnz_out = nnz;
    return 0;
}

extern "C" int saa_assemble_mass_load_dev(int device, int64_t n_nodes, int64_t n_elem, const int32_t *cells_dev,
                                          const double *coords_dev, double rho, double fz, double *m_node_out_dev,
                                          double *F_out_dev)
{
    if (!cells_dev || !coords_dev || !m_node_out_dev || !F_out_dev || n_nodes <= 0 || n_elem <= 0)
        return fail("saa_assemble_mass_load_dev: null or empty argument");
    if (saa_device_count() <= device) return fail("saa_assemble_mass_load_dev: CUDA device %d not available", device);
    CK(cudaSetDevice(device));
    DevBuf inc_ptr, inc_slot;
    if (build_incidence(n_nodes, n_elem, cells_dev, inc_ptr, inc_slot)) return -1;
    saa_k_asm_mass_load<<<nblk(n_nodes, 128), 128>>>(n_nodes, inc_ptr.as<int64_t>(), inc_slot.as<int32_t>(), cells_dev, coords_dev,
                                                     rho, fz, m_node_out_dev, F_out_dev);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    return 0;
}
