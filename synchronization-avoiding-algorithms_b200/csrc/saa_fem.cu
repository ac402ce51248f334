// saa_fem.cu — C ABI (include/saa_fem.h) of the explicit FE time-step path: plan construction
// (boundary-first / sigma-sorted sliced-ELL layout), state movement, stepping strategies (per-step
// launches, CUDA graph, cooperative persistent loop) and halo transports (in-process group, NCCL).
//
// Reference semantics restated here (paths under /root/reference): Tools/Dynamic_solver.py:9-34,
// Tools/Distributed_tools.py:77-92, Data_prepare.py:223-240, Online_predictor.py:251-318.
#include "saa_kernels.cuh"
#include "saa_energy.cuh"
#include "saa_matfree.cuh"
#include "saa_stress.cuh"
#include "saa_static.cuh"
#include "saa_multigrid.cuh"

#include <dlfcn.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <memory>
#include <numeric>
#include <string>
#include <vector>

#include "../../include/saa_fem.h"

#define SAA_SIGMA 1024          // nodes per sorting window (multiple of 32)
#define SAA_WARPS_PER_BLOCK 8
#define SAA_DEFAULT_KVARIANT (-1) // schedule variant of the step kernel: -1 = by partition size; SAA_KVARIANT overrides

static thread_local std::string g_err;

static int fail(const char *fmt, ...)
{
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return -1;
}

#define CK(call)                                                                                           \
    do {                                                                                                   \
        cudaError_t e_ = (call);                                                                           \
        if (e_ != cudaSuccess) return fail("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
    } while (0)

// ---- minimal NCCL binding resolved at run time (torch ships libnccl.so.2; no link-time dependency) ----
typedef struct { char internal[128]; } saa_ncclUniqueId;
typedef void *saa_ncclComm_t;
struct NcclApi {
    void *h = nullptr;
    int (*GetUniqueId)(saa_ncclUniqueId *) = nullptr;
    int (*CommInitRank)(saa_ncclComm_t *, int, saa_ncclUniqueId, int) = nullptr;
    int (*CommDestroy)(saa_ncclComm_t) = nullptr;
    int (*Send)(const void *, size_t, int, int, saa_ncclComm_t, cudaStream_t) = nullptr;
    int (*Recv)(void *, size_t, int, int, saa_ncclComm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
};
static NcclApi g_nccl;
static const int SAA_NCCL_DOUBLE = 8;   // ncclFloat64

static int load_nccl()
{
    if (g_nccl.h) return 0;
    const char *names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char *n : names) {
        g_nccl.h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (g_nccl.h) break;
    }
    if (!g_nccl.h) return fail("cannot dlopen libnccl.so.2 (%s); import torch first or set LD_LIBRARY_PATH", dlerror());
#define SYM(f, name)                                             \
    *(void **)(&g_nccl.f) = dlsym(g_nccl.h, name);               \
    if (!g_nccl.f) return fail("libnccl: missing symbol %s", name)
    SYM(GetUniqueId, "ncclGetUniqueId");
    SYM(CommInitRank, "ncclCommInitRank");
    SYM(CommDestroy, "ncclCommDestroy");
    SYM(Send, "ncclSend");
    SYM(Recv, "ncclRecv");
    SYM(GroupStart, "ncclGroupStart");
    SYM(GroupEnd, "ncclGroupEnd");
    SYM(GetErrorString, "ncclGetErrorString");
#undef SYM
    return 0;
}
#define NCK(call)                                                                                        \
    do {                                                                                                 \
        int e_ = (call);                                                                                 \
        if (e_ != 0) return fail("%s:%d %s -> NCCL error %d (%s)", __FILE__, __LINE__, #call, e_,        \
                                 g_nccl.GetErrorString ? g_nccl.GetErrorString(e_) : "?");               \
    } while (0)

// ---------------------------------------------------------------------------------------------------
struct saa_plan {
    int device = 0;
    bool finalized = false;
    // device-resident inputs (saa_plan_create_dev): borrowed until finalize
    bool dev_input = false;
    const int64_t *in_indptr = nullptr;
    const int32_t *in_indices = nullptr;
    const double *in_data = nullptr, *in_F = nullptr, *in_M = nullptr;
    // host copies of the inputs (released by finalize)
    int64_t n_dof = 0;
    std::vector<int32_t> indptr, indices;
    std::vector<double> data, F, M;
    std::vector<int64_t> dirichlet;
    double dt = 0, dt2 = 0, dt_half = 0, half_alpha = 0, alpha = 0;
    // halo description (host)
    int rank = 0, size = 1;
    std::vector<int64_t> shared_pos, nb_ptr, send_idx, holders_ptr, holders_slot;
    std::vector<int32_t> nb_rank, holders_rank;
    // layout
    int64_t nnz = 0, padded_entries = 0, n_rows = 0, n_slices = 0, sh_slices = 0;
    int64_t value_planes = 0;              // stored value planes (raw and coded)
    int64_t coded_planes = 0;              // of which coded (int64 base + 32 16-bit offsets)
    bool plane_mask = true;                // false: all nine planes of every block stored (SAA_PLANE_MASK=0, or the cp.async variant)
    bool value_code = true;                // false: every block-row raw (SAA_VALUE_CODE=0, or plane_mask false)
    std::vector<int32_t> iperm_h;          // external local DOF -> internal row
    std::vector<int32_t> node_order;       // optional base order of the nodes (saa_plan_set_node_order); empty = ascending
    // device
    SaaDev D{};
    SaaHaloDev H{};
    int64_t *d_slice_ptr = nullptr, *d_val_ptr = nullptr, *d_vb_ptr = nullptr;
    uint16_t *d_pmask = nullptr;
    long long *d_vbase = nullptr;
    double *d_val = nullptr, *d_M = nullptr, *d_F = nullptr;
    int32_t *d_col = nullptr, *d_iperm = nullptr;
    uint32_t *d_dir = nullptr;
    double *d_buf[2] = {nullptr, nullptr};  // displacement levels; d0 = d_buf[cur], dn = d_buf[cur^1]
    SaaClock *d_clk = nullptr;              // [2], (tn, sync_step) = d_clk[cur]
    int cur = 0;
    double *d_stage = nullptr;              // 3*n_dof staging in external order (state I/O)
    // halo device
    double *d_xbuf = nullptr, *d_send = nullptr;
    double *d_recv = nullptr;               // peer region: [2 parities x total_msg doubles | n_nb arrival flags (u64)]
    unsigned int *d_done = nullptr;          // [0] boundary completion counter, [1] error word, [32] finished-block tickets
    unsigned long long *d_own_ready = nullptr;
    int kvariant = SAA_DEFAULT_KVARIANT;    // SAA_KVARIANT: schedule variant of the step kernel
    bool peer_fused = true;                 // one fused launch per synchronised step (SAA_PEER_FUSED=0 / SAA_OPT_PEER_FUSED: three kernels)
    bool prefer_nccl = false;               // SAA_OPT_PREFER_NCCL: synchronised steps use the NCCL transport although peer memory is attached
    int32_t *d_dst_nb = nullptr;
    // peer-memory transport
    bool peer = false;
    SaaHaloDev Hp{};                        // H with the peer destination table
    int32_t *d_dst_pos_peer = nullptr;
    double **d_peer_recv = nullptr;
    int64_t *d_peer_stride = nullptr;
    unsigned long long **d_peer_flag = nullptr;
    std::vector<void *> peer_mapped;        // cudaIpcOpenMemHandle results (closed on destroy)
    cudaGraphExec_t graph_peer[2] = {nullptr, nullptr};
    int64_t *d_dst_ptr = nullptr, *d_src_ptr = nullptr;
    int32_t *d_dst_pos = nullptr, *d_src_pos = nullptr;
    std::vector<int32_t> dst_pos_h, dst_nb_h; // host copies of the pack table (rebased by saa_plan_peer_attach)
    std::vector<int64_t> msg_off;           // [n_nb+1] offsets (in doubles) of each neighbour's message
    int64_t total_msg = 0;
    // history ring
    int32_t *d_hist_rows = nullptr;
    double *d_hist = nullptr;
    int64_t hist_n = 0, hist_cap = 0, hist_every = 1, hist_count = 0, step_index = 0;
    // prediction table (sync-avoiding mode)
    int32_t *d_pred_rows = nullptr;
    const double *d_pred_table = nullptr;
    int64_t pred_n = 0, pred_rows = 0, pred_next = 0;
    std::vector<int32_t> pred_rows_h;       // internal rows of the predicted DOFs
    SaaHookDev hook_h{};                    // host mirror of the device-resident hook state
    SaaHookDev *d_hook = nullptr;
    int64_t hook_epoch = 0;                 // bumped when the hook configuration (not just the table) changes
    struct StepGraph { int mode, cur; int64_t epoch; cudaGraphExec_t exec; int launches; };
    std::vector<StepGraph> step_graphs;     // two-step graphs of steps with hooks
    // energy monitor (saa_plan_set_energy): per-slice / per-unit partials [slices | units of 256 shared rows], the
    // reduction's block sums and ticket, accumulators + ring; PREDICT steps: skipped-row mask, stashed d_{n-1}, partials
    int64_t energy_cap = 0, energy_every = 1, energy_count = 0;
    int64_t epart_n = 0, epred_n = 0;       // partials per field (stride) of the step and of the prediction scatter
    int energy_grid = 0;                    // blocks of the reduction (fixed per plan: fixed summation order)
    double *d_epart = nullptr, *d_estage = nullptr, *d_ering = nullptr, *d_epred = nullptr, *d_pred_stash = nullptr;
    unsigned int *d_eticket = nullptr;
    uint32_t *d_pred_skip = nullptr;
    SaaEnergyDev *d_energy = nullptr;
    // execution
    cudaStream_t stream = nullptr;
    cudaGraphExec_t graph_exec[2] = {nullptr, nullptr};   // LOCAL-mode two-step graphs captured at cur = 0 / 1
    int coop_blocks = 0, coop_blocks_sync = 0, n_sms = 0;
    int64_t launches = 0;
    saa_ncclComm_t comm = nullptr;
    saa_group *group = nullptr;
    cudaEvent_t ev_msg = nullptr;
    bool in_split_step = false;             // between saa_plan_step_begin_host and saa_plan_step_end_host
    int64_t state_epoch = 1, host_epoch = 0; // saa_step_host_ex: the device still holds the previous call's d0 iff equal
    // pipelined host call (saa_step_host_ex): chunks of external rows; upload / compute / download overlap
    struct HostPipe {
        int state = 0;                        // 0 not built yet, 1 usable, -1 not applicable
        int64_t first_slice = 0;              // slices below are boundary slices (table 1) and not part of the chunks
        std::vector<int64_t> row_off;         // [K+1] external row offsets of the chunks
        std::vector<int64_t> slice_end;       // [K] compute chunk c = internal slices [slice_end[c-1], slice_end[c])
        std::vector<int> need_upload;         // [K] compute chunk c needs the uploads of chunks <= need_upload[c]
        std::vector<char> has_shared;         // [K] table 1: chunk holds shared rows (downloaded after the shared-row update)
        int need_boundary = -1;               // table 1: the boundary slices need the uploads of chunks <= this
    } hp[2];                                  // [0] local steps, [1] synchronised steps of a plan with neighbours
    std::vector<cudaEvent_t> hp_ev_up, hp_ev_cmp;
    cudaStream_t hp_s_in = nullptr, hp_s_out = nullptr;
    double *d_force = nullptr;              // [2 * n_rows] scratch of the stand-alone force synchronisation
    // matrix-free mode (K5, saa_plan_set_matfree_dev)
    SaaMatFreeDev MF{};
    int64_t *d_mf_slice_ptr = nullptr;
    int32_t *d_mf_inc = nullptr, *d_mf_cells = nullptr;
    double *d_mf_X = nullptr;
    int64_t mf_elems = 0, mf_lanes = 0;
    int mf_minb = 3;                        // SAA_MF_MINB: minimum resident blocks per SM of the matrix-free kernel (register cap)
    bool matfree = false;                   // SAA_OPT_MATFREE: local steps evaluate B^T D B u_e instead of streaming the matrix
    // stress recovery (saa_plan_element_stress_dev / saa_plan_nodal_stress_dev), allocated on first use
    int32_t *d_st_ext = nullptr;            // external position of every internal node (-1: slice padding)
    unsigned long long *d_st_bad = nullptr; // lowest element index with detJ <= 0 of the last element call, ~0 if none
};

struct saa_group {
    std::vector<saa_plan *> plans;
    cudaStream_t stream = nullptr;
};

// stream a plan's work is ordered on: its own, or its group's once it has joined one
static inline cudaStream_t plan_stream(const saa_plan *p) { return p->group ? p->group->stream : p->stream; }

extern "C" int saa_version(void) { return 100; }
extern "C" const char *saa_last_error(void) { return g_err.c_str(); }
extern "C" int saa_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

extern "C" int saa_plan_create(saa_plan **out, int device, int64_t n_dof, const int32_t *indptr, const int32_t *indices,
                               const double *data, const double *F_rankwise, const double *l_M,
                               const int64_t *dirichlet, int64_t n_dirichlet, double dt, double dt2, double dt_half,
                               double half_alpha, double alpha)
{
    if (!out || n_dof <= 0 || !indptr || !indices || !data || !F_rankwise || !l_M)
        return fail("saa_plan_create: null or empty argument");
    if (n_dof % 3 != 0) return fail("saa_plan_create: n_dof=%lld is not a multiple of 3", (long long)n_dof);
    if (n_dirichlet > 0 && !dirichlet) return fail("saa_plan_create: dirichlet is null");
    if (saa_device_count() <= device) return fail("saa_plan_create: CUDA device %d not available (no CPU fallback)", device);
    const int64_t nnz = indptr[n_dof];
    for (int64_t i = 0; i < n_dof; ++i)
        if (indptr[i + 1] < indptr[i]) return fail("saa_plan_create: indptr not monotone at row %lld", (long long)i);
    for (int64_t k = 0; k < nnz; ++k)
        if (indices[k] < 0 || indices[k] >= n_dof) return fail("saa_plan_create: column index out of range at %lld", (long long)k);
    for (int64_t k = 0; k < n_dirichlet; ++k)
        if (dirichlet[k] < 0 || dirichlet[k] >= n_dof) return fail("saa_plan_create: Dirichlet DOF out of range");
    saa_plan *p = new saa_plan();
    p->device = device;
    p->n_dof = n_dof;
    p->indptr.assign(indptr, indptr + n_dof + 1);
    p->indices.assign(indices, indices + nnz);
    p->data.assign(data, data + nnz);
    p->F.assign(F_rankwise, F_rankwise + n_dof);
    p->M.assign(l_M, l_M + n_dof);
    p->dirichlet.assign(dirichlet, dirichlet + n_dirichlet);
    p->dt = dt; p->dt2 = dt2; p->dt_half = dt_half; p->half_alpha = half_alpha; p->alpha = alpha;
    p->nnz = nnz;
    *out = p;
    return 0;
}

extern "C" int saa_plan_set_halo(saa_plan *p, int rank, int size, int64_t n_shared, const int64_t *shared_pos, int n_nb,
                                 const int32_t *nb_rank, const int64_t *nb_ptr, const int64_t *send_idx,
                                 const int64_t *holders_ptr, const int32_t *holders_rank, const int64_t *holders_slot)
{
    if (!p) return fail("saa_plan_set_halo: null plan");
    if (p->finalized) return fail("saa_plan_set_halo: plan already finalized");
    if (rank < 0 || rank >= size) return fail("saa_plan_set_halo: bad rank %d of %d", rank, size);
    p->rank = rank; p->size = size;
    if (n_shared > 0) {
        if (!shared_pos || !nb_rank || !nb_ptr || !send_idx || !holders_ptr || !holders_rank || !holders_slot || n_nb <= 0)
            return fail("saa_plan_set_halo: null argument");
        for (int64_t j = 0; j < n_shared; ++j)
            if (shared_pos[j] < 0 || 3 * shared_pos[j] + 2 >= p->n_dof) return fail("saa_plan_set_halo: shared_pos out of range");
        p->shared_pos.assign(shared_pos, shared_pos + n_shared);
        p->nb_rank.assign(nb_rank, nb_rank + n_nb);
        p->nb_ptr.assign(nb_ptr, nb_ptr + n_nb + 1);
        p->send_idx.assign(send_idx, send_idx + nb_ptr[n_nb]);
        p->holders_ptr.assign(holders_ptr, holders_ptr + n_shared + 1);
        p->holders_rank.assign(holders_rank, holders_rank + holders_ptr[n_shared]);
        p->holders_slot.assign(holders_slot, holders_slot + holders_ptr[n_shared]);
        for (int64_t k = 0; k < nb_ptr[n_nb]; ++k)
            if (send_idx[k] < 0 || send_idx[k] >= n_shared) return fail("saa_plan_set_halo: send_idx out of range");
    }
    return 0;
}

extern "C" int saa_plan_set_node_order(saa_plan *p, const int32_t *order, int64_t n_nodes)
{
    if (!p) return fail("saa_plan_set_node_order: null plan");
    if (p->finalized) return fail("saa_plan_set_node_order: plan already finalized");
    if (!order || n_nodes != p->n_dof / 3) return fail("saa_plan_set_node_order: need one entry per node (%lld)", (long long)(p->n_dof / 3));
    std::vector<char> seen(n_nodes, 0);
    for (int64_t i = 0; i < n_nodes; ++i) {
        if (order[i] < 0 || order[i] >= n_nodes || seen[order[i]]) return fail("saa_plan_set_node_order: not a permutation of the nodes");
        seen[order[i]] = 1;
    }
    p->node_order.assign(order, order + n_nodes);
    return 0;
}

struct DevBuf {   // RAII scratch
    void *p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
    int alloc(size_t bytes)
    {
        cudaError_t e = cudaMalloc(&p, std::max<size_t>(bytes, 16));
        if (e != cudaSuccess) return fail("cudaMalloc(%zu) -> %s", bytes, cudaGetErrorString(e));
        return 0;
    }
    template <class T> T *as() { return (T *)p; }
};

template <class T>
static int upload(T **dptr, const std::vector<T> &h)
{
    size_t bytes = std::max<size_t>(h.size(), 1) * sizeof(T);
    CK(cudaMalloc((void **)dptr, bytes));
    if (!h.empty()) CK(cudaMemcpy(*dptr, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
    return 0;
}

// order nodes of one region: windows of SAA_SIGMA nodes sorted by decreasing block count (stable)
static void sigma_sort(std::vector<int64_t> &nodes, const std::vector<int32_t> &nblk)
{
    for (size_t w = 0; w < nodes.size(); w += SAA_SIGMA) {
        size_t e = std::min(nodes.size(), w + (size_t)SAA_SIGMA);
        std::stable_sort(nodes.begin() + w, nodes.begin() + e, [&](int64_t a, int64_t b) { return nblk[a] > nblk[b]; });
    }
}

static inline unsigned nblk(int64_t n, int per) { return (unsigned)((n + per - 1) / per); }
static int finalize_tail(saa_plan *p, int64_t sh_pad);
static int prepare_graphs(saa_plan *p, bool peer);
static int finalize_device(saa_plan *p);

extern "C" int saa_plan_finalize(saa_plan *p)
{
    if (!p) return fail("saa_plan_finalize: null plan");
    if (p->finalized) return 0;
    if (const char *kv = getenv("SAA_KVARIANT")) p->kvariant = atoi(kv);
    {   // value planes that are zero in every lane of a slice are not stored (SAA_PLANE_MASK=0 stores all nine); the
        // cp.async variant walks the values by block-row arithmetic and gets the full-plane layout
        const char *pm = getenv("SAA_PLANE_MASK");
        p->plane_mask = !(pm && pm[0] == '0') && p->kvariant < 6;
        // block-rows whose planes span at most 65535 ulps are stored as base + 16-bit offsets (SAA_VALUE_CODE=0: all raw)
        const char *vc = getenv("SAA_VALUE_CODE");
        p->value_code = p->plane_mask && !(vc && vc[0] == '0');
    }
    if (p->dev_input) return finalize_device(p);
    CK(cudaSetDevice(p->device));
    const int64_t n = p->n_dof, nn = n / 3;
    const int64_t n_shared = (int64_t)p->shared_pos.size();

    // 1. block pattern: distinct column nodes of every node (union over its three rows, ascending)
    std::vector<int64_t> bptr(nn + 1, 0);
    std::vector<int32_t> bcol;
    bcol.reserve((size_t)(p->nnz / 6 + nn));
    std::vector<int32_t> nblk(nn, 0);
    for (int64_t e = 0; e < nn; ++e) {
        int32_t q[3] = {p->indptr[3 * e], p->indptr[3 * e + 1], p->indptr[3 * e + 2]};
        const int32_t qe[3] = {p->indptr[3 * e + 1], p->indptr[3 * e + 2], p->indptr[3 * e + 3]};
        for (;;) {
            int32_t cn = INT32_MAX;
            for (int A = 0; A < 3; ++A)
                if (q[A] < qe[A]) cn = std::min(cn, p->indices[q[A]] / 3);
            if (cn == INT32_MAX) break;
            for (int A = 0; A < 3; ++A)
                while (q[A] < qe[A] && p->indices[q[A]] / 3 == cn) {
                    if (q[A] + 1 < qe[A] && p->indices[q[A] + 1] <= p->indices[q[A]])
                        return fail("saa_plan_finalize: LocalK must have sorted, duplicate-free column indices");
                    ++q[A];
                }
            bcol.push_back(cn);
        }
        bptr[e + 1] = (int64_t)bcol.size();
        nblk[e] = (int32_t)(bptr[e + 1] - bptr[e]);
    }

    // 2. internal node order: interface nodes (canonical interface order), then the rest ascending
    std::vector<char> is_shared(nn, 0);
    std::vector<int64_t> sh_nodes, in_nodes;
    sh_nodes.reserve(n_shared);
    for (int64_t j = 0; j < n_shared; ++j) {
        const int64_t e = p->shared_pos[j];
        if (is_shared[e]) return fail("saa_plan_finalize: duplicate shared node");
        is_shared[e] = 1;
        sh_nodes.push_back(e);
    }
    in_nodes.reserve(nn - sh_nodes.size());
    for (int64_t i = 0; i < nn; ++i) {
        const int64_t e = p->node_order.empty() ? i : p->node_order[i];     // caller's locality-preserving order, if any
        if (!is_shared[e]) in_nodes.push_back(e);
    }
    sigma_sort(sh_nodes, nblk);
    sigma_sort(in_nodes, nblk);
    auto pad32 = [](int64_t v) { return (v + 31) / 32 * 32; };
    const int64_t sh_padn = pad32((int64_t)sh_nodes.size());
    const int64_t in_padn = pad32((int64_t)in_nodes.size());
    const int64_t n_slots = sh_padn + in_padn;
    p->n_rows = 3 * n_slots;
    p->n_slices = n_slots / 32;
    p->sh_slices = sh_padn / 32;
    if (p->n_rows >= (int64_t)INT32_MAX) return fail("saa_plan_finalize: more than 2^31 rows per partition not supported");
    std::vector<int64_t> permn(n_slots, -1);            // internal node -> external node (-1: padding)
    for (size_t i = 0; i < sh_nodes.size(); ++i) permn[i] = sh_nodes[i];
    for (size_t i = 0; i < in_nodes.size(); ++i) permn[sh_padn + i] = in_nodes[i];
    p->iperm_h.assign(n, -1);
    for (int64_t i = 0; i < n_slots; ++i)
        if (permn[i] >= 0)
            for (int c = 0; c < 3; ++c) p->iperm_h[3 * permn[i] + c] = (int32_t)(3 * i + c);

    // 3. plane-masked node-block sliced ELL
    std::vector<int64_t> slice_ptr(p->n_slices + 1, 0);
    for (int64_t s = 0; s < p->n_slices; ++s) {
        int32_t mx = 0;
        for (int l = 0; l < 32; ++l) {
            const int64_t e = permn[s * 32 + l];
            if (e >= 0) mx = std::max(mx, nblk[e]);
        }
        slice_ptr[s + 1] = slice_ptr[s] + 32 * (int64_t)mx;
    }
    const int64_t lanes = slice_ptr[p->n_slices];
    p->padded_entries = 9 * lanes;
    // visits the stored entries of node e in stored order: fn(block j, plane 3A+B, entry k)
    auto for_each_entry = [&](int64_t e, auto &&fn) {
        int32_t q[3] = {p->indptr[3 * e], p->indptr[3 * e + 1], p->indptr[3 * e + 2]};
        const int32_t qe[3] = {p->indptr[3 * e + 1], p->indptr[3 * e + 2], p->indptr[3 * e + 3]};
        for (int64_t j = 0; j < nblk[e]; ++j) {
            const int32_t cn = bcol[bptr[e] + j];
            for (int A = 0; A < 3; ++A)
                while (q[A] < qe[A] && p->indices[q[A]] / 3 == cn) {
                    fn(j, 3 * A + p->indices[q[A]] % 3, q[A]);
                    ++q[A];
                }
        }
    };
    // stored planes of every block-row: the union of the stored patterns of its 32 lanes (the pattern, not the value
    // bits, so that an explicitly stored 0.0 is kept), and the column-node ids
    std::vector<uint16_t> pmask((size_t)(lanes / 32), p->plane_mask ? 0 : 0x1FF);
    std::vector<int32_t> col((size_t)lanes);
    for (int64_t s = 0; s < p->n_slices; ++s) {
        const int64_t L = (slice_ptr[s + 1] - slice_ptr[s]) / 32;
        uint16_t *ms = pmask.data() + slice_ptr[s] / 32;
        int32_t *cs = col.data() + slice_ptr[s];
        for (int l = 0; l < 32; ++l) {
            const int64_t inode = s * 32 + l;
            const int64_t e = permn[inode];
            int64_t cnt = 0;
            if (e >= 0) {
                cnt = nblk[e];
                for_each_entry(e, [&](int64_t j, int b, int32_t) { ms[j] |= (uint16_t)(1u << b); });
                for (int64_t j = 0; j < cnt; ++j) cs[32 * j + l] = p->iperm_h[3 * (int64_t)bcol[bptr[e] + j]] / 3;
            }
            // padding blocks: 0.0 * d0[own node] at the end of the rows leaves the sums unchanged
            for (int64_t j = cnt; j < L; ++j) cs[32 * j + l] = (int32_t)inode;
        }
    }
    // raw planes of every slice, then the coding decision of every block-row from their bits and the final layout
    std::vector<int64_t> raw_ptr(p->n_slices + 1, 0);
    for (int64_t s = 0; s < p->n_slices; ++s) {
        int64_t planes = 0;
        for (int64_t r = slice_ptr[s] / 32; r < slice_ptr[s + 1] / 32; ++r) planes += __builtin_popcount(pmask[r]);
        raw_ptr[s + 1] = raw_ptr[s] + 32 * planes;
    }
    p->value_planes = raw_ptr[p->n_slices] / 32;
    std::vector<double> raw((size_t)raw_ptr[p->n_slices], 0.0);
    for (int64_t s = 0; s < p->n_slices; ++s) {
        const int64_t L = (slice_ptr[s + 1] - slice_ptr[s]) / 32;
        const uint16_t *ms = pmask.data() + slice_ptr[s] / 32;
        std::vector<int64_t> off(L + 1, 0);              // planes stored for the blocks before j
        for (int64_t j = 0; j < L; ++j) off[j + 1] = off[j] + __builtin_popcount(ms[j]);
        double *vs = raw.data() + raw_ptr[s];
        for (int l = 0; l < 32; ++l) {
            const int64_t e = permn[s * 32 + l];
            if (e >= 0)
                for_each_entry(e, [&](int64_t j, int b, int32_t k) {
                    vs[32 * (off[j] + __builtin_popcount(ms[j] & ((1u << b) - 1u))) + l] = p->data[k];
                });
        }
    }
    auto bits = [](double x) { int64_t b; std::memcpy(&b, &x, 8); return b; };
    std::vector<int64_t> val_ptr(p->n_slices + 1, 0), vb_ptr(p->n_slices + 1, 0);
    for (int64_t s = 0; s < p->n_slices; ++s) {
        const double *pl = raw.data() + raw_ptr[s];     // next raw plane of the slice
        int64_t vals = 0, coded = 0;
        for (int64_t r = slice_ptr[s] / 32; r < slice_ptr[s + 1] / 32; ++r) {
            const int n = __builtin_popcount(pmask[r]);
            bool code = p->value_code && n > 0;
            for (int i = 0; i < n && code; ++i) {
                int64_t lo = INT64_MAX, hi = INT64_MIN;
                for (int l = 0; l < 32; ++l) { lo = std::min(lo, bits(pl[32 * i + l])); hi = std::max(hi, bits(pl[32 * i + l])); }
                code = (uint64_t)hi - (uint64_t)lo <= 65535u;
            }
            if (code) pmask[r] |= SAA_CODED;
            vals += (code ? 8 : 32) * n;
            coded += code ? n : 0;
            pl += 32 * n;
        }
        val_ptr[s + 1] = val_ptr[s] + vals;
        vb_ptr[s + 1] = vb_ptr[s] + coded;
    }
    p->coded_planes = vb_ptr[p->n_slices];
    std::vector<double> val((size_t)val_ptr[p->n_slices], 0.0);
    std::vector<long long> vbase((size_t)vb_ptr[p->n_slices], 0);
    for (int64_t s = 0; s < p->n_slices; ++s) {
        const double *pl = raw.data() + raw_ptr[s];
        char *v = (char *)(val.data() + val_ptr[s]);
        long long *vb = vbase.data() + vb_ptr[s];
        for (int64_t r = slice_ptr[s] / 32; r < slice_ptr[s + 1] / 32; ++r) {
            const int n = __builtin_popcount(pmask[r] & SAA_PLANES);
            for (int i = 0; i < n; ++i, pl += 32) {
                if (pmask[r] & SAA_CODED) {                // lane-major offsets (saa_coded_off)
                    int64_t lo = INT64_MAX;
                    for (int l = 0; l < 32; ++l) lo = std::min(lo, bits(pl[l]));
                    *vb++ = lo;
                    for (int l = 0; l < 32; ++l) {
                        const uint16_t o = (uint16_t)((uint64_t)bits(pl[l]) - (uint64_t)lo);
                        std::memcpy(v + saa_coded_off(n, i, l), &o, 2);
                    }
                } else {
                    std::memcpy(v + 256 * i, pl, 256);
                }
            }
            v += ((pmask[r] & SAA_CODED) ? 64 : 256) * n;
        }
    }
    std::vector<double>().swap(raw);
    std::vector<double> M(p->n_rows, 1.0), F(p->n_rows, 0.0);
    for (int64_t r = 0; r < n; ++r) { M[p->iperm_h[r]] = p->M[r]; F[p->iperm_h[r]] = p->F[r]; }
    std::vector<uint32_t> dir(p->n_rows / 32, 0u);
    for (int64_t k : p->dirichlet) {
        int32_t i = p->iperm_h[k];
        dir[i >> 5] |= (1u << (i & 31));
    }

    if (upload(&p->d_slice_ptr, slice_ptr) || upload(&p->d_val_ptr, val_ptr) || upload(&p->d_pmask, pmask) ||
        upload(&p->d_vb_ptr, vb_ptr) || upload(&p->d_vbase, vbase) || upload(&p->d_val, val) || upload(&p->d_col, col) ||
        upload(&p->d_M, M) || upload(&p->d_F, F) || upload(&p->d_dir, dir) || upload(&p->d_iperm, p->iperm_h))
        return -1;
    const int64_t sh_pad = 3 * sh_padn;
    return finalize_tail(p, sh_pad);
}

// second half of finalize, shared by the host-CSR and the device-CSR paths: state buffers, kernel parameter
// block, halo tables.  Needs n_rows / n_slices / sh_slices / iperm_h and the device layout arrays.
static int finalize_tail(saa_plan *p, int64_t sh_pad)
{
    const int64_t n = p->n_dof;
    const int64_t n_shared = (int64_t)p->shared_pos.size();
    for (int b = 0; b < 2; ++b) {
        CK(cudaMalloc((void **)&p->d_buf[b], p->n_rows * sizeof(double)));
        CK(cudaMemset(p->d_buf[b], 0, p->n_rows * sizeof(double)));
    }
    CK(cudaMalloc((void **)&p->d_clk, 2 * sizeof(SaaClock)));
    CK(cudaMemset(p->d_clk, 0, 2 * sizeof(SaaClock)));
    CK(cudaMalloc((void **)&p->d_hook, sizeof(SaaHookDev)));
    p->hook_h.hist_every = 1; p->hook_h.hist_cap = 1;
    CK(cudaMemcpy(p->d_hook, &p->hook_h, sizeof(SaaHookDev), cudaMemcpyHostToDevice));
    CK(cudaMalloc((void **)&p->d_stage, 3 * n * sizeof(double)));
    CK(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));

    p->D.n_rows = p->n_rows; p->D.n_slices = p->n_slices; p->D.sh_slices = p->sh_slices;
    p->D.slice_ptr = p->d_slice_ptr; p->D.val_ptr = p->d_val_ptr; p->D.pmask = p->d_pmask; p->D.val = p->d_val; p->D.col = p->d_col; p->D.dir_mask = p->d_dir;
    p->D.vb_ptr = p->d_vb_ptr; p->D.vbase = p->d_vbase;
    p->D.M = p->d_M; p->D.F = p->d_F;
    {   // one mass value per node when every node's three DOFs hold the same bits (SAA_NODE_MASS=0 keeps the per-DOF stream)
        const char *nm = getenv("SAA_NODE_MASS");
        int *d_flag = nullptr, differs = 0;
        const int64_t nn = p->n_rows / 3;
        if (!(nm && nm[0] == '0')) {
            CK(cudaMalloc((void **)&d_flag, sizeof(int)));
            CK(cudaMemset(d_flag, 0, sizeof(int)));
            saa_k_mass_check<<<nblk(nn, 256), 256>>>(nn, p->d_M, d_flag);
            CK(cudaMemcpy(&differs, d_flag, sizeof(int), cudaMemcpyDeviceToHost));
            cudaFree(d_flag);
            if (!differs) {
                double *mn = nullptr;
                CK(cudaMalloc((void **)&mn, nn * sizeof(double)));
                saa_k_mass_compact<<<nblk(nn, 256), 256>>>(nn, p->d_M, mn);
                CK(cudaDeviceSynchronize());
                cudaFree(p->d_M);
                p->d_M = mn; p->D.M = mn; p->D.node_mass = 1;
            }
        }
    }
    p->D.dt = p->dt; p->D.dt2 = p->dt2; p->D.dt_half = p->dt_half; p->D.half_alpha = p->half_alpha; p->D.alpha = p->alpha;

    // 3. halo: message layout, pack lists, rank-ordered source lists
    if (n_shared > 0) {
        const int n_nb = (int)p->nb_rank.size();
        p->msg_off.assign(n_nb + 1, 0);
        for (int k = 0; k < n_nb; ++k) p->msg_off[k + 1] = p->msg_off[k] + 3 * (p->nb_ptr[k + 1] - p->nb_ptr[k]);
        p->total_msg = p->msg_off[n_nb];
        if (sh_pad + 2 * p->total_msg >= (int64_t)INT32_MAX) return fail("halo too large");
        // internal row of (shared node j, component c)
        auto irow = [&](int64_t j, int c) { return (int64_t)p->iperm_h[3 * p->shared_pos[j] + c]; };
        std::vector<std::vector<int32_t>> dst(sh_pad), dstk(sh_pad), src(sh_pad);
        for (int k = 0; k < n_nb; ++k)
            for (int64_t e = p->nb_ptr[k]; e < p->nb_ptr[k + 1]; ++e)
                for (int c = 0; c < 3; ++c) {
                    dst[irow(p->send_idx[e], c)].push_back((int32_t)(p->msg_off[k] + 3 * (e - p->nb_ptr[k]) + c));
                    dstk[irow(p->send_idx[e], c)].push_back((int32_t)k);
                }
        for (int64_t j = 0; j < n_shared; ++j)
            for (int64_t h = p->holders_ptr[j]; h < p->holders_ptr[j + 1]; ++h) {
                if (h > p->holders_ptr[j] && p->holders_rank[h] <= p->holders_rank[h - 1])
                    return fail("saa_plan_finalize: holders of a shared node must be in ascending rank order");
                for (int c = 0; c < 3; ++c) {
                    if (p->holders_slot[h] < 0) {
                        src[irow(j, c)].push_back((int32_t)irow(j, c));
                    } else {
                        int k = (int)(std::find(p->nb_rank.begin(), p->nb_rank.end(), p->holders_rank[h]) - p->nb_rank.begin());
                        if (k >= n_nb) return fail("saa_plan_finalize: holder rank %d is not a neighbour", p->holders_rank[h]);
                        if (p->holders_slot[h] >= p->nb_ptr[k + 1] - p->nb_ptr[k]) return fail("holder slot out of range");
                        src[irow(j, c)].push_back((int32_t)(sh_pad + p->msg_off[k] + 3 * p->holders_slot[h] + c));
                    }
                }
            }
        std::vector<int64_t> dst_ptr(sh_pad + 1, 0), src_ptr(sh_pad + 1, 0);
        std::vector<int32_t> dst_pos, dst_nb, src_pos;
        for (int64_t r = 0; r < sh_pad; ++r) {
            dst_pos.insert(dst_pos.end(), dst[r].begin(), dst[r].end());
            dst_nb.insert(dst_nb.end(), dstk[r].begin(), dstk[r].end());
            src_pos.insert(src_pos.end(), src[r].begin(), src[r].end());
            dst_ptr[r + 1] = (int64_t)dst_pos.size();
            src_ptr[r + 1] = (int64_t)src_pos.size();
        }
        p->dst_pos_h = dst_pos; p->dst_nb_h = dst_nb;
        if (upload(&p->d_dst_ptr, dst_ptr) || upload(&p->d_dst_pos, dst_pos) || upload(&p->d_src_ptr, src_ptr) ||
            upload(&p->d_src_pos, src_pos))
            return -1;
        CK(cudaMalloc((void **)&p->d_xbuf, sh_pad * sizeof(double)));
        CK(cudaMemset(p->d_xbuf, 0, sh_pad * sizeof(double)));
        const size_t region = (size_t)(2 * p->total_msg) * sizeof(double) + (size_t)std::max(n_nb, 1) * sizeof(unsigned long long);
        CK(cudaMalloc((void **)&p->d_recv, region));
        CK(cudaMemset(p->d_recv, 0, region));
        CK(cudaMalloc((void **)&p->d_done, 64 * sizeof(unsigned int)));
        CK(cudaMemset(p->d_done, 0, 64 * sizeof(unsigned int)));
        CK(cudaMalloc((void **)&p->d_own_ready, sizeof(unsigned long long)));
        CK(cudaMemset(p->d_own_ready, 0, sizeof(unsigned long long)));
        if (upload(&p->d_dst_nb, dst_nb)) return -1;
        CK(cudaMalloc((void **)&p->d_send, std::max<int64_t>(p->total_msg, 1) * sizeof(double)));
        p->H.sh_rows = sh_pad; p->H.xbuf = p->d_xbuf; p->H.sendbuf = p->d_send;
        p->H.recv = p->d_recv; p->H.recv_stride = p->total_msg;
        p->H.dst_ptr = p->d_dst_ptr; p->H.dst_pos = p->d_dst_pos; p->H.dst_nb = p->d_dst_nb;
        p->H.src_ptr = p->d_src_ptr; p->H.src_pos = p->d_src_pos;
        p->H.n_nb = n_nb; p->H.done_ctr = p->d_done; p->H.err = p->d_done + 1; p->H.tail_ticket = p->d_done + 32; p->H.own_ready = p->d_own_ready;
        p->H.flags = (const unsigned long long *)(p->d_recv + 2 * p->total_msg);
    }

    // cooperative launch geometry for the persistent kernel
    int dev_sms = 0, occ = 0;
    CK(cudaDeviceGetAttribute(&dev_sms, cudaDevAttrMultiProcessorCount, p->device));
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, saa_k_persistent, 32 * SAA_WARPS_PER_BLOCK, 0));
    p->coop_blocks = dev_sms * occ;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, saa_k_persistent_sync, 32 * SAA_WARPS_PER_BLOCK, 0));
    p->coop_blocks_sync = dev_sms * occ;
    p->n_sms = dev_sms;

    // host copies are no longer needed
    std::vector<int32_t>().swap(p->indptr); std::vector<int32_t>().swap(p->indices);
    std::vector<double>().swap(p->data); std::vector<double>().swap(p->F); std::vector<double>().swap(p->M);
    CK(cudaDeviceSynchronize());   // set-up work ran on the default stream; the plan's stream is non-blocking
    // measured on B200 (profiles/r1/kernel_variants.md, profiles/r2/kernel_variants_r2.md, profiles/plane_mask/variants.md
    // and, with the coded values, profiles/value_coding/value_coding_probe.json): the plain schedule with 3 blocks per SM
    // (85-register cap, no spills; the 64-register cap of 4 blocks per SM spills) wins at 1.1 M and 104 M DOF, coded or raw
    if (p->kvariant < 0) p->kvariant = 2;
    p->finalized = true;
    return prepare_graphs(p, false);
}

extern "C" int saa_plan_destroy(saa_plan *p)
{
    if (!p) return 0;
    if (p->finalized) {
        cudaSetDevice(p->device);
        if (p->stream) cudaStreamSynchronize(p->stream);
        for (int i = 0; i < 2; ++i) {
            if (p->graph_exec[i]) cudaGraphExecDestroy(p->graph_exec[i]);
            if (p->graph_peer[i]) cudaGraphExecDestroy(p->graph_peer[i]);
        }
        for (void *m : p->peer_mapped) cudaIpcCloseMemHandle(m);
        for (auto &g : p->step_graphs) cudaGraphExecDestroy(g.exec);
        void *ptrs[] = {p->d_slice_ptr, p->d_val_ptr, p->d_vb_ptr, p->d_pmask, p->d_val, p->d_vbase, p->d_col, p->d_M, p->d_F, p->d_dir, p->d_iperm, p->d_buf[0], p->d_buf[1],
                        p->d_clk, p->d_stage, p->d_xbuf, p->d_send, p->d_dst_ptr, p->d_dst_pos, p->d_src_ptr, p->d_src_pos,
                        p->d_recv, p->d_done, p->d_own_ready, p->d_dst_nb, p->d_dst_pos_peer, p->d_peer_recv, p->d_peer_stride, p->d_peer_flag,
                        p->d_hist_rows, p->d_hist, p->d_pred_rows, p->d_force, p->d_hook,
                        p->d_epart, p->d_estage, p->d_ering, p->d_epred, p->d_pred_stash, p->d_eticket, p->d_pred_skip, p->d_energy,
                        p->d_mf_slice_ptr, p->d_mf_inc, p->d_mf_cells, p->d_mf_X, p->d_st_ext, p->d_st_bad};
        for (void *q : ptrs)
            if (q) cudaFree(q);
        if (p->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(p->comm);
        if (p->ev_msg) cudaEventDestroy(p->ev_msg);
        for (cudaEvent_t e : p->hp_ev_up) cudaEventDestroy(e);
        for (cudaEvent_t e : p->hp_ev_cmp) cudaEventDestroy(e);
        if (p->hp_s_in) cudaStreamDestroy(p->hp_s_in);
        if (p->hp_s_out) cudaStreamDestroy(p->hp_s_out);
        if (p->stream) cudaStreamDestroy(p->stream);
    }
    delete p;
    return 0;
}

extern "C" int64_t saa_plan_n_dof(const saa_plan *p) { return p ? p->n_dof : -1; }
extern "C" int64_t saa_plan_nnz(const saa_plan *p) { return p ? p->nnz : -1; }
extern "C" int64_t saa_plan_padded_entries(const saa_plan *p) { return p ? p->padded_entries : -1; }
extern "C" int64_t saa_plan_kernel_launches(const saa_plan *p) { return p ? p->launches : -1; }
extern "C" int64_t saa_plan_vector_bytes(const saa_plan *p)
{
    // fp64 streams of one step: d0 and dn read, d1 written, F read (one value per row each) + the lumped mass (per row, or per node)
    return p ? 4 * 8 * p->n_rows + 8 * (p->D.node_mass ? p->n_rows / 3 : p->n_rows) : -1;
}
extern "C" int64_t saa_plan_value_planes(const saa_plan *p) { return p ? p->value_planes : -1; }
extern "C" int64_t saa_plan_coded_planes(const saa_plan *p) { return p ? p->coded_planes : -1; }
extern "C" int64_t saa_plan_matrix_bytes(const saa_plan *p)
{
    // the plane-masked layout without value coding: stored value planes (32 fp64 each), one column-node id per
    // block-lane, one plane mask per block-row, slice and value offsets, Dirichlet mask words
    if (!p) return -1;
    const int64_t lanes = p->padded_entries / 9;
    return p->value_planes * 256 + lanes * 4 + (lanes / 32) * 2 + 2 * (p->n_slices + 1) * 8 + (p->n_rows / 32) * 4;
}
extern "C" int64_t saa_plan_streamed_matrix_bytes(const saa_plan *p)
{
    // what a matrix pass reads: raw planes 256 B, coded planes 64 B of offsets + an 8-B base, the ids, masks, the
    // slice, value and base offsets and the Dirichlet mask words
    if (!p) return -1;
    const int64_t lanes = p->padded_entries / 9;
    return (p->value_planes - p->coded_planes) * 256 + p->coded_planes * (64 + 8) + lanes * 4 + (lanes / 32) * 2 +
           3 * (p->n_slices + 1) * 8 + (p->n_rows / 32) * 4;
}
extern "C" void *saa_plan_stream(saa_plan *p) { return p ? (void *)plan_stream(p) : nullptr; }


#define NEED_FINAL(p, name)                                   \
    if (!(p)) return fail(name ": null plan");                \
    if (!(p)->finalized) return fail(name ": plan not finalized")

static int set_state_from_stage(saa_plan *p, cudaStream_t st, double tn, bool with_dn = true)
{
    // d_stage holds [d0_ext | dn_ext]; padding rows of the internal buffers stay 0
    p->state_epoch++;
    saa_k_scatter_to_internal<<<nblk(p->n_dof, 256), 256, 0, st>>>(p->n_dof, p->d_iperm, p->d_stage, p->d_buf[p->cur]);
    p->launches++;
    if (with_dn) {
        saa_k_scatter_to_internal<<<nblk(p->n_dof, 256), 256, 0, st>>>(p->n_dof, p->d_iperm, p->d_stage + p->n_dof, p->d_buf[p->cur ^ 1]);
        p->launches++;
    }
    CK(cudaMemcpyAsync(&p->d_clk[p->cur].tn, &tn, sizeof(double), cudaMemcpyHostToDevice, st));
    CK(cudaGetLastError());
    return 0;
}

extern "C" int saa_plan_set_state(saa_plan *p, const double *d0, const double *dn, double tn)
{
    NEED_FINAL(p, "saa_plan_set_state");
    if (!d0 || !dn) return fail("saa_plan_set_state: null argument");
    CK(cudaSetDevice(p->device));
    CK(cudaMemcpyAsync(p->d_stage, d0, p->n_dof * sizeof(double), cudaMemcpyHostToDevice, plan_stream(p)));
    CK(cudaMemcpyAsync(p->d_stage + p->n_dof, dn, p->n_dof * sizeof(double), cudaMemcpyHostToDevice, plan_stream(p)));
    if (set_state_from_stage(p, plan_stream(p), tn)) return -1;
    CK(cudaStreamSynchronize(plan_stream(p)));
    return 0;
}

extern "C" int saa_plan_set_state_dev(saa_plan *p, const double *d0, const double *dn, double tn)
{
    NEED_FINAL(p, "saa_plan_set_state_dev");
    if (!d0 || !dn) return fail("saa_plan_set_state_dev: null argument");
    CK(cudaSetDevice(p->device));
    CK(cudaMemcpyAsync(p->d_stage, d0, p->n_dof * sizeof(double), cudaMemcpyDeviceToDevice, plan_stream(p)));
    CK(cudaMemcpyAsync(p->d_stage + p->n_dof, dn, p->n_dof * sizeof(double), cudaMemcpyDeviceToDevice, plan_stream(p)));
    if (set_state_from_stage(p, plan_stream(p), tn)) return -1;
    CK(cudaStreamSynchronize(plan_stream(p)));
    return 0;
}

static int get_state_to_stage(saa_plan *p, cudaStream_t st, bool want_d0, bool want_dn)
{
    if (want_d0) { saa_k_gather_to_external<<<nblk(p->n_dof, 256), 256, 0, st>>>(p->n_dof, p->d_iperm, p->d_buf[p->cur], p->d_stage); p->launches++; }
    if (want_dn) { saa_k_gather_to_external<<<nblk(p->n_dof, 256), 256, 0, st>>>(p->n_dof, p->d_iperm, p->d_buf[p->cur ^ 1], p->d_stage + p->n_dof); p->launches++; }
    CK(cudaGetLastError());
    return 0;
}

extern "C" int saa_plan_get_state(saa_plan *p, double *d0, double *dn, double *tn)
{
    NEED_FINAL(p, "saa_plan_get_state");
    CK(cudaSetDevice(p->device));
    if (get_state_to_stage(p, plan_stream(p), d0 != nullptr, dn != nullptr)) return -1;
    if (d0) CK(cudaMemcpyAsync(d0, p->d_stage, p->n_dof * sizeof(double), cudaMemcpyDeviceToHost, plan_stream(p)));
    if (dn) CK(cudaMemcpyAsync(dn, p->d_stage + p->n_dof, p->n_dof * sizeof(double), cudaMemcpyDeviceToHost, plan_stream(p)));
    if (tn) CK(cudaMemcpyAsync(tn, &p->d_clk[p->cur].tn, sizeof(double), cudaMemcpyDeviceToHost, plan_stream(p)));
    CK(cudaStreamSynchronize(plan_stream(p)));
    return 0;
}

extern "C" int saa_plan_get_state_dev(saa_plan *p, double *d0, double *dn, double *tn)
{
    NEED_FINAL(p, "saa_plan_get_state_dev");
    CK(cudaSetDevice(p->device));
    if (get_state_to_stage(p, plan_stream(p), d0 != nullptr, dn != nullptr)) return -1;
    if (d0) CK(cudaMemcpyAsync(d0, p->d_stage, p->n_dof * sizeof(double), cudaMemcpyDeviceToDevice, plan_stream(p)));
    if (dn) CK(cudaMemcpyAsync(dn, p->d_stage + p->n_dof, p->n_dof * sizeof(double), cudaMemcpyDeviceToDevice, plan_stream(p)));
    if (tn) CK(cudaMemcpyAsync(tn, &p->d_clk[p->cur].tn, sizeof(double), cudaMemcpyDeviceToHost, plan_stream(p)));
    CK(cudaStreamSynchronize(plan_stream(p)));
    return 0;
}

// ---- energy monitor --------------------------------------------------------------------------------------
// PREDICT steps with the monitor on: K1E skips the d_{n+1} terms of the predicted rows (mask) and stashes their d_{n-1};
// the prediction scatter adds those terms after the overwrite, one partial per block of 256 predicted rows
static int energy_prepare_predict(saa_plan *p)
{
    CK(cudaStreamSynchronize(plan_stream(p)));       // earlier steps may still read the buffers replaced here
    for (void *q : {(void *)p->d_pred_skip, (void *)p->d_pred_stash, (void *)p->d_epred})
        if (q) cudaFree(q);
    p->d_pred_skip = nullptr; p->d_pred_stash = nullptr; p->d_epred = nullptr; p->epred_n = 0;
    if (p->pred_n <= 0) return 0;
    std::vector<uint32_t> skip(p->n_rows / 32, 0u);
    for (int32_t r : p->pred_rows_h) skip[r >> 5] |= 1u << (r & 31);
    if (upload(&p->d_pred_skip, skip)) return -1;
    CK(cudaMalloc((void **)&p->d_pred_stash, p->n_rows * sizeof(double)));
    p->epred_n = nblk(p->pred_n, 256);
    CK(cudaMalloc((void **)&p->d_epred, SAA_ENERGY_PARTS * p->epred_n * sizeof(double)));
    return 0;
}

extern "C" int saa_plan_set_energy(saa_plan *p, int64_t capacity, int64_t every)
{
    NEED_FINAL(p, "saa_plan_set_energy");
    if (capacity > 0 && every < 1) return fail("saa_plan_set_energy: every must be >= 1 (got %lld)", (long long)every);
    if (capacity > 0 && p->matfree)
        return fail("saa_plan_set_energy: the matrix-free kernel (SAA_OPT_MATFREE) computes a different force; the energy monitor needs the assembled-matrix step");
    CK(cudaSetDevice(p->device));
    CK(cudaStreamSynchronize(plan_stream(p)));
    if (p->d_ering) { cudaFree(p->d_ering); p->d_ering = nullptr; }
    p->energy_cap = p->energy_count = 0;
    p->hook_epoch++;
    if (capacity <= 0) return 0;
    if (!p->d_epart) {                               // layout-sized buffers: allocated once per plan
        const int64_t n_units = nblk(p->H.sh_rows, 256);
        p->epart_n = p->n_slices + n_units;
        p->energy_grid = (int)std::min<int64_t>(296, std::max<int64_t>(1, nblk(p->epart_n, 2048)));
        CK(cudaMalloc((void **)&p->d_epart, SAA_ENERGY_PARTS * p->epart_n * sizeof(double)));
        CK(cudaMemset(p->d_epart, 0, SAA_ENERGY_PARTS * p->epart_n * sizeof(double)));
        CK(cudaMalloc((void **)&p->d_estage, SAA_ENERGY_PARTS * p->energy_grid * sizeof(double)));
        CK(cudaMalloc((void **)&p->d_eticket, sizeof(unsigned int)));
        CK(cudaMemset(p->d_eticket, 0, sizeof(unsigned int)));
        CK(cudaMalloc((void **)&p->d_energy, sizeof(SaaEnergyDev)));
    }
    CK(cudaMalloc((void **)&p->d_ering, (size_t)capacity * SAA_ENERGY_FIELDS * sizeof(double)));
    SaaEnergyDev e{};
    e.arm = 1;
    e.every = every;
    e.first = (p->step_index + every - 1) / every;   // first recorded step is the next multiple of every
    e.cap = capacity;
    e.ring = p->d_ering;
    CK(cudaMemcpy(p->d_energy, &e, sizeof e, cudaMemcpyHostToDevice));
    p->energy_cap = capacity;
    p->energy_every = every;
    if (energy_prepare_predict(p)) return -1;
    return 0;
}
extern "C" int64_t saa_plan_energy_count(const saa_plan *p) { return p ? p->energy_count : -1; }
extern "C" int saa_plan_read_energy(saa_plan *p, int64_t first, int64_t count, double *out)
{
    NEED_FINAL(p, "saa_plan_read_energy");
    if (first < 0 || count < 0 || first + count > p->energy_count) return fail("saa_plan_read_energy: range out of bounds");
    if (first < p->energy_count - p->energy_cap) return fail("saa_plan_read_energy: records already overwritten");
    if (count > 0 && !out) return fail("saa_plan_read_energy: null output");
    CK(cudaSetDevice(p->device));
    CK(cudaStreamSynchronize(plan_stream(p)));
    for (int64_t s = 0; s < count;) {               // contiguous runs of the ring
        const int64_t slot = (first + s) % p->energy_cap;
        const int64_t run = std::min(count - s, p->energy_cap - slot);
        CK(cudaMemcpy(out + s * SAA_ENERGY_FIELDS, p->d_ering + slot * SAA_ENERGY_FIELDS, run * SAA_ENERGY_FIELDS * sizeof(double),
                      cudaMemcpyDeviceToHost));
        s += run;
    }
    return 0;
}

// ---- history / prediction ------------------------------------------------------------------------------
extern "C" int saa_plan_set_history(saa_plan *p, const int64_t *dofs, int64_t n_dofs, int64_t capacity, int64_t save_every)
{
    NEED_FINAL(p, "saa_plan_set_history");
    CK(cudaSetDevice(p->device));
    if (p->d_hist_rows) { cudaFree(p->d_hist_rows); p->d_hist_rows = nullptr; }
    if (p->d_hist) { cudaFree(p->d_hist); p->d_hist = nullptr; }
    p->hist_n = p->hist_cap = p->hist_count = 0;
    p->hook_epoch++;
    if (capacity <= 0) return 0;
    if (save_every <= 0) return fail("saa_plan_set_history: save_every must be positive");
    if (!dofs) n_dofs = p->n_dof;
    std::vector<int32_t> rows(n_dofs);
    for (int64_t i = 0; i < n_dofs; ++i) {
        int64_t d = dofs ? dofs[i] : i;
        if (d < 0 || d >= p->n_dof) return fail("saa_plan_set_history: DOF out of range");
        rows[i] = p->iperm_h[d];
    }
    if (upload(&p->d_hist_rows, rows)) return -1;
    CK(cudaMalloc((void **)&p->d_hist, (size_t)capacity * n_dofs * sizeof(double)));
    p->hist_n = n_dofs; p->hist_cap = capacity; p->hist_every = save_every;
    p->hook_h.hist_every = save_every; p->hook_h.hist_cap = capacity;
    p->hook_h.hist_first = (p->step_index + save_every - 1) / save_every;      // first recorded step is the next multiple of save_every
    p->hook_epoch++;
    CK(cudaMemcpyAsync(p->d_hook, &p->hook_h, sizeof(SaaHookDev), cudaMemcpyHostToDevice, plan_stream(p)));
    CK(cudaStreamSynchronize(plan_stream(p)));
    return 0;
}
extern "C" int64_t saa_plan_history_count(const saa_plan *p) { return p ? p->hist_count : -1; }
extern "C" int saa_plan_read_history(saa_plan *p, int64_t first, int64_t count, double *out)
{
    NEED_FINAL(p, "saa_plan_read_history");
    if (first < 0 || count < 0 || first + count > p->hist_count) return fail("saa_plan_read_history: range out of bounds");
    if (first < p->hist_count - p->hist_cap) return fail("saa_plan_read_history: snapshots already overwritten");
    CK(cudaSetDevice(p->device));
    CK(cudaStreamSynchronize(plan_stream(p)));
    for (int64_t s = 0; s < count; ++s) {
        const int64_t slot = (first + s) % p->hist_cap;
        CK(cudaMemcpy(out + s * p->hist_n, p->d_hist + slot * p->hist_n, p->hist_n * sizeof(double), cudaMemcpyDeviceToHost));
    }
    return 0;
}

extern "C" int saa_plan_read_history_dev(saa_plan *p, int64_t first, int64_t count, double *out)
{
    NEED_FINAL(p, "saa_plan_read_history_dev");
    if (first < 0 || count < 0 || first + count > p->hist_count) return fail("saa_plan_read_history_dev: range out of bounds");
    if (first < p->hist_count - p->hist_cap) return fail("saa_plan_read_history_dev: snapshots already overwritten");
    CK(cudaSetDevice(p->device));
    cudaStream_t st = plan_stream(p);
    for (int64_t s = 0; s < count;) {       // contiguous runs of the ring
        const int64_t slot = (first + s) % p->hist_cap;
        const int64_t run = std::min(count - s, p->hist_cap - slot);
        CK(cudaMemcpyAsync(out + s * p->hist_n, p->d_hist + slot * p->hist_n, run * p->hist_n * sizeof(double),
                           cudaMemcpyDeviceToDevice, st));
        s += run;
    }
    return 0;
}

extern "C" int saa_plan_set_prediction(saa_plan *p, const int64_t *dofs, int64_t n_dofs, const double *table_dev, int64_t n_rows)
{
    NEED_FINAL(p, "saa_plan_set_prediction");
    CK(cudaSetDevice(p->device));
    if (dofs) {
        if (p->d_pred_rows) { cudaFree(p->d_pred_rows); p->d_pred_rows = nullptr; }
        std::vector<int32_t> rows(n_dofs);
        for (int64_t i = 0; i < n_dofs; ++i) {
            if (dofs[i] < 0 || dofs[i] >= p->n_dof) return fail("saa_plan_set_prediction: DOF out of range");
            rows[i] = p->iperm_h[dofs[i]];
        }
        if (upload(&p->d_pred_rows, rows)) return -1;
        p->pred_n = n_dofs;
        p->pred_rows_h = rows;
        if (p->energy_cap > 0 && energy_prepare_predict(p)) return -1;
    } else if (n_dofs != p->pred_n) {
        return fail("saa_plan_set_prediction: n_dofs changed without a DOF list");
    }
    p->d_pred_table = table_dev; p->pred_rows = n_rows; p->pred_next = 0;
    p->hook_h.pred_table = table_dev; p->hook_h.pred_rows = n_rows; p->hook_h.pred_base_step = p->step_index;
    if (dofs) p->hook_epoch++;
    CK(cudaMemcpyAsync(p->d_hook, &p->hook_h, sizeof(SaaHookDev), cudaMemcpyHostToDevice, plan_stream(p)));
    CK(cudaStreamSynchronize(plan_stream(p)));      // hook_h is reused by the next call
    return 0;
}

// after a step: the new d0 is d_buf[cur]; the step read its clock from slot cur ^ 1.  Only kernels are enqueued here
// (graph-capturable); the host mirrors of the counters are advanced by count_step().
static void enqueue_hooks(saa_plan *p, cudaStream_t st, int mode)
{
    const SaaClock *clk_old = p->d_clk + (p->cur ^ 1);
    const bool energy = p->energy_cap > 0;
    if (mode == SAA_MODE_PREDICT && p->pred_n > 0) {                         // Online_predictor.py:298
        if (energy)
            saa_k_hook_scatter_energy<<<nblk(p->pred_n, 256), 256, 0, st>>>(p->D, p->H, p->pred_n, p->d_pred_rows, p->d_hook, clk_old,
                                                                            p->d_buf[p->cur], p->d_pred_stash, p->d_epred, p->epred_n);
        else
            saa_k_hook_scatter<<<nblk(p->pred_n, 256), 256, 0, st>>>(p->pred_n, p->d_pred_rows, p->d_hook, clk_old, p->d_buf[p->cur]);
        p->launches++;
    }
    if (p->hist_cap > 0 && p->hist_n > 0) {                                  // Data_prepare.py:238-240
        saa_k_hook_gather<<<nblk(p->hist_n, 256), 256, 0, st>>>(p->hist_n, p->d_hist_rows, p->d_hook, clk_old, p->d_buf[p->cur], p->d_hist);
        p->launches++;
    }
    if (energy) {
        // partials this step wrote: synchronised steps K1E over the interior slices + K3E units (contiguous), other
        // steps K1E over every slice (+ the prediction scatter's blocks)
        const bool sync = mode == SAA_MODE_SYNC && p->size > 1;
        const int64_t a0 = sync ? p->sh_slices : 0, na = (sync ? p->epart_n : p->n_slices) - a0;
        const bool pred = mode == SAA_MODE_PREDICT && p->pred_n > 0;
        saa_k_energy_reduce<<<p->energy_grid, 256, 0, st>>>(p->d_epart, p->epart_n, a0, na, p->d_epred, p->epred_n, 0, pred ? p->epred_n : 0,
                                                            p->d_estage, p->d_eticket, p->d_energy, clk_old, p->dt, p->dt2, p->alpha);
        p->launches++;
    }
}
static void count_step(saa_plan *p, int mode)
{
    if (mode == SAA_MODE_PREDICT) p->pred_next++;
    if (p->hist_cap > 0 && (p->step_index % p->hist_every) == 0) p->hist_count++;
    if (p->energy_cap > 0 && (p->step_index % p->energy_every) == 0) p->energy_count++;
    p->step_index++;
}
static int check_prediction(saa_plan *p, int mode, int64_t n_steps)
{
    if (mode != SAA_MODE_PREDICT) return 0;
    if (!p->d_pred_table && p->pred_n > 0) return fail("SAA_MODE_PREDICT: no prediction table set");
    if (p->hook_h.pred_base_step + p->pred_next != p->step_index) return fail("SAA_MODE_PREDICT: steps of another mode ran since the table was set; set it again");
    if (p->pred_next + n_steps > p->pred_rows) return fail("SAA_MODE_PREDICT: prediction table exhausted (%lld rows left, %lld steps asked)",
                                                            (long long)(p->pred_rows - p->pred_next), (long long)n_steps);
    return 0;
}
static int after_step(saa_plan *p, cudaStream_t st, int mode)
{
    if (check_prediction(p, mode, 1)) return -1;
    enqueue_hooks(p, st, mode);
    count_step(p, mode);
    return 0;
}

// ---- stepping --------------------------------------------------------------------------------------------
// instruction-schedule variants of the step kernel (same arithmetic, same bits): dot mode x minimum blocks per SM.
// Which one is fastest depends on the schedule ptxas happens to pick; profiles/r1/kernel_variants.md has the
// measurements behind the default.
static void launch_step_kernel(int variant, unsigned grid, cudaStream_t st, const SaaDev &D, const SaaHaloDev &H, const double *d0,
                               double *dn, const SaaClock *ci, SaaClock *co, int64_t slice_begin, unsigned max_waiters, unsigned count_sync)
{
    switch (variant) {
    case 0: saa_k_step<0, 6><<<grid, 256, 0, st>>>(D, H, d0, dn, ci, co, slice_begin, max_waiters, count_sync); break;
    case 1: saa_k_step<0, 4><<<grid, 256, 0, st>>>(D, H, d0, dn, ci, co, slice_begin, max_waiters, count_sync); break;
    case 2: saa_k_step<0, 3><<<grid, 256, 0, st>>>(D, H, d0, dn, ci, co, slice_begin, max_waiters, count_sync); break;
    case 3: saa_k_step<1, 6><<<grid, 256, 0, st>>>(D, H, d0, dn, ci, co, slice_begin, max_waiters, count_sync); break;
    case 5: saa_k_step<1, 3><<<grid, 256, 0, st>>>(D, H, d0, dn, ci, co, slice_begin, max_waiters, count_sync); break;
    default: saa_k_step<1, 4><<<grid, 256, 0, st>>>(D, H, d0, dn, ci, co, slice_begin, max_waiters, count_sync); break;
    }
}
template <int STAGES, int WARPS, int BR>
static void launch_stream(saa_plan *p, cudaStream_t st, const SaaDev &D, int64_t slice_begin, unsigned count_sync, bool advance_clock)
{
    const size_t smem = (size_t)WARPS * STAGES * SAA_STREAM_STAGE_BYTES(BR);
    cudaFuncSetAttribute(saa_k_step_stream<STAGES, WARPS, BR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);   // per device
    saa_k_step_stream<STAGES, WARPS, BR><<<p->n_sms, 32 * WARPS, smem, st>>>(D, p->d_buf[p->cur], p->d_buf[p->cur ^ 1], p->d_clk + p->cur,
                                                                       advance_clock ? p->d_clk + (p->cur ^ 1) : nullptr, slice_begin, count_sync);
    p->launches++;
}
// K1 only: slices [slice_begin, n_slices) as interior rows (no interface handling inside the kernel)
static void launch_interior(saa_plan *p, cudaStream_t st, int64_t slice_begin, unsigned count_sync, bool advance_clock, int64_t slice_end = -1,
                            bool predict = false)
{
    SaaDev D = p->D;
    D.sh_slices = 0;
    if (slice_end < 0) slice_end = p->n_slices;
    if (p->energy_cap > 0) {       // K1E (also for the cp.async variant: its full-plane layout is a layout with pmask = 0x1FF)
        const unsigned n_main = std::max(1u, nblk(slice_end - slice_begin, SAA_WARPS_PER_BLOCK));
        const bool skip = predict && p->pred_n > 0;
        saa_k_step_energy<1><<<n_main, 256, 0, st>>>(D, p->H, p->d_buf[p->cur], p->d_buf[p->cur ^ 1], p->d_clk + p->cur,
                                                     advance_clock ? p->d_clk + (p->cur ^ 1) : nullptr, slice_begin, count_sync,
                                                     p->d_epart, p->epart_n, skip ? p->d_pred_skip : nullptr, p->d_pred_stash);
        p->launches++;
        return;
    }
    if (p->kvariant >= 6 && p->n_slices > slice_begin) {       // cp.async streaming kernels, persistent grid
        launch_stream<3, 24, 1>(p, st, D, slice_begin, count_sync, advance_clock);   // the fastest streaming configuration measured
        return;
    }
    // slices [slice_begin, slice_end): slice_end - slice_begin is a multiple of the warps per block unless slice_end = n_slices
    const unsigned n_main = std::max(1u, nblk(slice_end - slice_begin, SAA_WARPS_PER_BLOCK));
    launch_step_kernel(p->kvariant, n_main, st, D, p->H, p->d_buf[p->cur], p->d_buf[p->cur ^ 1], p->d_clk + p->cur,
                       advance_clock ? p->d_clk + (p->cur ^ 1) : nullptr, slice_begin, 0u, count_sync);
    p->launches++;
}

static void launch_local_step(saa_plan *p, cudaStream_t st, bool predict = false)
{
    if (p->matfree) {
        const unsigned g = std::max(1u, nblk(p->n_slices, SAA_WARPS_PER_BLOCK));
        // register budget = occupancy of the gather-latency-bound kernel (SAA_MF_MINB: blocks per SM; measured in profiles/)
        switch (p->mf_minb) {
        case 3: saa_k_step_matfree<3><<<g, 256, 0, st>>>(p->D, p->MF, p->d_buf[p->cur], p->d_buf[p->cur ^ 1], p->d_clk + p->cur, p->d_clk + (p->cur ^ 1)); break;
        case 5: saa_k_step_matfree<5><<<g, 256, 0, st>>>(p->D, p->MF, p->d_buf[p->cur], p->d_buf[p->cur ^ 1], p->d_clk + p->cur, p->d_clk + (p->cur ^ 1)); break;
        case 6: saa_k_step_matfree<6><<<g, 256, 0, st>>>(p->D, p->MF, p->d_buf[p->cur], p->d_buf[p->cur ^ 1], p->d_clk + p->cur, p->d_clk + (p->cur ^ 1)); break;
        default: saa_k_step_matfree<4><<<g, 256, 0, st>>>(p->D, p->MF, p->d_buf[p->cur], p->d_buf[p->cur ^ 1], p->d_clk + p->cur, p->d_clk + (p->cur ^ 1)); break;
        }
        p->launches++;
    } else {
        launch_interior(p, st, 0, 0u, true, -1, predict);
    }
    p->cur ^= 1;
}

static bool needs_hooks(const saa_plan *p, int mode) { return mode == SAA_MODE_PREDICT || p->hist_cap > 0 || p->energy_cap > 0; }

// one step of `mode` (local / predict / peer-synchronised) with its hooks: kernels only
static void launch_peer_step(saa_plan *p, cudaStream_t st);
static void enqueue_step_with_hooks(saa_plan *p, cudaStream_t st, int mode)
{
    if (mode == SAA_MODE_SYNC) launch_peer_step(p, st);
    else launch_local_step(p, st, mode == SAA_MODE_PREDICT);
    enqueue_hooks(p, st, mode);
}
// steps with history / prediction hooks, replayed two at a time from a CUDA graph (the hooks take their row / slot
// from the device clock, the table pointer from the device hook state: nothing in the graph changes between replays)
static int step_hook_graph(saa_plan *p, int64_t n_steps, int mode)
{
    cudaStream_t st = p->stream;
    int64_t done = 0;
    saa_plan::StepGraph *g = nullptr;
    const int c0 = p->cur;
    for (auto &q : p->step_graphs)
        if (q.mode == mode && q.cur == c0 && q.epoch == p->hook_epoch) g = &q;
    if (!g) {
        for (size_t i = 0; i < p->step_graphs.size();)                       // drop graphs of older hook configurations
            if (p->step_graphs[i].epoch != p->hook_epoch) { cudaGraphExecDestroy(p->step_graphs[i].exec); p->step_graphs.erase(p->step_graphs.begin() + i); }
            else ++i;
        cudaGraph_t graph;
        CK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
        const int64_t l0 = p->launches;
        enqueue_step_with_hooks(p, st, mode);
        enqueue_step_with_hooks(p, st, mode);
        const int per = (int)(p->launches - l0);
        p->launches = l0;
        CK(cudaStreamEndCapture(st, &graph));
        saa_plan::StepGraph q{mode, c0, p->hook_epoch, nullptr, per};
        CK(cudaGraphInstantiate(&q.exec, graph, 0));
        CK(cudaGraphDestroy(graph));
        p->step_graphs.push_back(q);
        g = &p->step_graphs.back();
    }
    for (; done + 2 <= n_steps; done += 2) {
        CK(cudaGraphLaunch(g->exec, st));
        p->launches += g->launches;
        count_step(p, mode);
        count_step(p, mode);
    }
    for (; done < n_steps; ++done) {
        enqueue_step_with_hooks(p, st, mode);
        count_step(p, mode);
    }
    CK(cudaGetLastError());
    return 0;
}

// Two consecutive steps (LOCAL, or peer-synchronised) starting at the current buffer parity as an instantiated,
// uploaded CUDA graph.  Capture enqueues nothing, so this is also done ahead of time for BOTH parities
// (prepare_graphs, at finalize / peer attach): the first saa_plan_step call then costs what every later one does.
static void launch_peer_step(saa_plan *p, cudaStream_t st);
static int capture_two_steps(saa_plan *p, bool peer)
{
    cudaStream_t st = p->stream;
    cudaGraphExec_t *slot = peer ? &p->graph_peer[p->cur] : &p->graph_exec[p->cur];
    if (*slot) return 0;
    cudaGraph_t g;
    const int64_t energy_cap = p->energy_cap;
    p->energy_cap = 0;                               // these graphs run only while no hook is set: never the monitor's kernels
    CK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    const int64_t l0 = p->launches;
    for (int i = 0; i < 2; ++i) {
        if (peer) launch_peer_step(p, st);
        else launch_local_step(p, st);
    }
    p->launches = l0;
    p->energy_cap = energy_cap;
    CK(cudaStreamEndCapture(st, &g));
    CK(cudaGraphInstantiate(slot, g, 0));
    CK(cudaGraphDestroy(g));
    CK(cudaGraphUpload(*slot, st));
    return 0;
}
static int prepare_graphs(saa_plan *p, bool peer)
{
    if (p->kvariant >= 6) return 0;                  // the streaming variant sets a function attribute at launch: captured lazily
    for (int i = 0; i < 2; ++i) {
        if (capture_two_steps(p, peer)) return -1;
        p->cur ^= 1;                                 // the same two steps for the other buffer parity
    }
    CK(cudaStreamSynchronize(p->stream));
    return 0;
}

static int step_local(saa_plan *p, int64_t n_steps, int mode, int launch)
{
    cudaStream_t st = p->stream;
    const bool hooks = needs_hooks(p, mode);
    if (launch == SAA_LAUNCH_AUTO) launch = (n_steps >= 2 ? SAA_LAUNCH_GRAPH : SAA_LAUNCH_PER_STEP);   // graphs exist since finalize
    if (p->energy_cap > 0 && launch == SAA_LAUNCH_PERSISTENT)
        return fail("saa_plan_step: the energy monitor is not available in the persistent loop (disarm it, or use per-step or graph launches)");
    if (hooks && launch == SAA_LAUNCH_PERSISTENT) return fail("history / prediction hooks are not available in the persistent loop");
    if (p->matfree && launch == SAA_LAUNCH_PERSISTENT) return fail("the matrix-free kernel has no persistent form");
    if (check_prediction(p, mode, n_steps)) return -1;
    if (hooks && launch == SAA_LAUNCH_GRAPH && n_steps >= 2) return step_hook_graph(p, n_steps, mode);
    if (launch == SAA_LAUNCH_PERSISTENT) {
        if (p->coop_blocks <= 0) return fail("cooperative launch not available");
        double *a = p->d_buf[p->cur], *b = p->d_buf[p->cur ^ 1];
        SaaClock *tn = p->d_clk + p->cur;
        int64_t ns = n_steps;
        void *args[] = {&p->D, &a, &b, &tn, &ns};
        int64_t want = (p->n_slices + SAA_WARPS_PER_BLOCK - 1) / SAA_WARPS_PER_BLOCK;
        int blocks = (int)std::min<int64_t>(p->coop_blocks, want);
        CK(cudaLaunchCooperativeKernel((void *)saa_k_persistent, dim3(blocks), dim3(32 * SAA_WARPS_PER_BLOCK), args, 0, st));
        p->launches++;
        if (n_steps & 1) {   // an odd number of steps swaps the buffer roles; tn was written back to d_tn[cur]
            CK(cudaMemcpyAsync(p->d_clk + (p->cur ^ 1), p->d_clk + p->cur, sizeof(SaaClock), cudaMemcpyDeviceToDevice, st));
            p->cur ^= 1;
        }
        p->step_index += n_steps;
        return 0;
    }
    int64_t done = 0;
    if (launch == SAA_LAUNCH_GRAPH && n_steps >= 2) {
        const int c = p->cur;
        if (!p->graph_exec[c] && capture_two_steps(p, false)) return -1;
        for (; done + 2 <= n_steps; done += 2) {
            CK(cudaGraphLaunch(p->graph_exec[c], st));
            p->launches += 2;
        }
        p->step_index += done;
    }
    for (; done < n_steps; ++done) {
        launch_local_step(p, st, mode == SAA_MODE_PREDICT);
        enqueue_hooks(p, st, mode);
        count_step(p, mode);
    }
    CK(cudaGetLastError());
    return 0;
}

// one synchronised step of one plan, split in its three phases so that transports can interleave
static inline bool use_peer(const saa_plan *p) { return p->peer && !(p->prefer_nccl && p->comm); }
static void sync_phase_boundary(saa_plan *p, cudaStream_t st)
{
    if (p->sh_slices > 0) {
        if (use_peer(p))
            saa_k_boundary<true><<<nblk(p->sh_slices, SAA_WARPS_PER_BLOCK), 32 * SAA_WARPS_PER_BLOCK, 0, st>>>(p->D, p->Hp, p->d_buf[p->cur], p->d_clk + p->cur);
        else
            saa_k_boundary<false><<<nblk(p->sh_slices, SAA_WARPS_PER_BLOCK), 32 * SAA_WARPS_PER_BLOCK, 0, st>>>(p->D, p->H, p->d_buf[p->cur], p->d_clk + p->cur);
        p->launches++;
    }
}
static void sync_phase_interior(saa_plan *p, cudaStream_t st)
{
    // also advances the clock; runs even with zero interior slices so that tn moves
    launch_interior(p, st, p->sh_slices, 1u, true);
}
static void sync_phase_shared(saa_plan *p, cudaStream_t st)
{
    if (p->sh_slices > 0) {
        if (p->energy_cap > 0) {   // K3E: partials of the units of 256 shared rows after the slices' ones
            if (use_peer(p))
                saa_k_shared_update_energy<true><<<nblk(p->H.sh_rows, 256), 256, 0, st>>>(p->D, p->Hp, p->d_buf[p->cur], p->d_buf[p->cur ^ 1], p->d_clk + p->cur,
                                                                                         p->d_epart, p->epart_n, p->n_slices);
            else
                saa_k_shared_update_energy<false><<<nblk(p->H.sh_rows, 256), 256, 0, st>>>(p->D, p->H, p->d_buf[p->cur], p->d_buf[p->cur ^ 1], p->d_clk + p->cur,
                                                                                          p->d_epart, p->epart_n, p->n_slices);
        } else if (use_peer(p))
            saa_k_shared_update<true><<<nblk(p->H.sh_rows, 256), 256, 0, st>>>(p->D, p->Hp, p->d_buf[p->cur], p->d_buf[p->cur ^ 1], p->d_clk + p->cur);
        else
            saa_k_shared_update<false><<<nblk(p->H.sh_rows, 256), 256, 0, st>>>(p->D, p->H, p->d_buf[p->cur], p->d_buf[p->cur ^ 1], p->d_clk + p->cur);
        p->launches++;
    }
    p->cur ^= 1;
}

// the neighbour messages of one synchronised step through NCCL (grouped send / receive pairs on the plan's stream)
static int nccl_exchange(saa_plan *p, cudaStream_t st)
{
    const int n_nb = (int)p->nb_rank.size();
    if (n_nb > 0) {
        NCK(g_nccl.GroupStart());
        for (int k = 0; k < n_nb; ++k) {
            const size_t cnt = (size_t)(p->msg_off[k + 1] - p->msg_off[k]);
            NCK(g_nccl.Send(p->d_send + p->msg_off[k], cnt, SAA_NCCL_DOUBLE, p->nb_rank[k], p->comm, st));
            NCK(g_nccl.Recv(p->d_recv + p->msg_off[k], cnt, SAA_NCCL_DOUBLE, p->nb_rank[k], p->comm, st));
        }
        NCK(g_nccl.GroupEnd());
    }
    return 0;
}

static int step_sync_nccl(saa_plan *p, int64_t n_steps)
{
    cudaStream_t st = p->stream;
    for (int64_t s = 0; s < n_steps; ++s) {
        sync_phase_boundary(p, st);
        if (nccl_exchange(p, st)) return -1;
        sync_phase_interior(p, st);
        sync_phase_shared(p, st);
        if (after_step(p, st, SAA_MODE_SYNC)) return -1;
    }
    CK(cudaGetLastError());
    return 0;
}

// peer transport: three stream-ordered kernels per step, no host involvement -> replayed from a two-step graph
static void launch_peer_step(saa_plan *p, cudaStream_t st)
{
    if (p->peer_fused && p->sh_slices > 0 && p->energy_cap == 0) {     // the monitor has no fused form: three kernels
        // n_main slice blocks + one tail block per unit of 256 shared rows; at most one WAITING tail block per SM (every
        // schedule variant keeps >= 3 blocks per SM resident), so blocks that have not started always find a slot
        const unsigned n_main = nblk(p->n_slices, SAA_WARPS_PER_BLOCK);
        const unsigned n_units = nblk(p->H.sh_rows, 256);
        const unsigned waiters = std::max(1u, std::min(n_units, (unsigned)p->n_sms));
        launch_step_kernel(p->kvariant, n_main + n_units, st, p->D, p->Hp, p->d_buf[p->cur], p->d_buf[p->cur ^ 1], p->d_clk + p->cur,
                           p->d_clk + (p->cur ^ 1), 0, waiters, 1u);
        p->launches++;
        p->cur ^= 1;
        return;
    }
    sync_phase_boundary(p, st);
    sync_phase_interior(p, st);
    sync_phase_shared(p, st);
}

static int step_sync_peer(saa_plan *p, int64_t n_steps, int launch)
{
    cudaStream_t st = p->stream;
    const bool hooks = p->hist_cap > 0 || p->energy_cap > 0;
    int64_t done = 0;
    if (launch == SAA_LAUNCH_PERSISTENT) {
        // one cooperative launch for all n_steps synchronised steps (small shards: no launch per step); every rank must
        // make the same call, like any synchronised step
        if (p->energy_cap > 0)
            return fail("saa_plan_step: the energy monitor is not available in the persistent loop (disarm it, or use per-step or graph launches)");
        if (hooks) return fail("history hooks are not available in the persistent loop");
        if (p->coop_blocks_sync <= 0) return fail("cooperative launch not available");
        if (p->sh_slices == 0) return fail("saa_plan_step: the persistent synchronised loop needs an interface (this rank has none)");
        double *a = p->d_buf[p->cur], *b = p->d_buf[p->cur ^ 1];
        SaaClock *clk = p->d_clk + p->cur;
        int64_t ns = n_steps;
        void *args[] = {&p->D, &p->Hp, &a, &b, &clk, &ns};
        const int64_t want = (p->n_slices + SAA_WARPS_PER_BLOCK - 1) / SAA_WARPS_PER_BLOCK;
        const int blocks = (int)std::min<int64_t>(p->coop_blocks_sync, want);
        CK(cudaLaunchCooperativeKernel((void *)saa_k_persistent_sync, dim3(blocks), dim3(32 * SAA_WARPS_PER_BLOCK), args, 0, st));
        p->launches++;
        if (n_steps & 1) {   // an odd number of steps swaps the buffer roles; the clock was written back to slot cur
            CK(cudaMemcpyAsync(p->d_clk + (p->cur ^ 1), p->d_clk + p->cur, sizeof(SaaClock), cudaMemcpyDeviceToDevice, st));
            p->cur ^= 1;
        }
        p->step_index += n_steps;
        return 0;
    }
    if (hooks && launch != SAA_LAUNCH_PER_STEP && n_steps >= 2) return step_hook_graph(p, n_steps, SAA_MODE_SYNC);
    if (!hooks && launch != SAA_LAUNCH_PER_STEP && n_steps >= 2) {
        const int c = p->cur;
        if (!p->graph_peer[c] && capture_two_steps(p, true)) return -1;
        const int per = (p->sh_slices > 0 ? (p->peer_fused ? 1 : 3) : 1) * 2;
        for (; done + 2 <= n_steps; done += 2) {
            CK(cudaGraphLaunch(p->graph_peer[c], st));
            p->launches += per;
        }
        p->step_index += done;
    }
    for (; done < n_steps; ++done) {
        launch_peer_step(p, st);
        if (after_step(p, st, SAA_MODE_SYNC)) return -1;
    }
    CK(cudaGetLastError());
    return 0;
}

extern "C" int saa_plan_step(saa_plan *p, int64_t n_steps, int mode, int launch)
{
    NEED_FINAL(p, "saa_plan_step");
    if (n_steps < 0) return fail("saa_plan_step: negative n_steps");
    if (n_steps == 0) return 0;
    if (p->group) return fail("saa_plan_step: this plan belongs to a group; use saa_group_step");
    CK(cudaSetDevice(p->device));
    p->state_epoch++;
    if (mode == SAA_MODE_LOCAL || mode == SAA_MODE_PREDICT) return step_local(p, n_steps, mode, launch);
    if (mode == SAA_MODE_SYNC) {
        if (p->size == 1) return step_local(p, n_steps, SAA_MODE_LOCAL, launch);   // Dynamic_solver.py:25 `if size != 1`
        if (p->group) return fail("saa_plan_step: this plan belongs to a group; use saa_group_step");
        if (p->peer && !(p->prefer_nccl && p->comm)) return step_sync_peer(p, n_steps, launch);
        if (!p->comm) return fail("saa_plan_step: SAA_MODE_SYNC needs a transport (saa_plan_peer_attach, saa_plan_init_nccl or saa_group_create)");
        return step_sync_nccl(p, n_steps);
    }
    return fail("saa_plan_step: unknown mode %d", mode);
}

extern "C" int saa_plan_set_option(saa_plan *p, int option, int value)
{
    NEED_FINAL(p, "saa_plan_set_option");
    CK(cudaSetDevice(p->device));
    CK(cudaStreamSynchronize(plan_stream(p)));
    if (option == SAA_OPT_PEER_FUSED) {
        if ((value != 0) == p->peer_fused) return 0;
        p->peer_fused = value != 0;
        for (int i = 0; i < 2; ++i)
            if (p->graph_peer[i]) { cudaGraphExecDestroy(p->graph_peer[i]); p->graph_peer[i] = nullptr; }
        p->hook_epoch++;                                 // graphs of hooked synchronised steps hold the old form too
        return p->peer ? prepare_graphs(p, true) : 0;
    }
    if (option == SAA_OPT_MATFREE) {
        if (value && p->energy_cap > 0)
            return fail("saa_plan_set_option: the energy monitor is armed; the matrix-free kernel (SAA_OPT_MATFREE) computes a different force and has no energy form");
        if (value && !p->d_mf_inc) return fail("saa_plan_set_option: SAA_OPT_MATFREE needs saa_plan_set_matfree_dev first");
        if (!value && !p->d_val) return fail("saa_plan_set_option: the assembled matrix of this plan was released (SAA_OPT_MATFREE = 2)");
        if (value == 2 && p->d_val) {                    // release the assembled matrix: the plan is matrix-free for good
            if (p->size > 1) return fail("saa_plan_set_option: SAA_OPT_MATFREE = 2 is for single-partition plans (synchronised steps stream the matrix)");
            cudaFree(p->d_val); cudaFree(p->d_col); cudaFree(p->d_vbase);
            p->d_val = nullptr; p->d_col = nullptr; p->d_vbase = nullptr; p->D.val = nullptr; p->D.col = nullptr; p->D.vbase = nullptr;
        }
        if ((value != 0) == p->matfree) return 0;
        p->matfree = value != 0;
        for (int i = 0; i < 2; ++i)
            if (p->graph_exec[i]) { cudaGraphExecDestroy(p->graph_exec[i]); p->graph_exec[i] = nullptr; }
        p->hook_epoch++;
        return prepare_graphs(p, false);
    }
    if (option == SAA_OPT_PREFER_NCCL) {
        if (value && !p->comm) return fail("saa_plan_set_option: SAA_OPT_PREFER_NCCL needs saa_plan_init_nccl first");
        p->prefer_nccl = value != 0;
        return 0;
    }
    return fail("saa_plan_set_option: unknown option %d", option);
}

extern "C" int saa_plan_synchronize(saa_plan *p)
{
    NEED_FINAL(p, "saa_plan_synchronize");
    CK(cudaSetDevice(p->device));
    CK(cudaStreamSynchronize(plan_stream(p)));
    if (p->peer && p->d_done) {
        unsigned int err = 0;
        CK(cudaMemcpy(&err, p->d_done + 1, sizeof err, cudaMemcpyDeviceToHost));
        if (err) return fail("saa_plan_synchronize: a wait for a neighbour's halo message expired (ranks out of step?)");
    }
    return 0;
}

// ---- pipelined host call ------------------------------------------------------------------------------------------
// The reference-facing call moves d0 up and d1 down over PCIe around ONE step; done one after the other that is
// upload + step + download.  PCIe is full duplex and a row of the step only needs the d0 entries of its own column
// window, so the call is cut into K chunks of EXTERNAL rows and run as a three-stage pipeline on three streams:
//   upload  c : rows [row_off[c], row_off[c+1]) of d0 (and dn) -> staging -> internal order            (stream s_in)
//   compute c : internal slices [slice_end[c-1], slice_end[c]) — every slice holding a row of the chunks <= c —
//               after the uploads of all chunks its rows and column nodes live in (need_upload[c])     (plan stream)
//   download c: rows of chunk c of d1 -> external order -> host, after compute c                        (stream s_out)
// Same kernels on the same data, every row computed exactly once: same bits as the plain call.  With a layout whose
// column windows span everything (random node order) need_upload = K-1 and it degenerates to upload-all-then-compute.
// Synchronised steps of a multi-partition plan (table 1) chunk the INTERIOR slices the same way; the boundary slices
// (K2: partial forces -> neighbours) are launched as soon as the chunks they read have arrived, the shared-row update
// (K3) after the last interior chunk, and the chunks that hold shared rows are downloaded after it.
__global__ void saa_k_hp_inverse(int64_t n_ext_nodes, const int32_t *__restrict__ iperm, int32_t *__restrict__ ext_of_int)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < n_ext_nodes) ext_of_int[iperm[3 * e] / 3] = (int32_t)e;
}
// per slice: largest external node among its own nodes and among own + column nodes of its blocks (-1: all-padding slice)
__global__ void saa_k_hp_slice_reach(SaaDev P, const int32_t *__restrict__ ext_of_int, int32_t *__restrict__ reach_own, int32_t *__restrict__ reach_col)
{
    const int lane = threadIdx.x & 31;
    const int64_t slice = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (slice >= P.n_slices) return;
    const int32_t own = ext_of_int[slice * 32 + lane];
    int32_t mc = own;
    if (own >= 0) {                                              // padding lanes point at themselves
        const int64_t beg = P.slice_ptr[slice];
        const int len = (int)((P.slice_ptr[slice + 1] - beg) >> 5);
        for (int j = 0; j < len; ++j) mc = max(mc, ext_of_int[P.col[beg + 32 * j + lane]]);
    }
    int32_t mo = own;
    for (int o = 16; o > 0; o >>= 1) {
        mo = max(mo, __shfl_xor_sync(0xffffffffu, mo, o));
        mc = max(mc, __shfl_xor_sync(0xffffffffu, mc, o));
    }
    if (lane == 0) { reach_own[slice] = mo; reach_col[slice] = mc; }
}

// table 0: every slice as an interior slice (local steps); table 1: synchronised steps of a plan with an interface
static int host_pipe_build(saa_plan *p, int table)
{
    saa_plan::HostPipe &h = p->hp[table];
    h.state = -1;
    const char *env = getenv("SAA_STEP_HOST_PIPELINE");
    if (env && env[0] == '0') { h.state = 0; return 0; }        // switched off for now: decide again at the next call
    const int64_t nn = p->n_dof / 3;
    int K = (int)std::min<int64_t>(32, (p->n_dof * 8) / (2 << 20));      // chunks of at least 2 MiB (below that the launches cost more than the overlap gains)
    if (env && atoi(env) > 1) K = (int)std::min<int64_t>(std::min(atoi(env), 64), nn);
    if (K < 2) return 0;
    const int64_t sb = table == 1 ? p->sh_slices : 0;            // first slice handled as an interior slice
    DevBuf inv, r_own, r_col;
    const int64_t n_int = p->n_rows / 3;
    if (inv.alloc(n_int * sizeof(int32_t)) || r_own.alloc(p->n_slices * sizeof(int32_t)) || r_col.alloc(p->n_slices * sizeof(int32_t))) return -1;
    CK(cudaMemset(inv.p, 0xff, n_int * sizeof(int32_t)));                // -1: padding node
    saa_k_hp_inverse<<<nblk(nn, 256), 256>>>(nn, p->d_iperm, inv.as<int32_t>());
    saa_k_hp_slice_reach<<<nblk(p->n_slices, SAA_WARPS_PER_BLOCK), 32 * SAA_WARPS_PER_BLOCK>>>(p->D, inv.as<int32_t>(), r_own.as<int32_t>(), r_col.as<int32_t>());
    CK(cudaGetLastError());
    std::vector<int32_t> own(p->n_slices), col(p->n_slices);
    CK(cudaMemcpy(own.data(), r_own.p, p->n_slices * sizeof(int32_t), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(col.data(), r_col.p, p->n_slices * sizeof(int32_t), cudaMemcpyDeviceToHost));
    // chunks of external nodes of equal size
    std::vector<int64_t> node_off(K + 1);
    for (int c = 0; c <= K; ++c) node_off[c] = (nn * c) / K;
    auto chunk_of = [&](int64_t e) { return (int)(std::upper_bound(node_off.begin(), node_off.end(), e) - node_off.begin()) - 1; };
    // compute chunk c must cover every interior slice that holds an external node of the chunks <= c: attribute each slice
    // to the chunk of its SMALLEST external node (the earliest download that needs it) and take running maxima
    h.first_slice = sb;
    h.slice_end.assign(K, 0);
    h.need_upload.assign(K, 0);
    h.has_shared.assign(K, 0);
    h.need_boundary = -1;
    std::vector<int32_t> min_own(p->n_slices, INT32_MAX);
    for (int64_t e = 0; e < nn; ++e) {
        const int64_t s = (p->iperm_h[3 * e] / 3) >> 5;
        min_own[s] = std::min<int32_t>(min_own[s], (int32_t)e);
        if (s < sb) h.has_shared[chunk_of(e)] = 1;
    }
    std::vector<int64_t> last_slice(K, -1);
    for (int64_t s = sb; s < p->n_slices; ++s)
        if (own[s] >= 0) {
            const int c = chunk_of(min_own[s]);
            last_slice[c] = std::max(last_slice[c], s);
        }
    int64_t run = sb;
    for (int c = 0; c < K; ++c) {
        run = std::max(run, last_slice[c] + 1);
        // ranges start at sb and have a whole number of thread blocks' worth of slices, except the last one
        const int64_t end = (c == K - 1) ? p->n_slices
                                         : std::min<int64_t>(p->n_slices, sb + (run - sb + SAA_WARPS_PER_BLOCK - 1) / SAA_WARPS_PER_BLOCK * SAA_WARPS_PER_BLOCK);
        h.slice_end[c] = end;
        run = end;
    }
    for (int64_t s = sb; s < p->n_slices; ++s)                   // every slice is finished before the first download that reads it
        if (own[s] >= 0 && s >= h.slice_end[chunk_of(min_own[s])]) return fail("host_pipe_build: inconsistent chunk table");
    for (int c = 0; c < K; ++c) {
        int32_t reach = -1;
        for (int64_t s = (c ? h.slice_end[c - 1] : sb); s < h.slice_end[c]; ++s) reach = std::max(reach, col[s]);
        h.need_upload[c] = std::max(reach >= 0 ? chunk_of(reach) : 0, c ? h.need_upload[c - 1] : 0);
    }
    if (sb > 0) {
        int32_t reach = -1;
        for (int64_t s = 0; s < sb; ++s) reach = std::max(reach, col[s]);
        h.need_boundary = reach >= 0 ? chunk_of(reach) : 0;
    }
    h.row_off.resize(K + 1);
    for (int c = 0; c <= K; ++c) h.row_off[c] = 3 * node_off[c];
    if (!p->hp_s_in) {
        CK(cudaStreamCreateWithFlags(&p->hp_s_in, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&p->hp_s_out, cudaStreamNonBlocking));
    }
    while ((int)p->hp_ev_up.size() < K) {
        cudaEvent_t a, b;
        CK(cudaEventCreateWithFlags(&a, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&b, cudaEventDisableTiming));
        p->hp_ev_up.push_back(a); p->hp_ev_cmp.push_back(b);
    }
    CK(cudaDeviceSynchronize());
    h.state = 1;
    return 0;
}

static int host_pipe_step(saa_plan *p, int table, const double *d0, const double *dn, double tn, double *d1, bool keep_dn)
{
    saa_plan::HostPipe &h = p->hp[table];
    const int K = (int)h.slice_end.size();
    const bool sync = table == 1;
    const unsigned count_sync = sync ? 1u : 0u;
    cudaStream_t st = p->stream, s_in = p->hp_s_in, s_out = p->hp_s_out;
    CK(cudaStreamSynchronize(st));                               // earlier work of the plan (other entry points use this stream)
    p->state_epoch += 2;                                         // state upload + step, like the plain call
    CK(cudaMemcpyAsync(&p->d_clk[p->cur].tn, &tn, sizeof(double), cudaMemcpyHostToDevice, s_in));
    double *b0 = p->d_buf[p->cur], *b1 = p->d_buf[p->cur ^ 1];
    double *stage_dn = p->d_stage + p->n_dof, *stage_out = p->d_stage + 2 * p->n_dof;
    // stage 1: the copies of all chunks back to back on s_in (nothing but copies on the copy streams: a kernel between
    // two copies of a stream leaves the PCIe link idle for the kernel and two dependency hand-overs)
    for (int c = 0; c < K; ++c) {
        const int64_t off = h.row_off[c], cnt = h.row_off[c + 1] - off;
        CK(cudaMemcpyAsync(p->d_stage + off, d0 + off, cnt * sizeof(double), cudaMemcpyHostToDevice, s_in));
        if (!keep_dn) CK(cudaMemcpyAsync(stage_dn + off, dn + off, cnt * sizeof(double), cudaMemcpyHostToDevice, s_in));
        CK(cudaEventRecord(p->hp_ev_up[c], s_in));
    }
    // stage 2 on the plan's stream: caller order -> internal order of the chunks as they arrive, the step slice range by
    // slice range, internal -> caller order of the finished rows;  stage 3: their copies back to back on s_out
    int arrived = -1;
    auto take_uploads = [&](int upto) -> int {
        for (int c = arrived + 1; c <= upto; ++c) {
            const int64_t off = h.row_off[c], cnt = h.row_off[c + 1] - off;
            CK(cudaStreamWaitEvent(st, p->hp_ev_up[c], 0));
            saa_k_scatter_to_internal<<<nblk(cnt, 256), 256, 0, st>>>(cnt, p->d_iperm + off, p->d_stage + off, b0);
            if (!keep_dn) saa_k_scatter_to_internal<<<nblk(cnt, 256), 256, 0, st>>>(cnt, p->d_iperm + off, stage_dn + off, b1);
            p->launches += keep_dn ? 1 : 2;
        }
        arrived = std::max(arrived, upto);
        return 0;
    };
    auto download = [&](int c) -> int {
        const int64_t off = h.row_off[c], cnt = h.row_off[c + 1] - off;
        saa_k_gather_to_external<<<nblk(cnt, 256), 256, 0, st>>>(cnt, p->d_iperm + off, b1, stage_out + off);
        p->launches++;
        CK(cudaEventRecord(p->hp_ev_cmp[c], st));
        CK(cudaStreamWaitEvent(s_out, p->hp_ev_cmp[c], 0));
        CK(cudaMemcpyAsync(d1 + off, stage_out + off, cnt * sizeof(double), cudaMemcpyDeviceToHost, s_out));
        return 0;
    };
    bool boundary_done = !(sync && p->sh_slices > 0);
    for (int c = 0; c < K; ++c) {
        if (!boundary_done && (h.need_upload[c] >= h.need_boundary || c == K - 1)) {
            if (take_uploads(h.need_boundary)) return -1;
            sync_phase_boundary(p, st);                          // K2: partial forces of the shared rows -> neighbours
            if (!use_peer(p) && nccl_exchange(p, st)) return -1;
            boundary_done = true;
        }
        if (take_uploads(h.need_upload[c])) return -1;
        const int64_t s0 = c ? h.slice_end[c - 1] : h.first_slice, s1 = h.slice_end[c];
        if (s1 > s0) launch_interior(p, st, s0, count_sync, c == 0, s1);
        else if (c == 0) launch_interior(p, st, p->n_slices, count_sync, true, p->n_slices);   // no slice, the clock only
        if (!(sync && h.has_shared[c]) && download(c)) return -1;
    }
    if (take_uploads(K - 1)) return -1;                          // the whole state is resident afterwards, whatever the step read
    if (sync) {
        sync_phase_shared(p, st);                                // K3: rank-ordered sums + update of the shared rows; swaps the levels
        for (int c = 0; c < K; ++c)
            if (h.has_shared[c] && download(c)) return -1;
    } else {
        p->cur ^= 1;
    }
    CK(cudaGetLastError());
    p->step_index++;
    CK(cudaStreamSynchronize(s_out));
    CK(cudaStreamSynchronize(st));
    CK(cudaStreamSynchronize(s_in));
    return 0;
}

extern "C" int saa_plan_host_pipe_info(saa_plan *p, int mode, int *n_chunks, int64_t *slice_end, int32_t *need_upload, int cap)
{
    NEED_FINAL(p, "saa_plan_host_pipe_info");
    if (!n_chunks) return fail("saa_plan_host_pipe_info: null argument");
    CK(cudaSetDevice(p->device));
    const int table = (mode == SAA_MODE_SYNC && p->size > 1) ? 1 : 0;
    if (p->hp[table].state == 0 && host_pipe_build(p, table)) return -1;
    const saa_plan::HostPipe &h = p->hp[table];
    const int K = (h.state == 1 && !p->matfree) ? (int)h.slice_end.size() : 0;   // K5 steps take the plain sequence
    *n_chunks = K;
    if (K > 0 && slice_end && need_upload) {
        if (cap < K) return fail("saa_plan_host_pipe_info: capacity %d < %d chunks", cap, K);
        for (int c = 0; c < K; ++c) { slice_end[c] = h.slice_end[c]; need_upload[c] = h.need_upload[c]; }
    }
    return 0;
}

// pinned (page-locked) host memory for the vectors of saa_step_host[_ex]: asynchronous, full-speed PCIe copies
extern "C" void *saa_host_alloc(int64_t bytes)
{
    void *q = nullptr;
    if (bytes <= 0) { fail("saa_host_alloc: non-positive size"); return nullptr; }
    cudaError_t e = cudaHostAlloc(&q, (size_t)bytes, cudaHostAllocPortable);
    if (e != cudaSuccess) { fail("cudaHostAlloc(%lld) -> %s", (long long)bytes, cudaGetErrorString(e)); return nullptr; }
    return q;
}
extern "C" int saa_host_free(void *q)
{
    if (q) CK(cudaFreeHost(q));
    return 0;
}

extern "C" int saa_step_host_ex(saa_plan *p, const double *d0, const double *dn, double tn, int mode, double *d1, int flags)
{
    NEED_FINAL(p, "saa_step_host");
    if (!d0 || !dn || !d1) return fail("saa_step_host: null argument");
    if (p->group) return fail("saa_step_host: plan belongs to a group");
    CK(cudaSetDevice(p->device));
    cudaStream_t st = p->stream;
    // The reference's loop rotates d_n = d_0; d_0 = d1 (Data_prepare.py:233-234): the dn of this call is the d0 of the
    // previous one, which the device still holds in the other displacement level (the step overwrote the OLD dn with
    // d1 and swapped).  Valid only while nothing else touched the plan's state since that call.
    const bool keep_dn = (flags & SAA_HOST_DN_IS_PREVIOUS_D0) && p->host_epoch == p->state_epoch;
    const bool local = mode == SAA_MODE_LOCAL || (mode == SAA_MODE_SYNC && p->size == 1);
    const bool sync = mode == SAA_MODE_SYNC && p->size > 1 && (use_peer(p) || p->comm);
    const char *pipe_env = getenv("SAA_STEP_HOST_PIPELINE");  // "0": plain sequence (checked per call); K > 1: K chunks (read when the table is built)
    if ((local || sync) && !needs_hooks(p, mode) && !p->matfree && p->kvariant < 6 && !(pipe_env && pipe_env[0] == '0')) {
        const int table = sync ? 1 : 0;
        if (p->hp[table].state == 0 && host_pipe_build(p, table)) return -1;
        if (p->hp[table].state == 1) {
            if (host_pipe_step(p, table, d0, dn, tn, d1, keep_dn)) return -1;
            p->host_epoch = p->state_epoch;
            return keep_dn ? 1 : 0;
        }
    }
    CK(cudaMemcpyAsync(p->d_stage, d0, p->n_dof * sizeof(double), cudaMemcpyHostToDevice, st));
    if (!keep_dn) CK(cudaMemcpyAsync(p->d_stage + p->n_dof, dn, p->n_dof * sizeof(double), cudaMemcpyHostToDevice, st));
    if (set_state_from_stage(p, st, tn, !keep_dn)) return -1;
    if (saa_plan_step(p, 1, mode, SAA_LAUNCH_PER_STEP)) return -1;
    if (get_state_to_stage(p, st, true, false)) return -1;
    CK(cudaMemcpyAsync(d1, p->d_stage, p->n_dof * sizeof(double), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    p->host_epoch = p->state_epoch;
    return keep_dn ? 1 : 0;
}

extern "C" int saa_step_host(saa_plan *p, const double *d0, const double *dn, double tn, int mode, double *d1)
{
    return saa_step_host_ex(p, d0, dn, tn, mode, d1, 0) < 0 ? -1 : 0;
}

// ---- caller-provided transport (MPI through mpi4py, gloo, ...): the messages pass through host memory ----
extern "C" int saa_plan_halo_layout(const saa_plan *p, int *n_nb, int32_t *nb_rank, int64_t *msg_off, int cap)
{
    if (!p || !p->finalized) return fail("saa_plan_halo_layout: plan not finalized");
    const int n = (int)p->nb_rank.size();
    if (n_nb) *n_nb = n;
    if (nb_rank && msg_off) {
        if (cap < n) return fail("saa_plan_halo_layout: capacity %d < %d neighbours", cap, n);
        for (int k = 0; k < n; ++k) nb_rank[k] = p->nb_rank[k];
        for (int k = 0; k <= n; ++k) msg_off[k] = p->msg_off.empty() ? 0 : p->msg_off[k];
    }
    return 0;
}

extern "C" int saa_plan_step_begin_host(saa_plan *p, double *send_host)
{
    NEED_FINAL(p, "saa_plan_step_begin_host");
    if (p->group) return fail("saa_plan_step_begin_host: plan belongs to a group");
    CK(cudaSetDevice(p->device));
    p->state_epoch++;
    sync_phase_boundary(p, p->stream);
    if (p->total_msg > 0) {
        if (!send_host) return fail("saa_plan_step_begin_host: null send buffer");
        CK(cudaMemcpyAsync(send_host, p->d_send, p->total_msg * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
        if (!p->ev_msg) CK(cudaEventCreateWithFlags(&p->ev_msg, cudaEventDisableTiming));
        CK(cudaEventRecord(p->ev_msg, p->stream));
    }
    // interior rows do not depend on the exchange: enqueue them now so that they overlap the caller's transport
    sync_phase_interior(p, p->stream);
    CK(cudaGetLastError());
    if (p->total_msg > 0) CK(cudaEventSynchronize(p->ev_msg));   // wait for the messages only, not for the interior rows
    p->in_split_step = true;
    return 0;
}

extern "C" int saa_plan_step_end_host(saa_plan *p, const double *recv_host)
{
    NEED_FINAL(p, "saa_plan_step_end_host");
    if (!p->in_split_step) return fail("saa_plan_step_end_host without saa_plan_step_begin_host");
    CK(cudaSetDevice(p->device));
    if (p->total_msg > 0) {
        if (!recv_host) return fail("saa_plan_step_end_host: null receive buffer");
        CK(cudaMemcpyAsync(p->d_recv, recv_host, p->total_msg * sizeof(double), cudaMemcpyHostToDevice, p->stream));
    }
    sync_phase_shared(p, p->stream);
    p->in_split_step = false;
    if (after_step(p, p->stream, SAA_MODE_SYNC)) return -1;
    CK(cudaGetLastError());
    return 0;
}

// syn_cpus on a caller-provided force vector (external local DOF order, host memory)
extern "C" int saa_plan_forces_begin_host(saa_plan *p, const double *f_host, double *send_host)
{
    NEED_FINAL(p, "saa_plan_forces_begin_host");
    if (!f_host) return fail("saa_plan_forces_begin_host: null argument");
    CK(cudaSetDevice(p->device));
    cudaStream_t st = plan_stream(p);
    if (!p->d_force) CK(cudaMalloc((void **)&p->d_force, 2 * p->n_rows * sizeof(double)));
    CK(cudaMemsetAsync(p->d_force, 0, p->n_rows * sizeof(double), st));
    CK(cudaMemcpyAsync(p->d_stage, f_host, p->n_dof * sizeof(double), cudaMemcpyHostToDevice, st));
    saa_k_scatter_to_internal<<<nblk(p->n_dof, 256), 256, 0, st>>>(p->n_dof, p->d_iperm, p->d_stage, p->d_force);
    p->launches++;
    if (p->sh_slices > 0) {
        saa_k_pack_forces<<<nblk(p->H.sh_rows, 256), 256, 0, st>>>(p->H, p->d_force);
        p->launches++;
        if (p->total_msg > 0 && send_host)
            CK(cudaMemcpyAsync(send_host, p->d_send, p->total_msg * sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    CK(cudaStreamSynchronize(st));
    return 0;
}

extern "C" int saa_plan_forces_end_host(saa_plan *p, const double *recv_host, double *out_host)
{
    NEED_FINAL(p, "saa_plan_forces_end_host");
    if (!out_host || !p->d_force) return fail("saa_plan_forces_end_host: null argument or no begin call");
    CK(cudaSetDevice(p->device));
    cudaStream_t st = plan_stream(p);
    if (p->total_msg > 0 && recv_host)
        CK(cudaMemcpyAsync(p->d_recv, recv_host, p->total_msg * sizeof(double), cudaMemcpyHostToDevice, st));
    double *sum = p->d_force + p->n_rows;
    saa_k_sum_forces<<<nblk(p->n_rows, 256), 256, 0, st>>>(p->n_rows, p->H, p->d_force, sum);
    saa_k_gather_to_external<<<nblk(p->n_dof, 256), 256, 0, st>>>(p->n_dof, p->d_iperm, sum, p->d_stage);
    p->launches += 2;
    CK(cudaMemcpyAsync(out_host, p->d_stage, p->n_dof * sizeof(double), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return 0;
}

// ---- group transport: P partitions in one process, messages moved by device-to-device copies ------------
extern "C" int saa_group_create(saa_group **out, saa_plan **plans, int n_plans)
{
    if (!out || !plans || n_plans <= 0) return fail("saa_group_create: bad arguments");
    for (int i = 0; i < n_plans; ++i) {
        if (!plans[i] || !plans[i]->finalized) return fail("saa_group_create: plan %d is not finalized", i);
        if (plans[i]->size != n_plans || plans[i]->rank != i) return fail("saa_group_create: plan %d has rank %d of %d", i, plans[i]->rank, plans[i]->size);
        if (plans[i]->device != plans[0]->device) return fail("saa_group_create: all plans of a group must live on one device");
    }
    // message sizes must match pairwise
    for (int i = 0; i < n_plans; ++i) {
        saa_plan *a = plans[i];
        for (size_t k = 0; k < a->nb_rank.size(); ++k) {
            saa_plan *b = plans[a->nb_rank[k]];
            auto it = std::find(b->nb_rank.begin(), b->nb_rank.end(), i);
            if (it == b->nb_rank.end()) return fail("saa_group_create: rank %d lists %d as neighbour but not vice versa", i, a->nb_rank[k]);
            size_t kk = it - b->nb_rank.begin();
            if (b->msg_off[kk + 1] - b->msg_off[kk] != a->msg_off[k + 1] - a->msg_off[k])
                return fail("saa_group_create: interface %d<->%d has different sizes on the two sides", i, a->nb_rank[k]);
        }
    }
    saa_group *g = new saa_group();
    g->plans.assign(plans, plans + n_plans);
    CK(cudaSetDevice(plans[0]->device));
    CK(cudaStreamCreateWithFlags(&g->stream, cudaStreamNonBlocking));
    for (int i = 0; i < n_plans; ++i) plans[i]->group = g;
    *out = g;
    return 0;
}

extern "C" int saa_group_step(saa_group *g, int64_t n_steps, int mode, int launch)
{
    if (!g) return fail("saa_group_step: null group");
    (void)launch;
    CK(cudaSetDevice(g->plans[0]->device));
    cudaStream_t st = g->stream;
    // make sure earlier work on the plans' own streams (state uploads) is complete
    for (saa_plan *p : g->plans) { CK(cudaStreamSynchronize(p->stream)); p->state_epoch++; }
    for (int64_t s = 0; s < n_steps; ++s) {
        if (mode == SAA_MODE_SYNC && g->plans.size() > 1) {
            for (saa_plan *p : g->plans) sync_phase_boundary(p, st);
            for (size_t i = 0; i < g->plans.size(); ++i) {
                saa_plan *a = g->plans[i];
                for (size_t k = 0; k < a->nb_rank.size(); ++k) {
                    saa_plan *b = g->plans[a->nb_rank[k]];
                    size_t kk = std::find(b->nb_rank.begin(), b->nb_rank.end(), (int32_t)i) - b->nb_rank.begin();
                    // a receives from b the message b packed for a
                    CK(cudaMemcpyAsync(a->d_recv + a->msg_off[k], b->d_send + b->msg_off[kk],
                                       (a->msg_off[k + 1] - a->msg_off[k]) * sizeof(double), cudaMemcpyDeviceToDevice, st));
                }
            }
            for (saa_plan *p : g->plans) {
                sync_phase_interior(p, st);
                sync_phase_shared(p, st);
                if (after_step(p, st, mode)) return -1;
            }
        } else {
            for (saa_plan *p : g->plans) {
                launch_local_step(p, st, mode == SAA_MODE_PREDICT);
                if (after_step(p, st, mode == SAA_MODE_SYNC ? SAA_MODE_LOCAL : mode)) return -1;
            }
        }
    }
    CK(cudaGetLastError());
    return 0;
}

extern "C" int saa_group_synchronize(saa_group *g)
{
    if (!g) return fail("saa_group_synchronize: null group");
    CK(cudaSetDevice(g->plans[0]->device));
    CK(cudaStreamSynchronize(g->stream));
    return 0;
}

extern "C" int saa_group_destroy(saa_group *g)
{
    if (!g) return 0;
    cudaSetDevice(g->plans[0]->device);
    cudaStreamSynchronize(g->stream);
    for (saa_plan *p : g->plans) p->group = nullptr;
    cudaStreamDestroy(g->stream);
    delete g;
    return 0;
}

// ---- peer-memory transport over NVLink: one process per GPU of one node ------------------------------------
extern "C" int saa_plan_peer_export(saa_plan *p, void *handle64, int64_t *total_msg)
{
    NEED_FINAL(p, "saa_plan_peer_export");
    if (!handle64) return fail("saa_plan_peer_export: null argument");
    if (!p->d_recv) return fail("saa_plan_peer_export: this plan has no interface");
    CK(cudaSetDevice(p->device));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, p->d_recv));
    memcpy(handle64, &h, sizeof h);
    if (total_msg) *total_msg = p->total_msg;
    return 0;
}

extern "C" int saa_plan_peer_attach(saa_plan *p, int n_nb, const void *handles64, const int64_t *remote_off,
                                    const int64_t *remote_total, const int32_t *remote_slot, const int32_t *remote_n_nb)
{
    NEED_FINAL(p, "saa_plan_peer_attach");
    if (n_nb != (int)p->nb_rank.size()) return fail("saa_plan_peer_attach: %d handles for %d neighbours", n_nb, (int)p->nb_rank.size());
    if (p->peer) return fail("saa_plan_peer_attach: already attached");
    if (n_nb > 255) return fail("saa_plan_peer_attach: more than 255 neighbours");
    if (n_nb == 0) { p->peer = true; p->Hp = p->H; return prepare_graphs(p, true); }
    if (!handles64 || !remote_off || !remote_total || !remote_slot || !remote_n_nb) return fail("saa_plan_peer_attach: null argument");
    CK(cudaSetDevice(p->device));
    std::vector<double *> recv(n_nb);
    std::vector<unsigned long long *> flag(n_nb);
    std::vector<int64_t> stride(n_nb);
    for (int k = 0; k < n_nb; ++k) {
        cudaIpcMemHandle_t h;
        memcpy(&h, (const char *)handles64 + 64 * k, sizeof h);
        void *ptr = nullptr;
#ifdef SAA_DEBUG_PEER
        if (getenv("SAA_DEBUG_PEER_SELF")) ptr = p->d_recv;   // single-GPU timing probe: "the neighbour" is this plan itself
#endif
        if (!ptr) {
            CK(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
            p->peer_mapped.push_back(ptr);
        }
        if (remote_slot[k] < 0 || remote_slot[k] >= remote_n_nb[k]) return fail("saa_plan_peer_attach: bad remote slot");
        recv[k] = (double *)ptr;
        stride[k] = remote_total[k];
        flag[k] = (unsigned long long *)((double *)ptr + 2 * remote_total[k]) + remote_slot[k];
    }
    // destination table inside the neighbours' receive areas: same entries as the pack table, rebased
    std::vector<int32_t> pos(p->dst_pos_h.size());
    for (size_t i = 0; i < pos.size(); ++i) {
        const int k = p->dst_nb_h[i];
        pos[i] = (int32_t)(p->dst_pos_h[i] - p->msg_off[k] + remote_off[k]);
        if (pos[i] < 0 || pos[i] >= remote_total[k]) return fail("saa_plan_peer_attach: destination outside the neighbour's receive area");
    }
    if (upload(&p->d_dst_pos_peer, pos) || upload(&p->d_peer_recv, recv) || upload(&p->d_peer_stride, stride) || upload(&p->d_peer_flag, flag))
        return -1;
    p->Hp = p->H;
    p->Hp.dst_pos = p->d_dst_pos_peer;
    p->Hp.peer_recv = p->d_peer_recv; p->Hp.peer_stride = p->d_peer_stride; p->Hp.peer_flag = p->d_peer_flag;
    const char *fz = getenv("SAA_PEER_FUSED");
    p->peer_fused = !(fz && fz[0] == '0');
    p->Hp.dbg = 0;
#ifdef SAA_DEBUG_PEER                                  // profiling builds only (make DEBUG_PEER=1): results are wrong when set
    if (const char *dbg = getenv("SAA_DEBUG_PEER")) {
        p->Hp.dbg = atoi(dbg);
        fprintf(stderr, "[saa] SAA_DEBUG_PEER=%d: timing experiment, RESULTS ARE WRONG\n", p->Hp.dbg);
    }
#else
    if (getenv("SAA_DEBUG_PEER") || getenv("SAA_DEBUG_PEER_SELF"))
        return fail("saa_plan_peer_attach: SAA_DEBUG_PEER* is set but this library was built without -DSAA_DEBUG_PEER");
#endif
    p->peer = true;
    return prepare_graphs(p, true);
}

// ---- NCCL transport -----------------------------------------------------------------------------------------
extern "C" int saa_nccl_unique_id(void *id128)
{
    if (!id128) return fail("saa_nccl_unique_id: null argument");
    if (load_nccl()) return -1;
    saa_ncclUniqueId id;
    NCK(g_nccl.GetUniqueId(&id));
    memcpy(id128, &id, sizeof id);
    return 0;
}

extern "C" int saa_plan_init_nccl(saa_plan *p, const void *id128)
{
    NEED_FINAL(p, "saa_plan_init_nccl");
    if (!id128) return fail("saa_plan_init_nccl: null id");
    if (load_nccl()) return -1;
    CK(cudaSetDevice(p->device));
    saa_ncclUniqueId id;
    memcpy(&id, id128, sizeof id);
    NCK(g_nccl.CommInitRank(&p->comm, p->size, id, p->rank));
    return 0;
}

#include "saa_device_setup.cuh"

// ---- matrix-free mode (K5) ------------------------------------------------------------------------------------
extern "C" int saa_plan_set_matfree_dev(saa_plan *p, int64_t n_elem, const int32_t *cells_dev, const double *coords_dev, double lmd, double mu)
{
    NEED_FINAL(p, "saa_plan_set_matfree_dev");
    if (n_elem <= 0 || !cells_dev || !coords_dev) return fail("saa_plan_set_matfree_dev: null or empty argument");
    if (p->d_mf_inc) return fail("saa_plan_set_matfree_dev: already set");
    CK(cudaSetDevice(p->device));
    const int64_t nn_ext = p->n_dof / 3, nn_int = p->n_rows / 3;
    {   // every kernel below indexes by the node ids and K5 divides by 6 detJ: refuse bad cells before anything changes
        DevBuf b_first;
        if (b_first.alloc(2 * sizeof(unsigned long long))) return -1;
        unsigned long long *first_d = b_first.as<unsigned long long>();
        CK(cudaMemset(first_d, 0xff, 2 * sizeof(unsigned long long)));
        saa_k_mf_check_cells<<<nblk(n_elem, 256), 256>>>(n_elem, nn_ext, cells_dev, coords_dev, first_d);
        CK(cudaGetLastError());
        unsigned long long first[2] = {0, 0};
        CK(cudaMemcpy(first, first_d, sizeof first, cudaMemcpyDeviceToHost));
        if (first[0] != ~0ull)
            return fail("saa_plan_set_matfree_dev: element %llu has a node id outside [0, %lld)", first[0], (long long)nn_ext);
        if (first[1] != ~0ull)
            return fail("saa_plan_set_matfree_dev: element %llu has zero volume (a repeated corner, or 6 detJ of a corner "
                        "rounds to 0)", first[1]);
    }
    CK(cudaMalloc((void **)&p->d_mf_cells, 4 * n_elem * sizeof(int32_t)));
    CK(cudaMalloc((void **)&p->d_mf_X, 3 * nn_int * sizeof(double)));
    CK(cudaMemset(p->d_mf_X, 0, 3 * nn_int * sizeof(double)));
    saa_k_mf_cells_to_internal<<<nblk(4 * n_elem, 256), 256>>>(4 * n_elem, cells_dev, p->d_iperm, p->d_mf_cells);
    saa_k_mf_coords_to_internal<<<nblk(nn_ext, 256), 256>>>(nn_ext, coords_dev, p->d_iperm, p->d_mf_X);
    CK(cudaGetLastError());
    DevBuf inc_ptr, inc_slot, width;
    if (build_incidence(nn_int, n_elem, p->d_mf_cells, inc_ptr, inc_slot)) return -1;     // ascending element order per node
    if (width.alloc((p->n_slices + 1) * sizeof(int64_t))) return -1;
    CK(cudaMalloc((void **)&p->d_mf_slice_ptr, (p->n_slices + 1) * sizeof(int64_t)));
    saa_k_mf_slice_width<<<nblk(p->n_slices + 1, 256), 256>>>(p->n_slices, inc_ptr.as<int64_t>(), width.as<int64_t>());
    thrust::exclusive_scan(thrust::device, width.as<int64_t>(), width.as<int64_t>() + p->n_slices + 1, p->d_mf_slice_ptr);
    CK(cudaMemcpy(&p->mf_lanes, p->d_mf_slice_ptr + p->n_slices, sizeof(int64_t), cudaMemcpyDeviceToHost));
    CK(cudaMalloc((void **)&p->d_mf_inc, std::max<int64_t>(p->mf_lanes, 1) * sizeof(int32_t)));
    saa_k_mf_fill<<<nblk(nn_int, 256), 256>>>(nn_int, inc_ptr.as<int64_t>(), inc_slot.as<int32_t>(), p->d_mf_slice_ptr, p->d_mf_inc);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    p->mf_elems = n_elem;
    if (const char *mb = getenv("SAA_MF_MINB")) p->mf_minb = atoi(mb);
    p->MF.slice_ptr = p->d_mf_slice_ptr; p->MF.inc = p->d_mf_inc; p->MF.cells = (const int4 *)p->d_mf_cells; p->MF.X = p->d_mf_X;
    p->MF.lmd = lmd; p->MF.mu = mu;
    return 0;
}

// bytes the matrix-free kernel streams per time step besides the five vector streams: connectivity, incidence
// (incl. slice padding), coordinates, slice offsets, Dirichlet mask words
extern "C" int64_t saa_plan_matfree_bytes(const saa_plan *p)
{
    if (!p || !p->d_mf_inc) return -1;
    return 16 * p->mf_elems + 4 * p->mf_lanes + 24 * (p->n_rows / 3) + (p->n_slices + 1) * 8 + (p->n_rows / 32) * 4;
}

// ---- stress recovery (saa_stress.cuh) --------------------------------------------------------------------------
extern "C" int saa_plan_element_stress_dev(saa_plan *p, double *out_dev)
{
    NEED_FINAL(p, "saa_plan_element_stress_dev");
    if (!p->d_mf_inc) return fail("saa_plan_element_stress_dev: no element geometry attached; call saa_plan_set_matfree_dev first");
    if (!out_dev) return fail("saa_plan_element_stress_dev: null output");
    if ((uintptr_t)out_dev % 16) return fail("saa_plan_element_stress_dev: out_dev must be 16-byte aligned");
    CK(cudaSetDevice(p->device));
    const cudaStream_t st = plan_stream(p);
    if (!p->d_st_bad) CK(cudaMalloc((void **)&p->d_st_bad, sizeof(unsigned long long)));
    CK(cudaMemsetAsync(p->d_st_bad, 0xff, sizeof(unsigned long long), st));
    saa_k_stress_elem<<<nblk(p->mf_elems, 256), 256, 0, st>>>(p->mf_elems, p->MF.cells, p->MF.X, p->d_buf[p->cur], p->MF.lmd, p->MF.mu,
                                                             out_dev, p->d_st_bad);
    CK(cudaGetLastError());
    p->launches++;
    unsigned long long bad = 0;
    CK(cudaMemcpyAsync(&bad, p->d_st_bad, sizeof bad, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (bad != ~0ull)
        return fail("saa_plan_element_stress_dev: element %llu (in the order given to saa_plan_set_matfree_dev) has detJ <= 0: "
                    "inverted or degenerate tetrahedron", bad);
    return 0;
}

extern "C" int saa_plan_nodal_stress_dev(saa_plan *p, const double *elem_dev, double *out_dev)
{
    NEED_FINAL(p, "saa_plan_nodal_stress_dev");
    if (!p->d_mf_inc) return fail("saa_plan_nodal_stress_dev: no element geometry attached; call saa_plan_set_matfree_dev first");
    if (!elem_dev || !out_dev) return fail("saa_plan_nodal_stress_dev: null argument");
    if ((uintptr_t)elem_dev % 16) return fail("saa_plan_nodal_stress_dev: elem_dev must be 16-byte aligned");
    CK(cudaSetDevice(p->device));
    const cudaStream_t st = plan_stream(p);
    if (!p->d_st_ext) {
        CK(cudaMalloc((void **)&p->d_st_ext, (p->n_rows / 3) * sizeof(int32_t)));
        CK(cudaMemsetAsync(p->d_st_ext, 0xff, (p->n_rows / 3) * sizeof(int32_t), st));
        saa_k_hp_inverse<<<nblk(p->n_dof / 3, 256), 256, 0, st>>>(p->n_dof / 3, p->d_iperm, p->d_st_ext);
        CK(cudaGetLastError());
        p->launches++;
    }
    saa_k_stress_node<<<nblk(p->n_slices, SAA_WARPS_PER_BLOCK), 32 * SAA_WARPS_PER_BLOCK, 0, st>>>(p->n_slices, p->MF.slice_ptr, p->MF.inc,
                                                                                                   p->d_st_ext, elem_dev, out_dev);
    CK(cudaGetLastError());
    p->launches++;
    return 0;
}

// ---- static solve on the resident stiffness (saa_static.cuh, DESIGN.md §7c) ------------------------------------
// Work vectors of one plan for the duration of one call: one allocation, released when the call returns.  H is the
// plan's halo description with the pack and receive buffers pointed at the call's own scratch, so no buffer of the
// step path is written.
struct CgWork {
    saa_plan *p = nullptr;
    DevBuf mem;
    double *x = nullptr, *r = nullptr, *pv = nullptr, *q = nullptr, *z = nullptr, *binv = nullptr, *part = nullptr,
           *stage = nullptr, *recv = nullptr;
    uint32_t *free_mask = nullptr;
    int32_t *ext = nullptr;
    unsigned int *ticket = nullptr;
    SaaHaloDev H{};
    int64_t n_nodes = 0, n_blk = 0, n_units = 0, n_parts = 0;   // blocks of the slice / node kernels, shared-row units
};
#define SAA_CG_REDUCE_BLOCKS 256

static int cg_alloc(CgWork &w, saa_plan *p, bool solve, cudaStream_t st)
{
    const int64_t n = p->n_rows;
    w.p = p;
    w.H = p->H;
    w.n_nodes = n / 3;
    w.n_blk = nblk(p->n_slices, 8);                  // = blocks of 256 nodes
    w.n_units = nblk(p->H.sh_rows, 256);
    w.n_parts = w.n_blk + w.n_units;
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    const size_t ox = take(8 * n), oq = take(8 * n);
    size_t orr = 0, op = 0, oz = 0, ob = 0, opart = 0, ost = 0, ofm = 0, oext = 0, otk = 0;
    if (solve) {
        orr = take(8 * n); op = take(8 * n); oz = take(8 * n); ob = take(48 * w.n_nodes); opart = take(16 * w.n_parts);
        ost = take(16 * SAA_CG_REDUCE_BLOCKS); ofm = take(4 * (n / 32)); oext = take(4 * w.n_nodes); otk = take(4);
    }
    const size_t oxb = take(8 * p->H.sh_rows), osend = take(8 * p->total_msg), orecv = take(8 * p->total_msg);
    if (w.mem.alloc(off)) return -1;
    char *b = (char *)w.mem.p;
    w.x = (double *)(b + ox); w.q = (double *)(b + oq);
    if (solve) {
        w.r = (double *)(b + orr); w.pv = (double *)(b + op); w.z = (double *)(b + oz); w.binv = (double *)(b + ob);
        w.part = (double *)(b + opart); w.stage = (double *)(b + ost); w.free_mask = (uint32_t *)(b + ofm);
        w.ext = (int32_t *)(b + oext); w.ticket = (unsigned int *)(b + otk);
        CK(cudaMemsetAsync(w.ticket, 0, sizeof(unsigned int), st));   // ordered before the first reduction
    }
    w.recv = (double *)(b + orecv);
    w.H.xbuf = (double *)(b + oxb); w.H.sendbuf = (double *)(b + osend); w.H.recv = w.recv;
    return 0;
}

// syn_cpus on vector v of every plan of a group: pack the partial values of the shared rows, move the messages by
// device copies (as saa_group_step does); saa_k_sum_forces / saa_k_cg_shared then add them in ascending rank order
static int cg_exchange(CgWork *W, int P, double *CgWork::*v, cudaStream_t st)
{
    for (int i = 0; i < P; ++i)
        if (W[i].H.sh_rows > 0) saa_k_pack_forces<<<nblk(W[i].H.sh_rows, 256), 256, 0, st>>>(W[i].H, W[i].*v);
    for (int i = 0; i < P; ++i) {
        const saa_plan *a = W[i].p;
        for (size_t k = 0; k < a->nb_rank.size(); ++k) {
            const CgWork &b = W[a->nb_rank[k]];
            const size_t kk = std::find(b.p->nb_rank.begin(), b.p->nb_rank.end(), (int32_t)i) - b.p->nb_rank.begin();
            CK(cudaMemcpyAsync(W[i].recv + a->msg_off[k], b.H.sendbuf + b.p->msg_off[kk],
                               (a->msg_off[k + 1] - a->msg_off[k]) * sizeof(double), cudaMemcpyDeviceToDevice, st));
        }
    }
    CK(cudaGetLastError());
    return 0;
}

// out = S K in (DOT, with p.q partials) or b - S K in (RES, with r.r and b.b partials) on every plan, shared rows summed
template <int MODE>
static int cg_apply(CgWork *W, int P, double *CgWork::*in, double *CgWork::*out, cudaStream_t st, const long long *gate)
{
    for (int i = 0; i < P; ++i)
        saa_k_cg_apply<MODE><<<W[i].n_blk, 256, 0, st>>>(W[i].p->D, W[i].*in, W[i].*out, W[i].free_mask, W[i].part, W[i].n_parts, gate);
    if (P > 1) {
        if (cg_exchange(W, P, out, st)) return -1;
        for (int i = 0; i < P; ++i)
            if (W[i].n_units > 0)
                saa_k_cg_shared<MODE><<<W[i].n_units, 256, 0, st>>>(W[i].p->D, W[i].H, W[i].*in, W[i].*out, W[i].free_mask, W[i].part,
                                                                    W[i].n_parts, W[i].n_blk, gate);
    }
    CK(cudaGetLastError());
    return 0;
}

// the partials of the last apply (all n_parts) or update (n_blk, stride n_blk) of every plan -> rank slots rk[f * P + rank]
template <int NF>
static void cg_reduce(CgWork *W, int P, bool of_apply, double *rk, cudaStream_t st, const long long *gate)
{
    for (int i = 0; i < P; ++i) {
        const int64_t n = of_apply ? W[i].n_parts : W[i].n_blk;
        const unsigned G = std::min<unsigned>(nblk(n, 2048), SAA_CG_REDUCE_BLOCKS);
        saa_k_cg_reduce<NF><<<G, 256, 0, st>>>(W[i].part, n, n, W[i].stage, W[i].ticket, rk + i, P, gate);
    }
}

struct GraphExecGuard {
    cudaGraphExec_t e = nullptr;
    ~GraphExecGuard() { if (e) cudaGraphExecDestroy(e); }
};

// The iterations of a solve: chunks of check_every iterations, each replayed from one CUDA graph (SAA_STATIC_GRAPH=0:
// launched one by one), until the device-resident flags say done; hs then holds the final state.  A breakdown fails
// the call with its iteration index.
template <class Iteration>
static int cg_iterate(Iteration &iteration, const char *name, cudaStream_t st, SaaCgState *S, SaaCgState &hs, int64_t max_iter,
                      int64_t check_every)
{
    const int64_t chunk = std::min<int64_t>(check_every, std::max<int64_t>(max_iter, 1));
    const char *ge = getenv("SAA_STATIC_GRAPH");
    GraphExecGuard exec;
    if (max_iter > 0 && !(ge && ge[0] == '0')) {
        cudaGraph_t g;
        CK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
        int rc = 0;
        for (int64_t c = 0; c < chunk && rc == 0; ++c) rc = iteration();
        CK(cudaStreamEndCapture(st, &g));
        if (rc) { cudaGraphDestroy(g); return -1; }
        const cudaError_t e = cudaGraphInstantiate(&exec.e, g, 0);
        cudaGraphDestroy(g);
        CK(e);
    }
    auto read_state = [&]() -> int {
        CK(cudaMemcpyAsync(&hs, S, sizeof hs, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        return 0;
    };
    if (read_state()) return -1;
    for (int64_t launched = 0; !hs.done && launched < max_iter; launched += chunk) {
        if (exec.e) {
            CK(cudaGraphLaunch(exec.e, st));
        } else {
            for (int64_t c = 0; c < chunk; ++c)
                if (iteration()) return -1;
        }
        if (read_state()) return -1;
    }
    if (hs.fail) {
        const char *what = hs.fail == 1 ? "p.Ap <= 0 or not finite (A is not positive definite on the free DOFs)"
                         : hs.fail == 2 ? "r.z <= 0 or not finite before convergence" : "non-finite residual";
        return fail("%s: breakdown at iteration %lld: %s", name, hs.fail_it, what);
    }
    return 0;
}

static int cg_solve(saa_plan *const *plans, int P, const char *name, const double *const *x0, double *const *xout, double rtol,
                    int64_t max_iter, int64_t check_every, double *hist, int64_t *iters, double *rel_res, double *rel_res_true,
                    int *converged)
{
    if (!(rtol >= 0.0) || !std::isfinite(rtol)) return fail("%s: rtol must be finite and >= 0", name);
    if (max_iter < 0) return fail("%s: max_iter < 0", name);
    if (check_every < 1) return fail("%s: check_every must be >= 1", name);
    for (int i = 0; i < P; ++i) {
        if (!xout || !xout[i]) return fail("%s: null output", name);
        if (!plans[i]->d_val) return fail("%s: the assembled matrix of this plan was released (SAA_OPT_MATFREE = 2)", name);
    }
    saa_plan *p0 = plans[0];
    CK(cudaSetDevice(p0->device));
    for (int i = 0; i < P; ++i) CK(cudaStreamSynchronize(plans[i]->stream));   // earlier work on a plan's own stream
    const cudaStream_t st = plan_stream(p0);
    std::unique_ptr<CgWork[]> W(new CgWork[P]);
    for (int i = 0; i < P; ++i)
        if (cg_alloc(W[i], plans[i], true, st)) return -1;
    DevBuf sbuf;                                     // state, rank slots [2][P], bad node per plan
    if (sbuf.alloc(sizeof(SaaCgState) + 2 * P * sizeof(double) + P * sizeof(unsigned long long))) return -1;
    SaaCgState *S = sbuf.as<SaaCgState>();
    double *rk = (double *)(S + 1);
    unsigned long long *bad = (unsigned long long *)(rk + 2 * P);
    SaaCgState hs{};
    hs.rtol = rtol;
    hs.max_iter = max_iter;
    CK(cudaMemcpyAsync(S, &hs, sizeof hs, cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(bad, 0xff, P * sizeof(unsigned long long), st));

    // preconditioner: free rows, diagonal blocks (summed over the holders of a shared node), their inverses
    for (int i = 0; i < P; ++i) {
        CgWork &w = W[i];
        saa_plan *p = w.p;
        CK(cudaMemsetAsync(w.ext, 0xff, w.n_nodes * sizeof(int32_t), st));
        saa_k_hp_inverse<<<nblk(p->n_dof / 3, 256), 256, 0, st>>>(p->n_dof / 3, p->d_iperm, w.ext);
        saa_k_cg_free_mask<<<nblk(p->n_rows / 32, 256), 256, 0, st>>>(p->n_rows / 32, p->d_dir, w.ext, w.free_mask);
        saa_k_cg_diag<<<w.n_blk, 256, 0, st>>>(p->D, w.x, w.r, w.z);
    }
    if (P > 1)
        for (double *CgWork::*c : {&CgWork::x, &CgWork::r, &CgWork::z}) {
            if (cg_exchange(W.get(), P, c, st)) return -1;
            for (int i = 0; i < P; ++i) {
                saa_k_sum_forces<<<nblk(W[i].p->n_rows, 256), 256, 0, st>>>(W[i].p->n_rows, W[i].H, W[i].*c, W[i].q);
                CK(cudaMemcpyAsync(W[i].*c, W[i].q, W[i].p->n_rows * sizeof(double), cudaMemcpyDeviceToDevice, st));
            }
        }
    for (int i = 0; i < P; ++i)
        saa_k_cg_binv<<<nblk(W[i].n_nodes, 256), 256, 0, st>>>(W[i].n_nodes, W[i].x, W[i].r, W[i].z, W[i].free_mask, W[i].ext,
                                                               W[i].binv, bad + i);
    CK(cudaGetLastError());
    std::vector<unsigned long long> bad_h(P);
    CK(cudaMemcpyAsync(bad_h.data(), bad, P * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (int i = 0; i < P; ++i)
        if (bad_h[i] != ~0ull)
            return fail("%s: rank %d, local node %llu: its diagonal 3x3 block (clamped rows and columns replaced by the identity) "
                        "is not positive definite, Cholesky fails", name, plans[i]->rank, bad_h[i]);

    // x = S x0, r = b - A x, z = B^-1 r, p = z
    for (int i = 0; i < P; ++i) {
        CgWork &w = W[i];
        CK(cudaMemsetAsync(w.x, 0, w.p->n_rows * sizeof(double), st));
        if (x0 && x0[i]) {
            saa_k_scatter_to_internal<<<nblk(w.p->n_dof, 256), 256, 0, st>>>(w.p->n_dof, w.p->d_iperm, x0[i], w.x);
            saa_k_cg_mask<<<nblk(w.p->n_rows, 256), 256, 0, st>>>(w.p->n_rows, w.free_mask, w.x);
        }
    }
    if (cg_apply<SAA_APPLY_RES>(W.get(), P, &CgWork::x, &CgWork::r, st, nullptr)) return -1;
    cg_reduce<2>(W.get(), P, true, rk, st, nullptr);
    saa_k_cg_scalar<<<1, 32, 0, st>>>(S, rk, P, SAA_CG_RES0, hist);
    for (int i = 0; i < P; ++i)
        saa_k_cg_update<true><<<W[i].n_blk, 256, 0, st>>>(W[i].n_nodes, W[i].H, S, W[i].x, W[i].r, W[i].pv, W[i].q, W[i].z, W[i].binv,
                                                          W[i].free_mask, W[i].part, W[i].n_blk);
    cg_reduce<2>(W.get(), P, false, rk, st, nullptr);
    saa_k_cg_scalar<<<1, 32, 0, st>>>(S, rk, P, SAA_CG_INIT, hist);
    CK(cudaGetLastError());

    const long long *gate = &S->done;
    auto iteration = [&]() -> int {
        if (cg_apply<SAA_APPLY_DOT>(W.get(), P, &CgWork::pv, &CgWork::q, st, gate)) return -1;
        cg_reduce<1>(W.get(), P, true, rk, st, gate);
        saa_k_cg_scalar<<<1, 32, 0, st>>>(S, rk, P, SAA_CG_ALPHA, hist);
        for (int i = 0; i < P; ++i)
            saa_k_cg_update<false><<<W[i].n_blk, 256, 0, st>>>(W[i].n_nodes, W[i].H, S, W[i].x, W[i].r, W[i].pv, W[i].q, W[i].z,
                                                               W[i].binv, W[i].free_mask, W[i].part, W[i].n_blk);
        cg_reduce<2>(W.get(), P, false, rk, st, gate);
        saa_k_cg_scalar<<<1, 32, 0, st>>>(S, rk, P, SAA_CG_BETA, hist);
        for (int i = 0; i < P; ++i)
            saa_k_cg_direction<<<nblk(W[i].p->n_rows, 256), 256, 0, st>>>(W[i].p->n_rows, S, W[i].z, W[i].pv);
        CK(cudaGetLastError());
        return 0;
    };
    if (cg_iterate(iteration, name, st, S, hs, max_iter, check_every)) return -1;
    auto read_state = [&]() -> int {
        CK(cudaMemcpyAsync(&hs, S, sizeof hs, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        return 0;
    };
    // the true residual b - A x of the returned iterate, and x in local DOF order
    if (cg_apply<SAA_APPLY_RES>(W.get(), P, &CgWork::x, &CgWork::q, st, nullptr)) return -1;
    cg_reduce<2>(W.get(), P, true, rk, st, nullptr);
    saa_k_cg_scalar<<<1, 32, 0, st>>>(S, rk, P, SAA_CG_TRUE, hist);
    for (int i = 0; i < P; ++i)
        saa_k_gather_to_external<<<nblk(W[i].p->n_dof, 256), 256, 0, st>>>(W[i].p->n_dof, W[i].p->d_iperm, W[i].x, xout[i]);
    CK(cudaGetLastError());
    if (read_state()) return -1;
    const double bn = std::sqrt(hs.bb);
    if (iters) *iters = hs.it;
    if (rel_res) *rel_res = bn > 0.0 ? std::sqrt(hs.rr) / bn : std::sqrt(hs.rr);
    if (rel_res_true) *rel_res_true = bn > 0.0 ? std::sqrt(hs.rr_true) / bn : std::sqrt(hs.rr_true);
    if (converged) *converged = (int)hs.converged;
    return 0;
}

extern "C" int saa_plan_solve_static_dev(saa_plan *p, const double *x0_dev, double *x_dev, double rtol, int64_t max_iter,
                                         int64_t check_every, double *hist_dev, int64_t *iters, double *rel_res,
                                         double *rel_res_true, int *converged)
{
    NEED_FINAL(p, "saa_plan_solve_static_dev");
    if (p->size > 1)
        return fail("saa_plan_solve_static_dev: this plan is rank %d of a partition of size %d; solve all ranks together with "
                    "saa_group_solve_static_dev (the peer, NCCL and host-staged transports are not supported by the static solve)",
                    p->rank, p->size);
    return cg_solve(&p, 1, "saa_plan_solve_static_dev", &x0_dev, &x_dev, rtol, max_iter, check_every, hist_dev, iters, rel_res,
                    rel_res_true, converged);
}

extern "C" int saa_group_solve_static_dev(saa_group *g, const double *const *x0_dev, double *const *x_dev, double rtol,
                                          int64_t max_iter, int64_t check_every, double *hist_dev, int64_t *iters,
                                          double *rel_res, double *rel_res_true, int *converged)
{
    if (!g) return fail("saa_group_solve_static_dev: null group");
    return cg_solve(g->plans.data(), (int)g->plans.size(), "saa_group_solve_static_dev", x0_dev, x_dev, rtol, max_iter,
                    check_every, hist_dev, iters, rel_res, rel_res_true, converged);
}

// y = LocalK x of every plan (local DOF order); with `sum`, the shared rows hold the rank-ordered holder sums
static int apply_stiffness(saa_plan *const *plans, int P, const char *name, const double *const *x, double *const *y, bool sum)
{
    for (int i = 0; i < P; ++i) {
        if (!x || !y || !x[i] || !y[i]) return fail("%s: null argument", name);
        if (!plans[i]->d_val) return fail("%s: the assembled matrix of this plan was released (SAA_OPT_MATFREE = 2)", name);
    }
    CK(cudaSetDevice(plans[0]->device));
    for (int i = 0; i < P; ++i) CK(cudaStreamSynchronize(plans[i]->stream));
    const cudaStream_t st = plan_stream(plans[0]);
    std::unique_ptr<CgWork[]> W(new CgWork[P]);
    for (int i = 0; i < P; ++i) {
        CgWork &w = W[i];
        saa_plan *p = plans[i];
        if (cg_alloc(w, p, false, st)) return -1;
        CK(cudaMemsetAsync(w.x, 0, p->n_rows * sizeof(double), st));   // slice padding: finite, multiplied by 0.0
        saa_k_scatter_to_internal<<<nblk(p->n_dof, 256), 256, 0, st>>>(p->n_dof, p->d_iperm, x[i], w.x);
        saa_k_cg_apply<SAA_APPLY_RAW><<<w.n_blk, 256, 0, st>>>(p->D, w.x, w.q, nullptr, nullptr, 0, nullptr);
    }
    double *CgWork::*res = &CgWork::q;
    if (sum) {
        if (cg_exchange(W.get(), P, &CgWork::q, st)) return -1;
        for (int i = 0; i < P; ++i)
            saa_k_sum_forces<<<nblk(W[i].p->n_rows, 256), 256, 0, st>>>(W[i].p->n_rows, W[i].H, W[i].q, W[i].x);
        res = &CgWork::x;
    }
    for (int i = 0; i < P; ++i)
        saa_k_gather_to_external<<<nblk(plans[i]->n_dof, 256), 256, 0, st>>>(plans[i]->n_dof, plans[i]->d_iperm, W[i].*res, y[i]);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(st));
    return 0;
}

extern "C" int saa_plan_apply_stiffness_dev(saa_plan *p, const double *x_dev, double *y_dev)
{
    NEED_FINAL(p, "saa_plan_apply_stiffness_dev");
    return apply_stiffness(&p, 1, "saa_plan_apply_stiffness_dev", &x_dev, &y_dev, false);
}

extern "C" int saa_group_apply_stiffness_dev(saa_group *g, const double *const *x_dev, double *const *y_dev)
{
    if (!g) return fail("saa_group_apply_stiffness_dev: null group");
    return apply_stiffness(g->plans.data(), (int)g->plans.size(), "saa_group_apply_stiffness_dev", x_dev, y_dev, true);
}

// ---- geometric multigrid preconditioner (saa_multigrid.cuh, DESIGN.md §7d) -------------------------------------------
// One level: its plan, the block-Jacobi inverse and free rows (w: the fields cg_apply / cg_reduce use, w.x / w.q point
// at r / d for the power iteration), the level's vectors and the tables that connect it to its neighbours.
struct MgLevel {
    saa_plan *p = nullptr;
    DevBuf mem, tab, ttab;
    CgWork w;
    double *x = nullptr, *b = nullptr, *r = nullptr, *d = nullptr, *slot = nullptr;   // x, b: coarse levels only
    double lam = 0.0;
    std::vector<double> c1, c2;                                         // Chebyshev step k: d = c1 d + c2 B^-1 r
    int64_t *p_ptr = nullptr; int32_t *p_cnode = nullptr; double *p_w = nullptr;    // prolongation from level + 1
    int64_t *t_ptr = nullptr; int32_t *t_fnode = nullptr; double *t_w = nullptr;    // restriction from level - 1
};
struct saa_mg {
    int n = 0;
    std::unique_ptr<MgLevel[]> L;
    DevBuf cinv;                                                        // A^-1 of the coarsest level, internal order
    int64_t bytes = 0;
};

// Chebyshev polynomial of `degree` steps on [0.3, 1.1] x lam (the smoother of PETSc's PCMG default): step 0 is
// d = B^-1 r / theta, step k > 0 d = rho_k rho_{k-1} d + 2 rho_k / delta B^-1 r with rho_k = 1 / (2 sigma - rho_{k-1})
static void mg_chebyshev(MgLevel &l, int degree)
{
    const double hi = 1.1 * l.lam, lo = 0.3 * l.lam, theta = 0.5 * (hi + lo), delta = 0.5 * (hi - lo), sigma = theta / delta;
    double rho = 1.0 / sigma;
    l.c1.assign(degree, 0.0);
    l.c2.assign(degree, 1.0 / theta);
    for (int k = 1; k < degree; ++k) {
        const double rn = 1.0 / (2.0 * sigma - rho);
        l.c1[k] = rn * rho;
        l.c2[k] = 2.0 * rn / delta;
        rho = rn;
    }
}

// x = V b on level l (b, x: level vectors in internal order, b zero on non-free rows)
static void mg_vcycle(saa_mg *mg, int l, const double *b, double *x, cudaStream_t st, const long long *gate)
{
    MgLevel &L = mg->L[l];
    const SaaDev &D = L.p->D;
    const int64_t nn = L.w.n_nodes;
    const unsigned gs = (unsigned)L.w.n_blk, gn = nblk(nn, 256);
    if (l == mg->n - 1) {
        saa_k_mg_coarse<<<nblk(L.p->n_rows, 8), 256, 0, st>>>(L.p->n_rows, mg->cinv.as<double>(), b, x, L.w.free_mask, gate);
        return;
    }
    const int deg = (int)L.c2.size();
    auto residual = [&]() { saa_k_mg_residual<<<gs, 256, 0, st>>>(D, x, b, L.r, L.w.free_mask, gate); };
    auto next_steps = [&]() {
        for (int k = 1; k < deg; ++k) {
            residual();
            saa_k_mg_cheb<SAA_MG_CHEB_NEXT><<<gn, 256, 0, st>>>(nn, L.r, L.d, x, L.w.binv, L.w.free_mask, L.c1[k], L.c2[k], gate);
        }
    };
    saa_k_mg_cheb<SAA_MG_CHEB_FIRST_ZERO><<<gn, 256, 0, st>>>(nn, b, L.d, x, L.w.binv, L.w.free_mask, 0.0, L.c2[0], gate);
    next_steps();
    residual();
    MgLevel &C = mg->L[l + 1];
    saa_k_mg_restrict<<<nblk(C.w.n_nodes, 256), 256, 0, st>>>(C.w.n_nodes, C.w.ext, C.t_ptr, C.t_fnode, C.t_w, L.r, C.b,
                                                              C.w.free_mask, gate);
    mg_vcycle(mg, l + 1, C.b, C.x, st, gate);
    saa_k_mg_prolong<<<gn, 256, 0, st>>>(nn, L.w.ext, L.p_ptr, L.p_cnode, L.p_w, C.x, x, L.w.free_mask, gate);
    residual();
    saa_k_mg_cheb<SAA_MG_CHEB_FIRST><<<gn, 256, 0, st>>>(nn, L.r, L.d, x, L.w.binv, L.w.free_mask, 0.0, L.c2[0], gate);
    next_steps();
}

// level l's memory, free rows, block-Jacobi inverse and lambda_max(B^-1 A)
static int mg_level_setup(saa_mg *mg, int l, saa_plan *p, int power_iters, cudaStream_t st)
{
    MgLevel &L = mg->L[l];
    CgWork &w = L.w;
    const int64_t n = p->n_rows;
    L.p = w.p = p;
    w.H = p->H;
    w.n_nodes = n / 3;
    w.n_blk = nblk(p->n_slices, 8);
    w.n_units = 0;
    w.n_parts = w.n_blk;
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    const bool own_xb = l > 0;
    const size_t ox = own_xb ? take(8 * n) : 0, ob = own_xb ? take(8 * n) : 0, orr = take(8 * n), od = take(8 * n);
    const size_t obinv = take(48 * w.n_nodes), opart = take(16 * w.n_parts), ost = take(16 * SAA_CG_REDUCE_BLOCKS);
    const size_t ofm = take(4 * (n / 32)), oext = take(4 * w.n_nodes), otk = take(4), osl = take(16), obad = take(8);
    if (L.mem.alloc(off)) return -1;
    mg->bytes += off;
    char *base = (char *)L.mem.p;
    if (own_xb) { L.x = (double *)(base + ox); L.b = (double *)(base + ob); }
    L.r = (double *)(base + orr); L.d = (double *)(base + od);
    w.binv = (double *)(base + obinv); w.part = (double *)(base + opart); w.stage = (double *)(base + ost);
    w.free_mask = (uint32_t *)(base + ofm); w.ext = (int32_t *)(base + oext); w.ticket = (unsigned int *)(base + otk);
    L.slot = (double *)(base + osl);
    unsigned long long *bad = (unsigned long long *)(base + obad);
    w.x = L.r; w.q = L.d;
    CK(cudaMemsetAsync(w.ticket, 0, sizeof(unsigned int), st));
    CK(cudaMemsetAsync(bad, 0xff, sizeof(unsigned long long), st));
    CK(cudaMemsetAsync(w.ext, 0xff, w.n_nodes * sizeof(int32_t), st));
    saa_k_hp_inverse<<<nblk(p->n_dof / 3, 256), 256, 0, st>>>(p->n_dof / 3, p->d_iperm, w.ext);
    saa_k_cg_free_mask<<<nblk(n / 32, 256), 256, 0, st>>>(n / 32, p->d_dir, w.ext, w.free_mask);
    {
        DevBuf cols;                                   // the diagonal blocks' three columns
        if (cols.alloc(3 * 8 * n)) return -1;
        double *c = cols.as<double>();
        saa_k_cg_diag<<<w.n_blk, 256, 0, st>>>(p->D, c, c + n, c + 2 * n);
        saa_k_cg_binv<<<nblk(w.n_nodes, 256), 256, 0, st>>>(w.n_nodes, c, c + n, c + 2 * n, w.free_mask, w.ext, w.binv, bad);
        CK(cudaGetLastError());
        unsigned long long bad_h = 0;
        CK(cudaMemcpyAsync(&bad_h, bad, sizeof bad_h, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (bad_h != ~0ull)
            return fail("saa_mg_create: level %d, local node %llu: its diagonal 3x3 block (clamped rows and columns replaced by the "
                        "identity) is not positive definite, Cholesky fails", l, bad_h);
    }
    // power iteration of B^-1 A, Rayleigh quotient in the A inner product: lam = (A x)^T B^-1 (A x) / x^T A x
    saa_k_mg_start<<<nblk(w.n_nodes, 256), 256, 0, st>>>(w.n_nodes, w.ext, w.free_mask, w.x);
    for (int it = 0; it < power_iters; ++it) {
        if (cg_apply<SAA_APPLY_DOT>(&w, 1, &CgWork::x, &CgWork::q, st, nullptr)) return -1;
        cg_reduce<1>(&w, 1, true, L.slot, st, nullptr);
        saa_k_mg_power<<<w.n_blk, 256, 0, st>>>(w.n_nodes, w.q, w.x, w.binv, w.free_mask, L.slot, w.part, w.n_blk);
        cg_reduce<1>(&w, 1, false, L.slot + 1, st, nullptr);
    }
    CK(cudaGetLastError());
    double s[2];
    CK(cudaMemcpyAsync(s, L.slot, sizeof s, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    L.lam = s[1] / s[0];
    if (!(L.lam > 0.0) || !std::isfinite(L.lam))
        return fail("saa_mg_create: level %d: the estimate of lambda_max(B^-1 A) is %g (A is not positive definite on the free DOFs)",
                    l, L.lam);
    return 0;
}

// the prolongation from level l + 1 to level l (stored on level l) and its transpose (stored on level l + 1)
static int mg_tables(saa_mg *mg, int l, const int64_t *ptr, const int32_t *col, const double *wt, cudaStream_t st)
{
    MgLevel &F = mg->L[l], &C = mg->L[l + 1];
    const int64_t nf = F.p->n_dof / 3, nc = C.p->n_dof / 3;
    DevBuf badb;
    if (badb.alloc(8)) return -1;
    CK(cudaMemsetAsync(badb.p, 0xff, 8, st));
    saa_k_mg_check_table<<<nblk(nf, 256), 256, 0, st>>>(nf, nc, ptr, col, badb.as<unsigned long long>());
    CK(cudaGetLastError());
    unsigned long long bad = 0;
    int64_t nnz = 0;
    CK(cudaMemcpyAsync(&bad, badb.p, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (bad != ~0ull)
        return fail("saa_mg_create: prolongation %d -> %d, fine node %llu: p_ptr is not a CSR offset table over the %lld nodes of "
                    "level %d, or a column is outside the %lld nodes of level %d", l + 1, l, bad, (long long)nf, l, (long long)nc, l + 1);
    CK(cudaMemcpyAsync(&nnz, ptr + nf, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (nnz >= INT32_MAX) return fail("saa_mg_create: prolongation %d -> %d has 2^31 or more entries", l + 1, l);
    const size_t b_ptr = 8 * (nf + 1), b_col = 4 * std::max<int64_t>(nnz, 1), b_w = 8 * std::max<int64_t>(nnz, 1);
    const size_t bt_ptr = 8 * (nc + 1);
    if (F.tab.alloc(b_ptr + b_col + b_w + 64) || C.ttab.alloc(bt_ptr + b_col + b_w + 64)) return -1;
    mg->bytes += b_ptr + b_col + b_w + bt_ptr + b_col + b_w;
    F.p_ptr = F.tab.as<int64_t>(); F.p_w = (double *)(F.p_ptr + nf + 1); F.p_cnode = (int32_t *)(F.p_w + std::max<int64_t>(nnz, 1));
    C.t_ptr = C.ttab.as<int64_t>(); C.t_w = (double *)(C.t_ptr + nc + 1); C.t_fnode = (int32_t *)(C.t_w + std::max<int64_t>(nnz, 1));
    CK(cudaMemcpyAsync(F.p_ptr, ptr, b_ptr, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(F.p_w, wt, 8 * nnz, cudaMemcpyDeviceToDevice, st));
    DevBuf scratch;                                    // entry row, sort keys, sorted entries
    if (scratch.alloc(12 * std::max<int64_t>(nnz, 1))) return -1;
    int32_t *row_of = scratch.as<int32_t>(), *keys = row_of + nnz, *entry = keys + nnz;
    saa_k_mg_table_rows<<<nblk(nf, 256), 256, 0, st>>>(nf, ptr, col, C.p->d_iperm, row_of, F.p_cnode);
    CK(cudaMemcpyAsync(keys, col, 4 * nnz, cudaMemcpyDeviceToDevice, st));
    CK(cudaGetLastError());
    // transpose: entries stably sorted by coarse node keep their ascending fine-node order
    thrust::sequence(thrust::cuda::par.on(st), entry, entry + nnz);
    thrust::stable_sort_by_key(thrust::cuda::par.on(st), keys, keys + nnz, entry);
    thrust::lower_bound(thrust::cuda::par.on(st), keys, keys + nnz, thrust::counting_iterator<int32_t>(0),
                        thrust::counting_iterator<int32_t>((int32_t)nc + 1), C.t_ptr);
    saa_k_mg_table_transpose<<<nblk(nnz, 256), 256, 0, st>>>(nnz, entry, row_of, wt, F.p->d_iperm, C.t_fnode, C.t_w);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(st));
    return 0;
}

extern "C" int saa_mg_create(saa_mg **out, saa_plan *const *levels, int n_levels, const int64_t *const *p_ptr, const int32_t *const *p_col,
                             const double *const *p_w, const double *coarse_inv_dev, int degree, int power_iters, int64_t coarsest_max_dof)
{
    if (!out) return fail("saa_mg_create: null output");
    *out = nullptr;
    if (!levels || n_levels < 2) return fail("saa_mg_create: a hierarchy needs at least two levels (got %d)", n_levels);
    if (degree < 1 || power_iters < 1) return fail("saa_mg_create: degree and power_iters must be >= 1");
    if (!p_ptr || !p_col || !p_w || !coarse_inv_dev) return fail("saa_mg_create: null prolongation table or coarse inverse");
    for (int l = 0; l < n_levels; ++l) {
        saa_plan *p = levels[l];
        if (!p) return fail("saa_mg_create: level %d: null plan", l);
        if (!p->finalized) return fail("saa_mg_create: level %d: plan not finalized", l);
        if (p->size > 1)
            return fail("saa_mg_create: level %d is rank %d of a partition of size %d; the multigrid preconditioner needs size-1 plans",
                        l, p->rank, p->size);
        if (!p->d_val) return fail("saa_mg_create: level %d: the assembled matrix of this plan was released (SAA_OPT_MATFREE = 2)", l);
        if (p->device != levels[0]->device)
            return fail("saa_mg_create: level %d is on device %d, level 0 on device %d", l, p->device, levels[0]->device);
        if (l < n_levels - 1 && (!p_ptr[l] || !p_col[l] || !p_w[l])) return fail("saa_mg_create: null prolongation table %d", l);
    }
    const saa_plan *pc = levels[n_levels - 1];
    if (pc->n_dof > coarsest_max_dof)
        return fail("saa_mg_create: the coarsest level has %lld DOF, above coarsest_max_dof = %lld (its dense inverse would take %.2f GB)",
                    (long long)pc->n_dof, (long long)coarsest_max_dof, 8.0 * pc->n_rows * pc->n_rows / 1e9);
    CK(cudaSetDevice(levels[0]->device));
    for (int l = 0; l < n_levels; ++l) CK(cudaStreamSynchronize(levels[l]->stream));
    const cudaStream_t st = plan_stream(levels[0]);
    std::unique_ptr<saa_mg> mg(new saa_mg);
    mg->n = n_levels;
    mg->L.reset(new MgLevel[n_levels]);
    for (int l = 0; l < n_levels; ++l) {
        if (mg_level_setup(mg.get(), l, levels[l], power_iters, st)) return -1;
        mg_chebyshev(mg->L[l], degree);
    }
    for (int l = 0; l + 1 < n_levels; ++l)
        if (mg_tables(mg.get(), l, p_ptr[l], p_col[l], p_w[l], st)) return -1;
    const int64_t ne = pc->n_dof, ni = pc->n_rows;
    if (mg->cinv.alloc(8 * ni * ni)) return -1;
    mg->bytes += 8 * ni * ni;
    CK(cudaMemsetAsync(mg->cinv.p, 0, 8 * ni * ni, st));
    saa_k_mg_coarse_permute<<<nblk(ne * ne, 256), 256, 0, st>>>(ne, ni, pc->d_iperm, coarse_inv_dev, mg->cinv.as<double>());
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(st));
    *out = mg.release();
    return 0;
}

extern "C" int saa_mg_destroy(saa_mg *mg)
{
    if (!mg) return 0;
    cudaSetDevice(mg->L[0].p->device);
    delete mg;
    return 0;
}

extern "C" int saa_mg_info(const saa_mg *mg, double *lambda, int64_t *bytes)
{
    if (!mg) return fail("saa_mg_info: null hierarchy");
    if (lambda)
        for (int l = 0; l < mg->n; ++l) lambda[l] = mg->L[l].lam;
    if (bytes) *bytes = mg->bytes;
    return 0;
}

static int mg_check(saa_mg *mg, const char *name)
{
    if (!mg) return fail("%s: null hierarchy", name);
    for (int l = 0; l < mg->n; ++l)
        if (!mg->L[l].p->d_val) return fail("%s: level %d: the assembled matrix of this plan was released (SAA_OPT_MATFREE = 2)", name, l);
    CK(cudaSetDevice(mg->L[0].p->device));
    for (int l = 0; l < mg->n; ++l) CK(cudaStreamSynchronize(mg->L[l].p->stream));
    return 0;
}

extern "C" int saa_plan_solve_static_mg_dev(saa_mg *mg, const double *x0, double *xout, double rtol, int64_t max_iter,
                                            int64_t check_every, double *hist, int64_t *iters, double *rel_res, double *rel_res_true,
                                            int *converged)
{
    const char *name = "saa_plan_solve_static_mg_dev";
    if (!(rtol >= 0.0) || !std::isfinite(rtol)) return fail("%s: rtol must be finite and >= 0", name);
    if (max_iter < 0) return fail("%s: max_iter < 0", name);
    if (check_every < 1) return fail("%s: check_every must be >= 1", name);
    if (!xout) return fail("%s: null output", name);
    if (mg_check(mg, name)) return -1;
    MgLevel &F = mg->L[0];
    saa_plan *p = F.p;
    const cudaStream_t st = plan_stream(p);
    // the outer iteration's vectors; preconditioner, free rows and partials are the fine level's
    CgWork w;
    w.p = p; w.H = F.w.H; w.n_nodes = F.w.n_nodes; w.n_blk = F.w.n_blk; w.n_units = 0; w.n_parts = F.w.n_parts;
    w.binv = F.w.binv; w.part = F.w.part; w.stage = F.w.stage; w.free_mask = F.w.free_mask; w.ext = F.w.ext; w.ticket = F.w.ticket;
    const int64_t n = p->n_rows;
    if (w.mem.alloc(5 * 8 * n)) return -1;
    w.x = w.mem.as<double>(); w.r = w.x + n; w.pv = w.r + n; w.q = w.pv + n; w.z = w.q + n;
    DevBuf sbuf;
    if (sbuf.alloc(sizeof(SaaCgState) + 2 * sizeof(double))) return -1;
    SaaCgState *S = sbuf.as<SaaCgState>();
    double *rk = (double *)(S + 1);
    SaaCgState hs{};
    hs.rtol = rtol;
    hs.max_iter = max_iter;
    CK(cudaMemcpyAsync(S, &hs, sizeof hs, cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(w.x, 0, n * sizeof(double), st));
    if (x0) {
        saa_k_scatter_to_internal<<<nblk(p->n_dof, 256), 256, 0, st>>>(p->n_dof, p->d_iperm, x0, w.x);
        saa_k_cg_mask<<<nblk(n, 256), 256, 0, st>>>(n, w.free_mask, w.x);
    }
    const long long *gate = &S->done;
    const unsigned gn = (unsigned)w.n_blk;
    // r = b - A x, z = V r, p = z
    if (cg_apply<SAA_APPLY_RES>(&w, 1, &CgWork::x, &CgWork::r, st, nullptr)) return -1;
    cg_reduce<2>(&w, 1, true, rk, st, nullptr);
    saa_k_cg_scalar<<<1, 32, 0, st>>>(S, rk, 1, SAA_CG_RES0, hist);
    mg_vcycle(mg, 0, w.r, w.z, st, gate);
    saa_k_mg_rz<true><<<gn, 256, 0, st>>>(w.n_nodes, S, w.r, w.z, w.pv, w.part, w.n_blk);
    cg_reduce<2>(&w, 1, false, rk, st, nullptr);
    saa_k_cg_scalar<<<1, 32, 0, st>>>(S, rk, 1, SAA_CG_INIT, hist);
    CK(cudaGetLastError());
    auto iteration = [&]() -> int {
        if (cg_apply<SAA_APPLY_DOT>(&w, 1, &CgWork::pv, &CgWork::q, st, gate)) return -1;
        cg_reduce<1>(&w, 1, true, rk, st, gate);
        saa_k_cg_scalar<<<1, 32, 0, st>>>(S, rk, 1, SAA_CG_ALPHA, hist);
        saa_k_mg_update<<<gn, 256, 0, st>>>(w.n_nodes, S, w.x, w.r, w.pv, w.q, w.free_mask, w.part, w.n_blk);
        mg_vcycle(mg, 0, w.r, w.z, st, gate);
        saa_k_mg_rz<false><<<gn, 256, 0, st>>>(w.n_nodes, S, w.r, w.z, nullptr, w.part, w.n_blk);
        cg_reduce<2>(&w, 1, false, rk, st, gate);
        saa_k_cg_scalar<<<1, 32, 0, st>>>(S, rk, 1, SAA_CG_BETA, hist);
        saa_k_cg_direction<<<nblk(n, 256), 256, 0, st>>>(n, S, w.z, w.pv);
        CK(cudaGetLastError());
        return 0;
    };
    if (cg_iterate(iteration, name, st, S, hs, max_iter, check_every)) return -1;
    // the true residual b - A x of the returned iterate, and x in local DOF order
    if (cg_apply<SAA_APPLY_RES>(&w, 1, &CgWork::x, &CgWork::q, st, nullptr)) return -1;
    cg_reduce<2>(&w, 1, true, rk, st, nullptr);
    saa_k_cg_scalar<<<1, 32, 0, st>>>(S, rk, 1, SAA_CG_TRUE, hist);
    saa_k_gather_to_external<<<nblk(p->n_dof, 256), 256, 0, st>>>(p->n_dof, p->d_iperm, w.x, xout);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(&hs, S, sizeof hs, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const double bn = std::sqrt(hs.bb);
    if (iters) *iters = hs.it;
    if (rel_res) *rel_res = bn > 0.0 ? std::sqrt(hs.rr) / bn : std::sqrt(hs.rr);
    if (rel_res_true) *rel_res_true = bn > 0.0 ? std::sqrt(hs.rr_true) / bn : std::sqrt(hs.rr_true);
    if (converged) *converged = (int)hs.converged;
    return 0;
}

// ---- the hierarchy's operators one at a time, external order (tests) ----
extern "C" int saa_mg_vcycle_dev(saa_mg *mg, const double *r_dev, double *z_dev)
{
    if (mg_check(mg, "saa_mg_vcycle_dev")) return -1;
    if (!r_dev || !z_dev) return fail("saa_mg_vcycle_dev: null argument");
    saa_plan *p = mg->L[0].p;
    const cudaStream_t st = plan_stream(p);
    const int64_t n = p->n_rows;
    DevBuf t;
    if (t.alloc(16 * n)) return -1;
    double *b = t.as<double>(), *x = b + n;
    CK(cudaMemsetAsync(b, 0, 8 * n, st));
    saa_k_scatter_to_internal<<<nblk(p->n_dof, 256), 256, 0, st>>>(p->n_dof, p->d_iperm, r_dev, b);
    saa_k_cg_mask<<<nblk(n, 256), 256, 0, st>>>(n, mg->L[0].w.free_mask, b);
    mg_vcycle(mg, 0, b, x, st, nullptr);
    saa_k_gather_to_external<<<nblk(p->n_dof, 256), 256, 0, st>>>(p->n_dof, p->d_iperm, x, z_dev);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(st));
    return 0;
}

static int mg_transfer(saa_mg *mg, int level, const double *in, double *out, bool prolong, const char *name)
{
    if (mg_check(mg, name)) return -1;
    if (!in || !out) return fail("%s: null argument", name);
    if (level < 0 || level + 1 >= mg->n) return fail("%s: level %d is not in [0, %d)", name, level, mg->n - 1);
    MgLevel &F = mg->L[level], &C = mg->L[level + 1];
    saa_plan *pi = prolong ? C.p : F.p, *po = prolong ? F.p : C.p;
    const cudaStream_t st = plan_stream(F.p);
    DevBuf t;
    if (t.alloc(8 * (pi->n_rows + po->n_rows))) return -1;
    double *vi = t.as<double>(), *vo = vi + pi->n_rows;
    CK(cudaMemsetAsync(t.p, 0, 8 * (pi->n_rows + po->n_rows), st));
    saa_k_scatter_to_internal<<<nblk(pi->n_dof, 256), 256, 0, st>>>(pi->n_dof, pi->d_iperm, in, vi);
    if (prolong)
        saa_k_mg_prolong<<<nblk(F.w.n_nodes, 256), 256, 0, st>>>(F.w.n_nodes, F.w.ext, F.p_ptr, F.p_cnode, F.p_w, vi, vo, F.w.free_mask,
                                                                 nullptr);
    else
        saa_k_mg_restrict<<<nblk(C.w.n_nodes, 256), 256, 0, st>>>(C.w.n_nodes, C.w.ext, C.t_ptr, C.t_fnode, C.t_w, vi, vo,
                                                                  C.w.free_mask, nullptr);
    saa_k_gather_to_external<<<nblk(po->n_dof, 256), 256, 0, st>>>(po->n_dof, po->d_iperm, vo, out);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(st));
    return 0;
}

extern "C" int saa_mg_prolong_dev(saa_mg *mg, int level, const double *xc_dev, double *xf_dev)
{
    return mg_transfer(mg, level, xc_dev, xf_dev, true, "saa_mg_prolong_dev");
}

extern "C" int saa_mg_restrict_dev(saa_mg *mg, int level, const double *rf_dev, double *bc_dev)
{
    return mg_transfer(mg, level, rf_dev, bc_dev, false, "saa_mg_restrict_dev");
}
