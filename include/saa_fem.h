/*
 * saa_fem.h — C ABI of the B200-native explicit FE time-step path.
 *
 * This is the drop-in boundary for the hot path of desResLab/Synchronization-avoiding-algorithms.
 * The reference has no FFI: the path sits behind three Python functions (all paths below are
 * under /root/reference):
 *
 *   parallel_explicit_solver_dis_pre(LocalK, F_rankwise, Points, Local_nodes, Local_Dirichlet,
 *                                    T, Elas, l_M, alpha, size, rank, MODEL)   Tools/Dynamic_solver.py:9-34
 *   syn_cpus(size, rank, f, L_g, Local_nodes)                                  Tools/Distributed_tools.py:77-92
 *   Local_assembly_for_stiffness(...) -> scipy csr_matrix                      Tools/Mat_construction.py:122-150
 *
 * A maintainer binds the entry points below with ctypes (see INTEGRATION.md); the Python shims in
 * synchronization-avoiding-algorithms_b200/Tools/ keep the reference's signatures on top of them.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; every function returns 0 on success, <0 on error;
 *     saa_last_error() returns a message for the calling thread's last failure.
 *   - "host" pointers are ordinary CPU memory, "dev" pointers are CUDA device memory on the plan's GPU.
 *   - A plan belongs to one GPU and one partition (MPI rank of the reference); not thread-safe.
 *   - All floating-point data is IEEE binary64.  The kernels evaluate every row sum and the update
 *     formula in the reference's operation order with separately rounded multiply/add (no FMA), so
 *     results are bit-identical to the reference's numpy/scipy arithmetic.
 *   - There is no CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef SAA_FEM_H
#define SAA_FEM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct saa_plan saa_plan;     /* one partition's device-resident problem + state */
typedef struct saa_group saa_group;   /* several plans of ONE process stepped together (halo exchange by
                                         device copies) — used to run a P-way partition on fewer GPUs */

/* step modes (MODEL / size arguments of Dynamic_solver.py:9-10,22,25) */
#define SAA_MODE_LOCAL 0      /* size == 1, or MODEL=True: no exchange, F_int = LocalK.dot(d0)            */
#define SAA_MODE_SYNC 1       /* size != 1 and MODEL=False: partial forces of shared DOFs are summed over
                                 their holders in ascending rank order (Distributed_tools.py:83-86)       */
#define SAA_MODE_PREDICT 2    /* MODEL=True + Online_predictor.py:298: shared DOFs overwritten by rows of
                                 the prediction table set with saa_plan_set_prediction                    */

/* launch strategies for saa_plan_step / saa_group_step */
#define SAA_LAUNCH_AUTO 0
#define SAA_LAUNCH_PER_STEP 1   /* one fused kernel launch per time step                                  */
#define SAA_LAUNCH_GRAPH 2      /* two-step CUDA graph replayed n/2 times                                 */
#define SAA_LAUNCH_PERSISTENT 3 /* one cooperative kernel looping over all steps with grid-wide barriers:
                                   SAA_MODE_LOCAL, and SAA_MODE_SYNC with the peer transport (small shards)   */

int saa_version(void);
const char *saa_last_error(void);
int saa_device_count(void);

/*
 * Build a plan from the inputs of parallel_explicit_solver_dis_pre (Dynamic_solver.py:9-10):
 *   n_dof            3 * len(Local_nodes)
 *   indptr/indices/data   LocalK as scipy CSR (int32 indptr and indices, sorted columns, float64 data).
 *                    The stored order inside each row is kept: it is the summation order of csr_matvec.
 *   F_rankwise, l_M  (n_dof) un-ramped load and lumped mass
 *   dirichlet        Local_Dirichlet: local DOF ids forced to 0 (Dynamic_solver.py:20,32)
 *   dt               T.dt;  dt2 = T.dt**2, dt_half = T.dt/2, half_alpha = 0.5*alpha are the scalar
 *                    sub-expressions of Dynamic_solver.py:17 evaluated by the caller in Python (np.float64
 *                    `**` goes through libm pow) so that the kernel uses the very same constants
 *   alpha            mass-proportional damping factor (`alpha` argument, Damp in Data_prepare.py:41)
 * The arrays are copied; the caller may free them afterwards.  State starts at d0 = dn = 0, tn = 0.
 */
int saa_plan_create(saa_plan **out, int device, int64_t n_dof, const int32_t *indptr, const int32_t *indices,
                    const double *data, const double *F_rankwise, const double *l_M, const int64_t *dirichlet,
                    int64_t n_dirichlet, double dt, double dt2, double dt_half, double half_alpha, double alpha);

/*
 * Describe the partition interface of this plan (what syn_cpus, Distributed_tools.py:77-92, derives
 * from rank_local_node_list each step).  Must be called before saa_plan_finalize for size > 1.
 *   rank, size        this partition and the number of partitions
 *   n_shared          number of shared nodes of this rank
 *   shared_pos        (n_shared) their positions in Local_nodes, in the canonical interface order
 *                     (ascending global node id)
 *   n_nb, nb_rank     neighbouring ranks, ascending
 *   nb_ptr            (n_nb+1) offsets into send_idx
 *   send_idx          for neighbour k: positions (into shared_pos) of the nodes shared with it, ascending
 *                     global id — the neighbour lists the same nodes in the same order
 *   holders_ptr       (n_shared+1) CSR over shared nodes
 *   holders_rank      ranks holding the node, ASCENDING (own rank included)
 *   holders_slot      -1 for the own rank, else the index of the node inside the message from that rank
 */
int saa_plan_set_halo(saa_plan *plan, int rank, int size, int64_t n_shared, const int64_t *shared_pos,
                      int n_nb, const int32_t *nb_rank, const int64_t *nb_ptr, const int64_t *send_idx,
                      const int64_t *holders_ptr, const int32_t *holders_rank, const int64_t *holders_slot);

/*
 * Same as saa_plan_create for inputs that already live on the plan's GPU (set-up at scale, see
 * saa_assemble_stiffness_dev): LocalK as CSR with int64 indptr, int32 sorted indices, float64 data; F_rankwise
 * and l_M as (n_dof) device vectors.  `dirichlet` is a host list.  The device arrays are borrowed until
 * saa_plan_finalize returns (which builds the same layout as the host path, entirely on the GPU); the caller
 * may free them afterwards.
 */
int saa_plan_create_dev(saa_plan **out, int device, int64_t n_dof, const int64_t *indptr_dev, const int32_t *indices_dev,
                        const double *data_dev, const double *F_rankwise_dev, const double *l_M_dev,
                        const int64_t *dirichlet_host, int64_t n_dirichlet, double dt, double dt2, double dt_half,
                        double half_alpha, double alpha);

/*
 * Sparse assembly on the GPU — Local_assembly_for_stiffness (Tools/Mat_construction.py:122-150) without the
 * dense (3n)^2 accumulator.  cells_dev: (n_elem,4) int32 LOCAL node ids of the rank's elements in
 * Local_ele_list order; coords_dev: (n_nodes,3) coordinates in Local_nodal_list order.  Returns cudaMalloc'ed
 * CSR arrays (3*n_nodes rows, int64 indptr, int32 ascending columns, exact zeros dropped); release them with
 * saa_device_free.  Element contributions are added in ascending element order by the thread owning the row
 * (deterministic, no atomics).  Values agree with the reference's BLAS-evaluated B^T D B to a few 1e-16
 * relative, not bit for bit (DESIGN.md).
 */
int saa_assemble_stiffness_dev(int device, int64_t n_nodes, int64_t n_elem, const int32_t *cells_dev,
                               const double *coords_dev, double lmd, double mu, int64_t **indptr_out_dev,
                               int32_t **indices_out_dev, double **data_out_dev, int64_t *nnz_out);
/* Row-summed (lumped) mass per node and un-ramped load vector (3 per node) of the LOCAL elements only
 * (Local_MKF, Mat_construction.py:36-73; lumping_to_vec, commons.py:103-107); shared nodes still need the
 * sum over their holders.  Outputs are caller-allocated device arrays of n_nodes and 3*n_nodes doubles. */
int saa_assemble_mass_load_dev(int device, int64_t n_nodes, int64_t n_elem, const int32_t *cells_dev,
                               const double *coords_dev, double rho, double fz, double *m_node_out_dev,
                               double *F_out_dev);
int saa_device_free(void *ptr);
/* cudaMemcpy(dst, src, bytes, cudaMemcpyDefault) — lets bindings read the arrays above */
int saa_device_copy(void *dst, const void *src, int64_t bytes);

/*
 * Optional, before saa_plan_finalize: the order in which the (non-interface) nodes are laid out in HBM — a
 * permutation of 0 .. n_dof/3-1, e.g. a space-filling-curve or reverse Cuthill-McKee order.  It only changes where
 * rows live (gather locality); results are bit-identical, external numbering is untouched.  Default: ascending
 * local node id, i.e. the reference's first-appearance order (Distributed_tools.py:14-24), which is as coherent
 * as the element order of the mesh file.
 */
int saa_plan_set_node_order(saa_plan *plan, const int32_t *order_host, int64_t n_nodes);

/* Upload everything to the GPU (boundary-first row order, sliced-ELL storage). */
int saa_plan_finalize(saa_plan *plan);
int saa_plan_destroy(saa_plan *plan);

/* sizes / layout facts, e.g. for the roofline arithmetic of bench.py */
int64_t saa_plan_n_dof(const saa_plan *plan);
int64_t saa_plan_nnz(const saa_plan *plan);           /* stored entries of LocalK                         */
int64_t saa_plan_padded_entries(const saa_plan *plan);/* 9 x block-lanes: entries of the 3x3 blocks incl. slice padding */
int64_t saa_plan_value_planes(const saa_plan *plan);  /* value planes stored (32 fp64 each; at most padded_entries / 32) */
int64_t saa_plan_kernel_launches(const saa_plan *plan);/* kernels launched by this plan so far            */
int64_t saa_plan_matrix_bytes(const saa_plan *plan);  /* bytes of matrix storage streamed per step        */
int64_t saa_plan_vector_bytes(const saa_plan *plan);  /* bytes of the vector streams of one step (d0, dn, d1, F, M; padded rows) */

/* State = (d0, dn, tn) of Time_integration_displacement (commons.py:47-52), local DOF order. */
int saa_plan_set_state(saa_plan *plan, const double *d0_host, const double *dn_host, double tn);
int saa_plan_get_state(saa_plan *plan, double *d0_host, double *dn_host, double *tn);
int saa_plan_set_state_dev(saa_plan *plan, const double *d0_dev, const double *dn_dev, double tn);
int saa_plan_get_state_dev(saa_plan *plan, double *d0_dev, double *dn_dev, double *tn);

/*
 * n_steps iterations of the loop body of Data_prepare.py:223-235 with the state resident in HBM:
 *   d1 = step(d0, dn, tn);  dn <- d0;  d0 <- d1;  tn <- tn + dt.
 * mode SAA_MODE_SYNC needs a transport: a group (saa_group_create) or NCCL (saa_plan_init_nccl).
 * Work is enqueued on the plan's stream; saa_plan_synchronize waits for it.
 */
int saa_plan_step(saa_plan *plan, int64_t n_steps, int mode, int launch);
int saa_plan_synchronize(saa_plan *plan);
/*
 * Execution options of synchronised steps (same arithmetic, same bits; used for cross-path checks and measurements):
 *   SAA_OPT_PEER_FUSED   1 (default): one fused launch per step with the peer transport; 0: boundary / interior /
 *                        shared-row kernels as three launches.
 *   SAA_OPT_PREFER_NCCL  1: use the NCCL transport (saa_plan_init_nccl) although peer memory is attached too.
 *   SAA_OPT_MATFREE      1: un-synchronised steps evaluate f_int = sum_e B^T D B u_e element by element (kernel K5,
 *                        saa_plan_set_matfree_dev) instead of streaming the assembled matrix — NOT bit-identical to the
 *                        assembled path (different association; see DESIGN.md), a throughput / low-memory mode.
 *                        2: same, and the assembled matrix is released (single-partition plans; cannot be undone).
 */
#define SAA_OPT_PEER_FUSED 1
#define SAA_OPT_PREFER_NCCL 2
#define SAA_OPT_MATFREE 3   /* 1: LOCAL / PREDICT steps (and SYNC steps of a single partition) use the matrix-free kernel K5 */
int saa_plan_set_option(saa_plan *plan, int option, int value);

/*
 * Matrix-free internal force (north star: "matrix-free element-wise B^T.D.B.u_e gather/scatter ... made deterministic
 * with ... CSR row ownership rather than atomics"): the element kernel of Tools/Mat_construction.py:79-119 applied to
 * u_e instead of assembled (:122-150).  cells_dev: (n_elem, 4) int32 LOCAL node ids (positions in Local_nodal_list),
 * coords_dev: (n_dof/3, 3) float64 coordinates of the local nodes, both in device memory (copied); lmd, mu: Lame
 * constants (Data_prepare.py:47).  Enable with saa_plan_set_option(plan, SAA_OPT_MATFREE, 1).
 */
int saa_plan_set_matfree_dev(saa_plan *plan, int64_t n_elem, const int32_t *cells_dev, const double *coords_dev,
                             double lmd, double mu);
int64_t saa_plan_matfree_bytes(const saa_plan *plan); /* bytes K5 streams per step besides the vector streams     */
/* the cudaStream_t the plan enqueues on (as void*), so that callers can record events on it */
void *saa_plan_stream(saa_plan *plan);

/*
 * The reference-facing call with HOST buffers: one evaluation of
 * parallel_explicit_solver_dis_pre(..., T=(tn, dt, d0, dn), ...) -> d1 (Dynamic_solver.py:9-34).
 * Copies d0 and dn to the GPU, runs one step, copies d1 back; the plan's state becomes (d1, d0, tn+dt).
 */
int saa_step_host(saa_plan *plan, const double *d0_host, const double *dn_host, double tn, int mode,
                  double *d1_host);
/*
 * Same call with a hint about the caller's rotation (Data_prepare.py:233-234, Online_predictor.py:265-266:
 * `d_n = d_0; d_0 = d1`).  SAA_HOST_DN_IS_PREVIOUS_D0 asserts that dn_host holds, unchanged, the values passed as
 * d0_host to the previous saa_step_host[_ex] call on this plan; the device still has them, so only d0 crosses PCIe.
 * The hint is ignored (full upload) when anything else touched the plan's state since that call.  dn_host must
 * still be a valid pointer.  Returns 1 when the dn upload was skipped, 0 when everything was uploaded, < 0 on error.
 */
#define SAA_HOST_DN_IS_PREVIOUS_D0 1
int saa_step_host_ex(saa_plan *plan, const double *d0_host, const double *dn_host, double tn, int mode,
                     double *d1_host, int flags);
/*
 * How saa_step_host[_ex] runs for `mode` on this plan.  Plans of >= 4 MiB per vector cut the call into K <= 32 chunks of
 * caller-order rows and overlap the upload of d0, the step over the rows whose inputs have arrived and the download
 * of d1 (three streams; PCIe is full duplex) — same kernels, every row computed once, same bits as the plain
 * sequence.  n_chunks = 0: the plain upload-step-download sequence is used (small plans, hooks, matrix-free mode, or
 * SAA_STEP_HOST_PIPELINE=0 in the environment; SAA_STEP_HOST_PIPELINE=K forces K chunks).  slice_end[c] / need_upload[c]
 * (capacity `cap`, may be NULL): compute chunk c ends at this internal slice and starts once the uploads of chunks
 * <= need_upload[c] are in — need_upload[c] - c is the pipeline lag the memory layout allows.
 */
int saa_plan_host_pipe_info(saa_plan *plan, int mode, int *n_chunks, int64_t *slice_end, int32_t *need_upload, int cap);
/*
 * Page-locked host memory for the d0 / dn / d1 vectors of saa_step_host[_ex] (the reference allocates them with
 * numpy, Data_prepare.py:215-217 and Dynamic_solver.py:18): copies from / to such memory are asynchronous and run at
 * the full PCIe rate.  Any host pointer is accepted by saa_step_host; pageable ones are staged by the CUDA driver.
 */
void *saa_host_alloc(int64_t bytes);
int saa_host_free(void *ptr);

/*
 * Record rows of the solution on the device every `save_every` steps (the d1_save / d_sol_shared
 * arrays of Data_prepare.py:219,238-240 and Online_predictor.py:244,260,301).
 *   dofs       local DOF ids to record (NULL: all n_dof), n_dofs their number
 *   capacity   number of snapshots the device buffer can hold (ring)
 */
int saa_plan_set_history(saa_plan *plan, const int64_t *dofs, int64_t n_dofs, int64_t capacity, int64_t save_every);
int64_t saa_plan_history_count(const saa_plan *plan);
/* copy snapshots [first, first+count) (snapshot-major, n_dofs values each) to host memory */
int saa_plan_read_history(saa_plan *plan, int64_t first, int64_t count, double *out_host);
/* same, into device memory (asynchronous on the plan's stream) — feeds the on-device LSTM predictor */
int saa_plan_read_history_dev(saa_plan *plan, int64_t first, int64_t count, double *out_dev);

/*
 * Synchronization-avoiding mode (Online_predictor.py:280-301): `table` holds n_rows predictions of the
 * shared DOFs, row-major (n_rows, 3*n_shared_ref) in the order of the reference's loc_dof_shared
 * (`dofs`, local DOF ids, Online_predictor.py:129).  A SAA_MODE_PREDICT step overwrites those DOFs of d1
 * with the next unread row.
 */
int saa_plan_set_prediction(saa_plan *plan, const int64_t *dofs, int64_t n_dofs, const double *table_dev,
                            int64_t n_rows);

/* ---- caller-provided transport: the neighbour messages pass through HOST memory, so any communicator the
 * caller already has (mpi4py as in the reference, gloo, ...) can carry them.  Layout of the send / receive
 * buffers: neighbour k (ascending rank nb_rank[k]) owns doubles [msg_off[k], msg_off[k+1]); both sides of an
 * interface list the common nodes in ascending global node id, 3 doubles (x, y, z) per node. ----------- */
int saa_plan_halo_layout(const saa_plan *plan, int *n_nb, int32_t *nb_rank, int64_t *msg_off, int capacity);
/* One synchronised step in two halves (Dynamic_solver.py:12 ... syn_cpus ... :29-32):
 *   begin: partial forces of the shared rows -> send_host (returns when the messages are in host memory;
 *          the interior rows keep running on the GPU while the caller exchanges)
 *   end:   recv_host (the neighbours' send buffers, same layout) -> rank-ordered sum, update, rotation   */
int saa_plan_step_begin_host(saa_plan *plan, double *send_host);
int saa_plan_step_end_host(saa_plan *plan, const double *recv_host);
/* syn_cpus (Distributed_tools.py:77-92) on a caller-provided force vector f (host, local DOF order):
 *   begin: pack the shared entries of f into send_host;  end: out = f_global[dofs_local]               */
int saa_plan_forces_begin_host(saa_plan *plan, const double *f_host, double *send_host);
int saa_plan_forces_end_host(saa_plan *plan, const double *recv_host, double *out_host);

/* ---- several partitions in one process (P ranks on fewer GPUs; exchange by device copies) ---------- */
int saa_group_create(saa_group **out, saa_plan **plans, int n_plans);
int saa_group_step(saa_group *grp, int64_t n_steps, int mode, int launch);
int saa_group_synchronize(saa_group *grp);
int saa_group_destroy(saa_group *grp);

/* ---- one partition per process / GPU of one node: halo exchange by peer-memory stores over NVLink -----------
 * Every rank exports the CUDA IPC handle of its receive area (saa_plan_peer_export), the handles are
 * distributed by the caller (torch.distributed / MPI), and saa_plan_peer_attach maps the neighbours' areas:
 *   handles64     n_nb x 64 bytes, neighbour k = nb_rank[k] of saa_plan_halo_layout
 *   remote_off    offset (doubles) of THIS rank's message inside neighbour k's receive area (its msg_off)
 *   remote_total  neighbour k's total message length (its msg_off[n_nb]) — the parity stride of its area
 *   remote_slot   index of THIS rank in neighbour k's neighbour list (selects its arrival flag)
 *   remote_n_nb   neighbour k's number of neighbours
 * Afterwards SAA_MODE_SYNC steps run as three stream-ordered kernels per step (pack + peer store + flag,
 * interior rows, wait + rank-ordered sum + update) with no host or NCCL call, replayed from a CUDA graph.
 * All ranks must execute the same number of synchronised steps.                                           */
int saa_plan_peer_export(saa_plan *plan, void *handle64, int64_t *total_msg);
int saa_plan_peer_attach(saa_plan *plan, int n_nb, const void *handles64, const int64_t *remote_off,
                         const int64_t *remote_total, const int32_t *remote_slot, const int32_t *remote_n_nb);

/* ---- one partition per process / GPU: halo exchange over NCCL (NVLink) -------------------------------- */
/* 128-byte NCCL unique id, created on one rank and distributed by the caller (torch.distributed) */
int saa_nccl_unique_id(void *id128);
int saa_plan_init_nccl(saa_plan *plan, const void *id128);

#ifdef __cplusplus
}
#endif
#endif /* SAA_FEM_H */
