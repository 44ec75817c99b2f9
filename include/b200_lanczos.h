/*
 * b200_lanczos.h — C ABI of libb200lanczos.so (sm_100a).
 *
 * Drop-in boundary for ONE hot path of pnkraemer/experiments-lanczos-adjoints:
 * Arnoldi/Lanczos factorisation with full re-orthogonalisation, its hand-derived
 * adjoint sweep, and the matvec back-ends they call.  The reference has no native
 * boundary (it is pure JAX); each entry point below cites the reference function it
 * replaces.  A reference maintainer binds these through `jax.ffi` (see INTEGRATION.md)
 * or, as the Python host layer in this repo does, through ctypes.
 *
 * Conventions
 *   - plain pointers and sizes only; every `*_dev` / unmarked data pointer is DEVICE
 *     memory unless the name ends in `_host`;
 *   - `dtype`: BL_F32 or BL_F64 — the arithmetic type of every vector/matrix argument of
 *     that call (the reference follows the dtype of the input vector, arnoldi.py:64-65);
 *   - Krylov bases are stored as K contiguous rows of length `ld` (row j = j-th basis
 *     vector, i.e. the reference's `Q.T`, lanczos.py:165), `ld >= n`, `ld*sizeof(T)` a
 *     multiple of 16, base pointers 16-byte aligned;
 *   - small dense matrices (H, dH) are row-major K x K in `dtype`;
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*), no host
 *     synchronisation, no allocation inside the Krylov calls: the caller supplies a
 *     workspace of `*_workspace_bytes()` bytes;
 *   - return value 0 on success, otherwise a BL_E* code; `bl_last_error()` gives the
 *     message (thread-local).
 */
#ifndef B200_LANCZOS_H
#define B200_LANCZOS_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { BL_F32 = 0, BL_F64 = 1 };
enum {
  BL_OK = 0,
  BL_EINVAL = 1,   /* bad argument (shape, alignment, enum) */
  BL_EDEPTH = 2,   /* krylov depth outside [1, n]: arnoldi.py:58-60 -> ValueError("depth") */
  BL_ECUDA = 3,    /* CUDA runtime error, see bl_last_error() */
  BL_ENOMEM = 4,
  BL_ECALLBACK = 5 /* a user matvec callback returned non-zero */
};

const char* bl_last_error(void);
const char* bl_version(void);

/* ---- device runtime (thin wrappers so the host layer needs no other CUDA binding) ---- */
int bl_device_count(int* count);
int bl_set_device(int device);
int bl_get_device(int* device);
int bl_device_sm_count(int* count);
int bl_malloc(void** ptr, size_t bytes);
int bl_free(void* ptr);
int bl_host_alloc(void** ptr, size_t bytes); /* pinned host memory */
int bl_host_free(void* ptr);
int bl_memcpy_h2d(void* dst, const void* src_host, size_t bytes, void* stream);
int bl_memcpy_d2h(void* dst_host, const void* src, size_t bytes, void* stream);
int bl_memcpy_d2d(void* dst, const void* src, size_t bytes, void* stream);
int bl_memset(void* dst, int value, size_t bytes, void* stream);
int bl_stream_create(void** stream);
int bl_stream_destroy(void* stream);
int bl_stream_sync(void* stream);
int bl_device_sync(void);
int bl_event_create(void** event);
int bl_event_destroy(void* event);
int bl_event_record(void* event, void* stream);
int bl_stream_wait_event(void* stream, void* event); /* work enqueued on `stream` afterwards waits for `event` */
int bl_event_sync(void* event);
int bl_event_elapsed_ms(void* start, void* stop, float* ms);
/* number of kernels this library has launched in this process (bench.py `gpu_launches`) */
int bl_launch_count(uint64_t* count);
/* Blocks per SM of the basis-streaming kernels for launches from now on: 2 (default: one run alone fills the
 * memory system), 1 (several independent runs in flight on separate streams: kernels of different runs share an
 * SM and fill each other's ramps and reduction tails), 0 = back to the default / BL_BLOCKS_PER_SM. */
int bl_set_blocks_per_sm(int blocks);
int bl_get_blocks_per_sm(int* blocks); /* what bl_set_blocks_per_sm last set (0 = environment / default) */

/* Per-kernel-class device timing for the roofline report.  Between begin and end every
 * streaming launch of the Krylov loops is bracketed by CUDA events on its own stream; end
 * synchronises and returns, per class, the launch count, the summed event time (ms) and the
 * summed ALGORITHMIC bytes (rows*n*w for basis rows, n*w per dense vector read or written,
 * nnz*(w+4)+4(n+1) for the sparse operand; DESIGN.md).  Classes: */
enum { BL_PROF_DOTS = 0, BL_PROF_COMBINE = 1, BL_PROF_MATVEC = 2, BL_PROF_VJP = 3, BL_PROF_OTHER = 4,
       BL_PROF_FUSED = 5, /* fused combine + dots (one read of the basis for both) */
       BL_PROF_NCLASS = 6 };
int bl_profile_begin(void);
int bl_profile_end(uint64_t* counts, double* ms, double* bytes); /* arrays of BL_PROF_NCLASS */
/* Time stamps inside the one-launch Gram-Schmidt step kernel (k_step_tma), taken by its block 0: per launch 8
 * values -- [0] globaltimer (ns) at entry, [1..7] SM clock after the dependency wait, phase 0's loads, phase 0's
 * grid-wide reduction, phase 1's stream, phase 1's reduction, phase 2's stream, exit.  begin() arms the next
 * 2048 launches; end() synchronises the device, copies `launches` x 8 stamps out and says whether the driver
 * accepted cooperative + programmatic launch together. */
int bl_step_trace_begin(void);
int bl_step_trace_end(unsigned long long* stamps_host, int64_t max_launches, int64_t* launches, int* pdl_accepted);

/* ---- row sharding: one large operator split by rows over several GPUs (one process each) ----
 * Every rank owns the same row range of every Krylov vector (`n` in the Krylov calls is the LOCAL
 * length).  The only cross-rank data the loops need are the reduced dot products / norms: when a
 * hook is installed, each streaming kernel stops after its local reduction, the hook is called
 * with the device array of `count` doubles (it must enqueue an in-place SUM all-reduce on
 * `stream`, e.g. ncclAllReduce), and the epilogue that consumes the numbers runs afterwards.
 * The hook is per host thread; NULL removes it.  The matvec's own exchange (all-gather / halo)
 * belongs to the operator (bl_op_callback_create). */
typedef int (*bl_allreduce_cb)(void* user, double* values_dev, int count, void* stream);
int bl_dist_set_reduce_hook(bl_allreduce_cb hook, void* user);

/* ---- NCCL from the library itself (csrc/nccl_comm.cu): one process per GPU, no PyTorch ------
 * libnccl.so.2 is loaded with dlopen on first use (BL_NCCL_LIB overrides the name).  Rank 0 makes the
 * 128-byte unique id, the caller's host channel (comm.py: a socket rendezvous from MASTER_ADDR / MASTER_PORT /
 * RANK) hands it to the other ranks, every rank calls init on its own device.  Collectives are in place on the
 * caller's stream: the ONE all-reduce that closes a probe-sharded Hutchinson estimate (hutchinson.py:54 summed
 * over GPUs), the all-reduce of the per-step dot products and the all-gather of the Lanczos vector of a
 * row-sharded operand.  op: 0 = sum, 1 = max.  reduce_hook(comm) installs the communicator as this host
 * thread's bl_dist_set_reduce_hook (NULL removes it). */
typedef struct bl_nccl bl_nccl_t;
int bl_dist_nccl_available(int* yes, int* version);
int bl_dist_nccl_unique_id(void* id_128);
int bl_dist_nccl_init(const void* id_128, int rank, int world, bl_nccl_t** comm);
int bl_dist_nccl_allreduce(bl_nccl_t* comm, void* buf, int64_t count, int dtype, int op, void* stream);
int bl_dist_nccl_allgather(bl_nccl_t* comm, const void* send, void* recv, int64_t count_per_rank, int dtype,
                           void* stream);
int bl_dist_nccl_sendrecv(bl_nccl_t* comm, const void* send, int send_peer, void* recv, int recv_peer, int64_t count,
                          int dtype, void* stream); /* a peer of -1 skips that half */
int bl_dist_nccl_reduce_hook(bl_nccl_t* comm);
int bl_dist_nccl_destroy(bl_nccl_t* comm);

/* Peer-memory communicator (NVLink / NVSwitch, one process per GPU of one box; at most 8 ranks):
 * the native alternative to the hook.  Each rank allocates a mailbox in its own HBM, the ranks
 * exchange the CUDA-IPC handles out of band (the host layer uses torch.distributed's object
 * all-gather), map each other's mailboxes and meet at a barrier.  While a communicator is active on
 * a host thread, every reduction of the Krylov loops on that thread is ONE single-block kernel per
 * rank: store the local sums into the peers' mailboxes, publish a sequence number, wait for the
 * peers' numbers, add the contributions in rank order (bit-identical on every rank) and run the
 * epilogue -- no NCCL launch, no host callback.  Ranks must issue the same sequence of Krylov calls.
 * A rank that waits ~10 s for a peer gives up, poisons the sums with NaN and sets the error word.
 * (Several ranks inside ONE process -- host threads, same-process connect -- additionally need every
 * kernel of the route loaded before the first exchange, because a lazy kernel load may synchronise the
 * context while the peer spins: run one pass with a one-rank communicator first, or set
 * CUDA_MODULE_LOADING=EAGER.) */
typedef struct bl_comm bl_comm_t;
int bl_dist_comm_create(int rank, int world, bl_comm_t** comm);
/* own mailbox pointer and / or its 64-byte cudaIpcMemHandle_t (either may be NULL) */
int bl_dist_comm_local(bl_comm_t* comm, void** mailbox, void* ipc_handle_64);
/* handles: world x 64 bytes in rank order (the own entry is ignored) */
int bl_dist_comm_connect_ipc(bl_comm_t* comm, const void* handles);
/* same-process variant (tests; several ranks driven by several host threads): mailbox pointers */
int bl_dist_comm_connect_ptrs(bl_comm_t* comm, void* const* mailboxes);
/* All-gather window: 4 * slot_bytes of this rank's HBM ([2 parities][2 slots][slot_bytes]) that the peers
 * map like the mailbox; needed by operands that all-gather a sharded vector (bl_op_sharded_sparse_create). */
int bl_dist_comm_window_create(bl_comm_t* comm, size_t slot_bytes, void* ipc_handle_64);
int bl_dist_comm_window_local(bl_comm_t* comm, void** window);
int bl_dist_comm_window_connect_ipc(bl_comm_t* comm, const void* handles);
int bl_dist_comm_window_connect_ptrs(bl_comm_t* comm, void* const* windows);
int bl_dist_comm_activate(bl_comm_t* comm); /* NULL deactivates; per host thread; wins over the hook */
int bl_dist_comm_error(bl_comm_t* comm, int* timed_out);
int bl_dist_comm_destroy(bl_comm_t* comm);

/* ---- operators: the `matvec(v, *params)` callback of the reference ------------------
 * An operator owns its index structures and a gradient accumulator for its parameters.
 *   set_params : bind parameter values (device pointers, reference order)
 *   matvec     : y = A(x; params)                     [what `matvec(v, *params)` returns]
 *   vjp        : z = A^T lam  and  grad += d<lam, A(q; params)>/dparams
 *                [what jax.vjp(lambda u, p: matvec(u, *p), q, params)(lam) returns,
 *                 arnoldi.py:207-209]; z may be NULL (three-term adjoint, lanczos.py:328-329)
 *   grad_zero / grad_export : reset / read the accumulator (one buffer per parameter).
 */
typedef struct bl_operator bl_operator_t;

/* Sparse COO/BCOO operand (suite_sparse/benchmark.py:61-68, util/exp_util.py:35-42).
 * One parameter: the COO `data` array (nnz values, COO order; duplicates are summed by the
 * matvec and stay independent parameters).  Index work (COO -> CSR -> SELL-32 for A and
 * A^T) happens here, on the host, and is bit-exact against oracle/operators.py. */
int bl_op_sparse_create(int64_t n_rows, int64_t n_cols, int64_t nnz, const int32_t* coo_row_host,
                        const int32_t* coo_col_host, bl_operator_t** op);
/* A second handle on the same sparsity pattern with values and cotangent accumulator of its own (independent Krylov
 * runs on different streams need one operator each): the finished index work is shared, not redone. */
int bl_op_sparse_clone(const bl_operator_t* op, bl_operator_t** clone);
/* CSR view of the index work, for the bit-exact tests: row_ptr[n_rows+1], col_idx[nnz],
 * perm[nnz] (perm[k] = COO position of CSR slot k).  Any pointer may be NULL. */
int bl_op_sparse_export_csr(const bl_operator_t* op, int32_t* row_ptr_host, int32_t* col_idx_host,
                            int32_t* perm_host);
/* SELL-32 view: slice_ptr[n_slices+1] (int64), slot_of_csr[nnz] (int64). */
int bl_op_sparse_export_sell(const bl_operator_t* op, int transpose, int64_t* slice_ptr_host,
                             int64_t* slot_of_csr_host);

/* Row-sharded sparse operand over peer memory ("one large operator"): rank r owns rows [r*chunk, (r+1)*chunk)
 * of every vector (chunk a multiple of 32; width = world * chunk).  A_local / B_local are rectangular
 * chunk x width sparse operands holding the local rows of A and of A^T (they must outlive this object).
 * matvec: all-gather of the vector through the communicator's window (one kernel: NVLink stores into every
 * peer's window, sequence-number handshake), then the local rows of A.  vjp: gathers q and lambda, applies
 * the local rows of A^T, accumulates the cotangent of the entries of the local rows.  Two parameters:
 * the values of A_local and of B_local; the second gradient is zero (every entry is owned by its row). */
int bl_op_sharded_sparse_create(bl_operator_t* A_local, bl_operator_t* B_local, bl_comm_t* comm, int64_t chunk,
                                int64_t width, bl_operator_t** op);

/* Dense operand of the reference's tests: mode 0 `p @ s` (test_hessenberg_forward.py:20),
 * mode 1 `(p + p.T) @ s` (test_tridiag_adjoint.py:20-21).  One parameter: p (n x n row-major). */
int bl_op_dense_create(int64_t n, int mode, bl_operator_t** op);

/* Matrix-free Gram operator `(K(X,X) + noise I) v` (util/gp_util.py:69-184, 525-543).
 * kind 0 Matern-3/2, 1 Matern-1/2, 2 RBF.  X_host is n x d row-major doubles (converted per
 * dtype on bind).  Three parameters: raw_lengthscale (d), raw_outputscale (1), noise (1). */
int bl_op_gram_create(int64_t n, int64_t d, int kind, const double* X_host, bl_operator_t** op);
/* Which kernel evaluates the pairwise distances of an fp32 Gram operator: 0 automatic (tensor cores
 * when d <= 20), 1 FP32 ALU kernel, 2 tcgen05 kernel (TF32 hi/lo split operands, fp32 accumulator in
 * TMEM; gram_tc.cuh).  fp64 always uses the FP64 ALU kernel.  Takes effect at the next bind. */
int bl_op_gram_set_path(bl_operator_t* op, int path);
/* Diagnostic for the parity tests of the contraction itself: the tensor-core accumulator
 * x_i.x_j - |x_j|^2/2 of the scaled inputs (gp_util.py:87-92; s2_ij = |x_i|^2 - 2 acc_ij, the row term
 * is added in the epilogue) for the tile of rows [128 row_tile, +128) x columns [256 col_tile, +256),
 * written to out_host[128][256] (fp32; entries beyond n are padding).  col_tile must be the first tile of a column split.  Synchronises `stream`. */
int bl_op_gram_tile_distances(bl_operator_t* op, int64_t row_tile, int64_t col_tile, float* out_host, void* stream);
/* Cross-covariance of a Gram operator with m test points X* (the prediction half of a GP): the test points
 * are scaled (and packed for the tensor-core path) with the kernel parameters bound to `gram`, and again
 * whenever `gram` is re-bound; its noise is never read.  `gram` must outlive the object.  Xtest_host is
 * m x d row-major doubles.  dtype must be the dtype `gram` was last bound with.
 *   matvec     : y (m) = K(X*, X) v (v of length n), the square sweeps' kernels on a rectangular operand;
 *   columns    : out[b * ld + j] = k(x*_{first+b}, x_j), b < count <= 65535, j < n (ld >= n);
 *   prior_diag : out[t] = k(x*_t, x*_t), the kernel formula at s2 = 0 (Matern: sigma (1 + sqrt(eps)) e^-sqrt(eps)).
 * fp32 on tensor cores: s2 = |x|^2 + |y|^2 - 2 x.y is exact only on the square operator's diagonal, so a test
 * point that coincides with a training point gets s2 = O(eps |x|^2) rather than 0. */
typedef struct bl_gram_cross bl_gram_cross_t;
int bl_gram_cross_create(bl_operator_t* gram, int64_t m, const double* Xtest_host, bl_gram_cross_t** out);
int bl_gram_cross_destroy(bl_gram_cross_t* cross);
int bl_gram_cross_matvec(bl_gram_cross_t* cross, int dtype, const void* v, void* y, void* stream);
int bl_gram_cross_columns(bl_gram_cross_t* cross, int dtype, int64_t first, int64_t count, void* out, int64_t ld,
                          void* stream);
int bl_gram_cross_prior_diag(bl_gram_cross_t* cross, int dtype, void* out, void* stream);

/* Wave-equation stencil operand (util/pde_util.py:126-157): state (u, du) of 2 g^2 values,
 * A(u,du) = (du, scale^2 * conv3x3(stencil, edge_pad(u))).  One parameter: scale (g*g). */
int bl_op_wave_create(int64_t grid, const double* stencil3x3_host, bl_operator_t** op);
/* Row-sharded form: a slab of `rows` grid rows x `cols` columns with an optional neighbour above /
 * below.  State (u_slab, du_slab) of 2*rows*cols values; parameter scale (rows*cols).  Before each
 * matvec the caller writes the neighbours' boundary rows of u into halo buffers 0 (top) / 1 (bottom);
 * before each vjp: rows of q_u into 0/1, rows of lam_du into 2/3; the neighbours' rows of `scale`
 * into 4/5 once per bind.  bl_op_wave_halo returns the device pointer of buffer `which`
 * (cols values of the bound dtype). */
int bl_op_wave_slab_create(int64_t rows, int64_t cols, int has_top, int has_bottom, const double* stencil3x3_host,
                           bl_operator_t** op);
int bl_op_wave_halo(bl_operator_t* op, int which, void** ptr);
/* Native halo exchange: slab `rank` of `world` slabs stacked top to bottom.  With a communicator set,
 * matvec / vjp / set_params push the boundary rows into the neighbours' mailboxes themselves (one
 * single-block kernel per exchange, see bl_dist_comm_create) -- the operator is then a plain operand
 * of the Krylov calls, with no host callback on the path.  NULL returns to caller-filled halos. */
int bl_op_wave_set_comm(bl_operator_t* op, bl_comm_t* comm);

/* User-supplied matvec: the host layer passes C callbacks that enqueue work on `stream`.
 * matvec_cb(user, dtype, x, y, stream); vjp_cb(user, dtype, q, lam, z_or_null, stream). */
typedef int (*bl_matvec_cb)(void* user, int dtype, const void* x, void* y, void* stream);
typedef int (*bl_vjp_cb)(void* user, int dtype, const void* q, const void* lam, void* z, void* stream);
int bl_op_callback_create(int64_t n, bl_matvec_cb matvec_cb, bl_vjp_cb vjp_cb, void* user,
                          bl_operator_t** op);

int bl_op_destroy(bl_operator_t* op);
int bl_op_size(const bl_operator_t* op, int64_t* n);
int bl_op_num_params(const bl_operator_t* op, int* num);
int bl_op_param_size(const bl_operator_t* op, int index, int64_t* numel);
int bl_op_set_params(bl_operator_t* op, int dtype, const void* const* params, int num, void* stream);
int bl_op_matvec(bl_operator_t* op, int dtype, const void* x, void* y, void* stream);
int bl_op_vjp(bl_operator_t* op, int dtype, const void* q, const void* lam, void* z, void* stream);
int bl_op_grad_zero(bl_operator_t* op, int dtype, void* stream);
int bl_op_grad_export(bl_operator_t* op, int dtype, void* const* grads, int num, void* stream);

/* ---- Arnoldi with CGS2 re-orthogonalisation and its adjoint (arnoldi.py) --------------- */
size_t bl_arnoldi_workspace_bytes(int64_t n, int64_t krylov_depth, int dtype);

/* Bits of the `second_pass` argument of the forward entry points (0 / 1 keep their meaning). */
#define BL_FWD_SECOND_PASS 1 /* second Gram-Schmidt pass, arnoldi.py:91-92 */
#define BL_FWD_SYMMETRIC 2   /* with BL_FWD_SECOND_PASS, symmetric operand (lanczos.tridiag(reortho="full")):
                              * the first pass (arnoldi.py:87-88) takes h = Q^H v with rows i-1, i only -- the
                              * other entries are O(eps |A|) and H[j < i-1, i] is stored as zero; the second
                              * pass still projects against every row, so Q stays orthonormal to rounding.
                              * The basis is read twice per step instead of three times. */

/* arnoldi._forward (arnoldi.py:57-101).  second_pass & BL_FWD_SECOND_PASS performs the second
 * Gram-Schmidt pass (`reortho_ != "none"`, arnoldi.py:91; the reference's default always
 * does, arnoldi.py:26).  Outputs: Q (K rows, ld), H (K x K), r (n), c (1 element = 1/||v||).
 * Runs as bl_arnoldi_forward_batch with count = 1 and ldv = n; the workspace may be as small as what one run
 * uses (bl_arnoldi_workspace_bytes is always enough). */
int bl_arnoldi_forward(bl_operator_t* op, int dtype, int64_t n, int64_t krylov_depth, int second_pass,
                       const void* v, void* Q, int64_t ld, void* H, void* r, void* c,
                       void* workspace, size_t workspace_bytes, void* stream);

/* Bits of the `reortho_full` argument of the adjoint entry points (0 / 1 keep their meaning). */
#define BL_ADJ_REORTHO_FULL 1 /* `reortho == "full"`: re-project lambda, arnoldi.py:201-204 */
#define BL_ADJ_SYMMETRIC 2    /* the operand is symmetric and the forward ran with second_pass (what
                               * lanczos.tridiag(reortho="full") guarantees, lanczos.py:152-169): H is
                               * tridiagonal up to rounding, and `Lambda beta_plus` (arnoldi.py:218) keeps
                               * only its O(1) term H[idx, idx+1] Lambda[idx+1].  Results change by
                               * O(eps K |Lambda|); K^2/2 fewer basis rows are read per sweep. */
#define BL_ADJ_TRIDIAG_COTANGENT 4 /* with BL_ADJ_SYMMETRIC | BL_ADJ_REORTHO_FULL and dQ == NULL: dH is
                               * tridiagonal (the cotangent of lanczos.tridiag's (alpha, beta), lanczos.py:162-164).
                               * Gamma (arnoldi.py:213) is then banded up to rounding, because the re-projected
                               * lambda satisfies Q^T lambda = dH[:, idx] exactly: the dots Q^T(A^T lambda) are
                               * taken with rows idx-2..idx and Q (Gamma+Gamma^T)[idx] with rows idx-2..idx+2. */

/* arnoldi._adjoint (arnoldi.py:104-220).  reortho_full & BL_ADJ_REORTHO_FULL re-projects lambda
 * (`reortho == "full"`, arnoldi.py:201-204).  dQ (K rows, ld), dr, dc may be NULL (= zero
 * cotangent, the SLQ case of SURVEY 3.3).  Lambda is a K x ld scratch basis supplied by the
 * caller.  Output dv (n); parameter gradients accumulate in `op`.  Runs as bl_arnoldi_adjoint_batch with
 * count = 1 and lddv = n (same workspace rule as bl_arnoldi_forward). */
int bl_arnoldi_adjoint(bl_operator_t* op, int dtype, int64_t n, int64_t krylov_depth, int reortho_full,
                       const void* Q, int64_t ld, const void* H, const void* r, const void* c,
                       const void* dQ, const void* dH, const void* dr, const void* dc, void* dv,
                       void* Lambda, void* workspace, size_t workspace_bytes, void* stream);

/* Lockstep batch over `count` independent start vectors (Hutchinson probes; the reference's
 * `jax.vmap(integrand)` of hutchinson.py:14): the runs advance together and every step issues ONE batched
 * matvec (operators that share work between vectors -- the Gram operator evaluates each kernel tile once
 * for all of them -- make `count` runs cost little more than one).  Layouts: v (count, ldv), Q (count, K, ld),
 * H (count, K, K), r (count, ld), c (count); workspace = count * bl_arnoldi_workspace_bytes.  The adjoint
 * takes per-run cotangents dH (count, K, K) and, each optional (NULL = zero, the SLQ case), dQ (count, K, ld),
 * dr (count, ld), dc (count) -- the general cotangent of `jax.vmap(solve)` over initial conditions
 * (experiments/applications/partial_differential_equation/train.py:104-110) -- and writes dv (count, lddv) and
 * Lambda (count, K, ld).  The parameter cotangent is the SUM over the runs: operators with a deferred cotangent
 * (bl_op_deferred_grad) send all count*K (lambda, q) pairs through one batched pass at the end, the others
 * accumulate per step. */
int bl_arnoldi_forward_batch(bl_operator_t* op, int dtype, int64_t n, int64_t krylov_depth, int second_pass,
                             int64_t count, const void* v, int64_t ldv, void* Q, int64_t ld, void* H, void* r, void* c,
                             void* workspace, size_t workspace_bytes, void* stream);
int bl_arnoldi_adjoint_batch(bl_operator_t* op, int dtype, int64_t n, int64_t krylov_depth, int reortho_full,
                             int64_t count, const void* Q, int64_t ld, const void* H, const void* r, const void* c,
                             const void* dQ, const void* dH, const void* dr, const void* dc, void* dv, int64_t lddv,
                             void* Lambda, void* workspace, size_t workspace_bytes, void* stream);
/* 1 when the operator defers its parameter cotangent to one batched pass per adjoint sweep. */
int bl_op_deferred_grad(bl_operator_t* op, int dtype, int* yes);

/* ---- three-term Lanczos without re-orthogonalisation and its adjoint (lanczos.py:215-335) */
size_t bl_lanczos3_workspace_bytes(int64_t n, int64_t krylov_depth, int dtype);
/* xs: K+1 rows (ld); alphas[K]; betas[K] (betas[K-1] is the remainder norm). */
int bl_lanczos3_forward(bl_operator_t* op, int dtype, int64_t n, int64_t krylov_depth, const void* v,
                        void* xs, int64_t ld, void* alphas, void* betas, void* workspace,
                        size_t workspace_bytes, void* stream);
/* dxs: K+1 rows (ld) or NULL; dalphas[K], dbetas[K]; vnorm: 1 element (||v||, device).
 * Output dv (n); the single parameter's gradient accumulates in `op` (lanczos.py:329). */
int bl_lanczos3_adjoint(bl_operator_t* op, int dtype, int64_t n, int64_t krylov_depth, const void* xs,
                        int64_t ld, const void* alphas, const void* betas, const void* dxs,
                        const void* dalphas, const void* dbetas, const void* vnorm, void* dv,
                        void* workspace, size_t workspace_bytes, void* stream);

/* ---- linear solves of the GP path (cg.py, low_rank.py) -------------------------------------
 * Preconditioner of low_rank.py:10-60: v -> (s I + L L^T)^{-1} v (Woodbury).  `L_rows` holds the factor
 * as `rank` rows of length n (row k = k-th column of the reference's (n, rank) matrix), row stride ld;
 * the buffer must outlive the object.  create() forms L^T L on the device (synchronises `stream`);
 * set_shift(s) inverts the rank x rank capacitance matrix on the host (s = the noise); apply() is three
 * kernels on the stream. */
typedef struct bl_precond bl_precond_t;
int bl_precond_create(int dtype, int64_t n, int64_t rank, const void* L_rows, int64_t ld, void* stream,
                      bl_precond_t** out);
int bl_precond_set_shift(bl_precond_t* p, double shift, void* stream);
int bl_precond_apply(bl_precond_t* p, int dtype, const void* v, void* out, void* stream);
int bl_precond_destroy(bl_precond_t* p);

/* Preconditioned conjugate gradients, x0 = 0 (cg.py:20-131).  precond == NULL: plain CG.
 *   atol <  0 : pcg_fixed_step(max_steps) -- exactly max_steps iterations, nothing synchronises;
 *   atol >= 0 : pcg_adaptive(atol, rtol, maxiter = max_steps, miniter = min_steps) -- iterate while
 *               rms(r / (atol + |x| rtol)) > 1 or fewer than min_steps steps were taken.  The device
 *               freezes x and r at the iteration where that condition fails; the host reads the flag
 *               every `check_every` iterations (0 = default 8) and synchronises the stream to do so.
 * x, r: solution and residual b - A x (n values each); *num_steps_host: iterations taken.
 * Divisions are cg.py's _safe_divide (a / b where |b| > eps^2, else a). */
size_t bl_pcg_workspace_bytes(int64_t n, int dtype);
int bl_pcg_solve(bl_operator_t* op, int dtype, int64_t n, const void* b, bl_precond_t* precond, int64_t max_steps,
                 int64_t min_steps, double atol, double rtol, int check_every, void* x, void* r,
                 int64_t* num_steps_host, void* workspace, size_t workspace_bytes, void* stream);
/* `count` independent solves A X[c] = B[c] in lockstep, each column under bl_pcg_solve's rules (same
 * modes, _safe_divide, min_steps, its own freeze).  Every iteration takes one matvec_batch over the columns
 * the host still knows to be active (the Gram operator evaluates each kernel tile once for up to 16 of
 * them); dots, step lengths and updates are one launch per vector operation for all columns.  The host
 * reads the columns' flags back in one copy every `check_every` iterations.  B, X, R: count rows of n
 * values, row stride ld (ld >= n, ld * dtype size a multiple of 16 bytes); num_steps_host: count values.
 * The preconditioner is applied column by column. */
/* workspace of bl_pcg_solve_batch: pass the row stride ld as n */
size_t bl_pcg_batch_workspace_bytes(int64_t n, int64_t count, int dtype);
int bl_pcg_solve_batch(bl_operator_t* op, int dtype, int64_t n, int64_t count, const void* B, int64_t ld,
                       bl_precond_t* precond, int64_t max_steps, int64_t min_steps, double atol, double rtol,
                       int check_every, void* X, void* R, int64_t* num_steps_host, void* workspace,
                       size_t workspace_bytes, void* stream);
/* out[j] = <X[j], Y[j]> for j < count (rows of n values, row stride ld; out: count doubles on the device) */
int bl_rows_dot_pairs(int dtype, int64_t n, int64_t count, const void* X, const void* Y, int64_t ld, double* out,
                      void* stream);

/* Partial Cholesky factorisation of the lazily evaluated matrix of `op` (dense operand: its matrix; Gram
 * operand: the kernel matrix WITHOUT the noise term, gp_util.py:257-258).  pivot = 0: low_rank.py:63-118;
 * pivot = 1: low_rank.py:120-225 (first arg-max of |diag - sum L^2| over the permuted positions; the
 * factor is returned in the original row order).  L_rows: `rank` rows of length n, stride ld.
 * success_host / pivots_host (optional; reading them synchronises the stream): low_rank.py:198's flag and
 * the chosen pivots (original indices).  rank < 1 or rank > n -> BL_EINVAL with the reference's message. */
size_t bl_cholesky_workspace_bytes(int64_t n, int64_t rank, int dtype);
int bl_cholesky_partial(bl_operator_t* op, int dtype, int64_t n, int64_t rank, int pivot, void* L_rows, int64_t ld,
                        int* success_host, int64_t* pivots_host, void* workspace, size_t workspace_bytes,
                        void* stream);

/* ---- small vector helpers used by the host-side wrappers (lanczos.py:162-167, 24-26) ---- */
/* out[0] = sum_i x_i y_i  (device scalar, dtype) */
int bl_vec_dot(int dtype, int64_t n, const void* x, const void* y, void* out, void* workspace,
               size_t workspace_bytes, void* stream);
/* out = a*x + b*y  (host scalars; y may be NULL when b == 0; out may alias x or y) */
int bl_vec_axpby(int dtype, int64_t n, double a, const void* x, double b, const void* y, void* out,
                 void* stream);
/* rows x cols matrix, transpose copy (reference layout (n,K) <-> basis layout (K,ld)) */
int bl_transpose(int dtype, int64_t rows, int64_t cols, const void* src, int64_t ld_src, void* dst,
                 int64_t ld_dst, void* stream);
/* out[j] = sum_i M[j, i] x[i] for j < nrows (rows of length ld; device output in dtype) */
int bl_rows_dot(int dtype, int64_t n, int64_t nrows, const void* M, int64_t ld, const void* x,
                void* out, void* workspace, size_t workspace_bytes, void* stream);
/* out = sum_j coef_host[j] * M[j, :]  (+ out if accumulate) */
int bl_rows_combine(int dtype, int64_t n, int64_t nrows, const void* M, int64_t ld,
                    const double* coef_host, int accumulate, void* out, void* workspace,
                    size_t workspace_bytes, void* stream);
size_t bl_vec_workspace_bytes(void);

#ifdef __cplusplus
}
#endif
#endif /* B200_LANCZOS_H */
