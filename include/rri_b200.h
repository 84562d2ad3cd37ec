/*
 * rri_b200.h -- C-ABI of the B200-native RRI / HALS / WRRI sweep engine (librri_b200.so).
 *
 * The reference (maksimt/rri_nmf) has no FFI: its only seam for this path is the Python call
 *     nmf(X, k, **kwargs) -> dict            src/rri_nmf/nmf.py:98-108 (signature), :551-560 (return)
 * whose two inner loops (`for iter_no ... for t in range(k)`, nmf.py:377, :415-476) are what this
 * library replaces.  Each entry point below names the reference lines it stands in for.  All
 * pointers are plain device (or, where said, host) pointers; no torch types cross this boundary.
 *
 * Conventions: every call returns 0 on success, non-zero on failure; the message is available from
 * rri_last_error() (thread-local).  A handle is bound to one CUDA device and is not thread-safe.
 * Matrices are C-contiguous row-major like the reference's ndarrays: X[n,d] (leading dimension
 * ldX elements), W[n,k], T[k,d].  `stream` is a cudaStream_t passed as void*.
 */
#ifndef RRI_B200_H
#define RRI_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rri_handle_s* rri_handle_t;

enum { RRI_F32 = 0, RRI_F64 = 1 };                 /* element type of X, W, T (reference: dtype follows inputs) */
enum { RRI_MATH_IEEE = 0, RRI_MATH_TF32 = 1 };     /* contraction arithmetic of the two X passes (hals/f32 only) */
enum { RRI_ORDER_RRI = 0, RRI_ORDER_HALS = 1 };    /* interleaved (nmf.py:415-476) / block order */
enum { RRI_MASK_NONE = 0, RRI_MASK_REAL = 1, RRI_MASK_U8 = 2 };   /* W_mat storage: same dtype as X, or 0/1 bytes */

/* bits of the flags word written by rri_sweeps / rri_topics */
enum {
    RRI_FLAG_ZERO_T    = 1,   /* some sum(T[t,:]) <= 1e-10          nmf.py:757-758 */
    RRI_FLAG_ZERO_W    = 2,   /* some sum(W[:,t]) <= 1e-10          nmf.py:793-794, assert :476 */
    RRI_FLAG_UNBOUNDED = 4,   /* denominator <= 0 with no bound     optimization.py:60-67, :76-77, :105-107 */
    RRI_FLAG_NONFINITE = 8,   /* NaN/Inf produced */
    RRI_FLAG_NOT_IMPLEMENTED = 16  /* project_T_each_iter, block order: a denominator <= 0 with t_row_sum != 1
                                      (optimization.py:60-74 raises NotImplementedError) */
};

/* keyword arguments of nmf() that reach the hot path (nmf.py:98-108) */
typedef struct rri_params_s {
    double reg_w_l1, reg_w_l2, reg_t_l1, reg_t_l2;   /* nmf.py:437-438, :464-465 */
    double ub_w, ub_t;     /* qf_min `ub` (= w_row_sum / t_row_sum); <= 0 means None.  Only the
                              vector-c (masked) branch clips, optimization.py:82-83; the scalar
                              branch ignores ub for c>0 (:53-59) and uses it for c<=0 (:63-65) */
    double eps;            /* eps_div_by_zero = np.spacing(10), nmf.py:52, optimization.py:5 */
    int32_t fix_W, fix_T;  /* nmf.py:417, :460.  fix_T = W-only sweeps (transform()).  fix_W must be 0: the reference's
                              T-only sweep also rescales W (:450-452); the host shell drives it from rri_partials_T */
    int32_t simplex_T;     /* project_T_each_iter with s = ub_t: optimization.py:58-59 + nmf.py:759-761 (unmasked);
                              optimization.py:85-87 (masked / observed entries: rescale the clipped solution to sum s) */
    int32_t sp_refresh_every;  /* observed-entries handles, interleaved order: rebuild the residual copies from the factors
                              every this many sweeps of one rri_sweeps call (0 / 1 = every sweep: N sweeps in one call
                              == N calls of one sweep, bit for bit) */
} rri_params_t;

/* library / build information; never touches the GPU (safe on a CPU-only host) */
const char* rri_version(void);
const char* rri_last_error(void);

/* Create a sweep engine for one row shard X_i[n_local, d] with rank-k factors on CUDA device `device`.
 * Replaces the per-call setup of nmf(): nmf.py:272, :351-358. */
int rri_create(rri_handle_t* out, int64_t n_local, int64_t d, int32_t k,
               int32_t dtype, int32_t math, int32_t order, int32_t device);
int rri_destroy(rri_handle_t h);

/* Attach an NCCL communicator (ncclComm_t as void*) for row-sharded multi-GPU runs.  The shard
 * statistic that is all-reduced is the one the reference defines at nmf.py:680-686 / :706-713.
 * `nccl_lib_path` may be NULL when libnccl.so.2 is already loaded in the process. */
int rri_set_comm(rri_handle_t h, void* nccl_comm, int32_t rank, int32_t world, const char* nccl_lib_path);

/* NCCL bootstrap without torch types: rank 0 calls rri_nccl_unique_id, the 128 bytes are broadcast by
 * the host (torch.distributed), every rank calls rri_nccl_comm_create; the result is what
 * rri_set_comm takes.  (The reference has no communication backend; SURVEY.md §2.1.) */
int rri_nccl_unique_id(char id_out[128], const char* nccl_lib_path);
int rri_nccl_comm_create(void** comm_out, const char id[128], int32_t rank, int32_t world, int32_t device,
                         const char* nccl_lib_path);
int rri_nccl_comm_destroy(void* comm);

/* Peer-memory exchange for the block-order T half-step (optional; replaces the NCCL all-reduce of
 * [X_i'W_i | W_i'W_i] by in-place NVLink reads inside the update kernel).  After rri_bind every rank calls
 * rri_peer_export (64-byte CUDA IPC handle of its exchange buffer), the host all-gathers the handles
 * (rank-major, 64 bytes each) and every rank calls rri_peer_import.  Unmasked hals handles only. */
int rri_peer_export(rri_handle_t h, char handle_out[64]);
int rri_peer_import(rri_handle_t h, const char* handles, int32_t rank, int32_t world);
/* switch the exchange on once EVERY rank has imported successfully (the host checks); off = NCCL path */
int rri_peer_enable(rri_handle_t h, int32_t on);
/* unmap the peers' buffers; all ranks call it (and synchronise) BEFORE any rank destroys its handle */
int rri_peer_close(rri_handle_t h);

/* Optional, before rri_bind on a hals handle: storage [d, ldXt] (ldXt >= n rounded up to 16 bytes) owned by the
 * caller for the engine's transposed copy of X, so that it comes from the caller's allocator (torch's caching
 * allocator: no cudaMalloc/cudaFree of a data-sized buffer per fit).
 * With RRI_MATH_TF32 the same storage can hold, instead, 16-bit copies of X and X': fp16(tf32(x) * 2^e) with one
 * power-of-two scale, exact when every nonzero TF32 value of X lies within 30 binades of fp16's normal range under
 * that scale and X holds no inf / nan.  The block-order contractions then read half the bytes and see the same
 * operands.  rri_bind checks the data and takes that form when it is exact and the storage holds
 * 2 * (n * d8 + d * n8) bytes (d8, n8: d, n rounded up to 8); otherwise it builds the fp32 copy.  Environment
 * RRI_X16=0 (read at every rri_bind) keeps the fp32 copy.  rri_x_operand_bits reports the choice. */
int rri_set_transpose_storage(rri_handle_t h, void* Xt_dev, int64_t ldXt);

/* Bind the data (and optional elementwise weights W_mat) resident in device memory.  In hals order
 * the engine builds its own transposed copy of X (one extra pass, once).  nmf.py:98 (X, W_mat). */
int rri_bind(rri_handle_t h, const void* X_dev, int64_t ldX,
             const void* mask_dev, int32_t mask_kind, int64_t ldM, void* stream);
/* The storage of X the contractions of the block order read: 16 (the 16-bit copies described above), or the bits of
 * the handle's element type. */
int rri_x_operand_bits(rri_handle_t h, int32_t* bits);

/* Observed-entries binding for the recommender setting (SURVEY.md §8 f4): the (i, j, rating) triples of
 * sklearn_interface.py:78-83 as a CSR matrix of the LOCAL rows, instead of the densified X and the dense 0/1
 * W_mat of :97-102.  rowptr_dev[n_local+1] (int64), col_dev[nnz] (int32, strictly ascending inside a row),
 * val_dev[nnz] (element type of the handle); weight_dev[nnz] optional entry weights (NULL = 1, i.e. W_mat is the
 * indicator of the stored entries).  A stored entry is an observed one, whatever its value.  The engine builds its
 * column-major copy once (synchronises `stream`); the three CSR arrays must stay alive while the handle is used.
 * Every masked entry point (rri_sweeps, rri_topics, rri_objective, rri_partials_T, rri_topic_sums) then runs
 * nmf.py:687-701 / :735-746 with traffic proportional to nnz.  IEEE math only; a handle is bound once. */
int rri_bind_csr(rri_handle_t h, int64_t nnz, const int64_t* rowptr_dev, const int32_t* col_dev,
                 const void* val_dev, const void* weight_dev, void* stream);

/* Zero-filled sparse binding: the CSR matrix is an ordinary non-negative matrix stored sparsely (a tf-idf
 * document-term matrix); every entry is fitted, the unstored ones as 0.  Same CSR contract as rri_bind_csr
 * (int64 rowptr, int32 strictly ascending columns, nnz < 2^31, the three arrays stay alive while the handle is
 * used).  Handles created with RRI_MATH_IEEE (fp32 or fp64), in either order.  The column orientation and the chunk
 * plan of long rows / columns are built once (synchronises `stream`); the workspace grows with nnz and (n + d) * k,
 * never with n * d.  RRI_ORDER_HALS: the block-order half-steps take X T' and X' W from a sparse x dense contraction.
 * RRI_ORDER_RRI: the interleaved order of the dense path with one fused pass over the rows and the columns per topic
 * (y = X T_t', p = w_t+1' X), three launches per topic.  On such a handle: rri_sweeps (either order, and fix_T, which
 * runs the block-order W half), rri_objective and rri_objective_contraction (both through the identity, ||X||^2 from
 * the stored values in fp64), rri_partials_T (nw of length 1), rri_topic_sums, rri_stats, rri_spmm and
 * rri_profile_kernel (which = 0: the fused pass of an rri-order handle, 1 / 2: the W- / T-half contraction, 3 / 4:
 * the whole half-steps of a block-order handle).  rri_topics serves the rri-order handles and refuses the block-order
 * ones; rri_peer_export refuses both: row shards use the NCCL all-reduce. */
int rri_bind_csr_zero(rri_handle_t h, int64_t nnz, const int64_t* rowptr_dev, const int32_t* col_dev,
                      const void* val_dev, void* stream);

/* Sparse x dense product on a sparse handle (rri_bind_csr or rri_bind_csr_zero), for the randomized SVD of the NNDSVD
 * initialisation (nmf.py:840-843 initialises on W_mat o X):
 *     transpose = 0:  C[n_local, width] = X  B[d, width]        (over the CSR rows)
 *     transpose = 1:  C[d, width]       = X' B[n_local, width]  (over the CSC columns)
 * B and C are row-major with leading dimensions ldb, ldc >= width (in elements), element type of the handle, device
 * memory.  X is the zero-filled matrix of the stored entries; on an observed-entries handle with entry weights it is
 * w o x.  Operands wider than 256 columns run as panels of 256 columns, one launch each.  Summation order is fixed
 * (no float atomics): repeated calls give identical bits.  An observed-entries handle builds its chunk plans (and, with
 * weights, a weighted copy of the values: 2 * nnz elements, freed with the handle) on its first call, which
 * synchronises `stream`.  Calls and sweeps on one handle must be issued on one stream. */
int rri_spmm(rri_handle_t h, int32_t transpose, const void* B_dev, int64_t ldb, void* C_dev, int64_t ldc, int32_t width,
             void* stream);

/* Run n_sweeps full sweeps in place on W_dev[n_local,k], T_dev[k,d]:  nmf.py:377, :415-476
 * (+ masked branches :687-701, :735-746; qf_min optimization.py:51-59, :75-87).
 * flags_host (may be NULL): receives the OR of RRI_FLAG_* over all sweeps (forces a stream sync).
 * N sweeps in one call == N calls of one sweep, bit for bit (tests/test_nmf.py:97-109). */
int rri_sweeps(rri_handle_t h, void* W_dev, void* T_dev, int32_t n_sweeps,
               const rri_params_t* p, int32_t* flags_host, void* stream);

/* Run topics [t_begin, t_end) of ONE rri-order sweep (the body of the loop at nmf.py:415) so a host
 * policy (topic reset, nmf.py:762-783, :796-816) can act between topics.  rri order only (dense, masked,
 * observed-entries or zero-filled sparse data). */
int rri_topics(rri_handle_t h, void* W_dev, void* T_dev, int32_t t_begin, int32_t t_end,
               const rri_params_t* p, int32_t* flags_host, void* stream);

/* Per-topic sums of the last sweep, for zero-topic detection: sum_T[k], sum_W[k] (device -> host,
 * as doubles).  nmf.py:757, :793. */
int rri_topic_sums(rri_handle_t h, double* sum_T_host, double* sum_W_host, void* stream);

/* Objective of nmf.py:71-94 over the LOCAL rows:  out_host[0] = 0.5*sum M o (X-WT)^2,
 * out_host[1] = sum M o X^2 (for the relative error), out_host[2] = sum W^2, out_host[3] = sum |W|,
 * out_host[4] = sum T^2, out_host[5] = sum |T|.  The caller combines them with the regularisers
 * (and all-reduces entries 0-3 across shards). */
int rri_objective(rri_handle_t h, const void* W_dev, const void* T_dev, double* out_host, void* stream);

/* The same six numbers for UNMASKED dense data without a pass over X per call:
 *     ||X - W T||^2 = ||X||^2 - 2 <X T', W> + <W'W, T T'>          (fp64 sums; ||X||^2 once per binding)
 * where X T' is the contraction of the W half-step.  reuse_last_sweep != 0 states that W_dev / T_dev are exactly what
 * the last rri_sweeps call on a block-order handle left, so that call's own contraction is reused (an objective per
 * sweep then costs two k x k Gram products and one dot product over n*k, ~3 % of a config-3 sweep, instead of the
 * reference's "2x penalty", nmf.py:143-146); otherwise one contraction pass is made.  The difference of large terms
 * inherits the contraction's rounding: exact to ~1e-12 relative in fp64, ~1e-5 in IEEE fp32, and with TF32 operands
 * the relative error of <X T', W> (~1e-6) is amplified by ||X||^2 / ||X - WT||^2. */
int rri_objective_contraction(rri_handle_t h, const void* W_dev, const void* T_dev, int32_t reuse_last_sweep,
                              double* out_host, void* stream);

/* Test hook == the partial statistic of nmf.py:680-686 (unmasked) / :706-713 (masked) for the local
 * rows: out_wR_dev[d], out_nw_dev[1 (unmasked) | d (masked)], same dtype as X. */
int rri_partials_T(rri_handle_t h, const void* W_dev, const void* T_dev, int32_t t,
                   void* out_wR_dev, void* out_nw_dev, void* stream);

/* Row-wise Euclidean projection onto the simplex {x>=0, sum x = s} of a device matrix A[rows, cols]
 * in place (matrixops.py:5-69, :72-100); used for do_final_project_W (nmf.py:519-529),
 * project_W_each_iter (:481-484) and the initial projections (:870-878). */
int rri_project_rows_simplex(rri_handle_t h, void* A_dev, int64_t rows, int64_t cols, double s, void* stream);

/* Workspace blocks of destroyed handles are parked per device (cudaMalloc/cudaFree cost tens of ms each next to a
 * data-sized resident matrix); this really frees them. */
int rri_cache_trim(int32_t device);

/* Counters for bench.py: kernels launched by this handle since creation / bytes of workspace. */
int rri_stats(rri_handle_t h, int64_t* kernel_launches, int64_t* workspace_bytes);

/* Direct access to the contraction kernel for unit tests and roofline measurements:
 * C[M,N] = A[M,K] * B[N,K]^T, row-major, math as in rri_create (TF32 tcgen05 or IEEE SIMT). */
int rri_gemm_nt(rri_handle_t h, const void* A_dev, int64_t lda, const void* B_dev, int64_t ldb,
                void* C_dev, int64_t ldc, int64_t M, int32_t N, int64_t K, void* stream);

/* The streaming product of a block-order half-step on a dense, unmasked hals handle, through the operand copies
 * the sweeps read (the 16-bit ones where rri_x_operand_bits says 16):
 *     transpose = 0:  C[n_local, N] = X  B[N, d]'          transpose = 1:  C[d, N] = X' B[N, n_local]'
 * B row-major with leading dimension ldb (a multiple of 16 bytes in TF32 math), C row-major [., N]; 1 <= N <= k + 16
 * (at most 256).  With 16-bit copies B is rounded to TF32 and scaled into fp16 by a power of two taken from its
 * maximum; entries below ~2^-29 of that maximum become fp16 subnormals. */
int rri_contract_x(rri_handle_t h, int32_t transpose, const void* B_dev, int64_t ldb, int32_t N, void* C_dev,
                   void* stream);

/* Roofline hook for bench.py: launch the dominant streaming kernel of this handle `iters` times on
 * `stream` between two CUDA events and return the average launch duration in milliseconds.
 *   which = 0: the rri-order fused pass (y = X T_t', p = w_t' X)      -- reads X[n,d] once (zero-filled sparse
 *              handles: the stored entries once in each orientation)
 *   which = 1: the W half-step contraction  X T'  (n x d -> n x k)     -- reads X once
 *   which = 2: the T half-step contraction  X' W  (d x n -> d x k)     -- reads X' once (hals handles)
 *   which = 3 / 4: one whole T / W half-step of the block order (contraction, Gram, exchange, update); these
 *              advance W_dev / T_dev and, on row shards, are collective (every rank calls with the same iters)
 *   which = 5 / 6: one masked (or observed-entries) T-step / W-step of topic 0 -- the statistics pass of
 *              nmf.py:687-701 / :735-746 plus its solve; advances W_dev / T_dev; single-GPU handles */
int rri_profile_kernel(rri_handle_t h, int32_t which, const void* W_dev, const void* T_dev, int32_t iters,
                       float* avg_ms_host, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RRI_B200_H */
