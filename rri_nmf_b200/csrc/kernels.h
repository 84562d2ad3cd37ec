// kernels.h -- host-side launchers of the sweep kernels (internal; the public ABI is include/rri_b200.h)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace rri {

// ---------------------------------------------------------------------------------------------
// rri (interleaved) order, unmasked: three kernels per topic        (rri_kernels.cu)
// ---------------------------------------------------------------------------------------------
struct PassPlan {
    int vec;        // elements per 16-byte load (1 when X is not 16-byte tileable)
    int nch;        // column chunks per thread
    int ct;         // column tiles  (gridDim.x)
    int rg;         // row groups    (gridDim.y)
    int64_t cw;     // columns per tile
};
PassPlan plan_pass(int64_t n, int64_t d, int64_t ldx, const void* X, int elem_size, int sm_count);

// y[ct][i] = sum_{c in tile ct} X[i,c]*tvec[c]   and   p[rg][c] = sum_{i in group rg} W[i,tn]*X[i,c]
template <typename T>
void launch_rri_pass(const T* X, int64_t ldx, int64_t n, int64_t d, const T* tvec, const T* W, int k,
                     int tn, T* ypart, T* ppart, bool do_y, bool do_p, const PassPlan& pl,
                     cudaStream_t st);

struct SolveArgs {      // one half-step's scalar parameters, already in the element type's range
    double reg_l1, reg_l2, eps, ub;
    int has_ub;
};

int tstep_blocks(int64_t d);
int wstep_blocks(int64_t n, int sm_count);

// T-step of topic t (nmf.py:420-447) + partial h = T T_t' (nmf.py:730) for the following W-step
template <typename T>
void launch_rri_tstep(T* Tm, int64_t d, int k, int t, const T* ppart, int rg, int64_t pstride,
                      const T* gpart, int gb, const SolveArgs& a, T* hpart, double* sums, int t_prev,
                      int* flags, bool do_update, cudaStream_t st);

// W-step of topic t (nmf.py:462-469) + partial g = w_tn' W (nmf.py:673) for the following T-step
template <typename T>
void launch_rri_wstep(T* W, int64_t n, int k, int t, int tn, const T* ypart, int ct, int64_t ystride,
                      const T* hpart, int hb, const SolveArgs& a, T* gpart, double* sums, int* flags,
                      bool do_update, int blocks, cudaStream_t st);

// stat[0..d) = sum_rg ppart, stat[d..d+k] = sum_b gpart   (the row-shard statistic, nmf.py:680-686)
template <typename T>
void launch_reduce_stat(const T* ppart, int rg, int64_t d, const T* gpart, int gb, int k, T* stat,
                        cudaStream_t st);

// sums[k + t_prev] = sum over blocks of gpart slot k (sum of the last updated W column) + flags
template <typename T>
void launch_finalize_sums(const T* gpart, int gb, int k, int t_prev, double* sums, int* flags,
                          cudaStream_t st);

}  // namespace rri

namespace rri {
// ---------------------------------------------------------------------------------------------
// hals (block) order, unmasked: contraction + row update + Gram          (hals_kernels.cu)
// ---------------------------------------------------------------------------------------------
// IEEE SIMT contraction  C[p][M,N] = A[M, Kp] * B[N, Kp]^T  over `splits` K-slices p (deterministic:
// the consumer adds the slices in order).  N <= 256.
int simt_gemm_splits(int64_t M, int64_t K, int sm_count);
template <typename T>
void launch_simt_gemm_nt(const T* A, int64_t lda, const T* B, int64_t ldb, T* Cpart, int64_t M, int N,
                         int64_t K, int splits, cudaStream_t st);

// Sequential coordinate update of every row of F[m,k] (block-order HALS half-step):
//   for t: F[i,t] <- [ C[i,t] - sum_{j!=t} F[i,j] S[j,t] - reg_l1 ]_+ / (S[t,t] + reg_l2 + eps)
// C = sum of `parts` slices of Cpart.  Writes F in place, optionally Ft[k,m] = F', and per-block
// column sums colsum_part[blocks][k].   (nmf.py:420-447 / :462-469 applied with the other factor frozen)
int update_rows_blocks(int64_t m, int sm_count);
// Where the last block of an update kernel leaves the column sums: sums[off + t] (and the zero-topic flag bit
// `zero_flag`, 0 = none); counter = device word that is zero between launches.  sums == nullptr: per-block partials only.
struct ColsumOut {
    double* sums;
    int off, zero_flag;
    unsigned* counter;
};
// srcs (optional, device array of `parts` pointers): slice p is srcs[p] instead of Cpart + p*part_stride.
template <typename T>
void launch_update_rows(T* F, int64_t m, int k, const T* Cpart, int parts, int64_t part_stride,
                        const T* const* srcs, const T* S, const SolveArgs& a, T* Ft, int64_t ldft,
                        T* colsum_part, int* flags, int blocks, const ColsumOut& co, cudaStream_t st);

// Multi-GPU T half-step fused with its exchange over NVLink peer memory (hals_kernels.cu: peer_update_rows_kernel).
// Pointers of rank r's exchange buffer as mapped in THIS process; flag arrays hold one 128-byte slot per rank.
struct PeerExchange {
    int world, rank;
    unsigned epoch;
    int64_t row_lo, row_hi;        // rows of T' (columns of T) this rank updates
    int64_t ldtk;                  // row stride of the T replica [k, ldtk]
    const void* part[16];          // this epoch's partial statistic of every rank: [d*k | k*k]
    void* Tt[16];                  // every rank's replica of T' [d, k]
    void* Tk[16];                  // every rank's replica of T  [k, ldtk]
    void* tsum[16];                // every rank's table [world][k] of slice column sums
    unsigned* flag1[16];           // every rank's "partials published" flags  [world x 32 words]
    unsigned* flag2[16];           // every rank's "slice stored" flags         [world x 32 words]
    int* err;
};
int peer_update_blocks(int64_t rows, int sm_count);
// returns the number of kernels launched (2: Gram sum over the ranks into Gsum[k*k], then the row updates) or 0 (rank
// too wide for the fused kernel)
template <typename T>
int launch_peer_update_rows(const PeerExchange& px, int64_t d, int k, const SolveArgs& a, T* Gsum, T* colsum_part,
                            int* flags, double* sums, unsigned* counter, int blocks, cudaStream_t st);

// out[c] = sum_p srcs[p][c] for c < len (fixed order) -- Gram partials of all ranks read through peer memory
template <typename T>
void launch_sum_sources(const T* const* srcs, int parts, int64_t len, T* out, cudaStream_t st);

// Gram matrix G[k,k] = F'F of a row-major F[m,k]: per-chunk partials + fixed-order finalize.
int gram_chunks(int64_t m, int k, int sm_count);
template <typename T>
void launch_gram(const T* F, int64_t m, int k, T* part, int chunks, T* G, cudaStream_t st);

// out[c] = sum_b part[b][c]  (c < len) -- generic fixed-order reduction of per-block partials
template <typename T>
void launch_reduce_parts(const T* part, int parts, int64_t stride, int64_t len, T* out, cudaStream_t st);

// sums[off + t] = sum_b colsum_part[b][t]; sets zero-topic / non-finite flags
template <typename T>
void launch_colsum_finalize(const T* colsum_part, int blocks, int k, double* sums, int off,
                            int zero_flag, int* flags, cudaStream_t st);

// B[c, r] = A[r, c]  (A is rows x cols with leading dimension lda; B has leading dimension ldb)
template <typename T>
void launch_transpose(const T* A, int64_t rows, int64_t cols, int64_t lda, T* B, int64_t ldb,
                      cudaStream_t st);

// ---------------------------------------------------------------------------------------------
// 16-bit copies of TF32 operands for the block-order contraction (f16_gemm_run)      (x16_kernels.cu)
// ---------------------------------------------------------------------------------------------
// out[3] <- {bits of max |tf32(x)|, bits of the smallest nonzero |tf32(x)|, 1 if any value is inf / nan} over X
void launch_x16_scan(const float* X, int64_t rows, int64_t cols, int64_t ld, unsigned* out, int sm_count, cudaStream_t st);
// host: true (and the scale exponent e) when fp16(tf32(x) * 2^e) is exact for every x the scan saw
bool x16_exponent(const unsigned scan[3], int* e);
// Y[r, c] = Yt[c, r] = fp16(tf32(X[r, c]) * 2^e)  (Y [rows, ldy], Yt [cols, ldyt])
void launch_x16_copy(const float* X, int64_t rows, int64_t cols, int64_t ldx, int e, void* Y, int64_t ldy, void* Yt,
                     int64_t ldyt, cudaStream_t st);
// out [rows, ldo] = fp16(tf32(F) * 2^e) with e (written to *e_out) putting max |tf32(F)| into [2^15, 2^16);
// part: nparts = f16_factor_parts() block maxima
int f16_factor_parts(int sm_count);
void launch_f16_factor(const float* F, int rows, int64_t cols, int64_t ld, unsigned* part, int nparts, void* out,
                       int64_t ldo, int* e_out, cudaStream_t st);
}  // namespace rri

namespace rri {
// ---------------------------------------------------------------------------------------------
// masked / weighted WRRI half-steps and the objective                      (wrri_kernels.cu)
// ---------------------------------------------------------------------------------------------
enum { MK_NONE = 0, MK_REAL = 1, MK_U8 = 2, MK_SPARSE = 3 /* observed entries only: sparse_kernels.cu */ };

struct TilePlan { int tiles_r, tiles_c, groups; };      // groups = partial slices written
TilePlan plan_tstats(int64_t n, int64_t d, int sm_count);
TilePlan plan_wstats(int64_t n, int64_t d, int sm_count);

// T-step statistics of topic t over the local rows (nmf.py:687-701):
//   numer_part[g][c] = sum_{i in group g} W[i,t] * M[i,c] * (X[i,c] - sum_{j!=t} W[i,j] T[j,c])
//   denom_part[g][c] = sum_{i in group g} W[i,t]^2 * M[i,c]
template <typename T>
void launch_wrri_tstats(const T* X, int64_t ldx, const void* M, int mk, int64_t ldm, const T* W,
                        const T* Tm, int64_t n, int64_t d, int k, int t, T* numer_part, T* denom_part,
                        const TilePlan& pl, cudaStream_t st);
// W-step statistics of topic t (nmf.py:735-746): numer_part[g][i], denom_part[g][i] over column groups
template <typename T>
void launch_wrri_wstats(const T* X, int64_t ldx, const void* M, int mk, int64_t ldm, const T* W,
                        const T* Tm, int64_t n, int64_t d, int k, int t, T* numer_part, T* denom_part,
                        const TilePlan& pl, cudaStream_t st);
// vector-c solve (optimization.py:75-84) of out[idx*stride] for idx < len from `parts` partial slices
// (out2/out2_stride: optional second destination -- the padded operand copy of the tensor-core path)
template <typename T>
void launch_wrri_final(const T* numer_part, const T* denom_part, int parts, int64_t len,
                       const SolveArgs& a, T* out, int64_t out_stride, T* out2, int64_t out2_stride,
                       int* flags, cudaStream_t st);
// sums[slot] = sum_i v[i*stride]; zero/non-finite flags (single block, fixed order)
template <typename T>
void launch_vec_sum_flag(const T* v, int64_t len, int64_t stride, double* sums, int slot, int zero_flag,
                         int* flags, cudaStream_t st);
// sums[slot0 + r] = sum of row r of A[rows, ld] over len elements; zero / non-finite flags (one launch per sweep)
template <typename T>
void launch_rowsum_flag(const T* A, int rows, int64_t len, int64_t ld, double* sums, int slot0, int zero_flag,
                        int* flags, cudaStream_t st);
// v[i*stride] *= scale / sums[slot]   (vector-c branch with a sum constraint, optimization.py:85-87)
template <typename T>
void launch_vec_scale_to_sum(T* v, int64_t len, int64_t stride, const double* sums, int slot, double s,
                             cudaStream_t st);

// objective pieces over the local rows (nmf.py:71-94): out[0] = 0.5*sum M (X-WT)^2, out[1] = sum M X^2
int obj_blocks(int64_t n, int64_t d, int sm_count);
template <typename T>
void launch_objective(const T* X, int64_t ldx, const void* M, int mk, int64_t ldm, const T* W,
                      const T* Tm, int64_t n, int64_t d, int k, double* part, int blocks, double* out,
                      cudaStream_t st);
// pieces of the objective through the contraction (unmasked): ||X-WT||^2 = ||X||^2 - 2<X T', W> + <W'W, T T'>, fp64 sums
//   out[0] = sum A[r,c]^2 (A rows x cols, leading dimension lda);   part: >= 8*sm_count doubles of scratch
template <typename T>
void launch_sumsq_rows(const T* A, int64_t rows, int64_t cols, int64_t lda, double* part, double* out, int sm_count,
                       cudaStream_t st);
//   out[0] = sum_e (sum_p C[p*stride + e]) * W[e]
template <typename T>
void launch_dot_parts(const T* C, int parts, int64_t stride, const T* W, int64_t len, double* part, double* out,
                      int sm_count, cudaStream_t st);
//   out[0] = 0.5 * (acc[0] - 2 acc[1] + sum G o H), out[1] = acc[0]
template <typename T>
void launch_objective_identity(const T* G, const T* H, int k, const double* acc, double* out, cudaStream_t st);
// out[0] = sum v^2, out[1] = sum |v| over len contiguous elements (regulariser terms, nmf.py:72-75)
template <typename T>
void launch_norms(const T* v, int64_t len, double* part, double* out, cudaStream_t st);
}  // namespace rri

namespace rri {
// sets `zero_flag` when any sums[off + t] <= 1e-10 (after a cross-shard all-reduce of the sums)
void launch_flag_from_sums(const double* sums, int off, int k, int zero_flag, int* flags, cudaStream_t st);

// rows of A[rows, cols] <- Euclidean projection onto {x >= 0, sum x = s}   (simplex_kernels.cu;
// matrixops.py:5-69 computes the same threshold by sorting)
template <typename T>
void launch_project_rows_simplex(T* A, int64_t rows, int64_t cols, double s, cudaStream_t st);

// Block-order T half-step with the projection of every updated row of T onto the simplex of radius s
// (project_T_each_iter, nmf.py:420-447 + :759-761), from the contraction C = sum of `parts` slices [d, k] and the Gram
// matrix G [k, k]: updates T' = Tt [d, k] in place and writes T = Tout [k, ldo].  allow_fused: one cooperative launch
// when k and the grid fit it (else, and with allow_fused false, a chain of 2k + 1 launches).  Returns 0 or a
// cudaError_t; *launches = kernels launched.  slots: simplex_T_slots(d) doubles of scratch.
int simplex_T_slots(int64_t d);
template <typename T>
int launch_simplex_T_update(T* Tt, int64_t d, int k, const T* C, int parts, int64_t pstride, const T* G, const SolveArgs& a,
                            double s, T* Tout, int64_t ldo, double* slots, int* flags, int sm_count, bool allow_fused,
                            int* launches, cudaStream_t st);
}  // namespace rri

namespace rri {
// ---------------------------------------------------------------------------------------------
// observed-entries (sparse) WRRI: CSR + CSC residual copies                 (sparse_kernels.cu)
// ---------------------------------------------------------------------------------------------
struct SpSide {            // one compressed orientation of the observed entries
    int64_t nseg;          // rows (CSR) or columns (CSC)
    const int64_t* ptr;    // [nseg + 1]
    const int32_t* idx;    // [nnz] column (CSR) / row (CSC) of every entry, ascending inside a segment
    const void* x;         // [nnz] observed values in this order
    const void* wgt;       // [nnz] entry weights in this order, or null (all ones)
    void* E;               // [nnz] residual X - W T at the observed entries
    int group;             // threads that share a segment: 32 (a warp) or 256 (a block)
    // blocked passes (optional): the other factor's index range cut into nblk blocks of nb records
    const int64_t* ptr2;   // [nseg][nblk + 1] first entry of segment s with index >= b * nb, or null
    int nblk, nb;
    int64_t nother;        // length of the other factor's index range (d for CSR, n for CSC)
    const uint16_t* idx16; // [nnz] idx % nb (2 bytes instead of 4 per entry and pass), or null
};
int sp_block_len(int elem_size, int64_t nother, int* nblk_out);
void launch_sp_local_index(const int32_t* idx, int64_t nnz, int nb, uint16_t* out, int sm_count, cudaStream_t st);
void launch_sp_subptr(const int64_t* ptr, const int32_t* idx, int64_t nseg, int nblk, int nb, int64_t* ptr2,
                      int sm_count, cudaStream_t st);

// Column orientation of a CSR matrix: colptr[d+1], csc_row[nnz], x_csc[nnz] (, w_csc[nnz]); rows ascending inside
// a column; perm[nnz] (caller-owned) receives the CSR position of every CSC entry.  Returns 0, a cudaError_t (> 0), or -(bit mask) for a malformed CSR: 1 rowptr, 2 column range,
// 4 columns not strictly ascending inside a row.  Synchronises `st`.
template <typename T>
int sp_build_csc(const int64_t* rowptr, const int32_t* col, const T* x, const T* w, int64_t n, int64_t d,
                 int64_t nnz, int64_t* colptr, int32_t* csc_row, T* x_csc, T* w_csc, uint32_t* perm, int sm_count,
                 int* err_dev, cudaStream_t st);

// s.E[p] = s.x[p] - sum_l A[seg,l] * B[s.idx[p],l]   (A: own factor rows [nseg,k], B: other factor rows [.,k])
template <typename T>
void launch_sp_residual(const SpSide& s, const T* A, const T* B, int k, int sm_count, cudaStream_t st);

// The same for the row orientation with 16-byte gathers: B[., ldb] has a padded row stride (multiple of 16 bytes, zero
// pad columns); A[nseg, lda] is staged per segment through shared memory.
template <typename T>
void launch_sp_residual_rows(const SpSide& s, const T* A, int64_t lda, const T* B, int ldb, int k, int sm_count,
                             cudaStream_t st);
// dst[p] = src[perm[p]]
template <typename T>
void launch_sp_gather(const uint32_t* perm, const T* src, T* dst, int64_t nnz, int sm_count, cudaStream_t st);

// quad[i] = {po[i], pn[i], vold[i], vnew[i]}   (po/pn null -> 0): the 16/32-byte gather record of a pass
template <typename T>
void launch_sp_pack(const T* po, const T* pn, const T* vold, const T* vnew, void* quad, int64_t len, cudaStream_t st);

// One half-step statistic over one orientation (see sparse_kernels.cu): applies the pending rank-one change
// (own_po/own_pn null -> none), writes own_save[seg] = own_cur[seg] and `parts` slices numer[p][seg], denom[p][seg]
// (before the regularisers; the consumer adds the slices in order).  Returns parts (1, or s.nblk when blocked).
template <typename T>
int launch_sp_pass(const SpSide& s, const void* quad, const T* own_po, const T* own_pn, const T* own_cur,
                    T* own_save, T* numer, T* denom, int sm_count, cudaStream_t st);

// out[0] = 0.5 * sum m E^2, out[1] = sum m x^2 over the observed entries (fixed-order reduction)
template <typename T>
void launch_sp_objective(const SpSide& s, int64_t nnz, double* part, double* out, cudaStream_t st);
}  // namespace rri

namespace rri {
// ---------------------------------------------------------------------------------------------
// sparse x dense contraction on zero-filled sparse data (block order)          (spmm_kernels.cu)
// ---------------------------------------------------------------------------------------------
constexpr int SPMM_CHUNK = 1024;    // longest segment taken by one lane group; longer ones are cut into chunks
constexpr int SPMM_PANEL = 256;     // widest operand panel of one launch (accumulators in registers)
struct SpmmPlan {                   // one compressed orientation and its chunk plan (built once at bind time)
    int64_t nseg;                   // rows (CSR) or columns (CSC)
    const int64_t* ptr;             // [nseg + 1]
    const int32_t* idx;             // [nnz] column (CSR) / row (CSC) of every entry
    const void* val;                // [nnz]
    int64_t nlong_items;            // chunks of the segments longer than SPMM_CHUNK
    const int2* litem;              // [nlong_items] {long segment, chunk}
    const int32_t* lseg;            // [nlong] segment of long segment j
    const int64_t* lslot;           // [nlong] first partial slot of long segment j
    void* slots;                    // [nlong_items][panel width] chunk partials
    unsigned* counters;             // [nlong] arrivals, zero between launches
};
// C[r, :width] = sum_{e in segment r} val[e] * B[idx[e], :width]   (B [., ldb] and C [nseg, ldc] row-major; one launch per
// panel of at most SPMM_PANEL columns, in ascending order; p.slots holds [nlong_items][min(width, SPMM_PANEL)])
template <typename T>
void launch_spmm(const SpmmPlan& p, const T* B, int64_t ldb, int width, T* C, int64_t ldc, cudaStream_t st);
// out[i] = w[i] * x[i]
template <typename T>
void launch_spmm_weighted_values(const T* x, const T* w, int64_t nnz, T* out, int sm_count, cudaStream_t st);

// ---------------------------------------------------------------------------------------------
// interleaved-order pass on zero-filled sparse data: both statistics of rri_pass_kernel in one launch
//                                                                             (sparse_rri_kernels.cu)
// ---------------------------------------------------------------------------------------------
struct SparsePassPlan {
    int gy, gp;            // lanes per work item over the rows / the columns
    int blocks;            // resident blocks of one launch
    int blocks_y, blocks_p;    // their split between the orientations when both statistics are computed
};
template <typename T>
SparsePassPlan plan_sparse_rri_pass(const SpmmPlan& rows, const SpmmPlan& cols, int64_t nnz, int sm_count);
// y[i] = sum_{e in row i} val[e] * trow[col[e]]   (do_y)   and   p[j] = sum_{e in col j} val[e] * W[row[e] * k + tn]   (do_p)
template <typename T>
void launch_sparse_rri_pass(const SparsePassPlan& pl, const SpmmPlan& rows, const SpmmPlan& cols, const T* trow,
                            const T* W, int k, int tn, T* y, T* p, bool do_y, bool do_p, cudaStream_t st);
}  // namespace rri
