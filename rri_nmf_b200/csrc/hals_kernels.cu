// hals_kernels.cu -- block-order (HALS) half-steps, unmasked.
//
// With the other factor frozen, the k rank-one updates of one factor only need
//     C = A B'   (one streaming contraction over the data: X T' for W, X' W for T)
//     S = B B'   (k x k Gram)
// and then every row of the factor is updated independently by k sequential scalar solves --
// the arithmetic of nmf.py:670-676 + :437-447 (T) / :728-734 + :464-469 (W), reordered so that X
// is read twice per sweep instead of 2k times (BASELINE.json north_star groups (1)+(2)).
// This file holds the IEEE (fp32/fp64 SIMT) contraction, the row-update kernel and the Gram
// kernel; the TF32 tcgen05 contraction lives in gemm_tf32_sm100.cu.
#include "common.cuh"
#include "kernels.h"

namespace rri {

// ------------------------------------------------------------------------------------------------
// SIMT contraction C = A B^T   (A: M x K, B: N x K, both K-contiguous)
// ------------------------------------------------------------------------------------------------
constexpr int G_BM = 64, G_BK = 16, G_THREADS = 256;

template <typename T, int KT>
__global__ void __launch_bounds__(G_THREADS)
simt_gemm_nt_kernel(const T* __restrict__ A, int64_t lda, const T* __restrict__ B, int64_t ldb,
                    T* __restrict__ Cpart, int64_t M, int N, int64_t K)
{
    constexpr int BN = 16 * KT;
    __shared__ T As[G_BK][G_BM + 4];
    __shared__ T Bs[G_BK][BN + 4];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int64_t m0 = (int64_t)blockIdx.x * G_BM;
    int64_t k0, k1;
    part_range((K + G_BK - 1) / G_BK, gridDim.y, blockIdx.y, k0, k1);
    k0 *= G_BK; k1 = (k1 * G_BK < K) ? k1 * G_BK : K;

    T acc[4][KT];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < KT; ++j) acc[i][j] = T(0);

    const int arow = tid >> 2, akk = (tid & 3) * 4;
    for (int64_t kb = k0; kb < k1; kb += G_BK) {
        {   // A tile: 64 rows x 16
            const int64_t gm = m0 + arow;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int64_t gk = kb + akk + e;
                As[akk + e][arow] = (gm < M && gk < k1) ? ld_stream(A + gm * lda + gk) : T(0);
            }
        }
        for (int e = tid; e < BN * G_BK; e += G_THREADS) {
            const int row = e / G_BK, kk = e % G_BK;
            const int64_t gk = kb + kk;
            Bs[kk][row] = (row < N && gk < k1) ? B[(int64_t)row * ldb + gk] : T(0);
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < G_BK; ++kk) {
            T a[4], b[KT];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
            for (int j = 0; j < KT; ++j) b[j] = Bs[kk][tx + 16 * j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < KT; ++j) acc[i][j] = fma(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
    T* C = Cpart + (int64_t)blockIdx.y * M * N;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int64_t gm = m0 + ty * 4 + i;
        if (gm < M) {
#pragma unroll
            for (int j = 0; j < KT; ++j) {
                const int gn = tx + 16 * j;
                if (gn < N) C[gm * N + gn] = acc[i][j];
            }
        }
    }
}

int simt_gemm_splits(int64_t M, int64_t K, int sm_count)
{
    const int64_t tiles = (M + G_BM - 1) / G_BM;
    int64_t s = (2 * sm_count + tiles - 1) / tiles;
    const int64_t maxs = (K + 8 * G_BK - 1) / (8 * G_BK);        // >= 128 k-elements per slice
    if (s > maxs) s = maxs;
    if (s > 64) s = 64;
    return (int)(s < 1 ? 1 : s);
}

template <typename T>
void launch_simt_gemm_nt(const T* A, int64_t lda, const T* B, int64_t ldb, T* Cpart, int64_t M, int N,
                         int64_t K, int splits, cudaStream_t st)
{
    dim3 grid((unsigned)((M + G_BM - 1) / G_BM), splits);
    const int kt = (N + 15) / 16;
#define RRI_G_CASE(KT) simt_gemm_nt_kernel<T, KT><<<grid, G_THREADS, 0, st>>>(A, lda, B, ldb, Cpart, M, N, K)
    if (kt <= 1) RRI_G_CASE(1);
    else if (kt <= 2) RRI_G_CASE(2);
    else if (kt <= 4) RRI_G_CASE(4);
    else if (kt <= 8) RRI_G_CASE(8);
    else RRI_G_CASE(16);
#undef RRI_G_CASE
}

// ------------------------------------------------------------------------------------------------
// fused finalisation of the per-block column sums: the LAST block to finish (an arrival counter, nobody waits) adds
// the block partials in the fixed order of the former colsum_finalize_kernel (a warp per column, lanes stride over
// the blocks, shuffle tree) and sets the zero-topic / non-finite flags -- one launch less per half-step
// ------------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ void colsum_tail(const T* __restrict__ colsum_part, int k, double* __restrict__ sums, int off,
                                            int zero_flag, int* __restrict__ flags, unsigned* __restrict__ counter)
{
    __shared__ unsigned s_arrival;
    __threadfence();                                   // this block's partial sums before its arrival
    __syncthreads();
    if (threadIdx.x == 0) s_arrival = atomicAdd(counter, 1u);
    __syncthreads();
    if (s_arrival != gridDim.x - 1) return;
    __threadfence();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    for (int col = warp; col < k; col += nw) {
        T s = T(0);
        for (int b = lane; b < (int)gridDim.x; b += 32) s += __ldcg(colsum_part + (int64_t)b * k + col);
        s = warp_sum(s);
        if (lane == 0) {
            const double v = (double)s;
            sums[off + col] = v;
            if (zero_flag && !(v > 1e-10)) atomicOr(flags, zero_flag);
            if (!isfinite(v)) atomicOr(flags, 8);
        }
    }
    if (threadIdx.x == 0) *counter = 0u;              // ready for the next launch
}

// ------------------------------------------------------------------------------------------------
// row update: warp per row, lanes own coordinates t' = lane + 32 l
// ------------------------------------------------------------------------------------------------
constexpr int U_THREADS = 256, U_NW = U_THREADS / WARP, U_GROUP = 32;   // rows per block iteration

int update_rows_blocks(int64_t m, int sm_count)
{
    int64_t b = (m + 127) / 128;
    if (b > 4 * sm_count) b = 4 * sm_count;
    return (int)(b < 1 ? 1 : b);
}

template <typename T, int KL, bool S_SMEM>
__global__ void __launch_bounds__(U_THREADS)
update_rows_kernel(T* __restrict__ F, int64_t m, int k, const T* __restrict__ Cpart, int parts,
                   int64_t part_stride, const T* const* __restrict__ srcs, const T* __restrict__ S,
                   T reg_l1, T reg_l2, T eps, T ub, int has_ub,
                   T* __restrict__ Ft, int64_t ldft, T* __restrict__ colsum_part, int* __restrict__ flags,
                   double* __restrict__ sums, int sums_off, int zero_flag, unsigned* __restrict__ counter,
                   int64_t ldc, int64_t lds, int64_t s_stride)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T* ftile = reinterpret_cast<T*>(smem_raw);                 // [k][U_GROUP+1]
    T* csm = ftile + (size_t)k * (U_GROUP + 1);                // [U_NW][k]
    T* Ss = csm + (size_t)U_NW * k;                            // [k][k] when S_SMEM
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int z = blockIdx.y;                                  // model (RowBatch)
    F += (int64_t)z * m * k;
    S += (int64_t)z * s_stride;
    if (Ft) Ft += (int64_t)z * k * ldft;
    flags += z;
    colsum_part += (int64_t)z * gridDim.x * k;
    const int64_t coff = (int64_t)z * k;
    if (S_SMEM) {
        for (int e = tid; e < k * k; e += U_THREADS) Ss[e] = S[(e / k) * lds + e % k];
        __syncthreads();
    }
    const T* Sp = S_SMEM ? Ss : S;
    const int64_t sld = S_SMEM ? k : lds;

    T csum[KL];
#pragma unroll
    for (int l = 0; l < KL; ++l) csum[l] = T(0);
    bool unb = false;

    const int64_t ngroups = (m + U_GROUP - 1) / U_GROUP;
    for (int64_t g = blockIdx.x; g < ngroups; g += gridDim.x) {
        const int64_t i0 = g * U_GROUP;
#pragma unroll 1
        for (int q = 0; q < U_GROUP / U_NW; ++q) {
            const int ii = warp + U_NW * q;
            const int64_t i = i0 + ii;
            if (i < m) {
                T f[KL], r[KL];
#pragma unroll
                for (int l = 0; l < KL; ++l) {
                    const int tp = lane + 32 * l;
                    f[l] = T(0); r[l] = T(0);
                    if (tp < k) {
                        f[l] = F[i * k + tp];
                        T c = T(0);
                        for (int p = 0; p < parts; ++p)
                            c += (srcs ? srcs[p] : Cpart + (int64_t)p * part_stride)[coff + i * ldc + tp];
                        r[l] = c;
                    }
                }
                // r[t'] = C[i,t'] - sum_{j != t'} F[i,j] S[j,t']
#pragma unroll
                for (int l0 = 0; l0 < KL; ++l0) {
                    for (int tt = 0; tt < 32; ++tt) {
                        const int j = 32 * l0 + tt;
                        if (j >= k) break;
                        const T fj = __shfl_sync(0xffffffffu, f[l0], tt);
#pragma unroll
                        for (int l = 0; l < KL; ++l) {
                            const int tp = lane + 32 * l;
                            if (tp < k && tp != j) r[l] = fma(-fj, Sp[j * sld + tp], r[l]);
                        }
                    }
                }
                // sequential solves; after topic t changes by delta, r[t'] -= delta * S[t,t']
#pragma unroll
                for (int l0 = 0; l0 < KL; ++l0) {
                    for (int tt = 0; tt < 32; ++tt) {
                        const int t = 32 * l0 + tt;
                        if (t >= k) break;
                        T delta = T(0);
                        if (lane == tt) {
                            const T x = solve_scalar_c<T>(r[l0] - reg_l1, Sp[t * sld + t] + reg_l2, eps, ub,
                                                          has_ub != 0, unb);
                            delta = x - f[l0];
                            f[l0] = x;
                        }
                        delta = __shfl_sync(0xffffffffu, delta, tt);
#pragma unroll
                        for (int l = 0; l < KL; ++l) {
                            const int tp = lane + 32 * l;
                            if (tp < k && tp != t) r[l] = fma(-delta, Sp[t * sld + tp], r[l]);
                        }
                    }
                }
#pragma unroll
                for (int l = 0; l < KL; ++l) {
                    const int tp = lane + 32 * l;
                    if (tp < k) {
                        F[i * k + tp] = f[l];
                        csum[l] += f[l];
                        if (Ft) ftile[tp * (U_GROUP + 1) + ii] = f[l];
                    }
                }
            }
        }
        if (Ft) {
            __syncthreads();
            for (int e = tid; e < k * U_GROUP; e += U_THREADS) {
                const int tp = e / U_GROUP, ii = e % U_GROUP;
                if (i0 + ii < m) Ft[(int64_t)tp * ldft + i0 + ii] = ftile[tp * (U_GROUP + 1) + ii];
            }
            __syncthreads();
        }
    }
    if (unb) atomicOr(flags, 4);
#pragma unroll
    for (int l = 0; l < KL; ++l) {
        const int tp = lane + 32 * l;
        if (tp < k) csm[warp * k + tp] = csum[l];
    }
    __syncthreads();
    for (int tp = tid; tp < k; tp += U_THREADS) {
        T s = T(0);
#pragma unroll
        for (int w = 0; w < U_NW; ++w) s += csm[w * k + tp];
        colsum_part[(int64_t)blockIdx.x * k + tp] = s;
    }
    if (sums) colsum_tail<T>(colsum_part, k, sums, sums_off, zero_flag, flags, counter);
}

template <typename T, int KL>
static void launch_update_rows_kl(T* F, int64_t m, int k, const T* Cpart, int parts, int64_t part_stride,
                                  const T* const* srcs, const T* S, const SolveArgs& a, T* Ft, int64_t ldft, T* colsum_part,
                                  int* flags, int blocks, const ColsumOut& co, const RowBatch& rb, cudaStream_t st)
{
    const dim3 grid((unsigned)blocks, (unsigned)rb.models);
    size_t base = sizeof(T) * ((size_t)k * (U_GROUP + 1) + (size_t)U_NW * k);
    size_t with_s = base + sizeof(T) * (size_t)k * k;
    if (with_s <= 200 * 1024) {
        auto kern = update_rows_kernel<T, KL, true>;
        if (with_s > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)with_s);
        kern<<<grid, U_THREADS, with_s, st>>>(F, m, k, Cpart, parts, part_stride, srcs, S, (T)a.reg_l1,
                                               (T)a.reg_l2, (T)a.eps, (T)a.ub, a.has_ub, Ft, ldft,
                                               colsum_part, flags, co.sums, co.off, co.zero_flag, co.counter,
                                               rb.ldc, rb.lds, rb.s_stride);
    } else {
        auto kern = update_rows_kernel<T, KL, false>;
        if (base > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)base);
        kern<<<grid, U_THREADS, base, st>>>(F, m, k, Cpart, parts, part_stride, srcs, S, (T)a.reg_l1,
                                             (T)a.reg_l2, (T)a.eps, (T)a.ub, a.has_ub, Ft, ldft,
                                             colsum_part, flags, co.sums, co.off, co.zero_flag, co.counter,
                                             rb.ldc, rb.lds, rb.s_stride);
    }
}


// ------------------------------------------------------------------------------------------------
// row update, thread per row (k <= KM): the row's k factor entries live in registers (static
// indices only), the Gram row S[t,:] is a shared-memory broadcast read with 16-byte loads, the
// contraction row C[i,:] sits in a padded shared tile.  Direct form, as the reference computes it:
//     numer_t = C[i,t] - sum_{j != t} F[i,j] S[j,t]        (nmf.py:733 / :675 with the current factor)
// Rows are staged through shared memory so that global traffic stays coalesced.
// ------------------------------------------------------------------------------------------------
constexpr int TPR_ROWS = 128;       // rows (= threads) per block

// The k sequential scalar solves of one row (thread `tid` owns row `tid` of the staged tiles): topics in groups of
// 8, t = 8c + u with u unrolled, so the register holding f[t] can only be one of the 8 entries f[u], f[u+8], ... --
// 8 selects per step instead of KM.  ctile/ftile: [TPR_ROWS][KM+1] staged contraction / factor rows; Ss: [KM][KM].
template <typename T, int KM>
__device__ __forceinline__ void tpr_solve_row(const T* __restrict__ Ss, const T* __restrict__ ctile, T* __restrict__ ftile,
                                              int tid, int k, T reg_l1, T reg_l2, T eps, T ub, bool has_ub, bool& unb)
{
    using V = typename Vec<T>::type;
    constexpr int VN = Vec<T>::N;
    constexpr int LD = KM + 1;
    T f[KM];
#pragma unroll
    for (int j = 0; j < KM; ++j) f[j] = (j < k) ? ftile[tid * LD + j] : T(0);
#pragma unroll 1
    for (int c = 0; c < (k + 7) / 8; ++c) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int t = 8 * c + u;
            if (t < k) {
                const V* srow = reinterpret_cast<const V*>(Ss + t * KM);
                T acc[4] = {T(0), T(0), T(0), T(0)};
#pragma unroll
                for (int jv = 0; jv < KM / VN; ++jv) {
                    T sv[VN];
                    unpack(srow[jv], sv);
#pragma unroll
                    for (int v = 0; v < VN; ++v) acc[(jv * VN + v) & 3] = fma(f[jv * VN + v], sv[v], acc[(jv * VN + v) & 3]);
                }
                const T stt = Ss[t * KM + t];
                const T ft = ftile[tid * LD + t];
                // sum over j != t: remove the own term from the full dot product
                const T dot = ((acc[0] + acc[1]) + (acc[2] + acc[3])) - ft * stt;
                const T x = solve_scalar_c<T>(ctile[tid * LD + t] - dot - reg_l1, stt + reg_l2, eps, ub, has_ub, unb);
                ftile[tid * LD + t] = x;
#pragma unroll
                for (int jj = 0; jj < KM / 8; ++jj) f[8 * jj + u] = (jj == c) ? x : f[8 * jj + u];
            }
        }
    }
}

template <typename T, int KM>
__global__ void __launch_bounds__(TPR_ROWS)
update_rows_tpr_kernel(T* __restrict__ F, int64_t m, int k, const T* __restrict__ Cpart, int parts,
                       int64_t part_stride, const T* const* __restrict__ srcs, const T* __restrict__ S,
                       T reg_l1, T reg_l2, T eps, T ub, int has_ub,
                       T* __restrict__ Ft, int64_t ldft, T* __restrict__ colsum_part, int* __restrict__ flags,
                       double* __restrict__ sums, int sums_off, int zero_flag, unsigned* __restrict__ counter,
                       int64_t ldc, int64_t lds, int64_t s_stride)
{
    constexpr int LD = KM + 1;                              // padded row stride of the tiles
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T* Ss = reinterpret_cast<T*>(smem_raw);                 // [KM][KM], zero padded, 16-byte aligned rows
    T* ctile = Ss + KM * KM;                                // [TPR_ROWS][LD]  contraction rows
    T* ftile = ctile + TPR_ROWS * LD;                       // [TPR_ROWS][LD]  factor rows
    const int tid = threadIdx.x;
    const int z = blockIdx.y;                               // model (RowBatch)
    F += (int64_t)z * m * k;
    S += (int64_t)z * s_stride;
    if (Ft) Ft += (int64_t)z * k * ldft;
    flags += z;
    colsum_part += (int64_t)z * gridDim.x * k;
    const int64_t coff = (int64_t)z * k;
    for (int e = tid; e < KM * KM; e += TPR_ROWS) {
        const int a = e / KM, b = e % KM;
        Ss[e] = (a < k && b < k) ? S[a * lds + b] : T(0);
    }
    T csum = T(0);          // thread j < k accumulates the sum of column j over this block's rows
    bool unb = false;
    __syncthreads();

    const int64_t ngroups = (m + TPR_ROWS - 1) / TPR_ROWS;
    for (int64_t g = blockIdx.x; g < ngroups; g += gridDim.x) {
        const int64_t i0 = g * TPR_ROWS;
        const int nrow = (int)((m - i0) < TPR_ROWS ? (m - i0) : TPR_ROWS);
        {   // coalesced staging of the C and F rows, 8 independent loads in flight per thread (a plain loop
            // serialises one L2 round trip per element); (row, col) of e = tid + 128*it advance without divisions
            const int tot = nrow * k;
            int rr = tid / k, cc = tid - rr * k;
            const int dr = TPR_ROWS / k, dc = TPR_ROWS - dr * k;
            const T* Frow = F + i0 * k;
            const T* Crow = (srcs ? srcs[0] : Cpart) + coff + i0 * ldc;
            constexpr int UB = 8;
            for (int e0 = tid; e0 < tot; e0 += UB * TPR_ROWS) {
                T cv[UB], fv[UB];
                int co[UB];                                 // offset of element e in the contraction rows (row stride ldc)
                {
                    int r2 = rr, c2 = cc;
#pragma unroll
                    for (int u = 0; u < UB; ++u) {
                        co[u] = r2 * (int)ldc + c2;
                        r2 += dr; c2 += dc;
                        if (c2 >= k) { c2 -= k; ++r2; }
                    }
                }
#pragma unroll
                for (int u = 0; u < UB; ++u) {
                    const int e = e0 + u * TPR_ROWS;
                    cv[u] = T(0); fv[u] = T(0);
                    if (e < tot) {
                        cv[u] = Crow[co[u]];
                        fv[u] = Frow[e];
                    }
                }
                for (int p = 1; p < parts; ++p) {
                    const T* Cp = srcs ? srcs[p] + coff + i0 * ldc : Crow + (int64_t)p * part_stride;
#pragma unroll
                    for (int u = 0; u < UB; ++u) {
                        const int e = e0 + u * TPR_ROWS;
                        if (e < tot) cv[u] += Cp[co[u]];
                    }
                }
#pragma unroll
                for (int u = 0; u < UB; ++u) {
                    const int e = e0 + u * TPR_ROWS;
                    if (e < tot) {
                        ctile[rr * LD + cc] = cv[u];
                        ftile[rr * LD + cc] = fv[u];
                    }
                    rr += dr; cc += dc;
                    if (cc >= k) { cc -= k; ++rr; }
                }
            }
        }
        __syncthreads();
        if (tid < nrow) tpr_solve_row<T, KM>(Ss, ctile, ftile, tid, k, reg_l1, reg_l2, eps, ub, has_ub != 0, unb);
        __syncthreads();
        {   // write back: F (row-major, coalesced), column sums, transposed copy
            const int tot = nrow * k;
            int rr = tid / k, cc = tid - rr * k;
            const int dr = TPR_ROWS / k, dc = TPR_ROWS - dr * k;
            T* Frow = F + i0 * k;
            for (int e = tid; e < tot; e += TPR_ROWS) {
                Frow[e] = ftile[rr * LD + cc];
                rr += dr; cc += dc;
                if (cc >= k) { cc -= k; ++rr; }
            }
            if (tid < k) {
                T cs = T(0);
#pragma unroll 8
                for (int ii = 0; ii < nrow; ++ii) cs += ftile[ii * LD + tid];
                csum += cs;
            }
            if (Ft) {
                // thread ii writes element (tp, i0+ii): consecutive threads -> consecutive addresses
                if (tid < nrow)
                    for (int tp = 0; tp < k; ++tp) Ft[(int64_t)tp * ldft + i0 + tid] = ftile[tid * LD + tp];
            }
        }
        __syncthreads();
    }
    if (unb) atomicOr(flags, 4);
    if (tid < k) colsum_part[(int64_t)blockIdx.x * k + tid] = csum;
    if (sums) colsum_tail<T>(colsum_part, k, sums, sums_off, zero_flag, flags, counter);
}

template <typename T, int KM>
static void launch_update_rows_tpr(T* F, int64_t m, int k, const T* Cpart, int parts, int64_t part_stride,
                                   const T* const* srcs, const T* S, const SolveArgs& a, T* Ft, int64_t ldft, T* colsum_part,
                                   int* flags, int blocks, const ColsumOut& co, const RowBatch& rb, cudaStream_t st)
{
    const size_t smem = sizeof(T) * ((size_t)KM * KM + 2 * (size_t)TPR_ROWS * (KM + 1));
    auto kern = update_rows_tpr_kernel<T, KM>;
    if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    kern<<<dim3((unsigned)blocks, (unsigned)rb.models), TPR_ROWS, smem, st>>>(
        F, m, k, Cpart, parts, part_stride, srcs, S, (T)a.reg_l1, (T)a.reg_l2, (T)a.eps, (T)a.ub, a.has_ub, Ft, ldft,
        colsum_part, flags, co.sums, co.off, co.zero_flag, co.counter, rb.ldc, rb.lds, rb.s_stride);
}

// ------------------------------------------------------------------------------------------------
// row update, register-resident (the default when the contraction comes as one slice and k is a multiple of the
// 16-byte vector): only the Gram matrix sits in shared memory, so 2 (k = 128) to 8 blocks share an SM where the staged
// variant above fits one or two (its two staged tiles cost 66 KB at KM = 64, 132 KB at KM = 128).  A thread loads its
// own factor row into registers with 16-byte loads, reads the contraction entry of each step straight from global
// memory (16-byte loads, one group of 8 steps ahead), and writes the row and its transpose itself.  Same direct form
// and the same order of operations as update_rows_tpr_kernel -- the results are bit-identical.  Column sums are
// taken afterwards from the transposed copy (rowsum_flag_kernel).  Config-5 shard (125 000 rows, k = 128): W update
// 0.73 -> 0.43 ms, T update 0.23 -> 0.13 ms (profiles/r02_update_rows_reg_ab.txt).
// ------------------------------------------------------------------------------------------------
template <typename T, int KM>
__global__ void __launch_bounds__(128)
update_rows_reg_kernel(T* __restrict__ F, int64_t m, int k, const T* __restrict__ C, const T* __restrict__ S,
                       T reg_l1, T reg_l2, T eps, T ub, int has_ub, T* __restrict__ Ft, int64_t ldft,
                       int* __restrict__ flags, int64_t ldc, int64_t lds, int64_t s_stride)
{
    using V = typename Vec<T>::type;
    constexpr int VN = Vec<T>::N;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T* Ss = reinterpret_cast<T*>(smem_raw);                  // [KM][KM], zero padded
    const int tid = threadIdx.x;
    const int z = blockIdx.y;                                // model (RowBatch)
    F += (int64_t)z * m * k;
    C += (int64_t)z * k;
    S += (int64_t)z * s_stride;
    if (Ft) Ft += (int64_t)z * k * ldft;
    flags += z;
    for (int e = tid; e < KM * KM; e += 128) {
        const int a = e / KM, b = e % KM;
        Ss[e] = (a < k && b < k) ? S[a * lds + b] : T(0);
    }
    __syncthreads();
    bool unb = false;
    for (int64_t row = (int64_t)blockIdx.x * 128 + tid; row < m; row += (int64_t)gridDim.x * 128) {
        T f[KM];
        const V* frowv = reinterpret_cast<const V*>(F + row * k);                  // k % VN == 0 (checked by the launcher)
#pragma unroll
        for (int jv = 0; jv < KM / VN; ++jv) {
            T fv[VN];
#pragma unroll
            for (int v = 0; v < VN; ++v) fv[v] = T(0);
            if (VN * jv < k) unpack(frowv[jv], fv);
#pragma unroll
            for (int v = 0; v < VN; ++v) f[VN * jv + v] = fv[v];
        }
        // the contraction entries of 8 steps come as 16-byte loads, requested one group of steps ahead (a scalar load
        // per step leaves its line in L1 for the next 31 steps of the same thread -- with 16 warps per SM walking 32
        // rows each the lines do not survive, and every step waits for L2)
        const V* crowv = reinterpret_cast<const V*>(C + row * ldc);
        constexpr int GV = 8 / VN;                                                  // vectors per group of 8 steps
        T cn[8];
#pragma unroll
        for (int v = 0; v < GV; ++v) {
            T cv[VN];
#pragma unroll
            for (int x = 0; x < VN; ++x) cv[x] = T(0);
            if (VN * v < k) unpack(crowv[v], cv);
#pragma unroll
            for (int x = 0; x < VN; ++x) cn[VN * v + x] = cv[x];
        }
#pragma unroll 1
        for (int c = 0; c < (k + 7) / 8; ++c) {
            T cc[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) cc[u] = cn[u];
#pragma unroll
            for (int v = 0; v < GV; ++v) {
                const int jv = GV * (c + 1) + v;
                if (VN * jv < k) {
                    T cv[VN];
                    unpack(crowv[jv], cv);
#pragma unroll
                    for (int x = 0; x < VN; ++x) cn[VN * v + x] = cv[x];
                }
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int t = 8 * c + u;
                if (t < k) {
                    const V* srow = reinterpret_cast<const V*>(Ss + t * KM);
                    T acc[4] = {T(0), T(0), T(0), T(0)};
#pragma unroll
                    for (int jv = 0; jv < KM / VN; ++jv) {
                        T sv[VN];
                        unpack(srow[jv], sv);
#pragma unroll
                        for (int v = 0; v < VN; ++v) acc[(jv * VN + v) & 3] = fma(f[jv * VN + v], sv[v], acc[(jv * VN + v) & 3]);
                    }
                    T ft = f[u];
#pragma unroll
                    for (int jj = 1; jj < KM / 8; ++jj) ft = (jj == c) ? f[8 * jj + u] : ft;
                    const T stt = Ss[t * KM + t];
                    const T dot = ((acc[0] + acc[1]) + (acc[2] + acc[3])) - ft * stt;
                    const T x = solve_scalar_c<T>(cc[u] - dot - reg_l1, stt + reg_l2, eps, ub, has_ub != 0, unb);
#pragma unroll
                    for (int jj = 0; jj < KM / 8; ++jj) f[8 * jj + u] = (jj == c) ? x : f[8 * jj + u];
                }
            }
        }
        V* fout = reinterpret_cast<V*>(F + row * k);
#pragma unroll
        for (int jv = 0; jv < KM / VN; ++jv)
            if (VN * jv < k) {
                V o;
                T* op = reinterpret_cast<T*>(&o);
#pragma unroll
                for (int v = 0; v < VN; ++v) op[v] = f[VN * jv + v];
                fout[jv] = o;
            }
        if (Ft) {
#pragma unroll
            for (int t = 0; t < KM; ++t)
                if (t < k) Ft[(int64_t)t * ldft + row] = f[t];
        }
    }
    if (unb) atomicOr(flags, 4);
}

// fp32 form of update_rows_reg_kernel on packed arithmetic: the factor row lives in 64-bit register pairs and the
// dot product of a step is 32 fma.rn.f32x2 (two IEEE fp32 FMAs per instruction, sm_100) instead of 64 FFMA.  Lane 0 / 1
// of accumulator pair 0 are the chains acc[0] / acc[1] of the scalar kernel, pair 1 holds acc[2] / acc[3], and the
// products enter in the same order: the results are bit-identical.
__device__ __forceinline__ void ffma2(unsigned long long& acc, unsigned long long a, unsigned long long b)
{
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(b));
}
__device__ __forceinline__ float lo_f(unsigned long long v) { return __uint_as_float((unsigned)v); }
__device__ __forceinline__ float hi_f(unsigned long long v) { return __uint_as_float((unsigned)(v >> 32)); }
__device__ __forceinline__ unsigned long long pack_f(float lo, float hi)
{
    return (unsigned long long)__float_as_uint(lo) | ((unsigned long long)__float_as_uint(hi) << 32);
}

template <int KM>
__global__ void __launch_bounds__(128)
update_rows_reg_x2_kernel(float* __restrict__ F, int64_t m, int k, const float* __restrict__ C, const float* __restrict__ S,
                          float reg_l1, float reg_l2, float eps, float ub, int has_ub, float* __restrict__ Ft, int64_t ldft,
                          int* __restrict__ flags, int64_t ldc, int64_t lds, int64_t s_stride)
{
    using U64 = unsigned long long;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* Ss = reinterpret_cast<float*>(smem_raw);           // [KM][KM], zero padded
    const int tid = threadIdx.x;
    const int z = blockIdx.y;                                 // model (RowBatch)
    F += (int64_t)z * m * k;
    C += (int64_t)z * k;
    S += (int64_t)z * s_stride;
    if (Ft) Ft += (int64_t)z * k * ldft;
    flags += z;
    for (int e = tid; e < KM * KM; e += 128) {
        const int a = e / KM, b = e % KM;
        Ss[e] = (a < k && b < k) ? S[a * lds + b] : 0.f;
    }
    __syncthreads();
    bool unb = false;
    for (int64_t row = (int64_t)blockIdx.x * 128 + tid; row < m; row += (int64_t)gridDim.x * 128) {
        U64 fp[KM / 2];                                       // fp[j] = (f[2j], f[2j+1])
        const ulonglong2* frowv = reinterpret_cast<const ulonglong2*>(F + row * k);      // k % 4 == 0
#pragma unroll
        for (int jv = 0; jv < KM / 4; ++jv) {
            ulonglong2 v = make_ulonglong2(0ull, 0ull);
            if (4 * jv < k) v = frowv[jv];
            fp[2 * jv] = v.x; fp[2 * jv + 1] = v.y;
        }
        const float4* crowv = reinterpret_cast<const float4*>(C + row * ldc);
        float cn[8];
#pragma unroll
        for (int v = 0; v < 2; ++v) {
            float4 cv = make_float4(0.f, 0.f, 0.f, 0.f);
            if (4 * v < k) cv = crowv[v];
            cn[4 * v] = cv.x; cn[4 * v + 1] = cv.y; cn[4 * v + 2] = cv.z; cn[4 * v + 3] = cv.w;
        }
#pragma unroll 1
        for (int c = 0; c < (k + 7) / 8; ++c) {
            float cc[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) cc[u] = cn[u];
#pragma unroll
            for (int v = 0; v < 2; ++v) {
                const int jv = 2 * (c + 1) + v;
                if (4 * jv < k) {
                    const float4 cv = crowv[jv];
                    cn[4 * v] = cv.x; cn[4 * v + 1] = cv.y; cn[4 * v + 2] = cv.z; cn[4 * v + 3] = cv.w;
                }
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int t = 8 * c + u;
                if (t < k) {
                    const ulonglong2* srow = reinterpret_cast<const ulonglong2*>(Ss + t * KM);
                    U64 a01 = 0ull, a23 = 0ull;
#pragma unroll
                    for (int jv = 0; jv < KM / 4; ++jv) {
                        const ulonglong2 sv = srow[jv];
                        ffma2(a01, fp[2 * jv], sv.x);
                        ffma2(a23, fp[2 * jv + 1], sv.y);
                    }
                    // f[8 jj + u] = half (u & 1) of pair 4 jj + u / 2
                    U64 fpair = fp[u / 2];
#pragma unroll
                    for (int jj = 1; jj < KM / 8; ++jj) fpair = (jj == c) ? fp[4 * jj + u / 2] : fpair;
                    const float ft = (u & 1) ? hi_f(fpair) : lo_f(fpair);
                    const float stt = Ss[t * KM + t];
                    const float dot = ((lo_f(a01) + hi_f(a01)) + (lo_f(a23) + hi_f(a23))) - ft * stt;
                    const float x = solve_scalar_c<float>(cc[u] - dot - reg_l1, stt + reg_l2, eps, ub, has_ub != 0, unb);
#pragma unroll
                    for (int jj = 0; jj < KM / 8; ++jj) {
                        const U64 old = fp[4 * jj + u / 2];
                        const U64 upd = (u & 1) ? pack_f(lo_f(old), x) : pack_f(x, hi_f(old));
                        fp[4 * jj + u / 2] = (jj == c) ? upd : old;
                    }
                }
            }
        }
        ulonglong2* fout = reinterpret_cast<ulonglong2*>(F + row * k);
#pragma unroll
        for (int jv = 0; jv < KM / 4; ++jv)
            if (4 * jv < k) fout[jv] = make_ulonglong2(fp[2 * jv], fp[2 * jv + 1]);
        if (Ft) {
#pragma unroll
            for (int t = 0; t < KM; ++t)
                if (t < k) Ft[(int64_t)t * ldft + row] = (t & 1) ? hi_f(fp[t / 2]) : lo_f(fp[t / 2]);
        }
    }
    if (unb) atomicOr(flags, 4);
}

template <typename T, int KM>
static void launch_update_rows_reg(T* F, int64_t m, int k, const T* C, const T* S, const SolveArgs& a, T* Ft, int64_t ldft,
                                   int* flags, const ColsumOut& co, const RowBatch& rb, cudaStream_t st)
{
    const size_t smem = sizeof(T) * KM * KM;
    const dim3 nb((unsigned)((m + 127) / 128), (unsigned)rb.models);
    if constexpr (sizeof(T) == 4) {
        auto kx = update_rows_reg_x2_kernel<KM>;
        if (smem > 48 * 1024) cudaFuncSetAttribute(kx, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        kx<<<nb, 128, smem, st>>>(F, m, k, C, S, (T)a.reg_l1, (T)a.reg_l2, (T)a.eps, (T)a.ub, a.has_ub, Ft, ldft, flags,
                                  rb.ldc, rb.lds, rb.s_stride);
    } else {
        auto kern = update_rows_reg_kernel<T, KM>;
        if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        kern<<<nb, 128, smem, st>>>(F, m, k, C, S, (T)a.reg_l1, (T)a.reg_l2, (T)a.eps, (T)a.ub, a.has_ub, Ft, ldft, flags,
                                    rb.ldc, rb.lds, rb.s_stride);
    }
    if (co.sums) launch_rowsum_flag<T>(Ft, k, m, ldft, co.sums, co.off, co.zero_flag, flags, st);
}

// ------------------------------------------------------------------------------------------------
// Multi-GPU T half-step: exchange over NVLink peer memory FUSED with the rank-one updates (one launch).
//
// Every rank r holds, in an exchange buffer that all ranks have mapped, its partial statistic of this sweep
// [X_r'W_r (d x k) | W_r'W_r (k x k)] (nmf.py:680-686, batched over topics), a replica of T' (d x k, the factor
// rows this kernel updates) and of T (k x ldtk, the operand of the next W half-step).  Rank r owns the rows
// [row_lo, row_hi) of T':
//   1. publish "my partial is complete" to every peer (flag1, release at system scope) and wait for all peers';
//   2. add the k x k Gram partials and, per 128-row block, the contraction rows of all ranks in rank order
//      (in-place NVLink reads: the reduce-scatter half of an all-reduce, never materialised);
//   3. run the k sequential solves of those rows (nmf.py:437-447 with the Gram form of :672-676);
//   4. store the new rows into EVERY rank's T' and T replicas (NVLink writes: the all-gather half) and the slice's
//      column sums into every rank's tsum table;
//   5. the last block to finish publishes flag2 to every peer, waits for all peers' flag2 -- after which this rank's
//      replicas are complete -- and finalises sum(T[t,:]) (nmf.py:757) from the tsum table.
// Each T entry is computed by exactly one rank from sums taken in a fixed order: the replicas are bit-identical.
// The work of the T update is divided by the number of ranks instead of being repeated on each of them.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void peer_flag_store(unsigned* p, unsigned v)
{
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned peer_flag_load(const unsigned* p)
{
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// threads r < world wait until peer r has published `epoch` in this rank's flag array
__device__ __forceinline__ void peer_wait_all(const unsigned* flags_local, int world, unsigned epoch, int* err)
{
    const int r = threadIdx.x;
    if (r < world) {
        const long long t0 = clock64();
        while ((int)(peer_flag_load(flags_local + 32 * r) - epoch) < 0) {
            if (clock64() - t0 > 200000000000LL) {     // ~100 s: a lost peer must not hang the GPU for ever
                atomicExch(err, 1 + r);
                __trap();
            }
            __nanosleep(100);
        }
    }
}

// --- exchange, part 1: publish this rank's partial, wait for all ranks', add the k x k Gram partials in rank order into
// a local buffer.  A handful of blocks; every remote load of a batch is in flight before the first add (a remote
// load takes ~2 us: a dependent chain per element would cost world x latency).
template <typename T>
__global__ void __launch_bounds__(256)
peer_gram_kernel(PeerExchange px, int64_t d, int k, T* __restrict__ Gsum)
{
    const int tid = threadIdx.x;
    const int world = px.world, rank = px.rank;
    if (blockIdx.x == 0 && tid < world) {
        __threadfence_system();
        peer_flag_store(px.flag1[tid] + 32 * rank, px.epoch);
    }
    peer_wait_all(px.flag1[rank], world, px.epoch, px.err);
    __syncthreads();
    const int64_t goff = d * (int64_t)k;
    constexpr int GB = 4;
    const int e0 = (blockIdx.x * 256 + tid) * GB;
    if (e0 >= k * k) return;
    T v[16][GB];
#pragma unroll
    for (int r = 0; r < 16; ++r)
        if (r < world) {
            const T* Gp = reinterpret_cast<const T*>(px.part[r]) + goff;
#pragma unroll
            for (int u = 0; u < GB; ++u) v[r][u] = (e0 + u < k * k) ? __ldcg(Gp + e0 + u) : T(0);
        }
#pragma unroll
    for (int u = 0; u < GB; ++u)
        if (e0 + u < k * k) {
            T acc = T(0);
#pragma unroll
            for (int r = 0; r < 16; ++r)
                if (r < world) acc += v[r][u];
            Gsum[e0 + u] = acc;
        }
}

// --- exchange, part 2 (launched right behind part 1: all partials are visible): the rank's own rows of T' in blocks
// of PEER_ROWS = 32 rows -- many small blocks, so that the NVLink reads of a block are few dependent round trips and
// the blocks of a slice spread over the idle SMs (a slice is d/g rows: 20 blocks of 128 rows kept 128 SMs idle and
// serialised 16-32 remote round trips per block).  All 128 threads load and store; warp 0 runs the 32 row solves.
constexpr int PEER_ROWS = 32;
constexpr int PEER_THREADS = 128;

template <typename T, int KM>
__global__ void __launch_bounds__(PEER_THREADS)
peer_update_rows_kernel(PeerExchange px, int64_t d, int k, const T* __restrict__ Gsum, T reg_l1, T reg_l2, T eps, T ub,
                        int has_ub, T* __restrict__ colsum_part, int* __restrict__ flags, double* __restrict__ sums,
                        unsigned* __restrict__ counter)
{
    constexpr int LD = KM + 1;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T* Ss = reinterpret_cast<T*>(smem_raw);
    T* ctile = Ss + KM * KM;
    T* ftile = ctile + PEER_ROWS * LD;
    __shared__ unsigned s_arrival;
    const int tid = threadIdx.x;
    const int world = px.world, rank = px.rank;
    for (int e = tid; e < KM * KM; e += PEER_THREADS) {
        const int a = e / KM, b = e % KM;
        Ss[e] = (a < k && b < k) ? Gsum[a * k + b] : T(0);
    }
    T csum = T(0);
    bool unb = false;
    __syncthreads();
    const int64_t m = px.row_hi - px.row_lo;
    const int64_t ngroups = (m + PEER_ROWS - 1) / PEER_ROWS;
    T* Floc = reinterpret_cast<T*>(px.Tt[rank]);
    for (int64_t g = blockIdx.x; g < ngroups; g += gridDim.x) {
        const int64_t i0 = px.row_lo + g * PEER_ROWS;
        const int nrow = (int)((px.row_hi - i0) < PEER_ROWS ? (px.row_hi - i0) : PEER_ROWS);
        {   // staging: contraction rows summed over the ranks (in place, over NVLink), own factor rows; the loads of all
            // ranks for a batch of elements are in flight together
            const int tot = nrow * k;
            int rr = tid / k, cc = tid - rr * k;
            const int dr = PEER_THREADS / k, dc = PEER_THREADS - dr * k;
            const T* Frow = Floc + i0 * k;
            constexpr int UB = sizeof(T) == 8 ? 4 : 8;
            for (int e0 = tid; e0 < tot; e0 += UB * PEER_THREADS) {
                T acc[UB], fv[UB];
#pragma unroll
                for (int u = 0; u < UB; ++u) {
                    const int e = e0 + u * PEER_THREADS;
                    acc[u] = T(0);
                    fv[u] = e < tot ? Frow[e] : T(0);
                }
                for (int r0 = 0; r0 < world; r0 += 8) {                // ranks in groups of 8, added in rank order
                    T cv[8][UB];
#pragma unroll
                    for (int r = 0; r < 8; ++r)
                        if (r0 + r < world) {
                            const T* Cp = reinterpret_cast<const T*>(px.part[r0 + r]) + i0 * k;
#pragma unroll
                            for (int u = 0; u < UB; ++u) {
                                const int e = e0 + u * PEER_THREADS;
                                cv[r][u] = e < tot ? __ldcg(Cp + e) : T(0);
                            }
                        }
#pragma unroll
                    for (int r = 0; r < 8; ++r)
                        if (r0 + r < world) {
#pragma unroll
                            for (int u = 0; u < UB; ++u) acc[u] += cv[r][u];
                        }
                }
#pragma unroll
                for (int u = 0; u < UB; ++u) {
                    const int e = e0 + u * PEER_THREADS;
                    if (e < tot) {
                        ctile[rr * LD + cc] = acc[u];
                        ftile[rr * LD + cc] = fv[u];
                    }
                    rr += dr; cc += dc;
                    while (cc >= k) { cc -= k; ++rr; }
                }
            }
        }
        __syncthreads();
        // the k sequential solves (nmf.py:437-447 with the Gram form of :672-676), one thread per row
        if (tid < nrow) tpr_solve_row<T, KM>(Ss, ctile, ftile, tid, k, reg_l1, reg_l2, eps, ub, has_ub != 0, unb);
        __syncthreads();
        {   // fan-out: the new rows into every rank's T' (row-major) and T (transposed) replicas
            const int tot = nrow * k;
            for (int r = 0; r < world; ++r) {
                const int pr = (rank + r) % world;                     // start with the own copy, spread the peers
                T* Frow = reinterpret_cast<T*>(px.Tt[pr]) + i0 * k;
                int rr = tid / k, cc = tid - rr * k;
                const int dr = PEER_THREADS / k, dc = PEER_THREADS - dr * k;
                for (int e = tid; e < tot; e += PEER_THREADS) {
                    Frow[e] = ftile[rr * LD + cc];
                    rr += dr; cc += dc;
                    while (cc >= k) { cc -= k; ++rr; }
                }
                // transposed copy: thread (ii, tp0) writes (tp0 + 4j, i0 + ii): 32 consecutive addresses per warp
                T* Ft = reinterpret_cast<T*>(px.Tk[pr]);
                const int ii = tid % PEER_ROWS, tp0 = tid / PEER_ROWS;
                if (ii < nrow)
                    for (int tp = tp0; tp < k; tp += PEER_THREADS / PEER_ROWS) Ft[(int64_t)tp * px.ldtk + i0 + ii] = ftile[ii * LD + tp];
            }
            if (tid < k) {
                T cs = T(0);
#pragma unroll 8
                for (int ii = 0; ii < nrow; ++ii) cs += ftile[ii * LD + tid];
                csum += cs;
            }
        }
        __syncthreads();
    }
    if (unb) atomicOr(flags, 4);
    if (tid < k) colsum_part[(int64_t)blockIdx.x * k + tid] = csum;
    // last block: slice sums to every rank, flag2, wait for the peers, finalise sum(T[t,:])
    __threadfence_system();                            // this block's stores (local and remote) before its arrival
    __syncthreads();
    if (tid == 0) s_arrival = atomicAdd(counter, 1u);
    __syncthreads();
    if (s_arrival != gridDim.x - 1) return;
    __threadfence();
    if (tid < k) {
        T s = T(0);
        for (int b = 0; b < (int)gridDim.x; ++b) s += __ldcg(colsum_part + (int64_t)b * k + tid);
        for (int r = 0; r < world; ++r) reinterpret_cast<T*>(px.tsum[r])[rank * k + tid] = s;
    }
    __threadfence_system();
    __syncthreads();
    if (tid < world) {
        __threadfence_system();
        peer_flag_store(px.flag2[tid] + 32 * rank, px.epoch);
    }
    peer_wait_all(px.flag2[rank], world, px.epoch, px.err);
    __syncthreads();
    if (tid < k) {
        const T* ts = reinterpret_cast<const T*>(px.tsum[rank]);
        T s = T(0);
        for (int r = 0; r < world; ++r) s += __ldcg(ts + r * k + tid);
        const double v = (double)s;
        sums[tid] = v;
        if (!(v > 1e-10)) atomicOr(flags, 1);
        if (!isfinite(v)) atomicOr(flags, 8);
    }
    if (tid == 0) *counter = 0u;
}

int peer_update_blocks(int64_t rows, int sm_count)
{
    int64_t b = (rows + PEER_ROWS - 1) / PEER_ROWS;
    if (b > 4 * sm_count) b = 4 * sm_count;
    return (int)(b < 1 ? 1 : b);
}

template <typename T>
int launch_peer_update_rows(const PeerExchange& px, int64_t d, int k, const SolveArgs& a, T* Gsum, T* colsum_part,
                            int* flags, double* sums, unsigned* counter, int blocks, cudaStream_t st)
{
    const bool ok = sizeof(T) == 4 ? k <= 128 : k <= 64;
    if (!ok) return 0;                                 // rank too wide for the thread-per-row kernel: not fused
    peer_gram_kernel<T><<<(k * k + 1023) / 1024, 256, 0, st>>>(px, d, k, Gsum);
#define RRI_PEER(KM)                                                                                                  \
    do {                                                                                                              \
        const size_t smem = sizeof(T) * ((size_t)KM * KM + 2 * (size_t)PEER_ROWS * (KM + 1));                         \
        auto kern = peer_update_rows_kernel<T, KM>;                                                                   \
        if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);     \
        kern<<<blocks, PEER_THREADS, smem, st>>>(px, d, k, Gsum, (T)a.reg_l1, (T)a.reg_l2, (T)a.eps, (T)a.ub,         \
                                                a.has_ub, colsum_part, flags, sums, counter);                         \
        return 2;                                                                                                     \
    } while (0)
    if (k <= 16) RRI_PEER(16);
    if (k <= 32) RRI_PEER(32);
    if (k <= 64) RRI_PEER(64);
    if constexpr (sizeof(T) == 4) { if (k <= 128) RRI_PEER(128); }
#undef RRI_PEER
    return 0;
}

template <typename T>
void launch_update_rows(T* F, int64_t m, int k, const T* Cpart, int parts, int64_t part_stride,
                        const T* const* srcs, const T* S, const SolveArgs& a, T* Ft, int64_t ldft,
                        T* colsum_part, int* flags, int blocks, const ColsumOut& co, const RowBatch& rb,
                        cudaStream_t st)
{
    // thread-per-row variants while the row fits in registers / the tiles in shared memory
    // (fp32: k <= 128, fp64: k <= 64); wider ranks use the warp-per-row kernel
    {
        constexpr int VN = Vec<T>::N;
        // (16-byte loads of the factor and contraction rows: F and Cpart point at a model of a handle of several, which
        // need not start on a 16-byte boundary; such a model takes the staged kernel, which gives the same bits)
        const bool vec = (k % VN) == 0 && (rb.ldc % VN) == 0 && (reinterpret_cast<uintptr_t>(F) & 15) == 0 &&
                         (reinterpret_cast<uintptr_t>(Cpart) & 15) == 0;
        if (parts == 1 && !srcs && Ft && vec && k <= (sizeof(T) == 4 ? 128 : 64)) {
            if (k <= 16) launch_update_rows_reg<T, 16>(F, m, k, Cpart, S, a, Ft, ldft, flags, co, rb, st);
            else if (k <= 32) launch_update_rows_reg<T, 32>(F, m, k, Cpart, S, a, Ft, ldft, flags, co, rb, st);
            else if (k <= 64) launch_update_rows_reg<T, 64>(F, m, k, Cpart, S, a, Ft, ldft, flags, co, rb, st);
            else if constexpr (sizeof(T) == 4) launch_update_rows_reg<T, 128>(F, m, k, Cpart, S, a, Ft, ldft, flags, co, rb, st);
            return;
        }
    }
#define RRI_TPR(KM) launch_update_rows_tpr<T, KM>(F, m, k, Cpart, parts, part_stride, srcs, S, a, Ft, ldft, colsum_part, flags, blocks, co, rb, st)
    if (k <= 16) { RRI_TPR(16); return; }
    if (k <= 32) { RRI_TPR(32); return; }
    if (k <= 64) { RRI_TPR(64); return; }
    if (k <= 128 && sizeof(T) == 4) { RRI_TPR(128); return; }
#undef RRI_TPR
    const int kl = (k + 31) / 32;
    if (kl <= 1) launch_update_rows_kl<T, 1>(F, m, k, Cpart, parts, part_stride, srcs, S, a, Ft, ldft, colsum_part, flags, blocks, co, rb, st);
    else if (kl <= 2) launch_update_rows_kl<T, 2>(F, m, k, Cpart, parts, part_stride, srcs, S, a, Ft, ldft, colsum_part, flags, blocks, co, rb, st);
    else if (kl <= 4) launch_update_rows_kl<T, 4>(F, m, k, Cpart, parts, part_stride, srcs, S, a, Ft, ldft, colsum_part, flags, blocks, co, rb, st);
    else launch_update_rows_kl<T, 8>(F, m, k, Cpart, parts, part_stride, srcs, S, a, Ft, ldft, colsum_part, flags, blocks, co, rb, st);
}

// ------------------------------------------------------------------------------------------------
// Gram G = F'F
// ------------------------------------------------------------------------------------------------
constexpr int GR_ROWS = 32;      // rows staged per iteration

int gram_chunks(int64_t m, int k, int sm_count)
{
    const int kb = (k + 63) / 64;
    int64_t c = (2 * sm_count) / (kb * kb);
    const int64_t maxc = (m + 4 * GR_ROWS - 1) / (4 * GR_ROWS);
    if (c > maxc) c = maxc;
    return (int)(c < 1 ? 1 : c);
}

template <typename T>
__global__ void __launch_bounds__(256)
gram_kernel(const T* __restrict__ F, int64_t m, int k, T* __restrict__ part, int64_t f_stride)
{
    F += (int64_t)blockIdx.z * f_stride;                   // model z (launch_gram with models > 1)
    __shared__ T Fa[GR_ROWS][64 + 1];
    __shared__ T Fb[GR_ROWS][64 + 1];
    const int kb = (k + 63) / 64;
    const int a0 = (blockIdx.y / kb) * 64, b0 = (blockIdx.y % kb) * 64;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    int64_t r0, r1;
    part_range(m, gridDim.x, blockIdx.x, r0, r1);
    T acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = T(0);
    for (int64_t rb = r0; rb < r1; rb += GR_ROWS) {
        {   // all of this thread's loads first (one round trip per tile), then the shared-memory stores
            T va[GR_ROWS * 64 / 256], vb[GR_ROWS * 64 / 256];
#pragma unroll
            for (int u = 0; u < GR_ROWS * 64 / 256; ++u) {
                const int e = tid + u * 256;
                const int rr = e / 64, cc = e % 64;
                const int64_t gr = rb + rr;
                va[u] = (gr < r1 && a0 + cc < k) ? F[gr * k + a0 + cc] : T(0);
                vb[u] = (a0 == b0) ? va[u] : ((gr < r1 && b0 + cc < k) ? F[gr * k + b0 + cc] : T(0));
            }
#pragma unroll
            for (int u = 0; u < GR_ROWS * 64 / 256; ++u) {
                const int e = tid + u * 256;
                Fa[e / 64][e % 64] = va[u];
                Fb[e / 64][e % 64] = vb[u];
            }
        }
        __syncthreads();
#pragma unroll 8
        for (int rr = 0; rr < GR_ROWS; ++rr) {
            T a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = Fa[rr][ty + 16 * i];
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = Fb[rr][tx + 16 * j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fma(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
    T* P = part + ((int64_t)blockIdx.x * gridDim.z + blockIdx.z) * k * k;      // [chunks][models][k*k]
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int a = a0 + ty + 16 * i, b = b0 + tx + 16 * j;
            if (a < k && b < k) P[a * k + b] = acc[i][j];
        }
}

template <typename T>
__global__ void reduce_parts_kernel(const T* __restrict__ part, int parts, int64_t stride, int64_t len,
                                    T* __restrict__ out)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c < len) {
        T s = T(0);
        for (int p = 0; p < parts; ++p) s += part[(int64_t)p * stride + c];
        out[c] = s;
    }
}

// same sum with one warp per output element (lanes stride over the parts, fixed shuffle tree):
// for short outputs with many parts (Gram partials) the serial version is latency-bound
template <typename T>
__global__ void __launch_bounds__(256)
reduce_parts_warp_kernel(const T* __restrict__ part, int parts, int64_t stride, int64_t len, T* __restrict__ out)
{
    const int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (c >= len) return;
    T s = T(0);
    for (int p = lane; p < parts; p += 32) s += part[(int64_t)p * stride + c];
    s = warp_sum(s);
    if (lane == 0) out[c] = s;
}

template <typename T>
void launch_reduce_parts(const T* part, int parts, int64_t stride, int64_t len, T* out, cudaStream_t st)
{
    if (parts >= 16 && len <= 65536)
        reduce_parts_warp_kernel<T><<<(unsigned)((len * 32 + 255) / 256), 256, 0, st>>>(part, parts, stride, len, out);
    else
        reduce_parts_kernel<T><<<(unsigned)((len + 255) / 256), 256, 0, st>>>(part, parts, stride, len, out);
}

template <typename T>
__global__ void sum_sources_kernel(const T* const* __restrict__ srcs, int parts, int64_t len, T* __restrict__ out)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c < len) {
        T s = T(0);
        for (int p = 0; p < parts; ++p) s += srcs[p][c];
        out[c] = s;
    }
}

template <typename T>
void launch_sum_sources(const T* const* srcs, int parts, int64_t len, T* out, cudaStream_t st)
{
    sum_sources_kernel<T><<<(unsigned)((len + 255) / 256), 256, 0, st>>>(srcs, parts, len, out);
}

template <typename T>
void launch_gram(const T* F, int64_t m, int k, T* part, int chunks, T* G, cudaStream_t st, int models, int64_t f_stride)
{
    const int kb = (k + 63) / 64;
    dim3 grid(chunks, kb * kb, models);
    gram_kernel<T><<<grid, 256, 0, st>>>(F, m, k, part, f_stride);
    // (models * k * k <= 256 * 256: the reduction kernel, and with it the order of the sums, is the one model's)
    const int64_t len = (int64_t)models * k * k;
    launch_reduce_parts<T>(part, chunks, len, len, G, st);
}

template <typename T>
__global__ void __launch_bounds__(256)
colsum_finalize_kernel(const T* __restrict__ colsum_part, int blocks, int k, double* __restrict__ sums,
                       int off, int zero_flag, int* __restrict__ flags)
{
    // one warp per column; lanes stride over the block partials, fixed-order shuffle tree
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= k) return;
    T s = T(0);
    for (int b = lane; b < blocks; b += 32) s += colsum_part[(int64_t)b * k + warp];
    s = warp_sum(s);
    if (lane == 0) {
        const double v = (double)s;
        sums[off + warp] = v;
        if (zero_flag && !(v > 1e-10)) atomicOr(flags, zero_flag);
        if (!isfinite(v)) atomicOr(flags, 8);
    }
}

template <typename T>
void launch_colsum_finalize(const T* colsum_part, int blocks, int k, double* sums, int off,
                            int zero_flag, int* flags, cudaStream_t st)
{
    colsum_finalize_kernel<T><<<(k * 32 + 255) / 256, 256, 0, st>>>(colsum_part, blocks, k, sums, off, zero_flag, flags);
}

// ------------------------------------------------------------------------------------------------
// transpose
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
transpose_kernel(const T* __restrict__ A, int64_t rows, int64_t cols, int64_t lda, T* __restrict__ B, int64_t ldb)
{
    __shared__ T tile[32][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;     // 32 x 8
    const int64_t c0 = (int64_t)blockIdx.x * 32, r0 = (int64_t)blockIdx.y * 32;
#pragma unroll
    for (int j = 0; j < 32; j += 8) {
        const int64_t r = r0 + ty + j, c = c0 + tx;
        if (r < rows && c < cols) tile[ty + j][tx] = A[r * lda + c];
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 32; j += 8) {
        const int64_t c = c0 + ty + j, r = r0 + tx;
        if (r < rows && c < cols) B[c * ldb + r] = tile[tx][ty + j];
    }
}

template <typename T>
void launch_transpose(const T* A, int64_t rows, int64_t cols, int64_t lda, T* B, int64_t ldb, cudaStream_t st)
{
    // grid.y is limited to 65535 blocks -> tile rows over x when rows is the long side
    const int64_t bx = (cols + 31) / 32, by = (rows + 31) / 32;
    if (by <= 65535) {
        dim3 grid((unsigned)bx, (unsigned)by);
        transpose_kernel<T><<<grid, 256, 0, st>>>(A, rows, cols, lda, B, ldb);
    } else {
        for (int64_t r = 0; r < rows; r += 65535LL * 32) {
            const int64_t rr = (rows - r) < 65535LL * 32 ? (rows - r) : 65535LL * 32;
            dim3 grid((unsigned)bx, (unsigned)((rr + 31) / 32));
            transpose_kernel<T><<<grid, 256, 0, st>>>(A + r * lda, rr, cols, lda, B + r, ldb);
        }
    }
}

#define RRI_INST(T)                                                                                       \
    template void launch_simt_gemm_nt<T>(const T*, int64_t, const T*, int64_t, T*, int64_t, int, int64_t, \
                                         int, cudaStream_t);                                              \
    template void launch_update_rows<T>(T*, int64_t, int, const T*, int, int64_t, const T* const*,        \
                                        const T*, const SolveArgs&, T*, int64_t, T*, int*, int,            \
                                        const ColsumOut&, const RowBatch&, cudaStream_t);                  \
    template int launch_peer_update_rows<T>(const PeerExchange&, int64_t, int, const SolveArgs&, T*, T*,    \
                                            int*, double*, unsigned*, int, cudaStream_t);                  \
    template void launch_sum_sources<T>(const T* const*, int, int64_t, T*, cudaStream_t);                  \
    template void launch_gram<T>(const T*, int64_t, int, T*, int, T*, cudaStream_t, int, int64_t);        \
    template void launch_reduce_parts<T>(const T*, int, int64_t, int64_t, T*, cudaStream_t);              \
    template void launch_colsum_finalize<T>(const T*, int, int, double*, int, int, int*, cudaStream_t);   \
    template void launch_transpose<T>(const T*, int64_t, int64_t, int64_t, T*, int64_t, cudaStream_t);
RRI_INST(float)
RRI_INST(double)

}  // namespace rri
