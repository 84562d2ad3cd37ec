// wrri_kernels.cu -- masked / weighted WRRI half-step statistics (Ho's Alg. 10 as implemented by
// nmf.py:687-701 and :735-746) and the objective of nmf.py:71-94.
//
// The reference materialises R = W_mat o (X - W_{t->0} T) (an n x k x d GEMM plus three n x d
// temporaries) for every half-step.  Here R is never stored: each 64x64 tile of W_{t->0}T is formed
// in registers from staged factor tiles and consumed immediately against the X / W_mat tiles, which
// are each read once per half-step.
#include "common.cuh"
#include "kernels.h"

namespace rri {

constexpr int TL = 64;           // tile edge
constexpr int TKC = 32;          // k-chunk staged in shared memory
constexpr int TL_THREADS = 256;

template <typename T, int MK>
RRI_DEVINL T load_mask(const void* M, int64_t idx)
{
    if (MK == MK_NONE) return T(1);
    if (MK == MK_REAL) return ld_stream(reinterpret_cast<const T*>(M) + idx);
    return (T) reinterpret_cast<const unsigned char*>(M)[idx];
}

// acc[i][j] = sum_{jj != skip} W[r0 + ty*4+i, jj] * T[jj, c0 + tx+16j]
template <typename T>
RRI_DEVINL void tile_product(const T* __restrict__ W, const T* __restrict__ Tm, int64_t n, int64_t d,
                             int k, int skip, int64_t r0, int64_t c0, T (*Ws)[TKC + 1], T (*Ts)[TL + 1],
                             T acc[4][4])
{
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = T(0);
    for (int kb = 0; kb < k; kb += TKC) {
        for (int e = tid; e < TL * TKC; e += TL_THREADS) {
            const int rr = e / TKC, jj = e % TKC;
            const int64_t gr = r0 + rr;
            const int gj = kb + jj;
            Ws[rr][jj] = (gr < n && gj < k && gj != skip) ? W[gr * k + gj] : T(0);
        }
        for (int e = tid; e < TKC * TL; e += TL_THREADS) {
            const int jj = e / TL, cc = e % TL;
            const int64_t gc = c0 + cc;
            const int gj = kb + jj;
            Ts[jj][cc] = (gc < d && gj < k) ? Tm[(int64_t)gj * d + gc] : T(0);
        }
        __syncthreads();
#pragma unroll 8
        for (int jj = 0; jj < TKC; ++jj) {
            T a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = Ws[ty * 4 + i][jj];
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = Ts[jj][tx + 16 * j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fma(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
// T-step statistics: grid (col tiles, row groups); block loops over the row tiles of its group
// ------------------------------------------------------------------------------------------------
template <typename T, int MK>
__global__ void __launch_bounds__(TL_THREADS)
wrri_tstats_kernel(const T* __restrict__ X, int64_t ldx, const void* __restrict__ M, int64_t ldm,
                   const T* __restrict__ W, const T* __restrict__ Tm, int64_t n, int64_t d, int k, int t,
                   int tiles_r, T* __restrict__ numer_part, T* __restrict__ denom_part)
{
    __shared__ T Ws[TL][TKC + 1];
    __shared__ T Ts[TKC][TL + 1];
    // the cross-thread reduction buffer aliases the W staging tile (free once the tile loop is done)
    static_assert(2 * 16 * (TL + 1) <= TL * (TKC + 1), "reduction buffer must fit in the W tile");
    T (*red)[16][TL + 1] = reinterpret_cast<T (*)[16][TL + 1]>(&Ws[0][0]);
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int64_t c0 = (int64_t)blockIdx.x * TL;
    int64_t tb, te;
    part_range(tiles_r, gridDim.y, blockIdx.y, tb, te);
    T nacc[4] = {0, 0, 0, 0}, dacc[4] = {0, 0, 0, 0};
    for (int64_t tr = tb; tr < te; ++tr) {
        const int64_t r0 = tr * TL;
        T acc[4][4];
        tile_product<T>(W, Tm, n, d, k, t, r0, c0, Ws, Ts, acc);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int64_t gr = r0 + ty * 4 + i;
            if (gr < n) {
                const T wt = W[gr * k + t];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int64_t gc = c0 + tx + 16 * j;
                    if (gc < d) {
                        const T m = load_mask<T, MK>(M, gr * ldm + gc);
                        const T r = m * (ld_stream(X + gr * ldx + gc) - acc[i][j]);
                        nacc[j] = fma(wt, r, nacc[j]);
                        dacc[j] = fma(wt * wt, m, dacc[j]);
                    }
                }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) { red[0][ty][tx + 16 * j] = nacc[j]; red[1][ty][tx + 16 * j] = dacc[j]; }
    __syncthreads();
    if (tid < 2 * TL) {
        const int which = tid / TL, cc = tid % TL;
        T s = T(0);
#pragma unroll
        for (int y = 0; y < 16; ++y) s += red[which][y][cc];
        if (c0 + cc < d) (which ? denom_part : numer_part)[(int64_t)blockIdx.y * d + c0 + cc] = s;
    }
}

// ------------------------------------------------------------------------------------------------
// W-step statistics: grid (row tiles, col groups); block loops over the col tiles of its group
// ------------------------------------------------------------------------------------------------
template <typename T, int MK>
__global__ void __launch_bounds__(TL_THREADS)
wrri_wstats_kernel(const T* __restrict__ X, int64_t ldx, const void* __restrict__ M, int64_t ldm,
                   const T* __restrict__ W, const T* __restrict__ Tm, int64_t n, int64_t d, int k, int t,
                   int tiles_c, T* __restrict__ numer_part, T* __restrict__ denom_part)
{
    __shared__ T Ws[TL][TKC + 1];
    __shared__ T Ts[TKC][TL + 1];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int64_t r0 = (int64_t)blockIdx.x * TL;
    int64_t tb, te;
    part_range(tiles_c, gridDim.y, blockIdx.y, tb, te);
    T nacc[4] = {0, 0, 0, 0}, dacc[4] = {0, 0, 0, 0};
    for (int64_t tc = tb; tc < te; ++tc) {
        const int64_t c0 = tc * TL;
        T acc[4][4];
        tile_product<T>(W, Tm, n, d, k, t, r0, c0, Ws, Ts, acc);
        T tt[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int64_t gc = c0 + tx + 16 * j;
            tt[j] = (gc < d) ? Tm[(int64_t)t * d + gc] : T(0);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int64_t gr = r0 + ty * 4 + i;
            if (gr < n) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int64_t gc = c0 + tx + 16 * j;
                    if (gc < d) {
                        const T m = load_mask<T, MK>(M, gr * ldm + gc);
                        const T r = m * (ld_stream(X + gr * ldx + gc) - acc[i][j]);
                        nacc[i] = fma(r, tt[j], nacc[i]);
                        dacc[i] = fma(m * tt[j], tt[j], dacc[i]);
                    }
                }
            }
        }
    }
    // reduce over the 16 tx lanes that share a row (a half-warp)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) {
            nacc[i] += __shfl_xor_sync(0xffffffffu, nacc[i], o);
            dacc[i] += __shfl_xor_sync(0xffffffffu, dacc[i], o);
        }
        const int64_t gr = r0 + ty * 4 + i;
        if (tx == 0 && gr < n) {
            numer_part[(int64_t)blockIdx.y * n + gr] = nacc[i];
            denom_part[(int64_t)blockIdx.y * n + gr] = dacc[i];
        }
    }
}

TilePlan plan_tstats(int64_t n, int64_t d, int sm_count)
{
    TilePlan p;
    p.tiles_r = (int)((n + TL - 1) / TL);
    p.tiles_c = (int)((d + TL - 1) / TL);
    int g = (4 * sm_count + p.tiles_c - 1) / p.tiles_c;
    if (g > p.tiles_r) g = p.tiles_r;
    p.groups = g < 1 ? 1 : g;
    return p;
}

TilePlan plan_wstats(int64_t n, int64_t d, int sm_count)
{
    TilePlan p;
    p.tiles_r = (int)((n + TL - 1) / TL);
    p.tiles_c = (int)((d + TL - 1) / TL);
    int g = (4 * sm_count + p.tiles_r - 1) / p.tiles_r;
    if (g > p.tiles_c) g = p.tiles_c;
    p.groups = g < 1 ? 1 : g;
    return p;
}

template <typename T>
void launch_wrri_tstats(const T* X, int64_t ldx, const void* M, int mk, int64_t ldm, const T* W,
                        const T* Tm, int64_t n, int64_t d, int k, int t, T* numer_part, T* denom_part,
                        const TilePlan& pl, cudaStream_t st)
{
    dim3 grid(pl.tiles_c, pl.groups);
    if (mk == MK_NONE) wrri_tstats_kernel<T, MK_NONE><<<grid, TL_THREADS, 0, st>>>(X, ldx, M, ldm, W, Tm, n, d, k, t, pl.tiles_r, numer_part, denom_part);
    else if (mk == MK_REAL) wrri_tstats_kernel<T, MK_REAL><<<grid, TL_THREADS, 0, st>>>(X, ldx, M, ldm, W, Tm, n, d, k, t, pl.tiles_r, numer_part, denom_part);
    else wrri_tstats_kernel<T, MK_U8><<<grid, TL_THREADS, 0, st>>>(X, ldx, M, ldm, W, Tm, n, d, k, t, pl.tiles_r, numer_part, denom_part);
}

template <typename T>
void launch_wrri_wstats(const T* X, int64_t ldx, const void* M, int mk, int64_t ldm, const T* W,
                        const T* Tm, int64_t n, int64_t d, int k, int t, T* numer_part, T* denom_part,
                        const TilePlan& pl, cudaStream_t st)
{
    dim3 grid(pl.tiles_r, pl.groups);
    if (mk == MK_NONE) wrri_wstats_kernel<T, MK_NONE><<<grid, TL_THREADS, 0, st>>>(X, ldx, M, ldm, W, Tm, n, d, k, t, pl.tiles_c, numer_part, denom_part);
    else if (mk == MK_REAL) wrri_wstats_kernel<T, MK_REAL><<<grid, TL_THREADS, 0, st>>>(X, ldx, M, ldm, W, Tm, n, d, k, t, pl.tiles_c, numer_part, denom_part);
    else wrri_wstats_kernel<T, MK_U8><<<grid, TL_THREADS, 0, st>>>(X, ldx, M, ldm, W, Tm, n, d, k, t, pl.tiles_c, numer_part, denom_part);
}

// ------------------------------------------------------------------------------------------------
// vector-c solve + helpers
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void wrri_final_kernel(const T* __restrict__ numer_part, const T* __restrict__ denom_part,
                                  int parts, int64_t len, T reg_l1, T reg_l2, T eps, T ub, int has_ub,
                                  T* __restrict__ out, int64_t out_stride, T* __restrict__ out2,
                                  int64_t out2_stride, int* __restrict__ flags)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= len) return;
    T nu = T(0), de = T(0);
#pragma unroll 4
    for (int p = 0; p < parts; ++p) {
        nu += numer_part[(int64_t)p * len + i];
        de += denom_part[(int64_t)p * len + i];
    }
    bool unb = false;
    const T x = solve_vector_c<T>(nu - reg_l1, de + reg_l2, eps, ub, has_ub != 0, unb);
    out[i * out_stride] = x;
    if (out2) out2[i * out2_stride] = x;
    if (unb) atomicOr(flags, 4);
}

template <typename T>
void launch_wrri_final(const T* numer_part, const T* denom_part, int parts, int64_t len,
                       const SolveArgs& a, T* out, int64_t out_stride, T* out2, int64_t out2_stride,
                       int* flags, cudaStream_t st)
{
    wrri_final_kernel<T><<<(unsigned)((len + 255) / 256), 256, 0, st>>>(numer_part, denom_part, parts, len,
        (T)a.reg_l1, (T)a.reg_l2, (T)a.eps, (T)a.ub, a.has_ub, out, out_stride, out2, out2_stride, flags);
}

template <typename T>
__global__ void __launch_bounds__(1024)
vec_sum_flag_kernel(const T* __restrict__ v, int64_t len, int64_t stride, double* __restrict__ sums,
                    int slot, int zero_flag, int* __restrict__ flags)
{
    __shared__ double red[32];
    double s = 0.0;
    for (int64_t i = threadIdx.x; i < len; i += blockDim.x) s += (double)v[i * stride];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += red[w];
        sums[slot] = tot;
        if (!(tot > 1e-10)) atomicOr(flags, zero_flag);
        if (!isfinite(tot)) atomicOr(flags, 8);
    }
}

template <typename T>
void launch_vec_sum_flag(const T* v, int64_t len, int64_t stride, double* sums, int slot, int zero_flag,
                         int* flags, cudaStream_t st)
{
    vec_sum_flag_kernel<T><<<1, 1024, 0, st>>>(v, len, stride, sums, slot, zero_flag, flags);
}

// sums[slot0 + r] = sum_i A[r*ld + i] for r < rows (one block per row, same fixed order as vec_sum_flag_kernel):
// the per-topic sums of a whole sweep in one launch
template <typename T>
__global__ void __launch_bounds__(1024)
rowsum_flag_kernel(const T* __restrict__ A, int64_t len, int64_t ld, double* __restrict__ sums, int slot0,
                   int zero_flag, int* __restrict__ flags, const int* __restrict__ topic_model)
{
    __shared__ double red[32];
    const T* __restrict__ v = A + (int64_t)blockIdx.x * ld;
    double s = 0.0;
    for (int64_t i = threadIdx.x; i < len; i += blockDim.x) s += (double)v[i];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += red[w];
        sums[slot0 + blockIdx.x] = tot;
        int* f = topic_model ? flags + topic_model[blockIdx.x] : flags;
        if (zero_flag && !(tot > 1e-10)) atomicOr(f, zero_flag);
        if (!isfinite(tot)) atomicOr(f, 8);
    }
}

template <typename T>
void launch_rowsum_flag(const T* A, int rows, int64_t len, int64_t ld, double* sums, int slot0, int zero_flag,
                        int* flags, cudaStream_t st, const int* topic_model)
{
    if (rows > 0) rowsum_flag_kernel<T><<<rows, 1024, 0, st>>>(A, len, ld, sums, slot0, zero_flag, flags, topic_model);
}

template <typename T>
__global__ void vec_scale_to_sum_kernel(T* __restrict__ v, int64_t len, int64_t stride,
                                        const double* __restrict__ sums, int slot, double s)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < len) v[i * stride] = (T)(s) * v[i * stride] / (T)sums[slot];
}

template <typename T>
void launch_vec_scale_to_sum(T* v, int64_t len, int64_t stride, const double* sums, int slot, double s,
                             cudaStream_t st)
{
    vec_scale_to_sum_kernel<T><<<(unsigned)((len + 255) / 256), 256, 0, st>>>(v, len, stride, sums, slot, s);
}

// ------------------------------------------------------------------------------------------------
// objective
// ------------------------------------------------------------------------------------------------
int obj_blocks(int64_t n, int64_t d, int sm_count)
{
    const int64_t tiles = ((n + TL - 1) / TL) * ((d + TL - 1) / TL);
    int64_t b = 4 * sm_count;
    if (b > tiles) b = tiles;
    return (int)(b < 1 ? 1 : b);
}

template <typename T, int MK>
__global__ void __launch_bounds__(TL_THREADS)
objective_kernel(const T* __restrict__ X, int64_t ldx, const void* __restrict__ M, int64_t ldm,
                 const T* __restrict__ W, const T* __restrict__ Tm, int64_t n, int64_t d, int k,
                 double* __restrict__ part)
{
    __shared__ T Ws[TL][TKC + 1];
    __shared__ T Ts[TKC][TL + 1];
    __shared__ double red[2][TL_THREADS / WARP];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int64_t tiles_c = (d + TL - 1) / TL, tiles_r = (n + TL - 1) / TL;
    const int64_t tiles = tiles_r * tiles_c;
    double sq = 0.0, xsq = 0.0;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const int64_t r0 = (tile / tiles_c) * TL, c0 = (tile % tiles_c) * TL;
        T acc[4][4];
        tile_product<T>(W, Tm, n, d, k, -1, r0, c0, Ws, Ts, acc);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int64_t gr = r0 + ty * 4 + i;
            if (gr < n) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int64_t gc = c0 + tx + 16 * j;
                    if (gc < d) {
                        const double m = (double)load_mask<T, MK>(M, gr * ldm + gc);
                        const double x = (double)ld_stream(X + gr * ldx + gc);
                        const double r = x - (double)acc[i][j];
                        sq += m * r * r;
                        xsq += m * x * x;
                    }
                }
            }
        }
    }
    sq = warp_sum(sq); xsq = warp_sum(xsq);
    if ((tid & 31) == 0) { red[0][tid >> 5] = sq; red[1][tid >> 5] = xsq; }
    __syncthreads();
    if (tid < 2) {
        double s = 0.0;
        for (int w = 0; w < TL_THREADS / WARP; ++w) s += red[tid][w];
        part[2 * (int64_t)blockIdx.x + tid] = s;
    }
}

__global__ void objective_finalize_kernel(const double* __restrict__ part, int blocks, double* __restrict__ out)
{
    if (threadIdx.x < 2) {
        double s = 0.0;
        for (int b = 0; b < blocks; ++b) s += part[2 * (int64_t)b + threadIdx.x];
        out[threadIdx.x] = (threadIdx.x == 0) ? 0.5 * s : s;
    }
}

template <typename T>
void launch_objective(const T* X, int64_t ldx, const void* M, int mk, int64_t ldm, const T* W,
                      const T* Tm, int64_t n, int64_t d, int k, double* part, int blocks, double* out,
                      cudaStream_t st)
{
    if (mk == MK_NONE) objective_kernel<T, MK_NONE><<<blocks, TL_THREADS, 0, st>>>(X, ldx, M, ldm, W, Tm, n, d, k, part);
    else if (mk == MK_REAL) objective_kernel<T, MK_REAL><<<blocks, TL_THREADS, 0, st>>>(X, ldx, M, ldm, W, Tm, n, d, k, part);
    else objective_kernel<T, MK_U8><<<blocks, TL_THREADS, 0, st>>>(X, ldx, M, ldm, W, Tm, n, d, k, part);
    objective_finalize_kernel<<<1, 32, 0, st>>>(part, blocks, out);
}

template <typename T>
__global__ void __launch_bounds__(256)
norms_kernel(const T* __restrict__ v, int64_t len, double* __restrict__ part)
{
    __shared__ double red[2][8];
    double s2 = 0.0, s1 = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (int64_t)gridDim.x * blockDim.x) {
        const double x = (double)v[i];
        s2 += x * x; s1 += fabs(x);
    }
    s2 = warp_sum(s2); s1 = warp_sum(s1);
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = s2; red[1][threadIdx.x >> 5] = s1; }
    __syncthreads();
    if (threadIdx.x < 2) {
        double s = 0.0;
        for (int w = 0; w < 8; ++w) s += red[threadIdx.x][w];
        part[2 * (int64_t)blockIdx.x + threadIdx.x] = s;
    }
}

// out[j] = sum_b part[2b + j], j = 0, 1 (blocks <= 256): one partial per thread, fixed shared-memory tree
__global__ void __launch_bounds__(256)
norms_finalize_kernel(const double* __restrict__ part, int blocks, double* __restrict__ out)
{
    __shared__ double red[2][256];
    const int b = threadIdx.x;
    red[0][b] = b < blocks ? part[2 * b] : 0.0;
    red[1][b] = b < blocks ? part[2 * b + 1] : 0.0;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (b < o) { red[0][b] += red[0][b + o]; red[1][b] += red[1][b + o]; }
        __syncthreads();
    }
    if (b < 2) out[b] = red[b][0];
}

template <typename T>
void launch_norms(const T* v, int64_t len, double* part, double* out, cudaStream_t st)
{
    int blocks = (int)((len + 256 * 8 - 1) / (256 * 8));
    if (blocks > 256) blocks = 256;
    if (blocks < 1) blocks = 1;
    norms_kernel<T><<<blocks, 256, 0, st>>>(v, len, part);
    norms_finalize_kernel<<<1, 256, 0, st>>>(part, blocks, out);
}

// ------------------------------------------------------------------------------------------------
// objective through the contraction (unmasked data):  ||X - W T||^2 = ||X||^2 - 2 <X T', W> + <W'W, T T'>
// The contraction X T' is the W half-step's own (still in its buffer after a block-order sweep), so an objective per
// sweep costs two Gram products and a dot product instead of a pass over X.  All sums in fp64.
// ------------------------------------------------------------------------------------------------
// out[0] = sum over rows r < rows, columns c < cols of A[r*lda + c]^2
template <typename T>
__global__ void __launch_bounds__(256)
sumsq_rows_kernel(const T* __restrict__ A, int64_t rows, int64_t cols, int64_t lda, double* __restrict__ part)
{
    __shared__ double red[8];
    double s = 0.0;
    const int64_t total = rows * cols;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / cols, c = i - r * cols;
        const double x = (double)ld_stream(A + r * lda + c);
        s += x * x;
    }
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += red[w];
        part[blockIdx.x] = t;
    }
}

// part[b] = partial of sum_e (sum_p C[p*stride + c(e)]) * W[e]; c(e) = e, or (width > 0) the entry (e / width, e % width)
// of C [., ldc]
template <typename T>
__global__ void __launch_bounds__(256)
dot_parts_kernel(const T* __restrict__ C, int parts, int64_t stride, const T* __restrict__ W, int64_t len,
                 double* __restrict__ part, int64_t ldc, int width)
{
    __shared__ double red[8];
    double s = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t ci = width > 0 ? (i / width) * ldc + i % width : i;
        double c = 0.0;
        for (int p = 0; p < parts; ++p) c += (double)C[(int64_t)p * stride + ci];
        s += c * (double)W[i];
    }
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += red[w];
        part[blockIdx.x] = t;
    }
}

// out[0] = sum_b part[b]: 256 threads, strided partial sums, then a fixed shared-memory tree (deterministic)
__global__ void __launch_bounds__(256)
sum_partials_kernel(const double* __restrict__ part, int blocks, double* __restrict__ out)
{
    __shared__ double red[256];
    double s = 0.0;
    for (int b = threadIdx.x; b < blocks; b += 256) s += part[b];
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[0] = red[0];
}

template <typename T>
void launch_sumsq_rows(const T* A, int64_t rows, int64_t cols, int64_t lda, double* part, double* out, int sm_count,
                       cudaStream_t st)
{
    int64_t blocks = (rows * cols + 256 * 16 - 1) / (256 * 16);
    if (blocks > 8 * sm_count) blocks = 8 * sm_count;
    if (blocks < 1) blocks = 1;
    sumsq_rows_kernel<T><<<(unsigned)blocks, 256, 0, st>>>(A, rows, cols, lda, part);
    sum_partials_kernel<<<1, 256, 0, st>>>(part, (int)blocks, out);
}

template <typename T>
void launch_dot_parts(const T* C, int parts, int64_t stride, const T* W, int64_t len, double* part, double* out,
                      int sm_count, cudaStream_t st, int64_t ldc, int width)
{
    int64_t blocks = (len + 256 * 8 - 1) / (256 * 8);
    if (blocks > 8 * sm_count) blocks = 8 * sm_count;
    if (blocks < 1) blocks = 1;
    dot_parts_kernel<T><<<(unsigned)blocks, 256, 0, st>>>(C, parts, stride, W, len, part, ldc, ldc > width ? width : 0);
    sum_partials_kernel<<<1, 256, 0, st>>>(part, (int)blocks, out);
}

// out[0] = 0.5 * (xsq - 2 cross + sum_ab G[a,b] H[a,b]),  out[1] = xsq
template <typename T>
__global__ void __launch_bounds__(256)
objective_identity_kernel(const T* __restrict__ G, const T* __restrict__ H, int kk, const double* __restrict__ xsq,
                          const double* __restrict__ cross, double* __restrict__ out)
{
    __shared__ double red[8];
    double s = 0.0;
    for (int e = threadIdx.x; e < kk; e += blockDim.x) s += (double)G[e] * (double)H[e];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double q = 0.0;
        for (int w = 0; w < 8; ++w) q += red[w];
        out[0] = 0.5 * (xsq[0] - 2.0 * cross[0] + q);
        out[1] = xsq[0];
    }
}

template <typename T>
void launch_objective_identity(const T* G, const T* H, int k, const double* xsq, const double* cross, double* out,
                               cudaStream_t st)
{
    objective_identity_kernel<T><<<1, 256, 0, st>>>(G, H, k * k, xsq, cross, out);
}

#define RRI_INST(T)                                                                                         \
    template void launch_sumsq_rows<T>(const T*, int64_t, int64_t, int64_t, double*, double*, int, cudaStream_t); \
    template void launch_dot_parts<T>(const T*, int, int64_t, const T*, int64_t, double*, double*, int, cudaStream_t, \
                                      int64_t, int);                                                        \
    template void launch_objective_identity<T>(const T*, const T*, int, const double*, const double*, double*, \
                                               cudaStream_t);                                               \
    template void launch_wrri_tstats<T>(const T*, int64_t, const void*, int, int64_t, const T*, const T*,   \
                                        int64_t, int64_t, int, int, T*, T*, const TilePlan&, cudaStream_t); \
    template void launch_wrri_wstats<T>(const T*, int64_t, const void*, int, int64_t, const T*, const T*,   \
                                        int64_t, int64_t, int, int, T*, T*, const TilePlan&, cudaStream_t); \
    template void launch_wrri_final<T>(const T*, const T*, int, int64_t, const SolveArgs&, T*, int64_t,     \
                                       T*, int64_t, int*, cudaStream_t);                                    \
    template void launch_vec_sum_flag<T>(const T*, int64_t, int64_t, double*, int, int, int*, cudaStream_t);\
    template void launch_rowsum_flag<T>(const T*, int, int64_t, int64_t, double*, int, int, int*, cudaStream_t, \
                                        const int*);                                                        \
    template void launch_vec_scale_to_sum<T>(T*, int64_t, int64_t, const double*, int, double, cudaStream_t);\
    template void launch_objective<T>(const T*, int64_t, const void*, int, int64_t, const T*, const T*,     \
                                      int64_t, int64_t, int, double*, int, double*, cudaStream_t);          \
    template void launch_norms<T>(const T*, int64_t, double*, double*, cudaStream_t);
RRI_INST(float)
RRI_INST(double)

}  // namespace rri
