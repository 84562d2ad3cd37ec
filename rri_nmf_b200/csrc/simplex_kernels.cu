// simplex_kernels.cu -- Euclidean projection of matrix rows onto the simplex {x >= 0, sum x = s}, and the block-order
// T half-step with that projection after every topic (project_T_each_iter).
//
// The reference (matrixops.py:5-69, Duchi et al.) sorts the vector and finds
//     rho = max{ j : u_j * j > cumsum(u)_j - s },  theta = (cumsum(u)_rho - s) / rho,  w = max(v - theta, 0).
// The same theta is the fixed point of Michelot's iteration
//     theta <- (sum_{v_i > theta} v_i - s) / |{v_i > theta}|,   starting from the full set,
// which needs only reductions (no sort) and reaches the identical active set in a few rounds.
// Sums are accumulated in double for both element types.
#include <cooperative_groups.h>
#include <math.h>

#include "../../include/rri_b200.h"
#include "common.cuh"
#include "kernels.h"

namespace cg = cooperative_groups;

namespace rri {

// Michelot's iteration over one vector by one block, then v <- max(v - theta, 0).  tol >= 0: leave v as it is when
// |sum v - s| <= tol (the sum is the first round's total) -- the re-projection test of nmf.py:759-761.
template <typename T>
__device__ void block_project_simplex(T* __restrict__ v, int64_t cols, double s, double tol)
{
    __shared__ double rs[32];
    __shared__ double rc[32];
    __shared__ double bc[2];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
    double theta = -1.0e300;        // "everything active" on the first round
    double prev_cnt = -1.0;
    for (int iter = 0; iter < 10000; ++iter) {
        double sum = 0.0, cnt = 0.0;
        for (int64_t i = tid; i < cols; i += blockDim.x) {
            const double x = (double)v[i];
            if (x > theta) { sum += x; cnt += 1.0; }
        }
        sum = warp_sum(sum); cnt = warp_sum(cnt);
        if (lane == 0) { rs[warp] = sum; rc[warp] = cnt; }
        __syncthreads();
        if (tid == 0) {
            double a = 0.0, b = 0.0;
            for (int w = 0; w < nw; ++w) { a += rs[w]; b += rc[w]; }
            bc[0] = a; bc[1] = b;
        }
        __syncthreads();
        const double tot = bc[0], c = bc[1];
        __syncthreads();
        if (iter == 0 && tol >= 0.0 && fabs(tot - s) <= tol) return;
        if (c == prev_cnt || c == 0.0) break;       // active set unchanged: theta is final
        prev_cnt = c;
        theta = (tot - s) / c;
    }
    for (int64_t i = tid; i < cols; i += blockDim.x) {
        const double x = (double)v[i] - theta;
        v[i] = (T)(x > 0.0 ? x : 0.0);
    }
}

template <typename T>
__global__ void project_rows_simplex_kernel(T* __restrict__ A, int64_t rows, int64_t cols, double s)
{
    for (int64_t r = blockIdx.x; r < rows; r += gridDim.x) {
        block_project_simplex<T>(A + r * cols, cols, s, -1.0);
        __syncthreads();
    }
}

template <typename T>
void launch_project_rows_simplex(T* A, int64_t rows, int64_t cols, double s, cudaStream_t st)
{
    int threads = cols <= 64 ? 32 : (cols <= 4096 ? 256 : 1024);
    int64_t blocks = rows < 65535LL * 16 ? rows : 65535LL * 16;
    project_rows_simplex_kernel<T><<<(unsigned)blocks, threads, 0, st>>>(A, rows, cols, s);
}

template void launch_project_rows_simplex<float>(float*, int64_t, int64_t, double, cudaStream_t);
template void launch_project_rows_simplex<double>(double*, int64_t, int64_t, double, cudaStream_t);

__global__ void flag_from_sums_kernel(const double* __restrict__ sums, int off, int k, int zero_flag,
                                      int* __restrict__ flags)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < k) {
        const double v = sums[off + t];
        if (!(v > 1e-10)) atomicOr(flags, zero_flag);
        if (!isfinite(v)) atomicOr(flags, 8);
    }
}

void launch_flag_from_sums(const double* sums, int off, int k, int zero_flag, int* flags, cudaStream_t st)
{
    flag_from_sums_kernel<<<(k + 127) / 128, 128, 0, st>>>(sums, off, k, zero_flag, flags);
}

// ------------------------------------------------------------------------------------------------
// Block-order T half-step with project_T_each_iter (oracle/rri_oracle.py sweep(order='hals'), nmf.py:420-447 +
// :759-761): for every topic t in turn, over all d columns of T,
//     numer = C[:,t] - sum_{j != t} G[t,j] T[j,:] - reg_l1     (rows j < t already updated)
//     c = G[t,t] + reg_l2
//     c > 0 : x = max(numer, 0) / (c + eps), projected onto the simplex, projected again when |sum - s| > 1e-15
//     c <= 0: s == 1: one-hot at the first maximum of numer; otherwise RRI_FLAG_NOT_IMPLEMENTED (optimization.py:60-72)
// The projection threshold couples all d columns: it is a grid-wide quantity, k times per half-step.
// ------------------------------------------------------------------------------------------------
constexpr int SX_THREADS = 128;         // rows of T' (columns of T) per block of the fused kernel

int simplex_T_slots(int64_t d) { return (int)(2 * 3 * ((d + SX_THREADS - 1) / SX_THREADS)); }

// Grid-wide sums of three doubles: per block a shuffle tree and the warps in order, one slot per block, a grid
// barrier, then every block adds all slots in the same fixed order -- every block holds the same bits.  Two slot
// buffers alternate: a block can only overwrite buffer b again after the next barrier, which no block passes before it
// has finished reading b.
__device__ __forceinline__ void grid_sum3(cg::grid_group& grid, double a, double b, double c, double* __restrict__ slots,
                                          int& parity, double out[3])
{
    constexpr int NW = SX_THREADS / 32;
    __shared__ double ws[3][NW];
    __shared__ double res[3];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nb = gridDim.x;
    a = warp_sum(a); b = warp_sum(b); c = warp_sum(c);
    if (lane == 0) { ws[0][warp] = a; ws[1][warp] = b; ws[2][warp] = c; }
    __syncthreads();
    double* sl = slots + (size_t)parity * 3 * nb;
    parity ^= 1;
    if (threadIdx.x < 3) {
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < NW; ++w) v += ws[threadIdx.x][w];
        sl[(size_t)threadIdx.x * nb + blockIdx.x] = v;
        __threadfence();
    }
    grid.sync();
    if (warp == 0) {
        double v0 = 0.0, v1 = 0.0, v2 = 0.0;
        for (int q = lane; q < nb; q += 32) {
            v0 += __ldcg(sl + q); v1 += __ldcg(sl + nb + q); v2 += __ldcg(sl + 2 * nb + q);
        }
        v0 = warp_sum(v0); v1 = warp_sum(v1); v2 = warp_sum(v2);
        if (lane == 0) { res[0] = v0; res[1] = v1; res[2] = v2; }
    }
    __syncthreads();
    out[0] = res[0]; out[1] = res[1]; out[2] = res[2];
}

__device__ __forceinline__ bool argmax_before(double v1, double i1, double v2, double i2)
{
    return v1 > v2 || (v1 == v2 && i1 < i2);
}

// first index of the grid-wide maximum (order independent: max with the smallest index wins ties)
__device__ __forceinline__ double grid_argmax(cg::grid_group& grid, double v, double idx, double* __restrict__ slots,
                                              int& parity)
{
    constexpr int NW = SX_THREADS / 32;
    __shared__ double wv[NW], wi[NW];
    __shared__ double res;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nb = gridDim.x;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double v2 = __shfl_xor_sync(0xffffffffu, v, o), i2 = __shfl_xor_sync(0xffffffffu, idx, o);
        if (argmax_before(v2, i2, v, idx)) { v = v2; idx = i2; }
    }
    if (lane == 0) { wv[warp] = v; wi[warp] = idx; }
    __syncthreads();
    double* sl = slots + (size_t)parity * 3 * nb;
    parity ^= 1;
    if (threadIdx.x == 0) {
        double bv = wv[0], bi = wi[0];
        for (int w = 1; w < NW; ++w)
            if (argmax_before(wv[w], wi[w], bv, bi)) { bv = wv[w]; bi = wi[w]; }
        sl[blockIdx.x] = bv; sl[nb + blockIdx.x] = bi;
        __threadfence();
    }
    grid.sync();
    if (warp == 0) {
        double bv = -INFINITY, bi = 1e300;
        for (int q = lane; q < nb; q += 32) {
            const double v2 = __ldcg(sl + q), i2 = __ldcg(sl + nb + q);
            if (argmax_before(v2, i2, bv, bi)) { bv = v2; bi = i2; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double v2 = __shfl_xor_sync(0xffffffffu, bv, o), i2 = __shfl_xor_sync(0xffffffffu, bi, o);
            if (argmax_before(v2, i2, bv, bi)) { bv = v2; bi = i2; }
        }
        if (lane == 0) res = bi;
    }
    __syncthreads();
    return res;
}

// Michelot's iteration over the grid (one entry x per thread, `valid` = a real column), from theta with the previous
// round's active count prev_cnt.  psum: on return, the sum of the projected values (T)(x - theta) over the final active
// set, taken in the round that found the set unchanged -- the sum of what will be stored.
template <typename T>
__device__ __forceinline__ double grid_michelot(cg::grid_group& grid, double x, bool valid, double s, double theta,
                                                double prev_cnt, double* __restrict__ slots, int& parity, double& psum)
{
    for (int iter = 0; iter < 10000; ++iter) {
        const bool act = valid && x > theta;
        double r[3];
        grid_sum3(grid, act ? x : 0.0, act ? 1.0 : 0.0, act ? (double)(T)(x - theta) : 0.0, slots, parity, r);
        psum = r[2];
        if (r[1] == prev_cnt || r[1] == 0.0) break;
        prev_cnt = r[1];
        theta = (r[0] - s) / r[1];
    }
    return theta;
}

// Persistent, cooperatively launched: one thread per row i of T' (column i of T) with its k entries in registers,
// the Gram matrix in shared memory, the contraction read in `parts` slices in order.  Writes T' (in place) and
// Tout[k, ldo] (the caller's T, or the replica of the peer exchange).
// (a register cap, not launch bounds: with 128 threads ptxas spills the fp64 KM = 64 variant under its default choice)
template <typename T, int KM>
__global__ void __maxnreg__(255)
simplex_T_fused_kernel(T* __restrict__ Tt, int64_t d, int k, const T* __restrict__ C, int parts, int64_t pstride,
                       const T* __restrict__ G, T reg_l1, T reg_l2, T eps, double s, T* __restrict__ Tout, int64_t ldo,
                       double* __restrict__ slots, int* __restrict__ flags)
{
    using V = typename Vec<T>::type;
    constexpr int VN = Vec<T>::N;
    cg::grid_group grid = cg::this_grid();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T* Ss = reinterpret_cast<T*>(smem_raw);                  // [KM][KM], zero padded
    for (int e = threadIdx.x; e < KM * KM; e += SX_THREADS) {
        const int a = e / KM, b = e % KM;
        Ss[e] = (a < k && b < k) ? G[a * k + b] : T(0);
    }
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * SX_THREADS + threadIdx.x;
    const bool valid = i < d;
    T f[KM];
    {
        const V* frow = reinterpret_cast<const V*>(Tt + (valid ? i : 0) * k);      // k % VN == 0 (launcher)
#pragma unroll
        for (int jv = 0; jv < KM / VN; ++jv) {
            T fv[VN];
#pragma unroll
            for (int v = 0; v < VN; ++v) fv[v] = T(0);
            if (valid && VN * jv < k) unpack(frow[jv], fv);
#pragma unroll
            for (int v = 0; v < VN; ++v) f[VN * jv + v] = fv[v];
        }
    }
    int parity = 0;
    bool nonfinite = false;
#pragma unroll 1
    for (int t = 0; t < k; ++t) {
        const V* srow = reinterpret_cast<const V*>(Ss + t * KM);
        T acc[4] = {T(0), T(0), T(0), T(0)};
#pragma unroll
        for (int jv = 0; jv < KM / VN; ++jv) {
            T sv[VN];
            unpack(srow[jv], sv);
#pragma unroll
            for (int v = 0; v < VN; ++v) {
                const int j = jv * VN + v;
                acc[j & 3] = fma(j == t ? T(0) : f[j], sv[v], acc[j & 3]);
            }
        }
        T cv = T(0);
        if (valid)
            for (int p = 0; p < parts; ++p) cv += C[(int64_t)p * pstride + i * k + t];
        const T numer = cv - ((acc[0] + acc[1]) + (acc[2] + acc[3])) - reg_l1;
        if (valid && !isfinite(numer)) nonfinite = true;
        const T c = Ss[t * KM + t] + reg_l2;               // the same in every thread: the branches below are uniform
        T y = T(0);
        if (c > T(0)) {
            const T x = valid ? tmax(numer, T(0)) / (c + eps) : T(0);
            double psum = 0.0;
            const double th = grid_michelot<T>(grid, (double)x, valid, s, -1.0e300, -1.0, slots, parity, psum);
            y = (valid && (double)x > th) ? (T)((double)x - th) : T(0);
            if (fabs(psum - s) > 1e-15) {
                // nmf.py:759-761.  Round 1 of Michelot over y is known: every entry is active, the total is psum.
                const double th2 = grid_michelot<T>(grid, (double)y, valid, s, (psum - s) / (double)d, (double)d, slots,
                                                    parity, psum);
                y = (valid && (double)y > th2) ? (T)((double)y - th2) : T(0);
            }
        } else if (s == 1.0) {
            const double im = grid_argmax(grid, (valid && !isnan(numer)) ? (double)numer : -INFINITY,
                                          valid ? (double)i : 1e300, slots, parity);
            y = (valid && (double)i == im) ? T(1) : T(0);
        } else if (blockIdx.x == 0 && threadIdx.x == 0) {
            atomicOr(flags, RRI_FLAG_NOT_IMPLEMENTED);
        }
        if (valid) Tout[(int64_t)t * ldo + i] = y;
#pragma unroll
        for (int j = 0; j < KM; ++j) f[j] = (j == t) ? y : f[j];
    }
    if (valid) {
        V* fout = reinterpret_cast<V*>(Tt + i * k);
#pragma unroll
        for (int jv = 0; jv < KM / VN; ++jv)
            if (VN * jv < k) {
                V o;
                T* op = reinterpret_cast<T*>(&o);
#pragma unroll
                for (int v = 0; v < VN; ++v) op[v] = f[VN * jv + v];
                fout[jv] = o;
            }
    }
    if (nonfinite) atomicOr(flags, 8);
}

// Chain, step 1 of topic t: the numerator / scalar solve of every column (thread per column), into row t of Tk.
// c <= 0 with s == 1 leaves the numerator there for step 2.
template <typename T>
__global__ void __launch_bounds__(256)
simplex_topic_numer_kernel(T* __restrict__ Tk, int64_t ldt, int64_t d, int k, int t, const T* __restrict__ C, int parts,
                           int64_t pstride, const T* __restrict__ G, T reg_l1, T reg_l2, T eps, double s,
                           int* __restrict__ flags)
{
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= d) return;
    T acc[4] = {T(0), T(0), T(0), T(0)};
    for (int j0 = 0; j0 < k; j0 += 4) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int j = j0 + u;
            if (j < k) acc[u] = fma(j == t ? T(0) : Tk[(int64_t)j * ldt + i], G[t * k + j], acc[u]);
        }
    }
    T cv = T(0);
    for (int p = 0; p < parts; ++p) cv += C[(int64_t)p * pstride + i * k + t];
    const T numer = cv - ((acc[0] + acc[1]) + (acc[2] + acc[3])) - reg_l1;
    if (!isfinite(numer)) atomicOr(flags, 8);
    const T c = G[t * k + t] + reg_l2;
    T x = T(0);
    if (c > T(0)) x = tmax(numer, T(0)) / (c + eps);
    else if (s == 1.0) x = numer;
    else if (i == 0) atomicOr(flags, RRI_FLAG_NOT_IMPLEMENTED);
    Tk[(int64_t)t * ldt + i] = x;
}

// Chain, step 2 of topic t (one block): projection + re-projection test, or the one-hot of c <= 0, s == 1.
template <typename T>
__global__ void __launch_bounds__(1024)
simplex_topic_finish_kernel(T* __restrict__ row, int64_t d, double s, const T* __restrict__ Gtt, T reg_l2)
{
    const T c = *Gtt + reg_l2;
    if (c > T(0)) {
        block_project_simplex<T>(row, d, s, -1.0);
        __syncthreads();
        block_project_simplex<T>(row, d, s, 1e-15);       // nmf.py:759-761
        return;
    }
    if (s != 1.0) return;
    __shared__ double wv[32], wi[32];
    __shared__ double best;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
    double bv = -INFINITY, bi = 1e300;
    for (int64_t i = tid; i < d; i += blockDim.x) {
        const double v = (double)row[i];
        if (!isnan(v) && argmax_before(v, (double)i, bv, bi)) { bv = v; bi = (double)i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double v2 = __shfl_xor_sync(0xffffffffu, bv, o), i2 = __shfl_xor_sync(0xffffffffu, bi, o);
        if (argmax_before(v2, i2, bv, bi)) { bv = v2; bi = i2; }
    }
    if (lane == 0) { wv[warp] = bv; wi[warp] = bi; }
    __syncthreads();
    if (tid == 0) {
        double v = wv[0], ix = wi[0];
        for (int w = 1; w < nw; ++w)
            if (argmax_before(wv[w], wi[w], v, ix)) { v = wv[w]; ix = wi[w]; }
        best = ix;
    }
    __syncthreads();
    for (int64_t i = tid; i < d; i += blockDim.x) row[i] = ((double)i == best) ? T(1) : T(0);
}

template <typename T, int KM>
static int launch_fused_km(T* Tt, int64_t d, int k, const T* C, int parts, int64_t pstride, const T* G, const SolveArgs& a,
                           double s, T* Tout, int64_t ldo, double* slots, int* flags, int sm_count, cudaStream_t st)
{
    auto kern = simplex_T_fused_kernel<T, KM>;
    const size_t smem = sizeof(T) * KM * KM;
    if (smem > 48 * 1024 && cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
        return -(int)cudaGetLastError();
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, SX_THREADS, smem) != cudaSuccess)
        return -(int)cudaGetLastError();
    const int64_t blocks = (d + SX_THREADS - 1) / SX_THREADS;
    if (blocks > (int64_t)per_sm * sm_count) return 0;        // the grid cannot be co-resident: not fused
    T rl1 = (T)a.reg_l1, rl2 = (T)a.reg_l2, eps = (T)a.eps;
    void* args[] = {&Tt, &d, &k, &C, &parts, &pstride, &G, &rl1, &rl2, &eps, &s, &Tout, &ldo, &slots, &flags};
    const cudaError_t e = cudaLaunchCooperativeKernel((const void*)kern, dim3((unsigned)blocks), dim3(SX_THREADS), args, smem, st);
    return e == cudaSuccess ? 1 : -(int)e;
}

template <typename T>
static int fused_dispatch(T* Tt, int64_t d, int k, const T* C, int parts, int64_t pstride, const T* G, const SolveArgs& a,
                          double s, T* Tout, int64_t ldo, double* slots, int* flags, int sm_count, cudaStream_t st)
{
    if (k % Vec<T>::N != 0) return 0;
#define RRI_SX(KM) return launch_fused_km<T, KM>(Tt, d, k, C, parts, pstride, G, a, s, Tout, ldo, slots, flags, sm_count, st)
    if (k <= 16) RRI_SX(16);
    if (k <= 32) RRI_SX(32);
    if (k <= 64) RRI_SX(64);
    if constexpr (sizeof(T) == 4) { if (k <= 128) RRI_SX(128); }
#undef RRI_SX
    return 0;
}

template <typename T>
int launch_simplex_T_update(T* Tt, int64_t d, int k, const T* C, int parts, int64_t pstride, const T* G, const SolveArgs& a,
                            double s, T* Tout, int64_t ldo, double* slots, int* flags, int sm_count, bool allow_fused,
                            int* launches, cudaStream_t st)
{
    if (allow_fused) {
        const int r = fused_dispatch<T>(Tt, d, k, C, parts, pstride, G, a, s, Tout, ldo, slots, flags, sm_count, st);
        if (r < 0) return -r;
        if (r > 0) { *launches = 1; return 0; }
    }
    const unsigned nb = (unsigned)((d + 255) / 256);
    const int ft = d <= 4096 ? 256 : 1024;
    for (int t = 0; t < k; ++t) {
        simplex_topic_numer_kernel<T><<<nb, 256, 0, st>>>(Tout, ldo, d, k, t, C, parts, pstride, G, (T)a.reg_l1,
                                                          (T)a.reg_l2, (T)a.eps, s, flags);
        simplex_topic_finish_kernel<T><<<1, ft, 0, st>>>(Tout + (int64_t)t * ldo, d, s, G + (int64_t)t * k + t, (T)a.reg_l2);
    }
    launch_transpose<T>(Tout, k, d, ldo, Tt, k, st);
    *launches = 2 * k + 1;
    return (int)cudaGetLastError();
}

#define RRI_SX_INST(T)                                                                                                   \
    template int launch_simplex_T_update<T>(T*, int64_t, int, const T*, int, int64_t, const T*, const SolveArgs&, double, \
                                            T*, int64_t, double*, int*, int, bool, int*, cudaStream_t);
RRI_SX_INST(float)
RRI_SX_INST(double)
#undef RRI_SX_INST

}  // namespace rri
