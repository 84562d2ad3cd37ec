// sparse_kernels.cu -- observed-entries WRRI (SURVEY.md §8 row f4): the masked half-steps of nmf.py:687-701 and
// :735-746 for data given as (i, j, y) triples (sklearn_interface.py:78-83, :97-102) that are never densified.
//
// The reference recomputes Rt = M o (X - W_(t->0) T) with a dense n x k x d product for every topic.  Here the
// residual E = X - W T lives only at the observed entries, in two orientations that hold bit-identical values:
//   CSR (segments = rows)    -- read by the W-steps,
//   CSC (segments = columns) -- read by the T-steps.
// A half-step of topic t is ONE streaming pass over one orientation: 4 B index + 4 B residual read (+ 4 B written
// back) per observed entry and one 16-byte gather of the other factor's packed values.  While it streams, the pass
// also applies the rank-one change  w_old t_old' - w_new t_new'  left behind by the previous topic ("pending"
// update), with the same rounding sequence in both orientations, so the two copies never diverge.  The residual is
// rebuilt from X, W, T at the start of every sweep (so N sweeps == N x 1 sweep bit for bit, and rounding drift
// cannot accumulate).  No atomics: one warp (or one block) owns a whole segment.
#include <cub/device/device_radix_sort.cuh>

#include "common.cuh"
#include "kernels.h"

namespace rri {

template <typename T> struct alignas(16) Quad { T a, b, c, d; };

RRI_DEVINL float  mul_rn(float a, float b)   { return __fmul_rn(a, b); }
RRI_DEVINL double mul_rn(double a, double b) { return __dmul_rn(a, b); }
RRI_DEVINL float  add_rn(float a, float b)   { return __fadd_rn(a, b); }
RRI_DEVINL double add_rn(double a, double b) { return __dadd_rn(a, b); }
RRI_DEVINL float  sub_rn(float a, float b)   { return __fsub_rn(a, b); }
RRI_DEVINL double sub_rn(double a, double b) { return __dsub_rn(a, b); }

static int cap_blocks(int64_t want, int sm_count, int per_sm)
{
    int64_t cap = (int64_t)sm_count * per_sm;
    if (want > cap) want = cap;
    return (int)(want < 1 ? 1 : want);
}

// ------------------------------------------------------------------------------------------------
// building the column orientation from the caller's CSR (once per bind)
// ------------------------------------------------------------------------------------------------
__global__ void sp_check_kernel(const int64_t* __restrict__ rowptr, int64_t n, const int32_t* __restrict__ col,
                                int64_t nnz, int64_t d, int* __restrict__ err)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t r = i; r < n; r += stride) {
        const int64_t b = rowptr[r], e = rowptr[r + 1];
        if (b > e || b < 0 || e > nnz) { atomicOr(err, 1); continue; }
        for (int64_t p = b + 1; p < e; ++p)
            if (col[p] <= col[p - 1]) { atomicOr(err, 4); break; }       // ascending, no duplicates
    }
    for (int64_t p = i; p < nnz; p += stride)
        if (col[p] < 0 || (int64_t)col[p] >= d) atomicOr(err, 2);
    if (i == 0 && (rowptr[0] != 0 || rowptr[n] != nnz)) atomicOr(err, 1);
}

__global__ void sp_expand_rows_kernel(const int64_t* __restrict__ rowptr, int64_t n, int32_t* __restrict__ rowidx,
                                      uint32_t* __restrict__ iota)
{
    const int lane = threadIdx.x & 31;
    const int64_t w0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = w0; r < n; r += nw) {
        const int64_t b = rowptr[r], e = rowptr[r + 1];
        for (int64_t p = b + lane; p < e; p += 32) { rowidx[p] = (int32_t)r; iota[p] = (uint32_t)p; }
    }
}

template <typename T>
__global__ void sp_permute_kernel(const uint32_t* __restrict__ perm, const int32_t* __restrict__ rowidx,
                                  const T* __restrict__ x, const T* __restrict__ w, int64_t nnz,
                                  int32_t* __restrict__ csc_row, T* __restrict__ x_csc, T* __restrict__ w_csc)
{
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < nnz; p += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t q = perm[p];
        csc_row[p] = rowidx[q];
        x_csc[p] = x[q];
        if (w) w_csc[p] = w[q];
    }
}

// colptr[j] = first position whose (sorted) column key is >= j
__global__ void sp_colptr_kernel(const int32_t* __restrict__ keys, int64_t nnz, int64_t d, int64_t* __restrict__ colptr)
{
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j <= d; j += (int64_t)gridDim.x * blockDim.x) {
        int64_t lo = 0, hi = nnz;
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if ((int64_t)keys[mid] < j) lo = mid + 1; else hi = mid;
        }
        colptr[j] = lo;
    }
}

template <typename T>
int sp_build_csc(const int64_t* rowptr, const int32_t* col, const T* x, const T* w, int64_t n, int64_t d,
                 int64_t nnz, int64_t* colptr, int32_t* csc_row, T* x_csc, T* w_csc, uint32_t* perm, int sm_count,
                 int* err_dev, cudaStream_t st)
{
    cudaError_t e;
    const int nb = cap_blocks((nnz + 255) / 256 + (n + 7) / 8, sm_count, 8);
    sp_check_kernel<<<nb, 256, 0, st>>>(rowptr, n, col, nnz, d, err_dev);
    int err_host = 0;
    if ((e = cudaMemcpyAsync(&err_host, err_dev, sizeof(int), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return (int)e;
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return (int)e;
    if (err_host) return -err_host;                       // malformed CSR: nothing below may index with it
    if (nnz == 0) {
        sp_colptr_kernel<<<cap_blocks((d + 256) / 256, sm_count, 8), 256, 0, st>>>(nullptr, 0, d, colptr);
        return (int)cudaGetLastError();
    }
    int32_t *rowidx = nullptr, *keys_sorted = nullptr;
    uint32_t* iota = nullptr;
    void* tmp = nullptr;
    size_t tmp_bytes = 0;
    int end_bit = 1;
    while (end_bit < 31 && ((int64_t)1 << end_bit) < d) ++end_bit;
    int rc = 0;
    do {
        if ((e = cudaMalloc(&rowidx, sizeof(int32_t) * nnz)) != cudaSuccess) { rc = (int)e; break; }
        if ((e = cudaMalloc(&keys_sorted, sizeof(int32_t) * nnz)) != cudaSuccess) { rc = (int)e; break; }
        if ((e = cudaMalloc(&iota, sizeof(uint32_t) * nnz)) != cudaSuccess) { rc = (int)e; break; }
        sp_expand_rows_kernel<<<cap_blocks((n + 7) / 8, sm_count, 8), 256, 0, st>>>(rowptr, n, rowidx, iota);
        // stable LSD radix sort of (column, position): rows stay ascending inside every column
        if ((e = cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, col, keys_sorted, iota, perm, (int)nnz, 0, end_bit,
                                                 st)) != cudaSuccess) { rc = (int)e; break; }
        if ((e = cudaMalloc(&tmp, tmp_bytes ? tmp_bytes : 16)) != cudaSuccess) { rc = (int)e; break; }
        if ((e = cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, col, keys_sorted, iota, perm, (int)nnz, 0, end_bit,
                                                 st)) != cudaSuccess) { rc = (int)e; break; }
        sp_permute_kernel<T><<<cap_blocks((nnz + 255) / 256, sm_count, 8), 256, 0, st>>>(perm, rowidx, x, w, nnz, csc_row,
                                                                                         x_csc, w_csc);
        sp_colptr_kernel<<<cap_blocks((d + 256) / 256, sm_count, 8), 256, 0, st>>>(keys_sorted, nnz, d, colptr);
        if ((e = cudaGetLastError()) != cudaSuccess) { rc = (int)e; break; }
        if ((e = cudaStreamSynchronize(st)) != cudaSuccess) { rc = (int)e; break; }
    } while (0);
    cudaFree(rowidx); cudaFree(keys_sorted); cudaFree(iota); cudaFree(tmp);
    return rc;
}

// ------------------------------------------------------------------------------------------------
// residual from scratch:  E[p] = x[p] - sum_l A[seg,l] * B[idx[p],l]  in the row orientation (A = W, B = T'); the
// column copy is its permutation (sp_gather_kernel)
// Shifted mode (SH == 1): the stored value is S[p] = (m[p] - w0) E[p] + w0 x[p]  (m = 1 without entry weights).
// Rank-one mode (SH == 2, unstored weights u = w0 (a_i b_j), DESIGN.md §1 row f8): wgt holds mt = m - u per entry
// (sp_mtilde_kernel) and S[p] = mt E[p] + u x[p]; ab = a_i b_j from the segment's and the gathered entry's vector.
// ------------------------------------------------------------------------------------------------
template <typename T, int SH>
RRI_DEVINL T sp_stored(T e, T x, const T* __restrict__ wgt, int64_t p, T w0, T ab)
{
    if constexpr (SH == 1) return fma(sub_rn(wgt ? wgt[p] : T(1), w0), e, mul_rn(w0, x));
    if constexpr (SH == 2) return fma(wgt[p], e, mul_rn(mul_rn(w0, ab), x));
    return e;
}

// a_i b_j of entry p of segment s (a missing vector is all ones); only the rank-one mode reads the vectors
template <typename T, int SH>
RRI_DEVINL T sp_ab(const T* __restrict__ vseg, const T* __restrict__ vidx, int64_t s, int32_t j)
{
    if constexpr (SH == 2) return mul_rn(vseg ? vseg[s] : T(1), vidx ? vidx[j] : T(1));
    return T(1);
}

// Row-orientation residual with the segment's own factor row staged in shared memory and the gathered rows read
// with 16-byte loads: B has a padded row stride ldb (multiple of 16 bytes, pad columns zero), so an entry costs
// ceil(k/V) vector loads -- half the L1 tag look-ups of the 8-byte version at k = 50 -- and the own row costs none.
template <typename T, int G, int SH>
__global__ void __launch_bounds__(256)
sp_residual_rows_kernel(const int64_t* __restrict__ ptr, const int32_t* __restrict__ idx, const T* __restrict__ x,
                        const T* __restrict__ A, int64_t lda, const T* __restrict__ B, int ldb, int k,
                        T* __restrict__ E, int64_t nseg, const T* __restrict__ wgt, T w0, const T* __restrict__ vseg,
                        const T* __restrict__ vidx)
{
    using V = typename Vec<T>::type;
    constexpr int VN = Vec<T>::N;
    constexpr int GPB = 256 / G;
    __shared__ __align__(16) T a_s[GPB][256 + VN];
    const int lane = threadIdx.x % G, g = threadIdx.x / G;
    const int nv = (k + VN - 1) / VN;
    for (int64_t s = (int64_t)blockIdx.x * GPB + g; s < nseg; s += (int64_t)gridDim.x * GPB) {
        if (G == 256) __syncthreads(); else __syncwarp();              // the previous row has been consumed
        for (int l = lane; l < nv * VN; l += G) a_s[g][l] = l < k ? A[s * lda + l] : T(0);
        if (G == 256) __syncthreads(); else __syncwarp();
        const int64_t b = ptr[s], e = ptr[s + 1];
        const V* __restrict__ av = reinterpret_cast<const V*>(a_s[g]);
        for (int64_t p = b + lane; p < e; p += G) {
            const V* __restrict__ bv = reinterpret_cast<const V*>(B + (int64_t)idx[p] * ldb);
            T acc = x[p];
#pragma unroll 4
            for (int l = 0; l < nv; ++l) {
                T a[VN], c[VN];
                unpack(av[l], a);
                unpack(bv[l], c);
#pragma unroll
                for (int v = 0; v < VN; ++v) acc = fma(-a[v], c[v], acc);
            }
            E[p] = sp_stored<T, SH>(acc, x[p], wgt, p, w0, sp_ab<T, SH>(vseg, vidx, s, idx[p]));
        }
    }
}

template <typename T, int SH>
static void residual_rows_dispatch(const SpSide& s, const T* A, int64_t lda, const T* B, int ldb, int k, T w0, const T* vseg,
                                   const T* vidx, int sm_count, cudaStream_t st)
{
    const T* w = (const T*)s.wgt;
    if (s.group == 256)
        sp_residual_rows_kernel<T, 256, SH><<<cap_blocks(s.nseg, sm_count, 8), 256, 0, st>>>(s.ptr, s.idx, (const T*)s.x, A, lda, B,
                                                                                             ldb, k, (T*)s.E, s.nseg, w, w0,
                                                                                             vseg, vidx);
    else
        sp_residual_rows_kernel<T, 32, SH><<<cap_blocks((s.nseg + 7) / 8, sm_count, 8), 256, 0, st>>>(s.ptr, s.idx, (const T*)s.x, A,
                                                                                                      lda, B, ldb, k, (T*)s.E, s.nseg,
                                                                                                      w, w0, vseg, vidx);
}

// (rank-one mode when a vector is given: s.wgt is then the mt copy of this orientation)
template <typename T>
void launch_sp_residual_rows(const SpSide& s, const T* A, int64_t lda, const T* B, int ldb, int k, double w0, int sm_count,
                             cudaStream_t st, const T* vseg, const T* vidx)
{
    if (w0 > 0.0 && (vseg || vidx)) residual_rows_dispatch<T, 2>(s, A, lda, B, ldb, k, (T)w0, vseg, vidx, sm_count, st);
    else if (w0 > 0.0) residual_rows_dispatch<T, 1>(s, A, lda, B, ldb, k, (T)w0, nullptr, nullptr, sm_count, st);
    else residual_rows_dispatch<T, 0>(s, A, lda, B, ldb, k, T(0), nullptr, nullptr, sm_count, st);
}

// dst[p] = src[perm[p]]: the column copy of the residual taken from the row copy (bit-identical by construction)
template <typename T>
__global__ void sp_gather_kernel(const uint32_t* __restrict__ perm, const T* __restrict__ src, T* __restrict__ dst, int64_t nnz)
{
    constexpr int U = 4;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; p + (U - 1) * stride < nnz; p += U * stride) {
        uint32_t q[U]; T v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) q[u] = perm[p + u * stride];
#pragma unroll
        for (int u = 0; u < U; ++u) v[u] = src[q[u]];
#pragma unroll
        for (int u = 0; u < U; ++u) dst[p + u * stride] = v[u];
    }
    for (; p < nnz; p += stride) dst[p] = src[perm[p]];
}

template <typename T>
void launch_sp_gather(const uint32_t* perm, const T* src, T* dst, int64_t nnz, int sm_count, cudaStream_t st)
{
    sp_gather_kernel<T><<<cap_blocks((nnz + 1023) / 1024, sm_count, 8), 256, 0, st>>>(perm, src, dst, nnz);
}

// ------------------------------------------------------------------------------------------------
// the packed gather record of the "other" factor:  {pending old, pending new, current old, current new}
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void sp_pack_kernel(const T* __restrict__ po, const T* __restrict__ pn, const T* __restrict__ vold,
                               const T* __restrict__ vnew, Quad<T>* __restrict__ out, int64_t len)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= len) return;
    Quad<T> q;
    q.a = po ? po[i] : T(0);
    q.b = pn ? pn[i] : T(0);
    q.c = vold[i];
    q.d = vnew[i];
    out[i] = q;
}

template <typename T>
void launch_sp_pack(const T* po, const T* pn, const T* vold, const T* vnew, void* quad, int64_t len, cudaStream_t st)
{
    sp_pack_kernel<T><<<(unsigned)((len + 255) / 256), 256, 0, st>>>(po, pn, vold, vnew, (Quad<T>*)quad, len);
}

// ------------------------------------------------------------------------------------------------
// one half-step of topic t over one orientation
//   E'      = E + (w_po t_po - w_pn t_pn)            pending change of the previous topic (written back)
//   Eh      = E' + own_cur * other_old               residual without topic t  (nmf.py:689-691 / :737-739)
//   numer_s = sum m * other_new * Eh                 nmf.py:697 / :745  (before the l1 term)
//   denom_s = sum m * other_new^2                    nmf.py:699 / :746  (before the l2 term)
// T-step: segments = columns, own = T[t,:], other_old = other_new = W[:,t].
// W-step: segments = rows, own = W[:,t], other_old / other_new = T[t,:] before / after this topic's T-step.
// ------------------------------------------------------------------------------------------------
//
// Shifted mode (SH, a handle with unstored weight w0 > 0, DESIGN.md §1 row f7): the copies hold S = mt E + w0 x with
// mt = m - w0 (m = 1 without entry weights), so that
//   S'      = S + mt (w_po t_po - w_pn t_pn)
//   numer_s = sum other_new * (S' + mt own_cur other_old)     = sum other_new (mt Eh + w0 x)
//   denom_s = sum mt other_new^2
// and the solve adds the dense rank-k part  -w0 sum_{s!=t} G_ts own_s,  +w0 G_tt  (sp_implicit_final_kernel).
template <typename T, bool HASW, bool SH>
RRI_DEVINL void sp_entry(T ev, const Quad<T>& q, T m, T opo, T opn, T oc, bool apply, T* __restrict__ Eout,
                         T& num, T& den, T w0)
{
    if constexpr (SH) {
        const T mt = sub_rn(m, w0);
        if (apply) {
            const T a = mul_rn(q.a, opo);
            const T b = mul_rn(q.b, opn);
            ev = fma(mt, sub_rn(a, b), ev);
            *Eout = ev;
        }
        const T eh = fma(mul_rn(mt, q.c), oc, ev);
        num = fma(q.d, eh, num);
        den = fma(mul_rn(mt, q.d), q.d, den);
        return;
    }
    if (apply) {
        const T a = mul_rn(q.a, opo);
        const T b = mul_rn(q.b, opn);
        ev = add_rn(ev, sub_rn(a, b));
        *Eout = ev;
    }
    const T eh = fma(oc, q.c, ev);
    const T wn = HASW ? mul_rn(m, q.d) : q.d;
    num = fma(wn, eh, num);
    den = fma(wn, q.d, den);
}

template <typename T, int G, bool HASW, bool SH>
__global__ void __launch_bounds__(256)
sp_pass_kernel(const int64_t* __restrict__ ptr, const int32_t* __restrict__ idx, T* __restrict__ E,
               const T* __restrict__ wgt, const Quad<T>* __restrict__ Q, const T* __restrict__ own_po,
               const T* __restrict__ own_pn, const T* __restrict__ own_cur, T* __restrict__ own_save,
               T* __restrict__ numer, T* __restrict__ denom, int64_t nseg, T w0)
{
    constexpr int GPB = 256 / G;
    constexpr int U = 4;
    __shared__ T red[2][8];
    const int lane = threadIdx.x % G, g = threadIdx.x / G;
    const bool apply = own_po != nullptr;
    for (int64_t s = (int64_t)blockIdx.x * GPB + g; s < nseg; s += (int64_t)gridDim.x * GPB) {
        const int64_t b = ptr[s], e = ptr[s + 1];
        const T opo = apply ? own_po[s] : T(0), opn = apply ? own_pn[s] : T(0);
        const T oc = own_cur[s];
        T num = T(0), den = T(0);
        int64_t p = b + lane;
        for (; p + (U - 1) * G < e; p += U * G) {          // loads batched ahead of the arithmetic
            int32_t q[U]; T ev[U]; T m[U]; Quad<T> qq[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                q[u] = idx[p + u * G];
                ev[u] = E[p + u * G];
                m[u] = HASW ? wgt[p + u * G] : T(1);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) qq[u] = Q[q[u]];
#pragma unroll
            for (int u = 0; u < U; ++u)
                sp_entry<T, HASW, SH>(ev[u], qq[u], m[u], opo, opn, oc, apply, E + p + u * G, num, den, w0);
        }
        for (; p < e; p += G) {
            const Quad<T> qq = Q[idx[p]];
            sp_entry<T, HASW, SH>(E[p], qq, HASW ? wgt[p] : T(1), opo, opn, oc, apply, E + p, num, den, w0);
        }
        num = warp_sum(num);
        den = warp_sum(den);
        if (G == 32) {
            if (lane == 0) { numer[s] = num; denom[s] = den; own_save[s] = oc; }
        } else {
            if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = num; red[1][threadIdx.x >> 5] = den; }
            __syncthreads();
            if (threadIdx.x == 0) {
                T a = T(0), c = T(0);
#pragma unroll
                for (int w = 0; w < 8; ++w) { a += red[0][w]; c += red[1][w]; }
                numer[s] = a; denom[s] = c; own_save[s] = oc;
            }
            __syncthreads();
        }
    }
}

// Blocked variant.  The direct kernel above is bound by the gather: 32 lanes hit 32 different 128-byte lines of Q,
// one L1 tag look-up each (measured 0.38-0.68 ms per pass at 1e8 entries, against 0.12-0.18 ms of HBM time).  Here
// the index range of the gathered factor is cut into blocks of `nb` records that fit shared memory; CTA (b, c)
// stages block b of Q once and walks the sub-segments [ptr2[s][b], ptr2[s][b+1]) of its chunk c of the segments, a
// warp per sub-segment, so every gather is a shared-memory read.  Per-block partial sums are written to
// numer_part[b][s], denom_part[b][s] and added in block order by the solve kernel (deterministic).
template <typename T, bool HASW, bool SH, int U, int THREADS, int MINB>
__global__ void __launch_bounds__(THREADS, MINB)
sp_pass_blocked_kernel(const int64_t* __restrict__ ptr2, const uint16_t* __restrict__ idx16, T* __restrict__ E,
                       const T* __restrict__ wgt, const Quad<T>* __restrict__ Q, const T* __restrict__ own_po,
                       const T* __restrict__ own_pn, const T* __restrict__ own_cur, T* __restrict__ own_save,
                       T* __restrict__ numer_part, T* __restrict__ denom_part, int64_t nseg, int nblk, int nb,
                       int64_t nother, int chunks, T w0)
{
    extern __shared__ __align__(16) unsigned char sp_smem[];
    Quad<T>* __restrict__ qs = reinterpret_cast<Quad<T>*>(sp_smem);
    const int b = (int)(blockIdx.x % (unsigned)nblk), c = (int)(blockIdx.x / (unsigned)nblk);
    const int64_t base = (int64_t)b * nb;
    const int cnt = (int)((nother - base) < (int64_t)nb ? (nother - base) : (int64_t)nb);
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) qs[i] = Q[base + i];
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    int64_t s0, s1;
    part_range(nseg, chunks, c, s0, s1);
    const bool apply = own_po != nullptr;
    const int64_t pstride = (int64_t)nblk + 1;
    // the bounds and the per-segment scalars of the NEXT sub-segment are requested before this one is streamed: the
    // pointer load would otherwise sit in front of every sub-segment's first batch (two dependent round trips per ~3 KB)
    int64_t s = s0 + warp;
    int64_t beg = 0, end = 0;
    T opo = T(0), opn = T(0), oc = T(0);
    if (s < s1) {
        beg = ptr2[s * pstride + b]; end = ptr2[s * pstride + b + 1];
        opo = apply ? own_po[s] : T(0); opn = apply ? own_pn[s] : T(0); oc = own_cur[s];
    }
    while (s < s1) {
        const int64_t sn = s + nwarps;
        int64_t nbeg = 0, nend = 0;
        T nopo = T(0), nopn = T(0), noc = T(0);
        if (sn < s1) {
            nbeg = ptr2[sn * pstride + b]; nend = ptr2[sn * pstride + b + 1];
            nopo = apply ? own_po[sn] : T(0); nopn = apply ? own_pn[sn] : T(0); noc = own_cur[sn];
        }
        T num = T(0), den = T(0);
        for (int64_t p0 = beg + lane; p0 < end + lane; p0 += 32 * U) {        // (p0 - lane) < end: uniform per warp
            int32_t q[U]; T ev[U]; T m[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int64_t p = p0 + u * 32;
                const bool ok = p < end;
                q[u] = ok ? (int32_t)idx16[p] : -1;                                // block-local record index
                ev[u] = ok ? E[p] : T(0);
                m[u] = (HASW && ok) ? wgt[p] : T(1);
            }
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (q[u] >= 0) {
                    const Quad<T> qq = qs[q[u]];
                    sp_entry<T, HASW, SH>(ev[u], qq, m[u], opo, opn, oc, apply, E + p0 + u * 32, num, den, w0);
                }
        }
        num = warp_sum(num);
        den = warp_sum(den);
        if (lane == 0) {
            numer_part[(int64_t)b * nseg + s] = num;
            denom_part[(int64_t)b * nseg + s] = den;
            if (b == 0) own_save[s] = oc;
        }
        s = sn; beg = nbeg; end = nend; opo = nopo; opn = nopn; oc = noc;
    }
}

// Streamlined form of the blocked pass for 16-bit block-local indices.  Same entry -> lane mapping and the same order
// of additions as sp_pass_blocked_kernel (bit-identical sums), but
//   * a sub-segment is addressed with 32-bit offsets from three base pointers (no 64-bit compare per entry),
//   * trips with all 32*U entries present run without any predicate,
//   * the remainder issues only the slots the warp needs (warp-uniform tests) -- with U = 16 almost every sub-segment
//     of a config-4 shaped problem (~330-390 entries) is ONE batch of loads with 11-13 slots in flight per lane.
template <typename T, bool HASW, bool SH, int U, int THREADS, int MINB>
__global__ void __launch_bounds__(THREADS, MINB)
sp_pass_stream_kernel(const int64_t* __restrict__ ptr2, const uint16_t* __restrict__ idx16, T* __restrict__ E,
                      const T* __restrict__ wgt, const Quad<T>* __restrict__ Q, const T* __restrict__ own_po,
                      const T* __restrict__ own_pn, const T* __restrict__ own_cur, T* __restrict__ own_save,
                      T* __restrict__ numer_part, T* __restrict__ denom_part, int64_t nseg, int nblk, int nb,
                      int64_t nother, int chunks, T w0)
{
    extern __shared__ __align__(16) unsigned char sp_smem[];
    Quad<T>* __restrict__ qs = reinterpret_cast<Quad<T>*>(sp_smem);
    const int b = (int)(blockIdx.x % (unsigned)nblk), c = (int)(blockIdx.x / (unsigned)nblk);
    const int64_t base = (int64_t)b * nb;
    const int cnt = (int)((nother - base) < (int64_t)nb ? (nother - base) : (int64_t)nb);
    for (int i = threadIdx.x; i < cnt; i += THREADS) qs[i] = Q[base + i];
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int NWARPS = THREADS / 32;
    int64_t s0, s1;
    part_range(nseg, chunks, c, s0, s1);
    const bool apply = own_po != nullptr;
    const int64_t pstride = (int64_t)nblk + 1;
    int64_t s = s0 + warp;
    int64_t beg = 0, end = 0;
    T opo = T(0), opn = T(0), oc = T(0);
    if (s < s1) {
        beg = ptr2[s * pstride + b]; end = ptr2[s * pstride + b + 1];
        opo = apply ? own_po[s] : T(0); opn = apply ? own_pn[s] : T(0); oc = own_cur[s];
    }
    while (s < s1) {
        const int64_t sn = s + NWARPS;
        int64_t nbeg = 0, nend = 0;
        T nopo = T(0), nopn = T(0), noc = T(0);
        if (sn < s1) {
            nbeg = ptr2[sn * pstride + b]; nend = ptr2[sn * pstride + b + 1];
            nopo = apply ? own_po[sn] : T(0); nopn = apply ? own_pn[sn] : T(0); noc = own_cur[sn];
        }
        T num = T(0), den = T(0);
        const int len = (int)(end - beg);
        const uint16_t* __restrict__ ip = idx16 + beg + lane;
        T* __restrict__ Ep = E + beg + lane;
        const T* __restrict__ wp = HASW ? wgt + beg + lane : nullptr;
        int i = 0;
        for (; i + 32 * U <= len; i += 32 * U) {                 // full trips: no predicates
            uint32_t q[U]; T ev[U]; T m[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                q[u] = ip[i + 32 * u];
                ev[u] = Ep[i + 32 * u];
                m[u] = HASW ? wp[i + 32 * u] : T(1);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const Quad<T> qq = qs[q[u]];
                sp_entry<T, HASW, SH>(ev[u], qq, m[u], opo, opn, oc, apply, Ep + i + 32 * u, num, den, w0);
            }
        }
        const int rem = len - i;                                  // < 32 * U entries left (warp-uniform)
        if (rem > 0) {
            const int lrem = rem - lane;                          // slot u holds an entry for this lane iff 32u < lrem
            uint32_t q[U]; T ev[U]; T m[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                q[u] = 0; ev[u] = T(0); m[u] = T(1);
                if (32 * u < rem) {                               // warp-uniform: slots beyond the remainder are skipped
                    const bool ok = 32 * u < lrem;
                    if (ok) {
                        q[u] = ip[i + 32 * u];
                        ev[u] = Ep[i + 32 * u];
                        if (HASW) m[u] = wp[i + 32 * u];
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (32 * u < lrem) {
                    const Quad<T> qq = qs[q[u]];
                    sp_entry<T, HASW, SH>(ev[u], qq, m[u], opo, opn, oc, apply, Ep + i + 32 * u, num, den, w0);
                }
        }
        num = warp_sum(num);
        den = warp_sum(den);
        if (lane == 0) {
            numer_part[(int64_t)b * nseg + s] = num;
            denom_part[(int64_t)b * nseg + s] = den;
            if (b == 0) own_save[s] = oc;
        }
        s = sn; beg = nbeg; end = nend; opo = nopo; opn = nopn; oc = noc;
    }
}

// ptr2[s][b] = first entry of segment s whose index is >= b * nb   (b = 0..nblk)
__global__ void sp_subptr_kernel(const int64_t* __restrict__ ptr, const int32_t* __restrict__ idx, int64_t nseg, int nblk,
                                 int nb, int64_t* __restrict__ ptr2)
{
    const int64_t total = nseg * ((int64_t)nblk + 1);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t s = i / (nblk + 1);
        const int b = (int)(i - s * (nblk + 1));
        int64_t lo = ptr[s], hi = ptr[s + 1];
        const int64_t target = (int64_t)b * nb;
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if ((int64_t)idx[mid] < target) lo = mid + 1; else hi = mid;
        }
        ptr2[i] = lo;
    }
}

// Records per staged block of Q: at most SP_BLOCK_BYTES of shared memory (one 1024-thread CTA per SM; a block of
// <= 64 KB runs as two 512-thread CTAs per SM), and all blocks equally long (a short last block would leave its CTAs
// with a fraction of the work of the others).
constexpr int64_t SP_BLOCK_BYTES = 128 * 1024;
static_assert(SP_BLOCK_BYTES / (4 * sizeof(float)) <= 65536, "block-local indices must fit 16 bits (SpSide::idx16)");

int sp_block_len(int elem_size, int64_t nother, int* nblk_out)
{
    const int64_t cap = SP_BLOCK_BYTES / (4 * elem_size);
    const int64_t nblk = nother > 0 ? (nother + cap - 1) / cap : 1;
    int64_t nb = (nother + nblk - 1) / nblk;
    nb = (nb + 31) / 32 * 32;
    if (nb > cap) nb = cap;
    if (nb < 32) nb = 32;
    *nblk_out = (int)((nother + nb - 1) / nb > 0 ? (nother + nb - 1) / nb : 1);
    return (int)nb;
}

__global__ void sp_local_index_kernel(const int32_t* __restrict__ idx, int64_t nnz, int nb, uint16_t* __restrict__ out)
{
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < nnz; p += (int64_t)gridDim.x * blockDim.x)
        out[p] = (uint16_t)(idx[p] % nb);
}

void launch_sp_local_index(const int32_t* idx, int64_t nnz, int nb, uint16_t* out, int sm_count, cudaStream_t st)
{
    sp_local_index_kernel<<<cap_blocks((nnz + 255) / 256, sm_count, 8), 256, 0, st>>>(idx, nnz, nb, out);
}

void launch_sp_subptr(const int64_t* ptr, const int32_t* idx, int64_t nseg, int nblk, int nb, int64_t* ptr2,
                      int sm_count, cudaStream_t st)
{
    const int64_t total = nseg * ((int64_t)nblk + 1);
    sp_subptr_kernel<<<cap_blocks((total + 255) / 256, sm_count, 8), 256, 0, st>>>(ptr, idx, nseg, nblk, nb, ptr2);
}

template <typename T, bool SH>
static int sp_pass_dispatch(const SpSide& s, const Quad<T>* Q, const T* own_po, const T* own_pn, const T* own_cur,
                            T* own_save, T* numer, T* denom, T w0, int sm_count, cudaStream_t st)
{
    const T* w = (const T*)s.wgt;
    T* E = (T*)s.E;
    if (s.ptr2) {
        constexpr int U = sizeof(T) == 8 ? 4 : 8;
        const int64_t cnt = s.nother < (int64_t)s.nb ? s.nother : (int64_t)s.nb;
        const size_t smem = (size_t)cnt * sizeof(Quad<T>);
        int chunks = sm_count / s.nblk;
        if (chunks < 1) chunks = 1;
        if ((int64_t)chunks * 32 > s.nseg) chunks = (int)((s.nseg + 31) / 32);
        if (chunks < 1) chunks = 1;
        if (smem <= 64 * 1024) {
            // two CTAs of 512 threads per SM: one CTA's staging phase overlaps the other's streaming
            chunks = 2 * sm_count / s.nblk;
            if (chunks < 1) chunks = 1;
            if ((int64_t)chunks * 16 > s.nseg) chunks = (int)((s.nseg + 15) / 16);
            if (chunks < 1) chunks = 1;
            auto kern = w ? sp_pass_blocked_kernel<T, true, SH, U, 512, 2> : sp_pass_blocked_kernel<T, false, SH, U, 512, 2>;
            if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
            kern<<<(unsigned)(s.nblk * chunks), 512, smem, st>>>(s.ptr2, s.idx16, E, w, Q, own_po, own_pn, own_cur, own_save,
                                                                numer, denom, s.nseg, s.nblk, s.nb, s.nother, chunks, w0);
            return s.nblk;
        }
        if constexpr (sizeof(T) == 4) {
            // fp32: the streamlined kernel, 16 entries per lane and batch where no weights are read (64 registers, no
            // spills), 8 with weights
            if (w) {
                auto kv = sp_pass_stream_kernel<T, true, SH, 8, 1024, 1>;
                if (smem > 48 * 1024) cudaFuncSetAttribute(kv, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                kv<<<(unsigned)(s.nblk * chunks), 1024, smem, st>>>(s.ptr2, s.idx16, E, w, Q, own_po, own_pn, own_cur, own_save,
                                                                   numer, denom, s.nseg, s.nblk, s.nb, s.nother, chunks, w0);
            } else {
                // (shifted: 12 entries per lane and batch -- 16 spill there)
                auto kv = sp_pass_stream_kernel<T, false, SH, SH ? 12 : 16, 1024, 1>;
                if (smem > 48 * 1024) cudaFuncSetAttribute(kv, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                kv<<<(unsigned)(s.nblk * chunks), 1024, smem, st>>>(s.ptr2, s.idx16, E, w, Q, own_po, own_pn, own_cur, own_save,
                                                                   numer, denom, s.nseg, s.nblk, s.nb, s.nother, chunks, w0);
            }
        } else {
            auto kern = w ? sp_pass_blocked_kernel<T, true, SH, U, 1024, 1> : sp_pass_blocked_kernel<T, false, SH, U, 1024, 1>;
            if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            kern<<<(unsigned)(s.nblk * chunks), 1024, smem, st>>>(s.ptr2, s.idx16, E, w, Q, own_po, own_pn, own_cur, own_save,
                                                                 numer, denom, s.nseg, s.nblk, s.nb, s.nother, chunks, w0);
        }
        return s.nblk;
    }
    if (s.group == 256) {
        const int nb = cap_blocks(s.nseg, sm_count, 8);
        if (w) sp_pass_kernel<T, 256, true, SH><<<nb, 256, 0, st>>>(s.ptr, s.idx, E, w, Q, own_po, own_pn, own_cur, own_save, numer, denom, s.nseg, w0);
        else   sp_pass_kernel<T, 256, false, SH><<<nb, 256, 0, st>>>(s.ptr, s.idx, E, w, Q, own_po, own_pn, own_cur, own_save, numer, denom, s.nseg, w0);
    } else {
        const int nb = cap_blocks((s.nseg + 7) / 8, sm_count, 8);
        if (w) sp_pass_kernel<T, 32, true, SH><<<nb, 256, 0, st>>>(s.ptr, s.idx, E, w, Q, own_po, own_pn, own_cur, own_save, numer, denom, s.nseg, w0);
        else   sp_pass_kernel<T, 32, false, SH><<<nb, 256, 0, st>>>(s.ptr, s.idx, E, w, Q, own_po, own_pn, own_cur, own_save, numer, denom, s.nseg, w0);
    }
    return 1;
}

template <typename T>
int launch_sp_pass(const SpSide& s, const void* quad, const T* own_po, const T* own_pn, const T* own_cur,
                   T* own_save, T* numer, T* denom, double w0, int sm_count, cudaStream_t st, bool shifted)
{
    const Quad<T>* Q = (const Quad<T>*)quad;
    if (w0 > 0.0 || shifted) return sp_pass_dispatch<T, true>(s, Q, own_po, own_pn, own_cur, own_save, numer, denom, (T)w0, sm_count, st);
    return sp_pass_dispatch<T, false>(s, Q, own_po, own_pn, own_cur, own_save, numer, denom, T(0), sm_count, st);
}

// ------------------------------------------------------------------------------------------------
// objective pieces (nmf.py:71-94 on the observed entries): out[0] = 0.5 sum m E^2, out[1] = sum m x^2
// ------------------------------------------------------------------------------------------------
// SH (unstored weight w0 > 0): a third sum, out of the parts only, s2 = sum (x - E)^2 = sum (W T)^2 over the stored
// entries (the part of <W'W, T T'> that the unstored weight does not apply to)
template <typename T, bool SH>
__global__ void __launch_bounds__(256)
sp_objective_kernel(const T* __restrict__ E, const T* __restrict__ x, const T* __restrict__ wgt, int64_t nnz,
                    double* __restrict__ part)
{
    constexpr int NS = SH ? 3 : 2;
    __shared__ double red[NS][8];
    double s0 = 0.0, s1 = 0.0, s2 = 0.0;
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < nnz; p += (int64_t)gridDim.x * blockDim.x) {
        const double m = wgt ? (double)wgt[p] : 1.0;
        const double r = (double)E[p], v = (double)x[p];
        s0 += m * r * r;
        s1 += m * v * v;
        if (SH) s2 += (v - r) * (v - r);
    }
    s0 = warp_sum(s0); s1 = warp_sum(s1);
    if (SH) s2 = warp_sum(s2);
    if ((threadIdx.x & 31) == 0) {
        red[0][threadIdx.x >> 5] = s0; red[1][threadIdx.x >> 5] = s1;
        if (SH) red[NS - 1][threadIdx.x >> 5] = s2;
    }
    __syncthreads();
    if (threadIdx.x < NS) {
        double s = 0.0;
        for (int w = 0; w < 8; ++w) s += red[threadIdx.x][w];
        part[NS * (int64_t)blockIdx.x + threadIdx.x] = s;
    }
}

// Rank-one unstored weights (DESIGN.md §1 row f8): the same three sums with s2 = sum a_i b_j (x - E)^2; a warp per row
// (grid-stride over the rows, fixed order), b_j gathered by the column index
template <typename T>
__global__ void __launch_bounds__(256)
sp_objective_rows_kernel(const int64_t* __restrict__ ptr, const int32_t* __restrict__ idx, const T* __restrict__ E,
                         const T* __restrict__ x, const T* __restrict__ wgt, int64_t nseg, const T* __restrict__ va,
                         const T* __restrict__ vb, double* __restrict__ part)
{
    __shared__ double red[3][8];
    const int lane = threadIdx.x & 31;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0;
    for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < nseg; r += ((int64_t)gridDim.x * blockDim.x) >> 5) {
        const double ai = va ? (double)va[r] : 1.0;
        for (int64_t p = ptr[r] + lane; p < ptr[r + 1]; p += 32) {
            const double m = wgt ? (double)wgt[p] : 1.0;
            const double e = (double)E[p], v = (double)x[p];
            const double ab = vb ? ai * (double)vb[idx[p]] : ai;
            s0 += m * e * e;
            s1 += m * v * v;
            s2 += ab * (v - e) * (v - e);
        }
    }
    s0 = warp_sum(s0); s1 = warp_sum(s1); s2 = warp_sum(s2);
    if (lane == 0) { red[0][threadIdx.x >> 5] = s0; red[1][threadIdx.x >> 5] = s1; red[2][threadIdx.x >> 5] = s2; }
    __syncthreads();
    if (threadIdx.x < 3) {
        double s = 0.0;
        for (int w = 0; w < 8; ++w) s += red[threadIdx.x][w];
        part[3 * (int64_t)blockIdx.x + threadIdx.x] = s;
    }
}

__global__ void sp_objective_finalize_kernel(const double* __restrict__ part, int blocks, double* __restrict__ out)
{
    if (threadIdx.x < 2) {
        double s = 0.0;
        for (int b = 0; b < blocks; ++b) s += part[2 * (int64_t)b + threadIdx.x];
        out[threadIdx.x] = threadIdx.x == 0 ? 0.5 * s : s;
    }
}

// out[0] = 0.5 (sum m E^2 + w0 (<W'W, T T'> - sum (x - E)^2)) = 0.5 sum M (X - W T)^2 over all n x d entries,
// out[1] = sum m x^2; <W'W, T T'> from the fp64 Gram partials gw [k][cw][k] and gt [k][ct][k] (fixed order).  With
// rank-one weights the Grams are W' diag(a) W and T diag(b) T' and s2 carries a_i b_j.
__global__ void __launch_bounds__(256)
sp_objective_implicit_finalize_kernel(const double* __restrict__ part, int blocks, const double* __restrict__ gw, int cw,
                                      const double* __restrict__ gt, int ct, int k, double w0, double* __restrict__ out)
{
    __shared__ double red[8];
    double gh = 0.0;
    for (int q = threadIdx.x; q < k * k; q += blockDim.x) {
        const int a = q / k, b = q - a * k;
        double x = 0.0, y = 0.0;
        for (int c = 0; c < cw; ++c) x += gw[((int64_t)a * cw + c) * k + b];
        for (int c = 0; c < ct; ++c) y += gt[((int64_t)a * ct + c) * k + b];
        gh += x * y;
    }
    gh = warp_sum(gh);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = gh;
    __syncthreads();
    if (threadIdx.x == 0) {
        double g = 0.0, s0 = 0.0, s1 = 0.0, s2 = 0.0;
        for (int w = 0; w < 8; ++w) g += red[w];
        for (int b = 0; b < blocks; ++b) { s0 += part[3 * (int64_t)b]; s1 += part[3 * (int64_t)b + 1]; s2 += part[3 * (int64_t)b + 2]; }
        out[0] = 0.5 * (s0 + w0 * (g - s2));
        out[1] = s1;
    }
}

template <typename T>
void launch_sp_objective(const SpSide& s, int64_t nnz, double* part, double* out, double w0, const double* gw, int cw,
                         const double* gt, int ct, int k, cudaStream_t st, const T* va, const T* vb)
{
    int blocks = (int)((nnz + 256 * 8 - 1) / (256 * 8));
    if (blocks > 256) blocks = 256;
    if (blocks < 1) blocks = 1;
    if (w0 > 0.0 && (va || vb)) {
        sp_objective_rows_kernel<T><<<blocks, 256, 0, st>>>(s.ptr, s.idx, (const T*)s.E, (const T*)s.x, (const T*)s.wgt, s.nseg,
                                                            va, vb, part);
        sp_objective_implicit_finalize_kernel<<<1, 256, 0, st>>>(part, blocks, gw, cw, gt, ct, k, w0, out);
        return;
    }
    if (w0 > 0.0) {
        sp_objective_kernel<T, true><<<blocks, 256, 0, st>>>((const T*)s.E, (const T*)s.x, (const T*)s.wgt, nnz, part);
        sp_objective_implicit_finalize_kernel<<<1, 256, 0, st>>>(part, blocks, gw, cw, gt, ct, k, w0, out);
        return;
    }
    sp_objective_kernel<T, false><<<blocks, 256, 0, st>>>((const T*)s.E, (const T*)s.x, (const T*)s.wgt, nnz, part);
    sp_objective_finalize_kernel<<<1, 32, 0, st>>>(part, blocks, out);
}

// ------------------------------------------------------------------------------------------------
// the dense rank-k part of a half-step on a handle with unstored weight w0 (DESIGN.md §1 row f7)
// ------------------------------------------------------------------------------------------------
// Gram rows of F [k, ld] (row r = topic r over len entries): for z < gridDim.z, with t = t0 + z,
//   part[z][c][s] = sum_{i in chunk c} F[t, i] F[s, i]     (one block per (s, c, z); fixed-order block reduction)
// WV (rank-one unstored weights, row f8): sum F[t, i] v_i F[s, i] with the weight vector v over the len entries
// (a for W' diag(a) W, b for T diag(b) T'), the product F[t, i] v_i rounded in A first.
template <typename T, typename A, bool WV>
__global__ void __launch_bounds__(256)
sp_gram_rows_kernel(const T* __restrict__ F, int64_t ld, int64_t len, int k, int t0, int chunks, A* __restrict__ part,
                    const T* __restrict__ wv)
{
    __shared__ A red[8];
    const int s = blockIdx.x, c = blockIdx.y, z = blockIdx.z;
    int64_t b, e;
    part_range(len, chunks, c, b, e);
    const T* __restrict__ a = F + (int64_t)(t0 + z) * ld;
    const T* __restrict__ f = F + (int64_t)s * ld;
    A acc = A(0);
    if constexpr (WV) {
        for (int64_t i = b + threadIdx.x; i < e; i += 256) acc = fma((A)a[i] * (A)wv[i], (A)f[i], acc);
    } else {
        for (int64_t i = b + threadIdx.x; i < e; i += 256) acc = fma((A)a[i], (A)f[i], acc);
    }
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        A g = A(0);
#pragma unroll
        for (int w = 0; w < 8; ++w) g += red[w];
        part[((int64_t)z * chunks + c) * k + s] = g;
    }
}

int sp_gram_chunks(int64_t len, int pairs, int sm_count)
{
    int64_t c = (2 * (int64_t)sm_count + pairs - 1) / pairs;
    const int64_t cap = (len + 2047) / 2048;
    if (c > cap) c = cap;
    if (c > 64) c = 64;
    return (int)(c < 1 ? 1 : c);
}

template <typename T, typename A>
void launch_sp_gram_rows(const T* F, int64_t ld, int64_t len, int k, int t0, int rows, int chunks, A* part, cudaStream_t st,
                         const T* wv)
{
    const dim3 grid((unsigned)k, (unsigned)chunks, (unsigned)rows);
    if (wv) sp_gram_rows_kernel<T, A, true><<<grid, 256, 0, st>>>(F, ld, len, k, t0, chunks, part, wv);
    else sp_gram_rows_kernel<T, A, false><<<grid, 256, 0, st>>>(F, ld, len, k, t0, chunks, part, nullptr);
}

// The vector-c solve of wrri_final_kernel with the rank-k part of the statistic added first:
//   numer_i = sum_p numer_part[p][i] - w0 sum_{s != t} g_s F[s, i],   denom_i = sum_p denom_part[p][i] + w0 g_t
// g = the Gram row of topic t (sum of its `gchunks` partials), F [k, ldf] the factor being updated (rows s != t only:
// row t is the one written).  sc (rank-one unstored weights, row f8): w0 is w0 sc_i for entry i -- b_j in a T-step,
// a_i in a W-step -- in both terms.
template <typename T>
__global__ void __launch_bounds__(256)
sp_implicit_final_kernel(const T* __restrict__ numer_part, const T* __restrict__ denom_part, int parts, int64_t len,
                         const T* __restrict__ gpart, int gchunks, int k, int t, const T* __restrict__ F, int64_t ldf,
                         T w0, T reg_l1, T reg_l2, T eps, T ub, int has_ub, T* __restrict__ out, int64_t out_stride,
                         T* __restrict__ out2, int64_t out2_stride, int* __restrict__ flags, const T* __restrict__ sc)
{
    __shared__ T g[256];
    for (int s = threadIdx.x; s < k; s += blockDim.x) {
        T a = T(0);
        for (int c = 0; c < gchunks; ++c) a += gpart[(int64_t)c * k + s];
        g[s] = a;
    }
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= len) return;
    T nu = T(0), de = T(0);
#pragma unroll 4
    for (int p = 0; p < parts; ++p) {
        nu += numer_part[(int64_t)p * len + i];
        de += denom_part[(int64_t)p * len + i];
    }
    T corr = T(0);
    for (int s = 0; s < k; ++s)
        if (s != t) corr = fma(g[s], F[(int64_t)s * ldf + i], corr);
    const T wi = sc ? mul_rn(w0, sc[i]) : w0;
    nu = fma(-wi, corr, nu);
    de = fma(wi, g[t], de);
    bool unb = false;
    const T x = solve_vector_c<T>(nu - reg_l1, de + reg_l2, eps, ub, has_ub != 0, unb);
    out[i * out_stride] = x;
    if (out2) out2[i * out2_stride] = x;
    if (unb) atomicOr(flags, 4);
}

template <typename T>
void launch_sp_implicit_final(const T* numer_part, const T* denom_part, int parts, int64_t len, const T* gpart, int gchunks,
                              int k, int t, const T* F, int64_t ldf, double w0, const SolveArgs& a, T* out,
                              int64_t out_stride, T* out2, int64_t out2_stride, int* flags, cudaStream_t st, const T* sc)
{
    sp_implicit_final_kernel<T><<<(unsigned)((len + 255) / 256), 256, 0, st>>>(numer_part, denom_part, parts, len, gpart,
        gchunks, k, t, F, ldf, (T)w0, (T)a.reg_l1, (T)a.reg_l2, (T)a.eps, (T)a.ub, a.has_ub, out, out_stride, out2,
        out2_stride, flags, sc);
}

// ------------------------------------------------------------------------------------------------
// rank-one unstored weights u_ij = w0 (a_i b_j) (rri_set_unstored_weight_vectors, DESIGN.md §1 row f8), once per bind
// ------------------------------------------------------------------------------------------------
// err |= bit unless every v[i] is finite and >= 0
template <typename T>
__global__ void sp_check_weights_kernel(const T* __restrict__ v, int64_t len, int bit, int* __restrict__ err)
{
    bool bad = false;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (int64_t)gridDim.x * blockDim.x)
        bad |= !(isfinite((double)v[i]) && v[i] >= T(0));
    if (__syncthreads_or(bad) && threadIdx.x == 0) atomicOr(err, bit);
}

template <typename T>
void launch_sp_check_weights(const T* v, int64_t len, int bit, int* err, int sm_count, cudaStream_t st)
{
    if (v && len > 0) sp_check_weights_kernel<T><<<cap_blocks((len + 255) / 256, sm_count, 4), 256, 0, st>>>(v, len, bit, err);
}

// mt[p] = m[p] - w0 (a_i b_j) in CSR order (m = 1 without entry weights; a warp per row).  The column copy is the
// permutation of it (launch_sp_gather), so both orientations hold the same bits.
template <typename T>
__global__ void __launch_bounds__(256)
sp_mtilde_kernel(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col, const T* __restrict__ wgt, int64_t n,
                 const T* __restrict__ va, const T* __restrict__ vb, T w0, T* __restrict__ mt)
{
    const int lane = threadIdx.x & 31;
    for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n; r += ((int64_t)gridDim.x * blockDim.x) >> 5) {
        const T ai = va ? va[r] : T(1);
        for (int64_t p = rowptr[r] + lane; p < rowptr[r + 1]; p += 32) {
            const T u = mul_rn(w0, mul_rn(ai, vb ? vb[col[p]] : T(1)));
            mt[p] = sub_rn(wgt ? wgt[p] : T(1), u);
        }
    }
}

template <typename T>
void launch_sp_mtilde(const int64_t* rowptr, const int32_t* col, const T* wgt, int64_t n, const T* va, const T* vb,
                      double w0, T* mt, int sm_count, cudaStream_t st)
{
    sp_mtilde_kernel<T><<<cap_blocks((n + 7) / 8, sm_count, 8), 256, 0, st>>>(rowptr, col, wgt, n, va, vb, (T)w0, mt);
}

#define RRI_INST(T)                                                                                                 \
    template int sp_build_csc<T>(const int64_t*, const int32_t*, const T*, const T*, int64_t, int64_t, int64_t,    \
                                 int64_t*, int32_t*, T*, T*, uint32_t*, int, int*, cudaStream_t);                  \
    template void launch_sp_residual_rows<T>(const SpSide&, const T*, int64_t, const T*, int, int, double, int,    \
                                             cudaStream_t, const T*, const T*);                                    \
    template void launch_sp_gather<T>(const uint32_t*, const T*, T*, int64_t, int, cudaStream_t);                  \
    template void launch_sp_pack<T>(const T*, const T*, const T*, const T*, void*, int64_t, cudaStream_t);         \
    template int launch_sp_pass<T>(const SpSide&, const void*, const T*, const T*, const T*, T*, T*, T*, double,   \
                                   int, cudaStream_t, bool);                                                       \
    template void launch_sp_objective<T>(const SpSide&, int64_t, double*, double*, double, const double*, int,      \
                                         const double*, int, int, cudaStream_t, const T*, const T*);               \
    template void launch_sp_implicit_final<T>(const T*, const T*, int, int64_t, const T*, int, int, int, const T*, \
                                              int64_t, double, const SolveArgs&, T*, int64_t, T*, int64_t, int*,   \
                                              cudaStream_t, const T*);                                             \
    template void launch_sp_check_weights<T>(const T*, int64_t, int, int*, int, cudaStream_t);                     \
    template void launch_sp_mtilde<T>(const int64_t*, const int32_t*, const T*, int64_t, const T*, const T*, double, \
                                      T*, int, cudaStream_t);
RRI_INST(float)
RRI_INST(double)
// Gram rows: accumulated in the element type inside a half-step, in fp64 for the objective
template void launch_sp_gram_rows<float, float>(const float*, int64_t, int64_t, int, int, int, int, float*, cudaStream_t,
                                                const float*);
template void launch_sp_gram_rows<float, double>(const float*, int64_t, int64_t, int, int, int, int, double*, cudaStream_t,
                                                 const float*);
template void launch_sp_gram_rows<double, double>(const double*, int64_t, int64_t, int, int, int, int, double*, cudaStream_t,
                                                  const double*);

}  // namespace rri
