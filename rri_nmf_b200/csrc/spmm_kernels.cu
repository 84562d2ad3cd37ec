// spmm_kernels.cu -- the contraction of the block-order half-steps on a sparse matrix whose unstored entries are zeros
// (rri_bind_csr_zero):
//     C[r, :] = sum_{e in segment r} val[e] * B[idx[e], :]
// over the CSR rows (W half: B = T' [d, k], C = X T') or over the CSC columns (T half: B = W [n, k], C = X' W).
// Everything after C -- Gram, row updates, simplex T update, objective identity -- is the dense block order's.
//
// A group of G lanes owns one work item and keeps the k accumulators of its output row in registers (lane l holds the
// 16-byte units l, l + G, ... of the row, or single elements when k * sizeof(T) is not a multiple of 16).  The value and
// index streams are read once with evict-first loads; the gathered factor rows go through the normal cached path and
// stay L2-resident as long as the factor fits there.
//
// Load balance without float atomics: a segment longer than SPMM_CHUNK entries (a stop word's column can hold every
// row) is cut into chunks by a plan built once at bind time.  Each chunk writes its partial row to a slot; the chunk
// that arrives last (arrival counter, zero between launches) adds the slots in chunk order and writes the output row.
// Every output entry is therefore summed in an order fixed by the plan: N sweeps in one call equal N calls of one
// sweep, bit for bit.  One launch per half-step whatever k is.
//
// B and C have leading dimensions (ldb, ldc >= k), so that a column panel of a wider operand is computed in place:
// rri_spmm takes operands of up to k + 10 columns (the randomized SVD of the NNDSVD initialisation) as panels of at most
// SPMM_PANEL columns, one launch each, in ascending order.  The chunk slots of a panel are [chunks, panel width].
#include "common.cuh"
#include "kernels.h"

namespace rri {

template <typename T, int W>
RRI_DEVINL void ld_units(const T* p, T* o)
{
    if constexpr (W == 1) o[0] = __ldg(p);
    else unpack(__ldg(reinterpret_cast<const typename Vec<T>::type*>(p)), o);
}
template <typename T, int W>
RRI_DEVINL void ld_units_l2(const T* p, T* o)          // slots written by other blocks of this launch: bypass L1
{
    if constexpr (W == 1) o[0] = __ldcg(p);
    else unpack(__ldcg(reinterpret_cast<const typename Vec<T>::type*>(p)), o);
}
template <typename T, int W>
RRI_DEVINL void st_units(T* p, const T* v)
{
    if constexpr (W == 1) p[0] = v[0];
    else if constexpr (sizeof(T) == 4) *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    else *reinterpret_cast<double2*>(p) = make_double2(v[0], v[1]);
}

// W elements per load (Vec<T>::N or 1); NV loads per lane and entry
template <typename T, int W, int NV>
__global__ void __launch_bounds__(256)
spmm_kernel(SpmmPlan p, const T* __restrict__ B, int ldb, int k, int G, T* __restrict__ C, int ldc)
{
    // entries whose gathers are in flight together (2 for the widest fp64 rows: 4 spills there)
    constexpr int U = NV * W * sizeof(T) > 32 ? 2 : 4;
    const int gpb = 256 / G;
    const int lane = threadIdx.x % G;
    const int64_t item = (int64_t)blockIdx.x * gpb + threadIdx.x / G;
    if (item >= p.nlong_items + p.nseg) return;
    const int64_t* __restrict__ ptr = p.ptr;
    const int32_t* __restrict__ idx = p.idx;
    const T* __restrict__ val = static_cast<const T*>(p.val);
    int j = -1, c = 0;
    int64_t seg, b, e;
    if (item < p.nlong_items) {                        // long segments first: their chunks start early
        const int2 it = p.litem[item];
        j = it.x; c = it.y;
        seg = p.lseg[j];
        b = ptr[seg] + (int64_t)c * SPMM_CHUNK;
        const int64_t s1 = ptr[seg + 1];
        e = b + SPMM_CHUNK < s1 ? b + SPMM_CHUNK : s1;
    } else {
        seg = item - p.nlong_items;
        b = ptr[seg];
        e = ptr[seg + 1];
        if (e - b > SPMM_CHUNK) return;                // taken in chunks by the items above
    }
    const int units = k / W;
    T acc[NV * W];
#pragma unroll
    for (int i = 0; i < NV * W; ++i) acc[i] = T(0);
    int64_t q = b;
    for (; q + U <= e; q += U) {
        int32_t jj[U];
        T xv[U], bv[U][NV * W];
#pragma unroll
        for (int u = 0; u < U; ++u) { jj[u] = __ldcs(idx + q + u); xv[u] = __ldcs(val + q + u); }
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int v = 0; v < NV; ++v)
                if (lane + G * v < units) ld_units<T, W>(B + (int64_t)jj[u] * ldb + (lane + G * v) * W, &bv[u][v * W]);
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int v = 0; v < NV; ++v)
                if (lane + G * v < units)
#pragma unroll
                    for (int w = 0; w < W; ++w) acc[v * W + w] = fma(xv[u], bv[u][v * W + w], acc[v * W + w]);
    }
    for (; q < e; ++q) {
        const int32_t jq = __ldcs(idx + q);
        const T xq = __ldcs(val + q);
#pragma unroll
        for (int v = 0; v < NV; ++v)
            if (lane + G * v < units) {
                T bq[W];
                ld_units<T, W>(B + (int64_t)jq * ldb + (lane + G * v) * W, bq);
#pragma unroll
                for (int w = 0; w < W; ++w) acc[v * W + w] = fma(xq, bq[w], acc[v * W + w]);
            }
    }
    T* out = j < 0 ? C + seg * ldc : static_cast<T*>(p.slots) + (p.lslot[j] + c) * k;
#pragma unroll
    for (int v = 0; v < NV; ++v)
        if (lane + G * v < units) st_units<T, W>(out + (lane + G * v) * W, &acc[v * W]);
    if (j < 0) return;
    // fix-up of a chunked segment: the last chunk to arrive adds all slots in chunk order
    const int wl = threadIdx.x & 31, leader = wl & ~(G - 1);
    const unsigned gmask = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << leader);
    __threadfence();
    __syncwarp(gmask);
    unsigned ticket = 0;
    if (lane == 0) ticket = atomicAdd(p.counters + j, 1u);
    ticket = __shfl_sync(gmask, ticket, leader);
    const int nch = (int)((ptr[seg + 1] - ptr[seg] + SPMM_CHUNK - 1) / SPMM_CHUNK);
    if (ticket != (unsigned)(nch - 1)) return;
    __threadfence();
    const T* sl = static_cast<const T*>(p.slots) + p.lslot[j] * k;
#pragma unroll
    for (int v = 0; v < NV; ++v)
        if (lane + G * v < units) {
            const int off = (lane + G * v) * W;
            T s[W], t[W];
            ld_units_l2<T, W>(sl + off, s);
            for (int h = 1; h < nch; ++h) {
                ld_units_l2<T, W>(sl + (int64_t)h * k + off, t);
#pragma unroll
                for (int w = 0; w < W; ++w) s[w] += t[w];
            }
            st_units<T, W>(C + seg * ldc + off, s);
        }
    if (lane == 0) p.counters[j] = 0u;
}

template <typename T>
void launch_spmm(const SpmmPlan& p, const T* B, int64_t ldb, int width, T* C, int64_t ldc, cudaStream_t st)
{
    constexpr int VN = Vec<T>::N;
    const int64_t items = p.nlong_items + p.nseg;
    for (int off = 0; off < width; off += SPMM_PANEL) {
        const int k = width - off < SPMM_PANEL ? width - off : SPMM_PANEL;
        const T* Bp = B + off;
        T* Cp = C + off;
        const bool vec = (k % VN) == 0 && (ldb % VN) == 0 && (ldc % VN) == 0 &&
                         (reinterpret_cast<uintptr_t>(Bp) & 15) == 0 && (reinterpret_cast<uintptr_t>(Cp) & 15) == 0 &&
                         (reinterpret_cast<uintptr_t>(p.slots) & 15) == 0;
        const int units = vec ? k / VN : k;
        int G = 1;
        while (G < units && G < 32) G <<= 1;
        const int nv = (units + G - 1) / G;
        const unsigned blocks = (unsigned)((items + 256 / G - 1) / (256 / G));
        if (blocks == 0) return;
        const int lb = (int)ldb, lc = (int)ldc;
#define RRI_SPMM(W, NV) spmm_kernel<T, W, NV><<<blocks, 256, 0, st>>>(p, Bp, lb, k, G, Cp, lc)
        if (vec) {
            if (nv <= 1) RRI_SPMM(VN, 1);
            else if (nv <= 2) RRI_SPMM(VN, 2);
            else if constexpr (sizeof(T) == 8) RRI_SPMM(VN, 4);      // (fp64, k > 128; fp32 needs at most 2)
        } else {
            if (nv <= 1) RRI_SPMM(1, 1);
            else if (nv <= 2) RRI_SPMM(1, 2);
            else if (nv <= 4) RRI_SPMM(1, 4);
            else RRI_SPMM(1, 8);
        }
#undef RRI_SPMM
    }
}

// w o x of an observed-entries binding, the values rri_spmm applies there (built once, on the first call)
template <typename T>
__global__ void spmm_weighted_values_kernel(const T* __restrict__ x, const T* __restrict__ w, int64_t nnz, T* __restrict__ out)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = w[i] * x[i];
}

template <typename T>
void launch_spmm_weighted_values(const T* x, const T* w, int64_t nnz, T* out, int sm_count, cudaStream_t st)
{
    if (nnz <= 0) return;
    const int64_t want = (nnz + 255) / 256, cap = (int64_t)sm_count * 8;
    spmm_weighted_values_kernel<T><<<(unsigned)(want < cap ? want : cap), 256, 0, st>>>(x, w, nnz, out);
}

template void launch_spmm<float>(const SpmmPlan&, const float*, int64_t, int, float*, int64_t, cudaStream_t);
template void launch_spmm<double>(const SpmmPlan&, const double*, int64_t, int, double*, int64_t, cudaStream_t);
template void launch_spmm_weighted_values<float>(const float*, const float*, int64_t, float*, int, cudaStream_t);
template void launch_spmm_weighted_values<double>(const double*, const double*, int64_t, double*, int, cudaStream_t);

}  // namespace rri
