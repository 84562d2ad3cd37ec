// sparse_rri_kernels.cu -- the interleaved-order pass on a zero-filled sparse handle (rri_bind_csr_zero, RRI_ORDER_RRI).
// One launch per topic computes both statistics of the dense rri_pass_kernel from the two compressed orientations:
//     y[i] = sum_{e in row i} x[e] * T[t, col[e]]          (W-step t; over the CSR rows)
//     p[j] = sum_{e in col j} x[e] * W[row[e], tn]         (T-step tn = (t + 1) mod k; over the CSC columns)
// and writes them as ypart (ct = 1, stride n) and ppart (rg = 1, stride d): the dense order's T-step, W-step,
// statistic reduction and all-reduce then run unchanged.
//
// The blocks of the launch are split between the two orientations in proportion to their work.  A block is resident
// for the whole launch and walks the work items of its orientation: segments of at most SPMM_CHUNK entries and the
// chunks of longer ones, from the SpmmPlan of the block-order contraction (h->zrow, h->zcol) unchanged.  A group of G
// lanes owns one item; lane l accumulates entries l, l + G, ... (SRP_U of them in flight, values and indices read with
// evict-first loads) and the group adds its lanes with a butterfly.  A chunk writes its partial to the plan's slot at
// width 1; the last chunk to arrive (arrival counter, zero between launches) adds the slots in chunk order.  Every
// output entry is thus summed in an order fixed by the plan and G: N sweeps in one call equal N calls of one sweep,
// bit for bit.  Empty segments write 0.
//
// Both gathered vectors go through the cache: T[t, :] (contiguous, d elements) for the rows, W[:, tn] (row stride k) for
// the columns.  Staging T[t, :] in shared memory (two 512-thread blocks per SM at config 3) was measured slower:
// 0.41 against 0.32 ms per pass at config-3 shape and 0.69 % stored entries.
#include "common.cuh"
#include "kernels.h"

namespace rri {

constexpr int SRP_THREADS = 512;
constexpr int SRP_U = 4;                       // entries per lane in flight

template <typename T>
struct SrpSide {
    SpmmPlan pl;
    const T* vec;          // gathered vector: element idx[e] at vec[idx[e] * stride]
    int64_t stride;
    T* out;                // [nseg]
    int G;                 // lanes per work item (power of two, 4..32)
    int blocks;            // blocks of the launch on this orientation
};

template <typename T>
RRI_DEVINL void srp_side(const SrpSide<T>& s, int blk)
{
    constexpr int NW = SRP_THREADS / WARP;
    const int G = s.G, gpw = WARP / G;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gl = lane & (G - 1), gw = lane / G;
    const int64_t nlong = s.pl.nlong_items, nitems = nlong + s.pl.nseg;
    const int64_t* __restrict__ ptr = s.pl.ptr;
    const int32_t* __restrict__ idx = s.pl.idx;
    const T* __restrict__ val = static_cast<const T*>(s.pl.val);
    const T* __restrict__ g = s.vec;
    const int64_t gs = s.stride;
    const int64_t wstride = (int64_t)s.blocks * NW * gpw;
    // warp-uniform loop (every lane takes part in the group butterfly); long segments' chunks come first
    for (int64_t base = ((int64_t)blk * NW + warp) * gpw; base < nitems; base += wstride) {
        const int64_t item = base + gw;
        int j = -1, c = 0;
        int64_t seg = -1, b = 0, e = 0;
        if (item < nlong) {
            const int2 it = s.pl.litem[item];
            j = it.x; c = it.y;
            seg = s.pl.lseg[j];
            b = ptr[seg] + (int64_t)c * SPMM_CHUNK;
            const int64_t s1 = ptr[seg + 1];
            e = b + SPMM_CHUNK < s1 ? b + SPMM_CHUNK : s1;
        } else if (item < nitems) {
            seg = item - nlong;
            b = ptr[seg];
            e = ptr[seg + 1];
            if (e - b > SPMM_CHUNK) { seg = -1; b = e = 0; }       // taken in chunks by the items above
        }
        T acc = T(0);
        int64_t q = b + gl;
        for (; q + (SRP_U - 1) * G < e; q += SRP_U * G) {
            int32_t jj[SRP_U];
            T xv[SRP_U], gv[SRP_U];
#pragma unroll
            for (int u = 0; u < SRP_U; ++u) { jj[u] = __ldcs(idx + q + u * G); xv[u] = __ldcs(val + q + u * G); }
#pragma unroll
            for (int u = 0; u < SRP_U; ++u) gv[u] = __ldg(g + (int64_t)jj[u] * gs);
#pragma unroll
            for (int u = 0; u < SRP_U; ++u) acc = fma(xv[u], gv[u], acc);
        }
        for (; q < e; q += G) acc = fma(__ldcs(val + q), __ldg(g + (int64_t)__ldcs(idx + q) * gs), acc);
        for (int o = G >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (seg < 0 || gl != 0) continue;
        if (j < 0) { s.out[seg] = acc; continue; }
        // a chunk of a long segment: the last one to arrive adds all slots in chunk order
        T* slots = static_cast<T*>(s.pl.slots) + s.pl.lslot[j];
        slots[c] = acc;
        __threadfence();
        const unsigned ticket = atomicAdd(s.pl.counters + j, 1u);
        const int nch = (int)((ptr[seg + 1] - ptr[seg] + SPMM_CHUNK - 1) / SPMM_CHUNK);
        if (ticket != (unsigned)(nch - 1)) continue;
        __threadfence();
        T sum = __ldcg(slots);
        for (int h = 1; h < nch; ++h) sum += __ldcg(slots + h);
        s.out[seg] = sum;
        s.pl.counters[j] = 0u;
    }
}

template <typename T>
__global__ void __launch_bounds__(SRP_THREADS)
sparse_rri_pass_kernel(SrpSide<T> ys, SrpSide<T> ps)
{
    if ((int)blockIdx.x < ys.blocks) srp_side<T>(ys, blockIdx.x);
    else srp_side<T>(ps, blockIdx.x - ys.blocks);
}

static int srp_group(int64_t nnz, int64_t nseg)
{
    const int64_t avg = nseg > 0 ? (nnz + nseg - 1) / nseg : 0;
    int G = 4;
    while (G < 32 && (int64_t)G * SRP_U < avg) G <<= 1;
    return G;
}

template <typename T>
SparsePassPlan plan_sparse_rri_pass(const SpmmPlan& rows, const SpmmPlan& cols, int64_t nnz, int sm_count)
{
    SparsePassPlan pl;
    const int64_t n = rows.nseg, d = cols.nseg;
    pl.gy = srp_group(nnz, n);
    pl.gp = srp_group(nnz, d);
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sparse_rri_pass_kernel<T>, SRP_THREADS, 0) !=
            cudaSuccess || per_sm < 1)
        per_sm = 1;
    pl.blocks = per_sm * sm_count;
    // work of an orientation: its entries plus a per-item cost of one round of the group
    const double wy = (double)nnz + (double)(n + rows.nlong_items) * pl.gy * SRP_U;
    const double wp = (double)nnz + (double)(d + cols.nlong_items) * pl.gp * SRP_U;
    int by = (int)(pl.blocks * wy / (wy + wp) + 0.5);
    if (by < 1) by = 1;
    if (by > pl.blocks - 1) by = pl.blocks - 1 > 0 ? pl.blocks - 1 : 1;
    pl.blocks_y = by;
    pl.blocks_p = pl.blocks - by > 0 ? pl.blocks - by : 1;
    return pl;
}

// blocks that have an item: never more than the items need
static int srp_cap(int blocks, const SpmmPlan& p, int G)
{
    const int64_t per_block = (int64_t)(SRP_THREADS / WARP) * (WARP / G);
    const int64_t need = (p.nlong_items + p.nseg + per_block - 1) / per_block;
    return (int)(need < blocks ? (need < 1 ? 1 : need) : blocks);
}

template <typename T>
void launch_sparse_rri_pass(const SparsePassPlan& pl, const SpmmPlan& rows, const SpmmPlan& cols, const T* trow,
                            const T* W, int k, int tn, T* y, T* p, bool do_y, bool do_p, cudaStream_t st)
{
    if (!do_y && !do_p) return;
    SrpSide<T> ys{rows, trow, 1, y, pl.gy, 0};
    SrpSide<T> ps{cols, W + tn, k, p, pl.gp, 0};
    if (do_y) ys.blocks = srp_cap(do_p ? pl.blocks_y : pl.blocks, rows, pl.gy);
    if (do_p) ps.blocks = srp_cap(do_y ? pl.blocks_p : pl.blocks, cols, pl.gp);
    sparse_rri_pass_kernel<T><<<(unsigned)(ys.blocks + ps.blocks), SRP_THREADS, 0, st>>>(ys, ps);
}

template SparsePassPlan plan_sparse_rri_pass<float>(const SpmmPlan&, const SpmmPlan&, int64_t, int);
template SparsePassPlan plan_sparse_rri_pass<double>(const SpmmPlan&, const SpmmPlan&, int64_t, int);
template void launch_sparse_rri_pass<float>(const SparsePassPlan&, const SpmmPlan&, const SpmmPlan&, const float*,
                                            const float*, int, int, float*, float*, bool, bool, cudaStream_t);
template void launch_sparse_rri_pass<double>(const SparsePassPlan&, const SpmmPlan&, const SpmmPlan&, const double*,
                                             const double*, int, int, double*, double*, bool, bool, cudaStream_t);

}  // namespace rri
