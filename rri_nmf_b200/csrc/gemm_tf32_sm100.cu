// gemm_tf32_sm100.cu -- tall-skinny TF32 contraction on the 5th-generation tensor cores (sm_100a).
//
//     C[M, N] = A[M, K] * B[N, K]^T          A, B row-major with K contiguous, fp32 in HBM
//
// This is the streaming contraction of a block-order half-step (BASELINE.json north_star group (1)):
//   W half-step:  A = X  (n x d), B = T  (k x d)  ->  X T'   (n x k)
//   T half-step:  A = X' (d x n), B = W' (k x n)  ->  X' W   (d x k)
// N = k <= 256 is tiny, so the kernel is bound by reading A once from HBM; at k = 64 the 32 flop/byte
// it needs (210 TFLOP/s at 6.5 TB/s) is above the FP32 SIMT peak, hence tcgen05.mma kind::tf32.
//
// Design
//   * persistent grid, one CTA per SM, 320 threads = 10 warps: warp 0 TMA producer, warp 1 TMEM owner +
//     single-thread MMA issuer, warps 2-9 epilogue (two per TMEM lane quarter, half of the columns each);
//   * operands staged by TMA (cp.async.bulk.tensor.2d, 128-byte swizzle, zero fill out of bounds) into
//     a ring of NS stages: A stage = MT x 128 rows x 32 fp32, B stage = NPAD rows x 32 fp32.  The B tile
//     (whole factor slab for this K chunk) is shared by the MT row tiles a CTA works on at once, so the
//     factor is re-read from L2 only once per MT*128 rows of A; A uses an evict-first L2 policy, B evict-last;
//   * accumulators live in TMEM: two buffers of MT tiles x 128 lanes x NPAD fp32 columns.  The MMA warp
//     alternates buffers every FLUSH K-chunks (4 x 32 = 128 K); the epilogue warps drain the finished buffer into
//     fp32 registers while the next one fills.  Besides hiding the epilogue this bounds the length of any
//     tensor-core accumulation chain: the MMA accumulator truncates, which over K = 200 000 rows shows as a
//     systematic -6.5e-4 relative bias without a flush, -6.5e-6 with a flush every 1024 K and -6e-7 every 128 K
//     (profiles/r02_tf32_flush_sweep.txt; the shorter period costs 0.6 % of the sweep rate); the register adds are
//     round-to-nearest;
//   * stream-K work split: the (row super-tile, K chunk) units are divided evenly over the CTAs, so every
//     SM streams the same number of bytes whatever M is (no wave quantisation at 157 or 196 tiles).
//     A CTA whose segment covers a full K range writes C directly; first/last partial segments go to a
//     per-CTA slot, and the LAST contributor to arrive at a split tile (a per-tile counter) adds the slots in
//     CTA order and writes the tile (deterministic, no float atomics, no second kernel, nobody waits);
//   * optional auxiliary tile: one more row super-tile whose A operand is a second matrix A2 (in practice the
//     factor itself, so the tile is the k x k Gram matrix B B' of the same half-step) written to its own
//     output -- the Gram product of BASELINE.json's kernel group (2) rides on the streaming contraction
//     instead of costing two more launches per half-step;
//   * 16-bit operands (f16_gemm_run): exact fp16 copies of TF32 values under a power-of-two scale (x16_kernels.cu) go
//     through the same kernel with kind::f16 MMAs -- half the bytes per K, the same swizzle, split, fix-up and flush.
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>

#include "devmem.h"
#include "gemm_tf32_sm100.h"
#include "tc_sm100.cuh"

namespace rri {

namespace {

constexpr int BM = 128;            // rows per UMMA (M of the instruction, cta_group::1)
constexpr int BK = 32;             // fp32 elements per 128-byte swizzle row (64 for 16-bit operands)
constexpr int ROW_BYTES = 128;     // one swizzle row: the K extent of a stage in bytes, whatever the element type
constexpr int FLUSH = 4;            // K-chunks (x32 floats = 128 K) accumulated in TMEM before a flush into registers
constexpr int A_TILE_BYTES = BM * ROW_BYTES;   // 16 KB
constexpr int SMEM_LIMIT = 227 * 1024;

struct GemmParams {
    int64_t M, K;
    int N, NPAD;
    int64_t n_super, nk, units;    // work: n_super row super-tiles (the auxiliary one included) x nk K-chunks
    int64_t n_super_main;          // super-tiles of A; tile index n_super_main (when n_super is one more) reads A2
    float* C;
    int64_t ldc;
    float* C2;                     // output of the auxiliary tile: rows < M2, leading dimension ldc2
    int64_t ldc2;
    int M2;
    float* ws;                     // [grid][2][MT*BM*N] partial slots
    int* ctr;                      // [n_super] arrival counters of split tiles (all zero between launches)
    int stages;
    int tmem_cols;
    int nbuf;                      // TMEM accumulator buffers (2 when 2*MT*NPAD <= 512 columns)
    int flush;                     // K-chunks per TMEM accumulation run
    int reverse_tail;              // tails of split tiles stream K downward (see the producer)
    // 16-bit operands (F16): A holds fp16(a * 2^a_exp), B and A2 fp16(b * 2^(*b_exp)), exponents in [-126, 126]; the
    // epilogue scales the sums back
    int a_exp;
    const int* b_exp;
};

using namespace tc;

// balanced split of `units` over `parts`: first unit of part c
__host__ __device__ __forceinline__ int64_t part_start(int64_t units, int parts, int64_t c)
{
    const int64_t q = units / parts, r = units % parts;
    return c * q + (c < r ? c : r);
}
__host__ __device__ __forceinline__ int64_t part_of(int64_t units, int parts, int64_t u)
{
    const int64_t q = units / parts, r = units % parts;
    if (u < r * (q + 1)) return u / (q + 1);
    return r + (u - r * (q + 1)) / q;
}

// ------------------------------------------------------------------------------------------------
// main kernel
// ------------------------------------------------------------------------------------------------
// EWQ = epilogue warps per TMEM lane quarter (each takes NPAD/EWQ accumulator columns of every tile): 2 for
// k <= 64, 4 for wider ranks so that a thread never holds more than 64 accumulators.
// F16: fp16 operands and tcgen05.mma kind::f16 (fp32 accumulators) instead of fp32 operands rounded to TF32 on the way
// into shared memory.  A stage then holds 64 K-elements per row instead of 32, in the same bytes and the same swizzle.
template <int MT, int NPAD, int EWQ, bool F16>
__global__ void __launch_bounds__(64 + 128 * EWQ, 1)
tf32_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ CUtensorMap tmA2, GemmParams p, int* err)
{
    constexpr int BKE = F16 ? 2 * BK : BK;     // K-elements per chunk (one 128-byte swizzle row)
    constexpr int UK = F16 ? 16 : 8;           // K of one tcgen05.mma: 32 bytes of a row either way
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // carve: [A stages][B stages][barriers][tmem ptr]
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    constexpr int a_stage = MT * A_TILE_BYTES;
    constexpr int b_stage = NPAD * ROW_BYTES;
    uint8_t* smA = smem;
    uint8_t* smB = smem + (size_t)p.stages * a_stage;
    uint64_t* full = reinterpret_cast<uint64_t*>(smB + (size_t)p.stages * b_stage);
    uint64_t* empty = full + p.stages;
    uint64_t* tfull = empty + p.stages;       // [2] accumulator buffer filled
    uint64_t* tempty = tfull + 2;             // [2] accumulator buffer drained
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
    int* fix_info = reinterpret_cast<int*>(tmem_slot + 1);   // [3] arrival order / first / last contributor of a split tile
    const float** fix_src = reinterpret_cast<const float**>(full + 64);    // [<= gridDim.x] slot of every contributor

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t u_begin = part_start(p.units, gridDim.x, blockIdx.x);
    const int64_t u_end = part_start(p.units, gridDim.x, blockIdx.x + 1);

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&tmA);
        prefetch_tmap(&tmB);
        if (p.n_super > p.n_super_main) prefetch_tmap(&tmA2);
        for (int s = 0; s < p.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&tfull[b], 1); mbar_init(&tempty[b], 4 * EWQ); }
        fence_barrier_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(p.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===================================== TMA producer =====================================
        if (lane == 0) {
            const uint64_t polA = policy_evict_first(), polB = policy_evict_last();
            int stage = 0; uint32_t phase = 0;
            for (int64_t u = u_begin; u < u_end;) {
                const int64_t s = u / p.nk, kc0 = u % p.nk;
                const int64_t len = (u_end - u) < (p.nk - kc0) ? (u_end - u) : (p.nk - kc0);
                // K order of a segment: upward -- except, with p.reverse_tail, a segment that does not start at K = 0
                // (the tail of a tile whose head another CTA computes) runs downward from its end.  Every CTA starts
                // with such a tail, so all of them then read the SAME chunks of the factor B at the same time (they all
                // begin at the last chunk) and B is fetched from DRAM once instead of once per tile: with a stream-K
                // split the K offsets of the CTAs are otherwise spread over the whole range, and a 64 MB factor
                // (config 5, T half-step) does not survive in L2 next to the X stream.
                const bool down = p.reverse_tail && kc0 != 0;
                for (int64_t i = 0; i < len; ++i) {
                    const int64_t kc = down ? (kc0 + len - 1 - i) : (kc0 + i);
                    mbar_wait(&empty[stage], phase ^ 1, err, 1);
                    mbar_expect_tx(&full[stage], (uint32_t)(a_stage + b_stage));
                    if (s < p.n_super_main)
                        tma_load_2d(&tmA, smA + (size_t)stage * a_stage, &full[stage], (int)(kc * BKE), (int)(s * MT * BM), polA);
                    else        // auxiliary tile: rows of A2 (rows beyond M2 are zero-filled by TMA)
                        tma_load_2d(&tmA2, smA + (size_t)stage * a_stage, &full[stage], (int)(kc * BKE),
                                    (int)((s - p.n_super_main) * MT * BM), polB);
                    tma_load_2d(&tmB, smB + (size_t)stage * b_stage, &full[stage], (int)(kc * BKE), 0, polB);
                    if (++stage == p.stages) { stage = 0; phase ^= 1; }
                }
                u += len;
            }
        }
    } else if (warp == 1) {
        // ===================================== MMA issuer =======================================
        if (lane == 0) {
            const uint32_t idesc = F16 ? make_idesc_f16(BM, NPAD) : make_idesc_tf32(BM, NPAD);
            int stage = 0; uint32_t phase = 0;
            uint32_t run = 0;                                     // accumulation runs issued so far
            for (int64_t u = u_begin; u < u_end;) {
                const int64_t kc0 = u % p.nk;
                const int64_t len = (u_end - u) < (p.nk - kc0) ? (u_end - u) : (p.nk - kc0);
                for (int64_t i0 = 0; i0 < len; i0 += p.flush, ++run) {
                    const int64_t i1 = (i0 + p.flush) < len ? (i0 + p.flush) : len;
                    const uint32_t b = p.nbuf == 2 ? (run & 1u) : 0u;
                    const uint32_t use = p.nbuf == 2 ? (run >> 1) : run;       // how often buffer b was used before
                    mbar_wait(&tempty[b], (use & 1u) ^ 1u, err, 2);            // epilogue has drained this buffer
                    tc_fence_after();
                    const uint32_t tacc = tmem_base + b * (uint32_t)(MT * NPAD);
                    for (int64_t i = i0; i < i1; ++i) {
                        mbar_wait(&full[stage], phase, err, 3);               // TMA bytes have landed
                        tc_fence_after();
                        const uint32_t a0 = smem_u32(smA + (size_t)stage * a_stage);
                        const uint32_t b0 = smem_u32(smB + (size_t)stage * b_stage);
#pragma unroll
                        for (int mt = 0; mt < MT; ++mt) {
#pragma unroll
                            for (int ks = 0; ks < BKE / UK; ++ks) {
                                const uint64_t ad = make_desc(a0 + mt * A_TILE_BYTES + ks * 32);
                                const uint64_t bd = make_desc(b0 + ks * 32);
                                const uint32_t accum = (i > i0 || ks > 0) ? 1u : 0u;
                                if (F16) umma_f16(tacc + (uint32_t)(mt * NPAD), ad, bd, idesc, accum);
                                else umma_tf32(tacc + (uint32_t)(mt * NPAD), ad, bd, idesc, accum);
                            }
                        }
                        umma_commit(&empty[stage]);               // frees the smem slot when the MMAs retire
                        if (++stage == p.stages) { stage = 0; phase ^= 1; }
                    }
                    umma_commit(&tfull[b]);                       // this accumulation run is complete
                }
                u += len;
            }
        }
    } else {
        // ===================================== epilogue =========================================
        // 4*EWQ warps: warp (q, h) owns TMEM lanes [32q, 32q+32) and columns [h*NPAD/EWQ, (h+1)*NPAD/EWQ) of every tile
        const int q = warp & 3;
        const int h = (warp - 2) >> 2;
        constexpr int HC = NPAD / EWQ;                            // columns per thread and tile
        constexpr int EPI_THREADS = 128 * EWQ;
        constexpr int NACC = MT * HC;
        float acc[NACC];
        uint32_t run = 0;
        const int64_t slot_elems = (int64_t)MT * BM * p.N;
        for (int64_t u = u_begin; u < u_end;) {
            const int64_t s = u / p.nk, kc0 = u % p.nk;
            const int64_t len = (u_end - u) < (p.nk - kc0) ? (u_end - u) : (p.nk - kc0);
            const bool complete = (len == p.nk);
#pragma unroll
            for (int i = 0; i < NACC; ++i) acc[i] = 0.f;
            for (int64_t i0 = 0; i0 < len; i0 += p.flush, ++run) {
                const uint32_t b = p.nbuf == 2 ? (run & 1u) : 0u;
                const uint32_t use = p.nbuf == 2 ? (run >> 1) : run;
                mbar_wait(&tfull[b], use & 1u, err, 4);
                tc_fence_after();
                const uint32_t tacc = tmem_base + ((uint32_t)(q * 32) << 16) + b * (uint32_t)(MT * NPAD) + (uint32_t)(h * HC);
#pragma unroll
                for (int mt = 0; mt < MT; ++mt) {
#pragma unroll
                    for (int c0 = 0; c0 < HC; c0 += 16) {
                        float v[16];
                        tmem_ld16(tacc + (uint32_t)(mt * NPAD + c0), v);
#pragma unroll
                        for (int j = 0; j < 16; ++j) acc[mt * HC + c0 + j] += v[j];     // round-to-nearest fp32 adds
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tempty[b]);
            }
            // ---- the segment is done: a full K range goes straight to its output tile; a partial one goes to this
            // CTA's slot, and whichever contributor arrives last at the tile adds all slots in CTA order
            const bool aux = s >= p.n_super_main;
            if (F16) {
                // undo the operands' power-of-two scales (both exponents lie in [-126, 126]): exact, so slots scaled one
                // by one add up to the scaled sum
                const float sb = __int_as_float((127 - *p.b_exp) << 23);
                const float sa = aux ? sb : __int_as_float((127 - p.a_exp) << 23);
#pragma unroll
                for (int i = 0; i < NACC; ++i) acc[i] = acc[i] * sa * sb;
            }
            float* out = aux ? p.C2 : p.C;
            const int64_t out_ld = aux ? p.ldc2 : p.ldc;
            const int64_t out_row0 = (aux ? s - p.n_super_main : s) * MT * BM;
            const int64_t out_rows = aux ? (int64_t)p.M2 : p.M;
            int c_lo = 0, c_hi = 0;
            if (!complete) {
                const int slot = (u == u_begin) ? 0 : 1;
                float* dst = p.ws + ((int64_t)blockIdx.x * 2 + slot) * slot_elems;
#pragma unroll
                for (int mt = 0; mt < MT; ++mt) {
                    const int row = mt * BM + q * 32 + lane;
#pragma unroll
                    for (int c0 = 0; c0 < HC; c0 += 4) {
                        const int col = h * HC + c0;
                        float* o = dst + (int64_t)row * p.N + col;
                        if ((col + 4 <= p.N) && ((p.N & 3) == 0)) {
                            __stcg(reinterpret_cast<float4*>(o), make_float4(acc[mt * HC + c0], acc[mt * HC + c0 + 1], acc[mt * HC + c0 + 2], acc[mt * HC + c0 + 3]));
                        } else {
#pragma unroll
                            for (int j = 0; j < 4; ++j) if (col + j < p.N) __stcg(o + j, acc[mt * HC + c0 + j]);
                        }
                    }
                }
                __threadfence();                                              // slot visible before the arrival below
                asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS) : "memory");   // the epilogue warps
                if (threadIdx.x == 64) {
                    const int64_t u0 = s * p.nk;
                    const int lo = (int)part_of(p.units, gridDim.x, u0), hi = (int)part_of(p.units, gridDim.x, u0 + p.nk - 1);
                    fix_info[0] = atomicAdd(p.ctr + s, 1);
                    fix_info[1] = lo; fix_info[2] = hi;
                }
                asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS) : "memory");
                c_lo = fix_info[1]; c_hi = fix_info[2];
                if (fix_info[0] == c_hi - c_lo) {                             // every other contributor has arrived
                    __threadfence();
                    // flat, coalesced sum of all contributors' slots (own one included) straight into the output tile
                    const int et = (int)threadIdx.x - 64;
                    const int64_t u0 = s * p.nk;
                    const int ncontrib = c_hi - c_lo + 1;
                    for (int i = et; i < ncontrib; i += EPI_THREADS) {
                        const int64_t cta = c_lo + i;
                        const int cslot = part_start(p.units, gridDim.x, cta) >= u0 ? 0 : 1;
                        fix_src[i] = p.ws + (cta * 2 + cslot) * slot_elems;
                    }
                    asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS) : "memory");
                    const int64_t rows_left = out_rows - out_row0;
                    const int nvalid = (int)(rows_left < (int64_t)MT * BM ? rows_left : (int64_t)MT * BM) * p.N;
                    float* tile = out + out_row0 * out_ld;
                    if (out_ld == p.N && (p.N & 3) == 0) {
                        for (int e = et * 4; e < nvalid; e += EPI_THREADS * 4) {
                            float4 a4 = make_float4(0.f, 0.f, 0.f, 0.f);
                            for (int i = 0; i < ncontrib; ++i) {
                                const float4 v = __ldcg(reinterpret_cast<const float4*>(fix_src[i] + e));
                                a4.x += v.x; a4.y += v.y; a4.z += v.z; a4.w += v.w;
                            }
                            *reinterpret_cast<float4*>(tile + e) = a4;
                        }
                    } else {
                        for (int e = et; e < nvalid; e += EPI_THREADS) {
                            float a1 = 0.f;
                            for (int i = 0; i < ncontrib; ++i) a1 += __ldcg(fix_src[i] + e);
                            const int r = e / p.N, c = e - r * p.N;
                            tile[(int64_t)r * out_ld + c] = a1;
                        }
                    }
                    if (threadIdx.x == 64) p.ctr[s] = 0;                      // ready for the next launch
                }
                asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS) : "memory");   // fix_info / fix_src are reused by the next segment
            }
            if (complete) {
#pragma unroll
                for (int mt = 0; mt < MT; ++mt) {
                    const int64_t row = out_row0 + mt * BM + q * 32 + lane;
                    if (row < out_rows) {
#pragma unroll
                        for (int c0 = 0; c0 < HC; c0 += 4) {
                            const int col = h * HC + c0;
                            float* o = out + row * out_ld + col;
                            if ((col + 4 <= p.N) && ((out_ld & 3) == 0)) {
                                *reinterpret_cast<float4*>(o) = make_float4(acc[mt * HC + c0], acc[mt * HC + c0 + 1], acc[mt * HC + c0 + 2], acc[mt * HC + c0 + 3]);
                            } else {
#pragma unroll
                                for (int j = 0; j < 4; ++j) if (col + j < p.N) o[j] = acc[mt * HC + c0 + j];
                            }
                        }
                    }
                }
            }
            u += len;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

}  // namespace

struct Tf32Gemm {
    int sm_count = 148;
    int nmax = 0;
    EncodeTiledFn encode = nullptr;
    float* ws = nullptr;
    size_t ws_bytes = 0;
    int* err = nullptr;
    CUtensorMapDataType dtype = CU_TENSOR_MAP_DATA_TYPE_TFLOAT32;
    int force_mt = 0;
    int flush = FLUSH;
    int reverse_tail = -1;             // -1: automatic (on for N > 64), 0 / 1: forced by RRI_GEMM_REVERSE_TAIL
    int* ctr = nullptr;
    size_t ctr_len = 0;
};

Tf32Gemm* tf32_gemm_create(int sm_count, int nmax, std::string& err)
{
    Tf32Gemm* g = new Tf32Gemm();
    g->sm_count = sm_count;
    g->nmax = nmax;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) {
        err = "cuTensorMapEncodeTiled is not available from the driver";
        delete g;
        return nullptr;
    }
    g->encode = (EncodeTiledFn)fn;
    // per-CTA partial slots: 2 x (MT*128 x N) floats, MT <= 2
    g->ws_bytes = (size_t)sm_count * 2 * 2 * BM * (size_t)(nmax < 32 ? 32 : nmax) * sizeof(float);
    if (cached_malloc((void**)&g->ws, g->ws_bytes) != cudaSuccess || cached_malloc((void**)&g->err, sizeof(int)) != cudaSuccess) {
        err = "workspace allocation failed";
        delete g;
        return nullptr;
    }
    cudaMemset(g->err, 0, sizeof(int));
    // operand element type seen by TMA: TFLOAT32 (default) or plain FLOAT32 (RRI_TMA_F32=1), for the
    // rounding experiment described in DESIGN.md
    const char* ev = getenv("RRI_TMA_F32");
    if (ev && ev[0] == '1') g->dtype = CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
    const char* mt = getenv("RRI_GEMM_MT");
    if (mt) g->force_mt = atoi(mt);
    const char* rt = getenv("RRI_GEMM_REVERSE_TAIL");
    if (rt) g->reverse_tail = atoi(rt);
    const char* fl = getenv("RRI_GEMM_FLUSH");       // 0 = never flush (one TMEM accumulation per segment)
    if (fl) g->flush = atoi(fl);
    return g;
}

void tf32_gemm_destroy(Tf32Gemm* g)
{
    if (!g) return;
    if (g->ws) cached_free(g->ws);
    if (g->err) cached_free(g->err);
    if (g->ctr) cached_free(g->ctr);
    delete g;
}

// f16: a matrix of fp16 elements (box of 64 per 128-byte row), otherwise fp32 (the handle's TFLOAT32 / FLOAT32 map)
static bool encode_2d(Tf32Gemm* g, CUtensorMap* tm, const void* base, int64_t rows, int64_t cols, int64_t ld,
                      int box_rows, bool f16, std::string& err)
{
    const int es = f16 ? 2 : 4;
    if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || (ld * es) % 16 != 0) {
        err = "TMA needs 16-byte aligned rows (leading dimension a multiple of 16 bytes, base 16-byte aligned)";
        return false;
    }
    cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t gstr[1] = {(cuuint64_t)(ld * es)};
    cuuint32_t box[2] = {(cuuint32_t)(ROW_BYTES / es), (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = g->encode(tm, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : g->dtype, 2, const_cast<void*>(base), gdim, gstr, box,
                           estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        char buf[128];
        snprintf(buf, sizeof(buf), "cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld cols=%lld ld=%lld box=%d)", (int)r,
                 (long long)rows, (long long)cols, (long long)ld, box_rows);
        err = buf;
        return false;
    }
    return true;
}

template <int MT, int NPAD, bool F16>
static int run_cfg(Tf32Gemm* g, const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmA2, GemmParams p,
                   cudaStream_t st, std::string& err)
{
    const int a_stage = MT * A_TILE_BYTES, b_stage = NPAD * ROW_BYTES;
    const int bar_bytes = 4096;       // mbarriers, TMEM slot, fix-up scratch (one slot pointer per CTA of the grid)
    int stages = (SMEM_LIMIT - 1024 /*alignment slack*/ - bar_bytes) / (a_stage + b_stage);
    if (stages > 8) stages = 8;
    if (stages < 2) { err = "not enough shared memory for two pipeline stages"; return -1; }
    p.stages = stages;
    const size_t smem = (size_t)stages * (a_stage + b_stage) + bar_bytes + 1024;
    p.nbuf = (2 * MT * NPAD <= 512) ? 2 : 1;
    int cols = 32;
    while (cols < p.nbuf * MT * NPAD) cols <<= 1;
    p.tmem_cols = cols;
    // the flush period is a K length (RRI_GEMM_FLUSH counts 32-wide chunks): two 64-wide chunks of 16-bit operands
    p.flush = g->flush > 0 ? (F16 ? (g->flush + 1) / 2 : g->flush) : (1 << 30);
    // Measured (profiles/r02_gemm_reverse_tail_ab.txt): the shared B stream wins where B is half of A's traffic (k = 128:
    // T half-step of a config-5 shard 1.91 -> 1.76 ms) and loses where it is a quarter (k = 64: 2.49 -> 2.71 ms; streaming
    // all CTAs through the same columns at the same time costs more than the re-reads it saves).
    p.reverse_tail = g->reverse_tail >= 0 ? g->reverse_tail : (NPAD >= 128 ? 1 : 0);
    int64_t grid = p.units < g->sm_count ? p.units : g->sm_count;
    constexpr int EWQ = NPAD >= 128 ? 4 : 2;
    auto kern = tf32_gemm_kernel<MT, NPAD, EWQ, F16>;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
        err = "cudaFuncSetAttribute(max dynamic smem) failed";
        return -1;
    }
    kern<<<(unsigned)grid, 64 + 128 * EWQ, smem, st>>>(tmA, tmB, tmA2, p, g->err);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { err = cudaGetErrorString(e); return -1; }
    return 1;
}

static int gemm_run(Tf32Gemm* g, bool f16, const void* A, int64_t lda, int a_exp, const void* B, int64_t ldb,
                    const int* b_exp, float* C, int64_t ldc, int64_t M, int N, int64_t K, cudaStream_t st, std::string& err,
                    const void* A2, int64_t lda2, int M2, float* C2, int64_t ldc2)
{
    if (!g) { err = "null contraction handle"; return -1; }
    if (N < 1 || N > 256) { err = "N must be in [1,256]"; return -1; }
    const int npad = N <= 32 ? 32 : (N <= 64 ? 64 : (N <= 128 ? 128 : 256));     // TMEM columns per tile
    if (N > g->nmax && N > 32) { err = "N exceeds the rank this handle was created for"; return -1; }
    int mt = (M > BM) ? 2 : 1;
    if (npad == 256) mt = 1;                     // 128 accumulator registers per epilogue thread at most
    // fewer 256-row super-tiles than CTAs (the T half-step of a row shard: M = d) and a factor B small enough to stay
    // in L2 while twice as many tiles re-read it: 128-row tiles split more evenly -- measured 6-7 us per launch at
    // M = 20 000, N = 64, K = 25 000 / 50 000 (profiles/r02_gemm_tile_height_ab.txt).  At K = 200 000 (B = 51 MB) the
    // doubled re-reads cost 0.16 ms, and N = 128 gains nothing.
    if (npad <= 64 && (M + 2 * BM - 1) / (2 * BM) < g->sm_count && (int64_t)npad * K * 4 <= ((int64_t)16 << 20)) mt = 1;
    if (g->force_mt == 1 || (g->force_mt == 2 && npad < 256)) mt = g->force_mt;
    CUtensorMap tmA, tmB, tmA2;
    if (!encode_2d(g, &tmA, A, M, K, lda, mt * BM, f16, err)) return -1;
    if (!encode_2d(g, &tmB, B, N, K, ldb, npad, f16, err)) return -1;
    const bool aux = A2 != nullptr && M2 > 0 && C2 != nullptr;
    if (aux) { if (!encode_2d(g, &tmA2, A2, M2, K, lda2, mt * BM, f16, err)) return -1; }
    else tmA2 = tmA;
    GemmParams p;
    p.M = M; p.K = K; p.N = N; p.NPAD = npad;
    p.n_super_main = (M + (int64_t)mt * BM - 1) / ((int64_t)mt * BM);
    p.n_super = p.n_super_main + (aux ? (M2 + mt * BM - 1) / (mt * BM) : 0);
    const int bke = f16 ? 2 * BK : BK;
    p.nk = (K + bke - 1) / bke;
    p.units = p.n_super * p.nk;
    p.C = C; p.ldc = ldc; p.ws = g->ws;
    p.C2 = aux ? C2 : C; p.ldc2 = aux ? ldc2 : ldc; p.M2 = aux ? M2 : 0;
    if (p.n_super > (int64_t)g->ctr_len) {
        // arrival counters of split tiles: zero between launches (the last contributor resets its tile's counter)
        if (g->ctr) cached_free(g->ctr);
        g->ctr = nullptr; g->ctr_len = 0;
        const size_t len = (size_t)(p.n_super + 1023) / 1024 * 1024;
        if (cached_malloc((void**)&g->ctr, len * sizeof(int)) != cudaSuccess) { err = "tile counter allocation failed"; return -1; }
        if (cudaMemsetAsync(g->ctr, 0, len * sizeof(int), st) != cudaSuccess) { err = "tile counter reset failed"; return -1; }
        g->ctr_len = len;
    }
    p.ctr = g->ctr;
    p.stages = 0; p.tmem_cols = 0;
    p.nbuf = 1; p.flush = 0;
    p.a_exp = a_exp; p.b_exp = b_exp;
#define RRI_GEMM_CASE(MTv, NP)                                                                              \
    if (mt == MTv && npad == NP)                                                                            \
        return f16 ? run_cfg<MTv, NP, true>(g, tmA, tmB, tmA2, p, st, err) : run_cfg<MTv, NP, false>(g, tmA, tmB, tmA2, p, st, err)
    RRI_GEMM_CASE(2, 32); RRI_GEMM_CASE(2, 64); RRI_GEMM_CASE(2, 128);
    RRI_GEMM_CASE(1, 32); RRI_GEMM_CASE(1, 64); RRI_GEMM_CASE(1, 128); RRI_GEMM_CASE(1, 256);
#undef RRI_GEMM_CASE
    err = "no contraction kernel for this shape";
    return -1;
}

int tf32_gemm_run(Tf32Gemm* g, const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc,
                  int64_t M, int N, int64_t K, cudaStream_t st, std::string& err, const float* A2, int64_t lda2, int M2,
                  float* C2, int64_t ldc2)
{
    return gemm_run(g, false, A, lda, 0, B, ldb, nullptr, C, ldc, M, N, K, st, err, A2, lda2, M2, C2, ldc2);
}

int f16_gemm_run(Tf32Gemm* g, const __half* A, int64_t lda, int a_exp, const __half* B, int64_t ldb, const int* b_exp,
                 float* C, int64_t ldc, int64_t M, int N, int64_t K, cudaStream_t st, std::string& err, const __half* A2,
                 int64_t lda2, int M2, float* C2, int64_t ldc2)
{
    if (!b_exp) { err = "16-bit contraction without the factor's scale"; return -1; }
    return gemm_run(g, true, A, lda, a_exp, B, ldb, b_exp, C, ldc, M, N, K, st, err, A2, lda2, M2, C2, ldc2);
}

}  // namespace rri
