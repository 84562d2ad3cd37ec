// onepass_probe.cu -- streaming skeleton of a one-read-per-sweep block-order pass (sm_100a), for measuring whether L2
// can feed it before the row update that would sit in its middle is built.
//
// One persistent cooperative grid of P x R CTAs: CTA (c, r) owns the column slice [c*w, (c+1)*w) of X16 (n x d fp16,
// row-major) and the row tiles r, r + R, r + 2R, ... (128 rows each).  For its j-th tile a CTA
//   1. reads X[tile, slice] by TMA (128 x 128 fp16 per stage, two 64-column 128-byte-swizzled boxes) and runs
//      MMA1  D1[128 x 64] += X[tile, slice] * T16[:, slice]^T  (kind::f16, both operands K-major, T16 slice resident);
//   2. drains D1 and writes it as this slice's fp32 partial of (X T^T)[tile], then counts the partial in cnt1[tile];
//   3. (--reduce) once all P partials of tile j-L are counted: adds the P partials of 1/P of that tile's rows in slice
//      order into C (the traffic of the reduction a row update needs), then counts that in cnt2[tile];
//   4. after the lag of L tiles, once tile j-L is counted complete (cnt2 with --reduce, else cnt1), reads X[j-L, slice]
//      again together with W16[j-L] (the OLD factor tile stands in for the updated one) and runs
//      MMA2  D2[w x 64] += X[tile, slice]^T * W16[tile]  (M = 128 columns per piece, both operands MN-major: the same
//      swizzled boxes MMA1 reads K-major).  D2 stays in TMEM for the whole launch.
// No row update is done, and D2 is not flushed per tile: the time is the floor of the data movement alone.
// The re-reads either share the first reads' stage ring (one producer thread, one FIFO) or have a ring and a producer
// warp of their own (`sa sb` arguments).
//
// Deadlock freedom (given co-residency, which the cooperative launch guarantees or refuses): a CTA writes and counts its
// partial of tile j before it waits on anything about tile j (its epilogue waits only on tiles j - L, L >= 1); the MMA
// issuer never waits on a global counter, only on the stage rings and the drain; and a producer that waits for tile
// j - L has already issued the first reads of every tile up to j - 1, so every wait is on a tile whose first read every
// CTA has already issued.  Every spin is bounded (~4 s, then the launch fails).
//
// Build:  nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o build/onepass_probe tools/onepass_probe.cu -lcuda
// Run:    build/onepass_probe verify                (small ragged shapes, exact small-integer data, checks C and X^T W)
//         build/onepass_probe time n d w R L reduce hint iters [sa sb]
//             L = 0: no re-read, a plain single streaming pass; hint 1: first read evict-last, 0: no L2 hint;
//             sa, sb: stages of the first-read ring and of a separate re-read ring (default: one shared ring)
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../rri_nmf_b200/csrc/tc_sm100.cuh"

using namespace rri::tc;

#define CK(x)                                                                                   \
    do {                                                                                        \
        cudaError_t e_ = (x);                                                                   \
        if (e_ != cudaSuccess) {                                                                \
            fprintf(stderr, "%s:%d %s: %s\n", __FILE__, __LINE__, #x, cudaGetErrorString(e_)); \
            exit(1);                                                                            \
        }                                                                                       \
    } while (0)

constexpr int K = 64;                       // rank
constexpr int BOX = 64 * 128 * 2;           // 128 rows x 64 fp16 = 16 KB
constexpr int STAGE = 2 * BOX;              // 128 rows x 128 columns
constexpr int TBOX = 64 * 64 * 2;           // 64 rows of T16 x 64 columns = 8 KB
constexpr int NTHREADS = 64 + 128 + 32;     // producer warp, MMA warp, 4 epilogue warps, re-read producer warp

struct Params {
    int64_t n, d;
    int w, np, P, R, L, reduce, reread, hint;
    int ntiles, stages, stagesB, rd;
    float* ws;       // partials: [R][rd][P][64][128]
    int* cnt1;       // [ntiles] partials written
    int* cnt2;       // [ntiles] rows reduced
    float* C;        // [n][64]
    float* D2out;    // [R][d][64]
    int* err;
};

__device__ __forceinline__ int ld_acquire(const int* p)
{
    int v;
    asm volatile("ld.acquire.gpu.global.b32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ void wait_count(const int* p, int target, int* err, int code)
{
    if (ld_acquire(p) >= target) return;
    const long long t0 = clock64();
    while (ld_acquire(p) < target) {
        if (clock64() - t0 > 8000000000LL) {
            atomicExch(err, code);
            __trap();
        }
    }
}
// swizzled shared-memory descriptor with explicit leading / stride byte offsets (K-major: lbo unused, sbo = 1024;
// MN-major: lbo = distance between 64-element atoms along M/N, sbo = distance between 8-row groups along K)
__device__ __forceinline__ uint64_t desc_sw128(uint32_t saddr, uint32_t lbo, uint32_t sbo)
{
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

struct Ring {
    uint8_t* buf;
    uint64_t* full;
    uint64_t* empty;
    int n, stage;
    uint32_t phase;
    __device__ void advance() { if (++stage == n) { stage = 0; phase ^= 1; } }
};

__global__ void __launch_bounds__(NTHREADS, 1)
onepass_probe_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmT,
                     const __grid_constant__ CUtensorMap tmW, Params p)
{
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* smT = smem;                                  // np * 2 boxes of T16
    uint8_t* smW = smT + (size_t)p.np * 2 * TBOX;         // 2 W16 tiles
    uint8_t* smX = smW + 2 * BOX;                         // stages
    uint64_t* full = reinterpret_cast<uint64_t*>(smX + (size_t)(p.stages + p.stagesB) * STAGE);
    uint64_t* empty = full + p.stages;                    // ring B's full / empty follow: full + 2 * stages
    uint64_t* tfull = empty + p.stages + 2 * p.stagesB;   // [2]
    uint64_t* tempty = tfull + 2;                         // [2]
    uint64_t* wfull = tempty + 2;                         // [2]
    uint64_t* wempty = wfull + 2;                         // [2]
    uint64_t* tbar = wempty + 2;                          // T16 slice landed
    uint64_t* done = tbar + 1;                            // every MMA retired
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int c = blockIdx.x % p.P, r = blockIdx.x / p.P;
    const int col0 = c * p.w;
    const int nt = (p.ntiles - r + p.R - 1) / p.R;
    const int L = p.reread ? p.L : 0;
    const int nsteps = nt + L;

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&tmX); prefetch_tmap(&tmT); prefetch_tmap(&tmW);
        for (int s = 0; s < 2 * (p.stages + p.stagesB); ++s) mbar_init(&full[s], 1);
        for (int b = 0; b < 2; ++b) {
            mbar_init(&tfull[b], 1); mbar_init(&tempty[b], 4);
            mbar_init(&wfull[b], 1); mbar_init(&wempty[b], 1);
        }
        mbar_init(tbar, 1); mbar_init(done, 1);
        fence_barrier_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // stage rings: A carries the first reads; B the re-reads when p.stagesB > 0, else they share A (one producer thread)
    Ring ra{smX, full, empty, p.stages, 0, 0};
    Ring rb = p.stagesB ? Ring{smX + (size_t)p.stages * STAGE, full + 2 * p.stages, full + 2 * p.stages + p.stagesB, p.stagesB, 0, 0}
                        : ra;
    if (warp == 0 || warp == 6) {
        if (lane == 0) {
            const uint64_t pol_first = policy_evict_first(), pol_last = policy_evict_last();
            // first read: evict-last (hint 1) to keep it in L2 for the re-read, else no hint (hint 0), or evict-first (no
            // re-read)
            const uint64_t pol = !L ? pol_first : (p.hint ? pol_last : 0);
            auto load_piece = [&](Ring& g, int col, int row, uint64_t pl) {
                mbar_wait(&g.empty[g.stage], g.phase ^ 1, p.err, 1);
                mbar_expect_tx(&g.full[g.stage], STAGE);
                uint8_t* dst = g.buf + (size_t)g.stage * STAGE;
                if (pl) {
                    tma_load_2d(&tmX, dst, &g.full[g.stage], col, row, pl);
                    tma_load_2d(&tmX, dst + BOX, &g.full[g.stage], col + 64, row, pl);
                } else {
                    tma_load_2d(&tmX, dst, &g.full[g.stage], col, row);
                    tma_load_2d(&tmX, dst + BOX, &g.full[g.stage], col + 64, row);
                }
                g.advance();
            };
            int wr = 0;
            auto re_read = [&](Ring& g, int jj) {
                const int tile = r + jj * p.R, row = tile * 128;
                wait_count((p.reduce ? p.cnt2 : p.cnt1) + tile, p.P, p.err, 5);
                const int ws = wr & 1;
                mbar_wait(&wempty[ws], ((wr >> 1) & 1) ^ 1, p.err, 6);
                mbar_expect_tx(&wfull[ws], BOX);
                tma_load_2d(&tmW, smW + (size_t)ws * BOX, &wfull[ws], 0, row, pol_last);
                ++wr;
                // second read: the last use of these bytes
                for (int pc = 0; pc < p.np; ++pc) load_piece(g, col0 + pc * 128, row, pol_first);
            };
            if (warp == 0) {
                mbar_expect_tx(tbar, (uint32_t)(p.np * 2 * TBOX));
                for (int b = 0; b < 2 * p.np; ++b) tma_load_2d(&tmT, smT + (size_t)b * TBOX, tbar, col0 + 64 * b, 0, pol_last);
                for (int j = 0; j < nsteps; ++j) {
                    if (j < nt)
                        for (int pc = 0; pc < p.np; ++pc) load_piece(ra, col0 + pc * 128, (r + j * p.R) * 128, pol);
                    if (!p.stagesB && L > 0 && j >= L) re_read(ra, j - L);
                }
            } else if (p.stagesB && L > 0) {
                for (int j = L; j < nsteps; ++j) re_read(rb, j - L);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc1 = make_idesc_f16(128, K);
            const uint32_t idesc2 = make_idesc_f16(128, K) | (1u << 15) | (1u << 16);     // A and B MN-major
            mbar_wait(tbar, 0, p.err, 2);
            tc_fence_after();
            Ring& g2 = p.stagesB ? rb : ra;
            int wr = 0;
            for (int j = 0; j < nsteps; ++j) {
                if (j < nt) {
                    const uint32_t b = j & 1;
                    mbar_wait(&tempty[b], ((j >> 1) & 1) ^ 1, p.err, 3);
                    tc_fence_after();
                    const uint32_t d1 = tmem_base + b * K;
                    for (int pc = 0; pc < p.np; ++pc) {
                        mbar_wait(&ra.full[ra.stage], ra.phase, p.err, 4);
                        tc_fence_after();
                        const uint32_t a0 = smem_u32(ra.buf + (size_t)ra.stage * STAGE);
                        for (int h = 0; h < 2; ++h)
                            for (int ks = 0; ks < 4; ++ks)
                                umma_f16(d1, desc_sw128(a0 + h * BOX + ks * 32, 16, 1024),
                                         desc_sw128(smem_u32(smT + (size_t)(2 * pc + h) * TBOX) + ks * 32, 16, 1024), idesc1,
                                         (pc | h | ks) ? 1u : 0u);
                        umma_commit(&ra.empty[ra.stage]);
                        ra.advance();
                    }
                    umma_commit(&tfull[b]);
                }
                if (L > 0 && j >= L) {
                    const int ws = wr & 1;
                    mbar_wait(&wfull[ws], (wr >> 1) & 1, p.err, 7);
                    tc_fence_after();
                    const uint32_t w0 = smem_u32(smW + (size_t)ws * BOX);
                    for (int pc = 0; pc < p.np; ++pc) {
                        mbar_wait(&g2.full[g2.stage], g2.phase, p.err, 4);
                        tc_fence_after();
                        const uint32_t a0 = smem_u32(g2.buf + (size_t)g2.stage * STAGE);
                        const uint32_t d2 = tmem_base + 2 * K + pc * K;
                        for (int ks = 0; ks < 8; ++ks)       // 16 rows of the tile per MMA
                            umma_f16(d2, desc_sw128(a0 + ks * 2048, BOX, 1024), desc_sw128(w0 + ks * 2048, BOX, 1024), idesc2,
                                     (j > L || ks > 0) ? 1u : 0u);
                        umma_commit(&g2.empty[g2.stage]);
                        g2.advance();
                    }
                    umma_commit(&wempty[ws]);
                    ++wr;
                }
            }
            umma_commit(done);
        }
    } else if (warp < 6) {
        const int q = warp & 3;
        const int row = q * 32 + lane;                    // TMEM lane = row of the tile
        const int et = threadIdx.x - 64;
        float* ws_cta = p.ws;
        auto slot = [&](int jj, int cc) { return ws_cta + ((((int64_t)r * p.rd + jj % p.rd) * p.P + cc) * K) * 128; };
        const int rpc = (128 + p.P - 1) / p.P;           // rows of a tile this CTA reduces
        auto reduce_tile = [&](int jj) {
            const int tile = r + jj * p.R;
            if (et == 0) wait_count(p.cnt1 + tile, p.P, p.err, 8);
            asm volatile("bar.sync 1, 128;" ::: "memory");
            const int r0 = c * rpc, r1 = min(128, r0 + rpc);
            for (int e = et; e < (r1 - r0) * K; e += 128) {
                const int rr = r0 + e % (r1 - r0), col = e / (r1 - r0);
                float s = 0.f;
                for (int cc = 0; cc < p.P; ++cc) s += __ldcg(slot(jj, cc) + col * 128 + rr);
                const int64_t grow = (int64_t)tile * 128 + rr;
                if (grow < p.n) p.C[grow * K + col] = s;
            }
            __threadfence();
            asm volatile("bar.sync 1, 128;" ::: "memory");
            if (et == 0) atomicAdd(p.cnt2 + tile, 1);
        };
        for (int j = 0; j < nsteps; ++j) {
            if (j < nt) {
                const uint32_t b = j & 1;
                mbar_wait(&tfull[b], (j >> 1) & 1, p.err, 9);
                tc_fence_after();
                const uint32_t t = tmem_base + ((uint32_t)(q * 32) << 16) + b * K;
                float v[K];
                for (int c0 = 0; c0 < K; c0 += 16) tmem_ld16(t + c0, v + c0);
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tempty[b]);
                float* dst = slot(j, c);
#pragma unroll
                for (int col = 0; col < K; ++col) __stcg(dst + col * 128 + row, v[col]);
                __threadfence();
                asm volatile("bar.sync 1, 128;" ::: "memory");
                if (et == 0) atomicAdd(p.cnt1 + r + j * p.R, 1);
            }
            if (p.reduce && L > 0 && j >= L) reduce_tile(j - L);
        }
        // D2 -> global, once every MMA has retired
        mbar_wait(done, 0, p.err, 10);
        tc_fence_after();
        if (L > 0) {
            for (int pc = 0; pc < p.np; ++pc) {
                const uint32_t t = tmem_base + ((uint32_t)(q * 32) << 16) + 2 * K + pc * K;
                float v[K];
                for (int c0 = 0; c0 < K; c0 += 16) tmem_ld16(t + c0, v + c0);
                const int64_t gcol = (int64_t)col0 + pc * 128 + row;
                if (pc * 128 + row < p.w && gcol < p.d)
                    for (int k = 0; k < K; ++k) p.D2out[((int64_t)r * p.d + gcol) * K + k] = v[k];
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
    }
}

// small integers / 4 in [0, 0.75]: exact in fp16, and every product sum of this probe is exact in fp32
__global__ void fill_kernel(__half* a, int64_t count, uint32_t seed)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
        uint32_t h = (uint32_t)i * 2654435761u ^ seed;
        h ^= h >> 15; h *= 2246822519u; h ^= h >> 13;
        a[i] = __float2half(0.25f * (float)(h & 3u));
    }
}

typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                             const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                             CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeFn encode;

static CUtensorMap map2d(const __half* base, int64_t rows, int64_t cols, int box_rows)
{
    CUtensorMap tm;
    cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t gstr[1] = {(cuuint64_t)(cols * 2)};
    cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult e = encode(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<__half*>(base), gdim, gstr, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (e != CUDA_SUCCESS) { fprintf(stderr, "tensor map encode failed (%d)\n", (int)e); exit(1); }
    return tm;
}

struct Run {
    int64_t n, d;
    Params p;
    __half *X, *T, *W;
    CUtensorMap tmX, tmT, tmW;
    size_t smem;
};

static Run setup(int64_t n, int64_t d, int w, int R, int L, int reduce, int hint, int sa, int sb)
{
    Run u;
    u.n = n; u.d = d;
    Params& p = u.p;
    p.n = n; p.d = d; p.w = w; p.np = w / 128; p.R = R; p.L = L; p.reduce = reduce; p.reread = L > 0; p.hint = hint;
    p.P = (int)((d + w - 1) / w);
    p.ntiles = (int)((n + 127) / 128);
    p.rd = L + 2;
    const size_t fixed = (size_t)p.np * 2 * TBOX + 2 * BOX + 1024 /*barriers*/ + 1024 /*alignment*/;
    // sa = 0: as many stages as fit, one ring; else sa stages in ring A and sb in ring B (re-reads)
    p.stages = sa ? sa : (int)std::min<size_t>(8, (227 * 1024 - fixed) / STAGE);
    p.stagesB = sa ? sb : 0;
    u.smem = fixed + (size_t)(p.stages + p.stagesB) * STAGE;
    if (u.smem > 227 * 1024) { fprintf(stderr, "%zu bytes of shared memory do not fit\n", u.smem); exit(2); }
    CK(cudaMalloc(&u.X, n * d * 2));
    CK(cudaMalloc(&u.T, (size_t)K * d * 2));
    CK(cudaMalloc(&u.W, (size_t)n * K * 2));
    fill_kernel<<<1024, 256>>>(u.X, n * d, 0x1234u);
    fill_kernel<<<256, 256>>>(u.T, (int64_t)K * d, 0x777u);
    fill_kernel<<<256, 256>>>(u.W, n * K, 0x4242u);
    CK(cudaMalloc(&p.ws, (size_t)R * p.rd * p.P * K * 128 * 4));
    CK(cudaMalloc(&p.cnt1, (size_t)p.ntiles * 4));
    CK(cudaMalloc(&p.cnt2, (size_t)p.ntiles * 4));
    CK(cudaMalloc(&p.C, (size_t)n * K * 4));
    CK(cudaMalloc(&p.D2out, (size_t)R * d * K * 4));
    CK(cudaMalloc(&p.err, 4));
    CK(cudaMemset(p.err, 0, 4));
    CK(cudaMemset(p.C, 0, (size_t)n * K * 4));
    CK(cudaMemset(p.D2out, 0, (size_t)R * d * K * 4));
    u.tmX = map2d(u.X, n, d, 128);
    u.tmT = map2d(u.T, K, d, 64);
    u.tmW = map2d(u.W, n, K, 128);
    CK(cudaFuncSetAttribute(onepass_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)u.smem));
    CK(cudaDeviceSynchronize());
    return u;
}

static void launch(Run& u)
{
    CK(cudaMemsetAsync(u.p.cnt1, 0, (size_t)u.p.ntiles * 4));
    CK(cudaMemsetAsync(u.p.cnt2, 0, (size_t)u.p.ntiles * 4));
    void* args[] = {&u.tmX, &u.tmT, &u.tmW, &u.p};
    CK(cudaLaunchCooperativeKernel((const void*)onepass_probe_kernel, dim3(u.p.P * u.p.R), dim3(NTHREADS), args, u.smem, 0));
}

static void release(Run& u)
{
    cudaFree(u.X); cudaFree(u.T); cudaFree(u.W);
    cudaFree(u.p.ws); cudaFree(u.p.cnt1); cudaFree(u.p.cnt2); cudaFree(u.p.C); cudaFree(u.p.D2out); cudaFree(u.p.err);
}

static int verify(int64_t n, int64_t d, int w, int R, int L, int sa = 0, int sb = 0)
{
    Run u = setup(n, d, w, R, L, 1, 1, sa, sb);
    launch(u);
    CK(cudaDeviceSynchronize());
    std::vector<__half> X(n * d), T((size_t)K * d), W((size_t)n * K);
    std::vector<float> C((size_t)n * K), D2((size_t)R * d * K);
    CK(cudaMemcpy(X.data(), u.X, X.size() * 2, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(T.data(), u.T, T.size() * 2, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(W.data(), u.W, W.size() * 2, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(C.data(), u.p.C, C.size() * 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(D2.data(), u.p.D2out, D2.size() * 4, cudaMemcpyDeviceToHost));
    std::vector<float> Xf(X.size()), Tf(T.size()), Wf(W.size());
    for (size_t i = 0; i < X.size(); ++i) Xf[i] = __half2float(X[i]);
    for (size_t i = 0; i < T.size(); ++i) Tf[i] = __half2float(T[i]);
    for (size_t i = 0; i < W.size(); ++i) Wf[i] = __half2float(W[i]);
    int64_t bad_c = 0, bad_d = 0;
    for (int64_t i = 0; i < n; ++i)
        for (int k = 0; k < K; ++k) {
            double s = 0;
            for (int64_t j = 0; j < d; ++j) s += (double)Xf[i * d + j] * Tf[(size_t)k * d + j];
            if ((double)C[i * K + k] != s) ++bad_c;
        }
    for (int64_t j = 0; j < d; ++j)
        for (int k = 0; k < K; ++k) {
            double s = 0, g = 0;
            for (int64_t i = 0; i < n; ++i) s += (double)Xf[i * d + j] * Wf[i * K + k];
            for (int rr = 0; rr < R; ++rr) g += D2[((size_t)rr * d + j) * K + k];
            if (g != s) ++bad_d;
        }
    printf("verify n=%lld d=%lld w=%d R=%d L=%d P=%d rings=%d+%d: C mismatches %lld of %lld, X^T W mismatches %lld of %lld\n",
           (long long)n, (long long)d, w, R, L, u.p.P, u.p.stages, u.p.stagesB, (long long)bad_c, (long long)(n * K), (long long)bad_d,
           (long long)(d * K));
    release(u);
    return (bad_c || bad_d) ? 1 : 0;
}

int main(int argc, char** argv)
{
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    CK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
    if (!fn || q != cudaDriverEntryPointSuccess) { fprintf(stderr, "no cuTensorMapEncodeTiled\n"); return 1; }
    encode = (EncodeFn)fn;
    if (argc >= 2 && std::string(argv[1]) == "verify") {
        int bad = 0;
        bad |= verify(129, 520, 256, 2, 1);
        bad |= verify(1000, 520, 128, 3, 2);
        bad |= verify(16384 + 77, 2000, 384, 2, 4);
        bad |= verify(16384 + 77, 2000, 512, 3, 2, 2, 2);
        printf(bad ? "VERIFY FAILED\n" : "VERIFY OK\n");
        return bad;
    }
    if (argc < 10) { fprintf(stderr, "usage: %s verify | time n d w R L reduce hint iters\n", argv[0]); return 2; }
    const int64_t n = atoll(argv[2]), d = atoll(argv[3]);
    const int w = atoi(argv[4]), R = atoi(argv[5]), L = atoi(argv[6]), reduce = atoi(argv[7]), hint = atoi(argv[8]),
              iters = atoi(argv[9]);
    if (w % 128 || w / 128 > 6) { fprintf(stderr, "w must be a multiple of 128, at most 768\n"); return 2; }
    const int sa = argc > 10 ? atoi(argv[10]) : 0, sb = argc > 11 ? atoi(argv[11]) : 0;
    Run u = setup(n, d, w, R, L, reduce, hint, sa, sb);
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    for (int i = 0; i < 3; ++i) launch(u);
    CK(cudaDeviceSynchronize());
    std::vector<float> ms;
    for (int i = 0; i < iters; ++i) {
        CK(cudaEventRecord(e0));
        launch(u);
        CK(cudaEventRecord(e1));
        CK(cudaEventSynchronize(e1));
        float t; CK(cudaEventElapsedTime(&t, e0, e1));
        ms.push_back(t);
    }
    std::sort(ms.begin(), ms.end());
    const double med = ms[ms.size() / 2];
    const double xbytes = (double)n * d * 2;
    const double tile_mb = 128.0 * d * 2 / 1e6;
    printf("{\"n\": %lld, \"d\": %lld, \"w\": %d, \"P\": %d, \"R\": %d, \"ctas\": %d, \"L\": %d, \"reduce\": %d, \"hint\": %d, \"stages\": %d, \"stagesB\": %d, "
           "\"window_MB\": %.1f, \"ms_median\": %.4f, \"ms_min\": %.4f, \"ms_max\": %.4f, \"x_hbm_TBps\": %.3f, "
           "\"x_reads_TBps\": %.3f}\n",
           (long long)n, (long long)d, w, u.p.P, R, u.p.P * R, L, reduce, hint, u.p.stages, u.p.stagesB, R * (L + 1) * tile_mb, med, ms[0],
           ms.back(), xbytes / med / 1e9, (L > 0 ? 2 : 1) * xbytes / med / 1e9);
    release(u);
    return 0;
}
