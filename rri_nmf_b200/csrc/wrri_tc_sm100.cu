// wrri_tc_sm100.cu -- masked / weighted WRRI half-step statistics with the W T product on the tensor
// cores (sm_100a, fp32 data, TF32 operands).
//
// Reference arithmetic (src/rri_nmf/nmf.py:687-701 and :735-746), for topic t:
//     R      = M o (X - W_{t->0} T)                                   (never materialised here)
//     T-step : numer[c] = sum_i W[i,t] R[i,c]      denom[c] = sum_i W[i,t]^2 M[i,c]
//     W-step : numer[i] = sum_c R[i,c] T[t,c]      denom[i] = sum_c M[i,c] T[t,c]^2
// The SIMT kernels of wrri_kernels.cu spend k FMAs per matrix element on the CUDA cores.  Here every
// 128x128 tile of W T is one burst of tcgen05.mma kind::tf32 (K = k padded to 32) into TMEM; the
// epilogue warps move it to shared memory and then walk X and the mask in their own row-major,
// fully coalesced order, adding topic t back in fp32 (W_{t->0}T = WT - w_t T_t).  With a sparse
// mask the X loads of all-masked 16-byte groups are skipped, so the pass reads the mask once and only
// the observed neighbourhood of X.  Tiles are 128x64 so that two CTAs share an SM.
//
// Operands are engine-owned zero-padded copies Wp[n, KP], Tp[d, KP] (K-contiguous rows of KP = k
// rounded up to 32 floats -> legal TMA rows and whole 128-byte swizzle atoms).
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdio.h>

#include "devmem.h"
#include "kernels.h"
#include "tc_sm100.cuh"
#include "wrri_tc_sm100.h"

namespace rri {

namespace {

constexpr int TM = 128, TN = 64;           // tile: rows of X x columns of X (two CTAs per SM: a second tile
                                           // is in flight while this one waits on its loads)
constexpr int BK = 32;                     // floats per 128-byte swizzle row
constexpr int UK = 8;
constexpr int EPI_WARPS = 8;
constexpr int THREADS = 32 * (1 + EPI_WARPS);
constexpr int DS_LD = TN + 4;              // padded row stride of the staged product tile (floats)
constexpr int W_CHUNK_BYTES = TM * BK * 4;    // one 32-float K chunk of the 128-row W tile: 16 KB
constexpr int T_CHUNK_BYTES = TN * BK * 4;    // one 32-float K chunk of the  64-row T' tile:  8 KB
constexpr int ROWS_PER_THREAD = 8;            // element-wise pass: 128x64 tile / 256 threads / 4 columns

struct TcParams {
    const float* X; int64_t ldx;
    const void* M; int64_t ldm;
    const float* Wp; const float* Tp;      // padded operand copies [n,KP], [d,KP]
    const float* Tt;                       // T[t, :] of the caller's factor (contiguous row), TMA variant
    int64_t n, d;
    int KP, t;
    int tiles_r, tiles_c;                  // number of 128-row / 128-column tiles
    int groups;                            // T mode: row groups per column tile; W mode: column groups per row tile
    float* numer_part; float* denom_part;  // [groups][d] (T mode) or [groups][n] (W mode)
    int stages;
    int xm_stages;                         // TMA ring depth of the X / mask tiles (TMA variant)
};

using namespace tc;

__device__ __forceinline__ void epi_barrier()     // named barrier 1: the 8 epilogue warps only
{
    asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
}

// raw mask word(s) of one 16-byte X group: one 32-bit word of 4 bytes (u8) or one float4 (real weights)
template <int MK> struct MaskRaw;
template <> struct MaskRaw<MK_U8> {
    uint32_t w;
    __device__ __forceinline__ void load(const void* M, int64_t idx, bool ok)
    {
        w = ok ? __ldg(reinterpret_cast<const uint32_t*>(reinterpret_cast<const unsigned char*>(M) + idx)) : 0u;
    }
    __device__ __forceinline__ bool any() const { return w != 0u; }
    __device__ __forceinline__ void decode(float m[4]) const
    {
        m[0] = (float)(w & 0xffu); m[1] = (float)((w >> 8) & 0xffu); m[2] = (float)((w >> 16) & 0xffu); m[3] = (float)(w >> 24);
    }
};
template <> struct MaskRaw<MK_REAL> {
    float4 v;
    __device__ __forceinline__ void load(const void* M, int64_t idx, bool ok)
    {
        v = ok ? __ldcs(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(M) + idx)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __device__ __forceinline__ bool any() const { return (v.x != 0.f) | (v.y != 0.f) | (v.z != 0.f) | (v.w != 0.f); }
    __device__ __forceinline__ void decode(float m[4]) const { m[0] = v.x; m[1] = v.y; m[2] = v.z; m[3] = v.w; }
};

// MODE 0: T-step statistics (column sums; CTA = one 64-column tile x one group of 128-row tiles)
// MODE 1: W-step statistics (row sums;    CTA = one 128-row tile   x one group of 64-column tiles)
// 288 threads: warp 0 = TMA + MMA control, warps 1-8 = epilogue.  Two CTAs are resident per SM.
template <int MODE, int MK>
__global__ void __launch_bounds__(THREADS, 2)
wrri_tc_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmT, TcParams p)
{
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const int nchunk = p.KP / BK;
    const int w_bytes = nchunk * W_CHUNK_BYTES, t_bytes = nchunk * T_CHUNK_BYTES;     // W tile 128 rows, T' tile 64 rows
    const int fixed_bytes = MODE == 0 ? t_bytes : w_bytes;
    const int var_bytes = MODE == 0 ? w_bytes : t_bytes;
    const int var_chunk = MODE == 0 ? W_CHUNK_BYTES : T_CHUNK_BYTES;
    const int fixed_chunk = MODE == 0 ? T_CHUNK_BYTES : W_CHUNK_BYTES;
    uint8_t* sm_fixed = smem;                               // the operand that stays for the whole CTA
    uint8_t* sm_var = smem + fixed_bytes;                   // [stages] the operand that changes per tile
    float* Ds = reinterpret_cast<float*>(sm_var + (size_t)p.stages * var_bytes);      // [TM][DS_LD]
    uint64_t* bars = reinterpret_cast<uint64_t*>(Ds + TM * DS_LD);
    uint64_t* fixed_full = bars;            // 1
    uint64_t* var_full = bars + 1;          // [2]
    uint64_t* var_free = bars + 3;          // [2]
    uint64_t* acc_full = bars + 5;          // [2]
    uint64_t* acc_free = bars + 7;          // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int fixed_tile = blockIdx.x;      // column tile (MODE 0) / row tile (MODE 1)
    const int nvar_total = MODE == 0 ? p.tiles_r : p.tiles_c;
    int vb, ve;
    {
        const int q = nvar_total / (int)gridDim.y, r = nvar_total % (int)gridDim.y, g = blockIdx.y;
        vb = q * g + (g < r ? g : r);
        ve = vb + q + (g < r ? 1 : 0);
    }
    const int ntiles = ve - vb;
    const int var_rows = MODE == 0 ? TM : TN, fixed_rows = MODE == 0 ? TN : TM;       // rows per tile of each operand

    if (threadIdx.x == 0) {
        mbar_init(fixed_full, 1);
        for (int s = 0; s < 2; ++s) { mbar_init(&var_full[s], 1); mbar_init(&var_free[s], 1); mbar_init(&acc_full[s], 1); mbar_init(&acc_free[s], 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(128) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ================================ TMA + MMA control thread ================================
        if (lane == 0 && ntiles > 0) {
            const CUtensorMap* tm_fixed = MODE == 0 ? &tmT : &tmW;     // MODE 0: the column tile of T' is fixed
            const CUtensorMap* tm_var = MODE == 0 ? &tmW : &tmT;
            mbar_expect_tx(fixed_full, (uint32_t)fixed_bytes);
            for (int c = 0; c < nchunk; ++c) tma_load_2d(tm_fixed, sm_fixed + c * fixed_chunk, fixed_full, c * BK, fixed_tile * fixed_rows);
            const int S = p.stages;
            for (int s0 = 0; s0 < S && s0 < ntiles; ++s0) {           // prologue: fill the ring
                mbar_expect_tx(&var_full[s0], (uint32_t)var_bytes);
                for (int c = 0; c < nchunk; ++c)
                    tma_load_2d(tm_var, sm_var + (size_t)s0 * var_bytes + c * var_chunk, &var_full[s0], c * BK, (vb + s0) * var_rows);
            }
            mbar_wait(fixed_full, 0);
            // D[128 rows of X, 64 columns of X] = W tile (A, M = 128) x T' tile (B, N = 64), TF32 in, FP32 out
            const uint32_t idesc = make_idesc_tf32(TM, TN);
            for (int n = 0; n < ntiles; ++n) {
                const int s = n % S, a = n & 1;
                mbar_wait(&var_full[s], (n / S) & 1);
                mbar_wait(&acc_free[a], ((n >> 1) & 1) ^ 1);
                tc_fence_after();
                const uint32_t var0 = smem_u32(sm_var + (size_t)s * var_bytes), fix0 = smem_u32(sm_fixed);
                const uint32_t w0 = MODE == 0 ? var0 : fix0;      // W tile (A)
                const uint32_t t0 = MODE == 0 ? fix0 : var0;      // T' tile (B)
                for (int c = 0; c < nchunk; ++c) {
#pragma unroll
                    for (int ks = 0; ks < BK / UK; ++ks) {
                        umma_tf32(tmem_base + (uint32_t)(a * TN), make_desc(w0 + c * W_CHUNK_BYTES + ks * UK * 4),
                                  make_desc(t0 + c * T_CHUNK_BYTES + ks * UK * 4), idesc, (c > 0 || ks > 0) ? 1u : 0u);
                    }
                }
                umma_commit(&var_free[s]);
                umma_commit(&acc_full[a]);
                if (n + S < ntiles) {
                    // refill this stage for tile n+S once the MMAs that read it have retired
                    mbar_wait(&var_free[s], (n / S) & 1);
                    mbar_expect_tx(&var_full[s], (uint32_t)var_bytes);
                    for (int c = 0; c < nchunk; ++c)
                        tma_load_2d(tm_var, sm_var + (size_t)s * var_bytes + c * var_chunk, &var_full[s], c * BK, (vb + n + S) * var_rows);
                }
            }
        }
    } else {
        // ======================================= epilogue ========================================
        const int ew = warp - 1;                 // 0..7
        const int q = warp & 3;                  // TMEM lane quarter this warp may read
        // coalesced element-wise mapping: 16 lanes x 4 columns cover the 64 columns of a row; a warp takes
        // two rows per step, warp ew owns rows 2*ew + (lane >> 4) + 16*rr
        constexpr int R = ROWS_PER_THREAD;
        const int cl = 4 * (lane & 15);
        const int rsub = 2 * ew + (lane >> 4);
        float nacc[MODE == 0 ? 4 : R], dacc[MODE == 0 ? 4 : R];
#pragma unroll
        for (int i = 0; i < (MODE == 0 ? 4 : R); ++i) { nacc[i] = 0.f; dacc[i] = 0.f; }

        for (int n = 0; n < ntiles; ++n) {
            const int a = n & 1;
            const int rt = MODE == 0 ? (vb + n) : fixed_tile;         // row tile
            const int ctile = MODE == 0 ? fixed_tile : (vb + n);      // column tile
            const int64_t i0 = (int64_t)rt * TM, c0 = (int64_t)ctile * TN;
            const int64_t gc = c0 + cl;
            const bool cok = gc < p.d;                                // d % 4 == 0 is required by the launcher
            // the masks do not depend on the product tile: request them before blocking on the MMA
            MaskRaw<MK> mr[R];
#pragma unroll
            for (int rr = 0; rr < R; ++rr) {
                const int64_t gi = i0 + rsub + 16 * rr;
                mr[rr].load(p.M, gi * p.ldm + gc, cok && gi < p.n);
            }
            float tt[4] = {0.f, 0.f, 0.f, 0.f};
            if (cok) {
#pragma unroll
                for (int v = 0; v < 4; ++v) tt[v] = __ldg(p.Tp + (gc + v) * p.KP + p.t);
            }
            mbar_wait(&acc_full[a], (n >> 1) & 1);
            tc_fence_after();
            {   // TMEM -> shared: the two warps of a lane quarter take 32 columns each
                const int half = (warp - 1) >> 2;                     // warps 1-4 -> 0, warps 5-8 -> 1
                const int row = q * 32 + lane;
#pragma unroll
                for (int cc = 0; cc < 32; cc += 16) {
                    float v[16];
                    const int col = half * 32 + cc;
                    tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(a * TN + col), v);
                    float4* o = reinterpret_cast<float4*>(Ds + row * DS_LD + col);
                    o[0] = make_float4(v[0], v[1], v[2], v[3]);
                    o[1] = make_float4(v[4], v[5], v[6], v[7]);
                    o[2] = make_float4(v[8], v[9], v[10], v[11]);
                    o[3] = make_float4(v[12], v[13], v[14], v[15]);
                }
            }
            // observed X groups of this tile: all rows' loads in flight together (one round trip), issued
            // before the barrier so that part of their latency hides behind it.  (Loading X unconditionally,
            // without waiting for the mask, was measured slower: 0.54 s vs 0.40 s per config-4 sweep.)
            float4 xv[R];
            float wts[R];
#pragma unroll
            for (int rr = 0; rr < R; ++rr) {
                const int64_t gi = i0 + rsub + 16 * rr;
                xv[rr] = make_float4(0.f, 0.f, 0.f, 0.f);
                wts[rr] = 0.f;
                if (mr[rr].any()) {
                    xv[rr] = __ldcs(reinterpret_cast<const float4*>(p.X + gi * p.ldx + gc));
                    wts[rr] = __ldg(p.Wp + gi * p.KP + p.t);
                }
            }
            tc_fence_before();
            epi_barrier();                                            // product tile staged; TMEM reads done
            if (lane == 0 && ew < 4) mbar_arrive(&acc_free[a]);

            // ---- element-wise pass in X's own layout
#pragma unroll
            for (int rr = 0; rr < R; ++rr) {
                if (mr[rr].any()) {
                    const int r = rsub + 16 * rr;
                    float m[4];
                    mr[rr].decode(m);
                    const float4 dv = *reinterpret_cast<const float4*>(Ds + r * DS_LD + cl);
                    const float wt = wts[rr];
                    const float x[4] = {xv[rr].x, xv[rr].y, xv[rr].z, xv[rr].w};
                    const float dd[4] = {dv.x, dv.y, dv.z, dv.w};
#pragma unroll
                    for (int v = 0; v < 4; ++v) {
                        const float res = m[v] * (x[v] - dd[v] + wt * tt[v]);          // M o (X - W_{t->0} T)
                        if (MODE == 0) {
                            nacc[v] = fmaf(wt, res, nacc[v]);
                            dacc[v] = fmaf(wt * wt, m[v], dacc[v]);
                        } else {
                            nacc[rr] = fmaf(res, tt[v], nacc[rr]);
                            dacc[rr] = fmaf(m[v] * tt[v], tt[v], dacc[rr]);
                        }
                    }
                }
            }
            epi_barrier();                                            // Ds may be overwritten by the next tile
        }

        // ---- reductions and partial output
        if (MODE == 0) {
            // column sums: 16 thread rows (8 warps x 2 half-warps) per column, added through shared memory
            float* red = Ds;                                          // [16][2][TN]
            const int slot = 2 * ew + (lane >> 4);
#pragma unroll
            for (int v = 0; v < 4; ++v) {
                red[(slot * 2 + 0) * TN + cl + v] = nacc[v];
                red[(slot * 2 + 1) * TN + cl + v] = dacc[v];
            }
            epi_barrier();
            const int e = threadIdx.x - 32;                           // 0..255
            if (e < 2 * TN) {
                const int which = e / TN, cc = e % TN;
                float s = 0.f;
#pragma unroll
                for (int w = 0; w < 16; ++w) s += red[(w * 2 + which) * TN + cc];
                const int64_t gcol = (int64_t)fixed_tile * TN + cc;
                if (gcol < p.d) (which ? p.denom_part : p.numer_part)[(int64_t)blockIdx.y * p.d + gcol] = s;
            }
        } else {
            // row sums: the 16 lanes that share a row hold partials over their column slices
#pragma unroll
            for (int rr = 0; rr < R; ++rr) {
                float a = nacc[rr], b = dacc[rr];
#pragma unroll
                for (int o = 8; o > 0; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
                const int64_t gi = (int64_t)fixed_tile * TM + rsub + 16 * rr;
                if ((lane & 15) == 0 && gi < p.n) {
                    p.numer_part[(int64_t)blockIdx.y * p.n + gi] = a;
                    p.denom_part[(int64_t)blockIdx.y * p.n + gi] = b;
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(128) : "memory");
    }
}


// ------------------------------------------------------------------------------------------------
// TMA-staged variant (default).  Warp 0 = MMA issue, warp 1 = operand producer (the W / T' tile that changes with
// the tile, ring of 2), warp 2 = producer that streams the X tile and the mask tile through a ring of shared-memory
// stages several tiles ahead, warps 3-18 = epilogue.  One CTA per SM.  (With the operand refill issued by the MMA
// thread itself -- after waiting for its MMAs to retire -- the epilogue spent 37 % of its samples waiting for the
// next accumulator: profiles/r02_ncu_masked_v2.txt.)
//
// Epilogue without block barriers: epilogue warp (q, g) owns rows [32q, 32q+32) x columns [16g, 16g+16) of every
// 128 x 64 tile.  It reads exactly that block of the product straight from TMEM into registers (one tcgen05.ld,
// lane = row), the same elements of X from the stage -- written by TMA as two 32-column boxes with the 128-byte
// swizzle, so that a row-per-lane 16-byte read is bank-conflict free -- and of the mask, keeps its partial sums in
// registers across ALL tiles of the CTA, and hands the TMEM buffer and the stage back with one mbarrier arrival per
// warp.  Warps drift across the two accumulator buffers and the ring stages instead of marching in lockstep; the
// cross-warp reduction happens once per CTA.  (The previous version staged the product through shared memory between
// two 512-thread barriers per tile: ~3400 cycles per tile where the HBM rate needs ~1750.)
// ------------------------------------------------------------------------------------------------
constexpr int EPI_WARPS_TMA = 16;                    // 4 warps per TMEM lane quarter (16 columns each)
constexpr int SERVICE_WARPS_TMA = 3;                  // MMA issue, operand TMA, X / mask TMA
constexpr int THREADS_TMA = 32 * (SERVICE_WARPS_TMA + EPI_WARPS_TMA);
constexpr int X_BOX_BYTES = TM * 32 * 4;             // one 32-column swizzled box of the X tile: 16 KB
constexpr int X_TILE_BYTES = 2 * X_BOX_BYTES;        // 32 KB

__device__ __forceinline__ void epi_barrier_tma()
{
    asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS_TMA * 32) : "memory");
}

__device__ __forceinline__ float4 lds128(uint32_t saddr)
{
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr) : "memory");
    return v;
}
__device__ __forceinline__ uint4 lds128u(uint32_t saddr)
{
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(saddr) : "memory");
    return v;
}
// byte i of w (0..255) as a float without the conversion pipe: one PRMT builds the bits of 8388608 + b, one FADD
// removes the offset
__device__ __forceinline__ float byte_to_float(uint32_t w, int i)
{
    return __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7440u | (uint32_t)i)) - 8388608.0f;
}

template <int MODE, int MK>
__global__ void __launch_bounds__(THREADS_TMA, 1)
wrri_tc_tma_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmT,
                   const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmM, TcParams p)
{
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    constexpr int M_TILE_BYTES = MK == MK_U8 ? TM * TN : X_TILE_BYTES;
    constexpr int XM_STAGE = X_TILE_BYTES + M_TILE_BYTES;            // 40 KB / 64 KB: a multiple of 1024
    const int nchunk = p.KP / BK;
    const int w_bytes = nchunk * W_CHUNK_BYTES, t_bytes = nchunk * T_CHUNK_BYTES;
    const int fixed_bytes = MODE == 0 ? t_bytes : w_bytes;
    const int var_bytes = MODE == 0 ? w_bytes : t_bytes;
    const int var_chunk = MODE == 0 ? W_CHUNK_BYTES : T_CHUNK_BYTES;
    const int fixed_chunk = MODE == 0 ? T_CHUNK_BYTES : W_CHUNK_BYTES;
    uint8_t* sm_fixed = smem;
    uint8_t* sm_var = smem + fixed_bytes;
    uint8_t* sm_xm = sm_var + (size_t)p.stages * var_bytes;                       // [xm_stages][X tile | mask tile]
    uint64_t* bars = reinterpret_cast<uint64_t*>(sm_xm + (size_t)p.xm_stages * XM_STAGE);
    uint64_t* fixed_full = bars;            // 1
    uint64_t* var_full = bars + 1;          // [2]
    uint64_t* var_free = bars + 3;          // [2]
    uint64_t* acc_full = bars + 5;          // [2]
    uint64_t* acc_free = bars + 7;          // [2]
    uint64_t* xm_full = bars + 9;           // [4]
    uint64_t* xm_free = bars + 13;          // [4]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 17);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int fixed_tile = blockIdx.x;
    const int nvar_total = MODE == 0 ? p.tiles_r : p.tiles_c;
    int vb, ve;
    {
        const int q = nvar_total / (int)gridDim.y, r = nvar_total % (int)gridDim.y, g = blockIdx.y;
        vb = q * g + (g < r ? g : r);
        ve = vb + q + (g < r ? 1 : 0);
    }
    const int ntiles = ve - vb;
    const int var_rows = MODE == 0 ? TM : TN, fixed_rows = MODE == 0 ? TN : TM;

    if (threadIdx.x == 0) {
        mbar_init(fixed_full, 1);
        for (int s = 0; s < 2; ++s) {
            mbar_init(&var_full[s], 1); mbar_init(&var_free[s], 1);
            mbar_init(&acc_full[s], 1); mbar_init(&acc_free[s], EPI_WARPS_TMA);
        }
        for (int s = 0; s < 4; ++s) { mbar_init(&xm_full[s], 1); mbar_init(&xm_free[s], EPI_WARPS_TMA); }
        fence_barrier_init();
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(128) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ================================ MMA issue ================================================
        if (lane == 0 && ntiles > 0) {
            const int S = p.stages;
            mbar_wait(fixed_full, 0);
            const uint32_t idesc = make_idesc_tf32(TM, TN);
            int s = 0;
            uint32_t vph = 0;
            for (int n = 0; n < ntiles; ++n) {
                const int a = n & 1;
                mbar_wait(&var_full[s], vph);
                mbar_wait(&acc_free[a], ((n >> 1) & 1) ^ 1);
                tc_fence_after();
                const uint32_t var0 = smem_u32(sm_var + (size_t)s * var_bytes), fix0 = smem_u32(sm_fixed);
                const uint32_t w0 = MODE == 0 ? var0 : fix0;
                const uint32_t t0 = MODE == 0 ? fix0 : var0;
                for (int c = 0; c < nchunk; ++c) {
#pragma unroll
                    for (int ks = 0; ks < BK / UK; ++ks) {
                        umma_tf32(tmem_base + (uint32_t)(a * TN), make_desc(w0 + c * W_CHUNK_BYTES + ks * UK * 4),
                                  make_desc(t0 + c * T_CHUNK_BYTES + ks * UK * 4), idesc, (c > 0 || ks > 0) ? 1u : 0u);
                    }
                }
                umma_commit(&var_free[s]);            // the operand stage may be refilled when these MMAs retire
                umma_commit(&acc_full[a]);
                if (++s == S) { s = 0; vph ^= 1u; }
            }
        }
    } else if (warp == 1) {
        // ================================ operand producer =========================================
        if (lane == 0 && ntiles > 0) {
            const CUtensorMap* tm_fixed = MODE == 0 ? &tmT : &tmW;
            const CUtensorMap* tm_var = MODE == 0 ? &tmW : &tmT;
            mbar_expect_tx(fixed_full, (uint32_t)fixed_bytes);
            for (int c = 0; c < nchunk; ++c) tma_load_2d(tm_fixed, sm_fixed + c * fixed_chunk, fixed_full, c * BK, fixed_tile * fixed_rows);
            const int S = p.stages;
            int s = 0;
            uint32_t vph = 0;
            for (int n = 0; n < ntiles; ++n) {
                mbar_wait(&var_free[s], vph ^ 1u);    // the MMAs that read this stage have retired (free at the start)
                mbar_expect_tx(&var_full[s], (uint32_t)var_bytes);
                for (int c = 0; c < nchunk; ++c)
                    tma_load_2d(tm_var, sm_var + (size_t)s * var_bytes + c * var_chunk, &var_full[s], c * BK, (vb + n) * var_rows);
                if (++s == S) { s = 0; vph ^= 1u; }
            }
        }
    } else if (warp == 2) {
        // ================================ X / mask producer =======================================
        if (lane == 0) {
            const int NS = p.xm_stages;
            int s = 0;
            uint32_t xph = 0;
            for (int n = 0; n < ntiles; ++n, s = (s + 1 == NS ? 0 : s + 1), xph ^= (s == 0 ? 1u : 0u)) {
                const int rt = MODE == 0 ? (vb + n) : fixed_tile, ctile = MODE == 0 ? fixed_tile : (vb + n);
                mbar_wait(&xm_free[s], xph ^ 1u);                      // every epilogue warp has released this stage
                mbar_expect_tx(&xm_full[s], (uint32_t)XM_STAGE);
                uint8_t* dst = sm_xm + (size_t)s * XM_STAGE;
                tma_load_2d(&tmX, dst, &xm_full[s], ctile * TN, rt * TM);
                tma_load_2d(&tmX, dst + X_BOX_BYTES, &xm_full[s], ctile * TN + 32, rt * TM);
                if (MK == MK_U8) {
                    tma_load_2d(&tmM, dst + X_TILE_BYTES, &xm_full[s], ctile * TN, rt * TM);
                } else {
                    tma_load_2d(&tmM, dst + X_TILE_BYTES, &xm_full[s], ctile * TN, rt * TM);
                    tma_load_2d(&tmM, dst + X_TILE_BYTES + X_BOX_BYTES, &xm_full[s], ctile * TN + 32, rt * TM);
                }
            }
        }
    } else {
        // ======================================= epilogue ========================================
        const int ew = warp - SERVICE_WARPS_TMA; // 0..15
        const int q = warp & 3;                  // TMEM lane quarter this warp may read
        const int cgp = ew >> 2;                 // column group: tile columns [16*cgp, 16*cgp + 16)
        const int row = q * 32 + lane;           // row of the tile this thread owns
        const int c0 = 16 * cgp;
        const int NS = p.xm_stages;
        const float* Trow = p.Tt;                // T[t, :] (contiguous), W[:, t] = Wp[:, t] (stride KP)
        // shared-memory addresses of this thread's 4 x 16 bytes of an X (or fp32 weight) tile: box (c0 >> 5), row, and
        // the 16-byte chunks (c0 & 31)/4 + j with the 128-byte swizzle (chunk index XOR (row & 7)); loop invariant
        const uint32_t xrow = smem_u32(sm_xm) + (uint32_t)((c0 >> 5) * X_BOX_BYTES + row * 128);
        uint32_t xoff[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) xoff[j] = (uint32_t)(((((c0 & 31) >> 2) + j) ^ (row & 7)) << 4);
        // byte mask: 16 bytes of a 64-byte row, stored with the 64-byte swizzle (16-byte chunk index XOR (row >> 1) & 3:
        // eight consecutive rows then cover all 32 banks; unswizzled the read was a 4-way conflict, as many wavefronts
        // as the four X loads together)
        const uint32_t mrow = smem_u32(sm_xm) + (uint32_t)(X_TILE_BYTES + row * TN + (((c0 >> 4) ^ ((row >> 1) & 3)) << 4));
        const uint32_t tacc = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0;

        // With u = X - WT (the full residual) the statistics of nmf.py:687-701 / :735-746 are
        //   T-step: numer[c] = sum_r w_r m (u + w_r t_c) = A[c] + t_c D[c],  A[c] = sum_r (m w_r) u,  D[c] = sum_r (m w_r) w_r
        //   W-step: numer[r] = sum_c t_c m (u + w_r t_c) = A[r] + w_r D[r],  A[r] = sum_c (m t_c) u,  D[r] = sum_c (m t_c) t_c
        // i.e. four operations per element; the add-back of topic t happens once per CTA instead of once per element.
        float A[MODE == 0 ? 16 : 1], D[MODE == 0 ? 16 : 1];
#pragma unroll
        for (int i = 0; i < (MODE == 0 ? 16 : 1); ++i) { A[i] = 0.f; D[i] = 0.f; }

        auto load_tt = [&](int ctile, float out[16]) {
            const int64_t gc = (int64_t)ctile * TN + c0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (gc + 4 * j < p.d) v = __ldg(reinterpret_cast<const float4*>(Trow + gc) + j);     // d % 4 == 0
                out[4 * j] = v.x; out[4 * j + 1] = v.y; out[4 * j + 2] = v.z; out[4 * j + 3] = v.w;
            }
        };
        auto load_wt = [&](int rt) -> float {
            const int64_t gi = (int64_t)rt * TM + row;
            return gi < p.n ? __ldg(p.Wp + gi * p.KP + p.t) : 0.f;
        };
        // the factor entries that change with the tile (MODE 0: w_r, MODE 1: t_c) are requested one tile ahead
        float fac[MODE == 0 ? 1 : 16], facn[MODE == 0 ? 1 : 16];
        if (ntiles > 0) {
            if (MODE == 0) fac[0] = load_wt(vb); else load_tt(vb, fac);
        }
        int s = 0;
        uint32_t xph = 0;
        for (int n = 0; n < ntiles; ++n) {
            const int a = n & 1;
            if (n + 1 < ntiles) {
                if (MODE == 0) facn[0] = load_wt(vb + n + 1); else load_tt(vb + n + 1, facn);
            }
            // ---- this warp's 32 x 16 block of the product: TMEM -> registers
            mbar_wait(&acc_full[a], (n >> 1) & 1);
            tc_fence_after();
            uint32_t dr[16];
            tmem_ld16_issue(tacc + (uint32_t)(a * TN), dr);
            // ---- the same block of X and of the mask from the stage
            mbar_wait(&xm_full[s], xph);
            const uint32_t so = (uint32_t)s * XM_STAGE;
            float x[16], m[16];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float4 v = lds128(xrow + so + xoff[j]);
                x[4 * j] = v.x; x[4 * j + 1] = v.y; x[4 * j + 2] = v.z; x[4 * j + 3] = v.w;
            }
            if (MK == MK_U8) {
                const uint4 mw = lds128u(mrow + so);
                const uint32_t w4[4] = {mw.x, mw.y, mw.z, mw.w};
#pragma unroll
                for (int j = 0; j < 4; ++j)
#pragma unroll
                    for (int v = 0; v < 4; ++v) m[4 * j + v] = byte_to_float(w4[j], v);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 v = lds128(xrow + (uint32_t)X_TILE_BYTES + so + xoff[j]);
                    m[4 * j] = v.x; m[4 * j + 1] = v.y; m[4 * j + 2] = v.z; m[4 * j + 3] = v.w;
                }
            }
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_free[a]);                  // the accumulator block is in registers
            // ---- element-wise statistics
            if (MODE == 0) {
                const float wr = fac[0];
#pragma unroll
                for (int c = 0; c < 16; ++c) {
                    const float v = m[c] * wr;
                    A[c] = fmaf(v, x[c] - __uint_as_float(dr[c]), A[c]);
                    D[c] = fmaf(v, wr, D[c]);
                }
                fac[0] = facn[0];
                __syncwarp();
                if (lane == 0) mbar_arrive(&xm_free[s]);               // every lane has consumed its X / mask values
            } else {
                float a0 = 0.f, d0 = 0.f;
#pragma unroll
                for (int c = 0; c < 16; ++c) {
                    const float v = m[c] * fac[c];
                    a0 = fmaf(v, x[c] - __uint_as_float(dr[c]), a0);
                    d0 = fmaf(v, fac[c], d0);
                }
                A[0] += a0; D[0] += d0;
                __syncwarp();
                if (lane == 0) mbar_arrive(&xm_free[s]);
#pragma unroll
                for (int c = 0; c < 16; ++c) fac[c] = facn[c];
            }
            if (++s == NS) { s = 0; xph ^= 1u; }
        }
        // add topic t back (once per CTA): numer = A + (own factor entry) * D
        float nacc[MODE == 0 ? 16 : 1], dacc[MODE == 0 ? 16 : 1];
        if (MODE == 0) {
            float tt[16];
            load_tt(fixed_tile, tt);
#pragma unroll
            for (int c = 0; c < 16; ++c) { nacc[c] = fmaf(tt[c], D[c], A[c]); dacc[c] = D[c]; }
        } else {
            nacc[0] = fmaf(load_wt(fixed_tile), D[0], A[0]);
            dacc[0] = D[0];
        }

        // ---- once per CTA: cross-warp reduction through the (now idle) stage buffers, fixed order
        epi_barrier_tma();
        float* red = reinterpret_cast<float*>(sm_xm);
        const int et = threadIdx.x - 32 * SERVICE_WARPS_TMA;          // 0..511
        if (MODE == 0) {
            // red[which][col 0..63][row 0..127]: column sums over the 128 rows of the tile position
#pragma unroll
            for (int c = 0; c < 16; ++c) {
                red[(0 * TN + c0 + c) * TM + row] = nacc[c];
                red[(1 * TN + c0 + c) * TM + row] = dacc[c];
            }
            epi_barrier_tma();
            // 512 threads, 128 outputs: 4 threads per output add 32 rows each, then a 4-lane shuffle tree
            const int o = et >> 2, part = et & 3;
            float sacc = 0.f;
#pragma unroll 8
            for (int r = 0; r < 32; ++r) sacc += red[o * TM + part * 32 + ((r + lane) & 31)];      // bank = (r + lane) & 31
            sacc += __shfl_xor_sync(0xffffffffu, sacc, 1);
            sacc += __shfl_xor_sync(0xffffffffu, sacc, 2);
            if (part == 0) {
                const int which = o / TN, cc = o % TN;
                const int64_t gcol = (int64_t)fixed_tile * TN + cc;
                if (gcol < p.d) (which ? p.denom_part : p.numer_part)[(int64_t)blockIdx.y * p.d + gcol] = sacc;
            }
        } else {
            // red[which][column group][row]
            red[(0 * 4 + cgp) * TM + row] = nacc[0];
            red[(1 * 4 + cgp) * TM + row] = dacc[0];
            epi_barrier_tma();
            if (et < 2 * TM) {
                const int which = et / TM, r = et % TM;
                const float sacc = (red[(which * 4 + 0) * TM + r] + red[(which * 4 + 1) * TM + r]) +
                                   (red[(which * 4 + 2) * TM + r] + red[(which * 4 + 3) * TM + r]);
                const int64_t gi = (int64_t)fixed_tile * TM + r;
                if (gi < p.n) (which ? p.denom_part : p.numer_part)[(int64_t)blockIdx.y * p.n + gi] = sacc;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(128) : "memory");
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// dst[r, 0:KP] = (c < cols) ? src[r, c] (or src[c, r] when transposed) : 0
__global__ void pad_copy_kernel(const float* __restrict__ src, int64_t rows, int cols, int64_t ld, int transposed,
                                float* __restrict__ dst, int KP)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= rows * KP) return;
    const int64_t r = e / KP;
    const int c = (int)(e % KP);
    float v = 0.f;
    if (c < cols) v = transposed ? src[(int64_t)c * ld + r] : src[r * ld + c];
    dst[e] = v;
}

}  // namespace

struct WrriTc {
    int sm_count = 148;
    EncodeTiledFn encode = nullptr;
    int64_t n = 0, d = 0;
    int k = 0, KP = 0;
    float* Wp = nullptr;
    float* Tp = nullptr;
    CUtensorMap tmW, tmT;
    int stages[2] = {1, 2};
    size_t smem[2] = {0, 0};
    // TMA variant
    const void* mapX = nullptr; const void* mapM = nullptr; int64_t map_ldx = 0, map_ldm = 0; int map_mk = -1;
    CUtensorMap tmX, tmM;
    bool tma_ok = false;
    int tma_stages[2][3] = {{1, 1, 1}, {1, 1, 1}};      // [mode][mask kind] operand stages
    int tma_xm[2][3] = {{0, 0, 0}, {0, 0, 0}};          // [mode][mask kind] X/mask ring depth (0 = does not fit)
    size_t tma_smem[2][3] = {{0, 0, 0}, {0, 0, 0}};
};

WrriTc* wrri_tc_create(int sm_count, int64_t n, int64_t d, int k, std::string& err)
{
    if (k > 128) { err = "the tensor-core WRRI path supports k <= 128"; return nullptr; }
    if (d % 4 != 0) { err = "the tensor-core WRRI path needs d % 4 == 0"; return nullptr; }
    WrriTc* g = new WrriTc();
    g->sm_count = sm_count; g->n = n; g->d = d; g->k = k;
    g->KP = (k + 31) / 32 * 32;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess || !fn) {
        err = "cuTensorMapEncodeTiled is not available from the driver";
        delete g;
        return nullptr;
    }
    g->encode = (EncodeTiledFn)fn;
    if (cached_malloc((void**)&g->Wp, sizeof(float) * (size_t)n * g->KP) != cudaSuccess ||
        cached_malloc((void**)&g->Tp, sizeof(float) * (size_t)d * g->KP) != cudaSuccess) {
        err = "operand copy allocation failed";
        wrri_tc_destroy(g);
        return nullptr;
    }
    auto enc = [&](CUtensorMap* tm, float* base, int64_t rows, int box_rows) -> bool {
        cuuint64_t gdim[2] = {(cuuint64_t)g->KP, (cuuint64_t)rows};
        cuuint64_t gstr[1] = {(cuuint64_t)g->KP * 4};
        cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
        cuuint32_t estr[2] = {1, 1};
        return g->encode(tm, CU_TENSOR_MAP_DATA_TYPE_TFLOAT32, 2, base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
    };
    if (!enc(&g->tmW, g->Wp, n, TM) || !enc(&g->tmT, g->Tp, d, TN)) {
        err = "cuTensorMapEncodeTiled failed for the WRRI operands";
        wrri_tc_destroy(g);
        return nullptr;
    }
    // shared memory per CTA (two CTAs must fit in one SM): fixed operand + ring of the changing operand +
    // the staged product tile + barriers/alignment
    const int w_bytes = (g->KP / BK) * W_CHUNK_BYTES, t_bytes = (g->KP / BK) * T_CHUNK_BYTES;
    const size_t ds = sizeof(float) * TM * DS_LD + 256 + 1024;
    for (int mode = 0; mode < 2; ++mode) {
        const int fixed = mode == 0 ? t_bytes : w_bytes, var = mode == 0 ? w_bytes : t_bytes;
        g->stages[mode] = (fixed + 2 * (size_t)var + ds <= 112 * 1024) ? 2 : 1;
        g->smem[mode] = (size_t)fixed + (size_t)g->stages[mode] * var + ds;
    }
    return g;
}

void wrri_tc_destroy(WrriTc* g)
{
    if (!g) return;
    if (g->Wp) cached_free(g->Wp);
    if (g->Tp) cached_free(g->Tp);
    delete g;
}

float* wrri_tc_Wp(WrriTc* g) { return g->Wp; }
float* wrri_tc_Tp(WrriTc* g) { return g->Tp; }
int wrri_tc_KP(WrriTc* g) { return g->KP; }

int wrri_tc_groups(WrriTc* g, int mode)
{
    const int tiles_r = (int)((g->n + TM - 1) / TM), tiles_c = (int)((g->d + TN - 1) / TN);
    const int fixed = mode == 0 ? tiles_c : tiles_r, var = mode == 0 ? tiles_r : tiles_c;
    // enough CTAs for ~8 waves of one CTA per SM, at least 4 tiles per CTA when there are that many
    int groups = (16 * g->sm_count + fixed - 1) / fixed;
    if (groups > (var + 3) / 4) groups = (var + 3) / 4;
    if (groups < 1) groups = 1;
    return groups;
}

// refresh the padded operand copies from the caller's factors (start of a call)
void wrri_tc_load_factors(WrriTc* g, const float* W, const float* T, cudaStream_t st)
{
    int64_t e = g->n * g->KP;
    pad_copy_kernel<<<(unsigned)((e + 255) / 256), 256, 0, st>>>(W, g->n, g->k, g->k, 0, g->Wp, g->KP);
    e = g->d * g->KP;
    pad_copy_kernel<<<(unsigned)((e + 255) / 256), 256, 0, st>>>(T, g->d, g->k, g->d, 1, g->Tp, g->KP);
}

static bool tma_prepare(WrriTc* g, const float* X, int64_t ldx, const void* M, int mk, int64_t ldm)
{
    if (g->mapX == X && g->mapM == M && g->map_ldx == ldx && g->map_ldm == ldm && g->map_mk == mk) return g->tma_ok;
    g->mapX = X; g->mapM = M; g->map_ldx = ldx; g->map_ldm = ldm; g->map_mk = mk; g->tma_ok = false;
    const size_t mes = mk == MK_U8 ? 1 : 4;
    if ((reinterpret_cast<uintptr_t>(X) & 15) || (ldx * 4) % 16 || (reinterpret_cast<uintptr_t>(M) & 15) || (ldm * mes) % 16) return false;
    // fp32 tiles are fetched as 32-column boxes with the 128-byte swizzle (conflict-free row-per-lane reads in the
    // epilogue); the byte mask as one 64-column box with the 64-byte swizzle
    auto enc = [&](CUtensorMap* tm, const void* base, CUtensorMapDataType dt, size_t es, int64_t ld, int box_cols,
                   CUtensorMapSwizzle sw) -> bool {
        cuuint64_t gdim[2] = {(cuuint64_t)g->d, (cuuint64_t)g->n};
        cuuint64_t gstr[1] = {(cuuint64_t)ld * es};
        cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)TM};
        cuuint32_t estr[2] = {1, 1};
        return g->encode(tm, dt, 2, const_cast<void*>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
    };
    if (!enc(&g->tmX, X, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, ldx, 32, CU_TENSOR_MAP_SWIZZLE_128B)) return false;
    if (mk == MK_U8) {
        if (!enc(&g->tmM, M, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, ldm, TN, CU_TENSOR_MAP_SWIZZLE_64B)) return false;
    } else {
        if (!enc(&g->tmM, M, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, ldm, 32, CU_TENSOR_MAP_SWIZZLE_128B)) return false;
    }
    // shared-memory plan per mode: operands + as many X/mask stages as fit (at least 2) + barriers
    const int w_bytes = (g->KP / BK) * W_CHUNK_BYTES, t_bytes = (g->KP / BK) * T_CHUNK_BYTES;
    const size_t extra = 1024 /* barriers */ + 1024 /* alignment slack */;
    const size_t xm = (size_t)X_TILE_BYTES + (mk == MK_U8 ? (size_t)TM * TN : (size_t)X_TILE_BYTES);
    for (int mode = 0; mode < 2; ++mode) {
        const size_t fixed = mode == 0 ? t_bytes : w_bytes, var = mode == 0 ? w_bytes : t_bytes;
        // two operand stages first (with one, every tile waits a full L2 round trip for its W / T' tile after the
        // previous MMA retires), then as many X/mask stages as still fit (>= 2; the end-of-CTA reduction needs 64 KB)
        const size_t room = (size_t)227 * 1024;
        int S = 0, ns = 0;
        for (int s_try = 2; s_try >= 1; --s_try) {
            const size_t base = fixed + (size_t)s_try * var + extra;
            if (base >= room) continue;
            int n_try = (int)((room - base) / xm);
            if (n_try > 4) n_try = 4;
            if (n_try >= 2) { ns = n_try; S = s_try; break; }
        }
        if (S < 1 || ns < 2) { g->tma_xm[mode][mk] = 0; continue; }
        g->tma_stages[mode][mk] = S;
        g->tma_xm[mode][mk] = ns;
        g->tma_smem[mode][mk] = fixed + (size_t)S * var + extra + (size_t)ns * xm;
    }
    g->tma_ok = true;
    return true;
}

template <int MODE>
static int launch_mode(WrriTc* g, const float* X, int64_t ldx, const void* M, int mk, int64_t ldm, int t, const float* Trow,
                       float* numer_part, float* denom_part, int groups, cudaStream_t st, std::string& err)
{
    TcParams p;
    p.X = X; p.ldx = ldx; p.M = M; p.ldm = ldm; p.Wp = g->Wp; p.Tp = g->Tp; p.n = g->n; p.d = g->d; p.KP = g->KP; p.t = t;
    p.Tt = Trow;
    p.tiles_r = (int)((g->n + TM - 1) / TM); p.tiles_c = (int)((g->d + TN - 1) / TN);
    p.groups = groups; p.numer_part = numer_part; p.denom_part = denom_part; p.stages = g->stages[MODE]; p.xm_stages = 0;
    dim3 grid(MODE == 0 ? p.tiles_c : p.tiles_r, groups);
    if (mk != MK_U8 && mk != MK_REAL) { err = "the tensor-core WRRI path needs a mask"; return -1; }
    if (ldm % 4 != 0) { err = "mask rows need a stride that is a multiple of 4 elements"; return -1; }
    if (Trow && (reinterpret_cast<uintptr_t>(Trow) & 15) == 0 && tma_prepare(g, X, ldx, M, mk, ldm) &&
        g->tma_xm[MODE][mk] >= 2) {
        p.stages = g->tma_stages[MODE][mk];
        p.xm_stages = g->tma_xm[MODE][mk];
        const size_t smem = g->tma_smem[MODE][mk];
        if (mk == MK_U8) {
            auto kern = wrri_tc_tma_kernel<MODE, MK_U8>;
            cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            kern<<<grid, THREADS_TMA, smem, st>>>(g->tmW, g->tmT, g->tmX, g->tmM, p);
        } else {
            auto kern = wrri_tc_tma_kernel<MODE, MK_REAL>;
            cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            kern<<<grid, THREADS_TMA, smem, st>>>(g->tmW, g->tmT, g->tmX, g->tmM, p);
        }
    } else if (mk == MK_U8) {
        auto kern = wrri_tc_kernel<MODE, MK_U8>;
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g->smem[MODE]);
        kern<<<grid, THREADS, g->smem[MODE], st>>>(g->tmW, g->tmT, p);
    } else {
        auto kern = wrri_tc_kernel<MODE, MK_REAL>;
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g->smem[MODE]);
        kern<<<grid, THREADS, g->smem[MODE], st>>>(g->tmW, g->tmT, p);
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { err = cudaGetErrorString(e); return -1; }
    return 1;
}

int wrri_tc_stats(WrriTc* g, int mode, const float* X, int64_t ldx, const void* M, int mk, int64_t ldm, int t,
                  const float* Trow, float* numer_part, float* denom_part, int groups, cudaStream_t st, std::string& err)
{
    if ((reinterpret_cast<uintptr_t>(X) & 15) != 0 || ldx % 4 != 0) { err = "X rows must be 16-byte aligned"; return -1; }
    return mode == 0 ? launch_mode<0>(g, X, ldx, M, mk, ldm, t, Trow, numer_part, denom_part, groups, st, err)
                     : launch_mode<1>(g, X, ldx, M, mk, ldm, t, Trow, numer_part, denom_part, groups, st, err);
}

}  // namespace rri
