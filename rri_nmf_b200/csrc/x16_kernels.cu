// x16_kernels.cu -- 16-bit copies of the operands of the block-order TF32 contraction (f16_gemm_run).
//
// The TF32 tensor map rounds every fp32 element to TF32 (sign, 8 exponent bits, 10 mantissa bits) on its way into
// shared memory.  fp16 has the same 10-bit mantissa, so fp16(tf32(x) * 2^e) is exact -- and a kind::f16 MMA sees the
// very operand the TF32 path sees -- whenever tf32(x) * 2^e is 0 or lies in fp16's normal range [2^-14, 65504].  One
// power-of-two scale e per matrix; the contraction's epilogue multiplies the sums by 2^-(e_A + e_B), which is exact.
//
//   data   (once per rri_bind): x16_scan finds max |tf32(x)|, the smallest nonzero |tf32(x)| and any non-finite value;
//          x16_exponent decides (on the host) whether all nonzero values fit the 30 binades of fp16's normal range
//          under one scale; x16_copy then writes X16 [n, ldy] and its transpose Xt16 [d, ldyt] in one pass over X;
//   factor (once per contraction): f16_absmax_kernel reduces max |tf32(f)| per block, f16_factor_kernel re-reduces the
//          block maxima (fixed order: deterministic), picks the scale and writes the copy; the scale goes to device
//          memory, where the contraction's epilogue reads it.  Factor values below ~2^-29 of the factor's maximum become
//          fp16 subnormals and lose bits that TF32 keeps; their share of a sum is far below TF32's own rounding.
#include <cuda_fp16.h>

#include "kernels.h"

namespace rri {

namespace {

// round to TF32 as the TFLOAT32 tensor map does: to nearest, ties to even, subnormals kept (a value within half a TF32
// ulp of FLT_MAX becomes inf); inf and nan pass unchanged
__device__ __forceinline__ float to_tf32(float x)
{
    const uint32_t b = __float_as_uint(x);
    if ((b & 0x7f800000u) == 0x7f800000u) return x;
    return __uint_as_float((b + 0xfffu + ((b >> 13) & 1u)) & ~0x1fffu);
}

__device__ __forceinline__ float pow2(int e) { return __int_as_float((127 + e) << 23); }     // e in [-126, 127]

__global__ void x16_scan_kernel(const float* __restrict__ X, int64_t rows, int64_t cols, int64_t ld, unsigned* out)
{
    unsigned mx = 0u, mn = 0xffffffffu, bad = 0u;
    for (int64_t r = blockIdx.x; r < rows; r += gridDim.x) {
        const float* row = X + r * ld;
        for (int64_t c = threadIdx.x; c < cols; c += blockDim.x) {
            const unsigned b = __float_as_uint(fabsf(to_tf32(__ldcs(row + c))));
            if (b >= 0x7f800000u) bad = 1u;                        // inf / nan (or a finite value rounding to inf)
            else {
                mx = b > mx ? b : mx;
                if (b) mn = b < mn ? b : mn;
            }
        }
    }
    mx = __reduce_max_sync(0xffffffffu, mx);
    mn = __reduce_min_sync(0xffffffffu, mn);
    bad = __reduce_or_sync(0xffffffffu, bad);
    if ((threadIdx.x & 31) == 0) {
        if (mx) atomicMax(out + 0, mx);
        if (mn != 0xffffffffu) atomicMin(out + 1, mn);
        if (bad) atomicOr(out + 2, bad);
    }
}

// X16[r, c] = fp16(tf32(X[r, c]) * 2^e), Xt16[c, r] = the same value; 32 x 32 tiles, 256 threads
__global__ void x16_copy_kernel(const float* __restrict__ X, int64_t rows, int64_t cols, int64_t ldx, int e,
                                __half* __restrict__ Y, int64_t ldy, __half* __restrict__ Yt, int64_t ldyt)
{
    __shared__ __half tile[32][34];
    const int64_t c0 = (int64_t)blockIdx.x * 32, r0 = (int64_t)blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const float s = pow2(e);
    for (int i = ty; i < 32; i += 8) {
        const int64_t r = r0 + i, c = c0 + tx;
        if (r < rows && c < cols) {
            const __half h = __float2half_rn(to_tf32(X[r * ldx + c]) * s);
            Y[r * ldy + c] = h;
            tile[i][tx] = h;
        }
    }
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        const int64_t c = c0 + i, r = r0 + tx;
        if (r < rows && c < cols) Yt[c * ldyt + r] = tile[tx][i];
    }
}

// scale of a factor copy from the bits of max |tf32(f)|: the maximum lands in [2^15, 2^16)
__device__ __forceinline__ int factor_exp(unsigned m)
{
    if (m == 0u || m >= 0x7f800000u) return 0;                    // all zeros, or non-finite (propagates as in TF32)
    const int e = 15 - ((int)(m >> 23) - 127);
    return e < -126 ? -126 : (e > 126 ? 126 : e);
}

__device__ __forceinline__ unsigned block_max(unsigned v, unsigned* sh)
{
    v = __reduce_max_sync(0xffffffffu, v);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x < 32) {
        unsigned w = threadIdx.x < (blockDim.x >> 5) ? sh[threadIdx.x] : 0u;
        w = __reduce_max_sync(0xffffffffu, w);
        if (threadIdx.x == 0) sh[32] = w;
    }
    __syncthreads();
    return sh[32];
}

// Both passes over the factor go four elements per load (VEC: rows of a multiple of 4 columns, 16-byte aligned) with
// U loads in flight per thread before any of them is used: one dependent load per thread at a time left a 64 x 200 000
// factor (the T half-step's W') latency-bound.  The maximum does not depend on which block sees which element, and every
// element is converted on its own, so the copy and its scale are those of the one-element-at-a-time loops.
constexpr int FU = 4;

__device__ __forceinline__ unsigned absbits(float x) { return __float_as_uint(fabsf(to_tf32(x))); }

template <bool VEC>
__global__ void __launch_bounds__(256)
f16_absmax_kernel(const float* __restrict__ F, int rows, int64_t cols, int64_t ld, unsigned* __restrict__ part)
{
    __shared__ unsigned sh[33];
    unsigned m = 0u;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (VEC) {
        const int64_t cq = cols / 4, total = (int64_t)rows * cq;
        for (int64_t e0 = t0; e0 < total; e0 += FU * stride) {
            float4 v[FU];
#pragma unroll
            for (int u = 0; u < FU; ++u) {
                const int64_t e = e0 + u * stride;
                v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (e < total) v[u] = __ldg(reinterpret_cast<const float4*>(F + (e / cq) * ld) + e % cq);
            }
#pragma unroll
            for (int u = 0; u < FU; ++u)
                m = max(m, max(max(absbits(v[u].x), absbits(v[u].y)), max(absbits(v[u].z), absbits(v[u].w))));
        }
    } else {
        for (int r = 0; r < rows; ++r)
            for (int64_t c = t0; c < cols; c += stride) m = max(m, absbits(F[(int64_t)r * ld + c]));
    }
    m = block_max(m, sh);
    if (threadIdx.x == 0) part[blockIdx.x] = m;
}

__device__ __forceinline__ __half2 to_h2(float a, float b, float s)
{
    return __halves2half2(__float2half_rn(to_tf32(a) * s), __float2half_rn(to_tf32(b) * s));
}

template <bool VEC>
__global__ void __launch_bounds__(256)
f16_factor_kernel(const float* __restrict__ F, int rows, int64_t cols, int64_t ld, const unsigned* __restrict__ part,
                  int nparts, __half* __restrict__ out, int64_t ldo, int* __restrict__ e_out)
{
    __shared__ unsigned sh[33];
    unsigned m = 0u;
    for (int i = threadIdx.x; i < nparts; i += blockDim.x) m = part[i] > m ? part[i] : m;
    const int e = factor_exp(block_max(m, sh));
    const float s = pow2(e);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (VEC) {
        const int64_t cq = cols / 4, total = (int64_t)rows * cq;
        for (int64_t e0 = t0; e0 < total; e0 += FU * stride) {
            float4 v[FU];
#pragma unroll
            for (int u = 0; u < FU; ++u) {
                const int64_t q = e0 + u * stride;
                if (q < total) v[u] = __ldg(reinterpret_cast<const float4*>(F + (q / cq) * ld) + q % cq);
            }
#pragma unroll
            for (int u = 0; u < FU; ++u) {
                const int64_t q = e0 + u * stride;
                if (q < total) {
                    __half2* o = reinterpret_cast<__half2*>(out + (q / cq) * ldo + 4 * (q % cq));
                    o[0] = to_h2(v[u].x, v[u].y, s);
                    o[1] = to_h2(v[u].z, v[u].w, s);
                }
            }
        }
    } else {
        for (int r = 0; r < rows; ++r)
            for (int64_t c = t0; c < cols; c += stride)
                out[(int64_t)r * ldo + c] = __float2half_rn(to_tf32(F[(int64_t)r * ld + c]) * s);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *e_out = e;
}

}  // namespace

void launch_x16_scan(const float* X, int64_t rows, int64_t cols, int64_t ld, unsigned* out, int sm_count, cudaStream_t st)
{
    cudaMemsetAsync(out, 0, 3 * sizeof(unsigned), st);              // {max, min nonzero, non-finite} = {0, ~0u, 0}
    cudaMemsetAsync(out + 1, 0xff, sizeof(unsigned), st);
    const int64_t blocks = rows < (int64_t)sm_count * 8 ? rows : (int64_t)sm_count * 8;
    x16_scan_kernel<<<(unsigned)blocks, 512, 0, st>>>(X, rows, cols, ld, out);
}

bool x16_exponent(const unsigned scan[3], int* e)
{
    const unsigned mx = scan[0], mn = scan[1];
    *e = 0;
    if (scan[2]) return false;                                     // inf / nan
    if (mx == 0u) return true;                                     // all zeros
    if (mn < 0x00800000u) return false;                            // fp32 subnormals: keep what the TF32 path does with them
    const int emax = (int)(mx >> 23) - 127, emin = (int)(mn >> 23) - 127;
    int s = 15 - emax;                                             // the maximum lands in [2^15, 2^16): at most 65504
    if (s > 126) s = 126;
    *e = s;
    return emin + s >= -14;                                        // the smallest nonzero value stays a normal fp16
}

void launch_x16_copy(const float* X, int64_t rows, int64_t cols, int64_t ldx, int e, void* Y, int64_t ldy, void* Yt,
                     int64_t ldyt, cudaStream_t st)
{
    const int64_t bx = (cols + 31) / 32;
    for (int64_t r = 0; r < rows; r += 65535LL * 32) {             // grid.y is limited to 65535 blocks
        const int64_t rr = (rows - r) < 65535LL * 32 ? (rows - r) : 65535LL * 32;
        dim3 grid((unsigned)bx, (unsigned)((rr + 31) / 32));
        x16_copy_kernel<<<grid, 256, 0, st>>>(X + r * ldx, rr, cols, ldx, e, (__half*)Y + r * ldy, ldy, (__half*)Yt + r, ldyt);
    }
}

int f16_factor_parts(int sm_count) { return 4 * sm_count < 1024 ? 4 * sm_count : 1024; }

void launch_f16_factor(const float* F, int rows, int64_t cols, int64_t ld, unsigned* part, int nparts, void* out,
                       int64_t ldo, int* e_out, cudaStream_t st)
{
    const bool vec = cols % 4 == 0 && ld % 4 == 0 && ldo % 4 == 0 && (reinterpret_cast<uintptr_t>(F) & 15) == 0 &&
                     (reinterpret_cast<uintptr_t>(out) & 7) == 0;
    if (vec) {
        f16_absmax_kernel<true><<<nparts, 256, 0, st>>>(F, rows, cols, ld, part);
        f16_factor_kernel<true><<<nparts, 256, 0, st>>>(F, rows, cols, ld, part, nparts, (__half*)out, ldo, e_out);
    } else {
        f16_absmax_kernel<false><<<nparts, 256, 0, st>>>(F, rows, cols, ld, part);
        f16_factor_kernel<false><<<nparts, 256, 0, st>>>(F, rows, cols, ld, part, nparts, (__half*)out, ldo, e_out);
    }
}

}  // namespace rri
