// gemm_tf32_sm100.h -- TF32 tcgen05 contraction C[M,N] = A[M,K] * B[N,K]^T for tall-skinny outputs
// (N = rank k <= 256, M*K = the data matrix), sm_100a only.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>

namespace rri {
struct Tf32Gemm;
Tf32Gemm* tf32_gemm_create(int sm_count, int nmax, std::string& err);
void tf32_gemm_destroy(Tf32Gemm* g);
// returns the number of kernels launched, or -1 (err set).
// Optional auxiliary output in the same launch: C2[M2, N] (leading dimension ldc2) = A2[M2, K] * B[N, K]^T -- with
// A2 = B this is the k x k Gram matrix of the factor, computed as one more row tile of the streaming contraction.
int tf32_gemm_run(Tf32Gemm* g, const float* A, int64_t lda, const float* B, int64_t ldb, float* C,
                  int64_t ldc, int64_t M, int N, int64_t K, cudaStream_t st, std::string& err,
                  const float* A2 = nullptr, int64_t lda2 = 0, int M2 = 0, float* C2 = nullptr, int64_t ldc2 = 0);
// The same contraction over 16-bit copies: A holds fp16(a * 2^a_exp), B (and A2) fp16(b * 2^(*b_exp)) with the factor's
// exponent in device memory; C (C2) receive the products scaled back by 2^-(a_exp + *b_exp) (2^-2*b_exp), which is exact.
// The tensor cores run kind::f16 with fp32 accumulators; split, fix-up order and flush period (in K) are those of
// tf32_gemm_run, so operands that are exact TF32 values in fp16's normal range give what tf32_gemm_run gives.
int f16_gemm_run(Tf32Gemm* g, const __half* A, int64_t lda, int a_exp, const __half* B, int64_t ldb, const int* b_exp,
                 float* C, int64_t ldc, int64_t M, int N, int64_t K, cudaStream_t st, std::string& err,
                 const __half* A2 = nullptr, int64_t lda2 = 0, int M2 = 0, float* C2 = nullptr, int64_t ldc2 = 0);
}  // namespace rri
