// Internal interface between the fp32 HaplotypeModel path (haplotype.cu) and its tensor-core path (haplotype_tc.cu).
#pragma once
#include "common.cuh"

namespace nsnp {

// C[M][N] = A[M][K] . B[N][K]^T + bias[N] (tanh when act_tanh): A rows lda apart, C rows ldc apart; fp32 FFMA
int hap_sgemm_nt(const float* A, int64_t lda, const float* B, const float* bias, float* C, int64_t ldc, int64_t M, int N, int K, int act_tanh,
                 cudaStream_t st);
// genotype (10) / zygosity (3) heads + softmax from the dense output hid [n][256]
int hap_heads(const float* hid, const float* gw, const float* gb, const float* zw, const float* zb, float* gt, float* zy, int64_t n, cudaStream_t st);

}  // namespace nsnp
