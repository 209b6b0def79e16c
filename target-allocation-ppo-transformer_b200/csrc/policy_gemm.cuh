// policy_gemm.cuh - the dense contraction of the policy network: D[M,N] = act(A[M,K] W[N,K]^T + bias[N]) in bf16 with fp32
// accumulation on tcgen05 - the hand-written persistent TMA / TMEM kernel of policy_dense.cu.
#pragma once
#include <cstdint>
#include <cuda.h>
#include <cuda_runtime.h>

namespace uavp {
// A: bf16, row stride lda elements (lda % 8 == 0); W: bf16 [N,K] row-major; D: bf16 [M,N] row-major; bias fp32 [N] (or NULL).
// relu != 0 applies max(0, .).  N in {64,128,256,384}, K % 64 == 0, K <= 384.  Returns 0 or a negative code.
int gemm_bias_act(const void *A, int64_t lda, const void *W, const float *bias, void *D, int M, int N, int K, int relu,
                  cudaStream_t stream);
// D[M,N] = (A[M,K] W[N,K]^T) where aux[M,N] > 0, else 0 (aux: bf16, row stride ld_aux): ReLU backward fused into the
// epilogue of the activation-gradient GEMM.
int gemm_drelu(const void *A, int64_t lda, const void *W, const void *aux, int64_t ld_aux, void *D, int M, int N, int K,
               cudaStream_t stream);
// out[M,128] = LayerNorm(X[M,128] + A[M,K] W[128,K]^T + bias) * gamma + beta (eps 1e-5), plus what the backward keeps: the
// normalised rows xhat (bf16 [M,128]) and rstd (fp32 [M]).  X: bf16 with row stride ldx (the residual stream).
int gemm_add_ln(const void *A, int64_t lda, const void *W, const float *bias, const void *X, int64_t ldx, const float *gamma,
                const float *beta, void *out, void *xhat, float *rstd, int M, int K, cudaStream_t stream);

// TMA tensor maps of the dense and the weight-gradient kernels, built with the driver's cuTensorMapEncodeTiled (looked up
// once).  tensor_maps_available: the driver provides it.  make_tensor_map: row-major bf16 [rows, cols] with row stride ld
// (elements) as a 2-D map of [box_rows x 64] boxes with 128 B swizzle; false when the encoder is missing or rejects it.
bool tensor_maps_available();
bool make_tensor_map(CUtensorMap *m, const void *base, int64_t ld, int64_t rows, int cols, int box_rows);
}  // namespace uavp
