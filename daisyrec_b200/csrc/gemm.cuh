// gemm.cuh -- plain entry points of the dense-layer GEMM dispatcher in neumf.cu (dtype 0: fp32 CUDA cores, 1: bf16 tcgen05),
// and the dense optimiser step the tower / layer blocks of NeuMF, NGCF and NFM share.
#pragma once
#include "common.cuh"

namespace drb {

// C[M,N] = A[M,K] B[N,K]^T        (Linear forward: activations x weight^T)
int gemm_nt(int dtype, long long M, int N, int K, const float *A, long long lda, const float *B, long long ldb, float *C,
            long long ldc, cudaStream_t st);
// C[M,N] = A[M,K] B[K,N]          (input gradient: dZ x weight)
int gemm_nn(int dtype, long long M, int N, int K, const float *A, long long lda, const float *B, long long ldb, float *C,
            long long ldc, cudaStream_t st);
// C[N,M] += (A[K,M]^T B[K,N])^T   (weight gradient [out, in] += dZ^T X, computed with the wide dimension on the MMA rows; split-K)
int gemm_tn_acc_t(int dtype, long long M, int N, int K, const float *A, long long lda, const float *B, long long ldb, float *C,
                  long long ldc, cudaStream_t st);
// gb[n] += sum_m dZ[m, n]          (bias gradient, N <= 256)
int colsum_acc(const float *dZ, long long M, int N, float *gb, cudaStream_t st);

struct WsHeader;
// W -= step number adam_step + 1 of SGD or torch.optim.Adam's single-tensor rule (m, v: Adam's state) on a flat block of n
// floats, and g = 0; no-op once hdr->status is set (a NaN loss earlier in the step)
int dense_update(float *W, float *g, float *m, float *v, long long n, const drb_hyper *h, long long adam_step, const WsHeader *hdr,
                 cudaStream_t st);

}  // namespace drb
