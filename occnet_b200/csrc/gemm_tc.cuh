// tcgen05 / TMEM / TMA bf16 GEMM (gemm_tc.cu):  C[M,N] = act(A[M,K] . W[N,K]^T + bias) (+ residual)
#pragma once
#include "common.cuh"

namespace occ {

// shapes the tensor-core kernel handles: K % 64 == 0 (and the split point K1 % 64 == 0), N % 16 == 0, N <= 256 per pass
bool gemm_tc_supported(int M, int N, int K, int K1);

template <typename TC>
int gemm_tc(const bf16* A, const bf16* A2, int K1, const bf16* W, const float* bias, const float* residual, TC* C,
            int M, int N, int K, int act, cudaStream_t stream);

// Same GEMM with N = 256 and a fused epilogue  y = LayerNorm(A.W^T + bias + residual) (eps 1e-5):
// writes the fp32 residual stream, the bf16 operand copy and (optionally) the bf16 copy of y + pos.
int gemm_tc_ln(const bf16* A, const bf16* W, const float* bias, const float* residual, const float* gamma,
               const float* beta, const float* pos, float* y_f32, bf16* y_bf16, bf16* y_pos_bf16, int M, int K,
               cudaStream_t stream);

// C = A.W^T + bias with N = n*256: output written as n separate contiguous [M,256] bf16 matrices (C + i*M*256).
// Used to project the camera tokens with the value_proj weights of ALL encoder layers in one pass over the tokens.
int gemm_tc_blocked256(const bf16* A, const bf16* W, const float* bias, bf16* C, int M, int N, int K, cudaStream_t stream);

// TemporalSelfAttention's input projections in ONE launch (independent problems on disjoint CTAs): value_proj of 1-2 queue
// entries (bf16 [M,256]) + the concatenated sampling_offsets / attention_weights projection (fp16 [M,Nq], optional fp32
// epilogue constant rq [M,Nq] (rq_t32: the same constant in the T32 block layout, rows padded to 32), optional second K operand Aq2)
int gemm_tc_tsa_inputs(const bf16* const* Av, int nv, const bf16* Wv, const float* bv, bf16* const* Cv, const bf16* Aq,
                       const bf16* Aq2, int K1q, const bf16* Wq, const float* bq, const float* rq, const float* rq_t32, __half* Cq,
                       int M, int Nq, int Kq, cudaStream_t stream);

// fp32-grade product of an fp32 operand (given as its bf16 split S = [hi | lo], [M, 2*Ks]) with fp32 weights (given as
// W3 = [W_hi | W_hi | W_lo], [N, 3*Ks] bf16): 3 tensor-core passes in one launch, relative error ~2^-16.
int gemm_tc_split3(const bf16* S, int Ks, const bf16* W3, const float* bias, const float* residual, float* C, int M, int N,
                   int act, cudaStream_t stream);
// S[r] = [hi(a[r]) hi(b[r]) | lo(a[r]) lo(b[r])], hi = bf16(x), lo = bf16(x - hi); b may be null (Kb = 0)
int launch_split_bf16(const float* a, int Ka, const float* b, int Kb, int64_t rows, bf16* S, cudaStream_t stream);

int launch_bf16_to_f32(const bf16* src, float* dst, int64_t n, cudaStream_t stream);

}  // namespace occ
