// Fused tcgen05 kernels of the transformer layers (fused_tail.cu, fused_attn.cu).
#pragma once
#include "common.cuh"
#include "gemm_f32.cuh"   // ACT_* activation codes

namespace mocha {

// Block tail of a transformer layer, one launch (fused_tail.cu), width D = 256:
//   Y = LN1?(A0 W0^T + b0 + R0)                      A0 bf16 [M, K0] (row pitch lda), W0 bf16 [256, K0], R0 fp32 [M,256]
//   Z = LN2?(Y + act(Y W1^T + b1) W2^T + b2)         W1 bf16 [Hd, 256], W2 bf16 [256, Hd]; skipped when Hd == 0
// g1/be1, g2/be2 select the LayerNorms (NULL = none); outputs of the LAST stage: O32 fp32 and / or O16 bf16 [M,256].
bool tc_tail_supported(int M, int K0, int Hd);
int tc_tail(const __nv_bfloat16* A0, int lda, int K0, const __nv_bfloat16* W0, const float* b0, const float* R0,
            const float* g1, const float* be1, int Hd, int act, const __nv_bfloat16* W1, const float* b1,
            const __nv_bfloat16* W2, const float* b2, const float* g2, const float* be2, float eps, float* O32,
            __nv_bfloat16* O16, int M, cudaStream_t s, int r0_period = 0);   // r0_period > 0: R0 is a [period, 256] table, row r reads R0[r % period]

// Attention core in one launch (fused_attn.cu): out[b, :, h*dh:(h+1)*dh] = softmax(Q_h K_h^T / sqrt(dh)) V_h.
// q / k / v: bf16 views [B*nq | B*nkv, ld] with head h at columns h*dh (or h * the operand's head stride); out: bf16
// [B, nq, H*dh] (ldo = H*dh).
// dh in {64, 128, 256}, nkv <= 256, any nq.
bool tc_attn_fused_supported(int nq, int nkv, int dh);
int tc_attn_fused(const __nv_bfloat16* q, int ldq, const __nv_bfloat16* k, int ldk, const __nv_bfloat16* v, int ldv, int B, int H,
                  int nq, int nkv, int dh, __nv_bfloat16* out, int ldo, cudaStream_t s, bool q_shared = false,   // q_shared: one [nq, H*dh] query table for every clip
                  int q_hs = -1, int k_hs = -1, int v_hs = -1);   // column stride between heads per operand (-1: dh; 0: shared by all heads)

}  // namespace mocha
