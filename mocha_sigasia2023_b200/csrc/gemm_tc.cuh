// tcgen05 (5th-gen tensor core) GEMM family for sm_100a:
//   TMA (cp.async.bulk.tensor, 128B swizzle) -> shared memory ring -> tcgen05.mma (bf16 x bf16,
//   fp32 accumulators in TMEM, double-buffered) -> tcgen05.ld epilogue.
// Two epilogues share the main loop:
//   * linear:  C = act(A W^T + bias) (+ residual), optionally as an implicit temporal convolution
//              (taps shifted TMA row windows over a reflect-padded channel-last activation)
//   * matcher: coarse squared distances ||x||^2 - 2 q.x with a fused per-row running top-kc
#pragma once
#include <cuda.h>
#include "common.cuh"

namespace mocha {

// ---- tensor maps (shared with the fused kernels) -------------------------------------------------------
// operand map: [rows, K] row-major (row pitch pitch_elems, 0 = dense), box = box_rows x 128 bytes, 128 B swizzle,
// out-of-bounds reads return zero
int tc_make_tmap(CUtensorMap* tm, const void* ptr, unsigned long long rows, unsigned long long K, int box_rows,
                 unsigned long long pitch_elems = 0, bool f32 = false);
// output map {cols, rows per image, images}: boxes of 32 rows x 32 columns (fp32: 128 B-swizzled; bf16: 64 B-swizzled,
// or 64 columns / 128 B-swizzled with wide16); rows and columns past the tensor are clipped
int tc_make_out_tmap(CUtensorMap* tm, const void* ptr, unsigned long long cols, unsigned long long rows_per_img,
                     unsigned long long imgs, unsigned long long ld_elems, bool f32, unsigned long long img_pitch_rows = 0,
                     bool wide16 = false);
int tc_num_sms();

// ---- linear ------------------------------------------------------------------------------------
bool tc_linear_supported(int M, int N, int K);
// bytes of bf16 scratch needed to stage an [rows, K] A operand
size_t tc_scratch_bytes(size_t rows, size_t K);
void tc_set_workspace_precision(int precision);

// Registered bf16 mirror of an fp32 weight blob: W16 = blob16 + (W - blob32).
void tc_register_blob(const float* blob32, const void* blob16, size_t elems);
const __nv_bfloat16* tc_lookup_bf16(const float* W);

// C[M,N] fp32 = act(prologue(A)[M,K] W[N,K]^T + bias) (+res). A fp32 is cast to bf16 into ws first.
int tc_linear(const float* A, const float* W, const float* bias, int bias_period, const float* res, float* C,
              int M, int N, int K, int act, int a_lrelu, Workspace& ws, cudaStream_t s);

// Output of a tensor-core layer: fp32 and/or a bf16 copy (the operand of the next tensor-core layer);
// lrelu stores LeakyReLU(0.2)(x) in the bf16 copy for pre-activation consumers.
struct TcOut {
  float* f32;
  __nv_bfloat16* bf16;
  int lrelu;
};
// Same with operands already in bf16 (A16 [M,K] with row pitch lda, W16 [N,K], K-major, 16B-aligned rows).
int tc_linear_bf16(const __nv_bfloat16* A16, int lda, const __nv_bfloat16* W16, const float* bias, int bias_period,
                   const float* res, TcOut out, int M, int N, int K, int act, cudaStream_t s);
// nb stacked linear layers of one shape in one launch: out16[g] = A16[g] W16[g]^T, A16 [nb,R,K], W16 [nb,N,K], out16 [nb,R,N]
int tc_linear_bf16_grouped(const __nv_bfloat16* A16, const __nv_bfloat16* W16, __nv_bfloat16* out16, int nb, int R, int N,
                           int K, cudaStream_t s);
// fp32 -> bf16 (optionally through LeakyReLU(0.2))
int tc_cast(const float* x, __nv_bfloat16* y, long long n, int lrelu, cudaStream_t s);

// Reflect-padded temporal convolution on tensor cores: X fp32 [B,T,V,Cin] -> C [B*T*V, Cout].
// W [Cout, taps*Cin] (tap-major K). Stages a bf16 reflect-padded copy of X in ws.
bool tc_tconv_supported(int B, int T, int V, int Cin, int Cout, int taps);
size_t tc_tconv_scratch_bytes(int B, int T, int V, int Cin, int taps);
int tc_tconv(const float* X, const float* W, const float* bias, int bias_period, float* C, int B, int T, int V,
             int Cin, int Cout, int taps, int tdiv, Workspace& ws, cudaStream_t s, int repeat = 1);
// X or Xh (bf16 source) may be given; output fp32 and/or bf16
int tc_tconv_ex(const float* X, const __nv_bfloat16* Xh, const float* W, const float* bias, int bias_period, TcOut out,
                int B, int T, int V, int Cin, int Cout, int taps, int tdiv, Workspace& ws, cudaStream_t s, int repeat = 1,
                bool xh_is_padded = false);  // Xh already is the reflect-padded [B, T + 2*(taps/2), V, Cin] tensor
// GEMM over nb images whose outputs land at out + b * out_img_pitch_rows * N (TMA-store epilogue, column bias)
int tc_linear_bf16_img(const __nv_bfloat16* A16, int lda, const __nv_bfloat16* W16, const float* bias, TcOut out, int nb,
                       int rows_per_img, long long out_img_pitch_rows, int N, int K, int act, cudaStream_t s);

// ---- 3xTF32: fp32-grade GEMMs on the tensor cores (MOCHA_TF32X3) -------------------------------------
// fp32 operands split into tf32 hi / lo parts ([hi | lo | hi] x [hi | hi | lo] over a 3x longer K), fp32 accumulation in
// TMEM, the bf16 path's main loop and epilogues. Long problems run as row / image chunks sized by the free workspace.
bool tc_linear_tf32x3_supported(int M, int N, int K);
int tc_linear_tf32x3(const float* A, const float* W, const float* bias, int bias_period, const float* res, float* C, int M,
                     int N, int K, int act, int a_lrelu, Workspace& ws, cudaStream_t s);
bool tc_tconv_tf32x3_supported(int B, int T, int V, int Cin, int Cout, int taps);
int tc_tconv_tf32x3(const float* X, const float* W, const float* bias, int bias_period, float* C, int B, int T, int V, int Cin,
                    int Cout, int taps, int tdiv, Workspace& ws, cudaStream_t s);

bool tc_attention_tf32x3_supported(int nq, int nkv, int dh);
// softmax(Q K^T / sqrt(dh)) V with both products as split-fp32 batched-head GEMMs; S is the caller's [B, H, nq, nkv] scratch
int tc_attention_tf32x3(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv, int B, int H, int nq, int nkv,
                        int dh, float* S, float* out, int ldo, Workspace& ws, cudaStream_t s);

// ---- attention: softmax(Q K^T / sqrt(dh)) V for B*H (batch, head) problems on tensor cores ------------
// q/k/v are fp32 strided views [B*n, ld] with head h at columns h*dh; S is a [B,H,nq,nkv] fp32 scratch.
bool tc_attention_supported(int nq, int nkv, int dh);
size_t tc_attention_scratch_bytes(int B, int H, int nq, int nkv, int dh);
int tc_attention(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv, int B, int H, int nq,
                 int nkv, int dh, float* S, float* out, int ldo, Workspace& ws, cudaStream_t s);
int tc_attention_ex(const float* q, const __nv_bfloat16* qh, int ldq, const float* k, const __nv_bfloat16* kh, int ldk,
                    const float* v, const __nv_bfloat16* vh, int ldv, int B, int H, int nq, int nkv, int dh, float* S,
                    TcOut out, int ldo, Workspace& ws, cudaStream_t s);

// ---- matcher coarse pass ---------------------------------------------------------------------------
constexpr int MATCH_KC_MAX = 16;
// Number of N-splits the coarse pass will use for (nq, N); candidates are [nq, splits, kc].
int tc_match_splits(int nq, long long N);
// Every coarse pass takes optional per-query segments (seg_first / seg_rows [nq], NULL = all N rows): query q's
// candidates are then the rows seg_first[q] .. + seg_rows[q] only (clipped to [0, N)).
// split-K coarse pass for small problems (0 slices = not applicable); candidates are [nq, round_up(N,128)]
int tc_match_splitk_slices(int nq, long long N, int D);
size_t tc_match_splitk_ws_bytes(int nq, long long N, int D);
int tc_match_coarse_splitk(const __nv_bfloat16* Q16, int nq, const __nv_bfloat16* DB16, const float* dbnorm, long long N,
                           int D, float* partial, float* cand_score, int32_t* cand_idx, const int64_t* seg_first,
                           const int32_t* seg_rows, cudaStream_t s);
// cand_score [nq, splits, kc] fp32 (ascending), cand_idx [nq, splits, kc] int32 (-1 = empty)
int tc_match_coarse(const __nv_bfloat16* Q16, int nq, const __nv_bfloat16* DB16, const float* dbnorm,
                    long long N, int D, int kc, float* cand_score, int32_t* cand_idx, const int64_t* seg_first,
                    const int32_t* seg_rows, cudaStream_t s);

// fp32-storage DB: same pass with fp32 operands consumed as TF32 (dbnorm = ||x||^2 of the fp32 rows)
int tc_match_coarse_tf32(const float* Q, int nq, const float* DB, const float* dbnorm, long long N, int D, int kc,
                         float* cand_score, int32_t* cand_idx, const int64_t* seg_first, const int32_t* seg_rows,
                         cudaStream_t s);

}  // namespace mocha
