// MOCHA_BF16 (throughput) orchestration of the Generator / CVAE stages: every dense contraction runs on
// tcgen05 and activations that only feed another tensor-core layer live in bf16 ONLY — the producing
// epilogue (or normalisation kernel) writes the bf16 operand of its consumer directly, so there are no
// stand-alone cast kernels and no fp32 round trips between layers. fp32 copies are kept exactly where
// a residual add, a normalisation or a SIMT kernel reads them. Same math as networks.cu (fp32 mode).
#include "networks_bf16.cuh"

#include "fused.cuh"
#include "gemm_f32.cuh"
#include "gemm_tc.cuh"
#include "ops.cuh"

namespace mocha {

namespace {

typedef __nv_bfloat16 bf16;

struct Tc {
  cudaStream_t s;
  Workspace& ws;
  // C = act(A16 W^T + bias) (+res); out.f32 and/or out.bf16
  int lin(const bf16* A16, int lda, const float* W, const float* bias, int period, const float* res, TcOut out, int M,
          int N, int K, int act) const {
    const bf16* W16 = tc_lookup_bf16(W);
    if (!W16) return set_error(MOCHA_ERR_ARG, "bf16 path: weight %p has no registered bf16 mirror", (const void*)W);
    return tc_linear_bf16(A16, lda, W16, bias, period, res, out, M, N, K, act, s);
  }
};

// One side stream + fork / join events per host thread (created on first use; creating them is not a stream operation, so it
// is legal while the caller's stream is being captured).
struct SideStream {
  cudaStream_t stream = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
};
SideStream* side_stream() {
  // one set per (host thread, device): a stream belongs to the device that was current when it was created
  constexpr int MAXDEV = 16;
  static thread_local SideStream per_dev[MAXDEV];
  static thread_local bool failed[MAXDEV] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MAXDEV) return nullptr;
  SideStream& ss = per_dev[dev];
  if (!ss.stream && !failed[dev]) {
    bool ok = cudaStreamCreateWithFlags(&ss.stream, cudaStreamNonBlocking) == cudaSuccess &&
              cudaEventCreateWithFlags(&ss.fork, cudaEventDisableTiming) == cudaSuccess &&
              cudaEventCreateWithFlags(&ss.join, cudaEventDisableTiming) == cudaSuccess;
    if (!ok) {
      failed[dev] = true;
      (void)cudaGetLastError();
    }
  }
  return failed[dev] ? nullptr : &ss;
}

inline TcOut f32(float* p) { return TcOut{p, nullptr, 0}; }
inline TcOut h16(bf16* p, int lrelu = 0) { return TcOut{nullptr, p, lrelu}; }
inline TcOut both(float* p, bf16* q) { return TcOut{p, q, 0}; }

#define WS_OK(ws, name)                                                                            \
  do {                                                                                             \
    if ((ws).overflow)                                                                             \
      return set_error(MOCHA_ERR_WORKSPACE, "%s: workspace too small (%zu B given, %zu B needed)", \
                       name, (ws).cap, (ws).off);                                                  \
  } while (0)

inline int ntok(const mocha_dims& d) { return (d.T / d.tp) * d.P; }

// the fused block tail (fused_tail.cu) is built for D = 256; other widths run the unfused launch sequence
// (out-projection, LayerNorm, FFN GEMMs)
inline bool use_fused_tail(int D) { return D == 256; }

// Attention of the bf16 path: one fused launch (fused_attn.cu) when the geometry fits, else the two-launch sequence
// (scores + softmax epilogue, P V) of gemm_tc.cu.
int attn(cudaStream_t s, Workspace& ws, const bf16* q, int ldq, const bf16* k, int ldk, const bf16* v, int ldv, int B, int H, int nq,
         int nkv, int dh, bf16* out, int ldo) {
  if (tc_attn_fused_supported(nq, nkv, dh) && ldo == H * dh)
    return tc_attn_fused(q, ldq, k, ldk, v, ldv, B, H, nq, nkv, dh, out, ldo, s);
  return tc_attention_ex(nullptr, q, ldq, nullptr, k, ldk, nullptr, v, ldv, B, H, nq, nkv, dh, nullptr, h16(out), ldo, ws, s);
}

// fused block tail (fused_tail.cu) on fp32 weight pointers: looks up the registered bf16 mirrors
int tail(cudaStream_t s, const bf16* A0, int K0, const float* W0, const float* b0, const float* R0, const float* g1,
         const float* be1, int Hd, int act, const float* W1, const float* b1, const float* W2, const float* b2,
         const float* g2, const float* be2, float eps, float* O32, bf16* O16, int M, int r0_period = 0) {
  const bf16* W016 = tc_lookup_bf16(W0);
  const bf16* W116 = Hd > 0 ? tc_lookup_bf16(W1) : nullptr;
  const bf16* W216 = Hd > 0 ? tc_lookup_bf16(W2) : nullptr;
  if (!W016 || (Hd > 0 && (!W116 || !W216)))
    return set_error(MOCHA_ERR_ARG, "bf16 path: a block-tail weight has no registered bf16 mirror");
  return tc_tail(A0, K0, K0, W016, b0, R0, g1, be1, Hd, act, W116, b1, W216, b2, g2, be2, eps, O32, O16, M, s, r0_period);
}

}  // namespace

bool bf16_path_supported(const mocha_dims& d) {
  const int n = ntok(d);
  return d.C0 % 64 == 0 && d.D % 64 == 0 && d.mlp % 64 == 0 && (d.Kj * d.C0) % 64 == 0 && d.enc_dh % 64 == 0 &&
         d.dec_dh % 64 == 0 && n <= 256 && tc_attention_supported(n, n, d.enc_dh) &&
         tc_attention_supported(n, n, d.dec_dh);
}

// ---------------------------------------------------------------------------------------------------
int embed_bf16(const mocha_generator_weights* w, const float* X, int B, float* tokens, int add_pos_emb, Workspace& ws,
               cudaStream_t s) {
  const mocha_dims& d = w->dims;
  Tc tc{s, ws};
  const int R = B * d.T * d.V, Tp = d.T / d.tp, R2 = B * Tp * d.P;
  bf16* h1 = ws.take<bf16>((size_t)R * d.D);
  bf16* agg2 = ws.take<bf16>((size_t)R2 * d.Kb * d.D);
  bf16* g2 = ws.take<bf16>((size_t)R2 * d.D);
  WS_OK(ws, "mocha_embed_fwd(bf16)");
  const int KC = d.Kj * d.C0;
  if (w->jb_gcn_w_aug && w->jb_gcn_kaug >= KC + d.Kj && w->jb_gcn_kaug % 16 == 0 && (d.taps_j & 1)) {
    // bias folded into the GEMM (Kj extra K columns x adjacency column sums) -> plain single-pass epilogue,
    // and the GEMM's TMA stores land directly in the interior of the temporal conv's reflect-padded input
    const int Ka = w->jb_gcn_kaug, pad = d.taps_j / 2, Tpad = d.T + 2 * pad;
    const __nv_bfloat16* W16 = tc_lookup_bf16(w->jb_gcn_w_aug);
    if (!W16) return set_error(MOCHA_ERR_ARG, "mocha_embed_fwd: jb_gcn_w_aug has no registered bf16 mirror");
    bf16* agga = ws.take<bf16>((size_t)R * Ka);
    bf16* gpad = ws.take<bf16>((size_t)B * Tpad * d.V * d.D);
    WS_OK(ws, "mocha_embed_fwd(bf16)");
    MOCHA_TRY(embed_graph_agg(X, w->emb_w, w->emb_b, w->A_j, agga, B * d.T, d.V, d.Cin, d.C0, d.Kj, s, Ka));
    MOCHA_TRY(tc_linear_bf16_img(agga, Ka, W16, nullptr, h16(gpad + (size_t)pad * d.V * d.D), B, d.T * d.V,
                                 (long long)Tpad * d.V, d.D, Ka, ACT_NONE, s));
    MOCHA_TRY(reflect_border_fill(gpad, B, d.T, pad, (long long)d.V * d.D, s));
    MOCHA_TRY(tc_tconv_ex(nullptr, gpad, w->jb_tcn_w, w->jb_tcn_b, 0, h16(h1), B, d.T, d.V, d.D, d.D, d.taps_j, 1, ws, s, 1, true));
  } else {
    // Conv2d 1x1 Cin(15)->C0 + LeakyReLU + graph aggregation in one kernel (K = 15 is too short for a TMA row)
    bf16* agg = ws.take<bf16>((size_t)R * KC);
    bf16* g = ws.take<bf16>((size_t)R * d.D);
    WS_OK(ws, "mocha_embed_fwd(bf16)");
    MOCHA_TRY(embed_graph_agg(X, w->emb_w, w->emb_b, w->A_j, agg, B * d.T, d.V, d.Cin, d.C0, d.Kj, s));
    MOCHA_TRY(tc.lin(agg, KC, w->jb_gcn_w, w->jb_gcn_bias2d, d.V, nullptr, h16(g), R, d.D, KC, ACT_NONE));
    MOCHA_TRY(tc_tconv_ex(nullptr, g, w->jb_tcn_w, w->jb_tcn_b, 0, h16(h1), B, d.T, d.V, d.D, d.D, d.taps_j, 1, ws, s));
  }
  // joint -> body-part pooling + the BodyBlock's LeakyReLU and graph aggregation in one pass over h1
  MOCHA_TRY(pool_graph_agg(h1, w->pool_w, w->A_b, agg2, B, d.T, d.V, d.P, d.D, d.tp, d.Kb, s));
  MOCHA_TRY(tc.lin(agg2, d.Kb * d.D, w->bb_gcn_w, w->bb_gcn_bias2d, d.P, nullptr, h16(g2), R2, d.D, d.Kb * d.D, ACT_NONE));
  if (add_pos_emb)
    return tc_tconv_ex(nullptr, g2, w->bb_tcn_w, w->tok_bias_pos, Tp * d.P, f32(tokens), B, Tp, d.P, d.D, d.D, d.taps_b, 1, ws, s);
  return tc_tconv_ex(nullptr, g2, w->bb_tcn_w, w->bb_tcn_b, 0, f32(tokens), B, Tp, d.P, d.D, d.D, d.taps_b, 1, ws, s);
}

// ---------------------------------------------------------------------------------------------------
int encoder_bf16(const mocha_generator_weights* w, const float* tokens, int B, float* encoded, Workspace& ws,
                 cudaStream_t s) {
  const mocha_dims& d = w->dims;
  Tc tc{s, ws};
  const int n = ntok(d), R = B * n, inner = d.heads * d.enc_dh;
  bf16* x16 = ws.take<bf16>((size_t)R * d.D);
  bf16* qkv = ws.take<bf16>((size_t)R * 3 * inner);
  float* S = nullptr;   // scores stay in TMEM (softmax fused into the Q K^T epilogue)
  bf16* att = ws.take<bf16>((size_t)R * inner);
  float* xa = ws.take<float>((size_t)R * d.D);
  bf16* xa16 = ws.take<bf16>((size_t)R * d.D);
  float* xb = ws.take<float>((size_t)R * d.D);
  bf16* hid = ws.take<bf16>((size_t)R * d.mlp);
  WS_OK(ws, "mocha_encoder_fwd(bf16)");
  MOCHA_TRY(tc_cast(tokens, x16, (long long)R * d.D, 0, s));
  const float* x = tokens;
  for (int l = 0; l < d.enc_depth; ++l) {
    const mocha_enc_layer& L = w->enc[l];
    MOCHA_CHECK_ARG(L.wqkv && L.wo && L.bo && L.w1 && L.b1 && L.w2 && L.b2, "mocha_encoder_fwd: layer %d weights missing", l);
    const bool last = l == d.enc_depth - 1;
    MOCHA_TRY(tc.lin(x16, d.D, L.wqkv, nullptr, 0, nullptr, h16(qkv), R, 3 * inner, d.D, ACT_NONE));
    MOCHA_TRY(attn(s, ws, qkv, 3 * inner, qkv + inner, 3 * inner, qkv + 2 * inner, 3 * inner, B, d.heads, n, n, d.enc_dh, att, inner));
    float* dst = last ? encoded : xb;
    if (use_fused_tail(d.D) && tc_tail_supported(R, inner, d.mlp)) {
      // out-projection + residual + GELU FFN + residual in one launch (x and dst may alias: tiles are row-local)
      MOCHA_TRY(tail(s, att, inner, L.wo, L.bo, x, nullptr, nullptr, d.mlp, ACT_GELU, L.w1, L.b1, L.w2, L.b2, nullptr, nullptr,
                     0.f, dst, last ? nullptr : x16, R));
    } else {
      MOCHA_TRY(tc.lin(att, inner, L.wo, L.bo, 0, x, both(xa, xa16), R, d.D, inner, ACT_NONE));
      MOCHA_TRY(tc.lin(xa16, d.D, L.w1, L.b1, 0, nullptr, h16(hid), R, d.mlp, d.D, ACT_GELU));
      MOCHA_TRY(tc.lin(hid, d.mlp, L.w2, L.b2, 0, xa, last ? f32(dst) : both(dst, x16), R, d.D, d.mlp, ACT_NONE));
    }
    x = dst;
  }
  return MOCHA_OK;
}

// ---------------------------------------------------------------------------------------------------
int decoder_bf16(const mocha_generator_weights* w, const float* src, const float* cha, int B, float* decoded,
                 Workspace& ws, cudaStream_t s) {
  const mocha_dims& d = w->dims;
  Tc tc{s, ws};
  const int n = ntok(d), R = B * n, inner = d.heads * d.dec_dh;
  const float eps = 1e-5f;
  float* smean = ws.take<float>((size_t)B * d.D);
  bf16* smean16 = ws.take<bf16>((size_t)B * d.D);
  bf16* shid = ws.take<bf16>((size_t)B * 2 * d.D);
  float* gb_all = ws.take<float>((size_t)d.dec_depth * B * 2 * d.D);
  // the three projection inputs and outputs are stacked so that q / k / v run as ONE grouped GEMM launch
  bf16* in3 = ws.take<bf16>((size_t)3 * R * d.D);          // [IN(x1) | IN(style) | style]
  bf16* qin = in3;
  bf16* sty_in = in3 + (size_t)R * d.D;
  bf16* cha16 = in3 + (size_t)2 * R * d.D;
  float* x1 = ws.take<float>((size_t)R * d.D);
  float* x2 = ws.take<float>((size_t)R * d.D);
  bf16* x2h = ws.take<bf16>((size_t)R * d.D);
  float* xb = ws.take<float>((size_t)R * d.D);
  bf16* qkv3 = ws.take<bf16>((size_t)3 * R * inner);
  bf16* q = qkv3;
  bf16* k = qkv3 + (size_t)R * inner;
  bf16* v = qkv3 + (size_t)2 * R * inner;
  bf16* att = ws.take<bf16>((size_t)R * inner);
  float* S = nullptr;   // scores stay in TMEM (softmax fused into the Q K^T epilogue)
  bf16* hid = ws.take<bf16>((size_t)R * d.mlp);
  WS_OK(ws, "mocha_decoder_fwd(bf16)");
  // layer-independent functions of the style tokens
  // AdaIN parameters of every layer depend on the style only: one launch for the token mean and all MLPs
  bool fused_style = style_mlp_supported(d.D, d.dec_depth);
  const bf16 *w1[MOCHA_MAX_DEPTH], *w2[MOCHA_MAX_DEPTH];
  const float *b1[MOCHA_MAX_DEPTH], *b2[MOCHA_MAX_DEPTH];
  for (int l = 0; l < d.dec_depth && fused_style; ++l) {
    MOCHA_CHECK_ARG(w->dec[l].sw1 && w->dec[l].sw2, "mocha_decoder_fwd: layer %d weights missing", l);
    w1[l] = tc_lookup_bf16(w->dec[l].sw1); w2[l] = tc_lookup_bf16(w->dec[l].sw2);
    b1[l] = w->dec[l].sb1; b2[l] = w->dec[l].sb2;
    fused_style = w1[l] && w2[l];
  }
  // The style MLP (128 blocks, L2-latency-bound) and the two token-wise passes over the style (instance norm, bf16 copy)
  // are independent: the latter run on a side stream that forks from and joins the caller's stream through events, so the
  // fork is captured into a CUDA graph like any other dependency.
  SideStream* side = fused_style ? side_stream() : nullptr;
  cudaStream_t s2 = s;
  if (side) {
    MOCHA_CUDA(cudaEventRecord(side->fork, s));
    MOCHA_CUDA(cudaStreamWaitEvent(side->stream, side->fork, 0));
    s2 = side->stream;
  }
  if (fused_style) {
    MOCHA_TRY(style_mlp(cha, B, n, d.D, d.dec_depth, w1, b1, w2, b2, gb_all, s));
  } else {
    MOCHA_TRY(token_mean(cha, B, n, d.D, smean, s));
    MOCHA_TRY(tc_cast(smean, smean16, (long long)B * d.D, 0, s));
  }
  MOCHA_TRY(instance_norm_tokens(cha, B, n, d.D, eps, nullptr, nullptr, nullptr, nullptr, nullptr, s2, sty_in));
  MOCHA_TRY(tc_cast(cha, cha16, (long long)R * d.D, 0, s2));
  if (side) {
    MOCHA_CUDA(cudaEventRecord(side->join, side->stream));
    MOCHA_CUDA(cudaStreamWaitEvent(s, side->join, 0));
  }
  const float* x = src;
  for (int l = 0; l < d.dec_depth; ++l) {
    const mocha_dec_layer& L = w->dec[l];
    MOCHA_CHECK_ARG(L.sw1 && L.sw2 && L.wq && L.wk && L.wv && L.wo && L.w1 && L.w2, "mocha_decoder_fwd: layer %d weights missing", l);
    float* gb = gb_all + (size_t)l * B * 2 * d.D;
    if (!fused_style) {
      MOCHA_TRY(tc.lin(smean16, d.D, L.sw1, L.sb1, 0, nullptr, h16(shid), B, 2 * d.D, d.D, ACT_LRELU));
      MOCHA_TRY(tc.lin(shid, 2 * d.D, L.sw2, L.sb2, 0, nullptr, f32(gb), B, 2 * d.D, 2 * d.D, ACT_NONE));
    }
    if (n <= 128 && d.D % 64 == 0) {
      // x1 = AdaIN(x) and qin = IN(x1) from one pass (closed form for the second normalisation)
      MOCHA_TRY(adain_norm_tokens(x, B, n, d.D, eps, gb, x1, qin, s));
    } else {
      MOCHA_TRY(instance_norm_tokens(x, B, n, d.D, eps, gb, x1, nullptr, nullptr, nullptr, s));
      MOCHA_TRY(instance_norm_tokens(x1, B, n, d.D, eps, nullptr, nullptr, nullptr, nullptr, nullptr, s, qin));
    }
    const bf16* wq16 = tc_lookup_bf16(L.wq);
    if (wq16 && L.wk == L.wq + (size_t)inner * d.D && L.wv == L.wk + (size_t)inner * d.D && inner % 64 == 0) {
      // to_q / to_k / to_v sit back to back in the packed blob: three inputs x three weights in one launch
      MOCHA_TRY(tc_linear_bf16_grouped(in3, wq16, qkv3, 3, R, inner, d.D, s));
    } else {
      MOCHA_TRY(tc.lin(qin, d.D, L.wq, nullptr, 0, nullptr, h16(q), R, inner, d.D, ACT_NONE));
      MOCHA_TRY(tc.lin(sty_in, d.D, L.wk, nullptr, 0, nullptr, h16(k), R, inner, d.D, ACT_NONE));
      MOCHA_TRY(tc.lin(cha16, d.D, L.wv, nullptr, 0, nullptr, h16(v), R, inner, d.D, ACT_NONE));
    }
    MOCHA_TRY(attn(s, ws, q, inner, k, inner, v, inner, B, d.heads, n, n, d.dec_dh, att, inner));
    float* dst = (l == d.dec_depth - 1) ? decoded : xb;
    if (use_fused_tail(d.D) && tc_tail_supported(R, inner, d.mlp)) {
      MOCHA_TRY(tail(s, att, inner, L.wo, L.bo, x1, nullptr, nullptr, d.mlp, ACT_GELU, L.w1, L.b1, L.w2, L.b2, nullptr, nullptr,
                     0.f, dst, nullptr, R));
    } else {
      MOCHA_TRY(tc.lin(att, inner, L.wo, L.bo, 0, x1, both(x2, x2h), R, d.D, inner, ACT_NONE));
      MOCHA_TRY(tc.lin(x2h, d.D, L.w1, L.b1, 0, nullptr, h16(hid), R, d.mlp, d.D, ACT_GELU));
      MOCHA_TRY(tc.lin(hid, d.mlp, L.w2, L.b2, 0, x2, f32(dst), R, d.D, d.mlp, ACT_NONE));
    }
    x = dst;
  }
  return MOCHA_OK;
}

// ---------------------------------------------------------------------------------------------------
int to_mot_bf16(const mocha_generator_weights* w, const float* tokens, int B, float* Ytil, const float* Y_mean,
                const float* Y_std, float* Y, Workspace& ws, cudaStream_t s) {
  const mocha_dims& d = w->dims;
  Tc tc{s, ws};
  const int Tp = d.T / d.tp, R2 = B * Tp * d.P, R = B * d.T * d.V;
  bf16* agg = ws.take<bf16>((size_t)R2 * d.Kb * d.D);
  bf16* y1 = ws.take<bf16>((size_t)R2 * d.D);
  bf16* y2 = ws.take<bf16>((size_t)R2 * d.D);
  float* y3 = ws.take<float>((size_t)R2 * d.Kj * d.C0);
  const int padj = d.taps_j / 2;
  bf16* gp16 = ws.take<bf16>((size_t)B * (d.T + 2 * padj) * d.V * d.C0);   // reflect-padded, up-sampled conv input
  bf16* y4 = ws.take<bf16>((size_t)R * d.C0);
  // the 64 -> Cin(15) output conv writes rows padded to 16 floats so that its epilogue can use TMA stores;
  // the de-normalisation pass below reads the padded rows and emits the dense tensors
  const int Cp = (d.Cin + 7) / 8 * 8;
  float* ytp = ws.take<float>((size_t)R * Cp);
  WS_OK(ws, "mocha_to_mot_fwd(bf16)");
  MOCHA_TRY(graph_agg_first(tokens, w->tm_A_b, nullptr, B * Tp, d.P, d.D, d.Kb, 1, s, agg));
  MOCHA_TRY(tc.lin(agg, d.Kb * d.D, w->tm_bb_gcn_w, w->tm_bb_gcn_bias2d, d.P, nullptr, h16(y1), R2, d.D, d.Kb * d.D, ACT_NONE));
  // the two consumers below are pre-activation blocks: their bf16 operand is stored through LeakyReLU
  MOCHA_TRY(tc_tconv_ex(nullptr, y1, w->tm_bb_tcn_w, w->tm_bb_tcn_b, 0, h16(y2, 1), B, Tp, d.P, d.D, d.D, d.taps_b, 1, ws, s));
  MOCHA_TRY(tc.lin(y2, d.D, w->tm_jb_gcn_w, w->tm_jb_gcn_b, 0, nullptr, f32(y3), R2, d.Kj * d.C0, d.D, ACT_NONE));
  MOCHA_TRY(graph_agg_kv_pad16(y3, w->tm_A2, gp16, B, Tp, d.tp, padj, d.P, d.V, d.C0, d.Kj, s));
  MOCHA_TRY(tc_tconv_ex(nullptr, gp16, w->tm_jb_tcn_w, w->tm_jb_tcn_b, 0, h16(y4, 1), B, d.T, d.V, d.C0, d.C0, d.taps_j, 1, ws, s, 1,
                        true));
  if (out_conv_affine_supported(d.C0, d.Cin) && (Y || Ytil))
    return out_conv_affine(y4, w->tm_out_w, w->tm_out_b, Y_mean, Y_std, Ytil, Y, R, d.C0, d.Cin, d.V, s);
  MOCHA_TRY(tc.lin(y4, d.C0, w->tm_out_w, w->tm_out_b, 0, nullptr, f32(ytp), R, Cp, d.C0, ACT_NONE));
  if (Y || Ytil) MOCHA_TRY(affine_rows(ytp, Y_mean, Y_std, Y, R, d.Cin, d.V, s, Cp, Ytil));
  return MOCHA_OK;
}

// ---------------------------------------------------------------------------------------------------
int cvae_bf16(const mocha_cvae_weights* w, const float* cond, int B, int ncond, const float* eps, float* out, float* mu,
              float* logvar, const float* out_mean, const float* out_std, float* out_denorm, Workspace& ws,
              cudaStream_t s) {
  Tc tc{s, ws};
  const int D = w->D, H = w->heads, dh = D / H, np = ncond + 2, nm = ncond + 1, nq = w->out_seq;
  const int Rp = B * np, Rm = B * nm, Rq = B * nq;
  float* xa = ws.take<float>((size_t)Rp * D);
  float* xb = ws.take<float>((size_t)Rp * D);
  bf16* xa16 = ws.take<bf16>((size_t)Rp * D);
  bf16* xb16 = ws.take<bf16>((size_t)Rp * D);
  bf16* qkv = ws.take<bf16>((size_t)Rp * 3 * D);
  float* S = nullptr;   // scores stay in TMEM (softmax fused into the Q K^T epilogue)
  bf16* att = ws.take<bf16>((size_t)Rp * D);
  float* proj = ws.take<float>((size_t)Rp * D);
  bf16* hid = ws.take<bf16>((size_t)Rp * w->dff);
  bf16* mem = ws.take<bf16>((size_t)Rm * D);
  bf16* memkv = ws.take<bf16>((size_t)Rm * 2 * D);
  // memory K | V of the decoder layers after the first depend on `mem` only: they are projected on a side stream while
  // layer 0 runs (its 90-CTA block tails leave 58 SMs idle)
  bf16* memkv_ahead[MOCHA_MAX_DEPTH] = {nullptr, nullptr, nullptr, nullptr};
  for (int l = 1; l < w->depth; ++l) memkv_ahead[l] = ws.take<bf16>((size_t)Rm * 2 * D);
  bf16* dq = ws.take<bf16>((size_t)Rq * D);
  WS_OK(ws, "mocha_cvae_sample(bf16)");

  // ---- prior network: x (fp32 for the residual / LayerNorm) + x16 (operand of the next GEMM) ----
  MOCHA_TRY(cvae_prior_tokens(w->mu_token, w->logvar_token, cond, w->pe, xa, B, ncond, D, s, xa16));
  float* x = xa; bf16* x16 = xa16;
  float* y = xb; bf16* y16 = xb16;
  int prior_rows = np;  // rows per batch element in the prior's output tensor
  for (int l = 0; l < w->depth; ++l) {
    const mocha_cvae_enc_layer& L = w->prior[l];
    MOCHA_CHECK_ARG(L.in_w && L.in_b && L.out_w && L.out_b && L.l1_w && L.l2_w && L.n1_g && L.n2_g,
                    "mocha_cvae_sample: prior layer %d weights missing", l);
    if (l == w->depth - 1) {
      // Only the mu / logvar rows (tokens 0 and 1) of the last layer are ever read (model_CVAE.py:78):
      // keys / values still span all tokens, but queries, out-proj, LayerNorms and the FFN run on 2 rows.
      const int R2 = 2 * B;
      float* xq = y;          // [2B, D] gathered rows of x (residual)
      bf16* xq16 = y16;
      bf16* kv = qkv;         // [Rp, 2D]
      const bf16 *wq16 = tc_lookup_bf16(L.in_w), *wo16 = tc_lookup_bf16(L.out_w), *w116 = tc_lookup_bf16(L.l1_w),
                 *w216 = tc_lookup_bf16(L.l2_w);
      if (cvae_prior_last_supported(D, H, w->dff, np) && wq16 && wo16 && w116 && w216 && L.n1_b && L.n2_b) {
        // everything after the K / V projection acts on 2 rows per clip: one SIMT launch (ops.cu)
        MOCHA_TRY(tc.lin(x16, D, L.in_w + (size_t)D * D, L.in_b + D, 0, nullptr, h16(kv), Rp, 2 * D, D, ACT_NONE));
        MOCHA_TRY(cvae_prior_last(x, B, np, kv, wq16, L.in_b, wo16, L.out_b, L.n1_g, L.n1_b, w116, L.l1_b, w216, L.l2_b, L.n2_g,
                                  L.n2_b, H, w->dff, w->ln_eps, xq, s));
        x = xq;
        prior_rows = 2;
        break;
      }
      MOCHA_TRY(gather_token_rows(x, x16, np, 2, D, B, xq, xq16, s));
      bf16* q2 = att;         // [2B, D]
      bf16* att2 = hid;       // [2B, D]
      MOCHA_TRY(tc.lin(x16, D, L.in_w + (size_t)D * D, L.in_b + D, 0, nullptr, h16(kv), Rp, 2 * D, D, ACT_NONE));
      MOCHA_TRY(tc.lin(xq16, D, L.in_w, L.in_b, 0, nullptr, h16(q2), R2, D, D, ACT_NONE));
      MOCHA_TRY(attn(s, ws, q2, D, kv, 2 * D, kv + D, 2 * D, B, H, 2, np, dh, att2, D));
      if (use_fused_tail(D) && tc_tail_supported(R2, D, w->dff)) {
        MOCHA_TRY(tail(s, att2, D, L.out_w, L.out_b, xq, L.n1_g, L.n1_b, w->dff, ACT_RELU, L.l1_w, L.l1_b, L.l2_w, L.l2_b,
                       L.n2_g, L.n2_b, w->ln_eps, xq, nullptr, R2));
      } else {
        MOCHA_TRY(tc.lin(att2, D, L.out_w, L.out_b, 0, xq, f32(proj), R2, D, D, ACT_NONE));
        float* y2 = proj + (size_t)R2 * D;       // proj has Rp*D floats: plenty of room for the 2-row tensors
        bf16* y2h = q2;
        MOCHA_TRY(add_layernorm(proj, nullptr, L.n1_g, L.n1_b, y2, R2, D, w->ln_eps, nullptr, nullptr, 0, nullptr, s, y2h));
        bf16* hid2 = att2 + (size_t)R2 * D;
        MOCHA_TRY(tc.lin(y2h, D, L.l1_w, L.l1_b, 0, nullptr, h16(hid2), R2, w->dff, D, ACT_RELU));
        MOCHA_TRY(tc.lin(hid2, w->dff, L.l2_w, L.l2_b, 0, y2, f32(proj), R2, D, w->dff, ACT_NONE));
        MOCHA_TRY(add_layernorm(proj, nullptr, L.n2_g, L.n2_b, xq, R2, D, w->ln_eps, nullptr, nullptr, 0, nullptr, s));
      }
      x = xq;
      prior_rows = 2;
      break;
    }
    MOCHA_TRY(tc.lin(x16, D, L.in_w, L.in_b, 0, nullptr, h16(qkv), Rp, 3 * D, D, ACT_NONE));
    MOCHA_TRY(attn(s, ws, qkv, 3 * D, qkv + D, 3 * D, qkv + 2 * D, 3 * D, B, H, np, np, dh, att, D));
    if (use_fused_tail(D) && tc_tail_supported(Rp, D, w->dff)) {
      // x <- LN2(y + FF(y)), y = LN1(x + SA(x)): one launch, in place (tiles are row-local)
      MOCHA_TRY(tail(s, att, D, L.out_w, L.out_b, x, L.n1_g, L.n1_b, w->dff, ACT_RELU, L.l1_w, L.l1_b, L.l2_w, L.l2_b, L.n2_g,
                     L.n2_b, w->ln_eps, x, x16, Rp));
    } else {
      MOCHA_TRY(tc.lin(att, D, L.out_w, L.out_b, 0, x, f32(proj), Rp, D, D, ACT_NONE));      // proj = x + SA(x)
      MOCHA_TRY(add_layernorm(proj, nullptr, L.n1_g, L.n1_b, y, Rp, D, w->ln_eps, nullptr, nullptr, 0, nullptr, s, y16));
      MOCHA_TRY(tc.lin(y16, D, L.l1_w, L.l1_b, 0, nullptr, h16(hid), Rp, w->dff, D, ACT_RELU));
      MOCHA_TRY(tc.lin(hid, w->dff, L.l2_w, L.l2_b, 0, y, f32(proj), Rp, D, w->dff, ACT_NONE)); // proj = y + FF(y)
      MOCHA_TRY(add_layernorm(proj, nullptr, L.n2_g, L.n2_b, x, Rp, D, w->ln_eps, nullptr, nullptr, 0, nullptr, s, x16));
    }
  }
  MOCHA_TRY(cvae_memory(x, prior_rows, eps, cond, nullptr, mu, logvar, B, ncond, D, s, mem));
  SideStream* side = w->depth > 1 ? side_stream() : nullptr;
  bool ahead_pending = false;
  if (side) {
    MOCHA_CUDA(cudaEventRecord(side->fork, s));
    MOCHA_CUDA(cudaStreamWaitEvent(side->stream, side->fork, 0));
    Tc tc2{side->stream, ws};
    for (int l = 1; l < w->depth; ++l) {
      const mocha_cvae_dec_layer& L = w->dec[l];
      MOCHA_CHECK_ARG(L.ca_in_w && L.ca_in_b, "mocha_cvae_sample: decoder layer %d weights missing", l);
      MOCHA_TRY(tc2.lin(mem, D, L.ca_in_w + (size_t)D * D, L.ca_in_b + D, 0, nullptr, h16(memkv_ahead[l]), Rm, 2 * D, D, ACT_NONE));
    }
    MOCHA_CUDA(cudaEventRecord(side->join, side->stream));
    ahead_pending = true;
  }

  // ---- decoder (query rows reuse the prior's buffers: Rq <= Rp) ----
  float* dx = xa; bf16* dx16 = xa16;
  float* dy = xb; bf16* dy16 = xb16;
  if (!w->dec0_sa) MOCHA_TRY(broadcast_rows(w->pe, dx, B, (long long)nq * D, s, dx16));
  for (int l = 0; l < w->depth; ++l) {
    const mocha_cvae_dec_layer& L = w->dec[l];
    MOCHA_CHECK_ARG(L.sa_in_w && L.sa_out_w && L.ca_in_w && L.ca_out_w && L.l1_w && L.l2_w && L.n1_g && L.n2_g && L.n3_g,
                    "mocha_cvae_sample: decoder layer %d weights missing", l);
    const bool fused = use_fused_tail(D) && tc_tail_supported(Rq, D, w->dff);
    const bool last = l == w->depth - 1;
    // Layer 0 with both cached tables: the query rows are the same for every clip, so neither the broadcast [B, nq, D]
    // tensor nor its per-clip projection is materialised - the attention kernel reads the shared bf16 query table and the
    // block tail reads the fp32 table as a periodic residual.
    const bool shared_q = l == 0 && w->dec0_sa && w->dec0_q16 && fused && tc_attn_fused_supported(nq, nm, dh);
    const float* res_cross = dy;
    int res_period = 0;
    if (shared_q) {
      MOCHA_TRY(tc.lin(mem, D, L.ca_in_w + (size_t)D * D, L.ca_in_b + D, 0, nullptr, h16(memkv), Rm, 2 * D, D, ACT_NONE));
      MOCHA_TRY(tc_attn_fused((const bf16*)w->dec0_q16, D, memkv, 2 * D, memkv + D, 2 * D, B, H, nq, nm, dh, att, D, s, true));
      res_cross = w->dec0_sa;
      res_period = nq;
    } else {
    if (l == 0 && w->dec0_sa) {
      // layer 0's self-attention block acts on the constant query: cached table (mocha_cvae_precompute_dec0)
      MOCHA_TRY(broadcast_rows(w->dec0_sa, dy, B, (long long)nq * D, s, dy16));
    } else {
      MOCHA_TRY(tc.lin(dx16, D, L.sa_in_w, L.sa_in_b, 0, nullptr, h16(qkv), Rq, 3 * D, D, ACT_NONE));
      MOCHA_TRY(attn(s, ws, qkv, 3 * D, qkv + D, 3 * D, qkv + 2 * D, 3 * D, B, H, nq, nq, dh, att, D));
      if (use_fused_tail(D) && tc_tail_supported(Rq, D, 0)) {
        MOCHA_TRY(tail(s, att, D, L.sa_out_w, L.sa_out_b, dx, L.n1_g, L.n1_b, 0, ACT_NONE, nullptr, nullptr, nullptr, nullptr,
                       nullptr, nullptr, w->ln_eps, dy, dy16, Rq));
      } else {
        MOCHA_TRY(tc.lin(att, D, L.sa_out_w, L.sa_out_b, 0, dx, f32(proj), Rq, D, D, ACT_NONE));
        MOCHA_TRY(add_layernorm(proj, nullptr, L.n1_g, L.n1_b, dy, Rq, D, w->ln_eps, nullptr, nullptr, 0, nullptr, s, dy16));
      }
    }
    MOCHA_TRY(tc.lin(dy16, D, L.ca_in_w, L.ca_in_b, 0, nullptr, h16(dq), Rq, D, D, ACT_NONE));
    const bf16* mkv = memkv;
    if (side && l >= 1) {
      if (ahead_pending) { MOCHA_CUDA(cudaStreamWaitEvent(s, side->join, 0)); ahead_pending = false; }
      mkv = memkv_ahead[l];
    } else {
      MOCHA_TRY(tc.lin(mem, D, L.ca_in_w + (size_t)D * D, L.ca_in_b + D, 0, nullptr, h16(memkv), Rm, 2 * D, D, ACT_NONE));
    }
    MOCHA_TRY(attn(s, ws, dq, D, mkv, 2 * D, mkv + D, 2 * D, B, H, nq, nm, dh, att, D));
    }
    if (fused) {
      // cross-attention out-projection + LN2 + ReLU FFN (+ LN3 unless the de-normalising last LayerNorm follows)
      MOCHA_TRY(tail(s, att, D, L.ca_out_w, L.ca_out_b, res_cross, L.n2_g, L.n2_b, w->dff, ACT_RELU, L.l1_w, L.l1_b, L.l2_w, L.l2_b,
                     last ? nullptr : L.n3_g, last ? nullptr : L.n3_b, w->ln_eps, last ? proj : dy, last ? nullptr : dy16, Rq,
                     res_period));
      if (!last) {
        float* t = dx; dx = dy; dy = t;
        bf16* t16 = dx16; dx16 = dy16; dy16 = t16;
        continue;
      }
    } else {
      MOCHA_TRY(tc.lin(att, D, L.ca_out_w, L.ca_out_b, 0, dy, f32(proj), Rq, D, D, ACT_NONE));
      MOCHA_TRY(add_layernorm(proj, nullptr, L.n2_g, L.n2_b, dx, Rq, D, w->ln_eps, nullptr, nullptr, 0, nullptr, s, dx16));
      MOCHA_TRY(tc.lin(dx16, D, L.l1_w, L.l1_b, 0, nullptr, h16(hid), Rq, w->dff, D, ACT_RELU));
      MOCHA_TRY(tc.lin(hid, w->dff, L.l2_w, L.l2_b, 0, dx, f32(proj), Rq, D, w->dff, ACT_NONE));
    }
    if (l == w->depth - 1) {
      MOCHA_TRY(add_layernorm(proj, nullptr, L.n3_g, L.n3_b, out, Rq, D, w->ln_eps, out_mean, out_std, nq, out_denorm, s));
    } else {
      MOCHA_TRY(add_layernorm(proj, nullptr, L.n3_g, L.n3_b, dy, Rq, D, w->ln_eps, nullptr, nullptr, 0, nullptr, s, dy16));
      float* t = dx; dx = dy; dy = t;
      bf16* t16 = dx16; dx16 = dy16; dy16 = t16;
    }
  }
  if (side && ahead_pending) MOCHA_CUDA(cudaStreamWaitEvent(s, side->join, 0));
  return MOCHA_OK;
}

}  // namespace mocha
