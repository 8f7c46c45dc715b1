/*
 * mocha_b200.h — C ABI of libmocha_b200.so: the B200 (sm_100a) implementation of MOCHA's per-frame
 * characterization hot path (SURVEY.md §8a rows a1–a18).
 *
 * The reference (DK-Jang/MOCHA_SIGASIA2023) is pure Python and has no FFI of its own; the entry
 * points below are the operator boundary its Python call sites would bind (ctypes stubs in
 * INTEGRATION.md). Each function cites the reference call site / definition it replaces
 * (paths relative to the reference tree).
 *
 * Conventions
 *  - Every pointer named d_* / inside the weight structs is a DEVICE pointer owned by the caller.
 *    The library never allocates or frees device memory on the data path; scratch is passed in as
 *    (workspace, workspace_bytes) sized by the matching *_workspace_bytes() query.
 *  - All work is enqueued on `stream` (a cudaStream_t passed as void*); functions never synchronise
 *    and are safe under CUDA-graph capture. Weights are borrowed and must outlive the enqueued work.
 *  - Return value: 0 on success, negative on error (MOCHA_ERR_*); the message is available from
 *    mocha_last_error(). No exception crosses the boundary and there is NO CPU fallback: on a
 *    machine without an sm_100 device every compute entry point fails with MOCHA_ERR_ARCH/CUDA.
 *  - Layouts are channel-last and contiguous: pose windows [B,T,V,C] exactly as the reference feeds
 *    Generator.mot_embedding ('b t v c', model.py:43), token tensors [B,n,C], quaternions [w,x,y,z].
 *  - precision: MOCHA_FP32 computes every contraction in fp32 FFMA (parity mode, 1e-4 rel);
 *    MOCHA_BF16 runs the dense contractions on tcgen05 tensor cores with bf16 operands and fp32
 *    accumulation in TMEM (throughput mode, 2e-2 rel); MOCHA_TF32X3 is the parity mode on the tensor
 *    cores: every linear layer and temporal convolution splits its fp32 operands into tf32 hi / lo parts
 *    and runs a . w = a_hi w_hi + a_lo w_hi + a_hi w_lo as one tcgen05 kind::tf32 GEMM over a 3x longer K
 *    (fp32 accumulation in TMEM, same 1e-4 tolerance as MOCHA_FP32; attention products and the matcher
 *    stay on the fp32 / fp64 kernels). Its split operands live in whatever workspace is left after the
 *    stage's own buffers; long layers run as row chunks when that is short.
 */
#ifndef MOCHA_B200_H_
#define MOCHA_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MOCHA_OK 0
#define MOCHA_ERR_ARG (-1)
#define MOCHA_ERR_CUDA (-2)
#define MOCHA_ERR_WORKSPACE (-3)
#define MOCHA_ERR_ARCH (-4)
#define MOCHA_ERR_UNSUPPORTED (-5)

#define MOCHA_FP32 0
#define MOCHA_BF16 1
#define MOCHA_TF32X3 2

#define MOCHA_MAX_DEPTH 4

typedef void* mocha_stream_t; /* cudaStream_t */

/* ---- library ------------------------------------------------------------------------------ */
const char* mocha_last_error(void);
int mocha_version(void);
/* 0 if the current device is sm_100 (B200), MOCHA_ERR_ARCH otherwise. */
int mocha_check_device(void);
/* number of kernels this library launched since the last reset (bench.py "gpu_launches") */
long long mocha_launch_count(void);
void mocha_reset_launch_count(void);

/* sizeof() of the ABI structs in declaration order (dims, enc_layer, dec_layer, generator_weights,
 * cvae_enc_layer, cvae_dec_layer, cvae_weights, clip_state, post_params, frame_out): lets a binding
 * check its mirrored definitions at load time. */
int mocha_struct_sizes(size_t* out, int n);

/* MOCHA_BF16 layers look up the bf16 copy of a weight by address: register the bf16 mirror
 * (same element order) of each contiguous fp32 weight blob once after packing. */
int mocha_register_bf16_blob(const float* d_blob32, const void* d_blob16, size_t elems);

/* The mocha_*_workspace_bytes queries below answer for this precision mode from now on (process-wide).
 * The default covers MOCHA_FP32 and MOCHA_BF16; set MOCHA_TF32X3 before sizing the workspace of a
 * stage that will run in that mode (its split fp32 operands are three times the layer's A operand);
 * with less room the layers still run, as row chunks. */
int mocha_workspace_precision(int precision);

/* ---- model geometry (configs/config.yaml:13-43) -------------------------------------------- */
typedef struct {
  int T;        /* nframes 60 */
  int V;        /* njoints 24 */
  int Cin;      /* mot_in_dim 15 */
  int C0;       /* encoder_dim / temporal_patch_size = 64 */
  int D;        /* encoder_dim = decoder_dim = 256 */
  int P;        /* nbody 6 */
  int tp;       /* temporal_patch_size 4 */
  int Kj, Kb;   /* spatial kernel sizes: A_j.size(0)=3, A_b.size(0)=2 */
  int taps_j, taps_b; /* temporal kernel sizes 5 / 3 (model.py:121,149) */
  int heads;    /* 4 */
  int enc_dh, dec_dh; /* 128 / 256 */
  int mlp;      /* 512 */
  int enc_depth, dec_depth; /* 2 / 2 */
} mocha_dims;

/* Generator weights, repacked once on the host from the reference state_dict (see
 * mocha_sigasia2023_b200/packing.py). fp32, device, contiguous. */
typedef struct {
  const float* wqkv;              /* [3*heads*dh, D] = cat(to_q.1, to_k.1, to_v).weight (transformer.py:54-56) */
  const float* wo; const float* bo;   /* to_out.0 [D, heads*dh], [D] */
  const float* w1; const float* b1;   /* net.0 [mlp, D] */
  const float* w2; const float* b2;   /* net.3 [D, mlp] */
} mocha_enc_layer;

typedef struct {
  const float* sw1; const float* sb1; /* AdaIN style.2 [2D, D]  (transformer.py:104) */
  const float* sw2; const float* sb2; /* AdaIN style.4 [2D, 2D] (transformer.py:106) */
  const float* wq; const float* wk; const float* wv; /* [heads*dh, D] each */
  const float* wo; const float* bo;
  const float* w1; const float* b1;
  const float* w2; const float* b2;
} mocha_dec_layer;

typedef struct {
  mocha_dims dims;
  /* mot_embedding (model.py:42-50) */
  const float* emb_w; const float* emb_b;      /* .1  [C0,Cin],[C0] */
  const float* A_j;                            /* .2.A_j [Kj,V,V] */
  const float* jb_gcn_w;                       /* [D, Kj*C0]: w[co][k*C0+ci] = .2.blk.gcn.conv.weight[k*D+co][ci] */
  const float* jb_gcn_bias2d;                  /* [V, D]: sum_k bias[k*D+co] * sum_v A_j[k,v,w] */
  const float* jb_tcn_w; const float* jb_tcn_b;/* [D, taps_j*D]: w[co][tap*D+ci], [D] */
  const float* pool_w;                         /* .3.weight [V,P] */
  const float* A_b;                            /* .5.A_b [Kb,P,P] */
  const float* bb_gcn_w; const float* bb_gcn_bias2d; /* [D, Kb*D], [P, D] */
  const float* bb_tcn_w; const float* bb_tcn_b;      /* [D, taps_b*D], [D] */
  const float* pos_emb;                        /* [n_tok, D] */
  const float* tok_bias_pos;                   /* [n_tok, D] = bb_tcn_b + pos_emb (fused epilogue) */
  mocha_enc_layer enc[MOCHA_MAX_DEPTH];
  mocha_dec_layer dec[MOCHA_MAX_DEPTH];
  /* to_mot (model.py:71-80) */
  const float* tm_A_b;
  const float* tm_bb_gcn_w; const float* tm_bb_gcn_bias2d;
  const float* tm_bb_tcn_w; const float* tm_bb_tcn_b;
  const float* tm_jb_gcn_w; const float* tm_jb_gcn_b; /* [Kj*C0, D], [Kj*C0] (original layout) */
  const float* tm_A2;                                 /* [Kj,P,V]: sum_v unpool[p,v] * A_j[k,v,w] */
  const float* tm_jb_tcn_w; const float* tm_jb_tcn_b; /* [C0, taps_j*C0], [C0] */
  const float* tm_out_w; const float* tm_out_b;       /* .6 [Cin, C0], [Cin] */
  /* optional (tensor-core path): jb_gcn_w with the per-partition biases folded in as Kj extra K columns that
     multiply the adjacency column sums, K padded to a multiple of 16: [D, jb_gcn_kaug]; NULL = not provided */
  const float* jb_gcn_w_aug;
  int jb_gcn_kaug;
} mocha_generator_weights;

/* nn.TransformerEncoderLayer / DecoderLayer parameters exactly as PyTorch names them */
typedef struct {
  const float* in_w; const float* in_b;   /* self_attn.in_proj_{weight,bias} [3D,D],[3D] */
  const float* out_w; const float* out_b; /* self_attn.out_proj */
  const float* l1_w; const float* l1_b; const float* l2_w; const float* l2_b;
  const float* n1_g; const float* n1_b; const float* n2_g; const float* n2_b;
} mocha_cvae_enc_layer;

typedef struct {
  const float* sa_in_w; const float* sa_in_b; const float* sa_out_w; const float* sa_out_b;
  const float* ca_in_w; const float* ca_in_b; const float* ca_out_w; const float* ca_out_b;
  const float* l1_w; const float* l1_b; const float* l2_w; const float* l2_b;
  const float* n1_g; const float* n1_b; const float* n2_g; const float* n2_b;
  const float* n3_g; const float* n3_b;
} mocha_cvae_dec_layer;

typedef struct {
  int D, heads, dff, depth, out_seq; /* 256, 4, 512, 2, 90 (test_fullframework.py:52-55) */
  float ln_eps;                      /* 1e-5 */
  const float* mu_token; const float* logvar_token; /* prior_net.{mu,logvar}_token [D] */
  const float* pe;                                   /* sinusoidal table [>=ncond+2, D] (model_CVAE.py:168-186) */
  mocha_cvae_enc_layer prior[MOCHA_MAX_DEPTH];
  mocha_cvae_dec_layer dec[MOCHA_MAX_DEPTH];
  /* Optional [out_seq, D] table = norm1(pe + self_attn(pe)) of decoder layer 0. The decoder's query is
   * the constant positional table (model_CVAE.py:161-162), so this block is input-independent; fill it
   * once with mocha_cvae_precompute_dec0(). NULL = recompute it on every call. */
  const float* dec0_sa;
  /* Optional bf16 [out_seq, D] table = the layer-0 cross-attention QUERY projection of dec0_sa (rows of
   * ca_in_w[0:D], ca_in_b[0:D]): with it the tensor-core path neither materialises the broadcast query tensor nor
   * projects it per clip (every clip shares the table). Requires dec0_sa. NULL = project per call. */
  const void* dec0_q16;
} mocha_cvae_weights;

/* ---- (a1) Generator.mot_embedding  model.py:42-50, call site test_fullframework.py:190 ------ */
/* X [B,T,V,Cin] -> tokens [B, n_tok, D]; add_pos_emb != 0 also adds pos_emb (model.py:88 / :191). */
size_t mocha_embed_workspace_bytes(const mocha_dims* dims, int B);
int mocha_embed_fwd(const mocha_generator_weights* w, const float* d_X, int B, float* d_tokens,
                    int add_pos_emb, int precision, void* workspace, size_t workspace_bytes,
                    mocha_stream_t stream);

/* The JointBlock temporal convolution of mot_embedding alone (nn.Conv2d (5,1), reflect padding,
 * net/blocks.py:112-118): x [B*T*V, D] channel-last -> out [B*T*V, D]. Used by bench.py to time the
 * dominant kernel of the batched path in isolation: the operand is staged once (bf16 reflect-padded
 * copy in MOCHA_BF16 mode) and the GEMM kernel is launched gemm_repeats (>= 1) times back to back. */
int mocha_bench_tconv(const mocha_generator_weights* w, const float* d_x, int B, float* d_out, int precision,
                      int gemm_repeats, void* workspace, size_t workspace_bytes, mocha_stream_t stream);

/* bench.py `hbm_kernels`: `repeats` stand-alone launches of a bandwidth-bound kernel of the batched path at the
 * step's shapes; *algo_bytes = algorithmic bytes of ONE launch. which: 0 embed_graph_agg, 1 pool_graph_agg,
 * 2 add_layernorm (CVAE prior rows), 3 graph_agg_kv_pad16, 4 adain_norm_tokens, 5 instance_norm_tokens (bf16 out). */
int mocha_bench_hbm_kernel(const mocha_generator_weights* w, int which, int B, int repeats, void* workspace,
                           size_t workspace_bytes, double* algo_bytes, mocha_stream_t stream);

/* ---- (a3) Generator.encoder = Transformer(adain=False)  net/transformer.py:79-95 ------------ */
size_t mocha_encoder_workspace_bytes(const mocha_dims* dims, int B);
int mocha_encoder_fwd(const mocha_generator_weights* w, const float* d_tokens, int B, float* d_encoded,
                      int precision, void* workspace, size_t workspace_bytes, mocha_stream_t stream);

/* ---- (a4) mean_variance_norm  net/transformer.py:13-20 (+ matcher scaling :293,:442) ---------- */
/* x [B,n,C] normalised over n per (b,c). d_cnt and/or d_cnt_nm may be NULL.
 * d_cnt_nm = (cnt - cnt_mean)/cnt_std with tables [n,C]; d_cnt_nm16 (optional, bf16 [B,n*C]) is the
 * same query minus d_cnt_nm16_center ([n*C], optional) rounded to bf16: the operand of the tensor-core
 * matcher (mocha_match_tc's d_Q16) relative to the origin the bf16 DB rows were packed around. */
int mocha_cnt_features(const float* d_x, int B, int n, int C, float eps, float* d_cnt,
                       const float* d_cnt_mean, const float* d_cnt_std, float* d_cnt_nm, void* d_cnt_nm16,
                       const float* d_cnt_nm16_center, mocha_stream_t stream);

/* ---- fused transformer building blocks (bf16 operands, tcgen05; used by the bf16 stage bodies) ------- */
/* Block tail of a transformer layer in ONE launch (net/transformer.py:23-34,:70-76; nn.TransformerEncoder/
 * DecoderLayer of model_CVAE.py:70-79,:159-165), width 256:
 *   Y = LN1?(A0 W0^T + b0 + R0);  Z = LN2?(Y + act(Y W1^T + b1) W2^T + b2)   (FFN skipped when Hd == 0)
 * d_A0 bf16 [M,K0] (row pitch lda), d_W0 bf16 [256,K0], d_R0 fp32 [M,256] or NULL, d_W1 bf16 [Hd,256],
 * d_W2 bf16 [256,Hd]; g/be pairs select the LayerNorms (NULL = none); act: 0 none, 1 ReLU, 2 GELU, 3 LeakyReLU.
 * Outputs of the last stage: d_O32 fp32 and / or d_O16 bf16 [M,256]. K0 % 64 == 0, Hd % 128 == 0. */
int mocha_block_tail(const void* d_A0, int lda, int K0, const void* d_W0, const float* d_b0, const float* d_R0,
                     const float* d_g1, const float* d_be1, int Hd, int act, const void* d_W1, const float* d_b1,
                     const void* d_W2, const float* d_b2, const float* d_g2, const float* d_be2, float eps,
                     float* d_O32, void* d_O16, int M, mocha_stream_t stream);

/* Attention core in ONE launch (net/transformer.py:58-70; nn.MultiheadAttention): out[b, :, h*dh:(h+1)*dh] =
 * softmax(Q_h K_h^T / sqrt(dh)) V_h. d_q / d_k / d_v: bf16 views [B*nq | B*nkv, ld] with head h at columns h*dh
 * (16 B-aligned, ld % 8 == 0); d_out bf16 [B, nq, H*dh] with ldo == H*dh. dh in {64,128,256}, nkv <= 256. */
int mocha_attention_core(const void* d_q, int ldq, const void* d_k, int ldk, const void* d_v, int ldv, int B, int H,
                         int nq, int nkv, int dh, void* d_out, int ldo, mocha_stream_t stream);

/* ---- (a8) Generator.decoder = Transformer(adain=True)  transformer.py:79-113 ---------------- */
size_t mocha_decoder_workspace_bytes(const mocha_dims* dims, int B);
int mocha_decoder_fwd(const mocha_generator_weights* w, const float* d_src_encoded,
                      const float* d_cha_encoded, int B, float* d_decoded, int precision,
                      void* workspace, size_t workspace_bytes, mocha_stream_t stream);

/* ---- (a9) Generator.to_mot  model.py:71-80 -------------------------------------------------- */
/* tokens [B,n_tok,D] -> Ytil [B,T,V,Cin]. If d_Y_mean/d_Y_std ([V,Cin] tables) are non-NULL the
 * de-normalisation Ytil*Y_std+Y_mean (test_fullframework.py:457) is written to d_Y. */
size_t mocha_to_mot_workspace_bytes(const mocha_dims* dims, int B);
int mocha_to_mot_fwd(const mocha_generator_weights* w, const float* d_tokens, int B, float* d_Ytil,
                     const float* d_Y_mean, const float* d_Y_std, float* d_Y, int precision,
                     void* workspace, size_t workspace_bytes, mocha_stream_t stream);

/* ---- (a6,a7) CVAE.sample  model_CVAE.py:44-46 (PriorNet :70-92, Decoder :159-165) ----------- */
/* cond [B,ncond,D]; d_eps [B,D] standard-normal draw or NULL for deterministic=True;
 * out [B,out_seq,D]; d_mu/d_logvar [B,D] optional. If d_out_mean/d_out_std ([out_seq,D]) are given,
 * d_out_denorm = out*std+mean (test_fullframework.py:449) is also written.
 * With d_out == d_out_denorm == NULL and d_mu / d_logvar given only the token network runs: this is CVAE.prior
 * (model_CVAE.py:29-31) and, with the posterior Encoder's weights in the `prior` slots and cond = [c ; x]
 * (model_CVAE.py:116-126, up to 510 tokens), CVAE.encode (:33-35). */
size_t mocha_cvae_workspace_bytes(const mocha_cvae_weights* w, int B, int ncond);
int mocha_cvae_sample(const mocha_cvae_weights* w, const float* d_cond, int B, int ncond,
                      const float* d_eps, float* d_out, float* d_mu, float* d_logvar,
                      const float* d_out_mean, const float* d_out_std, float* d_out_denorm,
                      int precision, void* workspace, size_t workspace_bytes, mocha_stream_t stream);
/* Fills d_table [out_seq, D] for mocha_cvae_weights.dec0_sa (fp32 arithmetic). */
int mocha_cvae_precompute_dec0(const mocha_cvae_weights* w, float* d_table, void* workspace, size_t workspace_bytes,
                               mocha_stream_t stream);
/* condition = cat[(src_cnt-m0)/s0, (prev-m1)/s1] (test_fullframework.py:446-447); tables [n,D] */
int mocha_cvae_condition(const float* d_src_cnt, const float* d_prev, const float* d_m0, const float* d_s0,
                         const float* d_m1, const float* d_s1, float* d_cond, int B, int n, int D,
                         mocha_stream_t stream);

/* ---- (a5) context matching: BallTree(X).query(q, k)  test_fullframework.py:293-296,:440-443 -- */
/* Exact Euclidean k-NN of Q [nq,D] against DB [N,D] (both fp32), arithmetic in fp64 like
 * sklearn's BallTree64. idx [nq,k] int64 (+ index_offset, for row-sharded DBs), dist [nq,k] fp64
 * (may be NULL), sorted ascending by (distance, index). */
size_t mocha_match_exact_workspace_bytes(int nq, long long N, int k);
int mocha_match_exact(const float* d_Q, int nq, const float* d_DB, long long N, int D, int k,
                      long long index_offset, int64_t* d_idx, double* d_dist, void* workspace,
                      size_t workspace_bytes, mocha_stream_t stream);

/* Tensor-core matcher for large problems: coarse pass ||x||^2 - 2 q.x on tcgen05 (bf16 operands,
 * fp32 accumulate in TMEM) with a fused per-row running top-kc epilogue, cross-tile merge, then an
 * exact fp64 re-rank of the kc candidates in difference form against the stored rows.
 * d_Q16/d_DB16: bf16 copies [nq,D]/[N,D] (D % 64 == 0); d_dbnorm [N] = ||x||^2 of the bf16 rows;
 * exact re-rank reads d_Q (fp32) and, if d_DB32 != NULL, the fp32 rows, else the bf16 rows.
 * The bf16 operands only rank candidates, so they may be expressed relative to ANY common origin c
 * (d_Q16 = bf16(q - c), d_DB16 = bf16(x - c), d_dbnorm of those rows): distances do not depend on c, and
 * centring a DB whose rows share a large common component (feature DBs do: ||x|| >> ||x - x'||) removes
 * most of the bf16 rounding error from the ranking (BallTree / feature_db use the DB mean). With
 * d_DB32 == NULL the re-rank reads d_DB16 against d_Q, which must then share that origin. */
size_t mocha_match_tc_workspace_bytes(int nq, long long N, int D, int kc);
int mocha_match_tc(const float* d_Q, const void* d_Q16, int nq, const void* d_DB16, const float* d_DB32,
                   const float* d_dbnorm, long long N, int D, int k, int kc, long long index_offset,
                   int64_t* d_idx, double* d_dist, void* workspace, size_t workspace_bytes,
                   mocha_stream_t stream);
/* fp32-storage mode (BASELINE config 3 "fp32"): pass d_DB16 = d_Q16 = NULL and d_DB32 != NULL; the coarse
 * pass then feeds the fp32 rows to tcgen05 as TF32 (kind::tf32) and d_dbnorm = ||x||^2 of the fp32 rows
 * (mocha_db_norms_f32). */
int mocha_db_norms_f32(const float* d_rows, long long N, int D, float* d_norm, mocha_stream_t stream);
/* helpers to build the bf16 DB: rows fp32 -> bf16 (+ squared norms of the rounded rows) */
int mocha_db_pack_bf16(const float* d_rows, long long N, int D, void* d_rows16, float* d_norm,
                       mocha_stream_t stream);
/* merge per-shard candidate lists (dist fp64, idx int64), [nshard, nq, k] -> [nq, k] */
int mocha_topk_merge(const double* d_dist, const int64_t* d_idx, int nshard, int nq, int k,
                     double* d_out_dist, int64_t* d_out_idx, mocha_stream_t stream);

/* Seed of the autoregression for clips that start on this frame (test_fullframework.py:298, per clip): for every
 * b < B with d_start[b] != 0, d_dst[b] = d_table[d_idx[b * idx_stride]] (rows of row_elems floats, e.g. prev_cha[b] =
 * cha_encoded[match_idx[b, 0]]); other rows are not touched, and an index outside [0, N) leaves the row unchanged.
 * d_start uint8 [B]; d_table [N, row_elems] and d_dst [B, row_elems] 16 B aligned, row_elems % 4 == 0. */
int mocha_seed_rows(const uint8_t* d_start, const int64_t* d_idx, int idx_stride, const float* d_table, long long N,
                    long long row_elems, float* d_dst, int B, mocha_stream_t stream);

/* ---- peer-memory exchange of the DB-sharded matcher (one process per GPU, NVLink / NVSwitch P2P) ----
 * Fused replacement of "all-gather the [nq,k] lists, then merge" (sharded.py): ONE kernel per rank stores
 * its local lists into a slot of every peer's exchange buffer (plain P2P stores over NVLink), raises a
 * system-scope arrival counter on the peer, waits for the peers' counters in its own buffer and merges.
 * Buffers come from mocha_peer_alloc (cudaMalloc + CUDA IPC handle, 64 bytes, to be exchanged by the host
 * side, e.g. torch.distributed.all_gather_object) and are mapped with mocha_peer_open.
 * Layout of a buffer of mocha_topk_exchange_bytes(world, nq, k) bytes: 2 parities x world slots x
 * (nq*k fp64 + nq*k int64), then 2 x world uint32 arrival counters (zero-initialised by mocha_peer_alloc).
 * `epoch` counts calls on this group (0, 1, 2, ...): consecutive calls alternate between the two parities, so
 * a fast rank can never overwrite lists a slow rank is still merging. Every rank must launch with the same
 * nq, k, epoch; the grid is fixed (all blocks co-resident), so the cross-GPU wait cannot deadlock. */
size_t mocha_topk_exchange_bytes(int world, int nq, int k);
int mocha_peer_alloc(size_t bytes, void** d_ptr, unsigned char handle_out[64]);
int mocha_peer_open(const unsigned char handle[64], void** d_ptr);
int mocha_peer_close(void* d_ptr);
int mocha_peer_free(void* d_ptr);
int mocha_topk_exchange_merge(const double* d_local_dist, const int64_t* d_local_idx, int nq, int k, int rank, int world,
                              void* const* peer_bufs /* HOST array [world] of device pointers: every rank's buffer, own included */,
                              unsigned int epoch, double* d_out_dist, int64_t* d_out_idx, mocha_stream_t stream);

/* ---- dense primitive exposed for tests / reuse ----------------------------------------------- */
/* C[M,N] = act(A[M,K] * W[N,K]^T + bias) (+ residual). act: 0 none, 1 relu, 2 gelu(erf), 3 lrelu(0.2) */
int mocha_linear(const float* d_A, const float* d_W, const float* d_bias, const float* d_res, float* d_C,
                 int M, int N, int K, int act, int precision, void* workspace, size_t workspace_bytes,
                 mocha_stream_t stream);
size_t mocha_linear_workspace_bytes(int M, int N, int K, int precision);

/* ---- (a11) quat.from_xform_xy  motion/quat.py:96-107 (-> from_xform :69-94, normalize :15) --- */
/* xy [n,3,2] fp32 -> quat [n,4] fp32 */
int mocha_xy_to_quat(const float* d_xy, long long n, float* d_quat, mocha_stream_t stream);
/* quat.to_xform_xy motion/quat.py:42-55: quat [n,4] -> xy [n,3,2] */
int mocha_quat_to_xy(const float* d_quat, long long n, float* d_xy, mocha_stream_t stream);

/* ---- (a17) batch FK family  motion/quat.py:166-204, :175-187 --------------------------------- */
/* lrot [F,J,4], lpos [F,J,3] -> grot, gpos; parents int32 [J] on device (parents[0] = -1,
 * parents[i] < i). One warp walks one skeleton's chains. */
int mocha_fk(const float* d_lrot, const float* d_lpos, const int32_t* d_parents, long long F, int J,
             float* d_grot, float* d_gpos, mocha_stream_t stream);
int mocha_fk_vel(const float* d_lrot, const float* d_lpos, const float* d_lvel, const float* d_lang,
                 const int32_t* d_parents, long long F, int J, float* d_grot, float* d_gpos,
                 float* d_gvel, float* d_gang, mocha_stream_t stream);
/* quat.ik: global -> local */
int mocha_ik(const float* d_grot, const float* d_gpos, const int32_t* d_parents, long long F, int J,
             float* d_lrot, float* d_lpos, mocha_stream_t stream);

/* float64 variants (same layouts): the reference's final FK runs on float64 arrays (test_fullframework.py:672-694). */
int mocha_fk_f64(const double* d_lrot, const double* d_lpos, const int32_t* d_parents, long long F, int J,
                 double* d_grot, double* d_gpos, mocha_stream_t stream);
int mocha_fk_vel_f64(const double* d_lrot, const double* d_lpos, const double* d_lvel, const double* d_lang,
                     const int32_t* d_parents, long long F, int J, double* d_grot, double* d_gpos, double* d_gvel,
                     double* d_gang, mocha_stream_t stream);
int mocha_ik_f64(const double* d_grot, const double* d_gpos, const int32_t* d_parents, long long F, int J,
                 double* d_lrot, double* d_lpos, mocha_stream_t stream);

/* ---- (a10,a12-a16) per-frame post-process: test_fullframework.py:457-462, :492-509, :532-623 -- */
/* Persistent per-clip state carried frame to frame (all fp64 like the reference's NumPy state). */
typedef struct {
  double root_pos[3];          /* trans_Ypos_list[-1][0] */
  double root_rot[4];          /* trans_Yrot_list[-1][0] */
  double src_root_pos[3];      /* src_Ypos_list[-1][0] (float32 values, :478) */
  double src_root_rot[4];      /* src_Yrot_list[-1][0] */
  double prev_pos[25][3];      /* trans_Ypos_list[-1]   (blend history, :626) */
  double prev_ik_pos[25][3];   /* ik_trans_Ypos_list[-1] (:532) */
  /* contact state per foot (:403-431) */
  int32_t contact_state[2];
  int32_t contact_lock[2];
  double contact_position[2][3];
  double contact_velocity[2][3];
  double contact_point[2][3];
  double contact_target[2][3];
  double contact_offset_position[2][3];
  double contact_offset_velocity[2][3];
} mocha_clip_state;

typedef struct {
  int J;                       /* 25 bones (simulation root + 24 joints) */
  int32_t parents[32];
  int32_t contact_bones[2];    /* {5, 24} (test_fullframework.py:104) */
  double dt;                   /* 1/60 */
  double ik_max_length_buffer, ik_foot_height, ik_unlock_radius, ik_blending_halflife; /* :110-114 */
  int ik_enabled;
} mocha_post_params;

typedef struct {
  /* outputs for one frame of one clip, fp64 */
  double pos[25][3];           /* trans_Ypos (root + joints, before blending) */
  double rot[25][4];           /* trans_Yrot */
  double vel[25][3];           /* trans_Yvel */
  double ang[25][3];           /* trans_Yang */
  double blend_pos[25][3];     /* trans_Ypos_list entry (:626) */
  double ik_pos[25][3];        /* adjusted_bone_positions (:633) */
  double ik_rot[25][4];        /* adjusted_bone_rotations (:634) */
  double src_root_pos[3];      /* src_rootpos / rot / vel / ang (:476-479) */
  double src_root_rot[4];
  double src_root_vel[3];
  double src_root_ang[3];
} mocha_frame_out;

/* d_Y [B,T,V,Cin] de-normalised decoder output; d_src_hips_vel [B,T,3] = src_Yvel[i,:,1];
 * d_src_rvel/d_src_rang [B,3] = src_Yrvel[i,-1], src_Yrang[i,-1]; d_contacts [B,2] uint8 =
 * src_contact[i,-1]; init != 0 runs the frame-0 initialisation (:337-434) instead of a step. */
int mocha_post_frame(const mocha_post_params* params, const float* d_Y, const float* d_src_hips_vel,
                     const float* d_src_rvel, const float* d_src_rang, const uint8_t* d_contacts, int B,
                     int T, int V, int Cin, int init, mocha_clip_state* d_state, mocha_frame_out* d_out,
                     mocha_stream_t stream);

/* Same, with the source-motion inputs packed one row per clip: d_side [B, side_stride] floats =
 * [src_Yvel[i,:,1] (T*3) | src_Yrvel[i,-1] (3) | src_Yrang[i,-1] (3)], side_stride >= T*3+6. */
int mocha_post_frame_packed(const mocha_post_params* params, const float* d_Y, const float* d_side, int side_stride,
                            const uint8_t* d_contacts, int B, int T, int V, int Cin, int init,
                            mocha_clip_state* d_state, mocha_frame_out* d_out, mocha_stream_t stream);

/* Same as mocha_post_frame_packed with the frame-0 decision made per clip on the device (clip admission): clip b runs
 * the init frame (:337-434: root from the identity, blend / IK lists from the raw pose, contacts reset from the toe FK)
 * iff d_start[b] != 0 and a steady-state step otherwise, bit-identical to the init = 1 / init = 0 calls above.
 * d_start uint8 [B]. */
int mocha_post_frame_packed_masked(const mocha_post_params* params, const float* d_Y, const float* d_side, int side_stride,
                                   const uint8_t* d_contacts, const uint8_t* d_start, int B, int T, int V, int Cin,
                                   mocha_clip_state* d_state, mocha_frame_out* d_out, mocha_stream_t stream);

/* ---- window feature extraction: re-rooting block of the driver's set-up (test_fullframework.py:148-158,:180-186) ---
 * Inputs are quat.fk_vel's outputs over all frames of all windows, [W,T,J,{4,3,3,3}] fp32. Every window is expressed
 * relative to the simulation root of its last frame; d_X [W,T,J-1,15] receives (concat(Xpos, Xtxy, Xvel, Xang) -
 * X_mean)/X_std for joints 1.. (tables [J,15] as in norm.npz), d_xrot [W,T,J,4] / d_xpos [W,T,J,3] the re-rooted
 * rotations / positions the following quat.ik (:160) needs (either may be NULL).
 * d_X_mean == NULL selects the training-side twin convert_YtilToX (trainer.py:337-374): every FRAME relative to its own
 * root, all J joints, no normalisation: d_X [W,T,J,15]. */
int mocha_window_features(const float* d_grot, const float* d_gpos, const float* d_gvel, const float* d_gang, long long W,
                          int T, int J, const float* d_X_mean, const float* d_X_std, float* d_X, float* d_xrot,
                          float* d_xpos, mocha_stream_t stream);

/* ---- source windows: every slot's pose window built on the device from a bank of source clips (DESIGN §5b) ----
 * Bank: per-frame preprocess.process_frames arrays of many clips back to back, d_rot [n_frames,J,4], d_pos / d_vel /
 * d_ang [n_frames,J,3] fp32 (d_rot 16 B aligned), d_bank_contacts uint8 [n_frames,2]; clip c is frames
 * d_clip_first[c] .. + d_clip_frames[c] (int64 / int32 tables of n_clips entries; a frame count below T/4 + 1 marks an
 * unused entry). d_parents [J], d_X_mean / d_X_std [J,15] as for mocha_window_features.
 * Per slot b, each call: if d_start[b], d_slot_clip[b] = d_clip[b] and d_slot_cursor[b] = 0 (d_clip is read only there).
 * The slot then serves window w = min(cursor, nwin - 1) of its clip, nwin = F - T/4 (preprocess.sliding_windows' count
 * and edge padding), and the cursor becomes w + 1 (so it saturates at nwin: a finished clip repeats its last window).
 * Outputs are what features.extract computes for that window, bit for bit: d_X[b] [T,J-1,15]; d_side row b (stride
 * side_stride >= T*3+6 floats) = [velocity of joint 1 after ik, T*3 | root velocity 3 | root angular velocity 3] of the
 * last frame's body frame; d_contacts[b] [2] = contacts of the last frame. A slot whose clip id is outside
 * [0, n_clips), or names an unused entry, is idle (d_slot_clip[b] = -1): it writes zeros. One launch, graph-capturable. */
int mocha_source_windows(const float* d_rot, const float* d_pos, const float* d_vel, const float* d_ang,
                         const uint8_t* d_bank_contacts, long long n_frames, const int64_t* d_clip_first,
                         const int32_t* d_clip_frames, int n_clips, const int32_t* d_parents, int T, int J,
                         const float* d_X_mean, const float* d_X_std, const uint8_t* d_start, const int32_t* d_clip,
                         int32_t* d_slot_clip, int32_t* d_slot_cursor, int B, float* d_X, float* d_side, int side_stride,
                         uint8_t* d_contacts, mocha_stream_t stream);

/* ---- result bank: each served clip's motion recorded on the device, its bvh.save payload built per clip (DESIGN §5c)
 * One record row per (clip, window), at row d_clip_first[c] + w of arrays sized like the source bank's frames (w < nwin
 * < F keeps it inside the clip's frame range): the fields of mocha_frame_out the reference's final step reads, fp64,
 * and the matched DB row. 1464 B. */
typedef struct {
  double ik_pos[25][3];
  double ik_rot[25][4];
  double src_root_pos[3];
  double src_root_rot[4];
  int64_t match;
} mocha_frame_record;

/* Per slot b, the last launch of an admission frame (after mocha_post_frame_packed_masked): the slot's record count
 * d_slot_count[b] (int32 [B], session state) restarts at 0 if d_start[b]. If d_slot_clip[b] = c >= 0 (as
 * mocha_source_windows left it for this frame) and count < nwin(c) = d_clip_frames[c] - T/4, d_out[b]'s ik_pos /
 * ik_rot / src_root_pos / src_root_rot and d_match_idx[b * match_stride] go to d_rec[d_clip_first[c] + count]; then
 * count += 1, d_clip_done[c] = count and d_clip_built[c] = 0 (int32 [n_clips] each; a new row makes the clip's payload
 * stale). Idle slots and finished clips (whose last window the source
 * bank repeats) write nothing. Bank tables as for mocha_source_windows; d_rec has n_rows rows. Copies only; one launch,
 * graph-capturable. Two slots serving the same clip at once write the same rows: the caller must not do that. */
int mocha_record_frames(const mocha_frame_out* d_out, const int64_t* d_match_idx, int match_stride,
                        const uint8_t* d_start, const int32_t* d_slot_clip, int32_t* d_slot_count, int B,
                        const int64_t* d_clip_first, const int32_t* d_clip_frames, int n_clips, int T,
                        mocha_frame_record* d_rec, long long n_rows, int32_t* d_clip_done, int32_t* d_clip_built,
                        mocha_stream_t stream);

/* For the n_ids clip ids d_ids (int32, device), every recorded window w < min(d_clip_done[c], nwin(c)) of clip c: the
 * payload the reference hands to bvh.save (test_fullframework.py:672-721), at row r = d_clip_first[c] + w of the
 * outputs, [n_frames, 24, 3] each (joints 1..24; joint 1, the hips, takes its global transform; rotations as Euler 'xyz'
 * degrees):
 *   d_ours_pos / d_ours_rot fp64 from the recorded ik_pos / ik_rot;
 *   d_src_pos / d_src_rot fp32 from the local pose of window w's last frame, as features.extract gives it (fk of the
 *   bank frame d_rot / d_pos, re-rooting on its root, ik: bit for bit), with the recorded src_root_pos / src_root_rot
 *   (cast to fp32) as the root;
 *   d_match [n_frames] int64 the recorded matched DB row.
 * d_clip_built[c] becomes 1 if clip c was complete (d_clip_done[c] >= nwin), else 0: a reader of the payload rows
 * checks it, and the next record row of the clip clears it.
 * J must be 25 (the record's skeleton); max_nwin >= the largest nwin among the ids. Ids outside [0, n_clips) are
 * skipped. One warp per row, stream-ordered, off the frame. */
int mocha_clip_payload(const mocha_frame_record* d_rec, long long n_frames, const float* d_rot, const float* d_pos,
                       const int64_t* d_clip_first, const int32_t* d_clip_frames, int n_clips, const int32_t* d_clip_done,
                       int32_t* d_clip_built, const int32_t* d_parents, int T, int J, const int32_t* d_ids, int n_ids, int max_nwin,
                       float* d_src_rot, float* d_src_pos, double* d_ours_rot, double* d_ours_pos, int64_t* d_match,
                       mocha_stream_t stream);

/* ---- element-wise quaternion algebra of motion/quat.py in the caller's precision ------------- */
/* out[i] = op(a[i], b[i]) for i < n; dense [n, width] arrays, float32 (is_f64 == 0) or float64. Ops and widths
 * (a, b, out): 0 mul (4,4,4) quat.py:112 | 1 inv_mul :122 | 2 mul_inv :125 | 3 mul_vec (4,3,3) :128 |
 * 4 inv_mul_vec :132 | 5 inv (4,-,4) :109 | 6 abs :18 | 7 normalize quaternion (eps = param) :15 |
 * 8 normalize 3-vector (3,-,3) | 9 exp (3,-,4; eps = param) :154 | 10 log (4,-,3; eps = param) :149 |
 * 11 between (3,3,4) :143 | 12 from_angle_axis (1,3,4) :21 | 13 to_xform (4,-,9) :27 | 14 from_xform (9,-,4) :69 |
 * 15 to_euler 'xyz' (4,-,3) :346 | 16 to_euler 'yzx' | 17 _fast_cross (3,3,3) :3 | 18 to_xform_xy (4,-,6) :42 |
 * 19 from_xform_xy (6,-,4) :96 | 20 length of 3-vectors (3,-,1) :12 | 21 length of quaternions (4,-,1). */
int mocha_quat_op(int op, int is_f64, const void* d_a, const void* d_b, long long n, double param, void* d_out,
                  mocha_stream_t stream);

/* quat.fk_partial's chain walk (quat.py:241-272): n chains of m bones (bone c's parent is bone c-1); element 0
 * hangs off (d_start_pos [n,3], d_start_rot [n,4]) or, when both are NULL, is a root bone (global = local). */
int mocha_fk_chain(int is_f64, const void* d_start_pos, const void* d_start_rot, const void* d_lpos, const void* d_lrot,
                   long long n, int m, void* d_gpos, void* d_grot, mocha_stream_t stream);

/* ---- (a15) Inertialization.contact_update  motion/Inertialization.py:300-377 ----------------- */
/* Batched over n feet; state arrays are in/out, fp64; flags int32. */
int mocha_contact_update(int32_t* d_state, int32_t* d_lock, double* d_position, double* d_velocity,
                         double* d_point, double* d_target, double* d_off_pos, double* d_off_vel,
                         const double* d_input_position, const int32_t* d_input_state, long long n,
                         double unlock_radius, double foot_height, double halflife, double dt,
                         mocha_stream_t stream);
/* ---- (a16) quat.ik_two_bone  motion/quat.py:295-343; all arrays [n,·] fp64 ------------------- */
int mocha_ik_two_bone(const double* d_root_lr, const double* d_mid_lr, const double* d_root,
                      const double* d_mid, const double* d_end, const double* d_target, const double* d_fwd,
                      const double* d_root_gr, const double* d_mid_gr, const double* d_par_gr,
                      double max_length_buffer, long long n, double* d_out_root_lr, double* d_out_mid_lr,
                      mocha_stream_t stream);
/* ---- (a18) Inertialization.pose_update / pose_transition  Inertialization.py:136-297 ---------- */
/* Batched over n skeletons of J bones; fp64 arrays [n,J,3|4] updated in place as the reference does. */
int mocha_pose_transition(double* d_off_pos, double* d_off_vel, double* d_off_rot, double* d_off_ang,
                          const double* d_root_pos, const double* d_root_vel, const double* d_root_rot,
                          const double* d_root_ang, const double* d_src_pos, const double* d_src_vel,
                          const double* d_src_rot, const double* d_src_ang, const double* d_dst_pos,
                          const double* d_dst_vel, const double* d_dst_rot, const double* d_dst_ang,
                          long long n, int J, double* d_tr_src_pos, double* d_tr_src_rot,
                          double* d_tr_dst_pos, double* d_tr_dst_rot, mocha_stream_t stream);
int mocha_pose_update(double* d_pos, double* d_vel, double* d_rot, double* d_ang, double* d_off_pos,
                      double* d_off_vel, double* d_off_rot, double* d_off_ang, const double* d_in_pos,
                      const double* d_in_vel, const double* d_in_rot, const double* d_in_ang,
                      const double* d_tr_src_pos, const double* d_tr_src_rot, const double* d_tr_dst_pos,
                      const double* d_tr_dst_rot, double halflife, double dt, long long n, int J,
                      mocha_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* MOCHA_B200_H_ */
