// Fused "block tail" of a transformer layer on tcgen05 (sm_100a), one CTA per 128-row tile:
//
//     Y = LN1?( A0 W0^T + b0 + R0 )                       out-projection + bias + residual (+ LayerNorm)
//     Z = LN2?( Y + act(Y W1^T + b1) W2^T + b2 )          feed-forward + residual (+ LayerNorm)      [optional]
//
// i.e. net/transformer.py:23-34,:70-76 (Generator encoder / decoder: no norms, GELU) and the post-LN
// nn.TransformerEncoderLayer / DecoderLayer blocks of model_CVAE.py:70-79,:159-165 (LayerNorms, ReLU).
// What used to be 3 GEMM launches + 2 LayerNorm launches with four activation round trips through HBM is one
// launch whose intermediates never leave the SM:
//   * the out-projection accumulates in TMEM columns [0,256); its epilogue adds bias + residual (+ LN1), writes the
//     fp32 result Y BACK into the same TMEM columns and the bf16 copy into shared memory as the K-major,
//     128 B-swizzled A operand of the first FFN GEMM;
//   * the hidden layer is produced 128 columns at a time in TMEM columns [256,384) / [384,512) (double-buffered),
//     activated and stored to shared memory as the A operand of the second FFN GEMM,
//   * which accumulates ON TOP of Y in TMEM columns [0,256) - the residual add costs nothing and stays fp32;
//   * the final epilogue adds b2 (+ LN2) and hands fp32 and / or bf16 boxes to the TMA engine.
// Weights stream from L2 through a 3 x 32 KB ring; the A operand of the out-projection through 4 x 16 KB stages.
// Warp roles as in gemm_tc.cu: warp 0 TMA producer, warp 1 MMA issuer + TMEM owner, warps 2..9 epilogue (warp w reads
// TMEM lane quarter w % 4; the two warps of a quarter split the columns and exchange LayerNorm partial sums).
// Width is fixed at D = 256 (both models of the path); K0 % 64 == 0, hidden width % 128 == 0.
#include "fused.cuh"

#include "gemm_tc.cuh"
#include "tc_ptx.cuh"

namespace mocha {

using namespace tcx;

namespace {

constexpr int FT_THREADS = 320;
constexpr int FT_D = 256;
constexpr uint32_t FT_OFF_X = 0;            // X tile: bf16 Y, 4 k-blocks of [128 rows x 128 B]                     64 KB
constexpr uint32_t FT_OFF_HB = 65536;       // out-projection A stages (3 x 16 KB); first 32 KB later: hidden chunk  48 KB
constexpr int FT_NA = 3;
constexpr uint32_t FT_OFF_RING = 114688;    // weight ring 3 x 32 KB                                                 96 KB
constexpr uint32_t FT_SLOT = 32768;
constexpr int FT_NSLOT = 3;
constexpr uint32_t FT_OFF_PAR = 212992;     // bias / LayerNorm vectors staged once per CTA (2048 floats)             8 KB
constexpr uint32_t FT_OFF_BAR = 221184;     // mbarriers + TMEM slot                                                256 B
constexpr uint32_t FT_OFF_XCH = FT_OFF_BAR + 256;   // LayerNorm statistics exchange [2 halves][4][32][2] floats      2 KB
constexpr uint32_t FT_SMEM = FT_OFF_XCH + 2048;
static_assert(FT_SMEM <= 227 * 1024, "fused tail kernel: shared memory plan exceeds 227 KB");
// float offsets of the staged vectors
enum { PV_B0 = 0, PV_G1 = 256, PV_BE1 = 512, PV_B1 = 768, PV_B2 = 1280, PV_G2 = 1536, PV_BE2 = 1792, PV_COUNT = 2048 };
constexpr int FT_MAX_HD = 512;

enum { B_FULLW = 0, B_EMPTYW = 3, B_FULLA = 6, B_EMPTYA = 10, B_ACCP = 14, B_XREADY = 15, B_ACC1F = 16, B_ACC1E = 18,
       B_HREADY = 20, B_HEMPTY = 22, B_ACC2 = 24, B_COUNT = 25 };

#ifdef MOCHA_TRACE
// trace build: per-CTA clock64 time line of the pipeline roles (tools/tail_trace.py), 64 slots per CTA
__device__ unsigned long long* g_ft_trace = nullptr;
#define FT_TRACE(slot)                                                                                      \
  do {                                                                                                      \
    if (g_ft_trace) g_ft_trace[(size_t)blockIdx.x * 64 + (slot)] = (unsigned long long)clock64();            \
  } while (0)
#else
#define FT_TRACE(slot) do { } while (0)
#endif

struct TailParams {
  int M, K0, Hd, act;
  const float* b0;
  const float* R0;
  const float* g1;
  const float* be1;
  const float* b1;
  const float* b2;
  const float* g2;
  const float* be2;
  float eps;
  int out32, out16;
  int r0_period;     // > 0: the residual is a [period, 256] table shared by every group of `period` rows
};

// Hidden-layer GELU of the fused path: tanh form on the hardware tanh (MUFU.TANH), ~7 instructions per element instead of
// ~22 for the erf polynomial - the hidden epilogue is issue-bound (128 x 512 activations per tile on one SM).
// |gelu_tanh - gelu_erf| <= 5e-4 absolute (at |x| ~ 2), below the bf16 rounding (2^-9 relative) the activation gets anyway;
// the fp32 parity path keeps erff.
__device__ __forceinline__ float gelu_tanh_f(float x) {
  const float x2 = x * x;
  const float u = x * fmaf(0.0356774081f, x2, 0.7978845608f);
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(u));
  const float hx = 0.5f * x;
  return fmaf(hx, t, hx);
}

__device__ __forceinline__ void tma_store_3d(const CUtensorMap* tm, uint32_t smem_addr, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(tm), "r"(smem_addr),
               "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}

// per-warp epilogue context
struct EpiW {
  int lane, q, half, ew;
  int row_l;          // row inside the tile
  long long row;      // global row
  bool row_ok;
  uint32_t taddr;     // TMEM address of this warp's lane quarter, column 0
  uint32_t stage;     // staging for the final outputs: [2 x 4 KB fp32 boxes][2 x 4 KB bf16 boxes]
  int m0;
};

// v += vec[col .. col+31] from the CTA's staged copy (same address in every lane: shared-memory broadcast). Global loads
// here cost ~2000 cycles per chunk: every warp of the CTA sits in the same phase, so nothing hides an L2 round trip.
__device__ __forceinline__ void add_bias32(float (&f)[32], uint32_t vec_smem, int col) {
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float4 b = lds128f(vec_smem + (uint32_t)(col + 4 * j) * 4u);
    f[4 * j] += b.x; f[4 * j + 1] += b.y; f[4 * j + 2] += b.z; f[4 * j + 3] += b.w;
  }
}

// LayerNorm statistics of a 256-wide row whose halves live in the two warps that share a TMEM lane quarter. Each warp
// brings the shifted sums of its 128 columns (s1 = sum(x - k), s2 = sum((x - k)^2), k = its first element: one pass, no
// cancellation); the halves are combined with the parallel-variance formula. The buffer is reused by LN2: by then
// both warps have passed the CTA-wide accumulator barriers, so the partner has long read the LN1 values.
__device__ __forceinline__ void pair_stats(float k, float s1, float s2, float* xch, const EpiW& e, float eps,
                                           float& mean, float& rstd) {
  const int set = 0;
  const float n = 128.f;
  const float mean_h = k + s1 / n;
  const float m2_h = s2 - s1 * s1 / n;
  float* mine = xch + ((set * 2 + e.half) * 4 + e.q) * 64 + e.lane * 2;
  mine[0] = mean_h; mine[1] = m2_h;
  named_bar_sync(2 + e.q, 64);
  const float* other = xch + ((set * 2 + (e.half ^ 1)) * 4 + e.q) * 64 + e.lane * 2;
  const float mean_o = other[0], m2_o = other[1];
  const float dm = mean_h - mean_o;
  mean = 0.5f * (mean_h + mean_o);
  const float m2 = m2_h + m2_o + dm * dm * (n * 0.5f);
  rstd = rsqrtf(m2 * (1.f / 256.f) + eps);
}

// final outputs of one 32-column chunk: fp32 box and / or (half of) a 64-column bf16 box -> TMA stores.
// Staging per warp: [2 x 4 KB fp32 boxes][2 x 4 KB bf16 boxes]; a box is refilled only after the store before last has
// finished reading shared memory (one store group per chunk), so the warp never waits for the store it just issued.
#ifdef MOCHA_TRACE
#define FT_TRACE_E(slot) do { if (e.ew == 0 && e.lane == 0 && c < 2) FT_TRACE(44 + 6 * c + (slot)); } while (0)
#else
#define FT_TRACE_E(slot) do { } while (0)
#endif
__device__ __forceinline__ void emit_chunk(const float (&f)[32], int col, int c, const EpiW& e, const TailParams& p,
                                           const CUtensorMap* tmO32, const CUtensorMap* tmO16) {
  FT_TRACE_E(0);
  const int sw = e.lane & 7;
  const int hcol = c & 1;
  const uint32_t box32 = e.stage + (uint32_t)(c & 1) * 4096u;
  const uint32_t box16 = e.stage + 8192u + (uint32_t)((c >> 1) & 1) * 4096u;
  // groups committed so far: one per chunk. Chunk c reuses box32 of chunk c-2 and (at hcol == 0) box16 of chunks c-4/c-3
  // -> at most the previous chunk's group may still be reading
  if (e.lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
  __syncwarp();
  FT_TRACE_E(1);
  if (p.out32) {
#pragma unroll
    for (int j = 0; j < 8; ++j)
      sts128(box32 + (uint32_t)(e.lane * 128 + ((j ^ sw) << 4)), __float_as_uint(f[4 * j]), __float_as_uint(f[4 * j + 1]),
             __float_as_uint(f[4 * j + 2]), __float_as_uint(f[4 * j + 3]));
  }
  if (p.out16) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      sts128(box16 + (uint32_t)(e.lane * 128 + (((j + 4 * hcol) ^ sw) << 4)), pack_bf16(f[8 * j], f[8 * j + 1]),
             pack_bf16(f[8 * j + 2], f[8 * j + 3]), pack_bf16(f[8 * j + 4], f[8 * j + 5]), pack_bf16(f[8 * j + 6], f[8 * j + 7]));
  }
  FT_TRACE_E(2);
  fence_proxy_async_smem();
  __syncwarp();
  FT_TRACE_E(3);
  if (e.lane == 0) {
    if (p.out32) tma_store_3d(tmO32, box32, col, e.m0 + e.q * 32, 0);
    if (p.out16 && hcol == 1) tma_store_3d(tmO16, box16, col - 32, e.m0 + e.q * 32, 0);
    bulk_commit();
  }
  FT_TRACE_E(4);
}

// Residual chunk [32 rows x 32 fp32] of this warp's slab. Loaded COALESCED (8 lanes x 16 B = one 128 B row segment,
// 4 rows per instruction) and transposed to the accumulator's lane = row layout through a per-warp 4 KB shared-memory
// tile (16 B chunks XOR-swizzled by row: conflict-free both ways). Reading it lane = row straight from global memory
// made every LDG.128 touch 32 different lines - 256 line requests per warp and chunk, ~1900 cycles per chunk on the
// L1 tag stage, the longest stall of this stage.
struct Res32 { float4 r[8]; };
__device__ __forceinline__ void load_res(Res32& x, const float* R0, long long slab_row0, int M, int col, int lane, int period) {
  const int rr = lane >> 3, c4 = (lane & 7) * 4;
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    const long long row = slab_row0 + rr + 4 * it;
    const long long src = period > 0 ? row % period : row;
    x.r[it] = (R0 && row < M) ? __ldg(reinterpret_cast<const float4*>(R0 + src * FT_D + col + c4)) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
}
// coalesced registers -> lane = row registers (warp-collective)
__device__ __forceinline__ void transpose_res(Res32& x, uint32_t tb, int lane) {
  const int rr = lane >> 3, cq = lane & 7;
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    const int r = rr + 4 * it;
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(tb + (uint32_t)(r * 128 + ((cq ^ (r & 7)) << 4))), "f"(x.r[it].x),
                 "f"(x.r[it].y), "f"(x.r[it].z), "f"(x.r[it].w)
                 : "memory");
  }
  __syncwarp();
#pragma unroll
  for (int j = 0; j < 8; ++j) x.r[j] = lds128f(tb + (uint32_t)(lane * 128 + ((j ^ (lane & 7)) << 4)));
  __syncwarp();
}
__device__ __forceinline__ void add_res(float (&f)[32], const Res32& x) {
#pragma unroll
  for (int j = 0; j < 8; ++j) { f[4 * j] += x.r[j].x; f[4 * j + 1] += x.r[j].y; f[4 * j + 2] += x.r[j].z; f[4 * j + 3] += x.r[j].w; }
}
__device__ __forceinline__ void ln_apply(float (&f)[32], uint32_t g_smem, uint32_t be_smem, int col, float mean, float rstd) {
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float4 gg = lds128f(g_smem + (uint32_t)(col + 4 * j) * 4u), bb = lds128f(be_smem + (uint32_t)(col + 4 * j) * 4u);
    f[4 * j] = (f[4 * j] - mean) * rstd * gg.x + bb.x;
    f[4 * j + 1] = (f[4 * j + 1] - mean) * rstd * gg.y + bb.y;
    f[4 * j + 2] = (f[4 * j + 2] - mean) * rstd * gg.z + bb.z;
    f[4 * j + 3] = (f[4 * j + 3] - mean) * rstd * gg.w + bb.w;
  }
}

__global__ void __launch_bounds__(FT_THREADS, 1)
tail_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmW0,
            const __grid_constant__ CUtensorMap tmW1, const __grid_constant__ CUtensorMap tmW2,
            const __grid_constant__ CUtensorMap tmO32, const __grid_constant__ CUtensorMap tmO16, const TailParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  pdl_trigger();
  if (threadIdx.x == 0) FT_TRACE(0);
  const uint32_t sbase = smem_u32(smem);
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + FT_OFF_BAR);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + B_COUNT);
  float* xch = reinterpret_cast<float*>(smem + FT_OFF_XCH);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0 && (sbase & 1023u) != 0) {
    printf("mocha tail kernel: dynamic shared memory base %u is not 1 KB aligned\n", sbase);
    __trap();
  }
  const int nkb0 = p.K0 / 64, nch = p.Hd / 128;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA0); tma_prefetch_desc(&tmW0);
    if (p.Hd > 0) { tma_prefetch_desc(&tmW1); tma_prefetch_desc(&tmW2); }
    for (int i = 0; i < FT_NSLOT; ++i) { mbar_init(&bar[B_FULLW + i], 1); mbar_init(&bar[B_EMPTYW + i], 1); }
    for (int i = 0; i < FT_NA; ++i) { mbar_init(&bar[B_FULLA + i], 1); mbar_init(&bar[B_EMPTYA + i], 1); }
    mbar_init(&bar[B_ACCP], 1);
    mbar_init(&bar[B_XREADY], 8);
    for (int i = 0; i < 2; ++i) { mbar_init(&bar[B_ACC1F + i], 1); mbar_init(&bar[B_ACC1E + i], 8); }
    mbar_init(&bar[B_HREADY], 8);
    mbar_init(&bar[B_HEMPTY], 1);
    mbar_init(&bar[B_ACC2], 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    // Weights are constants: pull every tile this CTA will stream into L2 now, under the previous kernel's tail. All
    // CTAs of the launch walk the same weight tiles in lockstep, so without this each ring refill is a fresh HBM miss
    // for everybody; the prefetches of different CTAs coalesce in L2. One box per lane: the issue cost stays off the
    // producer's critical path.
    const int nbox = nkb0 + nch * 6;
    for (int i = lane; i < nbox; i += 32) {
      if (i < nkb0) {
        tma_prefetch_l2_2d(&tmW0, i * 64, 0);
      } else {
        const int j = (i - nkb0) / 6, r = (i - nkb0) % 6;
        if (r < 4) tma_prefetch_l2_2d(&tmW1, r * 64, j * 128);
        else tma_prefetch_l2_2d(&tmW2, j * 128 + (r - 4) * 64, 0);
      }
    }
  }
  if (warp >= 2) {
    // bias / LayerNorm vectors -> shared memory with cp.async (constants: requested before the grid dependency is waited
    // for and NOT awaited here - the epilogue warps wait for them right before their first use, several microseconds
    // later; a blocking load here cost 4400 cycles of prologue on the critical path)
    const uint32_t par_s = sbase + FT_OFF_PAR;
    const int t = (int)threadIdx.x - 64;
#pragma unroll
    for (int it = 0; it < PV_COUNT / 4 / 256; ++it) {
      const int i = (t + it * 256) * 4;
      const float* src = i < PV_G1 ? p.b0 : i < PV_BE1 ? p.g1 : i < PV_B1 ? p.be1 : i < PV_B2 ? p.b1 : i < PV_G2 ? p.b2 : i < PV_BE2 ? p.g2 : p.be2;
      const int base = i < PV_G1 ? PV_B0 : i < PV_BE1 ? PV_G1 : i < PV_B1 ? PV_BE1 : i < PV_B2 ? PV_B1 : i < PV_G2 ? PV_B2 : i < PV_BE2 ? PV_G2 : PV_BE2;
      const int len = base == PV_B1 ? p.Hd : FT_D;
      if (src && i - base < len) {
        asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(par_s + (uint32_t)i * 4u), "l"(src + (i - base)) : "memory");
      } else {
        asm volatile("st.shared.v4.f32 [%0], {%1, %1, %1, %1};" ::"r"(par_s + (uint32_t)i * 4u), "f"(0.f) : "memory");
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  pdl_wait();   // PDL: the prologue above overlapped the previous kernel's tail
  if (threadIdx.x == 0) FT_TRACE(1);

  const int m0 = blockIdx.x * 128;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int sw = 0; uint32_t pw = 0;
      int sa = 0; uint32_t pa = 0;
      for (int kb = 0; kb < nkb0; ++kb) {
        mbar_wait(&bar[B_EMPTYA + sa], pa ^ 1);
        mbar_expect_tx(&bar[B_FULLA + sa], 16384);
        tma_load_2d(sbase + FT_OFF_HB + sa * 16384, &tmA0, &bar[B_FULLA + sa], kb * 64, m0);
        if (++sa == FT_NA) { sa = 0; pa ^= 1; }
        mbar_wait(&bar[B_EMPTYW + sw], pw ^ 1);
        mbar_expect_tx(&bar[B_FULLW + sw], FT_SLOT);
        tma_load_2d(sbase + FT_OFF_RING + sw * FT_SLOT, &tmW0, &bar[B_FULLW + sw], kb * 64, 0);
        if (++sw == FT_NSLOT) { sw = 0; pw ^= 1; }
      }
      FT_TRACE(2);   // producer: all prefix loads issued
      for (int step = 0; step <= nch && nch > 0; ++step) {
        if (step < nch) {               // W1 rows [128 j, +128): two slots of two k-blocks each
          const int j = step;
          for (int s2 = 0; s2 < 2; ++s2) {
            mbar_wait(&bar[B_EMPTYW + sw], pw ^ 1);
            mbar_expect_tx(&bar[B_FULLW + sw], FT_SLOT);
            tma_load_2d(sbase + FT_OFF_RING + sw * FT_SLOT, &tmW1, &bar[B_FULLW + sw], (2 * s2) * 64, j * 128);
            tma_load_2d(sbase + FT_OFF_RING + sw * FT_SLOT + 16384, &tmW1, &bar[B_FULLW + sw], (2 * s2 + 1) * 64, j * 128);
            if (++sw == FT_NSLOT) { sw = 0; pw ^= 1; }
          }
        }
        if (step >= 1) {                // W2 columns [128 j, +128): two k-blocks of 256 rows
          const int j = step - 1;
          for (int kk = 0; kk < 2; ++kk) {
            mbar_wait(&bar[B_EMPTYW + sw], pw ^ 1);
            mbar_expect_tx(&bar[B_FULLW + sw], FT_SLOT);
            tma_load_2d(sbase + FT_OFF_RING + sw * FT_SLOT, &tmW2, &bar[B_FULLW + sw], j * 128 + kk * 64, 0);
            if (++sw == FT_NSLOT) { sw = 0; pw ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      constexpr uint32_t idesc256 = make_idesc(128, 256), idesc128 = make_idesc(128, 128);
      const uint32_t accY = tmem;                 // columns [0,256): out-projection, then Y + FFN output
      int sw = 0; uint32_t pw = 0;
      int sa = 0; uint32_t pa = 0;
      for (int kb = 0; kb < nkb0; ++kb) {
        mbar_wait(&bar[B_FULLA + sa], pa);
        mbar_wait(&bar[B_FULLW + sw], pw);
        tc_fence_after();
        if (kb == 0) FT_TRACE(4);   // MMA: first operands landed
        const uint64_t adesc = make_smem_desc(sbase + FT_OFF_HB + sa * 16384);
        const uint64_t bdesc = make_smem_desc(sbase + FT_OFF_RING + sw * FT_SLOT);
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_bf16(accY, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc256, (kb | k) != 0);
        umma_commit(&bar[B_EMPTYA + sa]);
        umma_commit(&bar[B_EMPTYW + sw]);
        if (++sa == FT_NA) { sa = 0; pa ^= 1; }
        if (++sw == FT_NSLOT) { sw = 0; pw ^= 1; }
      }
      umma_commit(&bar[B_ACCP]);
      FT_TRACE(5);     // MMA: prefix issued
      if (nch > 0) {
        mbar_wait(&bar[B_XREADY], 0);   // X tile in shared memory, Y in TMEM
        tc_fence_after();
        FT_TRACE(6);   // MMA: X ready
        for (int step = 0; step <= nch; ++step) {
          if (step < nch) {
            const int j = step, b = j & 1, u = j >> 1;
            if (j >= 2) { mbar_wait(&bar[B_ACC1E + b], (uint32_t)((u - 1) & 1)); tc_fence_after(); }
            const uint32_t acc1 = tmem + 256u + 128u * (uint32_t)b;
            for (int s2 = 0; s2 < 2; ++s2) {
              mbar_wait(&bar[B_FULLW + sw], pw);
              tc_fence_after();
#pragma unroll
              for (int kk = 0; kk < 2; ++kk) {
                const int kb = 2 * s2 + kk;
                const uint64_t adesc = make_smem_desc(sbase + FT_OFF_X + kb * 16384);
                const uint64_t bdesc = make_smem_desc(sbase + FT_OFF_RING + sw * FT_SLOT + kk * 16384);
#pragma unroll
                for (int k = 0; k < 4; ++k)
                  umma_bf16(acc1, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc128, (kb | k) != 0);
              }
              umma_commit(&bar[B_EMPTYW + sw]);
              if (++sw == FT_NSLOT) { sw = 0; pw ^= 1; }
            }
            umma_commit(&bar[B_ACC1F + b]);
            FT_TRACE(8 + j);    // MMA: G1(j) issued
          }
          if (step >= 1) {
            const int j = step - 1;
            mbar_wait(&bar[B_HREADY], (uint32_t)(j & 1));
            tc_fence_after();
            for (int kk = 0; kk < 2; ++kk) {
              mbar_wait(&bar[B_FULLW + sw], pw);
              tc_fence_after();
              const uint64_t adesc = make_smem_desc(sbase + FT_OFF_HB + kk * 16384);
              const uint64_t bdesc = make_smem_desc(sbase + FT_OFF_RING + sw * FT_SLOT);
#pragma unroll
              for (int k = 0; k < 4; ++k) umma_bf16(accY, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc256, 1u);
              umma_commit(&bar[B_EMPTYW + sw]);
              if (++sw == FT_NSLOT) { sw = 0; pw ^= 1; }
            }
            umma_commit(&bar[B_HEMPTY]);
            FT_TRACE(16 + j);   // MMA: G2(j) issued
          }
        }
        umma_commit(&bar[B_ACC2]);
      }
    }
  } else {
    // ===================== epilogue (warps 2..9) =====================
    EpiW e;
    e.lane = lane; e.ew = warp - 2; e.q = warp & 3; e.half = e.ew >> 2;
    e.row_l = e.q * 32 + lane;
    e.row = (long long)m0 + e.row_l;
    e.row_ok = e.row < p.M;
    e.taddr = tmem + ((uint32_t)(e.q * 32) << 16);
    e.m0 = m0;
    e.stage = sbase + (uint32_t)e.ew * 16384u;   // over X / HB / first ring slot: all free whenever outputs are emitted
    const uint32_t par = sbase + FT_OFF_PAR;
    const int colbase = 128 * e.half;
    const int sw7 = lane & 7;

    // ---- stage P: Y = LN1?(acc + b0 + R0) -> TMEM (fp32) + X tile (bf16)   or, without an FFN, -> outputs ----
    // the residual of the first chunk is requested before the accumulator is waited for, the next chunk's while the
    // current one is processed: the L2 latency of these strided row reads was the longest stall of this stage
    Res32 res;
    const long long slab_row0 = (long long)m0 + e.q * 32;
    // transposition tile: the A stages are free once the out-projection has completed; without an FFN the ring is
    const uint32_t tb = sbase + (nch > 0 ? FT_OFF_HB : FT_OFF_RING + FT_SLOT) + (uint32_t)e.ew * 4096u;
    load_res(res, p.R0, slab_row0, p.M, colbase, lane, p.r0_period);
    // the staged vectors: every epilogue thread's own cp.async requests have landed, then all of them have
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    named_bar_sync(1, 256);
    mbar_wait(&bar[B_ACCP], 0);
    tc_fence_after();
    if (warp == 2 && lane == 0) FT_TRACE(24);   // epilogue: out-projection accumulator ready
    const bool ln1 = p.g1 != nullptr;
    float mean = 0.f, rstd = 1.f;
    if (ln1) {
      float k = 0.f, s1 = 0.f, s2 = 0.f;
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        const int col = colbase + 32 * c;
        uint32_t v[32];
        tmem_ld32(e.taddr + (uint32_t)col, v);
        float f[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[i]);
        if (p.R0) { transpose_res(res, tb, lane); add_res(f, res); }
        if (c < 3) load_res(res, p.R0, slab_row0, p.M, col + 32, lane, p.r0_period);
        if (p.b0) add_bias32(f, par + PV_B0 * 4u, col);
        if (c == 0) k = f[0];
#pragma unroll
        for (int i = 0; i < 32; ++i) { const float d = f[i] - k; s1 += d; s2 = fmaf(d, d, s2); v[i] = __float_as_uint(f[i]); }
        tmem_st32(e.taddr + (uint32_t)col, v);
      }
      pair_stats(k, s1, s2, xch, e, p.eps, mean, rstd);
      if (warp == 2 && lane == 0) FT_TRACE(25);   // epilogue: LN1 statistics done
    }
#pragma unroll 1
    for (int c = 0; c < 4; ++c) {
      const int col = colbase + 32 * c;
      uint32_t v[32];
      tmem_ld32(e.taddr + (uint32_t)col, v);
      float f[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[i]);
      if (ln1) {
        ln_apply(f, par + PV_G1 * 4u, par + PV_BE1 * 4u, col, mean, rstd);
      } else {
        if (p.R0) { transpose_res(res, tb, lane); add_res(f, res); }
        if (c < 3) load_res(res, p.R0, slab_row0, p.M, col + 32, lane, p.r0_period);
        if (p.b0) add_bias32(f, par + PV_B0 * 4u, col);
      }
      if (nch > 0) {
        // Y stays in TMEM as the accumulation base of the second FFN GEMM; its bf16 copy is the first one's A operand
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = __float_as_uint(f[i]);
        tmem_st32(e.taddr + (uint32_t)col, v);
        const int kb = col >> 6, c16 = (col & 63) >> 3;     // k-block of the X tile, first 16 B chunk inside its row
        const uint32_t xrow = sbase + FT_OFF_X + (uint32_t)kb * 16384u + (uint32_t)e.row_l * 128u;
#pragma unroll
        for (int t = 0; t < 4; ++t)
          sts128(xrow + (uint32_t)(((c16 + t) ^ sw7) << 4), pack_bf16(f[8 * t], f[8 * t + 1]), pack_bf16(f[8 * t + 2], f[8 * t + 3]),
                 pack_bf16(f[8 * t + 4], f[8 * t + 5]), pack_bf16(f[8 * t + 6], f[8 * t + 7]));
      } else {
        emit_chunk(f, col, c, e, p, &tmO32, &tmO16);
      }
    }
    if (nch > 0) {
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar[B_XREADY]);
      if (warp == 2 && lane == 0) FT_TRACE(26);   // epilogue: stage P done

      // ---- hidden chunks: H_j = act(acc1 + b1) -> bf16 A operand of the second FFN GEMM ----
#pragma unroll 1
      for (int j = 0; j < nch; ++j) {
        const int b = j & 1, u = j >> 1;
        mbar_wait(&bar[B_ACC1F + b], (uint32_t)(u & 1));
        tc_fence_after();
        if (warp == 2 && lane == 0) FT_TRACE(28 + 2 * j);   // epilogue: hidden chunk j ready
        const uint32_t hrow = sbase + FT_OFF_HB + (uint32_t)e.half * 16384u + (uint32_t)e.row_l * 128u;
        float hf[2][32];
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
          uint32_t v[32];
          tmem_ld32(e.taddr + 256u + 128u * (uint32_t)b + (uint32_t)(64 * e.half + 32 * cc), v);
          float (&f)[32] = hf[cc];
#pragma unroll
          for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[i]);
          if (p.b1) add_bias32(f, par + PV_B1 * 4u, j * 128 + 64 * e.half + 32 * cc);
          if (p.act == ACT_RELU) {
#pragma unroll
            for (int i = 0; i < 32; ++i) f[i] = fmaxf(f[i], 0.f);
          } else if (p.act == ACT_GELU) {
#pragma unroll
            for (int i = 0; i < 32; ++i) f[i] = gelu_tanh_f(f[i]);
          } else if (p.act == ACT_LRELU) {
#pragma unroll
            for (int i = 0; i < 32; ++i) f[i] = lrelu02(f[i]);
          }
        }
        // the accumulator is drained: the next-but-one hidden GEMM may overwrite it
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar[B_ACC1E + b]);
        // single hidden buffer: the previous chunk's second GEMM must have finished reading it
        if (j >= 1) mbar_wait(&bar[B_HEMPTY], (uint32_t)((j - 1) & 1));
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
          const float (&f)[32] = hf[cc];
#pragma unroll
          for (int t = 0; t < 4; ++t)
            sts128(hrow + (uint32_t)(((4 * cc + t) ^ sw7) << 4), pack_bf16(f[8 * t], f[8 * t + 1]), pack_bf16(f[8 * t + 2], f[8 * t + 3]),
                   pack_bf16(f[8 * t + 4], f[8 * t + 5]), pack_bf16(f[8 * t + 6], f[8 * t + 7]));
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar[B_HREADY]);
        if (warp == 2 && lane == 0) FT_TRACE(29 + 2 * j);   // epilogue: hidden chunk j stored
      }

      // ---- final: Z = LN2?(acc + b2) -> outputs ----
      mbar_wait(&bar[B_ACC2], 0);
      tc_fence_after();
      if (warp == 2 && lane == 0) FT_TRACE(40);   // epilogue: FFN accumulator ready
      const bool ln2 = p.g2 != nullptr;
      float mean2 = 0.f, rstd2 = 1.f;
      if (ln2) {
        float k = 0.f, s1 = 0.f, s2 = 0.f;
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
          const int col = colbase + 32 * c;
          uint32_t v[32];
          tmem_ld32(e.taddr + (uint32_t)col, v);
          float f[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[i]);
          if (p.b2) add_bias32(f, par + PV_B2 * 4u, col);
          if (c == 0) k = f[0];
#pragma unroll
          for (int i = 0; i < 32; ++i) { const float d = f[i] - k; s1 += d; s2 = fmaf(d, d, s2); v[i] = __float_as_uint(f[i]); }
          tmem_st32(e.taddr + (uint32_t)col, v);
        }
        pair_stats(k, s1, s2, xch, e, p.eps, mean2, rstd2);
      }
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        const int col = colbase + 32 * c;
        uint32_t v[32];
        tmem_ld32(e.taddr + (uint32_t)col, v);
        float f[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[i]);
        if (warp == 2 && lane == 0 && c < 2) FT_TRACE(56 + 2 * c);       // final stage: accumulator chunk in registers
        if (ln2) ln_apply(f, par + PV_G2 * 4u, par + PV_BE2 * 4u, col, mean2, rstd2);
        else if (p.b2) add_bias32(f, par + PV_B2 * 4u, col);
        emit_chunk(f, col, c, e, p, &tmO32, &tmO16);
      }
    }
    if (warp == 2 && lane == 0) FT_TRACE(41);     // epilogue: all output chunks handed to TMA
    if (lane == 0) bulk_wait_read0();   // staging must outlive the stores that read it
    if (warp == 2 && lane == 0) FT_TRACE(42);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
  if (threadIdx.x == 0) FT_TRACE(43);
}

}  // namespace

bool tc_tail_supported(int M, int K0, int Hd) {
  return M >= 1 && K0 >= 64 && (K0 % 64) == 0 && Hd >= 0 && (Hd % 128) == 0 && Hd <= FT_MAX_HD;
}

int tc_tail(const __nv_bfloat16* A0, int lda, int K0, const __nv_bfloat16* W0, const float* b0, const float* R0,
            const float* g1, const float* be1, int Hd, int act, const __nv_bfloat16* W1, const float* b1,
            const __nv_bfloat16* W2, const float* b2, const float* g2, const float* be2, float eps, float* O32,
            __nv_bfloat16* O16, int M, cudaStream_t s, int r0_period) {
  MOCHA_CHECK_ARG(tc_tail_supported(M, K0, Hd), "tc_tail: unsupported shape M=%d K0=%d hidden=%d", M, K0, Hd);
  MOCHA_CHECK_ARG(A0 && W0 && (O32 || O16), "tc_tail: null operand");
  MOCHA_CHECK_ARG(Hd == 0 || (W1 && W2), "tc_tail: FFN weights missing");
  MOCHA_CHECK_ARG((g1 == nullptr) == (be1 == nullptr) && (g2 == nullptr) == (be2 == nullptr), "tc_tail: LayerNorm needs gamma and beta");
  const uintptr_t al = reinterpret_cast<uintptr_t>(b0) | reinterpret_cast<uintptr_t>(R0) | reinterpret_cast<uintptr_t>(g1) |
                       reinterpret_cast<uintptr_t>(be1) | reinterpret_cast<uintptr_t>(b1) | reinterpret_cast<uintptr_t>(b2) |
                       reinterpret_cast<uintptr_t>(g2) | reinterpret_cast<uintptr_t>(be2) | reinterpret_cast<uintptr_t>(O32) |
                       reinterpret_cast<uintptr_t>(O16);
  MOCHA_CHECK_ARG((al & 15) == 0, "tc_tail: vectors and outputs must be 16 B aligned");
  CUtensorMap tmA0, tmW0, tmW1, tmW2, tmO32, tmO16;
  MOCHA_TRY(tc_make_tmap(&tmA0, A0, (unsigned long long)M, (unsigned long long)K0, 128, (unsigned long long)lda));
  MOCHA_TRY(tc_make_tmap(&tmW0, W0, FT_D, (unsigned long long)K0, 256));
  if (Hd > 0) {
    MOCHA_TRY(tc_make_tmap(&tmW1, W1, (unsigned long long)Hd, FT_D, 128));
    MOCHA_TRY(tc_make_tmap(&tmW2, W2, FT_D, (unsigned long long)Hd, 256));
  } else {
    tmW1 = tmW0; tmW2 = tmW0;
  }
  if (O32) MOCHA_TRY(tc_make_out_tmap(&tmO32, O32, FT_D, (unsigned long long)M, 1, FT_D, true));
  else tmO32 = tmW0;
  if (O16) MOCHA_TRY(tc_make_out_tmap(&tmO16, O16, FT_D, (unsigned long long)M, 1, FT_D, false, 0, true));
  else tmO16 = tmW0;
  TailParams p{};
  p.M = M; p.K0 = K0; p.Hd = Hd; p.act = act;
  p.b0 = b0; p.R0 = R0; p.g1 = g1; p.be1 = be1; p.b1 = b1; p.b2 = b2; p.g2 = g2; p.be2 = be2;
  p.eps = eps; p.out32 = O32 != nullptr; p.out16 = O16 != nullptr;
  p.r0_period = r0_period;
  static bool configured = false;
  if (!configured) {
    MOCHA_CUDA(cudaFuncSetAttribute(tail_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FT_SMEM));
    configured = true;
  }
  launch_k(tail_kernel, dim3((unsigned)ceil_div(M, 128)), dim3(FT_THREADS), (size_t)FT_SMEM, s, tmA0, tmW0, tmW1, tmW2, tmO32,
           tmO16, p);
  count_launch();
  MOCHA_LAUNCH_CHECK("tail_kernel");
  return MOCHA_OK;
}

}  // namespace mocha

#ifdef MOCHA_TRACE
extern "C" int mocha_debug_set_tail_trace(unsigned long long* buf) {
  return cudaMemcpyToSymbol(mocha::g_ft_trace, &buf, sizeof(buf)) == cudaSuccess ? 0 : 1;
}
#endif
