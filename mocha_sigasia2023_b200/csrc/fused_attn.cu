// Fused attention core on tcgen05 (sm_100a): softmax(Q K^T / sqrt(dh)) V for B x H (clip, head) problems in ONE launch
// (net/transformer.py:37-76; nn.MultiheadAttention inside model_CVAE.py's encoder / decoder layers).
//
// One persistent CTA per SM walks units (clip b, head h, 128-row query tile). Per unit:
//   S = Q_h K_h^T            tcgen05.mma, fp32 scores in TMEM columns [0, npad)              (npad = keys rounded up to 64)
//   P = exp2((S - max) c)    softmax in the epilogue warps straight from TMEM; the unnormalised bf16 probabilities go to
//                            shared memory as the K-major, 128 B-swizzled A operand of the second GEMM (they used to
//                            round-trip through HBM between two launches)
//   O = P V_h                V read in place as an MN-major B operand, fp32 accumulators in TMEM columns [256, 256 + dh)
//   out = O / sum(P)         bf16, TMA store into the [B, nq, H*dh] tensor the out-projection reads
// Q, K, V, P each have ONE shared-memory buffer with its own full / empty barrier, so the TMA producer refills Q and K
// for the next unit as soon as the score GEMM has read them (under the softmax, the second GEMM and the output
// epilogue of the current unit) and V as soon as the second GEMM has; the score GEMM of unit u+1 is issued before the
// P V GEMM of unit u. Warp roles as in gemm_tc.cu: warp 0 TMA producer, warp 1 MMA issuer + TMEM owner, warps 2..9
// epilogue (two warps per TMEM lane quarter split the key columns / the head dimension and exchange row maxima and sums).
#include "fused.cuh"

#include "gemm_tc.cuh"
#include "tc_ptx.cuh"

namespace mocha {

using namespace tcx;

namespace {

constexpr int FA_THREADS = 320;
// per-buffer barriers come in pairs ([0], [1]) for the two-group mode
enum { A_QKFULL = 0, A_QKEMPTY = 2, A_VFULL = 4, A_VEMPTY, A_SFULL, A_SEMPTY = A_SFULL + 2, A_PREADY = A_SEMPTY + 2, A_OFULL = A_PREADY + 2,
       A_OEMPTY = A_OFULL + 2, A_COUNT = A_OEMPTY + 2 };

#ifdef MOCHA_TRACE
// trace build: per-CTA clock64 time line (tools/attn_trace.py), 64 slots per CTA: 16 per unit for the first 4 units
__device__ unsigned long long* g_fa_trace = nullptr;
#define FA_TRACE(it, slot)                                                                                          \
  do {                                                                                                              \
    if (g_fa_trace && (it) < 4) g_fa_trace[(size_t)blockIdx.x * 64 + (it) * 16 + (slot)] = (unsigned long long)clock64(); \
  } while (0)
#else
#define FA_TRACE(it, slot) do { } while (0)
#endif

struct AttnParams {
  int B, H, nq, nkv, dh, npad;   // npad = nkv rounded up to a multiple of 64 (<= 256)
  int q_rows_b;                  // Q rows per clip: nq, or 0 when every clip shares one [nq, H*dh] query table
  int nqt;                       // query tiles per (clip, head)
  int units;
  float scale_log2e;             // log2(e) / sqrt(dh)
  uint32_t off_k, off_v, off_p, off_bar, off_xch;   // shared-memory plan (Q at 0)
  uint32_t p_bytes;              // one P buffer
  int qk_stages;                 // 1 or 2 Q / K buffers (stride qk_stride bytes; K at off_k inside a stage)
  uint32_t qk_stride;
  int groups;                    // 2: the two warps of a TMEM lane quarter alternate units (double-buffered S / O / P)
};

__device__ __forceinline__ void tma_store_3d(const CUtensorMap* tm, uint32_t smem_addr, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(tm), "r"(smem_addr),
               "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__global__ void __launch_bounds__(FA_THREADS, 1)
attn_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
            const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmO, const AttnParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  pdl_trigger();
  if (threadIdx.x == 0) FA_TRACE(0, 14);   // CTA start
  const uint32_t sbase = smem_u32(smem);
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + p.off_bar);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + A_COUNT);
  float* xch = reinterpret_cast<float*>(smem + p.off_xch);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0 && (sbase & 1023u) != 0) {
    printf("mocha attention kernel: dynamic shared memory base %u is not 1 KB aligned\n", sbase);
    __trap();
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmQ); tma_prefetch_desc(&tmK); tma_prefetch_desc(&tmV); tma_prefetch_desc(&tmO);
    for (int i = 0; i < 2; ++i) { mbar_init(&bar[A_QKFULL + i], 1); mbar_init(&bar[A_QKEMPTY + i], 1); }
    mbar_init(&bar[A_VFULL], 1); mbar_init(&bar[A_VEMPTY], 1);
    const uint32_t narr = p.groups == 2 ? 4 : 8;      // epilogue warps per unit
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bar[A_SFULL + i], 1); mbar_init(&bar[A_SEMPTY + i], narr);
      mbar_init(&bar[A_PREADY + i], narr);
      mbar_init(&bar[A_OFULL + i], 1); mbar_init(&bar[A_OEMPTY + i], narr);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  pdl_wait();
  if (threadIdx.x == 0) FA_TRACE(0, 15);   // prologue done

  const int dkb = p.dh / 64;          // k-blocks of the head dimension
  const int nkb = p.npad / 64;        // k-blocks of the key dimension
  const uint32_t q_bytes = (uint32_t)dkb * 16384u, k_bytes = (uint32_t)dkb * (uint32_t)p.npad * 128u;
  const uint32_t v_bytes = (uint32_t)nkb * (uint32_t)dkb * 8192u;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      uint32_t n = 0;
      for (int u = blockIdx.x; u < p.units; u += gridDim.x) ++n;
      const uint32_t QS = (uint32_t)p.qk_stages;
      auto load_qk = [&](uint32_t it) {
        const int u = blockIdx.x + (int)it * gridDim.x;
        const int qt = u % p.nqt, h = (u / p.nqt) % p.H, b = u / (p.nqt * p.H);
        const uint32_t st = it % QS, ph = (it / QS) & 1;
        mbar_wait(&bar[A_QKEMPTY + st], ph ^ 1);
        FA_TRACE(it, 0);   // producer: Q / K buffer free
        mbar_expect_tx(&bar[A_QKFULL + st], q_bytes + k_bytes);
        const uint32_t base = sbase + st * p.qk_stride;
        for (int kb = 0; kb < dkb; ++kb) {
          tma_load_2d(base + (uint32_t)kb * 16384u, &tmQ, &bar[A_QKFULL + st], h * p.dh + kb * 64, b * p.q_rows_b + qt * 128);
          tma_load_2d(base + p.off_k + (uint32_t)kb * (uint32_t)p.npad * 128u, &tmK, &bar[A_QKFULL + st], h * p.dh + kb * 64, b * p.nkv);
        }
      };
      auto load_v = [&](uint32_t it) {
        const int u = blockIdx.x + (int)it * gridDim.x;
        const int h = (u / p.nqt) % p.H, b = u / (p.nqt * p.H);
        mbar_wait(&bar[A_VEMPTY], (it & 1) ^ 1);
        FA_TRACE(it, 1);   // producer: V buffer free
        mbar_expect_tx(&bar[A_VFULL], v_bytes);
        for (int kb = 0; kb < nkb; ++kb)
          for (int a = 0; a < dkb; ++a)
            tma_load_2d(sbase + p.off_v + (uint32_t)(kb * dkb + a) * 8192u, &tmV, &bar[A_VFULL], h * p.dh + a * 64, b * p.nkv + kb * 64);
      };
      // Q / K run QS units ahead of V: the score GEMM of a later unit never waits behind the V refill, which has to wait
      // for the previous unit's second GEMM
      for (uint32_t it = 0; it < QS && it < n; ++it) load_qk(it);
      for (uint32_t it = 0; it < n; ++it) {
        load_v(it);
        if (it + QS < n) load_qk(it + QS);
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc_s = make_idesc(128, p.npad), idesc_o = make_idesc(128, p.dh, true);
      const int G = p.groups;
      // TMEM plan: one group: S at [0, npad), O at [256, 256 + dh); two groups: S[b] at b*npad, O[b] at 2*npad + b*dh
      auto acc_s = [&](int b) { return tmem + (uint32_t)(b * p.npad); };
      auto acc_o = [&](int b) { return tmem + (G == 2 ? (uint32_t)(2 * p.npad + b * p.dh) : 256u); };
      auto issue_s = [&](uint32_t it) {
        const int b = G == 2 ? (int)(it & 1) : 0;
        const uint32_t ub = G == 2 ? it >> 1 : it;     // use count of buffer b
        const uint32_t QS = (uint32_t)p.qk_stages, st = it % QS;
        mbar_wait(&bar[A_QKFULL + st], (it / QS) & 1);
        FA_TRACE(it, 2);   // MMA: Q / K landed
        mbar_wait(&bar[A_SEMPTY + b], (ub & 1) ^ 1);
        tc_fence_after();
        FA_TRACE(it, 3);   // MMA: score accumulator free, issuing S
        for (int kb = 0; kb < dkb; ++kb) {
          const uint64_t adesc = make_smem_desc(sbase + st * p.qk_stride + (uint32_t)kb * 16384u);
          const uint64_t bdesc = make_smem_desc(sbase + st * p.qk_stride + p.off_k + (uint32_t)kb * (uint32_t)p.npad * 128u);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_bf16(acc_s(b), adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc_s, (kb | k) != 0);
        }
        umma_commit(&bar[A_QKEMPTY + st]);
        umma_commit(&bar[A_SFULL + b]);
      };
      auto issue_o = [&](uint32_t it) {
        const int b = G == 2 ? (int)(it & 1) : 0;
        const uint32_t ub = G == 2 ? it >> 1 : it;
        mbar_wait(&bar[A_PREADY + b], ub & 1);
        FA_TRACE(it, 4);   // MMA: P ready
        mbar_wait(&bar[A_VFULL], it & 1);
        mbar_wait(&bar[A_OEMPTY + b], (ub & 1) ^ 1);
        tc_fence_after();
        FA_TRACE(it, 5);   // MMA: V landed + output accumulator free, issuing P V
        for (int kb = 0; kb < nkb; ++kb) {
          const uint64_t adesc = make_smem_desc(sbase + p.off_p + (uint32_t)b * p.p_bytes + (uint32_t)kb * 16384u);
          // MN-major V: one MMA consumes 16 key rows = 2 KB of every 64-column atom
          const uint64_t bdesc = make_smem_desc_mn(sbase + p.off_v + (uint32_t)(kb * dkb) * 8192u, 8192u);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_bf16(acc_o(b), adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(128 * k), idesc_o, (kb | k) != 0);
        }
        umma_commit(&bar[A_VEMPTY]);
        umma_commit(&bar[A_OFULL + b]);
      };
      uint32_t n = 0;
      for (int u = blockIdx.x; u < p.units; u += gridDim.x) ++n;
      // the score GEMMs run G units ahead of the P V products
      for (uint32_t it = 0; it < (uint32_t)G && it < n; ++it) issue_s(it);
      for (uint32_t it = 0; it < n; ++it) {
        if (G == 1 && it + 1 < n) issue_s(it + 1);
        issue_o(it);
        if (G == 2 && it + 2 < n) issue_s(it + 2);
      }
    }
  } else {
    // ===================== epilogue (warps 2..9) =====================
    // One group: the two warps of a TMEM lane quarter split the key columns / the head dimension of EVERY unit and
    // exchange row maxima and sums. Two groups (when 2 x (npad + dh) TMEM columns and two P buffers fit): warp `half`
    // of each quarter owns whole rows of the units with (it & 1) == half, so one group's softmax runs while the other
    // group waits for its P V product - the kernel is epilogue-bound, and this hides the waits.
    const int ew = warp - 2, q = warp & 3, half = ew >> 2;
    const int G = p.groups;
    const int row_l = q * 32 + lane, sw7 = lane & 7;
    const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16);
    const int scols = G == 2 ? p.npad : p.npad / 2;             // score columns of this warp
    const int sc0 = G == 2 ? 0 : half * scols;
    const bool o_active = G == 2 || p.dh >= 128 || half == 0;
    const int ocols = G == 2 ? p.dh : (p.dh >= 128 ? p.dh / 2 : p.dh);   // head-dimension columns of this warp
    const int oc0 = G == 2 ? 0 : (p.dh >= 128 ? half * ocols : 0);
    uint32_t it = 0;
    for (int u = blockIdx.x; u < p.units; u += gridDim.x, ++it) {
      if (G == 2 && (int)(it & 1) != half) continue;
      const int bsel = G == 2 ? half : 0;                        // S / O / P buffer of this unit
      const uint32_t ub = G == 2 ? it >> 1 : it;
      const uint32_t ph = ub & 1;
      const int qt = u % p.nqt, h = (u / p.nqt) % p.H, b = u / (p.nqt * p.H);
      const uint32_t t_s = taddr + (uint32_t)(bsel * p.npad);
      const uint32_t t_o = taddr + (G == 2 ? (uint32_t)(2 * p.npad + bsel * p.dh) : 256u);
      const uint32_t pbuf = sbase + p.off_p + (uint32_t)bsel * p.p_bytes;
      // output staging inside this unit's (then idle) P buffer: one group: 4 KB per warp; two groups: 2 x 4 KB per warp
      const uint32_t stage = pbuf + (G == 2 ? (uint32_t)q * 8192u : (uint32_t)ew * 4096u);
      // ---- softmax ----
      mbar_wait(&bar[A_SFULL + bsel], ph);
      tc_fence_after();
      if (warp == 2 && lane == 0) FA_TRACE(it, 8);    // epilogue: scores ready
      float m = -INFINITY;
#pragma unroll 1
      for (int c = 0; c < scols; c += 32) {
        uint32_t v[32];
        tmem_ld32(t_s + (uint32_t)(sc0 + c), v);
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (sc0 + c + j < p.nkv) m = fmaxf(m, __uint_as_float(v[j]));
      }
      if (G == 1) {
        xch[(half * 4 + q) * 32 + lane] = m;
        named_bar_sync(2 + q, 64);
        m = fmaxf(m, xch[((half ^ 1) * 4 + q) * 32 + lane]);
      }
      // the previous output stores of this buffer read their staging boxes out of the P buffer: they must have left it,
      // in every warp that shares it, before new probabilities are written
      if (ub > 0) {
        if (lane == 0) bulk_wait_read0();
        if (G == 2) named_bar_sync(6 + half, 128);
        else named_bar_sync(1, 256);
      }
      if (warp == 2 && lane == 0) FA_TRACE(it, 9);    // epilogue: row max known, P buffer free
      const float ms = m * p.scale_log2e;
      float sum = 0.f;
#pragma unroll 1
      for (int c = 0; c < scols; c += 32) {
        const int col = sc0 + c;
        uint32_t v[32];
        tmem_ld32(t_s + (uint32_t)col, v);
        float e[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) e[j] = col + j < p.nkv ? ex2(fmaf(__uint_as_float(v[j]), p.scale_log2e, -ms)) : 0.f;
        const uint32_t prow = pbuf + (uint32_t)(col >> 6) * 16384u + (uint32_t)row_l * 128u;
        const int c16 = (col & 63) >> 3;
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          uint32_t pk[4];
#pragma unroll
          for (int w2 = 0; w2 < 4; ++w2) {
            __nv_bfloat162 h2 = __floats2bfloat162_rn(e[8 * t + 2 * w2], e[8 * t + 2 * w2 + 1]);
            sum += __low2float(h2) + __high2float(h2);       // the denominator sums what the second GEMM multiplies
            pk[w2] = *reinterpret_cast<uint32_t*>(&h2);
          }
          sts128(prow + (uint32_t)(((c16 + t) ^ sw7) << 4), pk[0], pk[1], pk[2], pk[3]);
        }
      }
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) { mbar_arrive(&bar[A_SEMPTY + bsel]); mbar_arrive(&bar[A_PREADY + bsel]); }
      if (warp == 2 && lane == 0) FA_TRACE(it, 10);   // epilogue: P written
      if (G == 1) {
        xch[256 + (half * 4 + q) * 32 + lane] = sum;
        named_bar_sync(2 + q, 64);
        sum += xch[256 + ((half ^ 1) * 4 + q) * 32 + lane];
      }
      const float inv = 1.f / sum;
      // ---- output ----
      mbar_wait(&bar[A_OFULL + bsel], ph);
      tc_fence_after();
      if (warp == 2 && lane == 0) FA_TRACE(it, 11);   // epilogue: output accumulator ready
      if (o_active) {
#pragma unroll 1
        for (int c = 0; c < ocols; c += 32) {
          uint32_t v[32];
          tmem_ld32(t_o + (uint32_t)(oc0 + c), v);
          const int hc = (c >> 5) & 1;                        // half of the 64-column staging box
          const int box = G == 2 ? (c >> 6) & 1 : 0;          // two groups: two boxes per warp, alternating
          if (hc == 0 && c > 0 && (G == 1 || c >= 128)) {     // reusing a box: its previous store must have read it
            if (lane == 0) bulk_wait_read0();
            __syncwarp();
          }
          const uint32_t sbox = stage + (uint32_t)box * 4096u;
#pragma unroll
          for (int t = 0; t < 4; ++t)
            sts128(sbox + (uint32_t)(lane * 128 + (((t + 4 * hc) ^ sw7) << 4)),
                   pack_bf16(__uint_as_float(v[8 * t]) * inv, __uint_as_float(v[8 * t + 1]) * inv),
                   pack_bf16(__uint_as_float(v[8 * t + 2]) * inv, __uint_as_float(v[8 * t + 3]) * inv),
                   pack_bf16(__uint_as_float(v[8 * t + 4]) * inv, __uint_as_float(v[8 * t + 5]) * inv),
                   pack_bf16(__uint_as_float(v[8 * t + 6]) * inv, __uint_as_float(v[8 * t + 7]) * inv));
          if (hc == 1 || c + 32 >= ocols) {
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              tma_store_3d(&tmO, sbox, h * p.dh + oc0 + (c & ~63), qt * 128 + q * 32, b);
              bulk_commit();
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar[A_OEMPTY + bsel]);
      if (warp == 2 && lane == 0) FA_TRACE(it, 12);   // epilogue: output handed to TMA
    }
    if (lane == 0) bulk_wait_read0();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

}  // namespace

bool tc_attn_fused_supported(int nq, int nkv, int dh) {
  if (!(nq >= 1 && nkv >= 1 && nkv <= 256 && (dh == 64 || dh == 128 || dh == 256))) return false;
  const int npad = (nkv + 63) / 64 * 64, dkb = dh / 64, nkb = npad / 64;
  const size_t bytes = (size_t)dkb * 16384 + (size_t)dkb * npad * 128 + (size_t)nkb * dkb * 8192 + (size_t)nkb * 16384 + 256 + 2048;
  return bytes <= 227 * 1024 && (size_t)nkb * 16384 >= 8 * 4096;   // the P buffer also hosts the output staging boxes
}

// q/k/v: bf16 views [B*nq | B*nkv, ld*] with head h at columns h*dh; out bf16 [B, nq, H*dh]
int tc_attn_fused(const __nv_bfloat16* q, int ldq, const __nv_bfloat16* k, int ldk, const __nv_bfloat16* v, int ldv, int B, int H,
                  int nq, int nkv, int dh, __nv_bfloat16* out, int ldo, cudaStream_t s, bool q_shared) {
  MOCHA_CHECK_ARG(tc_attn_fused_supported(nq, nkv, dh), "tc_attn_fused: unsupported geometry nq=%d nkv=%d dh=%d", nq, nkv, dh);
  MOCHA_CHECK_ARG(q && k && v && out && B > 0 && H > 0, "tc_attn_fused: null operand");
  MOCHA_CHECK_ARG(ldo == H * dh && (ldq % 8) == 0 && (ldk % 8) == 0 && (ldv % 8) == 0, "tc_attn_fused: bad leading dimensions");
  AttnParams p{};
  p.B = B; p.H = H; p.nq = nq; p.nkv = nkv; p.dh = dh;
  p.q_rows_b = q_shared ? 0 : nq;
  p.npad = (nkv + 63) / 64 * 64;
  p.nqt = ceil_div(nq, 128);
  p.units = B * H * p.nqt;
  p.scale_log2e = 1.4426950408889634f / sqrtf((float)dh);
  const int dkb = dh / 64, nkb = p.npad / 64;
  p.off_k = (uint32_t)dkb * 16384u;                                 // K inside a Q / K stage
  p.qk_stride = (p.off_k + (uint32_t)dkb * (uint32_t)p.npad * 128u + 1023u) & ~1023u;
  p.p_bytes = (uint32_t)nkb * 16384u;
  const uint32_t v_bytes = (uint32_t)nkb * (uint32_t)dkb * 8192u;
  // two-group mode: double-buffered scores / outputs in TMEM, two P buffers (each also hosts 4 warps x 2 staging boxes);
  // a second Q / K stage when it still fits
  const size_t fixed = 256 + 2048;
  p.groups = (2 * (p.npad + dh) <= 512 && p.p_bytes >= 32768u &&
              (size_t)p.qk_stride + v_bytes + 2 * (size_t)p.p_bytes + fixed <= 227 * 1024) ? 2 : 1;
  p.qk_stages = (p.groups == 2 && 2 * (size_t)p.qk_stride + v_bytes + 2 * (size_t)p.p_bytes + fixed <= 227 * 1024) ? 2 : 1;
  p.off_v = (uint32_t)p.qk_stages * p.qk_stride;
  p.off_p = p.off_v + v_bytes;
  p.off_bar = p.off_p + (uint32_t)p.groups * p.p_bytes;
  p.off_xch = p.off_bar + 256u;
  const size_t smem = (size_t)p.off_xch + 2048;
  MOCHA_CHECK_ARG(smem <= 227 * 1024, "tc_attn_fused: shared-memory plan of %zu B exceeds 227 KB", smem);
  const int inner = H * dh;
  CUtensorMap tmQ, tmK, tmV, tmO;
  MOCHA_TRY(tc_make_tmap(&tmQ, q, (unsigned long long)(q_shared ? 1 : B) * nq, (unsigned long long)inner, 128, (unsigned long long)ldq));
  MOCHA_TRY(tc_make_tmap(&tmK, k, (unsigned long long)B * nkv, (unsigned long long)inner, p.npad, (unsigned long long)ldk));
  MOCHA_TRY(tc_make_tmap(&tmV, v, (unsigned long long)B * nkv, (unsigned long long)inner, 64, (unsigned long long)ldv));
  MOCHA_TRY(tc_make_out_tmap(&tmO, out, (unsigned long long)ldo, (unsigned long long)nq, (unsigned long long)B,
                             (unsigned long long)ldo, false, 0, true));
  static size_t configured = 0;
  if (smem > configured) {
    MOCHA_CUDA(cudaFuncSetAttribute(attn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    configured = 227 * 1024;
  }
  const int grid = p.units < tc_num_sms() ? p.units : tc_num_sms();
  launch_k(attn_kernel, dim3((unsigned)grid), dim3(FA_THREADS), smem, s, tmQ, tmK, tmV, tmO, p);
  count_launch();
  MOCHA_LAUNCH_CHECK("attn_kernel");
  return MOCHA_OK;
}

}  // namespace mocha

#ifdef MOCHA_TRACE
extern "C" int mocha_debug_set_attn_trace(unsigned long long* buf) {
  return cudaMemcpyToSymbol(mocha::g_fa_trace, &buf, sizeof(buf)) == cudaSuccess ? 0 : 1;
}
#endif
