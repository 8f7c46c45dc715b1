// tcgen05 / TMEM / TMA GEMM family for sm_100a (see gemm_tc.cuh).
//
// Kernel anatomy (one persistent CTA per SM, 384 threads in three warpgroups; setmaxnreg moves registers from the
// producer group, 88 per thread, to the epilogue groups, 208 per thread, so the epilogue does not spill):
//   warp 0      TMA producer: cp.async.bulk.tensor 2D tiles (128B swizzle) into a STAGES-deep ring
//   warp 1      MMA issuer:   one elected thread issues tcgen05.mma.cta_group::1.kind::f16
//               (M=128, N=BN, K=16) x4 per 64-wide k-block; tcgen05.commit frees ring slots and
//               publishes finished accumulators; also owns tcgen05.alloc / dealloc
//   warps 2, 3  idle (they complete the producer warpgroup)
//   warps 4..11 epilogue: tcgen05.ld 32x32b (lane = output row) from one of two TMEM accumulator
//               buffers, so the epilogue of tile i overlaps the main loop of tile i+1
// Operands are K-major bf16: A tile 128 x 64, B tile BN x 64, both landing in the canonical
// SWIZZLE_128B layout the UMMA shared-memory descriptors describe (8-row groups 1024 B apart).
#include <cuda.h>

#include "gemm_tc.cuh"

#include <mutex>
#include <type_traits>
#include <vector>
#include "gemm_f32.cuh"
#include "ops.cuh"

namespace mocha {

namespace {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;  // 64 bf16 = 128 B = one swizzle atom row
constexpr int UMMA_K = 16;
// Warp roles. Ten warps put three warps on one scheduler partition (16 K registers each), which caps every thread at
// 168 registers and made the epilogue spill. Twelve warps in three warpgroups: warps 0-3 are the producer group (TMA
// warp, MMA warp, two idle warps) and shrink to TC_REGS_PRODUCER with setmaxnreg, warps 4-11 (the epilogue) grow to
// TC_REGS_EPI.
constexpr int TC_EPI_WARP0 = 4;
constexpr int TC_THREADS = TC_EPI_WARP0 * 32 + 8 * 32;
constexpr int TC_REGS_PRODUCER = 88, TC_REGS_EPI = 208;   // 4 x 88 + 8 x 208 = 2016 = the 12 x 168 registers per lane slot the launch allocates
constexpr int A_STAGE_BYTES = BLOCK_M * BLOCK_K * 2;

// ------------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Bounded wait: a protocol bug becomes a trap (reported as a CUDA error) instead of a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t ok = 0;
  long long t0 = 0;
  for (uint32_t it = 0;; ++it) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
    if (ok) return;
    if (it == 64) t0 = clock64();
    if (it > 64 && (it & 1023) == 0 && clock64() - t0 > 6000000000LL) {
      printf("mocha tc kernel: mbarrier wait timed out (block %d thread %d)\n", blockIdx.x, threadIdx.x);
      __trap();
    }
  }
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// L2 eviction-priority policies for TMA loads (createpolicy encodings)
constexpr uint64_t L2_EVICT_NORMAL = 0x1000000000000000ull;
constexpr uint64_t L2_EVICT_FIRST = 0x12F0000000000000ull;
constexpr uint64_t L2_EVICT_LAST = 0x14F0000000000000ull;
__device__ __forceinline__ void tma_load_2d_hint(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar, int c0, int c1,
                                                 uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_u32(smem_dst)), "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tmap) : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, bf16 inputs, fp32 accumulate
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// same with fp32 operands consumed as TF32 (K = 8 per instruction, 32 B per k-step like bf16's 16 x 2 B)
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// UMMA shared-memory descriptor, K-major operand in SWIZZLE_128B canonical layout:
//   start address >> 4 | LBO (ignored for swizzled K-major, 1) | SBO = 1024 B (8 rows x 128 B)
//   | version 1 (sm_100) | layout type 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// MN-major operand (rows of the tile are K, the MN dimension is contiguous), 128 B swizzle: 64-element
// MN atoms of [8 K-rows x 128 B]; SBO = 1024 B between 8-row K groups, LBO = bytes between MN atoms.
__device__ __forceinline__ uint64_t make_smem_desc_mn(uint32_t smem_addr, uint32_t atom_stride_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((atom_stride_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// kind::f16 instruction descriptor: D=f32, A=B=bf16, both K-major, N>>3 at [17,23), M>>4 at [24,29)
// fmt: 1 = BF16 (kind::f16), 2 = TF32 (kind::tf32)
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, uint32_t fmt = 1) {
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ------------------------------------------------------------------------------------------------
// work decomposition shared by both epilogues
// ------------------------------------------------------------------------------------------------
struct TcShape {
  int nb;                  // independent row groups ("images"); 1 for a plain GEMM
  int rows_out_per_b;      // output rows per image
  int tiles_m_per_b;       // ceil(rows_out_per_b / 128)
  long long src_rows_per_b;  // A rows per image in the (padded) source tensor
  int taps;                // temporal taps (1 for a plain GEMM)
  int kb_per_tap;          // k-blocks per tap
  int tap_row_stride;      // A row shift per tap
  int tiles_n;             // ceil(N / BN)
  int tiles_per_unit;      // consecutive n-tiles handled by one unit
  int units;               // tiles_m_total * splits
  int tiles_m_total;
  // batched-head mode (attention): image z = zb * H + zh selects operand windows and the output block
  int H;                   // 0 = plain mode
  long long a_rows_h;      // A row offset per head (rows per batch come from src_rows_per_b)
  int a_cols_h;            // A column offset per head
  long long b_rows_b, b_rows_h;  // B row offsets per batch / head
  int b_cols_h;            // B column offset per head
  long long c_img_b, c_img_h;    // output element offsets per batch / head
  // L2-aware unit order: m-tiles are walked in groups of group_m (0 = all) so that the group's A
  // rows stay L2-resident while every split streams its B rows past them
  int group_m;
  int splits;
  // B operand given MN-major: tmB describes [K rows, N cols] (N contiguous) and is loaded as 64 x 64
  // boxes (attention's P V product reads V in place instead of a transposed copy)
  int b_mn;
};

// n / d for 0 <= n < 2^22 and d >= 1 through a float reciprocal with an integer correction step: the tile
// bookkeeping of every role runs once per tile, and four dependent hardware-less integer divisions were
// ~770 cycles between two tiles of the epilogue warps
__device__ __forceinline__ int fast_div(int n, int d) {
  int q = __float2int_rz(__int2float_rn(n) * __frcp_rn(__int2float_rn(d)));
  int r = n - q * d;
  if (r < 0) { --q; r += d; }
  if (r >= d) ++q;
  return q;
}

// unit -> (m tile, n split). Within a group of group_m m-tiles the m index runs fastest, so CTAs that
// run concurrently share both the group's A tiles and the same few B ranges.
__device__ __forceinline__ void decode_unit(const TcShape& sh, int u, int& mt, int& split) {
  if (sh.group_m <= 0 || sh.group_m >= sh.tiles_m_total) {
    if (u < (1 << 22)) {
      split = fast_div(u, sh.tiles_m_total);
      mt = u - split * sh.tiles_m_total;
    } else {
      mt = u % sh.tiles_m_total;
      split = u / sh.tiles_m_total;
    }
    return;
  }
  const int per_group = sh.group_m * sh.splits;
  const int g = u / per_group;
  const int r = u - g * per_group;
  const int m0 = g * sh.group_m;
  const int gm = min(sh.group_m, sh.tiles_m_total - m0);  // the last group may be smaller
  // full groups come first, so r indexes into a gm x splits block only when the group is full;
  // for the last (short) group recompute from the units that remain
  if (gm == sh.group_m) {
    mt = m0 + r % gm;
    split = r / gm;
  } else {
    const int r2 = u - g * per_group;
    mt = m0 + r2 % gm;
    split = r2 / gm;
  }
}

// Per-warp epilogue context. Eight epilogue warps: warp w reads TMEM lane quarter (w & 3), i.e. a
// 32-row slab of the 128-row tile, and column half (w - 2) / 4 of the tile.
constexpr int EPI_WARPS = 8;
constexpr int EPI_LD = 36;  // floats per staged row: 16 B aligned, conflict-free for 128-bit accesses
struct EpiCtx {
  uint32_t stage;        // shared-space address of this warp's [32][EPI_LD] float staging buffer
  int lane;
  int half;              // column half handled by this warp
  long long slab_row0;   // output row of the slab's first row (global, or within the image in batched mode)
  int slab_rows;         // valid rows in the slab (0..32)
  long long c_off;       // element offset of the output block (batched-head mode), else 0
  uint32_t res_bar;      // shared-space address of this warp's residual-prefetch mbarrier
  uint32_t bias_smem;    // shared-space address of the CTA's staged column bias (TMA epilogues)
  int etid;              // thread index among the epilogue warps (0..255)
  int col_off;           // column offset of the output block inside its TMA map (batched-head PV output)
  int z;                 // image index b of the tile (batched-head mode: z = zb * H + zh)
  int img;               // batch image of the tile: third TMA-store coordinate
  int row0_in_img;       // first row of the slab inside its image: second TMA-store coordinate
};

// TMA store of one [32 rows x 32 cols] box from shared memory (bulk async-group of the issuing thread)
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* tm, uint32_t smem_addr, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(tm),
               "r"(smem_addr), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t smem_dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(smem_dst),
      "l"(tm), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until every committed bulk store of this thread has finished READING shared memory
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// ... until at most ONE committed bulk store of this thread is still reading shared memory (double-buffered staging)
__device__ __forceinline__ void bulk_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void sts64(uint32_t addr, uint32_t a, uint32_t b) {
  asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(a), "r"(b) : "memory");
}
__device__ __forceinline__ void sts128f(uint32_t addr, const float4& v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}

// GELU(x) = x/2 (1 + erf(x/sqrt 2)) for the bf16 tensor-core path: erf through Abramowitz & Stegun 7.1.28,
// erf(t) = 1 - (1 + a1 t + ... + a6 t^6)^-16 for t >= 0 (|error| <= 3e-7, two orders below bf16's half ulp),
// ~16 instructions and one MUFU instead of erff's ~28 on the issue-bound epilogue. The fp32 path keeps erff.
__device__ __forceinline__ float gelu_fast(float x) {
  const float t = fabsf(x) * 0.70710678118654752f;
  float p = fmaf(0.0000430638f, t, 0.0002765672f);
  p = fmaf(p, t, 0.0001520143f);
  p = fmaf(p, t, 0.0092705272f);
  p = fmaf(p, t, 0.0422820123f);
  p = fmaf(p, t, 0.0705230784f);
  p = fmaf(p, t, 1.0f);
  p *= p; p *= p; p *= p; p *= p;                 // ^16 (overflows to +inf for large |x|: erf -> 1)
  float rp;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rp) : "f"(p));   // one MUFU (rcp.rn is a ~10-instruction sequence)
  const float e = 1.0f - rp;                      // erf(|x| / sqrt 2)
  return 0.5f * x * (1.0f + copysignf(e, x));
}

template <int ACT>
__device__ __forceinline__ float act_fn(float x) {
  if (ACT == ACT_RELU) return fmaxf(x, 0.f);
  if (ACT == ACT_GELU) return gelu_fast(x);
  if (ACT == ACT_LRELU) return lrelu02(x);
  return x;
}

#ifdef MOCHA_TRACE
// Debug build only (python -m mocha_sigasia2023_b200.build --trace): per-CTA clock64 time line of the
// pipeline roles, read back by tools/tc_trace.py. 32 u64 slots per CTA.
__device__ unsigned long long* g_tc_trace = nullptr;
__device__ int g_tc_dbg_mode = 0;  // 1: no TMA loads (pure MMA rate), 2: no MMAs (pure fill rate), 3: no epilogue work
__device__ __forceinline__ unsigned long long gtimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define TC_TRACE(slot, val)                                                         \
  do {                                                                              \
    const unsigned long long tv_ = (val);                                           \
    if (trace_buf && (slot) < 32) trace_buf[(size_t)blockIdx.x * 32 + (slot)] = tv_; \
  } while (0)
__device__ unsigned long long g_epi_dbg[16];
#define EPI_DBG(i) do { if (blockIdx.x == 0 && threadIdx.x == 64) g_epi_dbg[i] = (unsigned long long)clock64(); } while (0)
#else
#define EPI_DBG(i) do { } while (0)
#define TC_TRACE(slot, val) do { } while (0)
#endif

struct LinearEpiData {
  float* C;
  int ldc;
  int N;
  const float* bias;
  int bias_period;
  const float* res;
  int act;
  __nv_bfloat16* C16;   // optional bf16 copy of the output (operand of the next tensor-core layer); C may be null
  int c16_lrelu;        // store LeakyReLU(0.2)(x) in the bf16 copy (pre-activation consumers)
  // TMA-store path (plain / tconv mode with 16 B-aligned outputs): 3-D maps {cols, rows per image, images}
  int tma;      // 1: TMA-store path; 2: additionally the residual is TMA-prefetched (needs bias_period == 0)
  CUtensorMap tmC, tmC16, tmR;
  // optional per-row scale (TMA-store path only): out = act(acc * row_scale[z * rs_rows + row] + bias) ...
  // (attention: the softmax denominator is applied to P V here, flash-attention style)
  const float* row_scale;
  int rs_rows;
  // bf16-only outputs with N % 64 == 0 and tiles >= 128 wide: two 32-column chunks share one 64-column
  // (128 B rows, 128 B-swizzled) TMA box, halving the fence / issue / wait overhead per byte
  int c16_wide;
  CUtensorMap tmC16w;
};
using LinearEpi = LinearEpiData;

// MODE 0: LSU epilogue; 1: TMA stores; 2: TMA stores + TMA-prefetched residual; 4: MODE 1 with TWO staging boxes per
// warp - a TMA store needs ~1000 cycles to finish reading its box, and with one box every chunk (64 bf16 / 32 fp32
// columns) stalled on the previous chunk's store; with two the warp only waits for the store before last.
// One kernel instantiation per mode keeps each epilogue's register footprint and code small.
template <int MODE>
struct LinearEpiT : LinearEpiData {
  struct State {
    uint32_t rphase;  // parity of the residual-prefetch barrier
    int col_begin;    // first column of this warp's share of the current tile
    float rs;         // this lane's row scale for the current tile
    uint32_t par;     // MODE 4: which of the two staging boxes the next chunk fills
  };
  static constexpr bool kM1 = MODE == 1 || MODE == 4;   // single-output TMA-store epilogue
  static constexpr bool kDouble = MODE == 4;
  // per warp: 4 KB fp32 box [32][128 B] (128 B-swizzled, 1 KB aligned) + 2 KB bf16 box [32][64 B]
  // (64 B-swizzled) + 4 KB residual box (128 B-swizzled); the LSU path uses a [32][EPI_LD] float
  // transposition buffer
  // MODE 1 writes one output per launch (the host falls back to MODE 0 otherwise), so its bf16 box
  // aliases the fp32 box and a fourth operand stage fits beside a 128 x 256 tile's staging
  // The per-warp stride is a multiple of 1 KB (128 B-swizzled boxes must be 1 KB aligned); the whole column
  // bias (N <= 2048) is staged once per CTA in an 8 KB area behind the warps' buffers.
  // MODE 3 = MODE 2 without a bf16 output (no bf16 box): 8 KB per warp leaves room for 128 x 256 tiles
  static constexpr bool kRes = MODE == 2 || MODE == 3;
  static constexpr int kResOff = MODE == 3 ? 4096 : 6144;
  static constexpr int kWarpStageBytes = MODE == 2 ? 10240 : MODE == 3 ? 8192 : MODE == 1 ? 4096 : MODE == 4 ? 8192 : 5120;
  static_assert(kWarpStageBytes % 1024 == 0, "swizzled TMA boxes need 1 KB alignment");
  static constexpr int kBiasBytes = MODE == 0 ? 0 : 8192;
  static constexpr int kStageBytes = EPI_WARPS * kWarpStageBytes + kBiasBytes;
  static constexpr uint64_t kHintA = 0, kHintB = 0;                // default L2 policy
  static constexpr bool kTf32 = false;
  static constexpr bool kWholeTile = false;
  __device__ __forceinline__ void unit_begin(State&) const {}
  __device__ __forceinline__ void kernel_begin(State& st, const EpiCtx& e) const {
    st.rphase = 0; st.col_begin = 0; st.rs = 1.f; st.par = 0;
    if (MODE != 0) {
      // the epilogue's only global loads that are not TMA: the column bias, once per CTA, while the first
      // tile's main loop runs (per-chunk or per-tile loads see >1000-cycle latencies under store traffic)
      if (bias && bias_period == 0)
        for (int c = 4 * e.etid; c < N; c += 4 * EPI_WARPS * 32)
          sts128f(e.bias_smem + 4u * c, __ldg(reinterpret_cast<const float4*>(bias + c)));
      asm volatile("bar.sync 1, 256;" ::: "memory");   // the eight epilogue warps only
    }
  }
  // issue the TMA prefetch of a chunk's residual box (does not depend on the accumulator)
  __device__ __forceinline__ void prefetch_res(const EpiCtx& e, int col0) const {
    if (kRes && col0 >= 0 && col0 < N && e.slab_rows > 0 && e.lane == 0) {
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(e.res_bar), "r"(4096u) : "memory");
      tma_load_3d(e.stage + kResOff, &tmR, e.res_bar, col0, e.row0_in_img, e.img);
    }
  }
  // Global loads issued from the epilogue see multi-thousand-cycle latencies while every SM is streaming
  // stores, so nothing on a chunk's critical path may come from global memory: the warp's slice of the
  // column bias is staged in shared memory once per tile BEFORE the accumulator is waited for (the load
  // overlaps the tile's main loop), and in MODE 2 the residual box is TMA-prefetched one chunk ahead.
  __device__ __forceinline__ void tile_begin(State& st, const EpiCtx& e, int col_begin, int ncols) const {
    st.col_begin = col_begin;
    if (kM1 && row_scale)
      st.rs = e.lane < e.slab_rows ? __ldg(row_scale + (long long)e.z * rs_rows + e.row0_in_img + e.lane) : 0.f;
    (void)ncols;
    prefetch_res(e, col_begin);
  }
  __device__ __forceinline__ void prefetch_chunk(State&, const EpiCtx& e, int col0) const { prefetch_res(e, col0); }

  // LSU epilogue (batched-head attention outputs and unaligned tensors), second half of the transposed
  // path: 8 passes of 4 rows x 32 columns, 8 lanes x float4 = one 128 B line per row, as a fixed
  // sequence of unrolled phases - residual loads, staged reads, bias, activation, stores - with one
  // base address and constant row strides. Ragged / unaligned chunks take the scalar path below.
  template <int ACT>
  __device__ __forceinline__ void drain_fast(const EpiCtx& e, int col0) const {
    const int rr = e.lane >> 3, cc = (e.lane & 7) * 4;
    const int c = col0 + cc;
    const long long step = 4LL * ldc;
    const uint32_t sbase0 = e.stage + (uint32_t)((rr * EPI_LD + cc) * 4);
    float4 bc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (bias && bias_period == 0) bc = __ldg(reinterpret_cast<const float4*>(bias + c));
    // two half-chunks of 4 passes (16 rows): written for the 168-register cap of the ten-warp layout, kept as is
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const long long base = e.c_off + (e.slab_row0 + rr + 16 * h) * (long long)ldc + c;
      const int nrows = e.slab_rows - rr - 16 * h;  // pass `it` is live iff 4*it < nrows
      const uint32_t sbase = sbase0 + (uint32_t)(h * 16 * EPI_LD * 4);
      float4 rv[4];
      if (res) {
        const float* rp = res + base;
#pragma unroll
        for (int it = 0; it < 4; ++it)
          if (4 * it < nrows) rv[it] = __ldg(reinterpret_cast<const float4*>(rp + it * step));
      }
      float4 o[4];
      if (h == 0) EPI_DBG(2);
#pragma unroll
      for (int it = 0; it < 4; ++it) o[it] = lds128(sbase + (uint32_t)(it * 4 * EPI_LD * 4));
      if (h == 0) EPI_DBG(3);
      if (bias) {
        if (bias_period == 0) {
#pragma unroll
          for (int it = 0; it < 4; ++it) { o[it].x += bc.x; o[it].y += bc.y; o[it].z += bc.z; o[it].w += bc.w; }
        } else {
          const unsigned p = (unsigned)bias_period;
          unsigned m = (unsigned)((unsigned long long)(e.slab_row0 + rr + 16 * h) % p);
          float4 bv[4];
#pragma unroll
          for (int it = 0; it < 4; ++it) {
            bv[it] = __ldg(reinterpret_cast<const float4*>(bias + (size_t)m * N + c));
            m += 4;
            m = m >= p ? m - p : m;
            m = m >= p ? m - p : m;
          }
#pragma unroll
          for (int it = 0; it < 4; ++it) { o[it].x += bv[it].x; o[it].y += bv[it].y; o[it].z += bv[it].z; o[it].w += bv[it].w; }
        }
      }
      if (ACT != ACT_NONE) {
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          o[it].x = act_fn<ACT>(o[it].x); o[it].y = act_fn<ACT>(o[it].y);
          o[it].z = act_fn<ACT>(o[it].z); o[it].w = act_fn<ACT>(o[it].w);
        }
      }
      if (res) {
#pragma unroll
        for (int it = 0; it < 4; ++it)
          if (4 * it < nrows) { o[it].x += rv[it].x; o[it].y += rv[it].y; o[it].z += rv[it].z; o[it].w += rv[it].w; }
      }
      if (h == 0) EPI_DBG(4);
      if (C) {
        float* cp = C + base;
#pragma unroll
        for (int it = 0; it < 4; ++it)
          if (4 * it < nrows) *reinterpret_cast<float4*>(cp + it * step) = o[it];
      }
      if (h == 0) EPI_DBG(5);
      if (C16) {
        if (c16_lrelu) {
#pragma unroll
          for (int it = 0; it < 4; ++it) {
            o[it].x = lrelu02(o[it].x); o[it].y = lrelu02(o[it].y); o[it].z = lrelu02(o[it].z); o[it].w = lrelu02(o[it].w);
          }
        }
        __nv_bfloat16* cp = C16 + base;
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          __nv_bfloat162 lo = __floats2bfloat162_rn(o[it].x, o[it].y), hi = __floats2bfloat162_rn(o[it].z, o[it].w);
          uint2 pk;
          pk.x = *reinterpret_cast<uint32_t*>(&lo);
          pk.y = *reinterpret_cast<uint32_t*>(&hi);
          if (4 * it < nrows) *reinterpret_cast<uint2*>(cp + it * step) = pk;
        }
      }
    }
  }

  // TMA-store epilogue. The SM -> L2 write path is 32 B/clk/SM whether driven by STG or by the TMA
  // engine (tools/probes/store_probe.cu), and a K=256 tile's MMAs take no longer than its stores, so
  // the stores must never wait for the warps: each warp stages a 32x32 box in shared memory, one lane
  // hands it to the TMA engine and the warp moves on to the next chunk while the engine drains it.
  //   pass 1  lane = row: accumulator row -> 128 B-swizzled box (16 B chunk j of row r at j ^ (r & 7))
  //   pass 2  8 lanes x float4 = one row: coalesced bias / residual loads, activation, in-place write
  //           back (+ bf16 box), then fence.proxy.async and one elected TMA store per output.
  template <int ACT>
  __device__ __forceinline__ void drain_tma(State& st, const EpiCtx& e, int col0, int next_col0, const uint32_t (&v)[32]) const {
    EPI_DBG(14);
    if (bias_period == 0 || !bias) {
      // lane = row all the way (no transposed pass): column bias broadcast from the CTA's shared-memory copy,
      // row scale is one scalar per lane, results go straight into the TMA boxes
      float f[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
      if (row_scale) {
        const float rs = st.rs;
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] *= rs;
      }
      if (bias) {
        const uint32_t bs = e.bias_smem + (uint32_t)(col0 * 4);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 b4 = lds128(bs + 16u * j);   // same address in every lane: broadcast
          f[4 * j] += b4.x; f[4 * j + 1] += b4.y; f[4 * j + 2] += b4.z; f[4 * j + 3] += b4.w;
        }
      }
      if (ACT != ACT_NONE) {
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] = act_fn<ACT>(f[j]);
      }
      EPI_DBG(8);
      const uint32_t sbuf = e.stage + (kDouble ? st.par * 4096u : 0u);   // this chunk's staging box
      if (!(c16_wide && !C && (((col0 - st.col_begin) >> 5) & 1))) {
        // the store that last used this box has finished reading it (double-buffered: the store before last)
        if (e.lane == 0) { if (kDouble) bulk_wait_read1(); else bulk_wait_read0(); }
        __syncwarp();
      }
      EPI_DBG(9);
      if (C) {
        const int sw = e.lane & 7;
#pragma unroll
        for (int j = 0; j < 8; ++j)
          sts128(sbuf + (uint32_t)(e.lane * 128 + ((j ^ sw) << 4)), __float_as_uint(f[4 * j]), __float_as_uint(f[4 * j + 1]),
                 __float_as_uint(f[4 * j + 2]), __float_as_uint(f[4 * j + 3]));
      } else if (c16_wide) {
        const int hcol = ((col0 - st.col_begin) >> 5) & 1;   // which half of the 64-column box
        const int sw = e.lane & 7;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint32_t pk[4];
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            float a = f[8 * j + 2 * t], b = f[8 * j + 2 * t + 1];
            if (c16_lrelu) { a = lrelu02(a); b = lrelu02(b); }
            __nv_bfloat162 h2 = __floats2bfloat162_rn(a, b);
            pk[t] = *reinterpret_cast<uint32_t*>(&h2);
          }
          sts128(sbuf + (uint32_t)(e.lane * 128 + (((j + 4 * hcol) ^ sw) << 4)), pk[0], pk[1], pk[2], pk[3]);
        }
        if (hcol == 0) return;   // the box goes out with its second half
        fence_async_smem();
        __syncwarp();
        if (e.lane == 0) {
          tma_store_3d(&tmC16w, sbuf, col0 - 32 + e.col_off, e.row0_in_img, e.img);
          bulk_commit();
        }
        if (kDouble) st.par ^= 1u;
        return;
      } else {
        const int sw16 = (e.lane >> 1) & 3;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint32_t pk[4];
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            float a = f[8 * j + 2 * t], b = f[8 * j + 2 * t + 1];
            if (c16_lrelu) { a = lrelu02(a); b = lrelu02(b); }
            __nv_bfloat162 h2 = __floats2bfloat162_rn(a, b);
            pk[t] = *reinterpret_cast<uint32_t*>(&h2);
          }
          sts128(sbuf + (uint32_t)(e.lane * 64 + ((j ^ sw16) << 4)), pk[0], pk[1], pk[2], pk[3]);
        }
      }
      EPI_DBG(11);
      fence_async_smem();
      __syncwarp();
      EPI_DBG(12);
      if (e.lane == 0) {
        if (C) tma_store_3d(&tmC, sbuf, col0 + e.col_off, e.row0_in_img, e.img);
        else tma_store_3d(&tmC16, sbuf, col0 + e.col_off, e.row0_in_img, e.img);
        bulk_commit();
      }
      if (kDouble) st.par ^= 1u;
      EPI_DBG(13);
      return;
    }
    // bf16 box aliases the fp32 box: rows 16h..16h+15 of the bf16 box cover fp32 rows 8h..8h+7, which
    // the warp has already read when half h is written back (warp-synchronous, program order)
    const uint32_t buf32 = e.stage, buf16 = e.stage;
    EPI_DBG(8);
    if (e.lane == 0) bulk_wait_read0();  // the previous chunk's stores have left the staging buffers
    __syncwarp();
    EPI_DBG(9);
#pragma unroll
    for (int j = 0; j < 8; ++j)
      sts128(buf32 + (uint32_t)(e.lane * 128 + ((j ^ (e.lane & 7)) << 4)), v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    __syncwarp();
    EPI_DBG(10);
    const int rr = e.lane >> 3, cq = e.lane & 7;
    const int c = col0 + cq * 4;
    const bool col_ok = c < N;  // N % 4 == 0 on this path
    if (bias || res || ACT != ACT_NONE || C16 || row_scale) {
      const long long step = 4LL * ldc;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const long long base = e.c_off + (e.slab_row0 + rr + 16 * h) * (long long)ldc + c;
        const int nrows = col_ok ? e.slab_rows - rr - 16 * h : 0;  // pass `it` is live iff 4*it < nrows
        float4 rv[4];
        if (res) {
          const float* rp = res + base;
#pragma unroll
          for (int it = 0; it < 4; ++it)
            if (4 * it < nrows) rv[it] = __ldg(reinterpret_cast<const float4*>(rp + it * step));
        }
        float4 o[4];
        uint32_t addr[4];
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          const int r = 16 * h + 4 * it + rr;
          addr[it] = buf32 + (uint32_t)(r * 128 + ((cq ^ (r & 7)) << 4));
          o[it] = lds128(addr[it]);
        }
        if (row_scale) {
          const float* rsp = row_scale + (long long)e.z * rs_rows + e.row0_in_img + 16 * h + rr;
#pragma unroll
          for (int it = 0; it < 4; ++it) {
            const float f = 4 * it < nrows ? __ldg(rsp + 4 * it) : 0.f;
            o[it].x *= f; o[it].y *= f; o[it].z *= f; o[it].w *= f;
          }
        }
        if (bias) {
          {
            const unsigned p = (unsigned)bias_period;   // column biases take the single-pass path above
            unsigned m = (unsigned)((unsigned long long)(e.slab_row0 + rr + 16 * h) % p);
            float4 bv[4];
#pragma unroll
            for (int it = 0; it < 4; ++it) {
              bv[it] = make_float4(0.f, 0.f, 0.f, 0.f);
              if (4 * it < nrows) bv[it] = __ldg(reinterpret_cast<const float4*>(bias + (size_t)m * N + c));
              m += 4;
              m = m >= p ? m - p : m;
              m = m >= p ? m - p : m;
            }
#pragma unroll
            for (int it = 0; it < 4; ++it) { o[it].x += bv[it].x; o[it].y += bv[it].y; o[it].z += bv[it].z; o[it].w += bv[it].w; }
          }
        }
        if (ACT != ACT_NONE) {
#pragma unroll
          for (int it = 0; it < 4; ++it) {
            o[it].x = act_fn<ACT>(o[it].x); o[it].y = act_fn<ACT>(o[it].y);
            o[it].z = act_fn<ACT>(o[it].z); o[it].w = act_fn<ACT>(o[it].w);
          }
        }
        if (res) {
#pragma unroll
          for (int it = 0; it < 4; ++it)
            if (4 * it < nrows) { o[it].x += rv[it].x; o[it].y += rv[it].y; o[it].z += rv[it].z; o[it].w += rv[it].w; }
        }
        if (C) {
#pragma unroll
          for (int it = 0; it < 4; ++it) sts128f(addr[it], o[it]);
        }
        if (C16) {
          if (c16_lrelu) {
#pragma unroll
            for (int it = 0; it < 4; ++it) {
              o[it].x = lrelu02(o[it].x); o[it].y = lrelu02(o[it].y); o[it].z = lrelu02(o[it].z); o[it].w = lrelu02(o[it].w);
            }
          }
#pragma unroll
          for (int it = 0; it < 4; ++it) {
            __nv_bfloat162 lo = __floats2bfloat162_rn(o[it].x, o[it].y), hi = __floats2bfloat162_rn(o[it].z, o[it].w);
            const int r = 16 * h + 4 * it + rr;  // 64 B-swizzled box: 16 B chunk k of row r at k ^ ((r >> 1) & 3)
            sts64(buf16 + (uint32_t)(r * 64 + (((cq >> 1) ^ ((r >> 1) & 3)) << 4) + (cq & 1) * 8),
                  *reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
          }
        }
      }
    }
    EPI_DBG(11);
    fence_async_smem();
    __syncwarp();
    EPI_DBG(12);
    if (e.lane == 0) {
      // rows past the image and columns past the tensor are clipped by the tensor map
      if (C) tma_store_3d(&tmC, buf32, col0 + e.col_off, e.row0_in_img, e.img);
      if (C16) tma_store_3d(&tmC16, buf16, col0 + e.col_off, e.row0_in_img, e.img);
      bulk_commit();
    }
    EPI_DBG(13);
  }

  // Residual GEMMs (x + f(x) feeding both an fp32 stream and a bf16 operand): the residual box is
  // TMA-prefetched one chunk ahead into a 128 B-swizzled buffer, so everything stays in the lane = row
  // layout of tcgen05.ld: v = act(v + bias) + res, fp32 box and 64 B-swizzled bf16 box, TMA stores.
  template <int ACT>
  __device__ __forceinline__ void drain_tma_res(State& st, const EpiCtx& e, int col0, int next_col0, uint32_t (&v)[32]) const {
    const uint32_t buf32 = e.stage, buf16 = e.stage + 4096, bufr = e.stage + kResOff;   // MODE 3 never has C16
    const int sw = e.lane & 7;
    if (bias) {
      const uint32_t bs = e.bias_smem + (uint32_t)(col0 * 4);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 b4 = lds128(bs + 16u * j);   // same address in every lane: broadcast
        v[4 * j] = __float_as_uint(__uint_as_float(v[4 * j]) + b4.x);
        v[4 * j + 1] = __float_as_uint(__uint_as_float(v[4 * j + 1]) + b4.y);
        v[4 * j + 2] = __float_as_uint(__uint_as_float(v[4 * j + 2]) + b4.z);
        v[4 * j + 3] = __float_as_uint(__uint_as_float(v[4 * j + 3]) + b4.w);
      }
    }
    if (ACT != ACT_NONE) {
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(act_fn<ACT>(__uint_as_float(v[j])));
    }
    // residual box landed? (rows / columns past the tensor are zero-filled by the TMA load)
    {
      uint32_t done = 0;
      while (!done) {
        asm volatile(
            "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.b32 %0, 1, 0, p;\n}\n"
            : "=r"(done)
            : "r"(e.res_bar), "r"(st.rphase)
            : "memory");
      }
      st.rphase ^= 1;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 r4 = lds128(bufr + (uint32_t)(e.lane * 128 + ((j ^ sw) << 4)));
      v[4 * j] = __float_as_uint(__uint_as_float(v[4 * j]) + r4.x);
      v[4 * j + 1] = __float_as_uint(__uint_as_float(v[4 * j + 1]) + r4.y);
      v[4 * j + 2] = __float_as_uint(__uint_as_float(v[4 * j + 2]) + r4.z);
      v[4 * j + 3] = __float_as_uint(__uint_as_float(v[4 * j + 3]) + r4.w);
    }
    __syncwarp();                  // every lane has read the residual box: refill it for the next chunk
    prefetch_chunk(st, e, next_col0);
    if (e.lane == 0) bulk_wait_read0();  // the previous chunk's stores have left the staging buffers
    __syncwarp();
    if (C) {
#pragma unroll
      for (int j = 0; j < 8; ++j)
        sts128(buf32 + (uint32_t)(e.lane * 128 + ((j ^ sw) << 4)), v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    }
    if (C16) {
      const int sw16 = (e.lane >> 1) & 3;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint32_t pk[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          float a = __uint_as_float(v[8 * j + 2 * t]), b = __uint_as_float(v[8 * j + 2 * t + 1]);
          if (c16_lrelu) { a = lrelu02(a); b = lrelu02(b); }
          __nv_bfloat162 h2 = __floats2bfloat162_rn(a, b);
          pk[t] = *reinterpret_cast<uint32_t*>(&h2);
        }
        sts128(buf16 + (uint32_t)(e.lane * 64 + ((j ^ sw16) << 4)), pk[0], pk[1], pk[2], pk[3]);
      }
    }
    fence_async_smem();
    __syncwarp();
    if (e.lane == 0) {
      if (C) tma_store_3d(&tmC, buf32, col0 + e.col_off, e.row0_in_img, e.img);
      if (C16) tma_store_3d(&tmC16, buf16, col0 + e.col_off, e.row0_in_img, e.img);
      bulk_commit();
    }
  }

  // scalar path for ragged / unaligned chunks (attention score tiles, N not a multiple of 4)
  __device__ __forceinline__ void drain_slow(const EpiCtx& e, int col0) const {
    const int rr = e.lane >> 3, cc = (e.lane & 7) * 4;
    const int c = col0 + cc;
    if (c >= N) return;
#pragma unroll 1
    for (int it = 0; it < 8; ++it) {
      const int r = it * 4 + rr;
      if (r >= e.slab_rows) break;
      const long long grow = e.slab_row0 + r;
      const float4 x4 = lds128(e.stage + (uint32_t)((r * EPI_LD + cc) * 4));
      const float xs[4] = {x4.x, x4.y, x4.z, x4.w};
      const float* bp = !bias ? nullptr : bias_period > 0 ? bias + (size_t)((unsigned long long)grow % (unsigned)bias_period) * N : bias;
      const long long o_ = e.c_off + grow * (long long)ldc;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (c + k >= N) break;
        float x = xs[k];
        if (bp) x += __ldg(bp + c + k);
        x = act == ACT_RELU ? fmaxf(x, 0.f) : act == ACT_GELU ? gelu_erf(x) : act == ACT_LRELU ? lrelu02(x) : x;
        if (res) x += __ldg(res + o_ + c + k);
        if (C) C[o_ + c + k] = x;
        if (C16) C16[o_ + c + k] = __float2bfloat16_rn(c16_lrelu ? lrelu02(x) : x);
      }
    }
  }

  // Warp-collective: the accumulator slab (lane = row, 32 columns in registers) is transposed through
  // shared memory so that bias / residual loads and the stores are row-contiguous and coalesced.
  __device__ __forceinline__ void chunk(State& st, const EpiCtx& e, long long, bool, int col0, uint32_t (&v)[32],
                                        int next_col0) const {
    if (col0 >= N) return;
    if constexpr (kRes) {
      if (e.slab_rows <= 0) return;
      switch (act) {
        case ACT_RELU: drain_tma_res<ACT_RELU>(st, e, col0, next_col0, v); break;
        case ACT_GELU: drain_tma_res<ACT_GELU>(st, e, col0, next_col0, v); break;
        case ACT_LRELU: drain_tma_res<ACT_LRELU>(st, e, col0, next_col0, v); break;
        default: drain_tma_res<ACT_NONE>(st, e, col0, next_col0, v); break;
      }
    } else if constexpr (kM1) {
      if (e.slab_rows <= 0) return;
      switch (act) {
        case ACT_RELU: drain_tma<ACT_RELU>(st, e, col0, next_col0, v); break;
        case ACT_GELU: drain_tma<ACT_GELU>(st, e, col0, next_col0, v); break;
        case ACT_LRELU: drain_tma<ACT_LRELU>(st, e, col0, next_col0, v); break;
        default: drain_tma<ACT_NONE>(st, e, col0, next_col0, v); break;
      }
    } else {
    EPI_DBG(0);
#pragma unroll
    for (int j = 0; j < 32; j += 4)
      sts128(e.stage + (uint32_t)((e.lane * EPI_LD + j) * 4), v[j], v[j + 1], v[j + 2], v[j + 3]);
    __syncwarp();
    EPI_DBG(1);
    const bool fast = col0 + 32 <= N && ((ldc | N) & 3) == 0 && (e.c_off & 3) == 0 &&
                      (((reinterpret_cast<uintptr_t>(C) | reinterpret_cast<uintptr_t>(res) | reinterpret_cast<uintptr_t>(bias)) & 15) == 0) &&
                      ((reinterpret_cast<uintptr_t>(C16) & 7) == 0);
    if (fast) {
      switch (act) {
        case ACT_RELU: drain_fast<ACT_RELU>(e, col0); break;
        case ACT_GELU: drain_fast<ACT_GELU>(e, col0); break;
        case ACT_LRELU: drain_fast<ACT_LRELU>(e, col0); break;
        default: drain_fast<ACT_NONE>(e, col0); break;
      }
    } else {
      drain_slow(e, col0);
    }
    EPI_DBG(6);
    __syncwarp();
    EPI_DBG(7);
    }
  }
  __device__ __forceinline__ void unit_end(State&, const EpiCtx&, long long, bool, int) const {}
  // staging buffers must outlive the stores that read them: one wait when the CTA is done, not one per
  // tile (a store needs ~1000 cycles to leave shared memory; every chunk already waits before re-filling)
  __device__ __forceinline__ void kernel_end(const EpiCtx& e) const {
    if (MODE != 0 && e.lane == 0) bulk_wait_read0();
  }
};

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// Attention scores with the softmax fused into the epilogue: one tile holds every key of its 128
// query rows (nkv <= BN), so the warp that owns a 32-row TMEM lane quarter makes three passes over
// the accumulator - row max, then exp - without leaving TMEM, and hands the unnormalised bf16
// probabilities P[z, row, 0:ldp] (zero beyond nkv) to the TMA engine; the reciprocal row sums are
// applied by the P V GEMM's epilogue (flash-attention style). Replaces the fp32 score
// round trip through HBM and the stand-alone softmax launch.
struct SoftmaxEpi {
  float scale_log2e;  // log2(e) / sqrt(dh)
  int nkv;
  int ldp;
  int nq;
  float* inv_sum;     // [Z, nq] reciprocal softmax denominators, applied by the P V epilogue
  CUtensorMap tmP;    // {ldp, nq, Z} bf16, 64 B-swizzled 32 x 32 boxes
  struct State {};
  static constexpr int kWarpStageBytes = 2048;
  static constexpr int kStageBytes = EPI_WARPS * kWarpStageBytes;
  static constexpr uint64_t kHintA = 0, kHintB = 0;
  static constexpr bool kTf32 = false;
  static constexpr bool kWholeTile = true;
  __device__ __forceinline__ void unit_begin(State&) const {}
  __device__ __forceinline__ void kernel_begin(State&, const EpiCtx&) const {}
  __device__ __forceinline__ void tile_begin(State&, const EpiCtx&, int, int) const {}
  __device__ __forceinline__ void unit_end(State&, const EpiCtx&, long long, bool, int) const {}
  __device__ __forceinline__ void kernel_end(const EpiCtx& e) const {
    if (e.lane == 0) bulk_wait_read0();
  }
  __device__ __forceinline__ void tile(State&, const EpiCtx& e, uint32_t taddr, int acc_stage) const {
    // one warp per lane quarter owns whole rows of a tile; the two warps of a quarter alternate tiles
    // (accumulator stage 0 / 1), so two tiles' softmax passes run concurrently
    if (e.half != acc_stage || e.slab_rows <= 0) return;
    const int nch = (nkv + 31) >> 5;
    float m = -INFINITY;
#pragma unroll 1
    for (int ch = 0; ch < nch; ++ch) {
      uint32_t v[32];
      tmem_ld32(taddr + (uint32_t)(ch * 32), v);
      if (ch * 32 + 32 <= nkv) {
#pragma unroll
        for (int j = 0; j < 32; ++j) m = fmaxf(m, __uint_as_float(v[j]));
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (ch * 32 + j < nkv) m = fmaxf(m, __uint_as_float(v[j]));
      }
    }
    const float ms = m * scale_log2e;
    float sum = 0.f;
    const uint32_t buf16 = e.stage;
    const int sw16 = (e.lane >> 1) & 3;
    const int nbox = (ldp + 31) >> 5;
    // one exp per score: unnormalised probabilities go out as bf16, the row sums go to the P V epilogue
#pragma unroll 1
    for (int ch = 0; ch < nbox; ++ch) {
      uint32_t v[32];
      tmem_ld32(taddr + (uint32_t)(ch * 32), v);
      float ev[32];
      if (ch * 32 + 32 <= nkv) {
#pragma unroll
        for (int j = 0; j < 32; ++j) ev[j] = fast_exp2(fmaf(__uint_as_float(v[j]), scale_log2e, -ms));
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          ev[j] = ch * 32 + j < nkv ? fast_exp2(fmaf(__uint_as_float(v[j]), scale_log2e, -ms)) : 0.f;
      }
      if (e.lane == 0) bulk_wait_read0();
      __syncwarp();
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint32_t pk[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          __nv_bfloat162 h2 = __floats2bfloat162_rn(ev[8 * j + 2 * t], ev[8 * j + 2 * t + 1]);
          // the denominator sums what the P V GEMM will actually multiply
          sum += __low2float(h2) + __high2float(h2);
          pk[t] = *reinterpret_cast<uint32_t*>(&h2);
        }
        sts128(buf16 + (uint32_t)(e.lane * 64 + ((j ^ sw16) << 4)), pk[0], pk[1], pk[2], pk[3]);
      }
      fence_async_smem();
      __syncwarp();
      if (e.lane == 0) {
        tma_store_3d(&tmP, buf16, ch * 32, e.row0_in_img, e.z);
        bulk_commit();
      }
    }
    if (e.lane < e.slab_rows) inv_sum[(long long)e.z * nq + e.row0_in_img + e.lane] = 1.f / sum;
  }
  __device__ __forceinline__ void chunk(State&, const EpiCtx&, long long, bool, int, const uint32_t (&)[32], int) const {}
};

template <int KC, bool TF32 = false>
struct MatchEpi {
  static constexpr bool kTf32 = TF32;  // fp32-storage DB: operands fed to the tensor cores as TF32
  const float* dbnorm;
  long long N;
  float* cand_score;
  int32_t* cand_idx;
  int lists;  // candidate lists per query = 2 * splits (one per column half)
  static constexpr int kWarpStageBytes = 0;
  static constexpr int kStageBytes = 0;
  static constexpr bool kWholeTile = false;
  // query tiles are re-read for every DB tile: keep them in L2; DB rows stream through once per group
  static constexpr uint64_t kHintA = L2_EVICT_LAST, kHintB = L2_EVICT_FIRST;
  struct State {
    float s[KC];
    int32_t i[KC];
  };
  __device__ __forceinline__ void unit_begin(State& st) const {
#pragma unroll
    for (int t = 0; t < KC; ++t) { st.s[t] = INFINITY; st.i[t] = -1; }
  }
  __device__ __forceinline__ void kernel_begin(State&, const EpiCtx&) const {}
  __device__ __forceinline__ void tile_begin(State&, const EpiCtx&, int, int) const {}
  __device__ __forceinline__ void chunk(State& st, const EpiCtx&, long long, bool row_ok, int col0,
                                        const uint32_t (&v)[32], int) const {
    if (!row_ok || col0 >= N) return;
    float nrm[32];
    if ((long long)col0 + 32 <= N) {
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(dbnorm + col0 + j));
        nrm[j] = t.x; nrm[j + 1] = t.y; nrm[j + 2] = t.z; nrm[j + 3] = t.w;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j) nrm[j] = ((long long)col0 + j < N) ? __ldg(dbnorm + col0 + j) : INFINITY;
    }
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      // coarse squared distance up to the per-query constant ||q||^2 (+inf beyond the last row)
      float sc = fmaf(-2.f, __uint_as_float(v[j]), nrm[j]);
      if (sc < st.s[KC - 1]) {
        int32_t ci = col0 + j;
#pragma unroll
        for (int t = 0; t < KC; ++t) {
          if (sc < st.s[t]) {
            const float ts = st.s[t]; st.s[t] = sc; sc = ts;
            const int32_t ti = st.i[t]; st.i[t] = ci; ci = ti;
          }
        }
      }
    }
  }
  __device__ __forceinline__ void kernel_end(const EpiCtx&) const {}
  __device__ __forceinline__ void unit_end(State& st, const EpiCtx& e, long long row, bool row_ok, int split) const {
    if (!row_ok) return;
    const long long o = (row * lists + split * 2 + e.half) * KC;
#pragma unroll
    for (int t = 0; t < KC; ++t) { cand_score[o + t] = st.s[t]; cand_idx[o + t] = st.i[t]; }
  }
};

// Shared-memory plan: as many TMA stages as fit next to the epilogue staging the epilogue needs.
constexpr int SMEM_LIMIT = 227 * 1024;
template <int BN, int EPI_BYTES>
struct TcSmem {
  static constexpr int B_STAGE_BYTES = BN * BLOCK_K * 2;
  static constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
  static constexpr int FIXED = 1024 /*alignment slack*/ + 256 /*barriers*/ + EPI_BYTES;
  static constexpr int FIT = (SMEM_LIMIT - FIXED) / STAGE_BYTES;
  static constexpr int STAGES = FIT > 8 ? 8 : FIT;
  static constexpr int TOTAL = STAGES * STAGE_BYTES + FIXED;
  static_assert(STAGES >= 2, "not enough shared memory for a pipeline");
};


// Halo variant of the temporal convolution (HALO = true; 64 input channels, 5 taps, 24 rows per frame): the taps of one
// output tile read the SAME rows shifted by multiples of 24, so the general kernel fetches every activation row five times
// from L2 and the conv was bound by L2 -> SM traffic (ncu: 189 MB at 5.9 TB/s for a 24 MB tensor, tensor pipe 11 %).
// Here one TMA box of 128 + 4 x 24 = 224 rows lands per tile and tap t's A operand is that box at byte offset
// t x 24 x 128 = t x 3 KB - a whole number of 8-row swizzle atoms, so the UMMA descriptor just starts three atoms later -
// and the weights (5 taps x BN rows x 128 B) are loaded once per CTA and stay resident.
constexpr int HALO_TAPS = 5, HALO_SHIFT = 24, HALO_ROWS = BLOCK_M + (HALO_TAPS - 1) * HALO_SHIFT;
static_assert((HALO_SHIFT * 128) % 1024 == 0, "tap shifts must be whole swizzle atoms");
template <int BN, int EPI_BYTES>
struct HaloSmem {
  static constexpr int W_BYTES = HALO_TAPS * BN * BLOCK_K * 2;
  static constexpr int STAGE_BYTES = HALO_ROWS * BLOCK_K * 2;
  static constexpr int FIXED = 1024 /*alignment slack*/ + 256 /*barriers*/ + EPI_BYTES + W_BYTES;
  static constexpr int FIT = (SMEM_LIMIT - FIXED) / STAGE_BYTES;
  static constexpr int STAGES = FIT > 6 ? 6 : FIT;
  static constexpr int TOTAL = STAGES * STAGE_BYTES + FIXED;
  static_assert(STAGES >= 2, "not enough shared memory for a pipeline");
};

// Register re-partition between the producer warpgroup and the two epilogue warpgroups (see TC_EPI_WARP0): warpgroup-
// uniform, executed by every warp of the CTA once the prologue is done.
__device__ __forceinline__ void tc_regs_producer() {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(TC_REGS_PRODUCER));
}
__device__ __forceinline__ void tc_regs_epilogue() {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(TC_REGS_EPI));
}

template <int BN, class Epi, bool HALO = false>
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const TcShape sh, const int num_kb, const __grid_constant__ Epi epi) {
  using SM = typename std::conditional<HALO, HaloSmem<BN, Epi::kStageBytes>, TcSmem<BN, Epi::kStageBytes>>::type;
  constexpr int STAGES = SM::STAGES;
  constexpr uint32_t TMEM_COLS = 2 * BN < 32 ? 32 : 2 * BN;
  constexpr int KELEMS = Epi::kTf32 ? 32 : BLOCK_K;  // elements per 128-byte k-block row
  constexpr int W_RESIDENT = HALO ? HALO_TAPS * BN * BLOCK_K * 2 : 0;
  static_assert(!HALO || !Epi::kTf32, "the halo variant is bf16 only");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  // [operand stages][resident weights (HALO)][epilogue staging (1 KB aligned: stage sizes are multiples of 1 KB)][barriers]
  uint8_t* wres = smem + STAGES * SM::STAGE_BYTES;
  uint8_t* epi_stage = wres + W_RESIDENT;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(epi_stage + Epi::kStageBytes);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tfull_bar = empty_bar + STAGES;   // [2]
  uint64_t* tempty_bar = tfull_bar + 2;       // [2]
  uint64_t* res_bar = tempty_bar + 2;         // [EPI_WARPS] residual-prefetch barriers (LinearEpi)
  uint64_t* w_bar = res_bar + EPI_WARPS;      // resident weights landed (HALO)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(w_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_trigger();
#ifdef MOCHA_TRACE
  unsigned long long* const trace_buf = g_tc_trace;
  const int dbg_mode = g_tc_dbg_mode;
  if (threadIdx.x == 0) { TC_TRACE(0, gtimer()); TC_TRACE(1, (unsigned long long)clock64()); }
#endif

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], EPI_WARPS); }
    for (int i = 0; i < EPI_WARPS; ++i) mbar_init(&res_bar[i], 1);
    mbar_init(w_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // PDL: everything above (barriers, TMEM, descriptor prefetch) ran under the previous kernel's tail; operands and
  // outputs may only be touched once that kernel has completed
  pdl_wait();
#ifdef MOCHA_TRACE
  if (threadIdx.x == 0) TC_TRACE(2, (unsigned long long)clock64());
  int trace_tile = 0;
#endif

  if (warp < TC_EPI_WARP0) {
  tc_regs_producer();
  if (warp == 0) {
    // ===================== TMA producer =====================
    if (HALO && lane == 0) {
      // weights: constants, but read after the grid dependency like every other global read of the kernel
      mbar_expect_tx(w_bar, (uint32_t)W_RESIDENT);
#pragma unroll
      for (int tap = 0; tap < HALO_TAPS; ++tap)
        tma_load_2d(wres + tap * BN * BLOCK_K * 2, &tmB, w_bar, tap * BLOCK_K, 0);
      int stage = 0; uint32_t phase = 0;
      for (int u = blockIdx.x; u < sh.units; u += gridDim.x) {
        int mt, split;
        decode_unit(sh, u, mt, split);
        const int b = sh.nb == 1 ? 0 : fast_div(mt, sh.tiles_m_per_b), mtb = mt - b * sh.tiles_m_per_b;
        const long long a_row0 = (long long)b * sh.src_rows_per_b + (long long)mtb * BLOCK_M;
        mbar_wait(&empty_bar[stage], phase ^ 1);
        mbar_expect_tx(&full_bar[stage], SM::STAGE_BYTES);
        tma_load_2d(smem + stage * SM::STAGE_BYTES, &tmA, &full_bar[stage], 0, (int)a_row0);   // 224-row box: all five taps
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    } else if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int u = blockIdx.x; u < sh.units; u += gridDim.x) {
        int mt, split;
        decode_unit(sh, u, mt, split);
        const int b = sh.nb == 1 ? 0 : fast_div(mt, sh.tiles_m_per_b), mtb = mt - b * sh.tiles_m_per_b;
        long long a_row0 = (long long)b * sh.src_rows_per_b + (long long)mtb * BLOCK_M;
        long long b_row0 = 0;
        int a_col0 = 0, b_col0 = 0;
        if (sh.H > 0) {
          const int zb = fast_div(b, sh.H), zh = b - zb * sh.H;
          a_row0 = (long long)zb * sh.src_rows_per_b + (long long)zh * sh.a_rows_h + (long long)mtb * BLOCK_M;
          a_col0 = zh * sh.a_cols_h;
          b_row0 = (long long)zb * sh.b_rows_b + (long long)zh * sh.b_rows_h;
          b_col0 = zh * sh.b_cols_h;
        }
        const int nt_end = min(sh.tiles_n, (split + 1) * sh.tiles_per_unit);
        for (int nt = split * sh.tiles_per_unit; nt < nt_end; ++nt) {
          for (int kb = 0; kb < num_kb; ++kb) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            uint8_t* sa = smem + stage * SM::STAGE_BYTES;
            uint8_t* sb = sa + A_STAGE_BYTES;
#ifdef MOCHA_TRACE
            if (dbg_mode == 1) {
              mbar_arrive(&full_bar[stage]);
              if (++stage == STAGES) { stage = 0; phase ^= 1; }
              continue;
            }
#endif
            mbar_expect_tx(&full_bar[stage], SM::STAGE_BYTES);
            const int tap = kb / sh.kb_per_tap, kc = kb - tap * sh.kb_per_tap;
            if (Epi::kHintA != 0) {
              tma_load_2d_hint(sa, &tmA, &full_bar[stage], a_col0 + kc * KELEMS,
                               (int)(a_row0 + (long long)tap * sh.tap_row_stride), Epi::kHintA);
              tma_load_2d_hint(sb, &tmB, &full_bar[stage], b_col0 + kb * KELEMS, (int)(b_row0 + (long long)nt * BN),
                               Epi::kHintB);
            } else if (sh.b_mn) {
              tma_load_2d(sa, &tmA, &full_bar[stage], a_col0 + kc * KELEMS,
                          (int)(a_row0 + (long long)tap * sh.tap_row_stride));
#pragma unroll
              for (int a = 0; a < (BN >= 64 ? BN / 64 : 1); ++a)
                tma_load_2d(sb + a * 8192, &tmB, &full_bar[stage], b_col0 + nt * BN + a * 64, (int)(b_row0 + (long long)kb * BLOCK_K));
            } else {
              tma_load_2d(sa, &tmA, &full_bar[stage], a_col0 + kc * KELEMS,
                          (int)(a_row0 + (long long)tap * sh.tap_row_stride));
              tma_load_2d(sb, &tmB, &full_bar[stage], b_col0 + kb * KELEMS, (int)(b_row0 + (long long)nt * BN));
            }
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
#ifdef MOCHA_TRACE
          TC_TRACE(4 + trace_tile, (unsigned long long)clock64());  // all loads of the tile issued
          if (trace_tile < 3) ++trace_tile;
#endif
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (HALO && lane == 0) {
      constexpr uint32_t idesc = make_idesc(BLOCK_M, BN, 1u);
      int stage = 0; uint32_t phase = 0;
      int as = 0; uint32_t aphase = 0;
      mbar_wait(w_bar, 0);
      const uint32_t wb = smem_u32(wres);
      for (int u = blockIdx.x; u < sh.units; u += gridDim.x) {
        mbar_wait(&tempty_bar[as], aphase ^ 1);
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(as * BN);
        const uint32_t sa = smem_u32(smem + stage * SM::STAGE_BYTES);
#pragma unroll
        for (int tap = 0; tap < HALO_TAPS; ++tap) {
          const uint64_t adesc = make_smem_desc(sa + (uint32_t)(tap * HALO_SHIFT * BLOCK_K * 2));
          const uint64_t bdesc = make_smem_desc(wb + (uint32_t)(tap * BN * BLOCK_K * 2));
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k)
            umma_bf16(tmem_d, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (tap | k) != 0);
        }
        umma_commit(&empty_bar[stage]);
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
        umma_commit(&tfull_bar[as]);
        if (++as == 2) { as = 0; aphase ^= 1; }
      }
    } else if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(BLOCK_M, BN, Epi::kTf32 ? 2u : 1u);
      int stage = 0; uint32_t phase = 0;
      int as = 0; uint32_t aphase = 0;
      for (int u = blockIdx.x; u < sh.units; u += gridDim.x) {
        int mt, split;
        decode_unit(sh, u, mt, split);
        const int nt_end = min(sh.tiles_n, (split + 1) * sh.tiles_per_unit);
        for (int nt = split * sh.tiles_per_unit; nt < nt_end; ++nt) {
          mbar_wait(&tempty_bar[as], aphase ^ 1);
          tc_fence_after();
          const uint32_t tmem_d = tmem_base + (uint32_t)(as * BN);
          for (int kb = 0; kb < num_kb; ++kb) {
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after();
#ifdef MOCHA_TRACE
            if (kb == 0) TC_TRACE(8 + trace_tile, (unsigned long long)clock64());  // first operands landed
#endif
            const uint32_t sa = smem_u32(smem + stage * SM::STAGE_BYTES);
            const uint64_t adesc = make_smem_desc(sa);
#ifdef MOCHA_TRACE
            if (dbg_mode == 2) {
              mbar_arrive(&empty_bar[stage]);
              if (++stage == STAGES) { stage = 0; phase ^= 1; }
              continue;
            }
#endif
            if (!Epi::kTf32 && sh.b_mn) {
              // MN-major B: one MMA consumes 16 K-rows = 2 KB of every 64-column atom
              const uint64_t bdesc = make_smem_desc_mn(sa + A_STAGE_BYTES, 8192);
#pragma unroll
              for (int k = 0; k < BLOCK_K / UMMA_K; ++k)
                umma_bf16(tmem_d, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(128 * k), idesc | (1u << 16), (kb | k) != 0);
            } else {
              const uint64_t bdesc = make_smem_desc(sa + A_STAGE_BYTES);
#pragma unroll
              for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
                // advance 32 B (16 bf16) inside the 128 B swizzle atom: +2 in 16 B units
                if (Epi::kTf32) umma_tf32(tmem_d, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb | k) != 0);
                else umma_bf16(tmem_d, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb | k) != 0);
              }
            }
            umma_commit(&empty_bar[stage]);
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
          umma_commit(&tfull_bar[as]);
          if (++as == 2) { as = 0; aphase ^= 1; }
#ifdef MOCHA_TRACE
          TC_TRACE(12 + trace_tile, (unsigned long long)clock64());  // tile's MMAs issued + committed
          if (trace_tile < 3) ++trace_tile;
#endif
        }
      }
    }
  }
  } else {
    tc_regs_epilogue();
    // ===================== epilogue (the last eight warps) =====================
    const int q = warp & 3;  // TMEM lane quarter this warp may read
    int as = 0; uint32_t aphase = 0;
    typename Epi::State st;
    EpiCtx ectx;
    ectx.stage = smem_u32(epi_stage + (warp - TC_EPI_WARP0) * Epi::kWarpStageBytes);
    ectx.res_bar = smem_u32(&res_bar[warp - TC_EPI_WARP0]);
    ectx.bias_smem = smem_u32(epi_stage + EPI_WARPS * Epi::kWarpStageBytes);
    ectx.etid = (int)threadIdx.x - TC_EPI_WARP0 * 32;
    ectx.lane = lane;
    epi.kernel_begin(st, ectx);
    // Tile bookkeeping off the critical path: the unit -> (m tile, split, image) decode is ~200 dependent
    // scalar instructions (~1000 cycles between two tiles of a warp that has only one partner on its
    // scheduler). Lane i decodes the CTA's i-th unit once, up front, while the first main loop runs; each
    // tile then fetches its numbers with four shuffles.
    int pre_mt = 0, pre_split = 0, pre_b = 0, pre_zb = 0;
    {
      const long long u = (long long)blockIdx.x + (long long)lane * gridDim.x;
      if (u < sh.units) {
        decode_unit(sh, (int)u, pre_mt, pre_split);
        pre_b = sh.nb == 1 ? 0 : fast_div(pre_mt, sh.tiles_m_per_b);
        pre_zb = sh.H > 0 ? fast_div(pre_b, sh.H) : 0;
      }
    }
    int unit_it = 0;
    for (int u = blockIdx.x; u < sh.units; u += gridDim.x, ++unit_it) {
      int mt, split, b, zb_pre;
      if (unit_it < 32) {
        mt = __shfl_sync(0xffffffffu, pre_mt, unit_it);
        split = __shfl_sync(0xffffffffu, pre_split, unit_it);
        b = __shfl_sync(0xffffffffu, pre_b, unit_it);
        zb_pre = __shfl_sync(0xffffffffu, pre_zb, unit_it);
      } else {
        decode_unit(sh, u, mt, split);
        b = sh.nb == 1 ? 0 : fast_div(mt, sh.tiles_m_per_b);
        zb_pre = sh.H > 0 ? fast_div(b, sh.H) : 0;
      }
      const int mtb = mt - b * sh.tiles_m_per_b;
      const int r_in_b = mtb * BLOCK_M + q * 32 + lane;
      const bool row_ok = r_in_b < sh.rows_out_per_b;
      const long long row = (long long)b * sh.rows_out_per_b + r_in_b;
      ectx.col_off = 0;
      ectx.z = b;
      ectx.img = b;
      ectx.row0_in_img = mtb * BLOCK_M + q * 32;
      ectx.lane = lane;
      ectx.half = (warp - TC_EPI_WARP0) >> 2;
      ectx.slab_row0 = (long long)b * sh.rows_out_per_b + mtb * BLOCK_M + q * 32;
      ectx.slab_rows = max(0, min(32, sh.rows_out_per_b - (mtb * BLOCK_M + q * 32)));
      ectx.c_off = 0;
      if (sh.H > 0) {
        const int zb = zb_pre, zh = b - zb * sh.H;
        ectx.slab_row0 = mtb * BLOCK_M + q * 32;
        ectx.c_off = (long long)zb * sh.c_img_b + (long long)zh * sh.c_img_h;
        ectx.img = zb;                      // TMA-store view of a [B, rows, H*cols] output (host checks the layout)
        ectx.col_off = zh * (int)sh.c_img_h;
      }
      epi.unit_begin(st);
      const int nt_end = min(sh.tiles_n, (split + 1) * sh.tiles_per_unit);
      for (int nt = split * sh.tiles_per_unit; nt < nt_end; ++nt) {
        // the tile's BN/32 column chunks are split between the two warps that share a lane quarter
        constexpr int kSplitCol = ((BN / 32 + 1) / 2) * 32;
        const int c_begin = ectx.half == 0 ? 0 : kSplitCol, c_end = ectx.half == 0 ? kSplitCol : BN;
#ifdef MOCHA_TRACE
        if (warp == TC_EPI_WARP0 && lane == 0 && trace_tile == 1) TC_TRACE(29, (unsigned long long)clock64());
#endif
        if (c_begin < c_end) epi.tile_begin(st, ectx, nt * BN + c_begin, c_end - c_begin);  // overlaps the main loop
#ifdef MOCHA_TRACE
        if (warp == TC_EPI_WARP0 && lane == 0 && trace_tile == 1) TC_TRACE(30, (unsigned long long)clock64());
#endif
        mbar_wait(&tfull_bar[as], aphase);
        tc_fence_after();
#ifdef MOCHA_TRACE
        if (warp == TC_EPI_WARP0 && lane == 0) TC_TRACE(16 + trace_tile, (unsigned long long)clock64());  // accumulator ready
#endif
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * BN);
        if constexpr (Epi::kWholeTile) epi.tile(st, ectx, taddr, as);
#ifdef MOCHA_TRACE
        const int c_stop = dbg_mode == 3 ? c_begin : c_end;
#else
        const int c_stop = c_end;
#endif
#pragma unroll 1
        for (int c0 = c_begin; c0 < (Epi::kWholeTile ? c_begin : c_stop); c0 += 32) {
          uint32_t v[32];
          tmem_ld32(taddr + (uint32_t)c0, v);
#ifdef MOCHA_TRACE
          if (warp == TC_EPI_WARP0 && lane == 0 && trace_tile == 0 && c0 == c_begin) TC_TRACE(26, (unsigned long long)clock64());
#endif
          epi.chunk(st, ectx, row, row_ok, nt * BN + c0, v, c0 + 32 < c_end ? nt * BN + c0 + 32 : -1);
#ifdef MOCHA_TRACE
          if (warp == TC_EPI_WARP0 && lane == 0 && trace_tile == 0 && c0 == c_begin) TC_TRACE(27, (unsigned long long)clock64());
          if (warp == TC_EPI_WARP0 && lane == 0 && trace_tile == 0 && c0 == c_begin + 32) TC_TRACE(28, (unsigned long long)clock64());
#endif
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty_bar[as]);
        if (++as == 2) { as = 0; aphase ^= 1; }
#ifdef MOCHA_TRACE
        if (warp == TC_EPI_WARP0 && lane == 0) TC_TRACE(20 + trace_tile, (unsigned long long)clock64());  // tile drained
        if (trace_tile < 3) ++trace_tile;
#endif
      }
      epi.unit_end(st, ectx, row, row_ok, split);
    }
    epi.kernel_end(ectx);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
#ifdef MOCHA_TRACE
  if (threadIdx.x == 0) { TC_TRACE(24, (unsigned long long)clock64()); TC_TRACE(25, gtimer()); }
#endif
}

// ------------------------------------------------------------------------------------------------
// CTA-pair GEMM kernel: a thread-block cluster of two CTAs (one TPC) computes a 256 x 256 tile with
// tcgen05.mma.cta_group::2. Each CTA stages its own 128 activation rows (A) and HALF of the weight rows (B)
// per k-block, so the shared-memory fill and operand-read traffic per SM drop by 1/3 and 1/3 vs the
// 1-CTA kernel; the leader CTA's single MMA thread issues for the pair, tcgen05.commit multicasts the
// "slot free" / "accumulator ready" signals to both CTAs, and each CTA's epilogue warps drain their
// own 128 TMEM lanes.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t cta) {
  asm volatile(
      "{\n"
      ".reg .b32 ra;\n"
      "mapa.shared::cluster.u32 ra, %0, %1;\n"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(cta)
      : "memory");
}
// TMA load whose completion is signalled on the LEADER CTA's mbarrier (same smem offset, peer bit cleared)
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar, int c0, int c1,
                                                 uint64_t policy) {
  const uint32_t leader_bar = smem_u32(bar) & 0xFEFFFFFFu;
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_u32(smem_dst)), "l"(tmap), "r"(leader_bar), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"((uint16_t)3)
               : "memory");
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

constexpr int M2_BN = 256;                               // pair tile: 256 (M) x 256 (N)
constexpr int M2_STAGE_BYTES = A_STAGE_BYTES + 128 * BLOCK_K * 2;  // 128 A rows + 128 B rows per CTA
template <int EPI_BYTES>
struct PairSmem {
  static constexpr int FIXED = 1024 /*alignment slack*/ + 256 /*barriers*/ + EPI_BYTES;
  static constexpr int FIT = (SMEM_LIMIT - FIXED) / M2_STAGE_BYTES;
  static constexpr int STAGES = FIT > 6 ? 6 : FIT;
  static constexpr int TOTAL = STAGES * M2_STAGE_BYTES + FIXED;
};

// Works on the same TcShape as the 1-CTA kernel with tiles_m_per_b counted in 256-row PAIR tiles
// (plain / tconv mode; no batched-head mode). CTA `rank` of the pair owns rows [rank*128, +128) of the
// pair tile and stages B rows [rank*128, +128) of the 256-wide n-tile.
template <class Epi>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TC_THREADS, 1)
tc_gemm2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const TcShape sh,
                const int num_kb, const __grid_constant__ Epi epi) {
  pdl_trigger();
  using SM = PairSmem<Epi::kStageBytes>;
  constexpr int STAGES = SM::STAGES;
  constexpr int BN = M2_BN;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* epi_stage = smem + STAGES * M2_STAGE_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(epi_stage + Epi::kStageBytes);     // used in the leader
  uint64_t* empty_bar = full_bar + STAGES;                                            // per CTA
  uint64_t* tfull_bar = empty_bar + STAGES;                                           // per CTA [2]
  uint64_t* tempty_bar = tfull_bar + 2;                                               // leader [2]
  uint64_t* res_bar = tempty_bar + 2;                                                 // per CTA [EPI_WARPS]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_bar + EPI_WARPS);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int cid = blockIdx.x >> 1, ncl = gridDim.x >> 1;
#ifdef MOCHA_TRACE
  unsigned long long* const trace_buf = g_tc_trace;
  if (threadIdx.x == 0) { TC_TRACE(0, gtimer()); TC_TRACE(1, (unsigned long long)clock64()); }
  int trace_tile = 0;
#endif

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], 2); mbar_init(&empty_bar[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], 2 * EPI_WARPS); }
    for (int i = 0; i < EPI_WARPS; ++i) mbar_init(&res_bar[i], 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc_pair(tmem_slot, 512);
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();   // PDL: the prologue above overlaps the previous kernel's tail (see tc_gemm_kernel)
#ifdef MOCHA_TRACE
  if (threadIdx.x == 0) TC_TRACE(2, (unsigned long long)clock64());
#endif

  if (warp < TC_EPI_WARP0) {
  tc_regs_producer();
  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int u = cid; u < sh.units; u += ncl) {
        int mt, split;
        decode_unit(sh, u, mt, split);
        const int b = sh.nb == 1 ? 0 : fast_div(mt, sh.tiles_m_per_b), mtb = mt - b * sh.tiles_m_per_b;
        const long long a_row0 = (long long)b * sh.src_rows_per_b + (long long)mtb * 256 + (int)rank * 128;
        const int nt_end = min(sh.tiles_n, (split + 1) * sh.tiles_per_unit);
        for (int nt = split * sh.tiles_per_unit; nt < nt_end; ++nt) {
          const int b_row0 = nt * BN + (int)rank * 128 + (sh.H > 0 ? b * (int)sh.b_rows_b : 0);   // H > 0: one weight per image
          for (int kb = 0; kb < num_kb; ++kb) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            uint8_t* sa = smem + stage * M2_STAGE_BYTES;
            uint8_t* sb = sa + A_STAGE_BYTES;
            if (rank == 0) mbar_expect_tx(&full_bar[stage], 2 * M2_STAGE_BYTES);
            const int tap = kb / sh.kb_per_tap, kc = kb - tap * sh.kb_per_tap;
            tma_load_2d_pair(sa, &tmA, &full_bar[stage], kc * BLOCK_K, (int)(a_row0 + (long long)tap * sh.tap_row_stride), L2_EVICT_NORMAL);
            tma_load_2d_pair(sb, &tmB, &full_bar[stage], kb * BLOCK_K, b_row0, L2_EVICT_NORMAL);
            if (rank != 0) mbar_arrive_remote(&full_bar[stage], 0);
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
#ifdef MOCHA_TRACE
          TC_TRACE(4 + trace_tile, (unsigned long long)clock64());
          if (trace_tile < 3) ++trace_tile;
#endif
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (lane == 0 && rank == 0) {
      constexpr uint32_t idesc = make_idesc(256, BN);
      int stage = 0; uint32_t phase = 0;
      int as = 0; uint32_t aphase = 0;
      for (int u = cid; u < sh.units; u += ncl) {
        int mt, split;
        decode_unit(sh, u, mt, split);
        const int nt_end = min(sh.tiles_n, (split + 1) * sh.tiles_per_unit);
        for (int nt = split * sh.tiles_per_unit; nt < nt_end; ++nt) {
          mbar_wait(&tempty_bar[as], aphase ^ 1);
          tc_fence_after();
          const uint32_t tmem_d = tmem_base + (uint32_t)(as * BN);
          for (int kb = 0; kb < num_kb; ++kb) {
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after();
#ifdef MOCHA_TRACE
            if (kb == 0) TC_TRACE(8 + trace_tile, (unsigned long long)clock64());
#endif
            const uint32_t sa = smem_u32(smem + stage * M2_STAGE_BYTES);
            const uint64_t adesc = make_smem_desc(sa);
            const uint64_t bdesc = make_smem_desc(sa + A_STAGE_BYTES);
#pragma unroll
            for (int k = 0; k < BLOCK_K / UMMA_K; ++k)
              umma_bf16_pair(tmem_d, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb | k) != 0);
            umma_commit_pair(&empty_bar[stage]);
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
          umma_commit_pair(&tfull_bar[as]);
          if (++as == 2) { as = 0; aphase ^= 1; }
#ifdef MOCHA_TRACE
          TC_TRACE(12 + trace_tile, (unsigned long long)clock64());
          if (trace_tile < 3) ++trace_tile;
#endif
        }
      }
    }
  }
  } else {
    tc_regs_epilogue();
    // ===================== epilogue (the last eight warps of both CTAs) =====================
    const int q = warp & 3;
    int as = 0; uint32_t aphase = 0;
    typename Epi::State st;
    EpiCtx ectx;
    ectx.stage = smem_u32(epi_stage + (warp - TC_EPI_WARP0) * Epi::kWarpStageBytes);
    ectx.res_bar = smem_u32(&res_bar[warp - TC_EPI_WARP0]);
    ectx.bias_smem = smem_u32(epi_stage + EPI_WARPS * Epi::kWarpStageBytes);
    ectx.etid = (int)threadIdx.x - TC_EPI_WARP0 * 32;
    ectx.lane = lane; ectx.half = (warp - TC_EPI_WARP0) >> 2; ectx.c_off = 0; ectx.col_off = 0;
    epi.kernel_begin(st, ectx);
    // lane i decodes the cluster's i-th unit up front (see tc_gemm_kernel); tiles fetch it with shuffles
    int pre_mt = 0, pre_split = 0, pre_b = 0;
    {
      const long long u = (long long)cid + (long long)lane * ncl;
      if (u < sh.units) {
        decode_unit(sh, (int)u, pre_mt, pre_split);
        pre_b = sh.nb == 1 ? 0 : fast_div(pre_mt, sh.tiles_m_per_b);
      }
    }
    int unit_it = 0;
    for (int u = cid; u < sh.units; u += ncl, ++unit_it) {
      int mt, split, b;
      if (unit_it < 32) {
        mt = __shfl_sync(0xffffffffu, pre_mt, unit_it);
        split = __shfl_sync(0xffffffffu, pre_split, unit_it);
        b = __shfl_sync(0xffffffffu, pre_b, unit_it);
      } else {
        decode_unit(sh, u, mt, split);
        b = sh.nb == 1 ? 0 : fast_div(mt, sh.tiles_m_per_b);
      }
      const int mtb = mt - b * sh.tiles_m_per_b;
      const int r0 = mtb * 256 + (int)rank * 128 + q * 32;   // first row of the slab inside its image
      const bool row_ok = r0 + lane < sh.rows_out_per_b;
      const long long row = (long long)b * sh.rows_out_per_b + r0 + lane;
      ectx.slab_row0 = (long long)b * sh.rows_out_per_b + r0;
      ectx.slab_rows = max(0, min(32, sh.rows_out_per_b - r0));
      ectx.img = b; ectx.z = b; ectx.row0_in_img = r0;
      epi.unit_begin(st);
      const int nt_end = min(sh.tiles_n, (split + 1) * sh.tiles_per_unit);
      for (int nt = split * sh.tiles_per_unit; nt < nt_end; ++nt) {
        const int c_begin = ectx.half * (BN / 2), c_end = c_begin + BN / 2;
        epi.tile_begin(st, ectx, nt * BN + c_begin, c_end - c_begin);
        mbar_wait(&tfull_bar[as], aphase);
        tc_fence_after();
#ifdef MOCHA_TRACE
        if (warp == TC_EPI_WARP0 && lane == 0) TC_TRACE(16 + trace_tile, (unsigned long long)clock64());
#endif
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * BN);
#pragma unroll 1
        for (int c0 = c_begin; c0 < c_end; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(taddr + (uint32_t)c0, v);
          epi.chunk(st, ectx, row, row_ok, nt * BN + c0, v, c0 + 32 < c_end ? nt * BN + c0 + 32 : -1);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_remote(&tempty_bar[as], 0);
        if (++as == 2) { as = 0; aphase ^= 1; }
#ifdef MOCHA_TRACE
        if (warp == TC_EPI_WARP0 && lane == 0) TC_TRACE(20 + trace_tile, (unsigned long long)clock64());
        if (trace_tile < 3) ++trace_tile;
#endif
      }
      epi.unit_end(st, ectx, row, row_ok, split);
    }
    epi.kernel_end(ectx);
  }

  // the peer must stay resident until the leader's last MMA has read its shared memory
  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, 512);
  }
#ifdef MOCHA_TRACE
  if (threadIdx.x == 0) { TC_TRACE(24, (unsigned long long)clock64()); TC_TRACE(25, gtimer()); }
#endif
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// bf16 [rows, K] row-major, box = box_rows x 64 elements, 128B swizzle, OOB reads return zero
int make_tmap(CUtensorMap* tm, const void* ptr, unsigned long long rows, unsigned long long K, int box_rows,
              unsigned long long pitch_elems = 0, bool f32 = false) {
  if (pitch_elems == 0) pitch_elems = K;
  const unsigned long long esz = f32 ? 4 : 2;
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return set_error(MOCHA_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
  MOCHA_CHECK_ARG((reinterpret_cast<uintptr_t>(ptr) & 15) == 0, "tensor map: base not 16B aligned");
  MOCHA_CHECK_ARG((pitch_elems * esz) % 16 == 0, "tensor map: row pitch %llu B not a multiple of 16", pitch_elems * esz);
  cuuint64_t gdim[2] = {K, rows};
  cuuint64_t gstride[1] = {pitch_elems * esz};
  cuuint32_t box[2] = {(cuuint32_t)(128 / esz), (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(tm, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(MOCHA_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  return MOCHA_OK;
}

// Output maps of the TMA-store epilogue: {cols, rows per image, images}, box 32 cols x 32 rows x 1.
// fp32 boxes are 128 B-swizzled (the epilogue transposes through them), bf16 boxes 64 B-swizzled.
int make_out_tmap(CUtensorMap* tm, const void* ptr, unsigned long long cols, unsigned long long rows_per_img,
                  unsigned long long imgs, unsigned long long ld_elems, bool f32, unsigned long long img_pitch_rows = 0,
                  bool wide16 = false) {
  if (img_pitch_rows == 0) img_pitch_rows = rows_per_img;
  const unsigned long long esz = f32 ? 4 : 2;
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return set_error(MOCHA_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
  cuuint64_t gdim[3] = {cols, rows_per_img, imgs};
  cuuint64_t gstride[2] = {ld_elems * esz, img_pitch_rows * ld_elems * esz};
  cuuint32_t box[3] = {wide16 ? 64u : 32u, 32, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(tm, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), gdim,
                  gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  (f32 || wide16) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(MOCHA_ERR_CUDA, "cuTensorMapEncodeTiled (output) failed (%d)", (int)r);
  return MOCHA_OK;
}

// Switch a LinearEpi to the TMA-store path when its outputs allow it (plain / tconv mode only).
int setup_out_tma(LinearEpi& epi, unsigned long long rows_per_img, unsigned long long imgs, unsigned long long cols = 0,
                  unsigned long long img_pitch_rows = 0) {
  epi.tma = 0;
  if (cols == 0) cols = (unsigned long long)epi.N;
  const bool ok = (epi.N % 4) == 0 && (epi.ldc % 8) == 0 && (epi.N <= 2048 || !epi.bias || epi.bias_period > 0) &&
                  ((reinterpret_cast<uintptr_t>(epi.C) | reinterpret_cast<uintptr_t>(epi.C16) |
                    reinterpret_cast<uintptr_t>(epi.res) | reinterpret_cast<uintptr_t>(epi.bias)) & 15) == 0;
  if (!ok) return MOCHA_OK;
  const bool with_res = epi.res && epi.bias_period == 0;
  if (epi.C && epi.C16 && !with_res) return MOCHA_OK;  // two outputs without a residual: LSU epilogue
  if (epi.C) MOCHA_TRY(make_out_tmap(&epi.tmC, epi.C, cols, rows_per_img, imgs, (unsigned long long)epi.ldc, true, img_pitch_rows));
  if (epi.C16) MOCHA_TRY(make_out_tmap(&epi.tmC16, epi.C16, cols, rows_per_img, imgs, (unsigned long long)epi.ldc, false, img_pitch_rows));
  epi.tma = 1;
  epi.c16_wide = 0;
  if (epi.C16 && !epi.C && !with_res && epi.bias_period == 0 && epi.N % 64 == 0 && cols % 64 == 0) {
    // the launcher clears this again when the tile is narrower than 128 columns (odd chunk count per warp)
    MOCHA_TRY(make_out_tmap(&epi.tmC16w, epi.C16, cols, rows_per_img, imgs, (unsigned long long)epi.ldc, false, img_pitch_rows, true));
    epi.c16_wide = 1;
  }
  if (with_res) {
    MOCHA_TRY(make_out_tmap(&epi.tmR, epi.res, cols, rows_per_img, imgs, (unsigned long long)epi.ldc, true, img_pitch_rows));
    epi.tma = 2;
  }
  return MOCHA_OK;
}

int num_sms() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

template <int BN, class Epi>
int launch_tc(const CUtensorMap& tmA, const CUtensorMap& tmB, const TcShape& sh, int num_kb, const Epi& epi,
              cudaStream_t s) {
  using SM = TcSmem<BN, Epi::kStageBytes>;
  static bool configured = false;
  if (!configured) {
    MOCHA_CUDA(cudaFuncSetAttribute(tc_gemm_kernel<BN, Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM::TOTAL));
    configured = true;
  }
  const int grid = sh.units < num_sms() ? sh.units : num_sms();
  launch_k(tc_gemm_kernel<BN, Epi>, grid, TC_THREADS, SM::TOTAL, s, tmA, tmB, sh, num_kb, epi);
  count_launch();
  MOCHA_LAUNCH_CHECK("tc_gemm_kernel");
  return MOCHA_OK;
}

// Halo variant (see HaloSmem): tmA boxes are HALO_ROWS x 64, tmB boxes BN x 64 over the [BN, taps * 64] weight; one n-tile.
template <int BN, class Epi>
int launch_tc_halo(const CUtensorMap& tmA, const CUtensorMap& tmB, const TcShape& sh, const Epi& epi, cudaStream_t s) {
  using SM = HaloSmem<BN, Epi::kStageBytes>;
  static bool configured = false;
  if (!configured) {
    MOCHA_CUDA(cudaFuncSetAttribute(tc_gemm_kernel<BN, Epi, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM::TOTAL));
    configured = true;
  }
  const int grid = sh.units < num_sms() ? sh.units : num_sms();
  launch_k(tc_gemm_kernel<BN, Epi, true>, grid, TC_THREADS, SM::TOTAL, s, tmA, tmB, sh, HALO_TAPS, epi);
  count_launch();
  MOCHA_LAUNCH_CHECK("tc_gemm_kernel(halo)");
  return MOCHA_OK;
}

template <class Epi>
int launch_pair(const CUtensorMap& tmA, const CUtensorMap& tmB, const TcShape& sh, int num_kb, const Epi& epi,
                cudaStream_t s) {
  using SM = PairSmem<Epi::kStageBytes>;
  static bool configured = false;
  if (!configured) {
    MOCHA_CUDA(cudaFuncSetAttribute(tc_gemm2_kernel<Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM::TOTAL));
    configured = true;
  }
  int grid = 2 * sh.units;
  const int cap = num_sms() & ~1;
  if (grid > cap) grid = cap;
  launch_k(tc_gemm2_kernel<Epi>, grid, TC_THREADS, SM::TOTAL, s, tmA, tmB, sh, num_kb, epi);
  count_launch();
  MOCHA_LAUNCH_CHECK("tc_gemm2_kernel");
  return MOCHA_OK;
}

__global__ void cast_act_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, long long n,
                                     int lrelu) {
  pdl_trigger();
  pdl_wait();
  const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i + 3 < n) {
    float4 v = *reinterpret_cast<const float4*>(x + i);
    if (lrelu) { v.x = lrelu02(v.x); v.y = lrelu02(v.y); v.z = lrelu02(v.z); v.w = lrelu02(v.w); }
    __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
    uint2 pk;
    pk.x = *reinterpret_cast<uint32_t*>(&lo);
    pk.y = *reinterpret_cast<uint32_t*>(&hi);
    *reinterpret_cast<uint2*>(y + i) = pk;
  } else {
    for (long long j = i; j < n; ++j) {
      float v = x[j];
      y[j] = __float2bfloat16_rn(lrelu ? lrelu02(v) : v);
    }
  }
}

// X fp32 [B,T,V,C] -> bf16 [B, T+2*pad, V, C] with reflect padding along T
__global__ void reflect_pad_cast_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, int T, int V,
                                        int C, int pad, int tdiv, long long total4) {
  pdl_trigger();
  pdl_wait();
  const long long i4 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i4 >= total4) return;
  const long long i = i4 * 4;
  const int c = (int)(i % C);
  const long long r = i / C;
  const int v = (int)(r % V);
  const long long bt = r / V;
  const int Tp = T + 2 * pad;
  const int tp = (int)(bt % Tp);
  const long long b = bt / Tp;
  int t = tp - pad;
  if (t < 0) t = -t;
  if (t >= T) t = 2 * (T - 1) - t;
  t /= tdiv;  // nearest-neighbour temporal up-sampling folded into the gather (source has T/tdiv frames)
  const float4 val = *reinterpret_cast<const float4*>(x + (((b * (T / tdiv) + t) * V + v) * (long long)C + c));
  __nv_bfloat162 lo = __floats2bfloat162_rn(val.x, val.y), hi = __floats2bfloat162_rn(val.z, val.w);
  uint2 pk;
  pk.x = *reinterpret_cast<uint32_t*>(&lo);
  pk.y = *reinterpret_cast<uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(y + i) = pk;
}

// bf16 source variant (8 elements = 16 B per thread)
__global__ void reflect_pad_copy_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y, int T, int V,
                                        int C, int pad, int tdiv, long long total8) {
  pdl_trigger();
  pdl_wait();
  const long long i8 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i8 >= total8) return;
  const long long i = i8 * 8;
  const int c = (int)(i % C);
  const long long r = i / C;
  const int v = (int)(r % V);
  const long long bt = r / V;
  const int Tp = T + 2 * pad;
  const int tp = (int)(bt % Tp);
  const long long b = bt / Tp;
  int t = tp - pad;
  if (t < 0) t = -t;
  if (t >= T) t = 2 * (T - 1) - t;
  t /= tdiv;
  *reinterpret_cast<uint4*>(y + i) =
      *reinterpret_cast<const uint4*>(x + (((b * (T / tdiv) + t) * V + v) * (long long)C + c));
}

struct Blob {
  const float* b32;
  const __nv_bfloat16* b16;
  size_t elems;
};
// registry of bf16 weight mirrors: any number of live blobs, guarded for concurrent host threads (sessions / models are
// built and destroyed from Python threads; look-ups happen on every tensor-core layer call)
std::vector<Blob> g_blobs;
std::mutex g_blob_mutex;

// k_blocks > 0 lets long-K problems keep 256-wide tiles below one wave: a 128-wide tile needs twice the
// shared-memory fill per MMA (fill-bound at ~64 B/clk/SM), measured 16.3 -> 12.0 us on 11520 x 256 x 1024
int pick_bn(long long tiles_m, int N, int k_blocks = 0) {
  // largest BN that still gives about one wave of CTAs; tiles that would be mostly padding are skipped
  if (k_blocks >= 8 && N >= 256 && tiles_m * ((N + 255) / 256) * 2 >= num_sms()) return 256;
  const int cands[4] = {256, 128, 64, 32};
  for (int i = 0; i < 4; ++i) {
    const int bn = cands[i];
    if (bn > 32 && bn / 2 >= N) continue;
    if (tiles_m * ((N + bn - 1) / bn) >= num_sms()) return bn;
  }
  return N >= 128 ? 64 : 32;  // latency-bound problem: more, narrower CTAs
}

template <class Epi>
int dispatch_bn_impl(int bn, const CUtensorMap& tmA, const void* Wptr, unsigned long long wrows, unsigned long long K,
                TcShape sh, int N, int num_kb, const Epi& epi, cudaStream_t s, unsigned long long wpitch = 0) {
  CUtensorMap tmB;
  MOCHA_TRY(make_tmap(&tmB, Wptr, wrows, K, sh.b_mn ? 64 : bn, wpitch, Epi::kTf32));
  sh.tiles_n = ceil_div(N, bn);
  sh.tiles_per_unit = 1;
  sh.units = sh.tiles_m_total * sh.tiles_n;
  sh.splits = sh.tiles_n;
  sh.group_m = 0;
  switch (bn) {
    case 256: return launch_tc<256, Epi>(tmA, tmB, sh, num_kb, epi, s);
    case 128: return launch_tc<128, Epi>(tmA, tmB, sh, num_kb, epi, s);
    case 64: return launch_tc<64, Epi>(tmA, tmB, sh, num_kb, epi, s);
    default: return launch_tc<32, Epi>(tmA, tmB, sh, num_kb, epi, s);
  }
}

// LinearEpi launches: one kernel family per epilogue mode
int dispatch_bn(int bn, const CUtensorMap& tmA, const void* Wptr, unsigned long long wrows, unsigned long long K,
                TcShape sh, int N, int num_kb, const LinearEpi& epi, cudaStream_t s, unsigned long long wpitch = 0) {
  if (epi.tma == 2 && !epi.C16)   // residual, fp32 output only: no bf16 box, 128 x 256 tiles fit
    return dispatch_bn_impl(bn, tmA, Wptr, wrows, K, sh, N, num_kb, LinearEpiT<3>{epi}, s, wpitch);
  if (epi.tma == 2 && bn == 256) bn = 128;  // the residual / two-output staging leaves room for 32 KB stages only
  if (epi.c16_wide && bn < 128) {
    LinearEpi e2 = epi;
    e2.c16_wide = 0;
    return dispatch_bn_impl(bn, tmA, Wptr, wrows, K, sh, N, num_kb, LinearEpiT<4>{e2}, s, wpitch);
  }
  if (epi.tma == 2) return dispatch_bn_impl(bn, tmA, Wptr, wrows, K, sh, N, num_kb, LinearEpiT<2>{epi}, s, wpitch);
  if (epi.tma == 1) return dispatch_bn_impl(bn, tmA, Wptr, wrows, K, sh, N, num_kb, LinearEpiT<4>{epi}, s, wpitch);
  return dispatch_bn_impl(bn, tmA, Wptr, wrows, K, sh, N, num_kb, LinearEpiT<0>{epi}, s, wpitch);
}

// fp32 operands consumed as TF32 (kind::tf32, 32 elements per 128-byte k-block row): the 3xTF32 parity mode's GEMMs.
// Same epilogues; fp32 output only (modes 0 / 3 / 4).
template <int MODE>
struct LinearEpiTf : LinearEpiT<MODE> {
  static constexpr bool kTf32 = true;
};
int dispatch_bn_tf32(int bn, const CUtensorMap& tmA, const void* Wptr, unsigned long long wrows, unsigned long long K,
                     TcShape sh, int N, int num_kb, const LinearEpi& epi, cudaStream_t s) {
  if (epi.tma == 2) return dispatch_bn_impl(bn, tmA, Wptr, wrows, K, sh, N, num_kb, LinearEpiTf<3>{LinearEpiT<3>{epi}}, s);
  if (epi.tma == 1) return dispatch_bn_impl(bn, tmA, Wptr, wrows, K, sh, N, num_kb, LinearEpiTf<4>{LinearEpiT<4>{epi}}, s);
  return dispatch_bn_impl(bn, tmA, Wptr, wrows, K, sh, N, num_kb, LinearEpiTf<0>{LinearEpiT<0>{epi}}, s);
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// public (library-internal) API
// ------------------------------------------------------------------------------------------------
// tensor-map builders shared with the fused kernels (fused_tail.cu, fused_attn.cu)
int tc_make_tmap(CUtensorMap* tm, const void* ptr, unsigned long long rows, unsigned long long K, int box_rows,
                 unsigned long long pitch_elems, bool f32) {
  return make_tmap(tm, ptr, rows, K, box_rows, pitch_elems, f32);
}
int tc_make_out_tmap(CUtensorMap* tm, const void* ptr, unsigned long long cols, unsigned long long rows_per_img,
                     unsigned long long imgs, unsigned long long ld_elems, bool f32, unsigned long long img_pitch_rows,
                     bool wide16) {
  return make_out_tmap(tm, ptr, cols, rows_per_img, imgs, ld_elems, f32, img_pitch_rows, wide16);
}
int tc_num_sms() { return num_sms(); }

bool tc_linear_supported(int M, int N, int K) { return M >= 1 && N >= 8 && K >= 64 && (K % 8) == 0; }

// Workspace queries answer for the precision mode set by mocha_workspace_precision() (default: bf16, which also covers
// fp32): the 3xTF32 mode stages [rows, 3K] fp32 split operands plus the split weights (allowance: 2048 output rows).
int g_ws_precision = MOCHA_BF16;
void tc_set_workspace_precision(int precision) { g_ws_precision = precision; }
size_t tc_scratch_bytes(size_t rows, size_t K) {
  if (g_ws_precision == MOCHA_TF32X3) return align_up((rows + 2048) * K * 12, 256) + 1024;
  return align_up(rows * K * 2, 256) + 256;
}

void tc_register_blob(const float* blob32, const void* blob16, size_t elems) {
  std::lock_guard<std::mutex> lock(g_blob_mutex);
  // drop every entry that overlaps the new range (stale mirrors of freed / re-used allocations)
  size_t n = 0;
  for (size_t i = 0; i < g_blobs.size(); ++i) {
    const Blob& b = g_blobs[i];
    const bool overlap = blob32 < b.b32 + b.elems && b.b32 < blob32 + elems;
    if (!overlap) g_blobs[n++] = b;
  }
  g_blobs.resize(n);
  if (!blob16) return;  // unregister only
  g_blobs.push_back(Blob{blob32, (const __nv_bfloat16*)blob16, elems});
}

const __nv_bfloat16* tc_lookup_bf16(const float* W) {
  std::lock_guard<std::mutex> lock(g_blob_mutex);
  for (size_t i = g_blobs.size(); i-- > 0;) {   // newest first
    const Blob& b = g_blobs[i];
    if (b.b16 && W >= b.b32 && W < b.b32 + b.elems) return b.b16 + (W - b.b32);
  }
  return nullptr;
}

namespace {
// plain / image-batched linear layers on the CTA-pair kernel: single TMA-stored output, whole 256-wide n-tiles
bool pair_linear_wanted(const LinearEpi& epi, int rows_per_img, int nb, int N) {
  return epi.tma == 1 && N % 256 == 0 && (long long)ceil_div(rows_per_img, 256) * nb * (N / 256) >= num_sms() / 4;
}
TcShape pair_shape(const TcShape& sh, int rows_per_img, int nb, int N) {
  TcShape sp = sh;
  sp.tiles_m_per_b = ceil_div(rows_per_img, 256);
  sp.tiles_m_total = sp.tiles_m_per_b * nb;
  sp.tiles_n = N / 256;
  sp.tiles_per_unit = 1;
  sp.units = sp.tiles_m_total * sp.tiles_n;
  sp.splits = sp.tiles_n;
  sp.group_m = 0;
  return sp;
}
}  // namespace

int tc_linear_bf16(const __nv_bfloat16* A16, int lda, const __nv_bfloat16* W16, const float* bias, int bias_period,
                   const float* res, TcOut out, int M, int N, int K, int act, cudaStream_t s) {
  MOCHA_CHECK_ARG(A16 && W16 && (out.f32 || out.bf16), "tc_linear: null operand");
  MOCHA_CHECK_ARG(tc_linear_supported(M, N, K), "tc_linear: unsupported shape M=%d N=%d K=%d", M, N, K);
  CUtensorMap tmA;
  MOCHA_TRY(make_tmap(&tmA, A16, (unsigned long long)M, (unsigned long long)K, BLOCK_M, (unsigned long long)lda));
  TcShape sh{};
  sh.nb = 1;
  sh.rows_out_per_b = M;
  sh.tiles_m_per_b = ceil_div(M, BLOCK_M);
  sh.tiles_m_total = sh.tiles_m_per_b;
  sh.src_rows_per_b = M;
  sh.taps = 1;
  sh.kb_per_tap = ceil_div(K, BLOCK_K);
  sh.tap_row_stride = 0;
  LinearEpi epi{out.f32, N, N, bias, bias_period, res, act, out.bf16, out.lrelu};
  MOCHA_TRY(setup_out_tma(epi, (unsigned long long)M, 1));
  // CTA pairs (256 x 256 pair tiles, each CTA stages half of the weight rows) for the plain projections too: a 128 x 256 tile
  // of a K = 256 layer pulls 192 KB of operands per CTA from L2, a pair tile 128 KB, and these short-K launches turned out to
  // be sensitive to exactly that (same-box A/B: -15 us per step; 128-wide tiles, which re-read A twice as often: +28 us).
  if (pair_linear_wanted(epi, M, 1, N)) {
    CUtensorMap tmB;
    MOCHA_TRY(make_tmap(&tmB, W16, (unsigned long long)N, (unsigned long long)K, 128));
    return launch_pair(tmA, tmB, pair_shape(sh, M, 1, N), ceil_div(K, BLOCK_K), LinearEpiT<1>{epi}, s);
  }
  return dispatch_bn(pick_bn(sh.tiles_m_total, N, ceil_div(K, BLOCK_K)), tmA, W16, (unsigned long long)N, (unsigned long long)K, sh, N,
                     ceil_div(K, BLOCK_K), epi, s);
}

// Same GEMM over `nb` images of rows_per_img rows each (A dense [nb*rows_per_img, K]); image b's output
// rows start at out + b * out_img_pitch_rows * N, so the result can land inside a larger (e.g. time-padded)
// tensor. TMA-store epilogue only (column bias or none, one output).
int tc_linear_bf16_img(const __nv_bfloat16* A16, int lda, const __nv_bfloat16* W16, const float* bias, TcOut out, int nb,
                       int rows_per_img, long long out_img_pitch_rows, int N, int K, int act, cudaStream_t s) {
  MOCHA_CHECK_ARG(A16 && W16 && (out.f32 || out.bf16) && !(out.f32 && out.bf16), "tc_linear_img: bad operands");
  MOCHA_CHECK_ARG(tc_linear_supported(rows_per_img, N, K) && nb > 0, "tc_linear_img: unsupported shape");
  CUtensorMap tmA;
  MOCHA_TRY(make_tmap(&tmA, A16, (unsigned long long)nb * rows_per_img, (unsigned long long)K, BLOCK_M, (unsigned long long)lda));
  TcShape sh{};
  sh.nb = nb;
  sh.rows_out_per_b = rows_per_img;
  sh.tiles_m_per_b = ceil_div(rows_per_img, BLOCK_M);
  sh.tiles_m_total = sh.tiles_m_per_b * nb;
  sh.src_rows_per_b = rows_per_img;
  sh.taps = 1;
  sh.kb_per_tap = ceil_div(K, BLOCK_K);
  sh.tap_row_stride = 0;
  LinearEpi epi{out.f32, N, N, bias, 0, nullptr, act, out.bf16, out.lrelu};
  MOCHA_TRY(setup_out_tma(epi, (unsigned long long)rows_per_img, (unsigned long long)nb, 0, (unsigned long long)out_img_pitch_rows));
  if (epi.tma != 1) return set_error(MOCHA_ERR_ARG, "tc_linear_img: output is not TMA-storable");
  if (pair_linear_wanted(epi, rows_per_img, nb, N)) {
    CUtensorMap tmB;
    MOCHA_TRY(make_tmap(&tmB, W16, (unsigned long long)N, (unsigned long long)K, 128));
    return launch_pair(tmA, tmB, pair_shape(sh, rows_per_img, nb, N), ceil_div(K, BLOCK_K), LinearEpiT<1>{epi}, s);
  }
  return dispatch_bn(pick_bn(sh.tiles_m_total, N, ceil_div(K, BLOCK_K)), tmA, W16, (unsigned long long)N, (unsigned long long)K, sh, N,
                     ceil_div(K, BLOCK_K), epi, s);
}

// nb independent linear layers of one shape in ONE launch: out[g] = A[g] W[g]^T with A16 [nb, R, K], W16 [nb, N, K] and
// out16 [nb, R, N] stacked densely (the decoder's q / k / v projections: three inputs, three weights). Runs as the images
// of the batched-head mode (H = 1): image g selects its A rows, its weight rows and its output image, so the persistent
// CTAs walk nb x tiles without a launch ramp / tail per layer.
int tc_linear_bf16_grouped(const __nv_bfloat16* A16, const __nv_bfloat16* W16, __nv_bfloat16* out16, int nb, int R, int N,
                           int K, cudaStream_t s) {
  MOCHA_CHECK_ARG(A16 && W16 && out16 && nb >= 1, "tc_linear_grouped: bad operands");
  MOCHA_CHECK_ARG(tc_linear_supported(R, N, K) && N % 64 == 0, "tc_linear_grouped: unsupported shape R=%d N=%d K=%d", R, N, K);
  CUtensorMap tmA;
  MOCHA_TRY(make_tmap(&tmA, A16, (unsigned long long)nb * R, (unsigned long long)K, BLOCK_M));
  TcShape sh{};
  sh.nb = nb; sh.H = 1;
  sh.rows_out_per_b = R;
  sh.tiles_m_per_b = ceil_div(R, BLOCK_M);
  sh.tiles_m_total = sh.tiles_m_per_b * nb;
  sh.src_rows_per_b = R; sh.a_rows_h = 0; sh.a_cols_h = 0;
  sh.b_rows_b = N; sh.b_rows_h = 0; sh.b_cols_h = 0;
  sh.c_img_b = (long long)R * N; sh.c_img_h = 0;
  sh.taps = 1; sh.kb_per_tap = ceil_div(K, BLOCK_K); sh.tap_row_stride = 0;
  LinearEpi epi{nullptr, N, N, nullptr, 0, nullptr, ACT_NONE, out16, 0};
  MOCHA_TRY(setup_out_tma(epi, (unsigned long long)R, (unsigned long long)nb));
  if (epi.tma != 1) return set_error(MOCHA_ERR_ARG, "tc_linear_grouped: output is not TMA-storable");
  if (pair_linear_wanted(epi, R, nb, N)) {
    CUtensorMap tmB;
    MOCHA_TRY(make_tmap(&tmB, W16, (unsigned long long)nb * N, (unsigned long long)K, 128));
    return launch_pair(tmA, tmB, pair_shape(sh, R, nb, N), ceil_div(K, BLOCK_K), LinearEpiT<1>{epi}, s);   // sh.H = 1: per-image weights
  }
  return dispatch_bn(pick_bn(sh.tiles_m_total, N, ceil_div(K, BLOCK_K)), tmA, W16, (unsigned long long)nb * N, (unsigned long long)K, sh,
                     N, ceil_div(K, BLOCK_K), epi, s);
}

int tc_linear(const float* A, const float* W, const float* bias, int bias_period, const float* res, float* C, int M,
              int N, int K, int act, int a_lrelu, Workspace& ws, cudaStream_t s) {
  const __nv_bfloat16* W16 = tc_lookup_bf16(W);
  if (!W16) return set_error(MOCHA_ERR_ARG, "tc_linear: weight %p has no registered bf16 mirror", (const void*)W);
  const size_t mark = ws.off;
  __nv_bfloat16* A16 = ws.take<__nv_bfloat16>((size_t)M * K);
  if (!A16) return set_error(MOCHA_ERR_WORKSPACE, "tc_linear: workspace too small for the bf16 A operand");
  MOCHA_TRY(tc_cast(A, A16, (long long)M * K, a_lrelu, s));
  int rc = tc_linear_bf16(A16, K, W16, bias, bias_period, res, TcOut{C, nullptr, 0}, M, N, K, act, s);
  ws.off = mark;  // stream order makes the scratch reusable by the next layer
  return rc;
}

int tc_cast(const float* x, __nv_bfloat16* y, long long n, int lrelu, cudaStream_t s) {
  MOCHA_CHECK_ARG(x && y && n > 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0, "tc_cast: bad argument");
  launch_k(cast_act_bf16_kernel, (unsigned)((n / 4 + 255) / 256 + 1), 256, 0, s, x, y, n, lrelu);
  count_launch();
  MOCHA_LAUNCH_CHECK("cast_act_bf16");
  return MOCHA_OK;
}

// ------------------------------------------------------------------------------------------------
// 3xTF32: fp32-grade GEMMs on the tensor cores (MOCHA_TF32X3 precision mode).
//   x = hi + lo with hi = tf32(x), lo = tf32(x - hi) (both exactly representable, so the MMA's operand truncation is a
//   no-op);  a . w ~= a_hi w_hi + a_lo w_hi + a_hi w_lo  (the dropped lo x lo term is ~2^-22 relative), accumulated in
//   fp32 in TMEM. The three products run as ONE GEMM over a three times longer K: the A operand is written as
//   [hi | lo | hi] and the weights as [hi | hi | lo] per row (per tap for the temporal convolutions), so the main loop,
//   the implicit-convolution tap windows and every epilogue are the bf16 path's.
// ------------------------------------------------------------------------------------------------
namespace {

__device__ __forceinline__ float tf32_rna(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
__device__ __forceinline__ void split4(const float4& v, float4& hi, float4& lo) {
  hi.x = tf32_rna(v.x); hi.y = tf32_rna(v.y); hi.z = tf32_rna(v.z); hi.w = tf32_rna(v.w);
  lo.x = tf32_rna(v.x - hi.x); lo.y = tf32_rna(v.y - hi.y); lo.z = tf32_rna(v.z - hi.z); lo.w = tf32_rna(v.w - hi.w);
}

// two jobs in one launch: blocks [0, nblkA) split A [rowsA, K] -> [rowsA, 3K] as [hi | lo | hi], the rest split
// W [rowsW, K] -> [rowsW, 3K] as [hi | hi | lo]
__global__ void split3_kernel(const float* __restrict__ A, float* __restrict__ A3, long long rowsA, int a_lrelu,
                              const float* __restrict__ W, float* __restrict__ W3, long long rowsW, int K, int nblkA) {
  pdl_trigger();
  pdl_wait();
  const bool isw = (int)blockIdx.x >= nblkA;
  const float* x = isw ? W : A;
  float* y = isw ? W3 : A3;
  const long long rows = isw ? rowsW : rowsA;
  const int k4 = K / 4;
  const long long i4 = (long long)(isw ? blockIdx.x - nblkA : blockIdx.x) * blockDim.x + threadIdx.x;
  if (i4 >= rows * k4) return;
  const long long r = i4 / k4;
  const int c = (int)(i4 - r * k4) * 4;
  float4 v = *reinterpret_cast<const float4*>(x + r * K + c);
  if (!isw && a_lrelu) { v.x = lrelu02(v.x); v.y = lrelu02(v.y); v.z = lrelu02(v.z); v.w = lrelu02(v.w); }
  float4 hi, lo;
  split4(v, hi, lo);
  float* o = y + r * 3 * K + c;
  *reinterpret_cast<float4*>(o) = hi;
  *reinterpret_cast<float4*>(o + K) = isw ? hi : lo;
  *reinterpret_cast<float4*>(o + 2 * K) = isw ? lo : hi;
}

// X fp32 [nb, T/tdiv, V, C] -> [nb, T + 2*pad, V, 3C] reflect-padded along T, rows as [hi | lo | hi]
__global__ void reflect_pad_split3_kernel(const float* __restrict__ x, float* __restrict__ y, int T, int V, int C, int pad,
                                          int tdiv, long long total4) {
  pdl_trigger();
  pdl_wait();
  const long long i4 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i4 >= total4) return;
  const long long i = i4 * 4;
  const int c = (int)(i % C);
  const long long r = i / C;
  const int v = (int)(r % V);
  const long long bt = r / V;
  const int Tp = T + 2 * pad;
  const int tp = (int)(bt % Tp);
  const long long b = bt / Tp;
  int t = tp - pad;
  if (t < 0) t = -t;
  if (t >= T) t = 2 * (T - 1) - t;
  t /= tdiv;
  const float4 val = *reinterpret_cast<const float4*>(x + (((b * (T / tdiv) + t) * V + v) * (long long)C + c));
  float4 hi, lo;
  split4(val, hi, lo);
  float* o = y + r * 3 * C + c;
  *reinterpret_cast<float4*>(o) = hi;
  *reinterpret_cast<float4*>(o + C) = lo;
  *reinterpret_cast<float4*>(o + 2 * C) = hi;
}

constexpr int TF_K = 32;  // fp32 elements per 128-byte k-block row

}  // namespace

bool tc_linear_tf32x3_supported(int M, int N, int K) { return M >= 1 && N >= 8 && K >= 16 && (K % 4) == 0; }

int tc_linear_tf32x3(const float* A, const float* W, const float* bias, int bias_period, const float* res, float* C, int M,
                     int N, int K, int act, int a_lrelu, Workspace& ws, cudaStream_t s) {
  MOCHA_CHECK_ARG(A && W && C, "tc_linear_tf32x3: null operand");
  MOCHA_CHECK_ARG(tc_linear_tf32x3_supported(M, N, K), "tc_linear_tf32x3: unsupported shape M=%d N=%d K=%d", M, N, K);
  MOCHA_CHECK_ARG(((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(W)) & 15) == 0, "tc_linear_tf32x3: operands not 16 B aligned");
  const size_t mark = ws.off;
  const int K3 = 3 * K;
  float* W3 = ws.take<float>((size_t)N * K3);
  if (!W3) return set_error(MOCHA_ERR_WORKSPACE, "tc_linear_tf32x3: workspace too small for the split weights");
  // the split A operand takes whatever workspace is left; long problems run as row chunks (a multiple of 128 rows and of
  // the bias period, so tiles and the periodic bias keep their phase)
  const long long quantum = bias_period > 0 ? 128LL * bias_period : 128LL;
  const size_t avail = ws.cap > ws.off + 512 ? ws.cap - ws.off - 512 : 0;
  long long rows_fit = (long long)(avail / ((size_t)K3 * 4));
  if (rows_fit < M) rows_fit = rows_fit / quantum * quantum;
  if (rows_fit <= 0) return set_error(MOCHA_ERR_WORKSPACE, "tc_linear_tf32x3: workspace too small for the split A operand");
  if (rows_fit > M) rows_fit = M;
  float* A3 = ws.take<float>((size_t)rows_fit * K3);
  if (!A3) return set_error(MOCHA_ERR_WORKSPACE, "tc_linear_tf32x3: workspace too small for the split A operand");
  int rc = MOCHA_OK;
  bool w_done = false;
  for (long long m0 = 0; m0 < M && rc == MOCHA_OK; m0 += rows_fit) {
    const int mc = (int)((long long)M - m0 < rows_fit ? (long long)M - m0 : rows_fit);
    const int nblkA = (int)(((long long)mc * (K / 4) + 255) / 256);
    const int nblkW = w_done ? 0 : (int)(((long long)N * (K / 4) + 255) / 256);
    launch_k(split3_kernel, (unsigned)(nblkA + nblkW), 256, 0, s, A + m0 * K, A3, (long long)mc, a_lrelu, W, W3, (long long)N, K, nblkA);
    count_launch();
    MOCHA_LAUNCH_CHECK("split3_kernel");
    w_done = true;
    CUtensorMap tmA;
    MOCHA_TRY(make_tmap(&tmA, A3, (unsigned long long)mc, (unsigned long long)K3, BLOCK_M, 0, true));
    TcShape sh{};
    sh.nb = 1;
    sh.rows_out_per_b = mc;
    sh.tiles_m_per_b = ceil_div(mc, BLOCK_M);
    sh.tiles_m_total = sh.tiles_m_per_b;
    sh.src_rows_per_b = mc;
    sh.taps = 1;
    sh.kb_per_tap = ceil_div(K3, TF_K);
    sh.tap_row_stride = 0;
    LinearEpi epi{C + m0 * N, N, N, bias, bias_period, res ? res + m0 * N : nullptr, act, nullptr, 0};
    MOCHA_TRY(setup_out_tma(epi, (unsigned long long)mc, 1));
    rc = dispatch_bn_tf32(pick_bn(sh.tiles_m_total, N, sh.kb_per_tap), tmA, W3, (unsigned long long)N, (unsigned long long)K3, sh, N,
                          sh.kb_per_tap, epi, s);
  }
  ws.off = mark;
  return rc;
}

bool tc_tconv_tf32x3_supported(int B, int T, int V, int Cin, int Cout, int taps) {
  return B >= 1 && (Cin % TF_K) == 0 && Cout >= 8 && (taps & 1) && taps / 2 < T && (long long)T * V >= 1;
}

int tc_tconv_tf32x3(const float* X, const float* W, const float* bias, int bias_period, float* C, int B, int T, int V, int Cin,
                    int Cout, int taps, int tdiv, Workspace& ws, cudaStream_t s) {
  MOCHA_CHECK_ARG(X && W && C, "tc_tconv_tf32x3: null operand");
  MOCHA_CHECK_ARG(tdiv >= 1 && T % tdiv == 0, "tc_tconv_tf32x3: T=%d not a multiple of tdiv=%d", T, tdiv);
  MOCHA_CHECK_ARG(tc_tconv_tf32x3_supported(B, T, V, Cin, Cout, taps), "tc_tconv_tf32x3: unsupported geometry");
  MOCHA_CHECK_ARG(bias_period == 0 || (T * V) % bias_period == 0, "tc_tconv_tf32x3: bias period does not divide an image");
  const int pad = taps / 2, Tp = T + 2 * pad, C3 = 3 * Cin;
  const size_t mark = ws.off;
  // weights [Cout, taps * Cin] (tap-major K) -> [Cout, taps * 3 Cin], [hi | hi | lo] per tap
  float* W3 = ws.take<float>((size_t)Cout * taps * C3);
  if (!W3) return set_error(MOCHA_ERR_WORKSPACE, "tc_tconv_tf32x3: workspace too small for the split weights");
  const size_t img_bytes = (size_t)Tp * V * C3 * 4;
  const size_t avail = ws.cap > ws.off + 512 ? ws.cap - ws.off - 512 : 0;
  int imgs_fit = (int)(avail / img_bytes < (size_t)B ? avail / img_bytes : (size_t)B);
  if (imgs_fit <= 0) return set_error(MOCHA_ERR_WORKSPACE, "tc_tconv_tf32x3: workspace too small for the padded split operand");
  float* X3 = ws.take<float>((size_t)imgs_fit * Tp * V * C3);
  if (!X3) return set_error(MOCHA_ERR_WORKSPACE, "tc_tconv_tf32x3: workspace too small for the padded split operand");
  {
    const long long rowsW = (long long)Cout * taps;
    const int nblkW = (int)((rowsW * (Cin / 4) + 255) / 256);
    launch_k(split3_kernel, (unsigned)nblkW, 256, 0, s, (const float*)nullptr, (float*)nullptr, 0LL, 0, W, W3, rowsW, Cin, 0);
    count_launch();
    MOCHA_LAUNCH_CHECK("split3_kernel");
  }
  int rc = MOCHA_OK;
  for (int b0 = 0; b0 < B && rc == MOCHA_OK; b0 += imgs_fit) {
    const int nb = B - b0 < imgs_fit ? B - b0 : imgs_fit;
    const long long total4 = (long long)nb * Tp * V * Cin / 4;
    launch_k(reflect_pad_split3_kernel, (unsigned)((total4 + 255) / 256), 256, 0, s,
             X + (long long)b0 * (T / tdiv) * V * Cin, X3, T, V, Cin, pad, tdiv, total4);
    count_launch();
    MOCHA_LAUNCH_CHECK("reflect_pad_split3_kernel");
    CUtensorMap tmA;
    MOCHA_TRY(make_tmap(&tmA, X3, (unsigned long long)nb * Tp * V, (unsigned long long)C3, BLOCK_M, 0, true));
    TcShape sh{};
    sh.nb = nb;
    sh.rows_out_per_b = T * V;
    sh.tiles_m_per_b = ceil_div(T * V, BLOCK_M);
    sh.tiles_m_total = sh.tiles_m_per_b * nb;
    sh.src_rows_per_b = (long long)Tp * V;
    sh.taps = taps;
    sh.kb_per_tap = C3 / TF_K;
    sh.tap_row_stride = V;
    LinearEpi epi{C + (long long)b0 * T * V * Cout, Cout, Cout, bias, bias_period, nullptr, ACT_NONE, nullptr, 0};
    MOCHA_TRY(setup_out_tma(epi, (unsigned long long)T * V, (unsigned long long)nb));
    rc = dispatch_bn_tf32(pick_bn(sh.tiles_m_total, Cout, taps * sh.kb_per_tap), tmA, W3, (unsigned long long)Cout,
                          (unsigned long long)taps * C3, sh, Cout, taps * sh.kb_per_tap, epi, s);
  }
  ws.off = mark;
  return rc;
}

bool tc_tconv_supported(int B, int T, int V, int Cin, int Cout, int taps) {
  return B >= 1 && (Cin % BLOCK_K) == 0 && Cout >= 8 && (taps & 1) && taps / 2 < T && (long long)T * V >= 1;
}
size_t tc_tconv_scratch_bytes(int B, int T, int V, int Cin, int taps) {
  if (g_ws_precision == MOCHA_TF32X3)
    return align_up(((size_t)B * (T + 2 * (taps / 2)) * V + (size_t)2048 * taps) * Cin * 12, 256) + 1024;
  return align_up((size_t)B * (T + 2 * (taps / 2)) * V * Cin * 2, 256) + 256;
}

int tc_tconv(const float* X, const float* W, const float* bias, int bias_period, float* C, int B, int T, int V,
             int Cin, int Cout, int taps, int tdiv, Workspace& ws, cudaStream_t s, int repeat) {
  return tc_tconv_ex(X, nullptr, W, bias, bias_period, TcOut{C, nullptr, 0}, B, T, V, Cin, Cout, taps, tdiv, ws, s, repeat);
}

int tc_tconv_ex(const float* X, const __nv_bfloat16* Xh, const float* W, const float* bias, int bias_period, TcOut out,
                int B, int T, int V, int Cin, int Cout, int taps, int tdiv, Workspace& ws, cudaStream_t s, int repeat,
                bool xh_is_padded) {
  MOCHA_CHECK_ARG((X || Xh) && (out.f32 || out.bf16), "tc_tconv: null operand");
  MOCHA_CHECK_ARG(tdiv >= 1 && T % tdiv == 0, "tc_tconv: T=%d not a multiple of tdiv=%d", T, tdiv);
  MOCHA_CHECK_ARG(tc_tconv_supported(B, T, V, Cin, Cout, taps), "tc_tconv: unsupported geometry");
  const __nv_bfloat16* W16 = tc_lookup_bf16(W);
  if (!W16) return set_error(MOCHA_ERR_ARG, "tc_tconv: weight %p has no registered bf16 mirror", (const void*)W);
  const int pad = taps / 2, Tp = T + 2 * pad;
  const size_t mark = ws.off;
  const size_t elems = (size_t)B * Tp * V * Cin;
  MOCHA_CHECK_ARG(!xh_is_padded || (Xh && tdiv == 1), "tc_tconv: a pre-padded operand must be bf16 with tdiv = 1");
  const __nv_bfloat16* X16c = xh_is_padded ? Xh : nullptr;   // [B, Tp, V, Cin] reflect-padded by the producer
  __nv_bfloat16* X16 = xh_is_padded ? nullptr : ws.take<__nv_bfloat16>(elems);
  if (!xh_is_padded && !X16) return set_error(MOCHA_ERR_WORKSPACE, "tc_tconv: workspace too small for the padded bf16 operand");
  if (xh_is_padded) {
  } else if (Xh)
    launch_k(reflect_pad_copy_kernel, (unsigned)((elems / 8 + 255) / 256), 256, 0, s, Xh, X16, T, V, Cin, pad, tdiv,
                                                                               (long long)(elems / 8));
  else
    launch_k(reflect_pad_cast_kernel, (unsigned)((elems / 4 + 255) / 256), 256, 0, s, X, X16, T, V, Cin, pad, tdiv,
                                                                               (long long)(elems / 4));
  if (!xh_is_padded) {
    count_launch();
    MOCHA_LAUNCH_CHECK("reflect_pad_cast");
    X16c = X16;
  }
  CUtensorMap tmA;
  MOCHA_TRY(make_tmap(&tmA, X16c, (unsigned long long)B * Tp * V, (unsigned long long)Cin, BLOCK_M));
  TcShape sh{};
  sh.nb = B;
  sh.rows_out_per_b = T * V;
  sh.tiles_m_per_b = ceil_div(T * V, BLOCK_M);
  sh.tiles_m_total = sh.tiles_m_per_b * B;
  sh.src_rows_per_b = (long long)Tp * V;
  sh.taps = taps;
  sh.kb_per_tap = Cin / BLOCK_K;
  sh.tap_row_stride = V;
  LinearEpi epi{out.f32, Cout, Cout, bias, bias_period, nullptr, ACT_NONE, out.bf16, out.lrelu};
  MOCHA_TRY(setup_out_tma(epi, (unsigned long long)T * V, (unsigned long long)B));
  int rc = MOCHA_OK;
  // long-K, wide-N convolutions are bound by the shared-memory fill rate (~64 B/clk/SM) with 128 x 256
  // tiles: a CTA pair (cta_group::2) stages half of the weight rows each and runs 256 x 256 tiles
  const int pair_tiles = ceil_div(T * V, 256) * B;
  // images shorter than a pair tile (BodyBlock convs: 90 rows per clip) would run 256-row tiles that are mostly padding:
  // those keep the 1-CTA kernel's 128-row tiles
  const bool pair_fill_ok = ceil_div(T * V, 256) * 256 <= ceil_div(T * V, BLOCK_M) * BLOCK_M;
  if (pair_fill_ok && epi.tma == 1 && Cout % 256 == 0 && taps * sh.kb_per_tap >= 8 && pair_tiles >= num_sms() / 2) {
    CUtensorMap tmB;
    MOCHA_TRY(make_tmap(&tmB, W16, (unsigned long long)Cout, (unsigned long long)taps * Cin, 128));
    TcShape sp = sh;
    sp.tiles_m_per_b = ceil_div(T * V, 256);
    sp.tiles_m_total = sp.tiles_m_per_b * B;
    sp.tiles_n = Cout / 256;
    sp.tiles_per_unit = 1;
    sp.units = sp.tiles_m_total * sp.tiles_n;
    sp.splits = sp.tiles_n;
    sp.group_m = 0;
    for (int it = 0; it < (repeat < 1 ? 1 : repeat) && rc == MOCHA_OK; ++it)
      rc = launch_pair(tmA, tmB, sp, taps * sh.kb_per_tap, LinearEpiT<1>{epi}, s);
    ws.off = mark;
    return rc;
  }
  // 64 -> 64 channels, 5 taps, 24 rows per frame (to_mot's JointBlock conv): one 224-row box per tile serves all taps and the
  // weights stay resident (halo variant)
  if (epi.tma == 1 && !epi.C && epi.C16 && Cin == BLOCK_K && Cout == 64 && taps == HALO_TAPS && V == HALO_SHIFT &&
      bias_period == 0 && sh.tiles_m_total >= num_sms()) {
    CUtensorMap tmAh, tmB;
    MOCHA_TRY(make_tmap(&tmAh, X16c, (unsigned long long)B * Tp * V, (unsigned long long)Cin, HALO_ROWS));
    MOCHA_TRY(make_tmap(&tmB, W16, (unsigned long long)Cout, (unsigned long long)taps * Cin, 64));
    TcShape sp = sh;
    sp.tiles_n = 1; sp.tiles_per_unit = 1; sp.units = sp.tiles_m_total; sp.splits = 1; sp.group_m = 0;
    LinearEpi e2 = epi;
    e2.c16_wide = 0;   // a warp owns one 32-column chunk of the 64-wide tile
    for (int it = 0; it < (repeat < 1 ? 1 : repeat) && rc == MOCHA_OK; ++it)
      rc = launch_tc_halo<64, LinearEpiT<4>>(tmAh, tmB, sp, LinearEpiT<4>{e2}, s);
    ws.off = mark;
    return rc;
  }
  for (int it = 0; it < (repeat < 1 ? 1 : repeat) && rc == MOCHA_OK; ++it)  // repeat > 1: bench.py roofline pass
    rc = dispatch_bn(pick_bn(sh.tiles_m_total, Cout), tmA, W16, (unsigned long long)Cout,
                     (unsigned long long)taps * Cin, sh, Cout, taps * sh.kb_per_tap, epi, s);
  ws.off = mark;
  return rc;
}

// ------------------------------------------------------------------------------------------------
// attention on tensor cores: batched-head QK^T -> softmax (bf16 P) -> batched-head PV
// ------------------------------------------------------------------------------------------------
namespace {

// fp32 [rows, cols] view with row pitch ld -> compact bf16 [rows, cols]
__global__ void cast_strided_bf16_kernel(const float* __restrict__ x, int ld, int cols, long long total4,
                                         __nv_bfloat16* __restrict__ y) {
  pdl_trigger();
  pdl_wait();
  const long long i4 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i4 >= total4) return;
  const int c4 = cols >> 2;
  const long long r = i4 / c4;
  const int c = (int)(i4 - r * c4) * 4;
  const float4 v = *reinterpret_cast<const float4*>(x + r * (long long)ld + c);
  __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
  uint2 pk;
  pk.x = *reinterpret_cast<uint32_t*>(&lo);
  pk.y = *reinterpret_cast<uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(y + r * (long long)cols + c) = pk;
}

// V fp32 [B*nkv, ldv] (head h at columns h*dh..) -> VT bf16 [B*H, dh, ldp] (kv contiguous, zero padded)
__device__ __forceinline__ float to_f32(float x) { return x; }
__device__ __forceinline__ float to_f32(__nv_bfloat16 x) { return __bfloat162float(x); }
template <typename TV>
__global__ void transpose_v_bf16_kernel(const TV* __restrict__ v, int ldv, int H, int nkv, int dh, int ldp,
                                        __nv_bfloat16* __restrict__ vt) {
  pdl_trigger();
  pdl_wait();
  __shared__ float tile[32][33];
  const int z = blockIdx.z, b = z / H, h = z - b * H;
  const int j0 = blockIdx.x * 32, d0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int i = ty; i < 32; i += 8) {
    const int j = j0 + i, d = d0 + tx;
    tile[i][tx] = (j < nkv && d < dh) ? to_f32(v[((long long)b * nkv + j) * ldv + h * dh + d]) : 0.f;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int d = d0 + i, j = j0 + tx;
    if (d < dh && j < ldp) vt[((long long)z * dh + d) * ldp + j] = __float2bfloat16_rn(tile[tx][i]);
  }
}

}  // namespace

bool tc_attention_supported(int nq, int nkv, int dh) {
  return nq >= 1 && nkv >= 1 && nkv <= 256 && dh >= 64 && (dh % 64) == 0;
}

static int attn_ldp(int nkv) { return (nkv + 7) / 8 * 8; }

size_t tc_attention_tf32x3_scratch_bytes(int B, int H, int nq, int nkv, int dh);
size_t tc_attention_scratch_bytes(int B, int H, int nq, int nkv, int dh) {
  if (g_ws_precision == MOCHA_TF32X3) return tc_attention_tf32x3_scratch_bytes(B, H, nq, nkv, dh);
  const size_t Z = (size_t)B * H, ldp = attn_ldp(nkv);
  return align_up((size_t)B * nq * H * dh * 2, 256) + align_up((size_t)B * nkv * H * dh * 2, 256) +
         align_up(Z * dh * ldp * 2, 256) + align_up(Z * nq * ldp * 2, 256) + align_up(Z * nq * 4, 256) + 1024;
}

int tc_attention(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv, int B, int H, int nq,
                 int nkv, int dh, float* S, float* out, int ldo, Workspace& ws, cudaStream_t s) {
  return tc_attention_ex(q, nullptr, ldq, k, nullptr, ldk, v, nullptr, ldv, B, H, nq, nkv, dh, S, TcOut{out, nullptr, 0},
                         ldo, ws, s);
}

// Operands may be given as fp32 views (cast / transposed into scratch) or directly as bf16 views
// (qh/kh feed the TMA descriptors in place through their row pitch; vh is transposed from bf16).
int tc_attention_ex(const float* q, const __nv_bfloat16* qh, int ldq, const float* k, const __nv_bfloat16* kh, int ldk,
                    const float* v, const __nv_bfloat16* vh, int ldv, int B, int H, int nq, int nkv, int dh, float* S,
                    TcOut out, int ldo, Workspace& ws, cudaStream_t s) {
  MOCHA_CHECK_ARG(tc_attention_supported(nq, nkv, dh), "tc_attention: unsupported geometry nq=%d nkv=%d dh=%d", nq, nkv, dh);
  MOCHA_CHECK_ARG((q || qh) && (k || kh) && (v || vh) && (out.f32 || out.bf16), "tc_attention: null operand");
  const int inner = H * dh, Z = B * H, ldp = attn_ldp(nkv);
  const size_t mark = ws.off;
  const __nv_bfloat16* Q16 = qh;
  const __nv_bfloat16* K16 = kh;
  int pq = ldq, pk = ldk;
  if (!qh) {
    MOCHA_CHECK_ARG((ldq & 3) == 0 && ((uintptr_t)q & 15) == 0, "tc_attention: q view must be 16 B aligned");
    __nv_bfloat16* t = ws.take<__nv_bfloat16>((size_t)B * nq * inner);
    if (!t) return set_error(MOCHA_ERR_WORKSPACE, "tc_attention: workspace too small");
    const long long t4 = (long long)B * nq * inner / 4;
    launch_k(cast_strided_bf16_kernel, (unsigned)((t4 + 255) / 256), 256, 0, s, q, ldq, inner, t4, t);
    count_launch();
    Q16 = t; pq = inner;
  }
  if (!kh) {
    MOCHA_CHECK_ARG((ldk & 3) == 0 && ((uintptr_t)k & 15) == 0, "tc_attention: k view must be 16 B aligned");
    __nv_bfloat16* t = ws.take<__nv_bfloat16>((size_t)B * nkv * inner);
    if (!t) return set_error(MOCHA_ERR_WORKSPACE, "tc_attention: workspace too small");
    const long long u4 = (long long)B * nkv * inner / 4;
    launch_k(cast_strided_bf16_kernel, (unsigned)((u4 + 255) / 256), 256, 0, s, k, ldk, inner, u4, t);
    count_launch();
    K16 = t; pk = inner;
  }
  const bool v_in_place = vh != nullptr && (ldv % 8) == 0 && (reinterpret_cast<uintptr_t>(vh) & 15) == 0;
  __nv_bfloat16* VT16 = v_in_place ? nullptr : ws.take<__nv_bfloat16>((size_t)Z * dh * ldp);
  __nv_bfloat16* P16 = ws.take<__nv_bfloat16>((size_t)Z * nq * ldp);
  float* inv_sum = ws.take<float>((size_t)Z * nq);
  if (ws.overflow) return set_error(MOCHA_ERR_WORKSPACE, "tc_attention: workspace too small");
  MOCHA_CHECK_ARG(ldo == H * dh && (ldo % 8) == 0 && ((reinterpret_cast<uintptr_t>(out.f32) | reinterpret_cast<uintptr_t>(out.bf16)) & 15) == 0,
                  "tc_attention: output must be a dense, 16 B-aligned [B, nq, H*dh] tensor");
  if (!v_in_place) {
    dim3 g((ldp + 31) / 32, (dh + 31) / 32, Z);
    if (vh) launch_k(transpose_v_bf16_kernel<__nv_bfloat16>, g, 256, 0, s, vh, ldv, H, nkv, dh, ldp, VT16);
    else launch_k(transpose_v_bf16_kernel<float>, g, 256, 0, s, v, ldv, H, nkv, dh, ldp, VT16);
    count_launch();
    MOCHA_LAUNCH_CHECK("attention staging");
  }
  // scores S[z] = Q[z] K[z]^T  (fp32, [Z, nq, nkv])
  {
    CUtensorMap tmA;
    MOCHA_TRY(make_tmap(&tmA, Q16, (unsigned long long)B * nq, (unsigned long long)inner, BLOCK_M, (unsigned long long)pq));
    TcShape sh{};
    sh.nb = Z; sh.H = H;
    sh.rows_out_per_b = nq;
    sh.tiles_m_per_b = ceil_div(nq, BLOCK_M);
    sh.tiles_m_total = sh.tiles_m_per_b * Z;
    sh.src_rows_per_b = nq; sh.a_rows_h = 0; sh.a_cols_h = dh;
    sh.b_rows_b = nkv; sh.b_rows_h = 0; sh.b_cols_h = dh;
    sh.c_img_b = (long long)H * nq * nkv; sh.c_img_h = (long long)nq * nkv;
    sh.taps = 1; sh.kb_per_tap = dh / BLOCK_K; sh.tap_row_stride = 0;
    // softmax fused into the epilogue: one tile spans every key of its rows, P goes out through TMA
    SoftmaxEpi epi{};
    epi.scale_log2e = 1.4426950408889634f / sqrtf((float)dh);
    epi.nkv = nkv;
    epi.ldp = ldp;
    epi.nq = nq;
    epi.inv_sum = inv_sum;
    MOCHA_TRY(make_out_tmap(&epi.tmP, P16, (unsigned long long)ldp, (unsigned long long)nq, (unsigned long long)Z,
                            (unsigned long long)ldp, false));
    const int bn = nkv <= 32 ? 32 : nkv <= 64 ? 64 : nkv <= 128 ? 128 : 256;
    MOCHA_TRY(dispatch_bn_impl(bn, tmA, K16, (unsigned long long)B * nkv, (unsigned long long)inner, sh, nkv,
                               dh / BLOCK_K, epi, s, (unsigned long long)pk));
  }
  (void)S;  // scores no longer round-trip through HBM
  // out[b, :, h*dh:(h+1)*dh] = P[z] V[z]
  {
    CUtensorMap tmA;
    MOCHA_TRY(make_tmap(&tmA, P16, (unsigned long long)Z * nq, (unsigned long long)ldp, BLOCK_M));
    TcShape sh{};
    sh.nb = Z; sh.H = H;
    sh.rows_out_per_b = nq;
    sh.tiles_m_per_b = ceil_div(nq, BLOCK_M);
    sh.tiles_m_total = sh.tiles_m_per_b * Z;
    sh.src_rows_per_b = (long long)H * nq; sh.a_rows_h = nq; sh.a_cols_h = 0;
    sh.b_rows_b = (long long)H * dh; sh.b_rows_h = dh; sh.b_cols_h = 0;
    sh.c_img_b = (long long)nq * ldo; sh.c_img_h = dh;
    sh.taps = 1; sh.kb_per_tap = ceil_div(ldp, BLOCK_K); sh.tap_row_stride = 0;
    LinearEpi epi{out.f32, ldo, dh, nullptr, 0, nullptr, ACT_NONE, out.bf16, out.lrelu};
    // out is [B, nq, H*dh] with the head as a column offset: one {ldo, nq, B} map serves every head
    epi.row_scale = inv_sum;
    epi.rs_rows = nq;
    MOCHA_TRY(setup_out_tma(epi, (unsigned long long)nq, (unsigned long long)B, (unsigned long long)ldo));
    if (epi.tma != 1) return set_error(MOCHA_ERR_ARG, "tc_attention: TMA-store epilogue unavailable for the output");
    if (v_in_place) {
      // V is read where the projection left it: [B*nkv tokens, H*dh] with the head as a column offset
      sh.b_mn = 1;
      sh.b_rows_b = nkv; sh.b_rows_h = 0; sh.b_cols_h = dh;
      MOCHA_TRY(dispatch_bn(dh >= 256 ? 256 : dh >= 128 ? 128 : 64, tmA, vh, (unsigned long long)B * nkv,
                            (unsigned long long)inner, sh, dh, ceil_div(ldp, BLOCK_K), epi, s, (unsigned long long)ldv));
    } else {
      MOCHA_TRY(dispatch_bn(pick_bn(sh.tiles_m_total, dh), tmA, VT16, (unsigned long long)Z * dh,
                            (unsigned long long)ldp, sh, dh, ceil_div(ldp, BLOCK_K), epi, s));
    }
  }
  ws.off = mark;
  return MOCHA_OK;
}

// ------------------------------------------------------------------------------------------------
// attention in the 3xTF32 parity mode: Q K^T and P V as split-fp32 batched-head GEMMs (same [hi | lo | hi] x [hi | hi | lo]
// K-concatenation as tc_linear_tf32x3, per head), softmax in fp32 between them (softmax_rows_kernel via the caller's S)
// ------------------------------------------------------------------------------------------------
namespace {

// x [rows, ld] with head h at columns h*dh -> y [rows, H*3dh], per head [hi | lo | hi] (w_order = 0) or [hi | hi | lo] (1)
__global__ void split3_heads_kernel(const float* __restrict__ x, int ld, int H, int dh, long long total4, int w_order,
                                    float* __restrict__ y) {
  pdl_trigger();
  pdl_wait();
  const long long i4 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i4 >= total4) return;
  const int d4 = dh / 4, inner4 = H * d4;
  const long long r = i4 / inner4;
  const int rem = (int)(i4 - r * inner4), h = rem / d4, c = (rem - h * d4) * 4;
  const float4 v = *reinterpret_cast<const float4*>(x + r * ld + h * dh + c);
  float4 hi, lo;
  split4(v, hi, lo);
  float* o = y + (r * H + h) * 3 * dh + c;
  *reinterpret_cast<float4*>(o) = hi;
  *reinterpret_cast<float4*>(o + dh) = w_order ? hi : lo;
  *reinterpret_cast<float4*>(o + 2 * dh) = w_order ? lo : hi;
}

// P [rows, n] -> [rows, 3 kp] as [hi | lo | hi], each part zero-padded from n to kp columns
__global__ void split3_pad_rows_kernel(const float* __restrict__ x, int n, int kp, long long total, float* __restrict__ y) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long r = i / kp;
  const int j = (int)(i - r * kp);
  const float v = j < n ? x[r * n + j] : 0.f;
  const float hi = tf32_rna(v), lo = tf32_rna(v - hi);
  float* o = y + r * 3 * kp + j;
  o[0] = hi; o[kp] = lo; o[2 * kp] = hi;
}

// v view [B*nkv, ldv] (head h at columns h*dh) -> Vt3 [Z*dh, 3 kp]: row (z, d) = [hi | hi | lo] of v[b, :, h*dh + d], padded to kp
__global__ void transpose_split3_v_kernel(const float* __restrict__ v, int ldv, int H, int nkv, int dh, int kp,
                                          float* __restrict__ vt) {
  pdl_trigger();
  pdl_wait();
  __shared__ float tile[32][33];
  const int z = blockIdx.z, b = z / H, h = z - b * H;
  const int j0 = blockIdx.x * 32, d0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int i = ty; i < 32; i += 8) {
    const int j = j0 + i, d = d0 + tx;
    tile[i][tx] = (j < nkv && d < dh) ? v[((long long)b * nkv + j) * ldv + h * dh + d] : 0.f;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int d = d0 + i, j = j0 + tx;
    if (d < dh && j < kp) {
      const float x = tile[tx][i];
      const float hi = tf32_rna(x), lo = tf32_rna(x - hi);
      float* o = vt + ((long long)z * dh + d) * 3 * kp + j;
      o[0] = hi; o[kp] = hi; o[2 * kp] = lo;
    }
  }
}

inline int attn_kp(int nkv) { return (nkv + 3) / 4 * 4; }

}  // namespace

bool tc_attention_tf32x3_supported(int nq, int nkv, int dh) {
  return nq >= 1 && nkv >= 1 && nkv <= 256 && dh >= 32 && (dh % 32) == 0;
}

size_t tc_attention_tf32x3_scratch_bytes(int B, int H, int nq, int nkv, int dh) {
  const size_t Z = (size_t)B * H, kp = attn_kp(nkv), inner3 = (size_t)H * 3 * dh;
  return align_up((size_t)B * nq * inner3 * 4, 256) + align_up((size_t)B * nkv * inner3 * 4, 256) +
         align_up(Z * nq * 3 * kp * 4, 256) + align_up(Z * dh * 3 * kp * 4, 256) + 1024;
}

int tc_attention_tf32x3(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv, int B, int H, int nq, int nkv,
                        int dh, float* S, float* out, int ldo, Workspace& ws, cudaStream_t s) {
  MOCHA_CHECK_ARG(tc_attention_tf32x3_supported(nq, nkv, dh), "tc_attention_tf32x3: unsupported geometry nq=%d nkv=%d dh=%d", nq, nkv, dh);
  MOCHA_CHECK_ARG(q && k && v && S && out, "tc_attention_tf32x3: null operand");
  MOCHA_CHECK_ARG(((ldq | ldk) & 3) == 0 && ((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k)) & 15) == 0,
                  "tc_attention_tf32x3: q / k views must be 16 B aligned");
  const int inner = H * dh, inner3 = 3 * inner, Z = B * H, kp = attn_kp(nkv);
  const size_t mark = ws.off;
  float* Q3 = ws.take<float>((size_t)B * nq * inner3);
  float* K3 = ws.take<float>((size_t)B * nkv * inner3);
  float* P3 = ws.take<float>((size_t)Z * nq * 3 * kp);
  float* V3 = ws.take<float>((size_t)Z * dh * 3 * kp);
  if (ws.overflow) { ws.off = mark; ws.overflow = false; return set_error(MOCHA_ERR_WORKSPACE, "tc_attention_tf32x3: workspace too small"); }
  {
    const long long tq = (long long)B * nq * inner / 4, tk = (long long)B * nkv * inner / 4;
    launch_k(split3_heads_kernel, (unsigned)((tq + 255) / 256), 256, 0, s, q, ldq, H, dh, tq, 0, Q3);
    launch_k(split3_heads_kernel, (unsigned)((tk + 255) / 256), 256, 0, s, k, ldk, H, dh, tk, 1, K3);
    dim3 g((kp + 31) / 32, (dh + 31) / 32, Z);
    launch_k(transpose_split3_v_kernel, g, 256, 0, s, v, ldv, H, nkv, dh, kp, V3);
    count_launch(3);
    MOCHA_LAUNCH_CHECK("attention tf32x3 staging");
  }
  // scores S[z] = Q[z] K[z]^T (fp32, [Z, nq, nkv])
  {
    CUtensorMap tmA;
    MOCHA_TRY(make_tmap(&tmA, Q3, (unsigned long long)B * nq, (unsigned long long)inner3, BLOCK_M, 0, true));
    TcShape sh{};
    sh.nb = Z; sh.H = H;
    sh.rows_out_per_b = nq;
    sh.tiles_m_per_b = ceil_div(nq, BLOCK_M);
    sh.tiles_m_total = sh.tiles_m_per_b * Z;
    sh.src_rows_per_b = nq; sh.a_rows_h = 0; sh.a_cols_h = 3 * dh;
    sh.b_rows_b = nkv; sh.b_rows_h = 0; sh.b_cols_h = 3 * dh;
    sh.c_img_b = (long long)H * nq * nkv; sh.c_img_h = (long long)nq * nkv;
    sh.taps = 1; sh.kb_per_tap = 3 * dh / TF_K; sh.tap_row_stride = 0;
    LinearEpi epi{S, nkv, nkv, nullptr, 0, nullptr, ACT_NONE, nullptr, 0};
    epi.tma = 0;   // batched-head score blocks: LSU epilogue
    const int bn = nkv <= 32 ? 32 : nkv <= 64 ? 64 : nkv <= 128 ? 128 : 256;
    MOCHA_TRY(dispatch_bn_tf32(bn, tmA, K3, (unsigned long long)B * nkv, (unsigned long long)inner3, sh, nkv, sh.kb_per_tap, epi, s));
  }
  {
    // softmax over the keys, in place (fp32), then the split / padded A operand of the second GEMM
    MOCHA_TRY(softmax_rows(S, (long long)Z * nq, nkv, 1.0f / sqrtf((float)dh), s));
    const long long tp = (long long)Z * nq * kp;
    launch_k(split3_pad_rows_kernel, (unsigned)((tp + 255) / 256), 256, 0, s, (const float*)S, nkv, kp, tp, P3);
    count_launch();
    MOCHA_LAUNCH_CHECK("split3_pad_rows");
  }
  // out[b, :, h*dh:(h+1)*dh] = P[z] V[z]
  {
    CUtensorMap tmA;
    MOCHA_TRY(make_tmap(&tmA, P3, (unsigned long long)Z * nq, (unsigned long long)3 * kp, BLOCK_M, 0, true));
    TcShape sh{};
    sh.nb = Z; sh.H = H;
    sh.rows_out_per_b = nq;
    sh.tiles_m_per_b = ceil_div(nq, BLOCK_M);
    sh.tiles_m_total = sh.tiles_m_per_b * Z;
    sh.src_rows_per_b = (long long)H * nq; sh.a_rows_h = nq; sh.a_cols_h = 0;
    sh.b_rows_b = (long long)H * dh; sh.b_rows_h = dh; sh.b_cols_h = 0;
    sh.c_img_b = (long long)nq * ldo; sh.c_img_h = dh;
    sh.taps = 1; sh.kb_per_tap = ceil_div(3 * kp, TF_K); sh.tap_row_stride = 0;
    LinearEpi epi{out, ldo, dh, nullptr, 0, nullptr, ACT_NONE, nullptr, 0};
    if (ldo == H * dh) MOCHA_TRY(setup_out_tma(epi, (unsigned long long)nq, (unsigned long long)B, (unsigned long long)ldo));
    else epi.tma = 0;
    MOCHA_TRY(dispatch_bn_tf32(pick_bn(sh.tiles_m_total, dh), tmA, V3, (unsigned long long)Z * dh, (unsigned long long)3 * kp, sh, dh,
                               sh.kb_per_tap, epi, s));
  }
  ws.off = mark;
  return MOCHA_OK;
}

int tc_match_splits(int nq, long long N) {
  const int tiles_m = ceil_div(nq, BLOCK_M);
  const long long tiles_n = (N + 255) / 256;
  // ~8 units per SM for balance, but never more splits than n-tiles
  long long splits = (8LL * num_sms() + tiles_m - 1) / tiles_m;
  if (splits > tiles_n) splits = tiles_n;
  if (splits < 1) splits = 1;
  // recompute so that every split is non-empty
  const long long tpu = (tiles_n + splits - 1) / splits;
  splits = (tiles_n + tpu - 1) / tpu;
  return (int)splits * 2;  // x2: the two column halves of a tile keep separate lists
}

// fp32-storage variant: queries and DB rows stay fp32 in HBM and are consumed as TF32 by tcgen05
// (kind::tf32, K = 8 per instruction; 32 elements per 128-byte k-block row)
int tc_match_coarse_tf32(const float* Q, int nq, const float* DB, const float* dbnorm, long long N, int D, int kc,
                         float* cand_score, int32_t* cand_idx, cudaStream_t s) {
  MOCHA_CHECK_ARG(Q && DB && dbnorm && cand_score && cand_idx, "tc_match_coarse_tf32: null operand");
  MOCHA_CHECK_ARG(nq > 0 && N > 0 && N < 2147483647LL, "tc_match_coarse_tf32: bad sizes nq=%d N=%lld", nq, N);
  MOCHA_CHECK_ARG(D >= 32 && D % 4 == 0, "tc_match_coarse_tf32: D=%d must be >= 32 and a multiple of 4", D);
  MOCHA_CHECK_ARG(kc == 4 || kc == 8 || kc == 16, "tc_match_coarse_tf32: kc must be 4, 8 or 16");
  constexpr int BN = 256;
  CUtensorMap tmA, tmB;
  MOCHA_TRY(make_tmap(&tmA, Q, (unsigned long long)nq, (unsigned long long)D, BLOCK_M, 0, true));
  MOCHA_TRY(make_tmap(&tmB, DB, (unsigned long long)N, (unsigned long long)D, BN, 0, true));
  TcShape sh{};
  sh.nb = 1;
  sh.rows_out_per_b = nq;
  sh.tiles_m_per_b = ceil_div(nq, BLOCK_M);
  sh.tiles_m_total = sh.tiles_m_per_b;
  sh.src_rows_per_b = nq;
  sh.taps = 1;
  sh.kb_per_tap = ceil_div(D, 32);
  sh.tiles_n = (int)((N + BN - 1) / BN);
  const int splits = tc_match_splits(nq, N) / 2;
  sh.tiles_per_unit = ceil_div(sh.tiles_n, splits);
  sh.units = sh.tiles_m_total * splits;
  sh.splits = splits;
  {
    long long gm = (64LL << 20) / ((long long)BLOCK_M * D * 4);
    if (gm < 1) gm = 1;
    for (long long d = gm; d >= 1; --d)
      if (sh.tiles_m_total % d == 0) { if (2 * d > gm) gm = d; break; }
    sh.group_m = (int)gm;
  }
  const int num_kb = ceil_div(D, 32);
  if (kc == 4) return launch_tc<BN, MatchEpi<4, true>>(tmA, tmB, sh, num_kb, MatchEpi<4, true>{dbnorm, N, cand_score, cand_idx, 2 * splits}, s);
  if (kc == 8) return launch_tc<BN, MatchEpi<8, true>>(tmA, tmB, sh, num_kb, MatchEpi<8, true>{dbnorm, N, cand_score, cand_idx, 2 * splits}, s);
  return launch_tc<BN, MatchEpi<16, true>>(tmA, tmB, sh, num_kb, MatchEpi<16, true>{dbnorm, N, cand_score, cand_idx, 2 * splits}, s);
}

int tc_match_coarse(const __nv_bfloat16* Q16, int nq, const __nv_bfloat16* DB16, const float* dbnorm, long long N,
                    int D, int kc, float* cand_score, int32_t* cand_idx, cudaStream_t s) {
  MOCHA_CHECK_ARG(Q16 && DB16 && dbnorm && cand_score && cand_idx, "tc_match_coarse: null operand");
  MOCHA_CHECK_ARG(nq > 0 && N > 0 && N < 2147483647LL, "tc_match_coarse: bad sizes nq=%d N=%lld", nq, N);
  MOCHA_CHECK_ARG(D >= BLOCK_K && D % 8 == 0, "tc_match_coarse: D=%d must be >= 64 and a multiple of 8", D);
  MOCHA_CHECK_ARG(kc == 4 || kc == 8 || kc == 16, "tc_match_coarse: kc must be 4, 8 or 16");
  constexpr int BN = 256;
  CUtensorMap tmA, tmB;
  MOCHA_TRY(make_tmap(&tmA, Q16, (unsigned long long)nq, (unsigned long long)D, BLOCK_M));
  MOCHA_TRY(make_tmap(&tmB, DB16, (unsigned long long)N, (unsigned long long)D, BN));
  TcShape sh{};
  sh.nb = 1;
  sh.rows_out_per_b = nq;
  sh.tiles_m_per_b = ceil_div(nq, BLOCK_M);
  sh.tiles_m_total = sh.tiles_m_per_b;
  sh.src_rows_per_b = nq;
  sh.taps = 1;
  sh.kb_per_tap = ceil_div(D, BLOCK_K);
  sh.tap_row_stride = 0;
  sh.tiles_n = (int)((N + BN - 1) / BN);
  const int splits = tc_match_splits(nq, N) / 2;
  sh.tiles_per_unit = ceil_div(sh.tiles_n, splits);
  sh.units = sh.tiles_m_total * splits;
  sh.splits = splits;
  {
    // keep one group's query rows (group_m * 128 * D bf16) within about half of the 126 MB L2
    long long gm = (64LL << 20) / ((long long)BLOCK_M * D * 2);
    if (gm < 1) gm = 1;
    // prefer a group size that divides the m-tile count (balanced groups measured ~10 % faster)
    for (long long d = gm; d >= 1; --d)
      if (sh.tiles_m_total % d == 0) { if (2 * d > gm) gm = d; break; }
    sh.group_m = (int)gm;
  }
  const int num_kb = ceil_div(D, BLOCK_K);
  if (kc == 4) return launch_tc<BN, MatchEpi<4>>(tmA, tmB, sh, num_kb, MatchEpi<4>{dbnorm, N, cand_score, cand_idx, 2 * splits}, s);
  if (kc == 8) return launch_tc<BN, MatchEpi<8>>(tmA, tmB, sh, num_kb, MatchEpi<8>{dbnorm, N, cand_score, cand_idx, 2 * splits}, s);
  return launch_tc<BN, MatchEpi<16>>(tmA, tmB, sh, num_kb, MatchEpi<16>{dbnorm, N, cand_score, cand_idx, 2 * splits}, s);
}

// ------------------------------------------------------------------------------------------------
// Split-K coarse pass for small problems (few query x row tiles, very long rows): the batched
// characterization step matches 128 queries against a 385-row DB of 23040-d rows - 4 output tiles,
// 360 k-blocks each. The K range is cut into slices that run as independent images of the
// batched-head GEMM (slice z reads columns [z*Ks, (z+1)*Ks) of both operands and writes partial
// image z), and a reduction kernel forms ||x||^2 - 2 q.x as one candidate list per query.
// ------------------------------------------------------------------------------------------------
namespace {
__global__ void splitk_reduce_kernel(const float* __restrict__ partial, int slices, int nq, int Np, long long N,
                                     const float* __restrict__ dbnorm, float* __restrict__ cand_score,
                                     int32_t* __restrict__ cand_idx) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)nq * Np) return;
  const int n = (int)(i % Np);
  float acc = 0.f;
  const long long img = (long long)nq * Np;
  for (int z = 0; z < slices; ++z) acc += partial[z * img + i];
  const bool ok = n < N;
  cand_score[i] = ok ? fmaf(-2.f, acc, __ldg(dbnorm + n)) : INFINITY;
  cand_idx[i] = ok ? n : -1;
}
}  // namespace

int tc_match_splitk_slices(int nq, long long N, int D) {
  if (N > 8192 || D % 8 != 0) return 0;
  const int num_kb = ceil_div(D, BLOCK_K);
  const long long units0 = (long long)ceil_div(nq, BLOCK_M) * ((N + 127) / 128);
  if (num_kb < 16 || units0 * 2 > num_sms()) return 0;
  int slices = (int)((num_sms() + units0 - 1) / units0);
  if (slices > num_kb / 4) slices = num_kb / 4;
  if (slices < 2) return 0;
  const int kb_per = ceil_div(num_kb, slices);
  return ceil_div(num_kb, kb_per);
}

size_t tc_match_splitk_ws_bytes(int nq, long long N, int D) {
  const int slices = tc_match_splitk_slices(nq, N, D);
  if (!slices) return 0;
  const size_t Np = (size_t)((N + 127) / 128) * 128;
  return align_up((size_t)slices * nq * Np * 4, 256) + 256;
}

// candidate lists: cand_score / cand_idx are [nq, Np] with Np = round_up(N, 128) (index -1 past N)
int tc_match_coarse_splitk(const __nv_bfloat16* Q16, int nq, const __nv_bfloat16* DB16, const float* dbnorm, long long N,
                           int D, float* partial, float* cand_score, int32_t* cand_idx, cudaStream_t s) {
  const int slices = tc_match_splitk_slices(nq, N, D);
  MOCHA_CHECK_ARG(slices >= 2 && Q16 && DB16 && partial, "tc_match_coarse_splitk: not applicable");
  constexpr int BN = 128;
  const int num_kb = ceil_div(D, BLOCK_K), kb_per = ceil_div(num_kb, slices);
  const int Np = (int)((N + BN - 1) / BN) * BN;
  CUtensorMap tmA;
  MOCHA_TRY(make_tmap(&tmA, Q16, (unsigned long long)nq, (unsigned long long)D, BLOCK_M));
  TcShape sh{};
  sh.nb = slices; sh.H = slices;
  sh.rows_out_per_b = nq;
  sh.tiles_m_per_b = ceil_div(nq, BLOCK_M);
  sh.tiles_m_total = sh.tiles_m_per_b * slices;
  sh.src_rows_per_b = 0; sh.a_rows_h = 0; sh.a_cols_h = kb_per * BLOCK_K;
  sh.b_rows_b = 0; sh.b_rows_h = 0; sh.b_cols_h = kb_per * BLOCK_K;
  sh.c_img_b = 0; sh.c_img_h = (long long)nq * Np;
  sh.taps = 1; sh.kb_per_tap = kb_per; sh.tap_row_stride = 0;
  LinearEpi epi{partial, Np, Np, nullptr, 0, nullptr, ACT_NONE, nullptr, 0};
  MOCHA_TRY(dispatch_bn(BN, tmA, DB16, (unsigned long long)N, (unsigned long long)D, sh, Np, kb_per, epi, s));
  const long long total = (long long)nq * Np;
  launch_k(splitk_reduce_kernel, (unsigned)((total + 255) / 256), 256, 0, s, partial, slices, nq, Np, N, dbnorm, cand_score, cand_idx);
  count_launch();
  MOCHA_LAUNCH_CHECK("splitk_reduce_kernel");
  return MOCHA_OK;
}

}  // namespace mocha

#ifdef MOCHA_TRACE
extern "C" int mocha_debug_get_epi(unsigned long long* host16) {
  return cudaMemcpyFromSymbol(host16, mocha::g_epi_dbg, 16 * sizeof(unsigned long long)) == cudaSuccess ? 0 : 1;
}
// trace build only: bf16-in / bf16-out linear layer as the bf16 path runs it (A16 [M,K], W16 [N,K], out16 [M,N])
extern "C" int mocha_debug_linear_bf16(const void* A16, const void* W16, const float* bias, const float* res, float* out32,
                                       void* out16, int M, int N, int K, int act, void* stream) {
  return mocha::tc_linear_bf16((const __nv_bfloat16*)A16, K, (const __nv_bfloat16*)W16, bias, 0, res,
                               mocha::TcOut{out32, (__nv_bfloat16*)out16, 0}, M, N, K, act, (cudaStream_t)stream);
}
extern "C" int mocha_debug_set_mode(int mode) {
  return cudaMemcpyToSymbol(mocha::g_tc_dbg_mode, &mode, sizeof(mode)) == cudaSuccess ? 0 : 1;
}
extern "C" int mocha_debug_set_trace(unsigned long long* buf) {
  return cudaMemcpyToSymbol(mocha::g_tc_trace, &buf, sizeof(buf)) == cudaSuccess ? 0 : 1;
}
#endif
