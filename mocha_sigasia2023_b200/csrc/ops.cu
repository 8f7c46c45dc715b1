// Bandwidth/latency-bound building blocks (see ops.cuh for the reference citations).
#include "ops.cuh"

#include <cooperative_groups.h>

namespace mocha {

namespace {

// The 'distance' adjacency is sparse (24/46/52 non-zeros of 576 per partition for the joint graph):
// each (k, w) keeps a compact list of its non-zero sources in shared memory.
__global__ void graph_agg_first_kernel(const float* __restrict__ in, const float* __restrict__ A,
                                       float* __restrict__ out, __nv_bfloat16* __restrict__ out16, int V, int C,
                                       int Kk, int lrelu) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float sm[];
  float* xs = sm;                                   // [V][C]
  float* val = sm + V * C;                          // [Kk*V][V] non-zero values
  int* src = reinterpret_cast<int*>(val + Kk * V * V);  // [Kk*V][V] their source nodes
  int* cnt = src + Kk * V * V;                      // [Kk*V]
  const int bt = blockIdx.x;
  const float* xin = in + (long long)bt * V * C;
  for (int i = threadIdx.x; i < V * C; i += blockDim.x) {
    float v = xin[i];
    xs[i] = lrelu ? lrelu02(v) : v;
  }
  for (int kw = threadIdx.x; kw < Kk * V; kw += blockDim.x) {
    const int k = kw / V, w = kw - k * V;
    int n = 0;
    for (int u = 0; u < V; ++u) {
      const float a = A[(k * V + u) * V + w];
      if (a != 0.f) { val[kw * V + n] = a; src[kw * V + n] = u; ++n; }
    }
    cnt[kw] = n;
  }
  __syncthreads();
  const int KC = Kk * C;
  float* dst = out ? out + (long long)bt * V * KC : nullptr;
  __nv_bfloat16* dst16 = out16 ? out16 + (long long)bt * V * KC : nullptr;
  // thread -> channel c (fastest, coalesced stores) and a node stripe; no divisions in the loops. Rows wider than the
  // block (C > 256: a 512-wide model's body-part blocks) take several channel passes per thread.
  const int cw = C < (int)blockDim.x ? C : (int)blockDim.x;
  const int c0 = threadIdx.x % cw, stripe = threadIdx.x / cw, nstripes = blockDim.x / cw;
  if (stripe < nstripes) {
    for (int w = stripe; w < V; w += nstripes) {
      for (int k = 0; k < Kk; ++k) {
        const int kw = k * V + w;
        const int n = cnt[kw];
        for (int c = c0; c < C; c += cw) {
          float acc = 0.f;
          for (int i = 0; i < n; ++i) acc = fmaf(xs[src[kw * V + i] * C + c], val[kw * V + i], acc);
          if (dst) dst[w * KC + k * C + c] = acc;
          if (dst16) dst16[w * KC + k * C + c] = __float2bfloat16_rn(acc);
        }
      }
    }
  }
}

// Small graphs (V <= 8: the 6-node body-part graph of to_mot) with a bf16 output: one thread per (frame, 4 channels) keeps
// the V source vectors in registers and writes all Kk * V outputs (the adjacency is dense at this size); no per-block list
// building, loads and stores fully coalesced across channels. The list kernel above needed 19 us for 24 MB at 128 clips.
constexpr int GAS_VMAX = 8;
__global__ void __launch_bounds__(256)
graph_agg_small_kernel(const float* __restrict__ in, const float* __restrict__ A, __nv_bfloat16* __restrict__ out16,
                       long long total, int V, int C4, int Kk, int lrelu) {
  pdl_trigger();
  __shared__ float As[4 * GAS_VMAX * GAS_VMAX];
  for (int i = threadIdx.x; i < Kk * V * V; i += blockDim.x) As[i] = A[i];   // constant: before the grid dependency
  pdl_wait();
  __syncthreads();
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const long long bt = idx / C4;
  const int c = (int)(idx - bt * C4) * 4, C = C4 * 4, KC = Kk * C;
  float4 x[GAS_VMAX];
#pragma unroll
  for (int u = 0; u < GAS_VMAX; ++u)
    if (u < V) {
      float4 v = *reinterpret_cast<const float4*>(in + (bt * V + u) * C + c);
      if (lrelu) { v.x = lrelu02(v.x); v.y = lrelu02(v.y); v.z = lrelu02(v.z); v.w = lrelu02(v.w); }
      x[u] = v;
    }
  for (int k = 0; k < Kk; ++k)
    for (int w = 0; w < V; ++w) {
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int u = 0; u < GAS_VMAX; ++u)
        if (u < V) {
          const float av = As[(k * V + u) * V + w];
          a.x = fmaf(x[u].x, av, a.x); a.y = fmaf(x[u].y, av, a.y); a.z = fmaf(x[u].z, av, a.z); a.w = fmaf(x[u].w, av, a.w);
        }
      __nv_bfloat162 lo = __floats2bfloat162_rn(a.x, a.y), hi = __floats2bfloat162_rn(a.z, a.w);
      uint2 pk;
      pk.x = *reinterpret_cast<uint32_t*>(&lo);
      pk.y = *reinterpret_cast<uint32_t*>(&hi);
      *reinterpret_cast<uint2*>(out16 + (bt * V + w) * KC + k * C + c) = pk;
    }
}

// Fused front of mot_embedding's JointBlock for the tensor-core path (model.py:42-44, blocks.py:125-129):
//   h0 = Conv2d 1x1 (Cin -> C0) of the pose window, LeakyReLU(0.2), graph aggregation with the sparse
//   adjacency -> bf16 operand [BT*V, Kk*C0] of the 1x1 graph convolution GEMM.
// One block owns G consecutive frames: the adjacency lists, the 1x1 weights and the G x V x Cin inputs
// are staged once, h0 never leaves shared memory (saves a 2 x 47 MB round trip per 128 clips).
constexpr int EMB_MAXCIN = 16;
// The kernel is issue-bound (ncu: 81 % issue slots busy), so the layout minimises instructions per
// output: phase 2 computes 2 channels x 12 rows per thread with the 1x1 weights in registers, phase 3
// gives each half-warp one output row with 4 channels per lane (LDS.128 / 8 B stores) and walks exactly
// the non-zero neighbours; the padded tail of a row is copied from a per-node table.
template <int G>
__global__ void __launch_bounds__(256)
embed_graph_agg_kernel(const float* __restrict__ X, const float* __restrict__ Wemb, const float* __restrict__ bemb,
                       const float* __restrict__ A, __nv_bfloat16* __restrict__ out16, int BT, int V, int Cin, int C,
                       int Kk, int ldo) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float sm[];
  float* xs = sm;                                     // [G*V][C]   activated h0
  float* xin = xs + G * V * C;                        // [G*V][16]  raw inputs, rows padded to 16 floats
  float* val = xin + G * V * EMB_MAXCIN;              // [Kk*V][V]  adjacency A[k][u][w] staged as [k][w][u], then compacted
  int* src = reinterpret_cast<int*>(val + Kk * V * V);  // [Kk*V][V] source nodes of the non-zeros
  int* cnt = src + Kk * V * V;                        // [Kk*V]
  __nv_bfloat16* tails = reinterpret_cast<__nv_bfloat16*>(cnt + Kk * V);  // [V][ldo - Kk*C] row tails
  const int bt0 = blockIdx.x * G;
  const int rows = min(G, BT - bt0) * V;
  const int KC = Kk * C, tail = ldo - KC;
  {
    // all of this thread's input elements are requested before the first one is stored (the loop form paid one global
    // round trip per iteration: 19 % of the kernel's stall samples sat on its STS)
    constexpr int NIT = (G * 32 * EMB_MAXCIN + 255) / 256;   // V <= 32
    float vals[NIT];
#pragma unroll
    for (int j = 0; j < NIT; ++j) {
      const int i = threadIdx.x + 256 * j;
      const int r = i / EMB_MAXCIN, k = i - r * EMB_MAXCIN;
      vals[j] = (i < rows * EMB_MAXCIN && k < Cin) ? __ldg(X + ((long long)bt0 * V + r) * Cin + k) : 0.f;
    }
#pragma unroll
    for (int j = 0; j < NIT; ++j) {
      const int i = threadIdx.x + 256 * j;
      if (i < rows * EMB_MAXCIN) xin[i] = vals[j];
    }
  }
  for (int i = threadIdx.x; i < Kk * V * V; i += blockDim.x) {   // coalesced read, transposed to [k][w][u]
    const int k = i / (V * V), rem = i - k * V * V, u = rem / V, w = rem - u * V;
    val[(k * V + w) * V + u] = A[i];
  }
  __syncthreads();
  if (threadIdx.x < Kk * V) {   // one thread compacts one (k, w) list in place (ascending sources)
    const int kw = threadIdx.x;
    int n = 0;
    float sum = 0.f;
    for (int u = 0; u < V; ++u) {
      const float a = val[kw * V + u];
      if (a != 0.f) { val[kw * V + n] = a; src[kw * V + n] = u * C; sum += a; ++n; }
    }
    cnt[kw] = n;
    // tail of node w's rows: the Kk adjacency column sums (bias columns of the GEMM), then zeros
    const int k = kw / V, w = kw - k * V;
    if (k < tail) tails[w * tail + k] = __float2bfloat16_rn(sum);
  }
  for (int i = threadIdx.x; i < V * tail; i += blockDim.x)
    if (i % tail >= Kk) tails[i] = __float2bfloat16_rn(0.f);
  // h0 = lrelu(x W^T + b): thread = channel pair (weights in registers), rows striped over the block
  {
    const int C2 = C / 2;
    const int cp = threadIdx.x % C2, stripe = threadIdx.x / C2, nstripes = blockDim.x / C2;
    float w0[EMB_MAXCIN], w1[EMB_MAXCIN];
#pragma unroll
    for (int k = 0; k < EMB_MAXCIN; ++k) {
      w0[k] = k < Cin ? Wemb[(2 * cp) * Cin + k] : 0.f;
      w1[k] = k < Cin ? Wemb[(2 * cp + 1) * Cin + k] : 0.f;
    }
    const float b0 = bemb ? bemb[2 * cp] : 0.f, b1 = bemb ? bemb[2 * cp + 1] : 0.f;
    if (stripe < nstripes)
      for (int r = stripe; r < rows; r += nstripes) {
        const float4* xr = reinterpret_cast<const float4*>(xin + r * EMB_MAXCIN);
        float a0 = b0, a1 = b1;
#pragma unroll
        for (int k4 = 0; k4 < EMB_MAXCIN / 4; ++k4) {
          const float4 x4 = xr[k4];
          a0 = fmaf(x4.x, w0[4 * k4], a0); a1 = fmaf(x4.x, w1[4 * k4], a1);
          a0 = fmaf(x4.y, w0[4 * k4 + 1], a0); a1 = fmaf(x4.y, w1[4 * k4 + 1], a1);
          a0 = fmaf(x4.z, w0[4 * k4 + 2], a0); a1 = fmaf(x4.z, w1[4 * k4 + 2], a1);
          a0 = fmaf(x4.w, w0[4 * k4 + 3], a0); a1 = fmaf(x4.w, w1[4 * k4 + 3], a1);
        }
        *reinterpret_cast<float2*>(xs + r * C + 2 * cp) = make_float2(lrelu02(a0), lrelu02(a1));
      }
  }
  __syncthreads();
  // aggregation: a group of C/4 lanes owns one output row, 4 channels per lane
  const int C4 = C / 4, gpw = 32 / C4;                 // lanes per row, rows per warp pass
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int grp = lane / C4, l4 = (lane - grp * C4) * 4;
  const int ngroups = (blockDim.x >> 5) * gpw;
  for (int r = warp * gpw + grp; r < rows; r += ngroups) {
    const int g = r / V, w = r - g * V;
    const float* xg = xs + g * V * C + l4;
    __nv_bfloat16* dst = out16 + ((long long)bt0 * V + r) * ldo + l4;
    for (int k = 0; k < Kk; ++k) {
      const int kw = k * V + w, n = cnt[kw];
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int i = 0; i < n; ++i) {
        const float4 x = *reinterpret_cast<const float4*>(xg + src[kw * V + i]);
        const float av = val[kw * V + i];
        acc.x = fmaf(x.x, av, acc.x); acc.y = fmaf(x.y, av, acc.y);
        acc.z = fmaf(x.z, av, acc.z); acc.w = fmaf(x.w, av, acc.w);
      }
      __nv_bfloat162 lo = __floats2bfloat162_rn(acc.x, acc.y), hi = __floats2bfloat162_rn(acc.z, acc.w);
      uint2 pk;
      pk.x = *reinterpret_cast<uint32_t*>(&lo);
      pk.y = *reinterpret_cast<uint32_t*>(&hi);
      *reinterpret_cast<uint2*>(dst + k * C) = pk;
    }
    for (int t = l4; t < tail; t += C)   // tail <= C in practice: one 8 B copy per lane
      *reinterpret_cast<uint2*>(dst + KC - l4 + t) = *reinterpret_cast<const uint2*>(tails + w * tail + t);
  }
}

// ---- tensor-core variant (mma.sync m16n8k8, TF32 operands, fp32 accumulation) ----------------------------------------
// The sparse walk above is issue-bound (~30 K warp instructions per 96-row block, 0.2 of the HBM roof). Both steps are
// tiny dense products per frame: h0[V, C] = X[V, Cin] Wemb^T and out[(k, w), c] = sum_u A[k][u][w] h0[u, c], i.e.
// [Kk*V x V] x [V x C]. With the adjacency (transposed, zero rows up to a multiple of 16) and the 1x1 weights held as
// constant mma fragments in registers, a frame costs 8 + 15 mma per warp instead of ~900 FFMA / LDS instructions, and
// the kernel becomes what it should be: a stream of 512-byte output rows. Warp w owns channels 8w..8w+7 in both
// products; h0 goes through shared memory once (fp32, rounded to TF32, row stride 72 = conflict-free B fragments);
// finished rows are staged as bf16 (row stride ldo + 8) and leave with one 1-D bulk copy (cp.async.bulk) per row, so
// no thread waits for a store. Persistent over groups of G frames; the next group's inputs are in flight in registers
// while the current group is aggregated. TF32 rounding (2^-11) sits below the bf16 rounding of the output (2^-9).
__device__ __forceinline__ uint32_t f2tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
constexpr int EMB_XLD = 20;   // floats per staged input row: A-fragment loads (rows g, cols t / t+4) hit 32 distinct banks
constexpr int EMB_HLD = 72;   // floats per h0 row (C = 64): B-fragment loads (rows t, cols g) hit 32 distinct banks

template <int V, int KK, int G>
__global__ void __launch_bounds__(256, 2)
embed_graph_agg_mma_kernel(const float* __restrict__ X, const float* __restrict__ Wemb, const float* __restrict__ bemb,
                           const float* __restrict__ A, __nv_bfloat16* __restrict__ out16, int BT, int Cin, int ldo) {
  constexpr int C = 64, KC = KK * C, M = KK * V, MT = (M + 15) / 16, KS = V / 8, ROWS = G * V, XT = (ROWS + 15) / 16;
  constexpr int NLD = (ROWS * EMB_MAXCIN + 255) / 256;
  static_assert(V % 8 == 0 && ROWS <= 256 && ROWS % 8 == 0, "geometry");
  pdl_trigger();
  extern __shared__ __align__(16) unsigned char smraw[];
  float* xin = reinterpret_cast<float*>(smraw);                      // [XT*16][EMB_XLD]
  float* hs = xin + XT * 16 * EMB_XLD;                               // [ROWS][EMB_HLD]
  __nv_bfloat16* stg = reinterpret_cast<__nv_bfloat16*>(hs + ROWS * EMB_HLD);   // [ROWS][ldo + 8]
  const int sld = ldo + 8;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
  const int c0 = warp * 8;

  // ---- constants (weights: may be read before the grid dependency resolves) ----
  uint32_t wb[2][2];                      // 1x1 conv, B fragments: B[k = cin][n = c] = Wemb[c][cin]
#pragma unroll
  for (int ks = 0; ks < 2; ++ks) {
    const int k0 = ks * 8 + t, k1 = k0 + 4;
    wb[ks][0] = f2tf32(k0 < Cin ? __ldg(Wemb + (c0 + g) * Cin + k0) : 0.f);
    wb[ks][1] = f2tf32(k1 < Cin ? __ldg(Wemb + (c0 + g) * Cin + k1) : 0.f);
  }
  const float bias0 = bemb ? __ldg(bemb + c0 + 2 * t) : 0.f, bias1 = bemb ? __ldg(bemb + c0 + 2 * t + 1) : 0.f;
  uint32_t adj[MT][KS][4];                // aggregation, A fragments: At[(k, w)][u] = A[k][u][w]
#pragma unroll
  for (int mt = 0; mt < MT; ++mt)
#pragma unroll
    for (int ks = 0; ks < KS; ++ks)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int r = mt * 16 + g + (j & 1) * 8, u = ks * 8 + t + (j >> 1) * 4;
        const int k = r / V, w = r - k * V;
        adj[mt][ks][j] = f2tf32(r < M ? __ldg(A + (k * V + u) * V + w) : 0.f);
      }
  // staging offsets of this thread's output rows (row r = (k, w) -> staged row w, columns k*C + c0 + 2t)
  // (M is a multiple of 8, so whether a half tile of 8 rows exists is known at compile time)
  static_assert(M % 8 == 0, "half tiles are all-valid or all-padding");
  int soff[MT][2];
#pragma unroll
  for (int mt = 0; mt < MT; ++mt)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int r = mt * 16 + g + h * 8, k = r / V, w = r - k * V;
      soff[mt][h] = w * sld + k * C + c0 + 2 * t;
    }
  // zero the padded input columns / rows once; row tails (adjacency column sums = bias columns of the GEMM, then zeros)
  for (int i = threadIdx.x; i < XT * 16 * EMB_XLD; i += 256) xin[i] = 0.f;
  for (int i = threadIdx.x; i < ROWS * (ldo - KC); i += 256) {
    const int r = i / (ldo - KC), j = i - r * (ldo - KC), w = r % V;
    float sum = 0.f;
    if (j < KK)
      for (int u = 0; u < V; ++u) sum += __ldg(A + (j * V + u) * V + w);
    stg[r * sld + KC + j] = __float2bfloat16_rn(sum);
  }
  pdl_wait();

  const int ngroups = (BT + G - 1) / G;
  float xv[NLD];
  int xoff[NLD];   // shared-memory slot of this thread's j-th input element (row r, column k -> r * EMB_XLD + k); -1 = none
#pragma unroll
  for (int j = 0; j < NLD; ++j) {
    const int i = threadIdx.x + 256 * j, r = i / Cin;
    xoff[j] = i < ROWS * Cin ? r * EMB_XLD + (i - r * Cin) : -1;
  }
  auto load_x = [&](int grp) {
    const long long base = (long long)grp * ROWS * Cin;
    const int n = min(G, BT - grp * G) * V * Cin;
#pragma unroll
    for (int j = 0; j < NLD; ++j) {
      const int i = threadIdx.x + 256 * j;
      xv[j] = i < n ? __ldg(X + base + i) : 0.f;
    }
  };
  if ((int)blockIdx.x < ngroups) load_x(blockIdx.x);
  for (int grp = blockIdx.x; grp < ngroups; grp += gridDim.x) {
    const int rows = min(G, BT - grp * G) * V;
    __syncthreads();                                  // previous group's fragment reads of xin / hs are done
#pragma unroll
    for (int j = 0; j < NLD; ++j)
      if (xoff[j] >= 0) xin[xoff[j]] = xv[j];
    __syncthreads();
    if (grp + (int)gridDim.x < ngroups) load_x(grp + gridDim.x);   // in flight during both products
    // ---- h0 = lrelu(x Wemb^T + b) for this warp's 8 channels, all rows ----
#pragma unroll
    for (int mt = 0; mt < XT; ++mt) {
      float d[4] = {bias0, bias1, bias0, bias1};
#pragma unroll
      for (int ks = 0; ks < 2; ++ks) {
        const float* xr = xin + (mt * 16 + g) * EMB_XLD + ks * 8 + t;
        // raw fp32 bits: the MMA reads the top 19 bits (truncation, 2^-10 relative: below the bf16 rounding of the output)
        uint32_t a[4] = {__float_as_uint(xr[0]), __float_as_uint(xr[8 * EMB_XLD]), __float_as_uint(xr[4]),
                         __float_as_uint(xr[8 * EMB_XLD + 4])};
        mma_tf32(d, a, wb[ks][0], wb[ks][1]);
      }
      const int r0 = mt * 16 + g;
      if (mt * 16 < ROWS)
        *reinterpret_cast<float2*>(hs + r0 * EMB_HLD + c0 + 2 * t) =
            make_float2(__uint_as_float(f2tf32(lrelu02(d[0]))), __uint_as_float(f2tf32(lrelu02(d[1]))));
      if (mt * 16 + 8 < ROWS)
        *reinterpret_cast<float2*>(hs + (r0 + 8) * EMB_HLD + c0 + 2 * t) =
            make_float2(__uint_as_float(f2tf32(lrelu02(d[2]))), __uint_as_float(f2tf32(lrelu02(d[3]))));
    }
    // the previous group's bulk stores must have finished reading the staging rows before they are overwritten
    if (threadIdx.x < ROWS) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncthreads();
    // ---- aggregation: out[(k, w), c] = sum_u At[(k, w), u] h0[u, c] per frame ----
#pragma unroll 1
    for (int f = 0; f < G; ++f) {
      uint32_t hb[KS][2];
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
        const float* hr = hs + (f * V + ks * 8 + t) * EMB_HLD + c0 + g;
        hb[ks][0] = __float_as_uint(hr[0]);
        hb[ks][1] = __float_as_uint(hr[4 * EMB_HLD]);
      }
      __nv_bfloat16* sf = stg + f * V * sld;
#pragma unroll
      for (int mt = 0; mt < MT; ++mt) {
        float d[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) mma_tf32(d, adj[mt][ks], hb[ks][0], hb[ks][1]);
        if (mt * 16 < M) *reinterpret_cast<__nv_bfloat162*>(sf + soff[mt][0]) = __floats2bfloat162_rn(d[0], d[1]);
        if (mt * 16 + 8 < M) *reinterpret_cast<__nv_bfloat162*>(sf + soff[mt][1]) = __floats2bfloat162_rn(d[2], d[3]);
      }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    if ((int)threadIdx.x < rows) {
      const uint32_t src = (uint32_t)__cvta_generic_to_shared(stg + threadIdx.x * sld);
      __nv_bfloat16* dst = out16 + ((long long)grp * ROWS + threadIdx.x) * ldo;
      asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"((uint32_t)ldo * 2u)
                   : "memory");
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
  }
  if (threadIdx.x < ROWS) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

__global__ void graph_agg_kv_kernel(const float* __restrict__ in, const float* __restrict__ A2,
                                    float* __restrict__ out, int U, int Wn, int C, int Kk) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float sm[];
  const int KC = Kk * C;
  float* xs = sm;               // [U][Kk*C]
  float* As = sm + U * KC;      // [Kk][U][Wn]
  const int bt = blockIdx.x;
  const float* src = in + (long long)bt * U * KC;
  for (int i = threadIdx.x; i < U * KC; i += blockDim.x) xs[i] = src[i];
  for (int i = threadIdx.x; i < Kk * U * Wn; i += blockDim.x) As[i] = A2[i];
  __syncthreads();
  float* dst = out + (long long)bt * Wn * C;
  for (int idx = threadIdx.x; idx < Wn * C; idx += blockDim.x) {
    const int w = idx / C, c = idx - w * C;
    float acc = 0.f;
    for (int k = 0; k < Kk; ++k)
      for (int u = 0; u < U; ++u) {
        const float av = As[(k * U + u) * Wn + w];
        if (av != 0.f) acc = fmaf(xs[u * KC + k * C + c], av, acc);
      }
    dst[idx] = acc;
  }
}

constexpr int POOL_MAXP = 8;
__global__ void pool_joint_body_kernel(const float* __restrict__ in, const float* __restrict__ Wp,
                                       float* __restrict__ out, int T, int V, int P, int C, int tp) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float ws[];  // [V][P]
  for (int i = threadIdx.x; i < V * P; i += blockDim.x) ws[i] = Wp[i];
  __syncthreads();
  const int Tp = T / tp;
  const int b = blockIdx.x / Tp, t2 = blockIdx.x % Tp;
  const float inv = 1.f / (float)tp;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float acc[POOL_MAXP];
#pragma unroll
    for (int p = 0; p < POOL_MAXP; ++p) acc[p] = 0.f;
    for (int dt = 0; dt < tp; ++dt) {
      const float* src = in + ((long long)(b * T + t2 * tp + dt) * V) * C + c;
      for (int v = 0; v < V; ++v) {
        const float x = src[(long long)v * C];
#pragma unroll
        for (int p = 0; p < POOL_MAXP; ++p)
          if (p < P) acc[p] = fmaf(x, ws[v * P + p], acc[p]);
      }
    }
    float* dst = out + ((long long)(b * Tp + t2) * P) * C + c;
#pragma unroll
    for (int p = 0; p < POOL_MAXP; ++p)
      if (p < P) dst[(long long)p * C] = acc[p] * inv;
  }
}

// Tensor-core path: joint -> body-part pooling (graph.py:463-465 + AvgPool2d((tp,1)), model.py:47) of the
// bf16 JointBlock output fused with the BodyBlock's pre-activation and graph aggregation
// (blocks.py:125-129, :64): out16[(b,t2,w), k*C + c] = sum_u lrelu(pooled[b,t2,u,c]) * A[k,u,w].
// Block = one (b, t2); thread = a channel pair (bf162 loads, 128 B per warp row).
__global__ void __launch_bounds__(128)
pool_graph_agg_kernel(const __nv_bfloat16* __restrict__ in, const float* __restrict__ Wp, const float* __restrict__ A,
                      __nv_bfloat16* __restrict__ out16, int T, int V, int P, int C, int tp, int Kk) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float ws[];
  float* As = ws;                                   // [Kk][P][P] adjacency
  float* mw = As + Kk * P * P;                      // [P][V] member weights of each body part (compact)
  int* mv = reinterpret_cast<int*>(mw + P * V);     // [P][V] member joints
  int* mc = mv + P * V;                             // [P]
  for (int i = threadIdx.x; i < Kk * P * P; i += blockDim.x) As[i] = A[i];
  if (threadIdx.x < P) {
    // the pooling matrix is a (weighted) membership table: a handful of joints per part
    const int p = threadIdx.x;
    int n = 0;
    for (int v = 0; v < V; ++v) {
      const float wv = Wp[v * P + p];
      if (wv != 0.f) { mw[p * V + n] = wv; mv[p * V + n] = v; ++n; }
    }
    mc[p] = n;
  }
  __syncthreads();
  const int Tp = T / tp;
  const int b = blockIdx.x / Tp, t2 = blockIdx.x % Tp;
  const float inv = 1.f / (float)tp;
  const int KC = Kk * C, C2 = C / 2;
  for (int c2 = threadIdx.x; c2 < C2; c2 += blockDim.x) {
    float a0[POOL_MAXP], a1[POOL_MAXP];
    const __nv_bfloat162* src = reinterpret_cast<const __nv_bfloat162*>(in + ((long long)(b * T + t2 * tp) * V) * C) + c2;
#pragma unroll
    for (int p = 0; p < POOL_MAXP; ++p) {
      a0[p] = 0.f; a1[p] = 0.f;
      if (p < P) {
        const int n = mc[p];
        if (tp == 4) {
          // four frames of one member joint = four independent loads in flight per step
          const long long fs = (long long)V * C2;
#pragma unroll 2
          for (int i = 0; i < n; ++i) {
            const __nv_bfloat162* sj = src + (long long)mv[p * V + i] * C2;
            const float wv = mw[p * V + i];
            const float2 x0 = __bfloat1622float2(sj[0]), x1 = __bfloat1622float2(sj[fs]);
            const float2 x2 = __bfloat1622float2(sj[2 * fs]), x3 = __bfloat1622float2(sj[3 * fs]);
            a0[p] = fmaf((x0.x + x1.x) + (x2.x + x3.x), wv, a0[p]);
            a1[p] = fmaf((x0.y + x1.y) + (x2.y + x3.y), wv, a1[p]);
          }
        } else {
          for (int dt = 0; dt < tp; ++dt) {
            const __nv_bfloat162* sd = src + (long long)dt * V * C2;
#pragma unroll 4
            for (int i = 0; i < n; ++i) {
              const float2 x = __bfloat1622float2(sd[(long long)mv[p * V + i] * C2]);
              const float wv = mw[p * V + i];
              a0[p] = fmaf(x.x, wv, a0[p]);
              a1[p] = fmaf(x.y, wv, a1[p]);
            }
          }
        }
        a0[p] = lrelu02(a0[p] * inv);
        a1[p] = lrelu02(a1[p] * inv);
      }
    }
    __nv_bfloat16* dst = out16 + ((long long)(b * Tp + t2) * P) * KC + 2 * c2;
    for (int k = 0; k < Kk; ++k)
      for (int w = 0; w < P; ++w) {
        float o0 = 0.f, o1 = 0.f;
#pragma unroll
        for (int u = 0; u < POOL_MAXP; ++u)
          if (u < P) { const float av = As[(k * P + u) * P + w]; o0 = fmaf(a0[u], av, o0); o1 = fmaf(a1[u], av, o1); }
        *reinterpret_cast<__nv_bfloat162*>(dst + (long long)w * KC + k * C) = __floats2bfloat162_rn(o0, o1);
      }
  }
}

// Four channels per thread (8-byte loads): half the load / convert / FMA instructions of the bf162 kernel above for the same
// bytes (that one was issue- and latency-bound at 0.5 of the HBM roof: 16.7 M warp instructions for 94 MB). A (b, t2) group
// takes C / 4 threads; a block holds 128 / (C / 4) groups, so every warp still reads whole 256-byte row segments.
__global__ void __launch_bounds__(128)
pool_graph_agg_v4_kernel(const __nv_bfloat16* __restrict__ in, const float* __restrict__ Wp, const float* __restrict__ A,
                         __nv_bfloat16* __restrict__ out16, int groups, int T, int V, int P, int C, int tp, int Kk) {
  pdl_trigger();
  extern __shared__ float ws[];
  float* As = ws;                                   // [Kk][P][P] adjacency
  float* mw = As + Kk * P * P;                      // [P][V] member weights of each body part (compact)
  int* mv = reinterpret_cast<int*>(mw + P * V);     // [P][V] member joints
  int* mc = mv + P * V;                             // [P]
  for (int i = threadIdx.x; i < Kk * P * P; i += blockDim.x) As[i] = A[i];       // constants: before the grid dependency
  if (threadIdx.x < P) {
    const int p = threadIdx.x;
    int n = 0;
    for (int v = 0; v < V; ++v) {
      const float wv = Wp[v * P + p];
      if (wv != 0.f) { mw[p * V + n] = wv; mv[p * V + n] = v; ++n; }
    }
    mc[p] = n;
  }
  pdl_wait();
  __syncthreads();
  const int C4 = C / 4, gpb = blockDim.x / C4;
  const int grp = blockIdx.x * gpb + threadIdx.x / C4, c4 = threadIdx.x % C4;
  if (grp >= groups || threadIdx.x >= gpb * C4) return;
  const int Tp = T / tp, b = grp / Tp, t2 = grp - b * Tp;
  const float inv = 1.f / (float)tp;
  const int KC = Kk * C;
  const uint2* src = reinterpret_cast<const uint2*>(in + ((long long)(b * T + t2 * tp) * V) * C) + c4;   // row r at src[r * C4]
  float a[POOL_MAXP][4];
#pragma unroll
  for (int p = 0; p < POOL_MAXP; ++p) {
    a[p][0] = a[p][1] = a[p][2] = a[p][3] = 0.f;
    if (p < P) {
      const int n = mc[p];
      for (int i = 0; i < n; ++i) {
        const uint2* sj = src + (long long)mv[p * V + i] * C4;
        const float wv = mw[p * V + i];
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
        if (tp == 4) {
          // four frames of one member joint = four independent 8-byte loads in flight
          const long long fs = (long long)V * C4;
          const uint2 x0 = __ldg(sj), x1 = __ldg(sj + fs), x2 = __ldg(sj + 2 * fs), x3 = __ldg(sj + 3 * fs);
          s0 = (__uint_as_float(x0.x << 16) + __uint_as_float(x1.x << 16)) + (__uint_as_float(x2.x << 16) + __uint_as_float(x3.x << 16));
          s1 = (__uint_as_float(x0.x & 0xffff0000u) + __uint_as_float(x1.x & 0xffff0000u)) +
               (__uint_as_float(x2.x & 0xffff0000u) + __uint_as_float(x3.x & 0xffff0000u));
          s2 = (__uint_as_float(x0.y << 16) + __uint_as_float(x1.y << 16)) + (__uint_as_float(x2.y << 16) + __uint_as_float(x3.y << 16));
          s3 = (__uint_as_float(x0.y & 0xffff0000u) + __uint_as_float(x1.y & 0xffff0000u)) +
               (__uint_as_float(x2.y & 0xffff0000u) + __uint_as_float(x3.y & 0xffff0000u));
        } else {
          for (int dt = 0; dt < tp; ++dt) {
            const uint2 x = __ldg(sj + (long long)dt * V * C4);
            s0 += __uint_as_float(x.x << 16); s1 += __uint_as_float(x.x & 0xffff0000u);
            s2 += __uint_as_float(x.y << 16); s3 += __uint_as_float(x.y & 0xffff0000u);
          }
        }
        a[p][0] = fmaf(s0, wv, a[p][0]); a[p][1] = fmaf(s1, wv, a[p][1]);
        a[p][2] = fmaf(s2, wv, a[p][2]); a[p][3] = fmaf(s3, wv, a[p][3]);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) a[p][j] = lrelu02(a[p][j] * inv);
    }
  }
  __nv_bfloat16* dst = out16 + ((long long)grp * P) * KC + 4 * c4;
  for (int k = 0; k < Kk; ++k)
    for (int w = 0; w < P; ++w) {
      float o0 = 0.f, o1 = 0.f, o2 = 0.f, o3 = 0.f;
#pragma unroll
      for (int u = 0; u < POOL_MAXP; ++u)
        if (u < P) {
          const float av = As[(k * P + u) * P + w];
          o0 = fmaf(a[u][0], av, o0); o1 = fmaf(a[u][1], av, o1); o2 = fmaf(a[u][2], av, o2); o3 = fmaf(a[u][3], av, o3);
        }
      __nv_bfloat162 lo = __floats2bfloat162_rn(o0, o1), hi = __floats2bfloat162_rn(o2, o3);
      uint2 pk;
      pk.x = *reinterpret_cast<uint32_t*>(&lo);
      pk.y = *reinterpret_cast<uint32_t*>(&hi);
      *reinterpret_cast<uint2*>(dst + (long long)w * KC + k * C) = pk;
    }
}

// block = (batch b, group of 32 channels); lane = channel (coalesced 128 B rows), the 8 warps split the
// tokens; two-pass mean / unbiased variance like torch.std, partials combined through shared memory.
__global__ void __launch_bounds__(256)
instance_norm_tokens_kernel(const float* __restrict__ x, int n, int C, float eps,
                            const float* __restrict__ gb, float* __restrict__ y,
                            const float* __restrict__ tab_mean,
                            const float* __restrict__ tab_std, float* __restrict__ y2,
                            __nv_bfloat16* __restrict__ y16, __nv_bfloat16* __restrict__ y2h,
                            const float* __restrict__ y2h_center) {
  pdl_trigger();
  pdl_wait();
  __shared__ float part[8][32];
  __shared__ float stat[2][32];
  const int b = blockIdx.x, c = blockIdx.y * 32 + (threadIdx.x & 31), warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool ok = c < C;
  const float* xb = x + (long long)b * n * C;
  float s = 0.f;
  if (ok) for (int i = warp; i < n; i += 8) s += xb[(long long)i * C + c];
  part[warp][lane] = s;
  __syncthreads();
  if (warp == 0) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += part[w][lane];
    stat[0][lane] = t / (float)n;
  }
  __syncthreads();
  const float mean = stat[0][lane];
  float q = 0.f;
  if (ok) for (int i = warp; i < n; i += 8) {
    const float d = xb[(long long)i * C + c] - mean;
    q = fmaf(d, d, q);
  }
  part[warp][lane] = q;
  __syncthreads();
  if (warp == 0) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += part[w][lane];
    stat[1][lane] = sqrtf(t / (float)(n - 1)) + eps;
  }
  __syncthreads();
  if (!ok) return;
  const float den = stat[1][lane];
  float g = 1.f, be = 0.f;
  if (gb) {
    g = 1.f + gb[(long long)b * 2 * C + c];
    be = gb[(long long)b * 2 * C + C + c];
  }
  for (int i = warp; i < n; i += 8) {
    const long long o = (long long)i * C + c;
    // same operation order as the reference: divide, then modulate
    float v = (xb[o] - mean) / den;
    if (gb) v = g * v + be;
    if (y) y[(long long)b * n * C + o] = v;
    if (y16) y16[(long long)b * n * C + o] = __float2bfloat16_rn(v);
    if (y2 || y2h) {
      const float w = (v - tab_mean[o]) / tab_std[o];
      if (y2) y2[(long long)b * n * C + o] = w;
      if (y2h) y2h[(long long)b * n * C + o] = __float2bfloat16_rn(y2h_center ? w - y2h_center[o] : w);
    }
  }
}

// same statistics with the block's tokens held in registers (n <= 128): one pass over global memory
__global__ void __launch_bounds__(256)
instance_norm_tokens_reg_kernel(const float* __restrict__ x, int n, int C, float eps,
                                const float* __restrict__ gb, float* __restrict__ y,
                                const float* __restrict__ tab_mean,
                                const float* __restrict__ tab_std, float* __restrict__ y2,
                                __nv_bfloat16* __restrict__ y16, __nv_bfloat16* __restrict__ y2h,
                            const float* __restrict__ y2h_center) {
  pdl_trigger();
  pdl_wait();
  __shared__ float part[8][32];
  __shared__ float stat[2][32];
  const int b = blockIdx.x, c = blockIdx.y * 32 + (threadIdx.x & 31), warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool ok = c < C;
  const float* xb = x + (long long)b * n * C;
  float v[16];
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const int i = warp + 8 * j;
    v[j] = (ok && i < n) ? xb[(long long)i * C + c] : 0.f;
    s += v[j];
  }
  part[warp][lane] = s;
  __syncthreads();
  if (warp == 0) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += part[w][lane];
    stat[0][lane] = t / (float)n;
  }
  __syncthreads();
  const float mean = stat[0][lane];
  float q = 0.f;
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const float d = v[j] - mean;
    if (warp + 8 * j < n) q = fmaf(d, d, q);
  }
  part[warp][lane] = q;
  __syncthreads();
  if (warp == 0) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += part[w][lane];
    stat[1][lane] = sqrtf(t / (float)(n - 1)) + eps;
  }
  __syncthreads();
  if (!ok) return;
  const float den = stat[1][lane];
  float g = 1.f, be = 0.f;
  if (gb) {
    g = 1.f + gb[(long long)b * 2 * C + c];
    be = gb[(long long)b * 2 * C + C + c];
  }
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const int i = warp + 8 * j;
    if (i < n) {
      const long long o = (long long)i * C + c;
      float u = (v[j] - mean) / den;   // same operation order as the reference: divide, then modulate
      if (gb) u = g * u + be;
      if (y) y[(long long)b * n * C + o] = u;
      if (y16) y16[(long long)b * n * C + o] = __float2bfloat16_rn(u);
      if (y2 || y2h) {
        const float w = (u - tab_mean[o]) / tab_std[o];
        if (y2) y2[(long long)b * n * C + o] = w;
        if (y2h) y2h[(long long)b * n * C + o] = __float2bfloat16_rn(y2h_center ? w - y2h_center[o] : w);
      }
    }
  }
}

// float4 variant for the tensor-core path (C % 64 == 0, n <= 128): a block owns (batch b, 64 channels); 16 lanes x
// float4 cover the channels, the 16 row slots of the block (2 per warp) stride over the tokens. Four times
// fewer load / store instructions than the scalar kernels for the same bytes (which were request-bound at
// 1.4 TB/s); same two-pass statistics.
// (4 blocks per SM: at 80 registers only 3 fitted, and the 128-clip grid of 512 blocks ran as 1.15 waves)
__global__ void __launch_bounds__(256, 4)
instance_norm_tokens_v4_kernel(const float* __restrict__ x, int n, int C, float eps, const float* __restrict__ gb,
                               float* __restrict__ y, __nv_bfloat16* __restrict__ y16, __nv_bfloat16* __restrict__ q16,
                               const float* __restrict__ tab_mean = nullptr, const float* __restrict__ tab_std = nullptr,
                               float* __restrict__ y2 = nullptr, __nv_bfloat16* __restrict__ y2h = nullptr,
                               const float* __restrict__ y2h_center = nullptr) {
  pdl_trigger();
  pdl_wait();
  __shared__ float4 part[16][16];
  __shared__ float4 stat[2][16];
  const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int l16 = lane & 15, rs = warp * 2 + (lane >> 4);
  const int c = blockIdx.y * 64 + 4 * l16;
  const float* xb = x + (long long)b * n * C + c;
  float4 v[8];
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int i = rs + 16 * j;
    v[j] = i < n ? *reinterpret_cast<const float4*>(xb + (long long)i * C) : make_float4(0.f, 0.f, 0.f, 0.f);
    s.x += v[j].x; s.y += v[j].y; s.z += v[j].z; s.w += v[j].w;
  }
  part[rs][l16] = s;
  __syncthreads();
  if (threadIdx.x < 16) {
    float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int r = 0; r < 16; ++r) { const float4 p = part[r][threadIdx.x]; t.x += p.x; t.y += p.y; t.z += p.z; t.w += p.w; }
    const float inv = 1.f / (float)n;
    stat[0][threadIdx.x] = make_float4(t.x * inv, t.y * inv, t.z * inv, t.w * inv);
  }
  __syncthreads();
  const float4 mean = stat[0][l16];
  float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int j = 0; j < 8; ++j)
    if (rs + 16 * j < n) {
      const float dx = v[j].x - mean.x, dy = v[j].y - mean.y, dz = v[j].z - mean.z, dw = v[j].w - mean.w;
      q.x = fmaf(dx, dx, q.x); q.y = fmaf(dy, dy, q.y); q.z = fmaf(dz, dz, q.z); q.w = fmaf(dw, dw, q.w);
    }
  part[rs][l16] = q;
  __syncthreads();
  if (threadIdx.x < 16) {
    float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int r = 0; r < 16; ++r) { const float4 p = part[r][threadIdx.x]; t.x += p.x; t.y += p.y; t.z += p.z; t.w += p.w; }
    const float d = 1.f / (float)(n - 1);
    stat[1][threadIdx.x] = make_float4(sqrtf(t.x * d) + eps, sqrtf(t.y * d) + eps, sqrtf(t.z * d) + eps, sqrtf(t.w * d) + eps);
  }
  __syncthreads();
  const float4 den = stat[1][l16];
  float4 g = make_float4(1.f, 1.f, 1.f, 1.f), be = make_float4(0.f, 0.f, 0.f, 0.f);
  if (gb) {
    const float4 g0 = *reinterpret_cast<const float4*>(gb + (long long)b * 2 * C + c);
    be = *reinterpret_cast<const float4*>(gb + (long long)b * 2 * C + C + c);
    g = make_float4(1.f + g0.x, 1.f + g0.y, 1.f + g0.z, 1.f + g0.w);
  }
  // q16 = IN(AdaIN(x)) without a second pass: AdaIN(x) = g u + be with u = IN(x), whose mean is 0 and whose
  // unbiased std is std / (std + eps) = (den - eps) / den, so IN(g u + be) = u * g / (|g| (den - eps) / den + eps)
  float4 qs = make_float4(0.f, 0.f, 0.f, 0.f);
  if (q16) {
    qs.x = g.x / (fabsf(g.x) * (den.x - eps) / den.x + eps); qs.y = g.y / (fabsf(g.y) * (den.y - eps) / den.y + eps);
    qs.z = g.z / (fabsf(g.z) * (den.z - eps) / den.z + eps); qs.w = g.w / (fabsf(g.w) * (den.w - eps) / den.w + eps);
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int i = rs + 16 * j;
    if (i < n) {
      float4 u = make_float4((v[j].x - mean.x) / den.x, (v[j].y - mean.y) / den.y, (v[j].z - mean.z) / den.z,
                             (v[j].w - mean.w) / den.w);
      const long long o = ((long long)b * n + i) * C + c;
      if (q16) {
        __nv_bfloat162 lo = __floats2bfloat162_rn(u.x * qs.x, u.y * qs.y), hi = __floats2bfloat162_rn(u.z * qs.z, u.w * qs.w);
        uint2 pk;
        pk.x = *reinterpret_cast<uint32_t*>(&lo);
        pk.y = *reinterpret_cast<uint32_t*>(&hi);
        *reinterpret_cast<uint2*>(q16 + o) = pk;
      }
      if (gb) u = make_float4(g.x * u.x + be.x, g.y * u.y + be.y, g.z * u.z + be.z, g.w * u.w + be.w);
      if (y) *reinterpret_cast<float4*>(y + o) = u;
      if (y16) {
        __nv_bfloat162 lo = __floats2bfloat162_rn(u.x, u.y), hi = __floats2bfloat162_rn(u.z, u.w);
        uint2 pk;
        pk.x = *reinterpret_cast<uint32_t*>(&lo);
        pk.y = *reinterpret_cast<uint32_t*>(&hi);
        *reinterpret_cast<uint2*>(y16 + o) = pk;
      }
      if (y2 || y2h) {
        // matcher query (test_fullframework.py:442): (cnt - cnt_mean) / cnt_std with [n, C] tables; the bf16 copy is taken
        // relative to the origin the bf16 DB rows were packed around
        const long long ot = (long long)i * C + c;
        const float4 tm = *reinterpret_cast<const float4*>(tab_mean + ot), ts = *reinterpret_cast<const float4*>(tab_std + ot);
        float4 w = make_float4((u.x - tm.x) / ts.x, (u.y - tm.y) / ts.y, (u.z - tm.z) / ts.z, (u.w - tm.w) / ts.w);
        if (y2) *reinterpret_cast<float4*>(y2 + o) = w;
        if (y2h) {
          if (y2h_center) {
            const float4 cc = *reinterpret_cast<const float4*>(y2h_center + ot);
            w = make_float4(w.x - cc.x, w.y - cc.y, w.z - cc.z, w.w - cc.w);
          }
          __nv_bfloat162 lo = __floats2bfloat162_rn(w.x, w.y), hi = __floats2bfloat162_rn(w.z, w.w);
          uint2 pk;
          pk.x = *reinterpret_cast<uint32_t*>(&lo);
          pk.y = *reinterpret_cast<uint32_t*>(&hi);
          *reinterpret_cast<uint2*>(y2h + o) = pk;
        }
      }
    }
  }
}

__global__ void token_mean_kernel(const float* __restrict__ x, int n, int C, float* __restrict__ out) {
  pdl_trigger();
  pdl_wait();
  const int b = blockIdx.x;
  const float* xb = x + (long long)b * n * C;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float s = 0.f;
    for (int i = 0; i < n; ++i) s += xb[(long long)i * C + c];
    out[(long long)b * C + c] = s / (float)n;
  }
}

// AdaIN parameter MLP of every decoder layer in one launch (transformer.py:98-103 with the style token mean):
//   smean = mean over tokens of the style; per layer gb = W2 lrelu(W1 smean + b1) + b2   ([2D] = gamma | beta)
// Four 128-row GEMM launches + a token mean + a cast were ~54 us of pure launch / pipeline latency per step for
// 0.1 GFLOP. One block per clip: the mean with one column per thread, then a warp per output feature with the lanes
// across K (one coalesced 512-byte weight row segment per LDG.128, bf16 weights from the registered mirror, fp32
// activations), eight outputs reduced at a time with a transposing butterfly (9 shuffles per 8 outputs).
struct StyleMlpLayers {
  const __nv_bfloat16* w1[MOCHA_MAX_DEPTH];
  const float* b1[MOCHA_MAX_DEPTH];
  const __nv_bfloat16* w2[MOCHA_MAX_DEPTH];
  const float* b2[MOCHA_MAX_DEPTH];
};

// sums of NV (8 or 4) per-lane values across the warp with a transposing butterfly: lane L with L % 4 == 0 ends up with the
// total of value index 4*bit4(L) + 2*bit3(L) + bit2(L) (NV = 8) or 2*bit4(L) + bit3(L) (NV = 4, lanes with L % 8 == 0)
template <int NV>
__device__ __forceinline__ float warp_reduce_t(float (&v)[NV], int lane) {
  static_assert(NV == 8 || NV == 4, "NV");
  int bit = 16;
#pragma unroll
  for (int h = NV / 2; h >= 1; h /= 2) {
    const bool up = lane & bit;
#pragma unroll
    for (int i = 0; i < h; ++i) {
      const float send = up ? v[i] : v[i + h], keep = up ? v[i + h] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, bit);
    }
    bit >>= 1;
  }
#pragma unroll
  for (; bit >= 1; bit >>= 1) v[0] += __shfl_xor_sync(0xffffffffu, v[0], bit);
  return v[0];
}

// y[o] = act(W[o, :] . x + b[o]) for o in [0, N): W bf16 [N, K] row-major, x fp32 in shared memory, K = KCH * 256. A warp
// owns NV outputs per pass with its lanes across K: one coalesced 16-byte load per lane, row and 256-column chunk, all
// NV * KCH of them in flight before the first is used.
template <int KCH, int NV>
__device__ __forceinline__ void warp_matvec(const __nv_bfloat16* __restrict__ W, const float* __restrict__ b, const float* xs,
                                            float* ys, float* yg, int N, int lrelu, int warp, int nwarps, int lane) {
  constexpr int K = KCH * 256;
  float x[KCH * 8];
#pragma unroll
  for (int c = 0; c < KCH; ++c) {
    const float4 lo = *reinterpret_cast<const float4*>(xs + c * 256 + lane * 8);
    const float4 hi = *reinterpret_cast<const float4*>(xs + c * 256 + lane * 8 + 4);
    x[c * 8 + 0] = lo.x; x[c * 8 + 1] = lo.y; x[c * 8 + 2] = lo.z; x[c * 8 + 3] = lo.w;
    x[c * 8 + 4] = hi.x; x[c * 8 + 5] = hi.y; x[c * 8 + 6] = hi.z; x[c * 8 + 7] = hi.w;
  }
  for (int o0 = warp * NV; o0 < N; o0 += nwarps * NV) {
    uint4 wv[NV * KCH];
#pragma unroll
    for (int i = 0; i < NV; ++i)
#pragma unroll
      for (int c = 0; c < KCH; ++c)
        wv[i * KCH + c] = __ldg(reinterpret_cast<const uint4*>(W + (size_t)(o0 + i) * K + c * 256 + lane * 8));
    float v[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      float acc = 0.f;
#pragma unroll
      for (int c = 0; c < KCH; ++c) {
        const uint32_t u[4] = {wv[i * KCH + c].x, wv[i * KCH + c].y, wv[i * KCH + c].z, wv[i * KCH + c].w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {   // bf16 -> fp32 is a shift / mask of the packed pair
          acc = fmaf(__uint_as_float(u[j] << 16), x[c * 8 + 2 * j], acc);
          acc = fmaf(__uint_as_float(u[j] & 0xffff0000u), x[c * 8 + 2 * j + 1], acc);
        }
      }
      v[i] = acc;
    }
    const float tot = warp_reduce_t<NV>(v, lane);
    constexpr int STEP = 32 / NV;   // lanes per reduced value
    if ((lane & (STEP - 1)) == 0) {
      const int o = o0 + (NV == 8 ? ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1)
                                  : ((lane >> 4) & 1) * 2 + ((lane >> 3) & 1));
      float r = tot + (b ? __ldg(b + o) : 0.f);
      if (lrelu) r = lrelu02(r);
      if (ys) ys[o] = r;
      if (yg) yg[o] = r;
    }
  }
}

constexpr int STYLE_THREADS = 1024;
__global__ void __launch_bounds__(STYLE_THREADS, 1)
style_mlp_kernel(const float* __restrict__ cha, int n, const StyleMlpLayers L, int nlayers, float* __restrict__ gb, int B) {
  constexpr int D = 256, NW = STYLE_THREADS / 32;
  pdl_trigger();
  pdl_wait();
  __shared__ __align__(16) float part[4][D];
  __shared__ __align__(16) float smean[D];
  __shared__ __align__(16) float hid[2 * D];
  const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  {
    // token mean: four threads per column, each over a quarter of the tokens
    const int c = threadIdx.x & (D - 1), q = threadIdx.x >> 8;
    const float* xb = cha + (long long)b * n * D + c;
    float s0 = 0.f, s1 = 0.f;
    int i = q;
    for (; i + 4 < n; i += 8) { s0 += xb[(long long)i * D]; s1 += xb[(long long)(i + 4) * D]; }
    for (; i < n; i += 4) s0 += xb[(long long)i * D];
    part[q][c] = s0 + s1;
  }
  __syncthreads();
  if (threadIdx.x < D)
    smean[threadIdx.x] = ((part[0][threadIdx.x] + part[1][threadIdx.x]) + (part[2][threadIdx.x] + part[3][threadIdx.x])) / (float)n;
  __syncthreads();
  for (int l = 0; l < nlayers; ++l) {
    warp_matvec<1, 8>(L.w1[l], L.b1[l], smean, hid, nullptr, 2 * D, 1, warp, NW, lane);
    __syncthreads();
    warp_matvec<2, 4>(L.w2[l], L.b2[l], hid, nullptr, gb + ((long long)l * B + b) * 2 * D, 2 * D, 0, warp, NW, lane);
    __syncthreads();
  }
}

// ---- last CVAE prior layer on its two read rows, one launch ---------------------------------------------------------
// Only the mu / logvar token rows (tokens 0 and 1) of the last prior layer are read (model_CVAE.py:78). Keys / values
// still come from every token (one tensor-core GEMM), but everything that follows acts on 2 rows per clip: as tcgen05
// launches (gather, 256-row q projection, attention with 2 valid query rows per 128-row tile, a 2-CTA block tail) that
// was four launches and ~56 us of pure pipeline latency. Here one block per clip does all of it with the lanes of a warp
// across K (bf16 weights / keys / values, fp32 activations and statistics):
//   q = Wq x + bq;  p = softmax(q k^T / sqrt(dh)) per head;  a = p v;  y = LN1(x + Wo a + bo);  out = LN2(y + W2 relu(W1 y + b1) + b2)
// (nn.TransformerEncoderLayer, post-LN, ReLU: model_CVAE.py:60-79).
struct PriorLastW {
  const __nv_bfloat16 *wq, *wo, *w1, *w2;
  const float *bq, *bo, *b1, *b2, *g1, *be1, *g2, *be2;
};

// two-vector version of warp_matvec: ys[v * ldy + o] = act(W[o, :] . xs[v * ldx ...] + b[o]) (* scale) (+ res[v * ldy + o])
// ITER groups of NV outputs are loaded together (ITER * NV * KCH 16-byte loads in flight per lane): the phases are L2-latency
// chains, one round trip per pass of the loop.
template <int KCH, int NV, int ITER>
__device__ __forceinline__ void warp_matvec2(const __nv_bfloat16* __restrict__ W, const float* __restrict__ b, const float* xs,
                                             int ldx, float* ys, int ldy, const float* res, int N, int relu, float scale,
                                             int warp, int nwarps, int lane, float* ys_mirror = nullptr) {
  constexpr int K = KCH * 256;
  float x[2][KCH * 8];
#pragma unroll
  for (int v = 0; v < 2; ++v)
#pragma unroll
    for (int c = 0; c < KCH; ++c) {
      const float4 lo = *reinterpret_cast<const float4*>(xs + v * ldx + c * 256 + lane * 8);
      const float4 hi = *reinterpret_cast<const float4*>(xs + v * ldx + c * 256 + lane * 8 + 4);
      x[v][c * 8 + 0] = lo.x; x[v][c * 8 + 1] = lo.y; x[v][c * 8 + 2] = lo.z; x[v][c * 8 + 3] = lo.w;
      x[v][c * 8 + 4] = hi.x; x[v][c * 8 + 5] = hi.y; x[v][c * 8 + 6] = hi.z; x[v][c * 8 + 7] = hi.w;
    }
  for (int ob = warp * NV; ob < N; ob += nwarps * NV * ITER) {
    uint4 wv[ITER][NV * KCH];
#pragma unroll
    for (int it = 0; it < ITER; ++it) {
      const int o0 = ob + it * nwarps * NV;
      if (o0 < N) {
#pragma unroll
        for (int i = 0; i < NV; ++i)
#pragma unroll
          for (int c = 0; c < KCH; ++c)
            wv[it][i * KCH + c] = __ldg(reinterpret_cast<const uint4*>(W + (size_t)(o0 + i) * K + c * 256 + lane * 8));
      }
    }
#pragma unroll
    for (int it = 0; it < ITER; ++it) {
      const int o0 = ob + it * nwarps * NV;
      if (o0 >= N) break;
      float v0[NV], v1[NV];
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        float a0 = 0.f, a1 = 0.f;
#pragma unroll
        for (int c = 0; c < KCH; ++c) {
          const uint32_t u[4] = {wv[it][i * KCH + c].x, wv[it][i * KCH + c].y, wv[it][i * KCH + c].z, wv[it][i * KCH + c].w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float wl = __uint_as_float(u[j] << 16), wh = __uint_as_float(u[j] & 0xffff0000u);
            a0 = fmaf(wl, x[0][c * 8 + 2 * j], a0); a0 = fmaf(wh, x[0][c * 8 + 2 * j + 1], a0);
            a1 = fmaf(wl, x[1][c * 8 + 2 * j], a1); a1 = fmaf(wh, x[1][c * 8 + 2 * j + 1], a1);
          }
        }
        v0[i] = a0; v1[i] = a1;
      }
      const float t0 = warp_reduce_t<NV>(v0, lane), t1 = warp_reduce_t<NV>(v1, lane);
      constexpr int STEP = 32 / NV;
      if ((lane & (STEP - 1)) == 0) {
        const int o = o0 + (NV == 8 ? ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1)
                                    : ((lane >> 4) & 1) * 2 + ((lane >> 3) & 1));
        const float bo = b ? __ldg(b + o) : 0.f;
        float r0 = (t0 + bo) * scale, r1 = (t1 + bo) * scale;
        if (relu == 1) { r0 = fmaxf(r0, 0.f); r1 = fmaxf(r1, 0.f); }
        else if (relu == 2) { r0 = lrelu02(r0); r1 = lrelu02(r1); }   // LeakyReLU(0.2)
        if (res) { r0 += res[o]; r1 += res[ldy + o]; }
        ys[o] = r0; ys[ldy + o] = r1;
        if (ys_mirror) { ys_mirror[o] = r0; ys_mirror[ldy + o] = r1; }   // second copy (peer CTA's shared memory)
      }
    }
  }
}

// Two clips per CLUSTER of two CTAs (for even batches >= 64): one clip per block (style_mlp_kernel) is bound by the aggregate
// L2 -> SM bandwidth (128 blocks x 1.5 MB of the same weights), and two clips per block only moved the bound to the per-SM
// load rate (measured slower in the frame).
// Here CTA r of the pair owns HALF of every layer's output features for both clips: it reads half of each weight matrix
// (768 KB per CTA, 98 MB per launch), writes its half of the hidden vector into both CTAs' shared memory (DSMEM stores) and,
// after a cluster barrier, produces its half of gamma | beta. Same summation order per output as style_mlp_kernel.
constexpr int STYLEC_THREADS = 512;
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(STYLEC_THREADS, 1)
style_mlp_cluster_kernel(const float* __restrict__ cha, int n, const StyleMlpLayers L, int nlayers, float* __restrict__ gb, int B) {
  constexpr int D = 256, NW = STYLEC_THREADS / 32;
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  pdl_trigger();
  pdl_wait();
  __shared__ __align__(16) float smean[2][D];
  __shared__ __align__(16) float hid[2][2 * D];
  const int rank = (int)cluster.block_rank();
  const int b0 = 2 * (int)(blockIdx.x >> 1), lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* peer_hid = cluster.map_shared_rank(&hid[0][0], rank ^ 1);
  {
    // token means of both clips in both CTAs (same pairing as style_mlp_kernel)
    const int c = threadIdx.x & (D - 1), v = threadIdx.x >> 8;
    const float* xb = cha + (long long)(b0 + v) * n * D + c;
    float part[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      float s0 = 0.f, s1 = 0.f;
      int i = q;
      for (; i + 4 < n; i += 8) { s0 += xb[(long long)i * D]; s1 += xb[(long long)(i + 4) * D]; }
      for (; i < n; i += 4) s0 += xb[(long long)i * D];
      part[q] = s0 + s1;
    }
    smean[v][c] = ((part[0] + part[1]) + (part[2] + part[3])) / (float)n;
  }
  __syncthreads();
  for (int l = 0; l < nlayers; ++l) {
    // hidden features [rank * D, (rank + 1) * D) of both clips -> both CTAs
    warp_matvec2<1, 8, 2>(L.w1[l] + (size_t)rank * D * D, L.b1[l] + rank * D, &smean[0][0], D, &hid[0][0] + rank * D, 2 * D, nullptr,
                          D, 2, 1.f, warp, NW, lane, peer_hid + rank * D);
    cluster.sync();
    // outputs [rank * D, (rank + 1) * D) of gamma | beta for both clips
    warp_matvec2<2, 4, 2>(L.w2[l] + (size_t)rank * D * 2 * D, L.b2[l] + rank * D, &hid[0][0], 2 * D,
                          gb + ((long long)l * B + b0) * 2 * D + rank * D, 2 * D, nullptr, D, 0, 1.f, warp, NW, lane);
    cluster.sync();   // the peer has read this layer's hidden vector before the next layer overwrites it
  }
}

// LayerNorm of two 256-wide rows held in shared memory (warps 0 and 1), two-pass statistics; out may be shared or global
__device__ __forceinline__ void ln2_rows256(const float* in, int ldi, const float* __restrict__ g, const float* __restrict__ be,
                                            float eps, float* out, int ldo_, int warp, int lane) {
  if (warp < 2) {
    const float* r = in + warp * ldi;
    float v[8];
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) { v[j] = r[lane + 32 * j]; s += v[j]; }
    const float mean = warp_sum(s) * (1.f / 256.f);
    float q = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) { const float d = v[j] - mean; q = fmaf(d, d, q); }
    const float rstd = rsqrtf(warp_sum(q) * (1.f / 256.f) + eps);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = lane + 32 * j;
      out[warp * ldo_ + c] = (v[j] - mean) * rstd * __ldg(g + c) + __ldg(be + c);
    }
  }
}

constexpr int PL_THREADS = 512;
constexpr int PL_MAXKEYS = 256;
template <int KCH2>   // dff / 256
__global__ void __launch_bounds__(PL_THREADS, 1)
cvae_prior_last_kernel(const float* __restrict__ x, int np, const __nv_bfloat16* __restrict__ kv, const PriorLastW W, int H,
                       float eps, float* __restrict__ out) {
  constexpr int D = 256, NW = PL_THREADS / 32, DFF = KCH2 * 256;
  pdl_trigger();
  extern __shared__ __align__(128) float psm[];
  float* xs = psm;                       // [2][D] the two query rows (residual)
  float* qs = xs + 2 * D;                // [2][D] q * 1/sqrt(dh); later the attention output
  float* y1 = qs + 2 * D;                // [2][D]
  float* t1 = y1 + 2 * D;                // [2][D] pre-LayerNorm rows
  float* hid = t1 + 2 * D;               // [2][DFF]
  float* part = hid + 2 * DFF;           // [4][2][D] partial P V sums
  float* sc = part + 8 * D;              // [2][H][PL_MAXKEYS] scores / probabilities
  const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int dh = D / H, lph = dh / 8;    // lanes per head when a lane owns 8 consecutive columns
  const __nv_bfloat16* kb = kv + (long long)b * np * 2 * D;
  pdl_wait();
  for (int i = threadIdx.x; i < 2 * D; i += PL_THREADS) xs[i] = x[(long long)b * np * D + i];   // tokens 0 and 1 are adjacent
  __syncthreads();
  warp_matvec2<1, 8, 2>(W.wq, W.bq, xs, D, qs, D, nullptr, D, 0, rsqrtf((float)dh), warp, NW, lane);
  __syncthreads();
  {
    // scores: a warp per key, lane = 8 consecutive columns of the key row (one 512-byte row per load)
    float q0[8], q1[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { q0[j] = qs[lane * 8 + j]; q1[j] = qs[D + lane * 8 + j]; }
    for (int j0 = warp; j0 < np; j0 += 2 * NW) {
      const int j1 = j0 + NW;
      const uint4 k0 = *reinterpret_cast<const uint4*>(kb + (long long)j0 * 2 * D + lane * 8);
      uint4 k1 = make_uint4(0, 0, 0, 0);
      if (j1 < np) k1 = *reinterpret_cast<const uint4*>(kb + (long long)j1 * 2 * D + lane * 8);
      const uint32_t u0[4] = {k0.x, k0.y, k0.z, k0.w}, u1[4] = {k1.x, k1.y, k1.z, k1.w};
      float s00 = 0.f, s01 = 0.f, s10 = 0.f, s11 = 0.f;   // s[key][row]
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float a = __uint_as_float(u0[e] << 16), c = __uint_as_float(u0[e] & 0xffff0000u);
        const float a1 = __uint_as_float(u1[e] << 16), c1 = __uint_as_float(u1[e] & 0xffff0000u);
        s00 = fmaf(a, q0[2 * e], s00); s00 = fmaf(c, q0[2 * e + 1], s00);
        s01 = fmaf(a, q1[2 * e], s01); s01 = fmaf(c, q1[2 * e + 1], s01);
        s10 = fmaf(a1, q0[2 * e], s10); s10 = fmaf(c1, q0[2 * e + 1], s10);
        s11 = fmaf(a1, q1[2 * e], s11); s11 = fmaf(c1, q1[2 * e + 1], s11);
      }
      for (int o = 1; o < lph; o <<= 1) {
        s00 += __shfl_xor_sync(0xffffffffu, s00, o); s01 += __shfl_xor_sync(0xffffffffu, s01, o);
        s10 += __shfl_xor_sync(0xffffffffu, s10, o); s11 += __shfl_xor_sync(0xffffffffu, s11, o);
      }
      if ((lane & (lph - 1)) == 0) {
        const int h = lane / lph;
        sc[(0 * H + h) * PL_MAXKEYS + j0] = s00; sc[(1 * H + h) * PL_MAXKEYS + j0] = s01;
        if (j1 < np) { sc[(0 * H + h) * PL_MAXKEYS + j1] = s10; sc[(1 * H + h) * PL_MAXKEYS + j1] = s11; }
      }
    }
  }
  __syncthreads();
  for (int r = warp; r < 2 * H; r += NW) {   // softmax of one (row, head) list per warp
    float* row = sc + r * PL_MAXKEYS;
    float v[PL_MAXKEYS / 32];
    float m = -INFINITY;
#pragma unroll
    for (int j = 0; j < PL_MAXKEYS / 32; ++j) { const int i = lane + 32 * j; v[j] = i < np ? row[i] : -INFINITY; m = fmaxf(m, v[j]); }
    m = warp_max(m);
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < PL_MAXKEYS / 32; ++j) { v[j] = __expf(v[j] - m); sum += v[j]; }
    const float inv = 1.f / warp_sum(sum);
#pragma unroll
    for (int j = 0; j < PL_MAXKEYS / 32; ++j) { const int i = lane + 32 * j; if (i < np) row[i] = v[j] * inv; }
  }
  __syncthreads();
  {
    // a = p v: thread = 2 columns x one of 4 key groups
    const int c2 = (threadIdx.x & 127) * 2, kg = threadIdx.x >> 7, h = c2 / dh;
    const __nv_bfloat16* vb = kb + D + c2;
    const float* p0 = sc + (0 * H + h) * PL_MAXKEYS;
    const float* p1 = sc + (1 * H + h) * PL_MAXKEYS;
    float a00 = 0.f, a01 = 0.f, a10 = 0.f, a11 = 0.f;   // a[row][column]
#pragma unroll 16
    for (int j = kg; j < np; j += 4) {
      const uint32_t u = *reinterpret_cast<const uint32_t*>(vb + (long long)j * 2 * D);
      const float vl = __uint_as_float(u << 16), vh = __uint_as_float(u & 0xffff0000u);
      const float w0 = p0[j], w1 = p1[j];
      a00 = fmaf(w0, vl, a00); a01 = fmaf(w0, vh, a01);
      a10 = fmaf(w1, vl, a10); a11 = fmaf(w1, vh, a11);
    }
    *reinterpret_cast<float2*>(part + (kg * 2 + 0) * D + c2) = make_float2(a00, a01);
    *reinterpret_cast<float2*>(part + (kg * 2 + 1) * D + c2) = make_float2(a10, a11);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * D; i += PL_THREADS)
    qs[i] = (part[i] + part[2 * D + i]) + (part[4 * D + i] + part[6 * D + i]);
  __syncthreads();
  warp_matvec2<1, 8, 2>(W.wo, W.bo, qs, D, t1, D, xs, D, 0, 1.f, warp, NW, lane);        // x + Wo a + bo
  __syncthreads();
  ln2_rows256(t1, D, W.g1, W.be1, eps, y1, D, warp, lane);
  __syncthreads();
  warp_matvec2<1, 8, 2>(W.w1, W.b1, y1, D, hid, DFF, nullptr, DFF, 1, 1.f, warp, NW, lane);
  __syncthreads();
  warp_matvec2<KCH2, 4, (KCH2 <= 2 ? 2 : 1)>(W.w2, W.b2, hid, DFF, t1, D, y1, D, 0, 1.f, warp, NW, lane);  // y + W2 relu(.) + b2
  __syncthreads();
  ln2_rows256(t1, D, W.g2, W.be2, eps, out + (long long)b * 2 * D, D, warp, lane);
}

constexpr int SM_MAXPL = 16;  // up to 512 columns per row (the CVAE posterior attends over 272 tokens)
__global__ void softmax_rows_kernel(float* __restrict__ S, long long rows, int ncols, float scale) {
  pdl_trigger();
  pdl_wait();
  const int warps = blockDim.x >> 5, lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * warps + (threadIdx.x >> 5);
  if (row >= rows) return;
  float* r = S + row * ncols;
  float v[SM_MAXPL];
  float m = -INFINITY;
#pragma unroll
  for (int i = 0; i < SM_MAXPL; ++i) {
    const int c = lane + 32 * i;
    v[i] = c < ncols ? r[c] * scale : -INFINITY;
    m = fmaxf(m, v[i]);
  }
  m = warp_max(m);
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < SM_MAXPL; ++i) {
    const int c = lane + 32 * i;
    v[i] = c < ncols ? expf(v[i] - m) : 0.f;
    sum += v[i];
  }
  sum = warp_sum(sum);
  const float inv = 1.f / sum;
#pragma unroll
  for (int i = 0; i < SM_MAXPL; ++i) {
    const int c = lane + 32 * i;
    if (c < ncols) r[c] = v[i] * inv;
  }
}

__global__ void add_layernorm_kernel(const float* __restrict__ x, const float* __restrict__ r,
                                     const float* __restrict__ g, const float* __restrict__ b,
                                     float* __restrict__ y, long long rows, int C, float eps,
                                     const float* __restrict__ tab_mean, const float* __restrict__ tab_std,
                                     int period, float* __restrict__ y2, __nv_bfloat16* __restrict__ y16) {
  pdl_trigger();
  pdl_wait();
  const int warps = blockDim.x >> 5, lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * warps + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float* xr = x + row * C;
  const float* rr = r ? r + row * C : nullptr;
  float s = 0.f;
  for (int c = lane; c < C; c += 32) s += xr[c] + (rr ? rr[c] : 0.f);
  const float mean = warp_sum(s) / (float)C;
  float q = 0.f;
  for (int c = lane; c < C; c += 32) {
    const float d = xr[c] + (rr ? rr[c] : 0.f) - mean;
    q = fmaf(d, d, q);
  }
  const float rstd = rsqrtf(warp_sum(q) / (float)C + eps);
  for (int c = lane; c < C; c += 32) {
    const float v = (xr[c] + (rr ? rr[c] : 0.f) - mean) * rstd * g[c] + b[c];
    if (y) y[row * C + c] = v;
    if (y16) y16[row * C + c] = __float2bfloat16_rn(v);
    if (y2) {
      const long long o = (row % period) * C + c;
      y2[row * C + c] = v * tab_std[o] + tab_mean[o];
    }
  }
}

__device__ __forceinline__ void store_bf16x4(__nv_bfloat16* p, const float4& v) {
  __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
  uint2 pk;
  pk.x = *reinterpret_cast<uint32_t*>(&lo);
  pk.y = *reinterpret_cast<uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(p) = pk;
}
__device__ __host__ inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// C = 128 * NJ: the row lives in registers (float4 per lane per 128-column group), one pass over global memory
template <int NJ>
__global__ void __launch_bounds__(256)
add_layernorm_reg_kernel(const float* __restrict__ x, const float* __restrict__ r, const float* __restrict__ g,
                         const float* __restrict__ b, float* __restrict__ y, long long rows, float eps,
                         const float* __restrict__ tab_mean, const float* __restrict__ tab_std, int period,
                         float* __restrict__ y2, __nv_bfloat16* __restrict__ y16) {
  pdl_trigger();
  pdl_wait();
  constexpr int C = 128 * NJ;
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float4* xr = reinterpret_cast<const float4*>(x + row * C);
  const float4* rr = r ? reinterpret_cast<const float4*>(r + row * C) : nullptr;
  float4 v[NJ];
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    v[j] = xr[lane + 32 * j];
    if (rr) { const float4 t = rr[lane + 32 * j]; v[j].x += t.x; v[j].y += t.y; v[j].z += t.z; v[j].w += t.w; }
    s += (v[j].x + v[j].y) + (v[j].z + v[j].w);
  }
  const float mean = warp_sum(s) / (float)C;
  float q = 0.f;
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    v[j].x -= mean; v[j].y -= mean; v[j].z -= mean; v[j].w -= mean;
    q = fmaf(v[j].x, v[j].x, q); q = fmaf(v[j].y, v[j].y, q); q = fmaf(v[j].z, v[j].z, q); q = fmaf(v[j].w, v[j].w, q);
  }
  const float rstd = rsqrtf(warp_sum(q) / (float)C + eps);
  const long long prow = y2 ? row % period : 0;
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    const int c4 = lane + 32 * j;
    const float4 gg = reinterpret_cast<const float4*>(g)[c4], bb = reinterpret_cast<const float4*>(b)[c4];
    float4 o;
    o.x = v[j].x * rstd * gg.x + bb.x; o.y = v[j].y * rstd * gg.y + bb.y;
    o.z = v[j].z * rstd * gg.z + bb.z; o.w = v[j].w * rstd * gg.w + bb.w;
    if (y) reinterpret_cast<float4*>(y + row * C)[c4] = o;
    if (y16) store_bf16x4(y16 + row * C + 4 * c4, o);
    if (y2) {
      const float4 sd = reinterpret_cast<const float4*>(tab_std + prow * C)[c4];
      const float4 mu = reinterpret_cast<const float4*>(tab_mean + prow * C)[c4];
      reinterpret_cast<float4*>(y2 + row * C)[c4] = make_float4(o.x * sd.x + mu.x, o.y * sd.y + mu.y, o.z * sd.z + mu.z, o.w * sd.w + mu.w);
    }
  }
}

__global__ void cvae_prior_tokens_kernel(const float* __restrict__ mu_token, const float* __restrict__ lv_token,
                                         const float* __restrict__ cond, const float* __restrict__ pe,
                                         float* __restrict__ tok, __nv_bfloat16* __restrict__ tok16, int ncond, int C,
                                         long long total) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int n = ncond + 2;
  const int c = (int)(i % C);
  const int t = (int)((i / C) % n);
  const long long b = i / ((long long)C * n);
  float v;
  if (t == 0) v = mu_token[c];
  else if (t == 1) v = lv_token[c];
  else v = cond[(b * ncond + (t - 2)) * C + c];
  v += pe[(long long)t * C + c];
  tok[i] = v;
  if (tok16) tok16[i] = __float2bfloat16_rn(v);
}

__global__ void cvae_memory_kernel(const float* __restrict__ prior_out, int prior_tokens,
                                   const float* __restrict__ eps, const float* __restrict__ cond,
                                   float* __restrict__ mem, __nv_bfloat16* __restrict__ mem16,
                                   float* __restrict__ mu_out, float* __restrict__ lv_out, int ncond, int C,
                                   long long total) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int n = ncond + 1;
  const int c = (int)(i % C);
  const int t = (int)((i / C) % n);
  const long long b = i / ((long long)C * n);
  if (t == 0) {
    const float mu = prior_out[(b * prior_tokens + 0) * C + c];
    const float lv = prior_out[(b * prior_tokens + 1) * C + c];
    float z = mu;
    if (eps) z = mu + eps[b * C + c] * expf(0.5f * lv);
    if (mem) mem[i] = z;
    if (mem16) mem16[i] = __float2bfloat16_rn(z);
    if (mu_out) mu_out[b * C + c] = mu;
    if (lv_out) lv_out[b * C + c] = lv;
  } else {
    const float v = cond[(b * ncond + (t - 1)) * C + c];
    if (mem) mem[i] = v;
    if (mem16) mem16[i] = __float2bfloat16_rn(v);
  }
}

__global__ void cvae_condition_kernel(const float* __restrict__ src_cnt, const float* __restrict__ prev,
                                      const float* __restrict__ m0, const float* __restrict__ s0,
                                      const float* __restrict__ m1, const float* __restrict__ s1,
                                      float* __restrict__ cond, int n, int C, long long total) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long per = (long long)n * C;
  const long long b = i / (2 * per);
  const long long r = i - b * 2 * per;
  if (r < per) cond[i] = (src_cnt[b * per + r] - m0[r]) / s0[r];
  else cond[i] = (prev[b * per + (r - per)] - m1[r - per]) / s1[r - per];
}

// ---- float4 / 32-bit-index variants of the three CVAE assembly kernels (C % 4 == 0, < 2^31 elements) ----

__global__ void cvae_prior_tokens_v4_kernel(const float4* __restrict__ mu_token, const float4* __restrict__ lv_token,
                                            const float4* __restrict__ cond, const float4* __restrict__ pe,
                                            float4* __restrict__ tok, __nv_bfloat16* __restrict__ tok16, unsigned ncond,
                                            unsigned C4, unsigned total4) {
  pdl_trigger();
  pdl_wait();
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const unsigned n = ncond + 2;
  const unsigned row = i / C4, c = i - row * C4;
  const unsigned b = row / n, t = row - b * n;
  float4 v = t == 0 ? mu_token[c] : t == 1 ? lv_token[c] : cond[(b * ncond + (t - 2)) * C4 + c];
  const float4 p = pe[t * C4 + c];
  v.x += p.x; v.y += p.y; v.z += p.z; v.w += p.w;
  tok[i] = v;
  if (tok16) store_bf16x4(tok16 + 4ull * i, v);
}

__global__ void cvae_memory_v4_kernel(const float4* __restrict__ prior_out, unsigned prior_tokens,
                                      const float4* __restrict__ eps, const float4* __restrict__ cond,
                                      float4* __restrict__ mem, __nv_bfloat16* __restrict__ mem16,
                                      float4* __restrict__ mu_out, float4* __restrict__ lv_out, unsigned ncond, unsigned C4,
                                      unsigned total4) {
  pdl_trigger();
  pdl_wait();
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const unsigned n = ncond + 1;
  const unsigned row = i / C4, c = i - row * C4;
  const unsigned b = row / n, t = row - b * n;
  float4 v;
  if (t == 0) {
    const float4 mu = prior_out[(b * prior_tokens + 0) * C4 + c];
    const float4 lv = prior_out[(b * prior_tokens + 1) * C4 + c];
    v = mu;
    if (eps) {
      const float4 e = eps[b * C4 + c];
      v.x = mu.x + e.x * expf(0.5f * lv.x); v.y = mu.y + e.y * expf(0.5f * lv.y);
      v.z = mu.z + e.z * expf(0.5f * lv.z); v.w = mu.w + e.w * expf(0.5f * lv.w);
    }
    if (mu_out) mu_out[b * C4 + c] = mu;
    if (lv_out) lv_out[b * C4 + c] = lv;
  } else {
    v = cond[(b * ncond + (t - 1)) * C4 + c];
  }
  if (mem) mem[i] = v;
  if (mem16) store_bf16x4(mem16 + 4ull * i, v);
}

__global__ void cvae_condition_v4_kernel(const float4* __restrict__ src_cnt, const float4* __restrict__ prev,
                                         const float4* __restrict__ m0, const float4* __restrict__ s0,
                                         const float4* __restrict__ m1, const float4* __restrict__ s1,
                                         float4* __restrict__ cond, unsigned per4, unsigned total4) {
  pdl_trigger();
  pdl_wait();
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const unsigned b = i / (2 * per4);
  unsigned r = i - b * 2 * per4;
  float4 x, m, sd;
  if (r < per4) { x = src_cnt[b * per4 + r]; m = m0[r]; sd = s0[r]; }
  else { r -= per4; x = prev[b * per4 + r]; m = m1[r]; sd = s1[r]; }
  cond[i] = make_float4((x.x - m.x) / sd.x, (x.y - m.y) / sd.y, (x.z - m.z) / sd.z, (x.w - m.w) / sd.w);
}


__global__ void affine_rows_kernel(const float* __restrict__ x, const float* __restrict__ mu,
                                   const float* __restrict__ sd, float* __restrict__ out, long long total,
                                   int C, int period, int ld_in, float* __restrict__ copy) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long o = i % ((long long)period * C);
  const long long r = i / C;
  const float v = x[r * ld_in + (i - r * C)];
  if (out) out[i] = v * sd[o] + mu[o];
  if (copy) copy[i] = v;
}

// to_mot's output layer in one pass (model.py:77-78 + the driver's de-normalisation, test_fullframework.py:457):
//   Ytil = x W^T + b (x: bf16 rows that already went through LeakyReLU, K = 16 KS -> N <= 16 channels), Y = Ytil * std + mean
// on mma.sync m16n8k16 (bf16 operands, fp32 accumulation): the N x K weights are constant B fragments in registers, a
// warp takes 16 rows per pass with its A fragments loaded straight from global memory (4-byte pieces that L1 merges
// into whole sectors), results go through a staging tile so that the stores - and the table look-ups of the
// de-normalisation - are coalesced. Replaces a 15-wide tensor-core GEMM (16 us: all epilogue) and a scalar affine pass
// (14 us); a first SIMT version (thread per row, broadcast LDS.128 weights) was shared-memory-issue-bound at 27 us.
constexpr int OC_ROWS = 256;
__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
template <int KS>
__global__ void __launch_bounds__(OC_ROWS)
out_conv_affine_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ W, const float* __restrict__ bias,
                       const float* __restrict__ mu, const float* __restrict__ sd, float* __restrict__ ytil,
                       float* __restrict__ y, int R, int N, int period) {
  constexpr int K = KS * 16, PASSES = OC_ROWS / 128;
  pdl_trigger();
  extern __shared__ __align__(16) float osm[];
  float* stage = osm;                         // [OC_ROWS][N]
  float* tab = osm + OC_ROWS * N;             // [2][period * N] de-normalisation tables (std, mean)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
  const int pn = period * N;
  // constants (weights, tables): loaded before the grid dependency resolves
  if (y)
    for (int i = threadIdx.x; i < pn; i += OC_ROWS) { tab[i] = sd[i]; tab[pn + i] = mu[i]; }
  uint32_t wb[KS][2][2];                      // B fragments: B[k][n] = W[n][k], two n-tiles of 8 (columns >= N are zero)
#pragma unroll
  for (int ks = 0; ks < KS; ++ks)
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int n = nt * 8 + g, k = ks * 16 + 2 * t + 8 * h;
        float2 wv = make_float2(0.f, 0.f);
        if (n < N) wv = __ldg(reinterpret_cast<const float2*>(W + n * K + k));
        const __nv_bfloat162 p = __floats2bfloat162_rn(wv.x, wv.y);
        wb[ks][nt][h] = *reinterpret_cast<const uint32_t*>(&p);
      }
  float bz[2][2];
#pragma unroll
  for (int nt = 0; nt < 2; ++nt)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int n = nt * 8 + 2 * t + e;
      bz[nt][e] = (bias && n < N) ? __ldg(bias + n) : 0.f;
    }
  pdl_wait();
  const int ntiles = (R + OC_ROWS - 1) / OC_ROWS;
  uint32_t a[PASSES][KS][4];
  auto load_a = [&](int tile) {               // all of a tile's fragment loads in flight at once
    const int row0 = tile * OC_ROWS;
#pragma unroll
    for (int ps = 0; ps < PASSES; ++ps) {
      const int r0 = row0 + ps * 128 + warp * 16 + g, r1 = r0 + 8;
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
        const uint32_t* p0 = reinterpret_cast<const uint32_t*>(x + (long long)r0 * K + ks * 16 + 2 * t);
        const uint32_t* p1 = reinterpret_cast<const uint32_t*>(x + (long long)r1 * K + ks * 16 + 2 * t);
        a[ps][ks][0] = r0 < R ? __ldg(p0) : 0u;
        a[ps][ks][1] = r1 < R ? __ldg(p1) : 0u;
        a[ps][ks][2] = r0 < R ? __ldg(p0 + 4) : 0u;
        a[ps][ks][3] = r1 < R ? __ldg(p1 + 4) : 0u;
      }
    }
  };
  if ((int)blockIdx.x < ntiles) load_a(blockIdx.x);
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int row0 = tile * OC_ROWS;
#pragma unroll
    for (int ps = 0; ps < PASSES; ++ps) {
      const int lr = ps * 128 + warp * 16 + g;
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        float d[4] = {bz[nt][0], bz[nt][1], bz[nt][0], bz[nt][1]};
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) mma_bf16_16816(d, a[ps][ks], wb[ks][nt][0], wb[ks][nt][1]);
        const int n = nt * 8 + 2 * t;
        if (n < N) { stage[lr * N + n] = d[0]; stage[(lr + 8) * N + n] = d[2]; }
        if (n + 1 < N) { stage[lr * N + n + 1] = d[1]; stage[(lr + 8) * N + n + 1] = d[3]; }
      }
    }
    __syncthreads();
    if (tile + (int)gridDim.x < ntiles) load_a(tile + gridDim.x);   // next tile's rows arrive while this one is stored
    const int nvalid = min(OC_ROWS, R - row0) * N;
    const long long g0 = (long long)row0 * N;
    int o = (int)(g0 % pn) + (int)threadIdx.x;       // table index of this thread's first element
    for (int i = threadIdx.x; i < nvalid; i += OC_ROWS, o += OC_ROWS) {
      while (o >= pn) o -= pn;
      const float v = stage[i];
      if (ytil) ytil[g0 + i] = v;
      if (y) y[g0 + i] = fmaf(v, tab[o], tab[pn + o]);
    }
    __syncthreads();
  }
}

__global__ void broadcast_rows_kernel(const float* __restrict__ x, float* __restrict__ out,
                                      __nv_bfloat16* __restrict__ out16, long long n_elems, long long total) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const float v = x[i % n_elems];
  out[i] = v;
  if (out16) out16[i] = __float2bfloat16_rn(v);
}

__global__ void add_table_kernel(const float* __restrict__ a, const float* __restrict__ table,
                                 float* __restrict__ out, long long total, int C, int period) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  out[i] = a[i] + table[i % ((long long)period * C)];
}

__global__ void cast_f32_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, long long n) {
  pdl_trigger();
  pdl_wait();
  const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i + 3 < n) {
    const float4 v = *reinterpret_cast<const float4*>(x + i);
    __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
    uint2 pk;
    pk.x = *reinterpret_cast<uint32_t*>(&lo);
    pk.y = *reinterpret_cast<uint32_t*>(&hi);
    *reinterpret_cast<uint2*>(y + i) = pk;
  } else {
    for (long long j = i; j < n; ++j) y[j] = __float2bfloat16_rn(x[j]);
  }
}

// out[b, i, :] = x[b, i, :] for i < take (the first `take` tokens of every batch element), fp32 + bf16
__global__ void gather_token_rows_kernel(const float* __restrict__ x, const __nv_bfloat16* __restrict__ x16, int n,
                                         int take, int C, long long total, float* __restrict__ out,
                                         __nv_bfloat16* __restrict__ out16) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int c = (int)(i % C);
  const int t = (int)((i / C) % take);
  const long long b = i / ((long long)C * take);
  const long long src = (b * n + t) * C + c;
  if (out) out[i] = x[src];
  if (out16) out16[i] = x16 ? x16[src] : __float2bfloat16_rn(x[src]);
}

inline unsigned blocks_for(long long total, int bs) { return (unsigned)((total + bs - 1) / bs); }

}  // namespace

int graph_agg_first(const float* in, const float* A, float* out, int BT, int V, int C, int Kk, int lrelu,
                    cudaStream_t s, __nv_bfloat16* out16) {
  MOCHA_CHECK_ARG(in && A && (out || out16) && BT > 0 && V > 0 && C > 0 && Kk > 0, "graph_agg_first: bad args");
  if (!out && out16 && V <= GAS_VMAX && Kk <= 4 && (C & 3) == 0 && aligned16(in) && (reinterpret_cast<uintptr_t>(out16) & 7) == 0) {
    const long long total = (long long)BT * (C / 4);
    launch_k(graph_agg_small_kernel, blocks_for(total, 256), 256, 0, s, in, A, out16, total, V, C / 4, Kk, lrelu);
    count_launch();
    MOCHA_LAUNCH_CHECK("graph_agg_small");
    return MOCHA_OK;
  }
  size_t smem = (size_t)(V * C + 2 * Kk * V * V + Kk * V) * sizeof(float);
  MOCHA_CHECK_ARG(smem <= 48 * 1024, "graph_agg_first: tile too large (%zu B)", smem);
  launch_k(graph_agg_first_kernel, BT, 256, smem, s, in, A, out, out16, V, C, Kk, lrelu);
  count_launch();
  MOCHA_LAUNCH_CHECK("graph_agg_first");
  return MOCHA_OK;
}

int embed_graph_agg(const float* X, const float* Wemb, const float* bemb, const float* A, __nv_bfloat16* out16, int BT,
                    int V, int Cin, int C, int Kk, cudaStream_t s, int ldo) {
  if (ldo <= 0) ldo = Kk * C;
  MOCHA_CHECK_ARG(ldo >= Kk * C && (ldo & 3) == 0, "embed_graph_agg: bad output pitch %d", ldo);
  MOCHA_CHECK_ARG(X && Wemb && A && out16 && BT > 0 && V > 0 && Cin > 0 && Kk > 0, "embed_graph_agg: bad args");
  MOCHA_CHECK_ARG(C >= 8 && C <= 128 && (C & 3) == 0 && 128 % C == 0, "embed_graph_agg: C=%d unsupported", C);
  MOCHA_CHECK_ARG(Cin <= EMB_MAXCIN, "embed_graph_agg: Cin=%d > %d unsupported", Cin, EMB_MAXCIN);
  MOCHA_CHECK_ARG(V % 4 == 0 && V <= 32, "embed_graph_agg: V=%d must be a multiple of 4, at most 32", V);
  constexpr int G = 4;
  if (V == 24 && Kk == 3 && C == 64 && ldo % 8 == 0 && ldo <= 512 &&
      ((reinterpret_cast<uintptr_t>(out16) | reinterpret_cast<uintptr_t>(X)) & 15) == 0) {
    constexpr int XT = (G * 24 + 15) / 16;
    const size_t smem_mma = (size_t)(XT * 16 * EMB_XLD + G * 24 * EMB_HLD) * sizeof(float) + (size_t)G * 24 * (ldo + 8) * 2;
    static size_t configured_mma = 0;
    if (smem_mma > configured_mma) {
      MOCHA_CUDA(cudaFuncSetAttribute(embed_graph_agg_mma_kernel<24, 3, G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_mma));
      configured_mma = smem_mma;
    }
    static int sms = 0;
    if (!sms) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev); if (sms <= 0) sms = 148; }
    const int ngroups = (BT + G - 1) / G;
    const int grid = ngroups < 2 * sms ? ngroups : 2 * sms;
    launch_k(embed_graph_agg_mma_kernel<24, 3, G>, grid, 256, smem_mma, s, X, Wemb, bemb, A, out16, BT, Cin, ldo);
    count_launch();
    MOCHA_LAUNCH_CHECK("embed_graph_agg_mma");
    return MOCHA_OK;
  }
  const size_t smem = (size_t)(G * V * C + G * V * EMB_MAXCIN + 2 * Kk * V * V + Kk * V) * sizeof(float) +
                      (size_t)V * (ldo - Kk * C) * 2 + 16;
  static size_t configured = 0;
  if (smem > configured) {
    MOCHA_CHECK_ARG(smem <= 200 * 1024, "embed_graph_agg: tile too large (%zu B)", smem);
    if (smem > 48 * 1024)
      MOCHA_CUDA(cudaFuncSetAttribute(embed_graph_agg_kernel<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  launch_k(embed_graph_agg_kernel<G>, (BT + G - 1) / G, 256, smem, s, X, Wemb, bemb, A, out16, BT, V, Cin, C, Kk, ldo);
  count_launch();
  MOCHA_LAUNCH_CHECK("embed_graph_agg");
  return MOCHA_OK;
}

// to_mot's JointBlock input for the tensor-core path: the graph aggregation after the 1x1 conv (un-pooling
// folded into A2) written directly as the temporal conv's operand - bf16, nearest x tdiv up-sampling in time
// and reflect padding included - instead of an fp32 tensor plus a pad / cast pass.
// in [B*Ts, U, Kk*C] fp32 -> out16 [B, T + 2*pad, Wn, C] with T = Ts * tdiv.
__global__ void __launch_bounds__(256)
graph_agg_kv_pad16_kernel(const float* __restrict__ in, const float* __restrict__ A2, __nv_bfloat16* __restrict__ out16,
                          int Ts, int tdiv, int pad, int U, int Wn, int C, int Kk) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float sm[];
  const int KC = Kk * C, KU = Kk * U;
  float* xs = sm;                                   // [U][Kk*C]
  float* lval = sm + U * KC;                        // [Wn][Kk*U] non-zero weights of output node w
  int* loff = reinterpret_cast<int*>(lval + Wn * KU);  // [Wn][Kk*U] their source offsets u*KC + k*C
  int* lcnt = loff + Wn * KU;                       // [Wn]
  __shared__ int dst_tp[16];
  __shared__ int n_dst;
  const int b = blockIdx.x / Ts, t2 = blockIdx.x - b * Ts;
  const int T = Ts * tdiv, Tp = T + 2 * pad;
  const float* src = in + (long long)blockIdx.x * U * KC;
  for (int i = threadIdx.x * 4; i < U * KC; i += blockDim.x * 4)
    *reinterpret_cast<float4*>(xs + i) = *reinterpret_cast<const float4*>(src + i);
  if (threadIdx.x < Wn) {
    // compact list of the (k, u) pairs that feed output node w (ascending (k, u): fixed summation order)
    const int w = threadIdx.x;
    int n = 0;
    for (int k = 0; k < Kk; ++k)
      for (int u = 0; u < U; ++u) {
        const float av = A2[(k * U + u) * Wn + w];
        if (av != 0.f) { lval[w * KU + n] = av; loff[w * KU + n] = u * KC + k * C; ++n; }
      }
    lcnt[w] = n;
  }
  if (threadIdx.x == 255) {
    // padded frames whose (reflected, down-sampled) source frame is t2: tdiv interior ones plus borders
    int n = 0;
    for (int tp = 0; tp < Tp && n < 16; ++tp) {
      int t = tp - pad;
      if (t < 0) t = -t;
      if (t >= T) t = 2 * (T - 1) - t;
      if (t / tdiv == t2) dst_tp[n++] = tp;
    }
    n_dst = n;
  }
  __syncthreads();
  const int C4 = C / 4;
  for (int idx = threadIdx.x; idx < Wn * C4; idx += blockDim.x) {
    const int w = idx / C4, c = (idx - w * C4) * 4;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    const int n = lcnt[w];
    for (int i = 0; i < n; ++i) {
      const float4 x = *reinterpret_cast<const float4*>(xs + loff[w * KU + i] + c);
      const float av = lval[w * KU + i];
      a.x = fmaf(x.x, av, a.x); a.y = fmaf(x.y, av, a.y); a.z = fmaf(x.z, av, a.z); a.w = fmaf(x.w, av, a.w);
    }
    __nv_bfloat162 lo = __floats2bfloat162_rn(a.x, a.y), hi = __floats2bfloat162_rn(a.z, a.w);
    uint2 pk;
    pk.x = *reinterpret_cast<uint32_t*>(&lo);
    pk.y = *reinterpret_cast<uint32_t*>(&hi);
    for (int j = 0; j < n_dst; ++j)
      *reinterpret_cast<uint2*>(out16 + (((long long)b * Tp + dst_tp[j]) * Wn + w) * C + c) = pk;
  }
}

// Streaming variant: one thread per (source frame, group of 4 output nodes, 4 channels). The Kk * U source vectors of a
// frame are re-read by its 6 node groups through L1 (they are 4.6 KB), nothing is staged or built per block, and every
// store is an 8-byte piece of a coalesced 128-byte row segment. Geometry limits: Kk * U <= 24 adjacency terms per node.
constexpr int GKP_TERMS = 24;
__global__ void __launch_bounds__(256, 5)   // 5 blocks per SM: the 720-block grid of the 128-clip step runs as one wave
graph_agg_kv_pad16_stream_kernel(const float* __restrict__ in, const float* __restrict__ A2, __nv_bfloat16* __restrict__ out16,
                                 long long total, int Ts, int tdiv, int pad, int U, int Wn, int C4, int Kk) {
  pdl_trigger();
  __shared__ __align__(16) float As[GKP_TERMS * 32];     // [Kk*U][Wn] (Wn <= 32)
  const int KU = Kk * U;
  for (int i = threadIdx.x; i < KU * Wn; i += blockDim.x) As[i] = A2[i];   // constant: before the grid dependency
  pdl_wait();
  __syncthreads();
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int WG = Wn / 4, C = C4 * 4, KC = Kk * C;
  const int c = (int)(idx % C4) * 4;
  const long long r = idx / C4;
  const int wg = (int)(r % WG);
  const long long bt = r / WG;
  const int b = (int)(bt / Ts), t2 = (int)(bt - (long long)b * Ts);
  const float* src = in + bt * U * KC + c;
  float4 acc[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 6
  for (int ku = 0; ku < KU; ++ku) {            // ascending (k, u): the list kernel's summation order
    const int k = ku / U, u = ku - k * U;
    const float4 x = *reinterpret_cast<const float4*>(src + u * KC + k * C);
    const float4 a = *reinterpret_cast<const float4*>(As + ku * Wn + wg * 4);
    acc[0].x = fmaf(x.x, a.x, acc[0].x); acc[0].y = fmaf(x.y, a.x, acc[0].y); acc[0].z = fmaf(x.z, a.x, acc[0].z); acc[0].w = fmaf(x.w, a.x, acc[0].w);
    acc[1].x = fmaf(x.x, a.y, acc[1].x); acc[1].y = fmaf(x.y, a.y, acc[1].y); acc[1].z = fmaf(x.z, a.y, acc[1].z); acc[1].w = fmaf(x.w, a.y, acc[1].w);
    acc[2].x = fmaf(x.x, a.z, acc[2].x); acc[2].y = fmaf(x.y, a.z, acc[2].y); acc[2].z = fmaf(x.z, a.z, acc[2].z); acc[2].w = fmaf(x.w, a.z, acc[2].w);
    acc[3].x = fmaf(x.x, a.w, acc[3].x); acc[3].y = fmaf(x.y, a.w, acc[3].y); acc[3].z = fmaf(x.z, a.w, acc[3].z); acc[3].w = fmaf(x.w, a.w, acc[3].w);
  }
  uint2 pk[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    __nv_bfloat162 lo = __floats2bfloat162_rn(acc[j].x, acc[j].y), hi = __floats2bfloat162_rn(acc[j].z, acc[j].w);
    pk[j].x = *reinterpret_cast<uint32_t*>(&lo);
    pk[j].y = *reinterpret_cast<uint32_t*>(&hi);
  }
  // padded frames whose (reflected, down-sampled) source frame is t2: the tdiv interior ones plus reflected borders
  const int T = Ts * tdiv, Tp = T + 2 * pad;
  __nv_bfloat16* ob = out16 + (long long)b * Tp * Wn * C + (long long)(wg * 4) * C + c;
  for (int i = 0; i < tdiv; ++i) {
    __nv_bfloat16* o = ob + (long long)(pad + t2 * tdiv + i) * Wn * C;
#pragma unroll
    for (int j = 0; j < 4; ++j) *reinterpret_cast<uint2*>(o + j * C) = pk[j];
  }
  for (int e = 0; e < 2 * pad; ++e) {
    const int tp = e < pad ? e : T + e;          // border frame (front: 0..pad-1, back: T+pad..T+2pad-1)
    int t = tp - pad;
    t = t < 0 ? -t : 2 * (T - 1) - t;
    if (t / tdiv == t2) {
      __nv_bfloat16* o = ob + (long long)tp * Wn * C;
#pragma unroll
      for (int j = 0; j < 4; ++j) *reinterpret_cast<uint2*>(o + j * C) = pk[j];
    }
  }
}

// reflect-pad borders of a [B, T + 2*pad, V*C] bf16 tensor whose interior rows are already written
__global__ void reflect_border_kernel(__nv_bfloat16* __restrict__ xp, int T, int pad, long long row8, long long total8) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total8) return;
  const long long e = i % row8;
  const long long r = i / row8;
  const int j = (int)(r % (2 * pad));
  const long long b = r / (2 * pad);
  const int Tp = T + 2 * pad;
  const int tp = j < pad ? j : T + j;           // padded index of the border frame
  int t = tp - pad;
  t = t < 0 ? -t : 2 * (T - 1) - t;             // reflected source frame
  uint4* base = reinterpret_cast<uint4*>(xp) + b * Tp * row8;
  base[(long long)tp * row8 + e] = base[(long long)(t + pad) * row8 + e];
}

int reflect_border_fill(__nv_bfloat16* xp, int B, int T, int pad, long long row_elems, cudaStream_t s) {
  MOCHA_CHECK_ARG(xp && B > 0 && T > pad && pad > 0 && row_elems % 8 == 0, "reflect_border_fill: bad args");
  const long long row8 = row_elems / 8, total8 = (long long)B * 2 * pad * row8;
  launch_k(reflect_border_kernel, blocks_for(total8, 256), 256, 0, s, xp, T, pad, row8, total8);
  count_launch();
  MOCHA_LAUNCH_CHECK("reflect_border_fill");
  return MOCHA_OK;
}

int graph_agg_kv(const float* in, const float* A2, float* out, int BT, int U, int Wn, int C, int Kk,
                 cudaStream_t s) {
  MOCHA_CHECK_ARG(in && A2 && out && BT > 0 && U > 0 && Wn > 0 && C > 0 && Kk > 0, "graph_agg_kv: bad args");
  size_t smem = (size_t)(U * Kk * C + Kk * U * Wn) * sizeof(float);
  MOCHA_CHECK_ARG(smem <= 48 * 1024, "graph_agg_kv: tile too large (%zu B)", smem);
  launch_k(graph_agg_kv_kernel, BT, 256, smem, s, in, A2, out, U, Wn, C, Kk);
  count_launch();
  MOCHA_LAUNCH_CHECK("graph_agg_kv");
  return MOCHA_OK;
}

int graph_agg_kv_pad16(const float* in, const float* A2, __nv_bfloat16* out16, int B, int Ts, int tdiv, int pad, int U,
                       int Wn, int C, int Kk, cudaStream_t s) {
  MOCHA_CHECK_ARG(in && A2 && out16 && B > 0 && Ts > 0 && tdiv >= 1 && pad >= 0 && U > 0 && Wn > 0 && Wn <= 255 && C > 0 &&
                      (C & 3) == 0 && Kk > 0 && (reinterpret_cast<uintptr_t>(in) & 15) == 0,
                  "graph_agg_kv_pad16: bad args");
  MOCHA_CHECK_ARG(tdiv + 2 * pad <= 16 && pad < Ts * tdiv, "graph_agg_kv_pad16: tdiv / pad too large");
  if (Kk * U <= GKP_TERMS && Wn % 4 == 0 && Wn <= 32 && (reinterpret_cast<uintptr_t>(out16) & 7) == 0) {
    const long long total = (long long)B * Ts * (Wn / 4) * (C / 4);
    launch_k(graph_agg_kv_pad16_stream_kernel, blocks_for(total, 256), 256, 0, s, in, A2, out16, total, Ts, tdiv, pad, U, Wn, C / 4, Kk);
    count_launch();
    MOCHA_LAUNCH_CHECK("graph_agg_kv_pad16_stream");
    return MOCHA_OK;
  }
  const size_t smem = (size_t)(U * Kk * C + 2 * Kk * U * Wn + Wn) * sizeof(float);
  MOCHA_CHECK_ARG(smem <= 48 * 1024, "graph_agg_kv_pad16: tile too large (%zu B)", smem);
  launch_k(graph_agg_kv_pad16_kernel, B * Ts, 256, smem, s, in, A2, out16, Ts, tdiv, pad, U, Wn, C, Kk);
  count_launch();
  MOCHA_LAUNCH_CHECK("graph_agg_kv_pad16");
  return MOCHA_OK;
}

int pool_joint_body(const float* in, const float* Wp, float* out, int B, int T, int V, int P, int C, int tp,
                    cudaStream_t s) {
  MOCHA_CHECK_ARG(in && Wp && out && B > 0 && T > 0 && V > 0 && C > 0, "pool_joint_body: bad args");
  MOCHA_CHECK_ARG(P > 0 && P <= POOL_MAXP, "pool_joint_body: P=%d unsupported (max %d)", P, POOL_MAXP);
  MOCHA_CHECK_ARG(tp > 0 && T % tp == 0, "pool_joint_body: T=%d not a multiple of tp=%d", T, tp);
  launch_k(pool_joint_body_kernel, B * (T / tp), 256, (size_t)V * P * sizeof(float), s, in, Wp, out, T, V, P, C, tp);
  count_launch();
  MOCHA_LAUNCH_CHECK("pool_joint_body");
  return MOCHA_OK;
}

int pool_graph_agg(const __nv_bfloat16* in, const float* Wp, const float* A, __nv_bfloat16* out16, int B, int T, int V,
                   int P, int C, int tp, int Kk, cudaStream_t s) {
  MOCHA_CHECK_ARG(in && Wp && A && out16 && B > 0 && T > 0 && V > 0 && C > 0 && (C & 1) == 0 && Kk > 0, "pool_graph_agg: bad args");
  MOCHA_CHECK_ARG(P > 0 && P <= POOL_MAXP, "pool_graph_agg: P=%d unsupported (max %d)", P, POOL_MAXP);
  MOCHA_CHECK_ARG(tp > 0 && T % tp == 0, "pool_graph_agg: T=%d not a multiple of tp=%d", T, tp);
  const size_t smem = (size_t)(Kk * P * P + 2 * P * V + P) * sizeof(float);
  if (C % 4 == 0 && C / 4 <= 128 && 128 % (C / 4) == 0 && (reinterpret_cast<uintptr_t>(in) & 7) == 0 &&
      (reinterpret_cast<uintptr_t>(out16) & 7) == 0) {
    const int groups = B * (T / tp), gpb = 128 / (C / 4);
    launch_k(pool_graph_agg_v4_kernel, (groups + gpb - 1) / gpb, 128, smem, s, in, Wp, A, out16, groups, T, V, P, C, tp, Kk);
    count_launch();
    MOCHA_LAUNCH_CHECK("pool_graph_agg_v4");
    return MOCHA_OK;
  }
  launch_k(pool_graph_agg_kernel, B * (T / tp), 128, smem, s, in, Wp, A, out16, T, V, P, C, tp, Kk);
  count_launch();
  MOCHA_LAUNCH_CHECK("pool_graph_agg");
  return MOCHA_OK;
}

int instance_norm_tokens(const float* x, int B, int n, int C, float eps, const float* gb, float* y,
                         const float* tab_mean, const float* tab_std, float* y2, cudaStream_t s,
                         __nv_bfloat16* y16, __nv_bfloat16* y2h, const float* y2h_center) {
  MOCHA_CHECK_ARG(x && B > 0 && n > 1 && C > 0, "instance_norm_tokens: bad args");
  MOCHA_CHECK_ARG(y || y2 || y16 || y2h, "instance_norm_tokens: no output");
  MOCHA_CHECK_ARG(!(y2 || y2h) || (tab_mean && tab_std), "instance_norm_tokens: y2 needs its table");
  const bool al = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(gb)) & 15) == 0 &&
                  (reinterpret_cast<uintptr_t>(y16) & 7) == 0;
  const bool al2 = ((reinterpret_cast<uintptr_t>(tab_mean) | reinterpret_cast<uintptr_t>(tab_std) | reinterpret_cast<uintptr_t>(y2) |
                     reinterpret_cast<uintptr_t>(y2h_center)) & 15) == 0 && (reinterpret_cast<uintptr_t>(y2h) & 7) == 0;
  if (n <= 128 && (y16 || y2 || y2h) && (C % 64) == 0 && al && al2)   // float4 kernel (bf16 twin and / or matcher query)
    launch_k(instance_norm_tokens_v4_kernel, dim3(B, C / 64), 256, 0, s, x, n, C, eps, gb, y, y16, (__nv_bfloat16*)nullptr, tab_mean,
             tab_std, y2, y2h, y2h_center);
  else if (n <= 128)
    launch_k(instance_norm_tokens_reg_kernel, dim3(B, (C + 31) / 32), 256, 0, s, x, n, C, eps, gb, y, tab_mean, tab_std, y2, y16, y2h, y2h_center);
  else
    launch_k(instance_norm_tokens_kernel, dim3(B, (C + 31) / 32), 256, 0, s, x, n, C, eps, gb, y, tab_mean, tab_std, y2, y16, y2h, y2h_center);
  count_launch();
  MOCHA_LAUNCH_CHECK("instance_norm_tokens");
  return MOCHA_OK;
}

int adain_norm_tokens(const float* x, int B, int n, int C, float eps, const float* gb, float* y, __nv_bfloat16* q16,
                      cudaStream_t s) {
  MOCHA_CHECK_ARG(x && gb && y && q16 && B > 0 && n > 1 && n <= 128 && (C % 64) == 0, "adain_norm_tokens: bad args");
  MOCHA_CHECK_ARG(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(gb)) & 15) == 0 &&
                      (reinterpret_cast<uintptr_t>(q16) & 7) == 0, "adain_norm_tokens: operands must be 16 B aligned");
  launch_k(instance_norm_tokens_v4_kernel, dim3(B, C / 64), 256, 0, s, x, n, C, eps, gb, y, (__nv_bfloat16*)nullptr, q16,
           (const float*)nullptr, (const float*)nullptr, (float*)nullptr, (__nv_bfloat16*)nullptr, (const float*)nullptr);
  count_launch();
  MOCHA_LAUNCH_CHECK("adain_norm_tokens");
  return MOCHA_OK;
}

int token_mean(const float* x, int B, int n, int C, float* out, cudaStream_t s) {
  MOCHA_CHECK_ARG(x && out && B > 0 && n > 0 && C > 0, "token_mean: bad args");
  launch_k(token_mean_kernel, B, 256, 0, s, x, n, C, out);
  count_launch();
  MOCHA_LAUNCH_CHECK("token_mean");
  return MOCHA_OK;
}

bool style_mlp_supported(int D, int nlayers) { return D == 256 && nlayers >= 1 && nlayers <= MOCHA_MAX_DEPTH; }

int style_mlp(const float* cha, int B, int n, int D, int nlayers, const __nv_bfloat16* const* w1, const float* const* b1,
              const __nv_bfloat16* const* w2, const float* const* b2, float* gb, cudaStream_t s) {
  MOCHA_CHECK_ARG(cha && gb && B > 0 && n > 0 && style_mlp_supported(D, nlayers), "style_mlp: bad args");
  StyleMlpLayers L{};
  for (int l = 0; l < nlayers; ++l) {
    MOCHA_CHECK_ARG(w1[l] && w2[l] && aligned16(w1[l]) && aligned16(w2[l]), "style_mlp: layer %d weights missing / unaligned", l);
    L.w1[l] = w1[l]; L.b1[l] = b1[l]; L.w2[l] = w2[l]; L.b2[l] = b2[l];
  }
  if ((B & 1) == 0 && B >= 64)
    launch_k(style_mlp_cluster_kernel, B, STYLEC_THREADS, 0, s, cha, n, L, nlayers, gb, B);
  else
    launch_k(style_mlp_kernel, B, STYLE_THREADS, 0, s, cha, n, L, nlayers, gb, B);
  count_launch();
  MOCHA_LAUNCH_CHECK("style_mlp");
  return MOCHA_OK;
}

bool cvae_prior_last_supported(int D, int H, int dff, int np) {
  if (D != 256 || H < 1 || D % H != 0 || np < 2 || np > PL_MAXKEYS) return false;
  const int dh = D / H;
  if (dh % 8 != 0 || (dh / 8 & (dh / 8 - 1)) != 0) return false;   // a head = a power-of-two group of 8-column lanes
  return dff == 256 || dff == 512 || dff == 1024;
}

int cvae_prior_last(const float* x, int B, int np, const __nv_bfloat16* kv, const __nv_bfloat16* wq, const float* bq,
                    const __nv_bfloat16* wo, const float* bo, const float* g1, const float* be1, const __nv_bfloat16* w1,
                    const float* b1, const __nv_bfloat16* w2, const float* b2, const float* g2, const float* be2, int H, int dff,
                    float eps, float* out, cudaStream_t s) {
  MOCHA_CHECK_ARG(x && kv && wq && wo && w1 && w2 && g1 && be1 && g2 && be2 && out && B > 0, "cvae_prior_last: null argument");
  MOCHA_CHECK_ARG(cvae_prior_last_supported(256, H, dff, np), "cvae_prior_last: unsupported geometry");
  MOCHA_CHECK_ARG(aligned16(kv) && aligned16(wq) && aligned16(wo) && aligned16(w1) && aligned16(w2), "cvae_prior_last: unaligned operand");
  PriorLastW W{wq, wo, w1, w2, bq, bo, b1, b2, g1, be1, g2, be2};
  const size_t smem = (size_t)(8 * 256 + 2 * dff + 8 * 256 + 2 * H * PL_MAXKEYS) * sizeof(float) + 128;
  MOCHA_CHECK_ARG(smem <= 227 * 1024, "cvae_prior_last: too many heads");
  auto go = [&](auto kern) -> int {
    // (no cached flag: the variants share one function-pointer type, so a static here would be shared between them)
    if (smem > 48 * 1024) MOCHA_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    launch_k(kern, B, PL_THREADS, smem, s, x, np, kv, W, H, eps, out);
    return MOCHA_OK;
  };
  if (dff == 256) MOCHA_TRY(go(cvae_prior_last_kernel<1>));
  else if (dff == 512) MOCHA_TRY(go(cvae_prior_last_kernel<2>));
  else MOCHA_TRY(go(cvae_prior_last_kernel<4>));
  count_launch();
  MOCHA_LAUNCH_CHECK("cvae_prior_last");
  return MOCHA_OK;
}

int softmax_rows(float* S, long long rows, int ncols, float scale, cudaStream_t s) {
  MOCHA_CHECK_ARG(S && rows > 0 && ncols > 0, "softmax_rows: bad args");
  MOCHA_CHECK_ARG(ncols <= 32 * SM_MAXPL, "softmax_rows: ncols=%d > %d", ncols, 32 * SM_MAXPL);
  launch_k(softmax_rows_kernel, blocks_for(rows, 8), 256, 0, s, S, rows, ncols, scale);
  count_launch();
  MOCHA_LAUNCH_CHECK("softmax_rows");
  return MOCHA_OK;
}

int add_layernorm(const float* x, const float* r, const float* g, const float* b, float* y, long long rows,
                  int C, float eps, const float* tab_mean, const float* tab_std, int period, float* y2,
                  cudaStream_t s, __nv_bfloat16* y16) {
  MOCHA_CHECK_ARG(x && g && b && rows > 0 && C > 0, "add_layernorm: bad args");
  MOCHA_CHECK_ARG(y || y2 || y16, "add_layernorm: no output");
  MOCHA_CHECK_ARG(!y2 || (tab_mean && tab_std && period > 0), "add_layernorm: y2 needs its table");
  const bool vec = aligned16(x) && aligned16(r) && aligned16(g) && aligned16(b) && aligned16(y) && aligned16(y2) &&
                   aligned16(tab_mean) && aligned16(tab_std) && (reinterpret_cast<uintptr_t>(y16) & 7) == 0;
  if (vec && C == 256)
    launch_k(add_layernorm_reg_kernel<2>, blocks_for(rows, 8), 256, 0, s, x, r, g, b, y, rows, eps, tab_mean, tab_std, period, y2, y16);
  else if (vec && C == 128)
    launch_k(add_layernorm_reg_kernel<1>, blocks_for(rows, 8), 256, 0, s, x, r, g, b, y, rows, eps, tab_mean, tab_std, period, y2, y16);
  else if (vec && C == 512)
    launch_k(add_layernorm_reg_kernel<4>, blocks_for(rows, 8), 256, 0, s, x, r, g, b, y, rows, eps, tab_mean, tab_std, period, y2, y16);
  else
    launch_k(add_layernorm_kernel, blocks_for(rows, 8), 256, 0, s, x, r, g, b, y, rows, C, eps, tab_mean, tab_std,
                                                            period, y2, y16);
  count_launch();
  MOCHA_LAUNCH_CHECK("add_layernorm");
  return MOCHA_OK;
}

int cvae_prior_tokens(const float* mu_token, const float* logvar_token, const float* cond, const float* pe,
                      float* tok, int B, int ncond, int C, cudaStream_t s, __nv_bfloat16* tok16) {
  MOCHA_CHECK_ARG(mu_token && logvar_token && cond && pe && tok && B > 0 && ncond > 0 && C > 0,
                  "cvae_prior_tokens: bad args");
  const long long total = (long long)B * (ncond + 2) * C;
  if ((C & 3) == 0 && total < (1LL << 31) && aligned16(mu_token) && aligned16(logvar_token) && aligned16(cond) &&
      aligned16(pe) && aligned16(tok) && (!tok16 || (reinterpret_cast<uintptr_t>(tok16) & 7) == 0)) {
    const unsigned total4 = (unsigned)(total / 4);
    launch_k(cvae_prior_tokens_v4_kernel, (total4 + 255) / 256, 256, 0, s, reinterpret_cast<const float4*>(mu_token), reinterpret_cast<const float4*>(logvar_token),
        reinterpret_cast<const float4*>(cond), reinterpret_cast<const float4*>(pe), reinterpret_cast<float4*>(tok), tok16,
        (unsigned)ncond, (unsigned)(C / 4), total4);
    count_launch();
    MOCHA_LAUNCH_CHECK("cvae_prior_tokens");
    return MOCHA_OK;
  }
  launch_k(cvae_prior_tokens_kernel, blocks_for(total, 256), 256, 0, s, mu_token, logvar_token, cond, pe, tok, tok16,
                                                                  ncond, C, total);
  count_launch();
  MOCHA_LAUNCH_CHECK("cvae_prior_tokens");
  return MOCHA_OK;
}

int cvae_memory(const float* prior_out, int prior_tokens, const float* eps, const float* cond, float* mem,
                float* mu_out, float* logvar_out, int B, int ncond, int C, cudaStream_t s, __nv_bfloat16* mem16) {
  MOCHA_CHECK_ARG(prior_out && cond && (mem || mem16) && B > 0 && ncond > 0 && C > 0 && prior_tokens >= 2,
                  "cvae_memory: bad args");
  const long long total = (long long)B * (ncond + 1) * C;
  if ((C & 3) == 0 && total < (1LL << 31) && aligned16(prior_out) && aligned16(eps) && aligned16(cond) && aligned16(mem) &&
      aligned16(mu_out) && aligned16(logvar_out) && (reinterpret_cast<uintptr_t>(mem16) & 7) == 0) {
    const unsigned total4 = (unsigned)(total / 4);
    launch_k(cvae_memory_v4_kernel, (total4 + 255) / 256, 256, 0, s, reinterpret_cast<const float4*>(prior_out), (unsigned)prior_tokens, reinterpret_cast<const float4*>(eps),
        reinterpret_cast<const float4*>(cond), reinterpret_cast<float4*>(mem), mem16, reinterpret_cast<float4*>(mu_out),
        reinterpret_cast<float4*>(logvar_out), (unsigned)ncond, (unsigned)(C / 4), total4);
    count_launch();
    MOCHA_LAUNCH_CHECK("cvae_memory");
    return MOCHA_OK;
  }
  launch_k(cvae_memory_kernel, blocks_for(total, 256), 256, 0, s, prior_out, prior_tokens, eps, cond, mem, mem16, mu_out,
                                                            logvar_out, ncond, C, total);
  count_launch();
  MOCHA_LAUNCH_CHECK("cvae_memory");
  return MOCHA_OK;
}

int cvae_condition(const float* src_cnt, const float* prev, const float* m0, const float* s0, const float* m1,
                   const float* s1, float* cond, int B, int n, int C, cudaStream_t s) {
  MOCHA_CHECK_ARG(src_cnt && prev && m0 && s0 && m1 && s1 && cond && B > 0 && n > 0 && C > 0,
                  "cvae_condition: bad args");
  const long long total = (long long)B * 2 * n * C;
  if ((C & 3) == 0 && total < (1LL << 31) && aligned16(src_cnt) && aligned16(prev) && aligned16(m0) && aligned16(s0) &&
      aligned16(m1) && aligned16(s1) && aligned16(cond)) {
    const unsigned total4 = (unsigned)(total / 4);
    launch_k(cvae_condition_v4_kernel, (total4 + 255) / 256, 256, 0, s, reinterpret_cast<const float4*>(src_cnt), reinterpret_cast<const float4*>(prev), reinterpret_cast<const float4*>(m0),
        reinterpret_cast<const float4*>(s0), reinterpret_cast<const float4*>(m1), reinterpret_cast<const float4*>(s1),
        reinterpret_cast<float4*>(cond), (unsigned)((long long)n * C / 4), total4);
    count_launch();
    MOCHA_LAUNCH_CHECK("cvae_condition");
    return MOCHA_OK;
  }
  launch_k(cvae_condition_kernel, blocks_for(total, 256), 256, 0, s, src_cnt, prev, m0, s0, m1, s1, cond, n, C, total);
  count_launch();
  MOCHA_LAUNCH_CHECK("cvae_condition");
  return MOCHA_OK;
}

int affine_rows(const float* x, const float* mu, const float* sd, float* out, long long rows, int C, int period,
                cudaStream_t s, int ld_in, float* copy) {
  MOCHA_CHECK_ARG(x && (copy || (mu && sd && out)) && rows > 0 && C > 0 && period > 0, "affine_rows: bad args");
  const long long total = rows * C;
  launch_k(affine_rows_kernel, blocks_for(total, 256), 256, 0, s, x, mu, sd, out, total, C, period, ld_in > 0 ? ld_in : C, copy);
  count_launch();
  MOCHA_LAUNCH_CHECK("affine_rows");
  return MOCHA_OK;
}

bool out_conv_affine_supported(int K, int N) { return (K == 64 || K == 128) && N >= 1 && N <= 16; }

int out_conv_affine(const __nv_bfloat16* x, const float* W, const float* bias, const float* mu, const float* sd, float* ytil,
                    float* y, int R, int K, int N, int period, cudaStream_t s) {
  MOCHA_CHECK_ARG(x && W && (ytil || y) && R > 0 && out_conv_affine_supported(K, N) && aligned16(x), "out_conv_affine: bad args");
  MOCHA_CHECK_ARG(!y || (mu && sd && period > 0), "out_conv_affine: Y needs its tables");
  if (period <= 0) period = 1;
  const size_t smem = (size_t)(OC_ROWS * N + 2 * period * N) * sizeof(float);
  MOCHA_CHECK_ARG(smem <= 48 * 1024, "out_conv_affine: tables too large");
  static int sms = 0;
  if (!sms) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev); if (sms <= 0) sms = 148; }
  const int ntiles = (int)blocks_for(R, OC_ROWS);
  // persistent: at most 3 co-resident blocks per SM, every block the same number of tiles (no ragged last round)
  const int per = (ntiles + 3 * sms - 1) / (3 * sms);
  const int grid = (ntiles + per - 1) / per;
  if (K == 64)
    launch_k(out_conv_affine_kernel<4>, grid, OC_ROWS, smem, s, x, W, bias, mu, sd, ytil, y, R, N, period);
  else
    launch_k(out_conv_affine_kernel<8>, grid, OC_ROWS, smem, s, x, W, bias, mu, sd, ytil, y, R, N, period);
  count_launch();
  MOCHA_LAUNCH_CHECK("out_conv_affine");
  return MOCHA_OK;
}

int broadcast_rows(const float* x, float* out, int B, long long n_elems, cudaStream_t s, __nv_bfloat16* out16) {
  MOCHA_CHECK_ARG(x && out && B > 0 && n_elems > 0, "broadcast_rows: bad args");
  const long long total = (long long)B * n_elems;
  launch_k(broadcast_rows_kernel, blocks_for(total, 256), 256, 0, s, x, out, out16, n_elems, total);
  count_launch();
  MOCHA_LAUNCH_CHECK("broadcast_rows");
  return MOCHA_OK;
}

int add_table(const float* a, const float* table, float* out, long long rows, int C, int period,
              cudaStream_t s) {
  MOCHA_CHECK_ARG(a && table && out && rows > 0 && C > 0 && period > 0, "add_table: bad args");
  const long long total = rows * C;
  launch_k(add_table_kernel, blocks_for(total, 256), 256, 0, s, a, table, out, total, C, period);
  count_launch();
  MOCHA_LAUNCH_CHECK("add_table");
  return MOCHA_OK;
}

int gather_token_rows(const float* x, const __nv_bfloat16* x16, int n, int take, int C, int B, float* out,
                      __nv_bfloat16* out16, cudaStream_t s) {
  MOCHA_CHECK_ARG(x && (out || out16) && n >= take && take > 0 && C > 0 && B > 0, "gather_token_rows: bad args");
  const long long total = (long long)B * take * C;
  launch_k(gather_token_rows_kernel, blocks_for(total, 256), 256, 0, s, x, x16, n, take, C, total, out, out16);
  count_launch();
  MOCHA_LAUNCH_CHECK("gather_token_rows");
  return MOCHA_OK;
}

int cast_f32_bf16(const float* x, __nv_bfloat16* y, long long n, cudaStream_t s) {
  MOCHA_CHECK_ARG(x && y && n > 0, "cast_f32_bf16: bad args");
  MOCHA_CHECK_ARG((((uintptr_t)x) & 15) == 0 && (((uintptr_t)y) & 7) == 0, "cast_f32_bf16: misaligned");
  launch_k(cast_f32_bf16_kernel, blocks_for((n + 3) / 4, 256), 256, 0, s, x, y, n);
  count_launch();
  MOCHA_LAUNCH_CHECK("cast_f32_bf16");
  return MOCHA_OK;
}

}  // namespace mocha
