// Context matching (SURVEY §8 a5): exact Euclidean k-NN of encoded queries against the character
// feature DB. Semantics of sklearn.neighbors.BallTree(X).query(q, k) as called at
// test_fullframework.py:293-296 and :440-443 (float64 arithmetic on float32 inputs).
//   * mocha_match_exact : brute force in fp64, HBM-bound streaming of the DB (batch-1 / small N)
//   * mocha_match_tc    : tcgen05 coarse pass with fused top-kc epilogue (gemm_tc.cu) + this file's
//                         candidate merge and exact fp64 re-rank
#include "../../include/mocha_b200.h"
#include "common.cuh"
#include "gemm_tc.cuh"

using namespace mocha;

namespace {

constexpr int KMAX = 16;
constexpr int EXQ = 4;  // queries per pass of the exact kernel

// One CTA per (RB DB rows, QB queries) tile: every thread owns a slice of D and accumulates the RB x QB
// squared differences in fp64 registers (rows and queries are loaded once per tile, 128-bit loads,
// fp32 -> fp64 conversion amortised over the tile); warp shuffles + a small smem pass reduce over D.
// <1,4> serves batch-1 streaming (385 CTAs for the reference-size DB), <8,8> serves batched queries
// (L2 traffic per pair drops 5x, which is what bounds the small tile).
template <int RB, int QB>
__global__ void __launch_bounds__(256)
match_exact_tile_kernel(const float* __restrict__ Q, int nq, const float* __restrict__ DB, long long N, int D,
                        double* __restrict__ dist2) {
  pdl_trigger();
  pdl_wait();
  __shared__ double red[8][RB * QB];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row0 = (long long)blockIdx.x * RB;
  const int q0 = blockIdx.y * QB;
  const float* xr[RB];
  const float* qr[QB];
#pragma unroll
  for (int r = 0; r < RB; ++r) xr[r] = DB + (row0 + r < N ? row0 + r : N - 1) * (long long)D;   // clamped: result unused
#pragma unroll
  for (int j = 0; j < QB; ++j) qr[j] = Q + (long long)(q0 + j < nq ? q0 + j : nq - 1) * D;
  double acc[RB][QB];
#pragma unroll
  for (int r = 0; r < RB; ++r)
#pragma unroll
    for (int j = 0; j < QB; ++j) acc[r][j] = 0.0;
  if ((D & 3) == 0 && ((reinterpret_cast<uintptr_t>(DB) & 15) == 0) && ((reinterpret_cast<uintptr_t>(Q) & 15) == 0)) {
    for (int d = threadIdx.x * 4; d < D; d += 1024) {
      double xd[RB][4];
#pragma unroll
      for (int r = 0; r < RB; ++r) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(xr[r] + d));
        xd[r][0] = (double)v.x; xd[r][1] = (double)v.y; xd[r][2] = (double)v.z; xd[r][3] = (double)v.w;
      }
#pragma unroll
      for (int j = 0; j < QB; ++j) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(qr[j] + d));
        const double qd[4] = {(double)v.x, (double)v.y, (double)v.z, (double)v.w};
#pragma unroll
        for (int r = 0; r < RB; ++r) {
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const double a = qd[e] - xd[r][e];
            acc[r][j] = fma(a, a, acc[r][j]);
          }
        }
      }
    }
  } else {
    for (int d = threadIdx.x; d < D; d += 256) {
      double xd[RB];
#pragma unroll
      for (int r = 0; r < RB; ++r) xd[r] = (double)xr[r][d];
#pragma unroll
      for (int j = 0; j < QB; ++j) {
        const double qd = (double)qr[j][d];
#pragma unroll
        for (int r = 0; r < RB; ++r) {
          const double a = qd - xd[r];
          acc[r][j] = fma(a, a, acc[r][j]);
        }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < RB; ++r)
#pragma unroll
    for (int j = 0; j < QB; ++j) {
      const double v = warp_sum(acc[r][j]);
      if (lane == 0) red[warp][r * QB + j] = v;
    }
  __syncthreads();
  if (threadIdx.x < RB * QB) {
    const int r = threadIdx.x / QB, j = threadIdx.x - r * QB;
    if (row0 + r < N && q0 + j < nq) {
      double v = 0.0;
#pragma unroll
      for (int w = 0; w < 8; ++w) v += red[w][threadIdx.x];
      dist2[(long long)(q0 + j) * N + row0 + r] = v;
    }
  }
}

template <class T, class I>
__device__ __forceinline__ bool better(T d0, I i0, T d1, I i1) {
  return d0 < d1 || (d0 == d1 && i0 < i1);
}

// Block-wide top-k of (value, index) pairs by (value asc, index asc). Each thread feeds its own
// candidates through `local insert`, then k rounds of block arg-min pop the winners.
// The key type is a template parameter: fp64 compares issue on the slow FP64 pipe of this part, so lists
// whose values are fp32 (the tensor-core coarse scores) are merged with float keys and int indices.
template <int NT, class T, class I>
__device__ void block_topk_pop(T (&ls)[KMAX], I (&li)[KMAX], int k, T* out_d, I* out_i, T* red_d, I* red_i, int* red_t) {
  for (int r = 0; r < k; ++r) {
    // every thread proposes the head of its (ascending) local list
    T d = ls[0];
    I i = li[0];
    int t = threadIdx.x;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const T d2 = __shfl_xor_sync(0xffffffffu, d, o);
      const I i2 = __shfl_xor_sync(0xffffffffu, i, o);
      const int t2 = __shfl_xor_sync(0xffffffffu, t, o);
      const bool take = (i2 >= 0) && (i < 0 || better(d2, i2, d, i));
      if (take) { d = d2; i = i2; t = t2; }
    }
    if ((threadIdx.x & 31) == 0) { red_d[threadIdx.x >> 5] = d; red_i[threadIdx.x >> 5] = i; red_t[threadIdx.x >> 5] = t; }
    __syncthreads();
    if (threadIdx.x == 0) {
      T bd = red_d[0]; I bi = red_i[0]; int bt = red_t[0];
      for (int w = 1; w < NT / 32; ++w) {
        if (red_i[w] >= 0 && (bi < 0 || better(red_d[w], red_i[w], bd, bi))) { bd = red_d[w]; bi = red_i[w]; bt = red_t[w]; }
      }
      out_d[r] = bd; out_i[r] = bi; red_t[0] = bt;
    }
    __syncthreads();
    if (threadIdx.x == red_t[0] && out_i[r] >= 0) {
      // pop: shift the local list left (static indices keep it in registers)
#pragma unroll
      for (int j = 0; j + 1 < KMAX; ++j) { ls[j] = ls[j + 1]; li[j] = li[j + 1]; }
      ls[KMAX - 1] = INFINITY; li[KMAX - 1] = -1;
    }
    __syncthreads();
  }
}

// keep the k best (ascending by (value, index)) in ls/li; slots >= k stay empty
template <class T, class I>
__device__ __forceinline__ void local_insert(T (&ls)[KMAX], I (&li)[KMAX], int k, T d, I i) {
#pragma unroll
  for (int t = 0; t < KMAX; ++t) {
    if (t < k && i >= 0 && (li[t] < 0 || better(d, i, ls[t], li[t]))) {
      const T td = ls[t]; ls[t] = d; d = td;
      const I ti = li[t]; li[t] = i; i = ti;
    }
  }
}

// one block per query: top-k over a row of squared distances
__global__ void __launch_bounds__(256)
topk_rows_kernel(const double* __restrict__ dist2, long long N, int k, long long index_offset,
                 int64_t* __restrict__ out_idx, double* __restrict__ out_dist) {
  pdl_trigger();
  pdl_wait();
  __shared__ double red_d[8]; __shared__ long long red_i[8]; __shared__ int red_t[8];
  __shared__ double od[KMAX]; __shared__ long long oi[KMAX];
  const int q = blockIdx.x;
  const double* row = dist2 + (long long)q * N;
  double ls[KMAX]; long long li[KMAX];
#pragma unroll
  for (int t = 0; t < KMAX; ++t) { ls[t] = INFINITY; li[t] = -1; }
  for (long long n = threadIdx.x; n < N; n += 256) local_insert(ls, li, k, row[n], n);
  block_topk_pop<256, double, long long>(ls, li, k, od, oi, red_d, red_i, red_t);
  if (threadIdx.x < k) {
    out_idx[(long long)q * k + threadIdx.x] = oi[threadIdx.x] >= 0 ? oi[threadIdx.x] + index_offset : -1;
    if (out_dist) out_dist[(long long)q * k + threadIdx.x] = sqrt(od[threadIdx.x]);
  }
}

// one block per query: merge coarse candidates, exact fp64 re-rank of the best kc, emit top-k
__global__ void __launch_bounds__(256)
match_rerank_kernel(const float* __restrict__ Q, const __nv_bfloat16* __restrict__ DB16,
                    const float* __restrict__ DB32, int D, const float* __restrict__ cand_score,
                    const int32_t* __restrict__ cand_idx, int ncand, int kc, int k, long long index_offset,
                    int64_t* __restrict__ out_idx, double* __restrict__ out_dist) {
  pdl_trigger();
  pdl_wait();
  __shared__ double red_d[8]; __shared__ long long red_i[8]; __shared__ int red_t[8];
  __shared__ double od[KMAX]; __shared__ long long oi[KMAX];
  __shared__ double exact[KMAX];
  const int q = blockIdx.x;
  const float* cs = cand_score + (long long)q * ncand;
  const int32_t* ci = cand_idx + (long long)q * ncand;
  {
    // merge of the coarse lists on float keys / int indices (same (value, index) order as the fp64 version)
    __shared__ float fred_d[8]; __shared__ int fred_i[8];
    __shared__ float fod[KMAX]; __shared__ int foi[KMAX];
    float ls[KMAX]; int li[KMAX];
#pragma unroll
    for (int t = 0; t < KMAX; ++t) { ls[t] = INFINITY; li[t] = -1; }
    for (int n = threadIdx.x; n < ncand; n += 256) {
      const int32_t id = ci[n];
      if (id >= 0) local_insert(ls, li, kc, cs[n], (int)id);
    }
    block_topk_pop<256, float, int>(ls, li, kc, fod, foi, fred_d, fred_i, red_t);
    if (threadIdx.x < KMAX) { od[threadIdx.x] = (double)fod[threadIdx.x]; oi[threadIdx.x] = (long long)foi[threadIdx.x]; }
    __syncthreads();
  }
  // exact squared distances of the kc survivors: the whole block walks one candidate row at a time
  // (4 consecutive elements per thread, two fp64 accumulators) so the fp64 chains stay short
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* qv = Q + (long long)q * D;
  const bool vec4 = (D & 3) == 0 && ((reinterpret_cast<uintptr_t>(qv) & 15) == 0) &&
                    (DB32 ? (reinterpret_cast<uintptr_t>(DB32) & 15) == 0 : (reinterpret_cast<uintptr_t>(DB16) & 7) == 0);
  // Certified fp32 pre-filter. The FP64 pipe of this part sustains only ~4 ops/clk/SM (the exact pass over
  // kc rows of 23040 values was pipe-bound: 55 us for 128 queries), so the kc survivors are first measured
  // in fp32 (one accumulator of <= ceil(D/1024)*4 terms per thread, then 5 + 8 tree adds): the relative
  // error of such a sum of non-negative terms is below (ceil(D/1024)*4 + 20) * 2^-24. A row whose fp32
  // distance exceeds the k-th smallest fp32 one by more than twice that bound (x4 safety) cannot be among
  // the exact top k; only the rest - k rows unless there are near-ties - is re-evaluated in fp64.
  __shared__ float d32[KMAX];
  __shared__ int keep[KMAX];
  if (vec4 && DB32 && kc > k) {
    // all survivors at once: the query segment is loaded once and kc row segments are in flight per thread
    // (the loop is load-latency-bound: one block per SM streams kc rows of 92 KB); kc <= 8 doubles the depth
    float f[KMAX];
    const float* xr[KMAX];
#pragma unroll
    for (int c = 0; c < KMAX; ++c) {
      f[c] = 0.f;
      const long long id = c < kc ? oi[c] : -1;
      xr[c] = DB32 + (id >= 0 ? id : 0) * (long long)D;
    }
    int d = threadIdx.x * 4;
    if (kc <= 8) {
      for (; d + 1024 < D; d += 2048) {
        const float4 q0 = *reinterpret_cast<const float4*>(qv + d), q1 = *reinterpret_cast<const float4*>(qv + d + 1024);
        float4 x0[8], x1[8];
#pragma unroll
        for (int c = 0; c < 8; ++c)
          if (c < kc) {
            x0[c] = __ldg(reinterpret_cast<const float4*>(xr[c] + d));
            x1[c] = __ldg(reinterpret_cast<const float4*>(xr[c] + d + 1024));
          }
#pragma unroll
        for (int c = 0; c < 8; ++c)
          if (c < kc) {
            float e0 = q0.x - x0[c].x, e1 = q0.y - x0[c].y, e2 = q0.z - x0[c].z, e3 = q0.w - x0[c].w;
            f[c] = fmaf(e0, e0, f[c]); f[c] = fmaf(e1, e1, f[c]);
            f[c] = fmaf(e2, e2, f[c]); f[c] = fmaf(e3, e3, f[c]);
            e0 = q1.x - x1[c].x; e1 = q1.y - x1[c].y; e2 = q1.z - x1[c].z; e3 = q1.w - x1[c].w;
            f[c] = fmaf(e0, e0, f[c]); f[c] = fmaf(e1, e1, f[c]);
            f[c] = fmaf(e2, e2, f[c]); f[c] = fmaf(e3, e3, f[c]);
          }
      }
    }
    for (; d < D; d += 1024) {
      const float4 qq = *reinterpret_cast<const float4*>(qv + d);
      float4 xx[KMAX];
#pragma unroll
      for (int c = 0; c < KMAX; ++c)
        if (c < kc) xx[c] = __ldg(reinterpret_cast<const float4*>(xr[c] + d));
#pragma unroll
      for (int c = 0; c < KMAX; ++c)
        if (c < kc) {
          const float e0 = qq.x - xx[c].x, e1 = qq.y - xx[c].y, e2 = qq.z - xx[c].z, e3 = qq.w - xx[c].w;
          f[c] = fmaf(e0, e0, f[c]); f[c] = fmaf(e1, e1, f[c]);
          f[c] = fmaf(e2, e2, f[c]); f[c] = fmaf(e3, e3, f[c]);
        }
    }
    __shared__ float fpart[8][KMAX];
#pragma unroll
    for (int c = 0; c < KMAX; ++c) {
      const float acc = warp_sum(f[c]);
      if (lane == 0) fpart[warp][c] = acc;
    }
    __syncthreads();
    if (threadIdx.x < kc) {
      float t = 0.f;
      for (int w = 0; w < 8; ++w) t += fpart[w][threadIdx.x];
      d32[threadIdx.x] = oi[threadIdx.x] >= 0 ? t : INFINITY;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      float kth = INFINITY;   // k-th smallest fp32 distance (kc <= 16: selection by counting)
      for (int c = 0; c < kc; ++c) {
        int below = 0;
        for (int j = 0; j < kc; ++j) below += (d32[j] < d32[c]) || (d32[j] == d32[c] && j < c);
        if (below == k - 1) kth = d32[c];
      }
      const float eps = (float)(((D + 1023) / 1024) * 4 + 20) * 5.9604645e-8f;
      const float bound = kth * (1.f + 8.f * eps);
      for (int c = 0; c < kc; ++c) keep[c] = d32[c] <= bound;
    }
  } else {
    if (threadIdx.x < KMAX) keep[threadIdx.x] = 1;
  }
  __syncthreads();
  for (int c = 0; c < kc; ++c) {
    if (!keep[c]) {   // uniform across the block
      if (threadIdx.x == 0) { exact[c] = INFINITY; oi[c] = -1; }
      continue;
    }
    const long long id = oi[c];
    double a0 = 0.0, a1 = 0.0;
    if (id >= 0) {
      if (vec4 && DB32) {
        const float* xrow = DB32 + id * (long long)D;
        int d = threadIdx.x * 4;
        for (; d + 3 * 1024 < D; d += 4 * 1024) {   // four row segments in flight per thread
          float4 qq[4], xx[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            qq[u] = *reinterpret_cast<const float4*>(qv + d + u * 1024);
            xx[u] = __ldg(reinterpret_cast<const float4*>(xrow + d + u * 1024));
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const double e0 = (double)qq[u].x - (double)xx[u].x, e1 = (double)qq[u].y - (double)xx[u].y;
            const double e2 = (double)qq[u].z - (double)xx[u].z, e3 = (double)qq[u].w - (double)xx[u].w;
            a0 = fma(e0, e0, a0); a1 = fma(e1, e1, a1);
            a0 = fma(e2, e2, a0); a1 = fma(e3, e3, a1);
          }
        }
        for (; d < D; d += 1024) {
          const float4 qq = *reinterpret_cast<const float4*>(qv + d);
          const float4 xx = __ldg(reinterpret_cast<const float4*>(xrow + d));
          const double e0 = (double)qq.x - (double)xx.x, e1 = (double)qq.y - (double)xx.y;
          const double e2 = (double)qq.z - (double)xx.z, e3 = (double)qq.w - (double)xx.w;
          a0 = fma(e0, e0, a0); a1 = fma(e1, e1, a1);
          a0 = fma(e2, e2, a0); a1 = fma(e3, e3, a1);
        }
      } else if (vec4) {
        for (int d = threadIdx.x * 4; d < D; d += 1024) {
          const float4 qq = *reinterpret_cast<const float4*>(qv + d);
          float4 xx;
          if (DB32) {
            xx = __ldg(reinterpret_cast<const float4*>(DB32 + id * (long long)D + d));
          } else {
            const uint2 raw = __ldg(reinterpret_cast<const uint2*>(DB16 + id * (long long)D + d));
            const __nv_bfloat162 lo = *reinterpret_cast<const __nv_bfloat162*>(&raw.x);
            const __nv_bfloat162 hi = *reinterpret_cast<const __nv_bfloat162*>(&raw.y);
            xx = make_float4(__low2float(lo), __high2float(lo), __low2float(hi), __high2float(hi));
          }
          const double e0 = (double)qq.x - (double)xx.x, e1 = (double)qq.y - (double)xx.y;
          const double e2 = (double)qq.z - (double)xx.z, e3 = (double)qq.w - (double)xx.w;
          a0 = fma(e0, e0, a0); a1 = fma(e1, e1, a1);
          a0 = fma(e2, e2, a0); a1 = fma(e3, e3, a1);
        }
      } else if (DB32) {
        const float* x = DB32 + id * (long long)D;
        for (int d = threadIdx.x; d < D; d += 256) { const double a = (double)qv[d] - (double)x[d]; a0 = fma(a, a, a0); }
      } else {
        const __nv_bfloat16* x = DB16 + id * (long long)D;
        for (int d = threadIdx.x; d < D; d += 256) { const double a = (double)qv[d] - (double)__bfloat162float(x[d]); a0 = fma(a, a, a0); }
      }
    }
    double acc = warp_sum(a0 + a1);
    if (lane == 0) red_d[warp] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0.0;
      for (int w = 0; w < 8; ++w) t += red_d[w];
      exact[c] = id >= 0 ? t : INFINITY;
    }
    __syncthreads();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    // insertion sort of <= 16 entries by (distance, index)
    double d[KMAX]; long long id[KMAX];
    int m = 0;
    for (int c = 0; c < kc; ++c) {
      if (oi[c] < 0) continue;
      int p = m++;
      d[p] = exact[c]; id[p] = oi[c];
      while (p > 0 && better(d[p], id[p], d[p - 1], id[p - 1])) {
        const double td = d[p]; d[p] = d[p - 1]; d[p - 1] = td;
        const long long ti = id[p]; id[p] = id[p - 1]; id[p - 1] = ti;
        --p;
      }
    }
    for (int r = 0; r < k; ++r) {
      out_idx[(long long)q * k + r] = r < m ? id[r] + index_offset : -1;
      if (out_dist) out_dist[(long long)q * k + r] = r < m ? sqrt(d[r]) : INFINITY;
    }
  }
}

// warp per row: fp32 -> bf16 rows + squared norm of the rounded row
__global__ void __launch_bounds__(256)
db_pack_kernel(const float* __restrict__ rows, long long N, int D, __nv_bfloat16* __restrict__ rows16,
               float* __restrict__ norm) {
  pdl_trigger();
  pdl_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long r = (long long)blockIdx.x * 8 + warp;
  if (r >= N) return;
  const float* x = rows + r * (long long)D;
  __nv_bfloat16* y = rows16 + r * (long long)D;
  float acc = 0.f;
  for (int d = lane; d < D; d += 32) {
    const __nv_bfloat16 b = __float2bfloat16_rn(x[d]);
    y[d] = b;
    const float f = __bfloat162float(b);
    acc = fmaf(f, f, acc);
  }
  acc = warp_sum(acc);
  if (lane == 0 && norm) norm[r] = acc;
}

// thread per query: merge nshard sorted (dist, idx) lists of length k
__global__ void topk_merge_kernel(const double* __restrict__ dist, const int64_t* __restrict__ idx, int nshard,
                                  int nq, int k, double* __restrict__ out_dist, int64_t* __restrict__ out_idx) {
  pdl_trigger();
  pdl_wait();
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  int head[64];
  for (int s = 0; s < nshard; ++s) head[s] = 0;
  for (int r = 0; r < k; ++r) {
    int bs = -1; double bd = 0.0; long long bi = -1;
    for (int s = 0; s < nshard; ++s) {
      if (head[s] >= k) continue;
      const long long o = ((long long)s * nq + q) * k + head[s];
      const long long id = idx[o];
      if (id < 0) continue;
      const double d = dist[o];
      if (bs < 0 || better(d, id, bd, bi)) { bs = s; bd = d; bi = id; }
    }
    if (bs >= 0) ++head[bs];
    out_idx[(long long)q * k + r] = bi;
    if (out_dist) out_dist[(long long)q * k + r] = bs >= 0 ? bd : INFINITY;
  }
}

}  // namespace

extern "C" size_t mocha_match_exact_workspace_bytes(int nq, long long N, int k) {
  (void)k;
  if (nq <= 0 || N <= 0) return 0;
  return align_up((size_t)nq * (size_t)N * sizeof(double), 256) + 256;
}

extern "C" int mocha_match_exact(const float* Q, int nq, const float* DB, long long N, int D, int k,
                                 long long index_offset, int64_t* idx, double* dist, void* workspace,
                                 size_t workspace_bytes, mocha_stream_t stream) {
  MOCHA_CHECK_ARG(Q && DB && idx, "mocha_match_exact: null argument");
  MOCHA_CHECK_ARG(nq > 0 && N > 0 && D > 0, "mocha_match_exact: empty problem nq=%d N=%lld D=%d", nq, N, D);
  MOCHA_CHECK_ARG(k >= 1 && k <= KMAX && k <= N, "mocha_match_exact: k=%d out of range (1..min(%d,N))", k, KMAX);
  Workspace ws(workspace, workspace_bytes);
  double* dist2 = ws.take<double>((size_t)nq * (size_t)N);
  if (ws.overflow)
    return set_error(MOCHA_ERR_WORKSPACE, "mocha_match_exact: workspace too small (%zu B given, %zu B needed)",
                     workspace_bytes, ws.off);
  cudaStream_t s = (cudaStream_t)stream;
  MOCHA_CHECK_ARG(N <= 2147483647LL && (nq + EXQ - 1) / EXQ <= 65535, "mocha_match_exact: problem too large for the exact kernel (use mocha_match_tc)");
  if (nq >= 16 && N >= 64)
    launch_k(match_exact_tile_kernel<8, 8>, dim3((unsigned)((N + 7) / 8), (unsigned)((nq + 7) / 8)), 256, 0, s, Q, nq, DB, N, D, dist2);
  else
    launch_k(match_exact_tile_kernel<1, EXQ>, dim3((unsigned)N, (unsigned)((nq + EXQ - 1) / EXQ)), 256, 0, s, Q, nq, DB, N, D, dist2);
  count_launch();
  MOCHA_LAUNCH_CHECK("match_exact_tile_kernel");
  launch_k(topk_rows_kernel, nq, 256, 0, s, dist2, N, k, index_offset, idx, dist);
  count_launch();
  MOCHA_LAUNCH_CHECK("topk_rows_kernel");
  return MOCHA_OK;
}

extern "C" size_t mocha_match_tc_workspace_bytes(int nq, long long N, int D, int kc) {
  if (nq <= 0 || N <= 0 || kc <= 0) return 0;
  const size_t ncand = (size_t)tc_match_splits(nq, N) * kc;
  const size_t np = (size_t)((N + 127) / 128) * 128;  // split-K path: one candidate per (padded) row
  const size_t lists = ncand > np ? ncand : np;
  return 2 * (align_up((size_t)nq * lists * 4, 256)) + tc_match_splitk_ws_bytes(nq, N, D) + 512;
}

extern "C" int mocha_match_tc(const float* Q, const void* Q16, int nq, const void* DB16, const float* DB32,
                              const float* dbnorm, long long N, int D, int k, int kc, long long index_offset,
                              int64_t* idx, double* dist, void* workspace, size_t workspace_bytes,
                              mocha_stream_t stream) {
  MOCHA_CHECK_ARG(Q && dbnorm && idx && (DB16 || DB32), "mocha_match_tc: null argument");
  MOCHA_CHECK_ARG(!DB16 || Q16, "mocha_match_tc: bf16 DB needs the bf16 query copy");
  MOCHA_CHECK_ARG(k >= 1 && k <= kc && kc <= KMAX, "mocha_match_tc: need 1 <= k <= kc <= %d", KMAX);
  MOCHA_CHECK_ARG(k <= N, "mocha_match_tc: k=%d > N=%lld", k, N);
  Workspace ws(workspace, workspace_bytes);
  cudaStream_t s = (cudaStream_t)stream;
  if (DB16 && tc_match_splitk_slices(nq, N, D) > 0) {
    // small problem: K-sliced coarse pass, every row is a candidate of the fp64 re-rank's top-kc merge
    const size_t np = (size_t)((N + 127) / 128) * 128;
    float* cs = ws.take<float>((size_t)nq * np);
    int32_t* ci = ws.take<int32_t>((size_t)nq * np);
    float* partial = ws.take<float>(tc_match_splitk_ws_bytes(nq, N, D) / 4 - 64);
    if (ws.overflow)
      return set_error(MOCHA_ERR_WORKSPACE, "mocha_match_tc: workspace too small (%zu B given, %zu B needed)",
                       workspace_bytes, ws.off);
    MOCHA_TRY(tc_match_coarse_splitk((const __nv_bfloat16*)Q16, nq, (const __nv_bfloat16*)DB16, dbnorm, N, D, partial, cs, ci, s));
    launch_k(match_rerank_kernel, nq, 256, 0, s, Q, (const __nv_bfloat16*)DB16, DB32, D, cs, ci, (int)np, kc, k, index_offset,
                                           idx, dist);
    count_launch();
    MOCHA_LAUNCH_CHECK("match_rerank_kernel");
    return MOCHA_OK;
  }
  const int splits = tc_match_splits(nq, N);
  const size_t ncand = (size_t)splits * kc;
  float* cs = ws.take<float>((size_t)nq * ncand);
  int32_t* ci = ws.take<int32_t>((size_t)nq * ncand);
  if (ws.overflow)
    return set_error(MOCHA_ERR_WORKSPACE, "mocha_match_tc: workspace too small (%zu B given, %zu B needed)",
                     workspace_bytes, ws.off);
  if (DB16)
    MOCHA_TRY(tc_match_coarse((const __nv_bfloat16*)Q16, nq, (const __nv_bfloat16*)DB16, dbnorm, N, D, kc, cs, ci, s));
  else  // fp32-storage DB: TF32 tensor-core pass straight from the fp32 rows
    MOCHA_TRY(tc_match_coarse_tf32(Q, nq, DB32, dbnorm, N, D, kc, cs, ci, s));
  launch_k(match_rerank_kernel, nq, 256, 0, s, Q, (const __nv_bfloat16*)DB16, DB32, D, cs, ci, (int)ncand, kc, k,
                                         index_offset, idx, dist);
  count_launch();
  MOCHA_LAUNCH_CHECK("match_rerank_kernel");
  return MOCHA_OK;
}

extern "C" int mocha_db_pack_bf16(const float* rows, long long N, int D, void* rows16, float* norm,
                                  mocha_stream_t stream) {
  MOCHA_CHECK_ARG(rows && rows16 && N > 0 && D > 0, "mocha_db_pack_bf16: bad argument");
  launch_k(db_pack_kernel, (unsigned)((N + 7) / 8), 256, 0, (cudaStream_t)stream, rows, N, D, (__nv_bfloat16*)rows16, norm);
  count_launch();
  MOCHA_LAUNCH_CHECK("db_pack_kernel");
  return MOCHA_OK;
}

// squared norms of fp32 rows (dbnorm for the fp32-storage / TF32 matcher)
__global__ void __launch_bounds__(256) row_norm_kernel(const float* __restrict__ rows, long long N, int D, float* __restrict__ norm) {
  pdl_trigger();
  pdl_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long r = (long long)blockIdx.x * 8 + warp;
  if (r >= N) return;
  const float* x = rows + r * (long long)D;
  float acc = 0.f;
  for (int d = lane; d < D; d += 32) acc = fmaf(x[d], x[d], acc);
  acc = warp_sum(acc);
  if (lane == 0) norm[r] = acc;
}

extern "C" int mocha_db_norms_f32(const float* rows, long long N, int D, float* norm, mocha_stream_t stream) {
  MOCHA_CHECK_ARG(rows && norm && N > 0 && D > 0, "mocha_db_norms_f32: bad argument");
  launch_k(row_norm_kernel, (unsigned)((N + 7) / 8), 256, 0, (cudaStream_t)stream, rows, N, D, norm);
  count_launch();
  MOCHA_LAUNCH_CHECK("row_norm_kernel");
  return MOCHA_OK;
}

extern "C" int mocha_topk_merge(const double* dist, const int64_t* idx, int nshard, int nq, int k, double* out_dist,
                                int64_t* out_idx, mocha_stream_t stream) {
  MOCHA_CHECK_ARG(dist && idx && out_idx, "mocha_topk_merge: null argument");
  MOCHA_CHECK_ARG(nshard >= 1 && nshard <= 64 && nq > 0 && k >= 1 && k <= KMAX, "mocha_topk_merge: bad sizes");
  launch_k(topk_merge_kernel, (nq + 127) / 128, 128, 0, (cudaStream_t)stream, dist, idx, nshard, nq, k, out_dist, out_idx);
  count_launch();
  MOCHA_LAUNCH_CHECK("topk_merge_kernel");
  return MOCHA_OK;
}

// Seed of a started clip (clip admission): dst[b] = table[idx[b * idx_stride]] for the rows whose start byte is set,
// one block per row, 16-byte copies; rows that do not start exit after the grid dependency, and an index outside [0, N)
// leaves the row as it is.
__global__ void __launch_bounds__(256) seed_rows_kernel(const uint8_t* __restrict__ start, const int64_t* __restrict__ idx,
                                                        int idx_stride, const float4* __restrict__ table, long long N,
                                                        long long row4, float4* __restrict__ dst) {
  pdl_trigger();
  pdl_wait();
  const int b = blockIdx.x;
  if (!start[b]) return;
  const long long r = idx[(long long)b * idx_stride];
  if (r < 0 || r >= N) return;
  const float4* src = table + r * row4;
  float4* out = dst + (long long)b * row4;
#pragma unroll 4
  for (long long i = threadIdx.x; i < row4; i += 256) out[i] = src[i];
}

extern "C" int mocha_seed_rows(const uint8_t* start, const int64_t* idx, int idx_stride, const float* table, long long N,
                               long long row_elems, float* dst, int B, mocha_stream_t stream) {
  MOCHA_CHECK_ARG(start && idx && table && dst, "mocha_seed_rows: null argument");
  MOCHA_CHECK_ARG(B > 0 && N > 0 && row_elems > 0 && idx_stride >= 1, "mocha_seed_rows: bad sizes (B=%d, N=%lld, row=%lld)",
                  B, N, row_elems);
  MOCHA_CHECK_ARG(row_elems % 4 == 0 && ((reinterpret_cast<uintptr_t>(table) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0,
                  "mocha_seed_rows: rows must be 16 B aligned multiples of 4 floats");
  launch_k(seed_rows_kernel, (unsigned)B, 256, 0, (cudaStream_t)stream, start, idx, idx_stride,
           reinterpret_cast<const float4*>(table), N, row_elems / 4, reinterpret_cast<float4*>(dst));
  count_launch();
  MOCHA_LAUNCH_CHECK("seed_rows_kernel");
  return MOCHA_OK;
}

// ------------------------------------------------------------------------------------------------
// Peer-memory exchange + merge of the DB-sharded matcher (see include/mocha_b200.h)
// ------------------------------------------------------------------------------------------------
namespace {
constexpr int XCHG_BLOCKS = 16;   // fixed grid: all blocks co-resident on any GPU, so the cross-GPU wait is safe
constexpr int XCHG_MAX_WORLD = 16;

struct XchgPtrs {
  unsigned char* buf[XCHG_MAX_WORLD];
};

__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void red_release_sys_add(unsigned* p, unsigned v) {
  asm volatile("red.release.sys.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// One kernel per rank: (1) P2P-store the local [nq,k] lists into slot `rank` of every rank's buffer,
// (2) release-increment the peer's arrival counter, (3) acquire-wait for every source's counter in the own
// buffer, (4) merge the world lists of this block's queries.
__global__ void __launch_bounds__(256)
topk_exchange_merge_kernel(const double* __restrict__ ld, const long long* __restrict__ li, int nq, int k, int rank,
                           int world, XchgPtrs peers, unsigned epoch, double* __restrict__ out_d,
                           long long* __restrict__ out_i) {
  pdl_trigger();
  pdl_wait();
  const unsigned parity = epoch & 1u;
  const size_t list = (size_t)nq * k;                      // elements per list
  const size_t half_bytes = (list * 8 + 15) & ~(size_t)15; // each array starts 16 B aligned (uint4 stores), odd lists too
  const size_t slot_bytes = 2 * half_bytes;
  const size_t parity_bytes = (size_t)world * slot_bytes;
  const size_t flags_off = 2 * parity_bytes;
  // ---- (1) push: 16 B per thread-step, this block's contiguous share of the two arrays
  {
    const size_t n2 = list / 2 * 2;   // uint4 = 2 elements of 8 B
    for (int p = 0; p < world; ++p) {
      unsigned char* dst = peers.buf[p] + parity * parity_bytes + (size_t)rank * slot_bytes;
      double* dd = reinterpret_cast<double*>(dst);
      long long* di = reinterpret_cast<long long*>(dst + half_bytes);
      for (size_t e = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 2; e < n2; e += (size_t)gridDim.x * blockDim.x * 2) {
        *reinterpret_cast<uint4*>(dd + e) = *reinterpret_cast<const uint4*>(ld + e);
        *reinterpret_cast<uint4*>(di + e) = *reinterpret_cast<const uint4*>(li + e);
      }
      if (blockIdx.x == 0 && threadIdx.x == 0 && n2 < list) { dd[n2] = ld[n2]; di[n2] = li[n2]; }
    }
  }
  __threadfence_system();
  __syncthreads();
  // ---- (2) signal: one release-add per block and peer; (3) wait for gridDim.x arrivals per source and call
  const unsigned expected = (epoch / 2 + 1) * gridDim.x;
  if (threadIdx.x < world) {
    unsigned* peer_flag = reinterpret_cast<unsigned*>(peers.buf[threadIdx.x] + flags_off) + parity * world + rank;
    red_release_sys_add(peer_flag, 1u);
    const unsigned* my_flag = reinterpret_cast<const unsigned*>(peers.buf[rank] + flags_off) + parity * world + threadIdx.x;
    long long t0 = clock64();
    while (ld_acquire_sys(my_flag) < expected) {
      if (clock64() - t0 > 20000000000LL) {   // ~10 s: a peer never launched - report instead of hanging the GPU
        printf("mocha topk exchange: rank %d timed out waiting for rank %d\n", rank, (int)threadIdx.x);
        __trap();
      }
    }
  }
  __syncthreads();
  // ---- (4) merge: one thread per query
  const unsigned char* mine = peers.buf[rank] + parity * parity_bytes;
  for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += gridDim.x * blockDim.x) {
    double bd[KMAX]; long long bi[KMAX];
#pragma unroll
    for (int t = 0; t < KMAX; ++t) { bd[t] = INFINITY; bi[t] = -1; }
    for (int sidx = 0; sidx < world; ++sidx) {
      const double* sd = reinterpret_cast<const double*>(mine + (size_t)sidx * slot_bytes);
      const long long* si = reinterpret_cast<const long long*>(mine + (size_t)sidx * slot_bytes + half_bytes);
      for (int j = 0; j < k; ++j) {
        const long long id = __ldcv(si + (size_t)q * k + j);
        if (id >= 0) local_insert(bd, bi, k, __ldcv(sd + (size_t)q * k + j), id);
      }
    }
#pragma unroll
    for (int t = 0; t < KMAX; ++t)
      if (t < k) { out_d[(size_t)q * k + t] = bd[t]; out_i[(size_t)q * k + t] = bi[t]; }
  }
}
}  // namespace

extern "C" size_t mocha_topk_exchange_bytes(int world, int nq, int k) {
  if (world < 1 || nq < 1 || k < 1) return 0;
  const size_t half_bytes = ((size_t)nq * k * 8 + 15) & ~(size_t)15;   // kernel layout: [dist | idx], each 16 B aligned
  return 2 * (size_t)world * 2 * half_bytes + 2 * (size_t)world * 4 + 256;
}

extern "C" int mocha_peer_alloc(size_t bytes, void** d_ptr, unsigned char handle_out[64]) {
  MOCHA_CHECK_ARG(bytes > 0 && d_ptr && handle_out, "mocha_peer_alloc: bad argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle size");
  void* p = nullptr;
  MOCHA_CUDA(cudaMalloc(&p, bytes));
  MOCHA_CUDA(cudaMemset(p, 0, bytes));
  cudaIpcMemHandle_t h;
  MOCHA_CUDA(cudaIpcGetMemHandle(&h, p));
  memcpy(handle_out, &h, 64);
  *d_ptr = p;
  return MOCHA_OK;
}

extern "C" int mocha_peer_open(const unsigned char handle[64], void** d_ptr) {
  MOCHA_CHECK_ARG(handle && d_ptr, "mocha_peer_open: bad argument");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  MOCHA_CUDA(cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return MOCHA_OK;
}

extern "C" int mocha_peer_close(void* d_ptr) {
  MOCHA_CUDA(cudaIpcCloseMemHandle(d_ptr));
  return MOCHA_OK;
}

extern "C" int mocha_peer_free(void* d_ptr) {
  MOCHA_CUDA(cudaFree(d_ptr));
  return MOCHA_OK;
}

extern "C" int mocha_topk_exchange_merge(const double* d_local_dist, const int64_t* d_local_idx, int nq, int k, int rank,
                                         int world, void* const* d_peer_bufs, unsigned int epoch, double* d_out_dist,
                                         int64_t* d_out_idx, mocha_stream_t stream) {
  MOCHA_CHECK_ARG(d_local_dist && d_local_idx && d_peer_bufs && d_out_dist && d_out_idx, "mocha_topk_exchange_merge: null argument");
  MOCHA_CHECK_ARG(nq > 0 && k >= 1 && k <= KMAX && world >= 1 && world <= XCHG_MAX_WORLD && rank >= 0 && rank < world,
                  "mocha_topk_exchange_merge: bad sizes");
  MOCHA_CHECK_ARG(((reinterpret_cast<uintptr_t>(d_local_dist) | reinterpret_cast<uintptr_t>(d_local_idx)) & 15) == 0,
                  "mocha_topk_exchange_merge: local lists must be 16 B aligned");
  // d_peer_bufs is a HOST array of device pointers (copied into the kernel's parameter space)
  XchgPtrs peers{};
  for (int p = 0; p < world; ++p) {
    MOCHA_CHECK_ARG(d_peer_bufs[p], "mocha_topk_exchange_merge: peer buffer %d is null", p);
    peers.buf[p] = static_cast<unsigned char*>(d_peer_bufs[p]);
  }
  launch_k(topk_exchange_merge_kernel, XCHG_BLOCKS, 256, 0, (cudaStream_t)stream, d_local_dist, reinterpret_cast<const long long*>(d_local_idx), nq, k, rank, world, peers, epoch, d_out_dist,
      reinterpret_cast<long long*>(d_out_idx));
  count_launch();
  MOCHA_LAUNCH_CHECK("topk_exchange_merge_kernel");
  return MOCHA_OK;
}
