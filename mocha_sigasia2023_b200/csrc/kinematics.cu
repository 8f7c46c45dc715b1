// Quaternion forward kinematics, two-bone IK, inertialization and the per-frame post-process
// (SURVEY §8 rows a10-a18). Quaternion layout is [w,x,y,z] as in the reference's motion/quat.py.
// Bandwidth/latency-bound: batch kernels stage one skeleton per warp in shared memory (coalesced
// loads, joint hierarchy walked level by level with one lane per joint); the stateful per-clip
// post-process runs one thread per clip in fp64 like the reference's NumPy state.
#include "../../include/mocha_b200.h"
#include "common.cuh"

using namespace mocha;

namespace {

template <typename T>
struct V3 { T x, y, z; };
template <typename T>
struct Q4 { T w, x, y, z; };

template <typename T> __device__ __forceinline__ V3<T> v3(T x, T y, T z) { V3<T> r; r.x = x; r.y = y; r.z = z; return r; }
template <typename T> __device__ __forceinline__ V3<T> operator+(V3<T> a, V3<T> b) { return v3<T>(a.x + b.x, a.y + b.y, a.z + b.z); }
template <typename T> __device__ __forceinline__ V3<T> operator-(V3<T> a, V3<T> b) { return v3<T>(a.x - b.x, a.y - b.y, a.z - b.z); }
template <typename T> __device__ __forceinline__ V3<T> operator*(T s, V3<T> a) { return v3<T>(s * a.x, s * a.y, s * a.z); }
template <typename T> __device__ __forceinline__ T dot(V3<T> a, V3<T> b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
template <typename T> __device__ __forceinline__ V3<T> cross(V3<T> a, V3<T> b) {
  return v3<T>(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
template <typename T> __device__ __forceinline__ T vlen(V3<T> a) { return sqrt(dot(a, a)); }
// quat.normalize for 3-vectors: x / (|x| + eps)  (motion/quat.py:15)
template <typename T> __device__ __forceinline__ V3<T> vnormalize(V3<T> a) {
  const T d = vlen(a) + (T)1e-8;
  return v3<T>(a.x / d, a.y / d, a.z / d);
}
template <typename T> __device__ __forceinline__ Q4<T> q4(T w, T x, T y, T z) { Q4<T> r; r.w = w; r.x = x; r.y = y; r.z = z; return r; }
template <typename T> __device__ __forceinline__ V3<T> qvec(Q4<T> q) { return v3<T>(q.x, q.y, q.z); }

// quat.mul (motion/quat.py:112-120)
template <typename T> __device__ __forceinline__ Q4<T> qmul(Q4<T> a, Q4<T> b) {
  return q4<T>(b.w * a.w - b.x * a.x - b.y * a.y - b.z * a.z,
               b.w * a.x + b.x * a.w - b.y * a.z + b.z * a.y,
               b.w * a.y + b.x * a.z + b.y * a.w - b.z * a.x,
               b.w * a.z - b.x * a.y + b.y * a.x + b.z * a.w);
}
template <typename T> __device__ __forceinline__ Q4<T> qinv(Q4<T> q) { return q4<T>(q.w, -q.x, -q.y, -q.z); }
// quat.mul_vec (motion/quat.py:128-130)
template <typename T> __device__ __forceinline__ V3<T> qrot(Q4<T> q, V3<T> x) {
  const V3<T> t = (T)2 * cross(qvec(q), x);
  return x + q.w * t + cross(qvec(q), t);
}
// quat.mul_vec / quat.inv_mul_vec (motion/quat.py:128-133): mocha_quat_op's ops 3 and 4, and the source windows' root
// velocities
template <typename T> __device__ __forceinline__ V3<T> q_mul_vec(const T* q4p, const T* x, bool inv) {
  Q4<T> q = q4<T>(q4p[0], q4p[1], q4p[2], q4p[3]);
  if (inv) q = qinv(q);
  return qrot(q, v3<T>(x[0], x[1], x[2]));
}
template <typename T> __device__ __forceinline__ Q4<T> qnormalize(Q4<T> q) {
  const T d = sqrt(q.w * q.w + q.x * q.x + q.y * q.y + q.z * q.z) + (T)1e-8;
  return q4<T>(q.w / d, q.x / d, q.y / d, q.z / d);
}
template <typename T> __device__ __forceinline__ Q4<T> qabs(Q4<T> q) {
  return q.w > (T)0 ? q : q4<T>(-q.w, -q.x, -q.y, -q.z);
}
// quat.from_angle_axis (motion/quat.py:21-25)
template <typename T> __device__ __forceinline__ Q4<T> q_angle_axis(T angle, V3<T> axis) {
  const T c = cos(angle / (T)2), s = sin(angle / (T)2);
  return q4<T>(c, s * axis.x, s * axis.y, s * axis.z);
}
// quat.exp (motion/quat.py:154-158); np.sinc(h/pi) = sin(h)/h
template <typename T> __device__ __forceinline__ Q4<T> qexp(V3<T> x) {
  const T h = vlen(x);
  const T c = h < (T)1e-5 ? (T)1 : cos(h);
  const T s = h < (T)1e-5 ? (T)1 : sin(h) / h;
  return q4<T>(c, s * x.x, s * x.y, s * x.z);
}
// quat.log (motion/quat.py:149-152)
template <typename T> __device__ __forceinline__ V3<T> qlog(Q4<T> q) {
  const T len = vlen(qvec(q));
  const T ha = len < (T)1e-5 ? (T)1 : atan2(len, q.w) / len;
  return ha * qvec(q);
}
template <typename T> __device__ __forceinline__ Q4<T> q_from_scaled_angle_axis(V3<T> x) { return qexp((T)0.5 * x); }
template <typename T> __device__ __forceinline__ V3<T> q_to_scaled_angle_axis(Q4<T> q) { return (T)2 * qlog(q); }

// quat.from_xform (motion/quat.py:69-94): 4-branch matrix -> quaternion, then normalize
template <typename T> __device__ __forceinline__ Q4<T> q_from_xform(const T (&m)[3][3]) {
  Q4<T> q;
  if (m[2][2] < (T)0) {
    if (m[0][0] > m[1][1])
      q = q4<T>(m[2][1] - m[1][2], (T)1 + m[0][0] - m[1][1] - m[2][2], m[1][0] + m[0][1], m[0][2] + m[2][0]);
    else
      q = q4<T>(m[0][2] - m[2][0], m[1][0] + m[0][1], (T)1 - m[0][0] + m[1][1] - m[2][2], m[2][1] + m[1][2]);
  } else {
    if (m[0][0] < -m[1][1])
      q = q4<T>(m[1][0] - m[0][1], m[0][2] + m[2][0], m[2][1] + m[1][2], (T)1 - m[0][0] - m[1][1] + m[2][2]);
    else
      q = q4<T>((T)1 + m[0][0] + m[1][1] + m[2][2], m[2][1] - m[1][2], m[0][2] - m[2][0], m[1][0] - m[0][1]);
  }
  return qnormalize(q);
}
// quat.from_xform_xy (motion/quat.py:96-107): Gram-Schmidt through two cross products
template <typename T> __device__ __forceinline__ Q4<T> q_from_xy(V3<T> c0, V3<T> c1in) {
  V3<T> c2 = cross(c0, c1in);
  T n = sqrt(dot(c2, c2));
  c2 = v3<T>(c2.x / n, c2.y / n, c2.z / n);
  V3<T> c1 = cross(c2, c0);
  n = sqrt(dot(c1, c1));
  c1 = v3<T>(c1.x / n, c1.y / n, c1.z / n);
  const T m[3][3] = {{c0.x, c1.x, c2.x}, {c0.y, c1.y, c2.y}, {c0.z, c1.z, c2.z}};
  return q_from_xform(m);
}

// ------------------------------------------------------------------------------------------------
// element-wise rotation format conversions
// ------------------------------------------------------------------------------------------------
__global__ void xy_to_quat_kernel(const float* __restrict__ xy, long long n, float* __restrict__ out) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* p = xy + i * 6;  // [3][2]
  const Q4<float> q = q_from_xy(v3<float>(p[0], p[2], p[4]), v3<float>(p[1], p[3], p[5]));
  reinterpret_cast<float4*>(out)[i] = make_float4(q.w, q.x, q.y, q.z);
}

// quat.to_xform_xy (motion/quat.py:42-55)
__global__ void quat_to_xy_kernel(const float* __restrict__ quat, long long n, float* __restrict__ out) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 q = reinterpret_cast<const float4*>(quat)[i];
  const float qw = q.x, qx = q.y, qy = q.z, qz = q.w;
  const float x2 = qx + qx, y2 = qy + qy, z2 = qz + qz;
  const float xx = qx * x2, yy = qy * y2, wx = qw * x2;
  const float xy = qx * y2, yz = qy * z2, wy = qw * y2;
  const float xz = qx * z2, zz = qz * z2, wz = qw * z2;
  float* o = out + i * 6;
  o[0] = 1.0f - (yy + zz); o[1] = xy - wz;
  o[2] = xy + wz;          o[3] = 1.0f - (xx + zz);
  o[4] = xz - wy;          o[5] = yz + wx;
}

// ------------------------------------------------------------------------------------------------
// batch FK / FK with velocities / inverse (global -> local): one warp per skeleton
// ------------------------------------------------------------------------------------------------
constexpr int MAXJ = 32;
constexpr int FK_WARPS = 4;

template <typename T>
struct SkelSmem {
  T rot[MAXJ][4], pos[MAXJ][3], vel[MAXJ][3], ang[MAXJ][3];
  T grot[MAXJ][4], gpos[MAXJ][3], gvel[MAXJ][3], gang[MAXJ][3];
};

template <typename T>
__device__ __forceinline__ void warp_copy_in(T* dst, const T* __restrict__ src, int n, int lane) {
  for (int i = lane; i < n; i += 32) dst[i] = src[i];
}
template <typename T>
__device__ __forceinline__ void warp_copy_out(T* __restrict__ dst, const T* src, int n, int lane) {
  for (int i = lane; i < n; i += 32) dst[i] = src[i];
}

// Joint steps shared by the batch kernels and source_windows_kernel, which must reproduce their results bit for bit.
// quat.fk / quat.fk_vel (motion/quat.py:166-204): global transform of a joint from its parent's (pr, pp); rp is the
// parent-rotated offset the velocity step needs.
__device__ __forceinline__ void fk_joint_pose(Q4<float> pr, V3<float> pp, Q4<float> lr, V3<float> lp, V3<float>& rp,
                                              V3<float>& gp, Q4<float>& gr) {
  rp = qrot(pr, lp);
  gp = rp + pp;
  gr = qmul(pr, lr);
}
__device__ __forceinline__ void fk_joint_vel(Q4<float> pr, V3<float> rp, V3<float> pv, V3<float> pa, V3<float> lv,
                                             V3<float> la, V3<float>& gv, V3<float>& ga) {
  gv = qrot(pr, lv) + cross(pa, rp) + pv;
  ga = qrot(pr, la) + pa;
}
// quat.ik (motion/quat.py:175-187) of a non-root joint
template <typename T>
__device__ __forceinline__ void ik_joint(Q4<T> pr, V3<T> pp, Q4<T> gr, V3<T> gp, Q4<T>& lr, V3<T>& lp) {
  const Q4<T> pinv = qinv(pr);
  lr = qmul(pinv, gr);
  lp = qrot(pinv, gp - pp);
}

// depth of joint `lane` in the hierarchy (parents[i] < i)
__device__ __forceinline__ int joint_depth(const int32_t* par, int j, int J) {
  int d = 0;
  if (j < J) { int p = par[j]; while (p >= 0) { ++d; p = par[p]; } }
  return d;
}

template <bool WITH_VEL, typename T>
__global__ void __launch_bounds__(FK_WARPS * 32)
fk_kernel(const T* __restrict__ lrot, const T* __restrict__ lpos, const T* __restrict__ lvel,
          const T* __restrict__ lang, const int32_t* __restrict__ parents, long long F, int J,
          T* __restrict__ grot, T* __restrict__ gpos, T* __restrict__ gvel, T* __restrict__ gang) {
  pdl_trigger();
  pdl_wait();
  __shared__ SkelSmem<T> sm[FK_WARPS];
  __shared__ int32_t par[MAXJ];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x < J) par[threadIdx.x] = parents[threadIdx.x];
  __syncthreads();
  const int depth = joint_depth(par, lane, J);
  int maxd = depth;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) maxd = max(maxd, __shfl_xor_sync(0xffffffffu, maxd, o));
  SkelSmem<T>& s = sm[warp];
  for (long long f = (long long)blockIdx.x * FK_WARPS + warp; f < F; f += (long long)gridDim.x * FK_WARPS) {
    warp_copy_in(&s.rot[0][0], lrot + f * J * 4, J * 4, lane);
    warp_copy_in(&s.pos[0][0], lpos + f * J * 3, J * 3, lane);
    if (WITH_VEL) {
      warp_copy_in(&s.vel[0][0], lvel + f * J * 3, J * 3, lane);
      warp_copy_in(&s.ang[0][0], lang + f * J * 3, J * 3, lane);
    }
    __syncwarp();
    // quat.fk / quat.fk_vel (motion/quat.py:166-204): level-synchronous walk, one lane per joint
    for (int lvl = 0; lvl <= maxd; ++lvl) {
      if (lane < J && depth == lvl) {
        const int j = lane;
        const Q4<T> lr = q4<T>(s.rot[j][0], s.rot[j][1], s.rot[j][2], s.rot[j][3]);
        const V3<T> lp = v3<T>(s.pos[j][0], s.pos[j][1], s.pos[j][2]);
        if (lvl == 0) {
          s.grot[j][0] = lr.w; s.grot[j][1] = lr.x; s.grot[j][2] = lr.y; s.grot[j][3] = lr.z;
          s.gpos[j][0] = lp.x; s.gpos[j][1] = lp.y; s.gpos[j][2] = lp.z;
          if (WITH_VEL) {
            for (int c = 0; c < 3; ++c) { s.gvel[j][c] = s.vel[j][c]; s.gang[j][c] = s.ang[j][c]; }
          }
        } else {
          const int p = par[j];
          const Q4<T> pr = q4<T>(s.grot[p][0], s.grot[p][1], s.grot[p][2], s.grot[p][3]);
          const V3<T> pp = v3<T>(s.gpos[p][0], s.gpos[p][1], s.gpos[p][2]);
          const V3<T> rp = qrot(pr, lp);
          const V3<T> gp = rp + pp;
          const Q4<T> gr = qmul(pr, lr);
          s.gpos[j][0] = gp.x; s.gpos[j][1] = gp.y; s.gpos[j][2] = gp.z;
          s.grot[j][0] = gr.w; s.grot[j][1] = gr.x; s.grot[j][2] = gr.y; s.grot[j][3] = gr.z;
          if (WITH_VEL) {
            const V3<T> lv = v3<T>(s.vel[j][0], s.vel[j][1], s.vel[j][2]);
            const V3<T> la = v3<T>(s.ang[j][0], s.ang[j][1], s.ang[j][2]);
            const V3<T> pv = v3<T>(s.gvel[p][0], s.gvel[p][1], s.gvel[p][2]);
            const V3<T> pa = v3<T>(s.gang[p][0], s.gang[p][1], s.gang[p][2]);
            const V3<T> gv = qrot(pr, lv) + cross(pa, rp) + pv;
            const V3<T> ga = qrot(pr, la) + pa;
            s.gvel[j][0] = gv.x; s.gvel[j][1] = gv.y; s.gvel[j][2] = gv.z;
            s.gang[j][0] = ga.x; s.gang[j][1] = ga.y; s.gang[j][2] = ga.z;
          }
        }
      }
      __syncwarp();
    }
    warp_copy_out(grot + f * J * 4, &s.grot[0][0], J * 4, lane);
    warp_copy_out(gpos + f * J * 3, &s.gpos[0][0], J * 3, lane);
    if (WITH_VEL) {
      warp_copy_out(gvel + f * J * 3, &s.gvel[0][0], J * 3, lane);
      warp_copy_out(gang + f * J * 3, &s.gang[0][0], J * 3, lane);
    }
    __syncwarp();
  }
}

// Streaming fp32 FK for large batches (window feature extraction runs it over clips x windows x frames skeletons): one
// THREAD per skeleton instead of one warp. The level-synchronous walk above keeps 25 lanes busy for one joint level at a
// time, round-trips through shared memory per level and stages with 4-byte loops (0.18 of the HBM roof; ncu: issue-bound).
// Here a warp owns 32 consecutive skeletons, whose inputs are contiguous slabs of the global arrays: each slab arrives with
// ONE bulk copy (cp.async.bulk, completion on the warp's mbarrier) in its global layout, every lane walks its skeleton's
// joints in index order in place (parents precede children, so joint j's parent is already global; same expressions as
// above; quaternions move as 16-byte vectors - conflict-free at any row stride - and the 3-vectors as scalars, whose row
// stride 3 J is odd for the 25-bone skeleton), and each slab leaves with one bulk store. No staging loops at all: the
// instruction stream is the quaternion algebra. Warps of an SM sit in different phases, which overlaps one warp's
// copies with another's walk. A last, partly filled group (slab sizes not multiples of 16 bytes) uses element loops.
__device__ __forceinline__ void fk_bulk_in(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
               "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void fk_bulk_out(void* dst, uint32_t src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
}

template <bool WITH_VEL, int WARPS>
__global__ void __launch_bounds__(WARPS * 32)
fk_rows_kernel(const float* __restrict__ lrot, const float* __restrict__ lpos, const float* __restrict__ lvel,
               const float* __restrict__ lang, const int32_t* __restrict__ parents, long long F, int J,
               float* __restrict__ grot, float* __restrict__ gpos, float* __restrict__ gvel, float* __restrict__ gang) {
  pdl_trigger();
  extern __shared__ __align__(16) float fk_sm[];
  __shared__ int32_t par[MAXJ];
  __shared__ __align__(8) unsigned long long bars[WARPS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n4 = J * 4, n3 = J * 3;
  const int per_warp = 32 * (n4 + n3 * (WITH_VEL ? 3 : 1));
  float* rot = fk_sm + warp * per_warp;
  float* pos = rot + 32 * n4;
  float* vel = pos + 32 * n3;
  float* ang = vel + 32 * n3;
  const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&bars[warp]);
  if (lane == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  pdl_wait();
  if (threadIdx.x < J) par[threadIdx.x] = parents[threadIdx.x];
  __syncthreads();
  uint32_t parity = 0;
  const long long groups = (F + 31) / 32;
  for (long long grp = (long long)blockIdx.x * WARPS + warp; grp < groups; grp += (long long)gridDim.x * WARPS) {
    const long long f0 = grp * 32;
    const int cnt = (int)min(32LL, F - f0);
    const bool full = cnt == 32;     // warp-uniform
    if (full) {
      if (lane == 0) {
        // the previous group's bulk stores have finished reading this warp's buffers
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        const uint32_t b4 = 32u * n4 * 4u, b3 = 32u * n3 * 4u;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(b4 + b3 * (WITH_VEL ? 3u : 1u)) : "memory");
        fk_bulk_in((uint32_t)__cvta_generic_to_shared(rot), lrot + f0 * n4, b4, bar);
        fk_bulk_in((uint32_t)__cvta_generic_to_shared(pos), lpos + f0 * n3, b3, bar);
        if (WITH_VEL) {
          fk_bulk_in((uint32_t)__cvta_generic_to_shared(vel), lvel + f0 * n3, b3, bar);
          fk_bulk_in((uint32_t)__cvta_generic_to_shared(ang), lang + f0 * n3, b3, bar);
        }
      }
      uint32_t done = 0;
      while (!done)
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
      parity ^= 1u;
    } else {
      if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
      __syncwarp();
      for (int i = lane; i < cnt * n4; i += 32) rot[i] = lrot[f0 * n4 + i];
      for (int i = lane; i < cnt * n3; i += 32) pos[i] = lpos[f0 * n3 + i];
      if (WITH_VEL) {
        for (int i = lane; i < cnt * n3; i += 32) { vel[i] = lvel[f0 * n3 + i]; ang[i] = lang[f0 * n3 + i]; }
      }
      __syncwarp();
    }
    if (lane < cnt) {
      float4* r = reinterpret_cast<float4*>(rot + lane * n4);
      float* x = pos + lane * n3;
      float* v = vel + lane * n3;
      float* a = ang + lane * n3;
      // quat.fk / quat.fk_vel (motion/quat.py:166-204)
      for (int j = 0; j < J; ++j) {
        const int p = par[j];
        if (p < 0) continue;            // a root's global transform is its local one
        const float4 lr4 = r[j], pr4 = r[p];
        const Q4<float> lr = q4<float>(lr4.x, lr4.y, lr4.z, lr4.w);
        const Q4<float> pr = q4<float>(pr4.x, pr4.y, pr4.z, pr4.w);
        const V3<float> lp = v3<float>(x[3 * j], x[3 * j + 1], x[3 * j + 2]);
        const V3<float> pp = v3<float>(x[3 * p], x[3 * p + 1], x[3 * p + 2]);
        V3<float> rp, gp;
        Q4<float> gr;
        fk_joint_pose(pr, pp, lr, lp, rp, gp, gr);
        x[3 * j] = gp.x; x[3 * j + 1] = gp.y; x[3 * j + 2] = gp.z;
        r[j] = make_float4(gr.w, gr.x, gr.y, gr.z);
        if (WITH_VEL) {
          const V3<float> lv = v3<float>(v[3 * j], v[3 * j + 1], v[3 * j + 2]);
          const V3<float> la = v3<float>(a[3 * j], a[3 * j + 1], a[3 * j + 2]);
          const V3<float> pv = v3<float>(v[3 * p], v[3 * p + 1], v[3 * p + 2]);
          const V3<float> pa = v3<float>(a[3 * p], a[3 * p + 1], a[3 * p + 2]);
          V3<float> gv, ga;
          fk_joint_vel(pr, rp, pv, pa, lv, la, gv, ga);
          v[3 * j] = gv.x; v[3 * j + 1] = gv.y; v[3 * j + 2] = gv.z;
          a[3 * j] = ga.x; a[3 * j + 1] = ga.y; a[3 * j + 2] = ga.z;
        }
      }
    }
    if (full) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      if (lane == 0) {
        const uint32_t b4 = 32u * n4 * 4u, b3 = 32u * n3 * 4u;
        fk_bulk_out(grot + f0 * n4, (uint32_t)__cvta_generic_to_shared(rot), b4);
        fk_bulk_out(gpos + f0 * n3, (uint32_t)__cvta_generic_to_shared(pos), b3);
        if (WITH_VEL) {
          fk_bulk_out(gvel + f0 * n3, (uint32_t)__cvta_generic_to_shared(vel), b3);
          fk_bulk_out(gang + f0 * n3, (uint32_t)__cvta_generic_to_shared(ang), b3);
        }
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
    } else {
      __syncwarp();
      for (int i = lane; i < cnt * n4; i += 32) grot[f0 * n4 + i] = rot[i];
      for (int i = lane; i < cnt * n3; i += 32) gpos[f0 * n3 + i] = pos[i];
      if (WITH_VEL) {
        for (int i = lane; i < cnt * n3; i += 32) { gvel[f0 * n3 + i] = vel[i]; gang[f0 * n3 + i] = ang[i]; }
      }
      __syncwarp();
    }
  }
  if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// quat.ik (motion/quat.py:175-187)
template <typename T>
__global__ void __launch_bounds__(FK_WARPS * 32)
ik_kernel(const T* __restrict__ grot, const T* __restrict__ gpos, const int32_t* __restrict__ parents,
          long long F, int J, T* __restrict__ lrot, T* __restrict__ lpos) {
  pdl_trigger();
  pdl_wait();
  __shared__ SkelSmem<T> sm[FK_WARPS];
  __shared__ int32_t par[MAXJ];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x < J) par[threadIdx.x] = parents[threadIdx.x];
  __syncthreads();
  SkelSmem<T>& s = sm[warp];
  for (long long f = (long long)blockIdx.x * FK_WARPS + warp; f < F; f += (long long)gridDim.x * FK_WARPS) {
    warp_copy_in(&s.grot[0][0], grot + f * J * 4, J * 4, lane);
    warp_copy_in(&s.gpos[0][0], gpos + f * J * 3, J * 3, lane);
    __syncwarp();
    if (lane < J) {
      const int j = lane;
      const Q4<T> gr = q4<T>(s.grot[j][0], s.grot[j][1], s.grot[j][2], s.grot[j][3]);
      const V3<T> gp = v3<T>(s.gpos[j][0], s.gpos[j][1], s.gpos[j][2]);
      if (par[j] < 0) {
        s.rot[j][0] = gr.w; s.rot[j][1] = gr.x; s.rot[j][2] = gr.y; s.rot[j][3] = gr.z;
        s.pos[j][0] = gp.x; s.pos[j][1] = gp.y; s.pos[j][2] = gp.z;
      } else {
        const int p = par[j];
        const Q4<T> pr = q4<T>(s.grot[p][0], s.grot[p][1], s.grot[p][2], s.grot[p][3]);
        const V3<T> pp = v3<T>(s.gpos[p][0], s.gpos[p][1], s.gpos[p][2]);
        Q4<T> lr;
        V3<T> lp;
        ik_joint(pr, pp, gr, gp, lr, lp);
        s.rot[j][0] = lr.w; s.rot[j][1] = lr.x; s.rot[j][2] = lr.y; s.rot[j][3] = lr.z;
        s.pos[j][0] = lp.x; s.pos[j][1] = lp.y; s.pos[j][2] = lp.z;
      }
    }
    __syncwarp();
    warp_copy_out(lrot + f * J * 4, &s.rot[0][0], J * 4, lane);
    warp_copy_out(lpos + f * J * 3, &s.pos[0][0], J * 3, lane);
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------------------------
// fp64 scalar pieces of the post-process
// ------------------------------------------------------------------------------------------------
typedef V3<double> D3;
typedef Q4<double> DQ;

__device__ __forceinline__ D3 ld3(const double* p) { return v3<double>(p[0], p[1], p[2]); }
__device__ __forceinline__ void st3(double* p, D3 v) { p[0] = v.x; p[1] = v.y; p[2] = v.z; }
__device__ __forceinline__ DQ ld4(const double* p) { return q4<double>(p[0], p[1], p[2], p[3]); }
__device__ __forceinline__ void st4(double* p, DQ q) { p[0] = q.w; p[1] = q.x; p[2] = q.y; p[3] = q.z; }

// Inertialization.fast_negexpf / halflife_to_damping (Inertialization.py:10-14)
__device__ __forceinline__ double fast_negexp(double x) { return 1.0 / (1.0 + x + 0.48 * x * x + 0.235 * x * x * x); }
__device__ __forceinline__ double halflife_to_damping(double halflife) { return (4.0 * 0.693147180559945309417) / (halflife + 1e-5); }

// decay_spring_damper_exact, vec3 branch (Inertialization.py:39-54)
__device__ __forceinline__ void decay_spring_pos(D3& x, D3& v, double halflife, double dt) {
  const double y = halflife_to_damping(halflife) / 2.0;
  const double eydt = fast_negexp(y * dt);
  const D3 j1 = v + y * x;
  const D3 nx = eydt * (x + dt * j1);
  const D3 nv = eydt * (v - (y * dt) * j1);
  x = nx; v = nv;
}
// decay_spring_damper_exact_rot (Inertialization.py:28-37)
__device__ __forceinline__ void decay_spring_rot(DQ& x, D3& v, double halflife, double dt) {
  const double y = halflife_to_damping(halflife) / 2.0;
  const D3 j0 = q_to_scaled_angle_axis(x);
  const D3 j1 = v + y * j0;
  const double eydt = fast_negexp(y * dt);
  x = q_from_scaled_angle_axis(eydt * (j0 + dt * j1));
  v = eydt * (v - (y * dt) * j1);
}

struct ContactState {
  bool state, lock;
  D3 position, velocity, point, target, off_pos, off_vel;
};

// Inertialization.contact_update (Inertialization.py:300-377)
__device__ void contact_update_dev(ContactState& c, D3 input_position, bool input_state, double unlock_radius,
                                   double foot_height, double halflife, double dt) {
  const double eps = 1e-8;
  // finite-difference input velocity; the reference divides by (dt + eps)
  D3 iv = input_position - c.target;
  iv = v3<double>(iv.x / (dt + eps), iv.y / (dt + eps), iv.z / (dt + eps));
  c.target = input_position;
  // inertialize_update (:110-127): decay the offsets, then add them to the fed input
  decay_spring_pos(c.off_pos, c.off_vel, halflife, dt);
  const D3 in_x = c.lock ? c.point : input_position;
  const D3 in_v = c.lock ? v3<double>(0.0, 0.0, 0.0) : iv;
  c.position = in_x + c.off_pos;
  c.velocity = in_v + c.off_vel;
  const bool unlock = c.lock && (vlen(c.point - input_position) > unlock_radius);
  if (!c.state && input_state) {
    c.lock = true;
    c.point = c.position;
    c.point.y = foot_height;
    // inertialize_transition (:93-108), src = input, dst = contact point at rest
    c.off_pos = (input_position + c.off_pos) - c.point;
    c.off_vel = (iv + c.off_vel) - v3<double>(0.0, 0.0, 0.0);
  } else if ((c.lock && c.state && !input_state) || unlock) {
    c.lock = false;
    c.off_pos = (c.point + c.off_pos) - input_position;
    c.off_vel = (v3<double>(0.0, 0.0, 0.0) + c.off_vel) - iv;
  }
  c.state = input_state;
}

__device__ __forceinline__ double clip1(double x) { return fmin(1.0, fmax(-1.0, x)); }

// quat.ik_two_bone (motion/quat.py:295-343)
__device__ void ik_two_bone_dev(D3 bone_root, D3 bone_mid, D3 bone_end, D3 target, D3 fwd, DQ root_gr, DQ mid_gr,
                                DQ par_gr, double max_length_buffer, DQ& out_root_lr, DQ& out_mid_lr) {
  const double max_extension = vlen(bone_root - bone_mid) + vlen(bone_mid - bone_end) - max_length_buffer;
  D3 t = target;
  if (vlen(target - bone_root) > max_extension) t = bone_root + max_extension * vnormalize(target - bone_root);
  const D3 axis_dwn = vnormalize(bone_end - bone_root);
  const D3 axis_rot = vnormalize(cross(axis_dwn, fwd));
  const D3 a = bone_root, b = bone_mid, c = bone_end;
  const double lab = vlen(b - a), lcb = vlen(b - c), lat = vlen(t - a);
  const double ac_ab_0 = acos(clip1(dot(vnormalize(c - a), vnormalize(b - a))));
  const double ba_bc_0 = acos(clip1(dot(vnormalize(a - b), vnormalize(c - b))));
  const double ac_ab_1 = acos(clip1((lab * lab + lat * lat - lcb * lcb) / (2.0 * lab * lat)));
  const double ba_bc_1 = acos(clip1((lab * lab + lcb * lcb - lat * lat) / (2.0 * lab * lcb)));
  const DQ r0 = q_angle_axis(ac_ab_1 - ac_ab_0, axis_rot);
  const DQ r1 = q_angle_axis(ba_bc_1 - ba_bc_0, axis_rot);
  const D3 c_a = vnormalize(bone_end - bone_root);
  const D3 t_a = vnormalize(t - bone_root);
  const DQ r2 = q_angle_axis(acos(clip1(dot(c_a, t_a))), vnormalize(cross(c_a, t_a)));
  out_root_lr = qmul(qinv(par_gr), qmul(r2, qmul(r0, root_gr)));
  out_mid_lr = qmul(qinv(root_gr), qmul(r1, mid_gr));
}

// ------------------------------------------------------------------------------------------------
// Frame-0 pieces shared by both post-process kernels (one definition, so the general kernel's init frame and the
// step kernel's per-clip init agree bit for bit).
// ------------------------------------------------------------------------------------------------
// source root at frame 0 (:476-483): integrated from the identity in fp64, stored as float32 values like the reference
__device__ __forceinline__ void src_root_init_dev(mocha_frame_out& O, V3<float> rv, V3<float> ra, double dt) {
  const D3 p0 = dt * v3<double>((double)rv.x, (double)rv.y, (double)rv.z);
  const DQ r0 = q_from_scaled_angle_axis(dt * v3<double>((double)ra.x, (double)ra.y, (double)ra.z));
  st3(O.src_root_vel, v3<double>((double)rv.x, (double)rv.y, (double)rv.z));
  st3(O.src_root_ang, v3<double>((double)ra.x, (double)ra.y, (double)ra.z));
  st3(O.src_root_pos, v3<double>((double)(float)p0.x, (double)(float)p0.y, (double)(float)p0.z));
  st4(O.src_root_rot, q4<double>((double)(float)r0.w, (double)(float)r0.x, (double)(float)r0.y, (double)(float)r0.z));
}

// contact reset of foot f at frame 0 (:403-431): quat.fk_vel_bone (motion/quat.py:207-237) along the toe's ancestor
// chain (chain[0] = toe ... chain[n-1] = root) on the raw pose, then position = point = target = the toe
__device__ __forceinline__ void contact_init_dev(mocha_clip_state& S, const mocha_frame_out& O, const int* chain, int n,
                                                 int f) {
  D3 gp = ld3(O.pos[chain[n - 1]]), gv = ld3(O.vel[chain[n - 1]]), ga = ld3(O.ang[chain[n - 1]]);
  DQ gr = ld4(O.rot[chain[n - 1]]);
  for (int k = n - 2; k >= 0; --k) {
    const int j = chain[k];
    const D3 rp = qrot(gr, ld3(O.pos[j]));
    const D3 nv = gv + qrot(gr, ld3(O.vel[j])) + cross(ga, rp);
    const D3 na = qrot(gr, ld3(O.ang[j])) + ga;
    gp = rp + gp; gv = nv; ga = na;
    gr = qmul(gr, ld4(O.rot[j]));
  }
  S.contact_state[f] = 0; S.contact_lock[f] = 0;
  st3(S.contact_position[f], gp); st3(S.contact_velocity[f], gv);
  st3(S.contact_point[f], gp); st3(S.contact_target[f], gp);
  st3(S.contact_offset_position[f], v3<double>(0, 0, 0)); st3(S.contact_offset_velocity[f], v3<double>(0, 0, 0));
}

// ------------------------------------------------------------------------------------------------
// per-frame post-process, one WARP per clip: lanes split the 60-frame speed-ratio reduction, the 24
// joints of the pose assembly, the 25 bones of the blending and the two feet of the contact / IK step;
// lane 0 integrates the roots. Phases exchange data through the clip's output struct (__syncwarp).
// start != NULL: clip b runs the frame-0 branch iff start[b] != 0 (per-clip admission; `init` is ignored).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
post_frame_kernel(const mocha_post_params P, const float* __restrict__ Y,
                  const float* __restrict__ src_hips_vel, const float* __restrict__ src_rvel,
                  const float* __restrict__ src_rang, const uint8_t* __restrict__ contacts, int B,
                  int T, int V, int Cin, int init, const uint8_t* __restrict__ start, mocha_clip_state* __restrict__ states,
                  mocha_frame_out* __restrict__ outs, int hv_stride, int rv_stride) {
  pdl_trigger();
  pdl_wait();
  const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (b >= B) return;  // warp-uniform
  if (start) init = start[b] != 0;   // warp-uniform (one warp per clip)
  mocha_clip_state& S = states[b];
  mocha_frame_out& O = outs[b];
  const int J = P.J;
  const double dt = P.dt;
  const float* Yb = Y + (long long)b * T * V * Cin;
  const float* last = Yb + (long long)(T - 1) * V * Cin;

  // speed ratio (test_fullframework.py:492-496): mean |hips vel| over the window, fp32 like NumPy
  float num = 0.f, den = 0.f;
  for (int t = lane; t < T; t += 32) {
    const float* yv = Yb + ((long long)t * V + 0) * Cin + 9;
    num += sqrtf(yv[0] * yv[0] + yv[1] * yv[1] + yv[2] * yv[2]);
    const float* sv = src_hips_vel + (long long)b * hv_stride + t * 3;
    den += sqrtf(sv[0] * sv[0] + sv[1] * sv[1] + sv[2] * sv[2]);
  }
  num = warp_sum(num);
  den = warp_sum(den);
  float ratio = (num / (float)T) / (den / (float)T);
  if (ratio > 3.0f || ratio < 0.33f) ratio = 1.0f;

  DQ rootrot = q4<double>(1.0, 0.0, 0.0, 0.0);
  D3 rootpos = v3<double>(0.0, 0.0, 0.0);
  if (lane == 0) {
    const D3 yrvel = v3<double>((double)(src_rvel[(long long)b * rv_stride + 0] * ratio), (double)(src_rvel[(long long)b * rv_stride + 1] * ratio),
                                (double)(src_rvel[(long long)b * rv_stride + 2] * ratio));
    const D3 yrang = v3<double>((double)src_rang[(long long)b * rv_stride + 0], (double)src_rang[(long long)b * rv_stride + 1], (double)src_rang[(long long)b * rv_stride + 2]);
    // root integration (:500-503 / :345-348)
    const DQ prev_rot = init ? q4<double>(1.0, 0.0, 0.0, 0.0) : ld4(S.root_rot);
    const D3 prev_pos = init ? v3<double>(0.0, 0.0, 0.0) : ld3(S.root_pos);
    const D3 rootvel = qrot(prev_rot, yrvel);
    const D3 rootang = qrot(prev_rot, yrang);
    rootpos = prev_pos + dt * rootvel;
    rootrot = qmul(prev_rot, q_from_scaled_angle_axis(dt * rootang));
    st3(O.pos[0], rootpos); st3(O.vel[0], rootvel); st4(O.rot[0], rootrot); st3(O.ang[0], rootang);
  } else if (lane == 1) {
    // source root (:476-483): the reference keeps it in float32 arrays, so it integrates in fp32
    const V3<float> rv = v3<float>(src_rvel[(long long)b * rv_stride + 0], src_rvel[(long long)b * rv_stride + 1], src_rvel[(long long)b * rv_stride + 2]);
    const V3<float> ra = v3<float>(src_rang[(long long)b * rv_stride + 0], src_rang[(long long)b * rv_stride + 1], src_rang[(long long)b * rv_stride + 2]);
    if (init) {
      src_root_init_dev(O, rv, ra, dt);
    } else {
      const Q4<float> pr = q4<float>((float)S.src_root_rot[0], (float)S.src_root_rot[1], (float)S.src_root_rot[2],
                                     (float)S.src_root_rot[3]);
      const V3<float> pp = v3<float>((float)S.src_root_pos[0], (float)S.src_root_pos[1], (float)S.src_root_pos[2]);
      const float dtf = (float)dt;
      const V3<float> wv = qrot(pr, rv), wa = qrot(pr, ra);
      const V3<float> np_ = pp + dtf * wv;
      const Q4<float> nr = qmul(pr, q_from_scaled_angle_axis(dtf * wa));
      st3(O.src_root_vel, v3<double>((double)wv.x, (double)wv.y, (double)wv.z));
      st3(O.src_root_ang, v3<double>((double)wa.x, (double)wa.y, (double)wa.z));
      st3(O.src_root_pos, v3<double>((double)np_.x, (double)np_.y, (double)np_.z));
      st4(O.src_root_rot, q4<double>((double)nr.w, (double)nr.x, (double)nr.y, (double)nr.z));
    }
    for (int c = 0; c < 3; ++c) S.src_root_pos[c] = O.src_root_pos[c];
    for (int c = 0; c < 4; ++c) S.src_root_rot[c] = O.src_root_rot[c];
  }

  // assemble the 25-bone pose (:505-508): joint values are fp32 results promoted to fp64; lane = joint
  for (int j = lane; j < V; j += 32) {
    const float* y = last + (long long)j * Cin;
    O.pos[j + 1][0] = (double)y[0]; O.pos[j + 1][1] = (double)y[1]; O.pos[j + 1][2] = (double)y[2];
    const Q4<float> q = q_from_xy(v3<float>(y[3], y[5], y[7]), v3<float>(y[4], y[6], y[8]));
    O.rot[j + 1][0] = (double)q.w; O.rot[j + 1][1] = (double)q.x; O.rot[j + 1][2] = (double)q.y; O.rot[j + 1][3] = (double)q.z;
    O.vel[j + 1][0] = (double)y[9]; O.vel[j + 1][1] = (double)y[10]; O.vel[j + 1][2] = (double)y[11];
    O.ang[j + 1][0] = (double)y[12]; O.ang[j + 1][1] = (double)y[13]; O.ang[j + 1][2] = (double)y[14];
  }
  __syncwarp();

  if (init) {
    // frame 0 (:375-434): lists start from the raw pose; contacts reset from the toe's FK state
    for (int j = lane; j < J; j += 32) {
      for (int c = 0; c < 3; ++c) {
        O.blend_pos[j][c] = O.pos[j][c]; O.ik_pos[j][c] = O.pos[j][c];
        S.prev_pos[j][c] = O.pos[j][c]; S.prev_ik_pos[j][c] = O.pos[j][c];
      }
      for (int c = 0; c < 4; ++c) O.ik_rot[j][c] = O.rot[j][c];
    }
    if (lane < 2) {
      int chain[MAXJ]; int n = 0;
      for (int j = P.contact_bones[lane]; j >= 0; j = P.parents[j]) chain[n++] = j;
      contact_init_dev(S, O, chain, n, lane);
    }
    if (lane == 0) { st3(S.root_pos, rootpos); st4(S.root_rot, rootrot); }
    return;
  }

  // position blending (:532-536, :626); lane = bone
  for (int j = lane; j < J; j += 32) {
    for (int c = 0; c < 3; ++c) {
      O.ik_pos[j][c] = (S.prev_ik_pos[j][c] + O.vel[j][c] * dt) * 0.5 + O.pos[j][c] * 0.5;
      O.blend_pos[j][c] = (S.prev_pos[j][c] + O.vel[j][c] * dt) * 0.5 + O.pos[j][c] * 0.5;
    }
    for (int c = 0; c < 4; ++c) O.ik_rot[j][c] = O.rot[j][c];
  }
  __syncwarp();

  if (P.ik_enabled && lane < 2) {
    const int f = lane;  // the two feet touch disjoint bones and disjoint state slots
    const int toe = P.contact_bones[f], heel = P.parents[toe], knee = P.parents[heel], hip = P.parents[knee],
              rootb = P.parents[hip];
    // quat.fk_partial (motion/quat.py:241-272) along the toe's ancestor chain, on the blended pose
    int chain[MAXJ]; int n = 0;
    for (int j = toe; j >= 0; j = P.parents[j]) chain[n++] = j;
    D3 gpos[MAXJ]; DQ grot[MAXJ];
    {
      const int r = chain[n - 1];
      gpos[r] = ld3(O.ik_pos[r]); grot[r] = ld4(O.rot[r]);
      for (int k = n - 2; k >= 0; --k) {
        const int j = chain[k], p = chain[k + 1];
        gpos[j] = qrot(grot[p], ld3(O.ik_pos[j])) + gpos[p];
        grot[j] = qmul(grot[p], ld4(O.rot[j]));
      }
    }
    ContactState c;
    c.state = S.contact_state[f] != 0; c.lock = S.contact_lock[f] != 0;
    c.position = ld3(S.contact_position[f]); c.velocity = ld3(S.contact_velocity[f]);
    c.point = ld3(S.contact_point[f]); c.target = ld3(S.contact_target[f]);
    c.off_pos = ld3(S.contact_offset_position[f]); c.off_vel = ld3(S.contact_offset_velocity[f]);
    contact_update_dev(c, gpos[toe], contacts[b * 2 + f] != 0, P.ik_unlock_radius, P.ik_foot_height,
                       P.ik_blending_halflife, dt);
    // the clamp aliases contact_positions[bs] in the reference (:581-582): it persists
    c.position.y = fmax(c.position.y, P.ik_foot_height);
    S.contact_state[f] = c.state; S.contact_lock[f] = c.lock;
    st3(S.contact_position[f], c.position); st3(S.contact_velocity[f], c.velocity);
    st3(S.contact_point[f], c.point); st3(S.contact_target[f], c.target);
    st3(S.contact_offset_position[f], c.off_pos); st3(S.contact_offset_velocity[f], c.off_vel);

    const D3 target = c.position + (gpos[heel] - gpos[toe]);
    const D3 fwd = qrot(grot[knee], v3<double>(0.0, 1.0, 0.0));
    DQ new_hip, new_knee;
    ik_two_bone_dev(gpos[hip], gpos[knee], gpos[heel], target, fwd, grot[hip], grot[knee], grot[rootb],
                    P.ik_max_length_buffer, new_hip, new_knee);
    st4(O.ik_rot[hip], new_hip);
    st4(O.ik_rot[knee], new_knee);
  }
  __syncwarp();

  // carry state
  if (lane == 0) { st3(S.root_pos, ld3(O.blend_pos[0])); st4(S.root_rot, rootrot); }
  for (int j = lane; j < J; j += 32)
    for (int c = 0; c < 3; ++c) { S.prev_pos[j][c] = O.blend_pos[j][c]; S.prev_ik_pos[j][c] = O.ik_pos[j][c]; }
}

// ------------------------------------------------------------------------------------------------
// Steady-state frame (init == 0) of the same post-process, shaped for latency: the kernel above walks its phases through
// the clip's structs in GLOBAL memory (every phase boundary is an L2 round trip, the chain walk indexes local arrays), which
// made it a 20 us tail on a step whose last kernel it is. Here one single-warp block per clip (clips spread over the SMs)
// fetches everything the frame reads - state struct, last pose row, hips velocities, source root motion, contacts - in ONE
// round of independent loads, runs the phases on shared-memory copies of the two structs (same expressions, same order:
// fp64 results as above), and writes both structs back with 16-byte stores. The ancestor chains of the two contact bones
// depend only on the parameters and are built before the grid dependency resolves.
// MASKED: start[b] != 0 runs clip b's frame 0 instead (the general kernel's init branch: root from the identity, lists
// from the raw pose, contacts reset from the toe FK), so clips can start on any frame of a batch. The flag is one byte per
// block, read with the frame's other loads; the unmasked instantiation is the steady-state kernel alone.
// ------------------------------------------------------------------------------------------------
static_assert(sizeof(mocha_clip_state) % 16 == 0 && sizeof(mocha_frame_out) % 16 == 0, "struct copies use 16-byte vectors");
constexpr int PF_S16 = (int)(sizeof(mocha_clip_state) / 16), PF_O16 = (int)(sizeof(mocha_frame_out) / 16);
constexpr int PF_YMAX = 24 * 15;   // last pose row: V <= 24 joints x 15 features

template <bool MASKED>
__global__ void __launch_bounds__(32)
post_frame_step_kernel(const __grid_constant__ mocha_post_params P, const float* __restrict__ Y,
                       const float* __restrict__ src_hips_vel, const float* __restrict__ src_rvel,
                       const float* __restrict__ src_rang, const uint8_t* __restrict__ contacts,
                       const uint8_t* __restrict__ start, int T, int V, int Cin, mocha_clip_state* __restrict__ states,
                       mocha_frame_out* __restrict__ outs, int hv_stride, int rv_stride) {
  pdl_trigger();
  __shared__ __align__(16) mocha_frame_out Osh;
  __shared__ __align__(16) mocha_clip_state Ssh;
  __shared__ float ylast[PF_YMAX];
  __shared__ int chain_s[2][MAXJ];
  __shared__ int chain_n[2];
  const int b = blockIdx.x, lane = threadIdx.x;
  mocha_clip_state& S = Ssh;
  mocha_frame_out& O = Osh;
  const int J = P.J;
  const double dt = P.dt;
  // ---- before the grid dependency: parameters only ----
  for (int i = lane; i < PF_O16; i += 32) reinterpret_cast<double2*>(&Osh)[i] = make_double2(0.0, 0.0);
  if (lane < 2) {
    int n = 0;
    for (int j = P.contact_bones[lane]; j >= 0; j = P.parents[j]) chain_s[lane][n++] = j;
    chain_n[lane] = n;
  }
  pdl_wait();

  // ---- every global read of the frame, issued back to back ----
  const float* Yb = Y + (long long)b * T * V * Cin;
  const float* last = Yb + (long long)(T - 1) * V * Cin;
  const int nlast = V * Cin;
  const double2* Sg = reinterpret_cast<const double2*>(states + b);
  double2 sreg[(PF_S16 + 31) / 32];
#pragma unroll
  for (int k = 0; k < (PF_S16 + 31) / 32; ++k) {
    const int i = lane + 32 * k;
    sreg[k] = i < PF_S16 ? Sg[i] : make_double2(0.0, 0.0);
  }
  float yreg[(PF_YMAX + 31) / 32];
#pragma unroll
  for (int k = 0; k < (PF_YMAX + 31) / 32; ++k) {
    const int i = lane + 32 * k;
    yreg[k] = i < nlast ? last[i] : 0.f;
  }
  float yv[2][3], sv[2][3];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int t = lane + 32 * k;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      yv[k][c] = t < T ? Yb[((long long)t * V + 0) * Cin + 9 + c] : 0.f;
      sv[k][c] = t < T ? src_hips_vel[(long long)b * hv_stride + t * 3 + c] : 0.f;
    }
  }
  float rvf[3], raf[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) { rvf[c] = src_rvel[(long long)b * rv_stride + c]; raf[c] = src_rang[(long long)b * rv_stride + c]; }
  const bool contact_in = lane < 2 ? contacts[b * 2 + lane] != 0 : false;
  const bool init = MASKED && start[b] != 0;   // block-uniform

#pragma unroll
  for (int k = 0; k < (PF_S16 + 31) / 32; ++k) {
    const int i = lane + 32 * k;
    if (i < PF_S16) reinterpret_cast<double2*>(&Ssh)[i] = sreg[k];
  }
#pragma unroll
  for (int k = 0; k < (PF_YMAX + 31) / 32; ++k) {
    const int i = lane + 32 * k;
    if (i < nlast) ylast[i] = yreg[k];
  }

  // speed ratio (test_fullframework.py:492-496): mean |hips vel| over the window, fp32 like NumPy
  float num = 0.f, den = 0.f;
#pragma unroll
  for (int k = 0; k < 2; ++k)
    if (lane + 32 * k < T) {
      num += sqrtf(yv[k][0] * yv[k][0] + yv[k][1] * yv[k][1] + yv[k][2] * yv[k][2]);
      den += sqrtf(sv[k][0] * sv[k][0] + sv[k][1] * sv[k][1] + sv[k][2] * sv[k][2]);
    }
  for (int t = lane + 64; t < T; t += 32) {   // windows longer than 64 frames
    const float* y3 = Yb + ((long long)t * V + 0) * Cin + 9;
    num += sqrtf(y3[0] * y3[0] + y3[1] * y3[1] + y3[2] * y3[2]);
    const float* s3 = src_hips_vel + (long long)b * hv_stride + t * 3;
    den += sqrtf(s3[0] * s3[0] + s3[1] * s3[1] + s3[2] * s3[2]);
  }
  num = warp_sum(num);
  den = warp_sum(den);
  float ratio = (num / (float)T) / (den / (float)T);
  if (ratio > 3.0f || ratio < 0.33f) ratio = 1.0f;
  __syncwarp();   // state struct and pose row are in shared memory

  DQ rootrot = q4<double>(1.0, 0.0, 0.0, 0.0);
  if (lane == 0) {
    // root integration (:500-503 / :345-348)
    const D3 yrvel = v3<double>((double)(rvf[0] * ratio), (double)(rvf[1] * ratio), (double)(rvf[2] * ratio));
    const D3 yrang = v3<double>((double)raf[0], (double)raf[1], (double)raf[2]);
    const DQ prev_rot = init ? q4<double>(1.0, 0.0, 0.0, 0.0) : ld4(S.root_rot);
    const D3 prev_pos = init ? v3<double>(0.0, 0.0, 0.0) : ld3(S.root_pos);
    const D3 rootvel = qrot(prev_rot, yrvel);
    const D3 rootang = qrot(prev_rot, yrang);
    const D3 rootpos = prev_pos + dt * rootvel;
    rootrot = qmul(prev_rot, q_from_scaled_angle_axis(dt * rootang));
    st3(O.pos[0], rootpos); st3(O.vel[0], rootvel); st4(O.rot[0], rootrot); st3(O.ang[0], rootang);
  } else if (lane == 1) {
    // source root (:476-483): float32 arrays in the reference, so fp32 integration
    const V3<float> rv = v3<float>(rvf[0], rvf[1], rvf[2]);
    const V3<float> ra = v3<float>(raf[0], raf[1], raf[2]);
    if (init) {
      src_root_init_dev(O, rv, ra, dt);
    } else {
      const Q4<float> pr = q4<float>((float)S.src_root_rot[0], (float)S.src_root_rot[1], (float)S.src_root_rot[2],
                                     (float)S.src_root_rot[3]);
      const V3<float> pp = v3<float>((float)S.src_root_pos[0], (float)S.src_root_pos[1], (float)S.src_root_pos[2]);
      const float dtf = (float)dt;
      const V3<float> wv = qrot(pr, rv), wa = qrot(pr, ra);
      const V3<float> np_ = pp + dtf * wv;
      const Q4<float> nr = qmul(pr, q_from_scaled_angle_axis(dtf * wa));
      st3(O.src_root_vel, v3<double>((double)wv.x, (double)wv.y, (double)wv.z));
      st3(O.src_root_ang, v3<double>((double)wa.x, (double)wa.y, (double)wa.z));
      st3(O.src_root_pos, v3<double>((double)np_.x, (double)np_.y, (double)np_.z));
      st4(O.src_root_rot, q4<double>((double)nr.w, (double)nr.x, (double)nr.y, (double)nr.z));
    }
    for (int c = 0; c < 3; ++c) S.src_root_pos[c] = O.src_root_pos[c];
    for (int c = 0; c < 4; ++c) S.src_root_rot[c] = O.src_root_rot[c];
  }
  // assemble the pose (:505-508); lane = joint
  for (int j = lane; j < V; j += 32) {
    const float* y = ylast + j * Cin;
    O.pos[j + 1][0] = (double)y[0]; O.pos[j + 1][1] = (double)y[1]; O.pos[j + 1][2] = (double)y[2];
    const Q4<float> q = q_from_xy(v3<float>(y[3], y[5], y[7]), v3<float>(y[4], y[6], y[8]));
    O.rot[j + 1][0] = (double)q.w; O.rot[j + 1][1] = (double)q.x; O.rot[j + 1][2] = (double)q.y; O.rot[j + 1][3] = (double)q.z;
    O.vel[j + 1][0] = (double)y[9]; O.vel[j + 1][1] = (double)y[10]; O.vel[j + 1][2] = (double)y[11];
    O.ang[j + 1][0] = (double)y[12]; O.ang[j + 1][1] = (double)y[13]; O.ang[j + 1][2] = (double)y[14];
  }
  __syncwarp();

  if (init) {
    // frame 0 (:375-434): the lists start from the raw pose (the carry step below copies them into the state, and
    // blend_pos[0] is the identity-integrated root)
    for (int j = lane; j < J; j += 32) {
      for (int c = 0; c < 3; ++c) { O.blend_pos[j][c] = O.pos[j][c]; O.ik_pos[j][c] = O.pos[j][c]; }
      for (int c = 0; c < 4; ++c) O.ik_rot[j][c] = O.rot[j][c];
    }
  } else {
    // position blending (:532-536, :626); lane = bone
    for (int j = lane; j < J; j += 32) {
      for (int c = 0; c < 3; ++c) {
        O.ik_pos[j][c] = (S.prev_ik_pos[j][c] + O.vel[j][c] * dt) * 0.5 + O.pos[j][c] * 0.5;
        O.blend_pos[j][c] = (S.prev_pos[j][c] + O.vel[j][c] * dt) * 0.5 + O.pos[j][c] * 0.5;
      }
      for (int c = 0; c < 4; ++c) O.ik_rot[j][c] = O.rot[j][c];
    }
  }
  __syncwarp();

  if (init) {
    if (lane < 2) contact_init_dev(S, O, chain_s[lane], chain_n[lane], lane);
  } else if (P.ik_enabled && lane < 2) {
    const int f = lane;
    const int* ch = chain_s[f];
    const int n = chain_n[f];
    const int toe = ch[0], heel = ch[1], knee = ch[2], hip = ch[3];
    // quat.fk_partial (motion/quat.py:241-272) down the toe's ancestor chain on the blended pose: a running transform
    // from the top of the chain to the hip's parent, then the four bones the IK step needs by name
    D3 gp = ld3(O.ik_pos[ch[n - 1]]);
    DQ gr = ld4(O.rot[ch[n - 1]]);
    for (int k = n - 2; k >= 4; --k) {
      const int j = ch[k];
      gp = qrot(gr, ld3(O.ik_pos[j])) + gp;
      gr = qmul(gr, ld4(O.rot[j]));
    }
    const DQ r_rootb = gr;
    const D3 p_hip = qrot(gr, ld3(O.ik_pos[hip])) + gp;
    const DQ r_hip = qmul(gr, ld4(O.rot[hip]));
    const D3 p_knee = qrot(r_hip, ld3(O.ik_pos[knee])) + p_hip;
    const DQ r_knee = qmul(r_hip, ld4(O.rot[knee]));
    const D3 p_heel = qrot(r_knee, ld3(O.ik_pos[heel])) + p_knee;
    const DQ r_heel = qmul(r_knee, ld4(O.rot[heel]));
    const D3 p_toe = qrot(r_heel, ld3(O.ik_pos[toe])) + p_heel;
    ContactState c;
    c.state = S.contact_state[f] != 0; c.lock = S.contact_lock[f] != 0;
    c.position = ld3(S.contact_position[f]); c.velocity = ld3(S.contact_velocity[f]);
    c.point = ld3(S.contact_point[f]); c.target = ld3(S.contact_target[f]);
    c.off_pos = ld3(S.contact_offset_position[f]); c.off_vel = ld3(S.contact_offset_velocity[f]);
    contact_update_dev(c, p_toe, contact_in, P.ik_unlock_radius, P.ik_foot_height, P.ik_blending_halflife, dt);
    c.position.y = fmax(c.position.y, P.ik_foot_height);   // aliases contact_positions[bs] in the reference (:581-582)
    S.contact_state[f] = c.state; S.contact_lock[f] = c.lock;
    st3(S.contact_position[f], c.position); st3(S.contact_velocity[f], c.velocity);
    st3(S.contact_point[f], c.point); st3(S.contact_target[f], c.target);
    st3(S.contact_offset_position[f], c.off_pos); st3(S.contact_offset_velocity[f], c.off_vel);

    const D3 target = c.position + (p_heel - p_toe);
    const D3 fwd = qrot(r_knee, v3<double>(0.0, 1.0, 0.0));
    DQ new_hip, new_knee;
    ik_two_bone_dev(p_hip, p_knee, p_heel, target, fwd, r_hip, r_knee, r_rootb, P.ik_max_length_buffer, new_hip, new_knee);
    st4(O.ik_rot[hip], new_hip);
    st4(O.ik_rot[knee], new_knee);
  }
  __syncwarp();

  // carry state
  if (lane == 0) { st3(S.root_pos, ld3(O.blend_pos[0])); st4(S.root_rot, rootrot); }
  for (int j = lane; j < J; j += 32)
    for (int c = 0; c < 3; ++c) { S.prev_pos[j][c] = O.blend_pos[j][c]; S.prev_ik_pos[j][c] = O.ik_pos[j][c]; }
  __syncwarp();
  double2* Og = reinterpret_cast<double2*>(outs + b);
  for (int i = lane; i < PF_O16; i += 32) Og[i] = reinterpret_cast<const double2*>(&Osh)[i];
  double2* Sw = reinterpret_cast<double2*>(states + b);
  for (int i = lane; i < PF_S16; i += 32) Sw[i] = reinterpret_cast<const double2*>(&Ssh)[i];
}

// ------------------------------------------------------------------------------------------------
// batched stand-alone versions (API completeness + unit parity tests)
// ------------------------------------------------------------------------------------------------
__global__ void contact_update_kernel(int32_t* state, int32_t* lock, double* position, double* velocity,
                                      double* point, double* target, double* off_pos, double* off_vel,
                                      const double* input_position, const int32_t* input_state, long long n,
                                      double unlock_radius, double foot_height, double halflife, double dt) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  ContactState c;
  c.state = state[i] != 0; c.lock = lock[i] != 0;
  c.position = ld3(position + i * 3); c.velocity = ld3(velocity + i * 3); c.point = ld3(point + i * 3);
  c.target = ld3(target + i * 3); c.off_pos = ld3(off_pos + i * 3); c.off_vel = ld3(off_vel + i * 3);
  contact_update_dev(c, ld3(input_position + i * 3), input_state[i] != 0, unlock_radius, foot_height, halflife, dt);
  state[i] = c.state; lock[i] = c.lock;
  st3(position + i * 3, c.position); st3(velocity + i * 3, c.velocity); st3(point + i * 3, c.point);
  st3(target + i * 3, c.target); st3(off_pos + i * 3, c.off_pos); st3(off_vel + i * 3, c.off_vel);
}

__global__ void ik_two_bone_kernel(const double* root, const double* mid, const double* end, const double* target,
                                   const double* fwd, const double* root_gr, const double* mid_gr,
                                   const double* par_gr, double max_length_buffer, long long n, double* out_root_lr,
                                   double* out_mid_lr) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  DQ a, b;
  ik_two_bone_dev(ld3(root + i * 3), ld3(mid + i * 3), ld3(end + i * 3), ld3(target + i * 3), ld3(fwd + i * 3),
                  ld4(root_gr + i * 4), ld4(mid_gr + i * 4), ld4(par_gr + i * 4), max_length_buffer, a, b);
  st4(out_root_lr + i * 4, a);
  st4(out_mid_lr + i * 4, b);
}

// Inertialization.pose_transition (Inertialization.py:136-209): thread per (skeleton, bone)
__global__ void pose_transition_kernel(double* off_pos, double* off_vel, double* off_rot, double* off_ang,
                                       const double* root_pos, const double* root_vel, const double* root_rot,
                                       const double* root_ang, const double* src_pos, const double* src_vel,
                                       const double* src_rot, const double* src_ang, const double* dst_pos,
                                       const double* dst_vel, const double* dst_rot, const double* dst_ang,
                                       long long n, int J, double* tr_src_pos, double* tr_src_rot,
                                       double* tr_dst_pos, double* tr_dst_rot) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * J) return;
  const long long s = i / J;
  const int j = (int)(i - s * J);
  D3 ox = ld3(off_pos + i * 3), ov = ld3(off_vel + i * 3), oa = ld3(off_ang + i * 3);
  DQ orot = ld4(off_rot + i * 4);
  if (j == 0) {
    const DQ t_dst_rot = ld4(root_rot + s * 4);
    const DQ t_src_rot = ld4(dst_rot + i * 4);
    const D3 ws_vel = qrot(t_dst_rot, qrot(t_src_rot, ld3(dst_vel + i * 3)));
    const D3 ws_ang = qrot(t_dst_rot, qrot(t_src_rot, ld3(dst_ang + i * 3)));
    const D3 rp = ld3(root_pos + s * 3);
    // inertialize_transition_pos(off, off_v, root_position, root_velocity, root_position, ws_vel)
    ox = (rp + ox) - rp;
    ov = (ld3(root_vel + s * 3) + ov) - ws_vel;
    // inertialize_transition_rot(off, off_v, root_rotation, root_ang, root_rotation, ws_ang)
    orot = qabs(qmul(qmul(orot, t_dst_rot), qinv(t_dst_rot)));
    oa = (oa + ld3(root_ang + s * 3)) - ws_ang;
    st3(tr_dst_pos + s * 3, rp); st4(tr_dst_rot + s * 4, t_dst_rot);
    st3(tr_src_pos + s * 3, ld3(dst_pos + i * 3)); st4(tr_src_rot + s * 4, t_src_rot);
  } else {
    ox = (ld3(src_pos + i * 3) + ox) - ld3(dst_pos + i * 3);
    ov = (ld3(src_vel + i * 3) + ov) - ld3(dst_vel + i * 3);
    orot = qabs(qmul(qmul(orot, ld4(src_rot + i * 4)), qinv(ld4(dst_rot + i * 4))));
    oa = (oa + ld3(src_ang + i * 3)) - ld3(dst_ang + i * 3);
  }
  st3(off_pos + i * 3, ox); st3(off_vel + i * 3, ov); st4(off_rot + i * 4, orot); st3(off_ang + i * 3, oa);
}

// Inertialization.pose_update (Inertialization.py:217-297): thread per (skeleton, bone)
__global__ void pose_update_kernel(double* pos, double* vel, double* rot, double* ang, double* off_pos,
                                   double* off_vel, double* off_rot, double* off_ang, const double* in_pos,
                                   const double* in_vel, const double* in_rot, const double* in_ang,
                                   const double* tr_src_pos, const double* tr_src_rot, const double* tr_dst_pos,
                                   const double* tr_dst_rot, double halflife, double dt, long long n, int J) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * J) return;
  const long long s = i / J;
  const int j = (int)(i - s * J);
  D3 ix = ld3(in_pos + i * 3), iv = ld3(in_vel + i * 3), ia = ld3(in_ang + i * 3);
  DQ ir = ld4(in_rot + i * 4);
  if (j == 0) {
    const DQ dr = ld4(tr_dst_rot + s * 4), sr = ld4(tr_src_rot + s * 4);
    const D3 dp = ld3(tr_dst_pos + s * 3), sp = ld3(tr_src_pos + s * 3);
    ix = qrot(dr, qrot(qinv(sr), ix - sp)) + dp;
    iv = qrot(dr, qrot(qinv(sr), iv));
    ir = qnormalize(qmul(dr, qmul(qinv(sr), ir)));
    ia = qrot(dr, qrot(qinv(sr), ia));
  }
  D3 ox = ld3(off_pos + i * 3), ov = ld3(off_vel + i * 3), oa = ld3(off_ang + i * 3);
  DQ orot = ld4(off_rot + i * 4);
  decay_spring_pos(ox, ov, halflife, dt);
  decay_spring_rot(orot, oa, halflife, dt);
  st3(pos + i * 3, ix + ox); st3(vel + i * 3, iv + ov);
  st4(rot + i * 4, qmul(orot, ir)); st3(ang + i * 3, oa + ia);
  st3(off_pos + i * 3, ox); st3(off_vel + i * 3, ov); st4(off_rot + i * 4, orot); st3(off_ang + i * 3, oa);
}

int check_parents_arg(const int32_t* d_parents, int J) {
  MOCHA_CHECK_ARG(d_parents && J >= 1 && J <= MAXJ, "skeleton: need 1 <= J <= %d and a parents table", MAXJ);
  return MOCHA_OK;
}

inline unsigned nblk(long long n, int bs) { return (unsigned)((n + bs - 1) / bs); }

}  // namespace

extern "C" int mocha_xy_to_quat(const float* xy, long long n, float* quat, mocha_stream_t stream) {
  MOCHA_CHECK_ARG(xy && quat && n > 0, "mocha_xy_to_quat: bad argument");
  MOCHA_CHECK_ARG((reinterpret_cast<uintptr_t>(quat) & 15) == 0, "mocha_xy_to_quat: output not 16B aligned");
  launch_k(xy_to_quat_kernel, nblk(n, 256), 256, 0, (cudaStream_t)stream, xy, n, quat);
  count_launch();
  MOCHA_LAUNCH_CHECK("xy_to_quat_kernel");
  return MOCHA_OK;
}

extern "C" int mocha_quat_to_xy(const float* quat, long long n, float* xy, mocha_stream_t stream) {
  MOCHA_CHECK_ARG(xy && quat && n > 0, "mocha_quat_to_xy: bad argument");
  MOCHA_CHECK_ARG((reinterpret_cast<uintptr_t>(quat) & 15) == 0, "mocha_quat_to_xy: input not 16B aligned");
  launch_k(quat_to_xy_kernel, nblk(n, 256), 256, 0, (cudaStream_t)stream, quat, n, xy);
  count_launch();
  MOCHA_LAUNCH_CHECK("quat_to_xy_kernel");
  return MOCHA_OK;
}

static unsigned fk_grid(long long F) {
  long long g = (F + FK_WARPS - 1) / FK_WARPS;
  const long long cap = 148LL * 16;
  return (unsigned)(g < cap ? g : cap);
}

// thread-per-skeleton streaming kernel for batches that fill the GPU (>= 4096 skeletons); the warp-per-skeleton kernel keeps
// the small calls (a frame's clips), where parallelism inside the skeleton is all there is.
static bool fk_rows_wanted(long long F, int J, const void* a = nullptr, const void* b = nullptr, const void* c = nullptr,
                           const void* d = nullptr, const void* e = nullptr, const void* f = nullptr, const void* g = nullptr,
                           const void* h = nullptr) {
  const uintptr_t all = reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(c) |
                        reinterpret_cast<uintptr_t>(d) | reinterpret_cast<uintptr_t>(e) | reinterpret_cast<uintptr_t>(f) |
                        reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(h);
  return F >= 4096 && J >= 1 && J <= MAXJ && (all & 15) == 0;   // bulk copies move 16-byte aligned slabs
}
template <bool WITH_VEL, int WARPS>
static int fk_rows_launch(const float* lrot, const float* lpos, const float* lvel, const float* lang, const int32_t* parents,
                          long long F, int J, float* grot, float* gpos, float* gvel, float* gang, cudaStream_t s) {
  const size_t smem = (size_t)WARPS * 32 * (J * 4 + J * 3 * (WITH_VEL ? 3 : 1)) * sizeof(float);
  static size_t configured = 0;
  if (smem > configured) {
    MOCHA_CUDA(cudaFuncSetAttribute(fk_rows_kernel<WITH_VEL, WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  static int sms = 0;
  if (!sms) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev); if (sms <= 0) sms = 148; }
  const long long blocks = ((F + 31) / 32 + WARPS - 1) / WARPS;
  const long long resident = (long long)sms * (long long)max(1, (int)((220 * 1024) / (smem + 1024)));
  launch_k(fk_rows_kernel<WITH_VEL, WARPS>, (unsigned)min(blocks, resident), WARPS * 32, smem, s, lrot, lpos, lvel, lang, parents, F, J,
           grot, gpos, gvel, gang);
  return MOCHA_OK;
}

extern "C" int mocha_fk(const float* lrot, const float* lpos, const int32_t* parents, long long F, int J, float* grot,
                        float* gpos, mocha_stream_t stream) {
  MOCHA_CHECK_ARG(lrot && lpos && grot && gpos && F > 0, "mocha_fk: bad argument");
  MOCHA_TRY(check_parents_arg(parents, J));
  if (fk_rows_wanted(F, J, lrot, lpos, grot, gpos)) {
    MOCHA_TRY((fk_rows_launch<false, 8>(lrot, lpos, nullptr, nullptr, parents, F, J, grot, gpos, nullptr, nullptr, (cudaStream_t)stream)));
  } else {
    launch_k(fk_kernel<false, float>, fk_grid(F), FK_WARPS * 32, 0, (cudaStream_t)stream, lrot, lpos, nullptr, nullptr, parents, F, J,
                                                                            grot, gpos, nullptr, nullptr);
  }
  count_launch();
  MOCHA_LAUNCH_CHECK("fk_kernel");
  return MOCHA_OK;
}

extern "C" int mocha_fk_vel(const float* lrot, const float* lpos, const float* lvel, const float* lang,
                            const int32_t* parents, long long F, int J, float* grot, float* gpos, float* gvel,
                            float* gang, mocha_stream_t stream) {
  MOCHA_CHECK_ARG(lrot && lpos && lvel && lang && grot && gpos && gvel && gang && F > 0, "mocha_fk_vel: bad argument");
  MOCHA_TRY(check_parents_arg(parents, J));
  if (fk_rows_wanted(F, J, lrot, lpos, lvel, lang, grot, gpos, gvel, gang)) {
    MOCHA_TRY((fk_rows_launch<true, 5>(lrot, lpos, lvel, lang, parents, F, J, grot, gpos, gvel, gang, (cudaStream_t)stream)));
  } else {
    launch_k(fk_kernel<true, float>, fk_grid(F), FK_WARPS * 32, 0, (cudaStream_t)stream, lrot, lpos, lvel, lang, parents, F, J, grot,
                                                                           gpos, gvel, gang);
  }
  count_launch();
  MOCHA_LAUNCH_CHECK("fk_vel_kernel");
  return MOCHA_OK;
}

extern "C" int mocha_ik(const float* grot, const float* gpos, const int32_t* parents, long long F, int J, float* lrot,
                        float* lpos, mocha_stream_t stream) {
  MOCHA_CHECK_ARG(lrot && lpos && grot && gpos && F > 0, "mocha_ik: bad argument");
  MOCHA_TRY(check_parents_arg(parents, J));
  launch_k(ik_kernel<float>, fk_grid(F), FK_WARPS * 32, 0, (cudaStream_t)stream, grot, gpos, parents, F, J, lrot, lpos);
  count_launch();
  MOCHA_LAUNCH_CHECK("ik_kernel");
  return MOCHA_OK;
}

namespace {
int post_frame_launch(const mocha_post_params* params, const float* Y, const float* src_hips_vel, const float* src_rvel,
                      const float* src_rang, int hv_stride, int rv_stride, const uint8_t* contacts, int B, int T, int V,
                      int Cin, int init, const uint8_t* start, mocha_clip_state* state, mocha_frame_out* out,
                      mocha_stream_t stream) {
  MOCHA_CHECK_ARG(params && Y && src_hips_vel && src_rvel && src_rang && contacts && state && out && B > 0,
                  "mocha_post_frame: null/empty argument");
  MOCHA_CHECK_ARG(params->J == V + 1 && params->J <= 25, "mocha_post_frame: J=%d must equal V+1=%d and be <= 25",
                  params->J, V + 1);
  MOCHA_CHECK_ARG(Cin == 15 && T > 0, "mocha_post_frame: pose feature layout needs Cin=15");
  MOCHA_CHECK_ARG(params->parents[0] == -1, "mocha_post_frame: parents[0] must be -1");
  for (int j = 1; j < params->J; ++j)
    MOCHA_CHECK_ARG(params->parents[j] >= 0 && params->parents[j] < j, "mocha_post_frame: parents[%d] out of order", j);
  for (int f = 0; f < 2; ++f) {
    int depth = 0;
    for (int j = params->contact_bones[f]; j > 0 && j < params->J; j = params->parents[j]) ++depth;
    MOCHA_CHECK_ARG(params->contact_bones[f] > 0 && params->contact_bones[f] < params->J && depth >= 4,
                    "mocha_post_frame: contact bone %d needs 4 ancestors", params->contact_bones[f]);
  }
  // steady state: the latency-shaped kernel (shared-memory structs, one load round); frame 0 and unaligned struct arrays
  // take the general kernel. A per-clip start row (start != NULL) takes the masked step kernel under the same rule.
  const bool aligned = ((reinterpret_cast<uintptr_t>(state) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
  const bool step_kernel = aligned && V * Cin <= PF_YMAX;
  if (start && step_kernel)
    launch_k(post_frame_step_kernel<true>, B, 32, 0, (cudaStream_t)stream, *params, Y, src_hips_vel, src_rvel, src_rang, contacts,
             start, T, V, Cin, state, out, hv_stride, rv_stride);
  else if (!start && !init && step_kernel)
    launch_k(post_frame_step_kernel<false>, B, 32, 0, (cudaStream_t)stream, *params, Y, src_hips_vel, src_rvel, src_rang, contacts,
             nullptr, T, V, Cin, state, out, hv_stride, rv_stride);
  else
    launch_k(post_frame_kernel, nblk((long long)B * 32, 128), 128, 0, (cudaStream_t)stream, *params, Y, src_hips_vel, src_rvel, src_rang,
                                                                   contacts, B, T, V, Cin, init, start, state, out, hv_stride, rv_stride);
  count_launch();
  MOCHA_LAUNCH_CHECK("post_frame_kernel");
  return MOCHA_OK;
}
}  // namespace

extern "C" int mocha_post_frame(const mocha_post_params* params, const float* Y, const float* src_hips_vel,
                                const float* src_rvel, const float* src_rang, const uint8_t* contacts, int B, int T,
                                int V, int Cin, int init, mocha_clip_state* state, mocha_frame_out* out,
                                mocha_stream_t stream) {
  return post_frame_launch(params, Y, src_hips_vel, src_rvel, src_rang, T * 3, 3, contacts, B, T, V, Cin, init, nullptr, state,
                           out, stream);
}

// Same with the three per-clip source-motion inputs packed in ONE row per clip, [hips vel T*3 | rvel 3 | rang 3]
// (what a streaming caller uploads with a single H2D copy): no slicing copies in front of the kernel.
extern "C" int mocha_post_frame_packed(const mocha_post_params* params, const float* Y, const float* side, int side_stride,
                                       const uint8_t* contacts, int B, int T, int V, int Cin, int init,
                                       mocha_clip_state* state, mocha_frame_out* out, mocha_stream_t stream) {
  MOCHA_CHECK_ARG(side && side_stride >= T * 3 + 6, "mocha_post_frame_packed: side rows need T*3+6 floats");
  return post_frame_launch(params, Y, side, side + T * 3, side + T * 3 + 3, side_stride, side_stride, contacts, B, T, V,
                           Cin, init, nullptr, state, out, stream);
}

// Per-clip frame 0 (clip admission): clip b runs the init frame iff d_start[b] != 0, every other clip a steady-state step,
// in one launch that a captured graph can replay with a different start row every frame.
extern "C" int mocha_post_frame_packed_masked(const mocha_post_params* params, const float* Y, const float* side,
                                              int side_stride, const uint8_t* contacts, const uint8_t* start, int B, int T,
                                              int V, int Cin, mocha_clip_state* state, mocha_frame_out* out,
                                              mocha_stream_t stream) {
  MOCHA_CHECK_ARG(start, "mocha_post_frame_packed_masked: null start row");
  MOCHA_CHECK_ARG(side && side_stride >= T * 3 + 6, "mocha_post_frame_packed_masked: side rows need T*3+6 floats");
  return post_frame_launch(params, Y, side, side + T * 3, side + T * 3 + 3, side_stride, side_stride, contacts, B, T, V,
                           Cin, 0, start, state, out, stream);
}

extern "C" int mocha_contact_update(int32_t* state, int32_t* lock, double* position, double* velocity, double* point,
                                    double* target, double* off_pos, double* off_vel, const double* input_position,
                                    const int32_t* input_state, long long n, double unlock_radius, double foot_height,
                                    double halflife, double dt, mocha_stream_t stream) {
  MOCHA_CHECK_ARG(state && lock && position && velocity && point && target && off_pos && off_vel && input_position &&
                      input_state && n > 0,
                  "mocha_contact_update: null/empty argument");
  launch_k(contact_update_kernel, nblk(n, 128), 128, 0, (cudaStream_t)stream, state, lock, position, velocity, point, target,
                                                                       off_pos, off_vel, input_position, input_state,
                                                                       n, unlock_radius, foot_height, halflife, dt);
  count_launch();
  MOCHA_LAUNCH_CHECK("contact_update_kernel");
  return MOCHA_OK;
}

// float64 variants of the three batch operators: the reference driver's final FK (test_fullframework.py:672-694)
// runs on float64 arrays, and a drop-in must not narrow them
extern "C" int mocha_fk_f64(const double* lrot, const double* lpos, const int32_t* parents, long long F, int J, double* grot,
                            double* gpos, mocha_stream_t stream) {
  MOCHA_CHECK_ARG(lrot && lpos && grot && gpos && F > 0, "mocha_fk_f64: bad argument");
  MOCHA_TRY(check_parents_arg(parents, J));
  launch_k(fk_kernel<false, double>, fk_grid(F), FK_WARPS * 32, 0, (cudaStream_t)stream, lrot, lpos, nullptr, nullptr, parents, F, J,
                                                                                  grot, gpos, nullptr, nullptr);
  count_launch();
  MOCHA_LAUNCH_CHECK("fk_kernel<double>");
  return MOCHA_OK;
}

extern "C" int mocha_fk_vel_f64(const double* lrot, const double* lpos, const double* lvel, const double* lang,
                                const int32_t* parents, long long F, int J, double* grot, double* gpos, double* gvel,
                                double* gang, mocha_stream_t stream) {
  MOCHA_CHECK_ARG(lrot && lpos && lvel && lang && grot && gpos && gvel && gang && F > 0, "mocha_fk_vel_f64: bad argument");
  MOCHA_TRY(check_parents_arg(parents, J));
  launch_k(fk_kernel<true, double>, fk_grid(F), FK_WARPS * 32, 0, (cudaStream_t)stream, lrot, lpos, lvel, lang, parents, F, J, grot,
                                                                                 gpos, gvel, gang);
  count_launch();
  MOCHA_LAUNCH_CHECK("fk_vel_kernel<double>");
  return MOCHA_OK;
}

extern "C" int mocha_ik_f64(const double* grot, const double* gpos, const int32_t* parents, long long F, int J, double* lrot,
                            double* lpos, mocha_stream_t stream) {
  MOCHA_CHECK_ARG(lrot && lpos && grot && gpos && F > 0, "mocha_ik_f64: bad argument");
  MOCHA_TRY(check_parents_arg(parents, J));
  launch_k(ik_kernel<double>, fk_grid(F), FK_WARPS * 32, 0, (cudaStream_t)stream, grot, gpos, parents, F, J, lrot, lpos);
  count_launch();
  MOCHA_LAUNCH_CHECK("ik_kernel<double>");
  return MOCHA_OK;
}

extern "C" int mocha_ik_two_bone(const double* root_lr, const double* mid_lr, const double* root, const double* mid,
                                 const double* end, const double* target, const double* fwd, const double* root_gr,
                                 const double* mid_gr, const double* par_gr, double max_length_buffer, long long n,
                                 double* out_root_lr, double* out_mid_lr, mocha_stream_t stream) {
  (void)root_lr; (void)mid_lr;  // inputs the reference accepts but overwrites (motion/quat.py:340-341)
  MOCHA_CHECK_ARG(root && mid && end && target && fwd && root_gr && mid_gr && par_gr && out_root_lr && out_mid_lr && n > 0,
                  "mocha_ik_two_bone: null/empty argument");
  launch_k(ik_two_bone_kernel, nblk(n, 128), 128, 0, (cudaStream_t)stream, root, mid, end, target, fwd, root_gr, mid_gr,
                                                                    par_gr, max_length_buffer, n, out_root_lr,
                                                                    out_mid_lr);
  count_launch();
  MOCHA_LAUNCH_CHECK("ik_two_bone_kernel");
  return MOCHA_OK;
}

extern "C" int mocha_pose_transition(double* off_pos, double* off_vel, double* off_rot, double* off_ang,
                                     const double* root_pos, const double* root_vel, const double* root_rot,
                                     const double* root_ang, const double* src_pos, const double* src_vel,
                                     const double* src_rot, const double* src_ang, const double* dst_pos,
                                     const double* dst_vel, const double* dst_rot, const double* dst_ang, long long n,
                                     int J, double* tr_src_pos, double* tr_src_rot, double* tr_dst_pos,
                                     double* tr_dst_rot, mocha_stream_t stream) {
  MOCHA_CHECK_ARG(off_pos && off_vel && off_rot && off_ang && root_pos && root_vel && root_rot && root_ang && src_pos &&
                      src_vel && src_rot && src_ang && dst_pos && dst_vel && dst_rot && dst_ang && tr_src_pos &&
                      tr_src_rot && tr_dst_pos && tr_dst_rot && n > 0 && J > 0,
                  "mocha_pose_transition: null/empty argument");
  launch_k(pose_transition_kernel, nblk(n * J, 128), 128, 0, (cudaStream_t)stream, off_pos, off_vel, off_rot, off_ang, root_pos, root_vel, root_rot, root_ang, src_pos, src_vel, src_rot, src_ang,
      dst_pos, dst_vel, dst_rot, dst_ang, n, J, tr_src_pos, tr_src_rot, tr_dst_pos, tr_dst_rot);
  count_launch();
  MOCHA_LAUNCH_CHECK("pose_transition_kernel");
  return MOCHA_OK;
}

extern "C" int mocha_pose_update(double* pos, double* vel, double* rot, double* ang, double* off_pos, double* off_vel,
                                 double* off_rot, double* off_ang, const double* in_pos, const double* in_vel,
                                 const double* in_rot, const double* in_ang, const double* tr_src_pos,
                                 const double* tr_src_rot, const double* tr_dst_pos, const double* tr_dst_rot,
                                 double halflife, double dt, long long n, int J, mocha_stream_t stream) {
  MOCHA_CHECK_ARG(pos && vel && rot && ang && off_pos && off_vel && off_rot && off_ang && in_pos && in_vel && in_rot &&
                      in_ang && tr_src_pos && tr_src_rot && tr_dst_pos && tr_dst_rot && n > 0 && J > 0,
                  "mocha_pose_update: null/empty argument");
  launch_k(pose_update_kernel, nblk(n * J, 128), 128, 0, (cudaStream_t)stream, pos, vel, rot, ang, off_pos, off_vel, off_rot,
                                                                        off_ang, in_pos, in_vel, in_rot, in_ang,
                                                                        tr_src_pos, tr_src_rot, tr_dst_pos, tr_dst_rot,
                                                                        halflife, dt, n, J);
  count_launch();
  MOCHA_LAUNCH_CHECK("pose_update_kernel");
  return MOCHA_OK;
}

// ------------------------------------------------------------------------------------------------
// Element-wise quaternion algebra of motion/quat.py in the CALLER'S precision (float32 or float64): the
// reference driver's per-frame loop works on float64 NumPy arrays (test_fullframework.py:321-353, :476-509),
// so the drop-in `quat` module must not round its operands to float32. One thread per item; operands are dense
// [n, width] arrays (the host expands broadcasts). Widths per op: see quat_op_widths().
// ------------------------------------------------------------------------------------------------
namespace {

enum QuatOp {
  QOP_MUL = 0,          // quat.mul            (quat.py:112-120)  a[4] b[4] -> [4]
  QOP_INV_MUL = 1,      // quat.inv_mul        (:122-123)
  QOP_MUL_INV = 2,      // quat.mul_inv        (:125-126)
  QOP_MUL_VEC = 3,      // quat.mul_vec        (:128-130)         a[4] b[3] -> [3]
  QOP_INV_MUL_VEC = 4,  // quat.inv_mul_vec    (:132-133)
  QOP_INV = 5,          // quat.inv            (:109-110)         a[4] -> [4]
  QOP_ABS = 6,          // quat.abs            (:18-19)
  QOP_NORMALIZE4 = 7,   // quat.normalize on quaternions (:15-16); eps in `param`
  QOP_NORMALIZE3 = 8,   // quat.normalize on 3-vectors
  QOP_EXP = 9,          // quat.exp            (:154-158)         a[3] -> [4]; eps in `param`
  QOP_LOG = 10,         // quat.log            (:149-152)         a[4] -> [3]; eps in `param`
  QOP_BETWEEN = 11,     // quat.between        (:143-147)         a[3] b[3] -> [4]
  QOP_ANGLE_AXIS = 12,  // quat.from_angle_axis(:21-25)           a[1] b[3] -> [4]
  QOP_TO_XFORM = 13,    // quat.to_xform       (:27-40)           a[4] -> [9]
  QOP_FROM_XFORM = 14,  // quat.from_xform     (:69-94)           a[9] -> [4]
  QOP_TO_EULER_XYZ = 15,// quat.to_euler       (:346-358)         a[4] -> [3]
  QOP_TO_EULER_YZX = 16,
  QOP_CROSS = 17,       // quat._fast_cross    (:3-7)             a[3] b[3] -> [3]
  QOP_TO_XFORM_XY = 18, // quat.to_xform_xy    (:42-55)           a[4] -> [6]
  QOP_FROM_XFORM_XY = 19,// quat.from_xform_xy (:96-107)          a[6] -> [4]
  QOP_LENGTH3 = 20,     // quat.length         (:12-13)           a[3] -> [1]
  QOP_LENGTH4 = 21,     //                                        a[4] -> [1]
  QOP_COUNT = 22
};

struct QuatOpWidths { int a, b, o; };
__host__ __device__ inline QuatOpWidths quat_op_widths(int op) {
  switch (op) {
    case QOP_MUL: case QOP_INV_MUL: case QOP_MUL_INV: return {4, 4, 4};
    case QOP_MUL_VEC: case QOP_INV_MUL_VEC: return {4, 3, 3};
    case QOP_INV: case QOP_ABS: case QOP_NORMALIZE4: return {4, 0, 4};
    case QOP_NORMALIZE3: return {3, 0, 3};
    case QOP_EXP: return {3, 0, 4};
    case QOP_LOG: return {4, 0, 3};
    case QOP_BETWEEN: return {3, 3, 4};
    case QOP_ANGLE_AXIS: return {1, 3, 4};
    case QOP_TO_XFORM: return {4, 0, 9};
    case QOP_FROM_XFORM: return {9, 0, 4};
    case QOP_TO_EULER_XYZ: case QOP_TO_EULER_YZX: return {4, 0, 3};
    case QOP_CROSS: return {3, 3, 3};
    case QOP_TO_XFORM_XY: return {4, 0, 6};
    case QOP_FROM_XFORM_XY: return {6, 0, 4};
    case QOP_LENGTH3: return {3, 0, 1};
    case QOP_LENGTH4: return {4, 0, 1};
    default: return {0, 0, 0};
  }
}

template <typename T> __device__ __forceinline__ T clamp1(T x) { return x < (T)-1 ? (T)-1 : x > (T)1 ? (T)1 : x; }

// quat.to_euler(order='xyz') (quat.py:346-358), radians; shared by quat_op_kernel and clip_payload_kernel
template <typename T> __device__ __forceinline__ void to_euler_xyz(T q0, T q1, T q2, T q3, T* po) {
  po[0] = atan2((T)2 * (q0 * q1 + q2 * q3), (T)1 - (T)2 * (q1 * q1 + q2 * q2));
  po[1] = asin(clamp1((T)2 * (q0 * q2 - q3 * q1)));
  po[2] = atan2((T)2 * (q0 * q3 + q1 * q2), (T)1 - (T)2 * (q2 * q2 + q3 * q3));
}

template <typename T>
__global__ void quat_op_kernel(int op, const T* __restrict__ a, const T* __restrict__ b, long long n, T param,
                               T* __restrict__ out) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const QuatOpWidths w = quat_op_widths(op);
  const T* pa = a + i * w.a;
  const T* pb = b ? b + i * w.b : nullptr;
  T* po = out + i * w.o;
  switch (op) {
    case QOP_MUL: case QOP_INV_MUL: case QOP_MUL_INV: {
      Q4<T> x = q4<T>(pa[0], pa[1], pa[2], pa[3]), y = q4<T>(pb[0], pb[1], pb[2], pb[3]);
      if (op == QOP_INV_MUL) x = qinv(x);
      if (op == QOP_MUL_INV) y = qinv(y);
      const Q4<T> r = qmul(x, y);
      po[0] = r.w; po[1] = r.x; po[2] = r.y; po[3] = r.z;
      break;
    }
    case QOP_MUL_VEC: case QOP_INV_MUL_VEC: {
      const V3<T> r = q_mul_vec(pa, pb, op == QOP_INV_MUL_VEC);
      po[0] = r.x; po[1] = r.y; po[2] = r.z;
      break;
    }
    case QOP_INV: po[0] = pa[0]; po[1] = -pa[1]; po[2] = -pa[2]; po[3] = -pa[3]; break;
    case QOP_ABS: {
      const T s = pa[0] > (T)0 ? (T)1 : (T)-1;
      po[0] = s * pa[0]; po[1] = s * pa[1]; po[2] = s * pa[2]; po[3] = s * pa[3];
      break;
    }
    case QOP_NORMALIZE4: {
      const T d = sqrt(pa[0] * pa[0] + pa[1] * pa[1] + pa[2] * pa[2] + pa[3] * pa[3]) + param;
      po[0] = pa[0] / d; po[1] = pa[1] / d; po[2] = pa[2] / d; po[3] = pa[3] / d;
      break;
    }
    case QOP_NORMALIZE3: {
      const T d = sqrt(pa[0] * pa[0] + pa[1] * pa[1] + pa[2] * pa[2]) + param;
      po[0] = pa[0] / d; po[1] = pa[1] / d; po[2] = pa[2] / d;
      break;
    }
    case QOP_EXP: {
      const T h = sqrt(pa[0] * pa[0] + pa[1] * pa[1] + pa[2] * pa[2]);
      const T c = h < param ? (T)1 : cos(h);
      const T s = h < param ? (T)1 : sin(h) / h;
      po[0] = c; po[1] = s * pa[0]; po[2] = s * pa[1]; po[3] = s * pa[2];
      break;
    }
    case QOP_LOG: {
      const T len = sqrt(pa[1] * pa[1] + pa[2] * pa[2] + pa[3] * pa[3]);
      const T ha = len < param ? (T)1 : atan2(len, pa[0]) / len;
      po[0] = ha * pa[1]; po[1] = ha * pa[2]; po[2] = ha * pa[3];
      break;
    }
    case QOP_BETWEEN: {
      const V3<T> x = v3<T>(pa[0], pa[1], pa[2]), y = v3<T>(pb[0], pb[1], pb[2]);
      const V3<T> c = cross(x, y);
      po[0] = sqrt(dot(x, x) * dot(y, y)) + dot(x, y); po[1] = c.x; po[2] = c.y; po[3] = c.z;
      break;
    }
    case QOP_ANGLE_AXIS: {
      const Q4<T> r = q_angle_axis(pa[0], v3<T>(pb[0], pb[1], pb[2]));
      po[0] = r.w; po[1] = r.x; po[2] = r.y; po[3] = r.z;
      break;
    }
    case QOP_TO_XFORM: case QOP_TO_XFORM_XY: {
      const T qw = pa[0], qx = pa[1], qy = pa[2], qz = pa[3];
      const T x2 = qx + qx, y2 = qy + qy, z2 = qz + qz;
      const T xx = qx * x2, yy = qy * y2, wx = qw * x2;
      const T xy = qx * y2, yz = qy * z2, wy = qw * y2;
      const T xz = qx * z2, zz = qz * z2, wz = qw * z2;
      if (op == QOP_TO_XFORM) {
        po[0] = (T)1 - (yy + zz); po[1] = xy - wz; po[2] = xz + wy;
        po[3] = xy + wz; po[4] = (T)1 - (xx + zz); po[5] = yz - wx;
        po[6] = xz - wy; po[7] = yz + wx; po[8] = (T)1 - (xx + yy);
      } else {
        po[0] = (T)1 - (yy + zz); po[1] = xy - wz;
        po[2] = xy + wz; po[3] = (T)1 - (xx + zz);
        po[4] = xz - wy; po[5] = yz + wx;
      }
      break;
    }
    case QOP_FROM_XFORM: {
      const T m[3][3] = {{pa[0], pa[1], pa[2]}, {pa[3], pa[4], pa[5]}, {pa[6], pa[7], pa[8]}};
      const Q4<T> r = q_from_xform(m);
      po[0] = r.w; po[1] = r.x; po[2] = r.y; po[3] = r.z;
      break;
    }
    case QOP_FROM_XFORM_XY: {
      const Q4<T> r = q_from_xy(v3<T>(pa[0], pa[2], pa[4]), v3<T>(pa[1], pa[3], pa[5]));
      po[0] = r.w; po[1] = r.x; po[2] = r.y; po[3] = r.z;
      break;
    }
    case QOP_TO_EULER_XYZ: to_euler_xyz(pa[0], pa[1], pa[2], pa[3], po); break;
    case QOP_TO_EULER_YZX: {
      const T q0 = pa[0], q1 = pa[1], q2 = pa[2], q3 = pa[3];
      po[0] = atan2((T)2 * (q1 * q0 - q2 * q3), -q1 * q1 + q2 * q2 - q3 * q3 + q0 * q0);
      po[1] = atan2((T)2 * (q2 * q0 - q1 * q3), q1 * q1 - q2 * q2 - q3 * q3 + q0 * q0);
      po[2] = asin(clamp1((T)2 * (q1 * q2 + q3 * q0)));
      break;
    }
    case QOP_CROSS: {
      const V3<T> c = cross(v3<T>(pa[0], pa[1], pa[2]), v3<T>(pb[0], pb[1], pb[2]));
      po[0] = c.x; po[1] = c.y; po[2] = c.z;
      break;
    }
    case QOP_LENGTH3: po[0] = sqrt(pa[0] * pa[0] + pa[1] * pa[1] + pa[2] * pa[2]); break;
    case QOP_LENGTH4: po[0] = sqrt(pa[0] * pa[0] + pa[1] * pa[1] + pa[2] * pa[2] + pa[3] * pa[3]); break;
    default: break;
  }
}

// quat.fk_partial's chain walk (quat.py:241-272): n independent chains of m bones, bone c's parent is bone c-1 of
// the chain; chain element 0 hangs off (start_pos, start_rot) when has_start != 0, else it is a root bone whose
// global transform equals its local one. Sequential per chain (m <= 32), one thread per chain.
template <typename T>
__global__ void fk_chain_kernel(const T* __restrict__ start_pos, const T* __restrict__ start_rot, int has_start,
                                const T* __restrict__ lpos, const T* __restrict__ lrot, long long n, int m,
                                T* __restrict__ gpos, T* __restrict__ grot) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  V3<T> pp = v3<T>((T)0, (T)0, (T)0);
  Q4<T> pr = q4<T>((T)1, (T)0, (T)0, (T)0);
  if (has_start) {
    pp = v3<T>(start_pos[i * 3], start_pos[i * 3 + 1], start_pos[i * 3 + 2]);
    pr = q4<T>(start_rot[i * 4], start_rot[i * 4 + 1], start_rot[i * 4 + 2], start_rot[i * 4 + 3]);
  }
  for (int c = 0; c < m; ++c) {
    const T* lp = lpos + (i * m + c) * 3;
    const T* lr = lrot + (i * m + c) * 4;
    V3<T> gp = v3<T>(lp[0], lp[1], lp[2]);
    Q4<T> gr = q4<T>(lr[0], lr[1], lr[2], lr[3]);
    if (has_start || c > 0) {
      gp = qrot(pr, gp) + pp;
      gr = qmul(pr, gr);
    }
    T* op = gpos + (i * m + c) * 3;
    T* orr = grot + (i * m + c) * 4;
    op[0] = gp.x; op[1] = gp.y; op[2] = gp.z;
    orr[0] = gr.w; orr[1] = gr.x; orr[2] = gr.y; orr[3] = gr.z;
    pp = gp; pr = gr;
  }
}

}  // namespace

extern "C" int mocha_quat_op(int op, int is_f64, const void* a, const void* b, long long n, double param, void* out,
                             mocha_stream_t stream) {
  MOCHA_CHECK_ARG(op >= 0 && op < QOP_COUNT, "mocha_quat_op: unknown op %d", op);
  const QuatOpWidths w = quat_op_widths(op);
  MOCHA_CHECK_ARG(a && out && n > 0 && (w.b == 0 || b), "mocha_quat_op: null/empty argument");
  const unsigned grid = (unsigned)((n + 127) / 128);
  if (is_f64)
    launch_k(quat_op_kernel<double>, grid, 128, 0, (cudaStream_t)stream, op, (const double*)a, (const double*)b, n, param, (double*)out);
  else
    launch_k(quat_op_kernel<float>, grid, 128, 0, (cudaStream_t)stream, op, (const float*)a, (const float*)b, n, (float)param, (float*)out);
  count_launch();
  MOCHA_LAUNCH_CHECK("quat_op_kernel");
  return MOCHA_OK;
}

extern "C" int mocha_fk_chain(int is_f64, const void* start_pos, const void* start_rot, const void* lpos, const void* lrot,
                              long long n, int m, void* gpos, void* grot, mocha_stream_t stream) {
  MOCHA_CHECK_ARG(lpos && lrot && gpos && grot && n > 0 && m >= 1 && m <= 64, "mocha_fk_chain: bad argument");
  MOCHA_CHECK_ARG((start_pos == nullptr) == (start_rot == nullptr), "mocha_fk_chain: start transform needs both parts");
  const unsigned grid = (unsigned)((n + 63) / 64);
  const int hs = start_pos != nullptr;
  if (is_f64)
    launch_k(fk_chain_kernel<double>, grid, 64, 0, (cudaStream_t)stream, (const double*)start_pos, (const double*)start_rot, hs,
                                                                    (const double*)lpos, (const double*)lrot, n, m,
                                                                    (double*)gpos, (double*)grot);
  else
    launch_k(fk_chain_kernel<float>, grid, 64, 0, (cudaStream_t)stream, (const float*)start_pos, (const float*)start_rot, hs,
                                                                   (const float*)lpos, (const float*)lrot, n, m, (float*)gpos,
                                                                   (float*)grot);
  count_launch();
  MOCHA_LAUNCH_CHECK("fk_chain_kernel");
  return MOCHA_OK;
}

// ------------------------------------------------------------------------------------------------
// Window feature extraction (SURVEY §8f row 2): the re-rooting block of the driver's set-up,
// test_fullframework.py:148-158 + :180-186. Input: global transforms / velocities of every frame of every window
// (quat.fk_vel, :146). Every window is expressed relative to the simulation root of its LAST frame:
//   root := G[w, T-1, 0];  G[w, t, 0] := root for all t (:148-151)
//   Xpos = R0^-1 (Gpos - P0), Xrot = R0^-1 Grot, Xtxy = first two columns of Xrot's matrix, Xvel = R0^-1 Gvel,
//   Xang = R0^-1 Gang;  X = (concat(Xpos, Xtxy, Xvel, Xang)[joints 1..] - X_mean[1..]) / X_std[1..]
// One thread per (window, frame, joint); writes the normalised 15-channel rows the embedding reads and the re-rooted
// rotations / positions the following quat.ik (:160) needs.
// ------------------------------------------------------------------------------------------------
namespace {
// per-joint body of the re-rooting, shared with source_windows_kernel: a joint's global transform relative to the root
// (r0i = inverse root rotation, p0 = root position)
__device__ __forceinline__ void reroot_joint(Q4<float> r0i, V3<float> p0, Q4<float> gr, V3<float> gp, V3<float> gv,
                                             V3<float> ga, V3<float>& xp, Q4<float>& xr, V3<float>& xv, V3<float>& xa) {
  xp = qrot(r0i, gp - p0);
  xr = qmul(r0i, gr);
  xv = qrot(r0i, gv);
  xa = qrot(r0i, ga);
}
// the 15 channels of a joint row: position, first two columns of the rotation matrix (6-D encoding), velocity, angular
// velocity
__device__ __forceinline__ void feature_row(V3<float> xp, Q4<float> xr, V3<float> xv, V3<float> xa, float (&f)[15]) {
  const float qw = xr.w, qx = xr.x, qy = xr.y, qz = xr.z;
  const float x2 = qx + qx, y2 = qy + qy, z2 = qz + qz;
  const float xx = qx * x2, yy = qy * y2, wx = qw * x2;
  const float xy = qx * y2, yz = qy * z2, wy = qw * y2;
  const float xz = qx * z2, zz = qz * z2, wz = qw * z2;
  f[0] = xp.x; f[1] = xp.y; f[2] = xp.z;
  f[3] = 1.0f - (yy + zz); f[4] = xy - wz; f[5] = xy + wz; f[6] = 1.0f - (xx + zz); f[7] = xz - wy; f[8] = yz + wx;
  f[9] = xv.x; f[10] = xv.y; f[11] = xv.z; f[12] = xa.x; f[13] = xa.y; f[14] = xa.z;
}
__device__ __forceinline__ void store_normalised_row(float* __restrict__ o, const float (&f)[15], const float* __restrict__ mu,
                                                     const float* __restrict__ sd) {
#pragma unroll
  for (int c = 0; c < 15; ++c) o[c] = (f[c] - mu[c]) / sd[c];
}

__global__ void __launch_bounds__(256)
window_reroot_kernel(const float* __restrict__ grot, const float* __restrict__ gpos, const float* __restrict__ gvel,
                     const float* __restrict__ gang, long long W, int T, int J, const float* __restrict__ X_mean,
                     const float* __restrict__ X_std, float* __restrict__ X, float* __restrict__ xrot, float* __restrict__ xpos,
                     int per_frame_root) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = W * T * J;
  if (i >= total) return;
  const int j = (int)(i % J);
  const long long wt = i / J;
  const long long w = wt / T;
  // joint 0 of the window's last frame, or (training twin convert_YtilToX, trainer.py:356-362) of the frame itself
  const long long rootf = per_frame_root ? wt * J : (w * T + (T - 1)) * J;
  const Q4<float> r0 = q4<float>(grot[rootf * 4], grot[rootf * 4 + 1], grot[rootf * 4 + 2], grot[rootf * 4 + 3]);
  const Q4<float> r0i = qinv(r0);
  const V3<float> p0 = v3<float>(gpos[rootf * 3], gpos[rootf * 3 + 1], gpos[rootf * 3 + 2]);
  const long long src = j == 0 ? rootf : i;               // the root row of every frame is the last frame's root
  const Q4<float> gr = q4<float>(grot[src * 4], grot[src * 4 + 1], grot[src * 4 + 2], grot[src * 4 + 3]);
  const V3<float> gp = v3<float>(gpos[src * 3], gpos[src * 3 + 1], gpos[src * 3 + 2]);
  const V3<float> gv = v3<float>(gvel[src * 3], gvel[src * 3 + 1], gvel[src * 3 + 2]);
  const V3<float> ga = v3<float>(gang[src * 3], gang[src * 3 + 1], gang[src * 3 + 2]);
  V3<float> xp, xv, xa;
  Q4<float> xr;
  reroot_joint(r0i, p0, gr, gp, gv, ga, xp, xr, xv, xa);
  if (xrot) { xrot[i * 4] = xr.w; xrot[i * 4 + 1] = xr.x; xrot[i * 4 + 2] = xr.y; xrot[i * 4 + 3] = xr.z; }
  if (xpos) { xpos[i * 3] = xp.x; xpos[i * 3 + 1] = xp.y; xpos[i * 3 + 2] = xp.z; }
  if (j == 0 && !per_frame_root) return;                  // X drops the simulation root (:186)
  float f[15];
  feature_row(xp, xr, xv, xa, f);
  if (per_frame_root) {                                   // all J joints, not normalised (trainer.py:364-372)
    float* o = X + i * 15;
#pragma unroll
    for (int c = 0; c < 15; ++c) o[c] = f[c];
    return;
  }
  store_normalised_row(X + (wt * (J - 1) + (j - 1)) * 15, f, X_mean + j * 15, X_std + j * 15);
}

// ------------------------------------------------------------------------------------------------
// Source windows (DESIGN §5b): every slot's pose window built from a bank of preprocessed per-frame clip arrays, with
// the results of features.extract (fk_vel -> re-rooting -> ik -> central differences, quat_op inv_mul_vec) bit for bit.
// One CTA per slot. Window frames are staged SW_CHUNK at a time in shared memory (local transforms, edge-padded the way
// preprocess.sliding_windows pads: pose of the edge frame, zero velocities), the next chunk's loads in flight while the
// current one is processed; the hierarchy is walked level by level with one thread per (frame, joint), in place, through
// the same joint steps as fk_rows_kernel. Each joint row is then
// re-rooted on the last frame's root, encoded and normalised into X; the hips' local positions (ik of joint 1) collect
// in shared memory for the central difference once all frames are done.
// ------------------------------------------------------------------------------------------------
constexpr int SW_CHUNK = 15;
constexpr int SW_THREADS = SW_CHUNK * MAXJ;            // one (frame, joint) item of a chunk per thread

__host__ __device__ inline size_t source_windows_smem(int T, int J) {
  return (size_t)SW_CHUNK * J * (4 + 3 + 3 + 3) * sizeof(float) + (size_t)T * 3 * sizeof(float);
}

// sliding_windows' index map: clip frame of window w's frame t (F frames in the clip), and whether t is padding
__device__ __forceinline__ int window_frame(int t, int w, int F, int T, bool& pad) {
  const int L = min(T, F - w), sh = T - L, left = (sh + 1) / 2;
  const int k = t - left;
  pad = k < 0 || k >= L;
  return w + min(max(k, 0), L - 1);
}

// torch's (0.5 * (x[t+1] - x[t]) * 60.0 + 0.5 * (x[t] - x[t-1]) * 60.0), every op rounded on its own (no FMA)
__device__ __forceinline__ float central_diff(float xm, float x0, float xp) {
  return __fadd_rn(__fmul_rn(__fmul_rn(0.5f, __fsub_rn(xp, x0)), 60.0f), __fmul_rn(__fmul_rn(0.5f, __fsub_rn(x0, xm)), 60.0f));
}

__global__ void __launch_bounds__(SW_THREADS)
source_windows_kernel(const float* __restrict__ brot, const float* __restrict__ bpos, const float* __restrict__ bvel,
                      const float* __restrict__ bang, const uint8_t* __restrict__ bcontacts, long long n_frames,
                      const long long* __restrict__ clip_first, const int32_t* __restrict__ clip_frames, int n_clips,
                      const int32_t* __restrict__ parents, int T, int J, const float* __restrict__ X_mean,
                      const float* __restrict__ X_std, const uint8_t* __restrict__ start, const int32_t* __restrict__ clip,
                      int32_t* __restrict__ slot_clip, int32_t* __restrict__ slot_cursor, float* __restrict__ X,
                      float* __restrict__ side, int side_stride, uint8_t* __restrict__ contacts) {
  pdl_trigger();
  extern __shared__ __align__(16) float sw_sm[];
  __shared__ int32_t par[MAXJ];
  __shared__ int32_t depth[MAXJ];
  __shared__ int s_maxd, s_w, s_F;
  __shared__ long long s_first;
  const int b = blockIdx.x, tid = threadIdx.x;
  const int V = J - 1;
  float* out_X = X + (long long)b * T * V * 15;
  float* out_side = side + (long long)b * side_stride;
  pdl_wait();
  if (tid < J) par[tid] = parents[tid];
  if (tid == 0) {
    int c = slot_clip[b], cur = slot_cursor[b];
    if (start[b]) { c = clip[b]; cur = 0; }
    int w = -1, F = 0;
    long long first = 0;
    if (c >= 0 && c < n_clips) {
      F = clip_frames[c];
      first = clip_first[c];
      const int nwin = F - T / 4;                        // sliding_windows' count: range(0, F - T // 4)
      if (nwin >= 1 && first >= 0 && first + F <= n_frames) {
        w = min(cur, nwin - 1);
        cur = w + 1;                                     // saturates at nwin: a finished clip repeats its last window
      }
    }
    if (w < 0) { c = -1; cur = 0; }                      // idle: never started, bad id or empty table entry
    if (start[b] || c >= 0) { slot_clip[b] = c; slot_cursor[b] = cur; }
    s_w = w; s_F = F; s_first = first; s_maxd = 0;
  }
  __syncthreads();
  const int w = s_w;
  if (w < 0) {                                           // idle slot: finite (zero) inputs
    for (int i = tid; i < T * V * 15; i += blockDim.x) out_X[i] = 0.0f;
    for (int i = tid; i < T * 3 + 6; i += blockDim.x) out_side[i] = 0.0f;
    if (tid < 2) contacts[b * 2 + tid] = 0;
    return;
  }
  if (tid < J) {
    int d = 0;
    for (int p = par[tid]; p >= 0 && p < J && d < J; p = par[p]) ++d;
    depth[tid] = d;
    atomicMax(&s_maxd, d);
  }
  const int F = s_F;
  const long long first = s_first;
  float* rot = sw_sm;                                    // [SW_CHUNK][J][4]: local, then global transforms
  float* pos = rot + SW_CHUNK * J * 4;                   // [SW_CHUNK][J][3]
  float* vel = pos + SW_CHUNK * J * 3;
  float* ang = vel + SW_CHUNK * J * 3;
  float* hips = ang + SW_CHUNK * J * 3;                  // [T][3]: ik local position of joint 1
  // the window's last frame: its root (re-rooting), root velocities and contacts
  bool pad_last;
  const long long fl = first + window_frame(T - 1, w, F, T, pad_last);
  const Q4<float> r0 = q4<float>(brot[fl * J * 4], brot[fl * J * 4 + 1], brot[fl * J * 4 + 2], brot[fl * J * 4 + 3]);
  const V3<float> p0 = v3<float>(bpos[fl * J * 3], bpos[fl * J * 3 + 1], bpos[fl * J * 3 + 2]);
  const Q4<float> r0i = qinv(r0);
  const V3<float> zero3 = v3<float>(0.0f, 0.0f, 0.0f);
  if (tid == 0) {
    const float zeros[3] = {0.0f, 0.0f, 0.0f};           // padded frames have zero velocities
    const V3<float> rv = q_mul_vec(brot + fl * J * 4, pad_last ? zeros : bvel + fl * J * 3, true);
    const V3<float> ra = q_mul_vec(brot + fl * J * 4, pad_last ? zeros : bang + fl * J * 3, true);
    float* o = out_side + T * 3;
    o[0] = rv.x; o[1] = rv.y; o[2] = rv.z; o[3] = ra.x; o[4] = ra.y; o[5] = ra.z;
    contacts[b * 2] = bcontacts[fl * 2];
    contacts[b * 2 + 1] = bcontacts[fl * 2 + 1];
  }
  __syncthreads();
  const int maxd = s_maxd;
  // this thread's item of a chunk: frame t0 + tid / J, joint tid % J; its local transform is loaded one chunk ahead
  const int jt = tid % J, ft = tid / J;
  float4 nr = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  float np_[3], nv[3], na[3];
  auto fetch = [&](int t0) {
    if (ft < SW_CHUNK && t0 + ft < T) {
      bool pad;
      const long long f = (first + window_frame(t0 + ft, w, F, T, pad)) * J + jt;
      nr = make_float4(brot[f * 4], brot[f * 4 + 1], brot[f * 4 + 2], brot[f * 4 + 3]);
      for (int c = 0; c < 3; ++c) {
        np_[c] = bpos[f * 3 + c];
        nv[c] = pad ? 0.0f : bvel[f * 3 + c];
        na[c] = pad ? 0.0f : bang[f * 3 + c];
      }
    }
  };
  fetch(0);
  for (int t0 = 0; t0 < T; t0 += SW_CHUNK) {
    const int n = min(SW_CHUNK, T - t0) * J;
    if (tid < n) {                                       // stage the local transforms of the chunk
      reinterpret_cast<float4*>(rot)[tid] = nr;
      for (int c = 0; c < 3; ++c) { pos[tid * 3 + c] = np_[c]; vel[tid * 3 + c] = nv[c]; ang[tid * 3 + c] = na[c]; }
    }
    __syncthreads();
    fetch(t0 + SW_CHUNK);
    for (int lvl = 1; lvl <= maxd; ++lvl) {              // quat.fk_vel, one hierarchy level at a time
      for (int i = tid; i < n; i += blockDim.x) {
        const int j = i % J;
        if (depth[j] != lvl) continue;
        const int q = i - j + par[j];                    // the parent joint of the same frame
        const float4 lr4 = reinterpret_cast<const float4*>(rot)[i], pr4 = reinterpret_cast<const float4*>(rot)[q];
        const Q4<float> pr = q4<float>(pr4.x, pr4.y, pr4.z, pr4.w);
        V3<float> rp, gp, gv, ga;
        Q4<float> gr;
        fk_joint_pose(pr, v3<float>(pos[q * 3], pos[q * 3 + 1], pos[q * 3 + 2]), q4<float>(lr4.x, lr4.y, lr4.z, lr4.w),
                      v3<float>(pos[i * 3], pos[i * 3 + 1], pos[i * 3 + 2]), rp, gp, gr);
        fk_joint_vel(pr, rp, v3<float>(vel[q * 3], vel[q * 3 + 1], vel[q * 3 + 2]),
                     v3<float>(ang[q * 3], ang[q * 3 + 1], ang[q * 3 + 2]), v3<float>(vel[i * 3], vel[i * 3 + 1], vel[i * 3 + 2]),
                     v3<float>(ang[i * 3], ang[i * 3 + 1], ang[i * 3 + 2]), gv, ga);
        reinterpret_cast<float4*>(rot)[i] = make_float4(gr.w, gr.x, gr.y, gr.z);
        pos[i * 3] = gp.x; pos[i * 3 + 1] = gp.y; pos[i * 3 + 2] = gp.z;
        vel[i * 3] = gv.x; vel[i * 3 + 1] = gv.y; vel[i * 3 + 2] = gv.z;
        ang[i * 3] = ga.x; ang[i * 3 + 1] = ga.y; ang[i * 3 + 2] = ga.z;
      }
      __syncthreads();
    }
    for (int i = tid; i < n; i += blockDim.x) {          // re-root, encode, normalise; ik of the hips
      const int j = i % J, t = t0 + i / J;
      if (j == 0) continue;                              // X drops the simulation root
      const float4 g4 = reinterpret_cast<const float4*>(rot)[i];
      V3<float> xp, xv, xa;
      Q4<float> xr;
      reroot_joint(r0i, p0, q4<float>(g4.x, g4.y, g4.z, g4.w), v3<float>(pos[i * 3], pos[i * 3 + 1], pos[i * 3 + 2]),
                   v3<float>(vel[i * 3], vel[i * 3 + 1], vel[i * 3 + 2]), v3<float>(ang[i * 3], ang[i * 3 + 1], ang[i * 3 + 2]),
                   xp, xr, xv, xa);
      float fr[15];
      feature_row(xp, xr, xv, xa, fr);
      store_normalised_row(out_X + ((long long)t * V + (j - 1)) * 15, fr, X_mean + j * 15, X_std + j * 15);
      if (j != 1) continue;
      V3<float> lp = xp;                                 // a root joint's local transform is its global one
      const int pj = par[1];
      if (pj >= 0) {
        // the parent's re-rooted transform; every frame's joint 0 row is the last frame's root
        const int q = i - 1 + pj;
        const float4 q4v = reinterpret_cast<const float4*>(rot)[q];
        const Q4<float> qg = pj == 0 ? r0 : q4<float>(q4v.x, q4v.y, q4v.z, q4v.w);
        const V3<float> qp = pj == 0 ? p0 : v3<float>(pos[q * 3], pos[q * 3 + 1], pos[q * 3 + 2]);
        V3<float> pxp, pxv, pxa;
        Q4<float> pxr, lr;
        reroot_joint(r0i, p0, qg, qp, zero3, zero3, pxp, pxr, pxv, pxa);
        ik_joint(pxr, pxp, xr, xp, lr, lp);
      }
      hips[t * 3] = lp.x; hips[t * 3 + 1] = lp.y; hips[t * 3 + 2] = lp.z;
    }
    __syncthreads();
  }
  // hips velocity: features._central_diff_time, linear extrapolation at both ends
  for (int i = tid; i < T * 3; i += blockDim.x) {
    const int t = i / 3, c = i % 3;
    const float* x = hips + c;
    float v;
    if (t == 0) {
      v = __fsub_rn(central_diff(x[0], x[3], x[6]), __fsub_rn(central_diff(x[6], x[9], x[12]), central_diff(x[3], x[6], x[9])));
    } else if (t == T - 1) {
      const float a = central_diff(x[(T - 3) * 3], x[(T - 2) * 3], x[(T - 1) * 3]);
      const float bb = central_diff(x[(T - 4) * 3], x[(T - 3) * 3], x[(T - 2) * 3]);
      v = __fadd_rn(a, __fsub_rn(a, bb));
    } else {
      v = central_diff(x[(t - 1) * 3], x[t * 3], x[(t + 1) * 3]);
    }
    out_side[i] = v;
  }
}

// ------------------------------------------------------------------------------------------------
// Result bank (DESIGN §5c). record_frames_kernel is the last launch of a frame: one warp per slot copies the slot's
// ik_pos / ik_rot / src_root_pos / src_root_rot (one contiguous span of mocha_frame_out) and its matched DB row into
// record row clip_first[c] + count of the clip c the slot served this frame. Copies only: nothing here lengthens the
// frame's critical path beyond a ~1.5 KB store per slot.
// clip_payload_kernel runs off the frame, once per batch of finished clips: one warp per (clip, window) row, one lane
// per joint, builds what the reference hands to bvh.save (test_fullframework.py:672-721; final_payload).
// ------------------------------------------------------------------------------------------------
constexpr int RF_WARPS = 4;
constexpr int REC_SPAN = 25 * 3 + 25 * 4 + 3 + 4;     // doubles from mocha_frame_out::ik_pos through src_root_rot
static_assert(offsetof(mocha_frame_out, src_root_rot) + 4 * sizeof(double) ==
              offsetof(mocha_frame_out, ik_pos) + REC_SPAN * sizeof(double), "frame_out record span is not contiguous");
static_assert(offsetof(mocha_frame_record, match) == REC_SPAN * sizeof(double) && sizeof(mocha_frame_record) == 1464,
              "mocha_frame_record layout");

__global__ void __launch_bounds__(RF_WARPS * 32)
record_frames_kernel(const mocha_frame_out* __restrict__ out, const int64_t* __restrict__ match_idx, int match_stride,
                     const uint8_t* __restrict__ start, const int32_t* __restrict__ slot_clip,
                     int32_t* __restrict__ slot_count, int B, const long long* __restrict__ clip_first,
                     const int32_t* __restrict__ clip_frames, int n_clips, int T, mocha_frame_record* __restrict__ rec,
                     long long n_rows, int32_t* __restrict__ clip_done, int32_t* __restrict__ clip_built) {
  pdl_trigger();
  pdl_wait();
  const int b = blockIdx.x * RF_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;
  long long row = -1;
  if (lane == 0) {
    int n = start[b] ? 0 : slot_count[b];
    const int c = slot_clip[b];                          // as mocha_source_windows left it for this frame
    if (c >= 0 && c < n_clips) {
      const int nwin = clip_frames[c] - T / 4;
      const long long r = clip_first[c] + n;
      if (n < nwin && r >= 0 && r < n_rows) {            // a finished clip's repeated last window writes nothing
        row = r;
        clip_done[c] = ++n;
        clip_built[c] = 0;                               // a new row makes the clip's payload stale
      }
    }
    slot_count[b] = n;
  }
  row = __shfl_sync(0xffffffffu, row, 0);
  if (row < 0) return;
  const double* src = &out[b].ik_pos[0][0];
  double* dst = &rec[row].ik_pos[0][0];
  for (int i = lane; i < REC_SPAN; i += 32) dst[i] = src[i];
  if (lane == 0) rec[row].match = match_idx[(long long)b * match_stride];
}

constexpr int CP_WARPS = 4;
constexpr int REC_J = 25;

__global__ void __launch_bounds__(CP_WARPS * 32)
clip_payload_kernel(const mocha_frame_record* __restrict__ rec, long long n_frames, const float* __restrict__ brot,
                    const float* __restrict__ bpos, const long long* __restrict__ clip_first,
                    const int32_t* __restrict__ clip_frames, int n_clips, const int32_t* __restrict__ clip_done,
                    int32_t* __restrict__ clip_built,
                    const int32_t* __restrict__ parents, int T, const int32_t* __restrict__ ids,
                    float* __restrict__ src_rot, float* __restrict__ src_pos, double* __restrict__ ours_rot,
                    double* __restrict__ ours_pos, int64_t* __restrict__ match) {
  pdl_trigger();
  pdl_wait();
  constexpr int J = REC_J;
  constexpr unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31, w = blockIdx.x * CP_WARPS + (threadIdx.x >> 5);
  const int c = ids[blockIdx.y];
  if (c < 0 || c >= n_clips) return;
  const int F = clip_frames[c];
  const long long first = clip_first[c];
  const int nwin = F - T / 4;
  if (nwin < 1 || first < 0 || first + F > n_frames) return;
  const int done = clip_done[c];
  if (blockIdx.x == 0 && threadIdx.x == 0) clip_built[c] = done >= nwin;   // the payload of a complete clip
  if (w >= min(done, nwin)) return;                      // warp-uniform
  const long long row = first + w;
  const int j = lane;
  const bool on = j < J;
  const int pj = on ? parents[j] : -1;
  const int d = on ? joint_depth(parents, j, J) : 0;
  const int maxd = __reduce_max_sync(FULL, d);
  // src: the local pose of window w's last frame as features.extract gives it (Ypos[w, -1] / Yrot[w, -1]): fk of that
  // frame (sliding_windows' edge padding keeps the edge frame's pose), re-rooted on its own root, then ik
  bool pad;
  const long long f = (first + window_frame(T - 1, w, F, T, pad)) * J + (on ? j : 0);
  const Q4<float> lr = q4<float>(brot[f * 4], brot[f * 4 + 1], brot[f * 4 + 2], brot[f * 4 + 3]);
  const V3<float> lp = v3<float>(bpos[f * 3], bpos[f * 3 + 1], bpos[f * 3 + 2]);
  Q4<float> gr = lr;
  V3<float> gp = lp;
  const int src_lane = pj >= 0 ? pj : j;
  for (int lvl = 1; lvl <= maxd; ++lvl) {                // quat.fk, one hierarchy level at a time
    const Q4<float> pr = q4<float>(__shfl_sync(FULL, gr.w, src_lane), __shfl_sync(FULL, gr.x, src_lane),
                                   __shfl_sync(FULL, gr.y, src_lane), __shfl_sync(FULL, gr.z, src_lane));
    const V3<float> pp = v3<float>(__shfl_sync(FULL, gp.x, src_lane), __shfl_sync(FULL, gp.y, src_lane),
                                   __shfl_sync(FULL, gp.z, src_lane));
    if (d == lvl) {
      V3<float> rp;
      fk_joint_pose(pr, pp, lr, lp, rp, gp, gr);
    }
  }
  const Q4<float> r0 = q4<float>(__shfl_sync(FULL, gr.w, 0), __shfl_sync(FULL, gr.x, 0), __shfl_sync(FULL, gr.y, 0),
                                 __shfl_sync(FULL, gr.z, 0));
  const V3<float> p0 = v3<float>(__shfl_sync(FULL, gp.x, 0), __shfl_sync(FULL, gp.y, 0), __shfl_sync(FULL, gp.z, 0));
  const V3<float> zero3 = v3<float>(0.0f, 0.0f, 0.0f);
  V3<float> xp, xv, xa;
  Q4<float> xr;
  reroot_joint(qinv(r0), p0, gr, gp, zero3, zero3, xp, xr, xv, xa);
  const Q4<float> pxr = q4<float>(__shfl_sync(FULL, xr.w, src_lane), __shfl_sync(FULL, xr.x, src_lane),
                                  __shfl_sync(FULL, xr.y, src_lane), __shfl_sync(FULL, xr.z, src_lane));
  const V3<float> pxp = v3<float>(__shfl_sync(FULL, xp.x, src_lane), __shfl_sync(FULL, xp.y, src_lane),
                                  __shfl_sync(FULL, xp.z, src_lane));
  Q4<float> sr = xr;                                     // a root joint's local transform is its global one
  V3<float> sp = xp;
  if (pj >= 0) ik_joint(pxr, pxp, xr, xp, sr, sp);
  if (!on || j == 0) return;                             // the payload drops the simulation root
  const mocha_frame_record& R = rec[row];
  // ours (fp64): the recorded post-IK pose
  DQ orr = ld4(&R.ik_rot[j][0]);
  D3 op = ld3(&R.ik_pos[j][0]);
  if (j == 1 && pj == 0) {
    // hips: global transform under the recorded root; src in fp32 under the integrated source root (:478-488)
    const DQ r = ld4(&R.ik_rot[0][0]);
    op = qrot(r, op) + ld3(&R.ik_pos[0][0]);
    orr = qmul(r, orr);
    const Q4<float> qr = q4<float>((float)R.src_root_rot[0], (float)R.src_root_rot[1], (float)R.src_root_rot[2],
                                   (float)R.src_root_rot[3]);
    const V3<float> qp = v3<float>((float)R.src_root_pos[0], (float)R.src_root_pos[1], (float)R.src_root_pos[2]);
    V3<float> rp, hp;
    Q4<float> hr;
    fk_joint_pose(qr, qp, sr, sp, rp, hp, hr);
    sr = hr;
    sp = hp;
  }
  const long long o = (row * (J - 1) + (j - 1)) * 3;
  float fe[3];
  to_euler_xyz(sr.w, sr.x, sr.y, sr.z, fe);
  double de[3];
  to_euler_xyz(orr.w, orr.x, orr.y, orr.z, de);
  constexpr double DEG = 180.0 / 3.14159265358979323846;          // np.degrees
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    src_rot[o + k] = fe[k] * (float)DEG;
    ours_rot[o + k] = de[k] * DEG;
  }
  src_pos[o] = sp.x; src_pos[o + 1] = sp.y; src_pos[o + 2] = sp.z;
  ours_pos[o] = op.x; ours_pos[o + 1] = op.y; ours_pos[o + 2] = op.z;
  if (j == 1) match[row] = R.match;
}
}  // namespace

extern "C" int mocha_window_features(const float* grot, const float* gpos, const float* gvel, const float* gang, long long W,
                                     int T, int J, const float* X_mean, const float* X_std, float* X, float* xrot, float* xpos,
                                     mocha_stream_t stream) {
  MOCHA_CHECK_ARG(grot && gpos && gvel && gang && X, "mocha_window_features: null argument");
  MOCHA_CHECK_ARG(W > 0 && T > 0 && J > 1 && J <= MAXJ, "mocha_window_features: bad sizes W=%lld T=%d J=%d", W, T, J);
  // X_mean == NULL selects the training twin (trainer.py:337-374): per-frame root, all joints, no normalisation
  const int per_frame = X_mean == nullptr;
  MOCHA_CHECK_ARG(per_frame || X_std, "mocha_window_features: X_std missing");
  const long long total = W * T * J;
  launch_k(window_reroot_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, (cudaStream_t)stream, grot, gpos, gvel, gang, W,
           T, J, X_mean, X_std, X, xrot, xpos, per_frame);
  count_launch();
  MOCHA_LAUNCH_CHECK("window_reroot_kernel");
  return MOCHA_OK;
}

extern "C" int mocha_source_windows(const float* rot, const float* pos, const float* vel, const float* ang,
                                    const uint8_t* bank_contacts, long long n_frames, const int64_t* clip_first,
                                    const int32_t* clip_frames, int n_clips, const int32_t* parents, int T, int J,
                                    const float* X_mean, const float* X_std, const uint8_t* start, const int32_t* clip,
                                    int32_t* slot_clip, int32_t* slot_cursor, int B, float* X, float* side, int side_stride,
                                    uint8_t* contacts, mocha_stream_t stream) {
  MOCHA_CHECK_ARG(rot && pos && vel && ang && bank_contacts && clip_first && clip_frames && parents && X_mean && X_std,
                  "mocha_source_windows: null bank argument");
  MOCHA_CHECK_ARG(start && clip && slot_clip && slot_cursor && X && side && contacts, "mocha_source_windows: null slot argument");
  MOCHA_CHECK_ARG(B > 0 && n_frames > 0 && n_clips > 0, "mocha_source_windows: bad sizes B=%d n_frames=%lld n_clips=%d", B,
                  n_frames, n_clips);
  MOCHA_CHECK_ARG(J >= 2 && J <= MAXJ && T >= 5 && T <= 1024, "mocha_source_windows: need 2 <= J <= %d and 5 <= T <= 1024, "
                  "got J=%d T=%d", MAXJ, J, T);
  MOCHA_CHECK_ARG(side_stride >= T * 3 + 6, "mocha_source_windows: side rows need T*3+6 floats, stride %d", side_stride);
  MOCHA_CHECK_ARG((reinterpret_cast<uintptr_t>(rot) & 15) == 0, "mocha_source_windows: rotations not 16 B aligned");
  const size_t smem = source_windows_smem(T, J);
  static size_t configured = 0;
  if (smem > 48 * 1024 && smem > configured) {
    MOCHA_CUDA(cudaFuncSetAttribute(source_windows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  launch_k(source_windows_kernel, B, SW_THREADS, smem, (cudaStream_t)stream, rot, pos, vel, ang, bank_contacts, n_frames,
           reinterpret_cast<const long long*>(clip_first), clip_frames, n_clips, parents, T, J, X_mean, X_std, start, clip,
           slot_clip, slot_cursor, X, side, side_stride, contacts);
  count_launch();
  MOCHA_LAUNCH_CHECK("source_windows_kernel");
  return MOCHA_OK;
}

extern "C" int mocha_record_frames(const mocha_frame_out* out, const int64_t* match_idx, int match_stride,
                                   const uint8_t* start, const int32_t* slot_clip, int32_t* slot_count, int B,
                                   const int64_t* clip_first, const int32_t* clip_frames, int n_clips, int T,
                                   mocha_frame_record* rec, long long n_rows, int32_t* clip_done, int32_t* clip_built,
                                   mocha_stream_t stream) {
  MOCHA_CHECK_ARG(out && match_idx && start && slot_clip && slot_count, "mocha_record_frames: null slot argument");
  MOCHA_CHECK_ARG(clip_first && clip_frames && rec && clip_done && clip_built, "mocha_record_frames: null bank argument");
  MOCHA_CHECK_ARG(B > 0 && n_clips > 0 && n_rows > 0 && match_stride >= 1 && T >= 5,
                  "mocha_record_frames: bad sizes B=%d n_clips=%d n_rows=%lld match_stride=%d T=%d", B, n_clips, n_rows,
                  match_stride, T);
  launch_k(record_frames_kernel, ceil_div(B, RF_WARPS), RF_WARPS * 32, 0, (cudaStream_t)stream, out, match_idx,
           match_stride, start, slot_clip, slot_count, B, reinterpret_cast<const long long*>(clip_first), clip_frames,
           n_clips, T, rec, n_rows, clip_done, clip_built);
  count_launch();
  MOCHA_LAUNCH_CHECK("record_frames_kernel");
  return MOCHA_OK;
}

extern "C" int mocha_clip_payload(const mocha_frame_record* rec, long long n_frames, const float* rot, const float* pos,
                                  const int64_t* clip_first, const int32_t* clip_frames, int n_clips,
                                  const int32_t* clip_done, int32_t* clip_built, const int32_t* parents, int T, int J,
                                  const int32_t* ids,
                                  int n_ids, int max_nwin, float* src_rot, float* src_pos, double* ours_rot,
                                  double* ours_pos, int64_t* match, mocha_stream_t stream) {
  MOCHA_CHECK_ARG(rec && rot && pos && clip_first && clip_frames && clip_done && clip_built && parents,
                  "mocha_clip_payload: null bank argument");
  MOCHA_CHECK_ARG(ids && src_rot && src_pos && ours_rot && ours_pos && match, "mocha_clip_payload: null output argument");
  MOCHA_CHECK_ARG(n_frames > 0 && n_clips > 0 && n_ids > 0 && n_ids <= 65535 && max_nwin > 0,
                  "mocha_clip_payload: bad sizes n_frames=%lld n_clips=%d n_ids=%d max_nwin=%d", n_frames, n_clips, n_ids,
                  max_nwin);
  MOCHA_CHECK_ARG(J == REC_J && T >= 5, "mocha_clip_payload: need J=%d and T >= 5, got J=%d T=%d", REC_J, J, T);
  launch_k(clip_payload_kernel, dim3((unsigned)ceil_div(max_nwin, CP_WARPS), (unsigned)n_ids), CP_WARPS * 32, 0,
           (cudaStream_t)stream, rec, n_frames, rot, pos, reinterpret_cast<const long long*>(clip_first), clip_frames,
           n_clips, clip_done, clip_built, parents, T, ids, src_rot, src_pos, ours_rot, ours_pos, match);
  count_launch();
  MOCHA_LAUNCH_CHECK("clip_payload_kernel");
  return MOCHA_OK;
}
