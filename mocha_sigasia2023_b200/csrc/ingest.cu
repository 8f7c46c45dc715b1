// Raw clip ingestion (DESIGN §5d): preprocess.process_frames restated in fp64 for a whole batch of clips, written
// straight into the source bank's float32 rows. Every fp64 expression that restates a NumPy expression is spelled out
// op by op with __dmul_rn / __dadd_rn / __dsub_rn (no FMA contraction), in NumPy's evaluation order: sums over the
// last axis are sequential, np.cross is (a1 b2 - a2 b1, a2 b0 - a0 b2, a0 b1 - a1 b0), and scalar constants such as
// [1, 0, 1] or the zero components of an Euler axis are multiplied in (they decide the signs of zeros). Only sin, cos,
// atan2 and the savgol edge fits (scipy: polyfit; here: the same linear map as a table) are not NumPy's own bits.
//
// Five launches over a caller-sized fp64 workspace (the whole clip is needed between phases):
//   ingest_local_kernel     per (frame, joint): Euler -> quaternion, cm -> m; per frame: FK of the joints the root
//                           needs, raw root position and normalised root direction
//   ingest_unroll_kernel    per (clip, joint): quaternion sign recurrence over frames, a segmented parity scan
//   ingest_root_kernel      per frame: the two savgol filters, root direction -> root rotation
//   ingest_frames_kernel    per (frame, bone): re-rooting, central differences, angular velocity, float32 outputs;
//                           per (frame, toe): fk_vel down the toe's chain, toe speed < 0.5
//   ingest_contacts_kernel  per frame: median_filter(size=6, mode='nearest') of the toe flags as a count
// A clip whose table entry points outside the raw buffer or the bank, has fewer than 31 frames, more than
// max_clip_frames, or an unknown order code is skipped by every kernel: nothing of it is written.
#include "../../include/mocha_b200.h"
#include "common.cuh"

using namespace mocha;

namespace {

constexpr int IG_MAXJ = 31;            // raw joints; the bank adds the root bone
constexpr int IG_MIN_FRAMES = 31;      // savgol window of the root direction (scipy rejects shorter clips)
constexpr int IG_FT = 8;               // frames per CTA of the per-(frame, joint) kernels
constexpr int IG_ROOT_THREADS = 128;
constexpr int IG_UNROLL_WARPS = 4;

struct IngestSkel {
  int J0;                              // raw joints; bank bones J = J0 + 1
  int parents[IG_MAXJ];                // raw parents: parents[0] = -1, 0 <= parents[j] < j
  int spine2, shoulder_l, shoulder_r, upleg_l, upleg_r, toe_l, toe_r;   // raw joint indices
  unsigned fk_mask;                    // joints the root inputs need: spine2 .. upleg_r and their ancestors
};

struct IngestClips {
  const long long* first;              // raw frame of the clip's frame 0
  const int32_t* frames;
  const int32_t* order;                // Euler order code, 0..5 = xyz xzy yxz yzx zxy zyx
  int n_clips, max_frames;
  long long n_raw, bank_rows, row0;    // the clip's bank rows are row0 + first .. + frames
};

struct IngestWs {
  double *lrot, *lpos;                 // [N, J0, 4|3] local pose (unrolled in place)
  double *rp_raw, *rdir;               // [N, 3] root position before the filter, normalised root direction before it
  double *root_pos, *root_rot;         // [N, 3|4]
  uint8_t* toe;                        // [N, 2] toe speed < 0.5
};

__device__ __forceinline__ bool clip_ok(const IngestClips& cl, int c, long long& first, int& F) {
  first = cl.first[c];
  F = cl.frames[c];
  const int o = cl.order[c];
  return F >= IG_MIN_FRAMES && F <= cl.max_frames && first >= 0 && first + F <= cl.n_raw && o >= 0 && o < 6 &&
         cl.row0 + first + F <= cl.bank_rows;
}

struct D3 { double x, y, z; };
struct D4 { double w, x, y, z; };

__device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ D3 add3(D3 a, D3 b) { return {add(a.x, b.x), add(a.y, b.y), add(a.z, b.z)}; }
__device__ __forceinline__ D3 sub3(D3 a, D3 b) { return {sub(a.x, b.x), sub(a.y, b.y), sub(a.z, b.z)}; }
__device__ __forceinline__ D3 scale3(double s, D3 a) { return {mul(s, a.x), mul(s, a.y), mul(s, a.z)}; }
__device__ __forceinline__ double sumsq3(D3 a) { return add(add(mul(a.x, a.x), mul(a.y, a.y)), mul(a.z, a.z)); }
__device__ __forceinline__ D3 cross3(D3 a, D3 b) {    // np.cross
  return {sub(mul(a.y, b.z), mul(a.z, b.y)), sub(mul(a.z, b.x), mul(a.x, b.z)), sub(mul(a.x, b.y), mul(a.y, b.x))};
}
__device__ __forceinline__ D4 qneg(D4 q) { return {-q.w, -q.x, -q.y, -q.z}; }
__device__ __forceinline__ D4 qinv(D4 q) { return {q.w, -q.x, -q.y, -q.z}; }                 // q * [1, -1, -1, -1]
__device__ __forceinline__ D4 qmul(D4 a, D4 b) {      // preprocess._qmul
  return {sub(sub(sub(mul(b.w, a.w), mul(b.x, a.x)), mul(b.y, a.y)), mul(b.z, a.z)),
          add(sub(add(mul(b.w, a.x), mul(b.x, a.w)), mul(b.y, a.z)), mul(b.z, a.y)),
          sub(add(add(mul(b.w, a.y), mul(b.x, a.z)), mul(b.y, a.w)), mul(b.z, a.x)),
          add(add(sub(mul(b.w, a.z), mul(b.x, a.y)), mul(b.y, a.x)), mul(b.z, a.w))};
}
__device__ __forceinline__ D3 qrot(D4 q, D3 v) {      // preprocess._qrot: v + w t + u x t, t = 2 (u x v)
  const D3 u = {q.x, q.y, q.z};
  const D3 t = scale3(2.0, cross3(u, v));
  return add3(add3(v, scale3(q.w, t)), cross3(u, t));
}
__device__ __forceinline__ D3 qlog(D4 q) {            // preprocess._log, eps = 1e-5
  const D3 v = {q.x, q.y, q.z};
  const double ln = __dsqrt_rn(sumsq3(v));
  const double half = ln < 1e-5 ? 1.0 : __ddiv_rn(atan2(ln, q.w), ln);
  return scale3(half, v);
}
__device__ __forceinline__ D4 qabs(D4 q) { return q.w > 0.0 ? q : qneg(q); }

__device__ __forceinline__ D3 ld3(const double* p) { return {p[0], p[1], p[2]}; }
__device__ __forceinline__ D4 ld4(const double* p) { return {p[0], p[1], p[2], p[3]}; }
__device__ __forceinline__ void st3(double* p, D3 v) { p[0] = v.x; p[1] = v.y; p[2] = v.z; }
__device__ __forceinline__ void st4(double* p, D4 q) { p[0] = q.w; p[1] = q.x; p[2] = q.y; p[3] = q.z; }

// ---- phase 1: local pose, FK of the root inputs ------------------------------------------------------------------
// axis index (0 x, 1 y, 2 z) of each Euler angle for order codes xyz xzy yxz yzx zxy zyx
__constant__ int8_t c_order_axes[6][3] = {{0, 1, 2}, {0, 2, 1}, {1, 0, 2}, {1, 2, 0}, {2, 0, 1}, {2, 1, 0}};

__device__ __forceinline__ D4 axis_angle(double angle, int axis) {   // preprocess._axis_angle with a unit axis
  const double half = mul(angle, 0.5);                                 // angle / 2.0 (exact)
  double s, c;
  sincos(half, &s, &c);
  return {c, mul(s, axis == 0 ? 1.0 : 0.0), mul(s, axis == 1 ? 1.0 : 0.0), mul(s, axis == 2 ? 1.0 : 0.0)};
}

__global__ void __launch_bounds__(IG_FT * 32)
ingest_local_kernel(const double* __restrict__ raw_rot, const double* __restrict__ raw_pos, IngestClips cl, IngestSkel sk,
                    IngestWs ws) {
  pdl_trigger();
  __shared__ double s_lrot[IG_FT][32][4], s_lpos[IG_FT][32][3];
  __shared__ double s_grot[IG_FT][32][4], s_gpos[IG_FT][32][3];
  pdl_wait();
  const int c = blockIdx.x;
  long long first;
  int F;
  if (!clip_ok(cl, c, first, F)) return;
  const int j = threadIdx.x & 31, fr = threadIdx.x >> 5;
  const int f = blockIdx.y * IG_FT + fr;
  const int J0 = sk.J0;
  if (f < F && j < J0) {
    const long long i = (first + f) * J0 + j;
    const int8_t* ax = c_order_axes[cl.order[c]];
    constexpr double kRad = 3.141592653589793 / 180.0;                 // np.radians
    const D4 qa = axis_angle(mul(raw_rot[i * 3 + 0], kRad), ax[0]);
    const D4 qb = axis_angle(mul(raw_rot[i * 3 + 1], kRad), ax[1]);
    const D4 qc = axis_angle(mul(raw_rot[i * 3 + 2], kRad), ax[2]);
    const D4 q = qmul(qa, qmul(qb, qc));
    const D3 p = scale3(0.01, ld3(raw_pos + i * 3));                   // cm -> m (x * 0.01)
    st4(ws.lrot + i * 4, q);
    st3(ws.lpos + i * 3, p);
    st4(s_lrot[fr][j], q);
    st3(s_lpos[fr][j], p);
  }
  __syncthreads();
  if (j != 0 || f >= F) return;
  // One thread per frame walks the joints the root inputs need. The unroll comes later: q and -q give the same bits
  // through qrot and the same up to sign through qmul, so global positions do not depend on it.
  st4(s_grot[fr][0], ld4(s_lrot[fr][0]));
  st3(s_gpos[fr][0], ld3(s_lpos[fr][0]));
  for (int k = 1; k < J0; ++k) {
    if (!((sk.fk_mask >> k) & 1u)) continue;
    const int p = sk.parents[k];
    const D4 gr = ld4(s_grot[fr][p]);
    st3(s_gpos[fr][k], add3(qrot(gr, ld3(s_lpos[fr][k])), ld3(s_gpos[fr][p])));
    st4(s_grot[fr][k], qmul(gr, ld4(s_lrot[fr][k])));
  }
  const D3 s2 = ld3(s_gpos[fr][sk.spine2]);
  const D3 rp = {mul(1.0, s2.x), mul(0.0, s2.y), mul(1.0, s2.z)};      // [1, 0, 1] * gpos[spine2]
  const D3 across = add3(sub3(ld3(s_gpos[fr][sk.shoulder_l]), ld3(s_gpos[fr][sk.shoulder_r])),
                         sub3(ld3(s_gpos[fr][sk.upleg_l]), ld3(s_gpos[fr][sk.upleg_r])));
  const D3 cr = cross3(across, D3{0.0, 1.0, 0.0});
  D3 rd = {mul(1.0, cr.x), mul(0.0, cr.y), mul(1.0, cr.z)};
  const double n = __dsqrt_rn(sumsq3(rd));
  rd = {__ddiv_rn(rd.x, n), __ddiv_rn(rd.y, n), __ddiv_rn(rd.z, n)};
  st3(ws.rp_raw + (first + f) * 3, rp);
  st3(ws.rdir + (first + f) * 3, rd);
}

// ---- phase 2: unroll ----------------------------------------------------------------------------------------------
// preprocess._unroll negates frame i when (out[i] * out[i-1]).sum() < 0, out[i-1] being already unrolled. With
// d_i = (q_i * q_{i-1}).sum() on the un-flipped quaternions that dot is s_{i-1} d_i exactly (negation commutes with
// rounding), so the sign is s_i = (s_{i-1} d_i < 0) ? -1 : +1: it keeps s_{i-1} when d_i > 0, flips it when d_i < 0,
// and RESETS to +1 when d_i is +-0 or NaN (the comparison is false). Frame 0 is a reset. s is therefore the parity of
// the d < 0 frames since the last reset: a segmented parity scan, done 32 frames at a time per warp with ballot + popc
// (one warp per (clip, joint)). The previous frame's raw quaternion comes through a shuffle, never from the
// already-negated memory.
__global__ void __launch_bounds__(IG_UNROLL_WARPS * 32)
ingest_unroll_kernel(IngestClips cl, int J0, IngestWs ws) {
  pdl_trigger();
  pdl_wait();
  const int c = blockIdx.x;
  const int lane = threadIdx.x & 31;
  const int j = blockIdx.y * IG_UNROLL_WARPS + (threadIdx.x >> 5);
  long long first;
  int F;
  if (j >= J0 || !clip_ok(cl, c, first, F)) return;                   // warp-uniform
  const unsigned full = 0xffffffffu;
  const unsigned upto = lane == 31 ? full : (2u << lane) - 1u;          // lanes 0 .. lane
  D4 carry_q = {0.0, 0.0, 0.0, 0.0};                                    // raw quaternion of the frame before the chunk
  unsigned carry_s = 0;                                                 // its sign: 1 = negated
  for (int base = 0; base < F; base += 32) {
    const int i = base + lane;
    double* qp = ws.lrot + ((first + i) * J0 + j) * 4;
    D4 q = {0.0, 0.0, 0.0, 0.0};
    if (i < F) q = ld4(qp);
    D4 prev = {__shfl_up_sync(full, q.w, 1), __shfl_up_sync(full, q.x, 1), __shfl_up_sync(full, q.y, 1),
               __shfl_up_sync(full, q.z, 1)};
    if (lane == 0) prev = carry_q;
    bool neg = false, reset = true;
    if (i > 0 && i < F) {
      const double d = add(add(add(mul(q.w, prev.w), mul(q.x, prev.x)), mul(q.y, prev.y)), mul(q.z, prev.z));
      neg = d < 0.0;
      reset = !(d > 0.0) && !neg;
    }
    const unsigned nb = __ballot_sync(full, neg), rb = __ballot_sync(full, reset) & upto;
    unsigned s;
    if (rb) {
      const int last = 31 - __clz(rb);                                  // last reset at or before this frame
      const unsigned after = last == 31 ? 0u : ~((2u << last) - 1u);
      s = __popc(nb & upto & after) & 1u;
    } else {
      s = (carry_s + __popc(nb & upto)) & 1u;
    }
    carry_s = __shfl_sync(full, s, 31);
    carry_q = {__shfl_sync(full, q.w, 31), __shfl_sync(full, q.x, 31), __shfl_sync(full, q.y, 31),
               __shfl_sync(full, q.z, 31)};
    if (i < F && s) st4(qp, qneg(q));
  }
}

// ---- phase 3: root trajectory -------------------------------------------------------------------------------------
// savgol_filter(x, wl, 3, axis=0, mode='interp') on column k of x [F, 3]. tab = [w (wl) | left map (h, wl) | right
// map (h, wl)], h = wl / 2: w are the correlation weights ndimage applies (the coefficients reversed), the maps give
// the first / last h outputs from the first / last wl samples. ndimage treats weights that are equal within
// DBL_EPSILON as symmetric, which savgol's are, and then sums x[i] w[h] + (x[i-h+k] + x[i+h-k]) w[k] for k = 0 .. h-1
// in that order; the Python wrapper checks the symmetry before it hands the table over. The edge sums end with + 0:
// the columns process_frames multiplies by 0 hold +-0, and scipy's fit gives +0 at their edges where a sum of -0 terms
// would keep -0.
__device__ double savgol(const double* __restrict__ x, int F, int f, const double* __restrict__ tab, int wl) {
  const int h = wl / 2;
  if (f < h || f >= F - h) {
    const double* row = f < h ? tab + wl + f * wl : tab + wl + (h + f - (F - h)) * wl;
    const double* xs = f < h ? x : x + (F - wl) * 3;
    double t = mul(row[0], xs[0]);
    for (int k = 1; k < wl; ++k) t = add(t, mul(row[k], xs[k * 3]));
    return add(t, 0.0);                  // polyfit's edge values of an all-zero column are +0; -0 + 0 = +0, else exact
  }
  double t = mul(x[f * 3], tab[h]);
  for (int k = 0; k < h; ++k) t = add(t, mul(add(x[(f - h + k) * 3], x[(f + h - k) * 3]), tab[k]));
  return t;
}

__global__ void __launch_bounds__(IG_ROOT_THREADS)
ingest_root_kernel(IngestClips cl, const double* __restrict__ sg15, const double* __restrict__ sg31, IngestWs ws) {
  pdl_trigger();
  pdl_wait();
  const int c = blockIdx.x;
  long long first;
  int F;
  if (!clip_ok(cl, c, first, F)) return;
  const int f = blockIdx.y * IG_ROOT_THREADS + threadIdx.x;
  if (f >= F) return;
  const double* rp = ws.rp_raw + first * 3;
  const double* rd = ws.rdir + first * 3;
  const D3 pos = {savgol(rp, F, f, sg15, 15), savgol(rp + 1, F, f, sg15, 15), savgol(rp + 2, F, f, sg15, 15)};
  D3 dir = {savgol(rd, F, f, sg31, 31), savgol(rd + 1, F, f, sg31, 31), savgol(rd + 2, F, f, sg31, 31)};
  const double n = __dsqrt_rn(sumsq3(dir));
  dir = {__ddiv_rn(dir.x, n), __ddiv_rn(dir.y, n), __ddiv_rn(dir.z, n)};
  // quat.between(fwd = [0, 0, 1], dir), written as process_frames writes it, then normalised with + 1e-8
  const D4 b = {add(__dsqrt_rn(mul(1.0, sumsq3(dir))), add(add(mul(0.0, dir.x), mul(0.0, dir.y)), mul(1.0, dir.z))),
                sub(mul(0.0, dir.z), mul(1.0, dir.y)), sub(mul(1.0, dir.x), mul(0.0, dir.z)),
                sub(mul(0.0, dir.y), mul(0.0, dir.x))};
  const double bn = add(__dsqrt_rn(add(add(add(mul(b.w, b.w), mul(b.x, b.x)), mul(b.y, b.y)), mul(b.z, b.z))), 1e-8);
  st3(ws.root_pos + (first + f) * 3, pos);
  st4(ws.root_rot + (first + f) * 4, D4{__ddiv_rn(b.w, bn), __ddiv_rn(b.x, bn), __ddiv_rn(b.y, bn), __ddiv_rn(b.z, bn)});
}

// ---- phase 4: per-frame outputs -----------------------------------------------------------------------------------
// Bone b of the bank skeleton is raw joint b - 1; bone 0 is the root (root_pos / root_rot), bone 1 the hips re-rooted
// on it. Neighbouring frames' values are recomputed where a difference needs them (the same bits every time).
struct ClipFrames {
  const double *lrot, *lpos, *root_pos, *root_rot;   // at the clip's first frame
  int J0, F;
};

__device__ __forceinline__ D3 bone_pos(const ClipFrames& v, int f, int b) {
  const D3 rp = ld3(v.root_pos + f * 3);
  if (b == 0) return rp;
  const D3 p = ld3(v.lpos + ((long long)f * v.J0 + b - 1) * 3);
  return b == 1 ? qrot(qinv(ld4(v.root_rot + f * 4)), sub3(p, rp)) : p;
}
__device__ __forceinline__ D4 bone_rot(const ClipFrames& v, int f, int b) {
  const D4 rr = ld4(v.root_rot + f * 4);
  if (b == 0) return rr;
  const D4 q = ld4(v.lrot + ((long long)f * v.J0 + b - 1) * 4);
  return b == 1 ? qmul(qinv(rr), q) : q;
}
// preprocess._central_diff interior: 0.5 * (x[i+1] - x[i]) * 60 + 0.5 * (x[i] - x[i-1]) * 60
__device__ __forceinline__ double cdiff(double xm, double x0, double xp) {
  return add(mul(mul(0.5, sub(xp, x0)), 60.0), mul(mul(0.5, sub(x0, xm)), 60.0));
}
__device__ __noinline__ D3 vel_interior(const ClipFrames& v, int f, int b) {
  const D3 m = bone_pos(v, f - 1, b), o = bone_pos(v, f, b), p = bone_pos(v, f + 1, b);
  return {cdiff(m.x, o.x, p.x), cdiff(m.y, o.y, p.y), cdiff(m.z, o.z, p.z)};
}
// preprocess._angular_velocity interior: log(abs(q[i+1] q[i]^-1)) * 60 + log(abs(q[i] q[i-1]^-1)) * 60
__device__ __noinline__ D3 ang_interior(const ClipFrames& v, int f, int b) {
  const D4 m = bone_rot(v, f - 1, b), o = bone_rot(v, f, b), p = bone_rot(v, f + 1, b);
  return add3(scale3(60.0, qlog(qabs(qmul(p, qinv(o))))), scale3(60.0, qlog(qabs(qmul(o, qinv(m))))));
}
// the edge rule of both: v[0] = v[1] - (v[3] - v[2]), v[-1] = v[-2] + (v[-2] - v[-3])
__device__ D3 with_edges(const ClipFrames& v, int f, int b, bool angular) {
  auto at = [&](int k) { return angular ? ang_interior(v, k, b) : vel_interior(v, k, b); };
  if (f == 0) return sub3(at(1), sub3(at(3), at(2)));
  if (f == v.F - 1) {
    const D3 a = at(v.F - 2);
    return add3(a, sub3(a, at(v.F - 3)));
  }
  return at(f);
}

__global__ void __launch_bounds__(IG_FT * 32)
ingest_frames_kernel(IngestClips cl, IngestSkel sk, IngestWs ws, float* __restrict__ out_rot, float* __restrict__ out_pos,
                     float* __restrict__ out_vel, float* __restrict__ out_ang) {
  pdl_trigger();
  pdl_wait();
  const int c = blockIdx.x;
  long long first;
  int F;
  if (!clip_ok(cl, c, first, F)) return;
  const int b = threadIdx.x & 31;
  const int f = blockIdx.y * IG_FT + (threadIdx.x >> 5);
  if (f >= F) return;
  const int J0 = sk.J0, J = J0 + 1;
  const ClipFrames v = {ws.lrot + first * J0 * 4, ws.lpos + first * J0 * 3, ws.root_pos + first * 3,
                        ws.root_rot + first * 4, J0, F};
  if (b < J) {
    const long long o = (cl.row0 + first + f) * J + b;
    const D3 p = bone_pos(v, f, b), vel = with_edges(v, f, b, false), an = with_edges(v, f, b, true);
    const D4 q = bone_rot(v, f, b);
    out_pos[o * 3] = (float)p.x; out_pos[o * 3 + 1] = (float)p.y; out_pos[o * 3 + 2] = (float)p.z;
    out_vel[o * 3] = (float)vel.x; out_vel[o * 3 + 1] = (float)vel.y; out_vel[o * 3 + 2] = (float)vel.z;
    out_ang[o * 3] = (float)an.x; out_ang[o * 3 + 1] = (float)an.y; out_ang[o * 3 + 2] = (float)an.z;
    out_rot[o * 4] = (float)q.w; out_rot[o * 4 + 1] = (float)q.x; out_rot[o * 4 + 2] = (float)q.y;
    out_rot[o * 4 + 3] = (float)q.z;
  }
  if (b >= 2) return;
  // preprocess._fk_vel down the chain root -> toe; only the toe's global velocity is kept
  const int toe = (b == 0 ? sk.toe_l : sk.toe_r) + 1;
  int depth = 0;
  for (int k = toe; k > 0; k = sk.parents[k - 1] + 1) ++depth;         // bones above the toe, root excluded
  D4 gr = bone_rot(v, f, 0);
  D3 gv = with_edges(v, f, 0, false), ga = with_edges(v, f, 0, true);
  for (int s = depth - 1; s >= 0; --s) {
    int k = toe;                                                        // the chain's bone s steps above the toe
    for (int u = 0; u < s; ++u) k = sk.parents[k - 1] + 1;
    const D3 rp = qrot(gr, bone_pos(v, f, k));
    gv = add3(add3(qrot(gr, with_edges(v, f, k, false)), cross3(ga, rp)), gv);
    ga = add3(qrot(gr, with_edges(v, f, k, true)), ga);
    gr = qmul(gr, bone_rot(v, f, k));
  }
  ws.toe[(first + f) * 2 + b] = __dsqrt_rn(sumsq3(gv)) < 0.5;
}

// ---- phase 5: contacts --------------------------------------------------------------------------------------------
// median_filter(size=6, mode='nearest') of a boolean row is 1 iff at least 3 of frames clamp(i-3 .. i+2) are set.
__global__ void __launch_bounds__(IG_ROOT_THREADS)
ingest_contacts_kernel(IngestClips cl, IngestWs ws, uint8_t* __restrict__ out_contacts) {
  pdl_trigger();
  pdl_wait();
  const int c = blockIdx.x;
  long long first;
  int F;
  if (!clip_ok(cl, c, first, F)) return;
  const int f = blockIdx.y * IG_ROOT_THREADS + threadIdx.x;
  if (f >= F) return;
  const uint8_t* t = ws.toe + first * 2;
  int n0 = 0, n1 = 0;
  for (int k = f - 3; k <= f + 2; ++k) {
    const int kk = min(max(k, 0), F - 1);
    n0 += t[kk * 2];
    n1 += t[kk * 2 + 1];
  }
  const long long o = (cl.row0 + first + f) * 2;
  out_contacts[o] = n0 >= 3;
  out_contacts[o + 1] = n1 >= 3;
}

// workspace carve-up; with ws.base == nullptr it only sizes
void ingest_layout(Workspace& w, long long N, int J0, IngestWs& ws) {
  ws.lrot = w.take<double>((size_t)N * J0 * 4);
  ws.lpos = w.take<double>((size_t)N * J0 * 3);
  ws.rp_raw = w.take<double>((size_t)N * 3);
  ws.rdir = w.take<double>((size_t)N * 3);
  ws.root_pos = w.take<double>((size_t)N * 3);
  ws.root_rot = w.take<double>((size_t)N * 4);
  ws.toe = w.take<uint8_t>((size_t)N * 2);
}

}  // namespace

extern "C" size_t mocha_ingest_workspace_bytes(long long n_frames, int J) {
  if (n_frames <= 0 || J < 2 || J > IG_MAXJ + 1) return 0;
  Workspace w(nullptr, (size_t)-1);
  IngestWs ws;
  ingest_layout(w, n_frames, J - 1, ws);
  return w.off;
}

extern "C" int mocha_ingest_frames(const double* raw_rot, const double* raw_pos, long long n_frames,
                                   const int64_t* clip_first, const int32_t* clip_frames, const int32_t* clip_order,
                                   int n_clips, int max_clip_frames, const int32_t* parents, const int32_t* joints, int J,
                                   const double* savgol15, const double* savgol31, float* rot, float* pos, float* vel,
                                   float* ang, uint8_t* contacts, long long bank_rows, long long row0, void* workspace,
                                   size_t workspace_bytes, mocha_stream_t stream) {
  MOCHA_CHECK_ARG(parents && joints, "mocha_ingest_frames: null skeleton argument");
  MOCHA_CHECK_ARG(J >= 2 && J <= IG_MAXJ + 1, "mocha_ingest_frames: need 2 <= J <= %d, got %d", IG_MAXJ + 1, J);
  MOCHA_CHECK_ARG(n_frames > 0 && n_clips > 0 && bank_rows > 0 && row0 >= 0,
                  "mocha_ingest_frames: bad sizes n_frames=%lld n_clips=%d bank_rows=%lld row0=%lld", n_frames, n_clips,
                  bank_rows, row0);
  MOCHA_CHECK_ARG(max_clip_frames >= IG_MIN_FRAMES && max_clip_frames <= 65535 * IG_FT,
                  "mocha_ingest_frames: need %d <= max_clip_frames <= %d, got %d", IG_MIN_FRAMES, 65535 * IG_FT,
                  max_clip_frames);
  IngestSkel sk = {};
  sk.J0 = J - 1;
  MOCHA_CHECK_ARG(parents[0] == -1, "mocha_ingest_frames: joint 0 must be the skeleton's root (parent -1)");
  for (int j = 1; j < sk.J0; ++j) {
    MOCHA_CHECK_ARG(parents[j] >= 0 && parents[j] < j, "mocha_ingest_frames: parents[%d] = %d is not an earlier joint", j,
                    parents[j]);
  }
  for (int j = 0; j < sk.J0; ++j) sk.parents[j] = parents[j];
  for (int k = 0; k < 7; ++k) {
    MOCHA_CHECK_ARG(joints[k] >= 0 && joints[k] < sk.J0, "mocha_ingest_frames: joints[%d] = %d outside [0, %d)", k,
                    joints[k], sk.J0);
  }
  sk.spine2 = joints[0]; sk.shoulder_l = joints[1]; sk.shoulder_r = joints[2]; sk.upleg_l = joints[3];
  sk.upleg_r = joints[4]; sk.toe_l = joints[5]; sk.toe_r = joints[6];
  for (int k = 0; k < 5; ++k)
    for (int j = joints[k]; j >= 0; j = sk.parents[j]) sk.fk_mask |= 1u << j;
  MOCHA_CHECK_ARG(raw_rot && raw_pos && clip_first && clip_frames && clip_order && savgol15 && savgol31,
                  "mocha_ingest_frames: null input argument");
  MOCHA_CHECK_ARG(rot && pos && vel && ang && contacts, "mocha_ingest_frames: null bank argument");
  MOCHA_CHECK_ARG(workspace, "mocha_ingest_frames: null workspace");
  Workspace w(workspace, workspace_bytes);
  IngestWs ws;
  ingest_layout(w, n_frames, sk.J0, ws);
  if (w.overflow)
    return set_error(MOCHA_ERR_WORKSPACE, "mocha_ingest_frames: workspace of %zu B, need %zu", workspace_bytes, w.off);
  const IngestClips cl = {reinterpret_cast<const long long*>(clip_first), clip_frames, clip_order, n_clips,
                          max_clip_frames, n_frames, bank_rows, row0};
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned ft = (unsigned)ceil_div(max_clip_frames, IG_FT), rt = (unsigned)ceil_div(max_clip_frames, IG_ROOT_THREADS);
  launch_k(ingest_local_kernel, dim3((unsigned)n_clips, ft), IG_FT * 32, 0, st, raw_rot, raw_pos, cl, sk, ws);
  count_launch();
  MOCHA_LAUNCH_CHECK("ingest_local_kernel");
  launch_k(ingest_unroll_kernel, dim3((unsigned)n_clips, (unsigned)ceil_div(sk.J0, IG_UNROLL_WARPS)), IG_UNROLL_WARPS * 32,
           0, st, cl, sk.J0, ws);
  count_launch();
  MOCHA_LAUNCH_CHECK("ingest_unroll_kernel");
  launch_k(ingest_root_kernel, dim3((unsigned)n_clips, rt), IG_ROOT_THREADS, 0, st, cl, savgol15, savgol31, ws);
  count_launch();
  MOCHA_LAUNCH_CHECK("ingest_root_kernel");
  launch_k(ingest_frames_kernel, dim3((unsigned)n_clips, ft), IG_FT * 32, 0, st, cl, sk, ws, rot, pos, vel, ang);
  count_launch();
  MOCHA_LAUNCH_CHECK("ingest_frames_kernel");
  launch_k(ingest_contacts_kernel, dim3((unsigned)n_clips, rt), IG_ROOT_THREADS, 0, st, cl, ws, contacts);
  count_launch();
  MOCHA_LAUNCH_CHECK("ingest_contacts_kernel");
  return MOCHA_OK;
}
