// Device-side building blocks shared by the step kernels (bd_kernels.cu):
// Bullet's closed-form quaternion helpers, the two arithmetic flavours of the explicit
// dynamics, the reset logic and the per-task observation / reward / termination terms.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "bd_params.h"

namespace bd {

enum { TASK_HOVER = 0, TASK_MULTIHOVER = 1, TASK_SPIRAL = 2,
       // Meetup / Flock / LeaderFollower: rewards couple the drones of an env; one template instantiation
       // (TASK_SWARM) that branches on Params::task (warp-uniform)
       TASK_SWARM = 3, TASK_MEETUP = 3, TASK_FLOCK = 4, TASK_LEADERFOLLOWER = 5 };
enum { MODEL_CF2X = 0, MODEL_CF2P = 1, MODEL_RACE = 2 };
enum { AERO_GND = 1, AERO_DRAG = 2, AERO_DW = 4 };
enum { RESET_FIXED = 0, RESET_PHILOX = 1, RESET_BUFFER = 2 };

// ---------------------------------------------------------------- small maths
__device__ __forceinline__ float  sqrt_(float x)  { return sqrtf(x); }
__device__ __forceinline__ double sqrt_(double x) { return sqrt(x); }
__device__ __forceinline__ float  exp_(float x)  { return expf(x); }
__device__ __forceinline__ double exp_(double x) { return exp(x); }
__device__ __forceinline__ float  atan2_(float y, float x)  { return atan2f(y, x); }
__device__ __forceinline__ double atan2_(double y, double x) { return atan2(y, x); }
__device__ __forceinline__ float  asin_(float x)  { return asinf(x); }
__device__ __forceinline__ double asin_(double x) { return asin(x); }
__device__ __forceinline__ void sincos_(float x, float* s, float* c)  { sincosf(x, s, c); }
__device__ __forceinline__ void sincos_(double x, double* s, double* c) { sincos(x, s, c); }
__device__ __forceinline__ float  abs_(float x)  { return fabsf(x); }
__device__ __forceinline__ double abs_(double x) { return fabs(x); }

__device__ __forceinline__ float4  make4(float a, float b, float c, float d)   { return make_float4(a, b, c, d); }
__device__ __forceinline__ double4 make4(double a, double b, double c, double d) { return make_double4(a, b, c, d); }

template <int BYTES>
__device__ __forceinline__ void cp_async(void* smem_dst, const void* gmem_src) {
  unsigned d = static_cast<unsigned>(__cvta_generic_to_shared(smem_dst));
  if constexpr (BYTES == 16) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(gmem_src) : "memory");
  } else {
    asm volatile("cp.async.ca.shared.global [%0], [%1], %2;\n" ::"r"(d), "l"(gmem_src), "n"(BYTES) : "memory");
  }
}
// the same with an L2 eviction-priority descriptor (createpolicy), see L2Hints
template <int BYTES>
__device__ __forceinline__ void cp_async_hint(void* smem_dst, const void* gmem_src, uint64_t pol) {
  unsigned d = static_cast<unsigned>(__cvta_generic_to_shared(smem_dst));
  if constexpr (BYTES == 16) {
    asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %2;\n" ::"r"(d), "l"(gmem_src), "l"(pol) : "memory");
  } else {
    asm volatile("cp.async.ca.shared.global.L2::cache_hint [%0], [%1], %2, %3;\n" ::"r"(d), "l"(gmem_src), "n"(BYTES), "l"(pol)
                 : "memory");
  }
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;\n" ::: "memory"); }

// ------------------------------------------------------------------- Philox
__device__ __forceinline__ void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
    const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
    c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
}
__device__ __forceinline__ float  u01(uint32_t a, uint32_t, float)  { return (a >> 8) * (1.0f / 16777216.0f); }
__device__ __forceinline__ double u01(uint32_t a, uint32_t b, double) {
  return ((a >> 5) * 67108864.0 + (b >> 6)) * (1.0 / 9007199254740992.0);
}

// ------------------------------------------------- Bullet closed-form helpers
// btMatrix3x3::setRotation == pybullet getMatrixFromQuaternion (BaseAviary.py:836)
template <typename R>
__device__ __forceinline__ void quat_to_mat(R x, R y, R z, R w, R m[9]) {
  const R d = x * x + y * y + z * z + w * w;
  const R s = R(2) / d;
  const R xs = x * s, ys = y * s, zs = z * s;
  const R wx = w * xs, wy = w * ys, wz = w * zs;
  const R xx = x * xs, xy = x * ys, xz = x * zs;
  const R yy = y * ys, yz = y * zs, zz = z * zs;
  m[0] = R(1) - (yy + zz); m[1] = xy - wz;          m[2] = xz + wy;
  m[3] = xy + wz;          m[4] = R(1) - (xx + zz); m[5] = yz - wx;
  m[6] = xz - wy;          m[7] = yz + wx;          m[8] = R(1) - (xx + yy);
}

// btMatrix3x3::getRotation (what getBasePositionAndOrientation returns, :517)
template <typename R>
__device__ __forceinline__ void mat_to_quat(const R m[9], R& x, R& y, R& z, R& w) {
  const R trace = m[0] + m[4] + m[8];
  if (trace > R(0)) {
    R s = sqrt_(trace + R(1));
    w = s * R(0.5);
    s = R(0.5) / s;
    x = (m[7] - m[5]) * s;
    y = (m[2] - m[6]) * s;
    z = (m[3] - m[1]) * s;
  } else {
    const int i = m[0] < m[4] ? (m[4] < m[8] ? 2 : 1) : (m[0] < m[8] ? 2 : 0);
    if (i == 0) {
      R s = sqrt_(m[0] - m[4] - m[8] + R(1));
      x = s * R(0.5); s = R(0.5) / s;
      w = (m[7] - m[5]) * s; y = (m[3] + m[1]) * s; z = (m[6] + m[2]) * s;
    } else if (i == 1) {
      R s = sqrt_(m[4] - m[8] - m[0] + R(1));
      y = s * R(0.5); s = R(0.5) / s;
      w = (m[2] - m[6]) * s; z = (m[7] + m[5]) * s; x = (m[1] + m[3]) * s;
    } else {
      R s = sqrt_(m[8] - m[0] - m[4] + R(1));
      z = s * R(0.5); s = R(0.5) / s;
      w = (m[3] - m[1]) * s; x = (m[2] + m[6]) * s; y = (m[5] + m[7]) * s;
    }
  }
}

template <typename R>
__device__ __forceinline__ void bullet_roundtrip(R& x, R& y, R& z, R& w) {
  R m[9];
  quat_to_mat(x, y, z, w, m);
  mat_to_quat(m, x, y, z, w);
}

// Same map as bullet_roundtrip for float throughput: q/|q| with Bullet's sign rule
// (trace > 0 <=> 4w^2 > 1 -> w >= 0; else the largest diagonal's component >= 0).
__device__ __forceinline__ void fast_canonical(float& x, float& y, float& z, float& w) {
  const float rn = rsqrtf(fmaf(x, x, fmaf(y, y, fmaf(z, z, w * w))));
  x *= rn; y *= rn; z *= rn; w *= rn;
  bool neg;
  if (w * w > 0.25f) {
    neg = w < 0.0f;
  } else {
    const float xx = x * x, yy = y * y, zz = z * z;   // m00 < m11 <=> xx < yy
    const int i = xx < yy ? (yy < zz ? 2 : 1) : (xx < zz ? 2 : 0);
    neg = (i == 0 ? x : (i == 1 ? y : z)) < 0.0f;
  }
  if (neg) { x = -x; y = -y; z = -z; w = -w; }
}

// pybullet getEulerFromQuaternion (:518) incl. its gimbal branches
template <typename R>
__device__ __forceinline__ void quat_to_euler(R x, R y, R z, R w, R& roll, R& pitch, R& yaw) {
  const R sqx = x * x, sqy = y * y, sqz = z * z, squ = w * w;
  const R sarg = R(-2) * (x * z - w * y);
  const R half_pi = R(0.5 * 3.14159265358979323846);
  if (sarg <= R(-0.99999)) {
    roll = R(0); pitch = -half_pi; yaw = R(2) * atan2_(x, -y);
  } else if (sarg >= R(0.99999)) {
    roll = R(0); pitch = half_pi; yaw = R(2) * atan2_(-x, y);
  } else {
    roll = atan2_(R(2) * (y * z + w * x), squ - sqx - sqy + sqz);
    pitch = asin_(sarg);
    yaw = atan2_(R(2) * (x * y + w * z), squ + sqx - sqy - sqz);
  }
}

// `abs(roll) < pi/2 and abs(pitch) < pi/2` (the ground-effect gate, BaseAviary.py:735) without the three inverse
// trigonometric calls per substep: pitch = asin(sarg) is below pi/2 exactly when the gimbal branches are not taken,
// |atan2(ys, xs)| < pi/2 exactly when xs > 0 — except within rounding distance of 90 degrees.  There the reference
// compares the ROUNDED angle with the rounded constant: fl(atan2(ys, xs)) < fl(pi/2) holds iff the exact angle
// pi/2 - xs/|ys| lies below the midpoint of fl(pi/2) and its predecessor, i.e. iff
// xs/|ys| > (pi/2 - fl(pi/2)) + ulp/2 = 6.1232e-17 + 1.1102e-16.  Deciding it in this form (double) reproduces
// numpy / libm without depending on the last bit of the device's atan2 (found by the round-2 gimbal test: a roll
// that reaches pi/2 to 5e-16 after 30 substeps).
template <typename R>
__device__ __forceinline__ bool tilt_below_half_pi(R x, R y, R z, R w) {
  const R sarg = R(-2) * (x * z - w * y);
  if (sarg <= R(-0.99999) || sarg >= R(0.99999)) return false;   // pitch = -+pi/2 exactly
  const R xs = w * w - x * x - y * y + z * z, ys = R(2) * (y * z + w * x);
  if constexpr (sizeof(R) == 8) {
    return xs > R(1.7225464241988331e-16) * abs_(ys);
  }
  if (abs_(xs) <= R(1e-5) * abs_(ys)) {
    R roll, pitch, yaw;
    quat_to_euler(x, y, z, w, roll, pitch, yaw);
    const R half_pi = R(0.5 * 3.14159265358979323846);
    return abs_(roll) < half_pi && abs_(pitch) < half_pi;
  }
  return xs > R(0);
}

// atan2 for the float throughput path: one range reduction to |t| <= tan(pi/8) (through the half-angle identity
// atan(a) = pi/4 + atan((a - 1) / (a + 1)) when a > tan(pi/8), a = min/max), ONE division, a degree-4 minimax
// polynomial in t^2 (max error 3.3e-8 in float arithmetic), octant fix-ups.  |error| < 3e-7 rad overall,
// ~25 instructions against ~55 for atan2f.
__device__ __forceinline__ float atan2_fast(float y, float x) {
  const float ax = fabsf(x), ay = fabsf(y);
  const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
  const bool red = mn > 0.41421356f * mx;
  const float num = red ? mn - mx : mn;
  const float den = fmaxf(red ? mn + mx : mx, 1e-37f);   // atan2(0, 0) = 0
  const float t = __fdividef(num, den);
  const float s = t * t;
  float p = fmaf(s, 0.08044466376304626f, -0.13874448835849762f);
  p = fmaf(s, p, 0.1997736096382141f);
  p = fmaf(s, p, -0.33332937955856323f);
  p = fmaf(s * t, p, t);
  float r = red ? 0.78539816339744831f + p : p;
  r = ay > ax ? 1.57079632679489662f - r : r;
  r = x < 0.f ? 3.14159265358979324f - r : r;
  return copysignf(r, y);
}

// quat_to_euler with atan2_fast on the regular branch (float throughput kernel)
__device__ __forceinline__ void quat_to_euler_fast(float x, float y, float z, float w, float& roll, float& pitch, float& yaw) {
  const float sqx = x * x, sqy = y * y, sqz = z * z, squ = w * w;
  const float sarg = -2.f * (x * z - w * y);
  const float half_pi = 1.57079632679489662f;
  if (sarg <= -0.99999f) {
    roll = 0.f; pitch = -half_pi; yaw = 2.f * atan2f(x, -y);
  } else if (sarg >= 0.99999f) {
    roll = 0.f; pitch = half_pi; yaw = 2.f * atan2f(-x, y);
  } else {
    roll = atan2_fast(2.f * (y * z + w * x), squ - sqx - sqy + sqz);
    pitch = asinf(sarg);
    yaw = atan2_fast(2.f * (x * y + w * z), squ + sqx - sqy - sqz);
  }
}

// pybullet getQuaternionFromEuler (:488), normalised
template <typename R>
__device__ __forceinline__ void euler_to_quat(R roll, R pitch, R yaw, R& x, R& y, R& z, R& w) {
  R sp, cp, st, ct, ss, cs;
  sincos_(roll / R(2), &sp, &cp);
  sincos_(pitch / R(2), &st, &ct);
  sincos_(yaw / R(2), &ss, &cs);
  x = sp * ct * cs - cp * st * ss;
  y = cp * st * cs + sp * ct * ss;
  z = cp * ct * ss - sp * st * cs;
  w = cp * ct * cs + sp * st * ss;
  const R n = sqrt_(x * x + y * y + z * z + w * w);
  x /= n; y /= n; z /= n; w /= n;
}

// BaseAviary._integrateQ (:879-892): q <- cos(th) q + sin(th)/|w| Lambda(w) q
template <typename R>
__device__ __forceinline__ void integrate_q_exact(R& x, R& y, R& z, R& w, R p, R q, R r, R dt) {
  const R n = sqrt_(p * p + q * q + r * r);
  if (n <= R(1e-8)) return;                       // np.isclose(norm, 0): atol 1e-8
  R s, c;
  sincos_(n * dt / R(2), &s, &c);
  const R k = R(2) / n * R(0.5) * s;
  const R nx = c * x + k * (r * y - q * z + p * w);
  const R ny = c * y + k * (-r * x + p * z + q * w);
  const R nz = c * z + k * (q * x - p * y + r * w);
  const R nw = c * w + k * (-p * x - q * y - r * z);
  x = nx; y = ny; z = nz; w = nw;
}

// float fast path: cos(th) and sin(th)/|w| = (dt/2) sinc(th) as polynomials in th^2
__device__ __forceinline__ void integrate_q_fast(float& x, float& y, float& z, float& w,
                                                 float p, float q, float r, float half_dt) {
  const float n2 = fmaf(p, p, fmaf(q, q, r * r));
  const float u = n2 * half_dt * half_dt;         // th^2
  float c, k;
  if (u <= 0.25f) {
    c = fmaf(u, fmaf(u, fmaf(u, fmaf(u, 2.4801587e-5f, -1.3888889e-3f), 4.1666668e-2f), -0.5f), 1.0f);
    k = half_dt * fmaf(u, fmaf(u, fmaf(u, fmaf(u, 2.7557319e-6f, -1.9841270e-4f), 8.3333338e-3f),
                                    -1.6666667e-1f), 1.0f);
  } else {
    const float n = sqrtf(n2);
    float s;
    sincosf(n * half_dt, &s, &c);
    k = s / n;
  }
  const float nx = fmaf(k, fmaf(r, y, fmaf(-q, z, p * w)), c * x);
  const float ny = fmaf(k, fmaf(-r, x, fmaf(p, z, q * w)), c * y);
  const float nz = fmaf(k, fmaf(q, x, fmaf(-p, y, r * w)), c * z);
  const float nw = fmaf(k, -fmaf(p, x, fmaf(q, y, r * z)), c * w);
  x = nx; y = ny; z = nz; w = nw;
}

// --------------------------------------------------------------- reset logic
template <typename R>
struct Drone {
  R px, py, pz, qx, qy, qz, qw, vx, vy, vz, wx, wy, wz, tx, ty, tz;
};

// INIT pose of (env, drone) -> freshly reset drone (BaseAviary._housekeeping :451-505
// + kinematic refresh :509-519) and its 12 kinematic observation entries.
template <typename R, int TASK>
__device__ __forceinline__ void reset_drone(const Params<R>& P, int env, int drone, const R* cand,
                                            Drone<R>& d, float kin[12]) {
  const long long ib = (long long)env * P.init_env_stride + drone * 3;
  R ix = P.init_xyz[ib], iy = P.init_xyz[ib + 1], iz = P.init_xyz[ib + 2];
  if (TASK == TASK_MULTIHOVER && cand != nullptr) { ix = cand[0]; iy = cand[1]; iz = cand[2]; }
  d.px = ix; d.py = iy; d.pz = iz;
  euler_to_quat(P.init_rpy[ib], P.init_rpy[ib + 1], P.init_rpy[ib + 2], d.qx, d.qy, d.qz, d.qw);
  bullet_roundtrip(d.qx, d.qy, d.qz, d.qw);
  d.vx = d.vy = d.vz = R(0);
  d.wx = d.wy = d.wz = R(0);
  if (TASK == TASK_HOVER) { d.tx = R(0); d.ty = R(0); d.tz = R(1); }                 // HoverAviary.py:51
  else if (TASK == TASK_MULTIHOVER) { d.tx = ix; d.ty = iy; d.tz = iz + R(1) / R(drone + 1); }  // :72,106
  else { d.tx = d.ty = d.tz = R(0); }
  R roll, pitch, yaw;
  quat_to_euler(d.qx, d.qy, d.qz, d.qw, roll, pitch, yaw);
  kin[0] = (float)d.px; kin[1] = (float)d.py; kin[2] = (float)d.pz;
  kin[3] = (float)roll; kin[4] = (float)pitch; kin[5] = (float)yaw;
  kin[6] = kin[7] = kin[8] = kin[9] = kin[10] = kin[11] = 0.0f;
}

// MultiHoverAviary.reset (:83-102) for one env, run by its leader thread:
// ORIGINAL_INIT_XYZS + U(-0.25,0.25)^3, z clipped to [0.1,1], redraw until every
// pair is >= 0.5 m apart.  `cand` = shared-memory rows of this env's M drones.
// The reference loops forever when no draw can succeed; here kMaxJitterTries
// draws, then the un-jittered layout (documented deviation, DESIGN.md).
template <typename R>
__device__ void sample_jitter(const Params<R>& P, int env, int total_steps, int epoch, R* cand) {
  const int M = P.M;
  const long long ib = (long long)env * P.init_env_stride;
  for (int attempt = 0; attempt <= kMaxJitterTries; ++attempt) {
    const bool last = attempt == kMaxJitterTries;
    for (int i = 0; i < M; ++i) {
      R j[3] = {R(0), R(0), R(0)};
      if (!last) {
        if (P.reset_mode == RESET_BUFFER && P.jitter != nullptr) {
          const long long jb = ((long long)env * M + i) * 3;
          j[0] = P.jitter[jb]; j[1] = P.jitter[jb + 1]; j[2] = P.jitter[jb + 2];
        } else {
          uint32_t c[4] = {(uint32_t)env, (uint32_t)total_steps + P.philox_base, (uint32_t)(attempt * M + i), (uint32_t)epoch << 1};
          uint32_t c2[4] = {c[0], c[1], c[2], c[3] | 1u};
          philox4x32_10(c, (uint32_t)P.seed, (uint32_t)(P.seed >> 32));
          philox4x32_10(c2, (uint32_t)P.seed, (uint32_t)(P.seed >> 32));
          j[0] = R(-0.25) + R(0.5) * u01(c[0], c[1], R(0));
          j[1] = R(-0.25) + R(0.5) * u01(c[2], c[3], R(0));
          j[2] = R(-0.25) + R(0.5) * u01(c2[0], c2[1], R(0));
        }
      }
      R z = P.init_xyz[ib + i * 3 + 2] + j[2];
      z = z < R(0.1) ? R(0.1) : (z > R(1.0) ? R(1.0) : z);
      cand[i * 3 + 0] = P.init_xyz[ib + i * 3 + 0] + j[0];
      cand[i * 3 + 1] = P.init_xyz[ib + i * 3 + 1] + j[1];
      cand[i * 3 + 2] = z;
    }
    if (last || P.reset_mode == RESET_BUFFER) return;
    bool ok = true;
    for (int a = 0; a < M && ok; ++a)
      for (int b = a + 1; b < M; ++b) {
        const R dx = cand[a * 3] - cand[b * 3], dy = cand[a * 3 + 1] - cand[b * 3 + 1],
                dz = cand[a * 3 + 2] - cand[b * 3 + 2];
        if (sqrt_(dx * dx + dy * dy + dz * dz) < R(0.5)) { ok = false; break; }
      }
    if (ok) return;
  }
}

// --------------------------------------------------------------- task maths
template <typename R>
__device__ __forceinline__ void spiral_reference(const Params<R>& P, int step_counter, int drone,
                                                 R ref_p[3], R ref_v[3], R& sphi, R& cphi) {
  const R t = (R)((double)step_counter / P.pyb_freq);                            // SpiralAviary.py:84
  const R phase = P.sp_omega * t + R(2) * R(3.14159265358979323846) * R(drone) / R(P.M);
  sincos_(phase, &sphi, &cphi);
  ref_p[0] = P.sp_cx + P.sp_R * cphi;
  ref_p[1] = P.sp_cy + P.sp_R * sphi;
  ref_p[2] = R(0.3) + P.sp_vz * t;
  ref_v[0] = -P.sp_R * P.sp_omega * sphi;
  ref_v[1] = P.sp_R * P.sp_omega * cphi;
  ref_v[2] = P.sp_vz;
}

}  // namespace bd

namespace bd {

// ---------------------------------------------------------------------------
// Fast float flavour of S substeps (BaseAviary.py:343-374 with _dynamics :815-877).
// `onep[k]` = fl32(1 + 0.05 a_k) per motor, i.e. rpm_k / HOVER_RPM as numpy rounds it.
//   rpm_k = H (1 + s_k)  =>  rpm_k^2 = H^2 (1 + u_k),  u_k = s_k (2 + s_k).  With
//   4 KF H^2 = m g (BaseAviary.py:118) the hover terms cancel analytically, which
//   removes the float32 cancellation in thrust - gravity and in the torque mixes:
//   thrust/m = g (1 + e), e = sum(u)/4;  f_k = (m g / 4)(1 + u_k);  KM rpm_k^2 = KM H^2 (1 + u_k)
// Per substep only the rotation's third column is formed; the full matrix once, for the
// world angular velocity R_old w_new (:873) of the last substep.
// ---------------------------------------------------------------------------
// DW: pairwise downwash (BaseAviary.py:798-804) for envs that are lane groups of M (M | 32): the
// substep-start positions of the group's other drones arrive by warp shuffle (Jacobi snapshot,
// no shared memory, no barrier); the body-z force enters as F R[:,2] / m.
// MODE 0: plain DYN.  MODE 1: + downwash only.  MODE 2: any combination of ground effect / drag / downwash, chosen
// at run time by P.aero (warp-uniform).  An env is M consecutive lanes starting at `group_base` (a warp holds 32 / M whole
// envs; left-over lanes idle); `drone` = lane - group_base.  `last_sum` = sum over the motors of
// fl32(1 + 0.05 a) of the PREVIOUS control step (0 right after a reset): the drag model reads last_clipped_action,
// which during the first substep is still the previous step's (BaseAviary.py:359,372).
//   ground effect (:739-742): f_k <- f_k (1 + c_k), c_k = GND (r_prop / 4 h_k)^2, h_k = max(z + R20 x_k + R21 y_k, clip);
//       (1 + u_k)(1 + c_k) = 1 + u_k + e_k with e_k = (1 + u_k) c_k: thrust/m gains (g/4) sum e_k, the roll / pitch
//       mixes see u_k + e_k, the yaw torque (KM rpm^2) is unchanged; gated by |roll|, |pitch| < pi/2
//   drag (:773-774): F_world += k (.) v, k = -DRAG sum_k 2 pi rpm_k / 60, v = velocity at the start of the substep
// Single-instruction approximations for the pair terms of the fast flavour: `__fdividef` / `__expf` wrap MUFU.RCP / MUFU.EX2
// in denormal-range rescaling (a compare, two predicated multiplies and a select each) because this library is not built
// with flush-to-zero; in the O(M^2) downwash loop that is a fifth of the instructions.  Forces below 1e-38 N may flush.
__device__ __forceinline__ float rcp_ftz(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float ex2_ftz(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

template <int MODE>
__device__ __forceinline__ void fast_substeps(const Params<float>& P, Drone<float>& d, const float onep[4],
                                              float& avx, float& avy, float& avz, int group_base = 0, int drone = 0,
                                              float last_sum = 0.f) {
  const float dt = P.dt;
  float u[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float sk = onep[k] - 1.0f;                  // exact (Sterbenz)
    u[k] = sk * (2.0f + sk);
  }
  const bool gnd = (MODE == 2) && (P.aero & AERO_GND), drag = (MODE == 2) && (P.aero & AERO_DRAG);
  const bool dw = (MODE == 1) || ((MODE == 2) && (P.aero & AERO_DW));
  const float qf = 0.25f * P.gravity;                   // KF H^2
  const float qm = P.km * (P.hover_rpm * P.hover_rpm);  // KM H^2
  float tz = qm * ((-u[0] + u[1]) + (-u[2] + u[3]));
  float tx, ty;
  if (P.model == 0) { tx = -qf * ((u[0] + u[1]) - (u[2] + u[3])) * P.arm; ty = qf * ((-u[0] + u[1]) + (u[2] - u[3])) * P.arm; }
  else if (P.model == 1) { tx = qf * (u[1] - u[3]) * P.arm; ty = qf * (-u[0] + u[2]) * P.arm; }
  else { tx = qf * ((u[0] + u[1]) - (u[2] + u[3])) * P.arm; ty = qf * ((-u[0] + u[1]) + (u[2] - u[3])) * P.arm; tz = -tz; }
  const float kx = dt * P.ijx * tx, ky = dt * P.ijy * ty, kz = dt * P.ijz * tz;
  const float gx = dt * P.ijx * (P.jz - P.jy), gy = dt * P.ijy * (P.jx - P.jz), gz = dt * P.ijz * (P.jy - P.jx);
  const float e4 = 0.25f * ((u[0] + u[1]) + (u[2] + u[3]));
  const float cg = dt * P.gravity * P.inv_m;            // dt g
  const float c1 = cg * (1.0f + e4), c2 = cg * e4, c3 = -2.0f * cg;
  const float half_dt = 0.5f * dt;
  // drag factors dt k / m per axis: previous step's rpm in the first substep, this step's afterwards
  const float kd = -6.28318530717958647692f / 60.0f * P.hover_rpm * dt * P.inv_m;
  const float cur_sum = (onep[0] + onep[1]) + (onep[2] + onep[3]);
  // downwash constants of the power-of-two pair loop (see there)
  const float dwa = -0.0625f * P.dw1 * (P.prop_radius * P.prop_radius);
  const float dw2s = 1.17741002251547469101f * P.dw2, dw3s = 1.17741002251547469101f * P.dw3;   // / sqrt(log2(e) / 2)
#pragma unroll 1
  for (int s = 0; s < P.S; ++s) {
    const float x = d.qx, y = d.qy, z = d.qz, w = d.qw;   // unit up to rounding
    const float xxyy = fmaf(x, x, y * y);
    const float r02 = 2.0f * fmaf(x, z, w * y), r12 = 2.0f * fmaf(y, z, -w * x),
                r22 = fmaf(-2.0f, xxyy, 1.0f);
    float c1s = c1, c2s = c2, kxs = kx, kys = ky;
    float dvx = d.vx, dvy = d.vy, dvz = d.vz;
    if constexpr (MODE == 2) {
      if (gnd && tilt_below_half_pi(x, y, z, w)) {
        const float r20 = 2.0f * fmaf(x, z, -w * y), r21 = 2.0f * fmaf(y, z, w * x);
        float e[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          float h = d.pz + fmaf(r20, P.prop_x[k], r21 * P.prop_y[k]);
          h = fmaxf(h, P.gnd_h_clip);
          const float ratio = P.prop_radius * rcp_ftz(4.0f * h);
          // products that feed sums — and the sum 1 + u, whose u is itself a product — are rounded on their own (the _rn
          // intrinsics are never contracted): whether a multiply is fused into a following add depends on the surrounding kernel, and the one-launch K-step kernel must
          // reproduce the per-step kernel bit for bit
          e[k] = __fmul_rn(__fadd_rn(1.0f, u[k]), __fmul_rn(__fmul_rn(P.gnd_coeff, ratio), ratio));
        }
        const float es = __fmul_rn(cg * 0.25f, (e[0] + e[1]) + (e[2] + e[3]));
        c1s += es;
        c2s += es;
        float ex, ey;
        if (P.model == 0) { ex = -qf * ((e[0] + e[1]) - (e[2] + e[3])) * P.arm; ey = qf * ((-e[0] + e[1]) + (e[2] - e[3])) * P.arm; }
        else if (P.model == 1) { ex = qf * (e[1] - e[3]) * P.arm; ey = qf * (-e[0] + e[2]) * P.arm; }
        else { ex = qf * ((e[0] + e[1]) - (e[2] + e[3])) * P.arm; ey = qf * ((-e[0] + e[1]) + (e[2] - e[3])) * P.arm; }
        kxs = fmaf(dt * P.ijx, ex, kx);
        kys = fmaf(dt * P.ijy, ey, ky);
      }
      if (drag) {
        const float sum = kd * (s == 0 ? last_sum : cur_sum);
        dvx = fmaf(sum * P.drag_xy, d.vx, d.vx);
        dvy = fmaf(sum * P.drag_xy, d.vy, d.vy);
        dvz = fmaf(sum * P.drag_z, d.vz, d.vz);
      }
    }
    if constexpr (MODE != 0) {
      if (dw) {
        // Every unordered pair is evaluated ONCE: of two drones only the lower one feels the other's downwash (:801,
        // dz > 0), and the force depends on |dz| and the horizontal distance alone — so the lane that meets partner
        // drone + o computes f(|dz|, dxy^2) and keeps it (partner above me) or hands it to the partner (partner below
        // me) through one more shuffle; offsets 1 .. M/2 cover all pairs (for even M the offset M/2 is visited from both
        // ends: the lower-indexed drone owns it).  Half the exp / divide work of a loop over all M - 1 partners
        // (config-5 shape, M = 16: 493 -> see profiles/README.md), identical values, different summation order.
        const int M = P.M;
        float fdw = 0.f;
        const int half = M >> 1;
        if ((M & (M - 1)) == 0) {
          // Power-of-two teams (the tile kernel's M = 2 .. 32; configs[4]: 16): the loop was 46 instructions per pair (now 31.5), a
          // quarter of them lane arithmetic — an env is an aligned group of M lanes, so the shuffle's `width` does the
          // modulo (source lane drone + o, hand-back lane drone - o + M, no compare / select / add per index).  Constants
          // are folded (alpha = dw1 (R / 4 dz)^2 = c_a / dz^2; exp(-(dxy / beta)^2 / 2) = 2^-(dxy / beta')^2 with beta' =
          // beta / sqrt(log2(e) / 2), its two coefficients computed once per step) and the three conditions are three
          // chained predicates: "within 10 m" (and, for the doubly visited offset M / 2, "I own this pair"), "partner
          // above me" and "partner below me".
          const bool owner = drone < half;
          auto pair = [&](int o, bool last) {
            const float oz = __shfl_sync(0xffffffffu, d.pz, drone + o, M), ox = __shfl_sync(0xffffffffu, d.px, drone + o, M),
                        oy = __shfl_sync(0xffffffffu, d.py, drone + o, M);
            const float dz = oz - d.pz, dx = ox - d.px, dy = oy - d.py;
            const float adz = fabsf(dz);
            const float dxy2 = fmaf(dx, dx, dy * dy);
            const float r = rcp_ftz(adz);
            const float rb = rcp_ftz(fmaf(dw2s, adz, dw3s));
            const float f = ((r * r) * dwa) * ex2_ftz(-dxy2 * (rb * rb));      // < 0; inf / nan when dz == 0: never selected
            const bool near = (dxy2 < 100.f) && (!last || owner);                // :801 (delta_xy < 10)
            const float mine = (near && dz > 0.f) ? f : 0.f;                     // the partner is above me
            const float theirs = (near && dz < 0.f) ? f : 0.f;                   // the partner is below me: its force
            fdw += mine + __shfl_sync(0xffffffffu, theirs, drone - o + M, M);
          };
#pragma unroll 2
          for (int o = 1; o < half; ++o) pair(o, false);      // (four pairs in flight, one unified loop: 437 vs 431 us, 80 registers)
          if (half >= 1) pair(half, true);
        } else {
#pragma unroll 2
          for (int o = 1; o <= half; ++o) {
            int t = drone + o;
            t -= (t >= M) ? M : 0;
            int b = drone - o;
            b += (b < 0) ? M : 0;
            const int src = group_base + t;
            const float ox = __shfl_sync(0xffffffffu, d.px, src), oy = __shfl_sync(0xffffffffu, d.py, src),
                        oz = __shfl_sync(0xffffffffu, d.pz, src);
            const float dz = oz - d.pz, dx = ox - d.px, dy = oy - d.py;
            const float adz = fabsf(dz);
            const float dxy2 = fmaf(dx, dx, dy * dy);
            const float ratio = P.prop_radius * rcp_ftz(4.0f * adz);
            const float alpha = P.dw1 * ratio * ratio;
            const float beta = fmaf(P.dw2, adz, P.dw3);
            const float q2 = dxy2 * rcp_ftz(beta * beta);
            float f = -alpha * ex2_ftz(-0.72134752044448f * q2);          // exp(-q2 / 2) = 2^(-q2 log2(e) / 2)
            const bool mine_to_count = (2 * o != M) || (drone < half);     // the doubly visited offset: one owner
            if (!(adz > 0.f && dxy2 < 100.f && mine_to_count)) f = 0.f;       // :801 (delta_xy < 10)
            const float theirs = dz < 0.f ? f : 0.f;                          // the partner is below me
            const float recv = __shfl_sync(0xffffffffu, theirs, group_base + b);
            fdw += (dz > 0.f ? f : 0.f) + recv;
          }
        }
        const float k = dt * P.inv_m * fdw;                       // dt F / m along R[:,2]
        c1s += k;
        c2s += k;
      }
    }
    // a = g [(1+e) R[:,2] - e_z] (+ F_dw R[:,2] / m);  (1+e) r22 - 1 = e r22 - 2 (x^2 + y^2)
    d.vx = fmaf(c1s, r02, dvx);
    d.vy = fmaf(c1s, r12, dvy);
    d.vz = fmaf(c2s, r22, fmaf(c3, xxyy, dvz));
    const float owx = d.wx, owy = d.wy, owz = d.wz;
    d.wx = fmaf(-gx, owy * owz, owx + kxs);
    d.wy = fmaf(-gy, owz * owx, owy + kys);
    d.wz = fmaf(-gz, owx * owy, owz + kz);
    d.px = fmaf(dt, d.vx, d.px);
    d.py = fmaf(dt, d.vy, d.py);
    d.pz = fmaf(dt, d.vz, d.pz);
    if (s == P.S - 1) {
      const float r00 = fmaf(-2.0f, fmaf(y, y, z * z), 1.0f), r01 = 2.0f * fmaf(x, y, -w * z);
      const float r10 = 2.0f * fmaf(x, y, w * z), r11 = fmaf(-2.0f, fmaf(x, x, z * z), 1.0f);
      const float r20 = 2.0f * fmaf(x, z, -w * y), r21 = 2.0f * fmaf(y, z, w * x);
      avx = fmaf(r00, d.wx, fmaf(r01, d.wy, r02 * d.wz));
      avy = fmaf(r10, d.wx, fmaf(r11, d.wy, r12 * d.wz));
      avz = fmaf(r20, d.wx, fmaf(r21, d.wy, r22 * d.wz));
    }
    integrate_q_fast(d.qx, d.qy, d.qz, d.qw, d.wx, d.wy, d.wz, half_dt);
  }
  // Bullet's per-substep round trip (normalise + sign rule, :509-519) commutes with the
  // quaternion step, which is linear in q and norm-preserving: canon(step(canon(q))) ==
  // canon(step(q)).  Applying it once per control step gives the same quaternion up to float
  // rounding (|q|^2 drifts by ~1e-7 over 8 substeps) and saves ~10 % of the instructions.
  fast_canonical(d.qx, d.qy, d.qz, d.qw);
}

// Spiral env's 11 extra observation entries (SpiralAviary.py:120-146)
template <typename R>
__device__ __forceinline__ void spiral_extras(float* ext, const Drone<R>& d, const R rp[3], const R rv[3],
                                              R sphi, R cphi) {
  // SpiralAviary.py:130: "vel" = state[3:6] = quaternion x,y,z (reference quirk)
  ext[0] = (float)(rp[0] - d.px); ext[1] = (float)(rp[1] - d.py); ext[2] = (float)(rp[2] - d.pz);
  ext[3] = (float)(rv[0] - d.qx); ext[4] = (float)(rv[1] - d.qy); ext[5] = (float)(rv[2] - d.qz);
  ext[6] = (float)sphi; ext[7] = (float)cphi;
  ext[8] = (float)rv[0]; ext[9] = (float)rv[1]; ext[10] = (float)rv[2];
}

// Per-drone reward contribution and termination/truncation condition bits of the task
// (bit0: terminated condition, bit1: truncated condition), plus the spiral extras.
//   HoverAviary.py:77-117, MultiHoverAviary.py:128-241, SpiralAviary.py:150-191
template <typename R, int TASK>
__device__ __forceinline__ void task_terms(const Params<R>& P, const Drone<R>& d, R roll, R pitch,
                                           int step_counter, int drone, float* ext, R& contrib, int& flags) {
  contrib = R(0);
  flags = 0;
  if (TASK == 0) {
    const R ex = d.tx - d.px, ey = d.ty - d.py, ez = d.tz - d.pz;
    const R dist = sqrt_(ex * ex + ey * ey + ez * ez);
    const R d2 = dist * dist;
    const R r = R(2) - d2 * d2;                                                  // HoverAviary.py:78
    contrib = r > R(0) ? r : R(0);
    if (dist < R(.0001)) flags |= 1;                                             // :93
    if (abs_(d.px) > R(1.5) || abs_(d.py) > R(1.5) || d.pz > R(2.0) ||
        abs_(roll) > R(.4) || abs_(pitch) > R(.4)) flags |= 2;                   // :109-111
  } else if (TASK == 1) {
    const R ex = d.px - d.tx, ey = d.py - d.ty;
    const R err_xy = sqrt_(ex * ex + ey * ey);
    const R err_z = d.pz - d.tz;
    const R vel_z = d.vz;
    const R r_xy = R(1) / (R(1) + err_xy);
    const R r_z = exp_(R(-7.5) * abs_(err_z));
    const R r_vel = abs_(err_z) < R(0.2) ? R(-1.5) * (vel_z * vel_z) : R(0);
    const R bonus = (err_xy < R(0.03) && abs_(err_z) < R(0.03) && abs_(vel_z) < R(0.03)) ? R(0.5) : R(0);
    contrib = ((r_xy + r_z) + r_vel) + bonus;                                    // MultiHoverAviary.py:173-179
    if (d.pz < R(0.03)) flags |= 1;                                              // :226
    if (abs_(roll) > R(1.2) || abs_(pitch) > R(1.2)) flags |= 1;                 // :231
    if (abs_(d.px) > R(3.0) || abs_(d.py) > R(3.0)) flags |= 1;                  // :236
  } else {
    R rp[3], rv[3], sphi, cphi;
    spiral_reference(P, step_counter, drone, rp, rv, sphi, cphi);
    spiral_extras(ext, d, rp, rv, sphi, cphi);
    const R dpx = d.px - rp[0], dpy = d.py - rp[1], dpz = d.pz - rp[2];
    const R npos = sqrt_(dpx * dpx + dpy * dpy + dpz * dpz);
    const R dvx = d.qx - rv[0], dvy = d.qy - rv[1], dvz = d.qz - rv[2];           // :156 (same quirk)
    const R nvel = sqrt_(dvx * dvx + dvy * dvy + dvz * dvz);
    const R r_pos = exp_(R(-4.0) * (npos * npos));
    const R r_vel = exp_(R(-2.0) * (nvel * nvel));
    R r_tan = R(0);
    const R rx = d.px - P.sp_cx, ry = d.py - P.sp_cy;
    const R nr = sqrt_(rx * rx + ry * ry);
    if (nr > R(1e-3)) {
      const R tgx = -(ry / nr), tgy = rx / nr;
      const R nv = sqrt_(d.qx * d.qx + d.qy * d.qy);
      if (nv > R(1e-3)) {
        const R dot = (d.qx / nv) * tgx + (d.qy / nv) * tgy;
        r_tan = dot > R(0) ? dot : R(0);
      }
    }
    contrib = (R(1.0) * r_pos + R(2.0) * r_vel) + R(1.0) * r_tan;               // :179
    if (d.pz < R(0.05) || d.pz > R(3.0)) flags |= 1;                             // :188-190
  }
}

// Swarm tasks: per-drone part of the coupled reward / flags.  `ep`, `ev` = final positions / velocities
// of this env's M drones in shared memory.  flags bit1: truncation bound hit, bit2: my pair has not met.
//   MeetupAviary.py:74-154, FlockAviary.py:75-189, LeaderFollowerAviary.py:72-145
template <typename R>
__device__ __forceinline__ void swarm_terms(const Params<R>& P, const R* ep, const R* ev, int M, int drone,
                                            const Drone<R>& d, R roll, R pitch, R& contrib, R& aux, int& flags) {
  contrib = R(0); aux = R(0); flags = 0;
  const bool tilt = abs_(roll) > R(.4) || abs_(pitch) > R(.4);
  if (P.task == TASK_MEETUP) {
    if (drone < M / 2) {                                                         // :88-93
      const R* q = ep + (size_t)(M - 1 - drone) * 3;
      const R dx = d.px - q[0], dy = d.py - q[1], dz = d.pz - q[2];
      const R dist = sqrt_(dx * dx + dy * dy + dz * dz);
      contrib = (R(-1) * (dist * dist)) * R(2);
      if (dist > R(0.1)) flags |= 4;                                             // :115-118
    }
    if (abs_(d.px) > R(5.0) || abs_(d.py) > R(5.0) || d.pz > R(3.0) || d.pz < R(0.1) || tilt) flags |= 2;   // :142-147
  } else if (P.task == TASK_LEADERFOLLOWER) {
    if (drone == 0) {                                                            // :88
      const R ex = R(0) - d.px, ey = R(0) - d.py, ez = R(0.5) - d.pz;
      const R n = sqrt_(ex * ex + ey * ey + ez * ez);
      contrib = R(-1) * (n * n);
    } else {                                                                     // :91-97: target (x_i, y_i, z_leader)
      const R dz = ep[2] - d.pz;
      const R n = sqrt_(dz * dz);
      contrib = -(R(1) / R(M)) * (n * n);
    }
    if (abs_(d.px) > R(2.0) || abs_(d.py) > R(2.0) || d.pz > R(2.0) || tilt) flags |= 2;   // :135-140
  } else {                                                                       // Flock
    const R eps = R(1e-3);
    const R ni = sqrt_(d.vx * d.vx + d.vy * d.vy + d.vz * d.vz);
    R ali = R(0), sp = R(0);
    bool first = true;
    for (int j = 0; j < M; ++j) {
      if (j == drone) continue;
      const R* pj = ep + (size_t)j * 3;
      const R* vj = ev + (size_t)j * 3;
      const R nj = sqrt_(vj[0] * vj[0] + vj[1] * vj[1] + vj[2] * vj[2]);
      const R dot = d.vx * vj[0] + d.vy * vj[1] + d.vz * vj[2];
      ali += dot / (ni + eps) / (nj + eps);                                      // :98-103
      const R dx = pj[0] - d.px, dy = pj[1] - d.py, dz = pj[2] - d.pz;
      const R dist = sqrt_(dx * dx + dy * dy + dz * dz);
      sp = (first || dist < sp) ? dist : sp;                                     // :121-125 nearest neighbour
      first = false;
    }
    contrib = ali;
    aux = sp;
    if (abs_(d.px) > R(10.0) || abs_(d.py) > R(10.0) || d.pz > R(10.0) || tilt) flags |= 2;   // :181-184
  }
}

// env-level reward of the swarm tasks from the per-drone parts (run by the env's first drone)
template <typename R>
__device__ __forceinline__ R swarm_reward(const Params<R>& P, int M, const R* part, const R* aux, const R* ev) {
  R sum = R(0);
  for (int i = 0; i < M; ++i) sum += part[i];
  if (P.task != TASK_FLOCK) return sum;
  R cx = R(0), cy = R(0), cz = R(0);
  for (int i = 0; i < M; ++i) { cx += ev[i * 3]; cy += ev[i * 3 + 1]; cz += ev[i * 3 + 2]; }
  cx /= R(M); cy /= R(M); cz /= R(M);                                            // :111-112 centre-of-flock velocity
  const R speed = sqrt_(cx * cx + cy * cy + cz * cz);
  if (M == 1) return speed;                                                      // ali = spacing terms = 0 (:106-108,115-117)
  const R ali = sum / R(M * (M - 1));
  R avg = R(0);
  for (int i = 0; i < M; ++i) avg += aux[i];
  avg /= R(M);
  R var = R(0);
  for (int i = 0; i < M; ++i) { const R e = aux[i] - avg; var += e * e; }
  var /= R(M);                                                                   // np.var (:131)
  R pen = R(0);
  if (!(R(1.0) < avg && avg < R(3.0))) {                                         // :137-141
    const R a = abs_(avg - R(1.0)), b = abs_(avg - R(3.0));
    pen = a < b ? a : b;
  }
  return ((ali + speed) - pen) - var;                                            // :145
}

// ------------------------------------------------ DSL PID controller (ActionType.PID / VEL / ONE_D_PID)
// BaseRLAviary._preprocessAction (:193-235) turns these actions into motor RPMs through one
// DSLPIDControl per drone (control/DSLPIDControl.py:82-246).  The controller is always built for
// CF2X (BaseRLAviary.py:76): CF2X gains, mixer, mass and kf whatever airframe the env flies.
// Its memory — integral position error, integral attitude error, last rpy — is 9 numbers per
// drone, kept in plane-major device memory (ctrl[k * n_total + g]); planes 9..12 hold the
// commanded RPMs (`last_clipped_action`, BaseAviary.py:372, read by the drag model and bd_get_state).
enum { ACT_RPM = 0, ACT_ONE_D_RPM = 1, ACT_PID = 2, ACT_VEL = 3, ACT_ONE_D_PID = 4 };
constexpr int kCtrlPlanes = 13;

template <typename R>
__device__ __forceinline__ R clip_(R x, R lo, R hi) { return x < lo ? lo : (x > hi ? hi : x); }

// target position / yaw / velocity from the raw action (BaseRLAviary.py:193-235).
// `af` = the action as float (always valid), `ad` = the action as double when the caller passed
// doubles (`from_double`); numpy keeps float32 actions in float32 through the VEL unit-vector
// and speed arithmetic (norm = sqrt(sdot): float products summed in double, rounded to float).
template <typename R>
__device__ __forceinline__ void pid_targets(const Params<R>& P, const Drone<R>& d, R yaw, const float af[4],
                                            const double ad[4], bool from_double, R tp[3], R& tyaw, R tv[3]) {
  tp[0] = d.px; tp[1] = d.py; tp[2] = d.pz;
  tv[0] = tv[1] = tv[2] = R(0);
  tyaw = R(0);
  if (P.act_type == ACT_PID) {                      // :193-206 with _calculateNextStep (BaseAviary.py:1108-1150)
    R dest[3], dir[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) { dest[k] = from_double ? (R)ad[k] : (R)af[k]; }
    dir[0] = dest[0] - d.px; dir[1] = dest[1] - d.py; dir[2] = dest[2] - d.pz;
    const R dist = sqrt_(dir[0] * dir[0] + dir[1] * dir[1] + dir[2] * dir[2]);
    if (dist <= R(1)) { tp[0] = dest[0]; tp[1] = dest[1]; tp[2] = dest[2]; }
    else { tp[0] = d.px + dir[0] / dist; tp[1] = d.py + dir[1] / dist; tp[2] = d.pz + dir[2] / dist; }
  } else if (P.act_type == ACT_VEL) {               // :207-222
    tyaw = yaw;                                     // keep current yaw
    if (from_double) {
      const double n = sqrt(ad[0] * ad[0] + ad[1] * ad[1] + ad[2] * ad[2]);
      const double sp = (double)P.speed_limit * fabs(ad[3]);
      if (n != 0.0) { tv[0] = (R)(sp * (ad[0] / n)); tv[1] = (R)(sp * (ad[1] / n)); tv[2] = (R)(sp * (ad[2] / n)); }
    } else {
      const float p0 = __fmul_rn(af[0], af[0]), p1 = __fmul_rn(af[1], af[1]), p2 = __fmul_rn(af[2], af[2]);
      const float n = __fsqrt_rn((float)(((double)p0 + (double)p1) + (double)p2));
      const float sp = __fmul_rn(P.speed_limit_f, fabsf(af[3]));
      if (n != 0.f) {
        tv[0] = (R)__fmul_rn(sp, __fdiv_rn(af[0], n));
        tv[1] = (R)__fmul_rn(sp, __fdiv_rn(af[1], n));
        tv[2] = (R)__fmul_rn(sp, __fdiv_rn(af[2], n));
      }
    }
  } else {                                          // ONE_D_PID :226-235
    const R a0 = from_double ? (R)ad[0] : (R)af[0];
    tp[2] = d.pz + R(0.1) * a0;
  }
}

// DSLPIDControl.computeControl (:82-139): position loop -> thrust and target attitude,
// attitude loop -> PWM -> RPM.  c[0..2] integral_pos_e, c[3..5] integral_rpy_e, c[6..8] last_rpy.
// The scipy round trip of the target attitude (matrix -> 'XYZ' Euler -> quaternion -> matrix,
// :159-160,201-203) is the identity on an orthonormal matrix and is not performed.
template <typename R>
__device__ __forceinline__ void dsl_pid(const Params<R>& P, const Drone<R>& d, R roll, R pitch, R yaw,
                                        const R tp[3], R tyaw, const R tv[3], R c[9], R rpm[4]) {
  const R dt = P.ctrl_dt;
  R m[9];
  quat_to_mat(d.qx, d.qy, d.qz, d.qw, m);
  // ---- _dslPIDPositionControl (:143-197)
  const R pe[3] = {tp[0] - d.px, tp[1] - d.py, tp[2] - d.pz};
  const R ve[3] = {tv[0] - d.vx, tv[1] - d.vy, tv[2] - d.vz};
  c[0] = clip_(c[0] + pe[0] * dt, R(-2), R(2));
  c[1] = clip_(c[1] + pe[1] * dt, R(-2), R(2));
  c[2] = clip_(clip_(c[2] + pe[2] * dt, R(-2), R(2)), R(-0.15), R(0.15));
  R tt[3];
  tt[0] = (R(0.4) * pe[0] + R(0.05) * c[0]) + R(0.2) * ve[0];
  tt[1] = (R(0.4) * pe[1] + R(0.05) * c[1]) + R(0.2) * ve[1];
  tt[2] = ((R(1.25) * pe[2] + R(0.05) * c[2]) + R(0.5) * ve[2]) + P.ctrl_gravity;
  R scalar = (tt[0] * m[2] + tt[1] * m[5]) + tt[2] * m[8];
  scalar = scalar > R(0) ? scalar : R(0);
  const R thrust = (sqrt_(scalar / P.ctrl_4kf) - R(4070.3)) / R(0.2685);
  const R tn = sqrt_((tt[0] * tt[0] + tt[1] * tt[1]) + tt[2] * tt[2]);
  const R z[3] = {tt[0] / tn, tt[1] / tn, tt[2] / tn};
  R sy, cy;
  sincos_(tyaw, &sy, &cy);
  // y = z x x_c / |.|, x_c = (cos yaw, sin yaw, 0);  x = y x z
  R y[3] = {-z[2] * sy, z[2] * cy, z[0] * sy - z[1] * cy};
  const R yn = sqrt_((y[0] * y[0] + y[1] * y[1]) + y[2] * y[2]);
  y[0] /= yn; y[1] /= yn; y[2] /= yn;
  const R x[3] = {y[1] * z[2] - y[2] * z[1], y[2] * z[0] - y[0] * z[2], y[0] * z[1] - y[1] * z[0]};
  // ---- _dslPIDAttitudeControl (:201-246): rot_e from Rt^T Rc - Rc^T Rt, Rt = [x y z]
  const R c0[3] = {m[0], m[3], m[6]}, c1[3] = {m[1], m[4], m[7]}, c2[3] = {m[2], m[5], m[8]};
  auto dot3 = [](const R a[3], const R b[3]) { return (a[0] * b[0] + a[1] * b[1]) + a[2] * b[2]; };
  const R re[3] = {dot3(z, c1) - dot3(y, c2), dot3(x, c2) - dot3(z, c0), dot3(y, c0) - dot3(x, c1)};
  const R rpy[3] = {roll, pitch, yaw};
  R tq[3];
  const R ptor[3] = {R(70000), R(70000), R(60000)}, dtor[3] = {R(20000), R(20000), R(12000)};
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const R rate_e = R(0) - (rpy[k] - c[6 + k]) / dt;
    c[6 + k] = rpy[k];
    R ir = clip_(c[3 + k] - re[k] * dt, R(-1500), R(1500));
    if (k < 2) ir = clip_(ir, R(-1), R(1));
    c[3 + k] = ir;
    const R itor = k == 2 ? R(500) : R(0);
    tq[k] = clip_((-(ptor[k] * re[k]) + dtor[k] * rate_e) + itor * ir, R(-3200), R(3200));
  }
  // CF2X mixer (:48-53), PWM clip (:241), PWM -> RPM (:242)
  const R mix[4][3] = {{R(-.5), R(-.5), R(-1)}, {R(-.5), R(.5), R(1)}, {R(.5), R(.5), R(-1)}, {R(.5), R(-.5), R(1)}};
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const R pwm = clip_(thrust + ((mix[k][0] * tq[0] + mix[k][1] * tq[1]) + mix[k][2] * tq[2]), R(20000), R(65535));
    rpm[k] = R(0.2685) * pwm + R(4070.3);
  }
}

// ------------------------------------------------ async copies: TMA bulk store, cp.async history, PDL
// Observation rows are written once and never read back by the simulator: mark them evict-first
// in L2 so that they do not push out the persistent state / ring planes of the next step.
__device__ __forceinline__ void bulk_store_s2g(void* gdst, const void* ssrc, uint32_t bytes) {
  const unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(ssrc));
  uint64_t policy;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;\n" : "=l"(policy));
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;\n" ::"l"(gdst), "r"(s),
               "r"(bytes), "l"(policy)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
}
// L2 residency budget of the fast step kernel (DESIGN.md section 4): what the same tile reads again next step is
// marked evict_last, as far as the handle's budget (Params::l2_keep_state / l2_keep_slots) allows; data read for the
// last time is marked evict_first so that it goes before anything kept.  A ring slot's age is the number of steps
// since it was written (0: written by this step, read again at ages 1 .. B-1).  With the policy off every access
// carries evict_normal, the priority of an access without a hint.  Hints only choose where bytes come from.
__device__ __forceinline__ uint64_t l2_pol_last() {
  uint64_t p;
  asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;\n" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_pol_first() {
  uint64_t p;
  asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;\n" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_pol_normal() {
  uint64_t p;
  asm("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;\n" : "=l"(p));
  return p;
}
struct L2Hints {
  uint64_t state;       // state planes, step counter, episode return
  uint64_t slot_keep;   // ring slots younger than keep_slots
  uint64_t slot_drop;   // ring slots at or beyond keep_slots
  uint64_t once;        // caller's actions: read once
  int keep_slots;
};
template <typename R>
__device__ __forceinline__ L2Hints l2_hints(const Params<R>& P) {
  const uint64_t last = l2_pol_last(), first = l2_pol_first(), normal = l2_pol_normal();
  const bool on = P.l2_keep_state || P.l2_keep_slots > 0;
  return {P.l2_keep_state ? last : normal, last, on ? first : normal, first, P.l2_keep_slots};
}
__device__ __forceinline__ uint64_t l2_slot_pol(const L2Hints& h, int age) { return age < h.keep_slots ? h.slot_keep : h.slot_drop; }

__device__ __forceinline__ float4 ld_hint(const float4* p, uint64_t pol) {
  float4 v;
  asm volatile("ld.global.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;\n"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(pol) : "memory");
  return v;
}
__device__ __forceinline__ float ld_hint(const float* p, uint64_t pol) {
  float v;
  asm volatile("ld.global.L2::cache_hint.f32 %0, [%1], %2;\n" : "=f"(v) : "l"(p), "l"(pol) : "memory");
  return v;
}
__device__ __forceinline__ int ld_hint(const int* p, uint64_t pol) {
  int v;
  asm volatile("ld.global.L2::cache_hint.s32 %0, [%1], %2;\n" : "=r"(v) : "l"(p), "l"(pol) : "memory");
  return v;
}
__device__ __forceinline__ void st_hint(float4* p, float4 v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;\n" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w),
               "l"(pol)
               : "memory");
}
__device__ __forceinline__ void st_hint(float* p, float v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.f32 [%0], %1, %2;\n" ::"l"(p), "f"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_hint(int* p, int v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.s32 [%0], %1, %2;\n" ::"l"(p), "r"(v), "l"(pol) : "memory");
}

__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all0() { asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }

// action history of one tile, oldest -> second newest (BaseRLAviary.py:317-318): time-ordered
// entries j in [j0, j1) of B-1, entry j = ring slot (head+1+j) % B (age B-1-j) -> columns 12+jA.. of my row.
// HINT: each copy carries the L2 policy of its slot's age (L2Hints).
template <int A, bool VEC, bool HINT>
__device__ __forceinline__ void history_run(float*& dst, const float* src, size_t plane, int n, int& age, const L2Hints& h) {
#pragma unroll 2
  for (int j = 0; j < n; ++j) {
    if constexpr (HINT) {
      const uint64_t pol = l2_slot_pol(h, age);
      if constexpr (VEC) cp_async_hint<16>(dst, src, pol);
      else {
#pragma unroll
        for (int k = 0; k < A; ++k) cp_async_hint<4>(dst + k, src + k, pol);
      }
    } else {
      if constexpr (VEC) cp_async<16>(dst, src);
      else {
#pragma unroll
        for (int k = 0; k < A; ++k) cp_async<4>(dst + k, src + k);
      }
    }
    dst += A;
    src += plane;
    --age;
  }
}

template <typename R, int A, bool VEC, bool HINT = false>
__device__ __forceinline__ void issue_history(const Params<R>& P, long long g, int head, float* myrow,
                                              int j0, int j1, const L2Hints& h = L2Hints{}) {
  if (g < P.n_total) {
    const size_t plane = (size_t)P.n_total * A;
    const float* base = P.hist + (size_t)g * A;
    float* dst = myrow + 12 + j0 * A;
    // entries j0..j1-1 = slots head+1+j0 .. ; split at the ring wrap into two straight runs
    const int s0 = head + 1 + j0;            // may be >= B
    const int n = j1 - j0;
    int age = P.B - 1 - j0;
    if (s0 >= P.B) {
      history_run<A, VEC, HINT>(dst, base + (size_t)(s0 - P.B) * plane, plane, n, age, h);
    } else {
      const int n1 = min(n, P.B - s0);
      history_run<A, VEC, HINT>(dst, base + (size_t)s0 * plane, plane, n1, age, h);
      history_run<A, VEC, HINT>(dst, base, plane, n - n1, age, h);
    }
  }
}

__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ int ld_relaxed_gpu(const int* p) {
  int v;
  asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long ld_relaxed_gpu_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];\n" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(int* p, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;\n" ::"l"(p), "r"(v) : "memory");
}

__device__ __forceinline__ void st_relaxed_gpu(int* p, int v) {
  asm volatile("st.relaxed.gpu.global.s32 [%0], %1;\n" ::"l"(p), "r"(v) : "memory");
}

// gsteps layout: [0] total control steps, [1] CTA ticket (graph replays), [8..15] per-launch wait decisions
constexpr int kModeSlots = 8;
// Tile-level dependency on the previous control step (see bd_step_tile.cuh).  Returns nonzero when the CTA must
// still execute griddepcontrol.wait.  Two lanes work in parallel: lane 0 of warp 1 spins (ld.acquire) on this
// tile's epoch; lane 0 of warp 0 reads the launch's decision, made once per launch by the first CTA that finds
// the slot empty (or left over from an older launch): if the handle's previous step has not finished completely
// (finished-tile counter), the
// launch's programmatic primary can only be that step — anything else enqueued between two steps would itself
// have waited for the first one to finish — and the epochs cover everything: no grid-wide wait for any CTA of
// this launch (1).  Otherwise every CTA executes griddepcontrol.wait (2): free for our own finished kernel, and
// the usual completion + flush guarantee for a foreign kernel that produced the actions.
template <typename R>
__device__ __forceinline__ int pipe_gate(const Params<R>& P, int tile, int total, int tid) {
  int must_wait = 0;
  if (tid == 0) {
    // decision slots are tagged with the launch they belong to ((total + 1) << 2 | mode), so a slot left over from
    // the launch that used it eight steps earlier simply reads as empty: no recycling, no ordering to maintain
    unsigned* slot = reinterpret_cast<unsigned*>(P.gsteps + 8 + (total & (kModeSlots - 1)));
    const unsigned tag = ((unsigned)(total + 1) & 0x3fffffffu) << 2;
    unsigned v = (unsigned)ld_relaxed_gpu(reinterpret_cast<const int*>(slot));
    if ((v & ~3u) != tag || (v & 3u) == 0u) {
      const bool done = ld_relaxed_gpu_u64(P.finished) >= (unsigned long long)total * (unsigned long long)P.step_tiles;
      const unsigned want = tag | (done ? 2u : 1u);
      const unsigned old = atomicCAS(slot, v, want);
      v = (old == v) ? want : (((old & ~3u) == tag && (old & 3u) != 0u) ? old : want);   // lost the race: take the winner's
    }
    must_wait = ((v & 3u) == 2u);
  } else if (tid == 32) {
    // Bounded: the epoch is published by a CTA that is resident or already done, so the wait is a few
    // microseconds.  A protocol bug (an epoch that never arrives) must fail the launch, not hang the GPU:
    // after ~2^31 SM clocks (about one second) the CTA traps, like the actor kernel's mbarrier waits.
    long long t0 = 0;
    for (unsigned it = 0; ld_acquire_gpu(P.tile_epoch + tile) - total < 0; ++it) {
      __nanosleep(64);
      if ((it & 1023u) == 1023u) {
        const long long now = clock64();
        if (t0 == 0) t0 = now;
        else if (now - t0 > (1LL << 31)) __trap();
      }
    }
  }
  return __syncthreads_or(must_wait);
}

__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;\n" ::: "memory"); }

}  // namespace bd
