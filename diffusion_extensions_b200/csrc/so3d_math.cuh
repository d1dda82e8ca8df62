// so3d_math.cuh -- per-rotation SO(3) / IGSO(3) arithmetic shared by every kernel.
//
// One rotation lives in the registers of one thread (9 floats, row-major).  Everything here is a
// small inline function so that the kernels in so3d_kernels.cu can fuse axis-angle extraction,
// series/closed-form evaluation, sampling and composition without going through memory.
//
// The functions are __host__ __device__ on purpose: tests/host_math compiles this header with g++
// (SO3D_HOST_ONLY) so the CPU-only test tier can check the very same arithmetic against the oracle
// here, where no GPU exists.  That host build is a test harness -- the product never runs it.
//
// Reference behaviour is cited as file:line of qazwsxal/diffusion-extensions @ f100885d.
#pragma once

#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__) && !defined(SO3D_HOST_ONLY)
#define SO3D_HD __host__ __device__ __forceinline__
#define SO3D_D __device__ __forceinline__
#else
#define SO3D_HD inline
#define SO3D_D inline
#endif

namespace so3d {

constexpr float kPi = 3.14159265358979323846f;
constexpr float kTwoPi = 6.28318530717958647692f;
constexpr double kPiD = 3.14159265358979323846;
constexpr int kGrid = 1000;      // distributions.py:15 -- CDF grid points
constexpr int kCdf = kGrid - 1;  // entries per CDF row (trap / trap_loc)
constexpr float kNearPiCos = -0.9f;  // (tr R - 1)/2 below this: axis from the symmetric part

struct Vec3 {
  float x, y, z;
};
struct Mat3 {
  float m[9];  // row-major: m[3*i+j]
};

// ------------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------------
SO3D_HD float fast_ex2(float x) {
#if defined(__CUDA_ARCH__)
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));  // MUFU.EX2, 2 ulp
  return y;
#else
  return exp2f(x);
#endif
}

SO3D_HD float fast_rcp(float x) {
#if defined(__CUDA_ARCH__)
  return __frcp_rn(x);
#else
  return 1.0f / x;
#endif
}

SO3D_HD float rsqrt_f(float x) {
#if defined(__CUDA_ARCH__)
  return rsqrtf(x);
#else
  return 1.0f / sqrtf(x);
#endif
}

SO3D_HD void sincos_f(float x, float* s, float* c) {
#if defined(__CUDA_ARCH__)
  sincosf(x, s, c);
#else
  *s = sinf(x);
  *c = cosf(x);
#endif
}

SO3D_HD Mat3 identity() {
  Mat3 r;
  r.m[0] = 1.f; r.m[1] = 0.f; r.m[2] = 0.f;
  r.m[3] = 0.f; r.m[4] = 1.f; r.m[5] = 0.f;
  r.m[6] = 0.f; r.m[7] = 0.f; r.m[8] = 1.f;
  return r;
}

// C = A B
SO3D_HD Mat3 mul_nn(const Mat3& a, const Mat3& b) {
  Mat3 c;
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j)
      c.m[3 * i + j] = fmaf(a.m[3 * i + 2], b.m[6 + j], fmaf(a.m[3 * i + 1], b.m[3 + j], a.m[3 * i] * b.m[j]));
  return c;
}
// C = A^T B
SO3D_HD Mat3 mul_tn(const Mat3& a, const Mat3& b) {
  Mat3 c;
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j)
      c.m[3 * i + j] = fmaf(a.m[6 + i], b.m[6 + j], fmaf(a.m[3 + i], b.m[3 + j], a.m[i] * b.m[j]));
  return c;
}
// C = A B^T
SO3D_HD Mat3 mul_nt(const Mat3& a, const Mat3& b) {
  Mat3 c;
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j)
      c.m[3 * i + j] = fmaf(a.m[3 * i + 2], b.m[3 * j + 2], fmaf(a.m[3 * i + 1], b.m[3 * j + 1], a.m[3 * i] * b.m[3 * j]));
  return c;
}

// hat map, util.py:87-92
SO3D_HD Mat3 hat(Vec3 v) {
  Mat3 k;
  k.m[0] = 0.f;  k.m[1] = -v.z; k.m[2] = v.y;
  k.m[3] = v.z;  k.m[4] = 0.f;  k.m[5] = -v.x;
  k.m[6] = -v.y; k.m[7] = v.x;  k.m[8] = 0.f;
  return k;
}
// vee map, util.py:79-84: (m21, -m20, m10)
SO3D_HD Vec3 vee(const Mat3& a) { return Vec3{a.m[7], -a.m[6], a.m[3]}; }

// ------------------------------------------------------------------------------------------------
// log map / axis-angle.   util.py:164-192 (log_rmat), :208-219 (rmat_to_aa)
//   v = vee(R - R^T); s = |v|/2; c = (tr R - 1)/2; theta = atan2(s, c); log = theta/(2 s) * v.
// Deviation (SURVEY Q4/Q10): for c < kNearPiCos the axis is recovered from the symmetric part
// (R + R^T)/2 = c I + (1 - c) n n^T, which stays accurate up to and at theta = pi where the
// reference's skew-part formula is 0/0 and its eigh fallback picks a wrong axis; at the identity
// the axis is the fixed unit vector (0,0,1) instead of NaN.
// ------------------------------------------------------------------------------------------------
struct AxisAngle {
  Vec3 axis;    // unit
  float theta;  // [0, pi]
  float s, c;   // |v|/2 and (tr-1)/2 of the input (NOT renormalised): needed by the backward
};

SO3D_HD AxisAngle axis_angle(const Mat3& r) {
  AxisAngle o;
  const float vx = r.m[7] - r.m[5], vy = r.m[2] - r.m[6], vz = r.m[3] - r.m[1];
  const float n2 = fmaf(vx, vx, fmaf(vy, vy, vz * vz));
  const float nv = sqrtf(n2);
  o.s = 0.5f * nv;
  o.c = 0.5f * (r.m[0] + r.m[4] + r.m[8] - 1.0f);
  o.theta = atan2f(o.s, o.c);
  if (o.c >= kNearPiCos) {
    if (nv > 0.f) {
      const float inv = 1.0f / nv;
      o.axis = Vec3{vx * inv, vy * inv, vz * inv};
    } else {
      o.axis = Vec3{0.f, 0.f, 1.f};
    }
  } else {
    // symmetric part: d_i = R_ii, off-diagonals (R_ij + R_ji)/2; n_k from the largest diagonal
    const float omc = 1.0f - o.c;
    const float d0 = r.m[0], d1 = r.m[4], d2 = r.m[8];
    float nx, ny, nz;
    if (d0 >= d1 && d0 >= d2) {
      nx = sqrtf(fmaxf((d0 - o.c) / omc, 0.f));
      const float q = 0.5f / (omc * nx);
      ny = (r.m[1] + r.m[3]) * q;
      nz = (r.m[2] + r.m[6]) * q;
    } else if (d1 >= d2) {
      ny = sqrtf(fmaxf((d1 - o.c) / omc, 0.f));
      const float q = 0.5f / (omc * ny);
      nx = (r.m[1] + r.m[3]) * q;
      nz = (r.m[5] + r.m[7]) * q;
    } else {
      nz = sqrtf(fmaxf((d2 - o.c) / omc, 0.f));
      const float q = 0.5f / (omc * nz);
      nx = (r.m[2] + r.m[6]) * q;
      ny = (r.m[5] + r.m[7]) * q;
    }
    const float inv = rsqrt_f(fmaf(nx, nx, fmaf(ny, ny, nz * nz)));
    const float sgn = (fmaf(nx, vx, fmaf(ny, vy, nz * vz)) < 0.f) ? -inv : inv;
    o.axis = Vec3{nx * sgn, ny * sgn, nz * sgn};
  }
  return o;
}

// vee(log R) = theta * axis
SO3D_HD Vec3 log_vec(const Mat3& r) {
  const AxisAngle a = axis_angle(r);
  return Vec3{a.theta * a.axis.x, a.theta * a.axis.y, a.theta * a.axis.z};
}

// ------------------------------------------------------------------------------------------------
// exp map.  Replaces torch.matrix_exp + SVD re-orthogonalisation (util.py:195-205, :360,
// diffusion.py:294) by the Rodrigues closed form, always orthonormal to fp32 rounding.
//   R = I + sin(t) K + (1 - cos(t)) K^2,  K = hat(n), |n| = 1;   1 - cos t = 2 sin^2(t/2).
// ------------------------------------------------------------------------------------------------
SO3D_HD Mat3 rodrigues_sc(Vec3 n, float sn, float omc /* 1 - cos */) {
  Mat3 r;
  const float xx = n.x * n.x, yy = n.y * n.y, zz = n.z * n.z;
  const float xy = omc * n.x * n.y, xz = omc * n.x * n.z, yz = omc * n.y * n.z;
  const float sx = sn * n.x, sy = sn * n.y, sz = sn * n.z;
  r.m[0] = fmaf(-omc, yy + zz, 1.0f);
  r.m[1] = xy - sz;
  r.m[2] = xz + sy;
  r.m[3] = xy + sz;
  r.m[4] = fmaf(-omc, xx + zz, 1.0f);
  r.m[5] = yz - sx;
  r.m[6] = xz - sy;
  r.m[7] = yz + sx;
  r.m[8] = fmaf(-omc, xx + yy, 1.0f);
  return r;
}

SO3D_HD Mat3 rodrigues(Vec3 n_unit, float theta) {
  float sh, ch;
  sincos_f(0.5f * theta, &sh, &ch);
  return rodrigues_sc(n_unit, 2.0f * sh * ch, 2.0f * sh * sh);
}

// exp(hat(v)) for a rotation vector (no normalisation problem at |v| -> 0)
SO3D_HD Mat3 exp_vec(Vec3 v) {
  const float t2 = fmaf(v.x, v.x, fmaf(v.y, v.y, v.z * v.z));
  const float t = sqrtf(t2);
  float sh, ch;
  sincos_f(0.5f * t, &sh, &ch);
  // a = sin(t)/t, b = (1-cos t)/t^2 = (sin(t/2)/(t/2))^2 / 2
  float a, b;
  if (t > 1e-4f) {
    const float sinc_h = sh / (0.5f * t);
    a = sinc_h * ch;
    b = 0.5f * sinc_h * sinc_h;
  } else {
    a = 1.0f - t2 * (1.0f / 6.0f);
    b = 0.5f - t2 * (1.0f / 24.0f);
  }
  Mat3 r;
  const float xx = v.x * v.x, yy = v.y * v.y, zz = v.z * v.z;
  const float xy = b * v.x * v.y, xz = b * v.x * v.z, yz = b * v.y * v.z;
  r.m[0] = fmaf(-b, yy + zz, 1.0f);
  r.m[1] = fmaf(-a, v.z, xy);
  r.m[2] = fmaf(a, v.y, xz);
  r.m[3] = fmaf(a, v.z, xy);
  r.m[4] = fmaf(-b, xx + zz, 1.0f);
  r.m[5] = fmaf(-a, v.x, yz);
  r.m[6] = fmaf(-a, v.y, xz);
  r.m[7] = fmaf(a, v.x, yz);
  r.m[8] = fmaf(-b, xx + yy, 1.0f);
  return r;
}

// util.py:195-205: normalise the axis (0-axis -> NaN like the reference), rotate by `ang`.
SO3D_HD Mat3 aa_to_rmat(Vec3 axis, float ang) {
  const float inv = 1.0f / sqrtf(fmaf(axis.x, axis.x, fmaf(axis.y, axis.y, axis.z * axis.z)));
  return rodrigues(Vec3{axis.x * inv, axis.y * inv, axis.z * inv}, ang);
}

// util.py:349-361: exp(s log R) = rotation by s*theta about the axis of R.
SO3D_HD Mat3 scale_rot(const Mat3& r, float s) {
  const AxisAngle a = axis_angle(r);
  return rodrigues(a.axis, s * a.theta);
}

// util.py:222-252: real-first quaternion, un-normalised input allowed.
SO3D_HD Mat3 quat_to_rmat(float qr, float qi, float qj, float qk) {
  const float two_s = 2.0f / fmaf(qr, qr, fmaf(qi, qi, fmaf(qj, qj, qk * qk)));
  Mat3 o;
  o.m[0] = 1.0f - two_s * (qj * qj + qk * qk);
  o.m[1] = two_s * (qi * qj - qk * qr);
  o.m[2] = two_s * (qi * qk + qj * qr);
  o.m[3] = two_s * (qi * qj + qk * qr);
  o.m[4] = 1.0f - two_s * (qi * qi + qk * qk);
  o.m[5] = two_s * (qj * qk - qi * qr);
  o.m[6] = two_s * (qi * qk - qj * qr);
  o.m[7] = two_s * (qj * qk + qi * qr);
  o.m[8] = 1.0f - two_s * (qi * qi + qj * qj);
  return o;
}

// No reference counterpart (SURVEY D6).  Unit quaternion, real-first, real part >= 0.
SO3D_HD void rmat_to_quat(const Mat3& r, float q[4]) {
  const float tr = r.m[0] + r.m[4] + r.m[8];
  float w, x, y, z;
  if (tr > 0.f) {
    const float s = sqrtf(tr + 1.0f) * 2.0f;
    w = 0.25f * s; x = (r.m[7] - r.m[5]) / s; y = (r.m[2] - r.m[6]) / s; z = (r.m[3] - r.m[1]) / s;
  } else if (r.m[0] > r.m[4] && r.m[0] > r.m[8]) {
    const float s = sqrtf(1.0f + r.m[0] - r.m[4] - r.m[8]) * 2.0f;
    w = (r.m[7] - r.m[5]) / s; x = 0.25f * s; y = (r.m[1] + r.m[3]) / s; z = (r.m[2] + r.m[6]) / s;
  } else if (r.m[4] > r.m[8]) {
    const float s = sqrtf(1.0f + r.m[4] - r.m[0] - r.m[8]) * 2.0f;
    w = (r.m[2] - r.m[6]) / s; x = (r.m[1] + r.m[3]) / s; y = 0.25f * s; z = (r.m[5] + r.m[7]) / s;
  } else {
    const float s = sqrtf(1.0f + r.m[8] - r.m[0] - r.m[4]) * 2.0f;
    w = (r.m[3] - r.m[1]) / s; x = (r.m[2] + r.m[6]) / s; y = (r.m[5] + r.m[7]) / s; z = 0.25f * s;
  }
  const float n = rsqrt_f(fmaf(w, w, fmaf(x, x, fmaf(y, y, z * z)))) * (w < 0.f ? -1.f : 1.f);
  q[0] = w * n; q[1] = x * n; q[2] = y * n; q[3] = z * n;
}

// ------------------------------------------------------------------------------------------------
// Lean arithmetic for the HBM-bound fused kernels (forward noising, reverse step, closed-form score).
// At 84-92 B per rotation the instruction budget of an HBM-bound kernel on B200 is ~480 thread
// instructions per row (148 SMs x 128 lanes x 1.965 GHz / 7.7e10 rows/s); the general-purpose versions
// above (IEEE division and sqrt with slow-path calls, libdevice sincosf/atan2f, 3x3 products, divergent
// near-pi branch) cost ~1200.  These are branch-free, division-free (MUFU.RCP / MUFU.RSQ) and work on unit
// quaternions; each is accurate to ~2e-7 absolute, checked against the fp64 oracle in tests/test_host_math.py.
// ------------------------------------------------------------------------------------------------
SO3D_HD float rcp_approx(float x) {
#if defined(__CUDA_ARCH__)
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
#else
  return 1.0f / x;
#endif
}
SO3D_HD float rsqrt_approx(float x) {
#if defined(__CUDA_ARCH__)
  float y;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
#else
  return 1.0f / sqrtf(x);
#endif
}
SO3D_HD float fsel(bool p, float a, float b) { return p ? a : b; }

// sin and cos of x for |x| < ~1e5: k = rint(x 2/pi) by the magic-number add, two-FMA Cody-Waite reduction
// (pi/2 = 1.57079637 - 4.37113883e-8), cephes minimax polynomials on [-pi/4, pi/4], quadrant fix by selects.
SO3D_HD void sincos_fast(float x, float* s_out, float* c_out) {
  const float t = fmaf(x, 0.636619772f, 12582912.0f);  // 1.5 * 2^23: the integer lands in the low mantissa bits
  const float kf = t - 12582912.0f;
  float r = fmaf(kf, -1.57079637f, x);
  r = fmaf(kf, 4.37113883e-8f, r);
  const float r2 = r * r;
  float ps = fmaf(-1.9515295891e-4f, r2, 8.3321608736e-3f);
  ps = fmaf(ps, r2, -1.6666654611e-1f);
  const float sn = fmaf(ps * r2, r, r);
  float pc = fmaf(2.443315711809948e-5f, r2, -1.388731625493765e-3f);
  pc = fmaf(pc, r2, 4.166664568298827e-2f);
  pc = fmaf(pc, r2, -0.5f);
  const float cs = fmaf(pc, r2, 1.0f);
#if defined(__CUDA_ARCH__)
  const unsigned k = __float_as_uint(t);
#else
  unsigned k;
  memcpy(&k, &t, 4);
#endif
  const bool swap = k & 1u;
  const float s0 = fsel(swap, cs, sn), c0 = fsel(swap, sn, cs);
  *s_out = (k & 2u) ? -s0 : s0;
  *c_out = ((k + 1u) & 2u) ? -c0 : c0;
}

// atan2(y, x) for y >= 0: angle in [0, pi].  t = min/max in [0, 1], Abramowitz-Stegun 4.4.49 (|err| <= 2e-8).
SO3D_HD float atan2_pos(float y, float x) {
  const float ax = fabsf(x);
  const float hi = fmaxf(ax, y), lo = fminf(ax, y);
  const float t = lo * rcp_approx(fmaxf(hi, 1e-37f));
  const float z = t * t;
  float p = fmaf(0.0028662257f, z, -0.0161657367f);
  p = fmaf(p, z, 0.0429096138f);
  p = fmaf(p, z, -0.0752896400f);
  p = fmaf(p, z, 0.1065626393f);
  p = fmaf(p, z, -0.1420889944f);
  p = fmaf(p, z, 0.1999355085f);
  p = fmaf(p, z, -0.3333314528f);
  float r = fmaf(p * z, t, t);
  r = fsel(y > ax, 1.57079632679f - r, r);
  return fsel(x < 0.f, 3.14159265359f - r, r);
}

struct Quat {
  float w, x, y, z;
};

// Hamilton product a (x) b  (rotation a applied after b, i.e. R(a) R(b))
SO3D_HD Quat qmul(const Quat& a, const Quat& b) {
  Quat q;
  q.w = fmaf(-a.z, b.z, fmaf(-a.y, b.y, fmaf(-a.x, b.x, a.w * b.w)));
  q.x = fmaf(-a.z, b.y, fmaf(a.y, b.z, fmaf(a.x, b.w, a.w * b.x)));
  q.y = fmaf(a.z, b.x, fmaf(a.y, b.w, fmaf(-a.x, b.z, a.w * b.y)));
  q.z = fmaf(a.z, b.w, fmaf(-a.y, b.x, fmaf(a.x, b.y, a.w * b.z)));
  return q;
}

// unit quaternion of the rotation by `theta` about the unit axis n
SO3D_HD Quat quat_axis_angle(Vec3 n, float theta) {
  float sh, ch;
  sincos_fast(0.5f * theta, &sh, &ch);
  return Quat{ch, sh * n.x, sh * n.y, sh * n.z};
}

// exp(hat(v)) as a quaternion: (cos(|v|/2), sin(|v|/2) v/|v|), with the |v| -> 0 limit (1, v/2)
SO3D_HD Quat quat_exp_vec(Vec3 v) {
  const float t2 = fmaf(v.x, v.x, fmaf(v.y, v.y, v.z * v.z));
  const float rs = rsqrt_approx(fmaxf(t2, 1e-30f));
  const float t = t2 * rs;
  float sh, ch;
  sincos_fast(0.5f * t, &sh, &ch);
  const float k = fsel(t2 > 1e-12f, sh * rs, 0.5f);
  return Quat{ch, k * v.x, k * v.y, k * v.z};
}

// rotation matrix of a quaternion (normalised here, so the result is orthonormal to fp32 rounding)
SO3D_HD Mat3 quat_to_mat_unit(const Quat& q0) {
  const float inv = rsqrt_approx(fmaf(q0.w, q0.w, fmaf(q0.x, q0.x, fmaf(q0.y, q0.y, q0.z * q0.z))));
  const float w = q0.w * inv, x = q0.x * inv, y = q0.y * inv, z = q0.z * inv;
  const float x2 = x + x, y2 = y + y, z2 = z + z;
  const float wx = w * x2, wy = w * y2, wz = w * z2;
  Mat3 r;
  r.m[0] = fmaf(-y2, y, fmaf(-z2, z, 1.0f));
  r.m[4] = fmaf(-x2, x, fmaf(-z2, z, 1.0f));
  r.m[8] = fmaf(-x2, x, fmaf(-y2, y, 1.0f));
  r.m[1] = fmaf(x2, y, -wz);
  r.m[3] = fmaf(x2, y, wz);
  r.m[2] = fmaf(x2, z, wy);
  r.m[6] = fmaf(x2, z, -wy);
  r.m[5] = fmaf(y2, z, -wx);
  r.m[7] = fmaf(y2, z, wx);
  return r;
}

// Axis and angle of a rotation matrix, branch-free: same definition as axis_angle() above (theta = atan2(|v|/2,
// (tr-1)/2); axis from the skew part, or for (tr-1)/2 < kNearPiCos from the best-conditioned column of the
// symmetric part (R + R^T)/2 - c I = (1 - c) n n^T, sign fixed by the skew part), selects instead of branches.
//
// MUFU.RSQ (rsqrt.approx.ftz) flushes a subnormal input to zero and returns +inf, which made |v|^2 below FLT_MIN
// (theta below ~5e-20) come out as theta = pi/2 with an inf / NaN axis.  Such a skew part is scaled by 2^64 first
// (exact), so the axis and the angle keep full relative precision down to theta ~ 1e-38; below that the row is read as
// the identity.  For |v|^2 >= FLT_MIN the scale is 1 and every bit is what it was without it.
constexpr float kFltMin = 1.17549435e-38f;  // FLT_MIN = 2^-126
constexpr float kTinyUp = 18446744073709551616.0f;    // 2^64
constexpr float kTinyDown = 5.42101086242752217e-20f;  // 2^-64
struct AxisAngleF {
  Vec3 axis;
  float theta;
};
SO3D_HD AxisAngleF axis_angle_fast(const Mat3& r) {
  const float ux = r.m[7] - r.m[5], uy = r.m[2] - r.m[6], uz = r.m[3] - r.m[1];
  const bool tiny = fmaf(ux, ux, fmaf(uy, uy, uz * uz)) < kFltMin;
  const float k = fsel(tiny, kTinyUp, 1.0f);
  const float vx = ux * k, vy = uy * k, vz = uz * k;
  const float n2 = fmaf(vx, vx, fmaf(vy, vy, vz * vz));
  const bool pos = n2 >= kFltMin;
  const float rs = fsel(pos, rsqrt_approx(n2), 0.f);
  const float c = 0.5f * (r.m[0] + r.m[4] + r.m[8] - 1.0f);
  AxisAngleF o;
  o.theta = atan2_pos(fsel(tiny, 0.5f * kTinyDown, 0.5f) * n2 * rs, c);
  // symmetric-part candidate: column j of S - c I with the largest diagonal
  const float d0 = r.m[0] - c, d1 = r.m[4] - c, d2 = r.m[8] - c;
  const float s01 = 0.5f * (r.m[1] + r.m[3]), s02 = 0.5f * (r.m[2] + r.m[6]), s12 = 0.5f * (r.m[5] + r.m[7]);
  const bool p0 = (d0 >= d1) && (d0 >= d2);
  const bool p1 = d1 >= d2;
  const float cx = fsel(p0, d0, fsel(p1, s01, s02));
  const float cy = fsel(p0, s01, fsel(p1, d1, s12));
  const float cz = fsel(p0, s02, fsel(p1, s12, d2));
  const float cn = rsqrt_approx(fmaxf(fmaf(cx, cx, fmaf(cy, cy, cz * cz)), 1e-30f));
  const float sg = fsel(fmaf(cx, vx, fmaf(cy, vy, cz * vz)) < 0.f, -cn, cn);
  const bool near_pi = c < kNearPiCos;
  o.axis.x = fsel(near_pi, cx * sg, vx * rs);
  o.axis.y = fsel(near_pi, cy * sg, vy * rs);
  o.axis.z = fsel(near_pi, cz * sg, fsel(pos, vz * rs, 1.0f));
  return o;
}

// The L0 maps of util.py on the lean primitives (what the row-engine kernels run; the general-purpose versions
// above stay as the backward passes' and the host harness's definition).
SO3D_HD Vec3 log_vec_fast(const Mat3& r) {  // util.py:164-192: vee(log R) = theta axis
  const AxisAngleF a = axis_angle_fast(r);
  return Vec3{a.theta * a.axis.x, a.theta * a.axis.y, a.theta * a.axis.z};
}
SO3D_HD Mat3 scale_rot_fast(const Mat3& r, float s) {  // util.py:349-361: rotation by s theta about the axis of R
  const AxisAngleF a = axis_angle_fast(r);
  return quat_to_mat_unit(quat_axis_angle(a.axis, s * a.theta));
}

// half-angle in [0, pi/2] and unit axis of a (near-)unit quaternion, with q and -q identified (a vector part whose
// square is below FLT_MIN is scaled by 2^64 first, as in axis_angle_fast)
SO3D_HD void quat_axis_halfangle(const Quat& q, Vec3* n, float* half) {
  const bool tiny = fmaf(q.x, q.x, fmaf(q.y, q.y, q.z * q.z)) < kFltMin;
  const float sc = fsel(tiny, kTinyUp, 1.0f);
  const float x = q.x * sc, y = q.y * sc, z = q.z * sc;
  const float v2 = fmaf(x, x, fmaf(y, y, z * z));
  const bool pos = v2 >= kFltMin;
  const float rs = fsel(pos, rsqrt_approx(v2), 0.f);
  *half = atan2_pos(fsel(tiny, kTinyDown, 1.0f) * v2 * rs, fabsf(q.w));
  const float k = fsel(q.w < 0.f, -rs, rs);
  *n = Vec3{x * k, y * k, fsel(pos, z * k, 1.0f)};
}

// Kernel values on SO(3) for a pair of unit quaternions a, b (real part first), util.py:128-150:
//   gaussian: exp(-rmat_dist) = exp(-sqrt(2) theta),   cosine: cos(theta),   theta = angle of R(a)^T R(b).
// conj(a) (x) b has scalar part d = cos(theta/2) (up to sign) and a vector part v with |v| = sin(theta/2): both are
// computed directly (no 1 - d^2 cancellation), so theta/2 = atan2(|v|, |d|) is accurate to ~1e-7 rad from 0 to pi.
template <bool kGaussian>
SO3D_HD float so3_pair_kernel(const Quat& a, const Quat& b) {
  const float d = fmaf(a.w, b.w, fmaf(a.x, b.x, fmaf(a.y, b.y, a.z * b.z)));
  const float vx = fmaf(a.w, b.x, fmaf(-b.w, a.x, fmaf(a.z, b.y, -(a.y * b.z))));
  const float vy = fmaf(a.w, b.y, fmaf(-b.w, a.y, fmaf(a.x, b.z, -(a.z * b.x))));
  const float vz = fmaf(a.w, b.z, fmaf(-b.w, a.z, fmaf(a.y, b.x, -(a.x * b.y))));
  const float s2 = fmaf(vx, vx, fmaf(vy, vy, vz * vz));
  if (!kGaussian) return fmaf(d, d, -s2);  // cos(theta) = cos^2(theta/2) - sin^2(theta/2)
  const float s = s2 * rsqrt_approx(fmaxf(s2, 1e-37f));
  const float ad = fabsf(d);
  // s^2 + d^2 = 1, so max(s, |d|) >= 0.707: the quotient needs no zero guard
  const float hi = fmaxf(ad, s), lo = fminf(ad, s);
  const float t = lo * rcp_approx(hi);
  const float z = t * t;
  float p = fmaf(0.0028662257f, z, -0.0161657367f);  // Abramowitz-Stegun 4.4.49, |err| <= 2e-8 on [0, 1]
  p = fmaf(p, z, 0.0429096138f);
  p = fmaf(p, z, -0.0752896400f);
  p = fmaf(p, z, 0.1065626393f);
  p = fmaf(p, z, -0.1420889944f);
  p = fmaf(p, z, 0.1999355085f);
  p = fmaf(p, z, -0.3333314528f);
  float h = fmaf(p * z, t, t);
  h = fsel(s > ad, 1.57079632679f - h, h);
  return fast_ex2(-4.08055779f * h);  // exp(-sqrt(2) * 2h) = 2^(-2 sqrt(2) log2(e) h)
}

// The reverse step of diffusion.py:291-326 on quaternions (one atan2 per log, one sincos per exp):
//   x0_hat = so3_scale(x_t, a) @ exp(hat(b pred))^T ;  mean = so3_scale(x0_hat, c1) @ so3_scale(x_t, c2)
// Returns the mean as a quaternion; *x0h receives x0_hat.
SO3D_HD Quat p_mean_quat(const Mat3& x_t, Vec3 pred, float a, float b, float c1, float c2, Quat* x0h) {
  const AxisAngleF ax = axis_angle_fast(x_t);
  const Quat q1 = quat_axis_angle(ax.axis, a * ax.theta);
  const Quat q2 = quat_exp_vec(Vec3{-b * pred.x, -b * pred.y, -b * pred.z});
  const Quat qh = qmul(q1, q2);
  Vec3 n0;
  float h0;
  quat_axis_halfangle(qh, &n0, &h0);
  const Quat q3 = quat_axis_angle(n0, 2.0f * c1 * h0);
  const Quat q4 = quat_axis_angle(ax.axis, c2 * ax.theta);
  *x0h = qh;
  return qmul(q3, q4);
}

// The same step with pred = 0 (no denoiser / zero score: so3d_p_sample_loop_f32 with pred3 == NULL): exp(0) is the identity
// quaternion (1, 0, 0, 0) and q1 (x) (1, 0, 0, 0) = q1 exactly in floating point, so skipping the product gives the
// bits p_mean_quat() produces for pred = (0, 0, 0) (up to the sign of zero components, which no later operation sees).
SO3D_HD Quat p_mean_quat_nopred(const Mat3& x_t, float a, float c1, float c2, Quat* x0h) {
  const AxisAngleF ax = axis_angle_fast(x_t);
  const Quat qh = quat_axis_angle(ax.axis, a * ax.theta);
  Vec3 n0;
  float h0;
  quat_axis_halfangle(qh, &n0, &h0);
  const Quat q3 = quat_axis_angle(n0, 2.0f * c1 * h0);
  const Quat q4 = quat_axis_angle(ax.axis, c2 * ax.theta);
  *x0h = qh;
  return qmul(q3, q4);
}

// ------------------------------------------------------------------------------------------------
// Backward pieces (what autograd through the reference's torch ops yields, in closed form).
// ------------------------------------------------------------------------------------------------
// <G, hat(u)> = u . vee_adj(G)
SO3D_HD Vec3 vee_adj(const Mat3& g) { return Vec3{g.m[7] - g.m[5], g.m[2] - g.m[6], g.m[3] - g.m[1]}; }

// Gradient of  L(R) = <GL, log_rmat(R)>  w.r.t. the 9 entries of R, differentiating the reference's
// formula util.py:165-176 (theta = atan2(s, c), scale = theta/(2 s), log = scale (R - R^T)):
//   dL = a * dscale + scale <GL - GL^T, dR>,   a = <GL, R - R^T>
//   dscale = ds [ c/(2 s (s^2+c^2)) - theta/(2 s^2) ] - dc / (2 (s^2+c^2)),
//   ds = <R - R^T, dR>/(4 s),  dc = tr(dR)/2.
// For c < kNearPiCos the formula's component along SO(3) is ill-conditioned: R - R^T holds only ~2^-24 absolute
// precision, and evaluated on an fp32 matrix (orthonormal to ~6e-8) the formula's tangent part is off by ~2^-24/sin^2(theta).
// There the tangent component, vee_adj(R^T g), is replaced by the derivative of log along R exp(hat(xi)),
//   Jr^-T(theta n) vee_adj(GL) = u - (theta/2) n x u + (1 - (theta/2) sin(theta)/(1 - cos(theta))) n x (n x u),
// with theta and n from axis_angle's symmetric-part branch; the normal component (R times the symmetric part of R^T g)
// stays the reference formula's.  The error of the tangent part is then ~2^-24/sin(theta), the rounding of the fp32
// output, whose normal entries are of size 1/sin(theta).
SO3D_HD Mat3 log_bwd(const Mat3& r, const Mat3& gl) {
  const float vx = r.m[7] - r.m[5], vy = r.m[2] - r.m[6], vz = r.m[3] - r.m[1];
  const float s = 0.5f * sqrtf(fmaf(vx, vx, fmaf(vy, vy, vz * vz)));
  const float c = 0.5f * (r.m[0] + r.m[4] + r.m[8] - 1.0f);
  const float th = atan2f(s, c);
  const float den = fmaf(s, s, c * c);
  Mat3 a;  // R - R^T
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) a.m[3 * i + j] = r.m[3 * i + j] - r.m[3 * j + i];
  float ga = 0.f;
#pragma unroll
  for (int k = 0; k < 9; ++k) ga = fmaf(gl.m[k], a.m[k], ga);
  float scale, ks, kc;
  if (s > 1e-4f) {
    scale = th / (2.0f * s);
    ks = (c / (2.0f * s * den) - th / (2.0f * s * s)) / (4.0f * s);
    kc = -1.0f / (4.0f * den);
  } else if (c > 0.f) {
    // theta -> 0 limits: scale -> 1/2 + s^2/12 (orthonormal input); ks is the partial d scale/ds at fixed c, over 4 s,
    // -> -1/(12 c^3) = -1/12 (the total derivative along SO(3), 1/24, is not what the chain rule above needs)
    scale = 0.5f + s * s * (1.0f / 12.0f);
    ks = -(1.0f / 12.0f);
    kc = -1.0f / (4.0f * den);
  } else {
    // theta -> pi: the formula is singular (scale ~ pi/(2 s)); keep it finite, gradient is ill-defined
    const float sc = fmaxf(s, 1e-12f);
    scale = th / (2.0f * sc);
    ks = (c / (2.0f * sc * den) - th / (2.0f * sc * sc)) / (4.0f * sc);
    kc = -1.0f / (4.0f * den);
  }
  Mat3 g;
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      float v = ga * ks * a.m[3 * i + j] + scale * (gl.m[3 * i + j] - gl.m[3 * j + i]);
      if (i == j) v = fmaf(ga, kc, v);
      g.m[3 * i + j] = v;
    }
  if (c < kNearPiCos) {
    const AxisAngle aa = axis_angle(r);
    const Vec3 n = aa.axis, u = vee_adj(gl);
    const float ht = 0.5f * aa.theta;
    const float kq = 1.0f - ht * s / (1.0f - c);
    const Vec3 nu{n.y * u.z - n.z * u.y, n.z * u.x - n.x * u.z, n.x * u.y - n.y * u.x};        // n x u
    const Vec3 nnu{n.y * nu.z - n.z * nu.y, n.z * nu.x - n.x * nu.z, n.x * nu.y - n.y * nu.x};  // n x (n x u)
    const Vec3 cur = vee_adj(mul_tn(r, g));
    // g += R hat(d)/2 moves vee_adj(R^T g) by d
    const Vec3 d{0.5f * (fmaf(kq, nnu.x, fmaf(-ht, nu.x, u.x)) - cur.x), 0.5f * (fmaf(kq, nnu.y, fmaf(-ht, nu.y, u.y)) - cur.y),
                 0.5f * (fmaf(kq, nnu.z, fmaf(-ht, nu.z, u.z)) - cur.z)};
    const Mat3 corr = mul_nn(r, hat(d));
#pragma unroll
    for (int k = 0; k < 9; ++k) g.m[k] += corr.m[k];
  }
  return g;
}

// Gradient of <G, Rodrigues(n, t)> w.r.t. the (un-normalised) axis and the angle.
//   R = I + sin t K + (1 - cos t)(n n^T - I):  dR/dt = cos t K + sin t K^2,
//   dR/dn . dn = sin t hat(dn) + (1 - cos t)(dn n^T + n dn^T), then project through n = axis/|axis|.
SO3D_HD void aa_to_rmat_bwd(Vec3 axis, float ang, const Mat3& g, Vec3* g_axis, float* g_ang) {
  const float len = sqrtf(fmaf(axis.x, axis.x, fmaf(axis.y, axis.y, axis.z * axis.z)));
  const float inv = 1.0f / len;
  const Vec3 n{axis.x * inv, axis.y * inv, axis.z * inv};
  float sn, cs;
  sincos_f(ang, &sn, &cs);
  const Mat3 k = hat(n);
  const Mat3 k2 = mul_nn(k, k);
  float ga = 0.f;
#pragma unroll
  for (int i = 0; i < 9; ++i) ga = fmaf(g.m[i], fmaf(cs, k.m[i], sn * k2.m[i]), ga);
  *g_ang = ga;
  const Vec3 va = vee_adj(g);
  const float omc = 1.0f - cs;
  // (G + G^T) n
  const float sx = fmaf(2.f * g.m[0], n.x, fmaf(g.m[1] + g.m[3], n.y, (g.m[2] + g.m[6]) * n.z));
  const float sy = fmaf(g.m[1] + g.m[3], n.x, fmaf(2.f * g.m[4], n.y, (g.m[5] + g.m[7]) * n.z));
  const float sz = fmaf(g.m[2] + g.m[6], n.x, fmaf(g.m[5] + g.m[7], n.y, 2.f * g.m[8] * n.z));
  const float gx = fmaf(sn, va.x, omc * sx), gy = fmaf(sn, va.y, omc * sy), gz = fmaf(sn, va.z, omc * sz);
  const float dot = fmaf(gx, n.x, fmaf(gy, n.y, gz * n.z));
  *g_axis = Vec3{(gx - dot * n.x) * inv, (gy - dot * n.y) * inv, (gz - dot * n.z) * inv};
}

// Gradient of <G, exp(hat(w))> w.r.t. w:  d exp(W)[hat(dw)] = exp(W) hat(Jr(w) dw),
//   Jr(w) = I - (1-cos p)/p^2 hat(w) + (p - sin p)/p^3 hat(w)^2,  p = |w|;  grad = Jr^T vee_adj(R^T G).
SO3D_HD Vec3 exp_vec_bwd(Vec3 w, const Mat3& r_out, const Mat3& g) {
  const Vec3 u = vee_adj(mul_tn(r_out, g));
  const float p2 = fmaf(w.x, w.x, fmaf(w.y, w.y, w.z * w.z));
  const float p = sqrtf(p2);
  float b, cfac;
  if (p > 1e-2f) {
    float sh, ch;
    sincos_f(0.5f * p, &sh, &ch);
    b = 2.0f * sh * sh / p2;
    cfac = (p - 2.0f * sh * ch) / (p2 * p);
  } else {
    b = 0.5f - p2 * (1.0f / 24.0f);
    cfac = (1.0f / 6.0f) - p2 * (1.0f / 120.0f);
  }
  // Jr^T u = u + b (w x u) ... careful with signs: Jr^T = I + b hat(w) + cfac hat(w)^2
  const float cx = w.y * u.z - w.z * u.y, cy = w.z * u.x - w.x * u.z, cz = w.x * u.y - w.y * u.x;  // w x u
  const float dx = w.y * cz - w.z * cy, dy = w.z * cx - w.x * cz, dz = w.x * cy - w.y * cx;        // w x (w x u)
  return Vec3{fmaf(cfac, dx, fmaf(b, cx, u.x)), fmaf(cfac, dy, fmaf(b, cy, u.y)), fmaf(cfac, dz, fmaf(b, cz, u.z))};
}

// ------------------------------------------------------------------------------------------------
// IGSO(3) density: closed (Poisson-dual, 3-image) form.  distributions.py:53-72.
// ------------------------------------------------------------------------------------------------
// fp64, used only by the CDF-table builder (the reference evaluates in fp64 and rounds to fp32).
// quirks != 0 follows distributions.py:56-62 literally (0*inf = NaN -> 0 for w > 709 eps^2/pi, D5);
// the default uses the algebraically identical exp(-pi(pi -+ w)/v).
SO3D_HD double igso3_closed_f64(double t, double eps, int quirks) {
  const double v = eps * eps;
  const double pref = sqrt(kPiD) * pow(v, -1.5) * exp(v / 4) * exp(-((t / 2) * (t / 2)) / v);
  double inner;
  if (quirks) {
    inner = t - exp(-(kPiD * kPiD) / v) * ((t - 2 * kPiD) * exp(kPiD * t / v) + (t + 2 * kPiD) * exp(-kPiD * t / v));
  } else {
    inner = t - (t - 2 * kPiD) * exp(-kPiD * (kPiD - t) / v) - (t + 2 * kPiD) * exp(-kPiD * (kPiD + t) / v);
  }
  double val = pref * inner / (2 * sin(t / 2));
  if (isinf(val) || isnan(val)) val = 0.0;
  if (t == 0.0) {
    if (quirks) {
      val = sqrt(kPiD) * (v * exp(2 * kPiD * kPiD / v) - 2 * v * exp(kPiD * kPiD / v) + 4 * kPiD * kPiD * v * exp(kPiD * kPiD / v)) *
            exp(v / 4 - (2 * kPiD * kPiD) / v) / pow(v, 2.5);
    } else {
      const double e1 = exp(-(kPiD * kPiD) / v);
      val = sqrt(kPiD) * pow(v, -1.5) * exp(v / 4) * (1 - 2 * e1 + 4 * kPiD * kPiD * e1 / v);
    }
  }
  return val;
}

// e^x through MUFU.EX2 (2 ulp + the rounding of x log2 e: relative error ~1.2e-7 |x|; every use below has
// either |x| small or a result that is negligible against 1)
SO3D_HD float exp_fast(float x) {
#if defined(__CUDA_ARCH__)
  return fast_ex2(x * 1.4426950408889634f);
#else
  return expf(x);
#endif
}

// fp32 closed form: log f and g = d log f / d omega, stable for eps <= 1 (3 images: <= 1e-6 rel, measured).
//   f = sqrt(pi) v^-3/2 e^{v/4} e^{-w^2/4v} B(w) / (2 sin(w/2)),
//   B = w - (w - 2pi) E1 - (w + 2pi) E2,  E1 = e^{-pi(pi-w)/v}, E2 = e^{-pi(pi+w)/v}
//   g = -w/(2v) + (B'/B - 1/w) + (1/w - cot(w/2)/2)
//   w B' - B = E1 [-2pi - (pi w/v)(w - 2pi)] + E2 [2pi + (pi w/v)(w + 2pi)]
// Written in terms of dm = E1 - E2 = 2E sinh(y), sm = E1 + E2 = 2E cosh(y), E = e^{-pi^2/v}, y = pi w/v:
//   B/w        = (1 - sm) + 2 pi dm / w
//   (wB'-B)/w^2 = [ -(2pi + y w) dm + 2 pi y sm ] / w^2
// For y < 1/2 the sinh/cosh Taylor series remove the E1 - E2 and y cosh y - sinh y cancellations and
// every division by w, so w = 0 needs no special case (limit: B/w = 1 - 2E + 4 pi^2 E / v, g = 0).
// Division-free: reciprocals are MUFU.RCP (1/v with one Newton step, since it multiplies the large w^2/4);
// sin/cos of w/2 come from one sincos_fast; the three logarithms are merged into one.
SO3D_HD void igso3_closed_f32(float w, float eps, float* logf_out, float* g_out) {
  const float v = eps * eps;
  float iv = rcp_approx(v);
  iv = iv * fmaf(-v, iv, 2.0f);
  const float piv = kPi * iv;
  const float y = piv * w;
  const float rw = rcp_approx(fmaxf(w, 1e-30f));
  float bw, ratio;  // B/w and (wB' - B)/(w B)
  if (y < 0.5f) {
    const float E = exp_fast(-kPi * piv);
    const float y2 = y * y;
    const float sinhc = fmaf(y2, fmaf(y2, fmaf(y2, fmaf(y2, 2.7557319e-6f, 1.9841270e-4f), 8.3333333e-3f), 1.6666667e-1f), 1.0f);
    const float coshy = fmaf(y2, fmaf(y2, fmaf(y2, fmaf(y2, 2.4801587e-5f, 1.3888889e-3f), 4.1666667e-2f), 0.5f), 1.0f);
    const float p3 = y * fmaf(y2, fmaf(y2, fmaf(y2, 2.2045855e-5f, 1.1904762e-3f), 3.3333333e-2f), 3.3333333e-1f);  // (y cosh y - sinh y)/y^2
    const float dm_w = 2.0f * E * piv * sinhc;  // (E1 - E2)/w
    bw = (1.0f - 2.0f * E * coshy) + kTwoPi * dm_w;
    const float n2 = fmaf(-piv * w, dm_w, 2.0f * kTwoPi * E * piv * piv * p3);  // (wB' - B)/w^2
    ratio = n2 * rcp_approx(bw);
  } else {
    // pi - w with pi carried as hi + lo: near w = pi the image weight is e^{-(pi/v)(pi - w)} and an 8.7e-8
    // error in fp32 pi would be amplified by pi/v
    const float e1 = exp_fast(-piv * ((kPi - w) + (-8.742278e-8f)));
    const float e2 = exp_fast(-piv * (kPi + w));
    const float dm = e1 - e2, sm = e1 + e2;
    bw = (1.0f - sm) + kTwoPi * dm * rw;
    ratio = (fmaf(-(kTwoPi + y * w), dm, kTwoPi * y * sm)) * (rw * rw) * rcp_approx(bw);
  }
  float sh, ch;
  sincos_fast(0.5f * w, &sh, &ch);
  const float w2 = w * w;
  // w / (2 sin(w/2))  and  phi(w) = 1/w - cot(w/2)/2 (the part of g that cancels against the 1/w of the bracket)
  const float rsh = rcp_approx(fmaxf(sh, 1e-30f));
  const float wr = (w < 0.1f) ? fmaf(w2, fmaf(w2, 1.2152778e-3f, 4.1666667e-2f), 1.0f) : 0.5f * w * rsh;
  // w/12 + w^3/720 + w^5/30240 + w^7/1209600
  const float phi = (w < 0.5f) ? w * fmaf(w2, fmaf(w2, fmaf(w2, 8.2671958e-7f, 3.3068783e-5f), 1.3888889e-3f), 8.3333333e-2f)
                               : fmaf(-0.5f * ch, rsh, rw);
  // v^-3/2 from MUFU.RSQ with one Newton step
  float r = rsqrt_approx(v);
  r = r * fmaf(-0.5f * v * r, r, 1.5f);
  *logf_out = fmaf(0.25f, v, -0.25f * w2 * iv) + logf(1.7724538509055159f * (r * r * r) * (bw * wr));
  *g_out = fmaf(-0.5f * w, iv, ratio + phi);
}

// ------------------------------------------------------------------------------------------------
// IGSO(3) truncated series (SURVEY A.1) in character form,
//     f(w) = 2 F(w),   F = sum_{l<L} A_l chi_l(w),   A_l = (l+1/2) exp(-l(l+1) eps^2),
//     chi_l(w) = sin((l+1/2)w)/sin(w/2) = 1 + 2 sum_{m<=l} cos(m w)   (no 0/0 at w = 0),
// summed by Clenshaw's backward recurrence in Reinsch's difference form.  chi_l obeys
// chi_{l+1} = (2 - kappa) chi_l - chi_{l-1}, kappa = 4 sin^2(w/2), chi_0 = 1, chi_{-1} = -1, so with
//     d_l = A_l - kappa b_{l+1} + d_{l+1},        b_l = b_{l+1} + d_l          (b_L = d_L = 0)
// the sum is F = b_0 + b_1.  F depends on w only through kappa, so the recurrence is differentiated w.r.t. kappa:
//     d'_l = -b_{l+1} - kappa b'_{l+1} + d'_{l+1},   b'_l = b'_{l+1} + d'_l,   dF/dw = kappa' (b'_0 + b'_1),  kappa' = 2 sin w,
// hence d log f / dw = F'/F with no cancellation against cot(w/2) and nothing to special-case at w = 0 (kappa' = 0 there).
// (Differentiating w.r.t. w instead, d'_l = -kappa' b_{l+1} - kappa b'_{l+1} + d'_{l+1}, costs an fma where the kappa form
// has a subtraction: one more register operand per term.  SO3D_SERIES_DERIV=0 keeps that form.)
// No sin/cos of (l w) is ever formed: the previous design rotated (sin, cos)(m w) term by term and
// re-anchored it with an exact-product sincos every 32 terms (13 FP32 + 1 MUFU per term); this form
// needs 8 FP32 + 1 MUFU.EX2 per term, no anchors, and is MORE accurate (measured on the E-set,
// oracle/proto_series_fp32.py: max rel err of f 1.5e-6 vs 3.4e-6 for w <= 3.5 eps; the plain
// Clenshaw form with K = 2 cos w is 3e-4 there because of the rounding of K, hence Reinsch).
// Per term, all fp32:  x = mm * cexp;  A = ex2(x) * mh;  t = A + d;  d = fma(-kappa, b, t);
//   u = d' - b;  d' = fma(-kappa, b', u);  b += d;  b' += d'.
// m(m+1) is exact in fp32 for m < 2896.
//
// The row-invariant factors {m + 1/2, m(m+1)} come from a constant-memory table and reach the FP32 pipe
// as uniform-register operands (LDCU + FMUL R, R, UR).  Measured on B200 (profiles/microbench/pipes.cu)
// FP32 instruction throughput is set by vector-register operand reads: 3-register FFMA 85, 2-register
// forms 117, 1-register forms 129 lanes/clk/SM -- so each factor kept out of the vector register file
// is a direct saving.  Packing two rows per thread as f32x2 (igso3_series_branch_l2 in so3d_lanes.cuh) reads about as
// many operand words per flop, but cuts the issue slots per row-term from 9 to 5, and issue was the binding floor: measured 10.42 -> 8.66 ms at L = 2000, 2^24 rows, the same bits (profiles/r06a_series_lanes.jsonl).
// The kappa-form derivative then takes the packed term from 34 to 32 register words (profiles/sass_series_reads.py), with XU
// and operand reads both at 16 clk per packed term: measured 8.65 -> 8.36 ms on B200 (profiles/r07a_series_forms.jsonl).
// Also measured (profiles/r01l_series_ab.jsonl): deriving every second weight by a multiply, e_{l-1} = e_l rho_l,
// rho_{l-2} = rho_l 2^(4c) (half the MUFU, +0.5 FMUL per term) is SLOWER, 12.9 vs 12.2 clk per warp-term: the
// FP32 operand bandwidth is the wall, not the XU pipe.
// ------------------------------------------------------------------------------------------------
// Source-form knobs of the unrolled block.  The arithmetic is the same in every form; what changes is the order ptxas's
// list scheduler emits the 9 instructions per term in, and with it how often the FP32 pipe waits for register ports
// and the MUFU queue.  Measured on B200, L = 2000, 2^24 evaluations (profiles/r02m_series_variants.jsonl):
//   order 0 / block 32: 11.02 ms (12.22 clk per warp-term)     order 1 / block 64: 10.68 ms (11.85)  <- shipped
//   order 0 / block 64: 12.01      order 1 / block 32: 10.98      order 2 / block 64: 10.89      order 3 / block 64: 10.69
//   blocks 16, 48, 56, 72, 80, 96, 128 with the best order: 10.89 .. 11.64
#ifndef SO3D_SERIES_BLOCK
#define SO3D_SERIES_BLOCK 32
#endif
#ifndef SO3D_SERIES_ORDER
#define SO3D_SERIES_ORDER 0
#endif
#ifndef SO3D_SERIES_ROUNDUP
#define SO3D_SERIES_ROUNDUP 1
#endif
// Variable the derivative chain differentiates in: 1 (shipped) kappa, F' = kappa' (b'_0 + b'_1) after the loop; 0 w, the
// form before it (kappa' inside the loop, one more register operand per term).  The warp-split form below stays in w.
#ifndef SO3D_SERIES_DERIV
#define SO3D_SERIES_DERIV 1
#endif
constexpr int kSeriesBlock = SO3D_SERIES_BLOCK;       // unrolled terms per block
constexpr int kSeriesMaxTerms = 2896;  // m(m+1) is exact in fp32 below this

// Table layout.  0 (shipped): two float arrays, one LDCU.64 per term ({mh, mh'} and {mm, mm'} alternately).
// 1: one 16-byte record per PAIR of terms, {m+1/2, m(m+1)} for m = 2j and 2j+1, read with one ld.const.v4 -- meant to
// halve the constant loads (LDCU.128 per two terms, 9 -> 8.5 issue slots per term), but ptxas 12.9 splits the vector load
// into two LDCU.64 again (it keeps uniform-register live ranges short), so the layout buys nothing; kept as a knob.
#ifndef SO3D_SERIES_TAB4
#define SO3D_SERIES_TAB4 0
#endif
#if SO3D_SERIES_TAB4
struct alignas(16) SeriesPair {
  float x, y, z, w;  // mh(2j), mm(2j), mh(2j+1), mm(2j+1)
};
struct alignas(16) SeriesTab {
  SeriesPair pair[(kSeriesMaxTerms + kSeriesBlock) / 2 + 1];
};
constexpr SeriesTab make_series_tab() {
  SeriesTab t{};
  for (int j = 0; j < (kSeriesMaxTerms + kSeriesBlock) / 2 + 1; ++j) {
    const int m = 2 * j;
    t.pair[j].x = (float)m + 0.5f;
    t.pair[j].y = (float)((double)m * (double)(m + 1));
    t.pair[j].z = (float)(m + 1) + 0.5f;
    t.pair[j].w = (float)((double)(m + 1) * (double)(m + 2));
  }
  return t;
}
#else
struct alignas(16) SeriesTab {
  float mh[kSeriesMaxTerms + kSeriesBlock];  // m + 1/2
  float mm[kSeriesMaxTerms + kSeriesBlock];  // m (m + 1)
};
constexpr SeriesTab make_series_tab() {
  SeriesTab t{};
  for (int m = 0; m < kSeriesMaxTerms + kSeriesBlock; ++m) {
    t.mh[m] = (float)m + 0.5f;
    t.mm[m] = (float)((double)m * (double)(m + 1));
  }
  return t;
}
#endif
#if defined(__CUDACC__) && !defined(SO3D_HOST_ONLY)
__constant__ SeriesTab c_series_tab = make_series_tab();
#endif
static constexpr SeriesTab h_series_tab = make_series_tab();

#if SO3D_SERIES_TAB4
SO3D_HD SeriesPair series_pair(int j) {
#if defined(__CUDA_ARCH__)
  const float4 v = *reinterpret_cast<const float4*>(&c_series_tab.pair[j]);  // one ld.const.v4 -> LDCU.128
  return SeriesPair{v.x, v.y, v.z, v.w};
#else
  return h_series_tab.pair[j];
#endif
}
SO3D_HD float series_mh(int m) {
  const SeriesPair p = series_pair(m >> 1);
  return (m & 1) ? p.z : p.x;
}
SO3D_HD float series_mm(int m) {
  const SeriesPair p = series_pair(m >> 1);
  return (m & 1) ? p.w : p.y;
}
#else
SO3D_HD float series_mh(int m) {
#if defined(__CUDA_ARCH__)
  return c_series_tab.mh[m];
#else
  return h_series_tab.mh[m];
#endif
}
SO3D_HD float series_mm(int m) {
#if defined(__CUDA_ARCH__)
  return c_series_tab.mm[m];
#else
  return h_series_tab.mm[m];
#endif
}
#endif

struct SeriesAcc {
  float F, dF;  // sum (l+1/2) e_l chi_l  and its derivative w.r.t. w:  f = 2 F,  d log f / dw = dF / F
};

struct SeriesState {
  float b, d;    // b_{l+1}, d_{l+1}
  float bp, dp;  // b'_{l+1}, d'_{l+1}
  float b2, bp2; // b_{l+2}, b'_{l+2}
};

// The derivative chain's source term, the derivative of -kappa b_{l+1}: -b_{l+1} in the kappa form (a subtraction),
// -kappa' b_{l+1} in the w form (an fma with kappa' = 2 sin w)
SO3D_HD float series_dsrc(float kapp, float b, float dp) {
#if SO3D_SERIES_DERIV
  (void)kapp;
  return dp - b;
#else
  return fmaf(-kapp, b, dp);
#endif
}
// dF/dw from the chain's b'_0 + b'_1: times kappa' = dkappa/dw in the kappa form
SO3D_HD float series_dF(float kapp, float bp_sum) {
#if SO3D_SERIES_DERIV
  return kapp * bp_sum;
#else
  (void)kapp;
  return bp_sum;
#endif
}

// terms l = hi, hi-1, ..., hi-count+1 (descending)
template <int kUnroll>
SO3D_HD void igso3_series_run(SeriesState& st, float kap, float kapp, float cexp, int hi, int count) {
#pragma unroll kUnroll
  for (int i = 0; i < count; ++i) {
    const int l = hi - i;
#if SO3D_SERIES_ORDER == 0
    const float A = fast_ex2(series_mm(l) * cexp) * series_mh(l);
    const float dn = fmaf(-kap, st.b, A + st.d);
    const float dpn = fmaf(-kap, st.bp, series_dsrc(kapp, st.b, st.dp));
    st.b2 = st.b;
    st.bp2 = st.bp;
    st.b += dn;
    st.bp += dpn;
    st.d = dn;
    st.dp = dpn;
#elif SO3D_SERIES_ORDER == 1  // derivative chain first
    const float dpn = fmaf(-kap, st.bp, series_dsrc(kapp, st.b, st.dp));
    const float A = fast_ex2(series_mm(l) * cexp) * series_mh(l);
    const float dn = fmaf(-kap, st.b, A + st.d);
    st.b2 = st.b;
    st.bp2 = st.bp;
    st.bp += dpn;
    st.b += dn;
    st.dp = dpn;
    st.d = dn;
#elif SO3D_SERIES_ORDER == 3  // derivative chain first, each chain's updates kept together
    const float dpn = fmaf(-kap, st.bp, series_dsrc(kapp, st.b, st.dp));
    st.bp2 = st.bp;
    st.bp += dpn;
    st.dp = dpn;
    const float A = fast_ex2(series_mm(l) * cexp) * series_mh(l);
    const float dn = fmaf(-kap, st.b, A + st.d);
    st.b2 = st.b;
    st.b += dn;
    st.d = dn;
#else  // kap-products grouped: t = d - kap b, u = dp - kapp b
    const float t = fmaf(-kap, st.b, st.d);
    const float u = series_dsrc(kapp, st.b, st.dp);
    const float dn = fmaf(fast_ex2(series_mm(l) * cexp), series_mh(l), t);
    const float dpn = fmaf(-kap, st.bp, u);
    st.b2 = st.b;
    st.bp2 = st.bp;
    st.b += dn;
    st.bp += dpn;
    st.d = dn;
    st.dp = dpn;
#endif
  }
}

// Evaluate terms l = 0 .. L-1.
SO3D_HD SeriesAcc igso3_series_terms(float w, float eps, int L) {
  const float cexp = -(eps * eps) * 1.4426950408889634f;
  float sh, ch;
  sincos_f(0.5f * w, &sh, &ch);
  const float kap = 4.0f * sh * sh, kapp = 4.0f * sh * ch;
  SeriesState st;
  st.b = st.d = st.bp = st.dp = st.b2 = st.bp2 = 0.f;
  const int ragged = L % kSeriesBlock;  // top partial block first, so that full blocks are block-aligned
  if (ragged) igso3_series_run<1>(st, kap, kapp, cexp, L - 1, ragged);  // (an unrolled 16-term form of this partial block made the whole kernel 0.3 % slower)
  // block index as the loop variable: table offsets are provably 128-byte aligned -> LDCU.128
  for (int blk = L / kSeriesBlock - 1; blk >= 0; --blk)
    igso3_series_run<kSeriesBlock>(st, kap, kapp, cexp, blk * kSeriesBlock + (kSeriesBlock - 1), kSeriesBlock);
  return SeriesAcc{st.b + st.b2, series_dF(kapp, st.bp + st.bp2)};
}

// terms l = 0 .. L-1 in one rolled loop (igso3_series_run<1>): bit-identical to igso3_series_terms, tiny code
#ifndef SO3D_AUTO_SERIES_ROLLED
#define SO3D_AUTO_SERIES_ROLLED 1
#endif
SO3D_HD SeriesAcc igso3_series_terms_rolled(float w, float eps, int L) {
  const float cexp = -(eps * eps) * 1.4426950408889634f;
  float sh, ch;
  sincos_f(0.5f * w, &sh, &ch);
  const float kap = 4.0f * sh * sh, kapp = 4.0f * sh * ch;
  SeriesState st;
  st.b = st.d = st.bp = st.dp = st.b2 = st.bp2 = 0.f;
  igso3_series_run<1>(st, kap, kapp, cexp, L - 1, L);
  return SeriesAcc{st.b + st.b2, series_dF(kapp, st.bp + st.bp2)};
}

// ------------------------------------------------------------------------------------------------
// The same series with ONE WARP per rotation (small batches: a one-thread-per-rotation launch of 4096 rows is a single
// 2000-term dependent chain per thread, ~40 us, with most of the GPU idle).  The backward recurrence is linear in its
// state s = (b, d; b', d'), so the term range splits over the 32 lanes:
//   * lane j runs the recurrence over its own block of kLaneTerms terms, l = B j + B - 1 ... B j, from a zero state -> c_j;
//   * what the lower blocks' steps do to c_j is the HOMOGENEOUS recurrence (A = 0) applied B j times:
//         (b, d) <- P (b, d),   P = [[1 - kappa, 1], [-kappa, 1]],   and for the derivative parts  T = [[P, 0], [dP/dw, P]];
//     every lane obtains G = P^B (and dG/dw) by carrying the two unit vectors through its own B steps alongside the
//     block, raises it to the j-th power by binary exponentiation (pairs (M, dM/dw), product rule), applies it to c_j;
//   * the 32 propagated states are summed with __shfl_xor_sync:  F = 2 b - d,  F' = 2 b' - d'.
// ~20 instructions per term and lane instead of 9, but 64 terms per lane instead of 2000.  Not the same rounding path as
// the one-thread recurrence (the sums are associated differently): checked against the fp64 series to the same 1e-5
// bound (tests/test_host_math.py::test_series_warp_split, GPU: test_logp_score_series_small_batch_warp_split).
// ------------------------------------------------------------------------------------------------
struct SeriesLaneState {
  float b, d, bp, dp;
};
struct Mat2D {  // a 2x2 matrix and its derivative w.r.t. omega
  float a11, a12, a21, a22, d11, d12, d21, d22;
};
SO3D_HD Mat2D mat2d_mul(const Mat2D& x, const Mat2D& y) {  // (X Y, X' Y + X Y')
  Mat2D r;
  r.a11 = fmaf(x.a11, y.a11, x.a12 * y.a21);
  r.a12 = fmaf(x.a11, y.a12, x.a12 * y.a22);
  r.a21 = fmaf(x.a21, y.a11, x.a22 * y.a21);
  r.a22 = fmaf(x.a21, y.a12, x.a22 * y.a22);
  r.d11 = fmaf(x.d11, y.a11, fmaf(x.d12, y.a21, fmaf(x.a11, y.d11, x.a12 * y.d21)));
  r.d12 = fmaf(x.d11, y.a12, fmaf(x.d12, y.a22, fmaf(x.a11, y.d12, x.a12 * y.d22)));
  r.d21 = fmaf(x.d21, y.a11, fmaf(x.d22, y.a21, fmaf(x.a21, y.d11, x.a22 * y.d21)));
  r.d22 = fmaf(x.d21, y.a12, fmaf(x.d22, y.a22, fmaf(x.a21, y.d12, x.a22 * y.d22)));
  return r;
}
// Lane `lane` of 32: its block's state propagated to l = 0.  B = terms per lane (32 B >= L); terms l >= L weigh 0.
// (Carrying only ONE homogeneous sequence S_m = sin(m w)/sin(w) and deriving P^m = [[S_{m+1} - S_m, S_m], [-kappa S_m,
// S_m - S_{m-1}]] from it halves the homogeneous work, but the difference S_{m+1} - S_m loses 6 bits at small w and the
// powers amplify it: 1.1e-5 instead of 1.6e-6 on the E-set.  Both unit vectors are carried.)
SO3D_HD SeriesLaneState igso3_series_lane(float kap, float kapp, float cexp, int lane, int B, int L) {
  float b = 0.f, d = 0.f, bp = 0.f, dp = 0.f;
  // images of the unit vectors e_b = (1, 0) and e_d = (0, 1) under the homogeneous steps, and their derivatives
  float ub = 1.f, ud = 0.f, vb = 0.f, vd = 1.f, upb = 0.f, upd = 0.f, vpb = 0.f, vpd = 0.f;
  float lf = (float)(B * lane + B - 1);
  const float Lf = (float)L;
#pragma unroll 4
  for (int i = 0; i < B; ++i) {
    const float mm = fmaf(lf, lf, lf);  // l (l + 1), exact below 2^24
    const float A = lf < Lf ? fast_ex2(mm * cexp) * (lf + 0.5f) : 0.f;
    const float dpn = fmaf(-kap, bp, fmaf(-kapp, b, dp));
    const float dn = fmaf(-kap, b, A + d);
    bp += dpn;
    b += dn;
    dp = dpn;
    d = dn;
    const float updn = fmaf(-kap, upb, fmaf(-kapp, ub, upd)), vpdn = fmaf(-kap, vpb, fmaf(-kapp, vb, vpd));
    const float udn = fmaf(-kap, ub, ud), vdn = fmaf(-kap, vb, vd);
    upb += updn;
    vpb += vpdn;
    ub += udn;
    vb += vdn;
    upd = updn;
    vpd = vpdn;
    ud = udn;
    vd = vdn;
    lf -= 1.0f;
  }
  // G = P^B: columns are the images of e_b and e_d, rows are (b, d)
  Mat2D g{ub, vb, ud, vd, upb, vpb, upd, vpd};
  Mat2D acc{1.f, 0.f, 0.f, 1.f, 0.f, 0.f, 0.f, 0.f};
  for (int bit = 0; bit < 5; ++bit) {  // acc = G^lane
    if ((lane >> bit) & 1) acc = mat2d_mul(acc, g);
    if ((lane >> (bit + 1)) != 0) g = mat2d_mul(g, g);
  }
  SeriesLaneState o;
  o.b = fmaf(acc.a11, b, acc.a12 * d);
  o.d = fmaf(acc.a21, b, acc.a22 * d);
  o.bp = fmaf(acc.d11, b, fmaf(acc.d12, d, fmaf(acc.a11, bp, acc.a12 * dp)));
  o.dp = fmaf(acc.d21, b, fmaf(acc.d22, d, fmaf(acc.a21, bp, acc.a22 * dp)));
  return o;
}
// Terms the warp actually needs: the weights beyond igso3_series_live_terms(eps) are exactly 0 (ex2.approx.ftz flushes them), so
// summing min(L, live) terms gives the bits of summing L -- and with one rotation per warp the count is warp-uniform.
// Below 32 live terms the count is rounded up to one term per lane, but never past L: terms l >= L must not be summed.
SO3D_HD int igso3_series_live_terms(float eps, int L);
SO3D_HD int igso3_series_warp_terms(float eps, int L) {
  const int live = igso3_series_live_terms(eps, L);
  return live < 32 ? (L < 32 ? L : 32) : live;
}
SO3D_HD int igso3_series_lane_terms(int L) { return (L + 31) / 32; }
SO3D_HD void igso3_series_lane_setup(float w, float eps, float* kap, float* kapp, float* cexp) {
  *cexp = -(eps * eps) * 1.4426950408889634f;
  float sh, ch;
  sincos_f(0.5f * w, &sh, &ch);
  *kap = 4.0f * sh * sh;
  *kapp = 4.0f * sh * ch;
}
// host-side statement of the warp reduction (same butterfly order as __shfl_xor_sync with offsets 16, 8, 4, 2, 1)
SO3D_HD void igso3_series_warp_host(float w, float eps, int L, float* logf_out, float* g_out, bool guarded) {
  float kap, kapp, cexp;
  igso3_series_lane_setup(w, eps, &kap, &kapp, &cexp);
  const int Lw = igso3_series_warp_terms(eps, L);
  const int B = igso3_series_lane_terms(Lw);
  SeriesLaneState s[32];
  for (int j = 0; j < 32; ++j) s[j] = igso3_series_lane(kap, kapp, cexp, j, B, Lw);
  for (int off = 16; off > 0; off >>= 1) {
    SeriesLaneState t[32];
    for (int j = 0; j < 32; ++j) {
      const SeriesLaneState& o = s[j ^ off];
      t[j] = SeriesLaneState{s[j].b + o.b, s[j].d + o.d, s[j].bp + o.bp, s[j].dp + o.dp};
    }
    for (int j = 0; j < 32; ++j) s[j] = t[j];
  }
  const float F = 2.0f * s[0].b - s[0].d, dF = 2.0f * s[0].bp - s[0].dp;
  *logf_out = logf(2.0f * F);
  *g_out = dF / F;
  if (guarded && eps <= 1.0f && w > 4.2f * eps) igso3_closed_f32(w, eps, logf_out, g_out);
}

// Number of leading terms whose weight 2^(l(l+1) cexp) is not flushed to zero (ex2.approx.ftz
// returns 0 below 2^-126): skipping the rest is bit-identical to summing them.
SO3D_HD int igso3_series_live_terms(float eps, int L) {
  const float lim = 9.36f / eps + 2.0f;  // l(l+1) eps^2 log2(e) > 126  <=>  l > ~9.35/eps
  return lim < (float)L ? (int)lim : L;
}

enum IgsoMode { kSeries = 0, kClosed = 1, kAuto = 2, kSeriesAdaptive = 3, kSeriesPure = 4 };
constexpr float kAutoSeriesEps = 1.0f;  // auto: closed form up to eps = 1 (3 images: <= 1e-6 rel, measured), series (<= 12 live terms) above

// Conditioning guard of the fp32 series.  F = sum_l A_l chi_l(w) is an alternating sum whose condition number
// cond = sum |A_l chi_l| / |F| depends on w/eps only (fp64, eps = 6.4e-3 .. 0.5): 4.5 at w = 3.5 eps, 14 at 4.2 eps,
// 26 at 4.5 eps, 75 at 5 eps, 155 at 5.3 eps, 386 at 5.66 eps (the edge of the E-set, k = 4).  The fp32 evaluation
// measures ~4 u cond in the worst row (u = 6e-8): 3.5e-6 at 4.2 eps, 1.2e-5 at 4.9 eps, 6e-5 at 5.66 eps -- and that
// is not the recurrence's fault: with the recurrence carried in fp64 and only the weights A_l rounded to fp32 the
// E-set still shows 2.3e-5 at k ~ 4, with exactly rounded weights in the fp32 recurrence 5e-5 (DESIGN.md 4.1).
// north_star's 1e-5 is out of reach of ANY single-precision l-series beyond w ~ 4.8 eps.  The series modes therefore
// run every row's L terms (the loop is warp-uniform) and then REPLACE the result of the rows with
// w > kSeriesGuard eps, eps <= 1 by the closed form (the Poisson dual of the same series: 3 images, <= 2e-6 there).
// kSeriesPure keeps the raw series everywhere.
constexpr float kSeriesGuard = 4.2f;

// log f_eps(w) and g = d log f / dw by the evaluator kMode (a template parameter, so that a kernel contains one
// evaluator only and the exact-L series keeps a provably warp-uniform trip count: its table operands must stay
// uniform-register loads).
// Where the guard's closed form is evaluated relative to the L-term loop, and whether it is inlined.  The arithmetic is
// the same in every form; what changes is ptxas's register allocation and list schedule of the unrolled series block,
// which moves the kernel by +-15 % (measured, profiles/r03b_series_variants.jsonl; see the source-form knobs above):
//   0: after the loop, inlined        1: after the loop, out of line (__noinline__)
//   2: before the loop, inlined       3: before the loop, out of line
#ifndef SO3D_SERIES_GUARD_FORM
#define SO3D_SERIES_GUARD_FORM 3
#endif
#if defined(__CUDACC__) && !defined(SO3D_HOST_ONLY)
static __host__ __device__ __noinline__ void igso3_closed_f32_outofline(float w, float eps, float* logf_out, float* g_out) {
  igso3_closed_f32(w, eps, logf_out, g_out);
}
#else
inline void igso3_closed_f32_outofline(float w, float eps, float* logf_out, float* g_out) { igso3_closed_f32(w, eps, logf_out, g_out); }
#endif

// auto's series branch (eps > 1: at most 12 live terms) can be compiled out of line (SO3D_AUTO_SERIES_OUTOFLINE=1) so that the
// HBM-bound kernels that evaluate `auto` do not carry the unrolled series block inline.  Measured (profiles/r04u_probe.jsonl):
// 20 % fewer instructions in those kernels and SLOWER -- auto score 0.1675 -> 0.175 ms, forward noising with the score
// 0.3637 -> 0.378 ms (the call's register conventions cost more on the hot path than the inline block's size) -- so it is off.
// (Again with the closed form evaluated first and the call only on the rare override, r05i: 0.1655 -> 0.1735 ms, 0.3595 -> 0.376.)
#ifndef SO3D_AUTO_SERIES_OUTOFLINE
#define SO3D_AUTO_SERIES_OUTOFLINE 0
#endif
#ifndef SO3D_AUTO_CLOSED_FIRST
#define SO3D_AUTO_CLOSED_FIRST 1
#endif
template <int kMode>
SO3D_HD void igso3_series_branch(float w, float eps, int L, float* logf_out, float* g_out);
#if defined(__CUDACC__) && !defined(SO3D_HOST_ONLY)
static __host__ __device__ __noinline__ void igso3_auto_series_outofline(float w, float eps, int L, float* logf_out, float* g_out);
#else
inline void igso3_auto_series_outofline(float w, float eps, int L, float* logf_out, float* g_out);
#endif

template <int kMode>
SO3D_HD void igso3_logf_g_t(float w, float eps, int L, float* logf_out, float* g_out) {
  if (kMode == kAuto && SO3D_AUTO_CLOSED_FIRST) {
    // the closed form unconditionally and straight-line (so that ptxas can interleave it with the neighbouring row's / the
    // surrounding arithmetic), then the rare rows above eps = 1 are re-evaluated by the series: the same bits as branching first
    igso3_closed_f32(w, eps, logf_out, g_out);
    if (!(eps <= kAutoSeriesEps)) {
      if (SO3D_AUTO_SERIES_OUTOFLINE) igso3_auto_series_outofline(w, eps, L, logf_out, g_out);
      else igso3_series_branch<kAuto>(w, eps, L, logf_out, g_out);
    }
  } else if (kMode == kClosed || (kMode == kAuto && eps <= kAutoSeriesEps)) {
    igso3_closed_f32(w, eps, logf_out, g_out);
  } else if (kMode == kAuto && SO3D_AUTO_SERIES_OUTOFLINE) {
    igso3_auto_series_outofline(w, eps, L, logf_out, g_out);
  } else {
    igso3_series_branch<kMode>(w, eps, L, logf_out, g_out);
  }
}

template <int kMode>
SO3D_HD void igso3_series_branch(float w, float eps, int L, float* logf_out, float* g_out) {
  {
    int terms = L;
    if (kMode == kAuto || kMode == kSeriesAdaptive) {
      terms = igso3_series_live_terms(eps, L);
#if defined(__CUDA_ARCH__)
      // keep the trip count (and with it the constant-table index) the same across the warp: a lane-varying index
      // would serialise the constant loads.  The extra terms have weight exactly 0, so the result is unchanged.
      terms = __reduce_max_sync(__activemask(), terms);
#endif
#if SO3D_SERIES_ROUNDUP
      // whole blocks only: the extra terms have weight exactly 0 as well, and the partial-block loop is the slow one
      if (!(kMode == kAuto && SO3D_AUTO_SERIES_ROLLED)) {
        const int up = (terms + kSeriesBlock - 1) / kSeriesBlock * kSeriesBlock;
        terms = up <= L ? up : L;
      }
#endif
    }
    constexpr bool kGuarded = (kMode == kSeries || kMode == kSeriesAdaptive);
    const bool guard = kGuarded && eps <= kAutoSeriesEps && w > kSeriesGuard * eps;
    float lf_c = 0.f, g_c = 0.f;
    if (kGuarded && (SO3D_SERIES_GUARD_FORM == 2 || SO3D_SERIES_GUARD_FORM == 3) && guard) {
      if (SO3D_SERIES_GUARD_FORM == 3) igso3_closed_f32_outofline(w, eps, &lf_c, &g_c);
      else igso3_closed_f32(w, eps, &lf_c, &g_c);
    }
    // auto reaches this branch only above eps = 1, where at most 12 terms are live: a rolled loop over exactly those (the same
    // operations per term as the unrolled blocks, whose extra terms weigh exactly 0: the same bits) keeps the unrolled block out
    // of the HBM-bound kernels that evaluate `auto`
    const SeriesAcc a = (kMode == kAuto && SO3D_AUTO_SERIES_ROLLED) ? igso3_series_terms_rolled(w, eps, terms) : igso3_series_terms(w, eps, terms);
    *logf_out = logf(2.0f * a.F);
    *g_out = a.dF / a.F;
    if (kGuarded && guard) {
      if (SO3D_SERIES_GUARD_FORM == 0) igso3_closed_f32(w, eps, logf_out, g_out);
      else if (SO3D_SERIES_GUARD_FORM == 1) igso3_closed_f32_outofline(w, eps, logf_out, g_out);
      else { *logf_out = lf_c; *g_out = g_c; }
    }
  }
}
#if defined(__CUDACC__) && !defined(SO3D_HOST_ONLY)
static __host__ __device__ __noinline__ void igso3_auto_series_outofline(float w, float eps, int L, float* logf_out, float* g_out) {
  igso3_series_branch<kAuto>(w, eps, L, logf_out, g_out);
}
#else
inline void igso3_auto_series_outofline(float w, float eps, int L, float* logf_out, float* g_out) { igso3_series_branch<kAuto>(w, eps, L, logf_out, g_out); }
#endif

// runtime-mode dispatch (host harness, non-critical call sites)
SO3D_HD void igso3_logf_g(float w, float eps, int mode, int L, float* logf_out, float* g_out) {
  switch (mode) {
    case kSeries: igso3_logf_g_t<kSeries>(w, eps, L, logf_out, g_out); break;
    case kClosed: igso3_logf_g_t<kClosed>(w, eps, L, logf_out, g_out); break;
    case kAuto: igso3_logf_g_t<kAuto>(w, eps, L, logf_out, g_out); break;
    case kSeriesPure: igso3_logf_g_t<kSeriesPure>(w, eps, L, logf_out, g_out); break;
    default: igso3_logf_g_t<kSeriesAdaptive>(w, eps, L, logf_out, g_out); break;
  }
}

// ------------------------------------------------------------------------------------------------
// Inverse-CDF angle lookup.  distributions.py:38-49, float32 like the reference.
//   i1 = #{j : trap[j] <= u}  (binary search; trap is non-decreasing), i0 = max(i1 - 1, 0),
//   w = clamp((u - trap[i0]) / max(trap[i1] - trap[i0], 1e-6), 0, 1),  angle = lerp(loc[i0], loc[i1], w)
// `trap` may point to shared or global memory.  loc[j] = pi ((j+1)/999)^3 is passed as a table so
// the values are bit-identical to the reference's float32 grid.
// ------------------------------------------------------------------------------------------------
// number of entries of the non-decreasing row trap[0..998] that are <= u, known to lie in [lo, hi]
SO3D_HD int cdf_count_le(const float* trap, float u, int lo, int hi) {
#pragma unroll 1
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (trap[mid] <= u) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// angle for a given count i1 = #{trap <= u} (distributions.py:40-49)
SO3D_HD float igso3_angle_lerp(const float* trap, const float* loc, float u, int count) {
  const int i1 = count < kCdf - 1 ? count : kCdf - 1;  // u < 1 == trap[998] so count <= 998; clamp guards u >= 1 inputs
  const int i0 = i1 > 0 ? i1 - 1 : 0;
  const float t0 = trap[i0], t1 = trap[i1];
  const float diff = fmaxf(t1 - t0, 1e-6f);
  const float wgt = fminf(fmaxf((u - t0) / diff, 0.f), 1.f);
  const float a0 = loc[i0], a1 = loc[i1];
  const float d = a1 - a0;
  // torch.lerp: w < 0.5 ? a0 + w d : a1 - d (1 - w)
  return (wgt < 0.5f) ? fmaf(wgt, d, a0) : fmaf(-d, 1.0f - wgt, a1);
}

SO3D_HD float igso3_angle_from_uniform(const float* trap, const float* loc, float u) {
  return igso3_angle_lerp(trap, loc, u, cdf_count_le(trap, u, 0, kCdf));
}

// Guide of a CDF row: guide[k] = #{j : trap[j] <= k / kGuide}, k = 0..kGuide.  k / 1024 and u * 1024 are exact in
// fp32, so for u in [k/1024, (k+1)/1024) the count lies in [guide[k], guide[k+1]] and a search restricted to that
// range returns exactly the index of the full binary search, in ~1 probe instead of 10.
//   * shared-row kernels keep the guide as uint16 counts next to the row in shared memory (sg_bucket / sg_edge below);
//   * per-row lookups through L2 use 16-byte RECORDS, one per bucket: {lo | hi << 16, trap[lo-1], trap[lo],
//     trap[lo+1]} (indices clamped to [0, 998]).  When the bucket holds at most one grid point (hi - lo <= 1, the
//     common case) ONE 16-byte load resolves the lookup: the count is lo + (trap[lo] <= u) and both CDF values of
//     the interpolation are in the record -- a single dependent memory access instead of 4-5.
//     The record buckets are NOT uniform in u.  The grid angles are cubic in the index, so the CDF entries crowd
//     towards 0 like a power law (F ~ j^9 for broad distributions) and towards 1 like a Gaussian tail: with 1024
//     uniform buckets 5.1 % of the draws of the forward schedule land in a bucket that holds several grid points and
//     fall back to a dependent binary search through L2 -- 2 lanes of every warp, so 82 % of the warps paid for it
//     (r03u: 9 % of the issue slots and a quarter of the stall samples of the forward-noising kernel).  Records
//     therefore follow the float format in both tails (bucket_of below): [2^-13, 2^-3) of u and of 1 - u are cut
//     into 64 buckets per octave (the top 6 mantissa bits), the middle [1/8, 7/8] into 1/1024 steps, and one record
//     each covers u < 2^-13 and 1 - u < 2^-13.  0.2 % of the forward draws (0.02 % of the posterior's) are left on
//     the search path; 2051 records = 32.8 KB per row.  Every bucket edge and 1 - u (u >= 1/2) are exact in fp32, so
//     the bracket [lo, hi] of a record is exact for every u that maps to it.
constexpr int kGuide = 1024;
// Shared-memory guide (shared-row kernels): uint16 counts at kSgBuckets + 1 increasing edges of u, bucket b = [edge b,
// edge b + 1].  The same float-format idea within the shared-memory budget of the two-row reverse step (7 resident CTAs):
// 64 buckets per octave of u and of 1 - u on [2^-10, 2^-2), 1/512 steps on [1/4, 3/4) -- 1282 buckets instead of 1024
// uniform ones (+516 B), and the rows that need a search drop from 2.7 % to 0.2 % (posterior tables; forward 5.1 % -> 0.9 %).
constexpr int kSgOctLo = 10, kSgOctHi = 2, kSgMant = 6, kSgMid = 512;
constexpr int kSgLog = (kSgOctLo - kSgOctHi) << kSgMant;                // 512 log buckets per tail
constexpr int kSgBias = (127 - kSgOctLo) << kSgMant;                    // float bits >> 17 of 2^-10
constexpr int kSgMid0 = kSgMid >> kSgOctHi, kSgMid1 = kSgMid - kSgMid0;  // 128 .. 384
constexpr int kSgMidBase = 1 + kSgLog;                                  // 513: first middle bucket
constexpr int kSgUpBase = kSgMidBase + (kSgMid1 - kSgMid0);             // 769: first bucket of the upper tail
constexpr int kSgBuckets = kSgUpBase + 1 + kSgLog;                      // 1282
constexpr int kGuideStride = kSgBuckets + 2;  // uint16 entries per shared-memory guide (kSgBuckets + 1 used; even)
constexpr int kGuideRecWords = 4;         // 32-bit words per record of the global guide
constexpr int kRecOctLo = 13, kRecOctHi = 3, kRecMant = 6;                        // log part: [2^-13, 2^-3), 2^6 buckets per octave
constexpr int kRecLog = (kRecOctLo - kRecOctHi) << kRecMant;                      // 640 log buckets per tail
constexpr int kRecBias = ((127 - kRecOctLo) << kRecMant);                         // float bits >> 17 of 2^-13
constexpr int kRecMid0 = kGuide >> kRecOctHi, kRecMid1 = kGuide - kRecMid0;       // uniform buckets 128 .. 896 (inclusive)
constexpr int kRecMidBase = 1 + kRecLog;                                          // first middle record
constexpr int kRecUpBase = kRecMidBase + (kRecMid1 - kRecMid0 + 1);               // first record of the upper tail
constexpr int kGuideRecs = kRecUpBase + 1 + kRecLog;                              // 2051 records per row

SO3D_HD float sg_uint_as_float(uint32_t b) {
#if defined(__CUDA_ARCH__)
  return __uint_as_float(b);
#else
  float f;
  memcpy(&f, &b, sizeof f);
  return f;
#endif
}
SO3D_HD uint32_t sg_float_as_uint(float f) {
#if defined(__CUDA_ARCH__)
  return __float_as_uint(f);
#else
  uint32_t b;
  memcpy(&b, &f, sizeof b);
  return b;
#endif
}
SO3D_HD float sg_log_edge(int j) { return sg_uint_as_float((uint32_t)(j + kSgBias) << (23 - kSgMant)); }  // j = 0 .. kSgLog (2^-2)
// edge idx = 0 .. kSgBuckets of the shared-memory guide (non-decreasing in idx; all exact in fp32)
SO3D_HD float sg_edge(int idx) {
  if (idx <= 0) return 0.f;
  if (idx <= kSgMidBase) return sg_log_edge(idx - 1);
  if (idx <= kSgUpBase) return (float)(kSgMid0 + idx - kSgMidBase) * (1.0f / (float)kSgMid);
  if (idx < kSgBuckets) return 1.0f - sg_log_edge(kSgBuckets - idx - 1);
  return 1.0f;
}
// bucket of u: sg_edge(b) <= u <= sg_edge(b + 1) for every u in [0, 1) (any other float maps to some valid bucket)
SO3D_HD int sg_bucket(float u) {
  const bool upper = u >= 0.75f;
  const float v = upper ? 1.0f - u : u;  // exact for u >= 1/2
  int kl = (int)(sg_float_as_uint(v) >> (23 - kSgMant)) - (kSgBias - 1);
  kl = kl < 0 ? 0 : (kl > kSgLog ? kSgLog : kl);
  int b = (int)(u * (float)kSgMid) + (kSgMidBase - kSgMid0);
  b = (u < 0.25f) ? kl : (upper ? (kSgBuckets - 1) - kl : b);
  return b < 0 ? 0 : (b > kSgBuckets - 1 ? kSgBuckets - 1 : b);
}

SO3D_HD float igso3_angle_from_uniform_guided(const float* trap, const float* loc, const uint16_t* guide, float u) {
  const int k = sg_bucket(u);
  const int lo = (u >= 0.f) ? (int)guide[k] : 0;
  const int hi = (u < 1.0f) ? (int)guide[k + 1] : kCdf;
  return igso3_angle_lerp(trap, loc, u, cdf_count_le(trap, u, lo, hi));
}

struct GuideRec {
  uint32_t lohi;
  float tm1, t0, tp1;
};

SO3D_HD float rec_uint_as_float(uint32_t b) {
#if defined(__CUDA_ARCH__)
  return __uint_as_float(b);
#else
  float f;
  memcpy(&f, &b, sizeof f);
  return f;
#endif
}
SO3D_HD uint32_t rec_float_as_uint(float f) {
#if defined(__CUDA_ARCH__)
  return __float_as_uint(f);
#else
  uint32_t b;
  memcpy(&b, &f, sizeof b);
  return b;
#endif
}

// lower edge of log bucket j (j = 0 .. kRecLog; j = kRecLog is 2^-3) of a tail variable v = u or 1 - u
SO3D_HD float rec_log_edge(int j) { return rec_uint_as_float((uint32_t)(j + kRecBias) << (23 - kRecMant)); }

// [a, b]: every u that maps to record k satisfies a <= u <= b (b may be the first value of the next record)
SO3D_HD void guide_rec_range(int k, float* a, float* b) {
  if (k == 0) { *a = 0.f; *b = rec_log_edge(0); }
  else if (k < kRecMidBase) { *a = rec_log_edge(k - 1); *b = rec_log_edge(k); }
  else if (k < kRecUpBase) {
    const int q = k - kRecMidBase + kRecMid0;
    *a = (float)q * (1.0f / (float)kGuide);
    *b = (float)(q + 1) * (1.0f / (float)kGuide);
  } else if (k == kRecUpBase) { *a = 1.0f - rec_log_edge(0); *b = 1.0f; }
  else { *a = 1.0f - rec_log_edge(k - kRecUpBase); *b = 1.0f - rec_log_edge(k - kRecUpBase - 1); }
}

SO3D_HD GuideRec make_guide_rec(const float* trap, int k) {
  float a, b;
  guide_rec_range(k, &a, &b);
  const int lo = cdf_count_le(trap, a, 0, kCdf);
  const int hi = cdf_count_le(trap, b, 0, kCdf);
  auto at = [&](int j) { return trap[j < 0 ? 0 : (j > kCdf - 1 ? kCdf - 1 : j)]; };
  return GuideRec{(uint32_t)lo | ((uint32_t)hi << 16), at(lo - 1), at(lo), at(lo + 1)};
}

// `rec` = the record of bucket guide_bucket(u) of this row (already loaded); trap = the row, for the rare fallback
SO3D_HD float igso3_angle_from_record(const float* trap, const float* loc, const GuideRec& rec, float u) {
  const int lo = (int)(rec.lohi & 0xffffu), hi = (int)(rec.lohi >> 16);
  if (hi - lo <= 1 && lo < kCdf - 1 && u >= 0.f && u < 1.0f) {
    const bool up = (hi > lo) && (rec.t0 <= u);  // count = lo + up;  i1 = count, i0 = max(count - 1, 0)
    const int i1 = lo + (up ? 1 : 0);
    const int i0 = i1 > 0 ? i1 - 1 : 0;
    const float t0 = up ? rec.t0 : rec.tm1, t1 = up ? rec.tp1 : rec.t0;
    const float diff = fmaxf(t1 - t0, 1e-6f);
    const float wgt = fminf(fmaxf((u - t0) / diff, 0.f), 1.f);
    const float a0 = loc[i0], a1 = loc[i1];
    const float d = a1 - a0;
    return (wgt < 0.5f) ? fmaf(wgt, d, a0) : fmaf(-d, 1.0f - wgt, a1);
  }
  const bool in01 = (u >= 0.f) && (u < 1.0f);
  // (Measured, profiles/r01n_probe_engine.jsonl: resolving 2..8-point buckets with one batch of nine independent
  // loads instead of this dependent search is SLOWER, 0.459 vs 0.442 ms for the forward-noising kernel -- the kernel
  // is issue-bound, the search's latency is hidden by the other warps, and the batch costs more issue slots.)
  return igso3_angle_lerp(trap, loc, u, cdf_count_le(trap, u, in01 ? lo : 0, in01 ? hi : kCdf));
}

// The one-record resolution alone, straight-line: *fast tells whether it applies (otherwise the caller runs
// igso3_angle_from_record, which searches).  For kernels that resolve two rows per thread and guard the rare search with one
// warp vote instead of a divergent region per row.  Same operations as the fast branch of igso3_angle_from_record.
SO3D_HD float igso3_angle_record_fast(const float* loc, const GuideRec& rec, float u, bool* fast) {
  const int lo = (int)(rec.lohi & 0xffffu), hi = (int)(rec.lohi >> 16);
  *fast = hi - lo <= 1 && lo < kCdf - 1 && u >= 0.f && u < 1.0f;
  const bool up = (hi > lo) && (rec.t0 <= u);
  int i1 = lo + (up ? 1 : 0);
  i1 = i1 < kCdf - 1 ? i1 : kCdf - 1;  // (only matters when !*fast)
  const int i0 = i1 > 0 ? i1 - 1 : 0;
  const float t0 = up ? rec.t0 : rec.tm1, t1 = up ? rec.tp1 : rec.t0;
  const float diff = fmaxf(t1 - t0, 1e-6f);
  const float wgt = fminf(fmaxf((u - t0) / diff, 0.f), 1.f);
  const float a0 = loc[i0], a1 = loc[i1];
  const float d = a1 - a0;
  return (wgt < 0.5f) ? fmaf(wgt, d, a0) : fmaf(-d, 1.0f - wgt, a1);
}

// record index of u (any float: values outside [0, 1) map to some valid record and take the search path)
SO3D_HD int guide_bucket(float u) {
  const bool upper = u > 0.875f;
  const float v = upper ? 1.0f - u : u;  // exact for u >= 1/2
  int kl = (int)(rec_float_as_uint(v) >> (23 - kRecMant)) - (kRecBias - 1);  // 0 below 2^-13, 1 + log bucket above
  kl = kl < 0 ? 0 : kl;
  int k = (int)(u * (float)kGuide) + (kRecMidBase - kRecMid0);
  k = (u < 0.125f) ? kl : (upper ? kRecUpBase + kl : k);
  return k < 0 ? 0 : (k > kGuideRecs - 1 ? kGuideRecs - 1 : k);
}

// ------------------------------------------------------------------------------------------------
// Philox4x32-10 counter-based RNG: key = seed (64 bit), counter = (row index 64 bit, stream offset
// 64 bit).  The draws of a row do not depend on how the batch is split over GPUs.
// ------------------------------------------------------------------------------------------------
struct U4 {
  uint32_t x, y, z, w;
};

SO3D_HD uint32_t mulhi32(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32);
#endif
}

SO3D_HD U4 philox4x32_10(uint64_t seed, uint64_t row, uint64_t offset) {
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  U4 c{(uint32_t)row, (uint32_t)(row >> 32), (uint32_t)offset, (uint32_t)(offset >> 32)};
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const uint32_t hi0 = mulhi32(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = mulhi32(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = U4{hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0};
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return c;
}

// The same generator with everything that depends only on (seed, offset) -- the ten round keys and the half of
// round 0 that multiplies the offset -- computed once on the host and passed by value in the kernel parameters
// (constant-bank operands): bit-identical to philox4x32_10(seed, row, offset), ~22 issue slots fewer per warp and
// tile than leaving the key schedule to the uniform datapath inside the tile loop.
struct PhiloxKey {
  uint32_t k0[10], k1[10];  // k0[0] already xor-ed with mulhi(0xCD9E8D57, offset_lo); k1[0] with offset_hi
  uint32_t lo1;             // 0xCD9E8D57 * offset_lo
};
SO3D_HD PhiloxKey make_philox_key(uint64_t seed, uint64_t offset) {
  PhiloxKey k;
  uint32_t a = (uint32_t)seed, b = (uint32_t)(seed >> 32);
  for (int i = 0; i < 10; ++i) {
    k.k0[i] = a;
    k.k1[i] = b;
    a += 0x9E3779B9u;
    b += 0xBB67AE85u;
  }
  const uint32_t ol = (uint32_t)offset, oh = (uint32_t)(offset >> 32);
  k.k0[0] ^= (uint32_t)(((uint64_t)0xCD9E8D57u * (uint64_t)ol) >> 32);
  k.k1[0] ^= oh;
  k.lo1 = 0xCD9E8D57u * ol;
  return k;
}
SO3D_HD U4 philox4x32_10(const PhiloxKey& k, uint64_t row) {
  const uint32_t rl = (uint32_t)row, rh = (uint32_t)(row >> 32);
  U4 c{k.k0[0] ^ rh, k.lo1, mulhi32(0xD2511F53u, rl) ^ k.k1[0], 0xD2511F53u * rl};
#pragma unroll
  for (int i = 1; i < 10; ++i) {
    const uint32_t hi0 = mulhi32(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = mulhi32(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = U4{hi1 ^ c.y ^ k.k0[i], lo1, hi0 ^ c.w ^ k.k1[i], lo0};
  }
  return c;
}

// The generator with the ten round keys (functions of the seed only) supplied by the caller -- kernels that change the
// stream offset while they run (one offset per step of a multi-step launch) take them as kernel parameters:
// bit-identical to philox4x32_10(seed, row, offset).
struct PhiloxRoundKeys {
  uint32_t k0[10], k1[10];
};
SO3D_HD PhiloxRoundKeys make_philox_round_keys(uint64_t seed) {
  PhiloxRoundKeys k;
  uint32_t a = (uint32_t)seed, b = (uint32_t)(seed >> 32);
  for (int i = 0; i < 10; ++i) {
    k.k0[i] = a;
    k.k1[i] = b;
    a += 0x9E3779B9u;
    b += 0xBB67AE85u;
  }
  return k;
}
SO3D_HD U4 philox4x32_10(const PhiloxRoundKeys& k, uint64_t row, uint64_t offset) {
  U4 c{(uint32_t)row, (uint32_t)(row >> 32), (uint32_t)offset, (uint32_t)(offset >> 32)};
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const uint32_t hi0 = mulhi32(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = mulhi32(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = U4{hi1 ^ c.y ^ k.k0[i], lo1, hi0 ^ c.w ^ k.k1[i], lo0};
  }
  return c;
}

// 24-bit uniform in [0, 1), the same lattice torch.rand(float32) uses.  Device: one round-toward-zero conversion of the
// whole word (keeps exactly the top 24 bits) and a multiply -- the same value as (x >> 8) 2^-24 without the shift.
SO3D_HD float u01(uint32_t x) {
#if defined(__CUDA_ARCH__)
  return __uint2float_rz(x) * (1.0f / 4294967296.0f);
#else
  return (float)(x >> 8) * (1.0f / 16777216.0f);
#endif
}

// The random-number side of the fused kernels is pure instruction issue (the kernels are issue-bound, DESIGN.md 4.3), and
// nothing downstream depends on a DRAWN direction or normal beyond its distribution -- so on the device these use the
// hardware approximations (MUFU.SIN / MUFU.COS / MUFU.LG2: absolute error 2^-20.9, i.e. a 5e-7 perturbation of a random
// variate) instead of the 22-instruction polynomial sincos and libdevice's logf.  The noise ANGLE and everything
// computed from an existing rotation keep the accurate primitives.  SO3D_DRAW_MUFU=0 restores the polynomial versions
// (the host build always uses them).
#ifndef SO3D_DRAW_MUFU
#define SO3D_DRAW_MUFU 1
#endif
SO3D_HD void sincos_draw(float x, float* s, float* c) {  // x in [-pi, pi]
#if defined(__CUDA_ARCH__) && SO3D_DRAW_MUFU
  asm("sin.approx.ftz.f32 %0, %1;" : "=f"(*s) : "f"(x));
  asm("cos.approx.ftz.f32 %0, %1;" : "=f"(*c) : "f"(x));
#else
  sincos_fast(x, s, c);
#endif
}
SO3D_HD float neg2_log_draw(float u) {  // -2 ln u for u in (0, 1]
#if defined(__CUDA_ARCH__) && SO3D_DRAW_MUFU
  float l;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(u));
  return -1.3862943611198906f * l;
#else
  return -2.0f * logf(u);
#endif
}

// Uniform point on S^2 from two uniforms (same law as the reference's normalised N(0, I3) draw,
// distributions.py:35-36).  The azimuth is 2 pi ub - pi in [-pi, pi): uniform on the circle like 2 pi ub, and inside
// the range where MUFU.SIN / MUFU.COS are specified to 2^-20.9.
SO3D_HD Vec3 sphere_from_uniforms(float ua, float ub) {
  const float z = fmaf(-2.0f, ua, 1.0f);
  const float t = 4.0f * ua * (1.0f - ua);  // 1 - z^2 without cancellation
  const float r = t * rsqrt_approx(fmaxf(t, 1e-30f));
  float sp, cp;
  sincos_draw(fmaf(kTwoPi, ub, -kPi), &sp, &cp);
  return Vec3{r * cp, r * sp, z};
}

// Four independent standard normals from one Philox block (Box-Muller on two pairs of 24-bit uniforms; the radius
// uniforms live in (0, 1], so the logarithm is finite: |z| <= sqrt(2 * 24 ln 2) = 5.77).
struct Normal4 {
  float a, b, c, d;
};
SO3D_HD Normal4 normal4_from_u4(const U4& r) {
  const float ua = (float)((r.x >> 8) + 1u) * (1.0f / 16777216.0f);
  const float ub = (float)((r.z >> 8) + 1u) * (1.0f / 16777216.0f);
  const float ta = neg2_log_draw(ua), tb = neg2_log_draw(ub);
  const float ra = ta * rsqrt_approx(fmaxf(ta, 1e-30f)), rb = tb * rsqrt_approx(fmaxf(tb, 1e-30f));
  float sa, ca, sb, cb;
  sincos_draw(fmaf(kTwoPi, u01(r.y), -kPi), &sa, &ca);
  sincos_draw(fmaf(kTwoPi, u01(r.w), -kPi), &sb, &cb);
  return Normal4{ra * ca, ra * sa, rb * cb, rb * sb};
}

struct NoiseDraw {
  Vec3 axis;
  float u;
};
SO3D_HD NoiseDraw draw_from_block(const U4& r) {
  NoiseDraw d;
  d.axis = sphere_from_uniforms(u01(r.x), u01(r.y));
  d.u = u01(r.z);
  return d;
}
SO3D_HD NoiseDraw draw_axis_u(uint64_t seed, uint64_t row, uint64_t offset) { return draw_from_block(philox4x32_10(seed, row, offset)); }
SO3D_HD NoiseDraw draw_axis_u(const PhiloxKey& k, uint64_t row) { return draw_from_block(philox4x32_10(k, row)); }
SO3D_HD NoiseDraw draw_axis_u(const PhiloxRoundKeys& k, uint64_t row, uint64_t offset) { return draw_from_block(philox4x32_10(k, row, offset)); }

// ------------------------------------------------------------------------------------------------
// Exact IGSO(3) angle sampler (so3d_igso3_sample_exact_f32): w = F^{-1}(u) for the angle law
//     p(w) = f(w) (1 - cos w) / pi  on [0, pi],   F(w) = int_0^w p,
// found per row in registers by a safeguarded Newton iteration, with no CDF table (DESIGN.md, "Exact IGSO(3) sampler").
// ------------------------------------------------------------------------------------------------
constexpr float kExactSeriesEps = 0.3f;  // series antiderivative at eps >= this, Gauss-Legendre quadrature below
constexpr float kExactXMax = 5.0f;       // eps < kExactSeriesEps: the mass beyond x = w / (2 eps) = 5 is 7.8e-11
constexpr int kExactMaxTerms = 24;       // eps >= kExactSeriesEps: a_l < 1e-10 from l = 17 on
constexpr int kExactIters = 16;          // Newton / bisection steps at most
constexpr float kExactTol = 1e-6f;       // relative Newton step at which the iteration stops

struct AngleCdf {
  float F, p;  // F and dF/dz in the variable z the branch iterates in (w for the series, x = w / (2 eps) below)
};

// eps >= kExactSeriesEps.  With the density's series weights a_l = (2l+1) e^{-l(l+1) eps^2} and a_0 = 1,
//   f(w) (1 - cos w) = sum_{l>=0} a_l [cos(l w) - cos((l+1) w)], so
//   pi F(w) = w + sum_{l>=1} (a_l - a_{l-1}) sin(l w) / l,   pi p(w) = 1 + sum_{l>=1} (a_l - a_{l-1}) cos(l w),
// exact on [0, pi] (F(pi) = 1).  At eps >= 0.3 the |a_l - a_{l-1}| sum to < 5, so fp32 keeps F to ~1e-7 absolute.
// sin / cos(l w) come from the angle-addition recurrence; the sum stops once a_{l-1} < 1e-10.
SO3D_HD AngleCdf igso3_angle_cdf_series(float w, float v) {
  float s1, c1;
  sincos_fast(w, &s1, &c1);
  float sl = s1, cl = c1, F = w, p = 1.0f, a_prev = 1.0f;
#pragma unroll 1
  for (int l = 1; l <= kExactMaxTerms && a_prev >= 1e-10f; ++l) {
    const float a = (float)(2 * l + 1) * expf(-(float)(l * (l + 1)) * v);
    const float c = a - a_prev;
    F = fmaf(c / (float)l, sl, F);
    p = fmaf(c, cl, p);
    const float sn = fmaf(sl, c1, cl * s1), cn = fmaf(cl, c1, -sl * s1);
    sl = sn;
    cl = cn;
    a_prev = a;
  }
  return AngleCdf{F * (1.0f / kPi), p * (1.0f / kPi)};
}

// eps < kExactSeriesEps, in x = w / (2 eps).  The closed form without its images (they weigh < 1e-11 on w <= 10 eps < pi):
//   dF/dx = C x sin(eps x) e^{-x^2},   C = 4 e^{eps^2/4} / (sqrt(pi) eps),   int_0^inf dF = 1 exactly,
// integrated over [0, min(x, 5)] with 16-node Gauss-Legendre (quadrature error <= 1e-10 there for every eps < 0.3;
// 12 nodes leave 5e-7).  As eps -> 0 this is the Maxwell law of x, i.e. w / (sqrt(2) eps) ~ chi with 3 degrees of freedom.
SO3D_HD float igso3_angle_integrand(float x, float eps) {
  float s, c;
  sincos_fast(eps * x, &s, &c);
  return x * s * expf(-x * x);
}
SO3D_HD AngleCdf igso3_angle_cdf_quad(float x, float eps, float C) {
  constexpr float kNode[8] = {9.501250984e-02f, 2.816035508e-01f, 4.580167777e-01f, 6.178762444e-01f,
                              7.554044084e-01f, 8.656312024e-01f, 9.445750231e-01f, 9.894009350e-01f};
  constexpr float kWeight[8] = {1.894506105e-01f, 1.826034150e-01f, 1.691565194e-01f, 1.495959888e-01f,
                                1.246289713e-01f, 9.515851168e-02f, 6.225352394e-02f, 2.715245941e-02f};
  const float h = 0.5f * fminf(x, kExactXMax);
  float acc = 0.0f;
#pragma unroll
  for (int k = 7; k >= 0; --k)
    acc = fmaf(kWeight[k], igso3_angle_integrand(h * (1.0f - kNode[k]), eps) + igso3_angle_integrand(h * (1.0f + kNode[k]), eps), acc);
  return AngleCdf{C * h * acc, C * igso3_angle_integrand(x, eps)};
}

// Starting point: the Maxwell quantile (the eps -> 0 law in x).  Normal quantile by Abramowitz & Stegun 26.2.23
// (|error| < 4.5e-4), Wilson-Hilferty for chi^2_3 = 2 x^2, and in the lower tail, where Wilson-Hilferty undershoots,
// the cubic law F ~ 4 x^3 / (3 sqrt(pi)).
SO3D_HD float maxwell_quantile_approx(float u) {
  const float q = fminf(u, 1.0f - u);
  const float t = sqrtf(-2.0f * logf(q));
  float z = t - fmaf(fmaf(0.010328f, t, 0.802853f), t, 2.515517f) / fmaf(fmaf(fmaf(0.001308f, t, 0.189269f), t, 1.432788f), t, 1.0f);
  z = u < 0.5f ? -z : z;
  const float h = fmaf(z, 0.27216553f, 0.92592593f);  // 1 - 2/27 + z sqrt(2/27)
  const float xw = sqrtf(fmaxf(1.5f * h * h * h, 0.0f));
  return fmaxf(xw, cbrtf(1.32934039f * u));  // (3 sqrt(pi) / 4) u
}

// w = F^{-1}(u) in [0, pi].  u <= 0 or eps = 0 gives 0; a NaN u or eps gives NaN.  The law depends on eps^2 only.
// The iteration keeps a bracket [lo, hi] from the sign of F - u and replaces a Newton step that leaves it by bisection.
SO3D_HD float igso3_angle_icdf(float u, float eps) {
  eps = fabsf(eps);
  if (isnan(u) || isnan(eps)) return u + eps;
  if (u <= 0.0f || eps == 0.0f) return 0.0f;
  const bool series = eps >= kExactSeriesEps;
  const float v = eps * eps;
  const float C = 4.0f * expf(0.25f * v) / (1.7724538509055159f * eps);
  const float x0 = maxwell_quantile_approx(u);
  float lo = 0.0f, hi = series ? kPi : kExactXMax;
  float z = series ? fminf(2.0f * eps * x0, kPi) : fminf(x0, kExactXMax);
#pragma unroll 1
  for (int it = 0; it < kExactIters; ++it) {
    const AngleCdf c = series ? igso3_angle_cdf_series(z, v) : igso3_angle_cdf_quad(z, eps, C);
    const float r = c.F - u;
    if (r == 0.0f) break;
    if (r > 0.0f) hi = z;
    else lo = z;
    float zn = z - r / c.p;
    if (!(zn >= lo && zn <= hi)) zn = 0.5f * (lo + hi);
    const bool done = fabsf(zn - z) <= kExactTol * z;
    z = zn;
    if (done) break;
  }
  return series ? z : fminf(2.0f * eps * z, kPi);
}

// ------------------------------------------------------------------------------------------------
// Pathwise derivative of the exact sampler's angle (so3d_igso3_rsample_bwd_f32): dw/deps of w = F^{-1}(u; eps) at fixed u
// (DESIGN.md, "Reparameterised IGSO(3) sampling").  Implicit differentiation gives dw/deps = -(dF/deps)(w) / p(w).  The
// density solves the heat equation on SO(3), df/d(eps^2) = f'' + cot(w/2) f' = (sin^2(w/2) f')' / sin^2(w/2), and
// p = (2/pi) sin^2(w/2) f, so
//     dF/d(eps^2) = (2/pi) int_0^w (sin^2(t/2) f'(t))' dt = (2/pi) sin^2(w/2) f'(w)   and   dw/deps = -2 eps f'(w) / f(w):
// the pathwise derivative is -2 eps times the angle score d log f / dw, one evaluation at the known w.  Every image term of
// the closed form solves the heat equation by itself, so this holds for the image-free law of the quadrature regime too.
//   eps <  kExactSeriesEps (the sampler's quadrature regime: image-free law, log f = log x - x^2 - log sin(w/2) + const in
//          x = w / (2 eps)):  dw/deps = 2x - 2 eps phi(w),  phi = 1/w - cot(w/2)/2 = w/12 + w^3/720 + ...;  2 eps phi is at
//          most 2 % of 2x, so nothing cancels, and w = 0 gives 0.
//   eps >= kExactSeriesEps (the series regime): -2 eps g with g from the density's `auto` evaluator (igso3_logf_g_t<kAuto>:
//          the 3-image closed form up to eps = 1, the series above).  The series of F and p would not do here: in the upper
//          tail at eps near 0.3 their terms are 10^7 times the density, and f' / f would keep no digit.
// Special values follow the sampler: NaN eps gives NaN; the law depends on eps^2, so the result is sign(eps) dw/d|eps|.
constexpr float kDepsPhiTaylorW = 0.5f;  // phi(w) by its Taylor series below this (4 terms: <= 2e-9 relative)

SO3D_HD float igso3_angle_phi(float w) {
  if (w < kDepsPhiTaylorW) {
    const float w2 = w * w;
    return w * fmaf(w2, fmaf(w2, fmaf(w2, 8.2671958e-7f, 3.3068783e-5f), 1.3888889e-3f), 8.3333333e-2f);
  }
  float sh, ch;
  sincos_fast(0.5f * w, &sh, &ch);
  return 1.0f / w - 0.5f * ch / sh;
}

SO3D_HD float igso3_angle_deps(float w, float eps) {
  const float e = fabsf(eps);
  float d;
  if (isnan(e)) {
    d = e;
  } else if (e < kExactSeriesEps) {
    const float x = w / (2.0f * e);
    d = fmaf(-2.0f * e, igso3_angle_phi(w), 2.0f * x);
  } else {
    float lf, g;
    igso3_logf_g_t<kAuto>(w, e, kExactMaxTerms, &lf, &g);
    d = -2.0f * e * g;
  }
  return eps < 0.0f ? -d : d;
}

// eps = 0: the sampler returns w = 0 whatever u is, so the derivative comes from u.  As eps -> 0+, w = 2 eps x with x -> x0(u),
// the Maxwell quantile, so dw/deps -> 2 x0(u).  x0 is the sampler's own quadrature-regime inversion at eps = 2^-64 (where
// C sin(eps x) = (4/sqrt(pi)) x to fp32 and 2 eps x is exact): 2 x0 = 2^64 w.
SO3D_HD float igso3_angle_deps_eps0(float u) { return igso3_angle_icdf(u, kTinyDown) * kTinyUp; }

}  // namespace so3d
