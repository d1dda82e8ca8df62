// so3d_lanes.cuh -- the lean per-rotation arithmetic of so3d_math.cuh written ONCE over a "lanes" type, so that a thread
// can carry one rotation (L1) or TWO rotations (L2) through exactly the same sequence of IEEE operations.
//
// Why: the fused row kernels are instruction-ISSUE bound with the FMA pipe at 30-40 % (DESIGN.md 4.3): ~45 % of their
// issue slots are FFMA / FMUL / FADD.  Blackwell has packed FP32 instructions (FFMA2 / FMUL2 / FADD2, PTX
// fma.rn.f32x2 ...: one issue slot for two lanes, two passes through the FMA pipe), so a thread that processes two rows
// with its FP32 work packed spends half the issue slots on it.  ptxas keeps the two lanes in an aligned register pair,
// folds negations into operand modifiers and broadcast constants into immediates, and lets the per-lane instructions
// (MUFU, selects, compares, integer work) address the halves directly -- no packing moves (checked in SASS).
//
// Contract: every operation below is a single correctly rounded IEEE operation per lane (explicit *_rn intrinsics on the
// device: never contracted, never reassociated), so L1 and L2 instantiations -- and therefore one-row and two-row
// kernels -- produce bit-identical results.  tests/test_host_math.py checks L1 == L2 == the functions of so3d_math.cuh
// they restate on the host build.
#pragma once

#include "so3d_math.cuh"

namespace so3d {

struct L1 {
  float x;
};
struct alignas(8) L2 {
  float x, y;
};
struct M1 {
  bool x;
};
struct M2 {
  bool x, y;
};
template <class L>
struct MaskOf;
template <>
struct MaskOf<L1> {
  using type = M1;
};
template <>
struct MaskOf<L2> {
  using type = M2;
};

// ---- one correctly rounded operation per lane --------------------------------------------------------------------------
SO3D_HD float op_add(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fadd_rn(a, b);
#else
  return a + b;
#endif
}
SO3D_HD float op_mul(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fmul_rn(a, b);
#else
  return a * b;
#endif
}
SO3D_HD float op_fma(float a, float b, float c) {
#if defined(__CUDA_ARCH__)
  return __fmaf_rn(a, b, c);
#else
  return fmaf(a, b, c);
#endif
}

template <class L>
SO3D_HD L bc(float c);
template <>
SO3D_HD L1 bc<L1>(float c) {
  return L1{c};
}
template <>
SO3D_HD L2 bc<L2>(float c) {
  return L2{c, c};
}

SO3D_HD L1 neg(L1 a) { return L1{-a.x}; }
SO3D_HD L2 neg(L2 a) { return L2{-a.x, -a.y}; }
SO3D_HD L1 add(L1 a, L1 b) { return L1{op_add(a.x, b.x)}; }
SO3D_HD L1 mul(L1 a, L1 b) { return L1{op_mul(a.x, b.x)}; }
SO3D_HD L1 fma(L1 a, L1 b, L1 c) { return L1{op_fma(a.x, b.x, c.x)}; }
SO3D_HD L2 add(L2 a, L2 b) {
#if defined(__CUDA_ARCH__)
  const float2 r = __fadd2_rn(make_float2(a.x, a.y), make_float2(b.x, b.y));
  return L2{r.x, r.y};
#else
  return L2{op_add(a.x, b.x), op_add(a.y, b.y)};
#endif
}
SO3D_HD L2 mul(L2 a, L2 b) {
#if defined(__CUDA_ARCH__)
  const float2 r = __fmul2_rn(make_float2(a.x, a.y), make_float2(b.x, b.y));
  return L2{r.x, r.y};
#else
  return L2{op_mul(a.x, b.x), op_mul(a.y, b.y)};
#endif
}
SO3D_HD L2 fma(L2 a, L2 b, L2 c) {
#if defined(__CUDA_ARCH__)
  const float2 r = __ffma2_rn(make_float2(a.x, a.y), make_float2(b.x, b.y), make_float2(c.x, c.y));
  return L2{r.x, r.y};
#else
  return L2{op_fma(a.x, b.x, c.x), op_fma(a.y, b.y, c.y)};
#endif
}
template <class L>
SO3D_HD L sub(L a, L b) {
  return add(a, neg(b));  // a - b: the negation is an operand modifier
}
template <class L>
SO3D_HD L fnma(L a, L b, L c) {
  return fma(neg(a), b, c);  // -(a b) + c
}
template <class L>
SO3D_HD L mulc(float k, L a) {
  return mul(bc<L>(k), a);
}

// ---- per-lane operations (no packed form exists: MUFU, min/max, compares, selects) ---------------------------------------
#define SO3D_LANEWISE1(NAME, EXPR)                   \
  SO3D_HD L1 NAME(L1 a) {                            \
    const float v = a.x;                             \
    return L1{EXPR};                                 \
  }                                                  \
  SO3D_HD L2 NAME(L2 a) {                            \
    float v = a.x;                                   \
    const float r0 = EXPR;                           \
    v = a.y;                                         \
    const float r1 = EXPR;                           \
    return L2{r0, r1};                               \
  }
SO3D_LANEWISE1(vabs, fabsf(v))
SO3D_LANEWISE1(vrsqrt, rsqrt_approx(v))
SO3D_LANEWISE1(vrcp, rcp_approx(v))
SO3D_LANEWISE1(vex2, fast_ex2(v))
#undef SO3D_LANEWISE1
SO3D_HD L1 vmax(L1 a, L1 b) { return L1{fmaxf(a.x, b.x)}; }
SO3D_HD L2 vmax(L2 a, L2 b) { return L2{fmaxf(a.x, b.x), fmaxf(a.y, b.y)}; }
SO3D_HD L1 vmin(L1 a, L1 b) { return L1{fminf(a.x, b.x)}; }
SO3D_HD L2 vmin(L2 a, L2 b) { return L2{fminf(a.x, b.x), fminf(a.y, b.y)}; }
SO3D_HD M1 gt(L1 a, L1 b) { return M1{a.x > b.x}; }
SO3D_HD M2 gt(L2 a, L2 b) { return M2{a.x > b.x, a.y > b.y}; }
SO3D_HD M1 ge(L1 a, L1 b) { return M1{a.x >= b.x}; }
SO3D_HD M2 ge(L2 a, L2 b) { return M2{a.x >= b.x, a.y >= b.y}; }
SO3D_HD M1 lt(L1 a, L1 b) { return M1{a.x < b.x}; }
SO3D_HD M2 lt(L2 a, L2 b) { return M2{a.x < b.x, a.y < b.y}; }
SO3D_HD M1 mand(M1 a, M1 b) { return M1{a.x && b.x}; }
SO3D_HD M2 mand(M2 a, M2 b) { return M2{a.x && b.x, a.y && b.y}; }
SO3D_HD M1 mnot(M1 a) { return M1{!a.x}; }
SO3D_HD M2 mnot(M2 a) { return M2{!a.x, !a.y}; }
SO3D_HD L1 sel(M1 m, L1 a, L1 b) { return L1{m.x ? a.x : b.x}; }
SO3D_HD L2 sel(M2 m, L2 a, L2 b) { return L2{m.x ? a.x : b.x, m.y ? a.y : b.y}; }

template <class L>
struct Vec3L {
  L x, y, z;
};
template <class L>
struct QuatL {
  L w, x, y, z;
};
template <class L>
struct Mat3L {
  L m[9];
};

// ---- sincos_fast (so3d_math.cuh) ---------------------------------------------------------------------------------------
SO3D_HD void sincos_quadrant(float t, float sn, float cs, float* s_out, float* c_out) {
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
SO3D_HD void sincos_fix(L1 t, L1 sn, L1 cs, L1* s, L1* c) { sincos_quadrant(t.x, sn.x, cs.x, &s->x, &c->x); }
SO3D_HD void sincos_fix(L2 t, L2 sn, L2 cs, L2* s, L2* c) {
  sincos_quadrant(t.x, sn.x, cs.x, &s->x, &c->x);
  sincos_quadrant(t.y, sn.y, cs.y, &s->y, &c->y);
}
template <class L>
SO3D_HD void sincos_fast_l(L x, L* s_out, L* c_out) {
  const L t = fma(x, bc<L>(0.636619772f), bc<L>(12582912.0f));
  const L kf = add(t, bc<L>(-12582912.0f));
  L r = fma(kf, bc<L>(-1.57079637f), x);
  r = fma(kf, bc<L>(4.37113883e-8f), r);
  const L r2 = mul(r, r);
  L ps = fma(bc<L>(-1.9515295891e-4f), r2, bc<L>(8.3321608736e-3f));
  ps = fma(ps, r2, bc<L>(-1.6666654611e-1f));
  const L sn = fma(mul(ps, r2), r, r);
  L pc = fma(bc<L>(2.443315711809948e-5f), r2, bc<L>(-1.388731625493765e-3f));
  pc = fma(pc, r2, bc<L>(4.166664568298827e-2f));
  pc = fma(pc, r2, bc<L>(-0.5f));
  const L cs = fma(pc, r2, bc<L>(1.0f));
  sincos_fix(t, sn, cs, s_out, c_out);
}

// ---- atan2_pos ---------------------------------------------------------------------------------------------------------
template <class L>
SO3D_HD L atan2_pos_l(L y, L x) {
  const L ax = vabs(x);
  const L hi = vmax(ax, y), lo = vmin(ax, y);
  const L t = mul(lo, vrcp(vmax(hi, bc<L>(1e-37f))));
  const L z = mul(t, t);
  L p = fma(bc<L>(0.0028662257f), z, bc<L>(-0.0161657367f));
  p = fma(p, z, bc<L>(0.0429096138f));
  p = fma(p, z, bc<L>(-0.0752896400f));
  p = fma(p, z, bc<L>(0.1065626393f));
  p = fma(p, z, bc<L>(-0.1420889944f));
  p = fma(p, z, bc<L>(0.1999355085f));
  p = fma(p, z, bc<L>(-0.3333314528f));
  L r = fma(mul(p, z), t, t);
  r = sel(gt(y, ax), sub(bc<L>(1.57079632679f), r), r);
  return sel(lt(x, bc<L>(0.f)), sub(bc<L>(3.14159265359f), r), r);
}

// ---- quaternions -------------------------------------------------------------------------------------------------------
template <class L>
SO3D_HD QuatL<L> qmul_l(const QuatL<L>& a, const QuatL<L>& b) {
  QuatL<L> q;
  q.w = fnma(a.z, b.z, fnma(a.y, b.y, fnma(a.x, b.x, mul(a.w, b.w))));
  q.x = fnma(a.z, b.y, fma(a.y, b.z, fma(a.x, b.w, mul(a.w, b.x))));
  q.y = fma(a.z, b.x, fma(a.y, b.w, fnma(a.x, b.z, mul(a.w, b.y))));
  q.z = fma(a.z, b.w, fnma(a.y, b.x, fma(a.x, b.y, mul(a.w, b.z))));
  return q;
}
template <class L>
SO3D_HD QuatL<L> quat_axis_angle_l(const Vec3L<L>& n, L theta) {
  L sh, ch;
  sincos_fast_l(mulc(0.5f, theta), &sh, &ch);
  return QuatL<L>{ch, mul(sh, n.x), mul(sh, n.y), mul(sh, n.z)};
}
template <class L>
SO3D_HD QuatL<L> quat_exp_vec_l(const Vec3L<L>& v) {
  const L t2 = fma(v.x, v.x, fma(v.y, v.y, mul(v.z, v.z)));
  const L rs = vrsqrt(vmax(t2, bc<L>(1e-30f)));
  const L t = mul(t2, rs);
  L sh, ch;
  sincos_fast_l(mulc(0.5f, t), &sh, &ch);
  const L k = sel(gt(t2, bc<L>(1e-12f)), mul(sh, rs), bc<L>(0.5f));
  return QuatL<L>{ch, mul(k, v.x), mul(k, v.y), mul(k, v.z)};
}
template <class L>
SO3D_HD Mat3L<L> quat_to_mat_unit_l(const QuatL<L>& q0) {
  const L inv = vrsqrt(fma(q0.w, q0.w, fma(q0.x, q0.x, fma(q0.y, q0.y, mul(q0.z, q0.z)))));
  const L w = mul(q0.w, inv), x = mul(q0.x, inv), y = mul(q0.y, inv), z = mul(q0.z, inv);
  const L x2 = add(x, x), y2 = add(y, y), z2 = add(z, z);
  const L wx = mul(w, x2), wy = mul(w, y2), wz = mul(w, z2);
  const L one = bc<L>(1.0f);
  Mat3L<L> r;
  r.m[0] = fnma(y2, y, fnma(z2, z, one));
  r.m[4] = fnma(x2, x, fnma(z2, z, one));
  r.m[8] = fnma(x2, x, fnma(y2, y, one));
  r.m[1] = fma(x2, y, neg(wz));
  r.m[3] = fma(x2, y, wz);
  r.m[2] = fma(x2, z, wy);
  r.m[6] = fma(x2, z, neg(wy));
  r.m[5] = fma(y2, z, neg(wx));
  r.m[7] = fma(y2, z, wx);
  return r;
}

// ---- axis / angle of a rotation matrix (axis_angle_fast) ----------------------------------------------------------------
template <class L>
struct AxisAngleL {
  Vec3L<L> axis;
  L theta;
};
template <class L>
SO3D_HD AxisAngleL<L> axis_angle_fast_l(const Mat3L<L>& r) {
  using M = typename MaskOf<L>::type;
  const L zero = bc<L>(0.f);
  const L ux = sub(r.m[7], r.m[5]), uy = sub(r.m[2], r.m[6]), uz = sub(r.m[3], r.m[1]);
  const M tiny = lt(fma(ux, ux, fma(uy, uy, mul(uz, uz))), bc<L>(kFltMin));
  const L k = sel(tiny, bc<L>(kTinyUp), bc<L>(1.0f));
  const L vx = mul(ux, k), vy = mul(uy, k), vz = mul(uz, k);
  const L n2 = fma(vx, vx, fma(vy, vy, mul(vz, vz)));
  const M pos = ge(n2, bc<L>(kFltMin));
  const L rs = sel(pos, vrsqrt(n2), zero);
  const L c = mulc(0.5f, add(add(add(r.m[0], r.m[4]), r.m[8]), bc<L>(-1.0f)));
  AxisAngleL<L> o;
  o.theta = atan2_pos_l(mul(mul(sel(tiny, bc<L>(0.5f * kTinyDown), bc<L>(0.5f)), n2), rs), c);
  const L d0 = sub(r.m[0], c), d1 = sub(r.m[4], c), d2 = sub(r.m[8], c);
  const L s01 = mulc(0.5f, add(r.m[1], r.m[3])), s02 = mulc(0.5f, add(r.m[2], r.m[6])), s12 = mulc(0.5f, add(r.m[5], r.m[7]));
  const M p0 = mand(ge(d0, d1), ge(d0, d2));
  const M p1 = ge(d1, d2);
  const L cx = sel(p0, d0, sel(p1, s01, s02));
  const L cy = sel(p0, s01, sel(p1, d1, s12));
  const L cz = sel(p0, s02, sel(p1, s12, d2));
  const L cn = vrsqrt(vmax(fma(cx, cx, fma(cy, cy, mul(cz, cz))), bc<L>(1e-30f)));
  const L sg = sel(lt(fma(cx, vx, fma(cy, vy, mul(cz, vz))), zero), neg(cn), cn);
  const M near_pi = lt(c, bc<L>(kNearPiCos));
  o.axis.x = sel(near_pi, mul(cx, sg), mul(vx, rs));
  o.axis.y = sel(near_pi, mul(cy, sg), mul(vy, rs));
  o.axis.z = sel(near_pi, mul(cz, sg), sel(mnot(pos), bc<L>(1.0f), mul(vz, rs)));
  return o;
}
template <class L>
SO3D_HD void quat_axis_halfangle_l(const QuatL<L>& q, Vec3L<L>* n, L* half) {
  using M = typename MaskOf<L>::type;
  const L zero = bc<L>(0.f);
  const M tiny = lt(fma(q.x, q.x, fma(q.y, q.y, mul(q.z, q.z))), bc<L>(kFltMin));
  const L sc = sel(tiny, bc<L>(kTinyUp), bc<L>(1.0f));
  const L x = mul(q.x, sc), y = mul(q.y, sc), z = mul(q.z, sc);
  const L v2 = fma(x, x, fma(y, y, mul(z, z)));
  const M pos = ge(v2, bc<L>(kFltMin));
  const L rs = sel(pos, vrsqrt(v2), zero);
  *half = atan2_pos_l(mul(mul(sel(tiny, bc<L>(kTinyDown), bc<L>(1.0f)), v2), rs), vabs(q.w));
  const L k = sel(lt(q.w, zero), neg(rs), rs);
  *n = Vec3L<L>{mul(x, k), mul(y, k), sel(pos, mul(z, k), bc<L>(1.0f))};
}

// ---- the reverse step's posterior mean on quaternions (p_mean_quat / p_mean_quat_nopred) ---------------------------------
// a, b, c1, c2: the step's schedule scalars (shared by the lanes)
template <class L, bool kHasPred>
SO3D_HD QuatL<L> p_mean_quat_l(const Mat3L<L>& x_t, const Vec3L<L>& pred, float a, float b, float c1, float c2, QuatL<L>* x0h) {
  const AxisAngleL<L> ax = axis_angle_fast_l(x_t);
  QuatL<L> qh = quat_axis_angle_l(ax.axis, mulc(a, ax.theta));
  if (kHasPred) {
    const QuatL<L> q2 = quat_exp_vec_l(Vec3L<L>{mulc(-b, pred.x), mulc(-b, pred.y), mulc(-b, pred.z)});
    qh = qmul_l(qh, q2);
  }
  Vec3L<L> n0;
  L h0;
  quat_axis_halfangle_l(qh, &n0, &h0);
  const QuatL<L> q3 = quat_axis_angle_l(n0, mulc(2.0f * c1, h0));
  const QuatL<L> q4 = quat_axis_angle_l(ax.axis, mulc(c2, ax.theta));
  *x0h = qh;
  return qmul_l(q3, q4);
}

// the same with per-lane schedule scalars (rows with their own step index)
template <class L>
SO3D_HD QuatL<L> p_mean_quat_rows_l(const Mat3L<L>& x_t, const Vec3L<L>& pred, L a, L b, L c1, L c2, QuatL<L>* x0h) {
  const AxisAngleL<L> ax = axis_angle_fast_l(x_t);
  const L nb = neg(b);
  const QuatL<L> q1 = quat_axis_angle_l(ax.axis, mul(a, ax.theta));
  const QuatL<L> q2 = quat_exp_vec_l(Vec3L<L>{mul(nb, pred.x), mul(nb, pred.y), mul(nb, pred.z)});
  const QuatL<L> qh = qmul_l(q1, q2);
  Vec3L<L> n0;
  L h0;
  quat_axis_halfangle_l(qh, &n0, &h0);
  const QuatL<L> q3 = quat_axis_angle_l(n0, mul(mulc(2.0f, c1), h0));
  const QuatL<L> q4 = quat_axis_angle_l(ax.axis, mul(c2, ax.theta));
  *x0h = qh;
  return qmul_l(q3, q4);
}

// ---- drawn direction (sphere_from_uniforms): the azimuth's sin / cos are per-lane MUFU (or the polynomial on the host) ------
SO3D_HD void sincos_draw_l(L1 x, L1* s, L1* c) { sincos_draw(x.x, &s->x, &c->x); }
SO3D_HD void sincos_draw_l(L2 x, L2* s, L2* c) {
  sincos_draw(x.x, &s->x, &c->x);
  sincos_draw(x.y, &s->y, &c->y);
}
template <class L>
SO3D_HD Vec3L<L> sphere_from_uniforms_l(L ua, L ub) {
  const L z = fma(bc<L>(-2.0f), ua, bc<L>(1.0f));
  const L t = mul(mulc(4.0f, ua), sub(bc<L>(1.0f), ua));
  const L r = mul(t, vrsqrt(vmax(t, bc<L>(1e-30f))));
  L sp, cp;
  sincos_draw_l(fma(bc<L>(kTwoPi), ub, bc<L>(-kPi)), &sp, &cp);
  return Vec3L<L>{mul(r, cp), mul(r, sp), z};
}

// ---- the L-term series (igso3_series_terms, source form 0) on two rows ---------------------------------------------------
// Per term, for both rows: FMUL2, 2 MUFU.EX2 (each writes its half of the register pair), 3 FFMA2, 3 FADD2 (4 FFMA2 and
// 2 FADD2 in the w form), and the table factors as uniform-register operands broadcast to both halves (one LDCU.64 per two
// terms) -- 5 issue slots + 2 MUFU per two row-terms where the one-row kernel spends 2 x 9.  The one-row kernel's `A + d`
// with A = ex2(x) * mh is contracted by the compiler into FFMA e, mh, d; the fma below is that instruction, so every lane
// goes through the same operations and gives the same bits.  Same block structure as igso3_series_terms: the ragged top block first, then whole blocks by block index.
// Source-form knobs of the packed block, as SO3D_SERIES_ORDER / SO3D_SERIES_BLOCK for the one-row loop: the same operations
// per lane in every form, only the order ptxas's list scheduler sees them in (and with it its operand-reuse flags) changes.
//   order 0: t = fma(e, mh, d); d = t - kap b; u = d' - b; d' = u - kap b'; b += d; b' += d'
//   order 1: the two consumers of b (u, d), then the two of kap (d, d') back to back
//   order 2: the derivative chain first
//   order 3: every consumer of b together (d, b += d, u), then d'
// Measured on B200 (profiles/r07a_series_forms.jsonl, DESIGN.md 4.1): order 0 and 1 compile to the same SASS; order 3 runs
// `series` 2.4 % faster but series_adaptive 3.6 % and the 16 384-row batch 6 % slower; blocks 16 and 64 are slower.
#ifndef SO3D_SERIES2_ORDER
#define SO3D_SERIES2_ORDER 0
#endif
#ifndef SO3D_SERIES2_BLOCK
#define SO3D_SERIES2_BLOCK 32
#endif
constexpr int kSeries2Block = SO3D_SERIES2_BLOCK;
struct SeriesStateL2 {
  L2 b, d, bp, dp, b2, bp2;
};
// series_dsrc over lanes
SO3D_HD L2 series_dsrc_l2(L2 kapp, L2 b, L2 dp) {
#if SO3D_SERIES_DERIV
  (void)kapp;
  return sub(dp, b);
#else
  return fnma(kapp, b, dp);
#endif
}
template <int kUnroll>
SO3D_HD void igso3_series_run_l2(SeriesStateL2& st, L2 kap, L2 kapp, L2 cexp, int hi, int count) {
#pragma unroll kUnroll
  for (int i = 0; i < count; ++i) {
    const int l = hi - i;
    const L2 e = vex2(mul(bc<L2>(series_mm(l)), cexp));
    const L2 mh = bc<L2>(series_mh(l));
    st.b2 = st.b;
    st.bp2 = st.bp;
#if SO3D_SERIES2_ORDER == 0
    const L2 dn = fnma(kap, st.b, fma(e, mh, st.d));
    const L2 dpn = fnma(kap, st.bp, series_dsrc_l2(kapp, st.b, st.dp));
    st.b = add(st.b, dn);
    st.bp = add(st.bp, dpn);
#elif SO3D_SERIES2_ORDER == 1
    const L2 t = fma(e, mh, st.d);
    const L2 u = series_dsrc_l2(kapp, st.b, st.dp);
    const L2 dn = fnma(kap, st.b, t);
    const L2 dpn = fnma(kap, st.bp, u);
    st.b = add(st.b, dn);
    st.bp = add(st.bp, dpn);
#elif SO3D_SERIES2_ORDER == 2
    const L2 dpn = fnma(kap, st.bp, series_dsrc_l2(kapp, st.b, st.dp));
    const L2 dn = fnma(kap, st.b, fma(e, mh, st.d));
    st.bp = add(st.bp, dpn);
    st.b = add(st.b, dn);
#else
    const L2 dn = fnma(kap, st.b, fma(e, mh, st.d));
    const L2 bn = add(st.b, dn);
    const L2 u = series_dsrc_l2(kapp, st.b, st.dp);
    const L2 dpn = fnma(kap, st.bp, u);
    st.b = bn;
    st.bp = add(st.bp, dpn);
#endif
    st.d = dn;
    st.dp = dpn;
  }
}

// log f and d log f / dw of the series modes (igso3_series_branch<kMode>, guard form 3) for two rows; `L` is the same for both
template <int kMode>
SO3D_HD void igso3_series_branch_l2(L2 w, L2 eps, int L, float* logf_out, float* g_out) {
  static_assert(kMode == kSeries || kMode == kSeriesAdaptive || kMode == kSeriesPure, "series modes only");
  int terms = L;
  if (kMode == kSeriesAdaptive) {
    const int t0 = igso3_series_live_terms(eps.x, L), t1 = igso3_series_live_terms(eps.y, L);
    terms = t0 > t1 ? t0 : t1;
#if defined(__CUDA_ARCH__)
    terms = __reduce_max_sync(__activemask(), terms);  // warp-uniform trip count (table operands stay uniform loads)
#endif
#if SO3D_SERIES_ROUNDUP
    const int up = (terms + kSeries2Block - 1) / kSeries2Block * kSeries2Block;
    terms = up <= L ? up : L;
#endif
  }
  constexpr bool kGuarded = kMode != kSeriesPure;
  const bool guard0 = kGuarded && eps.x <= kAutoSeriesEps && w.x > kSeriesGuard * eps.x;
  const bool guard1 = kGuarded && eps.y <= kAutoSeriesEps && w.y > kSeriesGuard * eps.y;
  float lf_c[2] = {0.f, 0.f}, g_c[2] = {0.f, 0.f};
  if (guard0) igso3_closed_f32_outofline(w.x, eps.x, &lf_c[0], &g_c[0]);
  if (guard1) igso3_closed_f32_outofline(w.y, eps.y, &lf_c[1], &g_c[1]);
  L2 kap, kapp, cexp;
  igso3_series_lane_setup(w.x, eps.x, &kap.x, &kapp.x, &cexp.x);
  igso3_series_lane_setup(w.y, eps.y, &kap.y, &kapp.y, &cexp.y);
  const L2 zero = bc<L2>(0.f);
  SeriesStateL2 st{zero, zero, zero, zero, zero, zero};
  const int ragged = terms % kSeries2Block;
  if (ragged) igso3_series_run_l2<1>(st, kap, kapp, cexp, terms - 1, ragged);
  for (int blk = terms / kSeries2Block - 1; blk >= 0; --blk)
    igso3_series_run_l2<kSeries2Block>(st, kap, kapp, cexp, blk * kSeries2Block + (kSeries2Block - 1), kSeries2Block);
  const L2 F = add(st.b, st.b2);
#if SO3D_SERIES_DERIV
  const L2 dF = mul(kapp, add(st.bp, st.bp2));  // series_dF
#else
  const L2 dF = add(st.bp, st.bp2);
#endif
  logf_out[0] = guard0 ? lf_c[0] : logf(2.0f * F.x);
  g_out[0] = guard0 ? g_c[0] : dF.x / F.x;
  logf_out[1] = guard1 ? lf_c[1] : logf(2.0f * F.y);
  g_out[1] = guard1 ? g_c[1] : dF.y / F.y;
}

// ---- lane <-> scalar glue ------------------------------------------------------------------------------------------------
// diffusion.py:344-346 over lanes: the quaternion of x_t = so3_scale(x0, sc) . noise with noise = rot(axis, ang) (its
// quaternion goes to *qn_out) -- the operations of the one-row forward-noising kernel (QSampleOp::row) in the same order
template <class L>
SO3D_HD QuatL<L> q_sample_quat_l(const Mat3L<L>& x0, L sc, const Vec3L<L>& axis, L ang, QuatL<L>* qn_out) {
  const QuatL<L> qn = quat_axis_angle_l(axis, ang);
  const AxisAngleL<L> ax = axis_angle_fast_l(x0);
  *qn_out = qn;
  return qmul_l(quat_axis_angle_l(ax.axis, mul(sc, ax.theta)), qn);
}

SO3D_HD Mat3L<L1> lanes_of(const Mat3& a) {
  Mat3L<L1> r;
  for (int k = 0; k < 9; ++k) r.m[k] = L1{a.m[k]};
  return r;
}
SO3D_HD Mat3L<L2> lanes_of(const Mat3& a, const Mat3& b) {
  Mat3L<L2> r;
  for (int k = 0; k < 9; ++k) r.m[k] = L2{a.m[k], b.m[k]};
  return r;
}

}  // namespace so3d
