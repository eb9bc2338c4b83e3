// Outward-rounded interval arithmetic and the interval env steps IEnv<ID> of the region verifier (certify_region.cu).
//
// An IEnv<ID>::step encloses ONE closed-loop env step of the real-arithmetic system: the CONTROL_STEP explicit-Euler
// sub-steps of Env<ID>::step (env_dynamics.cuh) evaluated exactly, with the env's float32 constants (float64 for TwoLink's
// solve) read as exact reals.  Every operation rounds its lower bound down and its upper bound up (__f*_rd / __f*_ru,
// __d*_rd / __d*_ru); sin / cos / tanh are the CUDA functions widened outward by more than their documented maximum error
// (2 ulp) plus one ulp; interval sin / cos include +-1 whenever the interval may contain an extremum.  Algebraically equal
// forms of the env expressions are used where they are tighter (e.g. TwoLink's determinant as a quadratic in cos theta2).
// NaN bounds are widened to +-inf at each step, so a NaN never turns into a finite bound.
#pragma once
#include "env_dynamics.cuh"

namespace msacl {

struct If { float l, u; };
struct Id { double l, u; };

// Outward widening of a CUDA sinf / cosf / tanhf result: 2^-20 relative (>= 8 ulp of the true value) + 2^-126 absolute
__device__ __forceinline__ float wdn(float f) { return __fsub_rd(f, __fmaf_ru(fabsf(f), 0x1p-20f, 0x1p-126f)); }
__device__ __forceinline__ float wup(float f) { return __fadd_ru(f, __fmaf_ru(fabsf(f), 0x1p-20f, 0x1p-126f)); }
// the same for the float64 sin / cos: 2^-48 relative (>= 16 ulp) + 2^-1000 absolute
__device__ __forceinline__ double wdn(double f) { return __dsub_rd(f, __fma_ru(fabs(f), 0x1p-48, 0x1p-1000)); }
__device__ __forceinline__ double wup(double f) { return __dadd_ru(f, __fma_ru(fabs(f), 0x1p-48, 0x1p-1000)); }

__device__ __forceinline__ If sane(If a) { return {isnan(a.l) ? -INFINITY : a.l, isnan(a.u) ? INFINITY : a.u}; }
__device__ __forceinline__ If ipt(float c) { return {c, c}; }
__device__ __forceinline__ If iadd(If a, If b) { return {__fadd_rd(a.l, b.l), __fadd_ru(a.u, b.u)}; }
__device__ __forceinline__ If isub(If a, If b) { return {__fsub_rd(a.l, b.u), __fsub_ru(a.u, b.l)}; }
// products of an infinite and a zero bound are NaN; fminf / fmaxf skip them, which is the real product 0
__device__ __forceinline__ If imul(If a, If b) {
  return {fminf(fminf(__fmul_rd(a.l, b.l), __fmul_rd(a.l, b.u)), fminf(__fmul_rd(a.u, b.l), __fmul_rd(a.u, b.u))),
          fmaxf(fmaxf(__fmul_ru(a.l, b.l), __fmul_ru(a.l, b.u)), fmaxf(__fmul_ru(a.u, b.l), __fmul_ru(a.u, b.u)))};
}
__device__ __forceinline__ If iscale(float c, If a) {          // c * a, c a nonzero constant
  return c >= 0.f ? If{__fmul_rd(c, a.l), __fmul_ru(c, a.u)} : If{__fmul_rd(c, a.u), __fmul_ru(c, a.l)};
}
__device__ __forceinline__ If idiv(If a, float c) { return {__fdiv_rd(a.l, c), __fdiv_ru(a.u, c)}; }   // c > 0
__device__ __forceinline__ If isq(If a) {
  if (a.l >= 0.f) return {__fmul_rd(a.l, a.l), __fmul_ru(a.u, a.u)};
  if (a.u <= 0.f) return {__fmul_rd(a.u, a.u), __fmul_ru(a.l, a.l)};
  return {0.f, fmaxf(__fmul_ru(a.l, a.l), __fmul_ru(a.u, a.u))};
}
__device__ __forceinline__ If itanh(If a) {
  return {isnan(a.l) ? -1.f : fmaxf(wdn(tanhf(a.l)), -1.f), isnan(a.u) ? 1.f : fminf(wup(tanhf(a.u)), 1.f)};
}

// true when [l, u] may contain off + 2 k pi for an integer k (conservative: |l|, |u| < 1e6, slack 1e-9 periods)
__device__ __forceinline__ bool may_hit(double l, double u, double off) {
  const double a = (l - off) * (0.5 / kPi), b = (u - off) * (0.5 / kPi);
  return floor(b + 1e-9) >= ceil(a - 1e-9);
}
// sin (cos_phase = false) or cos of [l, u]: the endpoint values widened outward, and +-1 where an extremum may lie inside
__device__ __forceinline__ If isincos(If a, bool cos_phase) {
  if (!(fabsf(a.l) < 1e6f) || !(fabsf(a.u) < 1e6f)) return {-1.f, 1.f};
  const float fl = cos_phase ? cosf(a.l) : sinf(a.l), fu = cos_phase ? cosf(a.u) : sinf(a.u);
  float lo = fminf(wdn(fl), wdn(fu)), hi = fmaxf(wup(fl), wup(fu));
  const double top = cos_phase ? 0.0 : 0.5 * kPi;              // maxima at top + 2 k pi, minima at top + pi + 2 k pi
  if (may_hit(a.l, a.u, top)) hi = 1.f;
  if (may_hit(a.l, a.u, top - kPi)) lo = -1.f;
  return {fmaxf(lo, -1.f), fminf(hi, 1.f)};
}
__device__ __forceinline__ If isin(If a) { return isincos(a, false); }
__device__ __forceinline__ If icos(If a) { return isincos(a, true); }

// ---- float64
__device__ __forceinline__ Id dpt(double c) { return {c, c}; }
__device__ __forceinline__ Id dsane(Id a) { return {isnan(a.l) ? -INFINITY : a.l, isnan(a.u) ? INFINITY : a.u}; }
__device__ __forceinline__ Id dadd(Id a, Id b) { return {__dadd_rd(a.l, b.l), __dadd_ru(a.u, b.u)}; }
__device__ __forceinline__ Id dsub(Id a, Id b) { return {__dsub_rd(a.l, b.u), __dsub_ru(a.u, b.l)}; }
__device__ __forceinline__ Id dmul(Id a, Id b) {
  return {fmin(fmin(__dmul_rd(a.l, b.l), __dmul_rd(a.l, b.u)), fmin(__dmul_rd(a.u, b.l), __dmul_rd(a.u, b.u))),
          fmax(fmax(__dmul_ru(a.l, b.l), __dmul_ru(a.l, b.u)), fmax(__dmul_ru(a.u, b.l), __dmul_ru(a.u, b.u)))};
}
__device__ __forceinline__ Id dscale(double c, Id a) {
  return c >= 0.0 ? Id{__dmul_rd(c, a.l), __dmul_ru(c, a.u)} : Id{__dmul_rd(c, a.u), __dmul_ru(c, a.l)};
}
__device__ __forceinline__ Id dsq(Id a) {
  if (a.l >= 0.0) return {__dmul_rd(a.l, a.l), __dmul_ru(a.u, a.u)};
  if (a.u <= 0.0) return {__dmul_rd(a.u, a.u), __dmul_ru(a.l, a.l)};
  return {0.0, fmax(__dmul_ru(a.l, a.l), __dmul_ru(a.u, a.u))};
}
__device__ __forceinline__ Id ddivpos(Id a, Id d) {           // a / d for d > 0, else the whole line
  if (!(d.l > 0.0)) return {-INFINITY, INFINITY};
  return {fmin(__ddiv_rd(a.l, d.l), __ddiv_rd(a.l, d.u)), fmax(__ddiv_ru(a.u, d.l), __ddiv_ru(a.u, d.u))};
}
__device__ __forceinline__ Id dsincos(Id a, bool cos_phase) {
  if (!(fabs(a.l) < 1e6) || !(fabs(a.u) < 1e6)) return {-1.0, 1.0};
  const double fl = cos_phase ? cos(a.l) : sin(a.l), fu = cos_phase ? cos(a.u) : sin(a.u);
  double lo = fmin(wdn(fl), wdn(fu)), hi = fmax(wup(fl), wup(fu));
  const double top = cos_phase ? 0.0 : 0.5 * kPi;
  if (may_hit(a.l, a.u, top)) hi = 1.0;
  if (may_hit(a.l, a.u, top - kPi)) lo = -1.0;
  return {fmax(lo, -1.0), fmin(hi, 1.0)};
}

template <int ID> struct IEnv;   // VanderPol, Pendulum, DuctedFan, TwoLink; SingleTrackCar / QuadTracking are refused

template <> struct IEnv<kVanderPol> {
  static constexpr bool supported = true;
  static __device__ __forceinline__ void step(If (&o)[2], const If (&a)[1]) {
#pragma unroll 1
    for (int s = 0; s < Env<kVanderPol>::CONTROL_STEP; ++s) {
      const If x = sane(o[0]), dx = sane(o[1]);
      const If ddx = iadd(isub(imul(isub(ipt(1.f), isq(x)), dx), x), a[0]);   // mu (1 - x^2) xdot - x + u, mu = 1
      o[0] = iadd(x, iscale(kDt, dx));
      o[1] = iadd(dx, iscale(kDt, ddx));
    }
  }
};

template <> struct IEnv<kPendulum> {
  static constexpr bool supported = true;
  static __device__ __forceinline__ void step(If (&o)[2], const If (&a)[1]) {
    constexpr float mgl = (float)(0.15 * 9.81 * 0.5);
    constexpr float ml2 = (float)(0.15 * (0.5 * 0.5));
#pragma unroll 1
    for (int s = 0; s < Env<kPendulum>::CONTROL_STEP; ++s) {
      const If th = sane(o[0]), thd = sane(o[1]);
      const If dd = idiv(iadd(isub(iscale(mgl, isin(th)), iscale(0.1f, thd)), a[0]), ml2);
      o[0] = iadd(th, iscale(kDt, thd));
      o[1] = iadd(thd, iscale(kDt, dd));
    }
  }
};

template <> struct IEnv<kDuctedFan> {
  static constexpr bool supported = true;
  static __device__ __forceinline__ void step(If (&o)[6], const If (&a)[2]) {
    constexpr float m = 8.5f, d = 0.95f, r = 0.26f, J = 0.048f;
    constexpr float mg = (float)(8.5 * 9.81), nmg = (float)(-8.5 * 9.81);
#pragma unroll 1
    for (int s = 0; s < Env<kDuctedFan>::CONTROL_STEP; ++s) {
#pragma unroll
      for (int j = 0; j < 6; ++j) o[j] = sane(o[j]);
      const If sn = isin(o[2]), cs = icos(o[2]);
      const If u1 = a[0], u2 = a[1];
      const If ddx = idiv(isub(iadd(isub(iscale(nmg, sn), iscale(d, o[3])), imul(u1, cs)), imul(u2, sn)), m);
      const If ddy = idiv(iadd(iadd(isub(iscale(mg, isub(cs, ipt(1.f))), iscale(d, o[4])), imul(u1, sn)), imul(u2, cs)), m);
      const If ddth = idiv(iscale(r, u1), J);
      const If n0 = iadd(o[0], iscale(kDt, o[3])), n1 = iadd(o[1], iscale(kDt, o[4])), n2 = iadd(o[2], iscale(kDt, o[5]));
      o[3] = iadd(o[3], iscale(kDt, ddx));
      o[4] = iadd(o[4], iscale(kDt, ddy));
      o[5] = iadd(o[5], iscale(kDt, ddth));
      o[0] = n0; o[1] = n1; o[2] = n2;
    }
  }
};

template <> struct IEnv<kTwoLink> {
  static constexpr bool supported = true;
  // the whole step in float64 intervals (the real map has no float32 stage); constants as in Env<kTwoLink>::step
  static __device__ __forceinline__ void step(If (&o)[4], const If (&a)[2]) {
    constexpr double I = (1.0 / 12.0) * 1.0 * (1.0 * 1.0);
    constexpr double p11 = (float)(I + I + 1.0 * (0.5 * 0.5)), c125 = (float)(1.0 * 1.0 + 0.5 * 0.5), c2l = (float)(2 * 1.0 * 0.5);
    constexpr double i2 = (float)I, lc2sq = (float)(0.5 * 0.5), l1lc2 = (float)(1.0 * 0.5);
    constexpr double M22 = I + 1.0 * (0.5 * 0.5);
    constexpr double hk = (float)(-1.0 * 1.0 * 0.5), g1a = (float)(-(1.0 * 0.5 + 1.0 * 1.0) * 9.81);
    constexpr double g1b = (float)(1.0 * 0.5 * 9.81), g2k = (float)(-1.0 * 0.5 * 9.81);
    // det = m11 M22 - m12^2 = A0 + A1 c2 + A2 c2^2 with m11 = (p11 + c125) + c2l c2, m12 = (i2 + lc2sq) + l1lc2 c2
    const Id al = dadd(dpt(p11), dpt(c125)), ga = dadd(dpt(i2), dpt(lc2sq));
    const Id A0 = dsub(dscale(M22, al), dsq(ga));
    const Id A1 = dsub(Id{__dmul_rd(c2l, M22), __dmul_ru(c2l, M22)}, dscale(2.0 * l1lc2, ga));
    const Id A2 = dpt(-(l1lc2 * l1lc2));            // l1lc2 = 0.5: exact
    Id th1 = {o[0].l, o[0].u}, th2 = {o[1].l, o[1].u}, d1 = {o[2].l, o[2].u}, d2 = {o[3].l, o[3].u};
    const Id u0 = {a[0].l, a[0].u}, u1 = {a[1].l, a[1].u};
#pragma unroll 1
    for (int s = 0; s < Env<kTwoLink>::CONTROL_STEP; ++s) {
      th1 = dsane(th1); th2 = dsane(th2); d1 = dsane(d1); d2 = dsane(d2);
      const Id s2 = dsincos(th2, false), c2 = dsincos(th2, true);
      const Id m11 = dadd(al, dscale(c2l, c2));
      const Id m12 = dadd(ga, dscale(l1lc2, c2));
      const Id det = dadd(dadd(A0, dmul(A1, c2)), dmul(A2, dsq(c2)));
      const Id h = dscale(hk, s2);
      const Id Cq1 = dmul(h, dmul(d2, dadd(dscale(2.0, d1), d2)));     // C11 q1 + C12 q2 = h (2 d1 d2 + d2^2)
      const Id Cq2 = dmul(dscale(-1.0, h), dsq(d1));                   // C21 q1 = -h d1^2
      const Id s12 = dsincos(dadd(th1, th2), false);
      const Id G1 = dsub(dscale(g1a, dsincos(th1, false)), dscale(g1b, s12));
      const Id G2 = dscale(g2k, s12);
      const Id b1 = dsub(dsub(u0, Cq1), G1), b2 = dsub(dsub(u1, Cq2), G2);
      const Id x2 = ddivpos(dsub(dmul(m11, b2), dmul(m12, b1)), det);
      const Id x1 = ddivpos(dsub(dscale(M22, b1), dmul(m12, b2)), det);
      const Id n1 = dadd(th1, dscale(kDtD, d1)), n2 = dadd(th2, dscale(kDtD, d2));
      d1 = dadd(d1, dscale(kDtD, x1));
      d2 = dadd(d2, dscale(kDtD, x2));
      th1 = n1; th2 = n2;
    }
    const Id r[4] = {th1, th2, d1, d2};
#pragma unroll
    for (int j = 0; j < 4; ++j) o[j] = {__double2float_rd(r[j].l), __double2float_ru(r[j].u)};
  }
};

template <> struct IEnv<kSingleTrackCar> { static constexpr bool supported = false; };
template <> struct IEnv<kQuadTracking> { static constexpr bool supported = false; };

}  // namespace msacl
