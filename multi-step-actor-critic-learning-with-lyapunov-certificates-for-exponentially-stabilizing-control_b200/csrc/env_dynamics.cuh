// Device-side dynamics of the six MSACL control environments, one env instance per thread,
// state held in registers.  Each Env<ID>::step() is one reference `env.step(action)`:
// control_step explicit-Euler sub-steps, quadratic reward (+ origin bonus) and the raw
// observation.  Termination / truncation / autoreset live in the callers (env_step.cu,
// rollout_fused.cu) because they are identical for all envs.
//
// Numerics: this translation unit is compiled with -fmad=false.  The reference rounds every
// float32 operation separately (NumPy scalar math), so the dynamics below spell out the same
// association and never contract a*b+c; the only places that use FMA are the explicit
// __fmaf_rn calls of the actor GEMM.  float64 appears exactly where the reference's NumPy
// expressions promote to float64 (TwoLink solve, SingleTrackCar f/g arrays, Quadrotor
// translational/attitude-rate terms and the desired-frame pipeline).
//
// Reference (relative to the upstream repo root):
//   RL/env/VanderPol.py:89-130, RL/env/Pendulum.py:93-137, RL/env/DuctedFan.py:99-147,
//   RL/env/TwoLink.py:100-177, RL/env/SingleTrackCar.py:131-320, RL/env/QuadTracking.py:122-360
#pragma once
#include <cmath>
#include <cstdint>

#include "philox.cuh"

namespace msacl {

enum EnvId : int { kVanderPol = 0, kPendulum = 1, kDuctedFan = 2, kTwoLink = 3, kSingleTrackCar = 4, kQuadTracking = 5, kNumEnvs = 6 };

constexpr float kDt = 0.01f;
constexpr double kDtD = 0.01;
constexpr int kMaxStep = 1000;
constexpr double kPi = 3.141592653589793;

template <int ID> struct Env;

// ------------------------------------------------------------------------------------------
// helpers shared by the five "box" envs (state == observation)
// ------------------------------------------------------------------------------------------
template <class E>
__device__ __forceinline__ float box_reward(const float (&o)[E::D], const float (&a)[E::A]) {
  // obs_cost = sum(Q * obs**2), control_cost = sum(R * action**2): left-to-right float32 sums
  float oc = E::q(0) * (o[0] * o[0]);
#pragma unroll
  for (int j = 1; j < E::D; ++j) oc = oc + E::q(j) * (o[j] * o[j]);
  float cc = 0.1f * (a[0] * a[0]);
#pragma unroll
  for (int j = 1; j < E::A; ++j) cc = cc + 0.1f * (a[j] * a[j]);
  float reward = -(oc + cc);
  bool near = true;
#pragma unroll
  for (int j = 0; j < E::D; ++j) near = near && (fabsf(o[j]) <= 0.01f);
  if (near) reward = reward + 1.0f;
  return reward;
}

template <class E>
__device__ __forceinline__ void box_reset(float (&sf)[E::SF], uint64_t seed, uint64_t env, uint32_t episode) {
  // obs = low + (high - low) * u, u from Philox block(s) of the (env, episode) reset stream
#pragma unroll
  for (int b = 0; b < (E::D + 3) / 4; ++b) {
    const U4 r = philox_env(seed, env, episode, kStreamReset + b);
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int j = 4 * b + k;
      if (j < E::D) sf[j] = E::reset_low(j) + (E::reset_high(j) - E::reset_low(j)) * u01(w[k]);
    }
  }
}

#define MSACL_BOX_ENV_COMMON                                                                   \
  static constexpr int SF = D;      /* float32 state rows */                                   \
  static constexpr int SD = 0;      /* float64 state rows */                                   \
  static constexpr int OBS_OFF = 0; /* observation = sf[OBS_OFF .. OBS_OFF+D) */               \
  static constexpr int CONTROL_STEP = 5;                                                       \
  static __device__ __forceinline__ void reset(float (&sf)[SF], double*, uint64_t seed,        \
                                               uint64_t env, uint32_t episode) {               \
    box_reset<Env>(sf, seed, env, episode);                                                    \
  }

// ------------------------------------------------------------------------------------------
template <> struct Env<kVanderPol> {
  static constexpr int D = 2, A = 1;
  MSACL_BOX_ENV_COMMON
  static __device__ __forceinline__ float q(int j) { constexpr float v[D] = {2.f, 1.f}; return v[j]; }
  static __device__ __forceinline__ float obs_low(int j) { return -10.f; }
  static __device__ __forceinline__ float obs_high(int j) { return 10.f; }
  static __device__ __forceinline__ float act_low(int j) { return -5.f; }
  static __device__ __forceinline__ float act_high(int j) { return 5.f; }
  static __device__ __forceinline__ float reset_low(int j) { return -5.f; }
  static __device__ __forceinline__ float reset_high(int j) { return 5.f; }
  static __device__ __forceinline__ float step(float (&o)[SF], double*, const float (&a)[A]) {
#pragma unroll
    for (int s = 0; s < CONTROL_STEP; ++s) {
      const float x = o[0], dx = o[1];
      const float ddx = ((1.0f * (1.0f - x * x)) * dx - x) + a[0];   // mu (1 - x^2) xdot - x + u
      o[0] = x + dx * kDt;
      o[1] = dx + ddx * kDt;
    }
    return box_reward<Env>(o, a);
  }
};

// ------------------------------------------------------------------------------------------
template <> struct Env<kPendulum> {
  static constexpr int D = 2, A = 1;
  MSACL_BOX_ENV_COMMON
  static __device__ __forceinline__ float q(int j) { constexpr float v[D] = {2.f, 1.f}; return v[j]; }
  static __device__ __forceinline__ float obs_low(int j) { return j == 0 ? -(float)kPi : -10.f; }
  static __device__ __forceinline__ float obs_high(int j) { return j == 0 ? (float)kPi : 10.f; }
  static __device__ __forceinline__ float act_low(int j) { return -5.f; }
  static __device__ __forceinline__ float act_high(int j) { return 5.f; }
  static __device__ __forceinline__ float reset_low(int j) { return obs_low(j); }
  static __device__ __forceinline__ float reset_high(int j) { return obs_high(j); }
  static __device__ __forceinline__ float step(float (&o)[SF], double*, const float (&a)[A]) {
    constexpr float mgl = (float)(0.15 * 9.81 * 0.5);
    constexpr float ml2 = (float)(0.15 * (0.5 * 0.5));
#pragma unroll
    for (int s = 0; s < CONTROL_STEP; ++s) {
      const float th = o[0], thd = o[1];
      const float dd = ((mgl * sinf(th) - 0.1f * thd) + a[0]) / ml2;
      o[0] = th + thd * kDt;
      o[1] = thd + dd * kDt;
    }
    return box_reward<Env>(o, a);
  }
};

// ------------------------------------------------------------------------------------------
template <> struct Env<kDuctedFan> {
  static constexpr int D = 6, A = 2;
  MSACL_BOX_ENV_COMMON
  static __device__ __forceinline__ float q(int j) { return j < 3 ? 2.f : 1.f; }
  static __device__ __forceinline__ float obs_low(int j) { return j == 2 ? -(float)(kPi / 2) : -5.f; }
  static __device__ __forceinline__ float obs_high(int j) { return j == 2 ? (float)(kPi / 2) : 5.f; }
  static __device__ __forceinline__ float act_low(int j) { return -5.f; }
  static __device__ __forceinline__ float act_high(int j) { return 5.f; }
  static __device__ __forceinline__ float reset_low(int j) { return -0.5f; }
  static __device__ __forceinline__ float reset_high(int j) { return 0.5f; }
  static __device__ __forceinline__ float step(float (&o)[SF], double*, const float (&a)[A]) {
    constexpr float m = 8.5f, d = 0.95f, r = 0.26f, J = 0.048f;
    constexpr float mg = (float)(8.5 * 9.81), nmg = (float)(-8.5 * 9.81);
#pragma unroll
    for (int s = 0; s < CONTROL_STEP; ++s) {
      float sn, cs;
      sincosf(o[2], &sn, &cs);
      const float u1 = a[0], u2 = a[1];
      const float ddx = (((nmg * sn - d * o[3]) + u1 * cs) - u2 * sn) / m;
      const float ddy = (((mg * (cs - 1.0f) - d * o[4]) + u1 * sn) + u2 * cs) / m;
      const float ddth = (r * u1) / J;
      const float n0 = o[0] + o[3] * kDt, n1 = o[1] + o[4] * kDt, n2 = o[2] + o[5] * kDt;
      o[3] = o[3] + ddx * kDt;
      o[4] = o[4] + ddy * kDt;
      o[5] = o[5] + ddth * kDt;
      o[0] = n0; o[1] = n1; o[2] = n2;
    }
    return box_reward<Env>(o, a);
  }
};

// ------------------------------------------------------------------------------------------
template <> struct Env<kTwoLink> {
  static constexpr int D = 4, A = 2;
  MSACL_BOX_ENV_COMMON
  static __device__ __forceinline__ float q(int j) { return j < 2 ? 2.f : 1.f; }
  static __device__ __forceinline__ float obs_low(int j) { return j < 2 ? -(float)(kPi / 2) : -20.f; }
  static __device__ __forceinline__ float obs_high(int j) { return j < 2 ? (float)(kPi / 2) : 20.f; }
  static __device__ __forceinline__ float act_low(int j) { return -20.f; }
  static __device__ __forceinline__ float act_high(int j) { return 20.f; }
  static __device__ __forceinline__ float reset_low(int j) { return -0.5f; }
  static __device__ __forceinline__ float reset_high(int j) { return 0.5f; }
  static __device__ __forceinline__ float step(float (&o)[SF], double*, const float (&a)[A]) {
    // l1=l2=m1=m2=1, lc=0.5, I=1/12, g=9.81 (TwoLink.py:24-33); Python folds these in float64
    constexpr double I = (1.0 / 12.0) * 1.0 * (1.0 * 1.0);
    constexpr float p11 = (float)(I + I + 1.0 * (0.5 * 0.5));      // I1 + I2 + m1 lc1^2
    constexpr float c125 = (float)(1.0 * 1.0 + 0.5 * 0.5);         // l1^2 + lc2^2
    constexpr float c2l = (float)(2 * 1.0 * 0.5);                  // 2 l1 lc2
    constexpr float i2 = (float)I;
    constexpr float lc2sq = (float)(0.5 * 0.5);
    constexpr float l1lc2 = (float)(1.0 * 0.5);
    constexpr double M22 = I + 1.0 * (0.5 * 0.5);
    constexpr float hk = (float)(-1.0 * 1.0 * 0.5);
    constexpr float g1a = (float)(-(1.0 * 0.5 + 1.0 * 1.0) * 9.81);
    constexpr float g1b = (float)(1.0 * 0.5 * 9.81);
    constexpr float g2k = (float)(-1.0 * 0.5 * 9.81);
#pragma unroll 1
    for (int s = 0; s < CONTROL_STEP; ++s) {
      const float th1 = o[0], th2 = o[1], d1 = o[2], d2 = o[3];
      float s2, c2;
      sincosf(th2, &s2, &c2);
      const float M11 = p11 + 1.0f * (c125 + c2l * c2);
      const float M12 = i2 + 1.0f * (lc2sq + l1lc2 * c2);
      const float h = hk * s2;
      const float C11 = h * d2;
      const float C12 = h * d2 + h * d1;
      const float C21 = (-h) * d1;
      const float s12 = sinf(th1 + th2);
      const float G1 = g1a * sinf(th1) - g1b * s12;
      const float G2 = g2k * s12;
      // float64 from here: rhs = u - C dq - G ; solve [[M11,M12],[M12,M22]] x = rhs (LU, no pivot swap)
      const double q1 = (double)d1, q2 = (double)d2;
      const double Cq1 = (double)C11 * q1 + (double)C12 * q2;
      const double Cq2 = (double)C21 * q1 + 0.0 * q2;
      const double b1 = ((double)a[0] - Cq1) - (double)G1;
      const double b2 = ((double)a[1] - Cq2) - (double)G2;
      const double m11 = (double)M11, m12 = (double)M12;
      // The LU solve above written out: x2 = (m11 b2 - m12 b1) / det, x1 = (M22 b1 - m12 b2) / det with det = m11 M22 - m12^2
      // (>= 0.19 for every theta2; condition number < 50), ONE float64 division per sub-step instead of three.  The
      // result differs from LAPACK's by a few float64 ulps (as the LU form did: dgesv scales by the reciprocal pivot), far
      // below the float32 state it is rounded to; the golden-step tolerance (4e-6) is unchanged.
      const double rdet = 1.0 / (m11 * M22 - m12 * m12);
      const double x2 = (m11 * b2 - m12 * b1) * rdet;
      const double x1 = (M22 * b1 - m12 * b2) * rdet;
      o[0] = (float)((double)th1 + q1 * kDtD);
      o[1] = (float)((double)th2 + q2 * kDtD);
      o[2] = (float)((double)d1 + x1 * kDtD);
      o[3] = (float)((double)d2 + x2 * kDtD);
    }
    return box_reward<Env>(o, a);
  }
};

// ------------------------------------------------------------------------------------------
template <> struct Env<kSingleTrackCar> {
  static constexpr int D = 7, A = 2;
  MSACL_BOX_ENV_COMMON
  static __device__ __forceinline__ float q(int j) { return j < 2 ? 2.f : 1.f; }
  static __device__ __forceinline__ float obs_high(int j) {
    constexpr float v[D] = {1.f, 1.f, (float)1.066, 1.f, (float)(kPi / 2), (float)(kPi / 2), (float)(kPi / 3)};
    return v[j];
  }
  static __device__ __forceinline__ float obs_low(int j) { return -obs_high(j); }
  static __device__ __forceinline__ float act_low(int j) { return -5.f; }
  static __device__ __forceinline__ float act_high(int j) { return 5.f; }
  static __device__ __forceinline__ float reset_low(int j) { return -0.5f; }
  static __device__ __forceinline__ float reset_high(int j) { return 0.5f; }
  static __device__ __forceinline__ float step(float (&o)[SF], double*, const float (&a)[A]) {
    // SingleTrackCar.py:49-64 parameters; all pure-Python sub-expressions fold in float64 first
    constexpr double lf = 0.3048 * 3.793293, lr = 0.3048 * 4.667707, hs = 0.3048 * 2.01355;
    constexpr double m = 4.4482216152605 / 0.3048 * (74.91452), Iz = 4.4482216152605 * 0.3048 * (1321.416);
    constexpr double g = 9.81, mu = 0.1 * 1.0489, CS = -(-21.92) / 1.0489;
    constexpr float mum = (float)(mu * m), Izf = (float)Iz, lsum = (float)(lr + lf), muf = (float)mu;
    constexpr double K2 = mu * m / (Iz * (lr + lf));
    constexpr float f5k1 = (float)(lf * lf * CS * g * lr + lr * lr * CS * g * lf);
    constexpr float f5k2 = (float)(K2 * (lr * CS * g * lf - lf * CS * g * lr));
    constexpr float f5k3 = (float)(K2 * (lf * CS * g * lr));
    constexpr float f6k1 = (float)(CS * g * lf * lr - CS * g * lr * lf);
    constexpr float f6k2 = (float)(CS * g * lf + CS * g * lr);
    constexpr float f6k3 = (float)(CS * g * lr);
    constexpr float g5k1 = (float)(-(lf * lf) * CS * hs + lr * lr * CS * hs);
    constexpr float g5k2 = (float)(K2 * (lr * CS * hs + lf * CS * hs));
    constexpr float g5k3 = (float)(K2 * (lf * CS * hs));
    constexpr float g6k1 = (float)(CS * hs * lr + CS * hs * lf);
    constexpr float g6k2 = (float)(CS * hs - CS * hs);
    constexpr float CSf = (float)CS, hsf = (float)hs;
    constexpr float lwb = (float)(lf + lr), lrf = (float)lr, inv_lwb = (float)(1 / (lf + lr));
    const double u0 = (double)a[0], u1 = (double)a[1];
#pragma unroll 1
    for (int s = 0; s < CONTROL_STEP; ++s) {
      const float sye = o[1], delta = o[2], ve = o[3], psi_e = o[4], psi_e_dot = o[5], beta = o[6];
      const float v = ve + 1.0f;
      const float psi_dot = psi_e_dot + 0.0f;
      float sn, cs;
      sincosf(psi_e + beta, &sn, &cs);
      double f[7], g0[7], g1[7];
      f[0] = (double)((v * cs - 1.0f) + 0.0f * sye);
      f[1] = (double)(v * sn - 0.0f * o[0]);
      f[2] = 0.0;
      f[3] = -0.0;
#pragma unroll
      for (int j = 0; j < 7; ++j) { g0[j] = 0.0; g1[j] = 0.0; }
      if (!(fabsf(v) < 0.1f)) {
        // dynamic single-track model (:176-196, :241-256)
        const float a1 = mum / ((v * Izf) * lsum);
        f[4] = (double)psi_e_dot;
        f[5] = (double)((((-a1) * f5k1) * psi_dot + f5k2 * beta) + f5k3 * delta);
        const float bA = muf / ((v * v) * lsum);
        const float bB = muf / (v * lsum);
        f[6] = (double)((((bA * f6k1 - 1.0f) * psi_dot) - (bB * f6k2) * beta) + (bB * f6k3) * delta);
        g0[2] = 1.0;
        g1[3] = 1.0;
        g1[5] = (double)((((-a1) * g5k1) * psi_dot + g5k2 * beta) - g5k3 * delta);
        g1[6] = (double)((((bA * g6k1) * psi_dot) - (bB * g6k2) * beta) - ((bB * CSf) * hsf) * delta);
      } else {
        // kinematic model (:197-204, :257-277)
        const float td = tanf(delta), cd = cosf(delta), sb = sinf(beta), cb = cosf(beta);
        f[4] = (double)((((v * cb) / lwb) * td) - 0.0f);
        f[5] = 0.0;
        f[6] = 0.0;
        const float tl = (td * lrf) / lwb;
        const float beta_dot = ((1.0f / (1.0f + tl * tl)) * lrf) / (lwb * (cd * cd));
        g1[5] = (double)(inv_lwb * (cb * td));
        g0[5] = (double)(inv_lwb * (((((-v) * sb) * td) * beta_dot) + (v * cb) / (cd * cd)));
        g0[6] = (double)beta_dot;
      }
#pragma unroll
      for (int j = 0; j < 7; ++j) {
        const double dj = f[j] + (g0[j] * u0 + g1[j] * u1);
        o[j] = (float)((double)o[j] + dj * kDtD);
      }
    }
    return box_reward<Env>(o, a);
  }
};

// ------------------------------------------------------------------------------------------
// QuadTracking: float32 state x[0:3] v[3:6] R[6:15] (row-major) Omega[15:18] obs[18:30];
//               float64 state t[0], Rd_last[1:10] (row-major; t_last == previous t)
// ------------------------------------------------------------------------------------------
// Cold path of NormalizeOrientMatrix (QuadTracking.py:312-314): det(U Vh) < 0.  The reference flips the last column of
// U (the singular vector of the SMALLEST singular value) and recomputes U Vh, i.e. R' = Q (I - 2 v3 v3^T) with Q the
// orthogonal polar factor of M (det -1) and v3 the right-singular vector of the smallest singular value = the eigenvector
// of the smallest eigenvalue of P = Q^T M (symmetric positive definite).  v3 is the dominant eigenvector of adj(P)
// (= det(P) P^-1), found by repeated squaring.  Unreachable from the dynamics (the input there is a rotation times
// I + h hat(w), det ~ +1).  Written as rolled loops over local-memory arrays (dynamic indexing, float64): an out-of-line
// call here cost the hot path 8.5 % (the rotation matrix was forced into local memory around the call), a rolled inline
// block costs a predicate.
__device__ __forceinline__ void quad_polar_reflected(float (&R)[9]) {
  double M[9], Q[9], C[9], S[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) { M[i] = (double)R[i]; Q[i] = M[i]; }
  // signed cofactors by the cyclic rule: C_ij = X_(i+1)(j+1) X_(i+2)(j+2) - X_(i+1)(j+2) X_(i+2)(j+1), indices mod 3
  auto cofactors = [](const double* X, double* Cf) {
#pragma unroll 1
    for (int e = 0; e < 9; ++e) {
      const int i = e / 3, j = e - 3 * i;
      const int i1 = (i + 1) % 3, i2 = (i + 2) % 3, j1 = (j + 1) % 3, j2 = (j + 2) % 3;
      Cf[e] = X[3 * i1 + j1] * X[3 * i2 + j2] - X[3 * i1 + j2] * X[3 * i2 + j1];
    }
  };
#pragma unroll 1
  for (int it = 0; it < 40; ++it) {            // Newton: Q <- (Q + Q^-T)/2, converges to the orthogonal factor (det -1)
    cofactors(Q, C);
    const double det = Q[0] * C[0] + Q[1] * C[1] + Q[2] * C[2];
    double delta = 0.0;
#pragma unroll 1
    for (int e = 0; e < 9; ++e) { const double q = 0.5 * (Q[e] + C[e] / det); delta += fabs(q - Q[e]); Q[e] = q; }
    if (delta < 1e-15) break;
  }
#pragma unroll 1
  for (int e = 0; e < 9; ++e) {                 // S = Q^T M
    const int i = e / 3, j = e - 3 * i;
    S[e] = Q[i] * M[j] + Q[3 + i] * M[3 + j] + Q[6 + i] * M[6 + j];
  }
#pragma unroll 1
  for (int e = 0; e < 9; ++e) {                 // P = sym(S), kept in M
    const int i = e / 3, j = e - 3 * i;
    M[e] = 0.5 * (S[e] + S[3 * j + i]);
  }
  cofactors(M, C);                              // symmetric P: adj(P) = cofactor matrix
#pragma unroll 1
  for (int it = 0; it < 12; ++it) {             // C <- C^2 / trace: rank-1 projector on the smallest eigenvector of P
#pragma unroll 1
    for (int e = 0; e < 9; ++e) {
      const int i = e / 3, j = e - 3 * i;
      S[e] = C[3 * i] * C[j] + C[3 * i + 1] * C[3 + j] + C[3 * i + 2] * C[6 + j];
    }
    const double tr = S[0] + S[4] + S[8];
#pragma unroll 1
    for (int e = 0; e < 9; ++e) C[e] = S[e] / tr;
  }
  int best = 0;
  double bn = -1.0;
#pragma unroll 1
  for (int j = 0; j < 3; ++j) {
    const double nn = C[j] * C[j] + C[3 + j] * C[3 + j] + C[6 + j] * C[6 + j];
    if (nn > bn) { bn = nn; best = j; }
  }
  const double inv = rsqrt(bn);
#pragma unroll 1
  for (int i = 0; i < 3; ++i) S[i] = C[3 * i + best] * inv;          // v3
#pragma unroll 1
  for (int i = 0; i < 3; ++i) {                 // R' = Q - 2 (Q v) v^T
    const double qv = Q[3 * i] * S[0] + Q[3 * i + 1] * S[1] + Q[3 * i + 2] * S[2];
#pragma unroll 1
    for (int j = 0; j < 3; ++j) M[3 * i + j] = Q[3 * i + j] - 2.0 * qv * S[j];
  }
#pragma unroll
  for (int i = 0; i < 9; ++i) R[i] = (float)M[i];
}

__device__ __forceinline__ void quad_polar_f32(float (&R)[9], float theta2) {
  // Orthogonal polar factor of a near-rotation 3x3 (reference: U @ Vh of np.linalg.svd,
  // QuadTracking.py:308-315).  Newton iteration X <- (X + X^-T)/2: every singular value 1 + e goes to 1 + e^2/2.
  // The input is (rotation) x (I + h hat(w)), singular values sqrt(1 + theta^2), theta = h |w|, i.e. e0 = theta^2/2:
  // two sweeps leave e0^4/8 (< 1e-9 for theta^2 < 0.02, below float32 round-off); a third sweep only runs for
  // theta^2 >= 0.02 (|w| > 14 rad/s, at the edge of the observation box).
  // The det<0 branch of the reference (:312-314) cannot trigger for such inputs (det ~ +1); it is honoured by the
  // out-of-line quad_polar_reflected() behind the predicate on the first sweep's determinant.
  // (The sweep is not a restatement of a NumPy expression, so it uses explicit fused multiply-adds: fewer
  // instructions and fewer roundings; everything that mirrors reference arithmetic stays unfused.)
  auto sweep = [&](bool first) -> bool {
    auto cof = [](float a, float b, float c, float d) { return __fmaf_rn(a, b, -(c * d)); };   // a*b - c*d
    const float c00 = cof(R[4], R[8], R[5], R[7]), c01 = cof(R[5], R[6], R[3], R[8]), c02 = cof(R[3], R[7], R[4], R[6]);
    const float c10 = cof(R[2], R[7], R[1], R[8]), c11 = cof(R[0], R[8], R[2], R[6]), c12 = cof(R[1], R[6], R[0], R[7]);
    const float c20 = cof(R[1], R[5], R[2], R[4]), c21 = cof(R[2], R[3], R[0], R[5]), c22 = cof(R[0], R[4], R[1], R[3]);
    const float det = __fmaf_rn(R[2], c02, __fmaf_rn(R[1], c01, R[0] * c00));
    if (first && det < 0.0f) return false;
    const float hid = 0.5f / det;                 // (an approximate reciprocal here measured 1.5 % slower end to end)
    R[0] = __fmaf_rn(c00, hid, 0.5f * R[0]); R[1] = __fmaf_rn(c01, hid, 0.5f * R[1]); R[2] = __fmaf_rn(c02, hid, 0.5f * R[2]);
    R[3] = __fmaf_rn(c10, hid, 0.5f * R[3]); R[4] = __fmaf_rn(c11, hid, 0.5f * R[4]); R[5] = __fmaf_rn(c12, hid, 0.5f * R[5]);
    R[6] = __fmaf_rn(c20, hid, 0.5f * R[6]); R[7] = __fmaf_rn(c21, hid, 0.5f * R[7]); R[8] = __fmaf_rn(c22, hid, 0.5f * R[8]);
    return true;
  };
  if (!sweep(true)) { quad_polar_reflected(R); return; }
  sweep(false);
  if (theta2 >= 0.02f) sweep(false);
}

// desired frame at time t for position x / velocity v (QuadTracking.py:122-139, trajectory :29-36)
__device__ __forceinline__ void quad_desired(const float* x, const float* v, double t, double (&xd)[3],
                                             float (&vd)[3], double (&Rd)[9]) {
  double st, ct;
  sincos(t, &st, &ct);
  xd[0] = 0.4 * t; xd[1] = 0.4 * st; xd[2] = 0.6 * ct;
  vd[0] = (float)0.4; vd[1] = (float)(0.4 * ct); vd[2] = (float)(-0.6 * st);
  const float ad[3] = {0.0f, (float)(-0.4 * st), (float)(-0.6 * ct)};
  constexpr float nkx = (float)(-69.44), kv = (float)24.304, mf = (float)4.34;
  constexpr double gz = 9.8, m = 4.34;
  double fd[3];
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const float ex = (float)((double)x[j] - xd[j]);
    const float ev = v[j] - vd[j];
    const float p = nkx * ex - kv * ev;                  // float32 part
    const double mg = (j == 2) ? m * gz : m * 0.0;
    fd[j] = -(((double)p - mg) + (double)(mf * ad[j]));
  }
  // normalisations as x * rsqrt(|x|^2): differs from x / sqrt(|x|^2) by a few float64 ulps, far below the float32
  // resolution every consumer of the desired frame is rounded to (one reciprocal square root instead of a square
  // root and three divisions on the float64 pipe)
  const double ifn = rsqrt((fd[0] * fd[0] + fd[1] * fd[1]) + fd[2] * fd[2]);
  const double b3[3] = {fd[0] * ifn, fd[1] * ifn, fd[2] * ifn};
  const double b1[3] = {ct, st, 0.0};
  double c[3] = {b3[1] * b1[2] - b3[2] * b1[1], b3[2] * b1[0] - b3[0] * b1[2], b3[0] * b1[1] - b3[1] * b1[0]};
  const double icn = rsqrt((c[0] * c[0] + c[1] * c[1]) + c[2] * c[2]);
  const double b2[3] = {c[0] * icn, c[1] * icn, c[2] * icn};
  const double bn[3] = {b2[1] * b3[2] - b2[2] * b3[1], b2[2] * b3[0] - b2[0] * b3[2], b2[0] * b3[1] - b2[1] * b3[0]};
#pragma unroll
  for (int i = 0; i < 3; ++i) { Rd[3 * i + 0] = bn[i]; Rd[3 * i + 1] = b2[i]; Rd[3 * i + 2] = b3[i]; }
}

// tracking errors -> obs[12] (QuadTracking.py:317-338)
__device__ __forceinline__ void quad_errors(const float* x, const float* v, const float* R, const float* Om,
                                            const double (&xd)[3], const float (&vd)[3], const double (&Rd)[9],
                                            const double (&Omd)[3], float* obs) {
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    obs[j] = (float)((double)x[j] - xd[j]);
    obs[3 + j] = v[j] - vd[j];
  }
  // E = Rd^T R - R^T Rd ; eR = 0.5 * vee(E) with vee = (E[2][1], E[0][2], E[1][0]).  M = Rd^T R is formed once:
  // (R^T Rd)[i][j] = M[j][i] term by term (same products, same association), so nothing changes numerically.
  double M[9];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j)
      M[3 * i + j] = (Rd[0 + i] * (double)R[0 + j] + Rd[3 + i] * (double)R[3 + j]) + Rd[6 + i] * (double)R[6 + j];
  obs[6] = (float)(M[3 * 2 + 1] - M[3 * 1 + 2]) * 0.5f;
  obs[7] = (float)(M[3 * 0 + 2] - M[3 * 2 + 0]) * 0.5f;
  obs[8] = (float)(M[3 * 1 + 0] - M[3 * 0 + 1]) * 0.5f;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const double w = (M[3 * 0 + i] * Omd[0] + M[3 * 1 + i] * Omd[1]) + M[3 * 2 + i] * Omd[2];
    obs[9 + i] = (float)((double)Om[i] - w);
  }
}

template <> struct Env<kQuadTracking> {
  static constexpr int D = 12, A = 4;
  static constexpr int SF = 30, SD = 10, OBS_OFF = 18, CONTROL_STEP = 4;
  static __device__ __forceinline__ float obs_low(int j) { return -10.f; }
  static __device__ __forceinline__ float obs_high(int j) { return 10.f; }
  static __device__ __forceinline__ float act_low(int j) { return j == 0 ? (float)(0.0 * (4.34 * 9.8)) : -10.f; }
  static __device__ __forceinline__ float act_high(int j) { return j == 0 ? (float)(2.0 * (4.34 * 9.8)) : 10.f; }

  static __device__ __forceinline__ float step(float (&sf)[SF], double (&sd)[SD], const float (&a)[A]) {
    float* x = sf; float* v = sf + 3; float* Om = sf + 15; float* obs = sf + 18;
    float R[9];
#pragma unroll
    for (int j = 0; j < 9; ++j) R[j] = sf[6 + j];
    const float force = a[0];
    constexpr float mf = (float)4.34;
    constexpr double J0 = 0.0820, J1 = 0.0845, J2 = 0.1377;
    constexpr double iJ0 = 1.0 / 0.0820, iJ1 = 1.0 / 0.0845, iJ2 = 1.0 / 0.1377;
#pragma unroll 1
    for (int s = 0; s < CONTROL_STEP; ++s) {
      // derivatives from the OLD state (:212-217)
      const double dv0 = 0.0 - (double)((force * R[2]) / mf);
      const double dv1 = 0.0 - (double)((force * R[5]) / mf);
      const double dv2 = 9.8 - (double)((force * R[8]) / mf);
      const float w0 = Om[0], w1 = Om[1], w2 = Om[2];
      float dR[9];
#pragma unroll
      for (int i = 0; i < 3; ++i) {   // R @ hat(w), hat = [[0,-w2,w1],[w2,0,-w0],[-w1,w0,0]]
        dR[3 * i + 0] = R[3 * i + 1] * w2 + R[3 * i + 2] * (-w1);
        dR[3 * i + 1] = R[3 * i + 0] * (-w2) + R[3 * i + 2] * w0;
        dR[3 * i + 2] = R[3 * i + 0] * w1 + R[3 * i + 1] * (-w0);
      }
      const double jw0 = J0 * (double)w0, jw1 = J1 * (double)w1, jw2 = J2 * (double)w2;
      const double cr0 = (double)w1 * jw2 - (double)w2 * jw1;
      const double cr1 = (double)w2 * jw0 - (double)w0 * jw2;
      const double cr2 = (double)w0 * jw1 - (double)w1 * jw0;
      const double dO0 = iJ0 * ((double)a[1] - cr0), dO1 = iJ1 * ((double)a[2] - cr1), dO2 = iJ2 * ((double)a[3] - cr2);
      // explicit Euler, each state re-rounded to float32 (:219-224)
#pragma unroll
      for (int j = 0; j < 3; ++j) x[j] = x[j] + v[j] * kDt;
      v[0] = (float)((double)v[0] + dv0 * kDtD);
      v[1] = (float)((double)v[1] + dv1 * kDtD);
      v[2] = (float)((double)v[2] + dv2 * kDtD);
#pragma unroll
      for (int j = 0; j < 9; ++j) R[j] = R[j] + dR[j] * kDt;
      Om[0] = (float)((double)w0 + dO0 * kDtD);
      Om[1] = (float)((double)w1 + dO1 * kDtD);
      Om[2] = (float)((double)w2 + dO2 * kDtD);
      quad_polar_f32(R, (kDt * kDt) * ((w0 * w0 + w1 * w1) + w2 * w2));
    }
#pragma unroll
    for (int j = 0; j < 9; ++j) sf[6 + j] = R[j];
    // time, desired frame, numerical angular velocity of the desired frame (:229-238)
    const double t_last = sd[0];
    const double t = t_last + kDtD * 4;
    double xd[3], Rd[9], Omd[3];
    float vd[3];
    quad_desired(x, v, t, xd, vd, Rd);
    double dtt = t - t_last;
    if (dtt < 1e-6) dtt = 1e-6;
    const double inv_dtt = 1.0 / dtt;                  // one float64 division instead of nine (same argument as above)
    float Rdd[9];
#pragma unroll
    for (int j = 0; j < 9; ++j) Rdd[j] = (float)((Rd[j] - sd[1 + j]) * inv_dtt);
    auto RdT_Rdd = [&](int i, int j) {
      return (Rd[0 + i] * (double)Rdd[0 + j] + Rd[3 + i] * (double)Rdd[3 + j]) + Rd[6 + i] * (double)Rdd[6 + j];
    };
    Omd[0] = (double)(float)RdT_Rdd(2, 1);
    Omd[1] = (double)(float)RdT_Rdd(0, 2);
    Omd[2] = (double)(float)RdT_Rdd(1, 0);
    sd[0] = t;
#pragma unroll
    for (int j = 0; j < 9; ++j) sd[1 + j] = Rd[j];
    quad_errors(x, v, R, Om, xd, vd, Rd, Omd, obs);
    // reward (:250-267): five float32 partial sums, then the linear origin bonus
    const float s0 = (obs[0] * obs[0] + obs[1] * obs[1]) + obs[2] * obs[2];
    const float s1 = (obs[3] * obs[3] + obs[4] * obs[4]) + obs[5] * obs[5];
    const float s2 = (obs[6] * obs[6] + obs[7] * obs[7]) + obs[8] * obs[8];
    const float s3 = (obs[9] * obs[9] + obs[10] * obs[10]) + obs[11] * obs[11];
    const float s4 = ((0.0001f * (a[0] * a[0]) + 0.01f * (a[1] * a[1])) + 0.01f * (a[2] * a[2])) + 0.01f * (a[3] * a[3]);
    float reward = -((((s0 + s1) + s2) + s3) + s4);
    float dist = 0.f;
#pragma unroll
    for (int j = 0; j < 12; ++j) dist = fmaxf(dist, fabsf(obs[j]));
    if (dist <= 0.1f) reward = reward + 10.0f * (1.0f - dist / 0.1f);
    return reward;
  }

  static __device__ __forceinline__ void reset(float (&sf)[SF], double (&sd)[SD], uint64_t seed, uint64_t env,
                                               uint32_t episode) {
    // x, v, Omega ~ U(+-0.01); R = exp(hat(0.01 z)), z ~ N(0, I3)   (distribution of :169-188)
    const U4 r0 = philox_env(seed, env, episode, kStreamReset + 0);
    const U4 r1 = philox_env(seed, env, episode, kStreamReset + 1);
    const U4 r2 = philox_env(seed, env, episode, kStreamReset + 2);
    const U4 r3 = philox_env(seed, env, episode, kStreamReset + 3);
    const uint32_t w[9] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w, r2.x};
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      sf[j] = -0.01f + 0.02f * u01(w[j]);
      sf[3 + j] = -0.01f + 0.02f * u01(w[3 + j]);
      sf[15 + j] = -0.01f + 0.02f * u01(w[6 + j]);
    }
    float z[4];
    box_muller(r3.x, r3.y, z[0], z[1]);
    box_muller(r3.z, r3.w, z[2], z[3]);
    const float k0 = 0.01f * z[0], k1 = 0.01f * z[1], k2 = 0.01f * z[2];
    const float th2 = (k0 * k0 + k1 * k1) + k2 * k2;
    const float th = sqrtf(th2);
    float Ac, Bc;
    if (th < 1e-4f) { Ac = 1.0f - th2 / 6.0f; Bc = 0.5f - th2 / 24.0f; }
    else { Ac = sinf(th) / th; Bc = (1.0f - cosf(th)) / (th * th); }
    const float K[9] = {0.f, -k2, k1, k2, 0.f, -k0, -k1, k0, 0.f};
    float* R = sf + 6;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        const float kk = (K[3 * i] * K[j] + K[3 * i + 1] * K[3 + j]) + K[3 * i + 2] * K[6 + j];
        R[3 * i + j] = ((i == j ? 1.0f : 0.0f) + Ac * K[3 * i + j]) + Bc * kk;
      }
    // initial observation with Omega_d = 0 and Rd_last <- Rd(t=0) (:190-201)
    double xd[3], Rd[9];
    float vd[3];
    quad_desired(sf, sf + 3, 0.0, xd, vd, Rd);
    const double Omd[3] = {0.0, 0.0, 0.0};
    quad_errors(sf, sf + 3, R, sf + 15, xd, vd, Rd, Omd, sf + 18);
    sd[0] = 0.0;
#pragma unroll
    for (int j = 0; j < 9; ++j) sd[1 + j] = Rd[j];
  }
};

// cost = sum(real_next_obs^2) * cost_scale with NumPy's pairwise association
// (RL/utils/rew_plus_cost.py:20-21; see oracle.envs.np_pairwise_rowsum)
template <int D>
__device__ __forceinline__ float np_rowsum_sq(const float* o) {
  if constexpr (D < 8) {
    float acc = o[0] * o[0];
#pragma unroll
    for (int j = 1; j < D; ++j) acc = acc + o[j] * o[j];
    return acc;
  } else {
    float r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = o[j] * o[j];
    constexpr int full = D - (D % 8);
#pragma unroll
    for (int i = 8; i < full; i += 8)
#pragma unroll
      for (int j = 0; j < 8; ++j) r[j] = r[j] + o[i + j] * o[i + j];
    float res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
#pragma unroll
    for (int i = full; i < D; ++i) res = res + o[i] * o[i];
    return res;
  }
}

}  // namespace msacl
