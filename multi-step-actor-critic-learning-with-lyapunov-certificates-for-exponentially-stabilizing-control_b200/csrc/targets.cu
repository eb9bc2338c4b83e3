// MSACL learner targets over [B, n] replay windows, given the network outputs.
// Replaces the ~40 small elementwise/reduction torch ops of RL/algorithm/msacl.py:
//   soft-TD backup :249-252, Lyapunov risk :280-329 (+ analytic backward), stability
//   advantage :392-400.  One warp per window: lane k owns step k (n <= 32), the clipped
//   importance-ratio cumprod is a warp scan and the lambda-weighted sums are warp reductions.
// HBM-bound: algorithmic bytes per window = 4*n*(2D + 4) read + 4*n*2 written (risk).
#include <cstdlib>

#include "common.cuh"

namespace msacl {

__global__ void __launch_bounds__(256)
q_backup_kernel(int64_t count, const float* __restrict__ rew, const float* __restrict__ done,
                const float* __restrict__ q1, const float* __restrict__ q2, const float* __restrict__ logp, float gamma,
                float alpha, float* __restrict__ backup) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride) {
    const float nq = fminf(q1[i], q2[i]);
    backup[i] = rew[i] + ((1.0f - done[i]) * gamma) * (nq - alpha * logp[i]);   // msacl.py:250-252
  }
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// DT = compile-time obs_dim (0: run-time D).  The kernel is instruction-issue bound before it is HBM bound (a warp
// per 20-step window moves only 1.4 KB), so the per-window instruction stream is kept lean: no run-time loops over D,
// one running 64-bit element index, all loads of a window issued before the first use.
template <int WPB, int DT>
__global__ void __launch_bounds__(WPB * 32)
lyapunov_risk_kernel(int64_t B, int n, int D_rt, const float* __restrict__ obs, const float* __restrict__ obs2,
                     const float* __restrict__ logp_new, const float* __restrict__ logp_old,
                     const float* __restrict__ lya_obs, const float* __restrict__ lya_obs2,
                     const float* __restrict__ coef_son, const float* __restrict__ coef_diff,
                     const float* __restrict__ coef_sl, float alpha1, float alpha2, float diff_scale, float pos_scale,
                     double* __restrict__ loss_parts, float* __restrict__ g_obs, float* __restrict__ g_obs2,
                     float* __restrict__ is_clip_out, float* __restrict__ esl_out) {
  __shared__ float s_part[3][WPB];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool act = lane < n;
  const int D = DT > 0 ? DT : D_rt;
  const float son = act ? coef_son[lane] : 0.f, dif = act ? coef_diff[lane] : 0.f, sl = act ? coef_sl[lane] : 0.f;
  const float inv_bn = pos_scale / (float)((double)B * n);
  const float w_scale = diff_scale / (float)B;
  float p0 = 0.f, p1 = 0.f, p2 = 0.f;
  const int64_t wstride = (int64_t)gridDim.x * WPB;
  const int64_t estep = wstride * n;
  int64_t b = (int64_t)blockIdx.x * WPB + warp;
  for (int64_t e = b * n + lane; b < B; b += wstride, e += estep) {
    float ratio = 1.f, v1 = 0.f, v2 = 0.f, op = 0.f, op2 = 0.f;
    if (act) {
      const float ln = logp_new[e], lo_ = logp_old[e];
      v1 = lya_obs[e]; v2 = lya_obs2[e];
      const float* o = obs + e * D;
      const float* q = obs2 + e * D;
      if constexpr (DT > 0 && DT % 4 == 0) {            // rows are 16-byte aligned: vector loads
        float4 a[DT / 4], c[DT / 4];
#pragma unroll
        for (int d = 0; d < DT / 4; ++d) { a[d] = reinterpret_cast<const float4*>(o)[d]; c[d] = reinterpret_cast<const float4*>(q)[d]; }
#pragma unroll
        for (int d = 0; d < DT / 4; ++d) {
          op = __fmaf_rn(a[d].x, a[d].x, op); op = __fmaf_rn(a[d].y, a[d].y, op); op = __fmaf_rn(a[d].z, a[d].z, op); op = __fmaf_rn(a[d].w, a[d].w, op);
          op2 = __fmaf_rn(c[d].x, c[d].x, op2); op2 = __fmaf_rn(c[d].y, c[d].y, op2); op2 = __fmaf_rn(c[d].z, c[d].z, op2); op2 = __fmaf_rn(c[d].w, c[d].w, op2);
        }
      } else if constexpr (DT > 0 && DT % 2 == 0) {
        float2 a[DT / 2], c[DT / 2];
#pragma unroll
        for (int d = 0; d < DT / 2; ++d) { a[d] = reinterpret_cast<const float2*>(o)[d]; c[d] = reinterpret_cast<const float2*>(q)[d]; }
#pragma unroll
        for (int d = 0; d < DT / 2; ++d) {
          op = __fmaf_rn(a[d].x, a[d].x, op); op = __fmaf_rn(a[d].y, a[d].y, op);
          op2 = __fmaf_rn(c[d].x, c[d].x, op2); op2 = __fmaf_rn(c[d].y, c[d].y, op2);
        }
      } else if constexpr (DT > 0) {
        float a[DT], c[DT];
#pragma unroll
        for (int d = 0; d < DT; ++d) { a[d] = o[d]; c[d] = q[d]; }
#pragma unroll
        for (int d = 0; d < DT; ++d) { op = __fmaf_rn(a[d], a[d], op); op2 = __fmaf_rn(c[d], c[d], op2); }
      } else {
        for (int d = 0; d < D; ++d) { op = __fmaf_rn(o[d], o[d], op); op2 = __fmaf_rn(q[d], q[d], op2); }
      }
      ratio = fminf(fmaxf(expf(ln - lo_), 0.f), 1.f);   // clamp(ratio, 0, 1) :284-285
    }
    // inclusive cumprod over the window (:286)
    float c = ratio;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const float y = __shfl_up_sync(0xffffffffu, c, o);
      if (lane >= o) c *= y;
    }
    const float lo = alpha1 * op - v1, up = v1 - alpha2 * op;           // boundedness hinge :291-301
    const float start_norm = sqrtf(__shfl_sync(0xffffffffu, op, 0));    // ||o_0|| :306-307
    const float start_lya = __shfl_sync(0xffffffffu, v1, 0);
    const float esl = (start_norm * son - sqrtf(op2)) >= 0.f ? 1.f : -1.f;   // :308-312
    const float inner = esl * (v2 - start_lya * sl);                    // :318-323
    const float term = c * fmaxf(inner, 0.f);
    const float w = (act && inner > 0.f) ? dif * c * esl * w_scale : 0.f;
    const float back0 = warp_sum(w * sl);
    if (act) {
      p0 += fmaxf(lo, 0.f);
      p1 += fmaxf(up, 0.f);
      p2 += dif * term;
      float g1 = ((lo > 0.f) ? -inv_bn : 0.f) + ((up > 0.f) ? inv_bn : 0.f);
      if (lane == 0) g1 -= back0;
      g_obs[e] = g1;
      g_obs2[e] = w;
      if (is_clip_out) is_clip_out[e] = c;
      if (esl_out) esl_out[e] = esl;
    }
  }
  p0 = warp_sum(p0); p1 = warp_sum(p1); p2 = warp_sum(p2);
  if (lane == 0) { s_part[0][warp] = p0; s_part[1][warp] = p1; s_part[2][warp] = p2; }
  __syncthreads();
  if (threadIdx.x < 3) {
    double s = 0.0;
    for (int w = 0; w < WPB; ++w) s += (double)s_part[threadIdx.x][w];
    atomicAdd(&loss_parts[threadIdx.x], s);
  }
}

// All-lanes-live variant: a warp walks tiles of 32 P consecutive (window, step) elements, P = n / gcd(n, 32), so that a tile
// holds whole windows (n = 20: 160 elements = 8 windows in 5 passes; n = 16: 2 windows in 1 pass).  Lane l of pass p owns
// element 32 p + l of the tile -- coalesced loads, every lane busy (the warp-per-window kernel above keeps only n of 32
// lanes busy and is instruction-issue bound at ~0.47 of the HBM peak for n = 20).  A window spans at most two passes
// (n <= 32), so the clipped-ratio cumprod is a segmented warp scan plus one carry from the previous pass, the window
// head's (||o_0||, V(o_0)) come from this or the previous pass by one shuffle each, and the head's back-propagated sum is
// a segmented suffix sum plus the continuation at lane 0 of the next pass.  Same arithmetic per element as the kernel above; only the association of the cumprod / window sums
// differs for windows that straddle two passes.
template <int WPB, int P, int DT>
__global__ void __launch_bounds__(WPB * 32, 2)
lyapunov_risk_striped_kernel(int64_t B, int n, const float* __restrict__ obs, const float* __restrict__ obs2,
                             const float* __restrict__ logp_new, const float* __restrict__ logp_old,
                             const float* __restrict__ lya_obs, const float* __restrict__ lya_obs2,
                             const float* __restrict__ coef_son, const float* __restrict__ coef_diff,
                             const float* __restrict__ coef_sl, float alpha1, float alpha2, float diff_scale, float pos_scale,
                             double* __restrict__ loss_parts, float* __restrict__ g_obs, float* __restrict__ g_obs2,
                             float* __restrict__ is_clip_out, float* __restrict__ esl_out) {
  static_assert(DT > 0, "compile-time obs_dim");
  __shared__ float s_part[3][WPB];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int T = 32 * P;
  const int64_t total = B * (int64_t)n;
  const float inv_bn = pos_scale / (float)((double)B * n);
  const float w_scale = diff_scale / (float)B;
  // tile-relative step index of this lane's element in every pass, and the coefficients of that step
  int kk[P];
  float son[P], dif[P], sl[P];
#pragma unroll
  for (int p = 0; p < P; ++p) {
    kk[p] = (32 * p + lane) % n;
    son[p] = coef_son[kk[p]]; dif[p] = coef_diff[kk[p]]; sl[p] = coef_sl[kk[p]];
  }
  float p0 = 0.f, p1 = 0.f, p2 = 0.f;
  const int64_t tiles = (total + T - 1) / T;
  for (int64_t tile = (int64_t)blockIdx.x * WPB + warp; tile < tiles; tile += (int64_t)gridDim.x * WPB) {
    const int64_t e0 = tile * T + lane;
    float ratio[P], v1[P], v2[P], op[P], op2[P];
    // ---- loads, pass by pass (measured: hoisting all P passes' loads in front of the first use -- 30 loads in flight per
    //      lane -- is slower, 0.54 vs 0.59 of the HBM peak: the compute of pass p no longer overlaps the loads of pass p + 1)
#pragma unroll
    for (int p = 0; p < P; ++p) {
      const int64_t e = e0 + 32 * p;
      ratio[p] = 1.f; v1[p] = 0.f; v2[p] = 0.f; op[p] = 0.f; op2[p] = 0.f;
      if (e < total) {
        const float ln = logp_new[e], lo_ = logp_old[e];
        v1[p] = lya_obs[e]; v2[p] = lya_obs2[e];
        const float* o = obs + e * DT;
        const float* q = obs2 + e * DT;
        float a[DT], c[DT];
        if constexpr (DT % 4 == 0) {
#pragma unroll
          for (int d = 0; d < DT / 4; ++d) {
            const float4 x = reinterpret_cast<const float4*>(o)[d], y = reinterpret_cast<const float4*>(q)[d];
            a[4 * d] = x.x; a[4 * d + 1] = x.y; a[4 * d + 2] = x.z; a[4 * d + 3] = x.w;
            c[4 * d] = y.x; c[4 * d + 1] = y.y; c[4 * d + 2] = y.z; c[4 * d + 3] = y.w;
          }
        } else if constexpr (DT % 2 == 0) {
#pragma unroll
          for (int d = 0; d < DT / 2; ++d) {
            const float2 x = reinterpret_cast<const float2*>(o)[d], y = reinterpret_cast<const float2*>(q)[d];
            a[2 * d] = x.x; a[2 * d + 1] = x.y; c[2 * d] = y.x; c[2 * d + 1] = y.y;
          }
        } else {
#pragma unroll
          for (int d = 0; d < DT; ++d) { a[d] = o[d]; c[d] = q[d]; }
        }
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int d = 0; d < DT; ++d) { s1 = __fmaf_rn(a[d], a[d], s1); s2 = __fmaf_rn(c[d], c[d], s2); }
        op[p] = s1; op2[p] = s2;
        ratio[p] = fminf(fmaxf(expf(ln - lo_), 0.f), 1.f);   // clamp(ratio, 0, 1) :284-285
      }
    }
    // ---- per pass: segmented cumprod (:286), window-head values, hinge terms
    float cp[P], wv[P], g1[P], es[P], sfx[P];
    float carry = 1.f;
#pragma unroll
    for (int p = 0; p < P; ++p) {
      const int k = kk[p];
      float c = ratio[p];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const float y = __shfl_up_sync(0xffffffffu, c, o);
        if (lane >= o && k >= o) c *= y;
      }
      if (k > lane) c *= carry;                     // the window began in the previous pass
      carry = __shfl_sync(0xffffffffu, c, 31);
      cp[p] = c;
      const int src = (lane - k) & 31;              // lane of the window head, in this pass (k <= lane) or the previous one
      float h_op = __shfl_sync(0xffffffffu, op[p], src), h_v1 = __shfl_sync(0xffffffffu, v1[p], src);
      if (p > 0) {
        const float q_op = __shfl_sync(0xffffffffu, op[p > 0 ? p - 1 : 0], src), q_v1 = __shfl_sync(0xffffffffu, v1[p > 0 ? p - 1 : 0], src);
        if (k > lane) { h_op = q_op; h_v1 = q_v1; }
      }
      const bool live = e0 + 32 * p < total;
      const float lo = alpha1 * op[p] - v1[p], up = v1[p] - alpha2 * op[p];           // boundedness hinge :291-301
      const float start_norm = sqrtf(h_op);                                              // ||o_0|| :306-307
      const float esl = (start_norm * son[p] - sqrtf(op2[p])) >= 0.f ? 1.f : -1.f;      // :308-312
      const float inner = esl * (v2[p] - h_v1 * sl[p]);                                  // :318-323
      const float term = c * fmaxf(inner, 0.f);
      const float w = (live && inner > 0.f) ? dif[p] * c * esl * w_scale : 0.f;
      wv[p] = w; es[p] = esl;
      // suffix sum of w * sl inside the window, within this pass
      float sx = w * sl[p];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const float y = __shfl_down_sync(0xffffffffu, sx, o);
        if (lane + o < 32 && k + o < n) sx += y;
      }
      sfx[p] = sx;
      g1[p] = ((lo > 0.f) ? -inv_bn : 0.f) + ((up > 0.f) ? inv_bn : 0.f);
      if (live) {
        p0 += fmaxf(lo, 0.f);
        p1 += fmaxf(up, 0.f);
        p2 += dif[p] * term;
      }
    }
    // ---- window heads take the back-propagated sum (continued at lane 0 of the next pass when the window straddles)
#pragma unroll
    for (int p = 0; p < P; ++p) {
      const float next0 = __shfl_sync(0xffffffffu, sfx[p + 1 < P ? p + 1 : p], 0);
      if (kk[p] == 0) g1[p] -= sfx[p] + ((p + 1 < P && lane + n > 32) ? next0 : 0.f);
      const int64_t e = e0 + 32 * p;
      if (e < total) {
        g_obs[e] = g1[p];
        g_obs2[e] = wv[p];
        if (is_clip_out) is_clip_out[e] = cp[p];
        if (esl_out) esl_out[e] = es[p];
      }
    }
  }
  p0 = warp_sum(p0); p1 = warp_sum(p1); p2 = warp_sum(p2);
  if (lane == 0) { s_part[0][warp] = p0; s_part[1][warp] = p1; s_part[2][warp] = p2; }
  __syncthreads();
  if (threadIdx.x < 3) {
    double s = 0.0;
    for (int w = 0; w < WPB; ++w) s += (double)s_part[threadIdx.x][w];
    atomicAdd(&loss_parts[threadIdx.x], s);
  }
}

// Streaming form of the all-lanes-live kernel for tiles of P > 1 passes (n = 20: P = 5).  The version above keeps every
// pass's intermediates of a tile in registers until its last pass (128 registers at P = 5: 25 % occupancy, 0.59 of HBM against
// 0.75 for the single-pass window lengths).  Here a pass is finished as soon as it is computed: the only state carried from
// pass to pass is the running cumprod, the previous pass's (||o||^2, V) for window heads that lie one pass back, and ONE
// pending window head per lane -- the head of a window that continues into the next pass waits for that pass's lane-0 suffix
// sum before its gradient is written.  The loads of pass p + 1 are issued before pass p is computed.
template <int DT>
struct LyaRow {
  float ln, lo, v1, v2, a[DT], c[DT];
};

template <int DT>
__device__ __forceinline__ void lya_load(LyaRow<DT>& r, int64_t e, const float* __restrict__ obs, const float* __restrict__ obs2,
                                         const float* __restrict__ logp_new, const float* __restrict__ logp_old,
                                         const float* __restrict__ lya_obs, const float* __restrict__ lya_obs2) {
  r.ln = logp_new[e]; r.lo = logp_old[e]; r.v1 = lya_obs[e]; r.v2 = lya_obs2[e];
  const float* o = obs + e * DT;
  const float* q = obs2 + e * DT;
  if constexpr (DT % 4 == 0) {
#pragma unroll
    for (int d = 0; d < DT / 4; ++d) {
      const float4 x = reinterpret_cast<const float4*>(o)[d], y = reinterpret_cast<const float4*>(q)[d];
      r.a[4 * d] = x.x; r.a[4 * d + 1] = x.y; r.a[4 * d + 2] = x.z; r.a[4 * d + 3] = x.w;
      r.c[4 * d] = y.x; r.c[4 * d + 1] = y.y; r.c[4 * d + 2] = y.z; r.c[4 * d + 3] = y.w;
    }
  } else if constexpr (DT % 2 == 0) {
#pragma unroll
    for (int d = 0; d < DT / 2; ++d) {
      const float2 x = reinterpret_cast<const float2*>(o)[d], y = reinterpret_cast<const float2*>(q)[d];
      r.a[2 * d] = x.x; r.a[2 * d + 1] = x.y; r.c[2 * d] = y.x; r.c[2 * d + 1] = y.y;
    }
  } else {
#pragma unroll
    for (int d = 0; d < DT; ++d) { r.a[d] = o[d]; r.c[d] = q[d]; }
  }
}

template <int WPB, int P, int DT, int OCC>
__global__ void __launch_bounds__(WPB * 32, OCC)
lyapunov_risk_stream_kernel(int64_t B, int n, const float* __restrict__ obs, const float* __restrict__ obs2,
                            const float* __restrict__ logp_new, const float* __restrict__ logp_old,
                            const float* __restrict__ lya_obs, const float* __restrict__ lya_obs2,
                            const float* __restrict__ coef_son, const float* __restrict__ coef_diff,
                            const float* __restrict__ coef_sl, float alpha1, float alpha2, float diff_scale, float pos_scale,
                            double* __restrict__ loss_parts, float* __restrict__ g_obs, float* __restrict__ g_obs2,
                            float* __restrict__ is_clip_out, float* __restrict__ esl_out) {
  __shared__ float s_part[3][WPB];
  __shared__ float s_coef[3][32];
  if (threadIdx.x < 32) {
    const bool in = (int)threadIdx.x < n;
    s_coef[0][threadIdx.x] = in ? coef_son[threadIdx.x] : 0.f;
    s_coef[1][threadIdx.x] = in ? coef_diff[threadIdx.x] : 0.f;
    s_coef[2][threadIdx.x] = in ? coef_sl[threadIdx.x] : 0.f;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int T = 32 * P;
  const int64_t total = B * (int64_t)n;
  const float inv_bn = pos_scale / (float)((double)B * n);
  const float w_scale = diff_scale / (float)B;
  int kk[P];                                     // tile-relative step index of this lane's element in every pass
#pragma unroll
  for (int p = 0; p < P; ++p) kk[p] = (32 * p + lane) % n;
  float p0 = 0.f, p1 = 0.f, p2 = 0.f;
  const int64_t tiles = (total + T - 1) / T;
  for (int64_t tile = (int64_t)blockIdx.x * WPB + warp; tile < tiles; tile += (int64_t)gridDim.x * WPB) {
    const int64_t e0 = tile * T + lane;
    float carry = 1.f, prev_op = 0.f, prev_v1 = 0.f;
    float pend_g1 = 0.f, pend_sfx = 0.f;
    int64_t pend_e = -1;
    LyaRow<DT> cur, nxt;
    lya_load<DT>(cur, min(e0, total - 1), obs, obs2, logp_new, logp_old, lya_obs, lya_obs2);
#pragma unroll
    for (int p = 0; p < P; ++p) {
      const int64_t e = e0 + 32 * p;
      const bool live = e < total;
      if (p + 1 < P) lya_load<DT>(nxt, min(e + 32, total - 1), obs, obs2, logp_new, logp_old, lya_obs, lya_obs2);
      const int k = kk[p];
      const float son = s_coef[0][k], dif = s_coef[1][k], sl = s_coef[2][k];
      float op = 0.f, op2 = 0.f;
#pragma unroll
      for (int d = 0; d < DT; ++d) { op = __fmaf_rn(cur.a[d], cur.a[d], op); op2 = __fmaf_rn(cur.c[d], cur.c[d], op2); }
      float c = fminf(fmaxf(expf(cur.ln - cur.lo), 0.f), 1.f);     // clamp(ratio, 0, 1) :284-285
      float v1 = cur.v1, v2 = cur.v2;
      if (!live) { op = 0.f; op2 = 0.f; v1 = 0.f; v2 = 0.f; c = 1.f; }
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {                           // segmented inclusive cumprod (:286)
        const float y = __shfl_up_sync(0xffffffffu, c, o);
        if (lane >= o && k >= o) c *= y;
      }
      if (k > lane) c *= carry;                                    // the window began in the previous pass
      carry = __shfl_sync(0xffffffffu, c, 31);
      const int src = (lane - k) & 31;                             // lane of the window head, in this pass or the previous one
      float h_op = __shfl_sync(0xffffffffu, op, src), h_v1 = __shfl_sync(0xffffffffu, v1, src);
      if (p > 0) {
        const float q_op = __shfl_sync(0xffffffffu, prev_op, src), q_v1 = __shfl_sync(0xffffffffu, prev_v1, src);
        if (k > lane) { h_op = q_op; h_v1 = q_v1; }
      }
      const float lo = alpha1 * op - v1, up = v1 - alpha2 * op;                       // boundedness hinge :291-301
      const float start_norm = sqrtf(h_op);                                          // ||o_0|| :306-307
      const float esl = (start_norm * son - sqrtf(op2)) >= 0.f ? 1.f : -1.f;         // :308-312
      const float inner = esl * (v2 - h_v1 * sl);                                    // :318-323
      const float term = c * fmaxf(inner, 0.f);
      const float w = (live && inner > 0.f) ? dif * c * esl * w_scale : 0.f;
      float sx = w * sl;                                           // suffix sum of w * sl inside the window, within this pass
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const float y = __shfl_down_sync(0xffffffffu, sx, o);
        if (lane + o < 32 && k + o < n) sx += y;
      }
      // the pending head of the previous pass takes its window's continuation (this pass's lane-0 suffix)
      const float next0 = __shfl_sync(0xffffffffu, sx, 0);
      if (pend_e >= 0) { g_obs[pend_e] = pend_g1 - (pend_sfx + next0); pend_e = -1; }
      if (live) {
        p0 += fmaxf(lo, 0.f);
        p1 += fmaxf(up, 0.f);
        p2 += dif * term;
        float g1 = ((lo > 0.f) ? -inv_bn : 0.f) + ((up > 0.f) ? inv_bn : 0.f);
        const bool cont = k == 0 && p + 1 < P && lane + n > 32;    // a window head whose window continues in the next pass
        if (cont) { pend_g1 = g1; pend_sfx = sx; pend_e = e; }
        else { if (k == 0) g1 -= sx + 0.f; g_obs[e] = g1; }
        g_obs2[e] = w;
        if (is_clip_out) is_clip_out[e] = c;
        if (esl_out) esl_out[e] = esl;
      }
      prev_op = op; prev_v1 = v1;
      if (p + 1 < P) cur = nxt;
    }
  }
  p0 = warp_sum(p0); p1 = warp_sum(p1); p2 = warp_sum(p2);
  if (lane == 0) { s_part[0][warp] = p0; s_part[1][warp] = p1; s_part[2][warp] = p2; }
  __syncthreads();
  if (threadIdx.x < 3) {
    double s = 0.0;
    for (int w = 0; w < WPB; ++w) s += (double)s_part[threadIdx.x][w];
    atomicAdd(&loss_parts[threadIdx.x], s);
  }
}

// One THREAD per window (a window is only n floats: a warp per window spends an instruction per 80 bytes and is
// issue-bound at a fifth of the HBM peak).  A warp covers 32 consecutive windows = 32*n contiguous floats; each lane
// reads its own n floats as float4 vectors when n % 4 == 0 (every sector fetched is fully used by the warp).  The
// lambda-weighted sum runs in step order, the batch moments are reduced per warp and per block in float64.
template <int TPB>
__global__ void __launch_bounds__(TPB)
stability_adv_kernel(int64_t B, int n, const float* __restrict__ lya_obs0, const float* __restrict__ lya_obs2,
                     const float* __restrict__ coef_diff, const float* __restrict__ coef_sl, float* __restrict__ adv_raw,
                     double* __restrict__ moments) {
  __shared__ float s_dif[32], s_sl[32];
  __shared__ double s_m[2][TPB / 32];
  if (threadIdx.x < 32) {
    s_dif[threadIdx.x] = threadIdx.x < n ? coef_diff[threadIdx.x] : 0.f;
    s_sl[threadIdx.x] = threadIdx.x < n ? coef_sl[threadIdx.x] : 0.f;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool vec = (n & 3) == 0 && (reinterpret_cast<uintptr_t>(lya_obs2) & 15) == 0;
  double m1 = 0.0, m2 = 0.0;
  const int64_t stride = (int64_t)gridDim.x * TPB;
  for (int64_t b = (int64_t)blockIdx.x * TPB + threadIdx.x; b < B; b += stride) {
    const float v0 = lya_obs0[b];
    const float* row = lya_obs2 + b * n;
    float a = 0.f;
    if (vec) {
      for (int k = 0; k < n; k += 4) {
        const float4 v = *reinterpret_cast<const float4*>(row + k);
        a += s_dif[k] * (v0 * s_sl[k] - v.x);                 // msacl.py:395-399
        a += s_dif[k + 1] * (v0 * s_sl[k + 1] - v.y);
        a += s_dif[k + 2] * (v0 * s_sl[k + 2] - v.z);
        a += s_dif[k + 3] * (v0 * s_sl[k + 3] - v.w);
      }
    } else {
      for (int k = 0; k < n; ++k) a += s_dif[k] * (v0 * s_sl[k] - row[k]);
    }
    adv_raw[b] = a;
    m1 += (double)a;
    m2 += (double)a * (double)a;
  }
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    m1 += __shfl_xor_sync(0xffffffffu, m1, o);
    m2 += __shfl_xor_sync(0xffffffffu, m2, o);
  }
  if (lane == 0) { s_m[0][warp] = m1; s_m[1][warp] = m2; }
  __syncthreads();
  if (threadIdx.x < 2) {
    double s = 0.0;
    for (int w = 0; w < TPB / 32; ++w) s += s_m[threadIdx.x][w];
    atomicAdd(&moments[threadIdx.x], s);
  }
}

__global__ void __launch_bounds__(256)
adv_normalize_kernel(int64_t B, const float* __restrict__ adv_raw, const double* __restrict__ moments, float* __restrict__ adv) {
  const double mean = moments[0] / (double)B;
  const double var = (moments[1] - moments[0] * mean) / (double)(B - 1);     // unbiased, torch.std default
  const float fmean = (float)mean;
  const float denom = (float)sqrt(var > 0.0 ? var : 0.0) + 1e-8f;            // msacl.py:400
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < B; i += stride) adv[i] = (adv_raw[i] - fmean) / denom;
}

// Soft (Polyak) target update over a whole parameter list in ONE launch (RL/algorithm/msacl.py:445-460 does
// `p_targ.mul_(polyak); p_targ.add_((1 - polyak) * p)` per tensor: ~24 tiny launches per iteration).  blockIdx.y = tensor,
// grid-stride over its elements; the three float32 roundings of the reference expression are kept (no FMA).
__global__ void __launch_bounds__(256)
polyak_update_kernel(const float* const* __restrict__ src, float* const* __restrict__ dst, const int64_t* __restrict__ numel,
                     float polyak, float one_minus) {
  const int t = blockIdx.y;
  const float* __restrict__ s = src[t];
  float* __restrict__ d = dst[t];
  const int64_t n = numel[t];
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    d[i] = __fadd_rn(__fmul_rn(d[i], polyak), __fmul_rn(one_minus, s[i]));
}

// FP32 FFMA peak probes (roofline denominators for the fused rollout kernel).
//  mode 0: 8 independent accumulator chains per thread, multiplier/addend are compile-time
//          constants (ptxas emits the immediate form) -- the best case the FMA pipe can do.
//  mode 1: the register-tiled SGEMM inner product itself, without any memory traffic: 8x8
//          accumulators, acc[i][c] += a[i] * b[c] with all operands in registers (three-register
//          FFMA, operand-collector bound) -- the ceiling for any register-blocked FP32 GEMM.
__global__ void __launch_bounds__(256) ffma_probe_kernel(int iters, float* sink) {
  float a[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) a[j] = (float)(threadIdx.x + j) * 1e-3f;
  const float x = 1.0000001f, y = 1e-7f;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int u = 0; u < 16; ++u)
#pragma unroll
      for (int j = 0; j < 8; ++j) a[j] = __fmaf_rn(a[j], x, y);
  }
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) s += a[j];
  if (s == 123.456f) sink[0] = s;
}

__global__ void __launch_bounds__(256) ffma_probe_outer_kernel(int iters, const float* __restrict__ src, float* sink) {
  float a[8], b[8], acc[8][8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { a[j] = src[(threadIdx.x + j) & 63]; b[j] = src[(threadIdx.x * 3 + j) & 63]; }
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[i][c] = 0.f;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[i][c] = __fmaf_rn(a[i], b[c], acc[i][c]);
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int c = 0; c < 8; ++c) s += acc[i][c];
  if (s == 123.456f) sink[0] = s;
}

// mode 2: the same outer product with packed FFMA2 (fma.rn.f32x2, scalar-broadcast A operand)
__global__ void __launch_bounds__(256) ffma2_probe_outer_kernel(int iters, const float* __restrict__ src, float* sink) {
  typedef unsigned long long u64;
  float a[8];
  u64 b[4], acc[8][4];
#pragma unroll
  for (int j = 0; j < 8; ++j) a[j] = src[(threadIdx.x + j) & 63];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float lo = src[(threadIdx.x * 3 + 2 * j) & 63], hi = src[(threadIdx.x * 3 + 2 * j + 1) & 63];
    asm("mov.b64 %0, {%1, %2};" : "=l"(b[j]) : "f"(lo), "f"(hi));
  }
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[i][c] = 0ull;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        u64 aa;
        asm("mov.b64 %0, {%1, %1};" : "=l"(aa) : "f"(a[i]));
#pragma unroll
        for (int c = 0; c < 4; ++c) asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc[i][c]) : "l"(aa), "l"(b[c]));
      }
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      float lo, hi;
      asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(acc[i][c]));
      s += lo + hi;
    }
  if (s == 123.456f) sink[0] = s;
}

// mode 8: the mode-1 outer product with directed rounding, half FFMA.RM (__fmaf_rd) and half FFMA.RP (__fmaf_ru): the issue
// rate of the interval GEMMs of certify_region.cu
__global__ void __launch_bounds__(256) ffma_rmrp_probe_outer_kernel(int iters, const float* __restrict__ src, float* sink) {
  float a[8], b[8], acc[8][8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { a[j] = src[(threadIdx.x + j) & 63]; b[j] = src[(threadIdx.x * 3 + j) & 63]; }
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[i][c] = 0.f;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[i][c] = (i & 1) ? __fmaf_ru(a[i], b[c], acc[i][c]) : __fmaf_rd(a[i], b[c], acc[i][c]);
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int c = 0; c < 8; ++c) s += acc[i][c];
  if (s == 123.456f) sink[0] = s;
}

// mode 3: FP64 DFMA throughput (8 independent chains per thread)
__global__ void __launch_bounds__(256) dfma_probe_kernel(int iters, float* sink) {
  double a[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) a[j] = (double)(threadIdx.x + j) * 1e-3;
  const double x = (double)sink[64] * 1e-9 + 1.0, y = (double)sink[65] * 1e-9;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int j = 0; j < 8; ++j) a[j] = __fma_rn(a[j], x, y);
  }
  double s = 0.0;
#pragma unroll
  for (int j = 0; j < 8; ++j) s += a[j];
  if (s == 123.456) sink[0] = (float)s;
}

// modes 4-6: FP64 issue rate seen by ONE warp per SM sub-partition (the env phase of the fused rollout kernel: one env warp
// per sub-partition, separate DMUL / DADD because the dynamics round like NumPy): CH independent chains per thread of
// alternating DMUL, DADD.  4: CH = 8 (throughput of a lone warp), 5: CH = 2, 6: CH = 1 (dependent latency).
template <int CH>
__global__ void __launch_bounds__(128) dmul_dadd_probe_kernel(int iters, float* sink) {
  double a[CH];
#pragma unroll
  for (int j = 0; j < CH; ++j) a[j] = (double)(threadIdx.x + j) * 1e-3;
  const double x = (double)sink[64] * 1e-9 + 1.0, y = (double)sink[65] * 1e-9;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int u = 0; u < 32 / CH; ++u)
#pragma unroll
      for (int j = 0; j < CH; ++j) a[j] = __dadd_rn(__dmul_rn(a[j], x), y);
  }
  double s = 0.0;
#pragma unroll
  for (int j = 0; j < CH; ++j) s += a[j];
  if (s == 123.456) sink[0] = (float)s;
}

// mode 7: float32 <-> float64 round trips (F2F.F32.F64, F2F.F64.F32) plus one DMUL per round trip, 8 chains, one warp per
// sub-partition: the conversion cost of the reference's mixed-precision dtype flow
__global__ void __launch_bounds__(128) f2f_probe_kernel(int iters, float* sink) {
  double a[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) a[j] = (double)(threadIdx.x + j) * 1e-3 + 1.0;
  const double x = (double)sink[64] * 1e-9 + 1.0;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int j = 0; j < 8; ++j) a[j] = __dmul_rn((double)__double2float_rn(a[j]), x);
  }
  double s = 0.0;
#pragma unroll
  for (int j = 0; j < 8; ++j) s += a[j];
  if (s == 123.456) sink[0] = (float)s;
}

}  // namespace msacl

using namespace msacl;

static inline unsigned grid_for(int64_t work_items, int per_block) {
  const int64_t want = (work_items + per_block - 1) / per_block;
  const int64_t cap = (int64_t)kNumSMs * 8;
  return (unsigned)(want < cap ? (want > 0 ? want : 1) : cap);
}

extern "C" int msacl_q_backup(int64_t count, const float* rew, const float* done, const float* next_q1,
                              const float* next_q2, const float* next_logp, float gamma, float alpha, float* backup,
                              void* stream) {
  if (count <= 0 || !rew || !done || !next_q1 || !next_q2 || !next_logp || !backup) { set_error("q_backup: bad argument"); return MSACL_ERR_BAD_ARG; }
  q_backup_kernel<<<grid_for(count, 256), 256, 0, (cudaStream_t)stream>>>(count, rew, done, next_q1, next_q2, next_logp, gamma, alpha, backup);
  return check_launch("q_backup");
}

extern "C" int msacl_lyapunov_risk(int64_t B, int32_t n, int32_t D, const float* obs, const float* obs2,
                                   const float* logp_new, const float* logp_old, const float* lya_obs,
                                   const float* lya_obs2, const float* coef_son, const float* coef_diff,
                                   const float* coef_sl, float alpha1, float alpha2, float diff_scale, float pos_scale,
                                   double* loss_parts, float* grad_lya_obs, float* grad_lya_obs2, float* is_clip,
                                   float* esl, void* stream) {
  if (B <= 0 || n <= 0 || n > 32 || D <= 0 || !obs || !obs2 || !logp_new || !logp_old || !lya_obs || !lya_obs2 ||
      !coef_son || !coef_diff || !coef_sl || !loss_parts || !grad_lya_obs || !grad_lya_obs2) {
    set_error("lyapunov_risk: bad argument (n_step must be <= 32)");
    return MSACL_ERR_BAD_ARG;
  }
  cudaStream_t s = (cudaStream_t)stream;
  cudaMemsetAsync(loss_parts, 0, 3 * sizeof(double), s);
  constexpr int WPB = 8;
  // all-lanes-live kernel: tiles of 32 P elements hold whole windows when P = n / gcd(n, 32); instantiated for P = 1, 3, 5
  // (n = 32, 16, 8, 4, 2, 1 / 24, 12, 6, 3 / 20, 10, 5 -- the reference default is n = 20) and the six envs' obs_dim
  {
    int g = n, r = 32;
    while (r) { const int t = g % r; g = r; r = t; }
    const int P = n / g;
    const int64_t tiles = (B * (int64_t)n + 32 * P - 1) / (32 * P);
#define MSACL_LYA_STRIPED(P_, DT)                                                                                            \
    if (P == P_ && D == DT) {                                                                                                \
      if constexpr (P_ > 1) {      /* multi-pass tiles: the streaming kernel (n = 20: 0.62 of HBM against 0.51) */             \
        /* 64 registers (4 blocks per SM) for the narrow observations: n = 20, obs_dim 4 0.77 -> 0.86 of HBM */               \
        lyapunov_risk_stream_kernel<WPB, P_, DT, (DT <= 4 ? 4 : 3)><<<resident_grid(lyapunov_risk_stream_kernel<WPB, P_, DT, (DT <= 4 ? 4 : 3)>, WPB * 32, tiles, WPB), WPB * 32, 0, s>>>( \
                \
            B, n, obs, obs2, logp_new, logp_old, lya_obs, lya_obs2, coef_son, coef_diff, coef_sl, alpha1, alpha2, diff_scale, \
            pos_scale, loss_parts, grad_lya_obs, grad_lya_obs2, is_clip, esl);                                                \
      }                                                                                                                       \
      else     /* single-pass tiles (n = 32, 16, 8 ...): 0.86 of HBM as they are; the streaming kernel with 4-pass tiles measured 0.77 */ \
        lyapunov_risk_striped_kernel<WPB, P_, DT><<<resident_grid(lyapunov_risk_striped_kernel<WPB, P_, DT>, WPB * 32, tiles, WPB), WPB * 32, 0, s>>>( \
                                  \
            B, n, obs, obs2, logp_new, logp_old, lya_obs, lya_obs2, coef_son, coef_diff, coef_sl, alpha1, alpha2, diff_scale, \
            pos_scale, loss_parts, grad_lya_obs, grad_lya_obs2, is_clip, esl);                                                \
      return check_launch("lyapunov_risk");                                                                                   \
    }
#define MSACL_LYA_STRIPED_D(P_) MSACL_LYA_STRIPED(P_, 2) MSACL_LYA_STRIPED(P_, 4) MSACL_LYA_STRIPED(P_, 6) MSACL_LYA_STRIPED(P_, 7) MSACL_LYA_STRIPED(P_, 12)
    if (n > 1) { MSACL_LYA_STRIPED_D(1) MSACL_LYA_STRIPED_D(3) MSACL_LYA_STRIPED_D(5) }
#undef MSACL_LYA_STRIPED_D
#undef MSACL_LYA_STRIPED
  }
#define MSACL_LYA_LAUNCH(DT)                                                                                              \
  lyapunov_risk_kernel<WPB, DT><<<resident_grid(lyapunov_risk_kernel<WPB, DT>, WPB * 32, B, WPB), WPB * 32, 0, s>>>(B, n, D, obs, obs2, logp_new, logp_old, lya_obs,    \
                                                                      lya_obs2, coef_son, coef_diff, coef_sl, alpha1, alpha2, \
                                                                      diff_scale, pos_scale, loss_parts, grad_lya_obs,       \
                                                                      grad_lya_obs2, is_clip, esl)
  switch (D) {           // obs_dim of the six reference envs; anything else takes the run-time-D instantiation
    case 2: MSACL_LYA_LAUNCH(2); break;
    case 4: MSACL_LYA_LAUNCH(4); break;
    case 6: MSACL_LYA_LAUNCH(6); break;
    case 7: MSACL_LYA_LAUNCH(7); break;
    case 12: MSACL_LYA_LAUNCH(12); break;
    default: MSACL_LYA_LAUNCH(0); break;
  }
#undef MSACL_LYA_LAUNCH
  return check_launch("lyapunov_risk");
}

extern "C" int msacl_stability_advantage(int64_t B, int32_t n, const float* lya_obs0, const float* lya_obs2,
                                         const float* coef_diff, const float* coef_sl, float* adv_raw, double* moments,
                                         void* stream) {
  if (B <= 0 || n <= 0 || n > 32 || !lya_obs0 || !lya_obs2 || !coef_diff || !coef_sl || !adv_raw || !moments) {
    set_error("stability_advantage: bad argument");
    return MSACL_ERR_BAD_ARG;
  }
  cudaStream_t s = (cudaStream_t)stream;
  cudaMemsetAsync(moments, 0, 2 * sizeof(double), s);
  constexpr int TPB = 128;
  stability_adv_kernel<TPB><<<grid_for(B, TPB), TPB, 0, s>>>(       /* (whole resident waves measured slower here: 24.9 vs 22.2 us) */
      B, n, lya_obs0, lya_obs2, coef_diff, coef_sl, adv_raw, moments);
  return check_launch("stability_advantage");
}

extern "C" int msacl_advantage_normalize(int64_t B, const float* adv_raw, const double* moments, float* adv, void* stream) {
  if (B <= 1 || !adv_raw || !moments || !adv) { set_error("advantage_normalize: bad argument"); return MSACL_ERR_BAD_ARG; }
  adv_normalize_kernel<<<grid_for(B, 256), 256, 0, (cudaStream_t)stream>>>(B, adv_raw, moments, adv);
  return check_launch("advantage_normalize");
}

extern "C" int msacl_polyak_update(int32_t count, const float* const* src, float* const* dst, const int64_t* numel,
                                   int64_t max_numel, float polyak, float one_minus, void* stream) {
  if (count <= 0 || count > 65535 || !src || !dst || !numel || max_numel <= 0) { set_error("polyak_update: bad argument"); return MSACL_ERR_BAD_ARG; }
  const int64_t want = (max_numel + 255) / 256;
  const dim3 grid((unsigned)(want < 64 ? want : 64), (unsigned)count);
  polyak_update_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, dst, numel, polyak, one_minus);
  return check_launch("polyak_update");
}

extern "C" int msacl_ffma_probe(int32_t mode, int32_t iters, float* sink, double* flops, void* stream) {
  if (iters <= 0 || !sink || mode < 0 || mode > 8) { set_error("ffma_probe: bad argument"); return MSACL_ERR_BAD_ARG; }
  if (mode == 8) {
    const unsigned grid = 2 * kNumSMs * 4;
    ffma_rmrp_probe_outer_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(iters, sink + 64, sink);
    if (flops) *flops = 2.0 * 128.0 * (double)iters * 256.0 * (double)grid;
    return check_launch("ffma_probe");
  }
  if (mode >= 4) {          // one warp per sub-partition: 148 blocks x 128 threads; *flops = FP64 instructions per warp
    if (mode == 4) dmul_dadd_probe_kernel<8><<<kNumSMs, 128, 0, (cudaStream_t)stream>>>(iters, sink);
    else if (mode == 5) dmul_dadd_probe_kernel<2><<<kNumSMs, 128, 0, (cudaStream_t)stream>>>(iters, sink);
    else if (mode == 6) dmul_dadd_probe_kernel<1><<<kNumSMs, 128, 0, (cudaStream_t)stream>>>(iters, sink);
    else f2f_probe_kernel<<<kNumSMs, 128, 0, (cudaStream_t)stream>>>(iters, sink);
    if (flops) *flops = (mode == 7 ? 32.0 : 64.0) * (double)iters;     // mode 7: round trips (2 conversions + 1 DMUL each)
    return check_launch("ffma_probe");
  }
  const unsigned grid = 2 * kNumSMs * 4;
  if (mode == 0) {
    ffma_probe_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(iters, sink);
    if (flops) *flops = 2.0 * 8.0 * 16.0 * (double)iters * 256.0 * (double)grid;
  } else if (mode == 1) {
    ffma_probe_outer_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(iters, sink + 64, sink);   // sink[64..128) = operand source
    if (flops) *flops = 2.0 * 128.0 * (double)iters * 256.0 * (double)grid;
  } else if (mode == 2) {
    ffma2_probe_outer_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(iters, sink + 64, sink);
    if (flops) *flops = 2.0 * 128.0 * (double)iters * 256.0 * (double)grid;
  } else {
    dfma_probe_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(iters, sink);
    if (flops) *flops = 2.0 * 32.0 * (double)iters * 256.0 * (double)grid;
  }
  return check_launch("ffma_probe");
}
