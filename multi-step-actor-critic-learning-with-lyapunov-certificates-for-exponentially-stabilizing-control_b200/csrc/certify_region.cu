// Region verifier of the Lyapunov certificate: interval branch-and-bound over state boxes (include/msacl_b200.h,
// "Region verifier").  No counterpart in the reference.
//
// region_eval_kernel encloses, for a batch of boxes C, V(C), the m-step closed-loop image F^m(C) and V(F^m(C)) in
// outward-rounded interval arithmetic.  Its cost is the 256x256 layers: per cell the V net's two 256-wide layers twice (at C
// and at F^m(C)) and the policy's 256x256 layer m times, 4 FMAs per weight (lo = W+ l + W- u rounded down, hi = W+ u + W- l
// rounded up, __fmaf_rd / __fmaf_ru = FFMA.RM / FFMA.RP).  Structure as rollout_fused_kernel: one persistent CTA of 8 warps
// per SM; a warp owns 4 cells of the 32-cell tile for the whole pipeline (register tile 4 cells x 8 units, two bounds each),
// so the MLP needs no block barrier; the pre-split [k][W+ | W-] rows of the 256-wide matrices (2 KB per k, resident in L2)
// stream through a 4-stage TMA bulk-copy ring in the same order for every tile.  The small layers, the heads and the env
// step (IEnv<ID>, one lane per cell) run on the same warps.  Tensor cores are not used: the rounding of tcgen05 FP32
// accumulation is not specified, so no outward bound exists for it.
//
// The bounded disturbances of p.dist widen one closed-loop step by three boxes: N (sensor noise) the policy's layer-1 input,
// which the owner lanes write to sm.pl / sm.pu from the state box, so V and the env step keep reading the un-widened state;
// U the clipped action; W the state after IEnv<ID>::step.  A set that is exactly {0} is skipped by a uniform flag rather than
// added as [0, 0] (-0 + 0 rounded up is +0), so an all-zero p.dist runs the nominal closed loop bit for bit.
//
// The branch-and-bound round (msacl_region_round) is count / scan / scatter in the style of windows.cu: cells are dyadic
// ([depth, idx per dimension], depth t bisects dimension t mod D -- the widest one scaled by the box width, lowest index on
// ties), so the tree and every statistic are independent of the chunking; volumes are integers in units of 2^-50.
#include <cmath>

#include "common.cuh"
#include "interval_env.cuh"
#include "tcgen05.cuh"

namespace msacl {

constexpr int RH = MSACL_REGION_HIDDEN;
constexpr int RWARPS = 8;
constexpr int RT = RWARPS * 32;
constexpr int RC = 4;                  // cells per warp
constexpr int RTM = RWARPS * RC;       // cells per tile
constexpr int RKC = 8;                 // k rows per TMA chunk
constexpr int RNCH = RH / RKC;
constexpr int RSTAGE = 4;
constexpr int RPRE = RSTAGE - 2;
constexpr int RROW = 2 * RH;           // [W+ | W-] floats per k
constexpr uint32_t RCHUNK_BYTES = RKC * RROW * 4;
constexpr int RD = 8;                  // padded obs dim of the W1 images
constexpr int RB = 256;                // threads of the bookkeeping kernels

// image layout (floats); every section starts 16-byte aligned
constexpr int64_t kMat = (int64_t)RH * RROW;
constexpr int64_t P_W1 = 0, P_B1 = P_W1 + RH * RD, P_W2 = P_B1 + RH, P_B2 = P_W2 + kMat, P_W3 = P_B2 + RH, P_B3 = P_W3 + 2 * RH;
constexpr int64_t V_W1 = P_B3 + 4, V_B1 = V_W1 + RH * RD, V_W2 = V_B1 + RH, V_B2 = V_W2 + kMat, V_W3 = V_B2 + RH,
                  V_B3 = V_W3 + kMat, IMG_FLOATS = V_B3 + RH;
static_assert(P_W2 % 4 == 0 && V_W2 % 4 == 0 && V_W3 % 4 == 0, "TMA sources must be 16-byte aligned");

constexpr uint32_t kKeyPosInf = 0xFF800000u, kKeyNegInf = 0x007FFFFFu;
__device__ __forceinline__ uint32_t okey(float f) {
  const uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

struct RSmem {
  float wc[RSTAGE][RKC * RROW];        // W chunk ring
  float hl[RH * RTM], hu[RH * RTM];    // layer inputs [k][cell], lower / upper
  float xl[RTM][RD], xu[RTM][RD];      // state box
  float pl[RTM][RD], pu[RTM][RD];      // policy input box x + N (sensor noise only)
  unsigned long long full_bar[RSTAGE], empty_bar[RSTAGE];
};

// per disturbance set of p.dist, whether it is not exactly {0} (set on the host, uniform in the kernel)
struct RDist {
  int obs, act, state;
};
// region_eval_kernel's parameters as one by-value argument: the flags are then loaded where they are used, whereas a small
// argument of their own is held in registers over the whole kernel (VanderPol: 168 instead of 155)
struct REval {
  msacl_region_params_t p;
  RDist on;
};

// ----------------------------------------------------------------------------------------------------------------------
__global__ void region_pack_kernel(msacl_region_nets_t s, float* img) {
  const int64_t total = IMG_FLOATS;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    float v = 0.f;
    auto w1 = [&](const float* w, int h, int64_t off) {           // [n][d] padded
      const int n = (int)(off / RD), d = (int)(off % RD);
      return (n < h && d < s.obs_dim) ? w[n * s.obs_dim + d] : 0.f;
    };
    auto vec = [&](const float* b, int h, int64_t off) { return off < h ? b[off] : 0.f; };
    auto split = [&](const float* w, int hout, int hin, int64_t off) {   // row k: [W+(n, k) | W-(n, k)], W [hout][hin]
      const int k = (int)(off / RROW), c = (int)(off % RROW), n = c % RH;
      if (n >= hout || k >= hin) return 0.f;
      const float x = w[(int64_t)n * hin + k];
      return c < RH ? fmaxf(x, 0.f) : fminf(x, 0.f);
    };
    if (e < P_B1) v = w1(s.p_w1, s.p_h1, e - P_W1);
    else if (e < P_W2) v = vec(s.p_b1, s.p_h1, e - P_B1);
    else if (e < P_B2) v = split(s.p_w2, s.p_h2, s.p_h1, e - P_W2);
    else if (e < P_W3) v = vec(s.p_b2, s.p_h2, e - P_B2);
    else if (e < P_B3) {                                           // the mean rows only
      const int64_t o = e - P_W3;
      const int j = (int)(o / RH), k = (int)(o % RH);
      v = (j < s.act_dim && k < s.p_h2) ? s.p_w3[j * s.p_h2 + k] : 0.f;
    } else if (e < V_W1) v = vec(s.p_b3, s.act_dim, e - P_B3);
    else if (e < V_B1) v = w1(s.v_w1, s.v_h1, e - V_W1);
    else if (e < V_W2) v = vec(s.v_b1, s.v_h1, e - V_B1);
    else if (e < V_B2) v = split(s.v_w2, s.v_h2, s.v_h1, e - V_W2);
    else if (e < V_W3) v = vec(s.v_b2, s.v_h2, e - V_B2);
    else if (e < V_B3) v = split(s.v_w3, s.v_out, s.v_h2, e - V_W3);
    else v = vec(s.v_b3, s.v_out, e - V_B3);
    img[e] = v;
  }
}

// ----------------------------------------------------------------------------------------------------------------------
template <int ID, int VT>
__global__ void __launch_bounds__(RT, 1)
region_eval_kernel(REval args, const float* __restrict__ img, int64_t n_host, const int64_t* n_dev,
                   const float* __restrict__ in_lo, const float* __restrict__ in_hi, msacl_region_out_t out) {
  using E = Env<ID>;
  constexpr int D = E::D, A = E::A;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  RSmem& sm = *reinterpret_cast<RSmem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, m0 = warp * RC;
  const int64_t n = n_dev ? *n_dev : n_host;
  const int64_t tiles = (n + RTM - 1) / RTM;
  const msacl_region_params_t& p = args.p;
  const RDist& on = args.on;
  const int m = p.steps;
  if (tid == 0) {
#pragma unroll
    for (int i = 0; i < RSTAGE; ++i) { tc::mbar_init(&sm.full_bar[i], 1); tc::mbar_init(&sm.empty_bar[i], RWARPS); }
    tc::mbar_fence_init();
    tc::fence_async_smem();
  }
  __syncthreads();
  const int64_t my_tiles = tiles > blockIdx.x ? (tiles - 1 - blockIdx.x) / gridDim.x + 1 : 0;
  const int per_tile = (m + 4) * RNCH;   // matrices per tile: V2 V3 | P2 x m | V2 V3
  const int64_t total = my_tiles * per_tile;
  const bool producer = tid == 0;
  auto produce = [&](int64_t gi) {
    if (gi >= total) return;
    const int stg = (int)(gi % RSTAGE);
    if (gi >= RSTAGE) tc::mbar_wait(&sm.empty_bar[stg], (uint32_t)(((gi / RSTAGE) & 1) ^ 1));
    const int pos = (int)(gi % per_tile), seg = pos / RNCH, ch = pos % RNCH;
    const int64_t base = (seg == 0 || seg == m + 2) ? V_W2 : (seg == 1 || seg == m + 3) ? V_W3 : P_W2;
    tc::mbar_expect_tx(&sm.full_bar[stg], RCHUNK_BYTES);
    tc::tma_bulk_g2s(sm.wc[stg], img + base + (int64_t)ch * RKC * RROW, RCHUNK_BYTES, &sm.full_bar[stg]);
  };
  if (producer) {
#pragma unroll
    for (int i = 0; i < RPRE; ++i) produce(i);
  }
  int64_t g = 0;
  auto unit = [&](int c) { return c < 4 ? lane * 4 + c : 128 + lane * 4 + (c - 4); };

  float al[RC][8], ah[RC][8];
  // layer 1 from an input box in smem (bl / bu): sign-selected interval products, bias first
  auto layer1 = [&](int64_t w1, int64_t b1, const float (*bl)[RD], const float (*bu)[RD]) {
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const float b = __ldg(img + b1 + unit(c));
#pragma unroll
      for (int i = 0; i < RC; ++i) { al[i][c] = b; ah[i][c] = b; }
    }
#pragma unroll
    for (int d = 0; d < D; ++d) {
      float xl[RC], xu[RC];
#pragma unroll
      for (int i = 0; i < RC; ++i) { xl[i] = bl[m0 + i][d]; xu[i] = bu[m0 + i][d]; }
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const float w = __ldg(img + w1 + unit(c) * RD + d);
        const bool pos = w >= 0.f;
#pragma unroll
        for (int i = 0; i < RC; ++i) {
          al[i][c] = __fmaf_rd(w, pos ? xl[i] : xu[i], al[i][c]);
          ah[i][c] = __fmaf_ru(w, pos ? xu[i] : xl[i], ah[i][c]);
        }
      }
    }
  };
  // activation, then the layer input of the next GEMM into smem (read back by this warp only)
  auto act_store = [&](bool tanh_act) {
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      float l[RC], u[RC];
#pragma unroll
      for (int i = 0; i < RC; ++i) {
        if (tanh_act) {
          const If t = itanh(If{al[i][c], ah[i][c]});
          l[i] = t.l; u[i] = t.u;
        } else {
          l[i] = fmaxf(al[i][c], 0.f);
          u[i] = isnan(ah[i][c]) ? INFINITY : fmaxf(ah[i][c], 0.f);
        }
      }
      const int k = unit(c);
      *reinterpret_cast<float4*>(&sm.hl[k * RTM + m0]) = make_float4(l[0], l[1], l[2], l[3]);
      *reinterpret_cast<float4*>(&sm.hu[k * RTM + m0]) = make_float4(u[0], u[1], u[2], u[3]);
    }
    __syncwarp();
  };
  // 256x256 interval GEMM over the next RNCH ring chunks, accumulators start at the bias
  auto gemm = [&](int64_t bias) {
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const float b = __ldg(img + bias + unit(c));
#pragma unroll
      for (int i = 0; i < RC; ++i) { al[i][c] = b; ah[i][c] = b; }
    }
    for (int ch = 0; ch < RNCH; ++ch, ++g) {
      if (producer) produce(g + RPRE);
      const int stg = (int)(g % RSTAGE);
      tc::mbar_wait(&sm.full_bar[stg], (uint32_t)((g / RSTAGE) & 1));
      const float* wb = sm.wc[stg] + lane * 4;
#pragma unroll 2
      for (int kk = 0; kk < RKC; ++kk) {
        const int k = ch * RKC + kk;
        const float4 xa = *reinterpret_cast<const float4*>(&sm.hl[k * RTM + m0]);
        const float4 xb = *reinterpret_cast<const float4*>(&sm.hu[k * RTM + m0]);
        const float4 p0 = *reinterpret_cast<const float4*>(wb + kk * RROW);
        const float4 p1 = *reinterpret_cast<const float4*>(wb + kk * RROW + 128);
        const float4 q0 = *reinterpret_cast<const float4*>(wb + kk * RROW + RH);
        const float4 q1 = *reinterpret_cast<const float4*>(wb + kk * RROW + RH + 128);
        const float xl[RC] = {xa.x, xa.y, xa.z, xa.w}, xu[RC] = {xb.x, xb.y, xb.z, xb.w};
        const float wp[8] = {p0.x, p0.y, p0.z, p0.w, p1.x, p1.y, p1.z, p1.w};
        const float wn[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
#pragma unroll
        for (int i = 0; i < RC; ++i)
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            al[i][c] = __fmaf_rd(wn[c], xu[i], __fmaf_rd(wp[c], xl[i], al[i][c]));
            ah[i][c] = __fmaf_ru(wn[c], xl[i], __fmaf_ru(wp[c], xu[i], ah[i][c]));
          }
      }
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&sm.empty_bar[stg]);
    }
  };
  auto reduce_rd = [&](float v) {
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) v = __fadd_rd(v, __shfl_xor_sync(0xffffffffu, v, o));
    return __shfl_sync(0xffffffffu, v, 0);
  };
  auto reduce_ru = [&](float v) {
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) v = __fadd_ru(v, __shfl_xor_sync(0xffffffffu, v, o));
    return __shfl_sync(0xffffffffu, v, 0);
  };
  // V of the state boxes of this warp's cells: [vl, vu] (warp-uniform)
  auto vnet = [&](float (&vl)[RC], float (&vu)[RC]) {
    layer1(V_W1, V_B1, sm.xl, sm.xu);
    act_store(VT == 1);
    gemm(V_B2);
    act_store(VT == 1);
    gemm(V_B3);
#pragma unroll
    for (int i = 0; i < RC; ++i) {
      float sl = 0.f, su = 0.f;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const If z = isq(sane(If{al[i][c], ah[i][c]}));
        sl = __fadd_rd(sl, z.l);
        su = __fadd_ru(su, z.u);
      }
      vl[i] = reduce_rd(sl);
      vu[i] = reduce_ru(su);
    }
  };

  const int TR = 4 * A + 2 * D;
  for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const int64_t cell = tile * RTM + m0 + lane;          // valid for lane < RC
    const bool owner = lane < RC && cell < n;
    if (lane < RC) {
#pragma unroll
      for (int d = 0; d < D; ++d) {
        sm.xl[m0 + lane][d] = owner ? in_lo[cell * D + d] : 0.f;
        sm.xu[m0 + lane][d] = owner ? in_hi[cell * D + d] : 0.f;
      }
    }
    __syncwarp();
    float v_l[RC], v_u[RC];
    vnet(v_l, v_u);
    uint32_t flags = 0;
    float esc_margin = 0.f;
    for (int j = 1; j <= m; ++j) {
      if (on.obs) {
        if (lane < RC) {
#pragma unroll
          for (int d = 0; d < D; ++d) {
            sm.pl[m0 + lane][d] = __fadd_rd(sm.xl[m0 + lane][d], p.dist.obs_lo[d]);
            sm.pu[m0 + lane][d] = __fadd_ru(sm.xu[m0 + lane][d], p.dist.obs_hi[d]);
          }
        }
        __syncwarp();
      }
      layer1(P_W1, P_B1, on.obs ? sm.pl : sm.xl, on.obs ? sm.pu : sm.xu);
      act_store(false);
      gemm(P_B2);
      // ReLU, then the mean rows of the output layer (sign-selected) on the register tile
      float ml[RC][A], mu[RC][A];
#pragma unroll
      for (int q = 0; q < A; ++q) {
        float w3[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) w3[c] = __ldg(img + P_W3 + q * RH + unit(c));
        const float b3 = __ldg(img + P_B3 + q);
#pragma unroll
        for (int i = 0; i < RC; ++i) {
          float sl = 0.f, su = 0.f;
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            const float hl = fmaxf(al[i][c], 0.f), hu = isnan(ah[i][c]) ? INFINITY : fmaxf(ah[i][c], 0.f);
            const bool pos = w3[c] >= 0.f;
            sl = __fmaf_rd(w3[c], pos ? hl : hu, sl);
            su = __fmaf_ru(w3[c], pos ? hu : hl, su);
          }
          ml[i][q] = __fadd_rd(reduce_rd(sl), b3);
          mu[i][q] = __fadd_ru(reduce_ru(su), b3);
        }
      }
      if (lane < RC) {
        If mean[A], act[A], x[D];
#pragma unroll
        for (int q = 0; q < A; ++q) {
          float a = ml[0][q], b = mu[0][q];
#pragma unroll
          for (int i = 1; i < RC; ++i)
            if (lane == i) { a = ml[i][q]; b = mu[i][q]; }
          mean[q] = sane(If{a, b});
          const float half = (E::act_high(q) - E::act_low(q)) / 2.0f, mid = (E::act_high(q) + E::act_low(q)) / 2.0f;
          const If t = itanh(mean[q]);
          act[q] = {fminf(fmaxf(__fmaf_rd(half, t.l, mid), E::act_low(q)), E::act_high(q)),
                    fminf(fmaxf(__fmaf_ru(half, t.u, mid), E::act_low(q)), E::act_high(q))};
          if (on.act) act[q] = iadd(act[q], If{p.dist.act_lo[q], p.dist.act_hi[q]});   // after the clip, not re-clipped
        }
#pragma unroll
        for (int d = 0; d < D; ++d) x[d] = If{sm.xl[m0 + lane][d], sm.xu[m0 + lane][d]};
        IEnv<ID>::step(x, act);
#pragma unroll
        for (int d = 0; d < D; ++d) {
          if (on.state) x[d] = iadd(x[d], If{p.dist.state_lo[d], p.dist.state_hi[d]});
          if (!(x[d].l > E::obs_low(d) && x[d].u < E::obs_high(d))) flags |= MSACL_REGION_ESCAPED;
          const float out_by = fmaxf(__fsub_rd(x[d].l, E::obs_high(d)), __fsub_rd(E::obs_low(d), x[d].u));
          if (out_by > 0.f) { flags |= MSACL_REGION_REFUTE_ESCAPED; esc_margin = fmaxf(esc_margin, out_by); }
          sm.xl[m0 + lane][d] = x[d].l;
          sm.xu[m0 + lane][d] = x[d].u;
        }
        if (out.trace && owner) {
          float* tr = out.trace + (cell * m + (j - 1)) * TR;
#pragma unroll
          for (int q = 0; q < A; ++q) { tr[q] = mean[q].l; tr[A + q] = mean[q].u; tr[2 * A + q] = act[q].l; tr[3 * A + q] = act[q].u; }
#pragma unroll
          for (int d = 0; d < D; ++d) { tr[4 * A + d] = x[d].l; tr[4 * A + D + d] = x[d].u; }
        }
      }
      __syncwarp();
    }
    float w_l[RC], w_u[RC];
    vnet(w_l, w_u);
    if (owner) {
      float vl = v_l[0], vu = v_u[0], wl = w_l[0], wu = w_u[0];
#pragma unroll
      for (int i = 1; i < RC; ++i)
        if (lane == i) { vl = v_l[i]; vu = v_u[i]; wl = w_l[i]; wu = w_u[i]; }
      bool fin = isfinite(vl) && isfinite(vu) && isfinite(wl) && isfinite(wu);
      double sl = 0.0, su = 0.0;                            // inf / sup |x|^2 over the cell
      for (int d = 0; d < D; ++d) {
        const If b = {in_lo[cell * D + d], in_hi[cell * D + d]};
        const double l = b.l, u = b.u;
        const double ql = (l > 0.0) ? l * l : (u < 0.0 ? u * u : 0.0), qu = fmax(l * l, u * u);   // float^2: exact
        sl = __dadd_rd(sl, ql);
        su = __dadd_ru(su, qu);
        const float il = sm.xl[m0 + lane][d], iu = sm.xu[m0 + lane][d];
        fin = fin && isfinite(il) && isfinite(iu);
        if (!(il >= p.x0_lo[d] && iu <= p.x0_hi[d])) flags |= MSACL_REGION_LEAVES;
        out.img_lo[cell * D + d] = il;
        out.img_hi[cell * D + d] = iu;
      }
      if (!fin) flags |= MSACL_REGION_NONFINITE;
      if (!((double)wu <= __dmul_rd(p.decay_lo, (double)vl))) flags |= MSACL_REGION_DECREASE;
      if (!(__dmul_ru(p.alpha1, su) <= (double)vl && (double)vu <= __dmul_rd(p.alpha2, sl))) flags |= MSACL_REGION_BOUND;
      const double dec_margin = __dsub_rd((double)wl, __dmul_ru(p.decay_hi, (double)vu));
      float margin = 0.f;
      if (fin && dec_margin > 0.0) { flags |= MSACL_REGION_REFUTE_DECREASE; margin = __double2float_rd(dec_margin); }
      else if (flags & MSACL_REGION_REFUTE_ESCAPED) margin = esc_margin;
      if (!fin) flags &= ~(uint32_t)(MSACL_REGION_REFUTE_DECREASE | MSACL_REGION_REFUTE_ESCAPED);
      out.v_lo[cell] = vl; out.v_hi[cell] = vu; out.vm_lo[cell] = wl; out.vm_hi[cell] = wu;
      out.flags[cell] = (uint8_t)flags;
      out.margin[cell] = (flags & (MSACL_REGION_REFUTE_DECREASE | MSACL_REGION_REFUTE_ESCAPED)) ? margin : 0.f;
    }
    __syncwarp();
  }
}

// ----------------------------------------------------------------------------------------------------------------------
// branch and bound
__device__ __forceinline__ int cell_level(uint32_t depth, int d, int D) { return (int)((depth + D - 1 - d) / D); }

// outward box of the dyadic cell (lo rounded down, hi up) and the float centre; `centre_ok`: the centre provably lies in the
// closed cell
__device__ void cell_box(const uint32_t* c, int D, const msacl_region_params_t& p, float* lo, float* hi, float* ctr, bool& centre_ok) {
  centre_ok = true;
  for (int d = 0; d < D; ++d) {
    const double scale = ldexp(1.0, -cell_level(c[0], d, D));
    const double t0 = (double)c[1 + d] * scale, t1 = (double)(c[1 + d] + 1) * scale, tc = ((double)c[1 + d] + 0.5) * scale;
    const double x0 = p.x0_lo[d], wl = __dsub_rd((double)p.x0_hi[d], x0), wu = __dsub_ru((double)p.x0_hi[d], x0);
    lo[d] = __double2float_rd(__dadd_rd(x0, __dmul_rd(wl, t0)));
    hi[d] = __double2float_ru(__dadd_ru(x0, __dmul_ru(wu, t1)));
    ctr[d] = __double2float_rn(x0 + 0.5 * (wl + wu) * tc);
    const double in_lo = __dadd_ru(x0, __dmul_ru(wu, t0)), in_hi = __dadd_rd(x0, __dmul_rd(wl, t1));
    centre_ok = centre_ok && (double)ctr[d] >= in_lo && (double)ctr[d] <= in_hi;
  }
}

__device__ __forceinline__ bool cell_inner(const uint32_t* c, int D, const msacl_region_bnb_t& b) {
  bool in = true;
  for (int d = 0; d < D; ++d) {
    const int l = cell_level(c[0], d, D);
    const uint64_t i = c[1 + d];
    in = in && (i << b.inner_level) >= ((uint64_t)b.inner_lo[d] << l) && ((i + 1) << b.inner_level) <= ((uint64_t)b.inner_hi[d] << l);
  }
  return in;
}

__global__ void __launch_bounds__(RB) region_cells_kernel(msacl_region_params_t p, int D, const uint32_t* __restrict__ stack,
                                                          int64_t k, msacl_region_ws_t ws) {
  const int64_t i = (int64_t)blockIdx.x * RB + threadIdx.x;
  if (i >= k) return;
  const int W = 1 + D;
  uint32_t c[1 + 16];
  for (int j = 0; j < W; ++j) { c[j] = stack[i * W + j]; ws.cells[i * W + j] = c[j]; }
  float lo[16], hi[16], ctr[16];
  bool ok;
  cell_box(c, D, p, lo, hi, ctr, ok);
  for (int d = 0; d < D; ++d) { ws.lo[i * D + d] = lo[d]; ws.hi[i * D + d] = hi[d]; }
}

// block-wide exclusive scan of v (RB threads); returns the prefix, *tot = block total
__device__ __forceinline__ int64_t block_scan(int64_t v, int64_t* tot) {
  __shared__ int64_t ws_[RB / 32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int64_t x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int64_t y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) ws_[w] = x;
  __syncthreads();
  int64_t base = 0, t = 0;
  for (int j = 0; j < RB / 32; ++j) { if (j < w) base += ws_[j]; t += ws_[j]; }
  __syncthreads();
  *tot = t;
  return base + x - v;
}

__device__ __forceinline__ bool verified(uint32_t f) {
  return (f & (MSACL_REGION_NONFINITE | MSACL_REGION_DECREASE | MSACL_REGION_ESCAPED)) == 0;
}

// probe candidates: failing cells outside B whose centre is inside the cell and provably outside the snapped B
__device__ bool probe_cell(const msacl_region_params_t& p, const msacl_region_bnb_t& b, int D, const uint32_t* c, uint32_t f,
                           float* ctr) {
  if (verified(f) || cell_inner(c, D, b)) return false;
  float lo[16], hi[16];
  bool ok;
  cell_box(c, D, p, lo, hi, ctr, ok);
  bool outside_b = false;
  for (int d = 0; d < D; ++d) outside_b = outside_b || (double)ctr[d] < b.inner_box_lo[d] || (double)ctr[d] > b.inner_box_hi[d];
  return ok && outside_b;
}

__global__ void __launch_bounds__(RB) region_probe_kernel(msacl_region_params_t p, msacl_region_bnb_t b, int D, int64_t k,
                                                          msacl_region_ws_t ws, int scatter) {
  const int64_t i = (int64_t)blockIdx.x * RB + threadIdx.x;
  float ctr[16];
  const bool pr = i < k && probe_cell(p, b, D, ws.cells + i * (1 + D), ws.res.flags[i], ctr);
  int64_t tot;
  const int64_t off = block_scan(pr ? 1 : 0, &tot);
  if (!scatter) {
    if (threadIdx.x == 0) ws.scan[blockIdx.x] = tot;
    return;
  }
  if (i >= k) return;
  const int64_t slot = ws.scan[blockIdx.x] + off;
  ws.probe[i] = pr ? (int32_t)slot : -1;
  if (pr)
    for (int d = 0; d < D; ++d) { ws.plo[slot * D + d] = ctr[d]; ws.phi[slot * D + d] = ctr[d]; }
}

// exclusive scan of a[0, nb) in place (one block); *total = sum
__global__ void region_scan_kernel(int64_t* a, int64_t nb, int64_t* total) {
  __shared__ int64_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int64_t base = 0; base < nb; base += RB) {
    const int64_t i = base + threadIdx.x;
    const int64_t v = i < nb ? a[i] : 0;
    int64_t tot;
    const int64_t off = block_scan(v, &tot);
    if (i < nb) a[i] = carry + off;
    __syncthreads();
    if (threadIdx.x == 0) carry += tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) *total = carry;
}

__device__ __forceinline__ uint32_t cell_status(const msacl_region_bnb_t& b, int D, const uint32_t* c, uint32_t f, int32_t probe,
                                                const msacl_region_out_t& pres) {
  if (cell_inner(c, D, b)) return MSACL_REGION_INNER;
  if (verified(f)) return MSACL_REGION_VERIFIED;
  if (probe >= 0 && (pres.flags[probe] & (MSACL_REGION_REFUTE_DECREASE | MSACL_REGION_REFUTE_ESCAPED))) return MSACL_REGION_REFUTED;
  return (int)c[0] < b.max_depth ? MSACL_REGION_SPLIT : MSACL_REGION_UNDECIDED;
}

__global__ void __launch_bounds__(RB) region_decide_kernel(msacl_region_bnb_t b, int D, int64_t k, msacl_region_ws_t ws,
                                                           int64_t* stats) {
  __shared__ unsigned long long cnt[MSACL_REGION_ST_COUNT];
  __shared__ unsigned int kmin, kmax_in, kmax_v;
  if (threadIdx.x < MSACL_REGION_ST_COUNT) cnt[threadIdx.x] = 0;
  if (threadIdx.x == 0) { kmin = kKeyPosInf; kmax_in = kKeyNegInf; kmax_v = kKeyNegInf; }
  __syncthreads();
  const int64_t i = (int64_t)blockIdx.x * RB + threadIdx.x;
  int64_t children = 0, examples = 0;
  if (i < k) {
    const uint32_t* c = ws.cells + i * (1 + D);
    const uint32_t f = ws.res.flags[i];
    const uint32_t s = cell_status(b, D, c, f, ws.probe[i], ws.pres);
    ws.status[i] = (uint8_t)s;
    atomicAdd(&cnt[MSACL_REGION_ST_EVALUATED], 1ull);
    if (ws.probe[i] >= 0) atomicAdd(&cnt[MSACL_REGION_ST_PROBED], 1ull);
    const unsigned long long vol = 1ull << (MSACL_REGION_MAX_DEPTH - c[0]);
    const float vl = ws.res.v_lo[i];
    if (s == MSACL_REGION_SPLIT) {
      atomicAdd(&cnt[MSACL_REGION_ST_SPLIT], 1ull);
      children = 2;
    } else if (s == MSACL_REGION_INNER) {
      atomicAdd(&cnt[MSACL_REGION_ST_INNER], 1ull);
      atomicAdd(&cnt[MSACL_REGION_ST_VOLUME + 3], vol);
      if (f & (MSACL_REGION_NONFINITE | MSACL_REGION_ESCAPED | MSACL_REGION_LEAVES)) atomicAdd(&cnt[MSACL_REGION_ST_INNER_FAIL], 1ull);
      const float cin = ws.res.vm_hi[i], vh = ws.res.v_hi[i];
      atomicMax(&kmax_in, okey(isnan(cin) ? INFINITY : cin));
      atomicMax(&kmax_v, okey(isnan(vh) ? INFINITY : vh));
    } else {
      const int slot = s == MSACL_REGION_VERIFIED ? 0 : s == MSACL_REGION_REFUTED ? 1 : 2;
      atomicAdd(&cnt[MSACL_REGION_ST_VERIFIED + slot], 1ull);
      atomicAdd(&cnt[MSACL_REGION_ST_VOLUME + slot], vol);
      for (int bit = 0; bit < 5; ++bit)
        if (f & (1u << bit)) atomicAdd(&cnt[MSACL_REGION_ST_FLAGS + bit], 1ull);
      if (s != MSACL_REGION_VERIFIED || (f & MSACL_REGION_LEAVES)) atomicMin(&kmin, okey(isnan(vl) ? -INFINITY : vl));
      if (s == MSACL_REGION_REFUTED) examples = 1;
    }
  }
  int64_t tc, te;
  block_scan(children, &tc);
  block_scan(examples, &te);
  const int64_t nb = (k + RB - 1) / RB;
  if (threadIdx.x == 0) { ws.scan[nb + blockIdx.x] = tc; ws.scan[2 * nb + blockIdx.x] = te; }
  __syncthreads();
  unsigned long long* out = reinterpret_cast<unsigned long long*>(stats);
  if (threadIdx.x < MSACL_REGION_ST_COUNT && cnt[threadIdx.x]) atomicAdd(&out[threadIdx.x], cnt[threadIdx.x]);
  if (threadIdx.x == 0) {
    if (kmin != kKeyPosInf) atomicMin(&out[MSACL_REGION_ST_C_SOUND], (unsigned long long)kmin);
    if (kmax_in != kKeyNegInf) atomicMax(&out[MSACL_REGION_ST_C_IN], (unsigned long long)kmax_in);
    if (kmax_v != kKeyNegInf) atomicMax(&out[MSACL_REGION_ST_V_INNER], (unsigned long long)kmax_v);
  }
}

__global__ void __launch_bounds__(RB) region_scatter_kernel(msacl_region_bnb_t b, int D, int64_t k, msacl_region_ws_t ws,
                                                            uint32_t* __restrict__ child_out, const int64_t* stats,
                                                            float* examples) {
  const int64_t i = (int64_t)blockIdx.x * RB + threadIdx.x;
  const int64_t nb = (k + RB - 1) / RB;
  const uint32_t s = i < k ? ws.status[i] : 255u;
  int64_t tot;
  const int64_t co = block_scan(s == MSACL_REGION_SPLIT ? 2 : 0, &tot);
  const int64_t eo = block_scan(s == MSACL_REGION_REFUTED ? 1 : 0, &tot);
  if (i >= k) return;
  const int W = 1 + D;
  const uint32_t* c = ws.cells + i * W;
  if (s == MSACL_REGION_SPLIT) {
    const int64_t at = ws.scan[nb + blockIdx.x] + co;
    const int dim = (int)(c[0] % (uint32_t)D);
    for (int h = 0; h < 2; ++h) {
      uint32_t* o = child_out + (at + h) * W;
      o[0] = c[0] + 1;
      for (int d = 0; d < D; ++d) o[1 + d] = d == dim ? 2 * c[1 + d] + h : c[1 + d];
    }
  } else if (s == MSACL_REGION_REFUTED) {
    const int64_t before = stats[MSACL_REGION_ST_REFUTED] - ws.scan[3 * nb + 2];      // refuted cells of earlier rounds
    const int64_t slot = before + ws.scan[2 * nb + blockIdx.x] + eo;
    if (slot < b.max_examples) {
      const int32_t q = ws.probe[i];
      float* e = examples + slot * (D + 2);
      for (int d = 0; d < D; ++d) e[d] = ws.plo[(int64_t)q * D + d];
      const uint32_t pf = ws.pres.flags[q];
      e[D] = ws.pres.margin[q];
      e[D + 1] = (pf & MSACL_REGION_REFUTE_DECREASE) ? 1.f : 2.f;
    }
  }
}

template <int ID>
static int eval_launch(const msacl_region_params_t* p, const RDist& on, const float* image, int64_t n, const int64_t* n_dev,
                       const float* lo, const float* hi, const msacl_region_out_t* out, cudaStream_t s) {
  if constexpr (!IEnv<ID>::supported) {
    set_error("region_eval: env id %d is not supported (VanderPol, Pendulum, DuctedFan, TwoLink)", ID);
    return MSACL_ERR_BAD_ENV;
  } else {
    const int64_t tiles = (n + RTM - 1) / RTM;
    const unsigned grid = (unsigned)(tiles < kNumSMs ? (tiles > 0 ? tiles : 1) : kNumSMs);
    const size_t smem = sizeof(RSmem);
    auto launch = [&](auto kern) -> int {
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) { set_error("region_eval: smem attr: %s", cudaGetErrorString(e)); return (int)MSACL_ERR_CUDA; }
      kern<<<grid, RT, smem, s>>>(REval{*p, on}, image, n, n_dev, lo, hi, *out);
      return check_launch("region_eval");
    };
    return p->v_tanh ? launch(region_eval_kernel<ID, 1>) : launch(region_eval_kernel<ID, 0>);
  }
}

// Refuses bad parameters, and a disturbance bound in the first obs_dim / act_dim entries of p->dist that is non-finite or has
// lo > hi; *D = obs_dim, *on flags each disturbance set that is not exactly {0}.
static int check_params(const msacl_region_params_t* p, int* D, RDist* on) {
  if (!p || p->steps < 1 || !(p->decay_lo > 0.0) || !(p->decay_hi >= p->decay_lo) || !(p->alpha1 > 0.0) || !(p->alpha2 > 0.0)) {
    set_error("region: bad parameters (need steps >= 1, 0 < decay_lo <= decay_hi, alpha1, alpha2 > 0)");
    return MSACL_ERR_BAD_ARG;
  }
  int32_t dims[6];
  if (int rc = msacl_env_dims(p->env_id, dims)) return rc;
  *D = dims[0];
  if (p->env_id == kSingleTrackCar || p->env_id == kQuadTracking) {
    set_error("region: env id %d is not supported (VanderPol, Pendulum, DuctedFan, TwoLink)", p->env_id);
    return MSACL_ERR_BAD_ENV;
  }
  const msacl_region_disturbance_t& w = p->dist;
  *on = RDist{};
  const struct { const char* name; const float *lo, *hi; int n; int* on; } sets[3] = {
      {"obs", w.obs_lo, w.obs_hi, dims[0], &on->obs}, {"act", w.act_lo, w.act_hi, dims[1], &on->act},
      {"state", w.state_lo, w.state_hi, dims[0], &on->state}};
  for (const auto& s : sets)
    for (int d = 0; d < s.n; ++d) {
      if (!(std::isfinite(s.lo[d]) && std::isfinite(s.hi[d]) && s.lo[d] <= s.hi[d])) {
        set_error("region: disturbance %s[%d] = [%g, %g] is not a finite interval with lo <= hi", s.name, d, (double)s.lo[d],
                  (double)s.hi[d]);
        return MSACL_ERR_BAD_ARG;
      }
      if (s.lo[d] != 0.f || s.hi[d] != 0.f) *s.on = 1;
    }
  return MSACL_OK;
}

// msacl_region_eval after check_params
static int region_eval(const msacl_region_params_t* p, const RDist& on, const float* image, int64_t n, const int64_t* n_dev,
                       const float* lo, const float* hi, const msacl_region_out_t* out, void* stream) {
  if (n < 0 || !image || !lo || !hi || !out || !out->v_lo || !out->v_hi || !out->vm_lo || !out->vm_hi || !out->img_lo ||
      !out->img_hi || !out->flags || !out->margin) {
    set_error("region_eval: bad argument");
    return MSACL_ERR_BAD_ARG;
  }
  if ((reinterpret_cast<uintptr_t>(image) & 15) != 0) { set_error("region_eval: image must be 16-byte aligned"); return MSACL_ERR_BAD_ARG; }
  if (n == 0) return MSACL_OK;
  MSACL_DISPATCH_ENV(p->env_id, { return eval_launch<ID>(p, on, image, n, n_dev, lo, hi, out, (cudaStream_t)stream); });
  return MSACL_OK;
}

}  // namespace msacl

using namespace msacl;

extern "C" {

int64_t msacl_region_image_bytes(void) { return IMG_FLOATS * (int64_t)sizeof(float); }

int msacl_region_pack(const msacl_region_nets_t* s, float* image, void* stream) {
  if (!s || !image || !s->p_w1 || !s->p_b1 || !s->p_w2 || !s->p_b2 || !s->p_w3 || !s->p_b3 || !s->v_w1 || !s->v_b1 || !s->v_w2 ||
      !s->v_b2 || !s->v_w3 || !s->v_b3) {
    set_error("region_pack: null argument");
    return MSACL_ERR_BAD_ARG;
  }
  const int w[5] = {s->p_h1, s->p_h2, s->v_h1, s->v_h2, s->v_out};
  for (int v : w)
    if (v < 1 || v > RH) { set_error("region_pack: layer widths must be in [1, %d]", RH); return MSACL_ERR_BAD_ARG; }
  if (s->obs_dim < 1 || s->obs_dim > RD || s->act_dim < 1 || s->act_dim > 2) {
    set_error("region_pack: need 1 <= obs_dim <= %d and 1 <= act_dim <= 2", RD);
    return MSACL_ERR_BAD_ARG;
  }
  region_pack_kernel<<<2 * kNumSMs, 256, 0, (cudaStream_t)stream>>>(*s, image);
  return check_launch("region_pack");
}

int msacl_region_eval(const msacl_region_params_t* p, const float* image, int64_t n, const int64_t* n_dev, const float* lo,
                      const float* hi, const msacl_region_out_t* out, void* stream) {
  int D;
  RDist on;
  if (int rc = check_params(p, &D, &on)) return rc;
  return region_eval(p, on, image, n, n_dev, lo, hi, out, stream);
}

int msacl_region_round(const msacl_region_params_t* p, const msacl_region_bnb_t* b, const float* image, uint32_t* stack,
                       int64_t top, int64_t k, const msacl_region_ws_t* ws, int64_t* stats, float* examples, int64_t* children,
                       void* stream) {
  int D;
  RDist on;
  if (int rc = check_params(p, &D, &on)) return rc;
  if (!b || b->max_depth < 1 || b->max_depth > MSACL_REGION_MAX_DEPTH || b->inner_level < 0 || b->inner_level > 31 ||
      b->max_examples < 0 || !image || !stack || !ws || !stats || !children || k < 1 || top < k ||
      (b->max_examples > 0 && !examples)) {
    set_error("region_round: bad argument (need 1 <= max_depth <= %d, 1 <= k <= top)", (int)MSACL_REGION_MAX_DEPTH);
    return MSACL_ERR_BAD_ARG;
  }
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t nb = (k + RB - 1) / RB;
  uint32_t* cells = stack + (top - k) * (1 + D);
  region_cells_kernel<<<(unsigned)nb, RB, 0, s>>>(*p, D, cells, k, *ws);
  if (int rc = region_eval(p, on, image, k, nullptr, ws->lo, ws->hi, &ws->res, stream)) return rc;
  region_probe_kernel<<<(unsigned)nb, RB, 0, s>>>(*p, *b, D, k, *ws, 0);
  region_scan_kernel<<<1, RB, 0, s>>>(ws->scan, nb, ws->scan + 3 * nb);
  region_probe_kernel<<<(unsigned)nb, RB, 0, s>>>(*p, *b, D, k, *ws, 1);
  if (int rc = region_eval(p, on, image, k, ws->scan + 3 * nb, ws->plo, ws->phi, &ws->pres, stream)) return rc;
  region_decide_kernel<<<(unsigned)nb, RB, 0, s>>>(*b, D, k, *ws, stats);
  region_scan_kernel<<<1, RB, 0, s>>>(ws->scan + nb, nb, ws->scan + 3 * nb + 1);
  region_scan_kernel<<<1, RB, 0, s>>>(ws->scan + 2 * nb, nb, ws->scan + 3 * nb + 2);
  region_scatter_kernel<<<(unsigned)nb, RB, 0, s>>>(*b, D, k, *ws, cells, stats, examples);
  if (cudaMemcpyAsync(children, ws->scan + 3 * nb + 1, sizeof(int64_t), cudaMemcpyDeviceToDevice, s) != cudaSuccess)
    return check_launch("region_round");
  return check_launch("region_round");
}

}  // extern "C"
