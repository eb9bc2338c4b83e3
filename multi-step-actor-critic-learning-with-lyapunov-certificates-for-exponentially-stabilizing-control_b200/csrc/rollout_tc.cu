// Tensor-core fused rollout (tcgen05 / TMEM / TMA), sm_100a.
//
// Same contract as rollout_fused.cu (K iterations of BaseSampler._n_step,
// RL/trainer/sampler/base.py:118-163,220) but the two dense actor layers run on the 5th-gen tensor
// cores with a split-bf16 ("bf16x3") scheme that keeps FP32-class accuracy:
//     x = x1 + x2 (+ O(2^-17 |x|)),  w = w1 + w2   (all four bf16, round-to-nearest-even)
//     x.w ~= x1.w1 + x1.w2 + x2.w1                 (three UMMAs, FP32 accumulation in TMEM)
// Relative error of a product ~1e-5 (vs 4e-3 for single-pass bf16); tolerances in tests/test_gpu_tc.py.
//
// One persistent CTA per SM, NS = 3 tiles of 128 envs (slots) in flight, warp-specialised:
//   env warps (4*NS)  thread = env instance, state in registers for all K steps; sample action, integrate the ODE,
//                     reward/cost/autoreset, write the next observation as the layer-1 A operand (16-wide K block:
//                     obs, 1.0 for the bias, 0), then the transition.
//   MMA warp          one elected thread: layer 1 = 3 UMMAs (K=16, bias folded in as a K column), layer 2 =
//                     16 k-steps x 3 UMMAs of 128x256x16, FP32 accumulators in TMEM.  TMEM is used as TWO 256-column
//                     buffers; tile-step t keeps both its H1 and its H2 in buffer t&1 (H2 overwrites H1 once
//                     epilogue 1 has drained it), so the MLP of tile-step t+1 runs while epilogue 2 of t reads.
//   epilogue warps (8) both epilogues, split by column halves (two warps per TMEM lane quadrant):
//                     epilogue 1: TMEM(H1) -> ReLU -> split to bf16 hi/lo -> the shared-memory A operand of layer 2
//                     (the whole 128x256 tile is resident: 8 stages of 16 KB, UMMA canonical K-major layout, thread = row);
//                     epilogue 2: TMEM(H2) -> +b2, ReLU -> layer 3 (256 -> 2A) in packed FP32 FMAs, the two column
//                     halves combined through shared memory -> logits in shared memory.
//   TMA warp          pre-split W2 k-step images (16 KB) global/L2 -> shared ring (cp.async.bulk).
// All hand-offs are mbarriers (per-stage full/free for A and B, per-buffer full/free for H2, H1 full/free, X full,
// logits); tcgen05.commit signals the ones the tensor pipe produces.
// The alternatives measured against this layout (two tiles per env warpgroup, a dedicated epilogue-1 group, 2 or 4 tile
// slots) are in DESIGN.md §4.1.
#include "env_phase.cuh"
#include "tcgen05.cuh"

namespace msacl {

// Role timers for tools/tc_timing.py (build with MSACL_TC_TIMING=1): cycles spent by each warp role waiting on /
// working between hand-offs, accumulated into stats[5..18].
#ifdef MSACL_TC_TIMING
#define TC_T0(var) const long long var = clock64()
#define TC_ACC(slot, t0) do { if (stats) atomicAdd(&stats[slot], (double)(clock64() - (t0))); } while (0)
#else
#define TC_T0(var) do {} while (0)
#define TC_ACC(slot, t0) do {} while (0)
#endif

// Debug watchdog (build with MSACL_TC_WATCHDOG=1, tools/tc_watchdog.py): every mbarrier wait gives up after ~1.5 s,
// the first one to do so records {site, aux, block, parity, thread} in stats[25..29] and raises stats[24]; all other
// waits then fall through, so a protocol deadlock ends the launch (with garbage results) instead of hanging the GPU.
#ifdef MSACL_TC_WATCHDOG
__device__ __forceinline__ void wd_wait(void* bar, uint32_t parity, int site, uint32_t aux, double* stats) {
  const long long t0 = clock64();
  uint32_t spins = 0;
  volatile unsigned long long* flag = reinterpret_cast<volatile unsigned long long*>(&stats[24]);
  while (!tc::mbar_test(bar, parity)) {
    if ((++spins & 1023u) == 0u) {
      if (*flag != 0ull) return;
      if (clock64() - t0 > 3000000000LL) {
        if (atomicCAS(reinterpret_cast<unsigned long long*>(&stats[24]), 0ull, 0x3FF0000000000000ull) == 0ull) {
          stats[25] = site; stats[26] = aux; stats[27] = blockIdx.x; stats[28] = parity; stats[29] = threadIdx.x;
          __threadfence();
        }
        return;
      }
    }
  }
}
#define TC_WAIT(bar, par, site, aux) wd_wait(bar, par, site, (uint32_t)(aux), stats)
#else
#define TC_WAIT(bar, par, site, aux) tc::mbar_wait(bar, par)
#endif

constexpr int TC_NS = 3;            // tile slots in flight per CTA = env warpgroups
constexpr int TCM = 128;            // envs per tile
constexpr int TC_HID = 256;
constexpr int KC2 = 32;             // K per A stage
constexpr int NCH = TC_HID / KC2;   // 8 A stages = the whole layer-2 A operand of a tile
constexpr int KCB = 16;             // K per W2 stage (one UMMA k-step)
constexpr int NCHB = TC_HID / KCB;  // 16 W2 stages per tile-step
constexpr int NB_MAX = 4;           // W2 ring depth: see tc_ring_depth()
constexpr int A_HALF = TCM * KC2 * 2;       // 8 KB  (a1 or a2 image of a stage)
constexpr int B_HALF = TC_HID * KCB * 2;    // 8 KB  (b1 or b2 image of a stage)
constexpr int A_LBO = TCM * 16, B_LBO = TC_HID * 16, SBO = 128;
constexpr int X_HALF = TCM * 16 * 2;        // 4 KB  (x1 or x2: 128 rows x 16 k)
constexpr int W1_HALF = TC_HID * 16 * 2;    // 8 KB
// Launch geometry: TC_NS env warpgroups + 8 epilogue warps + {MMA, TMA, 2 idle warps}.  Registers are rebalanced with
// setmaxnreg (65536 per SM in total).  Per warp: launch regs * warps >= sum of the budgets below, or setmaxnreg.inc never
// returns; and all four warps of a warpgroup must execute the same setmaxnreg (the {MMA, TMA, idle, idle} group shares
// TC_MISC_REGS).  Launch 80*24 = 1920 = 12*112 + 8*56 + 4*32.
constexpr int TC_THREADS = 768, TC_ENV_REGS = 112, TC_EPI_REGS = 56, TC_MISC_REGS = 32;
constexpr int W2P_BYTES = NCHB * 2 * B_HALF;   // 256 KB packed W2 (hi/lo k-step images)
constexpr int W1P_BYTES = 2 * W1_HALF;

struct TcBars {
  unsigned long long xfull[TC_NS], logits[TC_NS];
  unsigned long long h1full[2], h1free[2], h2full[2], h2free[2];   // per TMEM buffer
  unsigned long long afull[NCH], afree[NCH], bfull[NB_MAX], bfree[NB_MAX];
  uint32_t tmem_slot;
};

// The share of the tile list one CTA walks (see the comment in the kernel): `share` contiguous tiles from `first`, in
// `rounds` rounds of per (+ 1 for the first `ex`) tiles.  Host + device: msacl_tc_tile_share() exposes the same arithmetic to the
// CPU tests (every tile exactly once, round sizes <= NS and non-increasing).
struct TcShare {
  int64_t first;
  int share, rounds, per, ex;
  __host__ __device__ TcShare(int64_t num_tiles, int64_t G, int64_t cta, int nt_max) {
    share = (int)(num_tiles / G + (cta < num_tiles % G ? 1 : 0));
    first = cta * (num_tiles / G) + (cta < num_tiles % G ? cta : num_tiles % G);
    rounds = (share + nt_max - 1) / nt_max;
    per = rounds ? share / rounds : 0;
    ex = rounds ? share % rounds : 0;
  }
  __host__ __device__ int tiles_in_round(int j) const { return per + (j < ex ? 1 : 0); }
  __host__ __device__ int64_t first_tile_of_round(int j) const { return first + (int64_t)j * per + (j < ex ? j : ex); }
};

// Layer-1 K block: obs (D) + bias column need 16 K columns only for the quadrotor (D + 1 = 13).  For the box envs
// (D + 1 <= 8) the second 8-column K block of both layer-1 operands is all zero, so it is not stored per slot: the
// operand descriptors' K-block stride (LBO) points at one shared zero block instead.  That and the narrower W3 (2A <= 4)
// free the shared memory for a fourth W2 ring stage.
template <int ID> __host__ __device__ constexpr bool tc_two_kblocks() { return Env<ID>::D + 1 > 8; }
template <int ID> __host__ __device__ constexpr int tc_ring_depth() { return tc_two_kblocks<ID>() ? 3 : 4; }
template <int ID> __host__ __device__ constexpr int tc_w3_stride() { return 2 * Env<ID>::A > 4 ? 8 : 4; }

template <int ID>
struct TcSmem {
  static constexpr bool X2 = tc_two_kblocks<ID>();
  static constexpr int NB = tc_ring_depth<ID>();
  static constexpr int XH = X2 ? X_HALF : X_HALF / 2;          // bytes of the hi (or lo) image of a slot's X operand
  static constexpr int W1H = X2 ? W1_HALF : W1_HALF / 2;       // bytes of the hi (or lo) image of the W1|b1 operand
  alignas(128) unsigned char bstage[NB][2 * B_HALF];     //  48 KB (box envs: 64 KB)
  alignas(128) unsigned char astage[NCH][2 * A_HALF];    // 128 KB
  alignas(128) unsigned char w1p[2 * W1H];               //  16 KB (box envs: 8 KB)
  alignas(128) unsigned char xop[TC_NS][2 * XH];         //   8 KB (4 KB) per env warpgroup; doubles as the slot's logits
  alignas(128) unsigned char zeros[X2 ? 128 : W1_HALF / 2];   // shared all-zero second K block (box envs)
  alignas(16) float w3t[TC_HID * tc_w3_stride<ID>()];   // layer-3 weights transposed: [unit n][output j] (zero padded)
  alignas(16) float b2[TC_HID];
  alignas(16) float b3[8];
  TcBars bars;
};

// packed FP32 FMA (FFMA2): two IEEE fma.rn per instruction; pack2(a, a) folds into the scalar-broadcast operand form
typedef unsigned long long u64;
__device__ __forceinline__ u64 pack2(float lo, float hi) { u64 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void unpack2(u64 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) { u64 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }

__device__ __forceinline__ uint32_t pack_bf16x2_rn(float lo, float hi) {   // {hi:lo} packed, RNE
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// 8 floats -> hi image (8 bf16) and lo image (8 bf16 of the residuals)
__device__ __forceinline__ void split8(const float (&v)[8], uint4& hi, uint4& lo) {
  uint32_t h[4], l[4];
#pragma unroll
  for (int p = 0; p < 4; ++p) {
    h[p] = pack_bf16x2_rn(v[2 * p], v[2 * p + 1]);
    const float r0 = v[2 * p] - __uint_as_float(h[p] << 16);
    const float r1 = v[2 * p + 1] - __uint_as_float(h[p] & 0xFFFF0000u);
    l[p] = pack_bf16x2_rn(r0, r1);
  }
  hi = make_uint4(h[0], h[1], h[2], h[3]);
  lo = make_uint4(l[0], l[1], l[2], l[3]);
}

// ---- one-time packing of the actor weights into UMMA operand images (device, per weight upload)
// w1p: [hi|lo] x [2 kb][256 n][8 k] bf16, K index d < D = W1[n][d], K index D = b1[n], rest 0
// w2p: 16 k-steps x [hi|lo] x [2 kb][256 n][8 k] bf16, K-major (B[n][k] = W2[n][k] = w2t[k][n])
__global__ void tc_pack_actor_kernel(msacl_actor_t actor, int D, unsigned char* __restrict__ w1p, unsigned char* __restrict__ w2p) {
  const int gid = blockIdx.x * blockDim.x + threadIdx.x;
  // W2: one thread per (k-step c, kb, n): 16 * 2 * 256 = 8192 threads
  if (gid < NCHB * 2 * TC_HID) {
    const int n = gid % TC_HID, kb = (gid / TC_HID) % 2, c = gid / (TC_HID * 2);
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = actor.w2t[(size_t)(c * KCB + kb * 8 + j) * TC_HID + n];
    uint4 hi, lo;
    split8(v, hi, lo);
    unsigned char* base = w2p + (size_t)c * 2 * B_HALF + kb * B_LBO + n * 16;
    *reinterpret_cast<uint4*>(base) = hi;
    *reinterpret_cast<uint4*>(base + B_HALF) = lo;
  }
  // W1 (+ bias column): one thread per (kb, n): 512 threads
  if (gid < 2 * TC_HID) {
    const int n = gid % TC_HID, kb = gid / TC_HID;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = kb * 8 + j;
      v[j] = k < D ? actor.w1[n * D + k] : (k == D ? actor.b1[n] : 0.f);
    }
    uint4 hi, lo;
    split8(v, hi, lo);
    unsigned char* base = w1p + kb * B_LBO + n * 16;
    *reinterpret_cast<uint4*>(base) = hi;
    *reinterpret_cast<uint4*>(base + W1_HALF) = lo;
  }
}

template <int ID>
__global__ void __launch_bounds__(TC_THREADS, 1)
rollout_tc_kernel(msacl_env_state_t st, msacl_actor_t actor, const unsigned char* __restrict__ w1p_g,
                  const unsigned char* __restrict__ w2p_g, int K, uint32_t step_base, int n_step,
                  float reward_scale, float cost_scale, const float* __restrict__ eps, int deterministic, msacl_transitions_t out,
                  double* stats) {
  using E = Env<ID>;
  using S = TcSmem<ID>;
  constexpr int D = E::D, A = E::A, A2 = 2 * A;
  constexpr int NS = TC_NS;                    // tiles in flight per CTA ("group"); tile slot s belongs to warpgroup s % NS
  constexpr int NB = S::NB, XH = S::XH, W1H = S::W1H, W3S = tc_w3_stride<ID>();
  constexpr bool X2 = S::X2;
  constexpr int W_EPI1 = 4 * NS, W_MMA = W_EPI1 + 8, W_TMA = W_MMA + 1;
  static_assert(D < 16, "layer-1 K block holds obs + bias column");
  static_assert(A2 * TCM * 4 <= XH && ((A2 + 1) / 2) * 2 * TCM * 4 <= XH, "logits and partial sums alias the two halves of the X-operand region");
  extern __shared__ __align__(128) unsigned char smem_raw[];
  S& sm = *reinterpret_cast<S*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // a slot's logits live in its X-operand region (free between layer 1 and the next write_xop)
  auto logits_of = [&](int s) { return reinterpret_cast<float*>(sm.xop[s]); };   // [2A][128] f32

  // ---- one-time setup
  // W1|b1 images: the packed global buffer always holds both K blocks per image; box envs keep only the first
  for (int i = tid; i < 2 * W1H / 16; i += TC_THREADS) {
    const int img = i / (W1H / 16), off = i % (W1H / 16);
    reinterpret_cast<uint4*>(sm.w1p)[i] = reinterpret_cast<const uint4*>(w1p_g + (size_t)img * W1_HALF)[off];
  }
  for (int i = tid; i < (int)sizeof(sm.zeros) / 16; i += TC_THREADS) reinterpret_cast<uint4*>(sm.zeros)[i] = make_uint4(0, 0, 0, 0);
  for (int i = tid; i < W3S * TC_HID; i += TC_THREADS) { const int n = i / W3S, j = i % W3S; sm.w3t[i] = j < A2 ? actor.w3[j * TC_HID + n] : 0.f; }
  for (int i = tid; i < TC_HID; i += TC_THREADS) sm.b2[i] = actor.b2[i];
  if (tid < 8) sm.b3[tid] = tid < A2 ? actor.b3[tid] : 0.f;
  if (tid == 0) {
    TcBars& b = sm.bars;
    for (int s = 0; s < NS; ++s) tc::mbar_init(&b.xfull[s], TCM);
    for (int s = 0; s < NS; ++s) tc::mbar_init(&b.logits[s], TCM);
    for (int i = 0; i < 2; ++i) {
      tc::mbar_init(&b.h1full[i], 1); tc::mbar_init(&b.h1free[i], 2 * TCM);     // drained by all warps of epilogue 1
      tc::mbar_init(&b.h2full[i], 1); tc::mbar_init(&b.h2free[i], 2 * TCM);
    }
    for (int i = 0; i < NCH; ++i) { tc::mbar_init(&b.afull[i], TCM); tc::mbar_init(&b.afree[i], 1); }
    for (int i = 0; i < NB; ++i) { tc::mbar_init(&b.bfull[i], 1); tc::mbar_init(&b.bfree[i], 1); }
    tc::mbar_fence_init();
  }
  if (warp == W_MMA) tc::tmem_alloc(&sm.bars.tmem_slot, 512);
  tc::fence_async_smem();      // w1p image was written with generic stores, read by UMMA
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = sm.bars.tmem_slot;     // buffer b of tile-step t (b = t & 1) = columns [256 b, 256 b + 256)

  const int64_t num_tiles = (st.n + TCM - 1) / TCM;
  // Groups ("pairs") of up to NS tiles in flight.  A CTA walks the group ids cta, cta + G, cta + 2 G, ... (G = gridDim.x).
  // The tiles are dealt to the CTAs in contiguous BALANCED shares -- CTA b owns T / G (+ 1) tiles and walks them in
  // ceil(share / NS) rounds of share / rounds (+ 1) tiles, the larger rounds first (so a warpgroup that has no tile in a round
  // has none in the later ones, and every earlier round of an active warpgroup was a full K steps: x_index below).  Cutting the
  // tile list into fixed groups of NS instead leaves most SMs idle for half the launch when the tile count is a small
  // multiple of the SM count: 65 536 envs = 512 tiles = 171 groups of 3 on 148 SMs are TWO rounds of 3 tiles for 23 CTAs and one
  // for the rest; balanced, 68 CTAs run two rounds of 2 tiles and 80 one round of 3.  Results do not depend on the mapping
  // (the RNG streams are keyed by the global env id).
  const int64_t G = gridDim.x, cta = blockIdx.x;
  const TcShare sh(num_tiles, G, cta, NS);
  const int64_t num_pairs = cta + (int64_t)sh.rounds * G;      // bound of `for (pair = cta; pair < num_pairs; pair += G)`
  // (32-bit division: round index = tiles / G at most)
  auto tiles_in_pair = [&](int64_t pair) -> int { return sh.tiles_in_round((int)(pair - cta) / (int)G); };
  auto first_tile = [&](int64_t pair) -> int64_t { return sh.first_tile_of_round((int)(pair - cta) / (int)G); };
  // X operands are written per warpgroup: group pi (all but the last are full), step k, tile slot s -> running index
  auto tiles_of_wg = [&](int w, int nt) { return nt > w ? (nt - w - 1) / NS + 1 : 0; };
  auto x_index = [&](uint32_t pi, int k, int s, int nt) { return pi * (uint32_t)K + (uint32_t)(k * tiles_of_wg(s % NS, nt) + s / NS); };

  if (warp < W_EPI1) {
    // =========================== env warps ===========================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(TC_ENV_REGS));
    const int w = warp >> 2;                 // env warpgroup: tile slots w, w + NS, ...
    const int r = tid & (TCM - 1);
    uint32_t lcount = 0;                     // logits deliveries each of its tile slots has consumed
    EpisodeStats epstats;
    auto write_xop = [&](const float* obs, bool valid) {
      float v[16];
#pragma unroll
      for (int k = 0; k < 16; ++k) v[k] = (k < D) ? (valid ? obs[k < D ? k : 0] : 0.f) : (k == D ? 1.f : 0.f);
#pragma unroll
      for (int kb = 0; kb < (X2 ? 2 : 1); ++kb) {
        float wv[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) wv[j] = v[kb * 8 + j];
        uint4 hi, lo;
        split8(wv, hi, lo);
        *reinterpret_cast<uint4*>(sm.xop[w] + kb * A_LBO + r * 16) = hi;
        *reinterpret_cast<uint4*>(sm.xop[w] + XH + kb * A_LBO + r * 16) = lo;
      }
      tc::fence_async_smem();
      tc::mbar_arrive(&sm.bars.xfull[w]);
    };
    for (int64_t pair = blockIdx.x; pair < num_pairs; pair += gridDim.x) {
      const int nt = tiles_in_pair(pair);
      if (w >= nt) break;
      const int64_t tile0 = first_tile(pair);
      EnvRegs<ID> e;
      // first observations of this group's tiles
#pragma unroll 1
      for (int s = w; s < nt; s += NS) {
        const int64_t gi = (tile0 + s) * TCM + r;
        const bool owner = gi < st.n;
        if (owner) e.load(st, gi);
        write_xop(e.obs(), owner);
      }
      for (int k = 0; k < K; ++k) {
#pragma unroll 1
        for (int s = w; s < nt; s += NS) {
        const int64_t gi = (tile0 + s) * TCM + r;
        const bool owner = gi < st.n;
        const int64_t row = (int64_t)k * st.n + gi;
        // the action noise of this step does not depend on the logits: draw it while the tile's MLP is still running
        float z[4];
        env_noise<A>(z, owner && !deterministic, eps, row, st.seed, st.env_base + (uint64_t)gi, step_base + (uint32_t)k);
#ifdef MSACL_TC_TIMING
        const long long t_w0 = clock64();
#endif
        TC_WAIT(&sm.bars.logits[s], lcount & 1, 1, lcount);
        // the logits of this slot were written into its X-operand region (free between layer 1 and the next
        // write_xop): take them into registers, then a slot-wide barrier so that no thread of the slot can overwrite
        // them with its next observation before every thread has read its own
        float lg[A2];
#pragma unroll
        for (int j = 0; j < A2; ++j) lg[j] = logits_of(s)[j * TCM + r];
        tc::bar_sync(1 + w, 128);
#ifdef MSACL_TC_TIMING
        const long long t_w1 = clock64();
#endif
        if (owner) {
          env_phase<ID>(e, lg, z, deterministic, actor.min_log_std, actor.max_log_std, st, gi, n_step, reward_scale, cost_scale,
                        out, row, epstats, [&](const float* obs) { if (k + 1 < K) write_xop(obs, true); });
        } else if (k + 1 < K) {
          write_xop(e.obs(), false);
        }
#ifdef MSACL_TC_TIMING
        if (stats && r == 0) {
          const long long t_e = clock64();
          atomicAdd(&stats[5], (double)(t_e - t_w1));
          atomicAdd(&stats[6], (double)(t_w1 - t_w0));
          atomicAdd(&stats[7], 1.0);
        }
#endif
        }
        ++lcount;
      }
      const int64_t gi = (tile0 + w) * TCM + r;
      if (gi < st.n) e.store(st, gi);
    }
    if (stats) epstats.flush(stats);
  } else if (warp < W_MMA) {
    // =========================== epilogue warps (8): both epilogues, column-split ===========================
    // Warp e = warp - W_EPI1: TMEM lane quadrant q = e & 3 (rows 32q..32q+31, thread = row), column half h = e >> 2.
    //   epilogue 1 of a tile-step: H1[:, 128h..128h+127] -> ReLU -> bf16 hi/lo -> A stages 4h..4h+3
    //   epilogue 2 of a tile-step: H2[:, 128h..128h+127] -> +b2, ReLU -> partial layer 3 (packed FP32 FMAs); half 1
    //                              parks its partial sums in the slot's shared-memory region, half 0 adds them,
    //                              writes the logits and signals the slot's env warps.
    // Job order per tile-step t (groups of >= 2 slots): epilogue 1 of t+1 (it trails layer 2 of t stage by stage), then
    // epilogue 2 of t (while layer 2 of t+1 runs).  With a single slot the X operand of t+1 needs the logits of t, so
    // the order is swapped.
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(TC_EPI_REGS));
    const int q = warp & 3;
    const int h = (warp - W_EPI1) >> 2;      // column half
    const int r = q * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const bool timer = lane == 0 && warp == W_EPI1;
    auto epi1 = [&](uint32_t t1) {
      const uint32_t buf = t1 & 1u, tmem_b = tmem + buf * 256u;
      TC_T0(t_a);
      TC_WAIT(&sm.bars.h1full[buf], (t1 >> 1) & 1, 2, t1);
      tc::tc_fence_after();
      if (timer) TC_ACC(8, t_a);                      // epi1: wait for H1
      TC_T0(t_b);
#pragma unroll 1
      for (int cc = 0; cc < NCH / 2; ++cc) {
        const int c = h * (NCH / 2) + cc;
        TC_T0(t_c);
        if (t1 > 0) TC_WAIT(&sm.bars.afree[c], (t1 - 1) & 1, 3, t1);   // layer 2 of the previous tile-step is done with stage c
        if (timer) TC_ACC(10, t_c);                   // epi1: wait for a free A stage
        uint32_t v[32];
        tc::tmem_ld32(tmem_b + lane_addr + (uint32_t)(c * 32), v);
        tc::tmem_ld_wait();
        if (cc == NCH / 2 - 1) { tc::tc_fence_before(); tc::mbar_arrive(&sm.bars.h1free[buf]); }   // layer 2 may overwrite the buffer
        unsigned char* base = sm.astage[c] + r * 16;
#pragma unroll
        for (int kb = 0; kb < 4; ++kb) {
          float w[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) w[j] = fmaxf(__uint_as_float(v[kb * 8 + j]), 0.f);
          uint4 hi, lo;
          split8(w, hi, lo);
          *reinterpret_cast<uint4*>(base + kb * A_LBO) = hi;
          *reinterpret_cast<uint4*>(base + A_HALF + kb * A_LBO) = lo;
        }
        tc::fence_async_smem();
        tc::mbar_arrive(&sm.bars.afull[c]);
      }
      if (timer) TC_ACC(9, t_b);                      // epi1: chunk loop total
    };
    auto epi2 = [&](uint32_t t0, int s) {
      const uint32_t buf = t0 & 1u, tmem_b = tmem + buf * 256u;
      TC_T0(t_a);
      TC_WAIT(&sm.bars.h2full[buf], (t0 >> 1) & 1, 4, t0);
      tc::tc_fence_after();
      if (timer) TC_ACC(11, t_a);                     // epi2: wait for H2
      TC_T0(t_b);
      constexpr int NP = (A2 + 1) / 2;                // logit pairs (j, j+1) accumulated with packed FFMA2
      u64 acc[NP];
#pragma unroll
      for (int p = 0; p < NP; ++p) acc[p] = h == 0 ? pack2(sm.b3[2 * p], sm.b3[2 * p + 1]) : pack2(0.f, 0.f);
#pragma unroll 1
      for (int cc = 0; cc < TC_HID / 32; ++cc) {        // 16 columns per TMEM load: leaves registers to prefetch W3 rows
        const int cb = h * (TC_HID / 32) + cc;
        uint32_t v[16];
        tc::tmem_ld16(tmem_b + lane_addr + (uint32_t)(cb * 16), v);
        tc::tmem_ld_wait();
        if (cc == TC_HID / 32 - 1) { tc::tc_fence_before(); tc::mbar_arrive(&sm.bars.h2free[buf]); }
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const float4 bb = *reinterpret_cast<const float4*>(&sm.b2[cb * 16 + 4 * g]);
          const float hv[4] = {fmaxf(__uint_as_float(v[4 * g + 0]) + bb.x, 0.f), fmaxf(__uint_as_float(v[4 * g + 1]) + bb.y, 0.f),
                               fmaxf(__uint_as_float(v[4 * g + 2]) + bb.z, 0.f), fmaxf(__uint_as_float(v[4 * g + 3]) + bb.w, 0.f)};
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const float* wrow = &sm.w3t[(cb * 16 + 4 * g + c) * W3S];    // all lanes read the same address: broadcast
            const u64 hh = pack2(hv[c], hv[c]);
            if constexpr (NP >= 1) {
              const float4 w0 = *reinterpret_cast<const float4*>(wrow);
              acc[0] = fma2(hh, pack2(w0.x, w0.y), acc[0]);
              if constexpr (NP >= 2) acc[1] = fma2(hh, pack2(w0.z, w0.w), acc[1]);
            }
            if constexpr (NP >= 3) {
              const float4 w1 = *reinterpret_cast<const float4*>(wrow + 4);
              acc[2] = fma2(hh, pack2(w1.x, w1.y), acc[2]);
              if constexpr (NP >= 4) acc[3] = fma2(hh, pack2(w1.z, w1.w), acc[3]);
            }
          }
        }
      }
      // combine the two column halves: rows of quadrant q are shared by warps (q, half 0) and (q, half 1)
      float* part = reinterpret_cast<float*>(sm.xop[s] + XH);      // second half of the slot's X-operand region
      float* lgs = logits_of(s);
      if (h == 1) {
#pragma unroll
        for (int p = 0; p < NP; ++p) {
          float lo, hi;
          unpack2(acc[p], lo, hi);
          part[(2 * p) * TCM + r] = lo;
          part[(2 * p + 1) * TCM + r] = hi;
        }
      }
      tc::bar_sync(4 + q, 64);
      if (h == 0) {
#pragma unroll
        for (int p = 0; p < NP; ++p) {
          float lo, hi;
          unpack2(acc[p], lo, hi);
          lgs[(2 * p) * TCM + r] = lo + part[(2 * p) * TCM + r];
          if (2 * p + 1 < A2) lgs[(2 * p + 1) * TCM + r] = hi + part[(2 * p + 1) * TCM + r];
        }
        tc::mbar_arrive(&sm.bars.logits[s]);
      }
      if (timer) TC_ACC(12, t_b);                     // epi2: compute
    };
    uint32_t ts = 0;
    for (int64_t pair = blockIdx.x; pair < num_pairs; pair += gridDim.x) {
      const int nt = tiles_in_pair(pair);
      for (int k = 0; k < K; ++k)
        for (int s = 0; s < nt; ++s, ++ts) {
          if (ts == 0) epi1(0u);
          const bool has_next = !(s + 1 == nt && k + 1 == K && pair + (int64_t)gridDim.x >= num_pairs);
          const bool epi2_first = nt <= 1;
          if (!epi2_first) {
            if (has_next) epi1(ts + 1);
            epi2(ts, s);
          } else {
            epi2(ts, s);
            if (has_next) epi1(ts + 1);
          }
        }
    }
  } else {
    // (setmaxnreg must be executed with the same value by all four warps of a warpgroup)
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(TC_MISC_REGS));
    if (warp == W_MMA) {
    // =========================== MMA issuer ===========================
    if (tc::elect_one()) {
      const uint32_t idesc = tc::make_idesc_bf16(TCM, TC_HID);
      const uint32_t w1base = tc::smem_u32(sm.w1p);
      // The issuing thread is the serial resource of the tensor pipeline, so its per-k-step instruction stream is kept
      // short: descriptors are (constant high word, low word = base + (byte offset >> 4)) -- the 14-bit address field
      // cannot carry because shared memory is < 256 KB -- and the W2 ring position is tracked incrementally.
      const uint32_t a_lo0 = (uint32_t)tc::make_smem_desc(tc::smem_u32(sm.astage[0]), A_LBO, SBO);
      const uint32_t b_lo0 = (uint32_t)tc::make_smem_desc(tc::smem_u32(sm.bstage[0]), B_LBO, SBO);
      const uint32_t d_hi = (uint32_t)(tc::make_smem_desc(0u, 0u, SBO) >> 32);
      auto mk = [&](uint32_t lo) { return ((uint64_t)d_hi << 32) | (uint64_t)lo; };
      uint32_t bs = 0, bph = 0;                       // W2 ring stage / phase parity of the next k-step
      // layer 1 of tile-step t1 (slot s; xn = number of X operands that slot has produced before) into buffer t1 & 1:
      // H1 = [obs | 1 | 0] . [W1 | b1 | 0]^T  (K = 16, three products)
      auto issue_l1 = [&](int s, uint32_t xn, uint32_t t1) {
        TC_T0(t_h);
        if (t1 >= 2) TC_WAIT(&sm.bars.h2free[t1 & 1], ((t1 >> 1) - 1) & 1, 10, t1);   // epilogue 2 of tile-step t1-2 has drained the buffer
        TC_ACC(17, t_h);                              // MMA: wait for a free TMEM buffer
        TC_T0(t_x);
        TC_WAIT(&sm.bars.xfull[s % NS], xn & 1, 7, t1);
        TC_ACC(13, t_x);                              // MMA: wait for X
        tc::tc_fence_after();
        const uint32_t tmem_b = tmem + (t1 & 1u) * 256u;
        // K-block stride: the next 8 K columns follow in place (quadrotor) or are the shared zero block (box envs)
        const uint32_t xbase = tc::smem_u32(sm.xop[s % NS]), zbase = tc::smem_u32(sm.zeros);
        const uint64_t dw1 = tc::make_smem_desc(w1base, X2 ? B_LBO : zbase - w1base, SBO);
        const uint64_t dw2 = tc::make_smem_desc(w1base + W1H, X2 ? B_LBO : zbase - (w1base + W1H), SBO);
        const uint64_t dx1 = tc::make_smem_desc(xbase, X2 ? A_LBO : zbase - xbase, SBO);
        const uint64_t dx2 = tc::make_smem_desc(xbase + XH, X2 ? A_LBO : zbase - (xbase + XH), SBO);
        tc::umma_bf16(tmem_b, dx1, dw1, idesc, 0u);
        tc::umma_bf16(tmem_b, dx1, dw2, idesc, 1u);
        tc::umma_bf16(tmem_b, dx2, dw1, idesc, 1u);
        tc::umma_commit(&sm.bars.h1full[t1 & 1]);
      };
      uint32_t ts = 0, pi = 0;                        // tile-step counter, local group counter
      for (int64_t pair = blockIdx.x; pair < num_pairs; pair += gridDim.x, ++pi) {
        const int nt = tiles_in_pair(pair);
        for (int k = 0; k < K; ++k)
          for (int s = 0; s < nt; ++s, ++ts) {
            if (ts == 0) issue_l1(0, 0u, 0u);
            const uint32_t buf = ts & 1u, tmem_b = tmem + buf * 256u;
            // ---- successor tile-step: its layer 1 goes into the other buffer as early as that buffer is drained and
            //      its X operand is there (probed without blocking before and between the layer-2 chunks), so that
            //      epilogue 1 of the successor trails this tile's layer 2 stage by stage; at the latest after layer 2
            int s2 = s + 1, k2 = k;
            int64_t pair2 = pair;
            uint32_t pi2 = pi;
            if (s2 == nt) { s2 = 0; if (++k2 == K) { k2 = 0; pair2 += gridDim.x; ++pi2; } }
            bool next_pending = pair2 < num_pairs;
            const uint32_t xn2 = x_index(pi2, k2, s2, (pair2 == pair || !next_pending) ? nt : tiles_in_pair(pair2)), t2 = ts + 1;
            auto try_next = [&]() {
              if (next_pending && (t2 < 2 || tc::mbar_test(&sm.bars.h2free[t2 & 1], ((t2 >> 1) - 1) & 1)) &&
                  tc::mbar_test(&sm.bars.xfull[s2 % NS], xn2 & 1)) {
                issue_l1(s2, xn2, t2);
                next_pending = false;
              }
            };
            try_next();
            // ---- layer 2: H2 = relu(H1) . W2^T, accumulated over H1's own buffer once epilogue 1 has drained it
            TC_T0(t_h);
            TC_WAIT(&sm.bars.h1free[buf], (ts >> 1) & 1, 8, ts);
            TC_ACC(14, t_h);                          // MMA: wait for epilogue 1 to finish reading H1
#pragma unroll 1
            for (int c = 0; c < NCH; ++c) {
              TC_T0(t_1);
              TC_WAIT(&sm.bars.afull[c], ts & 1, 9, ts);
              TC_ACC(15, t_1);                        // MMA: wait for A stage
              const uint32_t a_lo = a_lo0 + (uint32_t)c * (2 * A_HALF / 16);
#pragma unroll
              for (int j = 0; j < KC2 / KCB; ++j) {
                TC_T0(t_2);
                TC_WAIT(&sm.bars.bfull[bs], bph, 11, ts);
                TC_ACC(16, t_2);                      // MMA: wait for B stage
                tc::tc_fence_after();
                const uint32_t b_lo = b_lo0 + bs * (2 * B_HALF / 16);
                const uint64_t da1 = mk(a_lo + j * (2 * A_LBO / 16)), da2 = mk(a_lo + j * (2 * A_LBO / 16) + A_HALF / 16);
                const uint64_t db1 = mk(b_lo), db2 = mk(b_lo + B_HALF / 16);
                tc::umma_bf16(tmem_b, da1, db1, idesc, (c > 0 || j > 0) ? 1u : 0u);
                tc::umma_bf16(tmem_b, da1, db2, idesc, 1u);
                tc::umma_bf16(tmem_b, da2, db1, idesc, 1u);
                tc::umma_commit(&sm.bars.bfree[bs]);
                if (++bs == NB) { bs = 0; bph ^= 1u; }
              }
              tc::umma_commit(&sm.bars.afree[c]);
              try_next();
            }
            tc::umma_commit(&sm.bars.h2full[buf]);
            if (next_pending) issue_l1(s2, xn2, t2);
#ifdef MSACL_TC_TIMING
            if (stats) atomicAdd(&stats[18], 1.0);
#endif
          }
      }
    }
    } else if (warp == W_TMA) {
    // =========================== TMA producer: W2 k-step images ===========================
    if (tc::elect_one()) {
      int64_t tile_steps = 0;
      for (int64_t pair = blockIdx.x; pair < num_pairs; pair += gridDim.x) tile_steps += (int64_t)tiles_in_pair(pair) * K;
      const int64_t total = tile_steps * NCHB;
      uint32_t bs = 0, bph = 1, kk = 0;            // ring stage, parity of the "free" phase to wait for, k-step within the tile
      for (int64_t i = 0; i < total; ++i) {
        if (i >= NB) TC_WAIT(&sm.bars.bfree[bs], bph, 13, i);
        tc::mbar_expect_tx(&sm.bars.bfull[bs], 2 * B_HALF);
        tc::tma_bulk_g2s(sm.bstage[bs], w2p_g + (size_t)kk * 2 * B_HALF, 2 * B_HALF, &sm.bars.bfull[bs]);
        if (++bs == NB) { bs = 0; bph ^= 1u; }
        if (++kk == NCHB) kk = 0;
      }
    }
    }
  }
  // ---- teardown
  tc::tc_fence_before();
  __syncthreads();
  if (warp == W_MMA) tc::tmem_dealloc(tmem, 512);
}

}  // namespace msacl

using namespace msacl;

static int g_tc_max_ctas = 0;      // 0 = one persistent CTA per SM

extern "C" int msacl_rollout_tc_set_max_ctas(int32_t max_ctas) {
  if (max_ctas < 0 || max_ctas > kNumSMs) { set_error("rollout_tc_set_max_ctas: expected 0 (all SMs) .. %d", kNumSMs); return MSACL_ERR_BAD_ARG; }
  g_tc_max_ctas = max_ctas;
  return MSACL_OK;
}

extern "C" int msacl_tc_tile_share(int64_t n_envs, int32_t grid, int32_t cta, int64_t* out) {
  if (n_envs <= 0 || grid <= 0 || cta < 0 || cta >= grid || !out) { set_error("tc_tile_share: bad argument"); return MSACL_ERR_BAD_ARG; }
  const TcShare sh((n_envs + TCM - 1) / TCM, grid, cta, TC_NS);
  out[0] = sh.first; out[1] = sh.share; out[2] = sh.rounds; out[3] = sh.per; out[4] = sh.ex;
  return MSACL_OK;
}

extern "C" int msacl_tc_pack_bytes(int64_t* w1p_bytes, int64_t* w2p_bytes) {
  if (w1p_bytes) *w1p_bytes = W1P_BYTES;
  if (w2p_bytes) *w2p_bytes = W2P_BYTES;
  return MSACL_OK;
}

extern "C" int msacl_tc_pack_actor(const msacl_actor_t* actor, int32_t obs_dim, void* w1p, void* w2p, void* stream) {
  if (!actor || !w1p || !w2p || obs_dim < 1 || obs_dim > 15) { set_error("tc_pack_actor: bad argument"); return MSACL_ERR_BAD_ARG; }
  tc_pack_actor_kernel<<<(NCHB * 2 * TC_HID + 255) / 256, 256, 0, (cudaStream_t)stream>>>(*actor, obs_dim, (unsigned char*)w1p, (unsigned char*)w2p);
  return check_launch("tc_pack_actor");
}

extern "C" int msacl_rollout_fused_tc(const msacl_env_state_t* st, const msacl_actor_t* actor, const void* w1p,
                                      const void* w2p, int32_t K, uint32_t step_base, int32_t n_step, float reward_scale,
                                      float cost_scale, const float* eps, int32_t deterministic,
                                      const msacl_transitions_t* out, double* stats, void* stream) {
  if (!st || !actor || !out || !w1p || !w2p || st->n <= 0 || K <= 0 || n_step <= 0) { set_error("rollout_fused_tc: bad argument"); return MSACL_ERR_BAD_ARG; }
  if ((reinterpret_cast<uintptr_t>(w2p) & 15) || (reinterpret_cast<uintptr_t>(w1p) & 15)) { set_error("rollout_fused_tc: packed weights must be 16-byte aligned"); return MSACL_ERR_BAD_ARG; }
  const int64_t tiles = (st->n + TCM - 1) / TCM;
  MSACL_DISPATCH_ENV(st->env_id, {
    if (int rc = check_rollout_outputs<ID>("rollout_fused_tc", st, out)) return rc;
    static_assert(sizeof(TcSmem<ID>) + 128 <= 232448, "shared-memory layout exceeds the 227 KB per-CTA limit");
    const int64_t cap = g_tc_max_ctas > 0 ? g_tc_max_ctas : kNumSMs;
    const unsigned grid = (unsigned)(tiles < cap ? tiles : cap);      // balanced shares: every CTA owns >= 1 tile
    const size_t smem = sizeof(TcSmem<ID>) + 128;
    auto kern = rollout_tc_kernel<ID>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { set_error("rollout_fused_tc: smem attr (%zu B): %s", smem, cudaGetErrorString(e)); return MSACL_ERR_CUDA; }
    kern<<<grid, TC_THREADS, smem, (cudaStream_t)stream>>>(*st, *actor, (const unsigned char*)w1p, (const unsigned char*)w2p, K,
                                                           step_base, n_step, reward_scale, cost_scale, eps, deterministic, *out, stats);
  });
  return check_launch("rollout_fused_tc");
}
