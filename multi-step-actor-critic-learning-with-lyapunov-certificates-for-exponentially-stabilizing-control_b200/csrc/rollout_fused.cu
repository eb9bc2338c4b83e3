// Fused K-step rollout kernel: actor MLP (obs -> 256 -> 256 -> 2A) + TanhGauss sample + clip +
// env dynamics + reward/cost + same-step autoreset + n-step bookkeeping.  Replaces K iterations
// of BaseSampler._n_step (RL/trainer/sampler/base.py:118-163,220).
//
// Design (B200, sm_100a), v3 -- warp specialised, one persistent CTA of 12 warps per SM:
//   * warps 0-7 ("GEMM warps") run the MLP for two 64-env tiles A/B alternately; warps 8-9 own
//     the env instances of tile A, warps 10-11 those of tile B ("env warps": state in registers
//     for all K steps, so HBM sees the state once per launch and one transition record per step).
//     While the env warps of tile A sample the action and integrate the ODE, the GEMM warps are
//     already multiplying tile B: the latency-bound env phase is off the FFMA critical path.
//     Hand-offs use named barriers (bar.arrive / bar.sync): X_READY[T] (env -> GEMM, obs tile in
//     smem) and LOGITS[T] (GEMM -> env).
//   * the MLP is >99% of the FLOPs (SURVEY.md 8d) and is an FP32 contraction (parity with the
//     reference's fp32 torch actor rules out single-pass bf16/tf32 tensor-core MMA), so the
//     binding roofline is the FP32 FFMA pipe.  Every GEMM warp owns 8 envs of the tile for the
//     whole MLP (8x8 register tile per thread: envs warp*8..+8 x units {lane*4..+4,
//     128+lane*4..+4}), so layers 1-3 need no block-wide barrier at all: the hidden-1
//     activations a warp writes (K-major layout with an XOR granule swizzle: conflict-free float4
//     stores, warp-broadcast float4 reads) are only ever read by the same warp.
//   * W2^T (256 KB, shared by all CTAs, resident in the 126 MB L2) is streamed in 16-row chunks
//     by TMA bulk copies (cp.async.bulk -> UBLKCP) into a 4-stage shared-memory ring guarded by
//     full/empty mbarriers: one elected thread issues, consumers wait per warp and release per
//     warp, so warps drift freely and the FFMA pipe is not gated by block barriers.  The chunk
//     sequence is identical for every tile, so the ring never drains across tile boundaries.
//   * layer 3 (256 -> 2A) is applied to the layer-2 register tile and combined with a halving
//     warp-shuffle reduction (62 shuffles / 64 values).
// Compiled with -fmad=false: only the explicit __fmaf_rn calls below contract.
#include "env_phase.cuh"
#include "tcgen05.cuh"

namespace msacl {

constexpr int TM = 64;          // envs per tile
constexpr int HID = 256;        // hidden width (reference default, msacl_train.py policy_hidden_sizes)
constexpr int NGEMM = 256;      // GEMM threads (warps 0-7)
constexpr int NTILE = 2;        // tiles in flight per CTA
constexpr int NTHREADS = NGEMM + NTILE * TM;   // 384
constexpr int KC = 16;          // W2^T rows per TMA chunk
constexpr int NCHUNK = HID / KC;
constexpr int NSTAGE = 4;       // ring depth
constexpr int PREFETCH = NSTAGE - 2;   // chunks in flight ahead of the consumer
constexpr uint32_t CHUNK_BYTES = KC * HID * 4;
static_assert(NCHUNK % NSTAGE == 0, "stage index must be tile-invariant");

enum : int { BAR_LOGITS = 2, BAR_XREADY = 4 };

template <int ID>
struct Smem {
  using E = Env<ID>;
  static constexpr int A2 = 2 * E::A;
  float h1[HID * TM];            // [k][m]  hidden-1 activations of the tile in the GEMM
  float wc[NSTAGE][KC * HID];    // W2^T chunk ring [k][n]
  float w1t[E::D * HID];         // W1^T [d][n]
  float w3[A2 * HID];            // [j][k]
  float b1[HID];
  float b2[HID];
  float b3[8];
  float x[NTILE][E::D * TM];     // obs tiles [d][m]
  float out[NTILE][A2 * TM];     // logits [j][m]
  unsigned long long full_bar[NSTAGE];
  unsigned long long empty_bar[NSTAGE];
};

// Halving butterfly: V values per lane summed over the 32 lanes; afterwards value
// `orig` lives in v[0..V/32) of lane orig / (V/32) (V >= 32), or in v[0] of lanes
// (orig * 32/V) .. (V < 32, replicated).
template <int V>
__device__ __forceinline__ void warp_multi_reduce(float (&v)[V], int lane) {
  int c = V;
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {
    if (c > 1) {
      const bool upper = (lane & s) != 0;
      const int half = c / 2;
#pragma unroll
      for (int i = 0; i < V / 2; ++i) {
        if (i < half) {
          const float keep = upper ? v[i + half] : v[i];
          const float send = upper ? v[i] : v[i + half];
          v[i] = keep + __shfl_xor_sync(0xffffffffu, send, s);
        }
      }
      c = half;
    } else {
      v[0] = v[0] + __shfl_xor_sync(0xffffffffu, v[0], s);
    }
  }
}

template <int ID>
__global__ void __launch_bounds__(NTHREADS, 1)
rollout_fused_kernel(msacl_env_state_t st, msacl_actor_t actor, int K, uint32_t step_base, int n_step,
                     float reward_scale, float cost_scale, const float* __restrict__ eps, int deterministic,
                     msacl_transitions_t out, double* stats) {
  using E = Env<ID>;
  using S = Smem<ID>;
  constexpr int D = E::D, A = E::A, A2 = 2 * A;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  S& sm = *reinterpret_cast<S*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  // ---- stage the small weights once per CTA
  for (int i = tid; i < D * HID; i += NTHREADS) {
    const int d = i / HID, n = i % HID;
    sm.w1t[i] = actor.w1[n * D + d];
  }
  for (int i = tid; i < A2 * HID; i += NTHREADS) sm.w3[i] = actor.w3[i];
  for (int i = tid; i < HID; i += NTHREADS) { sm.b1[i] = actor.b1[i]; sm.b2[i] = actor.b2[i]; }
  if (tid < 8) sm.b3[tid] = tid < A2 ? actor.b3[tid] : 0.f;
  if (tid == 0) {
#pragma unroll
    for (int i = 0; i < NSTAGE; ++i) { tc::mbar_init(&sm.full_bar[i], 1); tc::mbar_init(&sm.empty_bar[i], NGEMM / 32); }
    tc::mbar_fence_init();
    tc::fence_async_smem();
  }
  __syncthreads();

  const int64_t num_tiles = (st.n + TM - 1) / TM;
  const int64_t num_pairs = (num_tiles + NTILE - 1) / NTILE;

  if (tid < NGEMM) {
    // =========================== GEMM warps ===========================
    // number of W2 chunks this CTA will consume (producer must not run past it)
    int64_t my_tile_steps = 0;
    for (int64_t pair = blockIdx.x; pair < num_pairs; pair += gridDim.x)
      my_tile_steps += ((num_tiles - NTILE * pair) < NTILE ? (num_tiles - NTILE * pair) : NTILE) * (int64_t)K;
    const int64_t total_chunks = my_tile_steps * NCHUNK;
    const bool producer = (tid == 0);
    auto produce = [&](int64_t gi) {          // issue chunk gi (global index) into stage gi % NSTAGE
      if (gi >= total_chunks) return;
      const int stg = (int)(gi % NSTAGE);
      if (gi >= NSTAGE) tc::mbar_wait(&sm.empty_bar[stg], (uint32_t)(((gi / NSTAGE) & 1) ^ 1));
      tc::mbar_expect_tx(&sm.full_bar[stg], CHUNK_BYTES);
      tc::tma_bulk_g2s(sm.wc[stg], actor.w2t + (size_t)(gi % NCHUNK) * KC * HID, CHUNK_BYTES, &sm.full_bar[stg]);
    };
    if (producer) {
#pragma unroll
      for (int i = 0; i < PREFETCH; ++i) produce(i);
    }
    int64_t g = 0;                            // global chunk counter (identical in all GEMM threads)
    const int m0 = warp * 8;                  // this warp's envs within the tile
    for (int64_t pair = blockIdx.x; pair < num_pairs; pair += gridDim.x) {
      const int nt = (int)((num_tiles - NTILE * pair) < NTILE ? (num_tiles - NTILE * pair) : NTILE);
      for (int k = 0; k < K; ++k) {
        for (int T = 0; T < nt; ++T) {
          tc::bar_sync(BAR_XREADY + T, NGEMM + TM);   // obs tile T is in smem
          float acc[8][8];
          // ---- layer 1 on the same thread tile as layer 2 (envs m0..m0+8 x 8 units)
          {
            const float4 q0 = *reinterpret_cast<const float4*>(&sm.b1[lane * 4]);
            const float4 q1 = *reinterpret_cast<const float4*>(&sm.b1[128 + lane * 4]);
            const float bb[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
              for (int c = 0; c < 8; ++c) acc[i][c] = bb[c];
#pragma unroll
            for (int d = 0; d < D; ++d) {
              const float4 a0 = *reinterpret_cast<const float4*>(&sm.x[T][d * TM + m0]);
              const float4 a1 = *reinterpret_cast<const float4*>(&sm.x[T][d * TM + m0 + 4]);
              const float4 b0 = *reinterpret_cast<const float4*>(&sm.w1t[d * HID + lane * 4]);
              const float4 b1 = *reinterpret_cast<const float4*>(&sm.w1t[d * HID + 128 + lane * 4]);
              const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
              const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
              for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int c = 0; c < 8; ++c) acc[i][c] = __fmaf_rn(av[i], bv[c], acc[i][c]);
            }
            // h1 row n holds 16 granules of 4 envs; granule g is stored at g ^ ((n>>2)&7).  For unit
            // n = 4*lane+c (or 128+4*lane+c) the key is lane&7, so a warp-wide float4 store touches
            // every bank exactly four times (conflict-free), and a warp's two granules {2w, 2w+1}
            // stay inside one aligned 32-byte pair, so the inner loop still reads them with two
            // warp-broadcast float4 loads at compile-time-known offsets.
            const int key = lane & 7;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
              const int n = (c < 4) ? (lane * 4 + c) : (128 + lane * 4 + (c - 4));
              float* row = &sm.h1[n * TM];
              *reinterpret_cast<float4*>(row + ((2 * warp) ^ key) * 4) =
                  make_float4(fmaxf(acc[0][c], 0.f), fmaxf(acc[1][c], 0.f), fmaxf(acc[2][c], 0.f), fmaxf(acc[3][c], 0.f));
              *reinterpret_cast<float4*>(row + ((2 * warp + 1) ^ key) * 4) =
                  make_float4(fmaxf(acc[4][c], 0.f), fmaxf(acc[5][c], 0.f), fmaxf(acc[6][c], 0.f), fmaxf(acc[7][c], 0.f));
            }
            __syncwarp();     // the activations are consumed by this warp only
          }

          // ---- layer 2: register-tiled SGEMM over K = 256, W2^T chunks from the TMA ring
#pragma unroll
          for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int c = 0; c < 8; ++c) acc[i][c] = 0.f;

          for (int ch = 0; ch < NCHUNK; ++ch, ++g) {
            if (producer) produce(g + PREFETCH);
            const int stg = (int)(g % NSTAGE);
            tc::mbar_wait(&sm.full_bar[stg], (uint32_t)((g / NSTAGE) & 1));
            const float* wb = sm.wc[stg] + lane * 4;
            // swizzle key of hidden unit kg = ch*16 + kk is (kg>>2)&7 = ((ch&1)<<2) | (kk>>2):
            // pair index = warp ^ (key>>1) (runtime, per 8 k's), order inside the pair = key&1 (compile time)
#pragma unroll 1
            for (int half = 0; half < 2; ++half) {
              const float* ha = sm.h1 + (size_t)(ch * KC + half * 8) * TM + ((warp ^ (((ch & 1) << 1) | half)) << 3);
              const float* wh = wb + half * 8 * HID;
#pragma unroll
              for (int kk = 0; kk < 8; ++kk) {
                const float4 lo = *reinterpret_cast<const float4*>(ha + kk * TM);
                const float4 hi = *reinterpret_cast<const float4*>(ha + kk * TM + 4);
                const float4 a0 = ((kk >> 2) & 1) ? hi : lo;     // envs m0..m0+3
                const float4 a1 = ((kk >> 2) & 1) ? lo : hi;     // envs m0+4..m0+7
                const float4 b0 = *reinterpret_cast<const float4*>(wh + kk * HID);
                const float4 b1 = *reinterpret_cast<const float4*>(wh + kk * HID + 128);
                const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
                const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                for (int i = 0; i < 8; ++i)
#pragma unroll
                  for (int c = 0; c < 8; ++c) acc[i][c] = __fmaf_rn(av[i], bv[c], acc[i][c]);
              }
            }
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&sm.empty_bar[stg]);   // this warp is done with the stage
          }

          // ---- bias + ReLU, then layer 3 on the register tile
          {
            const float4 q0 = *reinterpret_cast<const float4*>(&sm.b2[lane * 4]);
            const float4 q1 = *reinterpret_cast<const float4*>(&sm.b2[128 + lane * 4]);
            const float bb[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
              for (int c = 0; c < 8; ++c) acc[i][c] = fmaxf(acc[i][c] + bb[c], 0.f);
          }
          float part[8 * A2];   // index i*A2 + j
#pragma unroll
          for (int j = 0; j < A2; ++j) {
            const float4 w0 = *reinterpret_cast<const float4*>(&sm.w3[j * HID + lane * 4]);
            const float4 w1 = *reinterpret_cast<const float4*>(&sm.w3[j * HID + 128 + lane * 4]);
            const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              float p = 0.f;
#pragma unroll
              for (int c = 0; c < 8; ++c) p = __fmaf_rn(acc[i][c], wv[c], p);
              part[i * A2 + j] = p;
            }
          }
          warp_multi_reduce<8 * A2>(part, lane);
          {
            constexpr int V = 8 * A2;
            if constexpr (V >= 32) {
              constexpr int per = V / 32;
#pragma unroll
              for (int q = 0; q < per; ++q) {
                const int orig = lane * per + q;
                const int i = orig / A2, j = orig % A2;
                sm.out[T][j * TM + warp * 8 + i] = part[q] + sm.b3[j];
              }
            } else {
              constexpr int rep = 32 / V;
              if (lane % rep == 0) {
                const int orig = lane / rep;
                const int i = orig / A2, j = orig % A2;
                sm.out[T][j * TM + warp * 8 + i] = part[0] + sm.b3[j];
              }
            }
          }
          __threadfence_block();
          tc::bar_arrive(BAR_LOGITS + T, NGEMM + TM);   // logits of tile T are in smem
        }
      }
    }
  } else {
    // =========================== env warps ===========================
    const int T = (tid - NGEMM) >> 6;        // tile slot owned by this warp pair
    const int et = (tid - NGEMM) & (TM - 1); // env within the tile
    EpisodeStats epstats;
    for (int64_t pair = blockIdx.x; pair < num_pairs; pair += gridDim.x) {
      const int64_t tile = NTILE * pair + T;
      if (tile >= num_tiles) break;          // CTA-uniform per warp pair; GEMM warps skip this slot too
      const int64_t gi = tile * TM + et;
      const bool owner = gi < st.n;
      EnvRegs<ID> r;
      if (owner) {
        r.load(st, gi);
#pragma unroll
        for (int d = 0; d < D; ++d) sm.x[T][d * TM + et] = r.obs()[d];
      } else {
#pragma unroll
        for (int d = 0; d < D; ++d) sm.x[T][d * TM + et] = 0.f;
      }
      __threadfence_block();
      tc::bar_arrive(BAR_XREADY + T, NGEMM + TM);
      for (int k = 0; k < K; ++k) {
        tc::bar_sync(BAR_LOGITS + T, NGEMM + TM);
        if (owner) {
          const int64_t row = (int64_t)k * st.n + gi;
          float z[4];
          env_noise<A>(z, !deterministic, eps, row, st.seed, st.env_base + (uint64_t)gi, step_base + (uint32_t)k);
          float lg[A2];
#pragma unroll
          for (int j = 0; j < A2; ++j) lg[j] = sm.out[T][j * TM + et];
          env_phase<ID>(r, lg, z, deterministic, actor.min_log_std, actor.max_log_std, st, gi, n_step, reward_scale, cost_scale,
                        out, row, epstats, [&](const float* obs) {
#pragma unroll
            for (int d = 0; d < D; ++d) sm.x[T][d * TM + et] = obs[d];
          });
        }
        if (k + 1 < K) {
          __threadfence_block();
          tc::bar_arrive(BAR_XREADY + T, NGEMM + TM);
        }
      }
      if (owner) r.store(st, gi);
    }
    if (stats) epstats.flush(stats);
  }
}

}  // namespace msacl

using namespace msacl;

extern "C" int msacl_rollout_fused(const msacl_env_state_t* st, const msacl_actor_t* actor, int32_t K,
                                   uint32_t step_base, int32_t n_step, float reward_scale, float cost_scale,
                                   const float* eps, int32_t deterministic, const msacl_transitions_t* out,
                                   double* stats, void* stream) {
  if (!st || !actor || !out || st->n <= 0 || K <= 0 || n_step <= 0) { set_error("rollout_fused: bad argument"); return MSACL_ERR_BAD_ARG; }
  if (!actor->w1 || !actor->b1 || !actor->w2t || !actor->b2 || !actor->w3 || !actor->b3) { set_error("rollout_fused: null actor weights"); return MSACL_ERR_BAD_ARG; }
  if ((reinterpret_cast<uintptr_t>(actor->w2t) & 15) != 0) { set_error("rollout_fused: w2t must be 16-byte aligned"); return MSACL_ERR_BAD_ARG; }
  const int64_t pairs = ((st->n + TM - 1) / TM + NTILE - 1) / NTILE;
  const unsigned grid = (unsigned)(pairs < kNumSMs ? pairs : kNumSMs);
  MSACL_DISPATCH_ENV(st->env_id, {
    if (int rc = check_rollout_outputs<ID>("rollout_fused", st, out)) return rc;
    const size_t smem = sizeof(Smem<ID>);
    auto kern = rollout_fused_kernel<ID>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { set_error("rollout_fused: smem attr: %s", cudaGetErrorString(e)); return MSACL_ERR_CUDA; }
    kern<<<grid, NTHREADS, smem, (cudaStream_t)stream>>>(*st, *actor, K, step_base, n_step, reward_scale, cost_scale,
                                                        eps, deterministic, *out, stats);
  });
  return check_launch("rollout_fused");
}
