/*
 * msacl_b200 -- C ABI of the B200-native MSACL hot path (libmsacl_b200.so).
 *
 * The reference is pure Python and has no FFI; its "plugin API" is duck-typed Python
 * (SURVEY.md section 8b).  Each entry point below therefore names the reference Python
 * function whose arithmetic it replaces; the Python shims in the package
 * (envs.py / sampler.py / buffer.py / targets.py) keep the reference's call signatures and
 * forward to these symbols through ctypes.  INTEGRATION.md shows the binding.
 *
 * Conventions: all pointers are DEVICE pointers into caller-allocated, contiguous buffers
 * (torch tensors) unless noted; nothing is allocated or synchronised inside; every call is
 * stream-ordered on `stream` (a cudaStream_t passed as void*); return value 0 = success,
 * negative = error (message via msacl_last_error()).  There is no CPU fallback.
 */
#ifndef MSACL_B200_H_
#define MSACL_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSACL_ABI_VERSION 3

/* env ids: the fixed table of RL/env/make_env.py:19-32 */
enum {
  MSACL_ENV_VANDERPOL = 0,
  MSACL_ENV_PENDULUM = 1,
  MSACL_ENV_DUCTEDFAN = 2,
  MSACL_ENV_TWOLINK = 3,
  MSACL_ENV_SINGLETRACKCAR = 4,
  MSACL_ENV_QUADTRACKING = 5,
  MSACL_NUM_ENVS = 6
};

enum {
  MSACL_OK = 0,
  MSACL_ERR_BAD_ENV = -1,
  MSACL_ERR_BAD_ARG = -2,
  MSACL_ERR_CUDA = -3
};

/* Structure-of-arrays state of n env instances of one env type on one GPU.
 * sf: float32 [sf_rows][stride]; sd: float64 [sd_rows][stride] (NULL when sd_rows == 0).
 * Row counts / layout per env come from msacl_env_dims(). */
typedef struct {
  int32_t env_id;
  int32_t max_step;      /* time limit (reference: 1000, e.g. RL/env/VanderPol.py:67); <= 0 (msacl_env_step only): bare
                            env semantics -- no time limit, no autoreset, stepping continues from a terminal state */
  int64_t n;             /* env instances on this GPU */
  int64_t stride;        /* row pitch in elements, >= n */
  float* sf;
  double* sd;
  int32_t* step;         /* current_step per env */
  int32_t* episode;      /* index of the current episode per env (keys the reset stream) */
  float* ep_return;      /* running undiscounted return (RecordEpisodeStatistics) */
  int32_t* ep_len;       /* running episode length */
  int32_t* run;          /* n-step deque length, capped at n_step (sampler/base.py:95) */
  uint64_t seed;         /* Philox key */
  uint64_t env_base;     /* global id of local env 0 (multi-GPU sharding) */
} msacl_env_state_t;

/* dims[0]=obs_dim, [1]=act_dim, [2]=sf_rows, [3]=sd_rows, [4]=obs_offset (row of obs[0] in sf),
 * [5]=control_step.  Host call.  Replaces the space probing of RL/utils/init_args.py:33-43. */
int msacl_env_dims(int env_id, int32_t dims[6]);

/* Host call: observation / action boxes, each float[obs_dim] / float[act_dim] HOST arrays
 * (observation_space / action_space of the reference env classes). */
int msacl_env_bounds(int env_id, float* obs_low, float* obs_high, float* act_low, float* act_high);

/* env.reset() for every instance: episode[i] is used as the reset-stream index; step, run,
 * ep_return, ep_len are zeroed.  Replaces <env>.reset (e.g. RL/env/VanderPol.py:69-86,
 * RL/env/QuadTracking.py:152-202) with a Philox-keyed draw of the same distribution. */
int msacl_env_reset(const msacl_env_state_t* st, void* stream);

/* Recompute the QuadTracking hidden desired-frame state and observation from raw x,v,R,Omega
 * already stored in sf (t := 0).  Used to inject initial states (tests, golden vectors). */
int msacl_quad_init_from_raw(const msacl_env_state_t* st, void* stream);

/* One vectorised env step with gymnasium-0.28.1 same-step autoreset.
 * Replaces gymnasium.vector.SyncVectorEnv.step -> <env>.step (RL/env/ *.py::step) as called at
 * RL/trainer/sampler/base.py:148.
 *   action     [n][act_dim] (already clipped by the caller, as the reference does)
 *   next_obs   [n][obs_dim] post-reset observation for done envs
 *   reward     [n] raw env reward (float32)
 *   terminated, truncated [n] (0/1)
 *   final_obs  [n][obs_dim] pre-reset observation (info["final_observation"]) for every env */
int msacl_env_step(const msacl_env_state_t* st, const float* action, float* next_obs, float* reward,
                   uint8_t* terminated, uint8_t* truncated, float* final_obs, void* stream);

/* Actor weights, StochaPolicy (RL/apprfunc/mlp.py:111-136) with hidden sizes [256,256]. */
typedef struct {
  const float* w1;   /* [256][obs_dim]  (torch nn.Linear weight layout) */
  const float* b1;   /* [256] */
  const float* w2t;  /* [256 in][256 out] = W2 transposed */
  const float* b2;   /* [256] */
  const float* w3;   /* [2*act_dim][256] */
  const float* b3;   /* [2*act_dim] */
  float min_log_std; /* -20 */
  float max_log_std; /*   1 */
} msacl_actor_t;

/* Transition outputs of a K-step rollout, each [K][n][...] row-major.  Any pointer may be NULL
 * to skip that field.  obs / obs2 / act are written one row per thread with 16-byte (row length % 4 == 0 floats) or
 * 8-byte (even) vector stores: the pointers must be aligned accordingly (any [t][n][dim] slice of a 16-byte aligned
 * allocation is). */
typedef struct {
  float* obs;     /* [K][n][obs_dim]  observation the action was computed from */
  float* act;     /* [K][n][act_dim]  clipped action */
  float* rew;     /* [K][n]  reward * reward_scale */
  float* cost;    /* [K][n]  sum(real_next_obs^2) * cost_scale */
  float* obs2;    /* [K][n][obs_dim]  real_next_obs (pre-reset) */
  uint8_t* done;  /* [K][n]  terminated | truncated */
  float* logp;    /* [K][n]  log-prob of the sampled action */
  uint8_t* emit;  /* [K][n]  1 iff the env's n-step deque is full after this transition */
  float* logits;  /* [K][n][2*act_dim]  optional diagnostic: the policy MLP output the action was sampled from
                     (mean || log_std BEFORE clamp/exp, i.e. the pre-tanh Gaussian parameters); parity tests assert
                     the tensor-core engine's stated tolerance on it.  Ignored by msacl_window_store. */
} msacl_transitions_t;

/* Fused K-step rollout: actor forward + TanhGauss sample + clip + env step + reward/cost
 * post-processing + autoreset + n-step run bookkeeping, state resident in registers.
 * Replaces K iterations of BaseSampler._n_step (RL/trainer/sampler/base.py:118-163,220) incl.
 * StochaPolicy.forward (mlp.py:132-136), TanhGaussDistribution.sample
 * (act_distribution_cls.py:45-57) and rew_plus_cost (RL/utils/rew_plus_cost.py:18-21).
 *   eps        optional [K][n][act_dim] explicit N(0,1) draws (tests); NULL -> Philox(seed,
 *              env_base+i, step_base+k)
 *   stats      optional double[8], atomically accumulated: [0] finished episodes, [1] sum of their returns,
 *              [2] sum of their lengths, [3] terminated, [4] truncated; [5..7] reserved (not written by release
 *              builds; the MSACL_TC_TIMING debug build uses [5..18] for role timers)
 *   deterministic != 0 -> action = mode() (act_distribution_cls.py:90-95; evaluator path) */
int msacl_rollout_fused(const msacl_env_state_t* st, const msacl_actor_t* actor, int32_t K, uint32_t step_base,
                        int32_t n_step, float reward_scale, float cost_scale, const float* eps,
                        int32_t deterministic, const msacl_transitions_t* out, double* stats, void* stream);

/* Tensor-core variant of msacl_rollout_fused (same contract, same outputs): the two dense actor layers
 * run on tcgen05 UMMA with a split-bf16 ("bf16x3": x1*w1 + x1*w2 + x2*w1) scheme and FP32 accumulation
 * in TMEM; layer 3, sampling and the dynamics stay FP32.  Logits agree with the FP32 path to ~3e-5
 * relative (tolerances in tests/test_gpu_tc.py).  w1p / w2p are the operand images produced by
 * msacl_tc_pack_actor (sizes from msacl_tc_pack_bytes); repack after every weight update.  The w2p buffer is the
 * 256 KB W2 image; msacl_rollout_fused_tc only reads it. */
int msacl_tc_pack_bytes(int64_t* w1p_bytes, int64_t* w2p_bytes);
/* Process-wide grid cap of the persistent tensor-core rollout kernel: 0 (default) = one CTA per SM (148); a smaller value
 * leaves SMs free for a kernel that must run CONCURRENTLY with a rollout launch -- e.g. the NCCL all-gather of the replay
 * sub-batches on a side stream, whose CTAs would otherwise displace rollout CTAs and stretch the launch by the collective's
 * cross-rank wait.  Host call, takes effect at the next launch. */
int msacl_rollout_tc_set_max_ctas(int32_t max_ctas);

/* How msacl_rollout_fused_tc deals its 128-env tiles to the persistent CTAs (host-side arithmetic, no launch; for tests and
 * capacity planning): CTA `cta` of `grid` owns out[1] contiguous tiles starting at tile out[0] and walks them in out[2] rounds
 * of out[3] tiles (+ 1 in the first out[4] rounds), at most 3 tiles (one per env warpgroup) per round.  out = int64[5].
 * Replaces nothing in the reference (its sampler loops over the envs one by one, RL/trainer/sampler/base.py:141-220). */
int msacl_tc_tile_share(int64_t n_envs, int32_t grid, int32_t cta, int64_t* out);
int msacl_tc_pack_actor(const msacl_actor_t* actor, int32_t obs_dim, void* w1p, void* w2p, void* stream);
int msacl_rollout_fused_tc(const msacl_env_state_t* st, const msacl_actor_t* actor, const void* w1p, const void* w2p,
                           int32_t K, uint32_t step_base, int32_t n_step, float reward_scale, float cost_scale,
                           const float* eps, int32_t deterministic, const msacl_transitions_t* out, double* stats,
                           void* stream);

/* One BaseSampler._n_step (RL/trainer/sampler/base.py:118-163,220) for policy outputs computed by the caller: the rollout
 * path for policies the fused kernels are not specialised for (the reference builds MLPs of any depth, width and
 * activation, RL/apprfunc/mlp.py:18-33; the layers are then msacl_gemm_tc calls).
 *   logits [n][2*act_dim] = mean || log_std of StochaPolicy.forward (mlp.py:132-136, before the clamp / exp)
 *   step   = global step index (keys the Philox action-noise stream, like step_base + k of the fused kernels)
 *   out    = pointers to the [n][.] slices of THIS step; eps [n][act_dim] optional explicit N(0,1) draws
 * Sampling, clip, env step, reward / cost scaling, same-step autoreset, episode statistics and n-step run / emit
 * bookkeeping are those of msacl_rollout_fused (same arithmetic, same random streams). */
int msacl_rollout_step(const msacl_env_state_t* st, const float* logits, float min_log_std, float max_log_std, uint32_t step,
                       int32_t n_step, float reward_scale, float cost_scale, const float* eps, int32_t deterministic,
                       const msacl_transitions_t* out, double* stats, void* stream);

/* Diagnostic: out[i] = NormalizeOrientMatrix(in[i]) for n row-major 3x3 float32 matrices through the device polar
 * routine of the QuadTracking step (RL/env/QuadTracking.py:308-315), including its det < 0 branch (:312-314), which the
 * dynamics cannot reach.  theta2 = (h |Omega|)^2 hint (>= 0.02 -> a third Newton sweep). */
int msacl_selftest_quad_polar(const float* in, float* out, int64_t n, float theta2, void* stream);

/* Fill out[n][act_dim] with the N(0,1) draws the rollout uses at global step `step`. */
int msacl_action_noise(uint64_t seed, uint64_t env_base, int64_t n, int32_t act_dim, uint32_t step, float* out,
                       void* stream);

/* n-step replay ring, arrays [max_size][n_step][...] as RL/trainer/buffer/nstep_replay_buffer.py:52-67 */
typedef struct {
  int64_t max_size;
  int32_t n_step, obs_dim, act_dim;
  float* obs; float* act; float* rew; float* cost; float* obs2; float* done; float* logp;
} msacl_ring_t;

/* Assemble every emitted n-step window of a rollout chunk and store it in the ring in the
 * reference's order (step-major, env-minor) starting at *ptr.  Replaces the deque logic of
 * RL/trainer/sampler/base.py:178-217 plus NstepReplayBuffer.add_batch/store
 * (nstep_replay_buffer.py:91-125).
 *   tr        transitions of H + K steps: the first H = n_step-1 slices are the tail of the
 *             previous chunk (history), the last K are new; emit flags of history are ignored
 *   scratch   int64[msacl_window_store_scratch_elems(K, n)] device scratch (= 2 + ceil(K*n/256): a two-word
 *             header and one count per block of 256 emit flags)
 *   ptr_size  device int64[2] = {ptr, size}, updated in place
 *   count_out device int64[1]: number of windows stored by this call */
int64_t msacl_window_store_scratch_elems(int32_t K, int64_t n);
int msacl_window_store(const msacl_transitions_t* tr, int32_t H, int32_t K, int64_t n, const msacl_ring_t* ring,
                       int64_t* ptr_size, int64_t* count_out, int64_t* scratch, void* stream);

/* batch[k] = ring[idx[k]] for all 7 fields ([B][n_step][...]); replaces
 * NstepReplayBuffer.sample_batch's gather (nstep_replay_buffer.py:138-146). */
int msacl_ring_gather(const msacl_ring_t* ring, const int64_t* idx, int64_t B, const msacl_ring_t* batch,
                      void* stream);

/* Index-based n-step window store (SURVEY.md 8f-1): instead of copying every emitted window into a
 * [max_size][n_step][.] ring (2 * 4 * n_step * (2D + A + 4) bytes of traffic per window), only the flat position
 * (slice * n + env) of the window's NEWEST transition inside the caller's [T][n][.] transition store is appended to
 * an int64 ring `win_pos[max_size]`, in the reference's append order and with the reference's ptr / size arithmetic
 * (RL/trainer/sampler/base.py:178-217, nstep_replay_buffer.py:106-119); the n_step rows are gathered when a batch is
 * sampled (nstep_replay_buffer.py:138-146).  The caller keeps the n_step - 1 slices in front of a window's newest slice
 * contiguous in the store and retires windows before their slices are overwritten (buffer.B200IndexedReplayBuffer).
 *   emit_new  [K][n] emit flags of the K new slices;  base_pos = flat position of emit_new[0][0] in the store
 *   scratch   int64[msacl_window_store_scratch_elems(K, n)] */
int msacl_window_index_store(const uint8_t* emit_new, int32_t K, int64_t n, int64_t base_pos, int64_t* win_pos,
                             int64_t max_size, int64_t* ptr_size, int64_t* count_out, int64_t* scratch, void* stream);
/* batch[b] = the window whose newest transition sits at store position win_pos[idx[b]]: rows
 * pos - (n_step-1-r)*n, r = 0..n_step-1, of every field (done: uint8 -> 0.0/1.0 float), written as [B][n_step][.].
 * tr: base pointers of the whole [T][n][.] store (emit / logits unused). */
int msacl_window_gather_indexed(const msacl_transitions_t* tr, int64_t n, const int64_t* win_pos, const int64_t* idx,
                                int64_t B, const msacl_ring_t* batch, void* stream);

/* NstepReplayBuffer.sample_batch (nstep_replay_buffer.py:138-146) of the reference-layout ring: idx[b] ~ U{0..size-1} drawn on
 * the device (Philox keyed by (seed, draw, b); size = ptr_size[1] read on the device), then msacl_ring_gather.
 *   idx  device int64[B], receives the drawn slots */
int msacl_ring_sample(const msacl_ring_t* ring, const int64_t* ptr_size, uint64_t seed, uint64_t draw, int64_t B,
                      const msacl_ring_t* batch, int64_t* idx, void* stream);

/* NstepReplayBuffer.sample_batch (nstep_replay_buffer.py:138-146) of the index-based store in one launch, without a host
 * read of the counters: window b of the batch is drawn uniformly (with replacement) from the `valid` most recent ring
 * entries, valid = min(ptr_size[1], sum of launch_counts[0..n_counts)) -- the windows whose slices are still resident --
 * with a Philox4x32-10 draw keyed by (seed, draw, b), and gathered like msacl_window_gather_indexed.
 *   ptr_size       device int64[2] as maintained by msacl_window_index_store
 *   launch_counts  device int64[n_counts]: windows emitted by each of the launches that are still resident
 *   slots_out      optional device int64[B]: the ring slots that were drawn
 * valid == 0 leaves the batch untouched. */
int msacl_window_sample_indexed(const msacl_transitions_t* tr, int64_t n, const int64_t* win_pos, int64_t max_size,
                                const int64_t* ptr_size, const int64_t* launch_counts, int32_t n_counts, uint64_t seed,
                                uint64_t draw, int64_t B, const msacl_ring_t* batch, int64_t* slots_out, void* stream);

/* MSACL soft-TD backup (RL/algorithm/msacl.py:249-252), elementwise over B*n. */
int msacl_q_backup(int64_t count, const float* rew, const float* done, const float* next_q1, const float* next_q2,
                   const float* next_logp, float gamma, float alpha, float* backup, void* stream);

/* Lyapunov risk forward + analytic backward (RL/algorithm/msacl.py:280-329).
 *   obs, obs2 [B][n][D]; logp_new, logp_old, lya_obs, lya_obs2 [B][n]
 *   coef_son / coef_diff / coef_sl: float[n] device (msacl.py:153-164)
 *   loss_parts double[3] device, zeroed by the call: sum relu(a1|o|^2-V), sum relu(V-a2|o|^2),
 *              sum_b sum_k lambda_k c_k relu(ESL (V(o2_k) - (1-eta)^(k+1) V(o_0)))
 *   grad_lya_obs, grad_lya_obs2 [B][n]: d loss / d V  (loss = (p0+p1)/(B n) * pos_scale + p2/B * diff_scale)
 *   is_clip, esl optional [B][n] outputs */
int msacl_lyapunov_risk(int64_t B, int32_t n, int32_t D, const float* obs, const float* obs2, const float* logp_new,
                        const float* logp_old, const float* lya_obs, const float* lya_obs2, const float* coef_son,
                        const float* coef_diff, const float* coef_sl, float alpha1, float alpha2, float diff_scale,
                        float pos_scale, double* loss_parts, float* grad_lya_obs, float* grad_lya_obs2,
                        float* is_clip, float* esl, void* stream);

/* Stability advantage (RL/algorithm/msacl.py:392-400): adv_raw[b] = sum_k lambda_k ((1-eta)^(k+1) V(o_0) - V(o2_k));
 * moments double[2] device (zeroed by the call) receive sum and sum of squares for the batch
 * normalisation, which msacl_advantage_normalize applies (unbiased std + 1e-8). */
int msacl_stability_advantage(int64_t B, int32_t n, const float* lya_obs0, const float* lya_obs2,
                              const float* coef_diff, const float* coef_sl, float* adv_raw, double* moments,
                              void* stream);
int msacl_advantage_normalize(int64_t B, const float* adv_raw, const double* moments, float* adv, void* stream);

/* Soft target update of a whole parameter list in one launch (RL/algorithm/msacl.py:445-460):
 * dst[t][i] = dst[t][i] * polyak + one_minus * src[t][i] for t < count, i < numel[t], with the reference's three
 * float32 roundings (bit-exact with `p_targ.mul_(polyak); p_targ.add_((1 - polyak) * p)`).
 * src / dst / numel are DEVICE arrays (pointer tables of length count); max_numel = max_t numel[t] sizes the grid. */
int msacl_polyak_update(int32_t count, const float* const* src, float* const* dst, const int64_t* numel,
                        int64_t max_numel, float polyak, float one_minus, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Learner networks and update (RL/apprfunc/mlp.py:18-52,72-88,111-136; RL/algorithm/msacl.py:227-460;
 * RL/utils/act_distribution_cls.py:59-84).  With these entry points a whole MSACL.model_update runs as a fixed
 * sequence of launches without autograd: dense layers forward / backward on the tcgen05 tensor cores, every scalar
 * (alpha, losses, entropy) resident on the device.
 * --------------------------------------------------------------------------------------------------------------- */

/* One dense layer, forward or backward, as a split-bf16 tcgen05 GEMM with a fused epilogue:
 *     C[r][n] = epilogue( sum_k A(r,k) * B(n,k) ),   A(r,k) = a[r*a_row_stride + k*a_k_stride],  B likewise (FP32, device)
 *   forward  (mlp.py:18-33)  H = act(X W^T + b):       a = X [rows][in], b = W [out][in] (nn.Linear layout), bias, act
 *   dgrad                    dX = (dY W) * act'(Xpost): a = dY, B(n,k) = W[k][n] (b_row_stride 1, b_k_stride in), mask_src = Xpost
 *   wgrad                    dW = dY^T X:              A(r,k) = dY[k][r], B(n,k) = X[k][n], k = rows, split_k partials
 * act / mask_act: 0 none, 1 relu, 2 tanh.  mask_src holds POST-activation values (relu' = [h > 0], tanh' = 1 - h^2).
 * split_k > 1: split z writes its partial product to c + z * c_split_stride (no epilogue allowed); the consumer
 * (msacl_adam_multi / msacl_reduce_splits) adds the partials in a fixed order.
 * row_sumsq: optional [m], receives sum_n C[r][n]^2 (LyapunovValue.forward, mlp.py:86-88); needs n <= 256. */
typedef struct {
  const float* a; int64_t a_row_stride, a_k_stride;
  const float* b; int64_t b_row_stride, b_k_stride;
  int32_t m, n, k;
  float* c; int64_t ldc;
  int32_t split_k; int64_t c_split_stride;
  const float* bias;
  int32_t act;
  const float* mask_src; int64_t mask_ld; int32_t mask_act;
  float* row_sumsq;
  int32_t precision;   /* bf16 products per algorithmic product: 6 (or 0 = default; 3-term operand split, FP32-class ~2^-23)
                          or 3 (2-term split, ~1.5e-5 relative per product, half the tensor work) */
  const void* b_packed; /* optional: the B operand pre-converted by msacl_gemm_pack_b (same b / strides / n / k / precision);
                          the launch then takes 256-wide column tiles and the B stages are streamed by bulk copies instead
                          of being re-converted from `b` in every CTA.  `b` must still be valid. */
} msacl_gemm_t;
int msacl_gemm_tc(const msacl_gemm_t* g, void* stream);
/* Pre-convert the B operand described by g (b, b_row_stride, b_k_stride, n <= 256, k, precision) into the kernel's
 * shared-memory stage images; `packed` = device buffer of msacl_gemm_packed_b_bytes(k, precision) bytes, 16-byte aligned.
 * Repack whenever the weights change (tiny: one thread per 8 elements). */
int64_t msacl_gemm_packed_b_bytes(int32_t k, int32_t precision);
int msacl_gemm_pack_b(const msacl_gemm_t* g, void* packed, void* stream);

/* out[z][c] = sum over the rows of split z (rows divided evenly over `splits`) of x[r*ld + c].  Bias gradients. */
int msacl_colsum(const float* x, int64_t rows, int32_t cols, int64_t ld, int32_t splits, float* out, void* stream);
/* out[r] = [a[r] | b[r]]  (ActionValue input, mlp.py:50-52) */
int msacl_concat2(const float* a, int32_t da, const float* b, int32_t db, int64_t rows, float* out, void* stream);
/* out[i] = sum_z parts[z*numel + i], z ascending */
int msacl_reduce_splits(const float* parts, int64_t numel, int32_t nsplit, float* out, void* stream);

/* TanhGaussDistribution on logits = [mean || log_std] rows [rows][2*act_dim] (StochaPolicy output BEFORE clamp / exp,
 * mlp.py:132-136); act_low / act_high: device float[act_dim].
 *   rsample  (act_distribution_cls.py:59-71) with explicit N(0,1) draws eps [rows][act_dim] -> act, logp
 *   log_prob (act_distribution_cls.py:73-84) of given (limited) actions -> logp
 *   log_prob_bwd: grad_logits[r] (+)= grad_logp[r] * d logp / d logits  (the clamp of log_std passes gradients inside its range) */
int msacl_tanh_gauss_rsample(int64_t rows, int32_t act_dim, const float* logits, const float* eps, const float* act_low,
                             const float* act_high, float min_log_std, float max_log_std, float* act, float* logp, void* stream);
int msacl_tanh_gauss_log_prob(int64_t rows, int32_t act_dim, const float* logits, const float* act, const float* act_low,
                              const float* act_high, float min_log_std, float max_log_std, float* logp, void* stream);
int msacl_tanh_gauss_log_prob_bwd(int64_t rows, int32_t act_dim, const float* logits, const float* act, const float* act_low,
                                  const float* act_high, float min_log_std, float max_log_std, const float* grad_logp,
                                  int32_t accumulate, float* grad_logits, void* stream);

/* msacl_q_backup with alpha = exp(*log_alpha) read on the device (no host synchronisation; msacl.py:249-252,339-346). */
int msacl_q_backup_dev_alpha(int64_t count, const float* rew, const float* done, const float* next_q1, const float* next_q2,
                             const float* next_logp, float gamma, const float* log_alpha, float* backup, void* stream);
/* Critic loss (msacl.py:254-257): dq{1,2} = 2 (q - backup) / count; sums (device double[4], zeroed by the call) receive
 * sum (q1-y)^2, sum (q2-y)^2, sum q1, sum q2. */
int msacl_q_loss_grad(int64_t count, const float* q1, const float* q2, const float* backup, float* dq1, float* dq2, double* sums,
                      void* stream);
/* LyapunovValue backward through V = sum_j z_j^2: dz[r][j] = 2 z[r][j] dv[r] */
int msacl_sumsq_bwd(int64_t rows, int32_t cols, const float* z, const float* dv, float* dz, void* stream);
/* Policy update (msacl.py:349-411), loss_policy = -mean(min(Q1,Q2)(obs, a_new) - alpha logp_new) - L_lya.
 *   policy_q_route: d loss / d q1, q2 (torch.min routing) and sums (device double[3], zeroed by the call):
 *                   [0] sum (min_q - alpha logp_new), [1] sum logp_new
 *   policy_logits_grad: d loss / d logits through (a) the critics' input gradients dxq{1,2} [rows][obs_dim+act_dim]
 *                   (action columns) and the reparameterised tanh sample, (b) the entropy term, (c) the clipped
 *                   stability-advantage surrogate on the first step of every window (adv: normalised advantage [rows/n_step]);
 *                   sums[2] += sum_b min(surr1, surr2) */
int msacl_policy_q_route(int64_t rows, const float* q1, const float* q2, const float* logp_new, const float* log_alpha, float* dq1,
                         float* dq2, double* sums, void* stream);
int msacl_policy_logits_grad(int64_t rows, int32_t n_step, int32_t obs_dim, int32_t act_dim, const float* logits, const float* eps,
                             const float* dxq1, const float* dxq2, const float* log_alpha, const float* old_act,
                             const float* old_logp, const float* adv, float clip_coef, const float* act_low, const float* act_high,
                             float min_log_std, float max_log_std, float* grad_logits, double* sums, void* stream);
/* Entropy coefficient (msacl.py:425-438): entropy = -sums[1] / rows; one Adam step on log_alpha with gradient
 * exp(log_alpha) (entropy - target_entropy); adam_state = device float[2] {exp_avg, exp_avg_sq}; clamp_max = log(alpha_bound) or +inf. */
int msacl_alpha_update(float* log_alpha, const double* sums, int64_t rows, float target_entropy, float* adam_state,
                       float one_minus_beta1, float beta2, float one_minus_beta2, float step_size, float bc2_sqrt, float eps,
                       float clamp_max, float* entropy_out, const float* dyn, void* stream);
/* torch.optim.Adam step (defaults: no weight decay, no amsgrad) over a whole parameter list in one launch.  params / grads /
 * exp_avg / exp_avg_sq: DEVICE pointer tables of length count; grads[t] holds nsplit[t] partial gradients of numel[t]
 * elements each, summed in order.  step_size = lr / (1 - beta1^step), bc2_sqrt = sqrt(1 - beta2^step) (host, float64 -> float32). */
int msacl_adam_multi(int32_t count, float* const* params, const float* const* grads, float* const* exp_avg, float* const* exp_avg_sq,
                     const int64_t* numel, const int32_t* nsplit, int64_t max_numel, float one_minus_beta1, float beta2,
                     float one_minus_beta2, float step_size, float bc2_sqrt, float eps, const float* dyn, void* stream);
/* Adam bias-correction scalars on the device: *step += 1; dyn[0] = lr / (1 - beta1^step), dyn[1] = sqrt(1 - beta2^step)
 * (float64 arithmetic, as torch on the host).  msacl_adam_multi / msacl_alpha_update read step_size / bc2_sqrt from `dyn`
 * (device float[2]) when it is non-NULL, so a captured CUDA graph of the whole update advances correctly on every replay. */
int msacl_adam_tick(int32_t* step, float* dyn, double lr, double beta1, double beta2, void* stream);

/* Device FP32 FFMA peak probes used by bench.py for the roofline denominator.
 * mode 0: independent FFMA chains with immediate operands (pipe peak);
 * mode 1: register-resident 8x8 outer-product accumulation, i.e. a register-tiled SGEMM inner
 *         loop with no memory traffic (three-register FFMA ceiling);
 * mode 2: the same outer product with packed FFMA2 (fma.rn.f32x2);
 * mode 3: FP64 DFMA throughput at full occupancy;
 * modes 4-6: separate DMUL / DADD issued by ONE warp per SM sub-partition with 8 / 2 / 1 independent chains per thread
 *         (*flops then returns the FP64 instructions issued per warp): the FP64 issue rate the fused rollout's env phase sees;
 * mode 7: float32 <-> float64 round trips (two conversions + one DMUL each; *flops = round trips per warp);
 * mode 8: the mode-1 outer product with directed rounding (half FFMA.RM, half FFMA.RP), the interval GEMM ceiling.
 * sink: device float[128] (sink[64..128) is read as operand source in mode 1).
 * Returns the FLOPs issued in *flops (host). */
int msacl_ffma_probe(int32_t mode, int32_t iters, float* sink, double* flops, void* stream);

/* Diagnostic: D[128][256] = A[128][256] * W[256][256]^T on the tcgen05 tensor cores with the
 * split-bf16 scheme (splits = 1: plain bf16; 3: a1*b1 + a1*b2 + a2*b1), FP32 accumulation in TMEM.
 * Exercises the descriptor / TMEM plumbing of the tensor-core rollout path. */
int msacl_selftest_tc_gemm(const float* A, const float* W, float* D, int32_t splits, void* stream);

/* Diagnostic: average cycles per 128x256x16 bf16 UMMA when one thread per SM issues `iters` groups of three
 * back to back from no-swizzle K-major shared-memory operands (mode 0), or while the CTA's other warps
 * stream 16-byte shared-memory stores (mode 1) or tcgen05.ld reads of other TMEM columns (mode 2; the aggregate
 * read rate in bytes/cycle is returned in cycles_per_umma[1]); mode 3: a tcgen05.commit per group; mode 4: plus an
 * mbarrier wait per group.  cycles_per_umma: device double[4]. */
int msacl_umma_probe(int32_t mode, int32_t iters, double* cycles_per_umma, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Lyapunov-certificate verifier (no counterpart in the reference).  For every initial state i the caller runs the greedy
 * closed loop for up to `horizon` steps (msacl_rollout_fused* with deterministic = 1, n_step = 1, max_step > horizon) and
 * evaluates V = networks.lyapunov on the visited observations; these entry points check, per visited state k = 0..e
 * (e = the first step whose `done` is set, else horizon), with s_k = sum_j o_k[j]^2 accumulated in float64 in order j = 0..D-1,
 * c_k = decay[k] and every comparison in float64:
 *   NONFINITE       some o_k[j] or V_k is NaN / Inf
 *   BOUND_LO        V_k < alpha1 s_k - v_atol              BOUND_HI  V_k > alpha2 s_k + v_atol
 *   DECREASE        k >= 1 and V_k > c_k V_0 + v_atol       ESCAPED   done at some step k <= horizon
 *   NOT_EXP_STABLE  k >= 1 and s_k > (alpha2 / alpha1) c_k s_0   (model-free; independent of V)
 * A state is certified when it has none of the first five.  An empirical check over the sampled states and horizon, not
 * a proof.  Records are per state, structure-of-arrays, streamed chunk by chunk: memory is O(n), not O(n * horizon).
 * --------------------------------------------------------------------------------------------------------------- */
enum {
  MSACL_CERT_NONFINITE = 1,
  MSACL_CERT_BOUND_LO = 2,
  MSACL_CERT_BOUND_HI = 4,
  MSACL_CERT_DECREASE = 8,
  MSACL_CERT_ESCAPED = 16,
  MSACL_CERT_NOT_EXP_STABLE = 32,
  MSACL_CERT_FAIL_MASK = 31,          /* flags that make a state uncertified */
  MSACL_CERT_MAX_HORIZON = 8192
};

/* Layout of the int64 summary written by msacl_certify_finish / msacl_certify_roa: [MSACL_CERT_SUM_HIST + horizon] */
enum {
  MSACL_CERT_SUM_STATES = 0,          /* n */
  MSACL_CERT_SUM_FLAGS = 1,           /* [1 + b] = states with flag bit b set, b = 0..5 */
  MSACL_CERT_SUM_CERTIFIED = 7,
  MSACL_CERT_SUM_INCONSISTENT = 8,    /* states where DECREASE and NOT_EXP_STABLE disagree */
  MSACL_CERT_SUM_CSTAR_KEY = 9,       /* min V_0 over uncertified states with V_0 not NaN, as the order-preserving key of its
                                         float32 bits (bits | 0x80000000 for sign 0, ~bits for sign 1); +inf if none */
  MSACL_CERT_SUM_ROA = 10,            /* #{i : V_0,i < c_star} (msacl_certify_roa) */
  MSACL_CERT_SUM_HIST = 11            /* [11 + k - 1] = states whose first DECREASE is at step k, k = 1..horizon */
};

typedef struct {
  int32_t horizon;         /* T, 1..MSACL_CERT_MAX_HORIZON; steps k > T are ignored */
  double alpha1, alpha2;   /* > 0 */
  double v_atol;           /* >= 0, absolute slack on V */
  const double* decay;     /* device double[T + 1]: c_0 = 1, c_k = c_{k-1} (1 - eta) (repeated multiplication) */
} msacl_cert_params_t;

/* Per-state records, device arrays [n] */
typedef struct {
  float* v0;               /* V(o_0) */
  double* s0;              /* s_0 */
  uint8_t* flags;          /* MSACL_CERT_* bits */
  int32_t* first_violation;/* first k at which a flag of MSACL_CERT_FAIL_MASK was raised, -1 if none */
  int32_t* first_decrease; /* first k with DECREASE, -1 if none */
  int32_t* end_step;       /* e */
  double* worst_ratio;     /* max_{1<=k<=e} V_k / (c_k V_0); 0/0 = 0, x/0 = +inf for x > 0, NaN terms skipped; 0 if e = 0 */
} msacl_cert_records_t;

/* Box initial states: o_i[j] = lo[j] + (hi[j] - lo[j]) u (float32), u = top 24 bits of Philox4x32-10 word 0 for the counter
 * (env_base + i, j, 0x63657274) under key st->seed, written into the sf rows of the five box envs (state == observation).
 * lo / hi: HOST float[obs_dim], lo <= hi.  Call after msacl_env_reset (which zeroes the step counters). */
int msacl_certify_box_init(const msacl_env_state_t* st, const float* lo, const float* hi, void* stream);
/* Initialise the records from the initial observations obs0 [n][obs_dim] and v0 [n] (checks of k = 0). */
int msacl_certify_begin(int64_t n, int32_t obs_dim, const float* obs0, const float* v0, const msacl_cert_params_t* p,
                        const msacl_cert_records_t* rec, void* stream);
/* One rollout chunk of K steps k0 .. k0 + K - 1 (k0 >= 1) in the transition-store layout: obs2 [K][n][obs_dim] (the real
 * next observation), v [K][n] = V(obs2), done [K][n].  States that already ended are skipped; obs2 rows are read with
 * 16-byte (obs_dim % 4 == 0) or 8-byte (even) vector loads and must be aligned accordingly. */
int msacl_certify_steps(int64_t n, int32_t obs_dim, int32_t K, int32_t k0, const float* obs2, const float* v, const uint8_t* done,
                        const msacl_cert_params_t* p, const msacl_cert_records_t* rec, void* stream);
/* Reduce the records into summary (zeroed by the call except [MSACL_CERT_SUM_ROA]): counts, first-DECREASE histogram and
 * the c_star key.  One atomic per block and counter. */
int msacl_certify_finish(int64_t n, int32_t horizon, const msacl_cert_records_t* rec, int64_t* summary, void* stream);
/* summary[MSACL_CERT_SUM_ROA] = #{i < n : v0[i] < c_star} (zeroed by the call). */
int msacl_certify_roa(int64_t n, const float* v0, float c_star, int64_t* summary, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Region verifier of the Lyapunov certificate (no counterpart in the reference): interval branch-and-bound over state boxes.
 * For a box X0, an inner box B, eta, alpha1, alpha2 and m >= 1 closed-loop steps it partitions X0 \ B into dyadic cells and
 * proves per cell C, with outward-rounded interval arithmetic:
 *   DECREASE ok  sup V(F^m(C)) <= (1 - eta)^m inf V(C)
 *   ESCAPED ok   F^j(C) lies strictly inside the env's observation bounds for j = 1..m (the env cannot terminate)
 *   BOUND ok     alpha1 sup |x|^2 <= inf V(C) and sup V(C) <= alpha2 inf |x|^2 over C
 *   NONFINITE    some bound overflowed or is NaN; such a cell is never verified
 * F is one greedy closed-loop step: policy mean mu, a = half tanh(mu) + mid, clip to the action box, CONTROL_STEP
 * explicit-Euler sub-steps.  The verified object is the REAL-ARITHMETIC closed loop: the networks as exact real functions of
 * their stored float32 parameters, exact sin / cos / tanh, the Euler map in exact arithmetic (the env's constants read as
 * exact reals).  The rounding of any float implementation (split-bf16 rollout GEMMs, float32 env kernels) is not modelled.
 * Envs: VanderPol, Pendulum, DuctedFan, TwoLink.
 *
 * Bounded disturbances (msacl_region_params_t.dist): one disturbed closed-loop step is
 *   F_d(x) = Phi(x, clip(half tanh(mu(x + n)) + mid) + u) + w,   n in N, u in U, w in W
 * with Phi the CONTROL_STEP Euler map.  n is sensor noise seen by the policy only (V is evaluated at the true state); u is an
 * actuator disturbance added after the clip, not re-clipped, and held over the sub-steps; w is a process disturbance added
 * once after the sub-steps.  N, U, W are boxes (need not contain 0), and each of the m steps takes its own (n, u, w): every
 * condition above, LEAVES, the inner-cell conditions and c_in hold for EVERY admissible disturbance sequence.  A REFUTE flag
 * still evaluates the degenerate [c, c] with the sets as intervals, so its violation holds for every sequence and its margin
 * is the least violation over them.  A set that is exactly {0} is skipped, so an all-zero dist is the nominal closed loop F,
 * bit for bit.
 * --------------------------------------------------------------------------------------------------------------- */
enum {
  MSACL_REGION_NONFINITE = 1,         /* cell flags (msacl_region_out_t.flags) */
  MSACL_REGION_DECREASE = 2,          /* DECREASE not proven */
  MSACL_REGION_ESCAPED = 4,           /* ESCAPED not proven */
  MSACL_REGION_BOUND = 8,             /* BOUND not proven */
  MSACL_REGION_LEAVES = 16,           /* F^m(C) not proven inside X0 */
  MSACL_REGION_REFUTE_DECREASE = 32,  /* proven: inf V(F^m(C)) > (1 - eta)^m sup V(C), i.e. every point of C violates DECREASE */
  MSACL_REGION_REFUTE_ESCAPED = 64,   /* proven: some F^j(C), j <= m, lies entirely outside the observation bounds */
  MSACL_REGION_HIDDEN = 256,          /* network width of the kernels (narrower layers are zero-padded) */
  MSACL_REGION_MAX_DEPTH = 50
};

/* cell status written by msacl_region_round (msacl_region_ws_t.status) */
enum { MSACL_REGION_SPLIT = 0, MSACL_REGION_VERIFIED = 1, MSACL_REGION_REFUTED = 2, MSACL_REGION_UNDECIDED = 3, MSACL_REGION_INNER = 4 };

/* int64 statistics accumulated by msacl_region_round; volumes in units of 2^-50 of X0; keys are order keys of float32
 * (MSACL_CERT_SUM_CSTAR_KEY): C_SOUND min (init +inf), C_IN / V_INNER max (init -inf) */
enum {
  MSACL_REGION_ST_VERIFIED = 0, MSACL_REGION_ST_REFUTED = 1, MSACL_REGION_ST_UNDECIDED = 2, MSACL_REGION_ST_INNER = 3,
  MSACL_REGION_ST_SPLIT = 4, MSACL_REGION_ST_EVALUATED = 5, MSACL_REGION_ST_PROBED = 6,
  MSACL_REGION_ST_FLAGS = 7,          /* [7 + b]: non-inner leaf cells with flag bit b (NONFINITE .. LEAVES) */
  MSACL_REGION_ST_VOLUME = 12,        /* [12 + s]: volume of VERIFIED, REFUTED, UNDECIDED, INNER leaves */
  MSACL_REGION_ST_C_SOUND = 16,       /* min inf V(C) over non-inner leaves that are not verified or whose F^m(C) may leave X0 */
  MSACL_REGION_ST_C_IN = 17,          /* max sup V(F^m(C)) over inner leaves */
  MSACL_REGION_ST_V_INNER = 18,       /* max sup V(C) over inner leaves */
  MSACL_REGION_ST_INNER_FAIL = 19,    /* inner leaves that are NONFINITE, ESCAPED or LEAVES */
  MSACL_REGION_ST_COUNT = 20
};

typedef struct {
  int32_t env_id, obs_dim, act_dim;
  int32_t p_h1, p_h2;                 /* policy obs -> p_h1 -> p_h2 -> 2 act_dim, ReLU, torch Linear layout [out][in] */
  const float *p_w1, *p_b1, *p_w2, *p_b2, *p_w3, *p_b3;
  int32_t v_h1, v_h2, v_out;          /* V net obs -> v_h1 -> v_h2 -> v_out (<= 256 each), V = sum z^2 */
  const float *v_w1, *v_b1, *v_w2, *v_b2, *v_w3, *v_b3;
} msacl_region_nets_t;

typedef struct {                      /* disturbance boxes [lo, hi] (finite, lo <= hi); all zero: no disturbance */
  float obs_lo[16], obs_hi[16];       /* N, [obs_dim]: sensor noise added to the policy's input */
  float act_lo[2], act_hi[2];         /* U, [act_dim]: actuator disturbance added to the clipped action */
  float state_lo[16], state_hi[16];   /* W, [obs_dim]: process disturbance added to the state after the Euler sub-steps */
} msacl_region_disturbance_t;

typedef struct {
  int32_t env_id, steps;              /* m >= 1 */
  int32_t v_tanh;                     /* V hidden activation: 0 ReLU, 1 tanh */
  double decay_lo, decay_hi;          /* (1 - eta)^m rounded down / up */
  double alpha1, alpha2;
  float x0_lo[16], x0_hi[16];         /* X0 */
  msacl_region_disturbance_t dist;    /* N, U, W (see above); all zero: the nominal loop */
} msacl_region_params_t;

typedef struct {                      /* per cell outputs of msacl_region_eval, [n] unless noted */
  float *v_lo, *v_hi;                 /* inf / sup V(C) */
  float *vm_lo, *vm_hi;               /* inf / sup V(F^m(C)) */
  float *img_lo, *img_hi;             /* [n][obs_dim] box of F^m(C) */
  uint8_t* flags;                     /* MSACL_REGION_* cell flags */
  float* margin;                      /* proven violation of a REFUTE flag (decrease first), else 0 */
  float* trace;                       /* optional [n][steps][4 act_dim + 2 obs_dim]: mu lo, mu hi, a lo, a hi, F^j lo, F^j hi */
} msacl_region_out_t;

typedef struct {
  int32_t max_depth;                  /* 1..MSACL_REGION_MAX_DEPTH; depth t bisects dimension t mod obs_dim */
  int32_t inner_level;                /* B is snapped outward to the grid of 2^inner_level cells per dimension */
  uint32_t inner_lo[16], inner_hi[16];/* B = X0_lo + (X0_hi - X0_lo) [inner_lo, inner_hi] / 2^inner_level per dimension */
  double inner_box_lo[16], inner_box_hi[16];   /* the snapped B in coordinates, rounded outward */
  int64_t max_examples;               /* capacity of the counterexample list */
} msacl_region_bnb_t;

typedef struct {                      /* scratch of one msacl_region_round for k cells (device arrays) */
  uint32_t* cells;                    /* [k][1 + obs_dim] copy of the popped cells */
  float *lo, *hi;                     /* [k][obs_dim] their boxes */
  msacl_region_out_t res;             /* [k] their evaluation (trace unused) */
  float *plo, *phi;                   /* [k][obs_dim] centres probed for refutation */
  msacl_region_out_t pres;            /* [k] evaluation of the centres */
  int32_t* probe;                     /* [k] probe slot of cell i, -1 if none */
  uint8_t* status;                    /* [k] MSACL_REGION_SPLIT .. INNER */
  int64_t* scan;                      /* [3 * (k / 256 + 1) + 8] */
} msacl_region_ws_t;

/* Bytes of the packed network image (floats, 16-byte aligned). */
int64_t msacl_region_image_bytes(void);
/* Pack the policy and V net into the image: zero-padded to 256 units, the 256-wide matrices as [k][W+ | W-] rows. */
int msacl_region_pack(const msacl_region_nets_t* nets, float* image, void* stream);
/* Enclose F (F_d under p->dist), V and the cell conditions for the n boxes [lo, hi] ([n][obs_dim], float32); n is *n_dev
 * when n_dev != NULL (n is then an upper bound).  The trace's a and F^j are the disturbed action and state.  One persistent
 * CTA per SM, FP32 FFMA.RM / FFMA.RP interval GEMMs.  MSACL_ERR_BAD_ARG for a non-finite disturbance bound or lo > hi. */
int msacl_region_eval(const msacl_region_params_t* p, const float* image, int64_t n, const int64_t* n_dev, const float* lo,
                      const float* hi, const msacl_region_out_t* out, void* stream);
/* One branch-and-bound round over the k cells stack[top - k, top) (cell = [depth, idx_0 .. idx_{obs_dim-1}] uint32):
 * evaluate, probe the centres of failing cells outside B for a proven counterexample, classify, accumulate stats, append up to
 * max_examples counterexamples ([obs_dim centre, margin, kind 1 = decrease / 2 = escaped] floats) in a deterministic order,
 * and write the children of split cells to stack[top - k, ...); *children (device) = their number. */
int msacl_region_round(const msacl_region_params_t* p, const msacl_region_bnb_t* b, const float* image, uint32_t* stack,
                       int64_t top, int64_t k, const msacl_region_ws_t* ws, int64_t* stats, float* examples, int64_t* children,
                       void* stream);

const char* msacl_last_error(void);
int msacl_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* MSACL_B200_H_ */
