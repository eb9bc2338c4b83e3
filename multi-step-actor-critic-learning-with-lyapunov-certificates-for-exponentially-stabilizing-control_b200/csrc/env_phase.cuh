// The env phase of one rollout step, shared by every rollout kernel (rollout_tc.cu, rollout_fused.cu and rollout_step_kernel
// in env_step.cu): one BaseSampler._n_step (RL/trainer/sampler/base.py:118-163,220) for one env instance whose policy
// outputs are already in registers.  Thread = env instance, state in EnvRegs.  The kernels differ only in where the logits
// come from and where the next observation goes; the arithmetic and the bookkeeping are defined here once.
#pragma once
#include "common.cuh"

namespace msacl {

// N(0,1) action noise of one env-step: the explicit row eps[row], else the env's Philox stream; zeros unless `draw`
// (deterministic actions, or a thread that owns no env instance).
template <int A>
__device__ __forceinline__ void env_noise(float (&z)[4], bool draw, const float* __restrict__ eps, int64_t row, uint64_t seed,
                                          uint64_t env, uint32_t step) {
#pragma unroll
  for (int j = 0; j < 4; ++j) z[j] = 0.f;
  if (!draw) return;
  if (eps) {
#pragma unroll
    for (int j = 0; j < A; ++j) z[j] = eps[row * A + j];
  } else {
    action_noise4(seed, env, step, z);
  }
}

// Episode statistics: per-thread partials (episodes, sum of returns, sum of lengths, terminated, truncated), reduced once per
// launch -- no hot atomics.
struct EpisodeStats {
  float ep = 0.f, ret = 0.f, len = 0.f, term = 0.f, trunc = 0.f;

  template <int ID>
  __device__ __forceinline__ void record(const EnvRegs<ID>& e, bool terminated) {
    ep += 1.f; ret += e.ep_return; len += (float)e.ep_len;
    if (terminated) term += 1.f; else trunc += 1.f;
  }
  // warp-shuffle reduction, then one atomic per warp and statistic that saw an episode end; every lane of the warp calls it
  __device__ __forceinline__ void flush(double* stats) const {
    float v[5] = {ep, ret, len, term, trunc};
#pragma unroll
    for (int q = 0; q < 5; ++q) {
#pragma unroll
      for (int o = 16; o >= 1; o >>= 1) v[q] += __shfl_xor_sync(0xffffffffu, v[q], o);
      if ((threadIdx.x & 31) == 0 && v[q] != 0.f) atomicAdd(&stats[q], (double)v[q]);
    }
  }
};

// One env-step of env instance gi of the state st from its logits lg = [mean | log_std] and noise z; the
// transition goes to record `row` of `out`.  hand_off(obs) receives the next observation (post-reset) before the transition
// is stored: the tensor-core kernel's hand-off ends in a proxy fence that waits for the thread's outstanding memory
// operations, so the (uncoalesced) transition stores are issued after it and drain while the next MLP runs.
template <int ID, typename HandOff>
__device__ __forceinline__ void env_phase(EnvRegs<ID>& e, const float (&lg)[2 * Env<ID>::A], const float (&z)[4], int deterministic,
                                          float min_log_std, float max_log_std, const msacl_env_state_t& st, int64_t gi,
                                          int n_step, float reward_scale, float cost_scale, const msacl_transitions_t& out,
                                          int64_t row, EpisodeStats& stats, HandOff&& hand_off) {
  using E = Env<ID>;
  constexpr int D = E::D, A = E::A, A2 = 2 * A;
  if (out.obs) store_row<D>(out.obs, row, e.obs());
  if (out.logits) {      // diagnostic output, written here so that the logits do not stay live across the env step
#pragma unroll
    for (int j = 0; j < A2; ++j) out.logits[row * A2 + j] = lg[j];
  }
  float act[A];
  float lp_gauss = 0.f, lp_tanh = 0.f, lp_scale = 0.f;
#pragma unroll
  for (int j = 0; j < A; ++j) {      // TanhGaussDistribution.sample / mode (act_distribution_cls.py:45-57, 90-95)
    const float mean = lg[j];
    const float ls = lg[A + j];
    const float sd = expf(fminf(fmaxf(ls, min_log_std), max_log_std));
    const float half = (E::act_high(j) - E::act_low(j)) / 2.0f;
    const float mid = (E::act_high(j) + E::act_low(j)) / 2.0f;
    const float u = deterministic ? mean : (sd * z[j] + mean);      // torch.normal: z*std, then +mean
    const float th = tanhf(u);
    const float a_lim = half * th + mid;
    // Normal.log_prob(u) = -((u-mean)^2)/(2 var) - log(std) - log(sqrt(2 pi))
    const float diff = u - mean;
    const float g = ((-(diff * diff)) / (2.0f * (sd * sd)) - logf(sd)) - 0.91893853320467267f;
    const float t = logf(1.000001f - th * th);
    const float sc = logf(half);
    lp_gauss = (j == 0) ? g : lp_gauss + g;
    lp_tanh = (j == 0) ? t : lp_tanh + t;
    lp_scale = (j == 0) ? sc : lp_scale + sc;
    act[j] = fminf(fmaxf(a_lim, E::act_low(j)), E::act_high(j));   // base.py:141-143
  }
  const float logp = (lp_gauss - lp_tanh) - lp_scale;
  const float rew = E::step(e.sf, e.sd, act);
  const bool term = e.out_of_bounds();
  e.step += 1;
  const bool trunc = e.step >= st.max_step;
  const bool done = term || trunc;
  e.ep_return += rew;
  e.ep_len += 1;
  const float rew_s = rew * reward_scale;                            // rew_plus_cost.py:18
  const float cost = np_rowsum_sq<D>(e.obs()) * cost_scale;          // :20-21, on real_next_obs
  e.run = min(e.run + 1, n_step);
  const bool emit = e.run >= n_step;
  float obs2[D];                                                     // real_next_obs (pre-reset)
#pragma unroll
  for (int d = 0; d < D; ++d) obs2[d] = e.obs()[d];
  if (done) {      // gymnasium 0.28.1 SyncVectorEnv: reset in the same step
    stats.record(e, term);
    e.episode += 1;
    e.run = 0;
    e.reset(st.seed, st.env_base + (uint64_t)gi);
  }
  hand_off(e.obs());
  if (out.act) store_row<A>(out.act, row, act);
  if (out.obs2) store_row<D>(out.obs2, row, obs2);
  if (out.rew) out.rew[row] = rew_s;
  if (out.cost) out.cost[row] = cost;
  if (out.done) out.done[row] = done ? 1 : 0;
  if (out.logp) out.logp[row] = logp;
  if (out.emit) out.emit[row] = emit ? 1 : 0;
}

}  // namespace msacl
