// Unfused vector-env API: dims / bounds / reset / step with same-step autoreset.
// One thread per env instance; SoA state rows are read/written coalesced; the [n][D] API
// tensors are written row-per-thread (a warp covers 32*D contiguous floats).
// HBM-bound: algorithmic bytes per env-step = 4*(2*SF + 2*D + A + 1) + 8*2*SD + 2 + 32 (counters).
#include <cstdarg>

#include "env_phase.cuh"

namespace msacl {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return MSACL_ERR_CUDA;
  }
  return MSACL_OK;
}

template <int ID>
__global__ void __launch_bounds__(128) env_reset_kernel(msacl_env_state_t st) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= st.n) return;
  EnvRegs<ID> r;
  r.episode = st.episode[i];
  r.run = 0;
  r.reset(st.seed, st.env_base + (uint64_t)i);
  r.store(st, i);
}

__global__ void __launch_bounds__(128) quad_init_from_raw_kernel(msacl_env_state_t st) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= st.n) return;
  EnvRegs<kQuadTracking> r;
  r.load(st, i);
  double xd[3], Rd[9];
  float vd[3];
  quad_desired(r.sf, r.sf + 3, 0.0, xd, vd, Rd);
  const double Omd[3] = {0.0, 0.0, 0.0};
  quad_errors(r.sf, r.sf + 3, r.sf + 6, r.sf + 15, xd, vd, Rd, Omd, r.sf + 18);
  r.sd[0] = 0.0;
#pragma unroll
  for (int j = 0; j < 9; ++j) r.sd[1 + j] = Rd[j];
  r.store(st, i);
}

template <int ID>
__global__ void __launch_bounds__(128)
env_step_kernel(msacl_env_state_t st, const float* __restrict__ action, float* __restrict__ next_obs,
                float* __restrict__ reward, uint8_t* __restrict__ terminated, uint8_t* __restrict__ truncated,
                float* __restrict__ final_obs) {
  using E = Env<ID>;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= st.n) return;
  EnvRegs<ID> r;
  r.load(st, i);
  float a[E::A];
#pragma unroll
  for (int j = 0; j < E::A; ++j) a[j] = action[i * E::A + j];
  const float rew = E::step(r.sf, r.sd, a);
  const bool term = r.out_of_bounds();
  r.step += 1;
  // max_step <= 0: a bare env instance as the reference classes are outside a vector env -- no time limit and no
  // autoreset; the state keeps evolving from the terminal state exactly as <env>.step would (e.g. VanderPol.py:100-130)
  const bool vec = st.max_step > 0;
  const bool trunc = vec && r.step >= st.max_step;
  r.ep_return += rew;
  r.ep_len += 1;
  if (final_obs) store_row<E::D>(final_obs, i, r.obs());
  if (vec && (term || trunc)) {   // gymnasium 0.28.1 SyncVectorEnv: reset in the same step
    r.episode += 1;
    r.run = 0;
    r.reset(st.seed, st.env_base + (uint64_t)i);
  }
  store_row<E::D>(next_obs, i, r.obs());
  reward[i] = rew;
  terminated[i] = term ? 1 : 0;
  truncated[i] = trunc ? 1 : 0;
  r.store(st, i);
}

// One BaseSampler._n_step (RL/trainer/sampler/base.py:118-163,220) for policy outputs computed OUTSIDE the kernel: the
// path for policies the fused rollout kernels are not specialised for (any depth / width / activation; the reference
// builds arbitrary MLPs, RL/apprfunc/mlp.py:18-33).  Thread = env instance; the env phase is the one of the fused
// rollout kernels (env_phase.cuh).  The next observation is handed off through the env state, which the next step's first
// layer reads: the state is stored in the hand-off, so its counters are dead before the transition stores (this keeps the
// SingleTrackCar instance free of register spills).
template <int ID>
__global__ void __launch_bounds__(128)
rollout_step_kernel(msacl_env_state_t st, const float* __restrict__ logits, float min_log_std, float max_log_std, uint32_t step,
                    int n_step, float reward_scale, float cost_scale, const float* __restrict__ eps, int deterministic,
                    msacl_transitions_t out, double* stats) {
  constexpr int A2 = 2 * Env<ID>::A;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  EpisodeStats epstats;
  if (i < st.n) {
    EnvRegs<ID> e;
    e.load(st, i);
    float lg[A2];
#pragma unroll
    for (int j = 0; j < A2; ++j) lg[j] = logits[i * A2 + j];
    float z[4];
    env_noise<Env<ID>::A>(z, !deterministic, eps, i, st.seed, st.env_base + (uint64_t)i, step);
    env_phase<ID>(e, lg, z, deterministic, min_log_std, max_log_std, st, i, n_step, reward_scale, cost_scale, out, i, epstats,
                  [&](const float*) { e.store(st, i); });
  }
  if (stats) epstats.flush(stats);
}

__global__ void action_noise_kernel(uint64_t seed, uint64_t env_base, int64_t n, int act_dim, uint32_t step, float* out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float z[4];
  action_noise4(seed, env_base + (uint64_t)i, step, z);
  for (int j = 0; j < act_dim; ++j) out[i * act_dim + j] = z[j];
}

}  // namespace msacl

using namespace msacl;

__global__ void quad_polar_selftest_kernel(const float* __restrict__ in, float* __restrict__ out, int64_t n, float theta2) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float R[9];
#pragma unroll
  for (int j = 0; j < 9; ++j) R[j] = in[i * 9 + j];
  quad_polar_f32(R, theta2);
#pragma unroll
  for (int j = 0; j < 9; ++j) out[i * 9 + j] = R[j];
}

extern "C" {

const char* msacl_last_error(void) { return g_err; }
int msacl_abi_version(void) { return MSACL_ABI_VERSION; }

int msacl_env_dims(int env_id, int32_t dims[6]) {
  MSACL_DISPATCH_ENV(env_id, {
    using E = Env<ID>;
    dims[0] = E::D; dims[1] = E::A; dims[2] = E::SF; dims[3] = E::SD; dims[4] = E::OBS_OFF; dims[5] = E::CONTROL_STEP;
  });
  return MSACL_OK;
}

__global__ void bounds_kernel(int env_id, float* out) {
  // out: obs_low[12] obs_high[12] act_low[4] act_high[4]
  auto fill = [&](auto tag) {
    using E = decltype(tag);
    for (int j = 0; j < E::D; ++j) { out[j] = E::obs_low(j); out[12 + j] = E::obs_high(j); }
    for (int j = 0; j < E::A; ++j) { out[24 + j] = E::act_low(j); out[28 + j] = E::act_high(j); }
  };
  switch (env_id) {
    case kVanderPol: fill(Env<kVanderPol>{}); break;
    case kPendulum: fill(Env<kPendulum>{}); break;
    case kDuctedFan: fill(Env<kDuctedFan>{}); break;
    case kTwoLink: fill(Env<kTwoLink>{}); break;
    case kSingleTrackCar: fill(Env<kSingleTrackCar>{}); break;
    case kQuadTracking: fill(Env<kQuadTracking>{}); break;
  }
}

int msacl_env_bounds(int env_id, float* obs_low, float* obs_high, float* act_low, float* act_high) {
  int32_t dims[6];
  int rc = msacl_env_dims(env_id, dims);
  if (rc) return rc;
  float* d = nullptr;
  float h[32];
  if (cudaMalloc(&d, sizeof(h)) != cudaSuccess) { set_error("cudaMalloc failed (no CUDA device?)"); return MSACL_ERR_CUDA; }
  bounds_kernel<<<1, 1>>>(env_id, d);
  cudaError_t e = cudaMemcpy(h, d, sizeof(h), cudaMemcpyDeviceToHost);
  cudaFree(d);
  if (e != cudaSuccess) { set_error("bounds query: %s", cudaGetErrorString(e)); return MSACL_ERR_CUDA; }
  memcpy(obs_low, h, dims[0] * sizeof(float));
  memcpy(obs_high, h + 12, dims[0] * sizeof(float));
  memcpy(act_low, h + 24, dims[1] * sizeof(float));
  memcpy(act_high, h + 28, dims[1] * sizeof(float));
  return MSACL_OK;
}

static int validate_state(const msacl_env_state_t* st) {
  if (!st || st->n <= 0 || st->stride < st->n || !st->sf || !st->step || !st->episode || !st->ep_return ||
      !st->ep_len || !st->run) {
    set_error("invalid env state descriptor");
    return MSACL_ERR_BAD_ARG;
  }
  return MSACL_OK;
}

int msacl_env_reset(const msacl_env_state_t* st, void* stream) {
  if (int rc = validate_state(st)) return rc;
  const int threads = 128;
  const unsigned blocks = (unsigned)((st->n + threads - 1) / threads);
  MSACL_DISPATCH_ENV(st->env_id, (env_reset_kernel<ID><<<blocks, threads, 0, (cudaStream_t)stream>>>(*st)));
  return check_launch("env_reset");
}

int msacl_quad_init_from_raw(const msacl_env_state_t* st, void* stream) {
  if (int rc = validate_state(st)) return rc;
  if (st->env_id != kQuadTracking || !st->sd) { set_error("quad_init_from_raw needs a QuadTracking state"); return MSACL_ERR_BAD_ARG; }
  const int threads = 128;
  const unsigned blocks = (unsigned)((st->n + threads - 1) / threads);
  quad_init_from_raw_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(*st);
  return check_launch("quad_init_from_raw");
}

int msacl_env_step(const msacl_env_state_t* st, const float* action, float* next_obs, float* reward,
                   uint8_t* terminated, uint8_t* truncated, float* final_obs, void* stream) {
  if (int rc = validate_state(st)) return rc;
  if (!action || !next_obs || !reward || !terminated || !truncated) { set_error("env_step: null buffer"); return MSACL_ERR_BAD_ARG; }
  const int threads = 128;
  const unsigned blocks = (unsigned)((st->n + threads - 1) / threads);
  MSACL_DISPATCH_ENV(st->env_id, {
    if (row_store_misaligned<Env<ID>::D>(next_obs) || row_store_misaligned<Env<ID>::D>(final_obs)) {
      set_error("env_step: next_obs / final_obs rows must be aligned to their vector width (16 B if obs_dim %% 4 == 0, 8 B if even)");
      return MSACL_ERR_BAD_ARG;
    }
    env_step_kernel<ID><<<blocks, threads, 0, (cudaStream_t)stream>>>(*st, action, next_obs, reward, terminated, truncated, final_obs);
  });
  return check_launch("env_step");
}

int msacl_rollout_step(const msacl_env_state_t* st, const float* logits, float min_log_std, float max_log_std, uint32_t step,
                       int32_t n_step, float reward_scale, float cost_scale, const float* eps, int32_t deterministic,
                       const msacl_transitions_t* out, double* stats, void* stream) {
  if (int rc = validate_state(st)) return rc;
  if (!logits || !out || n_step <= 0) { set_error("rollout_step: bad argument"); return MSACL_ERR_BAD_ARG; }
  const int threads = 128;
  const unsigned blocks = (unsigned)((st->n + threads - 1) / threads);
  MSACL_DISPATCH_ENV(st->env_id, {
    if (int rc = check_rollout_outputs<ID>("rollout_step", st, out)) return rc;
    rollout_step_kernel<ID><<<blocks, threads, 0, (cudaStream_t)stream>>>(*st, logits, min_log_std, max_log_std, step, n_step, reward_scale,
                                                                          cost_scale, eps, deterministic, *out, stats);
  });
  return check_launch("rollout_step");
}

int msacl_selftest_quad_polar(const float* in, float* out, int64_t n, float theta2, void* stream) {
  if (!in || !out || n <= 0) { set_error("selftest_quad_polar: bad argument"); return MSACL_ERR_BAD_ARG; }
  quad_polar_selftest_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(in, out, n, theta2);
  return check_launch("selftest_quad_polar");
}

int msacl_action_noise(uint64_t seed, uint64_t env_base, int64_t n, int32_t act_dim, uint32_t step, float* out,
                       void* stream) {
  if (n <= 0 || act_dim < 1 || act_dim > 4 || !out) { set_error("action_noise: bad argument"); return MSACL_ERR_BAD_ARG; }
  const int threads = 128;
  const unsigned blocks = (unsigned)((n + threads - 1) / threads);
  action_noise_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(seed, env_base, n, act_dim, step, out);
  return check_launch("action_noise");
}

}  // extern "C"
