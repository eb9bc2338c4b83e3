// Shared host/device helpers for libmsacl_b200.so
#pragma once
#include <cuda_runtime.h>

#include <cstdio>
#include <cstring>
#include <mutex>
#include <unordered_map>

#include "../../include/msacl_b200.h"
#include "env_dynamics.cuh"

namespace msacl {

constexpr int kNumSMs = 148;  // B200

void set_error(const char* fmt, ...);
int check_launch(const char* what);

// Grid of a grid-stride ("persistent") kernel: whole waves of RESIDENT blocks.  A fixed cap of 8 blocks per SM is 1.6 waves for
// a kernel that fits 5 blocks per SM (48 registers x 256 threads) -- the last wave runs at 60 % occupancy; measured on
// lyapunov_risk: 0.77 -> 0.80 of HBM from the grid alone.  `waves` resident sets are launched (2: blocks that fall behind
// are balanced by the second set).  The occupancy query is a host-side table lookup (no stream operation: legal during
// graph capture) and is cached per kernel.
inline int cached_occupancy(const void* kern, int block_threads) {
  static std::mutex mu;
  static std::unordered_map<const void*, int> cache;      // per translation unit; a kernel is always launched with one block size
  std::lock_guard<std::mutex> lock(mu);
  auto it = cache.find(kern);
  if (it != cache.end()) return it->second;
  int o = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, kern, block_threads, 0) != cudaSuccess || o < 1) { o = 4; (void)cudaGetLastError(); }
  cache.emplace(kern, o);
  return o;
}

template <typename Kernel>
inline unsigned resident_grid(Kernel kern, int block_threads, int64_t work_items, int per_block, int waves = 2) {
  const int64_t want = (work_items + per_block - 1) / per_block;
  const int64_t cap = (int64_t)kNumSMs * cached_occupancy(reinterpret_cast<const void*>(kern), block_threads) * waves;
  return (unsigned)(want < cap ? (want > 0 ? want : 1) : cap);
}

#define MSACL_DISPATCH_ENV(env_id, ...)                                        \
  switch (env_id) {                                                            \
    case kVanderPol: { constexpr int ID = kVanderPol; __VA_ARGS__; break; }    \
    case kPendulum: { constexpr int ID = kPendulum; __VA_ARGS__; break; }      \
    case kDuctedFan: { constexpr int ID = kDuctedFan; __VA_ARGS__; break; }    \
    case kTwoLink: { constexpr int ID = kTwoLink; __VA_ARGS__; break; }        \
    case kSingleTrackCar: { constexpr int ID = kSingleTrackCar; __VA_ARGS__; break; } \
    case kQuadTracking: { constexpr int ID = kQuadTracking; __VA_ARGS__; break; }     \
    default: set_error("unknown env id %d", (int)(env_id)); return MSACL_ERR_BAD_ENV; \
  }

// register-resident state of one env instance
// Row-per-thread store of N floats at dst[row * N ..): 16-byte (N % 4 == 0) or 8-byte (N % 2 == 0) vectors when the row
// stride keeps them aligned (base pointers are torch allocations, >= 256-byte aligned), scalar otherwise.
template <int N>
__device__ __forceinline__ void store_row(float* __restrict__ dst, int64_t row, const float* v) {
  float* p = dst + row * N;
  if constexpr (N % 4 == 0) {
#pragma unroll
    for (int j = 0; j < N / 4; ++j) reinterpret_cast<float4*>(p)[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
  } else if constexpr (N % 2 == 0) {
#pragma unroll
    for (int j = 0; j < N / 2; ++j) reinterpret_cast<float2*>(p)[j] = make_float2(v[2 * j], v[2 * j + 1]);
  } else {
#pragma unroll
    for (int j = 0; j < N; ++j) p[j] = v[j];
  }
}

// host-side check matching store_row's vector width
template <int N>
inline bool row_store_misaligned(const void* p) {
  constexpr uintptr_t mask = (N % 4 == 0) ? 15 : ((N % 2 == 0) ? 7 : 3);
  return p != nullptr && (reinterpret_cast<uintptr_t>(p) & mask) != 0;
}

// host-side checks shared by the rollout entry points `what`: the sampler path needs a time limit, and the env phase writes
// the obs / obs2 / act rows of the transition record with store_row
template <int ID>
inline int check_rollout_outputs(const char* what, const msacl_env_state_t* st, const msacl_transitions_t* out) {
  if (st->max_step <= 0) {
    set_error("%s: the sampler path needs max_step > 0 (bare-env mode is msacl_env_step only)", what);
    return MSACL_ERR_BAD_ARG;
  }
  if (row_store_misaligned<Env<ID>::D>(out->obs) || row_store_misaligned<Env<ID>::D>(out->obs2) || row_store_misaligned<Env<ID>::A>(out->act)) {
    set_error("%s: transition obs/obs2/act rows must be aligned to their vector width (16 B if the row length is a multiple of 4 "
              "floats, 8 B if even)", what);
    return MSACL_ERR_BAD_ARG;
  }
  return MSACL_OK;
}

template <int ID>
struct EnvRegs {
  using E = Env<ID>;
  float sf[E::SF];
  double sd[E::SD > 0 ? E::SD : 1];
  int32_t step, episode, ep_len, run;
  float ep_return;

  __device__ __forceinline__ void load(const msacl_env_state_t& st, int64_t i) {
#pragma unroll
    for (int r = 0; r < E::SF; ++r) sf[r] = st.sf[(int64_t)r * st.stride + i];
#pragma unroll
    for (int r = 0; r < E::SD; ++r) sd[r] = st.sd[(int64_t)r * st.stride + i];
    step = st.step[i]; episode = st.episode[i]; ep_len = st.ep_len[i]; run = st.run[i];
    ep_return = st.ep_return[i];
  }
  __device__ __forceinline__ void store(const msacl_env_state_t& st, int64_t i) const {
#pragma unroll
    for (int r = 0; r < E::SF; ++r) st.sf[(int64_t)r * st.stride + i] = sf[r];
#pragma unroll
    for (int r = 0; r < E::SD; ++r) st.sd[(int64_t)r * st.stride + i] = sd[r];
    st.step[i] = step; st.episode[i] = episode; st.ep_len[i] = ep_len; st.run[i] = run;
    st.ep_return[i] = ep_return;
  }
  __device__ __forceinline__ const float* obs() const { return sf + E::OBS_OFF; }

  // strict out-of-box test on the float32-cast bounds (e.g. VanderPol.py:118-121);
  // NaN compares false, i.e. never terminates, as in the reference
  __device__ __forceinline__ bool out_of_bounds() const {
    bool t = false;
#pragma unroll
    for (int j = 0; j < E::D; ++j) {
      const float o = sf[E::OBS_OFF + j];
      t = t || (o < E::obs_low(j)) || (o > E::obs_high(j));
    }
    return t;
  }
  __device__ __forceinline__ void reset(uint64_t seed, uint64_t env) {
    E::reset(sf, sd, seed, env, (uint32_t)episode);
    step = 0; ep_len = 0; ep_return = 0.f;
  }
};

}  // namespace msacl
