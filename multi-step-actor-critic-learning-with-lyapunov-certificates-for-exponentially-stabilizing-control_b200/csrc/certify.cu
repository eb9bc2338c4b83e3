// Lyapunov-certificate verifier: closed-loop checks of boundedness and exponential decrease (include/msacl_b200.h).
// No counterpart in the reference.  One thread per initial state; the per-state records are structure-of-arrays in HBM and
// are updated once per rollout chunk, so memory scales with n, not n * horizon.  Every comparison is in float64 on values
// that are exact in float64 (float32 inputs, squares of float32, the host's decay table), so NumPy restates it bit for bit
// (oracle/certify.py).
// HBM-bound: algorithmic bytes per state-step = 4 D + 4 + 1 (obs2 row, V, done), plus 33 bytes of record read / 29 written
// per live state and chunk.
#include <cmath>

#include "common.cuh"
#include "philox.cuh"

namespace msacl {

constexpr int CB = 256;
constexpr uint32_t kStreamCertBox = 0x63657274u;   // Philox counter word 3 of the box draws ("cert"; resets use 1..4)
constexpr int kCertMaxD = 16;
constexpr uint32_t kKeyInf = 0xFF800000u;           // order key of +inf

struct CertArgs {
  int32_t T;
  double alpha1, alpha2, ratio, v_atol;               // ratio = alpha2 / alpha1, divided on the host
  const double* decay;
};

__device__ __forceinline__ uint32_t float_key(float f) {
  const uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

template <int N>
__device__ __forceinline__ void load_row(const float* __restrict__ src, int64_t row, float* v) {
  const float* p = src + row * N;
  if constexpr (N % 4 == 0) {
#pragma unroll
    for (int j = 0; j < N / 4; ++j) {
      const float4 q = __ldg(reinterpret_cast<const float4*>(p) + j);
      v[4 * j] = q.x; v[4 * j + 1] = q.y; v[4 * j + 2] = q.z; v[4 * j + 3] = q.w;
    }
  } else if constexpr (N % 2 == 0) {
#pragma unroll
    for (int j = 0; j < N / 2; ++j) {
      const float2 q = __ldg(reinterpret_cast<const float2*>(p) + j);
      v[2 * j] = q.x; v[2 * j + 1] = q.y;
    }
  } else {
#pragma unroll
    for (int j = 0; j < N; ++j) v[j] = __ldg(p + j);
  }
}

template <int D>
__device__ __forceinline__ double sumsq64(const float* o) {
  double s = 0.0;
#pragma unroll
  for (int j = 0; j < D; ++j) s = s + (double)o[j] * (double)o[j];
  return s;
}

// flags of visited state k; ck = c_k, v0 / s0 of the state's k = 0
template <int D>
__device__ __forceinline__ uint32_t visit_flags(const float* o, float v, double s, int k, double ck, double v0, double s0,
                                                const CertArgs& a) {
  bool fin = isfinite(v);
#pragma unroll
  for (int j = 0; j < D; ++j) fin = fin && isfinite(o[j]);
  uint32_t f = fin ? 0u : (uint32_t)MSACL_CERT_NONFINITE;
  const double vd = (double)v;
  if (vd < a.alpha1 * s - a.v_atol) f |= MSACL_CERT_BOUND_LO;
  if (vd > a.alpha2 * s + a.v_atol) f |= MSACL_CERT_BOUND_HI;
  if (k >= 1) {
    if (vd > ck * v0 + a.v_atol) f |= MSACL_CERT_DECREASE;
    if (s > a.ratio * ck * s0) f |= MSACL_CERT_NOT_EXP_STABLE;
  }
  return f;
}

struct CertBox { float lo[kCertMaxD], hi[kCertMaxD]; };

__global__ void __launch_bounds__(CB) certify_box_kernel(msacl_env_state_t st, int D, CertBox box) {
  const int64_t i = (int64_t)blockIdx.x * CB + threadIdx.x;
  if (i >= st.n) return;
  const uint64_t gid = st.env_base + (uint64_t)i;
  for (int j = 0; j < D; ++j) {
    const U4 r = philox4x32_10((uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)j, kStreamCertBox, (uint32_t)st.seed,
                               (uint32_t)(st.seed >> 32));
    const float span = box.hi[j] - box.lo[j];
    st.sf[(int64_t)j * st.stride + i] = box.lo[j] + span * u01(r.x);
  }
}

template <int D>
__global__ void __launch_bounds__(CB) certify_begin_kernel(int64_t n, const float* __restrict__ obs0, const float* __restrict__ v0,
                                                           CertArgs a, msacl_cert_records_t rec) {
  const int64_t i = (int64_t)blockIdx.x * CB + threadIdx.x;
  if (i >= n) return;
  float o[D];
  load_row<D>(obs0, i, o);
  const float v = v0[i];
  const double s = sumsq64<D>(o);
  const uint32_t f = visit_flags<D>(o, v, s, 0, 1.0, (double)v, s, a);
  rec.v0[i] = v;
  rec.s0[i] = s;
  rec.flags[i] = (uint8_t)f;
  rec.first_violation[i] = (f & MSACL_CERT_FAIL_MASK) ? 0 : -1;
  rec.first_decrease[i] = -1;
  rec.end_step[i] = a.T;
  rec.worst_ratio[i] = 0.0;
}

template <int D>
__global__ void __launch_bounds__(CB) certify_steps_kernel(int64_t n, int32_t K, int32_t k0, const float* __restrict__ obs2,
                                                           const float* __restrict__ V, const uint8_t* __restrict__ done,
                                                           CertArgs a, msacl_cert_records_t rec) {
  const int64_t i = (int64_t)blockIdx.x * CB + threadIdx.x;
  if (i >= n) return;
  uint32_t flags = rec.flags[i];
  if (flags & MSACL_CERT_ESCAPED) return;                   // trajectory ended in an earlier chunk
  const double v0 = (double)rec.v0[i], s0 = rec.s0[i];
  int32_t fv = rec.first_violation[i], fd = rec.first_decrease[i], end = rec.end_step[i];
  double worst = rec.worst_ratio[i];
  const int kend = min(K, a.T - k0 + 1);
  for (int t = 0; t < kend; ++t) {
    const int k = k0 + t;
    const int64_t r = (int64_t)t * n + i;
    float o[D];
    load_row<D>(obs2, r, o);
    const float v = V[r];
    const double s = sumsq64<D>(o);
    const double ck = a.decay[k];
    uint32_t f = visit_flags<D>(o, v, s, k, ck, v0, s0, a);
    const double vd = (double)v, den = ck * v0;
    const double ratio = den == 0.0 ? (vd > 0.0 ? (double)INFINITY : 0.0) : vd / den;
    if (ratio > worst) worst = ratio;                       // NaN ratios are skipped
    if (done[r]) f |= MSACL_CERT_ESCAPED;
    if ((f & MSACL_CERT_FAIL_MASK) && !(flags & MSACL_CERT_FAIL_MASK)) fv = k;
    if ((f & MSACL_CERT_DECREASE) && !(flags & MSACL_CERT_DECREASE)) fd = k;
    flags |= f;
    if (f & MSACL_CERT_ESCAPED) { end = k; break; }
  }
  rec.flags[i] = (uint8_t)flags;
  rec.first_violation[i] = fv;
  rec.first_decrease[i] = fd;
  rec.end_step[i] = end;
  rec.worst_ratio[i] = worst;
}

__global__ void certify_summary_init_kernel(int64_t* summary, int32_t T) {
  for (int j = threadIdx.x; j < MSACL_CERT_SUM_HIST + T; j += blockDim.x)
    if (j != MSACL_CERT_SUM_ROA) summary[j] = (j == MSACL_CERT_SUM_CSTAR_KEY) ? (int64_t)kKeyInf : 0;
}

constexpr int kCertCounters = 9;   // summary[0 .. 9)

__global__ void __launch_bounds__(CB) certify_finish_kernel(int64_t n, int32_t T, msacl_cert_records_t rec, int64_t* summary) {
  extern __shared__ unsigned int hist[];                    // [T]
  __shared__ unsigned long long cnt[kCertCounters];
  __shared__ unsigned int kmin;
  for (int j = threadIdx.x; j < T; j += CB) hist[j] = 0;
  if (threadIdx.x < kCertCounters) cnt[threadIdx.x] = 0;
  if (threadIdx.x == 0) kmin = kKeyInf;
  __syncthreads();
  unsigned c[kCertCounters] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  unsigned key = kKeyInf;
  for (int64_t i = (int64_t)blockIdx.x * CB + threadIdx.x; i < n; i += (int64_t)gridDim.x * CB) {
    const unsigned f = rec.flags[i];
    c[0] += 1;
#pragma unroll
    for (int b = 0; b < 6; ++b) c[1 + b] += (f >> b) & 1u;
    const bool certified = (f & MSACL_CERT_FAIL_MASK) == 0;
    c[7] += certified ? 1u : 0u;
    c[8] += ((f >> 3) ^ (f >> 5)) & 1u;                     // DECREASE (bit 3) != NOT_EXP_STABLE (bit 5)
    if (!certified) {
      const float v = rec.v0[i];
      if (!isnan(v)) key = min(key, float_key(v));
    }
    const int fd = rec.first_decrease[i];
    if (fd >= 1 && fd <= T) atomicAdd(&hist[fd - 1], 1u);
  }
#pragma unroll
  for (int j = 0; j < kCertCounters; ++j) {
    const unsigned w = __reduce_add_sync(0xffffffffu, c[j]);
    if ((threadIdx.x & 31) == 0 && w) atomicAdd(&cnt[j], (unsigned long long)w);
  }
  key = __reduce_min_sync(0xffffffffu, key);
  if ((threadIdx.x & 31) == 0) atomicMin(&kmin, key);
  __syncthreads();
  unsigned long long* out = reinterpret_cast<unsigned long long*>(summary);
  if (threadIdx.x < kCertCounters && cnt[threadIdx.x]) atomicAdd(&out[threadIdx.x], cnt[threadIdx.x]);
  if (threadIdx.x == 0 && kmin != kKeyInf) atomicMin(&out[MSACL_CERT_SUM_CSTAR_KEY], (unsigned long long)kmin);
  for (int j = threadIdx.x; j < T; j += CB)
    if (hist[j]) atomicAdd(&out[MSACL_CERT_SUM_HIST + j], (unsigned long long)hist[j]);
}

__global__ void __launch_bounds__(CB) certify_roa_kernel(int64_t n, const float* __restrict__ v0, float c_star, int64_t* summary) {
  __shared__ unsigned long long cnt;
  if (threadIdx.x == 0) cnt = 0;
  __syncthreads();
  unsigned c = 0;
  for (int64_t i = (int64_t)blockIdx.x * CB + threadIdx.x; i < n; i += (int64_t)gridDim.x * CB) c += v0[i] < c_star ? 1u : 0u;
  const unsigned w = __reduce_add_sync(0xffffffffu, c);
  if ((threadIdx.x & 31) == 0 && w) atomicAdd(&cnt, (unsigned long long)w);
  __syncthreads();
  if (threadIdx.x == 0 && cnt) atomicAdd(reinterpret_cast<unsigned long long*>(summary) + MSACL_CERT_SUM_ROA, cnt);
}

static int cert_args(const msacl_cert_params_t* p, CertArgs* a) {
  if (!p || p->horizon < 1 || p->horizon > MSACL_CERT_MAX_HORIZON || !p->decay || !(p->alpha1 > 0.0) || !std::isfinite(p->alpha1) ||
      !(p->alpha2 > 0.0) || !std::isfinite(p->alpha2) || !(p->v_atol >= 0.0) || !std::isfinite(p->v_atol)) {
    set_error("certify: bad parameters (need 1 <= horizon <= %d, decay table, alpha1, alpha2 > 0, v_atol >= 0)",
              (int)MSACL_CERT_MAX_HORIZON);
    return MSACL_ERR_BAD_ARG;
  }
  *a = CertArgs{p->horizon, p->alpha1, p->alpha2, p->alpha2 / p->alpha1, p->v_atol, p->decay};
  return MSACL_OK;
}

static int cert_records(const msacl_cert_records_t* r) {
  if (!r || !r->v0 || !r->s0 || !r->flags || !r->first_violation || !r->first_decrease || !r->end_step || !r->worst_ratio) {
    set_error("certify: every record array is required");
    return MSACL_ERR_BAD_ARG;
  }
  return MSACL_OK;
}

template <int D>
static bool misaligned(const void* p) {
  constexpr uintptr_t mask = (D % 4 == 0) ? 15 : ((D % 2 == 0) ? 7 : 3);
  return (reinterpret_cast<uintptr_t>(p) & mask) != 0;
}

#define MSACL_DISPATCH_OBS_DIM(obs_dim, ...)                                      \
  switch (obs_dim) {                                                              \
    case 2: { constexpr int D = 2; __VA_ARGS__; break; }                          \
    case 4: { constexpr int D = 4; __VA_ARGS__; break; }                          \
    case 6: { constexpr int D = 6; __VA_ARGS__; break; }                          \
    case 7: { constexpr int D = 7; __VA_ARGS__; break; }                          \
    case 12: { constexpr int D = 12; __VA_ARGS__; break; }                        \
    default: set_error("certify: obs_dim %d is not one of the env observation sizes (2, 4, 6, 7, 12)", (int)(obs_dim)); \
             return MSACL_ERR_BAD_ARG;                                            \
  }

}  // namespace msacl

using namespace msacl;

extern "C" {

int msacl_certify_box_init(const msacl_env_state_t* st, const float* lo, const float* hi, void* stream) {
  if (!st || st->n <= 0 || st->stride < st->n || !st->sf || !lo || !hi) {
    set_error("certify_box_init: invalid env state or box");
    return MSACL_ERR_BAD_ARG;
  }
  if (st->env_id == kQuadTracking) {
    set_error("certify_box_init: QuadTracking has no box initial states (its observation is not its state)");
    return MSACL_ERR_BAD_ARG;
  }
  int32_t dims[6];
  if (int rc = msacl_env_dims(st->env_id, dims)) return rc;
  const int D = dims[0];
  CertBox box{};
  for (int j = 0; j < D; ++j) {
    if (!std::isfinite(lo[j]) || !std::isfinite(hi[j]) || !(lo[j] <= hi[j])) {
      set_error("certify_box_init: need finite lo[j] <= hi[j] (j = %d)", j);
      return MSACL_ERR_BAD_ARG;
    }
    box.lo[j] = lo[j];
    box.hi[j] = hi[j];
  }
  certify_box_kernel<<<(unsigned)((st->n + CB - 1) / CB), CB, 0, (cudaStream_t)stream>>>(*st, D, box);
  return check_launch("certify_box_init");
}

int msacl_certify_begin(int64_t n, int32_t obs_dim, const float* obs0, const float* v0, const msacl_cert_params_t* p,
                        const msacl_cert_records_t* rec, void* stream) {
  CertArgs a;
  if (int rc = cert_args(p, &a)) return rc;
  if (int rc = cert_records(rec)) return rc;
  if (n <= 0 || !obs0 || !v0) { set_error("certify_begin: bad argument"); return MSACL_ERR_BAD_ARG; }
  MSACL_DISPATCH_OBS_DIM(obs_dim, {
    if (misaligned<D>(obs0)) { set_error("certify_begin: obs0 rows are not vector-aligned"); return MSACL_ERR_BAD_ARG; }
    certify_begin_kernel<D><<<(unsigned)((n + CB - 1) / CB), CB, 0, (cudaStream_t)stream>>>(n, obs0, v0, a, *rec);
  });
  return check_launch("certify_begin");
}

int msacl_certify_steps(int64_t n, int32_t obs_dim, int32_t K, int32_t k0, const float* obs2, const float* v, const uint8_t* done,
                        const msacl_cert_params_t* p, const msacl_cert_records_t* rec, void* stream) {
  CertArgs a;
  if (int rc = cert_args(p, &a)) return rc;
  if (int rc = cert_records(rec)) return rc;
  if (n <= 0 || K <= 0 || k0 < 1 || !obs2 || !v || !done) { set_error("certify_steps: bad argument (need n, K >= 1, k0 >= 1)"); return MSACL_ERR_BAD_ARG; }
  if (k0 > a.T) return MSACL_OK;                            // the whole chunk lies beyond the horizon
  MSACL_DISPATCH_OBS_DIM(obs_dim, {
    if (misaligned<D>(obs2)) { set_error("certify_steps: obs2 rows are not vector-aligned"); return MSACL_ERR_BAD_ARG; }
    certify_steps_kernel<D><<<(unsigned)((n + CB - 1) / CB), CB, 0, (cudaStream_t)stream>>>(n, K, k0, obs2, v, done, a, *rec);
  });
  return check_launch("certify_steps");
}

int msacl_certify_finish(int64_t n, int32_t horizon, const msacl_cert_records_t* rec, int64_t* summary, void* stream) {
  if (int rc = cert_records(rec)) return rc;
  if (n <= 0 || !summary || horizon < 1 || horizon > MSACL_CERT_MAX_HORIZON) {
    set_error("certify_finish: bad argument (need n >= 1, summary, 1 <= horizon <= %d)", (int)MSACL_CERT_MAX_HORIZON);
    return MSACL_ERR_BAD_ARG;
  }
  cudaStream_t s = (cudaStream_t)stream;
  certify_summary_init_kernel<<<1, 256, 0, s>>>(summary, horizon);
  const unsigned grid = resident_grid(certify_finish_kernel, CB, n, CB, 1);
  certify_finish_kernel<<<grid, CB, (size_t)horizon * sizeof(unsigned), s>>>(n, horizon, *rec, summary);
  return check_launch("certify_finish");
}

int msacl_certify_roa(int64_t n, const float* v0, float c_star, int64_t* summary, void* stream) {
  if (n <= 0 || !v0 || !summary) { set_error("certify_roa: bad argument"); return MSACL_ERR_BAD_ARG; }
  cudaStream_t s = (cudaStream_t)stream;
  if (cudaMemsetAsync(summary + MSACL_CERT_SUM_ROA, 0, sizeof(int64_t), s) != cudaSuccess) return check_launch("certify_roa");
  const unsigned grid = resident_grid(certify_roa_kernel, CB, n, CB, 1);
  certify_roa_kernel<<<grid, CB, 0, s>>>(n, v0, c_star, summary);
  return check_launch("certify_roa");
}

}  // extern "C"
