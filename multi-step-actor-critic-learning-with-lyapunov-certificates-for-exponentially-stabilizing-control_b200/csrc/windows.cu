// n-step window assembly + device replay ring.
// Replaces the per-env deque logic of RL/trainer/sampler/base.py:178-217 and
// NstepReplayBuffer.store/add_batch/sample_batch (RL/trainer/buffer/nstep_replay_buffer.py:91-150).
//
// The rollout kernel already recorded, per transition, whether the env's deque is full
// (`emit`).  The reference appends emitted windows in step-major / env-minor order and stores
// them at consecutive ring slots, so slot(t,i) = (ptr + exclusive_scan(emit)[t*n+i]) % max_size.
// Three small kernels: per-block counts, single-block scan of the counts, scatter.
// Integer bookkeeping is bit-exact; payload is copied verbatim.  HBM-bound:
// bytes per stored window = 2 * 4 * n_step * (2D + A + 4)  (read transitions + write ring).
#include "common.cuh"
#include "philox.cuh"

namespace msacl {

constexpr int WB = 256;   // flags per block

__global__ void __launch_bounds__(WB) window_count_kernel(const uint8_t* __restrict__ emit_new, int64_t total,
                                                          int64_t* __restrict__ block_counts) {
  const int64_t f = (int64_t)blockIdx.x * WB + threadIdx.x;
  const int flag = (f < total && emit_new[f]) ? 1 : 0;
  const int c = __syncthreads_count(flag);
  if (threadIdx.x == 0) block_counts[blockIdx.x] = c;
}

// exclusive scan of block_counts[0..nb) in place (single block); header[0]=old ptr, header[1]=total
__global__ void __launch_bounds__(1024) window_scan_kernel(int64_t* __restrict__ block_counts, int64_t nb,
                                                           int64_t* __restrict__ header, int64_t* __restrict__ ptr_size,
                                                           int64_t* __restrict__ count_out, int64_t max_size) {
  __shared__ int64_t warp_sums[32];
  __shared__ int64_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t base = 0; base < nb; base += 1024) {
    const int64_t idx = base + threadIdx.x;
    const int64_t v = idx < nb ? block_counts[idx] : 0;
    int64_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int64_t y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) warp_sums[warp] = x;
    __syncthreads();
    if (warp == 0) {
      int64_t w = warp_sums[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int64_t y = __shfl_up_sync(0xffffffffu, w, o);
        if (lane >= o) w += y;
      }
      warp_sums[lane] = w;   // inclusive
    }
    __syncthreads();
    const int64_t warp_off = warp > 0 ? warp_sums[warp - 1] : 0;
    const int64_t incl = carry + warp_off + x;
    if (idx < nb) block_counts[idx] = incl - v;
    __syncthreads();
    if (threadIdx.x == 1023) carry = incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const int64_t total = carry;
    header[0] = ptr_size[0];
    header[1] = total;
    ptr_size[0] = (ptr_size[0] + total) % max_size;
    const int64_t s = ptr_size[1] + total;
    ptr_size[1] = s < max_size ? s : max_size;
    if (count_out) count_out[0] = total;
  }
}

constexpr int SC_IT = 3;   // register-resident path of the copy: up to 96 obs vectors and 96 act scalars per window
template <int N> struct ObsVec;
template <> struct ObsVec<4> { using type = float4; };
template <> struct ObsVec<2> { using type = float2; };
template <> struct ObsVec<1> { using type = float; };

// One warp copies one n-step window out of the [T][n][.] transition store into entry `slot` of a [.][n_step][.] window
// array (the sampled batch of window_gather_indexed_kernel and window_sample_indexed_kernel).
// A window's rows come from ns transition slices (stride n rows), its destination entry is contiguous per field.  Work
// items are OW-float vectors of the obs / obs2 rows (OW = 4, 2 or 1: the widest that divides obs_dim), scalars of the act
// rows, and one lane per row for the four per-step scalars.  The item -> (row, offset) map is the same for every
// window: each lane derives it once and then walks it with additions only (no division per window).
template <int W>
struct WindowCopier {
  using VecT = typename ObsVec<W>::type;
  static constexpr int OW = W;
  const msacl_transitions_t& tr;
  const msacl_ring_t& ring;
  int64_t n, row_stride, arow_stride;
  int lane, ns, D, A, vpr, nv, na, r0, q0, dr, dq, ar0, aj0, adr, adj;

  __device__ __forceinline__ WindowCopier(const msacl_transitions_t& tr_, int64_t n_, const msacl_ring_t& ring_, int lane_)
      : tr(tr_), ring(ring_), n(n_), lane(lane_) {
    ns = ring.n_step; D = ring.obs_dim; A = ring.act_dim;
    vpr = D / OW;                         // obs vectors per row
    nv = ns * vpr; na = ns * A;
    r0 = lane / vpr; q0 = lane - r0 * vpr; dr = 32 / vpr; dq = 32 - dr * vpr;
    ar0 = lane / A; aj0 = lane - ar0 * A; adr = 32 / A; adj = 32 - adr * A;
    row_stride = n * (int64_t)D; arow_stride = n * (int64_t)A;
  }

  // newest = flat (t, i) index of the window's newest transition in the store
  __device__ __forceinline__ void copy(int64_t newest, int64_t slot) const {
    const int64_t first = newest - (int64_t)(ns - 1) * n;           // flat (t, i) row index of the window's oldest transition
    const float* so = tr.obs + first * D;
    const float* so2 = tr.obs2 + first * D;
    const float* sa = tr.act + first * A;
    float* dob = ring.obs + slot * ns * D;
    float* dob2 = ring.obs2 + slot * ns * D;
    float* da = ring.act + slot * ns * A;
    if (nv <= 32 * SC_IT && na <= 32 * SC_IT) {
      // every load of the window is issued before the first store (one memory round trip per window)
      VecT vo[SC_IT], vo2[SC_IT];
      float va[SC_IT], vr = 0.f, vc = 0.f, vl = 0.f;
      uint8_t vd = 0;
      int r = r0, q = q0;
#pragma unroll
      for (int it = 0; it < SC_IT; ++it) {
        if (it * 32 + lane < nv) {
          const int64_t src = r * row_stride + q * OW;
          vo[it] = *reinterpret_cast<const VecT*>(so + src);
          vo2[it] = *reinterpret_cast<const VecT*>(so2 + src);
        }
        r += dr; q += dq;
        if (q >= vpr) { q -= vpr; ++r; }
      }
      r = ar0;
      int j = aj0;
#pragma unroll
      for (int it = 0; it < SC_IT; ++it) {
        if (it * 32 + lane < na) va[it] = sa[r * arow_stride + j];
        r += adr; j += adj;
        if (j >= A) { j -= A; ++r; }
      }
      if (lane < ns) {
        const int64_t src = first + lane * n;
        vr = tr.rew[src]; vc = tr.cost[src]; vl = tr.logp[src]; vd = tr.done[src];
      }
#pragma unroll
      for (int it = 0; it < SC_IT; ++it) {
        const int v = it * 32 + lane;
        if (v < nv) {
          *reinterpret_cast<VecT*>(dob + (int64_t)v * OW) = vo[it];
          *reinterpret_cast<VecT*>(dob2 + (int64_t)v * OW) = vo2[it];
        }
        if (v < na) da[v] = va[it];
      }
      if (lane < ns) {
        ring.rew[slot * ns + lane] = vr;
        ring.cost[slot * ns + lane] = vc;
        ring.done[slot * ns + lane] = vd ? 1.0f : 0.0f;
        ring.logp[slot * ns + lane] = vl;
      }
      return;
    }
    {
      int r = r0, q = q0;
      for (int v = lane; v < nv; v += 32) {
        const int64_t src = r * row_stride + q * OW;
        *reinterpret_cast<VecT*>(dob + (int64_t)v * OW) = *reinterpret_cast<const VecT*>(so + src);
        *reinterpret_cast<VecT*>(dob2 + (int64_t)v * OW) = *reinterpret_cast<const VecT*>(so2 + src);
        r += dr; q += dq;
        if (q >= vpr) { q -= vpr; ++r; }
      }
    }
    {
      int r = ar0, j = aj0;
      for (int e = lane; e < na; e += 32) {
        da[e] = sa[r * arow_stride + j];
        r += adr; j += adj;
        if (j >= A) { j -= A; ++r; }
      }
    }
    for (int r = lane; r < ns; r += 32) {
      const int64_t src = first + r * n;
      ring.rew[slot * ns + r] = tr.rew[src];
      ring.cost[slot * ns + r] = tr.cost[src];
      ring.done[slot * ns + r] = tr.done[src] ? 1.0f : 0.0f;
      ring.logp[slot * ns + r] = tr.logp[src];
    }
  }
};

// G windows per warp, 32 / G lanes each (window_scatter_kernel; described for G = 4).  The windows a block stores are consecutive in (t, env)
// order, so the four windows of a warp are -- almost always -- four ADJACENT envs at the same step: for a given row the four
// 8-lane groups then read one contiguous piece of the transition store (TwoLink: 4 x 16 B = two full sectors) instead of 20
// lanes touching 20 different lines for a single window; ncu had the one-window-per-warp copy at ~150 LSU wavefronts per
// 1.1 KB window.  Nothing depends on the adjacency: every group addresses its own window.  Items are walked with additions
// only (the lane's first item and the (row, offset) increment per 8 items are derived once per call).
template <int W, int G>
struct WindowCopier4 {
  static constexpr int L = 32 / G;      // lanes per window
  using VecT = typename ObsVec<W>::type;
  static constexpr int CH = 3;          // items per lane whose loads are issued before the first store
  const msacl_transitions_t& tr;
  const msacl_ring_t& ring;
  int64_t n, row_stride, arow_stride;
  int j, ns, D, A, vpr, nv, na, r0, q0, dr, dq, ar0, aj0, adr, adj;

  __device__ __forceinline__ WindowCopier4(const msacl_transitions_t& tr_, int64_t n_, const msacl_ring_t& ring_, int lane)
      : tr(tr_), ring(ring_), n(n_), j(lane & (L - 1)) {
    ns = ring.n_step; D = ring.obs_dim; A = ring.act_dim;
    vpr = D / W; nv = ns * vpr; na = ns * A;
    r0 = j / vpr; q0 = j - r0 * vpr; dr = L / vpr; dq = L - dr * vpr;
    ar0 = j / A; aj0 = j - ar0 * A; adr = L / A; adj = L - adr * A;
    row_stride = n * (int64_t)D; arow_stride = n * (int64_t)A;
  }

  // the 8-lane group of this lane copies the window whose newest transition is `newest` into ring entry `slot` (< 0: none)
  __device__ __forceinline__ void copy(int64_t newest, int64_t slot) const {
    if (slot < 0) return;
    const int64_t first = newest - (int64_t)(ns - 1) * n;
    const float* so = tr.obs + first * D;
    const float* so2 = tr.obs2 + first * D;
    const float* sa = tr.act + first * A;
    float* dob = ring.obs + slot * ns * D;
    float* dob2 = ring.obs2 + slot * ns * D;
    float* da = ring.act + slot * ns * A;
    {
      int r = r0, q = q0;
      for (int v0 = j; v0 < nv; v0 += L * CH) {
        VecT a[CH], b[CH];
        int rr = r, qq = q;
#pragma unroll
        for (int c = 0; c < CH; ++c) {
          if (v0 + L * c < nv) {
            const int64_t src = rr * row_stride + qq * W;
            a[c] = *reinterpret_cast<const VecT*>(so + src);
            b[c] = *reinterpret_cast<const VecT*>(so2 + src);
          }
          rr += dr; qq += dq;
          if (qq >= vpr) { qq -= vpr; ++rr; }
        }
#pragma unroll
        for (int c = 0; c < CH; ++c) {
          const int v = v0 + L * c;
          if (v < nv) {
            *reinterpret_cast<VecT*>(dob + (int64_t)v * W) = a[c];
            *reinterpret_cast<VecT*>(dob2 + (int64_t)v * W) = b[c];
          }
        }
        r = rr; q = qq;
      }
    }
    {
      int r = ar0, jj = aj0;
      for (int e0 = j; e0 < na; e0 += L * CH) {
        float a[CH];
        int rr = r, q = jj;
#pragma unroll
        for (int c = 0; c < CH; ++c) {
          if (e0 + L * c < na) a[c] = sa[rr * arow_stride + q];
          rr += adr; q += adj;
          if (q >= A) { q -= A; ++rr; }
        }
#pragma unroll
        for (int c = 0; c < CH; ++c)
          if (e0 + L * c < na) da[e0 + L * c] = a[c];
        r = rr; jj = q;
      }
    }
    for (int r = j; r < ns; r += L) {
      const int64_t src = first + (int64_t)r * n;
      const float vr = tr.rew[src], vc = tr.cost[src], vl = tr.logp[src];
      const uint8_t vd = tr.done[src];
      ring.rew[slot * ns + r] = vr;
      ring.cost[slot * ns + r] = vc;
      ring.done[slot * ns + r] = vd ? 1.0f : 0.0f;
      ring.logp[slot * ns + r] = vl;
    }
  }
};

// W = obs vector width in floats (4 if obs_dim % 4 == 0, 2 if even, else 1)
template <int W>
__global__ void __launch_bounds__(WB)
window_scatter_kernel(msacl_transitions_t tr, int H, int64_t n, int64_t total_flags, msacl_ring_t ring,
                      const int64_t* __restrict__ block_offsets, const int64_t* __restrict__ header) {
  __shared__ int warp_counts[WB / 32];
  __shared__ int64_t s_slot[WB];
  __shared__ int64_t s_src[WB];   // flat (t, i) index of the newest transition of the window
  __shared__ int s_num;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t f = (int64_t)blockIdx.x * WB + tid;
  const uint8_t* emit_new = tr.emit + (int64_t)H * n;
  const int flag = (f < total_flags && emit_new[f]) ? 1 : 0;
  const unsigned ballot = __ballot_sync(0xffffffffu, flag);
  if (lane == 0) warp_counts[warp] = __popc(ballot);
  __syncthreads();
  int before = 0;
  for (int w = 0; w < warp; ++w) before += warp_counts[w];
  const int local = before + __popc(ballot & ((1u << lane) - 1u));
  if (tid == 0) {
    int s = 0;
    for (int w = 0; w < WB / 32; ++w) s += warp_counts[w];
    s_num = s;
  }
  const int64_t old_ptr = header[0], total = header[1];
  if (flag) {
    const int64_t order = block_offsets[blockIdx.x] + local;   // position in the reference's append order
    // windows that a later window of the same call would overwrite are skipped (sequential
    // store semantics: the last writer wins)
    const bool live = (total - order) <= ring.max_size;
    s_slot[local] = live ? (old_ptr + order) % ring.max_size : -1;
    s_src[local] = f + (int64_t)H * n;
  }
  __syncthreads();
  const int num = s_num;
  constexpr int G = 8;                 // windows per warp
  WindowCopier4<W, G> cp(tr, n, ring, lane);
  for (int w0 = warp * G; w0 < num; w0 += (WB / 32) * G) {
    const int w = w0 + lane / (32 / G);
    cp.copy(w < num ? s_src[w] : 0, w < num ? s_slot[w] : -1);
  }
}

// ---- index-based window store (SURVEY.md 8f-1): a window is the flat position of its newest transition in the
// [T][n][.] transition store the rollout kernel already wrote; nothing is copied at append time (8 bytes per window
// instead of 8 * n_step * (2D + A + 4)), and the n rows are gathered when a batch is sampled.
// Blocks of 256 threads x 16 flags (one 16-byte load per thread when the flag slice is 16-byte aligned): 4096 flags per
// block, so the single-CTA scan of the block counts has 16x fewer entries than with one flag per thread (2^25 flags:
// 8192 counts = 8 scan passes instead of 128 -- the scan was 0.2 ms of the 0.43 ms e2e overhead per launch).
constexpr int IPT = 16, IBF = WB * IPT;

__device__ __forceinline__ uint32_t load_flag_mask16(const uint8_t* __restrict__ emit, int64_t f0, int64_t total, bool vec) {
  uint32_t mask = 0;
  if (f0 >= total) return 0;
  if (vec && f0 + IPT <= total) {
    const uint4 v = *reinterpret_cast<const uint4*>(emit + f0);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int b = 0; b < 4; ++b)
        if ((w[q] >> (8 * b)) & 0xFFu) mask |= 1u << (4 * q + b);
  } else {
    for (int j = 0; j < IPT && f0 + j < total; ++j)
      if (emit[f0 + j]) mask |= 1u << j;
  }
  return mask;
}

__global__ void __launch_bounds__(WB) window_count16_kernel(const uint8_t* __restrict__ emit_new, int64_t total, int vec,
                                                            int64_t* __restrict__ block_counts) {
  __shared__ int warp_counts[WB / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int c = __popc(load_flag_mask16(emit_new, ((int64_t)blockIdx.x * WB + tid) * IPT, total, vec != 0));
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if (lane == 0) warp_counts[warp] = c;
  __syncthreads();
  if (tid == 0) {
    int s = 0;
    for (int w = 0; w < WB / 32; ++w) s += warp_counts[w];
    block_counts[blockIdx.x] = s;
  }
}

__global__ void __launch_bounds__(WB)
window_index_scatter_kernel(const uint8_t* __restrict__ emit_new, int64_t total_flags, int vec, int64_t base_pos,
                            int64_t* __restrict__ win_pos, int64_t max_size, const int64_t* __restrict__ block_offsets,
                            const int64_t* __restrict__ header) {
  __shared__ int warp_counts[WB / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t f0 = ((int64_t)blockIdx.x * WB + tid) * IPT;
  uint32_t mask = load_flag_mask16(emit_new, f0, total_flags, vec != 0);
  const int c = __popc(mask);
  int incl = c;                                    // inclusive warp scan of the per-thread counts
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += y;
  }
  if (lane == 31) warp_counts[warp] = incl;
  __syncthreads();
  if (!c) return;
  int before = incl - c;
  for (int w = 0; w < warp; ++w) before += warp_counts[w];
  int64_t order = block_offsets[blockIdx.x] + before;   // position of this thread's first window in the reference's append order
  const int64_t old_ptr = header[0], total = header[1];
  while (mask) {
    const int j = __ffs(mask) - 1;
    mask &= mask - 1;
    if ((total - order) <= max_size) win_pos[(old_ptr + order) % max_size] = base_pos + f0 + j;     // last writer wins
    ++order;
  }
}

template <int W>
__global__ void __launch_bounds__(256)
window_gather_indexed_kernel(msacl_transitions_t tr, int64_t n, const int64_t* __restrict__ win_pos,
                             const int64_t* __restrict__ idx, int64_t B, msacl_ring_t batch) {
  const int lane = threadIdx.x & 31;
  const int64_t wstride = (int64_t)gridDim.x * (blockDim.x / 32);
  WindowCopier<W> cp(tr, n, batch, lane);
  for (int64_t b = (int64_t)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5); b < B; b += wstride)
    cp.copy(win_pos[idx[b]], b);
}

// sample_batch of the index-based replay in ONE launch (nstep_replay_buffer.py:138-146: uniform with replacement over the
// stored windows): warp b draws u ~ U[0, 1) from Philox keyed by (seed, draw counter, b), walks `back = floor(u * valid)`
// entries back from the newest ring slot -- valid = min(size, windows emitted by the launches whose slices are still
// resident), all read from device counters, so the host never synchronises -- and gathers that window.
template <int W>
__global__ void __launch_bounds__(256)
window_sample_indexed_kernel(msacl_transitions_t tr, int64_t n, const int64_t* __restrict__ win_pos, int64_t max_size,
                             const int64_t* __restrict__ ptr_size, const int64_t* __restrict__ launch_counts, int n_counts,
                             uint64_t seed, uint64_t draw, int64_t B, msacl_ring_t batch, int64_t* __restrict__ slots_out) {
  const int lane = threadIdx.x & 31;
  const int64_t wstride = (int64_t)gridDim.x * (blockDim.x / 32);
  int64_t resident = 0;
  for (int i = 0; i < n_counts; ++i) resident += launch_counts[i];
  const int64_t ptr = ptr_size[0], size = ptr_size[1];
  const int64_t valid = size < resident ? size : resident;
  if (valid <= 0) return;                                  // nothing stored yet: the batch is left untouched
  WindowCopier<W> cp(tr, n, batch, lane);
  for (int64_t b = (int64_t)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5); b < B; b += wstride) {
    const U4 r = philox4x32_10((uint32_t)b, (uint32_t)((uint64_t)b >> 32), (uint32_t)draw, (uint32_t)(draw >> 32) ^ 0x5EED5A3Du,
                               (uint32_t)seed, (uint32_t)(seed >> 32));
    const uint64_t bits = ((uint64_t)(r.x >> 5) << 26) | (uint64_t)(r.y >> 6);          // 53 random bits
    const double u = (double)bits * 1.1102230246251565e-16;                               // * 2^-53: [0, 1)
    int64_t back = (int64_t)(u * (double)valid);
    if (back > valid - 1) back = valid - 1;
    int64_t slot = (ptr - 1 - back) % max_size;
    if (slot < 0) slot += max_size;
    if (slots_out && lane == 0) slots_out[b] = slot;
    cp.copy(win_pos[slot], b);
  }
}

// One warp per sampled window (grid-stride).  Every field of a window is a contiguous run of floats; with
// n_step % 4 == 0 (reference default 20) all runs are whole, 16-byte aligned float4 vectors, and the window is copied as
// ONE flat list of vectors (obs | obs2 | act | rew | cost | done | logp).  The vector -> (field, offset) map is the same
// for every window, so each lane resolves its (up to GATHER_MAX_VEC) vectors once, and per window only adds the slot
// offset: all loads of a window are in flight together, then the stores.  Other n_step: scalar run-by-run copy.
constexpr int GATHER_MAX_VEC = 6;     // covers n_step * (2D + A + 4) / 4 <= 192 vectors (e.g. n_step 24, D 12, A 4)

__device__ __forceinline__ void gather_vec_map(const msacl_ring_t& R, int i, int Lo, int La, int Ls, float*& base, int& stride) {
  const int ns = R.n_step;
  if (i < Lo) { base = R.obs + 4 * i; stride = ns * R.obs_dim; return; }
  i -= Lo;
  if (i < Lo) { base = R.obs2 + 4 * i; stride = ns * R.obs_dim; return; }
  i -= Lo;
  if (i < La) { base = R.act + 4 * i; stride = ns * R.act_dim; return; }
  i -= La;
  const int f = i / Ls, o = i - f * Ls;
  base = (f == 0 ? R.rew : (f == 1 ? R.cost : (f == 2 ? R.done : R.logp))) + 4 * o;
  stride = ns;
}

__device__ __forceinline__ void copy_run(float* __restrict__ dst, const float* __restrict__ src, int count, int lane) {
  for (int e = lane; e < count; e += 32) dst[e] = src[e];
}

// NV = float4 vectors per lane (ceil(vectors per window / 32)); 0 = scalar fallback
template <int NV>
__global__ void __launch_bounds__(256)
ring_gather_kernel(msacl_ring_t ring, const int64_t* __restrict__ idx, int64_t B, msacl_ring_t batch) {
  const int lane = threadIdx.x & 31;
  const int64_t wstride = (int64_t)gridDim.x * (blockDim.x / 32);
  int64_t b = (int64_t)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
  const int ns = ring.n_step, D = ring.obs_dim, A = ring.act_dim;
  const int Lo = ns * D / 4, La = ns * A / 4, Ls = ns / 4;
  const int total = 2 * Lo + La + 4 * Ls;
  if constexpr (NV > 0) {
    float* sbase[NV];
    float* dbase[NV];
    int stride[NV];
#pragma unroll
    for (int it = 0; it < NV; ++it) {
      const int i = it * 32 + lane;
      sbase[it] = nullptr; dbase[it] = nullptr; stride[it] = 0;
      if (i < total) { gather_vec_map(ring, i, Lo, La, Ls, sbase[it], stride[it]); gather_vec_map(batch, i, Lo, La, Ls, dbase[it], stride[it]); }
    }
    for (; b < B; b += wstride) {
      const int64_t s = idx[b];
      float4 v[NV];
#pragma unroll
      for (int it = 0; it < NV; ++it)
        if (it * 32 + lane < total) v[it] = *reinterpret_cast<const float4*>(sbase[it] + s * stride[it]);
#pragma unroll
      for (int it = 0; it < NV; ++it)
        if (it * 32 + lane < total) *reinterpret_cast<float4*>(dbase[it] + b * stride[it]) = v[it];
    }
  } else {
    for (; b < B; b += wstride) {
      const int64_t s = idx[b];
      copy_run(batch.obs + b * ns * D, ring.obs + s * ns * D, ns * D, lane);
      copy_run(batch.obs2 + b * ns * D, ring.obs2 + s * ns * D, ns * D, lane);
      copy_run(batch.act + b * ns * A, ring.act + s * ns * A, ns * A, lane);
      copy_run(batch.rew + b * ns, ring.rew + s * ns, ns, lane);
      copy_run(batch.cost + b * ns, ring.cost + s * ns, ns, lane);
      copy_run(batch.done + b * ns, ring.done + s * ns, ns, lane);
      copy_run(batch.logp + b * ns, ring.logp + s * ns, ns, lane);
    }
  }
}

}  // namespace msacl

using namespace msacl;

static int validate_ring(const msacl_ring_t* r) {
  if (!r || r->max_size <= 0 || r->n_step <= 0 || r->obs_dim <= 0 || r->act_dim <= 0 || !r->obs || !r->act ||
      !r->rew || !r->cost || !r->obs2 || !r->done || !r->logp) {
    set_error("invalid ring descriptor");
    return MSACL_ERR_BAD_ARG;
  }
  return MSACL_OK;
}

extern "C" int64_t msacl_window_store_scratch_elems(int32_t K, int64_t n) {
  if (K <= 0 || n <= 0) return 0;
  return 2 + ((int64_t)K * n + WB - 1) / WB;
}

extern "C" int msacl_window_store(const msacl_transitions_t* tr, int32_t H, int32_t K, int64_t n,
                                  const msacl_ring_t* ring, int64_t* ptr_size, int64_t* count_out, int64_t* scratch,
                                  void* stream) {
  if (int rc = validate_ring(ring)) return rc;
  if (!tr || !tr->obs || !tr->act || !tr->rew || !tr->cost || !tr->obs2 || !tr->done || !tr->logp || !tr->emit ||
      !ptr_size || !scratch || K <= 0 || n <= 0 || H < ring->n_step - 1) {
    set_error("window_store: bad argument (need all transition fields and H >= n_step-1)");
    return MSACL_ERR_BAD_ARG;
  }
  const int64_t total = (int64_t)K * n;
  const int64_t nb = (total + WB - 1) / WB;
  cudaStream_t s = (cudaStream_t)stream;
  window_count_kernel<<<(unsigned)nb, WB, 0, s>>>(tr->emit + (int64_t)H * n, total, scratch + 2);
  window_scan_kernel<<<1, 1024, 0, s>>>(scratch + 2, nb, scratch, ptr_size, count_out, ring->max_size);
  const int D = ring->obs_dim;
  auto misaligned = [&](const void* p, int w) { return (reinterpret_cast<uintptr_t>(p) & (uintptr_t)(4 * w - 1)) != 0; };
  int W = (D % 4 == 0) ? 4 : ((D % 2 == 0) ? 2 : 1);
  while (W > 1 && (misaligned(tr->obs, W) || misaligned(tr->obs2, W) || misaligned(ring->obs, W) || misaligned(ring->obs2, W))) W >>= 1;
  if (W == 4) window_scatter_kernel<4><<<(unsigned)nb, WB, 0, s>>>(*tr, H, n, total, *ring, scratch + 2, scratch);
  else if (W == 2) window_scatter_kernel<2><<<(unsigned)nb, WB, 0, s>>>(*tr, H, n, total, *ring, scratch + 2, scratch);
  else window_scatter_kernel<1><<<(unsigned)nb, WB, 0, s>>>(*tr, H, n, total, *ring, scratch + 2, scratch);
  return check_launch("window_store");
}

extern "C" int msacl_window_index_store(const uint8_t* emit_new, int32_t K, int64_t n, int64_t base_pos, int64_t* win_pos,
                                        int64_t max_size, int64_t* ptr_size, int64_t* count_out, int64_t* scratch,
                                        void* stream) {
  if (!emit_new || !win_pos || !ptr_size || !scratch || K <= 0 || n <= 0 || max_size <= 0 || base_pos < 0) {
    set_error("window_index_store: bad argument");
    return MSACL_ERR_BAD_ARG;
  }
  const int64_t total = (int64_t)K * n;
  const int64_t nb = (total + IBF - 1) / IBF;
  const int vec = (reinterpret_cast<uintptr_t>(emit_new) & 15) == 0 ? 1 : 0;
  cudaStream_t s = (cudaStream_t)stream;
  window_count16_kernel<<<(unsigned)nb, WB, 0, s>>>(emit_new, total, vec, scratch + 2);
  window_scan_kernel<<<1, 1024, 0, s>>>(scratch + 2, nb, scratch, ptr_size, count_out, max_size);
  window_index_scatter_kernel<<<(unsigned)nb, WB, 0, s>>>(emit_new, total, vec, base_pos, win_pos, max_size, scratch + 2, scratch);
  return check_launch("window_index_store");
}

extern "C" int msacl_window_gather_indexed(const msacl_transitions_t* tr, int64_t n, const int64_t* win_pos,
                                           const int64_t* idx, int64_t B, const msacl_ring_t* batch, void* stream) {
  if (int rc = validate_ring(batch)) return rc;
  if (!tr || !tr->obs || !tr->act || !tr->rew || !tr->cost || !tr->obs2 || !tr->done || !tr->logp || !win_pos || !idx ||
      B <= 0 || n <= 0) {
    set_error("window_gather_indexed: bad argument");
    return MSACL_ERR_BAD_ARG;
  }
  const int wpb = 8;
  const int64_t want = (B + wpb - 1) / wpb, cap = (int64_t)kNumSMs * 8;
  const unsigned grid = (unsigned)(want < cap ? want : cap);
  const int D = batch->obs_dim;
  auto misaligned = [&](const void* p, int w) { return (reinterpret_cast<uintptr_t>(p) & (uintptr_t)(4 * w - 1)) != 0; };
  int W = (D % 4 == 0) ? 4 : ((D % 2 == 0) ? 2 : 1);
  while (W > 1 && (misaligned(tr->obs, W) || misaligned(tr->obs2, W) || misaligned(batch->obs, W) || misaligned(batch->obs2, W))) W >>= 1;
  cudaStream_t st = (cudaStream_t)stream;
  if (W == 4) window_gather_indexed_kernel<4><<<grid, wpb * 32, 0, st>>>(*tr, n, win_pos, idx, B, *batch);
  else if (W == 2) window_gather_indexed_kernel<2><<<grid, wpb * 32, 0, st>>>(*tr, n, win_pos, idx, B, *batch);
  else window_gather_indexed_kernel<1><<<grid, wpb * 32, 0, st>>>(*tr, n, win_pos, idx, B, *batch);
  return check_launch("window_gather_indexed");
}

extern "C" int msacl_window_sample_indexed(const msacl_transitions_t* tr, int64_t n, const int64_t* win_pos, int64_t max_size,
                                           const int64_t* ptr_size, const int64_t* launch_counts, int32_t n_counts, uint64_t seed,
                                           uint64_t draw, int64_t B, const msacl_ring_t* batch, int64_t* slots_out, void* stream) {
  if (int rc = validate_ring(batch)) return rc;
  if (!tr || !tr->obs || !tr->act || !tr->rew || !tr->cost || !tr->obs2 || !tr->done || !tr->logp || !win_pos || !ptr_size ||
      !launch_counts || n_counts <= 0 || max_size <= 0 || B <= 0 || n <= 0) {
    set_error("window_sample_indexed: bad argument");
    return MSACL_ERR_BAD_ARG;
  }
  const int wpb = 8;
  const int64_t want = (B + wpb - 1) / wpb, cap = (int64_t)kNumSMs * 8;
  const unsigned grid = (unsigned)(want < cap ? want : cap);
  const int D = batch->obs_dim;
  auto misaligned = [&](const void* p, int w) { return (reinterpret_cast<uintptr_t>(p) & (uintptr_t)(4 * w - 1)) != 0; };
  int W = (D % 4 == 0) ? 4 : ((D % 2 == 0) ? 2 : 1);
  while (W > 1 && (misaligned(tr->obs, W) || misaligned(tr->obs2, W) || misaligned(batch->obs, W) || misaligned(batch->obs2, W))) W >>= 1;
  cudaStream_t st = (cudaStream_t)stream;
#define MSACL_SAMPLE_LAUNCH(W_)                                                                                                  \
  window_sample_indexed_kernel<W_><<<grid, wpb * 32, 0, st>>>(*tr, n, win_pos, max_size, ptr_size, launch_counts, n_counts, seed, draw, B, \
                                                              *batch, slots_out)
  if (W == 4) MSACL_SAMPLE_LAUNCH(4);
  else if (W == 2) MSACL_SAMPLE_LAUNCH(2);
  else MSACL_SAMPLE_LAUNCH(1);
#undef MSACL_SAMPLE_LAUNCH
  return check_launch("window_sample_indexed");
}

// idx[b] ~ U{0 .. size - 1} (nstep_replay_buffer.py:138 `np.random.randint(0, self.size, batch_size)`), Philox keyed by
// (seed, draw, b); size is read from the device counters
__global__ void __launch_bounds__(256) ring_draw_kernel(const int64_t* __restrict__ ptr_size, uint64_t seed, uint64_t draw, int64_t B,
                                                        int64_t* __restrict__ idx) {
  const int64_t size = ptr_size[1];
  for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (int64_t)gridDim.x * blockDim.x) {
    const U4 r = philox4x32_10((uint32_t)b, (uint32_t)((uint64_t)b >> 32), (uint32_t)draw, (uint32_t)(draw >> 32) ^ 0x5EED5A3Du,
                               (uint32_t)seed, (uint32_t)(seed >> 32));
    const uint64_t bits = ((uint64_t)(r.x >> 5) << 26) | (uint64_t)(r.y >> 6);
    int64_t i = (int64_t)((double)bits * 1.1102230246251565e-16 * (double)size);
    if (i > size - 1) i = size - 1;
    idx[b] = i < 0 ? 0 : i;
  }
}

extern "C" int msacl_ring_gather(const msacl_ring_t* ring, const int64_t* idx, int64_t B, const msacl_ring_t* batch, void* stream);

extern "C" int msacl_ring_sample(const msacl_ring_t* ring, const int64_t* ptr_size, uint64_t seed, uint64_t draw, int64_t B,
                                 const msacl_ring_t* batch, int64_t* idx, void* stream) {
  if (!ptr_size || !idx || B <= 0) { set_error("ring_sample: bad argument"); return MSACL_ERR_BAD_ARG; }
  const int64_t want = (B + 255) / 256;
  ring_draw_kernel<<<(unsigned)(want < 1184 ? want : 1184), 256, 0, (cudaStream_t)stream>>>(ptr_size, seed, draw, B, idx);
  if (int rc = check_launch("ring_sample")) return rc;
  return msacl_ring_gather(ring, idx, B, batch, stream);
}

extern "C" int msacl_ring_gather(const msacl_ring_t* ring, const int64_t* idx, int64_t B, const msacl_ring_t* batch,
                                 void* stream) {
  if (int rc = validate_ring(ring)) return rc;
  if (int rc = validate_ring(batch)) return rc;
  if (!idx || B <= 0) { set_error("ring_gather: bad argument"); return MSACL_ERR_BAD_ARG; }
  const int wpb = 8;
  const int ns = ring->n_step;
  const int total = ns * (2 * ring->obs_dim + ring->act_dim + 4) / 4;      // float4 vectors per window
  const int nv = ((ns & 3) == 0 && total <= 32 * GATHER_MAX_VEC) ? (total + 31) / 32 : 0;
  cudaStream_t st = (cudaStream_t)stream;
  switch (nv) {
    case 1: ring_gather_kernel<1><<<resident_grid(ring_gather_kernel<1>, wpb * 32, B, wpb), wpb * 32, 0, st>>>(*ring, idx, B, *batch); break;
    case 2: ring_gather_kernel<2><<<resident_grid(ring_gather_kernel<2>, wpb * 32, B, wpb), wpb * 32, 0, st>>>(*ring, idx, B, *batch); break;
    case 3: ring_gather_kernel<3><<<resident_grid(ring_gather_kernel<3>, wpb * 32, B, wpb), wpb * 32, 0, st>>>(*ring, idx, B, *batch); break;
    case 4: ring_gather_kernel<4><<<resident_grid(ring_gather_kernel<4>, wpb * 32, B, wpb), wpb * 32, 0, st>>>(*ring, idx, B, *batch); break;
    case 5: ring_gather_kernel<5><<<resident_grid(ring_gather_kernel<5>, wpb * 32, B, wpb), wpb * 32, 0, st>>>(*ring, idx, B, *batch); break;
    case 6: ring_gather_kernel<6><<<resident_grid(ring_gather_kernel<6>, wpb * 32, B, wpb), wpb * 32, 0, st>>>(*ring, idx, B, *batch); break;
    default: ring_gather_kernel<0><<<resident_grid(ring_gather_kernel<0>, wpb * 32, B, wpb), wpb * 32, 0, st>>>(*ring, idx, B, *batch); break;
  }
  return check_launch("ring_gather");
}
