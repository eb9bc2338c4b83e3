// tcgen05 split-bf16 GEMM with fused MLP epilogues: the dense layers of the MSACL learner's networks
// (ActionValue / LyapunovValue / StochaPolicy, RL/apprfunc/mlp.py:18-52,72-88,111-136) forward AND backward.
//
//     C[r][n] = epilogue( sum_k A(r, k) * B(n, k) ),   r < m, n < n_total, k < k_total
//
// A and B are FP32 in global memory behind (row stride, k stride) pairs, so the same kernel covers
//   forward   H = act(X W^T + b)          A = X [rows][in]      B = W [out][in]  (torch nn.Linear layout, K-major as is)
//   dgrad     dX = (dY W) * act'(X)       A = dY [rows][out]    B(n, k) = W[k][n]          (strided read of W)
//   wgrad     dW = dY^T X                 A(r, k) = dY[k][r]    B(n, k) = X[k][n]          (K = rows, split over CTAs)
// Operand tiles are converted on the fly by 4 loader warps: FP32 -> a sum of bf16 terms, written into the UMMA canonical
// K-major no-swizzle layout (tcgen05.cuh); one elected thread issues the cross products per 16-wide k-step with FP32
// accumulation in TMEM; 4 epilogue warps read the accumulator with tcgen05.ld and apply bias / activation /
// activation-derivative mask / row sum of squares, then store (or store split-K partials).  Two precisions:
//   NIMG = 3 ("bf16x6", default of the learner): x = x1 + x2 + x3 (24 mantissa bits), products a1b1 + a1b2 + a2b1 + a2b2 +
//            a1b3 + a3b1 -- error ~2^-23 per product, i.e. FP32-class: hidden units land on the same side of the ReLU kink
//            as an FP32 GEMM's, so post-Adam parameters reproduce the reference's at the cuBLAS engine's tolerance;
//   NIMG = 2 ("bf16x3", the rollout kernel's scheme): x = x1 + x2 (16 bits), a1b1 + a1b2 + a2b1 -- ~1.5e-5 per product,
//            half the tensor work and 2 CTAs per SM.
// CTA tile 128 x (<= 256) x 32 per stage, 2 stages (144 KB / 96 KB of shared memory).  Roofline: tensor.
#include "common.cuh"
#include "tcgen05.cuh"

namespace msacl {

constexpr int GM = 128, GN = 256, GK = 32;  // GN = widest column tile (template BN: 256, or 64 for small row counts)
constexpr int GA_HALF = GM * GK * 2;       // 8 KB: one bf16 image of an A stage
constexpr int GA_LBO = GM * 16, G_SBO = 128;
// 17 warps (five per SM sub-partition at most: 96 registers per thread).  Warp 16 issues the UMMAs; the other sixteen are
// split by operand mode:
//   streamed weights (pre-packed B by bulk copies, k-contiguous A):  warps 0-7 epilogue (two per TMEM lane quadrant, each
//       owning half of the columns), warps 8-15 convert the A tile (256 threads, software-pipelined);
//   converted B (weight gradient, un-packed weights):                warps 0-3 epilogue, warps 4-15 loaders (threads
//       0..127 of the group own the A tile, 128..383 the B tile).
constexpr int G_LOADERS = 384;
constexpr int G_MMA_WARP = 16;
constexpr int G_THREADS = 32 * (G_MMA_WARP + 1);

// streamed mode: the K blocks of an A image are 32 bytes further apart (LBO = 128 * 16 + 32), so that the loader's 16-byte
// stores -- a quarter-warp holds the 4 K blocks of 2 adjacent rows -- fall into 8 different 16-byte bank groups
constexpr int GA_LBO_S = GM * 16 + 32, GA_HALF_S = 4 * GA_LBO_S;
template <int NIMG, int BN, int STAGES, bool STREAMED = false>
struct GemmSmem {
  alignas(128) unsigned char a[STAGES][NIMG * (STREAMED ? GA_HALF_S : GA_HALF)];
  alignas(128) unsigned char b[STAGES][NIMG * BN * GK * 2];
  alignas(16) float bias[BN];
  float ss_part[GM];
  unsigned long long full[STAGES], empty[STAGES], accfull[2], accfree[2];
  uint32_t tmem_slot;
};

// 256-bit global accesses (sm_100: LDG / STG .ENL2.256); the address must be 32-byte aligned
__device__ __forceinline__ void g_stg256(float* p, const float (&v)[8]) {
  asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]),
               "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]) : "memory");
}
__device__ __forceinline__ void g_ldg256(const float* p, float (&v)[8]) {
  asm volatile("ld.global.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]),
               "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]) : "l"(p));
}

__device__ __forceinline__ uint32_t g_pack_bf16x2_rn(float lo, float hi) {   // {hi:lo} packed, RNE
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// 8 floats -> NIMG images of 8 bf16: image i holds bf16(x - sum of the previous images) (every subtraction is exact)
template <int NIMG>
__device__ __forceinline__ void g_split8(const float (&v)[8], uint4 (&img)[NIMG]) {
  float r[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) r[j] = v[j];
#pragma unroll
  for (int i = 0; i < NIMG; ++i) {
    uint32_t h[4];
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      h[p] = g_pack_bf16x2_rn(r[2 * p], r[2 * p + 1]);
      r[2 * p] -= __uint_as_float(h[p] << 16);
      r[2 * p + 1] -= __uint_as_float(h[p] & 0xFFFF0000u);
    }
    img[i] = make_uint4(h[0], h[1], h[2], h[3]);
  }
}

// k-contiguous operand (k stride 1, rows 16-byte aligned): a group of GSZ threads loads a `rows` x 32 tile as float4 chunks,
// consecutive lanes on consecutive chunks (a warp instruction covers 4 whole 128-byte rows: fully coalesced, 4 L1 tags
// instead of 32).  Thread t keeps chunk c = t % 8 (K block c / 2, half c % 2) of rows t / 8 + j * GSZ / 8; each chunk becomes one
// 8-byte store per image (4-way bank conflict among the 4 K blocks of a row group, ~1k cycles per stage).
template <int GSZ, int ROWS>
__device__ __forceinline__ void g_kcontig_load(float4 (&v)[ROWS * 8 / GSZ], const float* __restrict__ src, int64_t rs, int64_t row0,
                                               int64_t row_limit, int rows_used, int k0, int kend, int t) {
  constexpr int NIT = ROWS * 8 / GSZ;
  const int kk = k0 + (t & 7) * 4;
#pragma unroll
  for (int j = 0; j < NIT; ++j) {
    const int rl = (t >> 3) + j * (GSZ / 8);
    const int64_t row = row0 + rl;
    v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (rl < rows_used && row < row_limit) {
      const float* p = src + row * rs + kk;
      if (kk + 3 < kend) v[j] = *reinterpret_cast<const float4*>(p);
      else {
        if (kk < kend) v[j].x = p[0];
        if (kk + 1 < kend) v[j].y = p[1];
        if (kk + 2 < kend) v[j].z = p[2];
      }
    }
  }
}

template <int LBO, int HALF, int NIMG, int GSZ, int ROWS>
__device__ __forceinline__ void g_kcontig_store(unsigned char* img0, const float4 (&v)[ROWS * 8 / GSZ], int rows_used, int t) {
  constexpr int NIT = ROWS * 8 / GSZ;
  const int c = t & 7;
#pragma unroll
  for (int j = 0; j < NIT; ++j) {
    const int rl = (t >> 3) + j * (GSZ / 8);
    if (rl >= rows_used) continue;
    float r[4] = {v[j].x, v[j].y, v[j].z, v[j].w};
    unsigned char* dst = img0 + (c >> 1) * LBO + rl * 16 + (c & 1) * 8;
#pragma unroll
    for (int i = 0; i < NIMG; ++i) {
      const uint32_t h0 = g_pack_bf16x2_rn(r[0], r[1]), h1 = g_pack_bf16x2_rn(r[2], r[3]);
      r[0] -= __uint_as_float(h0 << 16); r[1] -= __uint_as_float(h0 & 0xFFFF0000u);
      r[2] -= __uint_as_float(h1 << 16); r[3] -= __uint_as_float(h1 & 0xFFFF0000u);
      *reinterpret_cast<uint2*>(dst + i * HALF) = make_uint2(h0, h1);
    }
  }
}

// Streamed mode, 256 loader threads, a 128 x 32 A stage: thread t owns K block kb = t & 3 (8 consecutive k = 32 bytes, one
// 256-bit load) of rows (t >> 2) + 64 j, j = 0, 1 -- a warp instruction covers 8 whole 128-byte rows -- and turns each into ONE
// 16-byte store per image.  Needs 32-byte aligned rows (row stride % 8 == 0); the host checks.
__device__ __forceinline__ void g_k8_load(float (&v)[2][8], const float* __restrict__ src, int64_t rs, int64_t row0, int64_t row_limit,
                                          int k0, int kend, int t) {
  const int kk = k0 + (t & 3) * 8;
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const int64_t row = row0 + (t >> 2) + 64 * j;
#pragma unroll
    for (int e = 0; e < 8; ++e) v[j][e] = 0.f;
    if (row < row_limit) {
      const float* p = src + row * rs + kk;
      if (kk + 7 < kend) g_ldg256(p, v[j]);
      else {
#pragma unroll
        for (int e = 0; e < 8; ++e) if (kk + e < kend) v[j][e] = p[e];
      }
    }
  }
}

template <int LBO, int HALF, int NIMG>
__device__ __forceinline__ void g_k8_store(unsigned char* img0, const float (&v)[2][8], int t) {
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    uint4 img[NIMG];
    g_split8<NIMG>(v[j], img);
    unsigned char* dst = img0 + (t & 3) * LBO + ((t >> 2) + 64 * j) * 16;
#pragma unroll
    for (int i = 0; i < NIMG; ++i) *reinterpret_cast<uint4*>(dst + i * HALF) = img[i];
  }
}

template <int LBO, int HALF, int NIMG, int GSZ, int ROWS>
__device__ __forceinline__ void g_load_tile_kcontig(unsigned char* img0, const float* __restrict__ src, int64_t rs, int64_t row0,
                                                    int64_t row_limit, int rows_used, int k0, int kend, int t) {
  float4 v[ROWS * 8 / GSZ];
  g_kcontig_load<GSZ, ROWS>(v, src, rs, row0, row_limit, rows_used, k0, kend, t);
  g_kcontig_store<LBO, HALF, NIMG, GSZ, ROWS>(img0, v, rows_used, t);
}

// One operand row (local index rl, global row index `row`) of a 32-wide K stage -> 4 K blocks of 8 into the hi / lo images.
// All 32 loads are issued before the first conversion (memory-level parallelism).
template <int LBO, int HALF, int NIMG>
__device__ __forceinline__ void g_load_row(unsigned char* img0, const float* __restrict__ src, int64_t rs,
                                           int64_t ks, int64_t row, bool row_ok, int k0, int kend, int rl, bool vec) {
  float v[4][8];
  if (row_ok && vec && k0 + GK <= kend) {
    const float4* p = reinterpret_cast<const float4*>(src + row * rs + k0);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float4 t = p[i];
      v[i >> 1][(i & 1) * 4 + 0] = t.x; v[i >> 1][(i & 1) * 4 + 1] = t.y; v[i >> 1][(i & 1) * 4 + 2] = t.z; v[i >> 1][(i & 1) * 4 + 3] = t.w;
    }
  } else {
#pragma unroll
    for (int kb = 0; kb < 4; ++kb)
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int k = k0 + kb * 8 + j;
        v[kb][j] = (row_ok && k < kend) ? src[row * rs + (int64_t)k * ks] : 0.f;
      }
  }
#pragma unroll
  for (int kb = 0; kb < 4; ++kb) {
    uint4 img[NIMG];
    g_split8<NIMG>(v[kb], img);
#pragma unroll
    for (int i = 0; i < NIMG; ++i) *reinterpret_cast<uint4*>(img0 + i * HALF + kb * LBO + rl * 16) = img[i];
  }
}

// Pre-packed B operand (weights): the bf16 images of every 32-wide K stage, exactly as a CTA's shared-memory B stage holds
// them ([NIMG][4 K blocks][256 rows][16 B], rows >= n and k >= k_total zero), so that a GEMM over many row tiles streams
// them with one cp.async.bulk per stage instead of re-converting the same 256 x 256 weights in every CTA.
template <int NIMG>
__global__ void __launch_bounds__(256) gemm_pack_b_kernel(msacl_gemm_t g, unsigned char* __restrict__ packed) {
  constexpr int GB_HALF = GN * GK * 2, GB_LBO = GN * 16;
  const int stages = (g.k + GK - 1) / GK;
  const int64_t total = (int64_t)stages * 4 * GN;            // one thread per (stage, K block, row)
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int row = (int)(i % GN), kb = (int)((i / GN) % 4), st = (int)(i / (4 * GN));
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = st * GK + kb * 8 + j;
      v[j] = (row < g.n && k < g.k) ? g.b[(int64_t)row * g.b_row_stride + (int64_t)k * g.b_k_stride] : 0.f;
    }
    uint4 img[NIMG];
    g_split8<NIMG>(v, img);
    unsigned char* dst = packed + (size_t)st * NIMG * GB_HALF + kb * GB_LBO + row * 16;
#pragma unroll
    for (int q = 0; q < NIMG; ++q) *reinterpret_cast<uint4*>(dst + q * GB_HALF) = img[q];
  }
}

// BN = column tile (UMMA N <= BN), STAGES = shared-memory stages.  Persistent CTAs (one per SM) walk the output tiles with a
// static stride; the accumulator is double-buffered in TMEM (2 x BN columns), so the epilogue of tile i (TMEM -> bias /
// activation -> global) overlaps the loads and UMMAs of tile i + 1 -- ncu had the epilogue at ~2/3 of a tile's lifetime
// with every other warp idle at the teardown barrier.  <*, 256, *>: large row counts (one column tile covers a 256-wide
// layer); <*, 128, *> / <*, 64, *>: small row counts -- more CTAs in the single wave, so a GEMM over a few thousand rows (the
// reference's replay batch: 256 windows x 20 steps) is not serialised behind one tile's load latency.
struct GemmTile {
  int m0, n0, z, kbeg, kend, nk, n_rem, n_mma;
};

template <int BN>
__device__ __forceinline__ GemmTile gemm_tile(const msacl_gemm_t& g, int64_t tile, int mtiles, int ntiles) {
  GemmTile t;
  const int64_t per_z = (int64_t)mtiles * ntiles;
  t.z = (int)(tile / per_z);
  const int64_t rem = tile - (int64_t)t.z * per_z;
  const int y = (int)(rem / mtiles);
  t.m0 = (int)(rem - (int64_t)y * mtiles) * GM;
  t.n0 = y * BN;
  const int kper = ((g.k + g.split_k - 1) / g.split_k + GK - 1) / GK * GK;     // K range of a split: multiples of the stage width
  t.kbeg = t.z * kper;
  t.kend = min(g.k, t.kbeg + kper);
  t.nk = t.kend > t.kbeg ? (t.kend - t.kbeg + GK - 1) / GK : 0;
  t.n_rem = g.n - t.n0;
  t.n_mma = t.n_rem >= BN ? BN : ((t.n_rem + 15) / 16) * 16;                   // UMMA N: multiple of 16, 16..256
  return t;
}

// STREAMED (BN = 256 only): the host found a pre-packed B operand behind a k-contiguous A -- its own instantiation, so that
// the software-pipelined A loader does not share a register allocation with the converting loaders of the other mode.
template <int NIMG, int BN, int STAGES, bool STREAMED>
__global__ void __launch_bounds__(G_THREADS, 1) gemm_tc_kernel(msacl_gemm_t g) {
  constexpr int G_STAGES = STAGES;
  constexpr int GN = BN, GB_HALF = BN * GK * 2, GB_LBO = BN * 16;
  constexpr uint32_t TMEM_COLS = 2 * BN < 32 ? 32 : 2 * BN;          // two accumulator buffers (512 / 256 / 128 columns)
  extern __shared__ __align__(128) unsigned char smem_raw[];
  GemmSmem<NIMG, BN, STAGES, STREAMED>& sm = *reinterpret_cast<GemmSmem<NIMG, BN, STAGES, STREAMED>*>(smem_raw);
  constexpr int A_LBO = STREAMED ? GA_LBO_S : GA_LBO, A_HALF = STREAMED ? GA_HALF_S : GA_HALF;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int mtiles = (g.m + GM - 1) / GM, ntiles = (g.n + BN - 1) / BN;
  const int64_t total_tiles = (int64_t)mtiles * ntiles * g.split_k;

  // packed B (BN = 256 only): the B tile arrives by one bulk copy per stage (expect_tx arrival of the issuing thread)
  const bool packed_b = STREAMED || (BN == 256 && g.b_packed != nullptr);
  constexpr bool streamed = STREAMED;                  // role split (see G_THREADS)
  const int epi_warps = streamed ? 8 : 4, epi_threads = 32 * epi_warps;
  // arrivals per full stage: streamed -- 256 A threads + the bulk-copy expect_tx of A thread 0; packed B behind a strided A --
  // 128 A threads + the issuer; else all 384 loaders
  if (tid == 0) {
    for (int s = 0; s < G_STAGES; ++s) { tc::mbar_init(&sm.full[s], streamed ? 256 + 1 : (packed_b ? 128 + 1 : G_LOADERS)); tc::mbar_init(&sm.empty[s], 1); }
    for (int b = 0; b < 2; ++b) { tc::mbar_init(&sm.accfull[b], 1); tc::mbar_init(&sm.accfree[b], epi_threads); }
    tc::mbar_fence_init();
  }
  if (warp == G_MMA_WARP) tc::tmem_alloc(&sm.tmem_slot, TMEM_COLS);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = sm.tmem_slot;

  if (warp >= epi_warps && warp < G_MMA_WARP) {
    // =========================== loaders: FP32 global -> split-bf16 operand images ===========================
    // threads 0..127 of the loader group own the A tile (128 rows), threads 128..383 the B tile (<= 256 rows): one row (or
    // 8 coalesced float4 chunks) per thread per stage, so a stage costs one global round trip.
    const int t = tid - epi_threads;
    if constexpr (streamed) {
      // ---- A tile, k-contiguous, many row tiles (packed B): software-pipelined with G_LOOK register buffers -- the global
      //      loads of the next G_LOOK - 1 stages (across tile boundaries) are in flight while a stage is converted and
      //      stored (ncu, one-stage version: loader samples 46 % long-scoreboard, a stage cost ~4 k cycles against 1.5 k of
      //      UMMAs).  The buffers rotate by unrolling, never by register moves (a move of an in-flight load's destination
      //      would wait for it).
      constexpr int G_LOOK = 3;
      // fetch cursor: the position (tile, k stage) G_LOOK stages ahead of the one being stored
      int64_t ctile = blockIdx.x;
      GemmTile ctl;
      int cit = 0;
      bool cok = ctile < total_tiles;
      auto settle = [&]() {                           // skip tiles without k stages, stop behind the last tile
        while (cok && cit >= ctl.nk) {
          ctile += gridDim.x; cit = 0;
          cok = ctile < total_tiles;
          if (cok) ctl = gemm_tile<BN>(g, ctile, mtiles, ntiles);
        }
      };
      if (cok) ctl = gemm_tile<BN>(g, ctile, mtiles, ntiles);
      settle();
      float r[G_LOOK][2][8];
      int kst[G_LOOK];
      bool ok[G_LOOK];
      auto refill = [&](int ph) {
        ok[ph] = cok;
        if (cok) {
          g_k8_load(r[ph], g.a, g.a_row_stride, ctl.m0, g.m, ctl.kbeg + cit * GK, ctl.kend, t);
          kst[ph] = (ctl.kbeg + cit * GK) / GK;
          ++cit;
          settle();
        }
      };
#pragma unroll
      for (int ph = 0; ph < G_LOOK; ++ph) refill(ph);
      uint32_t gs = 0;
      bool more = true;
      while (more) {
#pragma unroll
        for (int ph = 0; ph < G_LOOK; ++ph) {
          if (!more) break;
          if (!ok[ph]) { more = false; break; }
          const int s = gs % G_STAGES;
          if (gs >= G_STAGES) tc::mbar_wait(&sm.empty[s], (uint32_t)((gs / G_STAGES - 1) & 1));
          if (t == 0) {                                 // the stage's B tile: one bulk copy of the pre-packed images
            constexpr uint32_t bytes = NIMG * GB_HALF;
            tc::mbar_expect_tx(&sm.full[s], bytes);
            tc::tma_bulk_g2s(sm.b[s], static_cast<const unsigned char*>(g.b_packed) + (size_t)kst[ph] * bytes, bytes, &sm.full[s]);
          }
          g_k8_store<A_LBO, A_HALF, NIMG>(sm.a[s], r[ph], t);
          tc::fence_async_smem();
          tc::mbar_arrive(&sm.full[s]);
          ++gs;
          refill(ph);
        }
      }
    } else if (t < 128 || !packed_b || t == 128) {    // (packed B behind a strided A: thread 128 issues the bulk copies)
      const bool avec = g.a_k_stride == 1 && (g.a_row_stride & 3) == 0 && (reinterpret_cast<uintptr_t>(g.a) & 15) == 0;
      const bool bvec = g.b_k_stride == 1 && (g.b_row_stride & 3) == 0 && (reinterpret_cast<uintptr_t>(g.b) & 15) == 0;
      const bool a_role = t < 128;                    // A tile: one row (or 8 coalesced chunks) per thread
      uint32_t gs = 0;                                     // stage counter over all tiles of this CTA
      for (int64_t tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const GemmTile tl = gemm_tile<BN>(g, tile, mtiles, ntiles);
        for (int it = 0; it < tl.nk; ++it, ++gs) {
          const int s = gs % G_STAGES;
          if (gs >= G_STAGES) tc::mbar_wait(&sm.empty[s], (uint32_t)((gs / G_STAGES - 1) & 1));
          const int k0 = tl.kbeg + it * GK;
          if (a_role) {
            if (avec) g_load_tile_kcontig<A_LBO, A_HALF, NIMG, 128, GM>(sm.a[s], g.a, g.a_row_stride, tl.m0, g.m, GM, k0, tl.kend, t);
            else g_load_row<A_LBO, A_HALF, NIMG>(sm.a[s], g.a, g.a_row_stride, g.a_k_stride, tl.m0 + t, tl.m0 + t < g.m, k0, tl.kend, t, false);
          } else if (packed_b) {
            constexpr uint32_t bytes = NIMG * GB_HALF;
            tc::mbar_expect_tx(&sm.full[s], bytes);
            tc::tma_bulk_g2s(sm.b[s], static_cast<const unsigned char*>(g.b_packed) + (size_t)(k0 / GK) * bytes, bytes, &sm.full[s]);
            continue;                                 // (the expect_tx above is this thread's arrival)
          } else {
            const int tb = t - 128;
            if (bvec) g_load_tile_kcontig<GB_LBO, GB_HALF, NIMG, 256, (GN >= 32 ? GN : 32)>(sm.b[s], g.b, g.b_row_stride, tl.n0, g.n, tl.n_mma, k0, tl.kend, tb);
            else if (tb < tl.n_mma) g_load_row<GB_LBO, GB_HALF, NIMG>(sm.b[s], g.b, g.b_row_stride, g.b_k_stride, tl.n0 + tb, tl.n0 + tb < g.n, k0, tl.kend, tb, false);
          }
          tc::fence_async_smem();
          tc::mbar_arrive(&sm.full[s]);
        }
      }
    }
  } else if (warp == G_MMA_WARP) {
    // =========================== MMA issuer ===========================
    if (tc::elect_one()) {
      uint32_t gs = 0, li = 0;                            // stage counter, local tile counter
      for (int64_t tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++li) {
        const GemmTile tl = gemm_tile<BN>(g, tile, mtiles, ntiles);
        const uint32_t buf = li & 1u;
        if (li >= 2) tc::mbar_wait(&sm.accfree[buf], (uint32_t)(((li >> 1) - 1) & 1));     // epilogue of tile li - 2 has drained this buffer
        tc::tc_fence_after();
        const uint32_t tacc = tmem + buf * (uint32_t)BN;
        const uint32_t idesc = tc::make_idesc_bf16(GM, tl.n_mma);
        for (int it = 0; it < tl.nk; ++it, ++gs) {
          const int s = gs % G_STAGES;
          tc::mbar_wait(&sm.full[s], (uint32_t)((gs / G_STAGES) & 1));
          tc::tc_fence_after();
          const uint32_t ab = tc::smem_u32(sm.a[s]), bb = tc::smem_u32(sm.b[s]);
#pragma unroll
          for (int j = 0; j < GK / 16; ++j) {
            uint64_t da[NIMG], db[NIMG];
#pragma unroll
            for (int i = 0; i < NIMG; ++i) {
              da[i] = tc::make_smem_desc(ab + i * A_HALF + j * 2 * A_LBO, A_LBO, G_SBO);
              db[i] = tc::make_smem_desc(bb + i * GB_HALF + j * 2 * GB_LBO, GB_LBO, G_SBO);
            }
            tc::umma_bf16(tacc, da[0], db[0], idesc, (it > 0 || j > 0) ? 1u : 0u);
            tc::umma_bf16(tacc, da[0], db[1], idesc, 1u);
            tc::umma_bf16(tacc, da[1], db[0], idesc, 1u);
            if constexpr (NIMG == 3) {
              tc::umma_bf16(tacc, da[1], db[1], idesc, 1u);
              tc::umma_bf16(tacc, da[0], db[2], idesc, 1u);
              tc::umma_bf16(tacc, da[2], db[0], idesc, 1u);
            }
          }
          tc::umma_commit(&sm.empty[s]);
        }
        tc::umma_commit(&sm.accfull[buf]);
      }
    }
  } else {
    // =========================== epilogue: TMEM -> bias / activation / mask -> global ===========================
    const int q = warp & 3, half = warp >> 2;          // TMEM lane quadrant (rows 32 q ..), column half (streamed mode: two halves)
    const bool two_halves = epi_warps == 8;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const bool cvec = (g.ldc & 3) == 0 && (reinterpret_cast<uintptr_t>(g.c) & 15) == 0 && (g.c_split_stride & 3) == 0;
    const bool cvec8 = (g.ldc & 7) == 0 && (reinterpret_cast<uintptr_t>(g.c) & 31) == 0 && (g.c_split_stride & 7) == 0;
    const bool mvec8 = g.mask_src && (g.mask_ld & 7) == 0 && (reinterpret_cast<uintptr_t>(g.mask_src) & 31) == 0;
    const bool mvec = g.mask_src && (g.mask_ld & 3) == 0 && (reinterpret_cast<uintptr_t>(g.mask_src) & 15) == 0;
    uint32_t li = 0;
    for (int64_t tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++li) {
      const GemmTile tl = gemm_tile<BN>(g, tile, mtiles, ntiles);
      const uint32_t buf = li & 1u;
      const uint32_t tacc = tmem + buf * (uint32_t)BN;
      const int row = tl.m0 + q * 32 + lane;
      const bool row_ok = row < g.m;
      const int nchunks = (tl.n_mma + 31) / 32, c_mid = two_halves ? (nchunks + 1) / 2 : nchunks;
      const int c_lo = half == 0 ? 0 : c_mid, c_hi = half == 0 ? c_mid : nchunks;
      float* crow = g.c + (int64_t)tl.z * g.c_split_stride + (int64_t)row * g.ldc + tl.n0;
      const float* mrow = g.mask_src ? g.mask_src + (int64_t)row * g.mask_ld + tl.n0 : nullptr;
      // bias of this column tile -> shared memory (the per-column global loads were most of the epilogue's stall time)
      asm volatile("bar.sync 1, %0;" ::"r"(epi_threads) : "memory");   // every epilogue warp is done with the previous tile's bias
      if (g.bias)
        for (int c = tid; c < BN; c += epi_threads) sm.bias[c] = (c < tl.n_rem) ? g.bias[tl.n0 + c] : 0.f;
      asm volatile("bar.sync 1, %0;" ::"r"(epi_threads) : "memory");
      float ss = 0.f;
      tc::mbar_wait(&sm.accfull[buf], (uint32_t)((li >> 1) & 1));
      tc::tc_fence_after();
      if (c_lo >= c_hi) {                               // (narrow tiles: the second half has no columns)
        tc::tc_fence_before();
        tc::mbar_arrive(&sm.accfree[buf]);
      }
      for (int c = c_lo * 32; c < c_hi * 32; c += 32) {
        uint32_t v[32];
        if (tl.nk == 0) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = 0u;
        } else if (tl.n_mma - c >= 32) {
          tc::tmem_ld32(tacc + lane_addr + (uint32_t)c, v);
          tc::tmem_ld_wait();
        } else {
          uint32_t w[16];
          tc::tmem_ld16(tacc + lane_addr + (uint32_t)c, w);
          tc::tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) { v[j] = w[j]; v[16 + j] = 0u; }
        }
        if (c + 32 >= c_hi * 32) {                      // last accumulator read of this warp: hand the buffer back to the MMA thread
          tc::tc_fence_before();
          tc::mbar_arrive(&sm.accfree[buf]);
        }
        if (!row_ok) continue;
#pragma unroll
        for (int j8 = 0; j8 < 32; j8 += 8) {
          const int col8 = c + j8;                // tile-local column of this group of 8
          if (col8 >= tl.n_rem) break;
          float x[8];
          float m8[8];
          const bool m8ok = mrow && mvec8 && col8 + 7 < tl.n_rem;      // activation-derivative source: one 32-byte load
          if (m8ok) g_ldg256(mrow + col8, m8);
#pragma unroll
          for (int hq = 0; hq < 2; ++hq) {
            const int col = col8 + 4 * hq;
            float* xs = x + 4 * hq;
#pragma unroll
            for (int j = 0; j < 4; ++j) xs[j] = __uint_as_float(v[j8 + 4 * hq + j]);
            if (col >= tl.n_rem) continue;
            const bool full4 = col + 3 < tl.n_rem;
            if (g.bias) {
              const float4 bb = *reinterpret_cast<const float4*>(&sm.bias[col]);
              xs[0] += bb.x; xs[1] += bb.y; xs[2] += bb.z; xs[3] += bb.w;
            }
            if (g.act == 1) {
#pragma unroll
              for (int j = 0; j < 4; ++j) xs[j] = fmaxf(xs[j], 0.f);
            } else if (g.act == 2) {
#pragma unroll
              for (int j = 0; j < 4; ++j) xs[j] = tanhf(xs[j]);
            }
            if (mrow) {
              float hsrc[4];
              if (m8ok) {
#pragma unroll
                for (int j = 0; j < 4; ++j) hsrc[j] = m8[4 * hq + j];
              } else if (mvec && full4) {
                const float4 t4 = *reinterpret_cast<const float4*>(mrow + col);
                hsrc[0] = t4.x; hsrc[1] = t4.y; hsrc[2] = t4.z; hsrc[3] = t4.w;
              } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) hsrc[j] = (col + j < tl.n_rem) ? mrow[col + j] : 0.f;
              }
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                if (g.mask_act == 1) xs[j] = hsrc[j] > 0.f ? xs[j] : 0.f;                       // relu'(pre) = [post > 0]
                else if (g.mask_act == 2) xs[j] = xs[j] * (1.0f - hsrc[j] * hsrc[j]);           // tanh'(pre) = 1 - post^2
              }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) if (col + j < tl.n_rem) ss = __fmaf_rn(xs[j], xs[j], ss);
          }
          if (cvec8 && col8 + 7 < tl.n_rem) {
            // one 32-byte store per lane (STG.256): a whole sector, half the store instructions / LSU wavefronts of two
            // 16-byte stores (the thread-per-row epilogue touches 32 lines per instruction either way)
            g_stg256(crow + col8, x);
          } else {
#pragma unroll
            for (int hq = 0; hq < 2; ++hq) {
              const int col = col8 + 4 * hq;
              if (col >= tl.n_rem) break;
              if (cvec && col + 3 < tl.n_rem) {
                *reinterpret_cast<float4*>(crow + col) = make_float4(x[4 * hq], x[4 * hq + 1], x[4 * hq + 2], x[4 * hq + 3]);
              } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) if (col + j < tl.n_rem) crow[col + j] = x[4 * hq + j];
              }
            }
          }
        }
      }
      if (g.row_sumsq) {
        if (two_halves) {                               // combine the two column halves of a row
          if (half == 1) sm.ss_part[q * 32 + lane] = ss;
          asm volatile("bar.sync 1, 256;" ::: "memory");
          if (half == 0 && row_ok) g.row_sumsq[row] = ss + sm.ss_part[q * 32 + lane];
        } else if (row_ok) {
          g.row_sumsq[row] = ss;
        }
      }
    }
  }
  // ---- teardown
  tc::tc_fence_before();
  __syncthreads();
  if (warp == G_MMA_WARP) tc::tmem_dealloc(tmem, TMEM_COLS);
}

}  // namespace msacl

using namespace msacl;

extern "C" int64_t msacl_gemm_packed_b_bytes(int32_t k, int32_t precision) {
  if (k <= 0) return 0;
  const int nimg = precision == 3 ? 2 : 3;
  return (int64_t)((k + GK - 1) / GK) * nimg * GN * GK * 2;
}

extern "C" int msacl_gemm_pack_b(const msacl_gemm_t* g, void* packed, void* stream) {
  if (!g || !g->b || !packed || g->n <= 0 || g->n > GN || g->k <= 0 || (reinterpret_cast<uintptr_t>(packed) & 15)) {
    set_error("gemm_pack_b: bad argument (needs n <= 256 and a 16-byte aligned destination)");
    return MSACL_ERR_BAD_ARG;
  }
  const int stages = (g->k + GK - 1) / GK;
  const unsigned grid = (unsigned)((stages * 4 * GN + 255) / 256);
  if (g->precision == 3) gemm_pack_b_kernel<2><<<grid, 256, 0, (cudaStream_t)stream>>>(*g, (unsigned char*)packed);
  else gemm_pack_b_kernel<3><<<grid, 256, 0, (cudaStream_t)stream>>>(*g, (unsigned char*)packed);
  return check_launch("gemm_pack_b");
}

extern "C" int msacl_gemm_tc(const msacl_gemm_t* g, void* stream) {
  if (!g || !g->a || !g->b || !g->c || g->m <= 0 || g->n <= 0 || g->k <= 0 || g->split_k < 1 || g->ldc < 1) {
    set_error("gemm_tc: bad argument");
    return MSACL_ERR_BAD_ARG;
  }
  if (g->act < 0 || g->act > 2 || g->mask_act < 0 || g->mask_act > 2 || (g->mask_src && g->mask_act == 0)) {
    set_error("gemm_tc: unknown activation code (0 none, 1 relu, 2 tanh)");
    return MSACL_ERR_BAD_ARG;
  }
  if (g->split_k > 1 && (g->bias || g->act || g->mask_src || g->row_sumsq)) {
    set_error("gemm_tc: split-K partials take no epilogue (bias / act / mask / row_sumsq)");
    return MSACL_ERR_BAD_ARG;
  }
  if (g->b_packed && (g->split_k != 1 || (reinterpret_cast<uintptr_t>(g->b_packed) & 15) || g->n > GN)) {
    set_error("gemm_tc: b_packed needs split_k == 1, n <= 256 and 16-byte alignment");
    return MSACL_ERR_BAD_ARG;
  }
  if (g->row_sumsq && g->n > GN) { set_error("gemm_tc: row_sumsq needs n <= 256 (one column tile)"); return MSACL_ERR_BAD_ARG; }
  if (g->precision != 0 && g->precision != 3 && g->precision != 6) { set_error("gemm_tc: precision must be 6 (default, bf16x6) or 3 (bf16x3)"); return MSACL_ERR_BAD_ARG; }
  // Column tile.  Large problems (>= one CTA per SM from the row tiles alone): 256, the A tile is converted once per 256 output
  // columns.  Small problems are bound by the latency of ONE CTA (its K stages run back to back), so the tile that gives the
  // fewest waves over the 148 SMs wins, and among those the narrowest (most CTAs in flight).
  const int64_t mt = (g->m + GM - 1) / GM;
  int bn = 256;
  if (!g->row_sumsq && mt * g->split_k < kNumSMs) {
    int64_t best_waves = -1;
    for (int cand : {64, 128, 256}) {
      if (cand > 64 && g->n <= cand / 2) continue;
      const int64_t ctas = mt * ((g->n + cand - 1) / cand) * g->split_k;
      const int64_t waves = (ctas + kNumSMs - 1) / kNumSMs;
      if (best_waves < 0 || waves < best_waves) { best_waves = waves; bn = cand; }
    }
  }
  // a pre-packed weight operand is a 256-wide column tile: take the streamed-weights instantiation also for few row tiles
  // (measured at 40 row tiles: the learner's model_update at replay batch 256 drops from 1.14 to 1.00 ms -- bulk-copied
  // weights and the pipelined A loader beat the converting loaders' one memory round trip per K stage, even with 40 CTAs)
  if (g->b_packed) bn = 256;
  const int64_t tiles = mt * ((g->n + bn - 1) / bn) * g->split_k;
  const dim3 grid((unsigned)(tiles < kNumSMs ? tiles : kNumSMs));          // persistent: one CTA per SM
  static bool attr_set = false;
  auto set_attr = [&](auto kern, size_t bytes) {
    return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) == cudaSuccess;
  };
#define MSACL_GEMM_VARIANTS(X) X(2, 256, 4, false) X(3, 256, 3, false) X(2, 256, 4, true) X(3, 256, 3, true) X(2, 128, 4, false) X(3, 128, 4, false) \
  X(2, 64, 4, false) X(3, 64, 4, false)
  if (!attr_set) {
    bool ok = true;
#define X(NI, BN_, ST, SM_) ok = ok && set_attr(gemm_tc_kernel<NI, BN_, ST, SM_>, sizeof(GemmSmem<NI, BN_, ST, SM_>) + 128);
    MSACL_GEMM_VARIANTS(X)
#undef X
    if (!ok) { set_error("gemm_tc: cudaFuncSetAttribute(MaxDynamicSharedMemorySize) failed"); return MSACL_ERR_CUDA; }
    attr_set = true;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int nimg = g->precision == 3 ? 2 : 3;
  // streamed mode: pre-packed weights (BN = 256) behind a k-contiguous, 16-byte aligned A operand
  const bool streamed = bn == 256 && g->b_packed && g->a_k_stride == 1 && (g->a_row_stride & 7) == 0 && (reinterpret_cast<uintptr_t>(g->a) & 31) == 0;
#define X(NI, BN_, ST, SM_) \
  if (nimg == NI && bn == BN_ && streamed == SM_) gemm_tc_kernel<NI, BN_, ST, SM_><<<grid, G_THREADS, sizeof(GemmSmem<NI, BN_, ST, SM_>) + 128, st>>>(*g);
  MSACL_GEMM_VARIANTS(X)
#undef X
#undef MSACL_GEMM_VARIANTS
  return check_launch("gemm_tc");
}
