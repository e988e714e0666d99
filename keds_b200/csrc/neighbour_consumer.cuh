// Forward pass of the consumer of the retrieved neighbours (SURVEY.md §8 f2): the IM2TEXT MLP
// applied to the query and to every neighbour, then two 3-layer single-query cross-attention
// stacks (image neighbours / text neighbours) -- src/model/model.py:37-123, called at
// src/trainer.py:59-69 and src/eval_utils.py:378-383,515-519,661-668,806-810,943-947.
//
// Two kernels:
//   k_linear_tf32   C = act(A W^T + bias), nn.Linear layout (W: [out][in]), fp32 in / fp32 out,
//                   tcgen05.mma kind::tf32 with TMA-staged operands (the TMA unit rounds fp32 to
//                   tf32 on the way in: to nearest, ties to even, subnormals kept -- measured by
//                   tests/test_gpu_consumer_kernels.py), accumulators in TMEM, bias (+ReLU) fused
//                   in the epilogue.
//                   blockIdx.z selects one of two independent problems of the same shape (the two
//                   attention stacks), so both run in one launch.
//   k_cross_attend  softmax(q K^T / sqrt(dh)) V for ONE query token per batch row over its k
//                   neighbours, one warp per head (src/model/model.py:69-73 with n_q = 1).
#pragma once
#include "ptx.cuh"

namespace keds {

constexpr int LIN_M = 128;       // rows of A per tile (TMEM lanes)
constexpr int LIN_K = 32;        // fp32 words per k-block = one 128-byte swizzle row
constexpr int LIN_UK = 8;        // K per tcgen05.mma kind::tf32
constexpr int LIN_THREADS = 320;    // k_linear_tf32: TMA warp, MMA warp, 8 epilogue warps (2 per TMEM lane quadrant)
constexpr int SK_THREADS = 192;     // k_linear_tf32_splitk: TMA warp, MMA warp, 4 epilogue warps
constexpr uint32_t LIN_A_BYTES = LIN_M * LIN_K * 4;
constexpr int LIN_WBOX = 128;    // rows of W per TMA box (the descriptor's box height)

// BN = output features per tile (TMEM columns): 128 for the small products (more CTAs), 256 where
// there are enough tiles anyway (half the A re-reads per flop).
template <int BN>
struct LinCfg {
  static constexpr int kStages = BN == 128 ? 6 : 4;
  static constexpr uint32_t kBBytes = BN * LIN_K * 4;
  static constexpr uint32_t kStageBytes = LIN_A_BYTES + kBBytes;
  static constexpr uint32_t kOffBars = kStages * kStageBytes;
  static constexpr uint32_t kSmemBytes = kOffBars + 128 + BN * 4 + 1024;  // barriers, bias, alignment slack
};

struct LinearParams {
  int M, N, K;            // C[M][N] = act(A[M][K] W[N][K]^T + bias[N])
  int relu;
  const float* bias[2];   // per problem (blockIdx.z); nullable
  float* C[2];
  long long ldc;          // floats between rows of C
  uint32_t* err;          // device error word (0 = ok)
  unsigned long long* tdump;  // diagnostics: per CTA {start, prologue done, dependency met, accumulator ready, end} ns
  int nz;                 // problems (k_linear_tf32_persistent walks a flat tile list)
};

template <int BN>
__global__ void __launch_bounds__(LIN_THREADS, 1)
k_linear_tf32(const __grid_constant__ CUtensorMap tm_a0, const __grid_constant__ CUtensorMap tm_a1,
              const __grid_constant__ CUtensorMap tm_w0, const __grid_constant__ CUtensorMap tm_w1,
              const LinearParams p) {
  using Cfg = LinCfg<BN>;
  constexpr int LIN_STAGES = Cfg::kStages;
  constexpr uint32_t LIN_STAGE_BYTES = Cfg::kStageBytes;
  constexpr int LIN_N = BN;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gbase = smem_raw + (sbase - smem_u32(smem_raw));
  const uint32_t bars = sbase + Cfg::kOffBars;
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (LIN_STAGES + s); };
  const uint32_t tfull_bar = bars + 8u * (2 * LIN_STAGES);
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(gbase + Cfg::kOffBars + 112);
  volatile uint32_t* dead = reinterpret_cast<volatile uint32_t*>(gbase + Cfg::kOffBars + 116);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int z = blockIdx.z;
  const int n0 = blockIdx.x * LIN_N;
  const int m0 = blockIdx.y * LIN_M;
  const CUtensorMap* tm_a = z == 0 ? &tm_a0 : &tm_a1;
  const CUtensorMap* tm_w = z == 0 ? &tm_w0 : &tm_w1;
  const int kblocks = (p.K + LIN_K - 1) / LIN_K;  // a ragged tail reads zeros from both operands
  unsigned long long* td = p.tdump ? p.tdump + 5ull * (blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z)) : nullptr;
  if (td && threadIdx.x == 0) td[0] = global_timer_ns();

  if (threadIdx.x == 0) {
    prefetch_tensormap(tm_a);
    prefetch_tensormap(tm_w);
    for (int s = 0; s < LIN_STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(tfull_bar, 1);
    *dead = 0;
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_slot)), LIN_N);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (td && threadIdx.x == 0) td[1] = global_timer_ns();

  griddep_wait();  // A is the previous kernel's output
  if (td && threadIdx.x == 0) td[2] = global_timer_ns();

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int kb = 0; kb < kblocks; ++kb) {
        mbar_wait(empty_bar(stage), phase ^ 1u, dead, p.err, 0x700u + stage);
        const uint32_t sa = sbase + stage * LIN_STAGE_BYTES;
        mbar_arrive_expect_tx(full_bar(stage), LIN_STAGE_BYTES);
        tma_load_2d(sa, tm_a, full_bar(stage), kb * LIN_K, m0, kEvictNormal);
#pragma unroll
        for (int wb = 0; wb < BN / LIN_WBOX; ++wb)
          tma_load_2d(sa + LIN_A_BYTES + wb * (LIN_WBOX * LIN_K * 4), tm_w, full_bar(stage), kb * LIN_K,
                      n0 + wb * LIN_WBOX, kEvictLast);
        if (++stage == LIN_STAGES) {
          stage = 0;
          phase ^= 1u;
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = idesc_tf32_f32(LIN_M, LIN_N);
      int stage = 0;
      uint32_t phase = 0;
      for (int kb = 0; kb < kblocks; ++kb) {
        mbar_wait(full_bar(stage), phase, dead, p.err, 0x710u + stage);
        tc_fence_after();
        const uint32_t sa = sbase + stage * LIN_STAGE_BYTES;
        const uint64_t adesc = smem_desc_sw128(sa);
        const uint64_t bdesc = smem_desc_sw128(sa + LIN_A_BYTES);
#pragma unroll
        for (int k = 0; k < LIN_K / LIN_UK; ++k)  // +32 bytes per K = 8 step: +2 in 16-byte units
          umma_tf32(tmem_base, adesc + 2u * k, bdesc + 2u * k, idesc, (kb | k) != 0 ? 1u : 0u);
        umma_commit(empty_bar(stage));
        if (++stage == LIN_STAGES) {
          stage = 0;
          phase ^= 1u;
        }
      }
      umma_commit(tfull_bar);
    }
  } else {
    // epilogue: TMEM lane == row of C. A thread holds 32 consecutive columns of ONE row; written
    // as such, a warp's store touches 32 rows (one 16-byte piece of 32 different lines). So each
    // warp turns its 32 x 32 block through shared memory (the pipeline stages are idle by now) and
    // writes whole 128-byte row segments.
    const int quad = warp & 3;
    const int row0 = m0 + quad * 32;
    const float* bias = p.bias[z];
    float* cbase = p.C[z] + n0;
    const int half = (warp - 2) >> 2;  // the two warps of a quadrant take alternate 32-column chunks
    float* tr = reinterpret_cast<float*>(gbase) + (warp - 2) * (32 * 33);  // [32 rows][33] per warp
    // this tile's bias -> shared memory while the main loop runs (weights: no dependency on the
    // previous kernel); the column loop below then never waits on global memory
    float* sbias = reinterpret_cast<float*>(gbase + Cfg::kOffBars + 128);
    for (int j = threadIdx.x - 64; j < LIN_N; j += 256)
      sbias[j] = (bias != nullptr && n0 + j < p.N) ? __ldg(bias + n0 + j) : 0.f;
    asm volatile("bar.sync 1, 256;" ::: "memory");
    mbar_wait(tfull_bar, 0u, dead, p.err, 0x720u);
    tc_fence_after();
    if (td && threadIdx.x == 64) td[3] = global_timer_ns();
    const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    const bool vec_ok = (p.ldc & 3) == 0 && (p.N & 3) == 0 && (reinterpret_cast<uintptr_t>(p.C[z]) & 15) == 0;
#pragma unroll 1
    for (int ch = half; ch < LIN_N / 32; ch += 2) {
      uint32_t v[32];
      tmem_ld32(taddr + ch * 32, v);
      tmem_ld_wait(v);
      const int c0 = n0 + ch * 32;
      if (c0 >= p.N) break;
      // bias first, into registers: interleaved with the stores below the compiler must assume
      // the two shared-memory arrays alias and serialises 32 load -> store round trips
      float4 bv[8];
#pragma unroll
      for (int j4 = 0; j4 < 8; ++j4) bv[j4] = reinterpret_cast<const float4*>(sbias + ch * 32)[j4];
#pragma unroll
      for (int j4 = 0; j4 < 8; ++j4) {
        const float x0 = __uint_as_float(v[4 * j4 + 0]) + bv[j4].x, x1 = __uint_as_float(v[4 * j4 + 1]) + bv[j4].y;
        const float x2 = __uint_as_float(v[4 * j4 + 2]) + bv[j4].z, x3 = __uint_as_float(v[4 * j4 + 3]) + bv[j4].w;
        tr[lane * 33 + 4 * j4 + 0] = p.relu ? fmaxf(x0, 0.f) : x0;
        tr[lane * 33 + 4 * j4 + 1] = p.relu ? fmaxf(x1, 0.f) : x1;
        tr[lane * 33 + 4 * j4 + 2] = p.relu ? fmaxf(x2, 0.f) : x2;
        tr[lane * 33 + 4 * j4 + 3] = p.relu ? fmaxf(x3, 0.f) : x3;
      }
      __syncwarp();
      if (vec_ok) {
        // 8 lanes cover one row's 32 columns (128 bytes), 4 rows per store instruction
        const int cc = (lane & 7) * 4;
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          const int rr = it * 4 + (lane >> 3);
          const float* s = tr + rr * 33 + cc;
          if (row0 + rr < p.M && c0 + cc < p.N)
            *reinterpret_cast<float4*>(cbase + static_cast<long long>(row0 + rr) * p.ldc + ch * 32 + cc) =
                make_float4(s[0], s[1], s[2], s[3]);
        }
      } else {
        for (int rr = 0; rr < 32; ++rr)
          if (row0 + rr < p.M && c0 + lane < p.N)
            cbase[static_cast<long long>(row0 + rr) * p.ldc + ch * 32 + lane] = tr[rr * 33 + lane];
      }
      __syncwarp();
    }
  }

  tc_fence_before();
  __syncthreads();
  if (td && lane == 0) atomicMax(&td[4], global_timer_ns());  // every warp: see ktimer_end
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, LIN_N);
  }
}

// The same product for MANY tiles (more than two waves of CTAs: the key/value projection of the
// neighbour consumer). One CTA per SM walks a flat list of 128 x 256 tiles; two 256-column TMEM
// accumulators let the epilogue of tile t run under the main loop of tile t + 1, and CTA launch /
// retire costs are paid once. Tile order: the N index runs fastest, so concurrently running CTAs
// share their A rows in L2.
constexpr int PL_BN = 256;
constexpr int PL_STAGES = 4;
constexpr int PL_THREADS = 192;  // TMA warp, MMA warp, 4 epilogue warps (hidden under the next main loop)
constexpr uint32_t PL_STAGE_BYTES = LIN_A_BYTES + PL_BN * LIN_K * 4;   // 48 KB
constexpr uint32_t PL_OFF_TR = PL_STAGES * PL_STAGE_BYTES;             // 4 warps x [32][33] fp32
constexpr uint32_t PL_OFF_BIAS = PL_OFF_TR + 4 * 32 * 33 * 4;
constexpr uint32_t PL_OFF_BARS = PL_OFF_BIAS + 2 * PL_BN * 4;
constexpr uint32_t PL_SMEM_BYTES = PL_OFF_BARS + 256 + 1024;

__global__ void __launch_bounds__(PL_THREADS, 1)
k_linear_tf32_persistent(const __grid_constant__ CUtensorMap tm_a0, const __grid_constant__ CUtensorMap tm_a1,
                         const __grid_constant__ CUtensorMap tm_w0, const __grid_constant__ CUtensorMap tm_w1,
                         const LinearParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gbase = smem_raw + (sbase - smem_u32(smem_raw));
  const uint32_t bars = sbase + PL_OFF_BARS;
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (PL_STAGES + s); };
  auto tfull_bar = [&](int a) { return bars + 8u * (2 * PL_STAGES + a); };
  auto tempty_bar = [&](int a) { return bars + 8u * (2 * PL_STAGES + 2 + a); };
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(gbase + PL_OFF_BARS + 200);
  volatile uint32_t* dead = reinterpret_cast<volatile uint32_t*>(gbase + PL_OFF_BARS + 204);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int nt = (p.N + PL_BN - 1) / PL_BN;
  const int mt = (p.M + LIN_M - 1) / LIN_M;
  const int tiles = nt * mt * p.nz;
  const int kblocks = (p.K + LIN_K - 1) / LIN_K;

  if (threadIdx.x == 0) {
    prefetch_tensormap(&tm_a0);
    prefetch_tensormap(&tm_w0);
    if (p.nz > 1) {
      prefetch_tensormap(&tm_a1);
      prefetch_tensormap(&tm_w1);
    }
    for (int s = 0; s < PL_STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), 4);
    }
    *dead = 0;
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_slot)), 2 * PL_BN);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  griddep_wait();  // A is the previous kernel's output

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = blockIdx.x; t < tiles; t += gridDim.x) {
        const int n0 = (t % nt) * PL_BN, m0 = ((t / nt) % mt) * LIN_M, z = t / (nt * mt);
        const CUtensorMap* tm_a = z == 0 ? &tm_a0 : &tm_a1;
        const CUtensorMap* tm_w = z == 0 ? &tm_w0 : &tm_w1;
        for (int kb = 0; kb < kblocks; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u, dead, p.err, 0x900u + stage);
          const uint32_t sa = sbase + stage * PL_STAGE_BYTES;
          mbar_arrive_expect_tx(full_bar(stage), PL_STAGE_BYTES);
          tma_load_2d(sa, tm_a, full_bar(stage), kb * LIN_K, m0, kEvictNormal);
#pragma unroll
          for (int wb = 0; wb < PL_BN / LIN_WBOX; ++wb)
            tma_load_2d(sa + LIN_A_BYTES + wb * (LIN_WBOX * LIN_K * 4), tm_w, full_bar(stage), kb * LIN_K,
                        n0 + wb * LIN_WBOX, kEvictLast);
          if (++stage == PL_STAGES) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = idesc_tf32_f32(LIN_M, PL_BN);
      int stage = 0, acc = 0;
      uint32_t phase = 0, acc_phase = 0;
      for (int t = blockIdx.x; t < tiles; t += gridDim.x) {
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u, dead, p.err, 0x910u + acc);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * PL_BN);
        for (int kb = 0; kb < kblocks; ++kb) {
          mbar_wait(full_bar(stage), phase, dead, p.err, 0x920u + stage);
          tc_fence_after();
          const uint32_t sa = sbase + stage * PL_STAGE_BYTES;
          const uint64_t adesc = smem_desc_sw128(sa);
          const uint64_t bdesc = smem_desc_sw128(sa + LIN_A_BYTES);
#pragma unroll
          for (int k = 0; k < LIN_K / LIN_UK; ++k)
            umma_tf32(d_tmem, adesc + 2u * k, bdesc + 2u * k, idesc, (kb | k) != 0 ? 1u : 0u);
          umma_commit(empty_bar(stage));
          if (++stage == PL_STAGES) {
            stage = 0;
            phase ^= 1u;
          }
        }
        umma_commit(tfull_bar(acc));
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1u;
      }
    }
  } else {
    const int quad = warp & 3;
    float* tr = reinterpret_cast<float*>(gbase + PL_OFF_TR) + (warp - 2) * (32 * 33);
    float* sbias_all = reinterpret_cast<float*>(gbase + PL_OFF_BIAS);
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int t = blockIdx.x; t < tiles; t += gridDim.x) {
      const int n0 = (t % nt) * PL_BN, m0 = ((t / nt) % mt) * LIN_M, z = t / (nt * mt);
      const int row0 = m0 + quad * 32;
      const float* bias = p.bias[z];
      float* cbase = p.C[z] + n0;
      float* sbias = sbias_all + acc * PL_BN;
      for (int j = threadIdx.x - 64; j < PL_BN; j += 128)
        sbias[j] = (bias != nullptr && n0 + j < p.N) ? __ldg(bias + n0 + j) : 0.f;
      asm volatile("bar.sync 1, 128;" ::: "memory");
      mbar_wait(tfull_bar(acc), acc_phase, dead, p.err, 0x930u + acc);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + static_cast<uint32_t>(acc * PL_BN);
      const bool vec_ok = (p.ldc & 3) == 0 && (p.N & 3) == 0 && (reinterpret_cast<uintptr_t>(p.C[z]) & 15) == 0;
#pragma unroll 1
      for (int ch = 0; ch < PL_BN / 32; ++ch) {
        uint32_t v[32];
        tmem_ld32(taddr + ch * 32, v);
        tmem_ld_wait(v);
        const int c0 = n0 + ch * 32;
        if (c0 >= p.N) break;
        float4 bv[8];
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) bv[j4] = reinterpret_cast<const float4*>(sbias + ch * 32)[j4];
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
          const float x0 = __uint_as_float(v[4 * j4 + 0]) + bv[j4].x, x1 = __uint_as_float(v[4 * j4 + 1]) + bv[j4].y;
          const float x2 = __uint_as_float(v[4 * j4 + 2]) + bv[j4].z, x3 = __uint_as_float(v[4 * j4 + 3]) + bv[j4].w;
          tr[lane * 33 + 4 * j4 + 0] = p.relu ? fmaxf(x0, 0.f) : x0;
          tr[lane * 33 + 4 * j4 + 1] = p.relu ? fmaxf(x1, 0.f) : x1;
          tr[lane * 33 + 4 * j4 + 2] = p.relu ? fmaxf(x2, 0.f) : x2;
          tr[lane * 33 + 4 * j4 + 3] = p.relu ? fmaxf(x3, 0.f) : x3;
        }
        __syncwarp();
        if (vec_ok) {
          const int cc = (lane & 7) * 4;
#pragma unroll
          for (int it = 0; it < 8; ++it) {
            const int rr = it * 4 + (lane >> 3);
            const float* s = tr + rr * 33 + cc;
            if (row0 + rr < p.M && c0 + cc < p.N)
              *reinterpret_cast<float4*>(cbase + static_cast<long long>(row0 + rr) * p.ldc + ch * 32 + cc) =
                  make_float4(s[0], s[1], s[2], s[3]);
          }
        } else {
          for (int rr = 0; rr < 32; ++rr)
            if (row0 + rr < p.M && c0 + lane < p.N)
              cbase[static_cast<long long>(row0 + rr) * p.ldc + ch * 32 + lane] = tr[rr * 33 + lane];
        }
        __syncwarp();
      }
      // accumulator drained: the MMA warp may reuse it two tiles from now
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1u;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 2 * PL_BN);
  }
}

// The same product for SMALL problems (the single-query-token chain: M = batch rows, a handful of
// 128 x 128 tiles). One tile per CTA leaves most SMs idle and each busy SM limited by its 64 B/clk
// ingress port, so here the work is cut finer in both directions: 32-column tiles, and the K range
// of a tile split over a CLUSTER of SK_SPLIT CTAs. Each CTA accumulates its K slice in TMEM, parks
// the 128 x 32 partial in its shared memory, and after a cluster barrier CTA r sums columns
// [8r, 8r + 8) of all partials through distributed shared memory (fixed order: deterministic),
// adds the bias and stores. grid = (SK_SPLIT * n_tiles, m_tiles, problems), cluster (SK_SPLIT,1,1).
constexpr int SK_BN = 32;
constexpr int SK_MAX_SPLIT = 4;      // cluster size: 2 or 4 (template parameter)
constexpr int SK_STAGES = 6;
constexpr uint32_t SK_B_BYTES = SK_BN * LIN_K * 4;                 // 4 KB
constexpr uint32_t SK_STAGE_BYTES = LIN_A_BYTES + SK_B_BYTES;      // 20 KB
constexpr uint32_t SK_OFF_PART = SK_STAGES * SK_STAGE_BYTES;       // [32 columns][128 rows] fp32
constexpr uint32_t SK_OFF_BARS = SK_OFF_PART + SK_BN * LIN_M * 4;
constexpr uint32_t SK_SMEM_BYTES = SK_OFF_BARS + 128 + 1024;

template <int SK_SPLIT>
__global__ void __launch_bounds__(SK_THREADS, 1)
k_linear_tf32_splitk(const __grid_constant__ CUtensorMap tm_a0, const __grid_constant__ CUtensorMap tm_a1,
                     const __grid_constant__ CUtensorMap tm_w0, const __grid_constant__ CUtensorMap tm_w1,
                     const LinearParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gbase = smem_raw + (sbase - smem_u32(smem_raw));
  const uint32_t bars = sbase + SK_OFF_BARS;
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (SK_STAGES + s); };
  const uint32_t tfull_bar = bars + 8u * (2 * SK_STAGES);
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(gbase + SK_OFF_BARS + 112);
  volatile uint32_t* dead = reinterpret_cast<volatile uint32_t*>(gbase + SK_OFF_BARS + 116);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int z = blockIdx.z;
  const int split = static_cast<int>(cluster_ctarank());   // == blockIdx.x % SK_SPLIT
  const int n0 = (blockIdx.x / SK_SPLIT) * SK_BN;
  const int m0 = blockIdx.y * LIN_M;
  const CUtensorMap* tm_a = z == 0 ? &tm_a0 : &tm_a1;
  const CUtensorMap* tm_w = z == 0 ? &tm_w0 : &tm_w1;
  const int kblocks = (p.K + LIN_K - 1) / LIN_K;
  const int kb0 = kblocks * split / SK_SPLIT, kb1 = kblocks * (split + 1) / SK_SPLIT;
  unsigned long long* td = p.tdump ? p.tdump + 5ull * (blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z)) : nullptr;
  if (td && threadIdx.x == 0) td[0] = global_timer_ns();

  if (threadIdx.x == 0) {
    prefetch_tensormap(tm_a);
    prefetch_tensormap(tm_w);
    for (int s = 0; s < SK_STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(tfull_bar, 1);
    *dead = 0;
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_slot)), SK_BN);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (td && threadIdx.x == 0) td[1] = global_timer_ns();

  griddep_wait();
  if (td && threadIdx.x == 0) td[2] = global_timer_ns();

  float* part = reinterpret_cast<float*>(gbase + SK_OFF_PART);
  float bv[SK_BN / SK_SPLIT];  // bias of the columns this CTA reduces (epilogue warps)
  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(empty_bar(stage), phase ^ 1u, dead, p.err, 0x800u + stage);
        const uint32_t sa = sbase + stage * SK_STAGE_BYTES;
        mbar_arrive_expect_tx(full_bar(stage), SK_STAGE_BYTES);
        tma_load_2d(sa, tm_a, full_bar(stage), kb * LIN_K, m0, kEvictNormal);
        tma_load_2d(sa + LIN_A_BYTES, tm_w, full_bar(stage), kb * LIN_K, n0, kEvictLast);
        if (++stage == SK_STAGES) {
          stage = 0;
          phase ^= 1u;
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = idesc_tf32_f32(LIN_M, SK_BN);
      int stage = 0;
      uint32_t phase = 0;
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(full_bar(stage), phase, dead, p.err, 0x810u + stage);
        tc_fence_after();
        const uint32_t sa = sbase + stage * SK_STAGE_BYTES;
        const uint64_t adesc = smem_desc_sw128(sa);
        const uint64_t bdesc = smem_desc_sw128(sa + LIN_A_BYTES);
#pragma unroll
        for (int k = 0; k < LIN_K / LIN_UK; ++k)
          umma_tf32(tmem_base, adesc + 2u * k, bdesc + 2u * k, idesc, ((kb - kb0) | k) != 0 ? 1u : 0u);
        umma_commit(empty_bar(stage));
        if (++stage == SK_STAGES) {
          stage = 0;
          phase ^= 1u;
        }
      }
      umma_commit(tfull_bar);
    }
  } else {
    // this CTA's partial tile -> shared memory, column-major (thread == row: conflict-free)
    const int quad = warp & 3;
    const int r = quad * 32 + lane;
#pragma unroll
    for (int c = 0; c < SK_BN / SK_SPLIT; ++c) {
      const int col = n0 + split * (SK_BN / SK_SPLIT) + c;
      bv[c] = (p.bias[z] != nullptr && col < p.N) ? __ldg(p.bias[z] + col) : 0.f;
    }
    uint32_t v[32];
    if (kb1 > kb0) {
      mbar_wait(tfull_bar, 0u, dead, p.err, 0x820u);
      tc_fence_after();
      tmem_ld32(tmem_base + (static_cast<uint32_t>(quad * 32) << 16), v);
      tmem_ld_wait(v);
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = 0u;  // more splits than k-blocks: this slice is empty
    }
#pragma unroll
    for (int j = 0; j < 32; ++j) part[j * LIN_M + r] = __uint_as_float(v[j]);
  }
  if (td && threadIdx.x == 64) td[3] = global_timer_ns();

  tc_fence_before();
  __syncwarp();
  cluster_sync_all();  // every CTA's partial is parked

  if (warp >= 2) {
    // CTA `split` owns columns [8 split, 8 split + 8) of the tile: sum the SK_SPLIT partials in rank
    // order through distributed shared memory, add the bias, store 32 bytes per row
    const int r = (warp & 3) * 32 + lane;
    const int row = m0 + r;
    const int c0 = split * (SK_BN / SK_SPLIT);
    float acc[SK_BN / SK_SPLIT];
#pragma unroll
    for (int c = 0; c < SK_BN / SK_SPLIT; ++c) acc[c] = 0.f;
    const uint32_t pbase = sbase + SK_OFF_PART;
#pragma unroll
    for (int s = 0; s < SK_SPLIT; ++s) {
#pragma unroll
      for (int c = 0; c < SK_BN / SK_SPLIT; ++c)
        acc[c] += ld_dsmem_f32(pbase + static_cast<uint32_t>(((c0 + c) * LIN_M + r) * 4), static_cast<uint32_t>(s));
    }
#pragma unroll
    for (int c = 0; c < SK_BN / SK_SPLIT; ++c) {
      const float x = acc[c] + bv[c];
      acc[c] = p.relu ? fmaxf(x, 0.f) : x;
    }
    if (row < p.M) {
      float* crow = p.C[z] + static_cast<long long>(row) * p.ldc + n0 + c0;
      const bool vec_ok = (p.ldc & 3) == 0 && (p.N & 3) == 0 && (reinterpret_cast<uintptr_t>(p.C[z]) & 15) == 0;
      if (vec_ok) {
#pragma unroll
        for (int c = 0; c < SK_BN / SK_SPLIT; c += 4)
          if (n0 + c0 + c < p.N)
            *reinterpret_cast<float4*>(crow + c) = make_float4(acc[c], acc[c + 1], acc[c + 2], acc[c + 3]);
      } else {
#pragma unroll
        for (int c = 0; c < SK_BN / SK_SPLIT; ++c)
          if (n0 + c0 + c < p.N) crow[c] = acc[c];
      }
    }
  }

  __syncwarp();
  cluster_sync_all();  // nobody leaves while a peer may still read its partial
  if (td && lane == 0) atomicMax(&td[4], global_timer_ns());
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, SK_BN);
  }
}

struct AttendParams {
  int B, k, heads, dim_head;
  const float* Q[2];    // [B][heads * dim_head]
  const float* KV[2];   // [B * k][ld_kv]; keys at column k_off + h * dim_head, values at v_off + ...
  float* O[2];          // [B][heads * dim_head]
  long long ld_kv;
  int k_off, v_off;
  float scale;          // dim_head ** -0.5
};

// grid (B, problems), block = 32 * heads threads (one warp per head), dynamic smem =
// heads * (dim_head + k) floats. Scores: one LANE per neighbour (its key row is read with
// independent 16-byte loads against the query staged in shared memory); the weighted sum of the
// value rows: one lane per output column, coalesced over the row.
// DH = 64 (the reference's dim_head): every global load of a phase is issued before its first
// use (explicit register arrays -- left to itself the compiler keeps two loads in flight and the
// kernel is a chain of ~24 memory round trips). DH = 0: any dim_head, plain loops.
template <int DH>
__global__ void k_cross_attend(const AttendParams p) {
  extern __shared__ float att_sm[];
  griddep_wait();
  const int b = blockIdx.x;
  const int z = blockIdx.y;
  const int h = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int dh = DH > 0 ? DH : p.dim_head;
  const int inner = p.heads * dh;
  const float* q = p.Q[z] + static_cast<long long>(b) * inner + h * dh;
  const float* kv = p.KV[z] + static_cast<long long>(b) * p.k * p.ld_kv + h * dh;
  float* qs = att_sm + h * dh;
  float* w = att_sm + p.heads * dh + h * p.k;
  for (int d = lane; d < dh; d += 32) qs[d] = q[d];
  __syncwarp();
  float mx = -INFINITY;
  for (int j = lane; j < p.k; j += 32) {
    const float* kr = kv + j * p.ld_kv + p.k_off;
    float s;
    if constexpr (DH > 0) {
      float4 a[DH / 4];
#pragma unroll
      for (int d = 0; d < DH / 4; ++d) a[d] = __ldg(reinterpret_cast<const float4*>(kr) + d);
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
      for (int d = 0; d < DH / 4; ++d) {
        const float4 c = reinterpret_cast<const float4*>(qs)[d];
        s0 = fmaf(a[d].x, c.x, s0);
        s1 = fmaf(a[d].y, c.y, s1);
        s2 = fmaf(a[d].z, c.z, s2);
        s3 = fmaf(a[d].w, c.w, s3);
      }
      s = (s0 + s1) + (s2 + s3);
    } else {
      s = 0.f;
      for (int d = 0; d < dh; ++d) s = fmaf(kr[d], qs[d], s);
    }
    s *= p.scale;
    w[j] = s;
    mx = fmaxf(mx, s);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float den = 0.f;
  for (int j = lane; j < p.k; j += 32) {
    const float e = expf(w[j] - mx);
    w[j] = e;
    den += e;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) den += __shfl_xor_sync(0xffffffffu, den, o);
  __syncwarp();
  const float inv = 1.f / den;
  float* o = p.O[z] + static_cast<long long>(b) * inner + h * dh;
  if constexpr (DH > 0) {
    // lane owns columns lane and lane + 32; 16 value rows (2 x 16 loads) in flight per step
    float acc0 = 0.f, acc1 = 0.f;
    for (int j0 = 0; j0 < p.k; j0 += 16) {
      float t0[16], t1[16];
#pragma unroll
      for (int jj = 0; jj < 16; ++jj) {
        const bool live = j0 + jj < p.k;
        const float* vr = kv + (j0 + jj) * p.ld_kv + p.v_off;
        t0[jj] = live ? __ldg(vr + lane) : 0.f;
        t1[jj] = (live && DH > 32) ? __ldg(vr + 32 + lane) : 0.f;
      }
#pragma unroll
      for (int jj = 0; jj < 16; ++jj) {
        const float wj = j0 + jj < p.k ? w[j0 + jj] : 0.f;
        acc0 = fmaf(wj, t0[jj], acc0);
        acc1 = fmaf(wj, t1[jj], acc1);
      }
    }
    o[lane] = acc0 * inv;
    if (DH > 32) o[32 + lane] = acc1 * inv;
  } else {
    for (int d = lane; d < dh; d += 32) {
      const float* vr = kv + p.v_off + d;
      float acc = 0.f;
      for (int j = 0; j < p.k; ++j) acc = fmaf(w[j], __ldg(vr + j * p.ld_kv), acc);
      o[d] = acc * inv;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Training: the backward pass of the same modules (src/trainer.py:59-69 with the modules being
// optimised, backward at :462-474). The products are the same tf32 tcgen05 GEMMs with the operand
// roles turned (dX = dY W, dW = dY^T X); these kernels are what lies between them.

// Linear -> Dropout -> ReLU of IM2TEXT (src/model/model.py:110-116) behind the GEMM, in place:
// h = max(z * mask, 0), mask = 0 or 1 / (1 - p) per element (drawn by the caller).
__global__ void k_mask_relu(float* __restrict__ z, const float* __restrict__ mask, long long n) {
  griddep_wait();
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) z[i] = fmaxf(z[i] * mask[i], 0.f);
}

// dz = dh * [h > 0] * mask   (mask nullable: no dropout)
__global__ void k_relu_bwd(const float* dh, const float* __restrict__ h, const float* __restrict__ mask, float* dz,
                           long long n) {  // dz may alias dh
  griddep_wait();
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) dz[i] = h[i] > 0.f ? dh[i] * (mask != nullptr ? mask[i] : 1.f) : 0.f;
}

// Bias gradient: out[c] = sum_r in[r][c]. One block per 32 columns (32 x 8 threads), rows summed in
// a fixed order: deterministic.
__global__ void __launch_bounds__(256)
k_colsum(const float* __restrict__ in, long long ld, long long rows, int cols, float* __restrict__ out) {
  griddep_wait();
  __shared__ float part[8][33];
  const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cx;
  float acc = 0.f;
  if (c < cols)
    for (long long r = ry; r < rows; r += 8) acc += in[r * ld + c];
  part[ry][cx] = acc;
  __syncthreads();
  if (ry == 0 && c < cols) {
    float t = part[0][cx];
#pragma unroll
    for (int i = 1; i < 8; ++i) t += part[i][cx];
    out[c] = t;
  }
}

// out[r][:] = a[r][:] + b[r][:] + c[r][:] over `cols` columns (row strides lda / ldb / ldc / ldo)
__global__ void k_add3_rows(const float* __restrict__ a, long long lda, const float* __restrict__ b, long long ldb,
                            const float* __restrict__ c, long long ldc, float* __restrict__ out, long long ldo,
                            long long rows, int cols) {
  griddep_wait();
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= rows * cols) return;
  const long long r = i / cols;
  const int x = static_cast<int>(i % cols);
  out[r * ldo + x] = a[r * lda + x] + b[r * ldb + x] + c[r * ldc + x];
}

// Backward of k_cross_attend for one query token: with s_j = scale q.k_j, p = softmax(s),
// o = sum_j p_j v_j and the incoming dO:
//   dv_j = p_j dO,  dp_j = dO.v_j,  ds_j = p_j (dp_j - sum_i p_i dp_i),
//   dq = scale sum_j ds_j k_j,  dk_j = scale ds_j q.
// The probabilities are recomputed from Q and K (nothing is kept from the forward but Q).
// grid (B, problems), one warp per head, dynamic smem = heads * (2 dim_head + 2 k) floats.
struct AttendBwdParams {
  int B, k, heads, dim_head;
  const float* Q[2];     // [B][inner]
  const float* KV[2];    // [B * k][ld_kv]
  const float* dO[2];    // [B][inner]
  float* dQ[2];          // [B][inner]
  float* dKV[2];         // [B * k][ld_kv]: dK at k_off, dV at v_off of this layer
  long long ld_kv;
  int k_off, v_off;
  float scale;
};

__global__ void k_cross_attend_bwd(const AttendBwdParams p) {
  extern __shared__ float atb_sm[];
  griddep_wait();
  const int b = blockIdx.x, z = blockIdx.y;
  const int h = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int dh = p.dim_head, inner = p.heads * dh;
  float* qs = atb_sm + h * (2 * dh + 2 * p.k);
  float* gs = qs + dh;          // dO of this head
  float* pr = gs + dh;          // scores -> probabilities
  float* ds = pr + p.k;         // dp -> ds
  const float* q = p.Q[z] + static_cast<long long>(b) * inner + h * dh;
  const float* go = p.dO[z] + static_cast<long long>(b) * inner + h * dh;
  const long long row0 = static_cast<long long>(b) * p.k;
  const float* kv = p.KV[z] + row0 * p.ld_kv + h * dh;
  float* dkv = p.dKV[z] + row0 * p.ld_kv + h * dh;
  for (int d = lane; d < dh; d += 32) {
    qs[d] = q[d];
    gs[d] = go[d];
  }
  __syncwarp();
  float mx = -INFINITY;
  for (int j = lane; j < p.k; j += 32) {
    const float* kr = kv + j * p.ld_kv + p.k_off;
    const float* vr = kv + j * p.ld_kv + p.v_off;
    float s = 0.f, dp = 0.f;
    for (int d = 0; d < dh; ++d) {
      s = fmaf(__ldg(kr + d), qs[d], s);
      dp = fmaf(__ldg(vr + d), gs[d], dp);
    }
    s *= p.scale;
    pr[j] = s;
    ds[j] = dp;
    mx = fmaxf(mx, s);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float den = 0.f;
  for (int j = lane; j < p.k; j += 32) {
    const float e = expf(pr[j] - mx);
    pr[j] = e;
    den += e;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) den += __shfl_xor_sync(0xffffffffu, den, o);
  const float inv = 1.f / den;
  float dot = 0.f;
  for (int j = lane; j < p.k; j += 32) {
    const float pj = pr[j] * inv;
    pr[j] = pj;
    dot = fmaf(pj, ds[j], dot);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
  for (int j = lane; j < p.k; j += 32) ds[j] = pr[j] * (ds[j] - dot);
  __syncwarp();
  // one lane per column: coalesced over the key / value rows
  float* dq = p.dQ[z] + static_cast<long long>(b) * inner + h * dh;
  for (int d = lane; d < dh; d += 32) {
    float acc = 0.f;
    const float qd = qs[d], gd = gs[d];
    for (int j = 0; j < p.k; ++j) {
      const float dsj = ds[j];
      acc = fmaf(dsj, __ldg(kv + j * p.ld_kv + p.k_off + d), acc);
      dkv[j * p.ld_kv + p.k_off + d] = p.scale * dsj * qd;
      dkv[j * p.ld_kv + p.v_off + d] = pr[j] * gd;
    }
    dq[d] = p.scale * acc;
  }
}

}  // namespace keds
