// Fused 16-bit (fp16 or bf16 operands, fp32 accumulate) scoring GEMM + per-query candidate
// selection for sm_100a.
//
// Replaces the "SGEMM tile -> HBM -> k-select" pair inside the Faiss GPU flat index that KEDs
// calls at src/trainer.py:213,221,271 and src/eval_utils.py:169,177. The [queries x rows] score
// matrix lives only in TMEM; what reaches HBM is, per (row slice, query), one 128-byte line of
// candidate (approx score, row id) pairs plus the slice's drop threshold.
//
//   warp 0        TMA producer: per k-block one {64 x 128} query box + one row box
//   warp 1        tcgen05.mma issuer (one lane), owns the TMEM allocation
//   warps 2..5    epilogue: TMEM lane == query, so one thread owns one query's scores
//   warps 6..9    (CTA-pair variant) a second set of epilogue warps: the same 128 queries, the
//                 other 128 columns of the tile, their own candidate lists ("sub-slices")
//
// Tile: M = 128 queries (TMEM lanes) x N = 256 DB rows (TMEM columns), K streamed in 64-wide
// k-blocks (one 128-byte swizzle row). Two 256-column accumulators double-buffer MMA vs epilogue.
//
// Two variants of one kernel:
//   kPair = false  one CTA per tile (cta_group::1). Used for batches of <= 128 queries, where the
//                  kernel is HBM-bound and every SM streams its own row slice.
//   kPair = true   a cluster of two CTAs shares every 256-row tile (cta_group::2, M = 256): each
//                  CTA holds its own 128 queries and loads HALF of the row tile, the leader CTA
//                  issues one MMA for both. Per CTA and k-block 32 KB cross L2->SM instead of 48 KB,
//                  which is what bounds the single-CTA variant once the batch is compute-bound.
//                  Here the selection epilogue is the co-bottleneck (ncu, round 2: tensor pipe
//                  76 % busy at 4096 x 0.5M, 53 % at 4096 x 50k -- a tile's 48 MMAs take ~6,100
//                  cycles, one epilogue warp per sub-partition needed about as long and stalled
//                  the issuer at every compaction), so each sub-partition gets TWO epilogue warps
//                  that split the tile's columns; all latencies (tcgen05.ld, the select chain,
//                  votes) of one hide under the other.
#pragma once
#include "ptx.cuh"

namespace keds {

constexpr int BM = 128;
constexpr int BN = 256;
constexpr int BK = 64;
constexpr int UK = 16;
constexpr int LKEEP = 16;   // a compaction keeps scores above the LKEEP-th best seen
constexpr int CHUNK = 32;   // TMEM columns per tcgen05.ld
constexpr int SCORE_THREADS = 192;       // single-CTA variant: producer, issuer, 4 epilogue warps
constexpr int SCORE_PAIR_THREADS = 320;  // CTA-pair variant: 8 epilogue warps
constexpr uint32_t Q_STAGE_BYTES = BM * BK * 2;
constexpr uint32_t TMEM_COLS = 512;
// Search with exclusion: at most EXCLUDE_MAX rows left out per query. k_prep_rows stages them as
// local row ids per database, EX_NONE where a slot excludes nothing (unused, out of range, repeat).
constexpr int EXCLUDE_MAX = 8;
constexpr int EX_NONE = -1;

template <bool kPair>
struct ScoreCfg {
  // Single CTA (HBM-bound, one query tile): the kernel lives on bytes in flight, so the candidate
  // slots are cut to 32 per query (32 KB) to make room for a fourth 48-KB stage; the slot count
  // is then checked every 8 scores. CTA pair (compute-bound): 64 slots, checked every 32 scores --
  // compactions are what its epilogue can least afford.
  // CTA pair (compute-bound): 8 epilogue warps of 32 slots each (the same 64 KB as 4 x 64 before).
  // Four 32-KB stages: 195 KB, which leaves an SM room for re-rank blocks of another sub-pass next
  // to a scoring CTA (api.cu: pipelined sub-passes); a fifth stage measured no faster.
  static constexpr int kStages = 4;
  static constexpr int kEpiWarps = kPair ? 8 : 4;
  static constexpr int kSub = kEpiWarps / 4;                        // candidate lists ("sub-slices") per (slice, query)
  static constexpr int kThreads = 64 + 32 * kEpiWarps;
  static constexpr int kCap = 32;
  static constexpr int kAppend = 8;
  static constexpr uint32_t kCandWarpBytes = kCap * 32 * 8;
  static constexpr int kRowsPerCta = kPair ? BN / 2 : BN;           // row-tile rows this CTA loads
  static constexpr uint32_t kXBytes = kRowsPerCta * BK * 2;
  static constexpr uint32_t kStageBytes = Q_STAGE_BYTES + kXBytes;  // 48 KB / 32 KB
  // dynamic shared memory map (offsets from a 1024-aligned base)
  static constexpr uint32_t kOffCand = kStages * kStageBytes;
  static constexpr uint32_t kOffBias = kOffCand + kEpiWarps * kCandWarpBytes;
  static constexpr uint32_t kOffBars = kOffBias + 2 * BN * 4;
  static constexpr uint32_t kSmemBytes = kOffBars + 256 + 768;      // barriers + alignment slack (227 KB exactly for the single-CTA variant)
};
constexpr uint32_t SCORE_SMEM_BYTES = ScoreCfg<false>::kSmemBytes;
constexpr uint32_t SCORE_PAIR_SMEM_BYTES = ScoreCfg<true>::kSmemBytes;

struct ScoreParams {
  int n_db;          // 1 or 2 databases scored against the same queries
  int n_qt;          // query tiles of BM
  int n_qg;          // query groups per (db, slice): n_qt (single CTA) or ceil(n_qt / 2) (pair)
  int S;             // row slices per (db, query tile); the pair variant writes 2 candidate lines per slice
  int n_items;       // n_db * S * n_qg ; item = ((db * S) + s) * n_qg + qg
  int kblocks;       // d_pad / BK
  uint32_t fmt_bits; // operand format bits of the instruction descriptor (kIdescBf16Bits, or 0 = fp16)
  int nq;            // live queries
  int n_rows[2];     // rows per database
  int n_tiles[2];    // ceil(n_rows / BN)
  const float* bias[2];  // nullable; additive per-row bias padded with -inf to n_tiles * BN
  uint2* cand;       // [n_db * S * kSub * n_qt][BM][LKEEP] {approx score bits, row id}, padded {-inf, ~0}
  int* cand_cnt;     // [..][BM]
  float* cand_theta; // [..][BM]  everything the slice dropped scored <= theta
  float* theta0;     // [n_db][theta_ld] running per-query drop threshold shared by all lists of a query (see epilogue)
  int theta_ld;
  uint32_t* err;     // device error word (0 = ok)
  float* dump;       // debug: full approx scores [n_db][nq][ld_dump], or nullptr
  long long ld_dump;
  unsigned long long* timing;  // nullable: {min start ns, max end ns} of this launch (%globaltimer)
  // kRank only (gallery ranking by counting, database 0 = the gallery, inner product): per query
  // the error band [lo, hi] around its target's exact score and the two rows left out of the count
  const float* rk_lo;
  const float* rk_hi;
  const int* rk_target;
  const int* rk_exclude;     // -1: none
  // top-k search with exclusion (kRank = false): per database [nq][n_ex] local row ids that must
  // never enter a candidate list (EX_NONE: unused slot); nullptr / n_ex = 0: nothing excluded
  const int* ex_rows;
  int n_ex;
  long long ex_ld;           // ints per database
  // kRange only (range search, database 0): per query the band threshold in approximate-score
  // space (range_search.cuh: k_range_band); every row scoring at or above it is appended as
  // {query, row} to rg_out. rg_count counts every such row, also past rg_cap (overflow: the host
  // grows the buffer and reruns the pass).
  const float* rg_thr;
  uint2* rg_out;
  unsigned long long* rg_count;
  unsigned long long rg_cap;
};

struct ItemCoord {
  int db, s, qg, t0, t1;
};

__device__ __forceinline__ ItemCoord decode_item(const ScoreParams& p, int item) {
  ItemCoord c;
  c.qg = item % p.n_qg;
  const int t = item / p.n_qg;
  c.s = t % p.S;
  c.db = t / p.S;
  const long long T = p.n_tiles[c.db];
  c.t0 = static_cast<int>((T * c.s) / p.S);
  c.t1 = static_cast<int>((T * (c.s + 1)) / p.S);
  return c;
}

__device__ __forceinline__ void sts64(uint32_t addr, uint32_t a, uint32_t b) {
  asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(a), "r"(b) : "memory");
}
__device__ __forceinline__ uint2 lds64(uint32_t addr) {
  uint2 r;
  asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(r.x), "=r"(r.y) : "r"(addr) : "memory");
  return r;
}
__device__ __forceinline__ float lds32f(uint32_t addr) {
  float r;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(r) : "r"(addr) : "memory");
  return r;
}

struct CandState {
  int cnt;
  float theta;
};

// Per-thread compaction of one query's candidate slots (all 32 lanes of a warp run it in lock
// step on their own columns of the warp's interleaved buffer): find the LKEEP-th best score with
// a register sorting network, raise theta to it, keep only strictly better entries.
template <int CAP>
__device__ __noinline__ CandState compact_candidates(uint32_t slot0, int cnt, float theta) {
  float s[CAP];
#pragma unroll
  for (int e = 0; e < CAP; ++e) s[e] = (e < cnt) ? lds32f(slot0 + e * 256) : -INFINITY;
#pragma unroll
  for (int k = 2; k <= CAP; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
#pragma unroll
      for (int i = 0; i < CAP; ++i) {
        const int l = i ^ j;
        if (l > i) {
          const float a = s[i], b = s[l];
          const float mx = fmaxf(a, b), mn = fminf(a, b);
          const bool desc = (i & k) == 0;  // descending overall
          s[i] = desc ? mx : mn;
          s[l] = desc ? mn : mx;
        }
      }
    }
  }
  theta = fmaxf(theta, s[LKEEP - 1]);
  // keep the entries above theta, in place and in order: every entry is in registers before the
  // first store; positions come from the keep mask (see the append loop for why)
  int w = 0;
#pragma unroll
  for (int e0 = 0; e0 < CAP; e0 += 16) {
    uint2 en[16];
    uint32_t m = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      en[i] = lds64(slot0 + (e0 + i) * 256);
      m |= (e0 + i < cnt && __uint_as_float(en[i].x) > theta) ? (1u << i) : 0u;
    }
#pragma unroll
    for (int i = 0; i < 16; ++i)
      if (m & (1u << i)) sts64(slot0 + (w + __popc(m & ((1u << i) - 1u))) * 256, en[i].x, en[i].y);
    w += __popc(m);
  }
  CandState r;
  r.cnt = w;
  r.theta = theta;
  return r;
}

// kRank = false: candidate selection for the top-k search (everything above).
// kRank = true:  gallery ranking by counting. Per (candidate list, query) the epilogue counts the
//                rows whose approximate score is above hi = s_target + eps (they beat the target for
//                certain) and lists the rows inside [lo, hi] (at most LKEEP per list; more sets the
//                overflow mark and the query is recounted exactly). The target and the excluded row
//                are skipped by id. Output: the same 128-byte lines (band rows), cand_cnt = band
//                rows or -1 (overflow), cand_theta = the certain count (as int bits).
// kExclude = true (top-k search only): rows listed per query in p.ex_rows never enter a list. A
//                separate instantiation, so that the plain search keeps its code and registers.
// kRange = true: range search (kernel k_score_range). No candidate lists: every (query, row) whose
//                approximate score (L2 bias included) is not below the query's band threshold
//                p.rg_thr[q] is appended to p.rg_out, one atomic per warp and 32-column chunk that
//                has any.
// The kernels below are thin entry points around this body: the tensor maps are their
// __grid_constant__ parameters, p their parameter block.
template <bool kPair, bool kRank, bool kExclude, bool kRange>
__device__ __forceinline__ void score_topk_body(const CUtensorMap& tm_q, const CUtensorMap& tm_x0,
                                                const CUtensorMap& tm_x1, const ScoreParams& p) {
  static_assert(!(kRank && kExclude), "exclusion is a top-k search option");
  static_assert(!(kRange && (kRank || kExclude)), "range search is a mode of its own");
  using Cfg = ScoreCfg<kPair>;
  constexpr int NSTAGE = Cfg::kStages;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gbase = smem_raw + (sbase - smem_u32(smem_raw));

  {
    // the layout fills the 227 KB exactly up to the alignment slack: refuse to run rather than
    // overrun if the dynamic window starts less aligned than assumed
    uint32_t dyn;
    asm volatile("mov.u32 %0, %%dynamic_smem_size;" : "=r"(dyn));
    if (sbase - smem_u32(smem_raw) + (Cfg::kSmemBytes - 768u) > dyn) {
      if (threadIdx.x == 0) atomicCAS(p.err, 0u, 0x900u);
      return;
    }
  }
  const uint32_t bars = sbase + Cfg::kOffBars;
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (NSTAGE + s); };
  auto tfull_bar = [&](int a) { return bars + 8u * (2 * NSTAGE + a); };
  auto tempty_bar = [&](int a) { return bars + 8u * (2 * NSTAGE + 2 + a); };
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(gbase + Cfg::kOffBars + 200);
  volatile uint32_t* dead = reinterpret_cast<volatile uint32_t*>(gbase + Cfg::kOffBars + 204);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t crank = kPair ? cluster_ctarank() : 0u;   // 0 = leader of the pair
  const int unit = kPair ? static_cast<int>(blockIdx.x >> 1) : static_cast<int>(blockIdx.x);
  const int n_units = kPair ? static_cast<int>(gridDim.x >> 1) : static_cast<int>(gridDim.x);

  if (threadIdx.x == 0) {
    prefetch_tensormap(&tm_q);
    prefetch_tensormap(&tm_x0);
    if (p.n_db > 1) prefetch_tensormap(&tm_x1);
    for (int s = 0; s < NSTAGE; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), kPair ? 2 * Cfg::kEpiWarps : Cfg::kEpiWarps);  // pair: the leader collects both CTAs' epilogue warps
    }
    *dead = 0;
    fence_mbar_init();
  }
  if (warp == 1) {
    if constexpr (kPair) {
      tmem_alloc_2sm(smem_u32(const_cast<uint32_t*>(tmem_slot)), TMEM_COLS);
      tmem_relinquish_2sm();
    } else {
      tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_slot)), TMEM_COLS);
      tmem_relinquish();
    }
  }
  tc_fence_before();
  if constexpr (kPair) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // The database rows do not depend on the previous kernel (they only change in add(), which
  // synchronises the device): the producer sends the row half of its first stages now, under
  // k_prep_rows, and the query half once the wait below has passed.
  int pre_rows = 0;
  if constexpr (!kPair) {
    if (warp == 0 && lane == 0 && unit < p.n_items) {
      const ItemCoord c = decode_item(p, unit);
      if (c.t0 < c.t1) {
        const CUtensorMap* tmx = c.db == 0 ? &tm_x0 : &tm_x1;
        pre_rows = min(NSTAGE, p.kblocks);
        for (int kb = 0; kb < pre_rows; ++kb) {
          mbar_arrive_expect_tx(full_bar(kb), Cfg::kStageBytes);
          tma_load_2d(sbase + kb * Cfg::kStageBytes + Q_STAGE_BYTES, tmx, full_bar(kb), kb * BK, c.t0 * BN,
                      p.n_qt > 1 ? kEvictNormal : kEvictFirst);
        }
      }
    }
  }

  // Programmatic dependent launch: everything above overlapped the tail of the previous kernel
  // (k_prep_rows); from here on its outputs (bf16 queries) are needed. Let the next kernel
  // (k_select_rerank) be scheduled as soon as SMs free up.
  griddep_wait();
  griddep_launch_dependents();
  const unsigned long long t_start = ktimer_begin(p.timing);

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int item = unit; item < p.n_items; item += n_units) {
        const ItemCoord c = decode_item(p, item);
        const CUtensorMap* tmx = c.db == 0 ? &tm_x0 : &tm_x1;
        const int qt = kPair ? c.qg * 2 + static_cast<int>(crank) : c.qg;
        for (int tile = c.t0; tile < c.t1; ++tile) {
          for (int kb = 0; kb < p.kblocks; ++kb) {
            mbar_wait(empty_bar(stage), phase ^ 1u, dead, p.err, 0x100u + stage);
            const uint32_t sq = sbase + stage * Cfg::kStageBytes;
            const uint32_t sx = sq + Q_STAGE_BYTES;
            if constexpr (kPair) {
              // the leader's barrier counts the bytes of both CTAs; only the leader arms it
              if (crank == 0) mbar_arrive_expect_tx(full_bar(stage), 2 * Cfg::kStageBytes);
              tma_load_2d_2sm(sq, &tm_q, full_bar(stage), kb * BK, qt * BM, kEvictLast);
              tma_load_2d_2sm(sx, tmx, full_bar(stage), kb * BK,
                              tile * BN + static_cast<int>(crank) * Cfg::kRowsPerCta, kEvictNormal);
            } else if (pre_rows > 0) {
              // first stages of the first tile: armed, and their rows requested, before the wait
              --pre_rows;
              tma_load_2d(sq, &tm_q, full_bar(stage), kb * BK, qt * BM, kEvictLast);
            } else {
              mbar_arrive_expect_tx(full_bar(stage), Cfg::kStageBytes);
              tma_load_2d(sq, &tm_q, full_bar(stage), kb * BK, qt * BM, kEvictLast);
              tma_load_2d(sx, tmx, full_bar(stage), kb * BK, tile * BN,
                          p.n_qt > 1 ? kEvictNormal : kEvictFirst);
            }
            if (++stage == NSTAGE) {
              stage = 0;
              phase ^= 1u;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer (pair: leader only)
    if (lane == 0 && crank == 0) {
      const uint32_t idesc = idesc_f16_base(kPair ? 2 * BM : BM, BN) | p.fmt_bits;
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int item = unit; item < p.n_items; item += n_units) {
        const ItemCoord c = decode_item(p, item);
        for (int tile = c.t0; tile < c.t1; ++tile) {
          mbar_wait(tempty_bar(acc), acc_phase ^ 1u, dead, p.err, 0x200u + acc);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * BN);
          for (int kb = 0; kb < p.kblocks; ++kb) {
            mbar_wait(full_bar(stage), phase, dead, p.err, 0x300u + stage);
            tc_fence_after();
            const uint32_t sq = sbase + stage * Cfg::kStageBytes;
            const uint64_t adesc = smem_desc_sw128(sq);
            const uint64_t bdesc = smem_desc_sw128(sq + Q_STAGE_BYTES);
#pragma unroll
            for (int k = 0; k < BK / UK; ++k) {
              // +32 bytes per K=16 step inside the 128-byte swizzle row: +2 in 16-byte units
              if constexpr (kPair)
                umma_bf16_2sm(d_tmem, adesc + 2u * k, bdesc + 2u * k, idesc, (kb | k) != 0 ? 1u : 0u);
              else
                umma_bf16(d_tmem, adesc + 2u * k, bdesc + 2u * k, idesc, (kb | k) != 0 ? 1u : 0u);
            }
            if constexpr (kPair) umma_commit_2sm(empty_bar(stage), 0x3); else umma_commit(empty_bar(stage));
            if (++stage == NSTAGE) {
              stage = 0;
              phase ^= 1u;
            }
          }
          if constexpr (kPair) umma_commit_2sm(tfull_bar(acc), 0x3); else umma_commit(tfull_bar(acc));
          acc ^= 1;
          if (acc == 0) acc_phase ^= 1u;
        }
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue (lane == query)
    const int quad = warp & 3;                // TMEM lane quadrant this warp may read
    const int q_local = quad * 32 + lane;
    constexpr int CAP = Cfg::kCap;
    constexpr int APPEND = Cfg::kAppend;
    constexpr int SUB = Cfg::kSub;
    constexpr int CH_PER = (BN / CHUNK) / SUB;  // column chunks of a tile this warp scans
    const int half = (warp - 2) >> 2;           // which columns: 0 (the only set in the single-CTA variant) or 1
    const uint32_t wbuf = sbase + Cfg::kOffCand + static_cast<uint32_t>(warp - 2) * Cfg::kCandWarpBytes;
    const uint32_t slot0 = wbuf + lane * 8;   // entry e of this lane lives at slot0 + e * 256
    float* sbias = reinterpret_cast<float*>(gbase + Cfg::kOffBias);
    const int et = threadIdx.x - 64;          // 0 .. 32 * kEpiWarps - 1 among epilogue threads
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int item = unit; item < p.n_items; item += n_units) {
      const ItemCoord c = decode_item(p, item);
      const int qt = kPair ? c.qg * 2 + static_cast<int>(crank) : c.qg;
      const int q_glob = qt * BM + q_local;
      const bool active = q_glob < p.nq;
      float theta = active ? -INFINITY : INFINITY;
      int cnt = 0;
      // Warm start: a list may begin at the final threshold of ANY list of the same query that has
      // already finished. That threshold is the 16th best score of its list, and the certificate
      // needs every list's threshold below tau anyway, so rows at or below it can be dropped here
      // as well (the list's reported threshold only rises from there). Without it every work item
      // starts cold -- every score of its first columns is appended and the list compacted every
      // eight appends -- which is what made short slices (k = 200 galleries: two tiles per item)
      // spend more time warming lists than scoring. Any stale value is still a valid start.
      float* th0 = nullptr;
      if constexpr (!kRank && !kRange) {
        if (active && p.theta0 != nullptr) {
          th0 = p.theta0 + static_cast<long long>(c.db) * p.theta_ld + q_glob;
          theta = __ldcg(th0);
        }
      }
      // rank mode: theta plays "hi", rk_lo_q the lower band edge
      [[maybe_unused]] float rk_lo_q = INFINITY;
      [[maybe_unused]] int rk_t = -1, rk_e = -1, beats = 0;
      [[maybe_unused]] bool overflow = false;
      if constexpr (kRank) {
        if (active) {
          rk_lo_q = p.rk_lo[q_glob];
          theta = p.rk_hi[q_glob];
          rk_t = p.rk_target[q_glob];
          rk_e = p.rk_exclude != nullptr ? p.rk_exclude[q_glob] : -1;
        }
      }
      [[maybe_unused]] float rg_thr = 0.f;
      if constexpr (kRange) {
        if (active) rg_thr = p.rg_thr[q_glob];
      }
      // Exclusion: this query's excluded rows of this database, in registers (statically indexed:
      // every loop over them is unrolled). An excluded row is not a row of this query's problem --
      // it never enters a list, so no list's theta depends on it (DESIGN.md section 3).
      [[maybe_unused]] int ex[EXCLUDE_MAX];
      [[maybe_unused]] bool has_ex = false;
      if constexpr (kExclude) {
#pragma unroll
        for (int e = 0; e < EXCLUDE_MAX; ++e) ex[e] = EX_NONE;
        if (active && p.ex_rows != nullptr) {
          const int* xr = p.ex_rows + c.db * p.ex_ld + static_cast<long long>(q_glob) * p.n_ex;
#pragma unroll
          for (int e = 0; e < EXCLUDE_MAX; ++e) {
            if (e < p.n_ex) ex[e] = __ldg(xr + e);
            has_ex = has_ex || ex[e] != EX_NONE;
          }
        }
      }
      const float* bias = p.bias[c.db];
      const int n_rows = p.n_rows[c.db];
      for (int tile = c.t0; tile < c.t1; ++tile) {
        // one test per tile and query; the per-column path below runs only for a tile that holds
        // an excluded row
        [[maybe_unused]] bool tile_ex = false;
        if constexpr (kExclude) {
          if (has_ex) {
#pragma unroll
            for (int e = 0; e < EXCLUDE_MAX; ++e)
              tile_ex = tile_ex || static_cast<unsigned>(ex[e] - tile * BN) < static_cast<unsigned>(BN);
          }
        }
        if (bias != nullptr) {
          if constexpr (SUB == 2) {
            sbias[acc * BN + et] = bias[static_cast<long long>(tile) * BN + et];
            asm volatile("bar.sync 1, 256;" ::: "memory");
          } else {
            sbias[acc * BN + et] = bias[static_cast<long long>(tile) * BN + et];
            sbias[acc * BN + 128 + et] = bias[static_cast<long long>(tile) * BN + 128 + et];
            asm volatile("bar.sync 1, 128;" ::: "memory");
          }
        }
        mbar_wait(tfull_bar(acc), acc_phase, dead, p.err, 0x400u + acc);
        tc_fence_after();
        const uint32_t taddr =
            tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + static_cast<uint32_t>(acc * BN);
        const int nvalid = n_rows - tile * BN;  // >= BN for full tiles
#pragma unroll 1
        for (int ch = half * CH_PER; ch < (half + 1) * CH_PER; ++ch) {
          uint32_t v[CHUNK];
          tmem_ld32(taddr + ch * CHUNK, v);
          tmem_ld_wait(v);
          if (bias != nullptr) {
            const float4* b4 = reinterpret_cast<const float4*>(sbias + acc * BN + ch * CHUNK);
#pragma unroll
            for (int j4 = 0; j4 < CHUNK / 4; ++j4) {
              const float4 b = b4[j4];
              v[4 * j4 + 0] = __float_as_uint(__uint_as_float(v[4 * j4 + 0]) + b.x);
              v[4 * j4 + 1] = __float_as_uint(__uint_as_float(v[4 * j4 + 1]) + b.y);
              v[4 * j4 + 2] = __float_as_uint(__uint_as_float(v[4 * j4 + 2]) + b.z);
              v[4 * j4 + 3] = __float_as_uint(__uint_as_float(v[4 * j4 + 3]) + b.w);
            }
          } else if (nvalid < BN) {
            // zero-filled out-of-range rows score 0 under IP: take them out of the race
#pragma unroll
            for (int j = 0; j < CHUNK; ++j)
              if (ch * CHUNK + j >= nvalid) v[j] = 0xff800000u;  // -inf
          }
          const uint32_t idx0 = static_cast<uint32_t>(tile * BN + ch * CHUNK);
          if (p.dump != nullptr && active) {
            float* drow = p.dump + (static_cast<long long>(c.db) * p.nq + q_glob) * p.ld_dump;
#pragma unroll
            for (int j = 0; j < CHUNK; ++j)
              if (static_cast<int>(idx0) + j < n_rows) drow[idx0 + j] = __uint_as_float(v[j]);
          }
          if constexpr (kExclude) {
            if (tile_ex) {
              // rare: the chunk's excluded columns as a bit mask, then -inf there (never > theta)
              uint32_t xm = 0;
#pragma unroll
              for (int e = 0; e < EXCLUDE_MAX; ++e) {
                const unsigned o = static_cast<unsigned>(ex[e] - static_cast<int>(idx0));
                xm |= o < static_cast<unsigned>(CHUNK) ? (1u << o) : 0u;
              }
#pragma unroll
              for (int j = 0; j < CHUNK; ++j)
                if ((xm >> j) & 1u) v[j] = 0xff800000u;
            }
          }
          if constexpr (kRange) {
            // "not below" rather than ">=": a threshold of -inf (a query with an unbounded error)
            // takes every row, -inf and NaN scores included; rows past n_rows are padding
            uint32_t m = 0;
#pragma unroll
            for (int j = 0; j < CHUNK; ++j)
              m |= (active && !(__uint_as_float(v[j]) < rg_thr) && static_cast<int>(idx0) + j < n_rows) ? (1u << j) : 0u;
            if (__any_sync(0xffffffffu, m != 0u)) {
              // warp-wide exclusive prefix of the hit counts, one atomic for the warp's whole chunk
              const int nh = __popc(m);
              int incl = nh;
#pragma unroll
              for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
              }
              unsigned long long base = 0;
              if (lane == 31) base = atomicAdd(p.rg_count, static_cast<unsigned long long>(incl));
              base = __shfl_sync(0xffffffffu, base, 31);
              unsigned long long pos = base + static_cast<unsigned long long>(incl - nh);
              while (m != 0u) {
                const int j = __ffs(m) - 1;
                m &= m - 1u;
                if (pos < p.rg_cap) p.rg_out[pos] = make_uint2(static_cast<uint32_t>(q_glob), idx0 + j);
                ++pos;
              }
            }
            continue;
          }
          if constexpr (kRank) {
            // count the certain winners; rows inside the band are rare and take a plain branch
#pragma unroll
            for (int j = 0; j < CHUNK; ++j) {
              const float sc = __uint_as_float(v[j]);
              const int id = static_cast<int>(idx0) + j;
              const bool special = id == rk_t || id == rk_e;
              beats += (sc > theta && !special) ? 1 : 0;
              if (sc >= rk_lo_q && !(sc > theta) && !special) {
                if (cnt < LKEEP) {
                  sts64(slot0 + static_cast<uint32_t>(cnt) * 256u, v[j], static_cast<uint32_t>(id));
                  ++cnt;
                } else {
                  overflow = true;
                }
              }
            }
            continue;
          }
          // APPEND scores at a time, then make sure the next APPEND still fit. (The slot buffers
          // are small on purpose: 32 KB instead of 64 KB buys a fourth TMA stage, and the kernel
          // lives on bytes in flight.)
#pragma unroll
          for (int g = 0; g < CHUNK; g += APPEND) {
            // Eight slot addresses first (a chain of selects in eight DIFFERENT registers), then the
            // eight predicated stores. Written the obvious way -- store, bump one pointer, store --
            // every bump waits ~20 cycles for the store in front of it to have read that register
            // (a write-after-read hazard on a memory instruction), 25 cycles per score in all.
            uint32_t wptr = slot0 + static_cast<uint32_t>(cnt) * 256u;
#pragma unroll
            for (int j0 = g; j0 < g + APPEND; j0 += 8) {
              uint32_t a[9];
              a[0] = wptr;
#pragma unroll
              for (int i = 0; i < 8; ++i) a[i + 1] = a[i] + (__uint_as_float(v[j0 + i]) > theta ? 256u : 0u);
#pragma unroll
              for (int i = 0; i < 8; ++i)
                if (__uint_as_float(v[j0 + i]) > theta) sts64(a[i], v[j0 + i], idx0 + j0 + i);
              wptr = a[8];
            }
            cnt = static_cast<int>((wptr - slot0) >> 8);
            if (__any_sync(0xffffffffu, cnt > CAP - APPEND)) {
              const CandState st = compact_candidates<CAP>(slot0, cnt, theta);
              cnt = st.cnt;
              theta = st.theta;
            }
          }
        }
        // accumulator drained: hand the TMEM buffer back to the MMA warp (pair: of the leader CTA)
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if constexpr (kPair) mbar_arrive_cluster(tempty_bar(acc), 0); else mbar_arrive(tempty_bar(acc));
        }
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1u;
      }
      // Final compaction: at most LKEEP - 1 entries survive (those strictly above the slice's
      // LKEEP-th best, which becomes theta). They leave as one 128-byte line per (slice, query):
      // [(db, s, qt)][query][LKEEP] {score bits, row id}, padded with {-inf, ~0}; the re-rank
      // kernel reads a slice with a single coalesced half-warp load.
      if constexpr (kRange) continue;  // the candidates are out already
      if constexpr (!kRank) {
        if (__any_sync(0xffffffffu, cnt >= LKEEP)) {
          const CandState st = compact_candidates<CAP>(slot0, cnt, theta);
          cnt = st.cnt;
          theta = st.theta;
        }
      }
      if (!kPair || qt < p.n_qt) {
        // one candidate line per (slice, column half, query): the re-rank kernel sees S * SUB slices
        const long long oitem =
            (static_cast<long long>(c.db) * (p.S * SUB) + (c.s * SUB + half)) * p.n_qt + qt;
        uint2* cbase = p.cand + (oitem * BM + q_local) * LKEEP;
#pragma unroll
        for (int e = 0; e < LKEEP; e += 2) {
          uint2 a = make_uint2(0xff800000u, 0xffffffffu), b = a;
          if (e < cnt) a = lds64(slot0 + e * 256);
          if (e + 1 < cnt) b = lds64(slot0 + (e + 1) * 256);
          *reinterpret_cast<uint4*>(cbase + e) = make_uint4(a.x, a.y, b.x, b.y);
        }
        if constexpr (kRank) {
          p.cand_cnt[oitem * BM + q_local] = overflow ? -1 : cnt;
          p.cand_theta[oitem * BM + q_local] = __int_as_float(beats);
        } else {
          p.cand_cnt[oitem * BM + q_local] = cnt;
          p.cand_theta[oitem * BM + q_local] = theta;
          // publish for the lists that start later (float max through the sign-split integer trick)
          if (th0 != nullptr && theta > -INFINITY) {
            if (theta >= 0.f) atomicMax(reinterpret_cast<int*>(th0), __float_as_int(theta));
            else atomicMin(reinterpret_cast<unsigned int*>(th0), __float_as_uint(theta));
          }
        }
      }
      __syncwarp();
    }
  }

  tc_fence_before();
  if constexpr (kPair) cluster_sync_all(); else __syncthreads();
  ktimer_end(p.timing, t_start);  // kernel duration without stream events
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    if constexpr (kPair) tmem_dealloc_2sm(tmem_base, TMEM_COLS); else tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

template <bool kPair, bool kRank = false, bool kExclude = false>
__global__ void __launch_bounds__(ScoreCfg<kPair>::kThreads, 1)
k_score_topk(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_x0,
             const __grid_constant__ CUtensorMap tm_x1, const ScoreParams p) {
  score_topk_body<kPair, kRank, kExclude, false>(tm_q, tm_x0, tm_x1, p);
}

// Range search: the same mainloop with the range epilogue (database 0 only).
template <bool kPair>
__global__ void __launch_bounds__(ScoreCfg<kPair>::kThreads, 1)
k_score_range(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_x0,
              const __grid_constant__ CUtensorMap tm_x1, const ScoreParams p) {
  score_topk_body<kPair, false, false, true>(tm_q, tm_x0, tm_x1, p);
}

}  // namespace keds
