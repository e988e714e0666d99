// Exact fp32 fallback for the queries whose certificate failed (and the whole batch in exact-only
// mode): ONE kernel per pass, k_exact_fallback, which returns at once when nothing is flagged, so it
// can sit in every search's launch chain (programmatic dependent launch hides its launch latency)
// without a host round trip. Two phases; work units are claimed through counters and the second
// phase starts once every unit of the first is finished (no dependence on how many blocks are
// resident); every block skips both alike when nothing is flagged:
//
//   exact_scores   rank scores (IP, or -squared-L2) of up to f_cap flagged queries per database
//                  against every row -> scratch[db][f][row]
//   exact_select   one block per (flagged query, database): radix-select the k-th best, take ties
//                  in id order, order by (score desc, id asc), write D/I, then run the neighbour
//                  consumer for that query (the re-rank kernel skipped it)
//
// Pass p handles flagged[p * f_cap ... (p+1) * f_cap); the host launches ceil(nq / f_cap) passes.
// Included by aux_kernels.cuh (uses warp_exact_score, block_find_bin, consume_query).
#pragma once

namespace keds {

struct ExactDb {
  const float* x_f32;
  long long n_rows;
  const int* flagged;
  const int* n_flagged;
  float* scratch;  // [f_cap][n_rows]
  float* cmax;     // [f_cap][chunks] best rank score of each row chunk (phase 1 -> phase 2 pre-filter)
  long long cg;    // 32-row groups per chunk
  int chunks;      // row chunks = phase-1 work units per query group
  float* D;
  long long* I;
  long long id_offset;
};

struct ExactParams {
  ConsumeParams cons;
  ExactDb db[2];
  int n_db, d, metric, k, f_cap, pass;
  const float* q_f32;
  unsigned int* work;          // [0] phase-1 units handed out, [1] phase-2 items handed out (zero at launch)
  unsigned int* done;          // phase-1 units finished (zero at launch)
  int ck_cap;                  // chunk maxima that fit the shared-memory key array of phase 2
  unsigned int* err;           // status word: EXACT_ERR_BARRIER if the barrier watchdog fired
  const unsigned int* band_dev;  // status word written by the re-rank kernel: largest |C| of this search
  unsigned int* band_host;     // nullable: mapped host word that receives it (planner feedback, no copy node)
  PeerOut peer;                // row-sharded exchange; n == 0: off
  unsigned long long* timing;  // nullable in-kernel launch timer
  // search with exclusion: staged local row ids (ScoreParams::ex_rows); nullptr: nothing excluded
  const int* ex_rows;
  int n_ex;
  long long ex_ld;
};

constexpr unsigned int EXACT_ERR_BARRIER = 0xEB000000u;
// Score an excluded row gets in the scratch: the NaN whose order key is 0, below every real score,
// so the selection never takes it while keff (k capped at the rows left) rows remain; fmaxf drops
// it from the chunk maxima.
constexpr unsigned int EXACT_EXCLUDED_BITS = 0xFFFFFFFFu;

__device__ __forceinline__ bool row_in(const int* ex, int n_ex, long long row) {
  bool hit = false;
#pragma unroll
  for (int e = 0; e < EXCLUDE_MAX; ++e) hit = hit || (e < n_ex && ex[e] == row);
  return hit;
}
constexpr int EXACT_LIST_CAP = 2048;  // rows at or above the pre-filter threshold held in shared memory

// Work is handed out through counters, never by block index: the blocks that are resident drain
// all of it, so the wait between the phases cannot depend on a block that has not started yet
// (two handles searching at once may share the SMs between their grids).
__device__ __forceinline__ unsigned int exact_claim(unsigned int* counter, unsigned int* slot) {
  __syncthreads();  // the previous value of *slot has been read by everyone
  if (threadIdx.x == 0) *slot = atomicAdd(counter, 1u);
  __syncthreads();
  return *slot;
}

struct ExactShape {
  int F[2];          // flagged queries of this pass per database
  int qgroups[2];    // groups of EXACT_QG queries
  unsigned int units[2];
};

__device__ __forceinline__ ExactShape exact_shape(const ExactParams& p) {
  ExactShape sh;
  const int r0 = p.pass * p.f_cap;
#pragma unroll
  for (int dbi = 0; dbi < 2; ++dbi) {
    sh.F[dbi] = 0;
    sh.qgroups[dbi] = 0;
    sh.units[dbi] = 0;
    if (dbi < p.n_db) {
      const int nfl = *p.db[dbi].n_flagged;
      if (nfl > r0) {
        sh.F[dbi] = min(p.f_cap, nfl - r0);
        sh.qgroups[dbi] = (sh.F[dbi] + EXACT_QG - 1) / EXACT_QG;
        sh.units[dbi] = static_cast<unsigned int>(sh.qgroups[dbi]) * static_cast<unsigned int>(p.db[dbi].chunks);
      }
    }
  }
  return sh;
}

// phase 1: unit = (database, query group, row chunk); the finished-unit count is the barrier
__device__ __forceinline__ void exact_scores(const ExactParams& p, const ExactShape& sh, uint8_t* ex_smem,
                                             unsigned int* slot) {
  float* qs = reinterpret_cast<float*>(ex_smem);  // EXACT_QG * dq
  const int dq = (p.d + 3) & ~3;
  float* wmax = qs + EXACT_QG * dq;               // [warps][EXACT_QG] per-warp chunk maxima
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wpb = blockDim.x >> 5;
  const int r0 = p.pass * p.f_cap;
  const unsigned int total = sh.units[0] + sh.units[1];
  __shared__ int qex[EXACT_QG * EXCLUDE_MAX];  // the group's excluded rows (search with exclusion)
  int have_db = -1, have_g0 = -1;
  for (;;) {
    unsigned int u = exact_claim(p.work, slot);
    if (u >= total) break;
    const int dbi = u < sh.units[0] ? 0 : 1;
    if (dbi == 1) u -= sh.units[0];
    const ExactDb& e = p.db[dbi];
    const int g0 = static_cast<int>(u / e.chunks) * EXACT_QG;
    const long long chunk = u % e.chunks;
    const int G = min(EXACT_QG, sh.F[dbi] - g0);
    if (dbi != have_db || g0 != have_g0) {  // block-uniform; exact_claim's barrier covers the reuse of qs
      for (int i = tid; i < G * dq; i += blockDim.x) {
        const int qi = i / dq, c = i % dq;
        const int q = e.flagged[r0 + g0 + qi];
        qs[i] = c < p.d ? p.q_f32[static_cast<long long>(q) * p.d + c] : 0.f;
      }
      if (p.ex_rows != nullptr && tid < G * p.n_ex) {
        const int q = e.flagged[r0 + g0 + tid / p.n_ex];
        qex[(tid / p.n_ex) * EXCLUDE_MAX + tid % p.n_ex] =
            p.ex_rows[dbi * p.ex_ld + static_cast<long long>(q) * p.n_ex + tid % p.n_ex];
      }
      __syncthreads();
      have_db = dbi;
      have_g0 = g0;
    }
    const long long groups = (e.n_rows + 31) / 32;
    const long long g_end = min(groups, (chunk + 1) * e.cg);
    float best[EXACT_QG];
#pragma unroll
    for (int i = 0; i < EXACT_QG; ++i) best[i] = -INFINITY;
    for (long long g = chunk * e.cg + warp; g < g_end; g += wpb) {
      float keep[EXACT_QG];
#pragma unroll
      for (int i = 0; i < EXACT_QG; ++i) keep[i] = 0.f;
      for (int rr = 0; rr < 32; ++rr) {
        const long long row = g * 32 + rr;
        if (row >= e.n_rows) break;
        const float* xr = e.x_f32 + row * p.d;
#pragma unroll
        for (int i = 0; i < EXACT_QG; ++i) {
          if (i < G) {
            const float sc = warp_exact_score(qs + i * dq, xr, p.d, p.metric, lane);
            if (lane == rr) keep[i] = p.metric == METRIC_L2 ? -sc : sc;
          }
        }
      }
      const long long row = g * 32 + lane;
      if (row < e.n_rows) {
#pragma unroll
        for (int i = 0; i < EXACT_QG; ++i) {
          if (i < G) {
            if (p.ex_rows != nullptr && row_in(qex + i * EXCLUDE_MAX, p.n_ex, row))
              keep[i] = __uint_as_float(EXACT_EXCLUDED_BITS);
            e.scratch[static_cast<long long>(g0 + i) * e.n_rows + row] = keep[i];
            best[i] = fmaxf(best[i], keep[i]);
          }
        }
      }
    }
    // the chunk's best score per query: lanes -> warp -> block
#pragma unroll
    for (int i = 0; i < EXACT_QG; ++i) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) best[i] = fmaxf(best[i], __shfl_xor_sync(0xffffffffu, best[i], o));
      if (lane == 0) wmax[warp * EXACT_QG + i] = best[i];
    }
    __syncthreads();
    if (tid < G) {
      float m = wmax[tid];
      for (int w = 1; w < wpb; ++w) m = fmaxf(m, wmax[w * EXACT_QG + tid]);
      e.cmax[static_cast<long long>(g0 + tid) * e.chunks + chunk] = m;
    }
    __syncthreads();  // every warp's scores of this unit and its maxima are written
    if (tid == 0) {
      __threadfence();
      atomicAdd(p.done, 1u);
    }
  }
  // wait until every unit is finished (by whichever blocks took them)
  if (tid == 0) {
    const unsigned long long t0 = global_timer_ns();
    for (;;) {
      unsigned int v;
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p.done) : "memory");
      if (v >= total) break;
      __nanosleep(200);
      if (global_timer_ns() - t0 > 20000000000ull) {  // never hang the device: flag and go on
        atomicOr(p.err, EXACT_ERR_BARRIER);
        break;
      }
    }
    __threadfence();
  }
  __syncthreads();
}

// phase 2: one (database, flagged query) per call
__device__ __forceinline__ void exact_select(const ExactParams& p, uint8_t* ex_smem, int dbi, int f) {
  const ExactDb& e = p.db[dbi];
  const int r0 = p.pass * p.f_cap;

  float4* part = reinterpret_cast<float4*>(ex_smem);                            // cons.part4
  unsigned int* sel_key = reinterpret_cast<unsigned int*>(part + p.cons.part4); // k
  unsigned int* sel_id = sel_key + p.k;                                         // k
  unsigned int* top_id = sel_id + p.k;                                          // k (rank order)
  float* top_d = reinterpret_cast<float*>(top_id + p.k);                        // k
  float* top_w = top_d + p.k;                                                   // k
  unsigned int* hist = reinterpret_cast<unsigned int*>(top_w + p.k);            // 256
  unsigned int* bcast = hist + 256;                                             // 4
  int* counters = reinterpret_cast<int*>(bcast + 4);                            // 4
  int* wsum = counters + 4;                                                     // 8
  unsigned int* lk = reinterpret_cast<unsigned int*>(wsum + 8);                 // EXACT_LIST_CAP keys
  unsigned int* li = lk + EXACT_LIST_CAP;                                       // EXACT_LIST_CAP row ids
  unsigned int* ck = li + EXACT_LIST_CAP;                                       // chunk maxima (keys)

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wpb = blockDim.x >> 5;
  {
    const int q = e.flagged[r0 + f];
    const float* sc = e.scratch + static_cast<long long>(f) * e.n_rows;
    const long long n = e.n_rows;
    // excluded rows (distinct and in range once staged) are not candidates: k is capped at the rest
    int n_out = 0;
    if (p.ex_rows != nullptr) {
      const int* xr = p.ex_rows + dbi * p.ex_ld + static_cast<long long>(q) * p.n_ex;
      for (int j = 0; j < p.n_ex; ++j) n_out += xr[j] != EX_NONE;
    }
    const int keff = static_cast<int>(min(static_cast<long long>(p.k), n - n_out));
    __syncthreads();
    for (int r = tid; r < p.k; r += blockDim.x) top_id[r] = 0xFFFFFFFFu;
    // Pre-filter: the k-th best row is at least as good as the k-th best chunk maximum t0 (each of
    // the k best chunks holds such a row), so only chunks whose maximum reaches t0 can hold an
    // answer, and only their rows at or above t0 are candidates. A handful of chunks instead of
    // five passes over the whole score row; the dense path below stays for k > chunks and for
    // candidate lists that do not fit (heavily duplicated data).
    bool filled = keff == 0;  // every row excluded: padding only
    if (!filled && e.chunks >= keff && e.chunks <= p.ck_cap && 2 * keff <= EXACT_LIST_CAP) {
      const float* cm = e.cmax + static_cast<long long>(f) * e.chunks;
      for (int c = tid; c < e.chunks; c += blockDim.x) {
        float v = __ldcg(cm + c);
        if (v == 0.f) v = 0.f;
        ck[c] = f32_to_key(v);
      }
      if (tid < 4) counters[tid] = 0;
      __syncthreads();
      const unsigned int t0 = block_kth_largest(ck, e.chunks, keff, hist, bcast);
      for (int c = warp; c < e.chunks; c += wpb) {
        if (ck[c] < t0) continue;  // warp-uniform
        const long long lo = static_cast<long long>(c) * e.cg * 32;
        const long long hi = min(n, lo + e.cg * 32);
#pragma unroll 4
        for (long long i = lo + lane; i < hi; i += 32) {
          float v = __ldcg(sc + i);
          if (v == 0.f) v = 0.f;
          const unsigned int key = f32_to_key(v);
          if (key >= t0) {
            const int pos = atomicAdd(&counters[2], 1);
            if (pos < EXACT_LIST_CAP) {
              lk[pos] = key;
              li[pos] = static_cast<unsigned int>(i);
            }
          }
        }
      }
      __syncthreads();
      const int L = counters[2];
      if (L <= EXACT_LIST_CAP) {  // block-uniform
        const unsigned int kth = block_kth_largest(lk, L, keff, hist, bcast);  // L >= keff: one row per chunk at least
        for (int c = tid; c < L; c += blockDim.x) {
          if (lk[c] > kth) {
            const int pos = atomicAdd(&counters[0], 1);
            sel_key[pos] = lk[c];
            sel_id[pos] = li[c];
          }
        }
        __syncthreads();
        const int n_gt = counters[0], need = keff - n_gt;
        // rows equal to the k-th value: the `need` lowest ids
        for (int c = tid; c < L; c += blockDim.x) {
          if (lk[c] != kth) continue;
          const unsigned int mine = li[c];
          int r = 0;
          for (int j = 0; j < L; ++j) r += (lk[j] == kth) && (li[j] < mine);
          if (r < need) {
            sel_key[n_gt + r] = kth;
            sel_id[n_gt + r] = mine;
          }
        }
        filled = true;
      }
      __syncthreads();
    }
    if (!filled) {
      // k-th largest rank score: 4 x 8-bit radix passes over the score row (global / L2)
      unsigned int prefix = 0, mask = 0;
      int need = keff, n_eq = 0;
      for (int shift = 24; shift >= 0; shift -= 8) {
        for (int i = tid; i < 256; i += blockDim.x) hist[i] = 0;
        __syncthreads();
#pragma unroll 8
        for (long long i = tid; i < n; i += blockDim.x) {  // unrolled: eight loads in flight per thread
          float v = __ldcg(sc + i);
          if (v == 0.f) v = 0.f;
          const unsigned int key = f32_to_key(v);
          if ((key & mask) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1u);
        }
        __syncthreads();
        block_find_bin(hist, need, bcast);
        prefix |= bcast[0] << shift;
        mask |= 255u << shift;
        need = static_cast<int>(bcast[1]);
        if (shift == 0) n_eq = static_cast<int>(hist[bcast[0]]);  // rows scoring exactly the k-th value
        __syncthreads();
      }
      const unsigned int kth = prefix;  // `need` rows equal to kth are wanted, lowest ids first
      if (tid < 4) counters[tid] = 0;
      __syncthreads();
      if (n_eq == need) {
        // the usual case: every row that ties with the k-th value is wanted, so nothing has to be
        // taken in id order -- one pass, no block barriers (the rank sort below orders the output)
#pragma unroll 4
        for (long long i = tid; i < n; i += blockDim.x) {
          float v = __ldcg(sc + i);
          if (v == 0.f) v = 0.f;
          const unsigned int key = f32_to_key(v);
          if (key >= kth) {
            const int pos = key > kth ? atomicAdd(&counters[0], 1) : (keff - need) + atomicAdd(&counters[1], 1);
            sel_key[pos] = key;
            sel_id[pos] = static_cast<unsigned int>(i);
          }
        }
      } else
      // rows strictly better than kth: any order; rows equal to kth: in id order until `need`
      for (long long base = 0; base < n; base += blockDim.x) {
        const long long i = base + tid;
        unsigned int key = 0;
        bool gt = false, eq = false;
        if (i < n) {
          float v = __ldcg(sc + i);
          if (v == 0.f) v = 0.f;
          key = f32_to_key(v);
          gt = key > kth;
          eq = key == kth;
        }
        if (gt) {
          const int pos = atomicAdd(&counters[0], 1);
          sel_key[pos] = key;
          sel_id[pos] = static_cast<unsigned int>(i);
        }
        const int taken = counters[1];  // uniform: only updated between the syncs below
        if (taken < need) {
          const unsigned int bal = __ballot_sync(0xffffffffu, eq);
          if (lane == 0) wsum[warp] = __popc(bal);
          __syncthreads();
          int before = 0;
          for (int w = 0; w < warp; ++w) before += wsum[w];
          const int my = taken + before + __popc(bal & ((1u << lane) - 1u));
          if (eq && my < need) {
            const int pos = (keff - need) + my;  // ties fill the tail slots
            sel_key[pos] = key;
            sel_id[pos] = static_cast<unsigned int>(i);
          }
          __syncthreads();
          if (tid == 0) {
            int tot = 0;
            for (int w = 0; w < wpb; ++w) tot += wsum[w];
            counters[1] = taken + tot;
          }
          __syncthreads();
        }
      }
    }
    __syncthreads();
    float* Dq = e.D + static_cast<long long>(q) * p.k;
    long long* Iq = e.I + static_cast<long long>(q) * p.k;
    for (int c = tid; c < keff; c += blockDim.x) {
      const unsigned long long mine =
          (static_cast<unsigned long long>(sel_key[c]) << 32) | (0xFFFFFFFFu - sel_id[c]);
      int rank = 0;
      for (int j = 0; j < keff; ++j) {
        const unsigned long long other =
            (static_cast<unsigned long long>(sel_key[j]) << 32) | (0xFFFFFFFFu - sel_id[j]);
        rank += other > mine;
      }
      const float v = key_to_f32(sel_key[c]);
      // 0 - v, not -v: an exact match's distance is +0, as the re-rank writes it (v is +0 then)
      const float dv = p.metric == METRIC_L2 ? 0.f - v : v;
      Dq[rank] = dv;
      Iq[rank] = static_cast<long long>(sel_id[c]) + e.id_offset;
      top_id[rank] = sel_id[c];
      top_d[rank] = dv;
    }
    for (int r = keff + tid; r < p.k; r += blockDim.x) {
      Dq[r] = p.metric == METRIC_L2 ? FLT_MAX : -FLT_MAX;
      Iq[r] = -1;
    }
    if (p.cons.enabled || p.peer.n > 1) {
      __syncthreads();
      if (p.peer.n > 1) push_row_to_peers(p.peer, dbi, q, p.k, top_id, top_d, e.id_offset, p.metric);
      if (p.cons.enabled && p.cons.host_D[dbi] != nullptr)
        mirror_row_to_host(p.cons, dbi, q, p.k, top_id, top_d, e.id_offset, p.metric);
      if (p.cons.enabled)
        consume_query<1>(p.cons, LocalRows{e.x_f32, p.d}, dbi, q, p.k, p.d, p.metric, top_id, top_d, top_w, part);
    }
  }
}

// Any grid size is correct; the host launches about two blocks per SM.
__global__ void __launch_bounds__(EXACT_THREADS)
k_exact_fallback(const ExactParams p) {
  griddep_wait();  // no early trigger: when this kernel has real work its successor must not take its SM slots
  const unsigned long long t_start = ktimer_begin(p.timing);
  extern __shared__ __align__(16) uint8_t ex_smem[];
  __shared__ unsigned int slot;
  const ExactShape sh = exact_shape(p);  // the same in every block: the flag counts are final by now
  // planner feedback: the search's largest candidate band goes to a mapped host word (a posted
  // write; the host reads it, possibly a search late, when it plans the next call)
  if (p.band_host != nullptr && blockIdx.x == 0 && threadIdx.x == 0) *p.band_host = *p.band_dev;
  if (sh.F[0] + sh.F[1] > 0) {
    exact_scores(p, sh, ex_smem, &slot);
    const unsigned int items = static_cast<unsigned int>(sh.F[0] + sh.F[1]);
    for (;;) {
      const unsigned int it = exact_claim(p.work + 1, &slot);
      if (it >= items) break;
      const int dbi = it < static_cast<unsigned int>(sh.F[0]) ? 0 : 1;
      exact_select(p, ex_smem, dbi, static_cast<int>(dbi == 0 ? it : it - sh.F[0]));
    }
  }
  if (p.peer.n > 1 && p.peer.publish) {
    // Row-sharded exchange: every result row of this step has been stored to the peers by now --
    // by the re-rank kernel (complete before this grid started) or by the blocks of this grid,
    // each of which fenced its stores. The last block to get here publishes the epoch.
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) slot = atomicAdd(p.peer.ticket, 1u);
    __syncthreads();
    if (slot == gridDim.x - 1) {
      if (threadIdx.x < p.peer.n && static_cast<int>(threadIdx.x) != p.peer.my_rank) {
        __threadfence_system();
        st_release_sys(p.peer.flag[threadIdx.x], p.peer.epoch);
      }
      if (threadIdx.x == 0) *p.peer.ticket = 0u;
    }
  }
  ktimer_end(p.timing, t_start);
}

}  // namespace keds
