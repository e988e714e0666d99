// Candidate selection + exact fp32 re-rank + exactness certificate (+ neighbour consumer).
// One block per (query, database), launched right behind the scoring kernel.
//
// Certificate.  Let a(n) be the bf16-GEMM score of row n and s(n) the exact one, |a - s| <= eps
// for every row (Cauchy-Schwarz on the two bf16 rounding residuals + an fp32 accumulation
// allowance).  With a_(k) the k-th largest approximate score, every true top-k row has
// a(n) >= a_(k) - 2 eps.  So C = { n : a(n) >= tau }, tau = a_(k) - 2 eps, contains the exact answer
// provided no slice dropped a row scoring >= tau, i.e. every slice threshold theta < tau.  C is
// re-scored in fp32 and ordered by (score desc, id asc).  If the certificate fails (or |C| is too
// large) the query is queued for the exact fallback instead.
//
// Input: per (slice, query) one 128-byte line of <= LKEEP-1 candidates (score_topk_sm100.cuh).
// The dependency chain is kept short: one round trip for all candidate lines + query + norms,
// a few shared-memory selection steps, one round trip for the fp32 rows, then ordering/consumer.
#pragma once

namespace keds {

struct RerankParams {
  ConsumeParams cons;
  int n_db, n_qt, S, nq, k, d, metric;
  const uint2* cand;         // [item][BM][LKEEP]
  const int* cand_cnt;       // [item][BM]
  const float* cand_theta;   // [item][BM]
  const float* q_f32;        // [nq][d]
  const float4* qstat;       // [nq] {|q|^2, |bf16 q|, |q - bf16 q|}
  const float* x_f32[2];
  const unsigned int* dbstat[2];
  float* D[2];
  long long* I[2];
  long long id_offset[2];
  int* flagged[2];
  int* n_flagged[2];
  float eps_scale;           // 1.0 normally; tests shrink/grow it to exercise the fallback
  int rmax;                  // candidate capacity of this launch (<= R_MAX; sizes the shared arrays)
  unsigned int* band_max;    // status word: largest |C| of this search (feeds the planner's next slice count)
  PeerOut peer;              // row-sharded exchange; n == 0: off
  unsigned long long* timing;  // nullable in-kernel launch timer
};

constexpr unsigned int PAD_ID = 0xFFFFFFFFu;

// R = candidate rows per warp in flight during the fp32 re-score. <3, 2>: small batches, shortest
// dependency chain (two blocks per SM). <1, 4>: large batches, four blocks per SM so that many
// queries overlap their phases.
template <int R, int MINB, int THREADS = RERANK_THREADS>
__global__ void __launch_bounds__(THREADS, MINB)
k_select_rerank(const RerankParams p) {
  extern __shared__ uint8_t rr_smem[];
  const int q = blockIdx.x, db = blockIdx.y;
  const int qt = q / BM, ql = q % BM;
  const int slots = p.S * LKEEP;
  // shared layout
  float* qvec = reinterpret_cast<float*>(rr_smem);                       // d (16-B aligned)
  float4* part = reinterpret_cast<float4*>(qvec + ((p.d + 3) & ~3));     // cons.part4
  unsigned long long* okey = reinterpret_cast<unsigned long long*>(part + p.cons.part4);  // R_MAX order keys
  unsigned int* keys = reinterpret_cast<unsigned int*>(okey + p.rmax);   // slots
  unsigned int* ids = keys + slots;                                      // slots
  unsigned int* smax = ids + slots;                                      // S   slice maxima (keys)
  unsigned int* a_key = smax + p.S;                                      // rmax survivors
  unsigned int* a_id = a_key + p.rmax;                                   // rmax
  unsigned int* sel_id = a_id + p.rmax;                                  // rmax  the set C
  float* sel_sc = reinterpret_cast<float*>(sel_id + p.rmax);             // rmax
  unsigned int* hist = reinterpret_cast<unsigned int*>(sel_sc + p.rmax); // 256 (radix path only)
  float* red = reinterpret_cast<float*>(hist + 256);                     // 32
  unsigned int* bcast = reinterpret_cast<unsigned int*>(red + 32);       // 4
  int* counters = reinterpret_cast<int*>(bcast + 4);                     // 4
  unsigned int* top_id = reinterpret_cast<unsigned int*>(counters + 4);  // k  (rank order)
  float* top_d = reinterpret_cast<float*>(top_id + p.k);                 // k
  float* top_w = top_d + p.k;                                            // k

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  if (tid < 4) counters[tid] = 0;
  for (int r = tid; r < p.k; r += blockDim.x) top_id[r] = PAD_ID;
  // the query and the error-bound inputs do not depend on the scoring kernel
  for (int c = tid; c < p.d; c += blockDim.x) qvec[c] = p.q_f32[static_cast<long long>(q) * p.d + c];
  const float xb = __uint_as_float(p.dbstat[db][0]);
  const float xd = __uint_as_float(p.dbstat[db][1]);
  const float xn2 = __uint_as_float(p.dbstat[db][2]);
  griddep_wait();  // candidates (and qstat from k_prep_rows) are visible from here on
  const unsigned long long t_start = ktimer_begin(p.timing);

  // ---- A: every slice's candidate line, count and threshold in one round trip.
  // Half a warp per slice: lane e < LKEEP reads entry e (one 128-byte line per slice).
  const float4 qs = p.qstat[q];
  float th_max = -INFINITY;
  int n_valid = 0;
  constexpr int MAX_IT = 6;  // loads issued back to back before the first use
  const int e = lane & 15;
  for (int sb = 0; sb < p.S; sb += MAX_IT * nwarps * 2) {
    uint2 en[MAX_IT];
    float th[MAX_IT];
    int cn[MAX_IT];
#pragma unroll
    for (int it = 0; it < MAX_IT; ++it) {
      const int s = sb + (it * nwarps + warp) * 2 + (lane >> 4);
      en[it] = make_uint2(0xff800000u, PAD_ID);
      th[it] = -INFINITY;
      cn[it] = 0;
      if (s < p.S) {
        const long long item = (static_cast<long long>(db) * p.S + s) * p.n_qt + qt;
        en[it] = __ldcg(p.cand + (item * BM + ql) * LKEEP + e);
        if (e == 0) {
          th[it] = __ldcg(p.cand_theta + item * BM + ql);
          cn[it] = __ldcg(p.cand_cnt + item * BM + ql);
        }
      }
    }
#pragma unroll
    for (int it = 0; it < MAX_IT; ++it) {
      const int s = sb + (it * nwarps + warp) * 2 + (lane >> 4);
      float sc = __uint_as_float(en[it].x);
      if (sc == 0.f) sc = 0.f;
      const unsigned int id = en[it].y;
      const unsigned int key = id != PAD_ID ? f32_to_key(sc) : 0u;
      if (s < p.S) {
        keys[s * LKEEP + e] = key;
        ids[s * LKEEP + e] = id;
      }
      th_max = fmaxf(th_max, th[it]);
      n_valid += cn[it];
      // slice maximum over its 16 lanes
      unsigned int mx = key;
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      if (s < p.S && e == 0) smax[s] = mx;
    }
  }
  // block-wide: max theta, number of valid candidates
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    th_max = fmaxf(th_max, __shfl_xor_sync(0xffffffffu, th_max, o));
    n_valid += __shfl_xor_sync(0xffffffffu, n_valid, o);
  }
  if (lane == 0) {
    red[warp] = th_max;
    atomicAdd(&counters[3], n_valid);
  }
  __syncthreads();  // (1)
  th_max = red[0];
  for (int w = 1; w < nwarps; ++w) th_max = fmaxf(th_max, red[w]);
  const int n = counters[3];

  // eps: |a - s| <= |dq| |x16| + |q| |dx| + accumulation allowance (x16 / q16: the operands as
  // rounded to the 16-bit format, dq / dx the rounding residuals). Under L2 the approximate score
  // also carries bias = fl(-0.5 fl(|x|^2)) and one more fp32 add: |x|^2 is a 24-term chain per lane
  // plus a 5-level tree (<= 29 roundings), so 0.5 * 30 * 2^-24 |x|^2 covers the bias and
  // 2^-23 (|a| + |bias|) the add.
  const float qn = sqrtf(qs.x);
  const int d_pad = (p.d + BK - 1) / BK * BK;
  float eps = qs.z * xb + qn * xd + (static_cast<float>(d_pad) * 2.4e-7f) * qs.y * xb;
  if (p.metric == METRIC_L2) eps += 1.0e-6f * xn2 + 1.2e-7f * (qs.y * xb + 0.5f * xn2);
  eps *= 1.0001f * p.eps_scale;
  if (!(eps == eps)) eps = INFINITY;  // inf * 0 from a degenerate query: nothing is certified

  // ---- B: survivors A' = { a >= t0 - 2 eps } with t0 <= a_(k) a cheap lower bound, so that
  // C = { a >= a_(k) - 2 eps } is a subset of A'.
  float tau = -INFINITY;
  bool radix = false;
  unsigned int kth = 0u;
  if (n >= p.k) {
    if (p.S >= p.k) {
      // t0 = k-th largest slice maximum (each of the k best slices holds a row at least that good)
      for (int s = tid; s < p.S; s += blockDim.x) {
        const unsigned int mine = smax[s];
        int rank = 0;
#pragma unroll 8
        for (int u = 0; u < p.S; ++u) {
          const unsigned int o = smax[u];
          rank += (o > mine) || (o == mine && u < s);
        }
        if (rank == p.k - 1) bcast[2] = mine;
      }
      __syncthreads();  // (2)
      const float t0 = bcast[2] != 0u ? key_to_f32(bcast[2]) : -INFINITY;
      const float thr = t0 - 2.f * eps;
      // few slots survive: one shared-memory atomic per warp and pass, none for most warps
      for (int i0 = 0; i0 < slots; i0 += blockDim.x) {
        const int i = i0 + tid;
        unsigned int id = PAD_ID, key = 0u;
        if (i < slots) {
          id = ids[i];
          key = keys[i];
        }
        const bool hit = id != PAD_ID && key_to_f32(key) >= thr;
        const unsigned int bal = __ballot_sync(0xffffffffu, hit);
        if (bal != 0u) {
          int base = 0;
          if (lane == 0) base = atomicAdd(&counters[2], __popc(bal));
          base = __shfl_sync(0xffffffffu, base, 0);
          const int pos = base + __popc(bal & ((1u << lane) - 1u));
          if (hit && pos < p.rmax) {
            a_key[pos] = key;
            a_id[pos] = id;
          }
        }
      }
      __syncthreads();  // (3)
      const int na = counters[2];
      if (na <= p.rmax) {
        if (na <= 256) {
          // a_(k): the survivor with fewer than k keys above it and at least k keys at or above it
          for (int c = tid; c < na; c += blockDim.x) {
            const unsigned int mine = a_key[c];
            int gt = 0, ge = 0;
#pragma unroll 8
            for (int j = 0; j < na; ++j) {
              const unsigned int o = a_key[j];
              gt += o > mine;
              ge += o >= mine;
            }
            if (gt < p.k && ge >= p.k) bcast[3] = mine;
          }
          __syncthreads();  // (4)
          kth = bcast[3];
        } else {
          // crowded band (clustered data): the quadratic count would dominate -- radix select
          kth = block_kth_largest(a_key, na, p.k, hist, bcast);
        }
        tau = key_to_f32(kth) - 2.f * eps;
        // C = survivors at or above tau
        for (int c = tid; c < na; c += blockDim.x) {
          if (key_to_f32(a_key[c]) >= tau) {
            const int pos = atomicAdd(&counters[1], 1);
            sel_id[pos] = a_id[c];
          }
        }
      } else {
        radix = true;
      }
    } else if (slots <= 1024) {
      // fewer slices than k: no slice-maximum bound, but the candidate set is small -- find a_(k)
      // by rank counting over all of it (padding keys are 0 and never counted as >= a valid key
      // unless k exceeds the valid count, which n >= k excludes)
      for (int i = tid; i < slots; i += blockDim.x) {
        if (ids[i] == PAD_ID) continue;
        const unsigned int mine = keys[i];
        int gt = 0, ge = 0;
        for (int j = 0; j < slots; ++j) {
          const unsigned int o = keys[j];
          const bool valid = ids[j] != PAD_ID;
          gt += valid && o > mine;
          ge += valid && o >= mine;
        }
        if (gt < p.k && ge >= p.k) bcast[3] = mine;
      }
      __syncthreads();
      kth = bcast[3];
      tau = key_to_f32(kth) - 2.f * eps;
      for (int i = tid; i < slots; i += blockDim.x) {
        const unsigned int id = ids[i];
        if (id != PAD_ID && key_to_f32(keys[i]) >= tau) {
          const int pos = atomicAdd(&counters[1], 1);
          if (pos < p.rmax) sel_id[pos] = id;
        }
      }
    } else {
      radix = true;
    }
    if (radix) {
      // few slices or a crowded band: exact k-th largest by radix select over all candidates
      __syncthreads();
      kth = block_kth_largest(keys, slots, p.k, hist, bcast);  // padding keys are 0: never in the top n
      tau = key_to_f32(kth) - 2.f * eps;
      for (int i = tid; i < slots; i += blockDim.x) {
        const unsigned int id = ids[i];
        if (id != PAD_ID && key_to_f32(keys[i]) >= tau) {
          const int pos = atomicAdd(&counters[1], 1);
          if (pos < p.rmax) sel_id[pos] = id;
        }
      }
    }
  } else {
    // fewer candidates than k (tiny database): everything is a candidate
    for (int i = tid; i < slots; i += blockDim.x) {
      const unsigned int id = ids[i];
      if (id != PAD_ID) {
        const int pos = atomicAdd(&counters[1], 1);
        if (pos < p.rmax) sel_id[pos] = id;
      }
    }
  }
  __syncthreads();  // (5)
  int m = counters[1];
  const bool ok = (m <= p.rmax) && (th_max == -INFINITY || th_max < tau);
  if (tid == 0) {
    if (!ok) {
      const int pos = atomicAdd(p.n_flagged[db], 1);
      p.flagged[db][pos] = q;
    }
    // an unusually crowded band is reported to the host planner (more slices next time)
    if (p.band_max != nullptr && m > 2 * p.k) atomicMax(p.band_max, static_cast<unsigned int>(m));
  }
  m = min(m, p.rmax);

  // ---- C: exact fp32 scores of the candidates, R rows per warp in flight
  const float* xbase = p.x_f32[db];
  for (int c0 = warp * R; c0 < m; c0 += nwarps * R) {
    const float* xr[R];
#pragma unroll
    for (int r = 0; r < R; ++r)
      xr[r] = xbase + static_cast<long long>(sel_id[min(c0 + r, m - 1)]) * p.d;
    float sc[R];
    warp_exact_score_multi<R>(qvec, xr, p.d, p.metric, lane, sc);
    if (lane == 0) {
#pragma unroll
      for (int r = 0; r < R; ++r)
        if (c0 + r < m) sel_sc[c0 + r] = sc[r];
    }
  }
  __syncthreads();  // (6)

  // ---- D: order by (score desc, id asc), write the top k
  float* Dq = p.D[db] + static_cast<long long>(q) * p.k;
  long long* Iq = p.I[db] + static_cast<long long>(q) * p.k;
  if (m > 64) {
    // many candidates: build the 64-bit order keys once instead of inside the quadratic loop
    for (int c = tid; c < m; c += blockDim.x) {
      const float sc = sel_sc[c];
      okey[c] = order_key(p.metric == METRIC_L2 ? -sc : sc, sel_id[c]);
    }
    __syncthreads();
  }
  for (int c = tid; c < m; c += blockDim.x) {
    const float sc = sel_sc[c];
    const unsigned long long mine = order_key(p.metric == METRIC_L2 ? -sc : sc, sel_id[c]);
    int rank = 0;
    if (m > 64) {
#pragma unroll 8
      for (int j = 0; j < m; ++j) rank += okey[j] > mine;
    } else {
#pragma unroll 8
      for (int j = 0; j < m; ++j) {
        const float sj = sel_sc[j];
        rank += order_key(p.metric == METRIC_L2 ? -sj : sj, sel_id[j]) > mine;
      }
    }
    if (rank < p.k) {
      Dq[rank] = sc;
      Iq[rank] = static_cast<long long>(sel_id[c]) + p.id_offset[db];
      top_id[rank] = sel_id[c];
      top_d[rank] = sc;
    }
  }
  for (int r = m + tid; r < p.k; r += blockDim.x) {
    Dq[r] = p.metric == METRIC_L2 ? FLT_MAX : -FLT_MAX;
    Iq[r] = -1;
  }
  // a flagged query is consumed (and sent to the peers) by the exact fallback instead, once its
  // answer is final
  if (ok && (p.cons.enabled || p.peer.n > 1)) {
    __syncthreads();  // (7)
    if (p.peer.n > 1)
      push_row_to_peers(p.peer, db, q, p.k, top_id, top_d, p.id_offset[db], p.metric);
    if (p.cons.enabled && p.cons.host_D[db] != nullptr)
      mirror_row_to_host(p.cons, db, q, p.k, top_id, top_d, p.id_offset[db], p.metric);
    if (p.cons.enabled)
      consume_query<(R >= 2 ? 2 : 1)>(p.cons, LocalRows{xbase, p.d}, db, q, p.k, p.d, p.metric, top_id, top_d, top_w,
                                      part);
  }
  ktimer_end(p.timing, t_start);
}

}  // namespace keds
