// Range search (keds_index_range_search): every row closer than a radius, exact in fp32.
//
//   k_prep_rows      queries -> 16-bit operands + statistics (as for the top-k search)
//   k_range_band     per query the band threshold thr_q in approximate-score space
//   k_score_range    the search's tensor-core GEMM; appends every (query, row) with a >= thr_q
//   k_range_rescore  warp_exact_score of every candidate; the strict hits get an order key
//   k_range_scan     hits per query -> offsets (and the caller's lims); clears the counts
//   k_range_scatter  hit keys into their query's segment
//   k_range_sort_runs, k_range_merge   segmented sort by (score, label), runs of 32 then merges
//   k_range_emit     keys -> D (fp32 score bits) and I (labels)
//
// The band (DESIGN.md section 3, "range search"): |a - s| <= eps for the approximate score a and
// the real-valued score s, and the fp32 score s32 that decides a hit is within rho of s. A row whose
// s32 passes the radius therefore has a >= thr_q = (IP) r - eps - rho, (L2) (|q|^2 - r)/2 - eps -
// rho', so the candidates hold every hit: no candidate list can drop one, and no fallback exists.
#pragma once

namespace keds {

constexpr int RANGE_RUN = 32;  // sorted runs the first sort step leaves inside a query's segment

// Per query: thr_q (see above), with eps the search certificate's bound (k_select_rerank) and
//   IP: rho = gamma |q| max|x|              (|s32 - s| <= gamma sum |q_i x_i|)
//   L2: rho' = gamma (|q|^2 + r) / 2        (s32 >= (1 - gamma) s for a sum of squares, and |q|^2
//                                            itself is an fp32 sum of squares)
// gamma = m u / (1 - m u), u = 2^-24, m = the longest rounding chain of warp_exact_score: a lane's
// fma chain (<= d_pad / 32 + 3 terms) + the 5-level butterfly (+ the rounded difference under L2).
// Margins (1.001, and 2^-21 |r|) cover the fp32 evaluation of the threshold itself. An unbounded
// or NaN threshold becomes -inf: every row of that query is a candidate.
__global__ void k_range_band(const float4* __restrict__ qstat, const unsigned int* __restrict__ dbstat, int nq,
                             int d_pad, int metric, float radius, float eps_scale, float* __restrict__ thr) {
  griddep_wait();  // qstat comes from k_prep_rows
  griddep_launch_dependents();
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  const float4 qs = qstat[q];
  const float xb = __uint_as_float(dbstat[0]);
  const float xd = __uint_as_float(dbstat[1]);
  const float xn2 = __uint_as_float(dbstat[2]);
  const float qn = sqrtf(qs.x);
  float eps = qs.z * xb + qn * xd + (static_cast<float>(d_pad) * 2.4e-7f) * qs.y * xb;
  if (metric == METRIC_L2) eps += 1.0e-6f * xn2 + 1.2e-7f * (qs.y * xb + 0.5f * xn2);
  eps *= 1.0001f * eps_scale;
  const float mu = static_cast<float>(d_pad / 32 + 3 + 5 + 2) * 5.9604645e-8f;
  const float gamma = mu / (1.f - mu);
  float t;
  if (metric == METRIC_L2) {
    const float rho = 0.5f * gamma * (qs.x + fabsf(radius)) * 1.0001f;
    t = 0.5f * (qs.x - radius) - (eps + rho) * 1.001f - 4.8e-7f * (fabsf(radius) + qs.x);
  } else {
    const float rho = gamma * qn * sqrtf(xn2) * 1.0001f;
    t = radius - (eps + rho) * 1.001f - 4.8e-7f * fabsf(radius);
  }
  if (!(t == t) || !(eps < INFINITY)) t = -INFINITY;
  thr[q] = t;
}

// One warp per candidate {query, row}: its exact fp32 score (the search's routine, so the same
// bits as search() for that pair) and, for a strict hit, its order key (never 0) and a count.
__global__ void k_range_rescore(const uint2* __restrict__ cand, long long n, const float* __restrict__ q_f32,
                                const float* __restrict__ x_f32, int d, int metric, float radius,
                                unsigned long long* __restrict__ key, int* __restrict__ qcnt) {
  const int lane = threadIdx.x & 31;
  const long long w0 = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const long long nw = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  for (long long c = w0; c < n; c += nw) {
    const uint2 e = cand[c];
    const float s = warp_exact_score(q_f32 + static_cast<long long>(e.x) * d, x_f32 + static_cast<long long>(e.y) * d,
                                     d, metric, lane);
    const bool hit = metric == METRIC_L2 ? s < radius : s > radius;
    if (lane == 0) {
      key[c] = hit ? order_key(metric == METRIC_L2 ? -s : s, e.y) : 0ull;
      if (hit) atomicAdd(qcnt + e.x, 1);
    }
  }
}

// One block of 1024 threads: off[i] = hits of queries < i (i <= nq), lims[i] = base + off[i],
// qcnt cleared for the scatter's cursors; out[0] = total hits, out[1] = largest segment.
__global__ void __launch_bounds__(1024) k_range_scan(int* __restrict__ qcnt, int nq, long long base,
                                                     long long* __restrict__ off, long long* __restrict__ lims,
                                                     unsigned long long* __restrict__ out) {
  __shared__ long long wsum[32];
  __shared__ int wmax[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int per = (nq + blockDim.x - 1) / blockDim.x;
  const int i0 = min(nq, tid * per), i1 = min(nq, i0 + per);
  long long s = 0;
  int mx = 0;
  for (int i = i0; i < i1; ++i) {
    s += qcnt[i];
    mx = max(mx, qcnt[i]);
  }
  long long incl = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const long long t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if (lane == 31) wsum[warp] = incl;
  if (lane == 0) wmax[warp] = mx;
  __syncthreads();
  long long before = incl - s;
  for (int w = 0; w < warp; ++w) before += wsum[w];
  for (int i = i0; i < i1; ++i) {
    off[i] = before;
    lims[i] = base + before;
    before += qcnt[i];
    qcnt[i] = 0;
  }
  if (tid == blockDim.x - 1) {
    off[nq] = before;
    lims[nq] = base + before;
    int m = 0;
    for (int w = 0; w < static_cast<int>(blockDim.x >> 5); ++w) m = max(m, wmax[w]);
    out[0] = static_cast<unsigned long long>(before);
    out[1] = static_cast<unsigned long long>(m);
  }
}

__global__ void k_range_scatter(const uint2* __restrict__ cand, const unsigned long long* __restrict__ key_in,
                                long long n, const long long* __restrict__ off, int* __restrict__ cursor,
                                unsigned long long* __restrict__ key_out) {
  for (long long c = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; c < n;
       c += static_cast<long long>(gridDim.x) * blockDim.x) {
    const unsigned long long k = key_in[c];
    if (k != 0ull) {
      const int q = static_cast<int>(cand[c].x);
      key_out[off[q] + atomicAdd(cursor + q, 1)] = k;
    }
  }
}

// The query whose segment [off[q], off[q+1]) holds position e (binary search over nq + 1 offsets).
__device__ __forceinline__ int range_segment(const long long* __restrict__ off, int nq, long long e) {
  int lo = 0, hi = nq;  // off[lo] <= e < off[hi]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (off[mid] <= e) lo = mid; else hi = mid;
  }
  return lo;
}

// Sort runs of RANGE_RUN keys inside every segment, descending (keys are distinct within a
// segment: one per row), by counting the larger keys of the run.
__global__ void k_range_sort_runs(const unsigned long long* __restrict__ in, unsigned long long* __restrict__ out,
                                  long long n, const long long* __restrict__ off, int nq) {
  for (long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; e < n;
       e += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int q = range_segment(off, nq, e);
    const long long s0 = off[q], s1 = off[q + 1];
    const long long r0 = s0 + (e - s0) / RANGE_RUN * RANGE_RUN, r1 = min(r0 + RANGE_RUN, s1);
    const unsigned long long mine = in[e];
    int rank = 0;
    for (long long j = r0; j < r1; ++j) rank += in[j] > mine;
    out[r0 + rank] = mine;
  }
}

// Merge sorted runs of `run` keys pairwise inside every segment: a key's place is its place in
// its own run plus the number of larger keys in the sibling run (binary search).
__global__ void k_range_merge(const unsigned long long* __restrict__ in, unsigned long long* __restrict__ out,
                              long long n, const long long* __restrict__ off, int nq, long long run) {
  for (long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; e < n;
       e += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int q = range_segment(off, nq, e);
    const long long s0 = off[q], s1 = off[q + 1];
    const long long p = e - s0, r = p / run;
    const long long pair0 = s0 + (r & ~1ll) * run;
    const long long sib0 = s0 + (r ^ 1ll) * run, sib1 = min(sib0 + run, s1);
    const unsigned long long mine = in[e];
    long long lo = sib0, hi = max(sib0, sib1);  // first position in the sibling whose key is below mine
    while (lo < hi) {
      const long long mid = (lo + hi) >> 1;
      if (in[mid] > mine) lo = mid + 1; else hi = mid;
    }
    out[pair0 + (p - r * run) + (lo - sib0)] = mine;
  }
}

// Order keys -> results: D is the fp32 score (IP) or squared distance (L2) with the bits
// warp_exact_score produced (it never produces -0, which order_key folds into +0), I = row + id_offset.
__global__ void k_range_emit(const unsigned long long* __restrict__ key, long long n, int metric, long long id_offset,
                             float* __restrict__ D, long long* __restrict__ I) {
  for (long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; e < n;
       e += static_cast<long long>(gridDim.x) * blockDim.x) {
    const unsigned long long k = key[e];
    float s = key_to_f32(static_cast<uint32_t>(k >> 32));
    if (metric == METRIC_L2) s = -s;
    if (s == 0.f) s = 0.f;
    D[e] = s;
    I[e] = static_cast<long long>(0xFFFFFFFFu - static_cast<uint32_t>(k)) + id_offset;
  }
}

}  // namespace keds
