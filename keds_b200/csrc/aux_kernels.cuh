// Plain CUDA-core kernels around the tcgen05 scoring kernel: operand preparation, candidate
// selection + exact fp32 re-rank with an exactness certificate, the exact fp32 fallback, shard
// merge, neighbour gather / weighted pool, gallery rank counting and label-hit counting.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <float.h>
#include "score_topk_sm100.cuh"

namespace keds {

constexpr int METRIC_IP = 0;
constexpr int METRIC_L2 = 1;
constexpr int RERANK_THREADS = 256;  // ~112 regs/thread: two blocks per SM, one wave for 2 x 128 queries
constexpr int R_MAX = 1024;     // most candidates one query may send to the fp32 re-rank
constexpr int P2P_MAX_RANKS = 8;  // GPUs of one box taking part in a row-sharded exchange
constexpr int K_MAX = 2048;     // largest k (Faiss' GPU flat index has the same limit)
constexpr int EXACT_THREADS = 256;
constexpr int EXACT_QG = 8;     // queries scored together against one pass over the rows

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// The one fp32 scoring routine of the library (re-rank, fallback and gallery ranking all call it,
// so a (query,row) pair gets the same bits on every path). Warp-cooperative; q may be shared or
// global memory. IP: sum q*x. L2: sum (q-x)^2. Every lane returns the full sum.
__device__ __forceinline__ float warp_exact_score(const float* __restrict__ q,
                                                  const float* __restrict__ x, int d, int metric,
                                                  int lane) {
  float acc = 0.f;
  if ((d & 3) == 0 && ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(q)) & 15) == 0) {
    const float4* x4 = reinterpret_cast<const float4*>(x);
    const float4* q4 = reinterpret_cast<const float4*>(q);
    const int d4 = d >> 2;
    if (metric == METRIC_IP) {
      for (int c = lane; c < d4; c += 32) {
        const float4 a = __ldg(x4 + c);
        const float4 b = q4[c];
        acc = fmaf(a.x, b.x, acc);
        acc = fmaf(a.y, b.y, acc);
        acc = fmaf(a.z, b.z, acc);
        acc = fmaf(a.w, b.w, acc);
      }
    } else {
      for (int c = lane; c < d4; c += 32) {
        const float4 a = __ldg(x4 + c);
        const float4 b = q4[c];
        float t;
        t = b.x - a.x; acc = fmaf(t, t, acc);
        t = b.y - a.y; acc = fmaf(t, t, acc);
        t = b.z - a.z; acc = fmaf(t, t, acc);
        t = b.w - a.w; acc = fmaf(t, t, acc);
      }
    }
  } else {
    if (metric == METRIC_IP) {
      for (int c = lane; c < d; c += 32) acc = fmaf(__ldg(x + c), q[c], acc);
    } else {
      for (int c = lane; c < d; c += 32) {
        const float t = q[c] - __ldg(x + c);
        acc = fmaf(t, t, acc);
      }
    }
  }
  return warp_sum(acc);
}

// R rows against one query with the loads of all R rows in flight together. Per row the
// operations and their order are exactly those of warp_exact_score (bit-identical results).
template <int R>
__device__ __forceinline__ void warp_exact_score_multi(const float* __restrict__ q,
                                                       const float* const (&x)[R], int d, int metric,
                                                       int lane, float (&out)[R]) {
  bool vec = (d & 3) == 0 && (reinterpret_cast<uintptr_t>(q) & 15) == 0;
#pragma unroll
  for (int r = 0; r < R; ++r) vec = vec && (reinterpret_cast<uintptr_t>(x[r]) & 15) == 0;
  if (!vec) {
#pragma unroll
    for (int r = 0; r < R; ++r) out[r] = warp_exact_score(q, x[r], d, metric, lane);
    return;
  }
  const float4* q4 = reinterpret_cast<const float4*>(q);
  const int d4 = d >> 2;
  float acc[R];
#pragma unroll
  for (int r = 0; r < R; ++r) acc[r] = 0.f;
  constexpr int U = 6;  // float4 chunks per lane per block: d = 768 is exactly one block
  for (int cb = 0; cb < d4; cb += 32 * U) {
    float4 a[R][U];
    // issue every load of the block (R rows x U chunks) before the first use
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int c = cb + u * 32 + lane;
#pragma unroll
      for (int r = 0; r < R; ++r)
        a[r][u] = c < d4 ? __ldg(reinterpret_cast<const float4*>(x[r]) + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int c = cb + u * 32 + lane;
      if (c < d4) {
        const float4 b = q4[c];
#pragma unroll
        for (int r = 0; r < R; ++r) {
          if (metric == METRIC_IP) {
            acc[r] = fmaf(a[r][u].x, b.x, acc[r]);
            acc[r] = fmaf(a[r][u].y, b.y, acc[r]);
            acc[r] = fmaf(a[r][u].z, b.z, acc[r]);
            acc[r] = fmaf(a[r][u].w, b.w, acc[r]);
          } else {
            float t;
            t = b.x - a[r][u].x; acc[r] = fmaf(t, t, acc[r]);
            t = b.y - a[r][u].y; acc[r] = fmaf(t, t, acc[r]);
            t = b.z - a[r][u].z; acc[r] = fmaf(t, t, acc[r]);
            t = b.w - a[r][u].w; acc[r] = fmaf(t, t, acc[r]);
          }
        }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < R; ++r) out[r] = warp_sum(acc[r]);
}

// Total order used everywhere: better score first, then lower row id.
// `rank_score` is the IP value, or minus the squared distance under L2.
__device__ __forceinline__ unsigned long long order_key(float rank_score, uint32_t id) {
  if (rank_score == 0.f) rank_score = 0.f;  // -0 -> +0
  return (static_cast<unsigned long long>(f32_to_key(rank_score)) << 32) |
         static_cast<unsigned long long>(0xFFFFFFFFu - id);
}

// ---------------------------------------------------------------------------------------------
// Operand preparation: fp32 rows -> 16-bit rows padded to d_pad, plus the per-row statistics the
// exactness certificate needs. One warp per row. x16 = the row rounded to the operand format.
//   stat[r] = { |x|^2, |x16|, |x - x16|, 0 }                (optional)
//   bias[r] = -0.5 |x|^2                                    (optional; L2 ranking bias)
//   gmax[0] = max_r |x16_r| , gmax[1] = max_r |x_r - x16_r| , gmax[2] = max_r |x_r|^2   (float bits)
//
// Operand format (fmt). FMT_FP16: 11 significant bits -- on unit-norm embeddings the rounding
// residual |x - x16|, and with it the certificate's error bound, is 8x smaller than bf16's (8
// bits) at the same tensor-core rate and the same bytes. FMT_BF16 keeps fp32's exponent range and
// is chosen for data fp16 would overflow or flush (see choose_format in api.cu). Under FMT_FP16
// values beyond +-65504 are clamped and the row's residual is set to 3e38, so that such a query
// can only be answered by the exact path.
constexpr int FMT_BF16 = 0;
constexpr int FMT_FP16 = 1;

__device__ __forceinline__ unsigned int round_pair(int fmt, float a, float b, float& ra, float& rb, bool& bad) {
  if (fmt == FMT_FP16) {
    const float ca = fminf(fmaxf(a, -65504.f), 65504.f), cb = fminf(fmaxf(b, -65504.f), 65504.f);
    bad = bad || (ca != a) || (cb != b);  // out of range or NaN
    const __half2 h = __floats2half2_rn(ca, cb);
    const float2 f = __half22float2(h);
    ra = f.x;
    rb = f.y;
    return *reinterpret_cast<const unsigned int*>(&h);
  }
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  const float2 f = __bfloat1622float2(h);
  ra = f.x;
  rb = f.y;
  return *reinterpret_cast<const unsigned int*>(&h);
}

// Search with exclusion, staged by k_prep_rows: the caller's labels (as the search returns them,
// id_offset included; device memory or page-locked host memory read through the mapping, once)
// become local row ids per database in handle scratch, so that no later kernel reads the caller's
// array. A label that is -1, outside the database or a repeat of an earlier slot becomes EX_NONE.
struct ExcludeStage {
  const long long* labels;  // [nq][n_ex]; nullptr: no exclusion
  long long nq;
  int n_ex;                 // 1 .. EXCLUDE_MAX
  int n_db;
  long long id_offset[2];
  long long n_rows[2];
  int* rows;                // [n_db][nq][n_ex]
};

// fp32 rows -> 16-bit operand rows and their statistics (queries per search, database rows at add);
// every output is optional (nullptr: not written)
struct PrepParams {
  const float* x;                // [n][d]
  long long n;
  int d, d_pad, fmt;
  uint16_t* out;                 // [n][d_pad] 16-bit rows
  float4* stat;                  // [n] {|x|^2, |x16|, |x - x16|, 0}
  float* bias;                   // [n] -|x|^2 / 2 (L2)
  unsigned int* gmax;            // [3] running maxima of the statistics (float bits, atomicMax)
  unsigned int* zero_words;      // [n_zero] cleared by block 0 (a status block)
  int n_zero;
  float* neg_inf_words;          // [n_neg_inf] set to -inf (the warm-start thresholds)
  int n_neg_inf;
  unsigned long long* timing;
  float* copy_f32;               // [n][d] device copy of x (x in page-locked host memory or misaligned)
  ExcludeStage ex;
};

__global__ void k_prep_rows(const PrepParams p) {
  const float* __restrict__ x = p.x;
  const long long n = p.n;
  const int d = p.d, d_pad = p.d_pad, fmt = p.fmt;
  uint16_t* __restrict__ out = p.out;
  float4* __restrict__ stat = p.stat;
  float* __restrict__ bias = p.bias;
  unsigned int* __restrict__ gmax = p.gmax;
  unsigned int* __restrict__ zero_words = p.zero_words;
  const int n_zero = p.n_zero;
  float* __restrict__ neg_inf_words = p.neg_inf_words;
  const int n_neg_inf = p.n_neg_inf;
  unsigned long long* timing = p.timing;
  float* __restrict__ copy_f32 = p.copy_f32;
  const ExcludeStage& ex = p.ex;
  const int lane = threadIdx.x & 31;
  griddep_wait();               // earlier kernels of the stream may still read what is rewritten here
  griddep_launch_dependents();  // the scoring kernel may start its prologue
  const unsigned long long t_start = ktimer_begin(timing);
  if (ex.labels != nullptr) {
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < ex.nq;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
      int r[2][EXCLUDE_MAX];  // every loop below is unrolled: the arrays stay in registers
#pragma unroll
      for (int e = 0; e < EXCLUDE_MAX; ++e) {
        const long long lab = e < ex.n_ex ? ex.labels[i * ex.n_ex + e] : -1ll;
#pragma unroll
        for (int db = 0; db < 2; ++db) {
          const long long loc = lab - ex.id_offset[db];
          r[db][e] = (lab != -1ll && loc >= 0 && loc < ex.n_rows[db]) ? static_cast<int>(loc) : EX_NONE;
#pragma unroll
          for (int f = 0; f < e; ++f)
            if (r[db][f] == r[db][e]) r[db][e] = EX_NONE;
        }
      }
#pragma unroll
      for (int db = 0; db < 2; ++db) {
        if (db >= ex.n_db) break;
        int* o = ex.rows + (static_cast<long long>(db) * ex.nq + i) * ex.n_ex;
#pragma unroll
        for (int e = 0; e < EXCLUDE_MAX; ++e)
          if (e < ex.n_ex) o[e] = r[db][e];
      }
    }
  }
  // per-call control words (flag counters, error word) are cleared here instead of by a separate
  // memset node in front of every search; the shared per-query thresholds start at -inf
  if (zero_words != nullptr && blockIdx.x == 0)
    for (int i = threadIdx.x; i < n_zero; i += blockDim.x) zero_words[i] = 0u;
  if (neg_inf_words != nullptr)
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_neg_inf; i += gridDim.x * blockDim.x)
      neg_inf_words[i] = -INFINITY;
  const long long warp0 = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  float mx_b = 0.f, mx_d = 0.f, mx_n = 0.f;
  for (long long r = warp0; r < n; r += nwarps) {
    const float* xr = x + r * d;
    uint16_t* orow = out + r * d_pad;
    float n2 = 0.f, b2 = 0.f, e2 = 0.f;
    bool bad = false;
    if ((d & 3) == 0 && (reinterpret_cast<uintptr_t>(xr) & 15) == 0) {
      // 16-byte loads, 8-byte stores (d_pad is a multiple of 64, rows of `out` are 128-B aligned)
      const float4* x4 = reinterpret_cast<const float4*>(xr);
      uint2* o2 = reinterpret_cast<uint2*>(orow);
      const int d4 = d >> 2, dp4 = d_pad >> 2;
#pragma unroll 4
      for (int c = lane; c < dp4; c += 32) {
        const float4 v = c < d4 ? __ldg(x4 + c) : make_float4(0.f, 0.f, 0.f, 0.f);
        // x in page-locked host memory (read through the mapping, once): the kernels behind this
        // one take the fp32 rows from this device copy
        if (copy_f32 != nullptr && c < d4) reinterpret_cast<float4*>(copy_f32 + r * d)[c] = v;
        float4 f;
        uint2 pk;
        pk.x = round_pair(fmt, v.x, v.y, f.x, f.y, bad);
        pk.y = round_pair(fmt, v.z, v.w, f.z, f.w, bad);
        o2[c] = pk;
        n2 = fmaf(v.x, v.x, n2); n2 = fmaf(v.y, v.y, n2); n2 = fmaf(v.z, v.z, n2); n2 = fmaf(v.w, v.w, n2);
        b2 = fmaf(f.x, f.x, b2); b2 = fmaf(f.y, f.y, b2); b2 = fmaf(f.z, f.z, b2); b2 = fmaf(f.w, f.w, b2);
        float e;
        e = v.x - f.x; e2 = fmaf(e, e, e2);
        e = v.y - f.y; e2 = fmaf(e, e, e2);
        e = v.z - f.z; e2 = fmaf(e, e, e2);
        e = v.w - f.w; e2 = fmaf(e, e, e2);
      }
    } else {
      for (int c = lane; c < d_pad; c += 32) {
        const float v = c < d ? xr[c] : 0.f;
        if (copy_f32 != nullptr && c < d) copy_f32[r * d + c] = v;
        float bf, unused;
        const unsigned int pk = round_pair(fmt, v, 0.f, bf, unused, bad);
        orow[c] = static_cast<uint16_t>(pk & 0xFFFFu);
        n2 = fmaf(v, v, n2);
        b2 = fmaf(bf, bf, b2);
        const float e = v - bf;
        e2 = fmaf(e, e, e2);
      }
    }
    n2 = warp_sum(n2);
    b2 = warp_sum(b2);
    e2 = warp_sum(e2);
    bad = __any_sync(0xffffffffu, bad);
    const float bn = sqrtf(b2);
    const float dn = bad ? 3.0e38f : sqrtf(e2);
    if (lane == 0) {
      if (stat != nullptr) stat[r] = make_float4(n2, bn, dn, 0.f);
      if (bias != nullptr) bias[r] = -0.5f * n2;
    }
    mx_b = fmaxf(mx_b, bn);
    mx_d = fmaxf(mx_d, dn);
    mx_n = fmaxf(mx_n, n2);
  }
  if (gmax != nullptr && lane == 0) {
    // round the maxima up by an ulp-ish factor so they stay upper bounds
    atomicMax(gmax + 0, __float_as_uint(mx_b * 1.000001f));
    atomicMax(gmax + 1, __float_as_uint(fminf(mx_d * 1.000001f, 3.0e38f)));
    atomicMax(gmax + 2, __float_as_uint(fminf(mx_n * 1.000001f, 3.0e38f)));
  }
  ktimer_end(timing, t_start);
}

// Which 16-bit format loses less of these rows? One warp per row.
//   out[0] = max |x_rc|, out[1] = max_r |x_r - bf16(x_r)|, out[2] = max_r |x_r - fp16(x_r)|
// as float bit patterns (atomicMax; the caller zeroes them). NaN / inf elements count as inf.
__global__ void k_probe_rows(const float* __restrict__ x, long long n, int d, unsigned int* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const long long warp0 = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  float amax = 0.f, mx_bf = 0.f, mx_fp = 0.f;
  for (long long r = warp0; r < n; r += nwarps) {
    const float* xr = x + r * d;
    float e_bf = 0.f, e_fp = 0.f;
    for (int c = lane; c < d; c += 32) {
      const float v = __ldg(xr + c);
      const float av = (v == v) ? fabsf(v) : INFINITY;
      amax = fmaxf(amax, av);
      float eb = v - __bfloat162float(__float2bfloat16_rn(v));
      float eh = v - __half2float(__float2half_rn(fminf(fmaxf(v, -65504.f), 65504.f)));
      e_bf = fmaf(eb, eb, e_bf);
      e_fp = fmaf(eh, eh, e_fp);
    }
    e_bf = warp_sum(e_bf);
    e_fp = warp_sum(e_fp);
    mx_bf = fmaxf(mx_bf, sqrtf(e_bf));
    mx_fp = fmaxf(mx_fp, sqrtf(e_fp));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
  if (lane == 0) {
    const float big = 3.0e38f;
    atomicMax(out + 0, __float_as_uint(fminf(amax, big)));
    atomicMax(out + 1, __float_as_uint(mx_bf == mx_bf ? fminf(mx_bf, big) : big));
    atomicMax(out + 2, __float_as_uint(mx_fp == mx_fp ? fminf(mx_fp, big) : big));
  }
}

// In-place L2 normalisation of fp32 rows (x / |x|, zero rows stay zero): the database builder's
// `bases / bases.norm(dim=1, keepdim=True)` (src/main.py:465-466). One warp per row.
__global__ void k_normalize_rows(float* __restrict__ x, long long n, int d) {
  const int lane = threadIdx.x & 31;
  const long long warp0 = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  for (long long r = warp0; r < n; r += nwarps) {
    float* xr = x + r * d;
    float n2 = 0.f;
    for (int c = lane; c < d; c += 32) n2 = fmaf(xr[c], xr[c], n2);
    n2 = warp_sum(n2);
    const float nrm = sqrtf(n2);
    if (nrm > 0.f)
      for (int c = lane; c < d; c += 32) xr[c] = xr[c] / nrm;
  }
}

__global__ void k_fill_f32(float* p, long long n, float v) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

// ---------------------------------------------------------------------------------------------
// Candidate selection + fp32 re-rank + certificate. One block per (query, db).
//
// Let a(n) be the bf16-GEMM score, s(n) the exact one, |a - s| <= eps for every row (eps from
// Cauchy-Schwarz on the two rounding residuals + an fp32 accumulation allowance). With a_(k) the
// k-th largest approximate score, every true top-k row has a(n) >= a_(k) - 2 eps. So the set
// C = { n : a(n) >= tau }, tau = a_(k) - 2 eps, contains the exact answer provided no slice
// dropped a row scoring >= tau, i.e. every slice threshold theta < tau. If that (or |C| <= R_MAX)
// fails the query is queued for the exact fallback instead of being answered from C.
// ---------------------------------------------------------------------------------------------
// Neighbour consumer, run by the block that has just ranked query b of stream s (0 = image,
// 1 = text) while the neighbour rows are still hot in L1/L2:
//   feat[s][b][j][:] = rows_s[id[perm_s ? perm_s[j] : j]][:]                       (optional)
//   pool[s][b][:]    = sum_j w_j * rows_s[id[j]][:]                                (optional)
// w = 1/k (mode 1) or softmax_j(sign * tau * D[j]) (mode 2; sign = -1 under L2).
// Replaces the CPU index_select + randperm copy + H2D of src/trainer.py:214-230 and the attn@v
// shaped reduction of src/model/model.py:69-73.
struct ConsumeParams {
  int enabled;      // 0: plain search
  int mode;         // 0 no pool, 1 mean, 2 softmax
  int part4;        // float4 slots of shared scratch: warps per block * d / 4 (0 when d % 4 != 0)
  float tau;
  const int* perm[2];
  float* feat[2];   // [nq][k][d]
  float* pool[2];   // [nq][d]
  // Host mirror of the result rows ([nq][k] each, page-locked host memory addressed through its
  // device mapping, nullable): the block that has a query's final row stores it there as well, so
  // the (D, I) the reference reads on the host need no copy behind the search.
  float* host_D[2];
  long long* host_I[2];
};

// One query's final row to the host mirror (called by every thread of the block, row complete in
// shared memory). Posted writes: they are on their way while the block goes on to the consumer.
__device__ __forceinline__ void mirror_row_to_host(const ConsumeParams& c, int s, long long q, int k,
                                                   const unsigned int* top_id, const float* top_d,
                                                   long long id_offset, int metric) {
  float* Dh = c.host_D[s] + q * k;
  long long* Ih = c.host_I[s] + q * k;
  for (int j = threadIdx.x; j < k; j += blockDim.x) {
    const unsigned int id = top_id[j];
    const bool pad = id == 0xFFFFFFFFu;
    Dh[j] = pad ? (metric == METRIC_L2 ? FLT_MAX : -FLT_MAX) : top_d[j];
    Ih[j] = pad ? -1ll : static_cast<long long>(id) + id_offset;
  }
}

// Row-sharded exchange fused into the search (p2p_exchange.cuh): the block that has ranked query b
// of database s also stores that [k] result row into every peer's receive buffer (NVLink P2P
// stores), and the last block of the search's last kernel publishes the epoch flag. n == 0: off.
struct PeerOut {
  int n, my_rank;
  int publish;                          // this launch is the last writer of the step: publish the flags
  unsigned int epoch;
  float* D[P2P_MAX_RANKS];              // where THIS rank's [nq][k] score block of database 0 lives in rank r's buffer
  long long* I[P2P_MAX_RANKS];          // ... and its label block
  long long db_stride;                  // database 1's blocks follow at D[r] + db_stride, I[r] + db_stride
  unsigned int* flag[P2P_MAX_RANKS];    // "rank my_rank has delivered `epoch`" word in rank r's buffer
  unsigned int* ticket;                 // local counter for "last block publishes" (zero between launches)
};

// Store one query's final row of database s to the peers. top_id: local row ids in rank order
// (0xFFFFFFFF = padding); called by every thread of the block after the row is complete in shared memory.
__device__ __forceinline__ void push_row_to_peers(const PeerOut& po, int s, long long q, int k,
                                                  const unsigned int* top_id, const float* top_d,
                                                  long long id_offset, int metric) {
  for (int r = 0; r < po.n; ++r) {
    if (r == po.my_rank) continue;
    float* Dr = po.D[r] + s * po.db_stride + q * k;
    long long* Ir = po.I[r] + s * po.db_stride + q * k;
    for (int j = threadIdx.x; j < k; j += blockDim.x) {
      const unsigned int id = top_id[j];
      const bool pad = id == 0xFFFFFFFFu;
      Dr[j] = pad ? (metric == METRIC_L2 ? FLT_MAX : -FLT_MAX) : top_d[j];
      Ir[j] = pad ? -1ll : static_cast<long long>(id) + id_offset;
    }
  }
  __threadfence_system();  // ordered before the flag a later block publishes with release.sys
}

// Where the consumer finds neighbour row `id` (the id top_id holds). LocalRows: the search's own
// database, row id of a [n][d] matrix. The sharded consumer (k_shard_consume) addresses rows that
// live on several GPUs through a per-query table of row pointers instead.
struct LocalRows {
  const float* __restrict__ base;
  int d;
  __device__ __forceinline__ const float* operator()(unsigned int id) const {
    return base + static_cast<long long>(id) * d;
  }
  __device__ __forceinline__ uintptr_t align_bits() const { return reinterpret_cast<uintptr_t>(base); }
};

// top_id: row ids in rank order (0xFFFFFFFF = padding) as `rows` resolves them, top_d: their D values.
// NIF = neighbour rows in flight per warp (2 for latency, 1 where registers are scarce).
template <int NIF, class Rows>
__device__ __forceinline__ void consume_query(const ConsumeParams& c, const Rows& rows,
                                              int s, long long b, int k, int d, int metric,
                                              const unsigned int* top_id, const float* top_d,
                                              float* w, float4* part) {
  const int tid = threadIdx.x;
  float* pool = c.mode != 0 ? c.pool[s] : nullptr;
  float* feat = c.feat[s] ? c.feat[s] + b * k * d : nullptr;
  if (pool == nullptr && feat == nullptr) return;
  // the permutation entries of this warp's first neighbours: fetched before the weights so that
  // the global load overlaps them
  const int* perm = c.perm[s];
  int jr_first[NIF];
#pragma unroll
  for (int t = 0; t < NIF; ++t) {
    const int jo = (tid >> 5) * NIF + t;
    jr_first[t] = jo < k ? (perm ? perm[jo] : jo) : 0;
    if (static_cast<unsigned int>(jr_first[t]) >= static_cast<unsigned int>(k)) jr_first[t] = -1;  // bad perm entry: zero row
  }
  if (tid < 32) {
    // weights by one warp (k is small: 16 in KEDs)
    if (pool != nullptr && c.mode == 2) {
      const float sign = metric == METRIC_L2 ? -1.f : 1.f;
      float mx = -INFINITY;
      for (int j = tid; j < k; j += 32)
        if (top_id[j] != 0xFFFFFFFFu) mx = fmaxf(mx, sign * c.tau * top_d[j]);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      float sum = 0.f;
      for (int j = tid; j < k; j += 32) {
        const float e = top_id[j] != 0xFFFFFFFFu ? __expf(sign * c.tau * top_d[j] - mx) : 0.f;
        w[j] = e;
        sum += e;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
      const float inv = sum > 0.f ? 1.f / sum : 0.f;
      for (int j = tid; j < k; j += 32) w[j] *= inv;
    } else {
      for (int j = tid; j < k; j += 32) w[j] = 1.f / static_cast<float>(k);
    }
  }
  __syncthreads();
  const bool vec = c.part4 > 0 && ((rows.align_bits() | reinterpret_cast<uintptr_t>(c.feat[s]) |
                                    reinterpret_cast<uintptr_t>(c.pool[s])) & 15) == 0;
  if (vec) {
    // One warp per neighbour row, two neighbours per warp in flight: every lane issues all its
    // 16-byte loads of both rows before the first store, so the whole gather of a query costs
    // about one memory round trip. Each warp keeps the weighted sum of its own neighbours; the
    // per-warp partial pools meet in shared memory (part: [warps][d/4]).
    const int d4 = d >> 2;
    const int lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    constexpr int U = 6;  // float4 per lane per pass: d = 768 is one pass
    for (int cb = 0; cb < d4; cb += 32 * U) {
      float4 acc[U];
#pragma unroll
      for (int u = 0; u < U; ++u) acc[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int jo0 = warp * NIF; jo0 < k; jo0 += nwarps * NIF) {
        float4 v[NIF][U];
        unsigned int idv[NIF];
        int jr[NIF];
#pragma unroll
        for (int t = 0; t < NIF; ++t) {
          const int jo = jo0 + t;
          // output slot jo shows rank jr
          jr[t] = jo0 == warp * NIF ? jr_first[t] : (jo < k ? (perm ? perm[jo] : jo) : 0);
          const bool jr_ok = static_cast<unsigned int>(jr[t]) < static_cast<unsigned int>(k);
          if (!jr_ok) jr[t] = 0;
          idv[t] = (jo < k && jr_ok) ? top_id[jr[t]] : 0xFFFFFFFFu;
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int col = cb + u * 32 + lane;
            v[t][u] = (idv[t] != 0xFFFFFFFFu && col < d4)
                          ? __ldg(reinterpret_cast<const float4*>(rows(idv[t])) + col)
                          : make_float4(0.f, 0.f, 0.f, 0.f);
          }
        }
#pragma unroll
        for (int t = 0; t < NIF; ++t) {
          const int jo = jo0 + t;
          if (jo >= k) continue;
          const float wj = w[jr[t]];
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int col = cb + u * 32 + lane;
            if (col < d4) {
              if (feat) reinterpret_cast<float4*>(feat + static_cast<long long>(jo) * d)[col] = v[t][u];
              acc[u].x = fmaf(wj, v[t][u].x, acc[u].x);
              acc[u].y = fmaf(wj, v[t][u].y, acc[u].y);
              acc[u].z = fmaf(wj, v[t][u].z, acc[u].z);
              acc[u].w = fmaf(wj, v[t][u].w, acc[u].w);
            }
          }
        }
      }
      if (pool) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int col = cb + u * 32 + lane;
          if (col < d4) part[warp * d4 + col] = acc[u];
        }
      }
    }
    if (pool) {
      __syncthreads();
      for (int col = tid; col < d4; col += blockDim.x) {
        float4 acc = part[col];
#pragma unroll 8
        for (int gg = 1; gg < nwarps; ++gg) {
          const float4 o = part[gg * d4 + col];
          acc.x += o.x; acc.y += o.y; acc.z += o.z; acc.w += o.w;
        }
        reinterpret_cast<float4*>(pool + b * d)[col] = acc;
      }
    }
  } else {
    for (int col = tid; col < d; col += blockDim.x) {
      float acc = 0.f;
      for (int jo = 0; jo < k; ++jo) {
        int j = perm ? perm[jo] : jo;
        const bool j_ok = static_cast<unsigned int>(j) < static_cast<unsigned int>(k);
        if (!j_ok) j = 0;
        const unsigned int id = j_ok ? top_id[j] : 0xFFFFFFFFu;
        const float v = id != 0xFFFFFFFFu ? rows(id)[col] : 0.f;
        if (feat) feat[static_cast<long long>(jo) * d + col] = v;
        acc = fmaf(w[j], v, acc);
      }
      if (pool) pool[b * d + col] = acc;
    }
  }
}


__device__ __forceinline__ float block_max_f(float v, float* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float r = red[0];
  for (int w = 1; w < (blockDim.x >> 5); ++w) r = fmaxf(r, red[w]);
  __syncthreads();
  return r;
}

// Radix-select step: given a 256-bin histogram, find the bin b with
//   count(bins > b) < need <= count(bins >= b)
// and publish bcast[0] = b, bcast[1] = need - count(bins > b). Warp 0 does the work (lane l owns
// bins 8l .. 8l+7), so any block size works; uniform call; ends with a __syncthreads so every
// thread may read bcast.
__device__ __forceinline__ void block_find_bin(const unsigned int* hist, int need, unsigned int* bcast) {
  if (threadIdx.x < 32) {
    const int lane = threadIdx.x;
    unsigned int h[8], tot = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      h[i] = hist[lane * 8 + i];
      tot += h[i];
    }
    unsigned int suf = tot;  // inclusive suffix sum over lanes: bins 8*lane .. 255
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned int up = __shfl_down_sync(0xffffffffu, suf, o);
      if (lane + o < 32) suf += up;
    }
    unsigned int above = suf - tot;  // count of bins owned by higher lanes
#pragma unroll
    for (int i = 7; i >= 0; --i) {
      const unsigned int incl = above + h[i];
      if (static_cast<int>(above) < need && static_cast<int>(incl) >= need) {
        bcast[0] = static_cast<unsigned int>(lane * 8 + i);
        bcast[1] = static_cast<unsigned int>(need) - above;
      }
      above = incl;
    }
  }
  __syncthreads();
}

// k-th largest of keys[0..n) (1 <= k <= n), 4 x 8-bit radix passes with a shared histogram.
__device__ unsigned int block_kth_largest(const unsigned int* keys, int n, int k,
                                          unsigned int* hist /*256*/, unsigned int* bcast /*2*/) {
  unsigned int prefix = 0, mask = 0;
  int need = k;
  for (int shift = 24; shift >= 0; shift -= 8) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    // Scores of one query share their leading bytes, so in the first two passes a whole warp lands
    // in ONE or two bins: lanes with the same bin elect a leader that adds their count (one
    // shared-memory atomic per distinct bin and warp instead of 32 serialised ones on one address).
    // The low bytes spread over the bins; there plain atomics are cheaper than the matching loop.
    if (shift >= 16) {
      for (int i0 = 0; i0 < n; i0 += blockDim.x) {
        const int i = i0 + static_cast<int>(threadIdx.x);
        const unsigned int key = i < n ? keys[i] : 0u;
        const bool live = i < n && (key & mask) == prefix;
        const unsigned int bin = live ? ((key >> shift) & 255u) : 256u;
        const unsigned int peers = __match_any_sync(0xffffffffu, bin);
        if (live && (threadIdx.x & 31) == static_cast<unsigned int>(__ffs(peers) - 1)) atomicAdd(&hist[bin], __popc(peers));
      }
    } else {
      for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const unsigned int key = keys[i];
        if ((key & mask) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1u);
      }
    }
    __syncthreads();
    block_find_bin(hist, need, bcast);
    prefix |= bcast[0] << shift;
    mask |= 255u << shift;
    need = static_cast<int>(bcast[1]);
    __syncthreads();
  }
  return prefix;
}

}  // namespace keds

#include "rerank.cuh"

namespace keds {

__global__ void k_flag_all(int* flagged, int* n_flagged, int nq) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nq) flagged[i] = i;
  if (i == 0) *n_flagged = nq;
}

}  // namespace keds

#include "exact_fallback.cuh"
#include "label_hits.cuh"
#include "p2p_exchange.cuh"

namespace keds {

// ---------------------------------------------------------------------------------------------
// Merge `parts` per-shard results (part p at Dp + p*stride_d, Ip + p*stride_i, each [nq][k]) into the global top-k (same total order; ids are
// already global, every part is sorted best-first the way a search returns it). One block per query.
// Used behind the exchange of a row-sharded search.
// With `flags` set (peer-memory exchange, p2p_exchange.cuh) each block first waits until every
// peer has delivered its part for this `epoch`; Dp/Ip must not be __restrict__/read-only cached.
struct MergeWait {
  const unsigned int* flags;  // nullptr: parts are already complete (NCCL path)
  int my_rank;
  unsigned int epoch;
  unsigned int* err_word;
  unsigned long long* stats;  // nullable: {sum, max, count} of block 0's wait for the peers, ns (rank skew)
};

__global__ void k_topk_merge(const float* Dp, const long long* Ip,
                             long long stride_d, long long stride_i, int parts, long long nq, int k,
                             int metric, float* __restrict__ D, long long* __restrict__ I,
                             const MergeWait mw) {
  // Every part is a search result: sorted by (score desc, label asc), valid entries first, labels
  // distinct across parts. The global rank of an entry is its position in its own part plus, for
  // every other part, the number of entries there that precede it -- found by binary search
  // (parts * log2 k steps per entry). The all-pairs count this replaces was quadratic in parts * k:
  // 512^2 per query at 8 shards x k = 64, ~150 us, i.e. the whole "exchange cost" of round 1.
  extern __shared__ uint8_t mg_smem[];
  long long* idv = reinterpret_cast<long long*>(mg_smem);     // parts*k
  float* val = reinterpret_cast<float*>(idv + parts * k);     // parts*k rank scores (IP, or -distance)
  __shared__ int nvalid;
  const long long q = blockIdx.x;
  const int tot = parts * k;
  if (threadIdx.x == 0) nvalid = 0;
  griddep_wait();
  if (mw.flags != nullptr) {
    if (threadIdx.x == 0) {
      const unsigned long long t0 = global_timer_ns();
      p2p_wait_flags(mw.flags, parts, mw.my_rank, mw.epoch, mw.err_word);
      if (mw.stats != nullptr && blockIdx.x == 0) {
        const unsigned long long dt = global_timer_ns() - t0;
        atomicAdd(mw.stats, dt);
        atomicMax(mw.stats + 1, dt);
        atomicAdd(mw.stats + 2, 1ull);
      }
    }
    __syncthreads();
  }
  int mine = 0;
  for (int i = threadIdx.x; i < tot; i += blockDim.x) {
    const int pt = i / k, j = i % k;
    const long long src = q * k + j;
    const float v = Dp[pt * stride_d + src];
    const long long id = Ip[pt * stride_i + src];
    val[i] = metric == METRIC_L2 ? -v : v;
    idv[i] = id;
    mine += id >= 0;
  }
  atomicAdd(&nvalid, mine);
  __syncthreads();
  for (int i = threadIdx.x; i < tot; i += blockDim.x) {
    const long long idi = idv[i];
    if (idi < 0) continue;
    const float vi = val[i];
    const int pt = i / k;
    int rank = i - pt * k;  // its own part is sorted and holds its valid entries first
    for (int p2 = 0; p2 < parts; ++p2) {
      if (p2 == pt) continue;
      const float* v2 = val + p2 * k;
      const long long* i2 = idv + p2 * k;
      int lo = 0, hi = k;  // entries [0, lo) of part p2 precede this one
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const long long idm = i2[mid];
        const float vm = v2[mid];
        const bool before = idm >= 0 && (vm > vi || (vm == vi && idm < idi));
        if (before) lo = mid + 1; else hi = mid;
      }
      rank += lo;
    }
    if (rank < k) {
      D[q * k + rank] = metric == METRIC_L2 ? -vi : vi;
      I[q * k + rank] = idi;
    }
  }
  // padding when fewer than k valid entries exist
  for (int r = nvalid + threadIdx.x; r < k; r += blockDim.x) {
    D[q * k + r] = metric == METRIC_L2 ? FLT_MAX : -FLT_MAX;
    I[q * k + r] = -1;
  }
}

// ---------------------------------------------------------------------------------------------
// Neighbour gather (+ optional column permutation) and weighted pool.
//   gather: out[b][j][:] = base[I[b][perm ? perm[j] : j]][:]              (W == nullptr)
//   pool:   out[b][h][:] = sum_j W[b][h][j] * base[I[b][j]][:]
// Replaces the CPU index_select + randperm copy + H2D of src/trainer.py:214-230 and the attn@v
// shaped reduction of src/model/model.py:69-73. Rows with id < 0 or id >= n_base, and slots whose
// perm entry is outside [0, k), read as zeros.
__global__ void k_gather_rows(const float* __restrict__ base, long long n_base, const long long* __restrict__ I,
                              const int* __restrict__ perm, long long B, int k, int d,
                              float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const long long w = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  if (w >= B * k) return;
  const long long b = w / k;
  const int j = static_cast<int>(w % k);
  const int pj = perm ? perm[j] : j;
  long long id = static_cast<unsigned int>(pj) < static_cast<unsigned int>(k) ? I[b * k + pj] : -1;
  if (id >= n_base) id = -1;
  float* o = out + w * d;
  if ((d & 3) == 0 && ((reinterpret_cast<uintptr_t>(base) | reinterpret_cast<uintptr_t>(out)) & 15) == 0) {
    const float4* s4 = reinterpret_cast<const float4*>(base + (id < 0 ? 0 : id) * d);
    float4* o4 = reinterpret_cast<float4*>(o);
    for (int c = lane; c < (d >> 2); c += 32)
      o4[c] = id < 0 ? make_float4(0.f, 0.f, 0.f, 0.f) : __ldg(s4 + c);
  } else {
    for (int c = lane; c < d; c += 32) o[c] = id < 0 ? 0.f : base[id * d + c];
  }
}

// The neighbour consumer's MLP input in one launch: rows [queries | image neighbours | text
// neighbours] = [B | B k | B k] x d (src/trainer.py:59-65 feeds the same three blocks through
// IM2TEXT). One warp per row; image neighbours follow the shared permutation; `rows` resolves a
// neighbour id of either stream to its row, or to nullptr (a zero row): ConsumerLocalRows for bases
// resident on this GPU, ConsumerShardRows (p2p_exchange.cuh) for row-sharded bases.
struct ConsumerLocalRows {
  const float* __restrict__ base_img;
  long long n_img;
  const float* __restrict__ base_txt;
  long long n_txt;
  __device__ __forceinline__ const float* operator()(bool img, long long id, int d) const {
    return id >= 0 && id < (img ? n_img : n_txt) ? (img ? base_img : base_txt) + id * d : nullptr;
  }
};

template <class Rows>
__global__ void k_consumer_rows(const float* __restrict__ q, const Rows rows,
                                const long long* __restrict__ I_img, const long long* __restrict__ I_txt,
                                const int* __restrict__ perm, long long B, int k, int d, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const long long w = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const long long Bk = B * k;
  if (w >= B + 2 * Bk) return;
  const float* src = nullptr;   // nullptr: zero row
  if (w < B) {
    src = q + w * d;
  } else {
    const bool img = w < B + Bk;
    const long long r = img ? w - B : w - B - Bk;
    const long long b = r / k;
    const int j = static_cast<int>(r % k);
    const int pj = (img && perm) ? perm[j] : j;
    const long long id = static_cast<unsigned int>(pj) < static_cast<unsigned int>(k) ? (img ? I_img : I_txt)[b * k + pj] : -1;
    src = rows(img, id, d);
  }
  float* o = out + w * d;
  if ((d & 3) == 0 && src != nullptr && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(o)) & 15) == 0) {
    const float4* s4 = reinterpret_cast<const float4*>(src);
    float4* o4 = reinterpret_cast<float4*>(o);
    for (int c = lane; c < (d >> 2); c += 32) o4[c] = __ldg(s4 + c);
  } else {
    for (int c = lane; c < d; c += 32) o[c] = src != nullptr ? src[c] : 0.f;
  }
}

__global__ void k_weighted_pool(const float* __restrict__ base, long long n_base, const long long* __restrict__ I,
                                const float* __restrict__ W, long long B, int k, int H, int d,
                                float* __restrict__ out) {
  extern __shared__ uint8_t pl_smem[];
  long long* ids = reinterpret_cast<long long*>(pl_smem);  // k
  float* w = reinterpret_cast<float*>(ids + k);            // H*k
  const long long b = blockIdx.x;
  for (int j = threadIdx.x; j < k; j += blockDim.x) ids[j] = I[b * k + j];
  for (int i = threadIdx.x; i < H * k; i += blockDim.x) w[i] = W[b * H * k + i];
  __syncthreads();
  for (int h = 0; h < H; ++h) {
    for (int c = threadIdx.x; c < d; c += blockDim.x) {
      float acc = 0.f;
      for (int j = 0; j < k; ++j) {
        const long long id = ids[j];
        if (id >= 0 && id < n_base) acc = fmaf(w[h * k + j], __ldg(base + id * d + c), acc);
      }
      out[(b * H + h) * d + c] = acc;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Gallery ranking by counting (no sort): rank[q] = number of gallery rows, other than the target
// and the optional excluded row, that beat the target under (score desc, id asc).
// Covers the argsort-then-find of src/eval_utils.py:1008-1067 (COCO / FashionIQ / CIRR).
// With `qlist` (device list of query ids, *n_list entries) only those queries are ranked: the
// exact recount behind the tensor-core ranking; blocks past the end of the list leave at once.
__global__ void __launch_bounds__(256)
k_gallery_rank(const float* __restrict__ Q, long long nq, const float* __restrict__ G, long long ng,
               int d, const long long* __restrict__ target, const long long* __restrict__ exclude,
               long long* __restrict__ rank_out, const int* __restrict__ qlist, const int* __restrict__ n_list) {
  // GR_Q queries per block share every gallery row a warp reads (the row is fetched once for
  // all of them); per (query,row) the arithmetic is that of warp_exact_score.
  constexpr int GR_Q = 8;
  extern __shared__ uint8_t gr_smem[];
  const int dq = (d + 3) & ~3;
  float* qv = reinterpret_cast<float*>(gr_smem);  // [GR_Q][dq]
  __shared__ int total[GR_Q];
  __shared__ float s_target[GR_Q];
  __shared__ long long qid[GR_Q];
  griddep_wait();
  if (n_list != nullptr) nq = *n_list;
  const long long q0 = static_cast<long long>(blockIdx.x) * GR_Q;
  if (q0 >= nq) return;
  const int nqb = static_cast<int>(min(static_cast<long long>(GR_Q), nq - q0));
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  if (threadIdx.x < GR_Q) {
    total[threadIdx.x] = 0;
    qid[threadIdx.x] = static_cast<int>(threadIdx.x) < nqb ? (qlist != nullptr ? qlist[q0 + threadIdx.x] : q0 + threadIdx.x) : 0;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < GR_Q * dq; i += blockDim.x) {
    const int qi = i / dq, c = i % dq;
    qv[i] = (qi < nqb && c < d) ? Q[qid[qi] * d + c] : 0.f;
  }
  __syncthreads();
  for (int qi = warp; qi < nqb; qi += nw) {
    const float st = warp_exact_score(qv + qi * dq, G + target[qid[qi]] * d, d, METRIC_IP, lane);
    if (lane == 0) s_target[qi] = st;
  }
  __syncthreads();
  long long tg[GR_Q], ex[GR_Q];
  float st[GR_Q];
  int cnt[GR_Q];
#pragma unroll
  for (int i = 0; i < GR_Q; ++i) {
    tg[i] = i < nqb ? target[qid[i]] : -1;
    ex[i] = (i < nqb && exclude) ? exclude[qid[i]] : -1;
    st[i] = i < nqb ? s_target[i] : 0.f;
    cnt[i] = 0;
  }
  const bool vec = (d & 3) == 0 && (reinterpret_cast<uintptr_t>(G) & 15) == 0;
  for (long long g = warp; g < ng; g += nw) {
    const float* xr = G + g * d;
    float acc[GR_Q];
#pragma unroll
    for (int i = 0; i < GR_Q; ++i) acc[i] = 0.f;
    if (vec) {
      const float4* x4 = reinterpret_cast<const float4*>(xr);
      const int d4 = d >> 2;
      for (int c = lane; c < d4; c += 32) {
        const float4 a = __ldg(x4 + c);
#pragma unroll
        for (int i = 0; i < GR_Q; ++i) {
          const float4 b = reinterpret_cast<const float4*>(qv + i * dq)[c];
          acc[i] = fmaf(a.x, b.x, acc[i]);
          acc[i] = fmaf(a.y, b.y, acc[i]);
          acc[i] = fmaf(a.z, b.z, acc[i]);
          acc[i] = fmaf(a.w, b.w, acc[i]);
        }
      }
    } else {
      for (int c = lane; c < d; c += 32) {
        const float a = __ldg(xr + c);
#pragma unroll
        for (int i = 0; i < GR_Q; ++i) acc[i] = fmaf(a, qv[i * dq + c], acc[i]);
      }
    }
#pragma unroll
    for (int i = 0; i < GR_Q; ++i) {
      const float s = warp_sum(acc[i]);
      if (i < nqb && g != tg[i] && g != ex[i]) cnt[i] += (s > st[i]) || (s == st[i] && g < tg[i]);
    }
  }
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < GR_Q; ++i)
      if (i < nqb) atomicAdd(&total[i], cnt[i]);
  }
  __syncthreads();
  if (threadIdx.x < nqb) rank_out[qid[threadIdx.x]] = total[threadIdx.x];
}

// ---------------------------------------------------------------------------------------------
// Gallery ranking on the tensor cores (k_score_topk<*, true>), the two kernels around it.
//
// k_rank_targets: per query (one warp) the exact fp32 score of its target row and the error band
// around it in approximate-score space: a row with a > s_t + eps beats the target for certain
// (its exact score is at least a - eps), a row with a < s_t - eps loses for certain, the rows in
// between are listed and settled exactly by k_rank_finish. eps as in the search certificate.
__global__ void k_rank_targets(const float* __restrict__ Q, long long nq, const float* __restrict__ G, int d,
                               const long long* __restrict__ target, const long long* __restrict__ exclude,
                               const float4* __restrict__ qstat, const unsigned int* __restrict__ dbstat,
                               float eps_scale, float* __restrict__ s_t, float* __restrict__ lo,
                               float* __restrict__ hi, int* __restrict__ t32, int* __restrict__ e32) {
  const int lane = threadIdx.x & 31;
  const long long q = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  griddep_wait();  // qstat comes from k_prep_rows
  if (q >= nq) return;
  const long long t = target[q];
  const float st = warp_exact_score(Q + q * d, G + t * d, d, METRIC_IP, lane);
  if (lane == 0) {
    const float4 qs = qstat[q];
    const float xb = __uint_as_float(dbstat[0]), xd = __uint_as_float(dbstat[1]);
    const int d_pad = (d + BK - 1) / BK * BK;
    float eps = qs.z * xb + sqrtf(qs.x) * xd + (static_cast<float>(d_pad) * 2.4e-7f) * qs.y * xb;
    eps *= 1.0001f * eps_scale;
    if (!(eps == eps)) eps = INFINITY;
    s_t[q] = st;
    lo[q] = st - eps;
    hi[q] = st + eps;
    t32[q] = static_cast<int>(t);
    e32[q] = exclude != nullptr ? static_cast<int>(exclude[q]) : -1;
  }
}

// k_rank_finish: one warp per query. rank = sum over the candidate lists of the certain counts +
// the band rows that beat the target under the exact rule (fp32 score, then lower row id). A list
// that overflowed queues the query for the exact recount (k_gallery_rank over the queue).
__global__ void k_rank_finish(const float* __restrict__ Q, long long nq, const float* __restrict__ G, int d,
                              int n_lists, int n_qt, const uint2* __restrict__ cand,
                              const int* __restrict__ cand_cnt, const float* __restrict__ cand_beats,
                              const float* __restrict__ s_t, const int* __restrict__ t32,
                              long long* __restrict__ rank_out, int* __restrict__ queue, int* __restrict__ n_queue) {
  const int lane = threadIdx.x & 31;
  const long long q = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  griddep_wait();
  if (q >= nq) return;
  const int qt = static_cast<int>(q / BM), ql = static_cast<int>(q % BM);
  const float st = s_t[q];
  const int t = t32[q];
  int beats = 0;
  bool over = false;
  // certain counts: lanes stride the lists
  for (int s = lane; s < n_lists; s += 32) {
    const long long item = static_cast<long long>(s) * n_qt + qt;
    const int c = cand_cnt[item * BM + ql];
    over = over || c < 0;
    beats += __float_as_int(cand_beats[item * BM + ql]);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) beats += __shfl_xor_sync(0xffffffffu, beats, o);
  over = __any_sync(0xffffffffu, over);
  if (over) {
    if (lane == 0) queue[atomicAdd(n_queue, 1)] = static_cast<int>(q);
    return;
  }
  // band rows: exact score, exact rule
  for (int s = 0; s < n_lists; ++s) {
    const long long item = static_cast<long long>(s) * n_qt + qt;
    const int c = cand_cnt[item * BM + ql];
    for (int e = 0; e < c; ++e) {
      const uint2 en = cand[(item * BM + ql) * LKEEP + e];
      const int g = static_cast<int>(en.y);
      const float sg = warp_exact_score(Q + q * d, G + static_cast<long long>(g) * d, d, METRIC_IP, lane);
      beats += (sg > st) || (sg == st && g < t);
    }
  }
  if (lane == 0) rank_out[q] = beats;
}

// hits[q][i] = #{ j < ks[i] : labels[I[q][j]] == qlabel[q] }   (ImageNet-domain R@k / P@k,
// src/eval_utils.py:1107-1118 without the [100 x G] scatter masks)
__global__ void k_label_hits(const long long* __restrict__ I, long long nq, int kmax,
                             const long long* __restrict__ labels, const long long* __restrict__ qlabel,
                             const int* __restrict__ ks, int nks, int* __restrict__ hits) {
  const long long q = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  const long long ql = qlabel[q];
  int acc = 0, ki = 0;
  for (int j = 0; j < kmax && ki < nks; ++j) {
    const long long id = I[q * kmax + j];
    acc += (id >= 0 && labels[id] == ql);
    while (ki < nks && j + 1 == ks[ki]) hits[q * nks + ki++] = acc;
  }
  while (ki < nks) hits[q * nks + ki++] = acc;
}

}  // namespace keds
