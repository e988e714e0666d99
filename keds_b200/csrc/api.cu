// C ABI of libkeds_knn.so (see include/keds_knn.h). Host orchestration only: planning, buffers,
// TMA descriptors, launches. All arithmetic is in the kernels of score_topk_sm100.cuh and
// aux_kernels.cuh. There is no CPU path: without a CUDA device every compute call fails.
#include "../../include/keds_knn.h"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "aux_kernels.cuh"
#include "range_search.cuh"

using namespace keds;

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

#define CK(call)                                                                         \
  do {                                                                                   \
    cudaError_t e_ = (call);                                                             \
    if (e_ != cudaSuccess)                                                               \
      return fail(e_ == cudaErrorMemoryAllocation ? KEDS_ERR_OOM : KEDS_ERR_CUDA,        \
                  "%s failed: %s (%d) at %s:%d", #call, cudaGetErrorString(e_), (int)e_, \
                  __FILE__, __LINE__);                                                   \
  } while (0)

#define CKS(call)          \
  do {                     \
    int s_ = (call);       \
    if (s_ != 0) return s_; \
  } while (0)

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  // Bumped whenever the buffer moves: a CUDA graph captured over a handle bakes these addresses in,
  // and its owner compares keds_index_generation() before every replay (RetrievalStep.run()).
  uint64_t* gen = nullptr;
  bool borrowed = false;  // p points into memory owned by the caller (bound training parameters): never freed here
  void moved() {
    if (gen) ++*gen;
  }
  // view of caller-owned memory (replaces whatever was held)
  void borrow(void* ptr, size_t bytes) {
    release();
    p = ptr;
    cap = bytes;
    borrowed = true;
  }
  // grow without keeping contents
  int ensure(size_t bytes) {
    if (bytes <= cap && !borrowed) return 0;
    if (borrowed) {
      p = nullptr;
      cap = 0;
      borrowed = false;
    }
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    moved();
    CK(cudaMalloc(&p, bytes));
    cap = bytes;
    return 0;
  }
  // grow keeping the first `keep` bytes
  int grow_keep(size_t bytes, size_t keep) {
    if (bytes <= cap) return 0;
    void* np = nullptr;
    CK(cudaMalloc(&np, bytes));
    if (p && keep) CK(cudaMemcpy(np, p, keep, cudaMemcpyDeviceToDevice));
    if (p) cudaFree(p);
    p = np;
    cap = bytes;
    moved();
    return 0;
  }
  void release() {
    if (p && !borrowed) {
      cudaFree(p);
      moved();
    }
    p = nullptr;
    cap = 0;
    borrowed = false;
  }
  template <class T>
  T* as() const { return static_cast<T*>(p); }
};

// page-locked host staging (the numpy-in / numpy-out path: one DMA each way instead of the driver's
// pageable-memory staging, and no extra blocking copy for the status words)
struct HostBuf {
  void* p = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes) {
    if (bytes <= cap) return 0;
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    CK(cudaHostAlloc(&p, bytes, cudaHostAllocDefault));
    cap = bytes;
    return 0;
  }
  void release() {
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
  }
};

struct DeviceGuard {
  int prev = -1;
  bool ok = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess && cudaSetDevice(dev) == cudaSuccess) ok = true;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* sym = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) !=
          cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(sym);
  return fn;
}

// 16-bit [rows][d_pad] row-major -> boxes of {BK columns x box_rows rows}, 128-byte swizzle,
// out-of-range rows read as zeros.
int encode_rows_map(CUtensorMap* tm, const void* base, int64_t rows, int d_pad, int box_rows, int fmt) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return fail(KEDS_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(d_pad), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstr[1] = {static_cast<cuuint64_t>(d_pad) * 2};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(BK), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(tm, fmt == FMT_FP16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                  const_cast<void*>(base), gdim, gstr, box,
                  estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(KEDS_ERR_CUDA, "cuTensorMapEncodeTiled failed: CUresult %d", (int)r);
  return 0;
}

// Where a caller's pointer lives: the device that owns it (-1: not device or managed memory) and,
// for page-locked host memory, its device alias (kernels read and write it through the mapping).
// Converts to true for device memory.
struct PtrLoc {
  int device = -1;
  void* mapped = nullptr;
  explicit operator bool() const { return device >= 0; }
};

PtrLoc locate(const void* p) {
  PtrLoc l;
  cudaPointerAttributes a;
  if (!p) return l;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return l;
  }
  if (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) l.device = a.device;
  if (a.type == cudaMemoryTypeHost) l.mapped = a.devicePointer;
  return l;
}

// [0],[1] n_flagged per db, [2] err word, [3] spare, [4..5] range search: candidates found (64 bit),
// [6] largest candidate band |C| of the search (planner feedback), [7] spare
constexpr int CTRL_WORDS = 8;
constexpr int CTRL_RANGE = 4;
constexpr int CTRL_BAND = 6;
// One block of status words per pass of a multi-pass call, so that no pass has to be read back
// before the next one starts. Behind the status words: the exact fallback's work counters, one set
// of four words per launch of that kernel (k_prep_rows zeroes the whole block, so the launches of a
// search need no memset between them).
constexpr int EXACT_CTR_SETS = 64;
constexpr int CTRL_STRIDE = CTRL_WORDS + 4 * EXACT_CTR_SETS;
constexpr int S_MAX = 192;
constexpr size_t CAND_BUDGET = size_t(1) << 30;
constexpr int64_t Q_PASS_MAX = 16384;
constexpr size_t TIMING_RING = 8192;
constexpr size_t TIMING_PAIRS = 5;  // k_prep_rows, k_score_topk, k_select_rerank, k_exact_fallback, (reserved)

// keds_index_label_hits: the search chain with the hit-counting kernel in the re-rank's place
struct HitsMode {
  int nks;
  int ks[HITS_MAX_CUTS];
  const long long* row_labels;
  const long long* qlabel;  // [nq]
  int* hits;                // [nq][nks]
};

// keds_index_rank: the scoring kernel counts the rows that beat each query's target (k_rank_targets
// before it, k_rank_finish and the exact recount after it) instead of collecting the top-k
struct RankMode {
  const long long* target;   // [nq]
  const long long* exclude;  // [nq] or nullptr
  long long* out;            // [nq] ranks
};

// keds_index_range_search: the scoring kernel appends the rows inside each query's band, which are
// re-scored, kept when strictly inside the radius, and ordered per query (range_search.cuh)
struct RangeMode {
  float radius;
  long long* lims;  // [nq + 1] handle scratch; a pass writes its queries' entries and the one behind them
};

// How the scoring kernel covers nq queries: which kernel, its work units and query groups, and
// the most row slices the candidate budget holds.
struct Geometry {
  bool pair = false;  // CTA-pair scoring kernel (two query tiles per work item)
  int sub = 1;        // candidate lines per (slice, query): 2 in the pair kernel (one per column half)
  int n_qt = 1, n_qg = 1, units = 0;
  long long s_mem = 0;
};

struct Plan : Geometry {
  int exact_only = 0;
  int S = 1, n_items = 0, grid = 0;
  bool small_batch = true;  // one wave of re-rank blocks: the latency variant
  void set_slices(int n_db, int slices) {
    S = slices;
    n_items = n_db * n_qg * S;
    grid = std::min(n_items, units) * (pair ? 2 : 1);
  }
};

}  // namespace

struct keds_index {
  int d = 0, d_pad = 0, metric = 0, device = 0, num_sms = 0;
  int64_t n = 0;
  int64_t id_offset = 0;
  float eps_scale = 1.f;
  // 16-bit operand format of x_bf16 / q_bf16 (FMT_FP16 or FMT_BF16; the buffer names predate the
  // choice) and what it was chosen from: running maxima over every row added so far
  int fmt = FMT_FP16;
  int fmt_forced = -1;  // -1: automatic (KEDS_OPERAND / keds_index_set_operand_format override it)
  float amax = 0.f, res_bf16 = 0.f, res_fp16 = 0.f;
  uint64_t generation = 0;        // bumped when a buffer a captured graph may hold is reallocated
  unsigned int* h_feedback = nullptr;  // mapped host word: largest candidate band of a recent search
  DevBuf x_f32, x_bf16, bias, dbstat, probe;
  CUtensorMap tm_x;   // {64 x 256}-row boxes (one CTA per tile)
  CUtensorMap tm_xh;  // {64 x 128}-row boxes (CTA pair: half a tile each)
  bool tm_x_ok = false;
  bool use_pair = true;
  // per-call scratch (one search in flight per handle)
  DevBuf q_f32, q_bf16, qstat, cand, cand_cnt, cand_theta, flagged[2], ctrl, exact_scratch, rk, theta0;
  DevBuf ex_rows;  // search with exclusion: the staged local row ids [n_db][nq][n_ex] of the pass
  // range search: band thresholds, candidates, order keys (two halves), per-query counts and offsets,
  // read-back words, and the results of the last call (rg_total entries, valid until the next call)
  DevBuf rg_thr, rg_cand, rg_key, rg_qcnt, rg_off, rg_word, rg_lims, rg_D, rg_I;
  int64_t rg_total = 0;
  bool warm_start = true;  // lists start at a finished list's threshold (KEDS_NO_WARM_START=1: every list cold)
  DevBuf D_stage[2], I_stage[2];
  HostBuf h_q, h_out;  // pinned staging for host-pointer calls
  CUtensorMap tm_q;
  const void* tm_q_base = nullptr;
  int64_t tm_q_rows = 0;
  int tm_q_fmt = -1;
  keds_search_stats stats;
  bool attrs_set = false;
  bool use_pdl = true;
  unsigned int* ctrl_cur = nullptr;  // status block of the pass being launched
  int ctrl_passes = 1;             // status blocks the last call used (finish_sync reads them all)
  int ctrl_slot = 0;               // n_flagged slot of the blocks' first count (1: only the call's second database ran)
  int rerank_threads_large = 128;  // block size of the throughput re-rank variant (KEDS_RERANK_THREADS)
  int rerank_variant = 0;          // 0: by batch size; 1 / 2: force the latency / throughput variant
  // in-kernel timing of the scoring kernel (bench.py's roofline leg): {min start, max end} ns
  bool timing_on = false;
  DevBuf timing;
  size_t timing_launches = 0;
};

namespace {

int set_kernel_attrs(keds_index* ix) {
  if (ix->attrs_set) return 0;
  CK(cudaFuncSetAttribute(k_score_topk<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                          (int)SCORE_SMEM_BYTES));
  CK(cudaFuncSetAttribute(k_score_topk<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                          (int)SCORE_PAIR_SMEM_BYTES));
  CK(cudaFuncSetAttribute(k_score_topk<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                          (int)SCORE_SMEM_BYTES));

  CK(cudaFuncSetAttribute(k_score_topk<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                          (int)SCORE_PAIR_SMEM_BYTES));
  CK(cudaFuncSetAttribute(k_score_topk<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                          (int)SCORE_SMEM_BYTES));
  CK(cudaFuncSetAttribute(k_score_topk<true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                          (int)SCORE_PAIR_SMEM_BYTES));
  CK(cudaFuncSetAttribute(k_score_range<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                          (int)SCORE_SMEM_BYTES));
  CK(cudaFuncSetAttribute(k_score_range<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                          (int)SCORE_PAIR_SMEM_BYTES));
  const char* no_pair = getenv("KEDS_NO_PAIR");
  ix->use_pair = !(no_pair && no_pair[0] == '1');
  CK(cudaFuncSetAttribute(k_select_rerank<3, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  CK(cudaFuncSetAttribute(k_select_rerank<1, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  CK(cudaFuncSetAttribute(k_select_rerank<2, 6, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  CK(cudaFuncSetAttribute(k_exact_fallback, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
  CK(cudaFuncSetAttribute(k_select_hits<2, 6>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  CK(cudaFuncSetAttribute(k_shard_consume, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  const char* no_pdl = getenv("KEDS_NO_PDL");
  ix->use_pdl = !(no_pdl && no_pdl[0] == '1');
  if (const char* ws = getenv("KEDS_NO_WARM_START")) ix->warm_start = !(ws[0] == '1');
  if (const char* rv = getenv("KEDS_RERANK_VARIANT")) {
    if (!strcmp(rv, "latency")) ix->rerank_variant = 1;
    if (!strcmp(rv, "throughput")) ix->rerank_variant = 2;
  }
  if (const char* rt = getenv("KEDS_RERANK_THREADS")) {
    const int v = atoi(rt);
    if (v == 32 || v == 64 || v == 128 || v == 256) ix->rerank_threads_large = v;
  }
  ix->attrs_set = true;
  return 0;
}

// Launch on `st`; with pdl the kernel may be scheduled while its predecessor in the stream is
// still draining (programmatic dependent launch) -- every kernel of the search chain calls
// griddep_wait() before it touches anything an earlier kernel wrote.
// cluster > 1: thread-block cluster of that many CTAs along x (the CTA-pair scoring kernel).
template <typename... KArgs, typename... Args>
int launch_kc(bool pdl, int cluster, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
              cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (pdl) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  if (cluster > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = static_cast<unsigned>(cluster);
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  CK(cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...));
  return 0;
}

template <typename... KArgs, typename... Args>
int launch_k(bool pdl, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
             Args&&... args) {
  return launch_kc(pdl, 1, kernel, grid, block, smem, st, std::forward<Args>(args)...);
}

Geometry geometry(const keds_index* ix, int n_db, int64_t nq) {
  Geometry g;
  g.n_qt = static_cast<int>((nq + BM - 1) / BM);
  // more than one query tile: CTA pairs share each row tile (two query tiles per work item)
  g.pair = ix->use_pair && g.n_qt >= 2 && ix->num_sms >= 2;
  g.sub = g.pair ? ScoreCfg<true>::kSub : ScoreCfg<false>::kSub;
  g.n_qg = g.pair ? (g.n_qt + 1) / 2 : g.n_qt;
  g.units = g.pair ? ix->num_sms / 2 : ix->num_sms;
  g.s_mem = static_cast<long long>(CAND_BUDGET / (size_t(LKEEP) * BM * 8)) /
            (static_cast<long long>(n_db) * g.n_qt * g.sub);
  return g;
}

// Pick the number of row slices: enough that no slice is expected to hold more than a third of
// LKEEP of the top-k, enough work items to fill the SMs, then whatever minimises the longest CTA.
// band_hint: the largest candidate band |C| a recent search on this handle reported (0: none).
// On i.i.d. data about 2k rows sit at or above tau; clustered embeddings put a whole cluster there,
// and a slice that holds LKEEP of them fails the certificate -- so the expected-fallback term
// below takes whichever is larger and the planner answers crowded bands with more, shorter slices.
Plan make_plan(const keds_index* ix, int n_db, int64_t nq, int k, int64_t n_min, int64_t n_max,
               uint32_t flags, unsigned int band_hint = 0) {
  Plan pl;
  static_cast<Geometry&>(pl) = geometry(ix, n_db, nq);
  const int T_min = static_cast<int>((n_min + BN - 1) / BN);
  const int T_max = static_cast<int>((n_max + BN - 1) / BN);
  // a slice hands over its best LKEEP-1 rows and drops the rest (theta = its LKEEP-th best): for
  // the certificate to pass, theta must sit well below the k-th best score overall, i.e. the
  // top-k must be spread over many slices (expected share per slice <= LKEEP / 6)
  // (in candidate lists: the pair kernel keeps one per column half of every slice)
  const int S_sel = std::max(1, ((6 * k + LKEEP - 1) / LKEEP + pl.sub - 1) / pl.sub);
  const int groups = n_db * pl.n_qg;
  const int S_hi = static_cast<int>(std::min<long long>(std::min(T_min, S_MAX), pl.s_mem));
  if ((flags & KEDS_SEARCH_EXACT_ONLY) || S_hi < S_sel || k > R_MAX / 2) {
    pl.exact_only = 1;
    return pl;
  }
  // re-rank variant: one wave of blocks (two per SM) runs the latency variant, more the
  // four-per-SM throughput variant
  pl.small_batch = nq * n_db <= 2ll * ix->num_sms;
  if (ix->rerank_variant == 1) pl.small_batch = true;   // experiments: KEDS_RERANK_VARIANT=latency|throughput
  if (ix->rerank_variant == 2) pl.small_batch = false;
  double best = 1e300;
  // one exact scan of every fp32 row, in the cost unit below (one bf16 row tile per work unit)
  const double scan_cost = 2.0 * T_max / pl.units;
  for (int S = S_sel; S <= S_hi; ++S) {
    const long long items = static_cast<long long>(groups) * S;
    const long long G = std::min<long long>(items, pl.units);
    const long long per_cta = (items + G - 1) / G;
    double cost = static_cast<double>(per_cta) * ((T_max + S - 1) / S) + 0.35 * per_cta;
    // expected fallbacks: a query is flagged when one list holds LKEEP or more of the rows at or
    // above tau (Poisson tail, five-fold margin) -- large k wants more lists than the SM count.
    // Rows at or above tau on i.i.d. data: ~2.4k with bf16 operands (wide band), k plus a few with
    // fp16 (measured 18-24 at k = 16, ~215 at k = 200); crowded bands arrive through band_hint.
    {
      const double band = ix->fmt == FMT_FP16 ? 1.15 * k + 12.0 : 2.0 * k;
      const double lam = std::max(band, 1.25 * static_cast<double>(band_hint)) / (S * pl.sub);
      double term = std::exp(-lam), tail = 0.0;  // term_i = e^-lam lam^i / i!
      for (int i = 1; i <= LKEEP + 40; ++i) {
        term *= lam / i;
        if (i >= LKEEP) tail += term;
      }
      cost += 5.0 * tail * static_cast<double>(nq) * n_db * S * pl.sub * scan_cost;
    }
    if (cost < best - 1e-9) {
      best = cost;
      pl.S = S;
    }
  }
  if (const char* dbg = getenv("KEDS_DEBUG_SLICES")) {  // experiments only: force the slice count
    const int v = atoi(dbg);
    if (v >= S_sel && v <= S_hi) pl.S = v;
  }
  pl.set_slices(n_db, pl.S);
  return pl;
}

// Gallery ranking: as many candidate lists as the tiles and the candidate budget allow (the band
// around a mid-ranked target is crowded); never exact-only.
Plan rank_plan(const keds_index* ix, int64_t nq) {
  Plan pl{geometry(ix, 1, nq)};
  const int T = static_cast<int>((ix->n + BN - 1) / BN);
  pl.set_slices(1, static_cast<int>(std::max<long long>(1, std::min<long long>(std::min(T, S_MAX), pl.s_mem))));
  return pl;
}

int ensure_q_map(keds_index* ix, int64_t rows_needed, cudaStream_t st) {
  const size_t bytes = static_cast<size_t>(rows_needed) * ix->d_pad * 2;
  if (bytes > ix->q_bf16.cap) {
    // round up so repeated slightly larger batches do not re-encode every call
    const int64_t rows = (rows_needed + 1023) / 1024 * 1024;
    CKS(ix->q_bf16.ensure(static_cast<size_t>(rows) * ix->d_pad * 2));
    // on the caller's stream: a legacy-stream memset is not ordered against a non-blocking stream
    CK(cudaMemsetAsync(ix->q_bf16.p, 0, ix->q_bf16.cap, st));
    ix->tm_q_base = nullptr;
  }
  if (ix->tm_q_base != ix->q_bf16.p || ix->tm_q_fmt != ix->fmt) {
    const int64_t rows = static_cast<int64_t>(ix->q_bf16.cap / (static_cast<size_t>(ix->d_pad) * 2));
    CKS(encode_rows_map(&ix->tm_q, ix->q_bf16.p, rows, ix->d_pad, BM, ix->fmt));
    ix->tm_q_base = ix->q_bf16.p;
    ix->tm_q_rows = rows;
    ix->tm_q_fmt = ix->fmt;
  }
  return 0;
}

// One search call. The entry points fill it with the caller's arrays; search_impl puts host
// queries and results into device staging before the first pass, and every pass gets a slice.
struct Call {
  keds_index* owner = nullptr;  // scratch, status blocks, stats and tuning switches: the call's first handle
  keds_index* dbs[2] = {nullptr, nullptr};
  int n_db = 1;
  int slot0 = 0;  // which of the call's databases dbs[0] is: its flagged count is reported there
  int64_t nq = 0;
  int k = 0;
  uint32_t flags = 0;
  int pass = 0;                  // status block of this pass
  const float* q = nullptr;      // fp32 [nq][d]
  const float* q_src = nullptr;  // page-locked host queries (device alias) or a misaligned query tensor
                                 // (gallery ranking), or null: k_prep_rows reads them and leaves the fp32 copy in q
  float* D[2] = {nullptr, nullptr};  // [nq][k] per database
  long long* I[2] = {nullptr, nullptr};
  // optional parts, absent while zero
  ConsumeParams cons{};           // the fused neighbour consumer (retrieve2)
  PeerOut peer{};                 // the sharded search's push to the other ranks
  const long long* ex = nullptr;  // [nq][n_ex] labels to leave out (device memory or a mapped host alias);
  int n_ex = 0;                   // k_prep_rows stages them as local row ids in owner->ex_rows
  HitsMode hits{};                // label hits at cut points in the re-rank's place
  RankMode rank{};                // gallery ranks in the top-k's place (rank.out set)
  RangeMode range{};              // range search in the top-k's place (range.lims set)
  float* dump = nullptr;          // debug_scores: the raw scores, ld_dump per query
  int64_t ld_dump = 0;

  int metric() const { return (flags & KEDS_SEARCH_FORCE_IP) ? METRIC_IP : owner->metric; }
  // the entry points' (exclude, n_exclude): NULL with 0 = no exclusion
  int exclude(const int64_t* labels, int n) {
    if (labels ? n < 1 || n > EXCLUDE_MAX : n != 0)
      return fail(KEDS_ERR_ARG, "exclude must be NULL with n_exclude = 0, or an [nq][n_exclude] array with 1 <= n_exclude <= %d",
                  EXCLUDE_MAX);
    ex = reinterpret_cast<const long long*>(labels);
    n_ex = n;
    return 0;
  }
};

Call call(int n_db, keds_index* a, keds_index* b, const float* q, int64_t nq, int k, float* Da, int64_t* Ia,
          float* Db, int64_t* Ib, uint32_t flags) {
  Call c;
  c.owner = c.dbs[0] = a;
  c.dbs[1] = b;
  c.n_db = n_db;
  c.q = q;
  c.nq = nq;
  c.k = k;
  c.D[0] = Da;
  c.I[0] = reinterpret_cast<long long*>(Ia);
  c.D[1] = Db;
  c.I[1] = reinterpret_cast<long long*>(Ib);
  c.flags = flags;
  return c;
}

// The exact-fallback kernel, ceil(nq / f_cap) passes; every launch returns at once when its slice
// of the flagged list is empty.
int launch_exact(const Call& c, unsigned long long* timing, cudaStream_t st) {
  keds_index* ix = c.owner;
  keds_index* const* dbs = c.dbs;
  const int n_db = c.n_db, k = c.k;
  const int64_t nq = c.nq;
  ExactParams ep;
  memset(&ep, 0, sizeof ep);
  if (c.ex) {
    ep.ex_rows = ix->ex_rows.as<int>();
    ep.n_ex = c.n_ex;
    ep.ex_ld = nq * c.n_ex;
  }
  ep.cons = c.cons;
  ep.n_db = n_db;
  ep.d = ix->d;
  ep.metric = c.metric();
  ep.k = k;
  ep.q_f32 = c.q;
  // Queries per launch: as many as the score scratch holds (it is allocated for the batch at hand,
  // never beyond the budget). Up to 1 GB always -- all of a 128-query batch at 2 x 0.5M rows, all of
  // 4,096 queries at 50k rows in ONE launch; large batches get up to 4 GB so that a search is followed
  // by about eight launches of this kernel, not sixty (each of them costs a few microseconds even
  // when nothing is queued: at 65,536 x 0.5M they added up to 2 ms of a 40-ms call).
  int64_t rows_sum = 0;
  for (int i = 0; i < n_db; ++i) rows_sum += dbs[i]->n;
  const long long row_bytes = 4 * std::max<int64_t>(rows_sum, 1);
  long long budget = std::max(1ll << 30, std::min(4ll << 30, static_cast<long long>(nq) * row_bytes / 8));
  long long fc = budget / row_bytes;
  fc = std::max(1ll, std::min<long long>(fc, nq));
  ep.f_cap = static_cast<int>(fc);
  // row chunks (phase-1 work units): about four per block, at least one 32-row group per warp
  const unsigned blocks_ = static_cast<unsigned>(ix->num_sms * 2);
  int64_t chunks_sum = 0;
  int chunks_max = 0;
  for (int i = 0; i < n_db; ++i) {
    const int64_t groups = (dbs[i]->n + 31) / 32;
    const int64_t want = 4ll * blocks_;
    ep.db[i].cg = std::max<int64_t>(EXACT_THREADS / 32, (groups + want - 1) / want);
    ep.db[i].chunks = static_cast<int>((groups + ep.db[i].cg - 1) / ep.db[i].cg);
    chunks_sum += ep.db[i].chunks;
    chunks_max = std::max(chunks_max, ep.db[i].chunks);
  }
  CKS(ix->exact_scratch.ensure(static_cast<size_t>(fc) * (rows_sum + chunks_sum) * 4));
  float* scratch = ix->exact_scratch.as<float>();
  for (int i = 0; i < n_db; ++i) {
    ExactDb& e = ep.db[i];
    e.x_f32 = dbs[i]->x_f32.as<float>();
    e.n_rows = dbs[i]->n;
    e.flagged = ix->flagged[i].as<int>();
    e.n_flagged = reinterpret_cast<int*>(ix->ctrl_cur) + i;
    e.scratch = scratch;
    scratch += static_cast<size_t>(fc) * dbs[i]->n;
    e.cmax = scratch;
    scratch += static_cast<size_t>(fc) * e.chunks;
    e.D = c.D[i];
    e.I = c.I[i];
    e.id_offset = dbs[i]->id_offset;
  }
  const int dq = (ix->d + 3) & ~3;
  const size_t smem_sc = static_cast<size_t>(EXACT_QG) * dq * 4 + (EXACT_THREADS / 32) * EXACT_QG * 4;
  ep.ck_cap = std::min(chunks_max, 8192);
  const size_t smem_sel = static_cast<size_t>(c.cons.part4) * 16 + static_cast<size_t>(k) * 20 + 256 * 4 + 16 + 16 + 32 +
                          static_cast<size_t>(EXACT_LIST_CAP) * 8 + static_cast<size_t>(ep.ck_cap) * 4;
  const size_t smem = std::max(smem_sc, smem_sel);
  if (smem > 160 * 1024) return fail(KEDS_ERR_ARG, "d=%d / k=%d too large for the exact fallback", ix->d, k);
  const unsigned blocks = blocks_;
  ep.err = ix->ctrl_cur + 2;
  ep.band_dev = ix->ctrl_cur + CTRL_BAND;
  const int passes = static_cast<int>((nq + fc - 1) / fc);
  for (int pass = 0; pass < passes; ++pass) {
    ep.pass = pass;
    ep.band_host = pass == passes - 1 ? ix->h_feedback : nullptr;
    ep.peer = c.peer;
    ep.peer.publish = c.peer.publish && pass == passes - 1;  // only the step's very last launch publishes
    ep.timing = pass == 0 ? timing : nullptr;
    // work counters of this launch: its own zeroed set (the last set is shared, with a memset, by
    // launches beyond EXACT_CTR_SETS)
    const int set = std::min(pass, EXACT_CTR_SETS - 1);
    ep.work = ix->ctrl_cur + CTRL_WORDS + 4 * set;
    ep.done = ep.work + 2;
    if (pass >= EXACT_CTR_SETS) CK(cudaMemsetAsync(ep.work, 0, 16, st));
    CKS(launch_k(ix->use_pdl, k_exact_fallback, dim3(blocks), dim3(EXACT_THREADS), smem, st, ep));
    ix->stats.launches += 1;
  }
  return 0;
}

// Candidate lines of a pass, indexed by (db, slice, query tile) whatever the work-item grouping.
int ensure_cand(keds_index* a, size_t lines) {
  CKS(a->cand.ensure(lines * LKEEP * BM * 8));
  CKS(a->cand_cnt.ensure(lines * BM * 4));
  CKS(a->cand_theta.ensure(lines * BM * 4));
  return 0;
}

// What every launch of the scoring kernel of a pass is given: the plan, the databases, the
// candidate lists and the error word, and a search's epilogue inputs (row bias, warm-start
// thresholds, exclusion, debug dump). Gallery ranking adds its band edges (launch_rank_targets).
ScoreParams score_params(const Call& c, const Plan& pl, unsigned long long* tchain) {
  const keds_index* a = c.owner;
  ScoreParams sp;
  memset(&sp, 0, sizeof sp);
  sp.n_db = c.n_db;
  sp.n_qt = pl.n_qt;
  sp.n_qg = pl.n_qg;
  sp.S = pl.S;
  sp.n_items = pl.n_items;
  sp.kblocks = a->d_pad / BK;
  sp.fmt_bits = a->fmt == FMT_BF16 ? kIdescBf16Bits : 0u;
  sp.nq = static_cast<int>(c.nq);
  for (int i = 0; i < c.n_db; ++i) {
    sp.n_rows[i] = static_cast<int>(c.dbs[i]->n);
    sp.n_tiles[i] = static_cast<int>((c.dbs[i]->n + BN - 1) / BN);
  }
  sp.cand = a->cand.as<uint2>();
  sp.cand_cnt = a->cand_cnt.as<int>();
  sp.cand_theta = a->cand_theta.as<float>();
  sp.err = a->ctrl_cur + 2;
  if (c.rank.out) return sp;
  for (int i = 0; i < c.n_db; ++i) sp.bias[i] = c.metric() == METRIC_L2 ? c.dbs[i]->bias.as<float>() : nullptr;
  sp.theta0 = a->warm_start ? a->theta0.as<float>() : nullptr;
  sp.theta_ld = pl.n_qt * BM;
  sp.dump = c.dump;
  sp.ld_dump = c.ld_dump;
  sp.timing = tchain ? tchain + 2 : nullptr;
  if (c.ex) {
    sp.ex_rows = a->ex_rows.as<int>();
    sp.n_ex = c.n_ex;
    sp.ex_ld = static_cast<long long>(c.nq) * c.n_ex;
  }
  return sp;
}

// The front of a pass: the status block cleared, the exclusion labels staged, and the queries'
// 16-bit operand rows and statistics (with the fp32 device copy of queries read from q_src).
// On the exact-only route no query rows are prepared: every query is flagged for the fallback.
int launch_prep(const Call& c, const Plan& pl, unsigned long long* tchain, cudaStream_t st) {
  keds_index* a = c.owner;
  const int n_db = c.n_db;
  const int64_t nq = c.nq;
  PrepParams pp;
  memset(&pp, 0, sizeof pp);
  pp.d = a->d;
  pp.d_pad = a->d_pad;
  pp.fmt = a->fmt;
  if (c.ex) {
    CKS(a->ex_rows.ensure(static_cast<size_t>(n_db) * nq * c.n_ex * 4));
    pp.ex.labels = c.ex;
    pp.ex.nq = nq;
    pp.ex.n_ex = c.n_ex;
    pp.ex.n_db = n_db;
    pp.ex.rows = a->ex_rows.as<int>();
    for (int i = 0; i < n_db; ++i) {
      pp.ex.id_offset[i] = c.dbs[i]->id_offset;
      pp.ex.n_rows[i] = c.dbs[i]->n;
    }
  }
  if (pl.exact_only) {
    if (c.q_src) CK(cudaMemcpyAsync(const_cast<float*>(c.q), c.q_src, static_cast<size_t>(nq) * a->d * 4, cudaMemcpyDefault, st));
    CK(cudaMemsetAsync(a->ctrl_cur, 0, CTRL_STRIDE * 4, st));
    for (int i = 0; i < n_db; ++i) {
      k_flag_all<<<static_cast<unsigned>((nq + 255) / 256), 256, 0, st>>>(
          a->flagged[i].as<int>(), reinterpret_cast<int*>(a->ctrl_cur) + i, static_cast<int>(nq));
      a->stats.launches++;
    }
    if (c.ex) {
      // the staging half of k_prep_rows alone (no query rows to prepare on this route)
      const unsigned blocks = static_cast<unsigned>(std::min<long long>((nq + 255) / 256, 1024));
      k_prep_rows<<<blocks, 256, 0, st>>>(pp);
      a->stats.launches++;
    }
    return 0;
  }
  // operands: bf16 queries + per-query residual norms
  const int64_t q_rows = static_cast<int64_t>(pl.n_qt) * BM;
  CKS(ensure_q_map(a, q_rows, st));
  CKS(a->qstat.ensure(static_cast<size_t>(nq) * sizeof(float4)));
  pp.x = c.q_src ? c.q_src : c.q;
  pp.n = nq;
  pp.out = a->q_bf16.as<uint16_t>();
  pp.stat = a->qstat.as<float4>();
  pp.zero_words = a->ctrl_cur;
  pp.n_zero = CTRL_STRIDE;
  pp.timing = tchain;
  pp.copy_f32 = c.q_src ? const_cast<float*>(c.q) : nullptr;
  if (!c.rank.out) {  // the lists' warm-start thresholds (gallery ranking starts from its band edges)
    CKS(a->theta0.ensure(static_cast<size_t>(n_db) * q_rows * 4));
    pp.neg_inf_words = a->theta0.as<float>();
    pp.n_neg_inf = static_cast<int>(n_db * q_rows);
  }
  const unsigned blocks = static_cast<unsigned>(std::min<long long>((nq * 32 + 255) / 256, 4096));  // a warp per query
  CKS(launch_k(a->use_pdl, k_prep_rows, dim3(blocks), dim3(256), 0, st, pp));
  a->stats.launches++;
  return 0;
}

// The scoring kernel in the instantiation sp asks for: gallery ranking (rk_lo), top-k with
// exclusion (ex_rows: tests each tile against the query's excluded rows), range search (rg_out) or
// the plain top-k.
int launch_score(const Call& c, const Plan& pl, const ScoreParams& sp, cudaStream_t st) {
  keds_index* a = c.owner;
  const keds_index* x0 = c.dbs[0];
  const keds_index* x1 = c.n_db > 1 ? c.dbs[1] : c.dbs[0];
  if (pl.pair)
    CKS(launch_kc(a->use_pdl, 2,
                  sp.rk_lo     ? k_score_topk<true, true>
                  : sp.ex_rows ? k_score_topk<true, false, true>
                  : sp.rg_out  ? k_score_range<true>
                               : k_score_topk<true>,
                  dim3(pl.grid), dim3(SCORE_PAIR_THREADS), SCORE_PAIR_SMEM_BYTES, st, a->tm_q, x0->tm_xh, x1->tm_xh, sp));
  else
    CKS(launch_k(a->use_pdl,
                 sp.rk_lo     ? k_score_topk<false, true>
                 : sp.ex_rows ? k_score_topk<false, false, true>
                 : sp.rg_out  ? k_score_range<false>
                              : k_score_topk<false>,
                 dim3(pl.grid), dim3(SCORE_THREADS), SCORE_SMEM_BYTES, st, a->tm_q, x0->tm_x, x1->tm_x, sp));
  a->stats.launches++;
  CK(cudaGetLastError());
  return 0;
}

// Candidate capacity per query of the re-rank and hits blocks: room for the band a recent search
// reported (a query that does not fit is answered by the exact fallback and raises the next call's figure).
int cand_capacity(int k, unsigned int band_hint) {
  const unsigned int want =
      std::max<unsigned int>(static_cast<unsigned int>(k + k / 2 + 64), band_hint + band_hint / 2);
  int rmax = 256;
  while (rmax < static_cast<int>(std::min<unsigned int>(want, R_MAX))) rmax *= 2;
  return rmax;
}

// The top-k from the candidate lists: exact fp32 scores of the rows at or above the certified
// threshold, the queries the certificate rejects flagged for the fallback.
int launch_rerank(const Call& c, const Plan& pl, const ScoreParams& sp, unsigned int band_hint,
                  unsigned long long* tchain, cudaStream_t st) {
  keds_index* a = c.owner;
  const int n_db = c.n_db, k = c.k;
  const int64_t nq = c.nq;
  RerankParams rp;
  memset(&rp, 0, sizeof rp);
  rp.n_db = n_db;
  rp.n_qt = pl.n_qt;
  rp.S = pl.S * pl.sub;  // candidate lines per (database, query)
  rp.nq = static_cast<int>(nq);
  rp.k = k;
  rp.d = a->d;
  rp.metric = c.metric();
  rp.cand = sp.cand;
  rp.cand_cnt = sp.cand_cnt;
  rp.cand_theta = sp.cand_theta;
  rp.q_f32 = c.q;
  rp.qstat = a->qstat.as<float4>();
  for (int i = 0; i < n_db; ++i) {
    rp.x_f32[i] = c.dbs[i]->x_f32.as<float>();
    rp.dbstat[i] = c.dbs[i]->dbstat.as<unsigned int>();
    rp.D[i] = c.D[i];
    rp.I[i] = c.I[i];
    rp.id_offset[i] = c.dbs[i]->id_offset;
    rp.flagged[i] = a->flagged[i].as<int>();
    rp.n_flagged[i] = reinterpret_cast<int*>(a->ctrl_cur) + i;
  }
  rp.eps_scale = a->eps_scale;
  rp.band_max = a->ctrl_cur + CTRL_BAND;
  // A single wave (the latency variant) has the shared memory to spare: full candidate capacity.
  // Large batches live on blocks per SM, so they start small and follow the band a recent search reported.
  const int rmax = pl.small_batch ? R_MAX : cand_capacity(k, band_hint);
  rp.rmax = rmax;
  rp.peer = c.peer;
  rp.cons = c.cons;
  rp.timing = tchain ? tchain + 4 : nullptr;
  const size_t slots = static_cast<size_t>(pl.S) * pl.sub * LKEEP;
  // qvec | part | okey | keys, ids | smax | a_key, a_id, sel_id, sel_sc | hist | red | bcast | counters | top_*
  const size_t smem = static_cast<size_t>((a->d + 3) & ~3) * 4 + static_cast<size_t>(c.cons.part4) * 16 +
                      static_cast<size_t>(rmax) * 24 + slots * 8 + pl.S * pl.sub * 4 + 256 * 4 + 32 * 4 + 16 + 16 +
                      static_cast<size_t>(k) * 12;
  if (smem > 200 * 1024) return fail(KEDS_ERR_ARG, "re-rank shared memory %zu too large", smem);
  if (pl.small_batch)
    CKS(launch_k(a->use_pdl, k_select_rerank<3, 2>, dim3(static_cast<unsigned>(nq), n_db),
                 dim3(RERANK_THREADS), smem, st, rp));
  else if (k >= 128 && a->rerank_threads_large == 128)
    // hundreds of fp32 rows per query: two rows per warp in flight (80 registers, six blocks per
    // SM) measured 0.82-0.87 ms against 0.95-1.0 at 10,000 x 50k, k = 200; at k = 16 / 64 the
    // 64-register variant below is 5-10 % faster
    CKS(launch_k(a->use_pdl, k_select_rerank<2, 6, 128>, dim3(static_cast<unsigned>(nq), n_db),
                 dim3(128), smem, st, rp));
  else
    CKS(launch_k(a->use_pdl, k_select_rerank<1, 4>, dim3(static_cast<unsigned>(nq), n_db),
                 dim3(a->rerank_threads_large), smem, st, rp));
  a->stats.launches++;
  CK(cudaGetLastError());
  return 0;
}

// Label hits at the cut points instead of the ranked rows (label_hits.cuh): same lists, same
// certificate, exact scores only for the rows inside the error band around a cut.
int launch_hits(const Call& c, const Plan& pl, const ScoreParams& sp, unsigned int band_hint,
                unsigned long long* tchain, cudaStream_t st) {
  keds_index* a = c.owner;
  const HitsMode& hm = c.hits;
  HitsParams hp;
  memset(&hp, 0, sizeof hp);
  hp.n_qt = pl.n_qt;
  hp.S = pl.S * pl.sub;
  hp.nq = static_cast<int>(c.nq);
  hp.d = a->d;
  hp.metric = c.metric();
  hp.nks = hm.nks;
  for (int j = 0; j < hm.nks; ++j) hp.ks[j] = hm.ks[j];
  const int rmax = cand_capacity(c.k, band_hint);
  hp.rmax = rmax;
  hp.cand = sp.cand;
  hp.cand_cnt = sp.cand_cnt;
  hp.cand_theta = sp.cand_theta;
  hp.q_f32 = c.q;
  hp.qstat = a->qstat.as<float4>();
  hp.x_f32 = c.dbs[0]->x_f32.as<float>();
  hp.dbstat = c.dbs[0]->dbstat.as<unsigned int>();
  hp.row_labels = hm.row_labels;
  hp.qlabel = hm.qlabel;
  hp.hits = hm.hits;
  hp.flagged = a->flagged[0].as<int>();
  hp.n_flagged = reinterpret_cast<int*>(a->ctrl_cur);
  hp.eps_scale = a->eps_scale;
  hp.band_max = a->ctrl_cur + CTRL_BAND;
  hp.timing = tchain ? tchain + 4 : nullptr;
  const size_t hslots = static_cast<size_t>(pl.S) * pl.sub * LKEEP;
  // qvec | cs | keys, ids | c_sc, c_info, amb | hist | red | bcast | counters | n_cert, band_end, n_hit
  const size_t hsmem = static_cast<size_t>((a->d + 3) & ~3) * 4 + hslots * 8 + static_cast<size_t>(rmax) * 20 +
                       1024 * 4 + 32 * 4 + 16 + 16 + 3 * HITS_MAX_CUTS * 4;
  if (hsmem > 200 * 1024) return fail(KEDS_ERR_ARG, "label-hits shared memory %zu too large", hsmem);
  // <2 rows in flight per warp, 6 blocks per SM>: measured 0.55 ms at 10,000 x 50k against 0.68 (<3, 4>) / 0.57 (<1, 8>)
  CKS(launch_k(a->use_pdl, k_select_hits<2, 6>, dim3(static_cast<unsigned>(c.nq)), dim3(HITS_THREADS), hsmem, st, hp));
  a->stats.launches++;
  CK(cudaGetLastError());
  return 0;
}

// Label hits behind the exact fallback: the queued queries' exact rows (written by the fallback
// just now) -> their hits.
int launch_hits_from_rows(const Call& c, cudaStream_t st) {
  keds_index* a = c.owner;
  HitsParams hp;
  memset(&hp, 0, sizeof hp);
  hp.nks = c.hits.nks;
  for (int j = 0; j < c.hits.nks; ++j) hp.ks[j] = c.hits.ks[j];
  hp.hits = c.hits.hits;
  CKS(launch_k(a->use_pdl, k_hits_from_rows, dim3(static_cast<unsigned>(std::min<int64_t>((c.nq + 127) / 128, 64))),
               dim3(128), 0, st, a->flagged[0].as<int>(), reinterpret_cast<int*>(a->ctrl_cur), c.I[0], c.k,
               c.dbs[0]->id_offset, c.hits.row_labels, c.hits.qlabel, hp));
  a->stats.launches++;
  return 0;
}

// Shared memory of k_gallery_rank: 8 queries per block
size_t gallery_rank_smem(int d) { return static_cast<size_t>((d + 3) & ~3) * 4 * 8; }

// Gallery ranking, before the scoring kernel: each query's exact fp32 target score and the error
// band around it, which the scoring kernel's counting epilogue reads.
int launch_rank_targets(const Call& c, ScoreParams& sp, cudaStream_t st) {
  keds_index* a = c.owner;
  const keds_index* g = c.dbs[0];
  const int64_t nq = c.nq;
  CKS(a->rk.ensure(static_cast<size_t>(nq) * 5 * 4));
  float* rk_st = a->rk.as<float>();
  float* rk_lo = rk_st + nq;
  float* rk_hi = rk_lo + nq;
  int* rk_t = reinterpret_cast<int*>(rk_hi + nq);
  int* rk_e = rk_t + nq;
  CKS(launch_k(a->use_pdl, k_rank_targets, dim3(static_cast<unsigned>((nq * 32 + 255) / 256)), dim3(256), 0, st, c.q,
               nq, g->x_f32.as<float>(), g->d, c.rank.target, c.rank.exclude, a->qstat.as<float4>(),
               g->dbstat.as<unsigned int>(), a->eps_scale, rk_st, rk_lo, rk_hi, rk_t, rk_e));
  a->stats.launches++;
  sp.rk_lo = rk_lo;
  sp.rk_hi = rk_hi;
  sp.rk_target = rk_t;
  sp.rk_exclude = c.rank.exclude ? rk_e : nullptr;
  return 0;
}

// Gallery ranking, after the scoring kernel: the lists' certain counts plus the band rows settled
// exactly (k_rank_finish), then the exact recount of the queries whose band overflowed a list
// (k_gallery_rank over the queue; none, normally: its blocks leave at once).
int launch_rank_count(const Call& c, const Plan& pl, const ScoreParams& sp, cudaStream_t st) {
  keds_index* a = c.owner;
  const keds_index* g = c.dbs[0];
  const int64_t nq = c.nq;
  int* queue = a->flagged[0].as<int>();
  int* n_queue = reinterpret_cast<int*>(a->ctrl_cur);
  CKS(launch_k(a->use_pdl, k_rank_finish, dim3(static_cast<unsigned>((nq * 32 + 255) / 256)), dim3(256), 0, st, c.q,
               nq, g->x_f32.as<float>(), g->d, pl.S * pl.sub, pl.n_qt, sp.cand, sp.cand_cnt, sp.cand_theta,
               a->rk.as<float>(), sp.rk_target, c.rank.out, queue, n_queue));
  CKS(launch_k(a->use_pdl, k_gallery_rank, dim3(static_cast<unsigned>((nq + 7) / 8)), dim3(256), gallery_rank_smem(g->d),
               st, c.q, nq, g->x_f32.as<float>(), g->n, g->d, c.rank.target, c.rank.exclude, c.rank.out, queue, n_queue));
  a->stats.launches += 2;
  CK(cudaGetLastError());
  return 0;
}

// Range search: row slices for the scoring kernel alone (there are no candidate lists to certify),
// by the top-k planner's balance term.
Plan range_plan(const keds_index* ix, int64_t nq) {
  Plan pl{geometry(ix, 1, nq)};
  const int T = static_cast<int>((ix->n + BN - 1) / BN);
  double best = 1e300;
  for (int S = 1; S <= std::min(T, S_MAX); ++S) {
    const long long items = static_cast<long long>(pl.n_qg) * S;
    const long long G = std::min<long long>(items, pl.units);
    const long long per_cta = (items + G - 1) / G;
    const double cost = static_cast<double>(per_cta) * ((T + S - 1) / S) + 0.35 * per_cta;
    if (cost < best - 1e-9) {
      best = cost;
      pl.S = S;
    }
  }
  pl.set_slices(1, pl.S);
  return pl;
}

// Blocks for a grid-stride kernel over n work items of `per` threads each.
unsigned stride_grid(const keds_index* a, long long n, int per) {
  const long long want = (std::max(1ll, n) * per + 255) / 256;
  return static_cast<unsigned>(std::min<long long>(want, 16ll * a->num_sms));
}

// Wait for the queued work and read n 64-bit device words; a fired watchdog is the call's error.
int range_read(keds_index* a, const unsigned long long* words, unsigned long long* out, int n, cudaStream_t st) {
  uint32_t err = 0;
  CK(cudaMemcpyAsync(out, words, static_cast<size_t>(n) * 8, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(&err, a->ctrl_cur + 2, 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  a->stats.err_word = err;
  if (err != 0) return fail(KEDS_ERR_KERNEL, "device watchdog fired (range search): error word 0x%x", err);
  return 0;
}

// One pass of a range search. The result size is known only once the pass has run, so it reads
// back twice: the candidate count (a buffer that overflowed is grown and the scoring kernel rerun,
// so no candidate is ever dropped), then the hit count (the results grow, keeping earlier passes).
int range_pass(const Call& c, cudaStream_t st) {
  keds_index* a = c.owner;
  const keds_index* x = c.dbs[0];
  const int64_t nq = c.nq;
  const int metric = c.metric();
  const float radius = c.range.radius;
  const Plan pl = range_plan(a, nq);
  a->stats.slices = pl.S;
  a->stats.items = pl.n_items;
  a->stats.grid = pl.grid;

  CKS(launch_prep(c, pl, nullptr, st));  // also clears the status block, the candidate count included
  CKS(a->rg_thr.ensure(static_cast<size_t>(nq) * 4));
  CKS(launch_k(a->use_pdl, k_range_band, dim3(static_cast<unsigned>((nq + 255) / 256)), dim3(256), 0, st,
               a->qstat.as<float4>(), x->dbstat.as<unsigned int>(), static_cast<int>(nq), a->d_pad, metric, radius,
               a->eps_scale, a->rg_thr.as<float>()));
  ScoreParams sp = score_params(c, pl, nullptr);
  sp.theta0 = nullptr;
  sp.rg_thr = a->rg_thr.as<float>();
  unsigned long long* count = reinterpret_cast<unsigned long long*>(a->ctrl_cur + CTRL_RANGE);
  sp.rg_count = count;
  CKS(a->rg_cand.ensure(static_cast<size_t>(std::max<int64_t>(int64_t(1) << 16, nq * 64)) * 8));
  sp.rg_out = a->rg_cand.as<uint2>();
  sp.rg_cap = a->rg_cand.cap / 8;
  CKS(launch_score(c, pl, sp, st));
  a->stats.launches += 2;
  unsigned long long n_cand = 0;
  CKS(range_read(a, count, &n_cand, 1, st));
  if (n_cand > sp.rg_cap) {
    CKS(a->rg_cand.ensure(static_cast<size_t>(n_cand + n_cand / 4) * 8));
    sp.rg_out = a->rg_cand.as<uint2>();
    sp.rg_cap = a->rg_cand.cap / 8;
    CK(cudaMemsetAsync(count, 0, 8, st));
    CKS(launch_score(c, pl, sp, st));
    CKS(range_read(a, count, &n_cand, 1, st));
  }
  const long long nc = static_cast<long long>(n_cand);

  // exact scores, hits per query, offsets (and this pass's lims)
  CKS(a->rg_qcnt.ensure(static_cast<size_t>(nq) * 4));
  CKS(a->rg_off.ensure(static_cast<size_t>(nq + 1) * 8));
  CKS(a->rg_key.ensure(static_cast<size_t>(std::max(nc, 1ll)) * 16));
  CKS(a->rg_word.ensure(16));
  CK(cudaMemsetAsync(a->rg_qcnt.p, 0, static_cast<size_t>(nq) * 4, st));
  int* qcnt = a->rg_qcnt.as<int>();
  long long* off = a->rg_off.as<long long>();
  unsigned long long* k0 = a->rg_key.as<unsigned long long>();
  unsigned long long* k1 = k0 + std::max(nc, 1ll);
  if (nc > 0) {
    k_range_rescore<<<stride_grid(a, nc, 32), 256, 0, st>>>(a->rg_cand.as<uint2>(), nc, c.q, x->x_f32.as<float>(),
                                                            a->d, metric, radius, k0, qcnt);
    a->stats.launches++;
  }
  k_range_scan<<<1, 1024, 0, st>>>(qcnt, static_cast<int>(nq), a->rg_total, off, c.range.lims,
                                   a->rg_word.as<unsigned long long>());
  a->stats.launches++;
  unsigned long long w[2] = {0, 0};
  CKS(range_read(a, a->rg_word.as<unsigned long long>(), w, 2, st));
  const long long total = static_cast<long long>(w[0]), longest = static_cast<long long>(w[1]);
  if (total == 0) return 0;

  // the hits into their queries' segments, ordered by (score, label) inside each, then out
  const size_t keep = static_cast<size_t>(a->rg_total);
  const size_t need = keep + static_cast<size_t>(total);
  if (need * 8 > a->rg_I.cap) {  // by half again at least, so that passes of one call rarely copy
    CKS(a->rg_D.grow_keep(std::max(need * 4, a->rg_D.cap + a->rg_D.cap / 2), keep * 4));
    CKS(a->rg_I.grow_keep(std::max(need * 8, a->rg_I.cap + a->rg_I.cap / 2), keep * 8));
  }
  k_range_scatter<<<stride_grid(a, nc, 1), 256, 0, st>>>(a->rg_cand.as<uint2>(), k0, nc, off, qcnt, k1);
  unsigned long long* in = k1;
  unsigned long long* out = k0;
  k_range_sort_runs<<<stride_grid(a, total, 1), 256, 0, st>>>(in, out, total, off, static_cast<int>(nq));
  std::swap(in, out);
  a->stats.launches += 3;
  for (long long run = RANGE_RUN; run < longest; run *= 2) {
    k_range_merge<<<stride_grid(a, total, 1), 256, 0, st>>>(in, out, total, off, static_cast<int>(nq), run);
    std::swap(in, out);
    a->stats.launches++;
  }
  k_range_emit<<<stride_grid(a, total, 1), 256, 0, st>>>(in, total, metric, x->id_offset, a->rg_D.as<float>() + keep,
                                                         a->rg_I.as<long long>() + keep);
  CK(cudaGetLastError());
  a->rg_total += total;
  return 0;
}

// One pass (<= Q_PASS_MAX queries) of a call; q, D and I are device memory. The chain: prep, the
// scoring kernel and its epilogue (re-rank, label hits or the rank count), the exact fallback.
int search_pass(const Call& c, cudaStream_t st) {
  keds_index* a = c.owner;
  keds_index* const* ix = c.dbs;
  const int n_db = c.n_db;
  const int64_t nq = c.nq;
  CKS(set_kernel_attrs(a));
  // in-kernel %globaltimer stamps, one {min start, max end} pair per kernel of this chain
  // (prep, score, rerank, exact scores, exact select); the first TIMING_RING searches are timed
  unsigned long long* tchain = nullptr;
  if (a->timing_on && a->timing_launches < TIMING_RING && !c.dump && !c.rank.out) {
    tchain = a->timing.as<unsigned long long>() + TIMING_PAIRS * 2 * a->timing_launches;
    a->timing_launches++;
  }
  a->ctrl_cur = a->ctrl.as<unsigned int>() + static_cast<size_t>(c.pass) * CTRL_STRIDE;
  a->ctrl_passes = c.pass + 1;
  a->ctrl_slot = c.slot0;
  if (c.range.lims) return range_pass(c, st);
  for (int i = 0; i < n_db; ++i) CKS(a->flagged[i].ensure(static_cast<size_t>(nq) * 4));

  int64_t n_min = ix[0]->n, n_max = ix[0]->n;
  if (n_db > 1) {
    n_min = std::min(n_min, ix[1]->n);
    n_max = std::max(n_max, ix[1]->n);
  }
  const unsigned int band_hint = a->h_feedback ? *static_cast<volatile unsigned int*>(a->h_feedback) : 0u;
  const Plan pl = c.rank.out ? rank_plan(a, nq) : make_plan(a, n_db, nq, c.k, n_min, n_max, c.flags, band_hint);
  if (c.dump && pl.exact_only) return fail(KEDS_ERR_ARG, "debug_scores needs at least one 256-row tile");
  a->stats.exact_only = pl.exact_only;
  a->stats.slices = pl.S;
  a->stats.items = pl.n_items;
  a->stats.grid = pl.grid;

  CKS(launch_prep(c, pl, tchain, st));
  if (!pl.exact_only) {
    CKS(ensure_cand(a, static_cast<size_t>(n_db) * pl.S * pl.sub * pl.n_qt));
    ScoreParams sp = score_params(c, pl, tchain);
    if (c.rank.out) CKS(launch_rank_targets(c, sp, st));
    CKS(launch_score(c, pl, sp, st));
    if (c.dump) return 0;
    if (c.rank.out) return launch_rank_count(c, pl, sp, st);
    CKS(c.hits.nks ? launch_hits(c, pl, sp, band_hint, tchain, st) : launch_rerank(c, pl, sp, band_hint, tchain, st));
  }
  if (!(c.flags & KEDS_SEARCH_NO_FALLBACK) || pl.exact_only) CKS(launch_exact(c, tchain ? tchain + 6 : nullptr, st));
  if (c.hits.nks) CKS(launch_hits_from_rows(c, st));
  CK(cudaGetLastError());
  return 0;
}

__global__ void k_fill_pad(float* D, long long* I, long long n, float dv) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) {
    D[i] = dv;
    I[i] = -1;
  }
}

// Queries [q0, q0 + nb) of a call: every per-query pointer moved to q0, and only the call's last
// pass publishes to the peers.
Call slice(const Call& c, int64_t q0, int64_t nb) {
  Call p = c;
  const int64_t d = c.owner->d, k = c.k;
  p.nq = nb;
  p.pass = static_cast<int>(q0 / Q_PASS_MAX);
  p.q += q0 * d;
  if (p.q_src) p.q_src += q0 * d;
  // (label hits: D and I hold the fallback's rows of the queued queries, scratch every pass reuses)
  for (int i = 0; i < c.n_db && !c.hits.nks; ++i) {
    p.D[i] += q0 * k;
    p.I[i] += q0 * k;
  }
  for (int s = 0; s < 2; ++s) {
    if (p.cons.feat[s]) p.cons.feat[s] += q0 * k * d;
    if (p.cons.pool[s]) p.cons.pool[s] += q0 * d;
    if (p.cons.host_D[s]) p.cons.host_D[s] += q0 * k;
    if (p.cons.host_I[s]) p.cons.host_I[s] += q0 * k;
  }
  for (int r = 0; r < p.peer.n; ++r) {
    if (p.peer.D[r]) p.peer.D[r] += q0 * k;
    if (p.peer.I[r]) p.peer.I[r] += q0 * k;
  }
  if (p.peer.n) p.peer.publish = q0 + nb >= c.nq;  // the flags go out behind the step's last pass
  if (p.ex) p.ex += q0 * c.n_ex;
  if (p.hits.nks) {
    p.hits.qlabel += q0;
    p.hits.hits += q0 * p.hits.nks;
  }
  if (p.rank.out) {
    p.rank.target += q0;
    if (p.rank.exclude) p.rank.exclude += q0;
    p.rank.out += q0;
  }
  if (p.range.lims) p.range.lims += q0;
  return p;
}

// Every pass of a call, queued back to back: each pass has its own status block and the scratch is
// reused in stream order (each kernel of a chain waits for its predecessor to complete), so the
// passes need no host round trip between them. The status blocks are sized before the first launch:
// growing them later would free memory that kernels of an earlier pass still write.
int run_passes(const Call& c, cudaStream_t st) {
  CKS(c.owner->ctrl.ensure(static_cast<size_t>((c.nq + Q_PASS_MAX - 1) / Q_PASS_MAX) * CTRL_STRIDE * 4));
  for (int64_t q0 = 0; q0 < c.nq; q0 += Q_PASS_MAX)
    CKS(search_pass(slice(c, q0, std::min<int64_t>(Q_PASS_MAX, c.nq - q0)), st));
  return 0;
}

// Status of a call = its passes' status blocks folded: flagged queries summed, first error word.
// Sets last_stats; a fired watchdog is the call's error.
int fold_status(keds_index* a, const uint32_t* blocks) {
  uint32_t h[3] = {0, 0, 0};
  for (int p = 0; blocks && p < a->ctrl_passes; ++p) {
    const uint32_t* b = blocks + static_cast<size_t>(p) * CTRL_STRIDE;
    for (int i = a->ctrl_slot; i < 2; ++i) h[i] += b[i - a->ctrl_slot];
    if (h[2] == 0) h[2] = b[2];
  }
  a->stats.n_flagged[0] = static_cast<int32_t>(h[0]);
  a->stats.n_flagged[1] = static_cast<int32_t>(h[1]);
  a->stats.err_word = h[2];
  if (h[2] != 0)
    return fail(KEDS_ERR_KERNEL, "device watchdog fired (scoring pipeline or fallback barrier): error word 0x%x", h[2]);
  return 0;
}

int finish_sync(keds_index* a, cudaStream_t st) {
  CK(cudaStreamSynchronize(st));
  if (!a->ctrl.p) return fold_status(a, nullptr);
  std::vector<uint32_t> all(static_cast<size_t>(a->ctrl_passes) * CTRL_STRIDE);
  CK(cudaMemcpy(all.data(), a->ctrl.p, all.size() * 4, cudaMemcpyDeviceToHost));
  return fold_status(a, all.data());
}

// Where a call's caller arrays may live.
enum Io {
  IO_HOST,    // q, D and I host or device memory (host arrays are staged through the handle)
  IO_DEVICE,  // device memory, checked by the caller
  IO_MAPPED,  // D and I device memory, checked by the caller; q and the exclusion labels device or
              // page-locked host memory (read through the mapping)
};

int search_impl(Call c, Io io, void* stream) {
  keds_index** ix = c.dbs;
  keds_index* a = c.owner;
  const int n_db = c.n_db, k = c.k;
  const int64_t nq = c.nq;
  if (!a || !c.q || nq < 0 || k <= 0) return fail(KEDS_ERR_ARG, "search: null handle/query or bad nq/k");
  if (k > K_MAX) return fail(KEDS_ERR_ARG, "search: k=%d exceeds the maximum %d", k, K_MAX);
  for (int i = 0; i < n_db; ++i) {
    if (!ix[i] || !c.D[i] || !c.I[i]) return fail(KEDS_ERR_ARG, "search: null index or output pointer");
    if (ix[i]->d != a->d || ix[i]->metric != a->metric || ix[i]->device != a->device)
      return fail(KEDS_ERR_ARG, "search2: indices differ in d, metric or device");
    if (ix[i]->n > 0x7fffffffll - BN) return fail(KEDS_ERR_ARG, "index too large for 32-bit row ids");
  }
  DeviceGuard g(a->device);
  if (!g.ok) return fail(KEDS_ERR_NO_GPU, "cannot select CUDA device %d", a->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  memset(&a->stats, 0, sizeof a->stats);
  if (nq == 0) return 0;
  // one query operand feeds both databases: they must share the 16-bit format. bf16 is the one
  // every database can take, so a mixed pair settles there (once; the rows are re-rounded).
  if (n_db > 1 && ix[0]->fmt != ix[1]->fmt)
    for (int i = 0; i < 2; ++i)
      if (ix[i]->fmt != FMT_BF16) CKS(keds_index_set_operand_format(ix[i], FMT_BF16));

  const PtrLoc lq = io == IO_DEVICE ? PtrLoc{a->device, nullptr} : locate(c.q);
  if (!lq && io == IO_MAPPED && !lq.mapped)
    return fail(KEDS_ERR_ARG, "retrieve2: q is neither device memory nor page-locked host memory");
  bool out_dev = true;
  for (int i = 0; io == IO_HOST && i < n_db; ++i) {
    const bool dd = static_cast<bool>(locate(c.D[i])), di = static_cast<bool>(locate(c.I[i]));
    if (dd != di) return fail(KEDS_ERR_ARG, "search: D and I must both be host or both be device memory");
    if (i > 0 && dd != out_dev) return fail(KEDS_ERR_ARG, "search2: outputs must all be host or all be device memory");
    out_dev = dd;
  }
  if (c.ex) {
    const PtrLoc lex = locate(c.ex);
    if (lex.device != a->device) {
      if (io != IO_MAPPED || !lex.mapped)
        return fail(KEDS_ERR_ARG, io == IO_MAPPED ? "retrieve2: exclude is neither device memory of the index's GPU "
                                                    "nor page-locked host memory"
                                                  : "search: exclude must be device memory of the index's GPU");
      c.ex = static_cast<const long long*>(lex.mapped);
    }
  }
  // Host in, host out (the reference's numpy call): the call synchronises before it returns, so
  // page-locked staging buffers can be reused call after call (one real DMA each way instead of
  // the driver's chunked pageable copies). Letting the kernels work on those buffers through the
  // mapping (as keds_retrieve2 does with host mirrors for RetrievalStep) was measured here too and is no
  // faster for this path (two searches of 128 queries: 403-411 us with copies, 413-425 us mapped):
  // the call is dominated by its host side.
  // one database's I (8 B) and D (4 B) blocks in the staged result, labels first (8-byte aligned)
  const size_t res_per = (static_cast<size_t>(nq) * k * 12 + 15) & ~size_t(15);
  const float* q = c.q;
  if (!lq) {
    const size_t qb = static_cast<size_t>(nq) * a->d * 4;
    CKS(a->q_f32.ensure(qb));
    c.q = a->q_f32.as<float>();
    if (io == IO_MAPPED) {
      c.q_src = static_cast<const float*>(lq.mapped);
    } else {
      const void* src = q;
      if (!out_dev && qb <= (size_t(64) << 20)) {
        CKS(a->h_q.ensure(qb));
        memcpy(a->h_q.p, q, qb);
        src = a->h_q.p;
      }
      CK(cudaMemcpyAsync(a->q_f32.p, src, qb, cudaMemcpyHostToDevice, st));
    }
  }
  float* D[2] = {c.D[0], c.D[1]};
  long long* I[2] = {c.I[0], c.I[1]};
  for (int i = 0; i < n_db && !out_dev; ++i) {
    CKS(a->D_stage[i].ensure(static_cast<size_t>(nq) * k * 4));
    CKS(a->I_stage[i].ensure(static_cast<size_t>(nq) * k * 8));
    c.D[i] = a->D_stage[i].as<float>();
    c.I[i] = a->I_stage[i].as<long long>();
  }
  // status blocks of every pass (the empty-database route clears them)
  const int n_passes = static_cast<int>((nq + Q_PASS_MAX - 1) / Q_PASS_MAX);
  CKS(a->ctrl.ensure(static_cast<size_t>(n_passes) * CTRL_STRIDE * 4));
  if (ix[0]->n == 0 || (n_db > 1 && ix[1]->n == 0)) {
    // empty databases answer with padding only; a non-empty one is searched alone, still with the
    // owner's scratch, status blocks and switches
    if (c.cons.enabled) return fail(KEDS_ERR_ARG, "retrieve2: both databases must hold rows");
    // (with every database empty no chain runs: the status blocks must read clean)
    CK(cudaMemsetAsync(a->ctrl.p, 0, static_cast<size_t>(n_passes) * CTRL_STRIDE * 4, st));
    a->ctrl_passes = n_passes;
    Call rest = c;
    rest.n_db = 0;
    for (int i = 0; i < n_db; ++i) {
      if (ix[i]->n != 0) {
        rest.n_db = 1;
        rest.slot0 = i;
        rest.dbs[0] = ix[i];
        rest.D[0] = c.D[i];
        rest.I[0] = c.I[i];
      } else {
        const long long tot = static_cast<long long>(nq) * k;
        k_fill_pad<<<static_cast<unsigned>((tot + 255) / 256), 256, 0, st>>>(
            c.D[i], c.I[i], tot, c.metric() == METRIC_L2 ? FLT_MAX : -FLT_MAX);
      }
    }
    c = rest;
  }
  if (c.n_db) CKS(run_passes(c, st));
  if (!out_dev) {
    // results and status words into pinned memory with asynchronous copies, ONE synchronisation,
    // then plain memcpy into the caller's arrays
    const size_t db_ = static_cast<size_t>(nq) * k * 4, ib_ = static_cast<size_t>(nq) * k * 8;
    const size_t per = res_per;
    if (per * n_db > (size_t(256) << 20)) {
      // very large result blocks: not worth pinning that much host memory, copy straight out
      for (int i = 0; i < n_db; ++i) {
        CK(cudaMemcpyAsync(D[i], a->D_stage[i].p, db_, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(I[i], a->I_stage[i].p, ib_, cudaMemcpyDeviceToHost, st));
      }
      return finish_sync(a, st);
    }
    const size_t ctrl_bytes = static_cast<size_t>(a->ctrl_passes) * CTRL_STRIDE * 4;
    CKS(a->h_out.ensure(per * n_db + ctrl_bytes));
    uint8_t* h = static_cast<uint8_t*>(a->h_out.p);
    for (int i = 0; i < n_db; ++i) {
      CK(cudaMemcpyAsync(h + per * i, a->I_stage[i].p, ib_, cudaMemcpyDeviceToHost, st));
      CK(cudaMemcpyAsync(h + per * i + ib_, a->D_stage[i].p, db_, cudaMemcpyDeviceToHost, st));
    }
    uint32_t* hall = reinterpret_cast<uint32_t*>(h + per * n_db);
    memset(hall, 0, ctrl_bytes);
    if (a->ctrl.p) CK(cudaMemcpyAsync(hall, a->ctrl.p, ctrl_bytes, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (int i = 0; i < n_db; ++i) {
      memcpy(I[i], h + per * i, ib_);
      memcpy(D[i], h + per * i + ib_, db_);
    }
    return fold_status(a, hall);
  }
  return 0;
}

}  // namespace

extern "C" {

const char* keds_last_error(void) { return g_err.c_str(); }
const char* keds_version(void) { return "keds-knn-b200 0.2 (sm_100a)"; }

int keds_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int keds_index_create(int d, int metric, int device, keds_index_t** out) {
  if (!out) return fail(KEDS_ERR_ARG, "create: out is null");
  *out = nullptr;
  if (d <= 0 || d > 16384) return fail(KEDS_ERR_ARG, "create: bad dimension %d", d);
  if (metric != KEDS_METRIC_IP && metric != KEDS_METRIC_L2)
    return fail(KEDS_ERR_ARG, "create: metric must be 0 (IP) or 1 (L2)");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(KEDS_ERR_NO_GPU, "no CUDA device: libkeds_knn has no CPU fallback");
  }
  if (device < 0 || device >= ndev) return fail(KEDS_ERR_ARG, "create: device %d of %d", device, ndev);
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(KEDS_ERR_NO_GPU, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                prop.major, prop.minor);
  DeviceGuard g(device);
  if (!g.ok) return fail(KEDS_ERR_NO_GPU, "cannot select CUDA device %d", device);
  keds_index* ix = new keds_index();
  ix->d = d;
  ix->d_pad = (d + BK - 1) / BK * BK;
  ix->metric = metric;
  ix->device = device;
  ix->num_sms = prop.multiProcessorCount;
  memset(&ix->stats, 0, sizeof ix->stats);
  if (const char* op = getenv("KEDS_OPERAND")) {  // "bf16" / "fp16" pin the operand format; default: automatic
    if (!strcmp(op, "bf16")) ix->fmt_forced = FMT_BF16;
    if (!strcmp(op, "fp16")) ix->fmt_forced = FMT_FP16;
  }
  int s = ix->dbstat.ensure(16);
  if (s == 0 && cudaMemset(ix->dbstat.p, 0, 16) != cudaSuccess) s = fail(KEDS_ERR_CUDA, "memset failed");
  if (s == 0) s = ix->probe.ensure(16);
  if (s == 0) {
    void* h = nullptr;
    if (cudaHostAlloc(&h, 64, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess)
      s = fail(KEDS_ERR_CUDA, "cudaHostAlloc of the feedback word failed");
    else {
      memset(h, 0, 64);
      ix->h_feedback = static_cast<unsigned int*>(h);
    }
  }
  if (s != 0) {
    keds_index_free(ix);
    return s;
  }
  // every buffer whose address a captured search bakes in reports its moves
  DevBuf* tracked[] = {&ix->x_f32, &ix->x_bf16, &ix->bias, &ix->q_f32, &ix->q_bf16, &ix->qstat, &ix->cand,
                       &ix->cand_cnt, &ix->cand_theta, &ix->flagged[0], &ix->flagged[1], &ix->ctrl,
                       &ix->exact_scratch, &ix->D_stage[0], &ix->D_stage[1], &ix->I_stage[0], &ix->I_stage[1],
                       &ix->rk, &ix->theta0, &ix->ex_rows, &ix->rg_thr, &ix->rg_cand, &ix->rg_key,
                       &ix->rg_qcnt, &ix->rg_off, &ix->rg_word, &ix->rg_lims, &ix->rg_D, &ix->rg_I};
  for (DevBuf* b : tracked) b->gen = &ix->generation;
  *out = ix;
  return 0;
}

void keds_index_free(keds_index_t* ix) {
  if (!ix) return;
  DeviceGuard g(ix->device);
  DevBuf* bufs[] = {&ix->x_f32, &ix->x_bf16, &ix->bias, &ix->dbstat, &ix->q_f32, &ix->q_bf16,
                    &ix->qstat, &ix->cand, &ix->cand_cnt, &ix->cand_theta, &ix->flagged[0],
                    &ix->flagged[1], &ix->ctrl, &ix->exact_scratch, &ix->D_stage[0], &ix->D_stage[1],
                    &ix->I_stage[0], &ix->I_stage[1], &ix->timing, &ix->probe, &ix->rk, &ix->theta0,
                    &ix->ex_rows, &ix->rg_thr, &ix->rg_cand, &ix->rg_key, &ix->rg_qcnt, &ix->rg_off,
                    &ix->rg_word, &ix->rg_lims, &ix->rg_D, &ix->rg_I};
  for (DevBuf* b : bufs) b->release();
  ix->h_q.release();
  ix->h_out.release();
  if (ix->h_feedback) cudaFreeHost(ix->h_feedback);
  delete ix;
}

int keds_index_add(keds_index_t* ix, const float* x, int64_t n) { return keds_index_add_ex(ix, x, n, 0u); }

int keds_index_get_rows(const keds_index_t* ix, int64_t first, int64_t n, float* out) {
  if (!ix || !out || first < 0 || n < 0 || first + n > ix->n)
    return fail(KEDS_ERR_ARG, "get_rows: bad range [%lld, %lld) of %lld rows", (long long)first,
                (long long)(first + n), (long long)(ix ? ix->n : 0));
  if (n == 0) return 0;
  DeviceGuard g(ix->device);
  CK(cudaMemcpy(out, ix->x_f32.as<float>() + first * ix->d, static_cast<size_t>(n) * ix->d * 4,
                cudaMemcpyDefault));
  return 0;
}

// Operand format from what the rows look like (running maxima over every add): fp16 when nothing
// comes near its range limit and it keeps more of the rows than bf16 does (always the case for
// unit-norm embeddings: 11 significant bits against 8), bf16 otherwise.
static int choose_format(const keds_index* ix) {
  if (ix->fmt_forced >= 0) return ix->fmt_forced;
  return (ix->amax < 3.0e4f && ix->res_fp16 <= ix->res_bf16) ? FMT_FP16 : FMT_BF16;
}

// (re)build the 16-bit operand copy, the L2 bias and the certificate statistics of rows [r0, r1)
static int prep_db_rows(keds_index* ix, int64_t r0, int64_t r1) {
  const size_t d = ix->d, dp = ix->d_pad;
  const int64_t n = r1 - r0;
  const unsigned blocks = static_cast<unsigned>(std::min<int64_t>((n * 32 + 255) / 256, ix->num_sms * 16));
  PrepParams pp;
  memset(&pp, 0, sizeof pp);
  pp.x = ix->x_f32.as<float>() + r0 * d;
  pp.n = n;
  pp.d = ix->d;
  pp.d_pad = ix->d_pad;
  pp.fmt = ix->fmt;
  pp.out = ix->x_bf16.as<uint16_t>() + r0 * dp;
  pp.bias = ix->bias.as<float>() + r0;
  pp.gmax = ix->dbstat.as<unsigned int>();
  k_prep_rows<<<blocks, 256>>>(pp);
  CK(cudaGetLastError());
  return 0;
}

int keds_index_add_ex(keds_index_t* ix, const float* x, int64_t n, uint32_t flags) {
  if (!ix || (n > 0 && !x) || n < 0) return fail(KEDS_ERR_ARG, "add: null handle/data or negative n");
  if (n == 0) return 0;
  DeviceGuard g(ix->device);
  if (!g.ok) return fail(KEDS_ERR_NO_GPU, "cannot select CUDA device %d", ix->device);
  const int64_t n0 = ix->n, n1 = n0 + n;
  if (n1 > 0x7fffffffll - BN) return fail(KEDS_ERR_ARG, "add: more than 2^31 rows");
  const size_t d = ix->d, dp = ix->d_pad;
  const int64_t cap_rows = n0 == 0 ? n1 : std::max<int64_t>(n1, n0 + n0 / 2);
  const int64_t tiles_cap = (cap_rows + BN - 1) / BN;
  if (static_cast<size_t>(n1) * d * 4 > ix->x_f32.cap) {
    CKS(ix->x_f32.grow_keep(static_cast<size_t>(cap_rows) * d * 4, static_cast<size_t>(n0) * d * 4));
    CKS(ix->x_bf16.grow_keep(static_cast<size_t>(cap_rows) * dp * 2, static_cast<size_t>(n0) * dp * 2));
    CKS(ix->bias.grow_keep(static_cast<size_t>(tiles_cap) * BN * 4, static_cast<size_t>(n0) * 4));
  }
  CK(cudaMemcpy(ix->x_f32.as<float>() + n0 * d, x, static_cast<size_t>(n) * d * 4, cudaMemcpyDefault));
  const unsigned blocks = static_cast<unsigned>(std::min<int64_t>((n * 32 + 255) / 256, ix->num_sms * 16));
  if (flags & KEDS_ADD_NORMALIZE) k_normalize_rows<<<blocks, 256>>>(ix->x_f32.as<float>() + n0 * d, n, ix->d);
  // which 16-bit format keeps more of these rows (one extra read of the upload)
  {
    CK(cudaMemset(ix->probe.p, 0, 16));
    k_probe_rows<<<blocks, 256>>>(ix->x_f32.as<float>() + n0 * d, n, ix->d, ix->probe.as<unsigned int>());
    CK(cudaGetLastError());
    float h[4] = {0.f, 0.f, 0.f, 0.f};
    CK(cudaMemcpy(h, ix->probe.p, 12, cudaMemcpyDeviceToHost));
    ix->amax = std::max(ix->amax, h[0]);
    ix->res_bf16 = std::max(ix->res_bf16, h[1]);
    ix->res_fp16 = std::max(ix->res_fp16, h[2]);
  }
  const int want = choose_format(ix);
  if (n0 > 0 && want != ix->fmt) {
    // rows added earlier were rounded to the other format: redo them from the fp32 master
    ix->fmt = want;
    CK(cudaMemset(ix->dbstat.p, 0, 16));
    CKS(prep_db_rows(ix, 0, n1));
  } else {
    ix->fmt = want;
    CKS(prep_db_rows(ix, n0, n1));
  }
  const int64_t padded = (n1 + BN - 1) / BN * BN;
  if (padded > n1)
    k_fill_f32<<<static_cast<unsigned>((padded - n1 + 255) / 256), 256>>>(ix->bias.as<float>() + n1,
                                                                          padded - n1, -INFINITY);
  CK(cudaGetLastError());
  CK(cudaDeviceSynchronize());
  ix->n = n1;
  CKS(encode_rows_map(&ix->tm_x, ix->x_bf16.p, n1, ix->d_pad, BN, ix->fmt));
  CKS(encode_rows_map(&ix->tm_xh, ix->x_bf16.p, n1, ix->d_pad, BN / 2, ix->fmt));
  ix->tm_x_ok = true;
  ix->generation++;  // the row count and the tensor maps are part of what a captured search holds
  return 0;
}

int keds_index_operand_format(const keds_index_t* ix) { return ix ? ix->fmt : -1; }

int keds_index_set_operand_format(keds_index_t* ix, int fmt) {
  if (!ix || fmt < -1 || fmt > FMT_FP16) return fail(KEDS_ERR_ARG, "set_operand_format: fmt must be -1 (auto), 0 (bf16) or 1 (fp16)");
  DeviceGuard g(ix->device);
  if (!g.ok) return fail(KEDS_ERR_NO_GPU, "cannot select CUDA device %d", ix->device);
  ix->fmt_forced = fmt;
  const int want = choose_format(ix);
  if (want == ix->fmt) return 0;
  ix->fmt = want;
  ix->generation++;
  if (ix->n == 0) return 0;
  CK(cudaDeviceSynchronize());
  CK(cudaMemset(ix->dbstat.p, 0, 16));
  CKS(prep_db_rows(ix, 0, ix->n));
  CK(cudaDeviceSynchronize());
  CKS(encode_rows_map(&ix->tm_x, ix->x_bf16.p, ix->n, ix->d_pad, BN, ix->fmt));
  CKS(encode_rows_map(&ix->tm_xh, ix->x_bf16.p, ix->n, ix->d_pad, BN / 2, ix->fmt));
  return 0;
}

uint64_t keds_index_generation(const keds_index_t* ix) { return ix ? ix->generation : 0; }

int keds_index_reset(keds_index_t* ix) {
  if (!ix) return fail(KEDS_ERR_ARG, "reset: null handle");
  DeviceGuard g(ix->device);
  CK(cudaDeviceSynchronize());
  ix->x_f32.release();
  ix->x_bf16.release();
  ix->bias.release();
  ix->n = 0;
  ix->tm_x_ok = false;
  ix->amax = ix->res_bf16 = ix->res_fp16 = 0.f;
  ix->generation++;
  CK(cudaMemset(ix->dbstat.p, 0, 16));
  return 0;
}

int64_t keds_index_ntotal(const keds_index_t* ix) { return ix ? ix->n : -1; }
int keds_index_dim(const keds_index_t* ix) { return ix ? ix->d : -1; }
int keds_index_metric(const keds_index_t* ix) { return ix ? ix->metric : -1; }
int keds_index_device(const keds_index_t* ix) { return ix ? ix->device : -1; }
const float* keds_index_rows(const keds_index_t* ix) { return ix ? ix->x_f32.as<float>() : nullptr; }

int keds_index_set_id_offset(keds_index_t* ix, int64_t offset) {
  if (!ix) return fail(KEDS_ERR_ARG, "set_id_offset: null handle");
  ix->id_offset = offset;
  return 0;
}

int keds_index_set_pdl(keds_index_t* ix, int enable) {
  if (!ix) return fail(KEDS_ERR_ARG, "set_pdl: null handle");
  DeviceGuard g(ix->device);
  CKS(set_kernel_attrs(ix));
  ix->use_pdl = enable != 0;
  return 0;
}

int keds_index_set_eps_scale(keds_index_t* ix, float scale) {
  if (!ix || !(scale >= 0.f)) return fail(KEDS_ERR_ARG, "set_eps_scale: bad argument");
  ix->eps_scale = scale;
  return 0;
}

int keds_index_search(keds_index_t* ix, const float* q, int64_t nq, int k, float* D, int64_t* I,
                      void* stream) {
  return keds_index_search_ex(ix, q, nq, k, D, I, nullptr, 0, 0u, stream);
}

int keds_index_search_ex(keds_index_t* ix, const float* q, int64_t nq, int k, float* D, int64_t* I,
                         const int64_t* exclude, int n_exclude, uint32_t flags, void* stream) {
  Call c = call(1, ix, nullptr, q, nq, k, D, I, nullptr, nullptr, flags);
  CKS(c.exclude(exclude, n_exclude));
  return search_impl(c, IO_HOST, stream);
}

int keds_index_search2(keds_index_t* a, keds_index_t* b, const float* q, int64_t nq, int k, float* Da,
                       int64_t* Ia, float* Db, int64_t* Ib, const int64_t* exclude, int n_exclude, uint32_t flags,
                       void* stream) {
  Call c = call(2, a, b, q, nq, k, Da, Ia, Db, Ib, flags);
  CKS(c.exclude(exclude, n_exclude));
  return search_impl(c, IO_HOST, stream);
}

}  // extern "C"

namespace {

// The fused consumer's description (enabled: something to consume); `fn` names the entry point in
// the refusals of its limits.
int consume_params(const char* fn, const keds_index* img, int k, const int32_t* perm_img, const int32_t* perm_txt,
                   int pool_mode, float tau, float* feat_img, float* feat_txt, float* pool_img, float* pool_txt,
                   ConsumeParams& cp) {
  if (pool_mode < 0 || pool_mode > 2) return fail(KEDS_ERR_ARG, "%s: pool_mode must be 0, 1 or 2", fn);
  if (k > 1024) return fail(KEDS_ERR_ARG, "%s: k=%d too large for the fused consumer", fn, k);
  const bool want_pool = pool_mode != 0 && (pool_img || pool_txt);
  memset(&cp, 0, sizeof cp);
  cp.enabled = (feat_img || feat_txt || want_pool) ? 1 : 0;
  cp.mode = want_pool ? pool_mode : 0;
  cp.tau = tau;
  cp.perm[0] = perm_img;
  cp.perm[1] = perm_txt;
  cp.feat[0] = feat_img;
  cp.feat[1] = feat_txt;
  cp.pool[0] = want_pool ? pool_img : nullptr;
  cp.pool[1] = want_pool ? pool_txt : nullptr;
  // one warp per neighbour row; per-warp partial pools meet in shared memory ([warps][d/4] float4)
  static_assert(RERANK_THREADS == EXACT_THREADS, "the consumer scratch is sized for one block shape");
  cp.part4 = (img->d & 3) == 0 ? (RERANK_THREADS / 32) * (img->d >> 2) : 0;
  return 0;
}

}  // namespace

extern "C" {

// The fused consumer on top of the two-database search, always on the mapped route: device queries
// and labels are used in place, page-locked host ones are read through the mapping.
int keds_retrieve2(keds_index_t* img, keds_index_t* txt, const float* q, int64_t nq, int k,
                   const int32_t* perm_img, const int32_t* perm_txt, int pool_mode, float tau,
                   float* D_img, int64_t* I_img, float* D_txt, int64_t* I_txt, float* Dh_img,
                   int64_t* Ih_img, float* Dh_txt, int64_t* Ih_txt, float* feat_img, float* feat_txt,
                   float* pool_img, float* pool_txt, const int64_t* exclude, int n_exclude, uint32_t flags,
                   void* stream) {
  Call c = call(2, img, txt, q, nq, k, D_img, I_img, D_txt, I_txt, flags);
  CKS(c.exclude(exclude, n_exclude));
  if (!img || !txt || !q || !D_img || !I_img || !D_txt || !I_txt)
    return fail(KEDS_ERR_ARG, "retrieve2: null handle, query or result pointer");
  ConsumeParams cp;
  CKS(consume_params("retrieve2", img, k, perm_img, perm_txt, pool_mode, tau, feat_img, feat_txt, pool_img, pool_txt,
                     cp));
  if (!locate(D_img) || !locate(I_img) || !locate(D_txt) || !locate(I_txt))
    return fail(KEDS_ERR_ARG, "retrieve2: D and I must be device memory");
  if ((Dh_img == nullptr) != (Ih_img == nullptr) || (Dh_txt == nullptr) != (Ih_txt == nullptr))
    return fail(KEDS_ERR_ARG, "retrieve2: a host mirror needs both its D and its I block");
  {
    DeviceGuard g(img->device);
    if (!g.ok) return fail(KEDS_ERR_NO_GPU, "cannot select CUDA device %d", img->device);
    // the host mirrors: written through their device aliases
    void* mirror[4] = {Dh_img, Ih_img, Dh_txt, Ih_txt};
    for (void*& m : mirror) {
      if (!m) continue;
      m = locate(m).mapped;
      if (!m) return fail(KEDS_ERR_ARG, "retrieve2: a host result pointer is not page-locked (cudaHostAlloc / pin_memory)");
    }
    cp.host_D[0] = static_cast<float*>(mirror[0]);
    cp.host_I[0] = static_cast<long long*>(mirror[1]);
    cp.host_D[1] = static_cast<float*>(mirror[2]);
    cp.host_I[1] = static_cast<long long*>(mirror[3]);
  }
  if (Dh_img || Dh_txt) cp.enabled = 1;  // the host mirrors are the consumer's too
  if (cp.enabled) c.cons = cp;
  return search_impl(c, IO_MAPPED, stream);
}

int keds_index_sync(keds_index_t* ix, void* stream) {
  if (!ix) return fail(KEDS_ERR_ARG, "sync: null handle");
  DeviceGuard g(ix->device);
  return finish_sync(ix, static_cast<cudaStream_t>(stream));
}

int keds_index_set_profiling(keds_index_t* ix, int enable) {
  if (!ix) return fail(KEDS_ERR_ARG, "set_profiling: null handle");
  if (enable != 0 && enable != 1) return fail(KEDS_ERR_ARG, "set_profiling: mode must be 0 (off) or 1 (in-kernel timer)");
  DeviceGuard g(ix->device);
  ix->timing_on = enable == 1;  // in-kernel timer of the scoring kernel, launch chain untouched
  ix->timing_launches = 0;
  if (ix->timing_on) {
    const size_t words = TIMING_RING * TIMING_PAIRS * 2;
    CKS(ix->timing.ensure(words * 8));
    std::vector<unsigned long long> init(words);
    for (size_t i = 0; i < words; i += 2) {
      init[i] = ~0ull;
      init[i + 1] = 0ull;
    }
    CK(cudaMemcpy(ix->timing.p, init.data(), words * 8, cudaMemcpyHostToDevice));
  }
  return 0;
}

int keds_index_profile_chain(keds_index_t* ix, double* dur_ms, double* gap_ms, int64_t* searches, int n) {
  if (!ix || !dur_ms || !gap_ms || !searches || n < static_cast<int>(TIMING_PAIRS))
    return fail(KEDS_ERR_ARG, "profile_chain: need room for %d kernels", (int)TIMING_PAIRS);
  if (!ix->timing_on) return fail(KEDS_ERR_ARG, "profile_chain: call set_profiling(1) first");
  DeviceGuard g(ix->device);
  CK(cudaDeviceSynchronize());
  const size_t words = TIMING_RING * TIMING_PAIRS * 2;
  std::vector<unsigned long long> t(words);
  CK(cudaMemcpy(t.data(), ix->timing.p, words * 8, cudaMemcpyDeviceToHost));
  const size_t used = std::min(ix->timing_launches, TIMING_RING);
  double dur[TIMING_PAIRS] = {0}, gap[TIMING_PAIRS] = {0};
  int64_t nd[TIMING_PAIRS] = {0}, ng[TIMING_PAIRS] = {0};
  for (size_t s = 0; s < used; ++s) {
    const unsigned long long* c = t.data() + s * TIMING_PAIRS * 2;
    unsigned long long prev_end = 0;
    for (size_t i = 0; i < TIMING_PAIRS; ++i) {
      const unsigned long long b = c[2 * i], e = c[2 * i + 1];
      if (e <= b || b == ~0ull) continue;  // kernel not part of this search
      dur[i] += static_cast<double>(e - b) * 1e-6;
      nd[i]++;
      if (prev_end != 0 && b >= prev_end) {
        gap[i] += static_cast<double>(b - prev_end) * 1e-6;
        ng[i]++;
      } else if (prev_end != 0) {
        ng[i]++;  // overlapped its predecessor (programmatic launch): gap 0
      }
      prev_end = e;
    }
  }
  for (size_t i = 0; i < TIMING_PAIRS; ++i) {
    dur_ms[i] = nd[i] ? dur[i] / nd[i] : 0.0;
    gap_ms[i] = ng[i] ? gap[i] / ng[i] : 0.0;
  }
  *searches = static_cast<int64_t>(used);
  return 0;
}

int keds_index_profile(keds_index_t* ix, double* score_ms_total, int64_t* score_launches) {
  if (!ix || !score_ms_total || !score_launches) return fail(KEDS_ERR_ARG, "profile: null argument");
  double dur[TIMING_PAIRS], gap[TIMING_PAIRS];
  int64_t n = 0;
  CKS(keds_index_profile_chain(ix, dur, gap, &n, TIMING_PAIRS));
  *score_ms_total = dur[1] * static_cast<double>(n);
  *score_launches = n;
  return keds_index_set_profiling(ix, 1);  // re-arm the ring
}

int keds_index_last_stats(const keds_index_t* ix, keds_search_stats* out) {
  if (!ix || !out) return fail(KEDS_ERR_ARG, "last_stats: null argument");
  *out = ix->stats;
  return 0;
}

int keds_debug_scores(keds_index_t* ix, const float* q, int64_t nq, float* out, void* stream) {
  if (!ix || !q || !out || nq <= 0 || nq > Q_PASS_MAX) return fail(KEDS_ERR_ARG, "debug_scores: bad argument");
  if (!locate(q) || !locate(out)) return fail(KEDS_ERR_ARG, "debug_scores: device pointers only");
  if (ix->n == 0) return fail(KEDS_ERR_ARG, "debug_scores: empty index");
  DeviceGuard g(ix->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  memset(&ix->stats, 0, sizeof ix->stats);
  Call c = call(1, ix, nullptr, q, nq, 1, nullptr, nullptr, nullptr, nullptr, 0u);
  c.dump = out;
  c.ld_dump = ix->n;
  CKS(run_passes(c, st));
  return finish_sync(ix, st);
}

int keds_debug_plan(int n_db, int64_t nq, int k, int64_t n_rows, int num_sms, int32_t out[6]) {
  if (!out || n_db < 1 || n_db > 2 || nq <= 0 || k <= 0 || n_rows <= 0 || num_sms <= 0)
    return fail(KEDS_ERR_ARG, "debug_plan: bad argument");
  keds_index ix;  // never touches the device: only the planner's inputs are read
  ix.num_sms = num_sms;
  const char* no_pair = getenv("KEDS_NO_PAIR");
  ix.use_pair = !(no_pair && no_pair[0] == '1');
  const Plan pl = make_plan(&ix, n_db, nq, k, n_rows, n_rows, 0u);
  out[0] = pl.exact_only;
  out[1] = pl.pair ? 1 : 0;
  out[2] = pl.S;
  out[3] = pl.n_qt;
  out[4] = pl.n_items;
  out[5] = pl.grid;
  return 0;
}

int keds_gather_pool(const float* base, int64_t n_base, const int64_t* I, const float* W,
                     const int32_t* perm, int64_t B, int k, int H, int d, float* out, void* stream) {
  if (!base || !I || !out || B < 0 || k <= 0 || d <= 0 || n_base < 0)
    return fail(KEDS_ERR_ARG, "gather_pool: bad argument");
  if (B == 0) return 0;
  const int dev = locate(out).device;
  if (dev < 0 || locate(base).device != dev) return fail(KEDS_ERR_ARG, "gather_pool: base and out must be memory of one device");
  DeviceGuard g(dev);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!W) {
    const long long warps = static_cast<long long>(B) * k;
    k_gather_rows<<<static_cast<unsigned>((warps * 32 + 255) / 256), 256, 0, st>>>(
        base, static_cast<long long>(n_base), reinterpret_cast<const long long*>(I), perm, B, k, d, out);
  } else {
    if (H <= 0) return fail(KEDS_ERR_ARG, "gather_pool: H must be positive with weights");
    const size_t smem = static_cast<size_t>(k) * 8 + static_cast<size_t>(H) * k * 4;
    if (smem > 48 * 1024) return fail(KEDS_ERR_ARG, "gather_pool: H*k too large");
    k_weighted_pool<<<static_cast<unsigned>(B), 256, smem, st>>>(
        base, static_cast<long long>(n_base), reinterpret_cast<const long long*>(I), W, B, k, H, d, out);
  }
  CK(cudaGetLastError());
  return 0;
}

int keds_topk_merge(const float* Dp, const int64_t* Ip, int parts, int64_t nq, int k, int metric,
                    float* D, int64_t* I, void* stream) {
  return keds_topk_merge_strided(Dp, Ip, nq * k, nq * k, parts, nq, k, metric, D, I, stream);
}

static int merge_impl(const float* Dp, const int64_t* Ip, int64_t stride_d, int64_t stride_i, int parts,
                      int64_t nq, int k, int metric, float* D, int64_t* I, const MergeWait& mw,
                      void* stream) {
  if (!Dp || !Ip || !D || !I || parts <= 0 || nq < 0 || k <= 0)
    return fail(KEDS_ERR_ARG, "topk_merge: bad argument");
  if (nq == 0) return 0;
  const size_t tot = static_cast<size_t>(parts) * k;
  const size_t smem = tot * 8 + tot * 4;  // labels, rank scores
  if (smem > 200 * 1024) return fail(KEDS_ERR_ARG, "topk_merge: parts*k too large");
  const int dev = locate(D).device;
  if (dev < 0) return fail(KEDS_ERR_ARG, "topk_merge: device pointers only");
  DeviceGuard g(dev);
  // the attribute is per device; IndexShards / IndexReplicas search from one host thread per GPU
  static std::atomic<bool> attr[64];
  if (dev >= 64 || !attr[dev].load(std::memory_order_acquire)) {
    CK(cudaFuncSetAttribute(k_topk_merge, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    if (dev < 64) attr[dev].store(true, std::memory_order_release);
  }
  // launched behind the local search / the push kernel with the programmatic attribute: its
  // launch latency hides under their tails (it starts with griddepcontrol.wait)
  CKS(launch_k(true, k_topk_merge, dim3(static_cast<unsigned>(nq)), dim3(128), smem,
               static_cast<cudaStream_t>(stream), Dp, reinterpret_cast<const long long*>(Ip),
               static_cast<long long>(stride_d), static_cast<long long>(stride_i), parts,
               static_cast<long long>(nq), k, metric, D, reinterpret_cast<long long*>(I), mw));
  return 0;
}

int keds_topk_merge_strided(const float* Dp, const int64_t* Ip, int64_t stride_d, int64_t stride_i,
                            int parts, int64_t nq, int k, int metric, float* D, int64_t* I,
                            void* stream) {
  MergeWait mw;
  memset(&mw, 0, sizeof mw);
  return merge_impl(Dp, Ip, stride_d, stride_i, parts, nq, k, metric, D, I, mw, stream);
}

int keds_p2p_push(const void* src, int64_t bytes, void* const* peer_dst, uint32_t* const* peer_flag,
                  int n_ranks, int my_rank, uint32_t epoch, uint32_t* ticket, void* stream) {
  if (!src || !peer_dst || !peer_flag || !ticket || bytes <= 0 || (bytes & 15) || n_ranks < 1 ||
      n_ranks > P2P_MAX_RANKS || my_rank < 0 || my_rank >= n_ranks)
    return fail(KEDS_ERR_ARG, "p2p_push: bad argument (bytes must be a positive multiple of 16, <= %d ranks)",
                P2P_MAX_RANKS);
  P2PPush p;
  memset(&p, 0, sizeof p);
  p.n_ranks = n_ranks;
  p.my_rank = my_rank;
  p.epoch = epoch;
  p.n16 = bytes / 16;
  p.src = static_cast<const uint4*>(src);
  for (int r = 0; r < n_ranks; ++r) {
    p.dst[r] = static_cast<uint4*>(peer_dst[r]);
    p.flag[r] = peer_flag[r];
    if (r != my_rank && (!p.dst[r] || !p.flag[r])) return fail(KEDS_ERR_ARG, "p2p_push: null peer pointer");
  }
  p.ticket = ticket;
  const int dev = locate(src).device;
  if (dev < 0) return fail(KEDS_ERR_ARG, "p2p_push: src must be device memory");
  DeviceGuard g(dev);
  const unsigned blocks = static_cast<unsigned>(std::min<long long>(64, (p.n16 + 255) / 256));
  CKS(launch_k(true, k_p2p_push, dim3(std::max(1u, blocks)), dim3(256), 0, static_cast<cudaStream_t>(stream), p));
  return 0;
}

int keds_topk_merge_wait(const float* Dp, const int64_t* Ip, int64_t stride_d, int64_t stride_i, int parts,
                         int64_t nq, int k, int metric, float* D, int64_t* I, const uint32_t* flags,
                         int my_rank, uint32_t epoch, uint32_t* err_word, void* stream) {
  if (!flags || !err_word || my_rank < 0 || my_rank >= parts)
    return fail(KEDS_ERR_ARG, "topk_merge_wait: bad argument");
  MergeWait mw;
  memset(&mw, 0, sizeof mw);
  mw.flags = flags;
  mw.my_rank = my_rank;
  mw.epoch = epoch;
  mw.err_word = err_word;
  return merge_impl(Dp, Ip, stride_d, stride_i, parts, nq, k, metric, D, I, mw, stream);
}

// ---- row-sharded search with the exchange fused into the search kernels ------------------------
struct keds_exchange {
  int n_ranks = 0, my_rank = 0, device = 0;
  uint8_t* base[P2P_MAX_RANKS] = {nullptr};  // rank r's symmetric buffer as mapped into this process
  int64_t buf_bytes = 0, slot_bytes = 0, i_off = 0;
  uint32_t epoch = 0;
  DevBuf words;  // [0] ticket, [1] error word, [2..3] pad, then {sum, max, count} wait statistics (u64)
  // every rank's fp32 rows per database (keds_exchange_attach_rows): the sharded consumer reads them
  // in place. opened: a peer mapping this handle owns (cudaIpcCloseMemHandle on re-attach and free).
  bool attached[2] = {false, false};
  ShardRowsDb rows[2];
  bool opened[2][P2P_MAX_RANKS] = {};
};

namespace {
constexpr int64_t EX_FLAG_BYTES = 256;  // 2 parities x P2P_MAX_RANKS flag words at the start of every buffer
uint8_t* ex_slot(const keds_exchange* ex, int owner, int parity, int r) {
  return ex->base[owner] + EX_FLAG_BYTES + (static_cast<int64_t>(parity) * ex->n_ranks + r) * ex->slot_bytes;
}
uint32_t* ex_flag(const keds_exchange* ex, int owner, int parity, int r) {
  return reinterpret_cast<uint32_t*>(ex->base[owner]) + parity * P2P_MAX_RANKS + r;
}

// Handles keds_index_rows_ipc gave out in this process, with the rows they name: a process cannot
// open its own handle, so attach_rows finds its own rank's pointer here.
struct IpcExport {
  cudaIpcMemHandle_t h;
  const float* rows;
};
std::mutex g_ipc_mu;
std::vector<IpcExport> g_ipc;

void ex_detach_rows(keds_exchange* ex, int db) {
  for (int r = 0; r < P2P_MAX_RANKS; ++r) {
    if (ex->opened[db][r]) cudaIpcCloseMemHandle(const_cast<float*>(ex->rows[db].base[r]));
    ex->opened[db][r] = false;
  }
  memset(&ex->rows[db], 0, sizeof ex->rows[db]);
  ex->attached[db] = false;
}

// Every database of a sharded call must be attached and this rank's rows where they were then.
int ex_check_rows(const keds_exchange* ex, keds_index* const* dbs, int n_db) {
  for (int i = 0; i < n_db; ++i) {
    const ShardRowsDb& rd = ex->rows[i];
    const int me = ex->my_rank;
    if (!ex->attached[i])
      return fail(KEDS_ERR_ARG, "sharded: database %d has no rows attached to the exchange", i);
    if (rd.n[me] != dbs[i]->n || rd.lo[me] != dbs[i]->id_offset ||
        (dbs[i]->n > 0 && rd.base[me] != dbs[i]->x_f32.as<float>()))
      return fail(KEDS_ERR_ARG,
                  "sharded: the rows of database %d changed since keds_exchange_attach_rows "
                  "(re-attach on every rank after each add)", i);
  }
  return 0;
}

// The local search of a row-sharded call (c: this rank's handles, the queries, flags and exclusion)
// with every finished result row pushed to the peers, then one merge per database into D[i] / I[i].
// Database i's [nq][k] blocks sit at i * nq * k in the D and I halves of the exchange slot.
int sharded_search(Call c, keds_exchange* ex, float* const* D, int64_t* const* I, void* stream) {
  const int64_t nq = c.nq, blk = c.nq * c.k;
  if (c.n_db * blk > ex->i_off / 4)
    return fail(KEDS_ERR_ARG, "sharded: %d x nq*k = %lld exceeds the exchange capacity %lld", c.n_db,
                (long long)(c.n_db * blk), (long long)(ex->i_off / 4));
  if (c.flags & KEDS_SEARCH_NO_FALLBACK)
    return fail(KEDS_ERR_ARG, "sharded: KEDS_SEARCH_NO_FALLBACK is not supported (the fallback publishes the step)");
  keds_index* ix = c.owner;
  DeviceGuard g(ix->device);
  if (!g.ok) return fail(KEDS_ERR_NO_GPU, "cannot select CUDA device %d", ix->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const uint32_t epoch = ++ex->epoch;
  const int parity = static_cast<int>(epoch & 1u);
  const int me = ex->my_rank, R = ex->n_ranks;
  // this rank's blocks land in slot `me` of every rank's buffer (its own included: the merge reads them there)
  uint8_t* mine = ex_slot(ex, me, parity, me);
  for (int i = 0; i < c.n_db; ++i) {
    c.D[i] = reinterpret_cast<float*>(mine) + i * blk;
    c.I[i] = reinterpret_cast<long long*>(mine + ex->i_off) + i * blk;
  }
  PeerOut po;
  memset(&po, 0, sizeof po);
  po.n = R;
  po.my_rank = me;
  po.publish = 1;
  po.epoch = epoch;
  po.ticket = ex->words.as<unsigned int>();
  po.db_stride = blk;
  for (int r = 0; r < R; ++r) {
    uint8_t* there = ex_slot(ex, r, parity, me);
    po.D[r] = reinterpret_cast<float*>(there);
    po.I[r] = reinterpret_cast<long long*>(there + ex->i_off);
    po.flag[r] = ex_flag(ex, r, parity, me);
  }
  bool empty = false;
  for (int i = 0; i < c.n_db; ++i) empty = empty || c.dbs[i]->n == 0;
  if (!empty && R > 1) c.peer = po;
  CKS(search_impl(c, IO_DEVICE, stream));
  if (empty && R > 1) {
    // an empty shard database runs no search chain to carry its padding (search_impl has filled it):
    // the whole slot goes out with the stand-alone push, which publishes
    void* dst[P2P_MAX_RANKS];
    uint32_t* flg[P2P_MAX_RANKS];
    for (int r = 0; r < R; ++r) {
      dst[r] = ex_slot(ex, r, parity, me);
      flg[r] = ex_flag(ex, r, parity, me);
    }
    CKS(keds_p2p_push(mine, ex->slot_bytes, dst, flg, R, me, epoch, po.ticket, stream));
  }
  uint8_t* parts = ex_slot(ex, me, parity, 0);
  for (int i = 0; i < c.n_db; ++i) {
    MergeWait mw;
    memset(&mw, 0, sizeof mw);
    if (R > 1) {
      // both merges wait on the step's one set of flags; the first one reports the wait
      mw.flags = ex_flag(ex, me, parity, 0);
      mw.my_rank = me;
      mw.epoch = epoch;
      mw.err_word = ex->words.as<unsigned int>() + 1;
      if (i == 0) mw.stats = reinterpret_cast<unsigned long long*>(ex->words.as<uint8_t>() + 16);
    }
    CKS(merge_impl(reinterpret_cast<const float*>(parts) + i * blk,
                   reinterpret_cast<const int64_t*>(parts + ex->i_off) + i * blk, ex->slot_bytes / 4,
                   ex->slot_bytes / 8, R, nq, c.k, c.metric(), D[i], I[i], mw, stream));
  }
  return 0;
}
}  // namespace

int keds_exchange_create(int n_ranks, int my_rank, int device, void* const* peer_base, int64_t buf_bytes,
                         keds_exchange_t** out) {
  if (!out) return fail(KEDS_ERR_ARG, "exchange_create: out is null");
  *out = nullptr;
  if (n_ranks < 1 || n_ranks > P2P_MAX_RANKS || my_rank < 0 || my_rank >= n_ranks || !peer_base)
    return fail(KEDS_ERR_ARG, "exchange_create: 1..%d ranks, my_rank inside", P2P_MAX_RANKS);
  const int64_t slot = (buf_bytes - EX_FLAG_BYTES) / (2 * n_ranks) / 48 * 48;  // D : I = 1 : 2, both 16-byte aligned
  if (slot < 48) return fail(KEDS_ERR_ARG, "exchange_create: buffer of %lld bytes is too small", (long long)buf_bytes);
  for (int r = 0; r < n_ranks; ++r)
    if (!peer_base[r] || (reinterpret_cast<uintptr_t>(peer_base[r]) & 15))
      return fail(KEDS_ERR_ARG, "exchange_create: peer buffer %d is null or not 16-byte aligned", r);
  DeviceGuard g(device);
  if (!g.ok) return fail(KEDS_ERR_NO_GPU, "cannot select CUDA device %d", device);
  keds_exchange* ex = new keds_exchange();
  ex->n_ranks = n_ranks;
  ex->my_rank = my_rank;
  ex->device = device;
  for (int r = 0; r < n_ranks; ++r) ex->base[r] = static_cast<uint8_t*>(peer_base[r]);
  ex->buf_bytes = buf_bytes;
  ex->slot_bytes = slot;
  ex->i_off = slot / 3;
  memset(ex->rows, 0, sizeof ex->rows);
  int s = ex->words.ensure(64);
  if (s == 0 && cudaMemset(ex->words.p, 0, 64) != cudaSuccess) s = fail(KEDS_ERR_CUDA, "memset failed");
  if (s != 0) {
    ex->words.release();
    delete ex;
    return s;
  }
  *out = ex;
  return 0;
}

void keds_exchange_free(keds_exchange_t* ex) {
  if (!ex) return;
  DeviceGuard g(ex->device);
  for (int db = 0; db < 2; ++db) ex_detach_rows(ex, db);
  ex->words.release();
  delete ex;
}

int64_t keds_exchange_capacity(const keds_exchange_t* ex) { return ex ? ex->i_off / 4 : -1; }

int keds_index_rows_ipc(const keds_index_t* ix, void* handle64) {
  if (!ix || !handle64) return fail(KEDS_ERR_ARG, "index_rows_ipc: null handle or output");
  memset(handle64, 0, sizeof(cudaIpcMemHandle_t));
  if (ix->n == 0) return 0;  // no rows: nothing to map (the all-zero handle)
  DeviceGuard g(ix->device);
  if (!g.ok) return fail(KEDS_ERR_NO_GPU, "cannot select CUDA device %d", ix->device);
  IpcExport e;
  CK(cudaIpcGetMemHandle(&e.h, ix->x_f32.p));
  e.rows = ix->x_f32.as<float>();
  memcpy(handle64, &e.h, sizeof e.h);
  std::lock_guard<std::mutex> lk(g_ipc_mu);
  for (IpcExport& o : g_ipc)
    if (o.rows == e.rows) {
      o = e;
      return 0;
    }
  if (g_ipc.size() >= 256) g_ipc.erase(g_ipc.begin());
  g_ipc.push_back(e);
  return 0;
}

int keds_exchange_attach_rows(keds_exchange_t* ex, int db, const void* const* handles, const int64_t* lo,
                              const int64_t* n) {
  if (!ex || db < 0 || db > 1 || !handles || !lo || !n)
    return fail(KEDS_ERR_ARG, "exchange_attach_rows: null argument or db outside 0..1");
  for (int r = 0; r < ex->n_ranks; ++r)
    if (lo[r] < 0 || n[r] < 0 || (n[r] > 0 && !handles[r]))
      return fail(KEDS_ERR_ARG, "exchange_attach_rows: rank %d has a negative range or no handle", r);
  DeviceGuard g(ex->device);
  if (!g.ok) return fail(KEDS_ERR_NO_GPU, "cannot select CUDA device %d", ex->device);
  ex_detach_rows(ex, db);
  ShardRowsDb& rd = ex->rows[db];
  for (int r = 0; r < ex->n_ranks; ++r) {
    rd.lo[r] = lo[r];
    rd.n[r] = n[r];
    if (n[r] == 0) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, handles[r], sizeof h);
    if (r == ex->my_rank) {
      std::lock_guard<std::mutex> lk(g_ipc_mu);
      for (const IpcExport& e : g_ipc)
        if (!memcmp(&e.h, &h, sizeof h)) rd.base[r] = e.rows;
      if (!rd.base[r]) {
        ex_detach_rows(ex, db);
        return fail(KEDS_ERR_ARG, "exchange_attach_rows: this rank's handle was not made by keds_index_rows_ipc here");
      }
      continue;
    }
    void* p = nullptr;
    const cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      cudaGetLastError();
      ex_detach_rows(ex, db);
      return fail(KEDS_ERR_CUDA, "exchange_attach_rows: cudaIpcOpenMemHandle of rank %d failed: %s", r,
                  cudaGetErrorString(e));
    }
    rd.base[r] = static_cast<const float*>(p);
    ex->opened[db][r] = true;
  }
  ex->attached[db] = true;
  return 0;
}

int keds_index_search_sharded(keds_index_t* ix, keds_exchange_t* ex, const float* q, int64_t nq, int k, float* D,
                              int64_t* I, const int64_t* exclude, int n_exclude, void* stream) {
  Call c = call(1, ix, nullptr, q, nq, k, nullptr, nullptr, nullptr, nullptr, 0u);
  CKS(c.exclude(exclude, n_exclude));
  if (!ix || !ex || !q || !D || !I || nq <= 0 || k <= 0)
    return fail(KEDS_ERR_ARG, "search_sharded: null handle / pointer or bad nq / k");
  if (ex->device != ix->device) return fail(KEDS_ERR_ARG, "search_sharded: exchange and index live on different devices");
  if (!locate(q) || !locate(D) || !locate(I)) return fail(KEDS_ERR_ARG, "search_sharded: device pointers only");
  return sharded_search(c, ex, &D, &I, stream);
}

int keds_retrieve2_sharded(keds_index_t* img, keds_index_t* txt, keds_exchange_t* ex, const float* q, int64_t nq,
                           int k, const int32_t* perm_img, const int32_t* perm_txt, int pool_mode, float tau,
                           int64_t row_lo, int64_t row_hi, float* D_img, int64_t* I_img, float* D_txt,
                           int64_t* I_txt, float* feat_img, float* feat_txt, float* pool_img, float* pool_txt,
                           const int64_t* exclude, int n_exclude, uint32_t flags, void* stream) {
  Call c = call(2, img, txt, q, nq, k, nullptr, nullptr, nullptr, nullptr, flags);
  CKS(c.exclude(exclude, n_exclude));
  if (!img || !txt || !ex || !q || !D_img || !I_img || !D_txt || !I_txt || nq <= 0 || k <= 0)
    return fail(KEDS_ERR_ARG, "retrieve2_sharded: null handle / pointer or bad nq / k");
  ConsumeParams cp;
  CKS(consume_params("retrieve2_sharded", img, k, perm_img, perm_txt, pool_mode, tau, feat_img, feat_txt, pool_img,
                     pool_txt, cp));
  if (row_lo < 0 || row_hi < row_lo || row_hi > nq)
    return fail(KEDS_ERR_ARG, "retrieve2_sharded: rows [%lld, %lld) outside [0, %lld)", (long long)row_lo,
                (long long)row_hi, (long long)nq);
  if (ex->device != img->device || txt->device != img->device)
    return fail(KEDS_ERR_ARG, "retrieve2_sharded: exchange and indices live on different devices");
  const void* dev_ptrs[] = {q, D_img, I_img, D_txt, I_txt, feat_img, feat_txt, cp.pool[0], cp.pool[1], perm_img,
                            perm_txt};
  for (const void* p : dev_ptrs)
    if (p && locate(p).device != img->device)
      return fail(KEDS_ERR_ARG, "retrieve2_sharded: device pointers of the indices' GPU only");
  CKS(ex_check_rows(ex, c.dbs, 2));
  float* D[2] = {D_img, D_txt};
  int64_t* I[2] = {I_img, I_txt};
  CKS(sharded_search(c, ex, D, I, stream));
  const int64_t nb = row_hi - row_lo;
  if (nb == 0 || !cp.enabled) return 0;
  ShardConsume sc;
  memset(&sc, 0, sizeof sc);
  sc.cons = cp;
  sc.n_ranks = ex->n_ranks;
  sc.k = k;
  sc.d = img->d;
  sc.metric = c.metric();
  sc.row_lo = row_lo;
  for (int i = 0; i < 2; ++i) {
    sc.D[i] = D[i];
    sc.I[i] = reinterpret_cast<const long long*>(I[i]);
    sc.db[i] = ex->rows[i];
  }
  const size_t smem = static_cast<size_t>(sc.cons.part4) * 16 + static_cast<size_t>(k) * 20;
  DeviceGuard g(img->device);
  // (with both of this rank's shards empty no search pass ran to set the attributes)
  CKS(set_kernel_attrs(img));
  CKS(launch_k(img->use_pdl, k_shard_consume, dim3(static_cast<unsigned>(nb), 2), dim3(RERANK_THREADS), smem,
               static_cast<cudaStream_t>(stream), sc));
  return 0;
}

int keds_exchange_stats(keds_exchange_t* ex, void* stream, double* wait_us_avg, double* wait_us_max,
                        int64_t* steps, uint32_t* err_word) {
  if (!ex) return fail(KEDS_ERR_ARG, "exchange_stats: null handle");
  DeviceGuard g(ex->device);
  CK(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  uint8_t h[64];
  CK(cudaMemcpy(h, ex->words.p, 64, cudaMemcpyDeviceToHost));
  const uint32_t* w = reinterpret_cast<const uint32_t*>(h);
  const unsigned long long* st = reinterpret_cast<const unsigned long long*>(h + 16);
  if (wait_us_avg) *wait_us_avg = st[2] ? static_cast<double>(st[0]) / static_cast<double>(st[2]) * 1e-3 : 0.0;
  if (wait_us_max) *wait_us_max = static_cast<double>(st[1]) * 1e-3;
  if (steps) *steps = static_cast<int64_t>(st[2]);
  if (err_word) *err_word = w[1];
  CK(cudaMemset(ex->words.as<uint8_t>() + 16, 0, 24));  // statistics restart; ticket and error word stay
  if (w[1] != 0)
    return fail(KEDS_ERR_KERNEL, "sharded exchange: peer %u did not deliver within the watchdog window (error word 0x%x)",
                w[1] - 0x500u, w[1]);
  return 0;
}

int keds_index_range_search(keds_index_t* ix, const float* q, int64_t nq, float radius, int64_t* lims,
                            uint32_t flags, void* stream) {
  if (!ix || !lims || nq < 0 || (nq > 0 && !q)) return fail(KEDS_ERR_ARG, "range_search: null handle/query/lims or nq < 0");
  if (flags & ~KEDS_SEARCH_FORCE_IP) return fail(KEDS_ERR_ARG, "range_search: flags 0x%x; only KEDS_SEARCH_FORCE_IP applies", flags);
  if (radius != radius) return fail(KEDS_ERR_ARG, "range_search: radius is NaN");
  if (ix->n > 0x7fffffffll - BN) return fail(KEDS_ERR_ARG, "index too large for 32-bit row ids");
  DeviceGuard g(ix->device);
  if (!g.ok) return fail(KEDS_ERR_NO_GPU, "cannot select CUDA device %d", ix->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  memset(&ix->stats, 0, sizeof ix->stats);
  ix->rg_total = 0;
  const PtrLoc ll = locate(lims);
  if (ll && ll.device != ix->device) return fail(KEDS_ERR_ARG, "range_search: lims on device %d, index on %d", ll.device, ix->device);
  CKS(ix->rg_lims.ensure(static_cast<size_t>(nq + 1) * 8));
  Call c = call(1, ix, nullptr, q, nq, 1, nullptr, nullptr, nullptr, nullptr, flags);
  c.range.radius = radius;
  c.range.lims = ix->rg_lims.as<long long>();
  if (nq == 0 || ix->n == 0) {
    CK(cudaMemsetAsync(ix->rg_lims.p, 0, static_cast<size_t>(nq + 1) * 8, st));
  } else {
    const PtrLoc lq = locate(q);
    if (lq && lq.device != ix->device) return fail(KEDS_ERR_ARG, "range_search: q on device %d, index on %d", lq.device, ix->device);
    // host queries, and device queries off a 16-byte boundary (warp_exact_score would take its scalar
    // order and so differ from search()), are scored from the handle's copy
    if (!lq || (reinterpret_cast<uintptr_t>(q) & 15) != 0) {
      const size_t qb = static_cast<size_t>(nq) * ix->d * 4;
      CKS(ix->q_f32.ensure(qb));
      CK(cudaMemcpyAsync(ix->q_f32.p, q, qb, cudaMemcpyDefault, st));
      c.q = ix->q_f32.as<float>();
    }
    CKS(run_passes(c, st));
  }
  CK(cudaMemcpyAsync(lims, ix->rg_lims.p, static_cast<size_t>(nq + 1) * 8, cudaMemcpyDefault, st));
  CK(cudaStreamSynchronize(st));
  return 0;
}

int keds_index_range_results(keds_index_t* ix, float* D, int64_t* I, void* stream) {
  if (!ix) return fail(KEDS_ERR_ARG, "range_results: null handle");
  if (ix->rg_total == 0) return 0;
  if (!D || !I) return fail(KEDS_ERR_ARG, "range_results: null output for %lld results", (long long)ix->rg_total);
  DeviceGuard g(ix->device);
  if (!g.ok) return fail(KEDS_ERR_NO_GPU, "cannot select CUDA device %d", ix->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const PtrLoc ld = locate(D), li = locate(I);
  if ((ld && ld.device != ix->device) || (li && li.device != ix->device))
    return fail(KEDS_ERR_ARG, "range_results: outputs on another device than the index");
  const size_t n = static_cast<size_t>(ix->rg_total);
  CK(cudaMemcpyAsync(D, ix->rg_D.p, n * 4, cudaMemcpyDefault, st));
  CK(cudaMemcpyAsync(I, ix->rg_I.p, n * 8, cudaMemcpyDefault, st));
  if (!ld || !li) CK(cudaStreamSynchronize(st));
  return 0;
}

// Gallery ranking against the rows of an index, on the tensor cores: the same scoring kernel with
// a counting epilogue between two small kernels (target scores + error band before, exact
// settlement of the band rows after), and the exact fp32 recount for queries whose band overflowed.
int keds_index_rank(keds_index_t* ix, const float* q, int64_t nq, const int64_t* target, const int64_t* exclude,
                    int64_t* rank_out, void* stream) {
  if (!ix || !q || !target || !rank_out || nq < 0) return fail(KEDS_ERR_ARG, "index_rank: null argument or bad nq");
  if (nq == 0) return 0;
  if (ix->n == 0) return fail(KEDS_ERR_ARG, "index_rank: empty index");
  if (!locate(q) || !locate(target) || !locate(rank_out) || (exclude && !locate(exclude)))
    return fail(KEDS_ERR_ARG, "index_rank: device pointers only");
  DeviceGuard g(ix->device);
  if (!g.ok) return fail(KEDS_ERR_NO_GPU, "cannot select CUDA device %d", ix->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int d = ix->d;
  if (gallery_rank_smem(d) > 48 * 1024) return fail(KEDS_ERR_ARG, "index_rank: d too large");
  const RankMode rm{reinterpret_cast<const long long*>(target), reinterpret_cast<const long long*>(exclude),
                    reinterpret_cast<long long*>(rank_out)};
  if (ix->n <= BN) {
    // less than two row tiles: nothing for the tensor cores to win
    k_gallery_rank<<<static_cast<unsigned>((nq + 7) / 8), 256, gallery_rank_smem(d), st>>>(
        q, nq, ix->x_f32.as<float>(), ix->n, d, rm.target, rm.exclude, rm.out, nullptr, nullptr);
    CK(cudaGetLastError());
    return 0;
  }
  memset(&ix->stats, 0, sizeof ix->stats);
  Call c = call(1, ix, nullptr, q, nq, 0, nullptr, nullptr, nullptr, nullptr, 0u);
  c.rank = rm;
  // warp_exact_score sums in float4 chunks only when q is 16-byte aligned: a query tensor that
  // starts elsewhere is scored from an aligned copy (left by k_prep_rows), so that its ranks do not
  // depend on where it starts and equal those of the recount, which reads q from shared memory
  if ((d & 3) == 0 && (reinterpret_cast<uintptr_t>(q) & 15) != 0) {
    CKS(ix->q_f32.ensure(static_cast<size_t>(nq) * d * 4));
    c.q_src = q;
    c.q = ix->q_f32.as<float>();
  }
  return run_passes(c, st);
}

int keds_index_label_hits(keds_index_t* ix, const float* q, int64_t nq, const int64_t* row_labels,
                          const int64_t* qlabel, const int32_t* ks, int nks, int32_t* hits, void* stream) {
  if (!ix || !q || !row_labels || !qlabel || !ks || !hits || nq < 0 || nks <= 0 || nks > HITS_MAX_CUTS)
    return fail(KEDS_ERR_ARG, "index_label_hits: null argument, bad nq or more than %d cut points", HITS_MAX_CUTS);
  for (int j = 0; j < nks; ++j)
    if (ks[j] <= 0 || (j > 0 && ks[j] <= ks[j - 1])) return fail(KEDS_ERR_ARG, "index_label_hits: ks must be ascending and positive");
  if (ks[nks - 1] > K_MAX) return fail(KEDS_ERR_ARG, "index_label_hits: k=%d exceeds the maximum %d", ks[nks - 1], K_MAX);
  if (nq == 0) return 0;
  if (ix->n == 0) return fail(KEDS_ERR_ARG, "index_label_hits: empty index");
  if (ix->n > 0x7fffffffll - BN) return fail(KEDS_ERR_ARG, "index too large for 32-bit row ids");
  if (!locate(q) || !locate(row_labels) || !locate(qlabel) || !locate(hits))
    return fail(KEDS_ERR_ARG, "index_label_hits: device pointers only");
  DeviceGuard g(ix->device);
  if (!g.ok) return fail(KEDS_ERR_NO_GPU, "cannot select CUDA device %d", ix->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  memset(&ix->stats, 0, sizeof ix->stats);
  const int kmax = ks[nks - 1];
  // exact rows of the queries the certificate queues (the fallback writes them, k_hits_from_rows counts them)
  const int64_t nb_max = std::min<int64_t>(nq, Q_PASS_MAX);
  CKS(ix->D_stage[0].ensure(static_cast<size_t>(nb_max) * kmax * 4));
  CKS(ix->I_stage[0].ensure(static_cast<size_t>(nb_max) * kmax * 8));
  Call c = call(1, ix, nullptr, q, nq, kmax, ix->D_stage[0].as<float>(), ix->I_stage[0].as<int64_t>(), nullptr,
                nullptr, 0u);
  c.hits.nks = nks;
  for (int j = 0; j < nks; ++j) c.hits.ks[j] = ks[j];
  c.hits.row_labels = reinterpret_cast<const long long*>(row_labels);
  c.hits.qlabel = reinterpret_cast<const long long*>(qlabel);
  c.hits.hits = hits;
  CKS(run_passes(c, st));
  CK(cudaGetLastError());
  return 0;
}

int keds_gallery_rank(const float* Q, int64_t nq, const float* G, int64_t ng, int d,
                      const int64_t* target, const int64_t* exclude, int64_t* rank_out, void* stream) {
  if (!Q || !G || !target || !rank_out || nq < 0 || ng <= 0 || d <= 0)
    return fail(KEDS_ERR_ARG, "gallery_rank: bad argument");
  if (nq == 0) return 0;
  const size_t smem = static_cast<size_t>((d + 3) & ~3) * 4 * 8;  // 8 queries per block
  if (smem > 48 * 1024) return fail(KEDS_ERR_ARG, "gallery_rank: d too large");
  const int dev = locate(rank_out).device;
  if (dev < 0 || locate(Q).device != dev || locate(G).device != dev)
    return fail(KEDS_ERR_ARG, "gallery_rank: Q, G and rank_out must be memory of one device");
  DeviceGuard g(dev);
  if (ng >= 1024 && nq >= 64) {
    // worth a tensor-core pass: rank against a temporary index over the gallery (callers that score
    // many query sets against one gallery keep the index and call keds_index_rank themselves)
    keds_index_t* tmp = nullptr;
    CKS(keds_index_create(d, KEDS_METRIC_IP, dev, &tmp));
    int s = keds_index_add(tmp, G, ng);
    if (s == 0) s = keds_index_rank(tmp, Q, nq, target, exclude, rank_out, stream);
    if (s == 0) s = finish_sync(tmp, static_cast<cudaStream_t>(stream));
    keds_index_free(tmp);
    return s;
  }
  k_gallery_rank<<<static_cast<unsigned>((nq + 7) / 8), 256, smem, static_cast<cudaStream_t>(stream)>>>(
      Q, nq, G, ng, d, reinterpret_cast<const long long*>(target),
      reinterpret_cast<const long long*>(exclude), reinterpret_cast<long long*>(rank_out), nullptr, nullptr);
  CK(cudaGetLastError());
  return 0;
}

int keds_label_hits(const int64_t* I, int64_t nq, int kmax, const int64_t* labels, const int64_t* qlabel,
                    const int32_t* ks, int nks, int32_t* hits, void* stream) {
  if (!I || !labels || !qlabel || !ks || !hits || nq < 0 || kmax <= 0 || nks <= 0)
    return fail(KEDS_ERR_ARG, "label_hits: bad argument");
  if (nq == 0) return 0;
  const int dev = locate(hits).device;
  if (dev < 0 || locate(I).device != dev) return fail(KEDS_ERR_ARG, "label_hits: I and hits must be memory of one device");
  DeviceGuard g(dev);
  k_label_hits<<<static_cast<unsigned>((nq + 127) / 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const long long*>(I), nq, kmax, reinterpret_cast<const long long*>(labels),
      reinterpret_cast<const long long*>(qlabel), ks, nks, hits);
  CK(cudaGetLastError());
  return 0;
}

}  // extern "C"

// keds_consumer_*: the neighbour consumer (uses the helpers above)
#include "consumer_host.cuh"
// keds_clip_loss_*: the contrastive loss over the gathered features
#include "clip_loss_host.cuh"
// keds_consumer_bind_params / _forward_train / _backward: the consumer while it is being trained
#include "consumer_train_host.cuh"
