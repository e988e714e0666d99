/* keds_knn.h -- C ABI of libkeds_knn.so, the B200 (sm_100a) drop-in for the knowledge-retrieval
 * hot path of KEDs. Plain C: opaque handles, raw pointers, sizes. No C++ or torch types.
 *
 * Every entry point names the reference interface it replaces (paths relative to the KEDs tree).
 * The reference reaches this path through the Faiss Python module; a maintainer binds these
 * functions with ctypes (see INTEGRATION.md, keds_b200/_capi.py).
 *
 * Pointer residency: `const float*`/output pointers may be host or device memory (detected with
 * cudaPointerGetAttributes). Host pointers imply staged copies and a stream synchronisation before
 * return (Faiss' numpy contract). Device pointers make the call stream-ordered and asynchronous.
 * All matrices are C-contiguous row-major. Return value: 0 on success, negative keds_status
 * otherwise, with text in keds_last_error(). There is no CPU fallback.
 */
#ifndef KEDS_KNN_H
#define KEDS_KNN_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct keds_index keds_index_t;

enum keds_metric { KEDS_METRIC_IP = 0, KEDS_METRIC_L2 = 1 };

enum keds_status {
  KEDS_OK = 0,
  KEDS_ERR_ARG = -1,      /* bad argument (null, d mismatch, k out of range ...) */
  KEDS_ERR_CUDA = -2,     /* CUDA runtime/driver error, cudaError_t in the message */
  KEDS_ERR_NO_GPU = -3,   /* no usable sm_100 device */
  KEDS_ERR_KERNEL = -4,   /* device-side protocol watchdog fired (error word in the message) */
  KEDS_ERR_OOM = -5
};

/* search flags */
#define KEDS_SEARCH_EXACT_ONLY 1u  /* skip the 16-bit tensor-core pass, answer with the fp32 scan */
#define KEDS_SEARCH_NO_FALLBACK 2u /* debugging: do not run the exact fallback for flagged queries */
#define KEDS_SEARCH_FORCE_IP 4u    /* rank by inner product whatever the index metric (the reference's
                                      use_faiss=False branch, src/trainer.py:246-257) */

typedef struct keds_search_stats {
  int32_t n_flagged[2];  /* queries whose certificate failed (answered by the exact fallback) */
  int32_t slices;        /* row slices per (database, query tile) used by the last search */
  int32_t items;         /* work items of the scoring kernel */
  int32_t grid;          /* CTAs launched by the scoring kernel */
  int32_t exact_only;    /* 1 if the planner chose the fp32 scan for the whole batch */
  int32_t launches;      /* kernels launched by the last search call */
  uint32_t err_word;     /* device watchdog word, 0 = clean */
} keds_search_stats;

/* ---- index lifecycle ------------------------------------------------------------------------
 * Replaces faiss.IndexFlatL2(768) / IndexFlatIP + faiss.index_cpu_to_gpu(res, gpu, index)
 * (src/main.py:72-83, src/eval_retrieval.py:289-296). */
int keds_index_create(int d, int metric, int device, keds_index_t** out);
void keds_index_free(keds_index_t* idx);

/* index.add(x) (src/main.py:78,83; src/eval_retrieval.py:293,296). x: [n][d] float32, host or
 * device. Copies; the caller may free x on return. Builds the fp32 master, the 16-bit operand copy
 * (fp16 or bf16, see keds_index_operand_format) and the per-row norms on the index's device. */
int keds_index_add(keds_index_t* idx, const float* x, int64_t n);
/* add with options. KEDS_ADD_NORMALIZE: rows are L2-normalised on the device while they are added
 * (the database builder's `bases / bases.norm(dim=1, keepdim=True)`, src/main.py:465-466), so the
 * fp32 master, the bf16 operand copy and the norms come out of one pass over the upload. */
#define KEDS_ADD_NORMALIZE 1u
int keds_index_add_ex(keds_index_t* idx, const float* x, int64_t n, uint32_t flags);
/* copy rows [first, first+n) of the resident fp32 master to out (host or device) -- e.g. to save a
 * database built on the device back into the .pt layout */
int keds_index_get_rows(const keds_index_t* idx, int64_t first, int64_t n, float* out);
int keds_index_reset(keds_index_t* idx);                 /* index.reset() */
int64_t keds_index_ntotal(const keds_index_t* idx);      /* index.ntotal */
int keds_index_dim(const keds_index_t* idx);             /* index.d */
int keds_index_metric(const keds_index_t* idx);
int keds_index_device(const keds_index_t* idx);
/* device pointer to the resident fp32 rows [ntotal][d] (for keds_gather_pool); owned by idx */
const float* keds_index_rows(const keds_index_t* idx);
/* added to every returned label (row-sharded indices report global ids) */
int keds_index_set_id_offset(keds_index_t* idx, int64_t offset);
/* 16-bit operand format of the tensor-core pass: 0 = bf16, 1 = fp16 (fp32 accumulate either way,
 * same rate, same bytes). Chosen per index from the rows it holds: fp16 keeps 11 significant bits,
 * so on unit-norm embeddings the certificate's error bound is ~6x tighter (fewer candidates to
 * re-score, clustered data stays on the fast path); bf16 is used when a value would leave fp16's
 * range or fp16 would lose more of the rows. Results are exact fp32 under both. set: -1 = automatic
 * (default; also env KEDS_OPERAND=bf16|fp16), 0 / 1 pin the format (rows already added are
 * re-rounded from the fp32 master). */
int keds_index_operand_format(const keds_index_t* idx);
int keds_index_set_operand_format(keds_index_t* idx, int fmt);
/* Bumped whenever a device buffer of idx moves or its rows change (add / reset, a search with a
 * larger batch or k growing the per-call scratch). A CUDA graph captured over a search on idx holds
 * those addresses: compare before every replay and re-capture on a change. */
uint64_t keds_index_generation(const keds_index_t* idx);

/* ---- search ---------------------------------------------------------------------------------
 * D, I = index.search(q, k) (src/trainer.py:213,221,271; src/eval_utils.py:169,177).
 * q: [nq][d] float32. D: [nq][k] float32 (inner products, or squared L2 distances). I: [nq][k]
 * int64 labels, best first; ties by lower label; rows past ntotal are padded with label -1 and
 * D = -FLT_MAX (IP) / +FLT_MAX (L2). Results equal an exact fp32 flat search.
 *
 * Exclusion (every search call but keds_index_search): rows left out per query (training without
 * self-retrieval: a query whose own pair is in the knowledge base must not retrieve it).
 * exclude: NULL with n_exclude = 0 for none, or int64 [nq][n_exclude], 1 <= n_exclude <= 8, labels
 * as I returns them (id_offset included); -1 = unused slot, a label the index does not hold excludes
 * nothing. Device memory of the index's GPU (keds_retrieve2 also takes page-locked host memory). In
 * two-database calls one array applies to both databases (aligned row for row: a pair's image row
 * and caption row share a label). Each query's result equals an exact fp32 flat search over the rows
 * it does not exclude: same order, same ties, -1 / -+FLT_MAX padding when fewer than k rows remain;
 * an excluded row is never returned. Gather, pool and host mirrors follow the returned I. */
int keds_index_search(keds_index_t* idx, const float* q, int64_t nq, int k, float* D, int64_t* I,
                      void* cuda_stream);
int keds_index_search_ex(keds_index_t* idx, const float* q, int64_t nq, int k, float* D, int64_t* I,
                         const int64_t* exclude, int n_exclude, uint32_t flags, void* cuda_stream);
/* Two indices, one query batch: the image-DB and text-DB searches of src/trainer.py:213 and :221
 * fused into one pass over the queries. Both indices share d, metric and device. */
int keds_index_search2(keds_index_t* a, keds_index_t* b, const float* q, int64_t nq, int k,
                       float* Da, int64_t* Ia, float* Db, int64_t* Ib, const int64_t* exclude,
                       int n_exclude, uint32_t flags, void* cuda_stream);
/* The whole retrieval operator of src/trainer.py:198-230 in one call: search both databases, then
 * per stream s in {img, txt}
 *   feat_s[b][j][:] = rows_s[I_s[b][perm_s ? perm_s[j] : j]][:]      (nullable; [nq][k][d])
 *   pool_s[b][:]    = sum_j w_j rows_s[I_s[b][j]][:]                 (nullable; [nq][d])
 * pool_mode 0: no pool; 1: w = 1/k; 2: w = softmax_j(+-tau * D_s[b][j]) (minus under L2).
 * Padding (I = -1, fewer than k rows to return) is a zero row in feat and in the pool: mean pools
 * still divide by k, softmax pools give it weight 0.
 * Each neighbour row is read once for both outputs. perm_*: device int32[k] or NULL, and it must be a
 * permutation of 0..k-1. It is not checked (that would need a synchronisation): the pool is summed
 * over output slots, slot j adding w_{perm[j]} * rows_s[I_s[b][perm[j]]], so a repeated entry counts
 * one neighbour twice and drops another; an entry outside [0, k) gives a zero row in feat and adds
 * nothing but w_0 * 0 to the pool. The Python wrappers refuse a host perm that is not a permutation.
 * The summation order of the pool depends on the route a query takes (DESIGN.md section 3).
 * D_*, I_*, feat_*, pool_*: device memory. For a caller whose queries and results live on the HOST,
 * as the reference's do (q.cpu().numpy() in, numpy (D, I) out, src/trainer.py:207-221), the call
 * also runs without copies around the search:
 *   q        may be page-locked host memory (cudaHostAlloc / cudaHostRegister / torch pin_memory):
 *            the first kernel of the chain reads it through the device mapping, once; so may
 *            exclude, read through the mapping once per call, like q;
 *   Dh_x, Ih_x (nullable, in pairs) page-locked host blocks [nq][k]: the block that finishes a query's
 *            row stores it there as well as into D_x, I_x (posted writes that travel while the
 *            neighbour gather of that query runs).
 * Stream-ordered and asynchronous: the host blocks are complete once the stream has been
 * synchronised (or the graph that captured the call has finished). */
int keds_retrieve2(keds_index_t* img, keds_index_t* txt, const float* q, int64_t nq, int k,
                   const int32_t* perm_img, const int32_t* perm_txt, int pool_mode, float tau,
                   float* D_img, int64_t* I_img, float* D_txt, int64_t* I_txt, float* Dh_img,
                   int64_t* Ih_img, float* Dh_txt, int64_t* Ih_txt, float* feat_img, float* feat_txt,
                   float* pool_img, float* pool_txt, const int64_t* exclude, int n_exclude,
                   uint32_t flags, void* cuda_stream);
/* ---- range search ------------------------------------------------------------------------------
 * lims, D, I = index.range_search(q, radius) (Faiss' RangeSearchResult layout): every row n with
 *   IP: s(n) > radius        L2: d(n) < radius (squared distance)
 * strictly, where s / d is the library's exact fp32 score -- the same bits keds_index_search reports
 * for that (query, row). Query i owns entries [lims[i], lims[i+1]) of D / I, ordered best first,
 * ties by lower label (Faiss leaves this order open; here it is fixed). Labels include id_offset;
 * KEDS_SEARCH_FORCE_IP is the only flag that applies. The tensor-core pass lists every row whose
 * 16-bit-operand score lies above the radius minus the certificate's error bound and the rounding of
 * the fp32 score (DESIGN.md section 3), and those rows are re-scored in fp32, so the answer is exact
 * for every query, including queries the 16-bit format cannot hold.
 * The result size is known only after the search, so the call has two steps:
 *   range_search   q [nq][d] float32 and lims int64 [nq + 1]: host or device memory. Runs the search
 *                  on cuda_stream, writes lims and synchronises the stream before it returns (it
 *                  reads counts back between its kernels). D and I stay in handle-owned buffers.
 *   range_results  copies the lims[nq] results out: D float32, I int64, host or device memory
 *                  (device pointers: stream-ordered; host pointers: synchronous).
 * The results stay valid until the next call on idx; a results buffer that grows bumps generation. */
int keds_index_range_search(keds_index_t* idx, const float* q, int64_t nq, float radius, int64_t* lims,
                            uint32_t flags, void* cuda_stream);
int keds_index_range_results(keds_index_t* idx, float* D, int64_t* I, void* cuda_stream);

/* Wait for the last asynchronous search on idx and report its device status. */
int keds_index_sync(keds_index_t* idx, void* cuda_stream);
int keds_index_last_stats(const keds_index_t* idx, keds_search_stats* out);
/* Timing of the scoring kernel inside a running loop (bench.py's roofline leg).
 * set_profiling(1): every launch stamps %globaltimer at the start of its first CTA and the end of
 *   its last one -- no stream events, the launch chain (programmatic dependent launches) is left
 *   untouched; profile() returns the summed kernel duration in ms and the number of launches.
 * set_profiling(0): off; any other mode is KEDS_ERR_ARG. profile() and profile_chain() fail unless
 *   mode 1 is on. */
int keds_index_set_profiling(keds_index_t* idx, int enable);
int keds_index_profile(keds_index_t* idx, double* score_ms_total, int64_t* score_launches);
/* Mode 1, whole chain: average in-loop duration of each kernel of a search (0 k_prep_rows,
 * 1 k_score_topk, 2 k_select_rerank, 3 k_exact_fallback, 4 reserved = 0) and the average idle gap
 * in front of it (end of the previous kernel to its first CTA), in ms. n >= 5. Does not clear. */
int keds_index_profile_chain(keds_index_t* idx, double* dur_ms, double* gap_ms, int64_t* searches, int n);

/* ---- neighbour gather / weighted pool ---------------------------------------------------------
 * W == NULL:  out[b][j][:] = base[I[b][perm ? perm[j] : j]][:]   (out: [B][k][d])
 *             replaces base[I.reshape(-1)].reshape(B,k,-1), the shared randperm(k) shuffle and the
 *             .to(device) of src/trainer.py:214-230, src/eval_utils.py:170-183.
 * W != NULL:  out[b][h][:] = sum_j W[b][h][j] * base[I[b][j]][:]  (W: [B][H][k], out: [B][H][d])
 *             the attn@v-shaped pool of src/model/model.py:69-73.
 * base, out, W: device float32. I: device int64. perm: device int32[k] or NULL. id < 0 -> zeros. */
int keds_gather_pool(const float* base, int64_t n_base, const int64_t* I, const float* W,
                     const int32_t* perm, int64_t B, int k, int H, int d, float* out,
                     void* cuda_stream);

/* ---- row-sharded merge ------------------------------------------------------------------------
 * D_parts/I_parts: [parts][nq][k] per-shard results with global labels (device), each part sorted
 * best-first with its -1 padding last, exactly as keds_index_search returns it; writes the global
 * top-k with the same ordering rule. New relative to the reference (replicas only). */
int keds_topk_merge(const float* D_parts, const int64_t* I_parts, int parts, int64_t nq, int k,
                    int metric, float* D, int64_t* I, void* cuda_stream);
/* Same, with part p at D_parts + p*stride_d (floats) and I_parts + p*stride_i (int64s): lets one
 * packed all-gather buffer ([rank][D block | I block]) be merged in place. */
int keds_topk_merge_strided(const float* D_parts, const int64_t* I_parts, int64_t stride_d,
                            int64_t stride_i, int parts, int64_t nq, int k, int metric, float* D,
                            int64_t* I, void* cuda_stream);

/* Row-shard exchange over NVLink peer memory (no collective call in the step). The buffers are
 * symmetric allocations mapped into every rank of the box; the library only sees raw pointers.
 *   keds_p2p_push       copy this rank's block (src, bytes % 16 == 0) into peer_dst[r] for every
 *                       r != my_rank with P2P stores, then publish `epoch` (system-scope release)
 *                       to peer_flag[r]. peer_dst / peer_flag: host arrays of n_ranks device
 *                       pointers (entry my_rank ignored). ticket: a zeroed device word owned by
 *                       the caller. Ordered after earlier work on the stream.
 *   keds_topk_merge_wait  keds_topk_merge_strided that first waits (system-scope acquire, bounded)
 *                       until flags[r] >= epoch for every r != my_rank; flags: this rank's own
 *                       flag array [parts]; a peer that never arrives sets *err_word. */
int keds_p2p_push(const void* src, int64_t bytes, void* const* peer_dst, uint32_t* const* peer_flag,
                  int n_ranks, int my_rank, uint32_t epoch, uint32_t* ticket, void* cuda_stream);
int keds_topk_merge_wait(const float* D_parts, const int64_t* I_parts, int64_t stride_d, int64_t stride_i,
                         int parts, int64_t nq, int k, int metric, float* D, int64_t* I,
                         const uint32_t* flags, int my_rank, uint32_t epoch, uint32_t* err_word,
                         void* cuda_stream);

/* Row-sharded search with the exchange fused into the search kernels (the north_star's "local
 * top-k -> all-gather -> merge" as ONE launch chain, no collective call and no extra copy kernel):
 * the block that finishes query b's exact top-k stores that row straight into every peer's receive
 * buffer over NVLink, the last block of the chain publishes the epoch flag, and the merge kernel
 * waits for the peers' flags. Every rank passes the same queries, calls in the same order, and ends
 * with the global (D, I). Bit-identical to an unsharded index.
 *   exchange_create   peer_base[r] = rank r's symmetric buffer (buf_bytes each, zero-filled before
 *                     the first search) as mapped into this process; entry my_rank = the local one.
 *                     Layout is the library's: 256 flag bytes, then 2 parities x n_ranks slots.
 *   exchange_capacity largest nq * k one search may carry.
 *   search_sharded    q [nq][d], D [nq][k], I [nq][k]: device memory; idx holds this rank's rows
 *                     with keds_index_set_id_offset(first global row). Asynchronous on cuda_stream.
 *                     exclude (nullable, as keds_index_search_ex): [nq][n_exclude] global labels in
 *                     device memory, the same on every rank; each shard leaves out the ones it holds,
 *                     so the merged result equals keds_index_search_ex on an unsharded index.
 *   exchange_stats    synchronises; average / maximum time (us) block 0 of the merge waited for the
 *                     peers since the last call (rank skew), merges counted, and the error word
 *                     (non-zero: a peer never delivered). */
typedef struct keds_exchange keds_exchange_t;
int keds_exchange_create(int n_ranks, int my_rank, int device, void* const* peer_base, int64_t buf_bytes,
                         keds_exchange_t** out);
void keds_exchange_free(keds_exchange_t* ex);
int64_t keds_exchange_capacity(const keds_exchange_t* ex);
int keds_index_search_sharded(keds_index_t* idx, keds_exchange_t* ex, const float* q, int64_t nq, int k,
                              float* D, int64_t* I, const int64_t* exclude, int n_exclude, void* cuda_stream);
int keds_exchange_stats(keds_exchange_t* ex, void* cuda_stream, double* wait_us_avg, double* wait_us_max,
                        int64_t* steps, uint32_t* err_word);

/* Row-sharded retrieval step: keds_retrieve2 over two row-sharded bases that share one exchange.
 *   index_rows_ipc      cudaIpcMemHandle_t (64 bytes) of the index's fp32 rows; all zero for an
 *                       empty index. Valid until the next add / reset of the index.
 *   exchange_attach_rows  every rank's rows of database db (0 image, 1 text): handles[r] from
 *                       index_rows_ipc on rank r, lo[r] its first global label, n[r] its row count
 *                       (n = 0: no rows, handle ignored). Peers' rows are mapped (cudaIpc), this
 *                       rank's own handle must come from index_rows_ipc in this process. Collective
 *                       in effect: every rank re-attaches after every add on any rank.
 *   retrieve2_sharded   q [nq][d] identical on every rank; every rank receives the merged
 *                       D_* / I_* [nq][k] of all queries (bit-identical to keds_retrieve2 on an
 *                       unsharded index, exclusion included), and feat_* [row_hi-row_lo][k][d] /
 *                       pool_* [row_hi-row_lo][d] of queries [row_lo, row_hi) only, gathered from the
 *                       owners' rows over NVLink (pools: the same weights; summation order fixed, so
 *                       equal for every shard count). Device pointers only; exclude nullable;
 *                       refuses to run if this rank's rows moved or grew since the attach. */
int keds_index_rows_ipc(const keds_index_t* idx, void* handle64);
int keds_exchange_attach_rows(keds_exchange_t* ex, int db, const void* const* handles, const int64_t* lo,
                              const int64_t* n);
int keds_retrieve2_sharded(keds_index_t* img, keds_index_t* txt, keds_exchange_t* ex, const float* q, int64_t nq,
                           int k, const int32_t* perm_img, const int32_t* perm_txt, int pool_mode, float tau,
                           int64_t row_lo, int64_t row_hi, float* D_img, int64_t* I_img, float* D_txt,
                           int64_t* I_txt, float* feat_img, float* feat_txt, float* pool_img, float* pool_txt,
                           const int64_t* exclude, int n_exclude, uint32_t flags, void* cuda_stream);

/* ---- gallery ranking --------------------------------------------------------------------------
 * rank_out[q] = #{ g != target[q], g != exclude[q] : (s(q,g), -g) > (s(q,target), -target) } with
 * s = fp32 inner product. Replaces the similarity matrix + full argsort + name matching of
 * get_metrics_coco / _fashion / _cirr (src/eval_utils.py:1008-1067). All pointers device memory;
 * exclude may be NULL. */
int keds_gallery_rank(const float* Q, int64_t nq, const float* G, int64_t ng, int d,
                      const int64_t* target, const int64_t* exclude, int64_t* rank_out,
                      void* cuda_stream);
/* The same ranks against the rows of an index (the gallery added once, many query sets ranked
 * against it: the reference scores 30 checkpoints x 3 feature sets against one gallery,
 * src/eval_utils.py:617,735). The dense Q x G contraction runs on the tensor cores: the scoring
 * kernel counts the rows whose 16-bit-operand score beats the target's exact score by more than the
 * certificate's error bound, lists the rows inside the bound, and those are settled with exact fp32
 * scores -- so the ranks equal the fp32 count bit for bit. Inner product whatever the index metric.
 * Device pointers; asynchronous on cuda_stream. */
int keds_index_rank(keds_index_t* idx, const float* q, int64_t nq, const int64_t* target,
                    const int64_t* exclude, int64_t* rank_out, void* cuda_stream);
/* hits[q][i] = #{ j < ks[i] : labels[I[q][j]] == qlabel[q] } for ascending ks (device pointers).
 * The counting core of get_metrics_imgnet (src/eval_utils.py:1107-1118). */
int keds_label_hits(const int64_t* I, int64_t nq, int kmax, const int64_t* labels,
                    const int64_t* qlabel, const int32_t* ks, int nks, int32_t* hits,
                    void* cuda_stream);
/* The same hits straight from the index, without materialising the ranked rows: the whole counting
 * core of get_metrics_imgnet (feats @ G.t(), argsort, top-k masks, label products;
 * src/eval_utils.py:1101-1118) in one call. hits[q][i] = #{ rows of the index among the exact
 * top-ks[i] of query q (score descending, then lower row id: the order keds_index_search returns)
 * whose row_labels entry equals qlabel[q] }. Neither distances nor the order inside a top-k set are
 * needed, so only the rows whose 16-bit-operand score lies inside the certificate's error band
 * around a cut point are re-scored in fp32 (about 65 instead of 200+ at the 50k-gallery shape);
 * the sets, and therefore the counts, are those of an exact fp32 search.
 * ks: HOST array, ascending, nks <= 8, ks[nks-1] <= 2048. q, row_labels [ntotal], qlabel [nq],
 * hits [nq][nks]: device. Asynchronous on cuda_stream. */
int keds_index_label_hits(keds_index_t* idx, const float* q, int64_t nq, const int64_t* row_labels,
                          const int64_t* qlabel, const int32_t* ks, int nks, int32_t* hits,
                          void* cuda_stream);

/* ---- neighbour consumer (SURVEY.md §8 f2; eval forward here, training entry points below) ------
 * The modules that consume the retrieved neighbours, evaluated in one launch sequence:
 *   mapped = img2text(feat); nb_img = img2text(base_img[I_img]); nb_txt = img2text(base_txt[I_txt])
 *   tokens[:,0,:] = retrieval_fuse(mapped[:,None], nb_img, nb_img)   (CrossFormer, image stack = 0)
 *   tokens[:,1,:] = text_condition(mapped[:,None], nb_txt, nb_txt)   (CrossFormer, text stack = 1)
 *   tokens[:,2,:] = mapped
 * i.e. src/trainer.py:59-69 and src/eval_utils.py:378-383,515-519,661-668,806-810,943-947 with
 * IM2TEXT / CrossFormer / CrossAttention of src/model/model.py:37-123 in eval mode (dropout off).
 * Arithmetic: tf32 tensor-core products with fp32 accumulation, fp32 everywhere else.
 *
 * create: d_in = feature width (768), d_mid = IM2TEXT middle_dim (512), d_tok = IM2TEXT output_dim =
 *   CrossFormer q/k/v_dim (768), n_hidden = IM2TEXT n_layer (2), n_layers = CrossFormer num_layers
 *   (3), heads (8), dim_head (64). All widths multiples of 4.
 * set_linear: one nn.Linear, W [out][in] float32 row-major (torch layout), b [out] or NULL; host or
 *   device pointers; copied. kind MLP: layer 0..n_hidden-1 = layers[i][0], layer n_hidden = fc_out
 *   (stack ignored). Other kinds: to_q / to_k / to_v / to_out[0] of cross_layers[layer] of `stack`.
 * finalize: after every slot is set; forward fails before it. */
typedef struct keds_consumer keds_consumer_t;
enum keds_consumer_kind {
  KEDS_CONSUMER_MLP = 0,
  KEDS_CONSUMER_TO_Q = 1,
  KEDS_CONSUMER_TO_K = 2,
  KEDS_CONSUMER_TO_V = 3,
  KEDS_CONSUMER_TO_OUT = 4
};
int keds_consumer_create(int d_in, int d_mid, int d_tok, int n_hidden, int n_layers, int heads,
                         int dim_head, int device, keds_consumer_t** out);
void keds_consumer_free(keds_consumer_t* c);
int keds_consumer_set_linear(keds_consumer_t* c, int kind, int stack, int layer, const float* W,
                             const float* b, int out_features, int in_features);
int keds_consumer_finalize(keds_consumer_t* c);
/* feat [B][d_in], base_* [n_*][d_in] (keds_index_rows), I_* [B][k] int64 (ids < 0 read as zero rows),
 * perm int32[k] or NULL (the shared randperm of src/trainer.py:218-219, image neighbours only),
 * tokens [B][3][d_tok]: all device memory. Asynchronous on cuda_stream. */
int keds_consumer_forward(keds_consumer_t* c, const float* feat, const float* base_img, int64_t n_img,
                          const float* base_txt, int64_t n_txt, const int64_t* I_img,
                          const int64_t* I_txt, const int32_t* perm, int64_t B, int k, float* tokens,
                          void* cuda_stream);
/* synchronise the stream and report a device-side pipeline error, if any; launches (nullable) =
 * kernels launched by this handle so far */
int keds_consumer_check(keds_consumer_t* c, void* cuda_stream, int64_t* launches);

/* ---- the same modules while they are being trained (src/trainer.py:59-69, backward at :462-474) --
 * Parameters live in ONE flat caller-owned device buffer (e.g. a torch Parameter) that the optimiser
 * updates in place; the handle reads through it and nothing is copied per step. Layout (floats,
 * every block padded to a multiple of 4): IM2TEXT W_i, b_i for i = 0 .. n_hidden (fc_out last); then
 * per stack (image, text): to_k / to_v of all layers stacked as [L][k | v][inner] x d_tok with their
 * biases, then per layer to_q W, b and to_out W, b. param_offset gives any slot's offsets and shape.
 *   bind_params     adopt the buffer (replaces set_linear + finalize; set_linear afterwards writes
 *                   into the buffer).
 *   forward_train   keds_consumer_forward that keeps the activations the backward needs. masks:
 *                   NULL or n_hidden device pointers (entries nullable) to float [B(1+2k)][d_mid]
 *                   dropout multipliers (0 or 1/(1-p); rows ordered queries | image neighbours |
 *                   text neighbours), applied between Linear and ReLU as in IM2TEXT
 *                   (src/model/model.py:110-116); they must stay alive until the backward.
 *                   Refuses (before queuing anything) a k whose attention backward, heads x
 *                   (2 dim_head + 2k) floats of shared memory, would not fit one block. Every
 *                   other batch it accepts (B (1 + 2k) <= 2^30 rows) also runs its backward.
 *   backward        dtokens [B][3][d_tok] -> grads (param_count floats, same layout, overwritten).
 *                   One backward per forward_train. tf32 tensor-core products, fp32 accumulation. */
int64_t keds_consumer_param_count(const keds_consumer_t* c);
int keds_consumer_param_offset(const keds_consumer_t* c, int kind, int stack, int layer, int64_t* w_off,
                               int64_t* b_off, int64_t* rows, int64_t* cols);
int keds_consumer_bind_params(keds_consumer_t* c, float* params);
int keds_consumer_forward_train(keds_consumer_t* c, const float* feat, const float* base_img, int64_t n_img,
                                const float* base_txt, int64_t n_txt, const int64_t* I_img,
                                const int64_t* I_txt, const int32_t* perm, int64_t B, int k,
                                const float* const* masks, float* tokens, void* cuda_stream);
int keds_consumer_backward(keds_consumer_t* c, const float* dtokens, float* grads, void* cuda_stream);

/* The consumer over two row-sharded bases (keds_retrieve2_sharded): the neighbour rows are read in
 * place from the rank that owns them (its own fp32 rows, or a peer's over NVLink through the mapping
 * of keds_exchange_attach_rows), so no [B][k][d] features are materialised.
 *   I_img / I_txt   [B][k] GLOBAL labels, e.g. this rank's rows of the merged I of
 *                   keds_retrieve2_sharded; a label no shard holds (-1 padding) reads as a zero row.
 *   img / txt       this rank's index handles of the two bases (databases 0 and 1 of ex).
 * Everything else as keds_consumer_forward / keds_consumer_forward_train; keds_consumer_backward
 * follows either unchanged (it reads only the assembled MLP input). Refused with KEDS_ERR_ARG before
 * anything is queued: a NULL argument or a buffer that is not device memory, a base not attached to
 * ex, this rank's rows moved or grown since the attach (re-attach after every add), an index width
 * other than d_in, consumer / indices / exchange on different devices. No flag guards the peers'
 * rows: they do not change between adds, and an add synchronises every rank first. */
int keds_consumer_forward_sharded(keds_consumer_t* c, keds_index_t* img, keds_index_t* txt, keds_exchange_t* ex,
                                  const float* feat, const int64_t* I_img, const int64_t* I_txt,
                                  const int32_t* perm, int64_t B, int k, float* tokens, void* cuda_stream);
int keds_consumer_forward_train_sharded(keds_consumer_t* c, keds_index_t* img, keds_index_t* txt,
                                        keds_exchange_t* ex, const float* feat, const int64_t* I_img,
                                        const int64_t* I_txt, const int32_t* perm, int64_t B, int k,
                                        const float* const* masks, float* tokens, void* cuda_stream);
/* Test hook: hidden activations [B(1+2k)][d_mid] of IM2TEXT layer `layer` as the last forward_train
 * left them (after dropout and ReLU). Their signs are the ReLU gates the backward uses; a tf32
 * forward and a float64 one disagree on them for pre-activations within rounding of zero, so a
 * gradient comparison has to take the gates from here. Synchronises. */
int keds_consumer_debug_hidden(keds_consumer_t* c, int layer, float* out, int64_t n, void* cuda_stream);
/* Diagnostics: with debug on, every k_linear_tf32 launch of a forward records per CTA
 * {start, prologue done, dependency met, accumulator ready, end} (%globaltimer ns).
 * debug_timeline copies launch `launch` (index within the last forward) of n_ctas CTAs to
 * out[n_ctas][5] (host). Synchronises the device. */
int keds_consumer_set_debug(keds_consumer_t* c, int enable);
int keds_consumer_debug_timeline(keds_consumer_t* c, int launch, uint64_t* out, int64_t n_ctas);

/* ---- contrastive loss over the gathered features (forward + backward; SURVEY.md §8 f3) ---------
 * The step that follows the retrieval path in the training loop (src/trainer.py:85-135,164):
 *   logits = logit_scale * I_all @ T_all.t()
 *   loss   = (CrossEntropy(logits, arange(N)) + CrossEntropy(logits.t(), arange(N))) / 2
 * I_all, T_all: [N][d] float32 device, the image / text features of ALL ranks after the all-gather
 * (rows [row0, row0 + n_local) are this rank's own); logit_scale: 1 float, device (no host sync).
 * Outputs (device): loss (1 float), and -- both
 * or neither -- dI_local, dT_local [n_local][d] = d loss / d (this rank's rows), plus dscale
 * (1 float, nullable) = d loss / d logit_scale. Products run on tf32 tensor cores with a hi/lo
 * operand split (fp32-class accuracy). N and d multiples of 4. Asynchronous on cuda_stream. */
typedef struct keds_clip_loss keds_clip_loss_t;
int keds_clip_loss_create(int device, keds_clip_loss_t** out);
void keds_clip_loss_free(keds_clip_loss_t* h);
int keds_clip_loss_forward_backward(keds_clip_loss_t* h, const float* I_all, const float* T_all, int64_t N,
                                    int d, int64_t row0, int64_t n_local, const float* logit_scale, float* loss,
                                    float* dI_local, float* dT_local, float* dscale, void* cuda_stream);
/* synchronise the stream and report a device-side pipeline error, if any */
int keds_clip_loss_check(keds_clip_loss_t* h, void* cuda_stream);

/* ---- diagnostics ------------------------------------------------------------------------------
 * Approximate (16-bit operand tensor-core) scores of q against every row: out [nq][ntotal] device float32.
 * Test hook for the GEMM alone; not a product path. */
int keds_debug_scores(keds_index_t* idx, const float* q, int64_t nq, float* out, void* cuda_stream);
/* Host only, needs no GPU: the work decomposition the planner picks for n_db databases of n_rows
 * rows each, nq queries, k neighbours on a device with num_sms SMs.
 * out = {exact_only, cta_pair, slices S, query tiles, work items, grid (CTAs)}. */
int keds_debug_plan(int n_db, int64_t nq, int k, int64_t n_rows, int num_sms, int32_t out[6]);
/* Host only, needs no GPU: which kernel the consumer's tf32 linear product C[M][N] (nz independent
 * problems) takes on num_sms SMs. variant = 1: 128-column tiles, 2: 256-column tiles, 3: persistent
 * 256-column tiles, 4 / 5: 32-column tiles with K split over a cluster of 2 / 4 CTAs. */
int keds_debug_linear_plan(int64_t M, int N, int nz, int num_sms, int32_t* variant);
/* Test hook for the tf32 linear product alone: C[z] = act(A[z] W[z]^T + b[z]) for z < nz (1 or 2),
 * act = ReLU if relu else identity. A[z] [M][K] with lda floats between rows (lda a multiple of 4,
 * >= K); W[z] [N][K] with round4(K) floats between rows; b[z] [N] or NULL; C[z] [M][N] with ldc
 * floats between rows (ldc >= N). A and W 16-byte aligned, C 4-byte aligned; all device memory.
 * variant 0 = the production choice (keds_debug_linear_plan), 1..5 forces one kernel.
 * Asynchronous on cuda_stream; keds_consumer_check reports device-side errors. */
int keds_consumer_debug_linear(keds_consumer_t* c, int variant, const float* A0, const float* A1, int64_t lda,
                               int64_t M, int K, const float* W0, const float* W1, const float* b0,
                               const float* b1, int N, int relu, float* C0, float* C1, int64_t ldc, int nz,
                               void* cuda_stream);
/* Test hook for the single-query cross-attention alone: one launch over both stacks z = 0, 1 (as the
 * forward and backward launch it), heads and dim_head of the handle, scale 1.0f / sqrtf(dim_head).
 * Q[z], out[z] (and dO[z]) [B][heads * dim_head]; KV[z] [B * k][ld_kv] with the keys of head h at
 * columns k_off + h * dim_head and its values at v_off + h * dim_head.
 *   backward = 0: out[z] = O = softmax(scale q K^T) V per head. variant 0 = the production choice,
 *     1 forces k_cross_attend<0>, 2 forces k_cross_attend<64> (dim_head 64, ld_kv, k_off and v_off
 *     multiples of 4, KV 16-byte aligned; refused otherwise).
 *   backward = 1 (variant 0 only): out[z] = dQ, and dK / dV of every neighbour row written to dKV[z]
 *     at the same columns as K / V in KV[z] (ld_kv); nothing else of dKV[z] is touched.
 * Refused before any launch: NULL or non-device buffers, k outside [1, 1024], key / value columns
 * beyond ld_kv, shared memory beyond what one block can have. Asynchronous on cuda_stream. */
int keds_consumer_debug_attend(keds_consumer_t* c, int variant, int backward, int64_t B, int k, const float* Q0,
                               const float* Q1, const float* KV0, const float* KV1, int64_t ld_kv, int k_off,
                               int v_off, const float* dO0, const float* dO1, float* out0, float* out1,
                               float* dKV0, float* dKV1, void* cuda_stream);
/* Programmatic dependent launch between the kernels of a search (default on; env KEDS_NO_PDL=1
 * turns the default off). Tuning/diagnostic switch; results do not depend on it. */
int keds_index_set_pdl(keds_index_t* idx, int enable);
/* Scale the certificate's error bound (1.0 = rigorous bound). Test hook for the fallback. */
int keds_index_set_eps_scale(keds_index_t* idx, float scale);

const char* keds_last_error(void);
int keds_device_count(void);          /* faiss.get_num_gpus() (src/eval_retrieval.py:289) */
const char* keds_version(void);

#ifdef __cplusplus
}
#endif
#endif /* KEDS_KNN_H */
