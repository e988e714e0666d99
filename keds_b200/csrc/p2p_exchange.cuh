// Row-shard exchange over NVLink peer memory, without a collective library call in the step:
// every rank stores its [B][k] (score | label) block straight into each peer's receive buffer
// (P2P stores through NVSwitch), publishes an epoch flag with system-scope release, and the merge
// kernel of each rank waits for the peers' flags with system-scope acquire before it reads.
// The buffers are symmetric allocations mapped into every rank (torch symmetric memory); this
// file only sees raw peer pointers. Included by aux_kernels.cuh.
#pragma once

namespace keds {

struct P2PPush {
  int n_ranks, my_rank;
  unsigned int epoch;
  long long n16;                       // 16-byte units to copy
  const uint4* src;                    // this rank's block (local memory)
  uint4* dst[P2P_MAX_RANKS];           // where that block lives in each rank's buffer (peer pointers)
  unsigned int* flag[P2P_MAX_RANKS];   // flag word "rank my_rank has delivered" in each rank's buffer
  unsigned int* ticket;                // local counter for "last CTA publishes"
};

__global__ void __launch_bounds__(256)
k_p2p_push(const P2PPush p) {
  griddep_wait();  // the local search results must be complete
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (int r = 0; r < p.n_ranks; ++r) {
    if (r == p.my_rank) continue;
    uint4* d = p.dst[r];
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < p.n16; i += stride)
      d[i] = p.src[i];
  }
  __threadfence_system();  // this thread's peer stores are ordered before the ticket below
  __syncthreads();
  __shared__ bool last;
  if (threadIdx.x == 0) last = atomicAdd(p.ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (last) {
    // every CTA has fenced its stores: publish the epoch to the peers, reset the ticket
    if (threadIdx.x < p.n_ranks && static_cast<int>(threadIdx.x) != p.my_rank) {
      __threadfence_system();
      st_release_sys(p.flag[threadIdx.x], p.epoch);
    }
    if (threadIdx.x == 0) *p.ticket = 0u;
  }
}

// Spin (bounded) until every peer's flag has reached `epoch`. Called by one thread per block.
__device__ __forceinline__ bool p2p_wait_flags(const unsigned int* flags, int n_ranks, int my_rank,
                                               unsigned int epoch, unsigned int* err_word) {
  const long long t0 = clock64();
  for (int r = 0; r < n_ranks; ++r) {
    if (r == my_rank) continue;
    // epochs only grow; the signed difference also survives wrap-around
    while (static_cast<int>(ld_acquire_sys(flags + r) - epoch) < 0) {
      if (clock64() - t0 > (1ll << 32)) {  // ~2 s: a peer is gone; report instead of hanging
        atomicCAS(err_word, 0u, 0x500u + r);
        return false;
      }
      __nanosleep(200);
    }
  }
  return true;
}

// ---------------------------------------------------------------------------------------------
// Neighbour consumer of a row-sharded two-database step (keds_retrieve2_sharded): after the merges,
// one block per (query of this rank's block [row_lo, row_lo + gridDim.x), database) looks up the
// owner of each merged label in the lo table, reads the row in place from that rank's fp32 master
// (its own, or a peer's over NVLink through a cudaIpc mapping) and runs the same gather / weights /
// pool as the local consumer. The rows do not change between adds, so no flag guards them.
struct ShardRowsDb {
  const float* base[P2P_MAX_RANKS];  // rank r's [n][d] fp32 rows as mapped into this process (null: no rows)
  long long lo[P2P_MAX_RANKS];       // global label of its first row
  long long n[P2P_MAX_RANKS];
};

// Where global label `lab` lives: row lab - lo[r] of the rank r with lo[r] <= lab < lo[r] + n[r], read
// in place from that rank's fp32 master; nullptr when no shard holds it (-1 padding included).
__device__ __forceinline__ const float* shard_row(const ShardRowsDb& rd, int n_ranks, long long lab, int d) {
  const float* row = nullptr;
  for (int r = 0; r < n_ranks; ++r)
    if (lab >= rd.lo[r] && lab < rd.lo[r] + rd.n[r]) row = rd.base[r] + (lab - rd.lo[r]) * d;
  return row;
}

// Row source of k_consumer_rows for row-sharded bases: ids are global labels, resolved per stream
// (0 image, 1 text) through the owners' rows as keds_exchange_attach_rows mapped them.
struct ConsumerShardRows {
  ShardRowsDb db[2];
  int n_ranks;
  __device__ __forceinline__ const float* operator()(bool img, long long id, int d) const {
    return shard_row(db[img ? 0 : 1], n_ranks, id, d);
  }
};

struct ShardConsume {
  ConsumeParams cons;  // feat / pool of the output rows [0, gridDim.x)
  int n_ranks, k, d, metric;
  long long row_lo;
  const float* D[2];  // merged [nq][k] per database
  const long long* I[2];
  ShardRowsDb db[2];
};

// Row `id` = slot id of a per-query table of row pointers (filled from the owners' bases).
struct PtrRows {
  const float* const* ptr;
  uintptr_t bits;  // OR of every base the pointers derive from (alignment test)
  __device__ __forceinline__ const float* operator()(unsigned int id) const { return ptr[id]; }
  __device__ __forceinline__ uintptr_t align_bits() const { return bits; }
};

__global__ void __launch_bounds__(RERANK_THREADS)
k_shard_consume(const ShardConsume p) {
  extern __shared__ __align__(16) uint8_t sc_smem[];
  float4* part = reinterpret_cast<float4*>(sc_smem);                          // cons.part4
  const float** ptr = reinterpret_cast<const float**>(part + p.cons.part4);   // k
  unsigned int* top_id = reinterpret_cast<unsigned int*>(ptr + p.k);          // k
  float* top_d = reinterpret_cast<float*>(top_id + p.k);                      // k
  float* w = top_d + p.k;                                                     // k
  const int s = blockIdx.y;
  const long long b = blockIdx.x, q = p.row_lo + b;
  const ShardRowsDb& rd = p.db[s];
  uintptr_t bits = 0;
  for (int r = 0; r < p.n_ranks; ++r) bits |= reinterpret_cast<uintptr_t>(rd.base[r]);
  griddep_wait();  // the merged rows are complete
  for (int j = threadIdx.x; j < p.k; j += blockDim.x) {
    const float* row = shard_row(rd, p.n_ranks, p.I[s][q * p.k + j], p.d);
    ptr[j] = row;
    top_id[j] = row != nullptr ? static_cast<unsigned int>(j) : 0xFFFFFFFFu;  // -1 padding: a zero row
    top_d[j] = p.D[s][q * p.k + j];
  }
  __syncthreads();
  consume_query<2>(p.cons, PtrRows{ptr, bits}, s, b, p.k, p.d, p.metric, top_id, top_d, w, part);
}

}  // namespace keds
