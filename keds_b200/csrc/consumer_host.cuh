// Host side of the neighbour consumer (keds_consumer_* in include/keds_knn.h): weight storage,
// TMA descriptors and the launch sequence. Included by api.cu (same translation unit: it uses
// the error / buffer / launch helpers defined there). All arithmetic is in neighbour_consumer.cuh.
#pragma once
#include "neighbour_consumer.cuh"

namespace {

constexpr int CONS_MAX_MLP = 8;      // hidden layers of the IM2TEXT MLP
constexpr int CONS_MAX_LAYERS = 8;   // cross-attention layers per stack

struct LinearW {
  DevBuf w, b;
  int out = 0, in = 0;
  bool set = false;
  CUtensorMap tm;     // boxes of 128 weight rows (k_linear_tf32)
  CUtensorMap tm32;   // boxes of 32 weight rows (k_linear_tf32_splitk)
};

// fp32 [rows][cols] with `ld` floats between rows -> boxes of {32 columns x 128 rows}, 128-byte
// swizzle; the TMA unit rounds to tf32 (to nearest, ties to even) and zero-fills out-of-range rows /
// columns.
int encode_f32_map(CUtensorMap* tm, const void* base, int64_t rows, int64_t cols, int64_t ld,
                   int box_rows = LIN_M) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return fail(KEDS_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstr[1] = {static_cast<cuuint64_t>(ld) * 4};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(LIN_K), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_TFLOAT32, 2, const_cast<void*>(base), gdim, gstr, box,
                  estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(KEDS_ERR_CUDA, "cuTensorMapEncodeTiled (f32) failed: CUresult %d", (int)r);
  return 0;
}

}  // namespace

struct keds_consumer {
  int device = 0;
  int d_in = 0, d_mid = 0, d_tok = 0, n_hidden = 0, n_layers = 0, heads = 0, dim_head = 0, inner = 0;
  bool finalized = false, attrs_set = false;
  int num_sms = 0;
  int attend_max = 0;  // dynamic shared memory the attention kernels may use (the device's opt-in limit)
  LinearW mlp[CONS_MAX_MLP + 1];               // n_hidden x (Linear + ReLU), then fc_out
  LinearW wq[2][CONS_MAX_LAYERS], wk[2][CONS_MAX_LAYERS], wv[2][CONS_MAX_LAYERS], wo[2][CONS_MAX_LAYERS];
  LinearW wkv[2];                              // all layers' to_k / to_v stacked: [L][k | v][inner] x d_tok
  DevBuf xin, hid[2], xm, kv, qb, ob, qn[2], err;
  int64_t launches = 0;
  struct AMap {  // TMA descriptor of an activation operand: a pure function of (base, rows, K, ld)
    const float* base;
    int64_t rows, ld;
    int K, box_rows;
    CUtensorMap tm;
  };
  std::vector<AMap> amaps;
  // diagnostics (keds_consumer_set_debug): per-CTA timestamps of the k_linear_tf32 launches of the
  // last forward, slot = launch index within the call
  bool debug = false;
  DevBuf tdump;
  int dbg_launch = 0;
  // ---- training (consumer_train_host.cuh) ----
  float* bound = nullptr;  // caller-owned flat parameter buffer (keds_consumer_bind_params)
  LinearW mlpT[CONS_MAX_MLP + 1], wqT[2][CONS_MAX_LAYERS], woT[2][CONS_MAX_LAYERS], wkvT[2];  // W^T: the weight operand of dX = dY W
  bool t_ready = false;
  struct Train {
    bool valid = false;
    int64_t B = 0;
    int k = 0;
    const float* masks[CONS_MAX_MLP] = {nullptr};
    DevBuf h[CONS_MAX_MLP];                                              // hidden activations [M][d_mid]
    DevBuf q[CONS_MAX_LAYERS], o[CONS_MAX_LAYERS], qin[CONS_MAX_LAYERS];  // per layer, both stacks side by side
    DevBuf dq[2], dO, dQ, dkv, dy, dh[2], ta, tb, dtok;                   // backward scratch
  } tr;
};
constexpr int CONS_DBG_LAUNCHES = 32;
constexpr int CONS_DBG_CTAS = 1024;

namespace {

LinearW* consumer_slot(keds_consumer* c, int kind, int stack, int layer) {
  if (kind == KEDS_CONSUMER_MLP) return (layer >= 0 && layer <= c->n_hidden) ? &c->mlp[layer] : nullptr;
  if (stack < 0 || stack > 1 || layer < 0 || layer >= c->n_layers) return nullptr;
  switch (kind) {
    case KEDS_CONSUMER_TO_Q: return &c->wq[stack][layer];
    case KEDS_CONSUMER_TO_K: return &c->wk[stack][layer];
    case KEDS_CONSUMER_TO_V: return &c->wv[stack][layer];
    case KEDS_CONSUMER_TO_OUT: return &c->wo[stack][layer];
    default: return nullptr;
  }
}

void consumer_slot_dims(const keds_consumer* c, int kind, int layer, int* out, int* in) {
  if (kind == KEDS_CONSUMER_MLP) {
    *in = layer == 0 ? c->d_in : c->d_mid;
    *out = layer == c->n_hidden ? c->d_tok : c->d_mid;
  } else if (kind == KEDS_CONSUMER_TO_OUT) {
    *in = c->inner;
    *out = c->d_tok;
  } else {
    *in = c->d_tok;
    *out = c->inner;
  }
}

// Descriptors of operands that live in scratch buffers are cached: a descriptor is a pure function
// of (base, rows, K, ld, box rows), so after the first call of a given shape every lookup hits
// (encoding costs ~5 us of host time per descriptor, more than the kernels they feed).
int consumer_cached_map(keds_consumer* c, const float* A, int64_t rows, int K, int64_t ld, int box_rows,
                        CUtensorMap* out) {
  for (const auto& e : c->amaps)
    if (e.base == A && e.rows == rows && e.K == K && e.ld == ld && e.box_rows == box_rows) {
      *out = e.tm;
      return 0;
    }
  keds_consumer::AMap e;
  e.base = A;
  e.rows = rows;
  e.K = K;
  e.ld = ld;
  e.box_rows = box_rows;
  CKS(encode_f32_map(&e.tm, A, rows, K, ld, box_rows));
  if (c->amaps.size() >= 256) c->amaps.clear();
  c->amaps.push_back(e);
  *out = e.tm;
  return 0;
}

// The five kernels behind one linear product (keds_debug_linear_plan reports these numbers).
enum LinearVariant { LIN_AUTO = 0, LIN_TILE128 = 1, LIN_TILE256 = 2, LIN_PERSISTENT = 3, LIN_SPLITK2 = 4, LIN_SPLITK4 = 5 };

// Which kernel runs C[M][N] (nz problems) on num_sms SMs. Host only.
int linear_variant(int64_t M, int N, int nz, int num_sms) {
  // tile width: fewer, wider tiles re-read A half as often but fill the SMs worse; pick by waves x
  // bytes per k-block (32 KB for 128 columns, 48 KB for 256)
  const long long mt = (M + LIN_M - 1) / LIN_M;
  const long long c128 = mt * ((N + 127) / 128) * nz, c256 = mt * ((N + 255) / 256) * nz;
  const long long sms = std::max(1, num_sms);
  // the one-tile and split-K kernels put the row tiles on grid.y (at most 65 535); the persistent
  // kernel walks a flat tile list, so it takes any M the consumer accepts (B (1 + 2k) <= 2^30)
  if (mt > 65535) return LIN_PERSISTENT;
  const bool wide = ((c256 + sms - 1) / sms) * 48 < ((c128 + sms - 1) / sms) * 32;
  // a handful of tiles only: 32-column tiles with the K range split over a cluster of SK_SPLIT CTAs
  if (c128 * 6 <= sms && num_sms >= SK_MAX_SPLIT) {
    const long long tiles = mt * ((N + SK_BN - 1) / SK_BN) * nz;
    return tiles * 4 <= sms ? LIN_SPLITK4 : LIN_SPLITK2;  // keep it to one wave
  }
  // more than two waves of wide tiles: one persistent CTA per SM with the epilogue of a tile
  // hidden under the main loop of the next
  if (wide && c256 > 2 * sms) return LIN_PERSISTENT;
  return wide ? LIN_TILE256 : LIN_TILE128;
}

// Launch one variant: C[z] = act(A[z] W[z]^T + b[z]) for z < nz, C[z] [M][N] with ldc floats between
// rows. ta*: A maps with LIN_M-row boxes; tw*: W maps with SK_BN-row boxes for the split-K variants,
// LIN_WBOX-row boxes otherwise.
int linear_launch(keds_consumer* c, int variant, const CUtensorMap& ta0, const CUtensorMap& ta1, const CUtensorMap& tw0,
                  const CUtensorMap& tw1, int64_t M, int N, int K, const float* b0, const float* b1, int relu, float* C0,
                  float* C1, int64_t ldc, int nz, cudaStream_t st) {
  LinearParams p;
  memset(&p, 0, sizeof p);
  p.M = static_cast<int>(M);
  p.N = N;
  p.K = K;
  p.relu = relu;
  p.bias[0] = b0;
  p.bias[1] = nz > 1 ? b1 : nullptr;
  p.C[0] = C0;
  p.C[1] = C1;
  p.ldc = ldc;
  p.err = c->err.as<uint32_t>();
  p.nz = nz;
  const long long mt = (M + LIN_M - 1) / LIN_M;
  if (variant == LIN_SPLITK2 || variant == LIN_SPLITK4) {
    const int split = variant == LIN_SPLITK4 ? 4 : 2;
    const dim3 gs(static_cast<unsigned>(split * ((p.N + SK_BN - 1) / SK_BN)), static_cast<unsigned>(mt),
                  static_cast<unsigned>(nz));
    if (c->debug && c->dbg_launch < CONS_DBG_LAUNCHES && gs.x * gs.y * gs.z <= (unsigned)CONS_DBG_CTAS)
      p.tdump = c->tdump.as<unsigned long long>() + static_cast<size_t>(c->dbg_launch) * CONS_DBG_CTAS * 5;
    c->dbg_launch++;
    if (split == 4)
      CKS(launch_kc(true, 4, k_linear_tf32_splitk<4>, gs, dim3(SK_THREADS), SK_SMEM_BYTES, st, ta0, ta1, tw0, tw1, p));
    else
      CKS(launch_kc(true, 2, k_linear_tf32_splitk<2>, gs, dim3(SK_THREADS), SK_SMEM_BYTES, st, ta0, ta1, tw0, tw1, p));
    c->launches++;
    return 0;
  }
  const int bn = variant == LIN_TILE128 ? 128 : 256;
  const dim3 grid(static_cast<unsigned>((p.N + bn - 1) / bn), static_cast<unsigned>(mt), static_cast<unsigned>(nz));
  if (c->debug && c->dbg_launch < CONS_DBG_LAUNCHES && grid.x * grid.y * grid.z <= (unsigned)CONS_DBG_CTAS)
    p.tdump = c->tdump.as<unsigned long long>() + static_cast<size_t>(c->dbg_launch) * CONS_DBG_CTAS * 5;
  c->dbg_launch++;
  if (variant == LIN_PERSISTENT) {
    p.tdump = nullptr;  // (no per-CTA stamps: one CTA walks many tiles)
    CKS(launch_k(true, k_linear_tf32_persistent, dim3(static_cast<unsigned>(std::max(1, c->num_sms))), dim3(PL_THREADS),
                 PL_SMEM_BYTES, st, ta0, ta1, tw0, tw1, p));
  } else if (variant == LIN_TILE256) {
    CKS(launch_k(true, k_linear_tf32<256>, grid, dim3(LIN_THREADS), LinCfg<256>::kSmemBytes, st, ta0, ta1, tw0, tw1, p));
  } else {
    CKS(launch_k(true, k_linear_tf32<128>, grid, dim3(LIN_THREADS), LinCfg<128>::kSmemBytes, st, ta0, ta1, tw0, tw1, p));
  }
  c->launches++;
  return 0;
}

int64_t round4(int64_t x) { return (x + 3) & ~int64_t(3); }

// dynamic shared memory of k_cross_attend and of k_cross_attend_bwd (twice as much): forward_train
// accepts only what its backward can also launch
size_t attend_smem(const keds_consumer* c, int k) { return static_cast<size_t>(c->heads) * (c->dim_head + k) * 4; }
size_t attend_bwd_smem(const keds_consumer* c, int k) { return 2 * attend_smem(c, k); }

// Which attention forward runs: k_cross_attend<64> (every key row read with 16-byte loads) for the
// reference's dim_head = 64 when every key / value row is 16-byte aligned, k_cross_attend<0> otherwise.
bool attend_dh64(int dim_head, int64_t ld_kv, int k_off, int v_off, const float* KV0, const float* KV1) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(KV0) | reinterpret_cast<uintptr_t>(KV1);
  return dim_head == 64 && (ld_kv & 3) == 0 && (k_off & 3) == 0 && (v_off & 3) == 0 && (a & 15) == 0;
}

// opt the attention kernels into the device's whole shared memory per block, once per handle
int attend_init(keds_consumer* c) {
  if (c->attend_max != 0) return 0;
  int optin = 0;
  CK(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, c->device));
  CK(cudaFuncSetAttribute(k_cross_attend<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
  CK(cudaFuncSetAttribute(k_cross_attend<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
  CK(cudaFuncSetAttribute(k_cross_attend_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
  c->attend_max = optin;
  return 0;
}

// C[z] = act(A[z] W[z]^T + b[z]) for z < nz; A[z]: [M][K] with lda floats between rows
int consumer_linear(keds_consumer* c, const float* A0, const float* A1, int64_t lda, int64_t M,
                    const LinearW* W0, const LinearW* W1, int relu, float* C0, float* C1, int64_t ldc,
                    int nz, cudaStream_t st) {
  CUtensorMap ta0, ta1;
  CKS(consumer_cached_map(c, A0, M, W0->in, lda, LIN_M, &ta0));
  if (nz > 1) CKS(consumer_cached_map(c, A1, M, W1->in, lda, LIN_M, &ta1)); else ta1 = ta0;
  const int v = linear_variant(M, W0->out, nz, c->num_sms);
  const bool sk = v == LIN_SPLITK2 || v == LIN_SPLITK4;
  const LinearW* W1e = nz > 1 ? W1 : W0;
  return linear_launch(c, v, ta0, ta1, sk ? W0->tm32 : W0->tm, sk ? W1e->tm32 : W1e->tm, M, W0->out, W0->in,
                       W0->b.as<float>(), nz > 1 ? W1->b.as<float>() : nullptr, relu, C0, C1, ldc, nz, st);
}

// kernel attributes, SM count and the error word: what any linear launch on `c` needs
int linear_init(keds_consumer* c) {
  if (!c->attrs_set) {
    CK(cudaFuncSetAttribute(k_linear_tf32<128>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            (int)LinCfg<128>::kSmemBytes));
    CK(cudaFuncSetAttribute(k_linear_tf32<256>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            (int)LinCfg<256>::kSmemBytes));
    CK(cudaFuncSetAttribute(k_linear_tf32_persistent, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            (int)PL_SMEM_BYTES));
    CK(cudaFuncSetAttribute(k_linear_tf32_splitk<2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            (int)SK_SMEM_BYTES));
    CK(cudaFuncSetAttribute(k_linear_tf32_splitk<4>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            (int)SK_SMEM_BYTES));
    CK(cudaDeviceGetAttribute(&c->num_sms, cudaDevAttrMultiProcessorCount, c->device));
    c->attrs_set = true;
  }
  CKS(c->err.ensure(16));
  CK(cudaMemset(c->err.p, 0, 16));
  return 0;
}

}  // namespace

extern "C" {

int keds_consumer_create(int d_in, int d_mid, int d_tok, int n_hidden, int n_layers, int heads,
                         int dim_head, int device, keds_consumer_t** out) {
  if (!out) return fail(KEDS_ERR_ARG, "consumer_create: out is NULL");
  *out = nullptr;
  if (d_in <= 0 || d_mid <= 0 || d_tok <= 0 || (d_in & 3) || (d_mid & 3) || (d_tok & 3))
    return fail(KEDS_ERR_ARG, "consumer_create: widths must be positive multiples of 4");
  if (n_hidden < 1 || n_hidden > CONS_MAX_MLP || n_layers < 1 || n_layers > CONS_MAX_LAYERS)
    return fail(KEDS_ERR_ARG, "consumer_create: n_hidden in [1,%d], n_layers in [1,%d]", CONS_MAX_MLP,
                CONS_MAX_LAYERS);
  if (heads < 1 || heads > 32 || dim_head < 1 || ((heads * dim_head) & 3))
    return fail(KEDS_ERR_ARG, "consumer_create: heads in [1,32], heads*dim_head a multiple of 4");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) {
    cudaGetLastError();
    return fail(KEDS_ERR_NO_GPU, "consumer_create: CUDA device %d not available (this library has no CPU path)", device);
  }
  keds_consumer* c = new keds_consumer();
  c->device = device;
  c->d_in = d_in;
  c->d_mid = d_mid;
  c->d_tok = d_tok;
  c->n_hidden = n_hidden;
  c->n_layers = n_layers;
  c->heads = heads;
  c->dim_head = dim_head;
  c->inner = heads * dim_head;
  *out = c;
  return 0;
}

void keds_consumer_free(keds_consumer_t* c) {
  if (!c) return;
  DeviceGuard g(c->device);
  for (auto& l : c->mlp) { l.w.release(); l.b.release(); }
  for (int z = 0; z < 2; ++z) {
    for (int l = 0; l < CONS_MAX_LAYERS; ++l)
      for (LinearW* s : {&c->wq[z][l], &c->wk[z][l], &c->wv[z][l], &c->wo[z][l]}) { s->w.release(); s->b.release(); }
    c->wkv[z].w.release();
    c->wkv[z].b.release();
  }
  for (DevBuf* b : {&c->xin, &c->hid[0], &c->hid[1], &c->xm, &c->kv, &c->qb, &c->ob, &c->qn[0], &c->qn[1], &c->err, &c->tdump})
    b->release();
  for (auto& l : c->mlpT) l.w.release();
  for (int z = 0; z < 2; ++z) {
    for (int l = 0; l < CONS_MAX_LAYERS; ++l) {
      c->wqT[z][l].w.release();
      c->woT[z][l].w.release();
    }
    c->wkvT[z].w.release();
  }
  for (int i = 0; i < CONS_MAX_MLP; ++i) c->tr.h[i].release();
  for (int l = 0; l < CONS_MAX_LAYERS; ++l) {
    c->tr.q[l].release();
    c->tr.o[l].release();
    c->tr.qin[l].release();
  }
  for (DevBuf* b : {&c->tr.dq[0], &c->tr.dq[1], &c->tr.dO, &c->tr.dQ, &c->tr.dkv, &c->tr.dy, &c->tr.dh[0], &c->tr.dh[1],
                    &c->tr.ta, &c->tr.tb, &c->tr.dtok})
    b->release();
  delete c;
}

int keds_consumer_set_linear(keds_consumer_t* c, int kind, int stack, int layer, const float* W,
                             const float* b, int out_features, int in_features) {
  if (!c || !W) return fail(KEDS_ERR_ARG, "consumer_set_linear: NULL argument");
  LinearW* s = consumer_slot(c, kind, stack, layer);
  if (!s) return fail(KEDS_ERR_ARG, "consumer_set_linear: no slot kind=%d stack=%d layer=%d", kind, stack, layer);
  int eo = 0, ei = 0;
  consumer_slot_dims(c, kind, layer, &eo, &ei);
  if (out_features != eo || in_features != ei)
    return fail(KEDS_ERR_ARG, "consumer_set_linear: slot kind=%d layer=%d wants [%d][%d], got [%d][%d]", kind,
                layer, eo, ei, out_features, in_features);
  DeviceGuard g(c->device);
  if (!g.ok) return fail(KEDS_ERR_CUDA, "cudaSetDevice(%d) failed", c->device);
  const size_t wb = static_cast<size_t>(eo) * ei * 4;
  if (!s->w.borrowed) {  // (bound parameters: the values go into the caller's flat buffer)
    CKS(s->w.ensure(wb));
    CKS(s->b.ensure(static_cast<size_t>(eo) * 4));
  }
  CK(cudaMemcpy(s->w.p, W, wb, cudaMemcpyDefault));
  if (b) CK(cudaMemcpy(s->b.p, b, static_cast<size_t>(eo) * 4, cudaMemcpyDefault));
  else CK(cudaMemset(s->b.p, 0, static_cast<size_t>(eo) * 4));
  s->out = eo;
  s->in = ei;
  s->set = true;
  c->finalized = false;
  return 0;
}

int keds_consumer_finalize(keds_consumer_t* c) {
  if (!c) return fail(KEDS_ERR_ARG, "consumer_finalize: NULL handle");
  DeviceGuard g(c->device);
  if (!g.ok) return fail(KEDS_ERR_CUDA, "cudaSetDevice(%d) failed", c->device);
  for (int i = 0; i <= c->n_hidden; ++i)
    if (!c->mlp[i].set) return fail(KEDS_ERR_ARG, "consumer_finalize: MLP layer %d not set", i);
  for (int z = 0; z < 2; ++z)
    for (int l = 0; l < c->n_layers; ++l)
      if (!c->wq[z][l].set || !c->wk[z][l].set || !c->wv[z][l].set || !c->wo[z][l].set)
        return fail(KEDS_ERR_ARG, "consumer_finalize: attention stack %d layer %d incomplete", z, l);
  CKS(linear_init(c));
  CKS(attend_init(c));
  const size_t wl = static_cast<size_t>(c->inner) * c->d_tok;  // one to_k or to_v matrix
  for (int z = 0; z < 2; ++z) {
    LinearW& kv = c->wkv[z];
    kv.out = c->n_layers * 2 * c->inner;
    kv.in = c->d_tok;
    if (c->bound == nullptr) {  // (bound parameters already live stacked in the caller's buffer)
      CKS(kv.w.ensure(static_cast<size_t>(kv.out) * kv.in * 4));
      CKS(kv.b.ensure(static_cast<size_t>(kv.out) * 4));
    }
    for (int l = 0; l < c->n_layers && c->bound == nullptr; ++l) {
      CK(cudaMemcpy(kv.w.as<float>() + (2 * l) * wl, c->wk[z][l].w.p, wl * 4, cudaMemcpyDeviceToDevice));
      CK(cudaMemcpy(kv.w.as<float>() + (2 * l + 1) * wl, c->wv[z][l].w.p, wl * 4, cudaMemcpyDeviceToDevice));
      CK(cudaMemcpy(kv.b.as<float>() + (2 * l) * c->inner, c->wk[z][l].b.p, c->inner * 4, cudaMemcpyDeviceToDevice));
      CK(cudaMemcpy(kv.b.as<float>() + (2 * l + 1) * c->inner, c->wv[z][l].b.p, c->inner * 4, cudaMemcpyDeviceToDevice));
    }
    kv.set = true;
    CKS(encode_f32_map(&kv.tm, kv.w.p, kv.out, kv.in, kv.in));
    CKS(encode_f32_map(&kv.tm32, kv.w.p, kv.out, kv.in, kv.in, SK_BN));
    for (int l = 0; l < c->n_layers; ++l) {
      CKS(encode_f32_map(&c->wq[z][l].tm, c->wq[z][l].w.p, c->inner, c->d_tok, c->d_tok));
      CKS(encode_f32_map(&c->wo[z][l].tm, c->wo[z][l].w.p, c->d_tok, c->inner, c->inner));
      CKS(encode_f32_map(&c->wq[z][l].tm32, c->wq[z][l].w.p, c->inner, c->d_tok, c->d_tok, SK_BN));
      CKS(encode_f32_map(&c->wo[z][l].tm32, c->wo[z][l].w.p, c->d_tok, c->inner, c->inner, SK_BN));
    }
  }
  for (int i = 0; i <= c->n_hidden; ++i) {
    CKS(encode_f32_map(&c->mlp[i].tm, c->mlp[i].w.p, c->mlp[i].out, c->mlp[i].in, c->mlp[i].in));
    CKS(encode_f32_map(&c->mlp[i].tm32, c->mlp[i].w.p, c->mlp[i].out, c->mlp[i].in, c->mlp[i].in, SK_BN));
  }
  CK(cudaDeviceSynchronize());
  c->finalized = true;
  return 0;
}

}  // extern "C"

namespace {

// Where the neighbour rows come from: the two resident bases of keds_consumer_forward[_train]
// (local ids), or every rank's rows of two row-sharded bases (global labels; sharded = true).
struct ConsumerRowSource {
  bool sharded = false;
  ConsumerLocalRows local{};
  ConsumerShardRows shard{};
};

ConsumerRowSource local_rows(const float* base_img, int64_t n_img, const float* base_txt, int64_t n_txt) {
  ConsumerRowSource src;
  src.local = ConsumerLocalRows{base_img, static_cast<long long>(n_img), base_txt, static_cast<long long>(n_txt)};
  return src;
}

// img / txt: this rank's shards of the two bases of `ex` (databases 0 and 1). Refuses, before
// anything is queued, what the rows of the exchange cannot serve: another device or width, a base
// that is not attached, this rank's rows moved or grown since the attach.
int shard_rows(const keds_consumer* c, keds_index* img, keds_index* txt, const keds_exchange* ex,
               ConsumerRowSource* src) {
  if (!c || !img || !txt || !ex) return fail(KEDS_ERR_ARG, "consumer_forward_sharded: NULL argument");
  if (img->device != c->device || txt->device != c->device || ex->device != c->device)
    return fail(KEDS_ERR_ARG, "consumer_forward_sharded: consumer, indices and exchange live on different devices");
  if (img->d != c->d_in || txt->d != c->d_in)
    return fail(KEDS_ERR_ARG, "consumer_forward_sharded: database widths %d / %d differ from the consumer's d_in %d",
                img->d, txt->d, c->d_in);
  keds_index* const dbs[2] = {img, txt};
  CKS(ex_check_rows(ex, dbs, 2));
  src->sharded = true;
  src->shard.db[0] = ex->rows[0];
  src->shard.db[1] = ex->rows[1];
  src->shard.n_ranks = ex->n_ranks;
  return 0;
}

// The forward pass. train = false: eval (dropout is the identity), scratch reused across layers.
// train = true: hidden activations, per-layer queries / attention outputs and layer inputs are
// kept for keds_consumer_backward; masks[i] (nullable) is hidden layer i's dropout multiplier.
int consumer_forward_impl(keds_consumer_t* c, const float* q, const ConsumerRowSource& src, const int64_t* I_img,
                          const int64_t* I_txt, const int32_t* perm, int64_t B, int k, float* tokens, void* stream,
                          bool train, const float* const* masks) {
  const ConsumerLocalRows& lr = src.local;
  if (!c || !q || !I_img || !I_txt || !tokens || (!src.sharded && (!lr.base_img || !lr.base_txt)))
    return fail(KEDS_ERR_ARG, "consumer_forward: NULL argument");
  if (!c->finalized) return fail(KEDS_ERR_ARG, "consumer_forward: call keds_consumer_finalize first");
  if (B < 0 || k <= 0 || k > 1024 || (!src.sharded && (lr.n_img < 0 || lr.n_txt < 0)))
    return fail(KEDS_ERR_ARG, "consumer_forward: bad B or k");
  if (B == 0) return 0;
  if (B * (1 + 2 * (int64_t)k) > (int64_t(1) << 30)) return fail(KEDS_ERR_ARG, "consumer_forward: batch too large");
  if (attend_smem(c, k) > static_cast<size_t>(c->attend_max))
    return fail(KEDS_ERR_ARG, "consumer_forward: heads * (dim_head + k) too large for the attention kernel");
  if (train && attend_bwd_smem(c, k) > static_cast<size_t>(c->attend_max))
    return fail(KEDS_ERR_ARG, "consumer_forward_train: heads * (dim_head + k) too large for the attention backward");
  for (const void* ptr : {(const void*)q, (const void*)lr.base_img, (const void*)lr.base_txt, (const void*)I_img,
                          (const void*)I_txt, (const void*)tokens})
    if ((ptr || !src.sharded) && !locate(ptr))
      return fail(KEDS_ERR_ARG, "consumer_forward: all buffers must be device memory");
  DeviceGuard g(c->device);
  if (!g.ok) return fail(KEDS_ERR_CUDA, "cudaSetDevice(%d) failed", c->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t Bk = B * k, M = B + 2 * Bk;
  const int L = c->n_layers, inner = c->inner, dt = c->d_tok;
  const int64_t kvw = static_cast<int64_t>(L) * 2 * inner;
  CKS(c->xin.ensure(static_cast<size_t>(M) * c->d_in * 4));
  if (train) {
    c->tr.valid = false;
    for (int i = 0; i < c->n_hidden; ++i) {
      CKS(c->tr.h[i].ensure(static_cast<size_t>(M) * c->d_mid * 4));
      c->tr.masks[i] = masks ? masks[i] : nullptr;
      if (c->tr.masks[i] && !locate(c->tr.masks[i]))
        return fail(KEDS_ERR_ARG, "consumer_forward_train: dropout masks must be device memory");
    }
    for (int l = 0; l < L; ++l) {
      CKS(c->tr.q[l].ensure(static_cast<size_t>(2) * B * inner * 4));
      CKS(c->tr.o[l].ensure(static_cast<size_t>(2) * B * inner * 4));
      if (l > 0) CKS(c->tr.qin[l].ensure(static_cast<size_t>(2) * B * dt * 4));
    }
  } else {
    CKS(c->hid[0].ensure(static_cast<size_t>(M) * c->d_mid * 4));
    CKS(c->hid[1].ensure(static_cast<size_t>(M) * c->d_mid * 4));
  }
  CKS(c->xm.ensure(static_cast<size_t>(M) * dt * 4));
  CKS(c->kv.ensure(static_cast<size_t>(2) * Bk * kvw * 4));
  CKS(c->qb.ensure(static_cast<size_t>(2) * B * inner * 4));
  CKS(c->ob.ensure(static_cast<size_t>(2) * B * inner * 4));
  CKS(c->qn[0].ensure(static_cast<size_t>(2) * B * dt * 4));
  CKS(c->qn[1].ensure(static_cast<size_t>(2) * B * dt * 4));

  c->dbg_launch = 0;
  if (c->debug) {
    CKS(c->tdump.ensure(static_cast<size_t>(CONS_DBG_LAUNCHES) * CONS_DBG_CTAS * 5 * 8));
    CK(cudaMemsetAsync(c->tdump.p, 0, c->tdump.cap, st));
  }

  // rows of the MLP input: [queries | image neighbours | text neighbours], one launch
  float* xin = c->xin.as<float>();
  const unsigned gblocks = static_cast<unsigned>(((B + 2 * Bk) * 32 + 255) / 256);
  const long long* Ii = reinterpret_cast<const long long*>(I_img);
  const long long* It = reinterpret_cast<const long long*>(I_txt);
  if (src.sharded)
    k_consumer_rows<<<gblocks, 256, 0, st>>>(q, src.shard, Ii, It, perm, B, k, c->d_in, xin);
  else
    k_consumer_rows<<<gblocks, 256, 0, st>>>(q, src.local, Ii, It, perm, B, k, c->d_in, xin);
  CK(cudaGetLastError());
  c->launches += 1;

  // IM2TEXT: hidden layers (Linear + ReLU; dropout is the identity in eval), then fc_out
  const float* cur = xin;
  int cur_w = c->d_in;
  for (int i = 0; i < c->n_hidden; ++i) {
    float* h = train ? c->tr.h[i].as<float>() : c->hid[i & 1].as<float>();
    const float* mask = train ? c->tr.masks[i] : nullptr;
    CKS(consumer_linear(c, cur, nullptr, cur_w, M, &c->mlp[i], nullptr, mask ? 0 : 1, h, nullptr, c->d_mid, 1, st));
    if (mask) {  // Linear -> Dropout -> ReLU (src/model/model.py:110-116)
      const long long n = static_cast<long long>(M) * c->d_mid;
      CKS(launch_k(true, k_mask_relu, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, h, mask, n));
      c->launches++;
    }
    cur = h;
    cur_w = c->d_mid;
  }
  float* xm = c->xm.as<float>();
  CKS(consumer_linear(c, cur, nullptr, cur_w, M, &c->mlp[c->n_hidden], nullptr, 0, xm, nullptr, dt, 1, st));

  // keys and values of every layer of both stacks in one launch
  float* kv0 = c->kv.as<float>();
  float* kv1 = kv0 + Bk * kvw;
  CKS(consumer_linear(c, xm + B * dt, xm + (B + Bk) * dt, dt, Bk, &c->wkv[0], &c->wkv[1], 0, kv0, kv1, kvw, 2, st));

  // the single query token walks the layers; both stacks side by side (blockIdx.z / .y)
  float* qb0 = c->qb.as<float>();
  float* qb1 = qb0 + B * inner;
  float* ob0 = c->ob.as<float>();
  float* ob1 = ob0 + B * inner;
  const float* qc0 = xm;
  const float* qc1 = xm;
  int64_t ldq = dt;
  for (int l = 0; l < L; ++l) {
    if (train) {  // every layer keeps its own query and attention output for the backward
      qb0 = c->tr.q[l].as<float>();
      qb1 = qb0 + B * inner;
      ob0 = c->tr.o[l].as<float>();
      ob1 = ob0 + B * inner;
    }
    CKS(consumer_linear(c, qc0, qc1, ldq, B, &c->wq[0][l], &c->wq[1][l], 0, qb0, qb1, inner, 2, st));
    AttendParams ap;
    memset(&ap, 0, sizeof ap);
    ap.B = static_cast<int>(B);
    ap.k = k;
    ap.heads = c->heads;
    ap.dim_head = c->dim_head;
    ap.Q[0] = qb0;
    ap.Q[1] = qb1;
    ap.KV[0] = kv0;
    ap.KV[1] = kv1;
    ap.O[0] = ob0;
    ap.O[1] = ob1;
    ap.ld_kv = kvw;
    ap.k_off = (2 * l) * inner;
    ap.v_off = (2 * l + 1) * inner;
    ap.scale = 1.0f / sqrtf(static_cast<float>(c->dim_head));
    const bool dh64 = attend_dh64(c->dim_head, kvw, ap.k_off, ap.v_off, kv0, kv1);
    CKS(launch_k(true, dh64 ? k_cross_attend<64> : k_cross_attend<0>, dim3(static_cast<unsigned>(B), 2),
                 dim3(32 * c->heads), attend_smem(c, k), st, ap));
    c->launches++;
    float *o0, *o1;
    int64_t ldo;
    if (l == L - 1) {  // last layer writes tokens[:, 0, :] (image stack) and tokens[:, 1, :] (text stack)
      o0 = tokens;
      o1 = tokens + dt;
      ldo = 3 * static_cast<int64_t>(dt);
    } else {
      o0 = train ? c->tr.qin[l + 1].as<float>() : c->qn[l & 1].as<float>();
      o1 = o0 + B * dt;
      ldo = dt;
    }
    CKS(consumer_linear(c, ob0, ob1, inner, B, &c->wo[0][l], &c->wo[1][l], 0, o0, o1, ldo, 2, st));
    qc0 = o0;
    qc1 = o1;
    ldq = ldo;
  }
  // tokens[:, 2, :] = img2text(query features)
  CK(cudaMemcpy2DAsync(tokens + 2 * dt, static_cast<size_t>(3) * dt * 4, xm, static_cast<size_t>(dt) * 4,
                       static_cast<size_t>(dt) * 4, static_cast<size_t>(B), cudaMemcpyDeviceToDevice, st));
  if (train) {
    c->tr.B = B;
    c->tr.k = k;
    c->tr.valid = true;
  }
  return 0;
}

}  // namespace

extern "C" {

int keds_consumer_forward(keds_consumer_t* c, const float* q, const float* base_img, int64_t n_img,
                          const float* base_txt, int64_t n_txt, const int64_t* I_img, const int64_t* I_txt,
                          const int32_t* perm, int64_t B, int k, float* tokens, void* stream) {
  return consumer_forward_impl(c, q, local_rows(base_img, n_img, base_txt, n_txt), I_img, I_txt, perm, B, k, tokens,
                               stream, false, nullptr);
}

int keds_consumer_forward_sharded(keds_consumer_t* c, keds_index_t* img, keds_index_t* txt, keds_exchange_t* ex,
                                  const float* feat, const int64_t* I_img, const int64_t* I_txt, const int32_t* perm,
                                  int64_t B, int k, float* tokens, void* stream) {
  ConsumerRowSource src;
  CKS(shard_rows(c, img, txt, ex, &src));
  return consumer_forward_impl(c, feat, src, I_img, I_txt, perm, B, k, tokens, stream, false, nullptr);
}

int keds_consumer_set_debug(keds_consumer_t* c, int enable) {
  if (!c) return fail(KEDS_ERR_ARG, "consumer_set_debug: NULL handle");
  c->debug = enable != 0;
  return 0;
}

int keds_consumer_debug_timeline(keds_consumer_t* c, int launch, uint64_t* out, int64_t n_ctas) {
  if (!c || !out || launch < 0 || launch >= CONS_DBG_LAUNCHES || n_ctas < 0 || n_ctas > CONS_DBG_CTAS)
    return fail(KEDS_ERR_ARG, "consumer_debug_timeline: bad argument");
  if (!c->tdump.p) return fail(KEDS_ERR_ARG, "consumer_debug_timeline: debug was not enabled");
  DeviceGuard g(c->device);
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(out, c->tdump.as<unsigned long long>() + static_cast<size_t>(launch) * CONS_DBG_CTAS * 5,
                static_cast<size_t>(n_ctas) * 5 * 8, cudaMemcpyDeviceToHost));
  return 0;
}

int keds_consumer_check(keds_consumer_t* c, void* stream, int64_t* launches) {
  if (!c) return fail(KEDS_ERR_ARG, "consumer_check: NULL handle");
  DeviceGuard g(c->device);
  if (!g.ok) return fail(KEDS_ERR_CUDA, "cudaSetDevice(%d) failed", c->device);
  CK(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  if (launches) *launches = c->launches;
  if (!c->err.p) return 0;
  uint32_t e = 0;
  CK(cudaMemcpy(&e, c->err.p, 4, cudaMemcpyDeviceToHost));
  if (e != 0) {
    CK(cudaMemset(c->err.p, 0, 4));
    return fail(KEDS_ERR_KERNEL, "consumer kernel pipeline timed out (code 0x%x)", e);
  }
  return 0;
}

int keds_debug_linear_plan(int64_t M, int N, int nz, int num_sms, int32_t* variant) {
  if (!variant || M <= 0 || N <= 0 || nz < 1 || nz > 2 || num_sms <= 0)
    return fail(KEDS_ERR_ARG, "debug_linear_plan: bad argument");
  *variant = linear_variant(M, N, nz, num_sms);
  return 0;
}

int keds_consumer_debug_linear(keds_consumer_t* c, int variant, const float* A0, const float* A1, int64_t lda,
                               int64_t M, int K, const float* W0, const float* W1, const float* b0, const float* b1,
                               int N, int relu, float* C0, float* C1, int64_t ldc, int nz, void* stream) {
  if (!c || variant < LIN_AUTO || variant > LIN_SPLITK4 || nz < 1 || nz > 2 || M <= 0 || K <= 0 || N <= 0)
    return fail(KEDS_ERR_ARG, "consumer_debug_linear: bad handle, variant, nz or shape");
  if ((M + LIN_M - 1) / LIN_M > 65535 || ldc < N)
    return fail(KEDS_ERR_ARG, "consumer_debug_linear: M too large or ldc < N");
  const int64_t ldw = round4(K);
  if ((lda & 3) || lda < K) return fail(KEDS_ERR_ARG, "consumer_debug_linear: lda must be a multiple of 4 and >= K");
  for (int z = 0; z < nz; ++z) {
    const float* A = z ? A1 : A0;
    const float* W = z ? W1 : W0;
    const float* b = z ? b1 : b0;
    const float* C = z ? C1 : C0;
    if (!A || !W || !C || (reinterpret_cast<uintptr_t>(A) & 15) || (reinterpret_cast<uintptr_t>(W) & 15) ||
        (reinterpret_cast<uintptr_t>(C) & 3))
      return fail(KEDS_ERR_ARG, "consumer_debug_linear: A, W 16-byte and C 4-byte aligned, none NULL");
    if (!locate(A) || !locate(W) || !locate(C) || (b && !locate(b)))
      return fail(KEDS_ERR_ARG, "consumer_debug_linear: all buffers must be device memory");
  }
  DeviceGuard g(c->device);
  if (!g.ok) return fail(KEDS_ERR_CUDA, "cudaSetDevice(%d) failed", c->device);
  if (!c->attrs_set) CKS(linear_init(c));
  if (variant == LIN_AUTO) variant = linear_variant(M, N, nz, c->num_sms);
  const bool sk = variant == LIN_SPLITK2 || variant == LIN_SPLITK4;
  CUtensorMap ta[2], tw[2];
  for (int z = 0; z < nz; ++z) {
    CKS(encode_f32_map(&ta[z], z ? A1 : A0, M, K, lda, LIN_M));
    CKS(encode_f32_map(&tw[z], z ? W1 : W0, N, K, ldw, sk ? SK_BN : LIN_WBOX));
  }
  if (nz == 1) {
    ta[1] = ta[0];
    tw[1] = tw[0];
  }
  return linear_launch(c, variant, ta[0], ta[1], tw[0], tw[1], M, N, K, b0, b1, relu, C0, C1, ldc, nz,
                       static_cast<cudaStream_t>(stream));
}

int keds_consumer_debug_attend(keds_consumer_t* c, int variant, int backward, int64_t B, int k, const float* Q0,
                               const float* Q1, const float* KV0, const float* KV1, int64_t ld_kv, int k_off,
                               int v_off, const float* dO0, const float* dO1, float* out0, float* out1, float* dKV0,
                               float* dKV1, void* stream) {
  if (!c || variant < 0 || variant > 2 || (backward && variant != 0) || B < 1 || B > INT32_MAX || k < 1 || k > 1024)
    return fail(KEDS_ERR_ARG, "consumer_debug_attend: bad handle, variant, B or k");
  const int inner = c->inner;
  if (k_off < 0 || v_off < 0 || ld_kv < static_cast<int64_t>(std::max(k_off, v_off)) + inner)
    return fail(KEDS_ERR_ARG, "consumer_debug_attend: key / value columns outside ld_kv");
  const float* need[] = {Q0, Q1, KV0, KV1, out0, out1, backward ? dO0 : Q0, backward ? dO1 : Q0,
                         backward ? dKV0 : Q0, backward ? dKV1 : Q0};
  for (const float* p : need)
    if (!p) return fail(KEDS_ERR_ARG, "consumer_debug_attend: NULL buffer");
  for (const float* p : need)
    if (!locate(p)) return fail(KEDS_ERR_ARG, "consumer_debug_attend: all buffers must be device memory");
  if (variant == 2 && !attend_dh64(c->dim_head, ld_kv, k_off, v_off, KV0, KV1))
    return fail(KEDS_ERR_ARG, "consumer_debug_attend: k_cross_attend<64> needs dim_head 64, ld_kv, k_off, v_off "
                              "multiples of 4 and 16-byte aligned KV");
  DeviceGuard g(c->device);
  if (!g.ok) return fail(KEDS_ERR_CUDA, "cudaSetDevice(%d) failed", c->device);
  CKS(attend_init(c));
  const size_t smem = backward ? attend_bwd_smem(c, k) : attend_smem(c, k);
  if (smem > static_cast<size_t>(c->attend_max))
    return fail(KEDS_ERR_ARG, "consumer_debug_attend: heads * (dim_head + k) too large for the attention kernel");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const float scale = 1.0f / sqrtf(static_cast<float>(c->dim_head));  // as the forward and backward compute it
  const dim3 grid(static_cast<unsigned>(B), 2), block(32 * c->heads);
  if (backward) {
    AttendBwdParams ap;
    memset(&ap, 0, sizeof ap);
    ap.B = static_cast<int>(B);
    ap.k = k;
    ap.heads = c->heads;
    ap.dim_head = c->dim_head;
    ap.Q[0] = Q0;
    ap.Q[1] = Q1;
    ap.KV[0] = KV0;
    ap.KV[1] = KV1;
    ap.dO[0] = dO0;
    ap.dO[1] = dO1;
    ap.dQ[0] = out0;
    ap.dQ[1] = out1;
    ap.dKV[0] = dKV0;
    ap.dKV[1] = dKV1;
    ap.ld_kv = ld_kv;
    ap.k_off = k_off;
    ap.v_off = v_off;
    ap.scale = scale;
    CKS(launch_k(true, k_cross_attend_bwd, grid, block, smem, st, ap));
  } else {
    AttendParams ap;
    memset(&ap, 0, sizeof ap);
    ap.B = static_cast<int>(B);
    ap.k = k;
    ap.heads = c->heads;
    ap.dim_head = c->dim_head;
    ap.Q[0] = Q0;
    ap.Q[1] = Q1;
    ap.KV[0] = KV0;
    ap.KV[1] = KV1;
    ap.O[0] = out0;
    ap.O[1] = out1;
    ap.ld_kv = ld_kv;
    ap.k_off = k_off;
    ap.v_off = v_off;
    ap.scale = scale;
    const bool dh64 = variant == 0 ? attend_dh64(c->dim_head, ld_kv, k_off, v_off, KV0, KV1) : variant == 2;
    CKS(launch_k(true, dh64 ? k_cross_attend<64> : k_cross_attend<0>, grid, block, smem, st, ap));
  }
  c->launches++;
  return 0;
}

}  // extern "C"
