// Training side of the neighbour consumer (keds_consumer_bind_params / _forward_train / _backward
// in include/keds_knn.h): the modules of src/trainer.py:59-69 while they are being optimised
// (backward at src/trainer.py:462-474). Included by api.cu behind consumer_host.cuh.
//
// Parameters live in ONE flat caller-owned buffer (a torch Parameter): the optimiser updates it in
// place, the handle reads through it, nothing is copied per step. Gradients come back in a second
// flat buffer of the same layout:
//
//   for i in 0 .. n_hidden:       W_i [out][in], b_i [out]              (IM2TEXT layers.i.0, fc_out)
//   for stack in (image, text):   Wkv [L][k | v][inner][d_tok], bkv [L][k | v][inner]   (to_k / to_v, stacked)
//                                 for l in 0 .. L-1:  Wq [inner][d_tok], bq, Wo [d_tok][inner], bo
//
// Every product is the tf32 tcgen05 GEMM of neighbour_consumer.cuh with the operand roles turned:
// dX = dY W uses W^T as the "weight" operand (refreshed from the parameters at the start of every
// backward), dW = dY^T X uses the transposed activation as the weight operand.
#pragma once

namespace {

struct ConsLayout {
  int64_t mlp_w[CONS_MAX_MLP + 1], mlp_b[CONS_MAX_MLP + 1];
  int64_t kv_w[2], kv_b[2];
  int64_t q_w[2][CONS_MAX_LAYERS], q_b[2][CONS_MAX_LAYERS], o_w[2][CONS_MAX_LAYERS], o_b[2][CONS_MAX_LAYERS];
  int64_t total;
};

ConsLayout consumer_layout(const keds_consumer* c) {
  ConsLayout y;
  memset(&y, 0, sizeof y);
  int64_t off = 0;
  auto take = [&](int64_t n) {
    const int64_t o = off;
    off += (n + 3) & ~int64_t(3);  // every block 16-byte aligned (TMA base addresses)
    return o;
  };
  for (int i = 0; i <= c->n_hidden; ++i) {
    int out = 0, in = 0;
    consumer_slot_dims(c, KEDS_CONSUMER_MLP, i, &out, &in);
    y.mlp_w[i] = take(static_cast<int64_t>(out) * in);
    y.mlp_b[i] = take(out);
  }
  const int64_t kvw = static_cast<int64_t>(c->n_layers) * 2 * c->inner;
  for (int z = 0; z < 2; ++z) {
    y.kv_w[z] = take(kvw * c->d_tok);
    y.kv_b[z] = take(kvw);
    for (int l = 0; l < c->n_layers; ++l) {
      y.q_w[z][l] = take(static_cast<int64_t>(c->inner) * c->d_tok);
      y.q_b[z][l] = take(c->inner);
      y.o_w[z][l] = take(static_cast<int64_t>(c->d_tok) * c->inner);
      y.o_b[z][l] = take(c->d_tok);
    }
  }
  y.total = off;
  return y;
}

// a weight-like operand [out][in] with `ld` floats between rows, living in scratch memory
int train_weight(keds_consumer* c, const float* W, int out, int in, int64_t ld, LinearW* w) {
  w->out = out;
  w->in = in;
  w->set = true;
  CKS(consumer_cached_map(c, W, out, in, ld, LIN_WBOX, &w->tm));
  CKS(consumer_cached_map(c, W, out, in, ld, SK_BN, &w->tm32));
  return 0;
}

// out[c][r] = in[r][c]
int train_transpose(keds_consumer* c, const float* in, int64_t ld_in, int64_t rows, int cols, float* out, int64_t ld_out,
                    cudaStream_t st) {
  CKS(launch_k(true, k_transpose_f32, transpose_grid(rows, cols), dim3(32, 8), 0, st, in, static_cast<long long>(ld_in),
               static_cast<int>(rows), cols, out, static_cast<long long>(ld_out)));
  c->launches++;
  return 0;
}

int train_colsum(keds_consumer* c, const float* in, int64_t ld, int64_t rows, int cols, float* out, cudaStream_t st) {
  CKS(launch_k(true, k_colsum, dim3(static_cast<unsigned>((cols + 31) / 32)), dim3(256), 0, st, in,
               static_cast<long long>(ld), static_cast<long long>(rows), cols, out));
  c->launches++;
  return 0;
}

// dW[z] [n_out][n_in] = dY[z]^T X[z] for z < nz (dY[z]: [rows][n_out], X[z]: [rows][n_in]); the two
// transposed operands go through ta / tb ([nz][n][ld] each)
int train_weight_grad(keds_consumer* c, const float* dY0, const float* dY1, int64_t ld_dy, const float* X0,
                      const float* X1, int64_t ld_x, int64_t rows, int n_out, int n_in, float* dW0, float* dW1,
                      int nz, cudaStream_t st) {
  const int64_t ldr = round4(rows);
  float* ta = c->tr.ta.as<float>();
  float* tb = c->tr.tb.as<float>();
  float* ta1 = ta + static_cast<int64_t>(n_out) * ldr;
  float* tb1 = tb + static_cast<int64_t>(n_in) * ldr;
  CKS(train_transpose(c, dY0, ld_dy, rows, n_out, ta, ldr, st));
  CKS(train_transpose(c, X0, ld_x, rows, n_in, tb, ldr, st));
  if (nz > 1) {
    CKS(train_transpose(c, dY1, ld_dy, rows, n_out, ta1, ldr, st));
    CKS(train_transpose(c, X1, ld_x, rows, n_in, tb1, ldr, st));
  }
  LinearW w0, w1;
  CKS(train_weight(c, tb, n_in, static_cast<int>(rows), ldr, &w0));
  if (nz > 1) CKS(train_weight(c, tb1, n_in, static_cast<int>(rows), ldr, &w1));
  return consumer_linear(c, ta, nz > 1 ? ta1 : nullptr, ldr, n_out, &w0, nz > 1 ? &w1 : nullptr, 0, dW0, dW1, n_in, nz, st);
}

// (re)allocate the transposed-weight operands and refresh them from the current parameters
int consumer_refresh_transposes(keds_consumer* c, cudaStream_t st) {
  auto one = [&](const LinearW& w, LinearW& t) -> int {
    const size_t bytes = static_cast<size_t>(w.out) * w.in * 4;
    const bool fresh = t.w.cap < bytes || !t.set;
    CKS(t.w.ensure(bytes));
    t.out = w.in;
    t.in = w.out;
    if (fresh) {
      CKS(encode_f32_map(&t.tm, t.w.p, t.out, t.in, t.in));
      CKS(encode_f32_map(&t.tm32, t.w.p, t.out, t.in, t.in, SK_BN));
      t.set = true;
    }
    return train_transpose(c, w.w.as<float>(), w.in, w.out, w.in, t.w.as<float>(), w.out, st);
  };
  for (int i = 1; i <= c->n_hidden; ++i) CKS(one(c->mlp[i], c->mlpT[i]));
  for (int z = 0; z < 2; ++z) {
    CKS(one(c->wkv[z], c->wkvT[z]));
    for (int l = 0; l < c->n_layers; ++l) {
      CKS(one(c->wq[z][l], c->wqT[z][l]));
      CKS(one(c->wo[z][l], c->woT[z][l]));
    }
  }
  return 0;
}

}  // namespace

extern "C" {

int64_t keds_consumer_param_count(const keds_consumer_t* c) { return c ? consumer_layout(c).total : -1; }

int keds_consumer_param_offset(const keds_consumer_t* c, int kind, int stack, int layer, int64_t* w_off, int64_t* b_off,
                               int64_t* rows, int64_t* cols) {
  if (!c || !w_off || !b_off || !rows || !cols) return fail(KEDS_ERR_ARG, "consumer_param_offset: NULL argument");
  const ConsLayout y = consumer_layout(c);
  if (kind == KEDS_CONSUMER_MLP) {
    if (layer < 0 || layer > c->n_hidden) return fail(KEDS_ERR_ARG, "consumer_param_offset: no MLP layer %d", layer);
    int out = 0, in = 0;
    consumer_slot_dims(c, kind, layer, &out, &in);
    *w_off = y.mlp_w[layer];
    *b_off = y.mlp_b[layer];
    *rows = out;
    *cols = in;
    return 0;
  }
  if (stack < 0 || stack > 1 || layer < 0 || layer >= c->n_layers)
    return fail(KEDS_ERR_ARG, "consumer_param_offset: no slot stack=%d layer=%d", stack, layer);
  const int64_t wl = static_cast<int64_t>(c->inner) * c->d_tok;
  switch (kind) {
    case KEDS_CONSUMER_TO_Q: *w_off = y.q_w[stack][layer]; *b_off = y.q_b[stack][layer]; *rows = c->inner; *cols = c->d_tok; return 0;
    case KEDS_CONSUMER_TO_OUT: *w_off = y.o_w[stack][layer]; *b_off = y.o_b[stack][layer]; *rows = c->d_tok; *cols = c->inner; return 0;
    case KEDS_CONSUMER_TO_K:
      *w_off = y.kv_w[stack] + (2 * layer) * wl; *b_off = y.kv_b[stack] + (2 * layer) * c->inner; *rows = c->inner; *cols = c->d_tok; return 0;
    case KEDS_CONSUMER_TO_V:
      *w_off = y.kv_w[stack] + (2 * layer + 1) * wl; *b_off = y.kv_b[stack] + (2 * layer + 1) * c->inner; *rows = c->inner; *cols = c->d_tok; return 0;
    default: return fail(KEDS_ERR_ARG, "consumer_param_offset: unknown kind %d", kind);
  }
}

int keds_consumer_bind_params(keds_consumer_t* c, float* params) {
  if (!c || !params) return fail(KEDS_ERR_ARG, "consumer_bind_params: NULL argument");
  if (!locate(params) || (reinterpret_cast<uintptr_t>(params) & 15))
    return fail(KEDS_ERR_ARG, "consumer_bind_params: params must be 16-byte aligned device memory");
  if ((c->inner * c->d_tok) & 3) return fail(KEDS_ERR_ARG, "consumer_bind_params: inner * d_tok must be a multiple of 4");
  DeviceGuard g(c->device);
  if (!g.ok) return fail(KEDS_ERR_CUDA, "cudaSetDevice(%d) failed", c->device);
  const ConsLayout y = consumer_layout(c);
  auto view = [&](LinearW& s, int64_t w_off, int64_t b_off, int out, int in) {
    s.w.borrow(params + w_off, static_cast<size_t>(out) * in * 4);
    s.b.borrow(params + b_off, static_cast<size_t>(out) * 4);
    s.out = out;
    s.in = in;
    s.set = true;
  };
  for (int i = 0; i <= c->n_hidden; ++i) {
    int out = 0, in = 0;
    consumer_slot_dims(c, KEDS_CONSUMER_MLP, i, &out, &in);
    view(c->mlp[i], y.mlp_w[i], y.mlp_b[i], out, in);
  }
  const int64_t wl = static_cast<int64_t>(c->inner) * c->d_tok;
  const int kvw = c->n_layers * 2 * c->inner;
  for (int z = 0; z < 2; ++z) {
    view(c->wkv[z], y.kv_w[z], y.kv_b[z], kvw, c->d_tok);
    for (int l = 0; l < c->n_layers; ++l) {
      view(c->wk[z][l], y.kv_w[z] + (2 * l) * wl, y.kv_b[z] + (2 * l) * c->inner, c->inner, c->d_tok);
      view(c->wv[z][l], y.kv_w[z] + (2 * l + 1) * wl, y.kv_b[z] + (2 * l + 1) * c->inner, c->inner, c->d_tok);
      view(c->wq[z][l], y.q_w[z][l], y.q_b[z][l], c->inner, c->d_tok);
      view(c->wo[z][l], y.o_w[z][l], y.o_b[z][l], c->d_tok, c->inner);
    }
  }
  c->bound = params;
  c->amaps.clear();
  c->t_ready = false;
  return keds_consumer_finalize(c);
}

int keds_consumer_forward_train(keds_consumer_t* c, const float* feat, const float* base_img, int64_t n_img,
                                const float* base_txt, int64_t n_txt, const int64_t* I_img, const int64_t* I_txt,
                                const int32_t* perm, int64_t B, int k, const float* const* masks, float* tokens,
                                void* stream) {
  return consumer_forward_impl(c, feat, local_rows(base_img, n_img, base_txt, n_txt), I_img, I_txt, perm, B, k, tokens,
                               stream, true, masks);
}

int keds_consumer_forward_train_sharded(keds_consumer_t* c, keds_index_t* img, keds_index_t* txt, keds_exchange_t* ex,
                                        const float* feat, const int64_t* I_img, const int64_t* I_txt,
                                        const int32_t* perm, int64_t B, int k, const float* const* masks,
                                        float* tokens, void* stream) {
  ConsumerRowSource src;
  CKS(shard_rows(c, img, txt, ex, &src));
  return consumer_forward_impl(c, feat, src, I_img, I_txt, perm, B, k, tokens, stream, true, masks);
}

int keds_consumer_debug_hidden(keds_consumer_t* c, int layer, float* out, int64_t n, void* stream) {
  if (!c || !out || layer < 0 || layer >= c->n_hidden) return fail(KEDS_ERR_ARG, "consumer_debug_hidden: bad argument");
  const int64_t have = c->tr.B * (1 + 2 * static_cast<int64_t>(c->tr.k)) * c->d_mid;
  if (c->tr.h[layer].p == nullptr || n != have)
    return fail(KEDS_ERR_ARG, "consumer_debug_hidden: expected %lld floats of the last forward_train", (long long)have);
  DeviceGuard g(c->device);
  CK(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  CK(cudaMemcpy(out, c->tr.h[layer].p, static_cast<size_t>(n) * 4, cudaMemcpyDefault));
  return 0;
}

int keds_consumer_backward(keds_consumer_t* c, const float* dtokens, float* grads, void* stream) {
  if (!c || !dtokens || !grads) return fail(KEDS_ERR_ARG, "consumer_backward: NULL argument");
  if (!c->finalized || !c->tr.valid) return fail(KEDS_ERR_ARG, "consumer_backward: no keds_consumer_forward_train to differentiate");
  if (!locate(dtokens) || !locate(grads) || (reinterpret_cast<uintptr_t>(grads) & 15))
    return fail(KEDS_ERR_ARG, "consumer_backward: dtokens / grads must be device memory (grads 16-byte aligned)");
  DeviceGuard g(c->device);
  if (!g.ok) return fail(KEDS_ERR_CUDA, "cudaSetDevice(%d) failed", c->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const ConsLayout y = consumer_layout(c);
  const int64_t B = c->tr.B, Bk = B * c->tr.k, M = B + 2 * Bk;
  const int k = c->tr.k, L = c->n_layers, inner = c->inner, dt = c->d_tok, dm = c->d_mid, din = c->d_in;
  const int64_t kvw = static_cast<int64_t>(L) * 2 * inner;
  const int64_t ldB = round4(B), ldBk = round4(Bk), ldM = round4(M);
  if (attend_bwd_smem(c, k) > static_cast<size_t>(c->attend_max))  // (forward_train refuses such k first)
    return fail(KEDS_ERR_ARG, "consumer_backward: heads * (dim_head + k) too large for the attention backward");

  CKS(consumer_refresh_transposes(c, st));
  CKS(c->tr.dq[0].ensure(static_cast<size_t>(2) * B * dt * 4));
  CKS(c->tr.dq[1].ensure(static_cast<size_t>(2) * B * dt * 4));
  CKS(c->tr.dO.ensure(static_cast<size_t>(2) * B * inner * 4));
  CKS(c->tr.dQ.ensure(static_cast<size_t>(2) * B * inner * 4));
  CKS(c->tr.dkv.ensure(static_cast<size_t>(2) * Bk * kvw * 4));
  CKS(c->tr.dy.ensure(static_cast<size_t>(M) * dt * 4));
  CKS(c->tr.dh[0].ensure(static_cast<size_t>(M) * dm * 4));
  CKS(c->tr.dh[1].ensure(static_cast<size_t>(M) * dm * 4));
  {
    // transposed operands: [nz][n][ld]; the largest are dKV^T (2 x kvw x Bk) and the MLP's (dt | dm | din) x M
    const int64_t wmax = std::max<int64_t>(std::max(dt, dm), std::max(din, inner));
    const size_t need = static_cast<size_t>(std::max<int64_t>(2 * kvw * ldBk, std::max<int64_t>(2 * wmax * ldB, wmax * ldM))) * 4;
    CKS(c->tr.ta.ensure(need));
    CKS(c->tr.tb.ensure(need));
  }
  // the incoming gradient moves to a fixed buffer first: autograd hands over a fresh allocation every
  // step, and the GEMMs' operand descriptors are cached by address
  CKS(c->tr.dtok.ensure(static_cast<size_t>(B) * 3 * dt * 4));
  CK(cudaMemcpyAsync(c->tr.dtok.p, dtokens, static_cast<size_t>(B) * 3 * dt * 4, cudaMemcpyDeviceToDevice, st));
  dtokens = c->tr.dtok.as<float>();
  float* dO0 = c->tr.dO.as<float>();
  float* dO1 = dO0 + B * inner;
  float* dQ0 = c->tr.dQ.as<float>();
  float* dQ1 = dQ0 + B * inner;
  float* dkv0 = c->tr.dkv.as<float>();
  float* dkv1 = dkv0 + Bk * kvw;
  float* kv0 = c->kv.as<float>();
  float* kv1 = kv0 + Bk * kvw;
  float* xm = c->xm.as<float>();
  float* dy = c->tr.dy.as<float>();

  // ---- the two attention stacks, last layer first; both stacks ride in every launch
  const float* dq0 = dtokens;        // d tokens[:, 0, :] (image stack) and [:, 1, :] (text stack)
  const float* dq1 = dtokens + dt;
  int64_t ld_dq = 3 * static_cast<int64_t>(dt);
  for (int l = L - 1; l >= 0; --l) {
    const float* o0 = c->tr.o[l].as<float>();
    const float* o1 = o0 + B * inner;
    const float* q0 = c->tr.q[l].as<float>();
    const float* q1 = q0 + B * inner;
    const float* in0 = l == 0 ? xm : c->tr.qin[l].as<float>();
    const float* in1 = l == 0 ? xm : in0 + B * dt;
    // to_out: dO = dq Wo, dWo = dq^T O, dbo = column sums of dq
    CKS(consumer_linear(c, dq0, dq1, ld_dq, B, &c->woT[0][l], &c->woT[1][l], 0, dO0, dO1, inner, 2, st));
    CKS(train_weight_grad(c, dq0, dq1, ld_dq, o0, o1, inner, B, dt, inner, grads + y.o_w[0][l], grads + y.o_w[1][l], 2, st));
    CKS(train_colsum(c, dq0, ld_dq, B, dt, grads + y.o_b[0][l], st));
    CKS(train_colsum(c, dq1, ld_dq, B, dt, grads + y.o_b[1][l], st));
    // attention
    AttendBwdParams ap;
    memset(&ap, 0, sizeof ap);
    ap.B = static_cast<int>(B);
    ap.k = k;
    ap.heads = c->heads;
    ap.dim_head = c->dim_head;
    ap.Q[0] = q0;
    ap.Q[1] = q1;
    ap.KV[0] = kv0;
    ap.KV[1] = kv1;
    ap.dO[0] = dO0;
    ap.dO[1] = dO1;
    ap.dQ[0] = dQ0;
    ap.dQ[1] = dQ1;
    ap.dKV[0] = dkv0;
    ap.dKV[1] = dkv1;
    ap.ld_kv = kvw;
    ap.k_off = (2 * l) * inner;
    ap.v_off = (2 * l + 1) * inner;
    ap.scale = 1.0f / sqrtf(static_cast<float>(c->dim_head));
    CKS(launch_k(true, k_cross_attend_bwd, dim3(static_cast<unsigned>(B), 2), dim3(32 * c->heads), attend_bwd_smem(c, k),
                 st, ap));
    c->launches++;
    // to_q: dWq = dQ^T q_in, dbq, dq_in = dQ Wq
    CKS(train_weight_grad(c, dQ0, dQ1, inner, in0, in1, dt, B, inner, dt, grads + y.q_w[0][l], grads + y.q_w[1][l], 2, st));
    CKS(train_colsum(c, dQ0, inner, B, inner, grads + y.q_b[0][l], st));
    CKS(train_colsum(c, dQ1, inner, B, inner, grads + y.q_b[1][l], st));
    float* n0 = c->tr.dq[l & 1].as<float>();
    float* n1 = n0 + B * dt;
    CKS(consumer_linear(c, dQ0, dQ1, inner, B, &c->wqT[0][l], &c->wqT[1][l], 0, n0, n1, dt, 2, st));
    dq0 = n0;
    dq1 = n1;
    ld_dq = dt;
  }
  // d mapped = d tokens[:, 2, :] + what both stacks pass back through their first to_q
  {
    const long long n = static_cast<long long>(B) * dt;
    CKS(launch_k(true, k_add3_rows, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, dtokens + 2 * dt,
                 static_cast<long long>(3) * dt, dq0, static_cast<long long>(dt), dq1, static_cast<long long>(dt), dy,
                 static_cast<long long>(dt), static_cast<long long>(B), dt));
    c->launches++;
  }
  // to_k / to_v of every layer at once: dN = dKV Wkv, dWkv = dKV^T N, dbkv
  CKS(consumer_linear(c, dkv0, dkv1, kvw, Bk, &c->wkvT[0], &c->wkvT[1], 0, dy + B * dt, dy + (B + Bk) * dt, dt, 2, st));
  CKS(train_weight_grad(c, dkv0, dkv1, kvw, xm + B * dt, xm + (B + Bk) * dt, dt, Bk, static_cast<int>(kvw), dt,
                        grads + y.kv_w[0], grads + y.kv_w[1], 2, st));
  CKS(train_colsum(c, dkv0, kvw, Bk, static_cast<int>(kvw), grads + y.kv_b[0], st));
  CKS(train_colsum(c, dkv1, kvw, Bk, static_cast<int>(kvw), grads + y.kv_b[1], st));

  // ---- IM2TEXT over all M rows: fc_out, then the hidden layers backwards
  const int H = c->n_hidden;
  CKS(train_weight_grad(c, dy, nullptr, dt, c->tr.h[H - 1].as<float>(), nullptr, dm, M, dt, dm, grads + y.mlp_w[H], nullptr, 1, st));
  CKS(train_colsum(c, dy, dt, M, dt, grads + y.mlp_b[H], st));
  float* dh = c->tr.dh[0].as<float>();
  CKS(consumer_linear(c, dy, nullptr, dt, M, &c->mlpT[H], nullptr, 0, dh, nullptr, dm, 1, st));
  for (int i = H - 1; i >= 0; --i) {
    // through ReLU and dropout (in place: dh becomes dz)
    const long long n = static_cast<long long>(M) * dm;
    CKS(launch_k(true, k_relu_bwd, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st,
                 static_cast<const float*>(dh), static_cast<const float*>(c->tr.h[i].as<float>()), c->tr.masks[i], dh, n));
    c->launches++;
    const float* xin_i = i == 0 ? c->xin.as<float>() : c->tr.h[i - 1].as<float>();
    const int w_in = i == 0 ? din : dm;
    CKS(train_weight_grad(c, dh, nullptr, dm, xin_i, nullptr, w_in, M, dm, w_in, grads + y.mlp_w[i], nullptr, 1, st));
    CKS(train_colsum(c, dh, dm, M, dm, grads + y.mlp_b[i], st));
    if (i > 0) {
      float* dprev = c->tr.dh[(H - i) & 1].as<float>();
      CKS(consumer_linear(c, dh, nullptr, dm, M, &c->mlpT[i], nullptr, 0, dprev, nullptr, dm, 1, st));
      dh = dprev;
    }
  }
  c->tr.valid = false;  // the activations belong to one backward
  CK(cudaGetLastError());
  return 0;
}

}  // extern "C"
