// Host side of keds_clip_loss_* (include/keds_knn.h): the symmetric contrastive loss over the
// gathered features, forward and backward in one launch sequence (src/trainer.py:85-135,164).
// Included by api.cu after consumer_host.cuh, whose tf32 linear-layer launcher it reuses.
#pragma once
#include "contrastive.cuh"

struct keds_clip_loss {
  keds_consumer lin;  // launch context of k_linear_tf32: error word, descriptor cache, SM count
  int device = 0;
  DevBuf Ia, Ib, Ta, Tb;       // [N][3d] split operands ([hi|lo|hi] and [hi|hi|lo])
  DevBuf L1, L2;               // [N][N] I.T^T and T.I^T
  DevBuf lse;                  // [2][N]
  DevBuf G, Ga;                // [2][B][N] scale * dloss/dlogits of the local rows; split [2][B][3N]
  DevBuf Xt, Xtb;              // [2][d][N] transposed features; split [2][d][3N]
  DevBuf accum;                // 4 floats
};

namespace {

// a weight-like operand that lives in a scratch buffer: descriptors from the cache
int scratch_weight(keds_consumer* c, const float* W, int out, int in, LinearW* w) {
  w->out = out;
  w->in = in;
  w->set = true;
  CKS(consumer_cached_map(c, W, out, in, in, LIN_WBOX, &w->tm));
  CKS(consumer_cached_map(c, W, out, in, in, SK_BN, &w->tm32));
  return 0;
}

}  // namespace

extern "C" {

int keds_clip_loss_create(int device, keds_clip_loss_t** out) {
  if (!out) return fail(KEDS_ERR_ARG, "clip_loss_create: out is NULL");
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) {
    cudaGetLastError();
    return fail(KEDS_ERR_NO_GPU, "clip_loss_create: CUDA device %d not available (this library has no CPU path)", device);
  }
  DeviceGuard g(device);
  if (!g.ok) return fail(KEDS_ERR_CUDA, "cudaSetDevice(%d) failed", device);
  keds_clip_loss* h = new keds_clip_loss();
  h->device = device;
  h->lin.device = device;
  auto init = [&]() -> int {
    CKS(linear_init(&h->lin));
    CKS(h->accum.ensure(16));
    CK(cudaDeviceSynchronize());  // the memset above is on the legacy stream; callers may use any stream
    return 0;
  };
  const int rc = init();
  if (rc != 0) {
    h->lin.err.release();
    h->accum.release();
    delete h;
    return rc;
  }
  *out = h;
  return 0;
}

void keds_clip_loss_free(keds_clip_loss_t* h) {
  if (!h) return;
  DeviceGuard g(h->device);
  for (DevBuf* b : {&h->Ia, &h->Ib, &h->Ta, &h->Tb, &h->L1, &h->L2, &h->lse, &h->G, &h->Ga, &h->Xt, &h->Xtb,
                    &h->accum, &h->lin.err, &h->lin.tdump})
    b->release();
  delete h;
}

int keds_clip_loss_forward_backward(keds_clip_loss_t* h, const float* I_all, const float* T_all, int64_t N,
                                    int d, int64_t row0, int64_t n_local, const float* scale, float* loss,
                                    float* dI_local, float* dT_local, float* dscale, void* stream) {
  if (!h || !I_all || !T_all || !loss || !scale) return fail(KEDS_ERR_ARG, "clip_loss: NULL argument");
  if (N <= 0 || N > (1 << 20) || d <= 0 || (N & 3) || (d & 3))
    return fail(KEDS_ERR_ARG, "clip_loss: N and d must be positive multiples of 4 (N = %lld, d = %d)", (long long)N, d);
  if (row0 < 0 || n_local < 0 || row0 + n_local > N) return fail(KEDS_ERR_ARG, "clip_loss: local rows outside [0, N)");
  const bool want_grad = dI_local != nullptr || dT_local != nullptr;
  if (want_grad && (!dI_local || !dT_local || n_local == 0))
    return fail(KEDS_ERR_ARG, "clip_loss: pass both gradient buffers (and local rows) or neither");
  for (const void* p : {(const void*)I_all, (const void*)T_all, (const void*)loss, (const void*)scale})
    if (!locate(p)) return fail(KEDS_ERR_ARG, "clip_loss: all buffers must be device memory");
  DeviceGuard g(h->device);
  if (!g.ok) return fail(KEDS_ERR_CUDA, "cudaSetDevice(%d) failed", h->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  keds_consumer* c = &h->lin;
  const int64_t B = n_local;
  const int K3 = 3 * d;
  const int64_t N3 = 3 * N;
  CKS(h->Ia.ensure(static_cast<size_t>(N) * K3 * 4));
  CKS(h->Ib.ensure(static_cast<size_t>(N) * K3 * 4));
  CKS(h->Ta.ensure(static_cast<size_t>(N) * K3 * 4));
  CKS(h->Tb.ensure(static_cast<size_t>(N) * K3 * 4));
  CKS(h->L1.ensure(static_cast<size_t>(N) * N * 4));
  CKS(h->L2.ensure(static_cast<size_t>(N) * N * 4));
  CKS(h->lse.ensure(static_cast<size_t>(2) * N * 4));
  if (want_grad) {
    CKS(h->G.ensure(static_cast<size_t>(2) * B * N * 4));
    CKS(h->Ga.ensure(static_cast<size_t>(2) * B * N3 * 4));
    CKS(h->Xt.ensure(static_cast<size_t>(2) * d * N * 4));
    CKS(h->Xtb.ensure(static_cast<size_t>(2) * d * N3 * 4));
  }
  float* Ia = h->Ia.as<float>();
  float* Ib = h->Ib.as<float>();
  float* Ta = h->Ta.as<float>();
  float* Tb = h->Tb.as<float>();
  float* L1 = h->L1.as<float>();
  float* L2 = h->L2.as<float>();
  float* lse_r = h->lse.as<float>();
  float* lse_c = lse_r + N;
  float* accum = h->accum.as<float>();

  // operands split into tf32 hi / lo parts along a tripled K axis (fp32-accurate products)
  const unsigned sb = static_cast<unsigned>((N * d + 255) / 256);
  k_split3_tf32<<<sb, 256, 0, st>>>(I_all, d, static_cast<int>(N), d, Ia, Ib, K3);
  k_split3_tf32<<<sb, 256, 0, st>>>(T_all, d, static_cast<int>(N), d, Ta, Tb, K3);
  CK(cudaMemsetAsync(accum, 0, 16, st));
  CK(cudaGetLastError());

  // L1 = I T^T and L2 = T I^T in one launch (two problems)
  LinearW wT, wI;
  CKS(scratch_weight(c, Tb, static_cast<int>(N), K3, &wT));
  CKS(scratch_weight(c, Ib, static_cast<int>(N), K3, &wI));
  CKS(consumer_linear(c, Ia, Ta, K3, N, &wT, &wI, 0, L1, L2, N, 2, st));

  const int nthr = N >= 1024 ? 256 : 128;
  CKS(launch_k(true, k_row_lse, dim3(static_cast<unsigned>(N)), dim3(nthr), 0, st, (const float*)L1, (long long)N,
               static_cast<int>(N), static_cast<int>(N), (const float*)scale, lse_r));
  CKS(launch_k(true, k_row_lse, dim3(static_cast<unsigned>(N)), dim3(nthr), 0, st, (const float*)L2, (long long)N,
               static_cast<int>(N), static_cast<int>(N), (const float*)scale, lse_c));
  float* Gr = want_grad ? h->G.as<float>() : nullptr;
  float* Gc = want_grad ? Gr + B * N : nullptr;
  CKS(launch_k(true, k_clip_grad_rows, dim3(static_cast<unsigned>(N)), dim3(nthr), 0, st, (const float*)L1,
               (long long)N, static_cast<int>(N), static_cast<int>(row0), static_cast<int>(B), (const float*)scale,
               (const float*)lse_r, (const float*)lse_c, Gr, (long long)N, accum));
  CKS(launch_k(true, k_clip_grad_rows, dim3(static_cast<unsigned>(N)), dim3(nthr), 0, st, (const float*)L2,
               (long long)N, static_cast<int>(N), static_cast<int>(row0), static_cast<int>(B), (const float*)scale,
               (const float*)lse_c, (const float*)lse_r, Gc, (long long)N, accum + 2));
  CKS(launch_k(true, k_clip_finalize, dim3(1), dim3(32), 0, st, (const float*)accum, static_cast<int>(N), loss,
               dscale));
  c->launches += 8;

  if (want_grad) {
    // dI_local = (scale G[local rows]) T_all,  dT_local = (scale G^T[local rows]) I_all
    float* Tt = h->Xt.as<float>();          // [d][N]
    float* It = Tt + static_cast<size_t>(d) * N;
    float* Ttb = h->Xtb.as<float>();        // [d][3N], [hi|hi|lo]
    float* Itb = Ttb + static_cast<size_t>(d) * N3;
    float* Gra = h->Ga.as<float>();         // [B][3N], [hi|lo|hi]
    float* Gca = Gra + B * N3;
    const dim3 tg = transpose_grid(N, d);
    k_transpose_f32<<<tg, dim3(32, 8), 0, st>>>(T_all, d, static_cast<int>(N), d, Tt, N);
    k_transpose_f32<<<tg, dim3(32, 8), 0, st>>>(I_all, d, static_cast<int>(N), d, It, N);
    const unsigned s1 = static_cast<unsigned>((static_cast<long long>(d) * N + 255) / 256);
    k_split3_tf32<<<s1, 256, 0, st>>>(Tt, N, d, static_cast<int>(N), nullptr, Ttb, N3);
    k_split3_tf32<<<s1, 256, 0, st>>>(It, N, d, static_cast<int>(N), nullptr, Itb, N3);
    const unsigned s2 = static_cast<unsigned>((B * N + 255) / 256);
    k_split3_tf32<<<s2, 256, 0, st>>>(Gr, N, static_cast<int>(B), static_cast<int>(N), Gra, nullptr, N3);
    k_split3_tf32<<<s2, 256, 0, st>>>(Gc, N, static_cast<int>(B), static_cast<int>(N), Gca, nullptr, N3);
    CK(cudaGetLastError());
    LinearW wTt, wIt;
    CKS(scratch_weight(c, Ttb, d, static_cast<int>(N3), &wTt));
    CKS(scratch_weight(c, Itb, d, static_cast<int>(N3), &wIt));
    CKS(consumer_linear(c, Gra, Gca, N3, B, &wTt, &wIt, 0, dI_local, dT_local, d, 2, st));
    c->launches += 6;
  }
  return 0;
}

int keds_clip_loss_check(keds_clip_loss_t* h, void* stream) {
  if (!h) return fail(KEDS_ERR_ARG, "clip_loss_check: NULL handle");
  DeviceGuard g(h->device);
  CK(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  uint32_t e = 0;
  CK(cudaMemcpy(&e, h->lin.err.p, 4, cudaMemcpyDeviceToHost));
  if (e != 0) {
    CK(cudaMemset(h->lin.err.p, 0, 4));
    return fail(KEDS_ERR_KERNEL, "clip-loss kernel pipeline timed out (code 0x%x)", e);
  }
  return 0;
}

}  // extern "C"
