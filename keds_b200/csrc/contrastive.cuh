// The step right after the retrieval path (SURVEY.md §8 f3): the symmetric contrastive loss over
// the features gathered from all ranks, src/trainer.py:85-135,164:
//     logits = logit_scale * I_all @ T_all.t();  loss = (CE(logits, arange) + CE(logits.t(), arange)) / 2
// Forward and backward in one pass. The two N x N products (logits and logits^T, both row-major so
// that every reduction below runs along contiguous rows) and the two gradient products reuse
// k_linear_tf32 (neighbour_consumer.cuh); the kernels here are the row statistics in between.
#pragma once
#include "ptx.cuh"

namespace keds {

// lse[r] = log sum_j exp(scale * L[r][j]) for r < n_rows; block per row.
__global__ void k_row_lse(const float* __restrict__ L, long long ld, int n_rows, int n_cols,
                          const float* __restrict__ scale_p, float* __restrict__ lse) {
  griddep_wait();
  const float scale = *scale_p;
  __shared__ float red[33];
  const int r = blockIdx.x;
  if (r >= n_rows) return;
  const float* row = L + static_cast<long long>(r) * ld;
  float mx = -INFINITY;
  for (int j = threadIdx.x; j < n_cols; j += blockDim.x) mx = fmaxf(mx, scale * row[j]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  if (threadIdx.x < 32) {
    float m = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : -INFINITY;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (threadIdx.x == 0) red[32] = m;
  }
  __syncthreads();
  mx = red[32];
  float s = 0.f;
  for (int j = threadIdx.x; j < n_cols; j += blockDim.x) s += expf(scale * row[j] - mx);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (threadIdx.x == 0) lse[r] = mx + logf(t);
  }
}

// With P = scale * L (L = A_all @ B_all^T, rows = this side's samples, columns = the other side's):
//   G[r][j] = (exp(P[r][j] - lse_own[r]) + exp(P[r][j] - lse_other[j]) - 2 [r == j]) / (2 N)
// = d loss / d P[r][j]. One block per row r < N. Rows [row0, row0 + n_local) -- this rank's samples
// -- also write scale * G[r][:] (= d loss / d L, what the gradient product needs) to
// Gout[r - row0][:]; every row contributes to the two sums every rank needs in full:
// accum[0] += lse_own[r] - P[r][r]          (this side's loss numerator)
// accum[1] += sum_j G[r][j] * L[r][j]       (d loss / d scale)
__global__ void k_clip_grad_rows(const float* __restrict__ L, long long ld, int N, int row0, int n_local,
                                 const float* __restrict__ scale_p, const float* __restrict__ lse_own,
                                 const float* __restrict__ lse_other, float* __restrict__ Gout, long long ldg,
                                 float* __restrict__ accum) {
  griddep_wait();
  __shared__ float red[32];
  const float scale = *scale_p;
  const int r = blockIdx.x;
  if (r >= N) return;
  float* gout = (Gout != nullptr && r >= row0 && r < row0 + n_local) ? Gout + static_cast<long long>(r - row0) * ldg
                                                                      : nullptr;
  const float* row = L + static_cast<long long>(r) * ld;
  const float lo = lse_own[r];
  const float inv = 0.5f / static_cast<float>(N);
  float acc = 0.f;
  for (int j = threadIdx.x; j < N; j += blockDim.x) {
    const float l = row[j];
    const float pv = scale * l;
    const float g = (expf(pv - lo) + expf(pv - lse_other[j]) - (j == r ? 2.f : 0.f)) * inv;
    if (gout != nullptr) gout[j] = scale * g;
    acc = fmaf(g, l, acc);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (threadIdx.x == 0) {
      atomicAdd(accum + 1, t);
      atomicAdd(accum + 0, lo - scale * row[r]);
    }
  }
}

// out[c][r] = in[r][c]  (in: [rows][cols] with ld_in, out: [cols][ld_out]); 32 x 32 tiles. A block
// walks the row tiles blockIdx.y, blockIdx.y + gridDim.y, ...: grid.y stops at 65 535, the rows of a
// consumer backward (B (1 + 2k) up to 2^30) do not. Launch with transpose_grid.
__global__ void k_transpose_f32(const float* __restrict__ in, long long ld_in, int rows, int cols,
                                float* __restrict__ out, long long ld_out) {
  griddep_wait();
  __shared__ float tile[32][33];
  const int c0 = blockIdx.x * 32;
  for (int r0 = blockIdx.y * 32; r0 < rows; r0 += gridDim.y * 32) {
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
      const int r = r0 + i, c = c0 + threadIdx.x;
      tile[i][threadIdx.x] = (r < rows && c < cols) ? in[static_cast<long long>(r) * ld_in + c] : 0.f;
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
      const int c = c0 + i, r = r0 + threadIdx.x;
      if (c < cols && r < rows) out[static_cast<long long>(c) * ld_out + r] = tile[threadIdx.x][i];
    }
    __syncthreads();  // the next row tile reuses `tile`
  }
}

inline dim3 transpose_grid(long long rows, int cols) {
  return dim3(static_cast<unsigned>((cols + 31) / 32), static_cast<unsigned>(std::min((rows + 31) / 32, 65535LL)));
}

// fp32-accurate products on the tf32 tensor cores: x = hi + lo with hi = tf32(x) (10-bit mantissa,
// round to nearest) and lo = x - hi (exact in fp32). With the K axis tripled,
//     A' = [A_hi | A_lo | A_hi],  B' = [B_hi | B_hi | B_lo]   =>   A' B'^T = A B^T - A_lo B_lo^T
// i.e. one ordinary tf32 product of three times the depth, wrong by ~2^-22 relative.
// in: [rows][K] (ld_in) -> out_a, out_b: [rows][3K] (ld_out); either output may be null.
__global__ void k_split3_tf32(const float* __restrict__ in, long long ld_in, int rows, int K,
                              float* __restrict__ out_a, float* __restrict__ out_b, long long ld_out) {
  griddep_wait();
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(rows) * K) return;
  const int r = static_cast<int>(i / K), c = static_cast<int>(i % K);
  const float x = in[static_cast<long long>(r) * ld_in + c];
  uint32_t hb;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hb) : "f"(x));
  const float hi = __uint_as_float(hb);
  const float lo = x - hi;
  const long long o = static_cast<long long>(r) * ld_out + c;
  if (out_a != nullptr) {
    out_a[o] = hi;
    out_a[o + K] = lo;
    out_a[o + 2 * K] = hi;
  }
  if (out_b != nullptr) {
    out_b[o] = hi;
    out_b[o + K] = hi;
    out_b[o + 2 * K] = lo;
  }
}

// loss = (sum_i (lse_r[i] - P[i][i]) + sum_j (lse_c[j] - P[j][j])) / (2 N);  dscale = sum G * L
__global__ void k_clip_finalize(const float* __restrict__ accum, int N, float* __restrict__ loss,
                                float* __restrict__ dscale) {
  griddep_wait();
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    if (loss != nullptr) *loss = (accum[0] + accum[2]) * (0.5f / static_cast<float>(N));
    if (dscale != nullptr) *dscale = accum[1];
  }
}

}  // namespace keds
