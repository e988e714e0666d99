"""Bit-exact fp32 reference for the retrieval step's gathered neighbours and pools.

The fused consumer (`consume_query`, keds_b200/csrc/aux_kernels.cuh) writes, per query b and stream s,

    feat[b][jo][:] = rows[I[b][perm[jo]]][:]           (zero row: padding id, or perm[jo] outside [0, k))
    pool[b][:]     = sum over output slots jo of  w[perm[jo]] * feat[b][jo][:]

with w = RN32(1/k) for every slot (mode 1, padding included: a padding slot is a zero row) or
softmax_j(sign * tau * D[b][j]) over the valid slots (mode 2, sign = -1 under L2; padding gets weight 0).
A slot whose perm entry is outside [0, k) reads a zero row with weight w[0]. For a permutation
`perm` the pool is sum_j w_j rows[I[b][j]], whatever perm is; a perm that repeats or leaves out an
entry changes it, which is why the Python entry points refuse one.

The summation order depends on the caller of consume_query. Each order is a pair (warps, NIF):

  * vec path (d % 4 == 0, rows, feat and pool 16-byte aligned): warp g owns the slots
    g*NIF + t + i*warps*NIF (i outer, t = 0..NIF-1 inner), i.e. its slots in increasing order, and
    keeps acc_g = fma(w, x, acc_g) per slot, from +0; a slot past k adds nothing. The pool is then
    acc_0 + acc_1 + ... + acc_{warps-1}, plain fp32 adds in that order (a warp without slots adds +0).
  * scalar path (d % 4 != 0, or a feat / pool output not 16-byte aligned): one thread per column, one
    fma chain over slots 0..k-1. It is the order (1, 1).

  caller                                     order
  k_select_rerank<3,2>   (latency variant)   (8, 2)
  k_select_rerank<2,6,128> (throughput, k >= 128, 128 threads)   (4, 2)
  k_select_rerank<1,4>   (throughput, T threads)                  (T/32, 1)
  k_exact_fallback                                                (8, 1)
  k_shard_consume                                                 (8, 2)

The emulation is per column, so any d works (d > 768 only means more float4 passes in the kernel,
each column still sums its slots in the order above).

Mode 2 goes through __expf, which has no bit-exact emulation; `softmax_pool_bound` gives a float64
pool from D and a rigorous bound on the library's distance from it (derivation in its docstring).

`weighted_pool` emulates k_weighted_pool (keds_gather_pool with weights): per (b, h, column) one fma
chain over j = 0..k-1 that skips ids < 0 or >= n_base (no fma at all for them).

All arithmetic is fp32 emulated in float64 with `f32_fma` / `f32_add` of oracle/fp32_exact.py; the
helpers run on CPU tensors, and on a CUDA device for large batches.
"""
from __future__ import annotations

import math
from typing import Optional

import numpy as np
import torch

from .fp32_exact import f32_add, f32_fma

U = 2.0 ** -24                 # unit roundoff of fp32

# (warps, neighbours in flight per warp) of each consume_query caller; SCALAR is the element path
LATENCY = (8, 2)
THROUGHPUT_K128 = (4, 2)
FALLBACK = (8, 1)
SHARD = (8, 2)
SCALAR = (1, 1)


def throughput(threads: int):
    """k_select_rerank<1,4> at `threads` threads per block (KEDS_RERANK_THREADS)."""
    return (threads // 32, 1)


def mean_weight(k: int) -> float:
    """1.f / (float)k as the kernel computes it (IEEE fp32 division)."""
    return float(np.float32(1.0) / np.float32(k))


# ------------------------------------------------------------------------------------ gather
def _slot_ranks(perm: Optional[torch.Tensor], k: int, device):
    """(rank each output slot shows, clamped to [0, k); slot's perm entry is valid) -- [k] each."""
    if perm is None:
        jr = torch.arange(k, device=device)
    else:
        jr = torch.as_tensor(perm, dtype=torch.int64).to(device).reshape(k)
    ok = (jr >= 0) & (jr < k)
    return torch.where(ok, jr, torch.zeros_like(jr)), ok


def _slot_ids(I: torch.Tensor, perm, n_rows: int):
    """[B, k] row id each output slot reads (-1: zero row) and the rank whose weight it takes."""
    B, k = I.shape
    jr, ok = _slot_ranks(perm, k, I.device)
    ids = I[:, jr]
    ids = torch.where(ok[None, :] & (ids >= 0) & (ids < n_rows), ids, torch.full_like(ids, -1))
    return ids, jr


def gather(rows: torch.Tensor, I: torch.Tensor, perm=None) -> torch.Tensor:
    """feat[b][jo] = rows[I[b][perm[jo]]] (fp32 [B, k, d]); zero rows for ids -1 (padding) or outside
    rows, and for slots whose perm entry is outside [0, k) -- as k_gather_rows and consume_query."""
    I = I.to(rows.device)
    ids, _ = _slot_ids(I, perm, rows.shape[0])
    out = rows[ids.clamp(min=0)]
    return out.masked_fill((ids < 0)[..., None], 0.0)


# ------------------------------------------------------------------------------------ pools
def pool_order(vals: torch.Tensor, wslot: torch.Tensor, nwarps: int, nif: int, vec: bool = True) -> torch.Tensor:
    """consume_query's pool from per-slot operands: vals [B, k, d] (the slot's row, fp32 values in any
    float dtype), wslot [B, k] (the slot's weight) -> fp32 [B, d] in the order (nwarps, nif), or the
    scalar order when vec is False."""
    if not vec:
        nwarps, nif = SCALAR
    B, k, d = vals.shape
    grp = nwarps * nif
    steps = -(-k // grp)
    # slot of warp g at its s-th fma: i = s // nif, t = s % nif -> g*nif + t + i*grp
    own = torch.arange(steps * grp, device=vals.device).view(steps, nwarps, nif).permute(1, 0, 2).reshape(nwarps, -1)
    v64, w64 = vals.double(), wslot.double()
    acc = torch.zeros(B, nwarps, d, dtype=torch.float64, device=vals.device)
    for s in range(own.shape[1]):
        jo = own[:, s]
        live = (jo < k)[None, :, None]
        jc = jo.clamp(max=k - 1)
        new = f32_fma(w64[:, jc][..., None], v64[:, jc], acc)
        acc = torch.where(live, new, acc)
    out = acc[:, 0]
    for g in range(1, nwarps):
        out = f32_add(out, acc[:, g])
    return out.to(torch.float32)


def slot_weights(w: torch.Tensor, perm, k: int) -> torch.Tensor:
    """[B, k] weight of each output slot: w[b][perm[jo]], w[b][0] for an out-of-range perm entry."""
    jr, _ = _slot_ranks(perm, k, w.device)
    return w[:, jr]


def consume_pool(rows: torch.Tensor, I: torch.Tensor, w: torch.Tensor, perm, nwarps: int, nif: int,
                 vec: bool = True, chunk: int = 1 << 24) -> torch.Tensor:
    """consume_query's pool for given fp32 weights w [B, k] (per rank) of the neighbours I [B, k]
    (row ids of `rows`, -1 padding): fp32 [B, d], bit for bit, in the order (nwarps, nif) / scalar."""
    I = I.to(rows.device)
    w = w.to(rows.device)
    B, k = I.shape
    d = rows.shape[1]
    out = torch.empty(B, d, dtype=torch.float32, device=rows.device)
    step = max(1, chunk // max(1, k * d * max(1, nwarps)))
    for b0 in range(0, B, step):
        sl = slice(b0, b0 + step)
        vals = gather(rows, I[sl], perm)
        out[sl] = pool_order(vals, slot_weights(w[sl], perm, k), nwarps, nif, vec)
    return out


def mean_pool(rows, I, perm, nwarps, nif, vec=True) -> torch.Tensor:
    """Mode 1: every slot weighs RN32(1/k), padding included (a padding slot adds a zero row)."""
    B, k = I.shape
    w = torch.full((B, k), mean_weight(k), dtype=torch.float64, device=rows.device)
    return consume_pool(rows, I, w, perm, nwarps, nif, vec)


def softmax_weights(D: torch.Tensor, I: torch.Tensor, tau: float, l2: bool) -> torch.Tensor:
    """float64 softmax_j(sign * tau * D[b][j]) over the valid entries (I >= 0), padding 0: [B, k]."""
    z = (-tau if l2 else tau) * D.double()
    z = z.masked_fill(I < 0, -math.inf)
    w = torch.softmax(z, dim=1)
    return torch.nan_to_num(w, nan=0.0)


def _expf_ulps(x: torch.Tensor) -> torch.Tensor:
    """CUDA C Programming Guide, intrinsic functions: __expf(x) is within 2 + floor(|1.173 x|) ulp."""
    return 2.0 + torch.floor((1.173 * x).abs())


def softmax_weight_interval(D: torch.Tensor, I: torch.Tensor, tau: float, l2: bool, nwarps_sum: int = 32):
    """(w_lo, w_hi) float64 [B, k]: an interval that holds both the exact softmax weight and the one
    consume_query computes in fp32 (padding: [0, 0]). See softmax_pool_bound for the derivation."""
    D64 = D.double()
    valid = I >= 0
    st = -float(tau) if l2 else float(tau)
    z = (st * D64).masked_fill(~valid, -math.inf)           # exact sign*tau*D (one fp32 rounding away)
    mx = z.amax(1, keepdim=True)
    x = (z - mx).masked_fill(~valid, 0.0)                   # exact argument (<= 0)
    # |computed argument - x| <= delta: RN(st*D) and RN(mx) each within u of their value (mx is the
    # rounded max, rounding being monotone), then one more rounding of the difference (or one
    # rounding in all when the compiler contracts st*D - mx into an fma); 3u covers either
    zabs = z.abs().masked_fill(~valid, 0.0)
    delta = 3.0 * U * (zabs + mx.abs().expand_as(zabs))
    n = _expf_ulps(x.abs() + delta)
    E = torch.exp(x)                                        # exact up to float64 rounding (1e-15 below)
    rel = n * 2.0 ** -23 + 1e-15
    A = 2.0 ** -125                                          # absolute: flush-to-zero / subnormal results
    Lj = torch.exp(-delta) * (1.0 - rel)
    Uj = torch.exp(delta) * (1.0 + rel)
    e_lo = (E * Lj - A).clamp(min=0.0).masked_fill(~valid, 0.0)
    e_hi = (E * Uj + A).masked_fill(~valid, 0.0)
    k = D.shape[1]
    m = -(-k // nwarps_sum) - 1 + 5                          # adds on any path: lane's own, then 5 butterfly levels
    gam = m * U / (1.0 - m * U)
    S_lo = e_lo.sum(1, keepdim=True) * (1.0 - gam)
    S_hi = e_hi.sum(1, keepdim=True) * (1.0 + gam)
    w_lo = e_lo * (1.0 - U) ** 2 / S_hi
    w_hi = e_hi * (1.0 + U) ** 2 / S_lo.clamp(min=1e-300)
    exact = E.masked_fill(~valid, 0.0)
    exact = exact / exact.sum(1, keepdim=True).clamp(min=1e-300)
    return torch.minimum(w_lo, exact), torch.maximum(w_hi, exact)


def softmax_pool_bound(rows: torch.Tensor, I: torch.Tensor, D: torch.Tensor, perm, tau: float, l2: bool,
                       nwarps: int, chunk: int = 1 << 24):
    """Mode 2: (float64 pool [B, d] with the exact softmax weights of D, bound [B, d]) such that the
    library's pool p satisfies |p - pool| <= bound elementwise on the route with `nwarps` warps.

    Derivation. Write x_j = sign*tau*D_j - max_i(sign*tau*D_i) <= 0 (exact, D being the fp32 values the
    library returns), E_j = exp(x_j), S = sum_j E_j >= 1, w_j = E_j / S. The kernel computes
      * x'_j = RN(RN(sign*tau*D_j) - RN(max)) (or one rounding of an fma): |x'_j - x_j| <= delta_j =
        3u (|sign*tau*D_j| + |max|), u = 2^-24;
      * e_j = __expf(x'_j), documented within n_j = 2 + floor(|1.173 x'_j|) ulp, i.e. a relative error
        <= n_j 2^-23, plus an absolute 2^-125 for results the flush-to-zero path loses. So
        E_j L_j - A <= e_j <= E_j U_j + A, L_j = e^-delta_j (1 - n_j 2^-23), U_j = e^delta_j (1 + n_j 2^-23);
      * the warp sum of the e_j: each lane sums its ceil(k/32) terms, then 5 butterfly adds: m adds on
        any path, relative error <= gamma_m = m u / (1 - m u) (non-negative terms);
      * inv = RN(1/sum) and w'_j = RN(e_j * inv): two more factors (1 +- u).
    Hence w'_j lies in [w_lo_j, w_hi_j] = [(E_j L_j - A)(1-u)^2 / (S_hi), (E_j U_j + A)(1+u)^2 / (S_lo)]
    with S_lo = (1 - gamma_m) sum (E_i L_i - A), S_hi = (1 + gamma_m) sum (E_i U_i + A), and so does w_j.
    The pool is then accumulated as one fma chain per warp (at most k terms) and nwarps - 1 adds, so
    |p - sum_j w'_j r_j| <= gamma_{k + nwarps} sum_j w'_j |r_j|, and
    |sum_j w'_j r_j - sum_j w_j r_j| <= sum_j (w_hi_j - w_lo_j) |r_j|. The float64 evaluation of the
    reference pool adds at most 1e-15 sum_j w_j |r_j|. Padding slots have weight 0 on both sides and
    a zero row. A perm only reorders the terms, so the bound holds for any permutation.
    """
    I = I.to(rows.device)
    D = D.to(rows.device)
    B, k = I.shape
    d = rows.shape[1]
    w = softmax_weights(D, I, tau, l2)
    w_lo, w_hi = softmax_weight_interval(D, I, tau, l2)
    ga = (k + nwarps) * U / (1.0 - (k + nwarps) * U)
    ref = torch.empty(B, d, dtype=torch.float64, device=rows.device)
    bound = torch.empty(B, d, dtype=torch.float64, device=rows.device)
    step = max(1, chunk // max(1, k * d))
    for b0 in range(0, B, step):
        sl = slice(b0, b0 + step)
        r = gather(rows, I[sl], None).double()               # rank order: the pool does not depend on perm
        ra = r.abs()
        ref[sl] = torch.einsum("bk,bkd->bd", w[sl], r)
        bound[sl] = (torch.einsum("bk,bkd->bd", (w_hi[sl] - w_lo[sl]) + (ga + 1e-15) * w_hi[sl], ra) + 1e-30)
    return ref, bound


def weighted_pool(rows: torch.Tensor, I: torch.Tensor, W: torch.Tensor) -> torch.Tensor:
    """k_weighted_pool: out[b][h][:] = fma chain over j = 0..k-1 of W[b][h][j] * rows[I[b][j]][:], ids
    < 0 or >= n_base skipped (no fma). fp32 [B, H, d], bit for bit."""
    I = I.to(rows.device)
    W = W.to(rows.device).double()
    B, k = I.shape
    H, d = W.shape[1], rows.shape[1]
    ok = (I >= 0) & (I < rows.shape[0])
    acc = torch.zeros(B, H, d, dtype=torch.float64, device=rows.device)
    for j in range(k):
        v = rows[I[:, j].clamp(0, rows.shape[0] - 1)].double()       # [B, d]
        new = f32_fma(W[:, :, j][..., None], v[:, None, :], acc)
        acc = torch.where(ok[:, j][:, None, None], new, acc)
    return acc.to(torch.float32)


def equal_rows(got: torch.Tensor, want: torch.Tensor) -> torch.Tensor:
    """[B] bool: got[i] equals want[i] bit for bit (fp32 tensors of the same shape)."""
    g = got.contiguous().view(torch.int32).reshape(got.shape[0], -1)
    w = want.to(got.device).contiguous().view(torch.int32).reshape(got.shape[0], -1)
    return (g == w).all(1)
