"""Bit-exact fp32 reference for the library's exact answers.

Every answer of the library claims to equal an exact fp32 flat search: the scores of one fp32
routine, `warp_exact_score` (keds_b200/csrc/aux_kernels.cuh), ordered by score descending, then row
id ascending. This module emulates that routine bit for bit and builds the search, gallery-rank,
label-hit and merge results on it, so that a test can compare the library's D and I with `==` on
their bits instead of with a tolerance. It is plain torch and never calls the library: it runs on
CPU tensors, and in float64 on a CUDA device for large cases.

The emulated routine, for one (query, row) pair and a warp of 32 lanes:
  * lane order: if d % 4 == 0 (the library's row and query buffers are then 16-byte aligned), lane l
    takes float4 chunks l, l+32, ... and does four fmas per chunk in x, y, z, w order; otherwise lane
    l takes elements l, l+32, ... one at a time;
  * IP: acc = fma(x, q, acc).  L2: t = RN32(q - x), acc = fma(t, t, acc);
  * the lanes' partial sums meet in an xor butterfly over offsets 16, 8, 4, 2, 1.

fp32 arithmetic is emulated in float64: fma(a, b, c) = RN32(RO64(a*b + c)), where the product of two
fp32 values is exact in float64 and RO64 rounds the float64 sum to odd (TwoSum gives the exact
error; when it is non-zero and the sum's last mantissa bit is even, step one float64 ulp in the
error's direction). Rounding to odd at 53 bits followed by round-to-nearest at 24 bits equals one
correct rounding of the exact value, subnormal results included. Additions use the same helper.

Candidate filter. Emulating every (query, row) pair of a large database is slow, so the search and
rank helpers first score in float64 and bound how far the fp32 result can be from it:
|fp32 - float64| <= (d + 8) * 2^-23 * A + 1e-12 * (|q|^2 + |x|^2), A = sum |q_i x_i| (IP) or the
squared distance (L2) -- far above the true fp32 summation error of a d-term sum. Only rows whose
interval can reach the answer are emulated; the rest are decided by the float64 score alone.
"""
from __future__ import annotations

from typing import Optional, Sequence

import torch

FLT_MAX = float(torch.finfo(torch.float32).max)
_INF = float("inf")


# ------------------------------------------------------------------------------------ fp32 arithmetic
def _round_to_odd_sum(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """a + b (float64 tensors) rounded to odd at float64 precision."""
    s = a + b
    bb = s - a
    err = (a - (s - bb)) + (b - bb)  # TwoSum: s + err == a + b exactly
    even = (s.view(torch.int64) & 1) == 0
    # nextafter(s, s + err) would not move (s + err rounds back to s): step towards an infinity
    toward = torch.where(err > 0, torch.full_like(s, _INF), torch.full_like(s, -_INF))
    return torch.where((err != 0) & even, torch.nextafter(s, toward), s)


def _rn32(x: torch.Tensor) -> torch.Tensor:
    return x.to(torch.float32).to(torch.float64)


def f32_add(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """fp32 a + b, correctly rounded. Operands and result: float64 tensors holding fp32 values."""
    return _rn32(_round_to_odd_sum(a, b))


def f32_fma(a: torch.Tensor, b: torch.Tensor, c: torch.Tensor) -> torch.Tensor:
    """fp32 fmaf(a, b, c): one rounding of the exact a*b + c. float64 tensors holding fp32 values."""
    return _rn32(_round_to_odd_sum(a * b, c))  # the product of two fp32 values is exact in float64


# ------------------------------------------------------------------------------------ the scoring routine
def _lanes(v: torch.Tensor, w: int) -> torch.Tensor:
    """[P, d] -> [P, steps, 32, w]: element steps*32*w + lane*w + j is lane `lane`'s j-th operand of
    its step `steps`. Zero padding is harmless: fma(0, 0, acc) == acc."""
    P, d = v.shape
    pad = (-d) % (32 * w)
    if pad:
        v = torch.nn.functional.pad(v, (0, pad))
    return v.reshape(P, -1, 32, w)


def pair_scores(q: torch.Tensor, x: torch.Tensor, metric: str, order: str = "auto",
                chunk: int = 1 << 23) -> torch.Tensor:
    """warp_exact_score of row pairs: q[i] against x[i] ([P, d] fp32 each) -> fp32 [P].
    IP: sum q*x. L2: sum (q-x)^2. order: 'auto' (float4 lanes when d % 4 == 0), 'vec' or 'scalar'."""
    assert q.shape == x.shape and q.dim() == 2 and metric in ("ip", "l2")
    P, d = q.shape
    vec = (d % 4 == 0) if order == "auto" else order == "vec"
    assert not (vec and d % 4), "the float4 order needs d % 4 == 0"
    w = 4 if vec else 1
    out = torch.empty(P, dtype=torch.float32, device=q.device)
    step = max(1, chunk // max(1, d))
    lane = torch.arange(32, device=q.device)
    for p0 in range(0, P, step):
        ql = _lanes(q[p0:p0 + step].double(), w)
        xl = _lanes(x[p0:p0 + step].double(), w)
        acc = torch.zeros(ql.shape[0], 32, dtype=torch.float64, device=q.device)
        for s in range(ql.shape[1]):
            for j in range(w):
                a, b = xl[:, s, :, j], ql[:, s, :, j]
                if metric == "ip":
                    acc = f32_fma(a, b, acc)
                else:
                    t = f32_add(b, -a)
                    acc = f32_fma(t, t, acc)
        for o in (16, 8, 4, 2, 1):
            acc = f32_add(acc, acc[:, lane ^ o])
        out[p0:p0 + step] = acc[:, 0].to(torch.float32)
    return out


def scores(q: torch.Tensor, x: torch.Tensor, metric: str, order: str = "auto") -> torch.Tensor:
    """warp_exact_score of every (query, row) pair: fp32 [B, d] x [N, d] -> fp32 [B, N]."""
    B, N = q.shape[0], x.shape[0]
    qi = torch.arange(B, device=q.device).repeat_interleave(N)
    xi = torch.arange(N, device=q.device).repeat(B)
    return pair_scores(q[qi], x[xi], metric, order).view(B, N)


# ------------------------------------------------------------------------------------ float64 filter
def _f64_and_bound(q: torch.Tensor, x: torch.Tensor, metric: str):
    """(rank score in float64, bound on |fp32 - float64|), both [B, N]. Rank score: IP value, or minus
    the squared distance under L2 (larger is better)."""
    q64, x64 = q.double(), x.double()
    qn, xn = (q64 * q64).sum(1), (x64 * x64).sum(1)
    d = q.shape[1]
    slack = 1e-12 * (qn[:, None] + xn[None, :])
    if metric == "ip":
        r = q64 @ x64.t()
        a = q64.abs() @ x64.abs().t()
    else:
        dist = (qn[:, None] + xn[None, :] - 2.0 * (q64 @ x64.t())).clamp_min(0.0)
        r = -dist
        a = dist
    return r, (d + 8) * 2.0 ** -23 * a + 2.0 * slack


def _emulate_mask(q, x, metric, mask, order="auto") -> torch.Tensor:
    """fp32 rank scores (IP, or -distance) where mask is set, NaN elsewhere: float64 [B, N]."""
    out = torch.full(mask.shape, float("nan"), dtype=torch.float64, device=q.device)
    qi, xi = mask.nonzero(as_tuple=True)
    if qi.numel():
        s = pair_scores(q[qi], x[xi], metric, order).double()
        out[qi, xi] = s if metric == "ip" else -s
    return out


def _local_excluded(exclude, B: int, N: int, id_offset: int, device) -> torch.Tensor:
    """[B, N] bool: rows each query leaves out (labels as the search returns them, -1 unused)."""
    ex = torch.zeros(B, N, dtype=torch.bool, device=device)
    if exclude is None:
        return ex
    e = torch.as_tensor(exclude, dtype=torch.int64, device=device).reshape(B, -1) - id_offset
    ok = (e >= 0) & (e < N) & (e + id_offset != -1)
    rows = torch.arange(B, device=device)[:, None].expand_as(e)
    ex[rows[ok], e[ok]] = True
    return ex


# ------------------------------------------------------------------------------------ results
def _pad(metric: str) -> float:
    return FLT_MAX if metric == "l2" else -FLT_MAX


def topk(q: torch.Tensor, x: torch.Tensor, k: int, metric: str, exclude=None, id_offset: int = 0):
    """The exact fp32 flat search: (D fp32 [B, k], I int64 [B, k]) ordered by score descending, then
    row id ascending. D is the IP value or the squared L2 distance. Rows each query excludes are
    left out and k is capped at the rows left; missing entries are I = -1, D = -FLT_MAX (IP) or
    FLT_MAX (L2). Labels are row ids + id_offset, as the library returns them."""
    B, N = q.shape[0], x.shape[0]
    dev = q.device
    D = torch.full((B, k), _pad(metric), dtype=torch.float32, device=dev)
    I = torch.full((B, k), -1, dtype=torch.int64, device=dev)
    if B == 0 or N == 0:
        return D, I
    excl = _local_excluded(exclude, B, N, id_offset, dev)
    r, b = _f64_and_bound(q, x, metric)
    r = r.masked_fill(excl, -_INF)
    keff = (N - excl.sum(1)).clamp(max=k)  # [B]
    kk = min(k, N)
    # the k-th best fp32 score is at least the k-th best lower bound: rows that cannot reach it lose
    lo = (r - b).topk(kk, dim=1).values[:, kk - 1:kk]
    cand = (r + b >= lo) & ~excl
    r32 = _emulate_mask(q, x, metric, cand).masked_fill(~cand, -_INF)
    order = torch.sort(r32, dim=1, descending=True, stable=True).indices[:, :kk]  # ties: lower id first
    val = torch.gather(r32, 1, order)
    live = torch.arange(kk, device=dev)[None, :] < keff[:, None]
    d32 = (val if metric == "ip" else -val).to(torch.float32)
    D[:, :kk] = torch.where(live, d32, torch.full_like(d32, _pad(metric)))
    I[:, :kk] = torch.where(live, order + id_offset, torch.full_like(order, -1))
    return D, I


def target_rank(q: torch.Tensor, g: torch.Tensor, target, exclude=None) -> torch.Tensor:
    """rank[i] = number of gallery rows, other than target[i] and exclude[i] (-1: none), whose fp32
    inner product with q[i] beats the target's: a larger score, or an equal score and a lower row id.
    int64 [B]."""
    B, N = q.shape[0], g.shape[0]
    dev = q.device
    t = torch.as_tensor(target, dtype=torch.int64, device=dev).reshape(B)
    e = (torch.full((B,), -1, dtype=torch.int64, device=dev) if exclude is None
         else torch.as_tensor(exclude, dtype=torch.int64, device=dev).reshape(B))
    st = pair_scores(q, g[t], "ip").double()[:, None]
    r, b = _f64_and_bound(q, g, "ip")
    ids = torch.arange(N, device=dev)[None, :]
    out_rows = (ids == t[:, None]) | (ids == e[:, None])
    sure = (r - b > st) & ~out_rows
    band = (r + b >= st) & (r - b <= st) & ~out_rows
    s32 = _emulate_mask(q, g, "ip", band)
    beats = band & ((s32 > st) | ((s32 == st) & (ids < t[:, None])))
    return sure.sum(1) + beats.sum(1)


def label_hits(I: torch.Tensor, labels: torch.Tensor, qlabel: torch.Tensor, ks: Sequence[int]) -> torch.Tensor:
    """hits[i, j] = #{ c < ks[j] : I[i, c] >= 0 and labels[I[i, c]] == qlabel[i] }: int32 [B, len(ks)]."""
    labels = labels.to(I.device)
    hit = (I >= 0) & (labels[I.clamp(min=0)] == qlabel.to(I.device)[:, None])
    cum = torch.cumsum(hit.to(torch.int32), dim=1)
    cols = torch.tensor([min(int(k), I.shape[1]) - 1 for k in ks], device=I.device)
    return cum[:, cols].to(torch.int32)


def merge(Ds: Sequence[torch.Tensor], Is: Sequence[torch.Tensor], k: int, metric: str):
    """Global top-k of per-part search results ([B, k_p] each, labels distinct across parts): valid
    entries ordered by score descending (IP) or distance ascending (L2), then label ascending;
    D keeps each entry's bits. Padding as in topk."""
    D = torch.cat(list(Ds), 1)
    I = torch.cat(list(Is), 1)
    val = (D.double() if metric == "ip" else -D.double()).masked_fill(I < 0, -_INF)
    by_id = torch.sort(I.masked_fill(I < 0, torch.iinfo(torch.int64).max), dim=1, stable=True).indices
    val_i = torch.gather(val, 1, by_id)
    order = torch.gather(by_id, 1, torch.sort(val_i, dim=1, descending=True, stable=True).indices)[:, :k]
    Dk, Ik = torch.gather(D, 1, order), torch.gather(I, 1, order)
    live = Ik >= 0
    B, kk = Dk.shape
    Dout = torch.full((B, k), _pad(metric), dtype=torch.float32, device=D.device)
    Iout = torch.full((B, k), -1, dtype=torch.int64, device=D.device)
    Dout[:, :kk] = torch.where(live, Dk, torch.full_like(Dk, _pad(metric)))
    Iout[:, :kk] = torch.where(live, Ik, torch.full_like(Ik, -1))
    return Dout, Iout


def equal_bits(D_got, I_got, D_ref, I_ref) -> torch.Tensor:
    """[B] bool: row i of (D, I) equals the reference bit for bit."""
    Dg, Dr = D_got.contiguous().view(torch.int32), D_ref.to(D_got.device).contiguous().view(torch.int32)
    return (Dg == Dr).all(1) & (I_got == I_ref.to(I_got.device)).all(1)
