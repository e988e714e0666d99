"""Bit-exact fp32 reference for the library's range search (keds_index_range_search).

Built on oracle/fp32_exact.py: its float64 filter decides the rows that cannot reach the radius, and
its emulation of `warp_exact_score` scores every other row bit for bit, so a test can compare the
library's lims, D and I with `==`. Plain torch; runs on CPU tensors, and in float64 on a CUDA device
for large cases.
"""
from __future__ import annotations

import torch

from .fp32_exact import _emulate_mask, _f64_and_bound


def range_search(q: torch.Tensor, x: torch.Tensor, radius: float, metric: str, id_offset: int = 0):
    """The exact fp32 range search: every row with fp32 score > radius (IP) or fp32 squared distance
    < radius (L2), strictly. Returns (lims int64 [B + 1], D fp32 [lims[B]], I int64 [lims[B]]) in
    Faiss' layout, each query's entries ordered by score descending (distance ascending), then row
    id ascending; labels are row ids + id_offset. The radius is taken as the library takes it,
    rounded to fp32. Rows whose float64 interval cannot pass it are left out; every other row (the
    hits and the rows near the boundary) is emulated bit for bit, so D holds the fp32 bits."""
    B, N = q.shape[0], x.shape[0]
    dev = q.device
    if B == 0 or N == 0:
        return (torch.zeros(B + 1, dtype=torch.int64, device=dev), torch.zeros(0, dtype=torch.float32, device=dev),
                torch.zeros(0, dtype=torch.int64, device=dev))
    r32 = float(torch.tensor(float(radius), dtype=torch.float32))
    t = r32 if metric == "ip" else -r32  # a hit: rank score (IP value, or minus the distance) > t
    r, b = _f64_and_bound(q, x, metric)
    cand = r + b >= t
    s32 = _emulate_mask(q, x, metric, cand)
    hit = cand & (s32 > t)
    val = s32.masked_fill(~hit, -float("inf"))
    order = torch.sort(val, dim=1, descending=True, stable=True).indices  # ties: lower id first
    cnt = hit.sum(1)
    lims = torch.zeros(B + 1, dtype=torch.int64, device=dev)
    lims[1:] = torch.cumsum(cnt, 0)
    keep = torch.arange(N, device=dev)[None, :] < cnt[:, None]
    v = torch.gather(val, 1, order)[keep]
    D = (v if metric == "ip" else -v).to(torch.float32)
    return lims, D, order[keep] + id_offset
