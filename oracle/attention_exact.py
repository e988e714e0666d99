"""float64 reference for the consumer's single-query cross-attention, forward and backward, with a
per-element bound on how far the fp32 kernels (k_cross_attend<64>, k_cross_attend<0>,
k_cross_attend_bwd in keds_b200/csrc/neighbour_consumer.cuh) can be from it.

One head: q [dh], K, V [k][dh] (rows j = neighbours), dO [dh], all fp32 values, and sigma = the fp32
scale the library uses, RN32(1 / RN32(sqrt(dh))). The reference is exact arithmetic on those inputs
(evaluated in float64):

    s_j = sigma q.K_j,  p = softmax(s),  O = sum_j p_j V_j
    dp_j = dO.V_j,  dot = sum_j p_j dp_j,  ds_j = p_j (dp_j - dot)
    dQ = sigma sum_j ds_j K_j,  dK_j = sigma ds_j q,  dV_j = p_j dO

What the kernels do (u = 2^-24, gamma_n = n u / (1 - n u)):
  * score: an fma chain over d (k_cross_attend<64>: four chains over d = c mod 4, then
    (s0 + s1) + (s2 + s3)), then one multiply by sigma. At most dh + 1 roundings touch a term, so
    |s~_j - s_j| <= E_j = gamma_{dh+1} sigma sum_d |K_jd q_d|.
  * m = max_j s~_j (exact); t_j = RN(s~_j - m), |t_j - (s~_j - m)| <= u |s~_j - m|.
  * e_j = expf(t_j): CUDA's expf (no fast-math) is within 2 ulp of exp(t_j): relative 4u for a
    normal result, absolute 2^-148 below the normal range (an underflow to 0 is within that too).
    With m* = max_j s_j, w_j = exp(s_j - m*) and c = exp(m* - m):
        e_j = c w_j (1 + rho_j) + a_j,   |rho_j| <= exp(E_j + u |t_j|)(1 + 4u) - 1,   |a_j| <= 2^-148,
    |m - m*| <= max E, so |t_j| <= (m* - s_j) + 2 max E and a_j / c <= alpha = 2^-148 exp(max E).
  * den: lane l adds e_l, e_{l+32}, ... in order, then an xor butterfly over 16, 8, 4, 2, 1:
    every e_j passes through at most n = ceil(k / 32) + 5 roundings, |den~ - sum e| <= gamma_n sum e.
    inv = RN(1 / den~). Together: RN(x inv) = (x / sum e)(1 + phi), |phi| <= r = (2u + u^2 + gamma_n) / (1 - gamma_n).
  * forward: acc_d = fma chain over j of e_j V_jd (gamma_k), O~_d = RN(acc_d inv).
    Because sum_j w_j (V_jd - O_d) = 0, the exact ratio of the kernel's weights is off by
        (sum_j e_j V_jd) / (sum_j e_j) - O_d = sum_j (e_j - c w_j)(V_jd - O_d) / sum_j e_j,
    and sum_j e_j >= c D_lo with D_lo = sum_j w_j (1 - rho_j) - k alpha. With
    A_d = sum_j (w_j (1 + rho_j) + alpha) |V_jd| / D_lo (>= |sum e V| / sum e):
        |O~_d - O_d| <= sum_j (w_j rho_j + alpha) |V_jd - O_d| / D_lo + A_d (gamma_k + (1 + gamma_k) r).
  * backward: scores and dp_j each one fma chain over d: |dp~_j - dp_j| <= F_j = gamma_dh sum_d |V_jd dO_d|.
    p~_j = RN(e_j inv) lies in [P_lo (1 - r), P_hi (1 + r)] with P_hi = (w_j (1 + rho_j) + alpha) / D_lo,
    P_lo = (w_j (1 - rho_j) - alpha)^+ / D_hi, D_hi = sum_j w_j (1 + rho_j) + k alpha; Pi_j bounds
    |p~_j - p_j| and pbar_j = P_hi (1 + r) bounds p~_j.
    dot~: per-lane fma chains plus the butterfly (gamma_n again):
        |dot~ - dot| <= T = sum_j (Pi_j |dp_j| + pbar_j F_j) + gamma_n sum_j pbar_j (|dp_j| + F_j),
    i.e. the cancellation in dp_j - dot costs in proportion to sum_j p_j |dp_j|, not to |dp_j - dot|.
    x~_j = RN(dp~_j - dot~): |x~_j - x_j| <= Y_j = F_j + T + u (|x_j| + F_j + T), xbar_j = |x_j| + Y_j.
    ds~_j = RN(p~_j x~_j): |ds~_j - ds_j| <= S_j = Pi_j xbar_j + p_j Y_j + u pbar_j xbar_j, dsbar_j = |ds_j| + S_j.
    dK~_jd = RN(RN(sigma ds~_j) q_d):  |.| <= sigma |q_d| (S_j + gamma_2 dsbar_j).
    dV~_jd = RN(p~_j dO_d):            |.| <= |dO_d| (Pi_j + u pbar_j).
    dQ~_d = RN(sigma acc_d), acc_d an fma chain over j of ds~_j K_jd:
        |.| <= sigma ((1 + u)(sum_j S_j |K_jd| + gamma_k sum_j dsbar_j |K_jd|) + u sum_j dsbar_j |K_jd|).

Underflow: a product or fma rounded to a subnormal is off by up to MU = 2^-150 absolute, not u
relative (adds stay exact there). Each such rounding adds MU where it happens: (dh + 1) MU to E_j,
dh MU to F_j, MU to p~_j and ds~_j, (k + 32) MU to dot~, k MU to every fma chain over j, MU to each
final product; in the forward, k + 1 such errors in units of the weights cost (k + 1) alpha / D_lo.

The float64 evaluation of the reference and of the bound is itself rounded, by at most about
(k + dh) 2^-53 of the same sums of magnitudes that the bound multiplies by gamma_k >= 2^-24, so a
factor 1 + 2^-20 on the bound covers it.

TEST INFRASTRUCTURE ONLY (tests/ may import it; keds_b200/ never). Torch float64, any device.
Batched: q [N, dh], K and V [N, k, dh], dO [N, dh], one head per leading index.
"""
from __future__ import annotations

import math

import numpy as np
import torch

U = 2.0 ** -24
EXPF_ABS = 2.0 ** -148           # 2 ulp of expf below the normal range
MU = 2.0 ** -150                 # the absolute error of a product or fma rounded to a subnormal
SLACK = 1.0 + 2.0 ** -20         # the float64 evaluation of reference and bound


def gamma(n) -> float:
    return n * U / (1.0 - n * U)


def scale(dim_head: int) -> float:
    """1.0f / sqrtf(dim_head) as the library computes it (both operations correctly rounded)."""
    return float(np.float32(1.0) / np.sqrt(np.float32(dim_head)))


def _softmax_terms(q, K, sigma):
    """(w, rho, alpha, D_lo, D_hi): the weights exp(s_j - max s) and their error model (docstring)"""
    k, dh = K.shape[-2], K.shape[-1]
    prod = K * q[:, None, :]                               # products of two fp32 values: exact
    s = sigma * prod.sum(-1)
    E = gamma(dh + 1) * sigma * prod.abs().sum(-1) + (dh + 1) * MU
    Emax = E.amax(-1, keepdim=True)
    smax = s.amax(-1, keepdim=True)
    w = torch.exp(s - smax)
    t_abs = (smax - s) + 2 * Emax
    rho = torch.exp(E + U * t_abs) * (1 + 4 * U) - 1
    alpha = EXPF_ABS * torch.exp(Emax)
    D_lo = (w * (1 - rho)).sum(-1, keepdim=True) - k * alpha
    D_hi = (w * (1 + rho)).sum(-1, keepdim=True) + k * alpha
    assert bool((D_lo > 0).all())
    return w, rho, alpha, D_lo, D_hi


def _r(k: int) -> float:
    g = gamma(math.ceil(k / 32) + 5)
    return (2 * U + U * U + g) / (1 - g)


def forward(q: torch.Tensor, K: torch.Tensor, V: torch.Tensor, sigma: float):
    """(O [N, dh], bound [N, dh]) in float64 for fp32 inputs (any float dtype holding fp32 values)."""
    q, K, V = q.double(), K.double(), V.double()
    k = K.shape[-2]
    w, rho, alpha, D_lo, _ = _softmax_terms(q, K, sigma)
    O = (w[..., None] * V).sum(-2) / w.sum(-1, keepdim=True)
    gk = gamma(k)
    A = ((w * (1 + rho) + alpha)[..., None] * V.abs()).sum(-2) / D_lo
    weights = ((w * rho + alpha)[..., None] * (V - O[:, None, :]).abs()).sum(-2) / D_lo
    bound = weights + A * (gk + (1 + gk) * _r(k)) + (k + 1) * alpha / D_lo + MU
    return O, bound * SLACK


def backward(q: torch.Tensor, K: torch.Tensor, V: torch.Tensor, dO: torch.Tensor, sigma: float):
    """float64 dict {dQ [N, dh], dK [N, k, dh], dV [N, k, dh]} and a dict of bounds of the same shapes."""
    q, K, V, g = q.double(), K.double(), V.double(), dO.double()
    k, dh = K.shape[-2], K.shape[-1]
    w, rho, alpha, D_lo, D_hi = _softmax_terms(q, K, sigma)
    r = _r(k)
    gn = gamma(math.ceil(k / 32) + 5)
    p = w / w.sum(-1, keepdim=True)
    P_hi = (w * (1 + rho) + alpha) / D_lo
    P_lo = (w * (1 - rho) - alpha).clamp_min(0) / D_hi
    pbar = P_hi * (1 + r) + MU
    Pi = torch.maximum(pbar - p, p - P_lo * (1 - r) + MU)
    vg = V * g[:, None, :]
    dp = vg.sum(-1)
    F = gamma(dh) * vg.abs().sum(-1) + dh * MU
    dot = (p * dp).sum(-1, keepdim=True)
    T = ((Pi * dp.abs() + pbar * F).sum(-1, keepdim=True) + gn * (pbar * (dp.abs() + F)).sum(-1, keepdim=True)
         + (k + 32) * MU)
    x = dp - dot
    Y = F + T + U * (x.abs() + F + T)
    xbar = x.abs() + Y
    ds = p * x
    S = Pi * xbar + p * Y + U * pbar * xbar + MU
    dsbar = ds.abs() + S
    gk = gamma(k)
    ref = {
        "dQ": sigma * (ds[..., None] * K).sum(-2),
        "dK": sigma * ds[..., None] * q[:, None, :],
        "dV": p[..., None] * g[:, None, :],
    }
    bound = {
        "dQ": sigma * ((1 + U) * ((S[..., None] * K.abs()).sum(-2) + gk * (dsbar[..., None] * K.abs()).sum(-2))
                       + U * (dsbar[..., None] * K.abs()).sum(-2) + (1 + U) * k * MU) + MU,
        "dK": sigma * q.abs()[:, None, :] * (S + gamma(2) * dsbar)[..., None] + (1 + U) * MU * q.abs()[:, None, :] + MU,
        "dV": g.abs()[:, None, :] * (Pi + U * pbar)[..., None] + MU,
    }
    return ref, {n: b * SLACK for n, b in bound.items()}


# ------------------------------------------------------------------------------------ inputs
def inputs(n: int, k: int, dh: int, kind: str, seed: int, device="cpu"):
    """fp32 (q [n, dh], K [n, k, dh], V [n, k, dh], dO [n, dh]) of one of the kinds the kernels find hard:
      'random'  unit normal;
      'sharp'   scores spread evenly over [-80, 80] (p spans ~70 orders of magnitude, most expf
                results subnormal or zero);
      'ties'    small integer entries, so q.K_j is exact in fp32 and many scores tie exactly;
      'cancel'  every V_j the same row up to 2^-20: dp_j - dot cancels to a few ulps."""
    g = torch.Generator().manual_seed(seed)
    q = torch.randn(n, dh, generator=g, dtype=torch.float64)
    K = torch.randn(n, k, dh, generator=g, dtype=torch.float64)
    V = torch.randn(n, k, dh, generator=g, dtype=torch.float64)
    dO = torch.randn(n, dh, generator=g, dtype=torch.float64)
    if kind == "sharp":
        # K_j = (noise orthogonal to q) + target_j / (sigma |q|^2) q: s_j = target_j up to rounding
        target = torch.linspace(-80, 80, k, dtype=torch.float64)[torch.randperm(k, generator=g)]
        qq = (q * q).sum(-1, keepdim=True)
        K = K - (K * q[:, None, :]).sum(-1, keepdim=True) / qq[:, None] * q[:, None, :]
        K = K + (target[None, :, None] / (scale(dh) * qq[:, None])) * q[:, None, :]
    elif kind == "ties":
        q = torch.randint(-2, 3, (n, dh), generator=g).double()
        K = torch.randint(-1, 2, (n, max(1, k // 4), dh), generator=g).double()
        K = K[:, torch.randint(0, K.shape[1], (k,), generator=g)]
        dO = torch.randint(-3, 4, (n, dh), generator=g).double()
    elif kind == "cancel":
        V = V[:, :1] + 2.0 ** -20 * V
    elif kind != "random":
        raise ValueError(kind)
    return tuple(t.to(torch.float32).to(device) for t in (q, K, V, dO))
