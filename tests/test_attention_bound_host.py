"""CPU: the bound of oracle/attention_exact.py holds for the attention kernels' own fp32 operation
order, and it is tight enough to reject references that model a subtly wrong kernel.

The kernels are emulated step by step in fp32 (fmas through oracle.fp32_exact.f32_fma, adds,
multiplies and divisions as IEEE fp32 tensor operations), in the order neighbour_consumer.cuh uses:
four fma chains and (s0 + s1) + (s2 + s3) for k_cross_attend<64>'s scores, one chain otherwise and
in the backward; lane-strided partial sums of den and dot (lane l takes j = l, l + 32, ...) met in an
xor butterfly; the weighted sums as one fma chain over j. expf is the one step without a bit-exact
model: its results are taken anywhere within its documented 2 ulp of exp, pushed in the direction
that hurts most.
"""
import math

import pytest
import torch

from oracle import attention_exact as ax
from oracle.fp32_exact import f32_fma

F32 = torch.float32


def f32(x):
    return x.to(F32).double()


def ulp32(x):
    """ulp of the fp32 binade holding |x| (float64 tensor)"""
    a = x.abs().clamp_min(2.0 ** -126)
    return torch.exp2(torch.floor(torch.log2(a)) - 23)


def expf_pushed(t, direction):
    """an fp32 value within 2 ulp of exp(t): the farthest one in `direction` (+1 up, -1 down, 0 nearest)"""
    exact = torch.exp(t)
    r = exact.to(F32)
    if isinstance(direction, int):
        direction = torch.full_like(t, direction)
    out = r.double()
    for _ in range(3):
        step = torch.where(direction > 0, torch.nextafter(r, torch.full_like(r, math.inf)),
                           torch.nextafter(r, torch.full_like(r, -math.inf)))
        ok = (direction != 0) & ((step.double() - exact).abs() <= 2 * ulp32(exact)) & (step >= 0)
        r = torch.where(ok, step, r)
    out = r.double()
    assert bool(((out - exact).abs() <= 2 * ulp32(exact)).all())
    return out


def lane_sum(vals, fma_with=None):
    """vals [N, k] -> [N, 1]: lane l sums j = l, l + 32, ... in order (fma(vals, fma_with, acc) if
    given), then an xor butterfly over 16, 8, 4, 2, 1 (every lane ends with the same value)"""
    N, k = vals.shape
    pad = (-k) % 32
    v = torch.nn.functional.pad(vals, (0, pad)).reshape(N, -1, 32)
    b = None if fma_with is None else torch.nn.functional.pad(fma_with, (0, pad)).reshape(N, -1, 32)
    acc = torch.zeros(N, 32, dtype=torch.float64)
    for i in range(v.shape[1]):
        acc = f32_fma(v[:, i], b[:, i] if b is not None else torch.ones_like(acc), acc)
    lanes = torch.arange(32)
    for o in (16, 8, 4, 2, 1):
        acc = f32(acc.to(F32) + acc[:, lanes ^ o].to(F32))
    return acc[:, :1]


def scores(q, K, sigma, dh64):
    N, k, dh = K.shape
    if dh64:
        s = [torch.zeros(N, k, dtype=torch.float64) for _ in range(4)]
        for d4 in range(dh // 4):
            for c in range(4):
                d = 4 * d4 + c
                s[c] = f32_fma(K[:, :, d], q[:, None, d].expand(N, k), s[c])
        lo, hi = s[0].to(F32) + s[1].to(F32), s[2].to(F32) + s[3].to(F32)
        acc = f32(lo + hi)
    else:
        acc = torch.zeros(N, k, dtype=torch.float64)
        for d in range(dh):
            acc = f32_fma(K[:, :, d], q[:, None, d].expand(N, k), acc)
    return f32(acc.to(F32) * torch.tensor(sigma, dtype=F32))


def softmax_parts(q, K, sigma, dh64, direction):
    s = scores(q, K, sigma, dh64)
    m = s.amax(-1, keepdim=True)
    t = f32(s.to(F32) - m.to(F32))
    e = expf_pushed(t, direction)
    den = lane_sum(e)
    inv = f32(1.0 / den.to(F32))
    return e, inv


def emulate_forward(q, K, V, sigma, dh64, direction):
    q, K, V = q.double(), K.double(), V.double()
    N, k, dh = K.shape
    e, inv = softmax_parts(q, K, sigma, dh64, direction)
    acc = torch.zeros(N, dh, dtype=torch.float64)
    for j in range(k):
        acc = f32_fma(e[:, j, None].expand(N, dh), V[:, j], acc)
    return f32(acc.to(F32) * inv.to(F32))


def emulate_backward(q, K, V, dO, sigma, direction):
    q, K, V, g = q.double(), K.double(), V.double(), dO.double()
    N, k, dh = K.shape
    e, inv = softmax_parts(q, K, sigma, False, direction)
    dp = torch.zeros(N, k, dtype=torch.float64)
    for d in range(dh):
        dp = f32_fma(V[:, :, d], g[:, None, d].expand(N, k), dp)
    p = f32(e.to(F32) * inv.to(F32))
    dot = lane_sum(p, dp)
    ds = f32(p.to(F32) * f32(dp.to(F32) - dot.to(F32)).to(F32))
    acc = torch.zeros(N, dh, dtype=torch.float64)
    for j in range(k):
        acc = f32_fma(ds[:, j, None].expand(N, dh), K[:, j], acc)
    sg = torch.tensor(sigma, dtype=F32)
    return {
        "dQ": f32(sg * acc.to(F32)),
        "dK": f32((sg * ds.to(F32))[..., None] * q.to(F32)[:, None, :]),
        "dV": f32(p.to(F32)[..., None] * g.to(F32)[:, None, :]),
    }


def directions(q, K, V, sigma):
    """expf pushes: all up, all down, nearest, up where V_j0 is above the output, and alternating"""
    O, _ = ax.forward(q, K, V, sigma)
    k = K.shape[1]
    tilt = torch.sign(V[:, :, 0].double() - O[:, None, 0])
    alt = (torch.arange(k) % 2 * 2 - 1).double().expand(K.shape[0], k)
    return [1, -1, 0, tilt, alt]


SMALL = [(1, 4), (31, 4), (32, 4), (33, 4), (1, 64), (31, 64), (33, 64), (65, 16), (7, 40)]


@pytest.mark.parametrize("k,dh", SMALL)
@pytest.mark.parametrize("kind", ["random", "sharp", "ties", "cancel"])
def test_the_bound_holds_for_the_kernels_operation_order(k, dh, kind):
    q, K, V, dO = ax.inputs(6, k, dh, kind, seed=k * 100 + dh)
    sigma = ax.scale(dh)
    O, bo = ax.forward(q, K, V, sigma)
    ref, bb = ax.backward(q, K, V, dO, sigma)
    worst = {}
    for direction in directions(q, K, V, sigma):
        for dh64 in ((False, True) if dh % 4 == 0 else (False,)):
            got = emulate_forward(q, K, V, sigma, dh64, direction)
            over = float(((got - O).abs() / bo).max())
            assert over <= 1.0, (dh64, over)
            worst["O"] = max(worst.get("O", 0.0), over)
        got = emulate_backward(q, K, V, dO, sigma, direction)
        for name in ("dQ", "dK", "dV"):
            over = float(((got[name] - ref[name]).abs() / bb[name]).nan_to_num(0.0).max())
            assert over <= 1.0, (name, over)
            worst[name] = max(worst.get(name, 0.0), over)
    print(f"k={k} dh={dh} {kind}: error / bound", {n: f"{v:.2e}" for n, v in worst.items()})


# ------------------------------------------------------------------------------------ not vacuous
def within(got, ref, bound):
    return bool(((got - ref).abs() <= bound).all())


# (B, k, heads, dim_head) of the GPU test where a wrong kernel is easiest to hide: the widest k, two
# lane rounds, the generic kernel
REJECT_SHAPES = [(8, 1024, 8, 64), (2, 33, 6, 40), (3, 64, 16, 64)]


@pytest.mark.parametrize("B,k,heads,dh", REJECT_SHAPES)
def test_the_bound_rejects_subtly_wrong_references(B, k, heads, dh):
    """What a kernel fed by a subtly wrong rule would return must fall outside the bound: a dropped
    neighbour (the last, and the first of the second lane round), the scale of inner instead of
    dim_head, two heads or the two stacks swapped, the previous layer's keys; in the backward, ds
    without - dot, dK and dV swapped, dQ without sigma."""
    g = torch.Generator().manual_seed(B * k + heads)
    L, inner = 3, heads * dh
    Q = torch.randn(2, B, inner, generator=g).float()
    KV = torch.randn(2, B * k, L * 2 * inner, generator=g).float()
    dOut = torch.randn(2, B, inner, generator=g).float()
    sigma = ax.scale(dh)

    def split(layer_cols):
        x = KV[:, :, layer_cols:layer_cols + inner].reshape(2, B, k, heads, dh)
        return x.permute(0, 1, 3, 2, 4).reshape(-1, k, dh)

    q, Kh, Vh, g_ = Q.reshape(-1, dh), split(2 * inner), split(3 * inner), dOut.reshape(-1, dh)
    got = emulate_forward(q, Kh, Vh, sigma, dh == 64, 0)
    O, bo = ax.forward(q, Kh, Vh, sigma)
    assert within(got, O, bo)
    wrong = {}
    for j in {k - 1, min(32, k - 1)}:
        keep = [i for i in range(k) if i != j]
        wrong[f"neighbour {j} dropped"] = ax.forward(q, Kh[:, keep], Vh[:, keep], sigma)[0]
    wrong["scale of inner"] = ax.forward(q, Kh, Vh, ax.scale(inner))[0]
    per_head = O.reshape(2, B, heads, dh)
    if heads > 1:
        wrong["heads 0 and 1 swapped"] = per_head[:, :, [1, 0] + list(range(2, heads))].reshape(-1, dh)
    wrong["stacks swapped"] = per_head.flip(0).reshape(-1, dh)
    wrong["previous layer's keys"] = ax.forward(q, split(0), Vh, sigma)[0]
    for what, ref in wrong.items():
        assert not within(got, ref, bo), what

    if k > 256:
        return  # the backward's emulation is slow at k = 1024; its rejections are shown at the other shapes
    gb = emulate_backward(q, Kh, Vh, g_, sigma, 0)
    ref, bb = ax.backward(q, Kh, Vh, g_, sigma)
    for n in ref:
        assert within(gb[n], ref[n], bb[n]), n
    w, *_ = ax._softmax_terms(q.double(), Kh.double(), sigma)
    p = w / w.sum(-1, keepdim=True)
    dp = (Vh.double() * g_.double()[:, None, :]).sum(-1)
    ds_no_dot = p * dp
    assert not within(gb["dQ"], sigma * (ds_no_dot[..., None] * Kh.double()).sum(-2), bb["dQ"]), "ds without - dot"
    assert not within(gb["dK"], sigma * ds_no_dot[..., None] * q.double()[:, None, :], bb["dK"]), "ds without - dot"
    assert not within(gb["dK"], ref["dV"], bb["dK"]), "dK and dV swapped"
    assert not within(gb["dV"], ref["dK"], bb["dV"]), "dK and dV swapped"
    assert not within(gb["dQ"], ref["dQ"] / sigma, bb["dQ"]), "dQ without sigma"
