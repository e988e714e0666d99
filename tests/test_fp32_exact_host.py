"""CPU: the bit-exact fp32 reference (oracle/fp32_exact.py) checked on its own -- its fma and add
against exact rational rounding, its vectorised lanes against a plain per-lane loop, its power to
tell the library's summation order from others, and a mutation check that the bitwise comparison
the GPU tests use rejects small, realistic mistakes in a result."""
from fractions import Fraction

import numpy as np
import pytest
import torch

from oracle import fp32_exact as fx


def rn32_exact(v: Fraction) -> float:
    """Round a rational to the nearest fp32 value, ties to even (no overflow in these tests)."""
    if v == 0:
        return 0.0
    sign = -1 if v < 0 else 1
    a = abs(v)
    e = a.numerator.bit_length() - a.denominator.bit_length()
    if Fraction(2) ** e > a:
        e -= 1
    ulp_e = max(e, -126) - 23  # subnormals share the exponent of the smallest normal binade
    scaled = a / Fraction(2) ** ulp_e
    n = scaled.numerator // scaled.denominator
    rem = scaled - n
    if rem > Fraction(1, 2) or (rem == Fraction(1, 2) and n % 2 == 1):
        n += 1
    return sign * float(Fraction(n) * Fraction(2) ** ulp_e)


def f32(v) -> torch.Tensor:
    return torch.tensor(v, dtype=torch.float32).double()


def random_f32(rng, n, lo_exp, hi_exp):
    m = rng.uniform(1.0, 2.0, n) * rng.choice([-1.0, 1.0], n)
    return (m * np.exp2(rng.integers(lo_exp, hi_exp, n))).astype(np.float32)


def test_fma_and_add_equal_exact_rounding():
    rng = np.random.default_rng(1)
    n = 4000
    a, b, c = random_f32(rng, n, -20, 20), random_f32(rng, n, -20, 20), random_f32(rng, n, -40, 40)
    # a tenth of the products subnormal in fp32 (and results near them)
    s = n // 10
    a[:s] = random_f32(rng, s, -80, -70)
    b[:s] = random_f32(rng, s, -80, -60)
    c[:s] = random_f32(rng, s, -150, -125)
    # c close to -a*b: cancellation, the error term decides the rounding
    c[s:2 * s] = -(a[s:2 * s].astype(np.float64) * b[s:2 * s]).astype(np.float32)
    fma = fx.f32_fma(f32(a), f32(b), f32(c)).numpy()
    add = fx.f32_add(f32(a), f32(c)).numpy()
    for i in range(n):
        A, B, Cc = Fraction(float(a[i])), Fraction(float(b[i])), Fraction(float(c[i]))
        assert fma[i] == rn32_exact(A * B + Cc), (i, a[i], b[i], c[i])
        assert add[i] == rn32_exact(A + Cc), (i, a[i], c[i])


def test_fma_double_rounding_trap():
    """a*b + c rounded once to float64 and then to fp32 lands on the wrong side of a tie; the
    round-to-odd sum does not."""
    a = (2 ** 23 + 2896) * 2.0 ** -23
    b = (2 ** 23 - 2895) * 2.0 ** -47
    c = 1.0
    exact = rn32_exact(Fraction(a) * Fraction(b) + Fraction(c))
    naive = float(np.float32(a * b + c))
    assert naive != exact
    assert fx.f32_fma(f32([a]), f32([b]), f32([c])).item() == exact
    # and nextafter towards s + err would have left the sum where it was
    s = torch.tensor([a * b + c], dtype=torch.float64)
    assert torch.nextafter(s, s + 1e-300).item() == s.item()


def loop_score(q: np.ndarray, x: np.ndarray, metric: str, vec: bool) -> np.float32:
    """warp_exact_score written out lane by lane, one fp32 operation at a time (Fraction rounding)."""
    d = q.shape[0]
    r = lambda v: Fraction(rn32_exact(v))
    acc = [Fraction(0)] * 32
    for lane in range(32):
        idx = ([4 * c + j for c in range(lane, d // 4, 32) for j in range(4)] if vec
               else list(range(lane, d, 32)))
        for i in idx:
            qi, xi = Fraction(float(q[i])), Fraction(float(x[i]))
            if metric == "ip":
                acc[lane] = r(xi * qi + acc[lane])
            else:
                t = r(qi - xi)
                acc[lane] = r(t * t + acc[lane])
    for o in (16, 8, 4, 2, 1):
        acc = [r(acc[l] + acc[l ^ o]) for l in range(32)]
    assert len(set(acc)) == 1  # every lane holds the full sum
    return np.float32(float(acc[0]))


@pytest.mark.parametrize("d,order", [(8, "vec"), (8, "scalar"), (132, "vec"), (132, "scalar"),
                                     (260, "vec"), (50, "scalar"), (33, "scalar")])
@pytest.mark.parametrize("metric", ["ip", "l2"])
def test_lanes_equal_a_per_lane_loop(d, order, metric):
    g = torch.Generator().manual_seed(d)
    q, x = torch.randn(6, d, generator=g), torch.randn(6, d, generator=g)
    x[0] = q[0]  # L2 of a row with itself: +0
    got = fx.pair_scores(q, x, metric, order).numpy()
    for i in range(6):
        want = loop_score(q[i].numpy(), x[i].numpy(), metric, order == "vec")
        assert got[i].view(np.int32) == want.view(np.int32), (i, got[i], want)


def test_the_emulated_order_is_told_apart_from_other_orders():
    """At d = 768 the float4 order, the element order and float64-then-round give different fp32
    bits on most IP pairs and on a third of the L2 pairs (squared distances of unit rows sit near 2,
    where the fp32 step is coarser): a kernel that summed in another order fails a bitwise test."""
    g = torch.Generator().manual_seed(7)
    q = torch.nn.functional.normalize(torch.randn(400, 768, generator=g), dim=1)
    x = torch.nn.functional.normalize(torch.randn(400, 768, generator=g), dim=1)
    for metric, share in (("ip", 0.5), ("l2", 0.25)):
        v = fx.pair_scores(q, x, metric, "vec")
        s = fx.pair_scores(q, x, metric, "scalar")
        q64, x64 = q.double(), x.double()
        f64 = ((q64 * x64).sum(1) if metric == "ip" else ((q64 - x64) ** 2).sum(1)).float()
        assert (v != s).float().mean() > share, metric
        assert (v != f64).float().mean() > share, metric
        assert ((v.double() - f64.double()).abs() < 1e-5).all()  # all are fp32 sums of the same terms


def test_scores_and_topk_follow_the_tie_rule():
    g = torch.Generator().manual_seed(3)
    x = torch.randn(300, 20, generator=g)
    x[200:210] = x[5]                      # ten copies of row 5 at higher ids
    q = torch.randn(9, 20, generator=g)
    q[0] = x[5]
    for metric in ("ip", "l2"):
        S = fx.scores(q, x, metric)
        r = S.double() if metric == "ip" else -S.double()
        for k in (1, 11, 300, 310):
            D, I = fx.topk(q, x, k, metric)
            for b in range(9):
                want = sorted(range(300), key=lambda j: (-r[b, j].item(), j))[:k]
                assert I[b, :len(want)].tolist() == want
                assert torch.equal(D[b, :len(want)], S[b, want])
                assert (I[b, len(want):] == -1).all()
                assert (D[b, len(want):] == (fx.FLT_MAX if metric == "l2" else -fx.FLT_MAX)).all()
        D, I = fx.topk(q, x, 11, metric)
        assert I[0].tolist()[:11] == [5] + list(range(200, 210)) or metric == "ip"
        if metric == "l2":
            assert (D[0, :11].view(torch.int32) == 0).all()   # +0, not -0
        # exclusion: labels with an offset, -1 and repeats ignored, k capped at the rows left
        ex = torch.full((9, 8), -1, dtype=torch.int64)
        ex[:, 0] = ex[:, 1] = I[:, 0] + 1000    # the best row, twice
        ex[:, 2] = 1000 + 299
        ex[:, 3] = 999                          # outside the database
        D2, I2 = fx.topk(q, x, 300, metric, exclude=ex, id_offset=1000)
        for b in range(9):
            gone = {int(I[b, 0]), 299}
            want = [j for j in sorted(range(300), key=lambda j: (-r[b, j].item(), j)) if j not in gone]
            assert (I2[b, :298] - 1000).tolist() == want and (I2[b, 298:] == -1).all()


def test_target_rank_and_label_hits_count_what_the_definition_says():
    g = torch.Generator().manual_seed(4)
    gal = torch.randn(200, 12, generator=g)
    gal[150] = gal[40]
    gal[20] = gal[40]                       # copies of row 40 below and above it
    q = torch.randn(30, 12, generator=g)
    t = torch.randint(0, 200, (30,), generator=g)
    t[:3] = 40
    e = torch.randint(-1, 200, (30,), generator=g)
    e[0], e[1] = 20, -1
    q[1] = q[0]
    S = fx.scores(q, gal, "ip")
    got = fx.target_rank(q, gal, t, e)
    for b in range(30):
        st, tb = S[b, t[b]], int(t[b])
        want = sum(1 for j in range(200) if j not in (tb, int(e[b])) and (S[b, j] > st or (S[b, j] == st and j < tb)))
        assert got[b].item() == want
    assert got[1] - got[0] == 1  # row 20 ties the target at 40 and wins on its lower id unless excluded
    labels = torch.randint(0, 3, (200,), generator=g)
    qlab = torch.randint(0, 3, (30,), generator=g)
    _, I = fx.topk(q, gal, 210, "ip")
    H = fx.label_hits(I, labels, qlab, [1, 5, 200, 210])
    for b in range(30):
        for c, k in enumerate([1, 5, 200, 210]):
            assert H[b, c] == sum(1 for j in I[b, :k].tolist() if j >= 0 and labels[j] == qlab[b])


def test_merge_orders_parts_by_score_then_label():
    g = torch.Generator().manual_seed(5)
    lat = (torch.randint(-2, 3, (400, 8), generator=g) / 8.0)
    q = (torch.randint(-2, 3, (6, 8), generator=g) / 8.0)
    for metric in ("ip", "l2"):
        D, I = fx.topk(q, lat, 40, metric)
        parts = [(fx.topk(q, lat[lo:hi], 40, metric, id_offset=lo)) for lo, hi in ((0, 150), (150, 390), (390, 400))]
        Dm, Im = fx.merge([p[0] for p in parts], [p[1] for p in parts], 40, metric)
        assert fx.equal_bits(Dm, Im, D, I).all()


def mutations(D, I, metric):
    """Small, realistic mistakes: each returns a mutated copy of (D, I)."""
    out = {}
    tie = None
    for b in range(D.shape[0]):
        for c in range(D.shape[1] - 1):
            if D[b, c] == D[b, c + 1] and I[b, c + 1] >= 0:
                tie = (b, c)
                break
        if tie:
            break
    assert tie is not None
    m = I.clone()
    b, c = tie
    m[b, c], m[b, c + 1] = I[b, c + 1], I[b, c]
    out["tied rows swapped"] = (D, m)
    m = D.clone()
    m[1, 3] = torch.nextafter(D[1, 3], torch.tensor(float("inf")))
    out["D one ulp off"] = (m, I)
    return out


def test_bitwise_comparison_rejects_each_mutation():
    g = torch.Generator().manual_seed(6)
    lat = torch.randint(-2, 3, (3000, 64), generator=g) / 8.0      # lattice: many exact ties
    q = torch.randint(-2, 3, (8, 64), generator=g) / 8.0
    k = 10
    for metric in ("ip", "l2"):
        D, I = fx.topk(q, lat, k, metric)
        assert fx.equal_bits(D, I, D, I).all()
        muts = mutations(D, I, metric)
        Dk1, Ik1 = fx.topk(q, lat, k + 1, metric)
        D3, I3 = D.clone(), I.clone()
        D3[:, -1], I3[:, -1] = Dk1[:, -1], Ik1[:, -1]                  # the (k+1)-th row in the k-th place
        muts["k-th row replaced by the (k+1)-th"] = (D3, I3)
        Ds, Is = fx.topk(q, lat[:5], k, metric)                       # short result: padding
        Dp = Ds.clone()
        Dp[:, 5:] = -Dp[:, 5:]                                         # wrong sign of the padding
        muts["wrong padding"] = (Dp, Is)
        Ip = Is.clone()
        Ip[:, 5:] = 0
        muts["padding ids"] = (Ds, Ip)
        for name, (Dm, Im) in muts.items():
            ref = (Ds, Is) if "padding" in name else (D, I)
            assert not fx.equal_bits(Dm, Im, *ref).all(), name
