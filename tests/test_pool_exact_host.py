"""CPU: the pool reference (oracle/pool_exact.py) against a per-slot loop in exact rational arithmetic,
its power to tell the library's summation orders apart and to reject wrong pools, the softmax
bound against exact evaluation with worst-case weights, and the Python entry points' refusal of a
perm that is not a permutation."""
from fractions import Fraction

import numpy as np
import pytest
import torch

from keds_b200 import retrieval as kr
from oracle import pool_exact as pe

# every distinct (warps, NIF) order of the consume_query callers: latency re-rank and the shard
# consumer (8, 2), the 128-thread two-row throughput re-rank (4, 2), the one-row throughput re-rank
# at 256 / 128 / 64 threads and the fallback (8, 1) (4, 1) (2, 1); at 32 threads it sums like the
# element path (one chain over the slots), SCALAR
ORDERS = {"8w-nif2": pe.LATENCY, "4w-nif2": pe.THROUGHPUT_K128, "8w-nif1": pe.FALLBACK,
          "4w-nif1": pe.throughput(128), "2w-nif1": pe.throughput(64), "scalar": pe.SCALAR}


def unit(n, d, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, d, generator=g, dtype=torch.float64)
    return (x / x.norm(dim=1, keepdim=True)).float()


# ------------------------------------------------------------------ exact rational fp32 arithmetic
def rn32(x: Fraction) -> float:
    """x rounded to the nearest fp32 value, ties to even (normal and subnormal range)."""
    if x == 0:
        return 0.0
    s, a = (-1, -x) if x < 0 else (1, x)
    e = a.numerator.bit_length() - a.denominator.bit_length()
    if Fraction(2) ** e > a:
        e -= 1
    ulp = Fraction(2) ** (max(e, -126) - 23)
    q, r = divmod(a, ulp)
    if r * 2 > ulp or (r * 2 == ulp and q % 2 == 1):
        q += 1
    return s * float(q * ulp)


def fma32(a, b, c):
    return rn32(Fraction(a) * Fraction(b) + Fraction(c))


def loop_pool(vals, wslot, nwarps, nif, vec):
    """The kernel's loops written out slot by slot (consume_query, aux_kernels.cuh)."""
    B, k, d = vals.shape
    out = np.zeros((B, d), np.float32)
    for b in range(B):
        for c in range(d):
            v = lambda jo: float(vals[b, jo, c])
            w = lambda jo: float(wslot[b, jo])
            if not vec:
                acc = 0.0
                for jo in range(k):
                    acc = fma32(w(jo), v(jo), acc)
                out[b, c] = acc
                continue
            part = []
            for warp in range(nwarps):
                acc = 0.0
                jo0 = warp * nif
                while jo0 < k:
                    for t in range(nif):
                        if jo0 + t < k:
                            acc = fma32(w(jo0 + t), v(jo0 + t), acc)
                    jo0 += nwarps * nif
                part.append(acc)
            acc = part[0]
            for g in range(1, nwarps):
                acc = rn32(Fraction(acc) + Fraction(part[g]))
            out[b, c] = acc
    return torch.from_numpy(out)


@pytest.mark.parametrize("nwarps,nif,vec,k,d,perm", [
    (8, 2, True, 16, 8, None), (8, 2, True, 5, 4, [4, 0, 3, 1, 2]), (4, 2, True, 13, 4, "rand"),
    (8, 1, True, 20, 8, None), (2, 1, True, 7, 4, "rand"), (4, 1, True, 1, 4, None), (1, 1, True, 3, 4, None),
    (8, 2, True, 27, 4, "rand"), (4, 2, False, 9, 5, "rand"), (8, 1, True, 16, 4, [0, 0, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 99]),
    (8, 2, True, 6, 4, [-1, 1, 2, 3, 4, 6])])
def test_vectorised_emulation_equals_the_slot_loop(nwarps, nif, vec, k, d, perm):
    """k below warps * NIF, k not a multiple of it, padding ids, bad perm entries (repeated, out of
    range: zero row with the weight of rank 0)."""
    g = torch.Generator().manual_seed(k * 100 + d)
    rows = unit(50, d, k + d)
    I = torch.randint(0, 50, (3, k), generator=g)
    I[1, -1] = -1                                            # padding
    if perm == "rand":
        perm = torch.randperm(k, generator=g)
    perm = None if perm is None else torch.as_tensor(perm)
    w = torch.rand(3, k, generator=g, dtype=torch.float64).float().double() - 0.3   # signed weights
    got = pe.consume_pool(rows, I, w, perm, nwarps, nif, vec)
    vals = pe.gather(rows, I, perm)
    want = loop_pool(vals.numpy(), pe.slot_weights(w, perm, k).numpy(), nwarps, nif, vec)
    assert torch.equal(got.view(torch.int32), want.view(torch.int32))
    # mode 1 through the same helper
    wm = torch.full((3, k), pe.mean_weight(k), dtype=torch.float64)
    assert torch.equal(pe.mean_pool(rows, I, perm, nwarps, nif, vec), pe.consume_pool(rows, I, wm, perm, nwarps, nif, vec))


def test_scalar_path_is_the_one_warp_one_row_order():
    rows, I = unit(100, 12, 1), torch.randint(0, 100, (4, 16), generator=torch.Generator().manual_seed(2))
    a = pe.mean_pool(rows, I, None, 1, 1, True)
    assert torch.equal(a, pe.mean_pool(rows, I, None, 8, 2, False))
    assert pe.mean_weight(3) == float(np.float32(1) / np.float32(3)) and pe.mean_weight(16) == 1 / 16


def test_gather_zero_rows():
    rows = unit(10, 4, 3)
    I = torch.tensor([[3, -1, 12, 5]])
    f = pe.gather(rows, I, torch.tensor([1, 0, 7, -2]))
    assert torch.equal(f[0, 1], rows[3]) and (f[0, 0] == 0).all() and (f[0, 2:] == 0).all()
    f = pe.gather(rows, I)
    assert torch.equal(f[0, 3], rows[5]) and (f[0, 1] == 0).all() and (f[0, 2] == 0).all()


# ------------------------------------------------------------------ the orders differ
def test_the_orders_can_be_told_apart():
    """Random unit rows at k = 16, mean weights: every pair of distinct orders disagrees in a large
    share of the pool entries, so a bitwise comparison names the route that ran."""
    rows = unit(4000, 256, 5)
    I = torch.randint(0, 4000, (16, 16), generator=torch.Generator().manual_seed(6))
    pools = {n: pe.mean_pool(rows, I, None, *o) for n, o in ORDERS.items()}
    names = list(pools)
    for i, a in enumerate(names):
        for b in names[i + 1:]:
            share = (pools[a].view(torch.int32) != pools[b].view(torch.int32)).double().mean().item()
            assert share > 0.5, (a, b, share)


# ------------------------------------------------------------------ mutations are rejected
def _case(k=16, B=6, d=64, seed=7):
    g = torch.Generator().manual_seed(seed)
    rows = unit(500, d, seed)
    I = torch.stack([torch.randperm(500, generator=g)[:k] for _ in range(B)])
    # D in rank order, neighbours 1e-3 apart
    D = (0.4 - 1e-3 * torch.arange(k, dtype=torch.float64)).float().expand(B, k).contiguous()
    return rows, I, D


def _kernel_like_softmax(D, I, tau, l2):
    """fp32 weights as consume_query forms them, with a correctly rounded exp in place of __expf."""
    z = ((-tau if l2 else tau) * D.double()).float()
    mx = z.amax(1, keepdim=True)
    e = torch.exp((z - mx).double()).float()
    e = e.masked_fill(I < 0, 0.0)
    s = torch.zeros(D.shape[0], dtype=torch.float32)
    for j in range(D.shape[1]):
        s = s + e[:, j]
    return (e * (1.0 / s)[:, None]).double()


def _outside(p, ref, bound):
    return ((p.double() - ref).abs() > bound).any(1)


@pytest.mark.parametrize("name", list(ORDERS))
def test_mean_pool_mutations_are_rejected(name):
    nw, nif = ORDERS[name]
    rows, I, _ = _case()
    k = I.shape[1]
    ref = pe.mean_pool(rows, I, None, nw, nif)
    ulp = ref.clone()
    ulp[:, 3] = torch.nextafter(ulp[:, 3], torch.full_like(ulp[:, 3], 1.0))
    dropped = I.clone()
    dropped[:, 5] = -1
    twice = torch.arange(k)
    twice[5] = 6                                              # neighbour 6 twice, neighbour 5 never
    for what, p in (("1 ulp", ulp), ("dropped", pe.mean_pool(rows, dropped, None, nw, nif)),
                    ("twice", pe.mean_pool(rows, I, twice, nw, nif))):
        assert not pe.equal_rows(p, ref).any(), what
    for other, o in ORDERS.items():
        if o != (nw, nif):
            assert (~pe.equal_rows(pe.mean_pool(rows, I, None, *o), ref)).sum() >= 5, other


@pytest.mark.parametrize("tau", [50.0, 0.5])
@pytest.mark.parametrize("l2", [False, True])
def test_softmax_bound_accepts_the_kernel_and_rejects_mutations(tau, l2):
    rows, I, D = _case()
    if l2:
        D = (2.0 - 2.0 * D.double()).float()                   # distances ascend in rank order
    k = I.shape[1]
    ref, bound = pe.softmax_pool_bound(rows, I, D, None, tau, l2, 8)
    w = _kernel_like_softmax(D, I, tau, l2)
    for o in ORDERS.values():
        p = pe.consume_pool(rows, I, w, None, *o)
        assert not _outside(p, ref, bound).any(), o
    lo, hi = pe.softmax_weight_interval(D, I, tau, l2)
    assert ((w >= lo) & (w <= hi)).all()
    # the weights of ranks 3 and 4 (D 1e-3 apart) swapped
    ws = w.clone()
    ws[:, [3, 4]] = ws[:, [4, 3]]
    # the lightest neighbour dropped, and one neighbour counted twice (another lost)
    dropped = I.clone()
    dropped[:, k - 1] = -1
    twice = torch.arange(k)
    twice[k - 1] = 0
    for what, p in (("swapped", pe.consume_pool(rows, I, ws, None, *pe.LATENCY)),
                    ("dropped", pe.consume_pool(rows, dropped, w, None, *pe.LATENCY)),
                    ("twice", pe.consume_pool(rows, I, w, twice, *pe.LATENCY))):
        assert _outside(p, ref, bound).all(), what


def test_softmax_bound_holds_against_exact_evaluation():
    """Small cases, weights pushed to the ends of the interval in the direction that moves each
    column furthest (and __expf results off by their documented ulps): the fp32 pool of those
    weights, in every order, stays within the bound of the exact pool sum_j w_j r_j."""
    g = torch.Generator().manual_seed(11)
    for case in range(6):
        k, d = (3, 4, 5, 6, 7, 8)[case], 4
        tau, l2 = (50.0, 0.5, 20.0)[case % 3], bool(case % 2)
        rows = unit(40, d, 20 + case)
        I = torch.randperm(40, generator=g)[:k][None, :]
        if case == 5:
            I[0, -2:] = -1                                     # padding: weight 0
        D = torch.sort(torch.rand(1, k, generator=g) * 0.5, dim=1, descending=not l2).values
        ref, bound = pe.softmax_pool_bound(rows, I, D, None, tau, l2, 8)
        lo, hi = pe.softmax_weight_interval(D, I, tau, l2)
        # exact pool: exp in float64 (its rounding is inside the bound's 1e-15 term), the rest rational
        st = -tau if l2 else tau
        valid = [int(i) >= 0 for i in I[0]]
        z = [st * float(D[0, j]) for j in range(k)]
        mx = max(z[j] for j in range(k) if valid[j])
        E = [Fraction(np.exp(z[j] - mx)) if valid[j] else Fraction(0) for j in range(k)]
        S = sum(E)
        r = pe.gather(rows, I)[0].double()
        for c in range(d):
            exact = sum(E[j] / S * Fraction(float(r[j, c])) for j in range(k))
            for up in (True, False):
                # each weight at the end of its interval that moves column c up (down), rounded inwards
                wj = []
                for j in range(k):
                    want_hi = (float(r[j, c]) >= 0) == up
                    x = float(hi[0, j] if want_hi else lo[0, j])
                    f = np.float32(x)
                    if want_hi and float(f) > x:
                        f = np.nextafter(f, np.float32(0))
                    if not want_hi and float(f) < x:
                        f = np.nextafter(f, np.float32(1))
                    wj.append(float(f))
                wt = torch.tensor([wj], dtype=torch.float64)
                for o in ORDERS.values():
                    p = pe.consume_pool(rows, I, wt, None, *o)[0, c]
                    assert abs(Fraction(float(p)) - exact) <= Fraction(float(bound[0, c])), (case, c, up, o)
        # __expf off by its documented ulps in either direction, then the kernel's fp32 steps: inside
        for sgn in (1, -1):
            xs = [np.float32(np.float32(z[j]) - np.float32(mx)) for j in range(k)]
            e = []
            for j in range(k):
                if not valid[j]:
                    e.append(np.float32(0))
                    continue
                v = np.float32(np.exp(np.float64(xs[j])))
                n = 2 + int(abs(1.173 * float(xs[j])))
                for _ in range(n):
                    v = np.nextafter(v, np.float32(np.inf if (sgn > 0) == (j == 0) else 0))
                e.append(v)
            s = np.float32(0)
            for v in e:
                s = np.float32(s + v)
            inv = np.float32(np.float32(1) / s)
            wk = torch.tensor([[float(np.float32(v * inv)) for v in e]], dtype=torch.float64)
            assert ((wk >= lo) & (wk <= hi)).all(), (case, sgn)


def test_weighted_pool_skips_invalid_ids():
    rows = unit(20, 5, 9)
    I = torch.tensor([[0, -1, 3, 25], [19, 19, -4, 2]])
    W = torch.randn(2, 3, 4, generator=torch.Generator().manual_seed(1))
    got = pe.weighted_pool(rows, I, W)
    for b in range(2):
        for h in range(3):
            for c in range(5):
                acc = 0.0
                for j in range(4):
                    i = int(I[b, j])
                    if 0 <= i < 20:
                        acc = fma32(float(W[b, h, j]), float(rows[i, c]), acc)
                assert float(got[b, h, c]) == acc


# ------------------------------------------------------------------ perm must be a permutation
@pytest.mark.parametrize("perm", [[0, 0, 1, 2], [0, 1, 2, 4], [-1, 0, 1, 2], [3, 2, 1], [0, 1, 2, 3, 4]])
def test_entry_points_refuse_a_host_perm_that_is_no_permutation(perm):
    p = torch.tensor(perm)
    with pytest.raises(ValueError, match="perm"):
        kr.check_perm(p, 4, "perm")
    # checked before the call touches its indices or query
    with pytest.raises(ValueError, match="perm_img"):
        kr.retrieve2(None, None, torch.zeros(2, 4), 4, perm_img=p)
    with pytest.raises(ValueError, match="perm_txt"):
        kr.retrieve2(None, None, torch.zeros(2, 4), 4, perm_txt=p.to(torch.int32))
    with pytest.raises(ValueError, match="perm_img"):
        kr.RetrievalStep(None, None, 2, 4, perm_img=p)
    kr.check_perm(torch.tensor([2, 0, 3, 1], dtype=torch.int32), 4)
