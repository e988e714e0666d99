"""GPU: range search against the bit-exact fp32 reference (oracle/range_exact.py).

`GpuIndexFlat.range_search(q, r)` returns every row with fp32 score > r (IP) or fp32 squared
distance < r (L2), in Faiss' (lims, D, I) layout, best first and ties by lower label. Here lims, the
bits of D and I are compared with `==` on both metrics and operand formats, widths that are and are
not multiples of 64 and of 4, row counts off the 256-row tile, radii with no, about 16 and about 1000
hits per query, hard data (clusters, 32-fold duplicates with ties at the radius, values beyond fp16,
a query beyond fp16), a radius that admits every row (the candidate buffer grows), several passes,
and the other entry points. Every call is followed by a clean device status."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from keds_b200.database import drop_near_duplicates  # noqa: E402
from keds_b200.index import METRIC_INNER_PRODUCT, METRIC_L2, GpuIndexFlat, IndexReplicas  # noqa: E402
from oracle import range_exact as rx  # noqa: E402

Q_PASS_MAX = 16384  # api.cu: queries per pass


def unit(n, d, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, d, generator=g)
    return (x / x.norm(dim=1, keepdim=True)).cuda()


def build(db, metric, fmt=None):
    ix = GpuIndexFlat(db.shape[1], METRIC_L2 if metric == "l2" else METRIC_INNER_PRODUCT, 0)
    ix.add(db)
    if fmt is not None:
        ix.set_operand_format(fmt)
    return ix


def range_search(ix, q, radius, **kw):
    lims, D, I = ix.range_search(q, radius, **kw)
    ix.sync()
    assert ix.last_stats()["err_word"] == 0
    return lims, D, I


def assert_same(got, ref, what):
    lims, D, I = got
    lr, Dr, Ir = (t.to(lims.device) for t in ref)
    assert torch.equal(lims, lr), f"{what}: lims differ at queries {(lims != lr).nonzero().flatten()[:8].tolist()}"
    bad = (D.view(torch.int32) != Dr.view(torch.int32)) | (I != Ir)
    if bool(bad.any()):
        e = int(bad.nonzero()[0])
        qi = int(torch.searchsorted(lims, torch.tensor(e, device=lims.device), right=True)) - 1
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} entries differ; first at {e} (query {qi}): "
                             f"got ({float(D[e])!r}, {int(I[e])}), want ({float(Dr[e])!r}, {int(Ir[e])})")


def radius_for(q, x, metric, hits):
    """an fp32 radius at which the median query gets about `hits` rows (float64 scores)"""
    q64, x64 = q.double(), x.double()
    if metric == "ip":
        s = q64 @ x64.t()
        return float(s.topk(hits, dim=1).values[:, -1].median().float())
    dist = (q64 * q64).sum(1)[:, None] + (x64 * x64).sum(1)[None, :] - 2 * q64 @ x64.t()
    return float(dist.topk(hits, dim=1, largest=False).values[:, -1].median().float())


def no_hit_radius(metric):
    return 1e30 if metric == "ip" else -1.0


def check(ix, q, x, radius, metric, what, **kw):
    got = range_search(ix, q, radius)
    assert_same(got, rx.range_search(q, x, radius, metric, **kw), what)
    return got


# ------------------------------------------------------------------ the matrix
@pytest.mark.parametrize("metric", ["ip", "l2"])
@pytest.mark.parametrize("fmt", ["bf16", "fp16"])
@pytest.mark.parametrize("d", [768, 200, 130])
def test_matches_oracle(metric, fmt, d):
    n, nq = 10037, 300  # not a multiple of 256; more than one query tile (the CTA-pair kernel)
    x, q = unit(n, d, 1), unit(nq, d, 2)
    ix = build(x, metric, fmt)
    for hits in (16, 1000):
        r = radius_for(q, x, metric, hits)
        lims, _, _ = check(ix, q, x, r, metric, f"{metric}/{fmt}/d={d}/~{hits} hits")
        per = (lims[1:] - lims[:-1]).double()
        assert hits / 4 <= float(per.median()) <= hits * 4
    lims, D, I = check(ix, q, x, no_hit_radius(metric), metric, f"{metric}/{fmt}/d={d}/no hits")
    assert int(lims[-1]) == 0 and D.numel() == 0 and I.numel() == 0


@pytest.mark.parametrize("metric", ["ip", "l2"])
def test_equals_the_search_prefix(metric):
    n, nq = 2000, 64
    x, q = unit(n, 96, 3), unit(nq, 96, 4)
    ix = build(x, metric)
    D, I = ix.search(q, n)
    ix.sync()
    r = radius_for(q, x, metric, 40)
    lims, Dr, Ir = range_search(ix, q, r)
    for i in range(nq):
        a, b = int(lims[i]), int(lims[i + 1])
        c = b - a
        assert torch.equal(Dr[a:b].view(torch.int32), D[i, :c].view(torch.int32)) and torch.equal(Ir[a:b], I[i, :c])
        if c < n:  # the next row of the search is not strictly beyond the radius
            assert not (float(D[i, c]) > r if metric == "ip" else float(D[i, c]) < r)


@pytest.mark.parametrize("metric", ["ip", "l2"])
def test_strict_boundary(metric):
    n = 5000
    x, q = unit(n, 768, 5), unit(8, 768, 6)
    ix = build(x, metric)
    D, I = ix.search(q, 64)
    ix.sync()
    for i in range(8):
        j = 20
        r = float(D[i, j])  # an exact D of row I[i, j]
        lims, Dr, Ir = range_search(ix, q[i:i + 1], r)
        got = Ir.tolist()
        assert int(I[i, j]) not in got
        assert int(I[i, j - 1]) in got
        assert got == I[i, :len(got)].tolist()
        assert len(got) == int(((D[i] > r) if metric == "ip" else (D[i] < r)).sum())


@pytest.mark.parametrize("metric", ["ip", "l2"])
def test_every_row_and_no_row(metric):
    n, nq = 3000, 200  # 600,000 candidates: more than the first candidate buffer holds
    x, q = unit(n, 64, 7), unit(nq, 64, 8)
    ix = build(x, metric)
    lims, D, I = check(ix, q, x, no_hit_radius(metric), metric, "no row")
    assert torch.equal(lims, torch.zeros(nq + 1, dtype=torch.int64, device=lims.device))
    gen = ix.generation
    lims, D, I = check(ix, q, x, -1e30 if metric == "ip" else 1e30, metric, "every row")
    assert torch.equal(lims, torch.arange(nq + 1, device=lims.device) * n)
    assert ix.generation != gen  # the candidate and result buffers grew
    gen = ix.generation
    assert_same(range_search(ix, q, -1e30 if metric == "ip" else 1e30), (lims, D, I), "every row, again")
    assert ix.generation == gen  # and are reused as they are


def test_no_queries():
    x = unit(1000, 64, 9)
    ix = build(x, "ip")
    lims, D, I = range_search(ix, torch.zeros(0, 64, device="cuda"), 0.1)
    assert lims.tolist() == [0] and D.numel() == 0 and I.numel() == 0
    lims, D, I = ix.range_search(np.zeros((0, 64), np.float32), 0.1)
    assert lims.tolist() == [0] and D.shape == (0,) and I.shape == (0,)


# ------------------------------------------------------------------ hard data
@pytest.mark.parametrize("metric", ["ip", "l2"])
def test_clustered(metric):
    g = torch.Generator().manual_seed(10)
    d = 768
    cent = torch.randn(1024, d, generator=g)
    cent = cent / cent.norm(dim=1, keepdim=True)
    x = cent[torch.randint(0, 1024, (20000,), generator=g)] + 0.05 * torch.randn(20000, d, generator=g) / d ** 0.5
    q = cent[torch.randint(0, 1024, (256,), generator=g)] + 0.05 * torch.randn(256, d, generator=g) / d ** 0.5
    x, q = x.cuda(), q.cuda()
    ix = build(x, metric)
    for hits in (16, 200):
        check(ix, q, x, radius_for(q, x, metric, hits), metric, f"clustered ~{hits}")


@pytest.mark.parametrize("metric", ["ip", "l2"])
def test_duplicates_tie_at_the_radius(metric):
    base = unit(600, 128, 11)
    x = base.repeat_interleave(32, dim=0)  # every row 32 times: groups of exact ties
    q = unit(100, 128, 12)
    ix = build(x, metric)
    D, _ = ix.search(q, 100)
    ix.sync()
    for col in (31, 32, 64):  # the last row of the first group, the first of the second, the third group
        r = float(D[0, col])
        lims, _, _ = check(ix, q, x, r, metric, f"duplicates, radius at column {col}")
        assert int(lims[1]) % 32 == 0  # a tie group is all in or all out


@pytest.mark.parametrize("metric", ["ip", "l2"])
def test_beyond_fp16(metric):
    x = unit(5000, 256, 13) * 1e6  # rows beyond fp16's range: the automatic choice is bf16
    q = unit(130, 256, 14)
    ix = build(x, metric)
    assert ix.operand_format == "bf16"
    check(ix, q, x, radius_for(q, x, metric, 16), metric, "bf16-range rows")

    x = unit(5000, 256, 15)
    q = unit(130, 256, 16)
    q[7] *= 1e7  # one query beyond fp16's range: its error bound is unbounded, every row a candidate
    ix = build(x, metric, "fp16")
    check(ix, q, x, radius_for(q[:7], x, metric, 16), metric, "a query beyond fp16")


# ------------------------------------------------------------------ passes and other paths
def test_passes():
    n, nq = 3000, Q_PASS_MAX + 300
    x, q = unit(n, 64, 17), unit(nq, 64, 18)
    ix = build(x, "ip")
    r = radius_for(q[:512], x, "ip", 16)
    lims, D, I = range_search(ix, q, r)
    assert int(lims[0]) == 0 and bool((lims[1:] >= lims[:-1]).all()) and int(lims[-1]) == D.numel() == I.numel()
    g = torch.Generator().manual_seed(19)
    pick = torch.cat([torch.arange(0, 40), torch.arange(Q_PASS_MAX - 40, Q_PASS_MAX + 40), torch.arange(nq - 40, nq),
                      torch.randint(0, nq, (200,), generator=g)]).unique()
    lr, Dr, Ir = rx.range_search(q[pick.cuda()], x, r, "ip")
    for j, i in enumerate(pick.tolist()):
        a, b = int(lims[i]), int(lims[i + 1])
        assert b - a == int(lr[j + 1] - lr[j]), f"query {i}"
        assert torch.equal(D[a:b].view(torch.int32), Dr[int(lr[j]):int(lr[j + 1])].view(torch.int32)), f"query {i}"
        assert torch.equal(I[a:b], Ir[int(lr[j]):int(lr[j + 1])]), f"query {i}"


def test_id_offset_and_force_ip():
    x, q = unit(4000, 96, 20), unit(150, 96, 21)
    ix = build(x, "l2")
    ix.set_id_offset(1000)
    check(ix, q, x, radius_for(q, x, "l2", 16), "l2", "id_offset", id_offset=1000)
    r = radius_for(q, x, "ip", 16)
    got = ix.range_search(q, r, flags=4)  # KEDS_SEARCH_FORCE_IP
    ix.sync()
    assert_same(got, rx.range_search(q, x, r, "ip", id_offset=1000), "force IP")


def test_numpy_and_tensor_calls_agree():
    x, q = unit(4000, 130, 22), unit(150, 130, 23)
    ix = build(x, "ip")
    r = radius_for(q, x, "ip", 16)
    lims, D, I = range_search(ix, q, r)
    ln, Dn, In = ix.range_search(q.cpu().numpy(), r)
    assert isinstance(ln, np.ndarray) and ln.dtype == np.int64 and Dn.dtype == np.float32 and In.dtype == np.int64
    assert np.array_equal(ln, lims.cpu().numpy()) and np.array_equal(In, I.cpu().numpy())
    assert np.array_equal(Dn.view(np.int32), D.cpu().numpy().view(np.int32))
    # a query tensor off a 16-byte boundary scores as the aligned one does
    qa = torch.empty(q.numel() + 1, device="cuda")[1:].view_as(q).copy_(q)
    assert_same(range_search(ix, qa, r), (lims, D, I), "misaligned query tensor")


def test_replicas_equal_one_index():
    x, q = unit(4000, 64, 24), unit(301, 64, 25)
    one = build(x, "ip")
    r = radius_for(q, x, "ip", 16)
    lims, D, I = one.range_search(q.cpu().numpy(), r)
    rep = IndexReplicas(64, METRIC_INNER_PRODUCT, [0, 0])
    rep.add(x.cpu().numpy())
    lr, Dr, Ir = rep.range_search(q.cpu().numpy(), r)
    assert np.array_equal(lims, lr) and np.array_equal(I, Ir) and np.array_equal(D.view(np.int32), Dr.view(np.int32))
    for s in rep.subs:
        s.sync()


# ------------------------------------------------------------------ the builder's near-duplicate filter
def test_drop_near_duplicates():
    g = torch.Generator().manual_seed(26)
    n, d = 5000, 768
    img = torch.randn(n, d, generator=g)
    txt = torch.randn(n, d, generator=g)
    names = [f"pair_{i:05d}.pt" for i in range(n)]
    src = torch.randperm(n, generator=g)[:40]
    pairs = [(int(a), int(b)) for a, b in zip(src[:20], src[20:])]
    later = []
    for a, b in pairs:  # row max(a, b) becomes a near-copy of row min(a, b)
        lo, hi = min(a, b), max(a, b)
        c = img[lo] / img[lo].norm() + 1e-3 * torch.randn(d, generator=g)
        img[hi] = c / c.norm() * 3.0  # any scale: the filter compares normalised rows
        later.append(hi)
    ki, kt, kn, dropped = drop_near_duplicates(img, txt, names, radius=0.99, device=0, batch=1024)
    assert sorted(dropped.tolist()) == sorted(later)
    keep = [i for i in range(n) if i not in set(later)]
    assert kn == [names[i] for i in keep]
    assert torch.equal(ki, img[keep]) and torch.equal(kt, txt[keep])
    again = drop_near_duplicates(img, txt, names, radius=0.99, device=0, batch=65536)
    assert torch.equal(again[3], dropped)
