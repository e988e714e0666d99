"""GPU: every exact answer of the library against the bit-exact fp32 reference (oracle/fp32_exact.py).

The library answers as an exact fp32 flat search would: scores of warp_exact_score, ordered by
score descending, then row id ascending. Here that is checked bit for bit -- D as int32 bits, I as
ids -- for every query, on each route a query can take (certified re-rank in all its variants, the
exact fallback's selection routes, exact-only searches, several passes), with lattice data whose
exact ties spread over thousands of distinct rows, and for the other entry points built on the same
scores: the fused two-database calls, the shard merge, gallery ranks and label hits. Each case also
checks, through last_stats, that it reached the route it is about."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from keds_b200 import _capi  # noqa: E402
from keds_b200 import metrics as km  # noqa: E402
from keds_b200 import retrieval as kr  # noqa: E402
from keds_b200.index import METRIC_INNER_PRODUCT, METRIC_L2, GpuIndexFlat, _stream_ptr, search2  # noqa: E402
from oracle import fp32_exact as fx  # noqa: E402

EXACT_LIST_CAP = 2048   # exact_fallback.cuh: rows the fallback's pre-filter holds in shared memory
# error-bound scales that queue every query for the exact fallback: lattice rows are exact in the
# 16-bit operand, so their bound is only the accumulation allowance and needs a far larger factor
EPS_ALL = 1e4
EPS_ALL_LATTICE = 1e9


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


def assert_bits(D, I, Dr, Ir, what):
    ok = fx.equal_bits(D, I, Dr, Ir)
    if not bool(ok.all()):
        b = int((~ok).nonzero()[0])
        cols = ((D[b].view(torch.int32) != Dr[b].to(D.device).view(torch.int32)) | (I[b] != Ir[b].to(I.device)))
        c = cols.nonzero().flatten()[:6].tolist()
        raise AssertionError(f"{what}: {int((~ok).sum())} of {ok.numel()} queries differ; query {b} columns {c}: "
                             f"got I {I[b, c].tolist()} D {D[b, c].tolist()}, want I {Ir[b, c].tolist()} "
                             f"D {Dr[b, c].tolist()}")


def search(ix, q, k, exclude=None):
    D, I = ix.search(q, k, exclude=exclude)
    ix.sync()
    st = ix.last_stats()
    assert st["err_word"] == 0, st
    return D, I, st


def certified(st, nq, most=True):
    """the tensor-core pass + re-rank answered (most of) the queries"""
    assert st["exact_only"] == 0, st
    assert st["n_flagged"][0] <= (nq // 10 if most else nq - 1), st


def fallback_route(n, k, n_excluded=0):
    """(pre-filter possible, chunks): the exact fallback's choice of selection route for one
    query (exact_fallback.cuh, exact_select; chunk layout from launch_exact in api.cu). With the
    pre-filter possible, it is taken when the rows at or above the k-th best chunk maximum fit
    EXACT_LIST_CAP; otherwise the dense radix route runs."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    groups = -(-n // 32)
    cg = max(8, -(-groups // (8 * sms)))
    chunks = -(-groups // cg)
    keff = min(k, n - n_excluded)
    return chunks >= keff and 2 * keff <= EXACT_LIST_CAP, chunks, cg


def prefilter_list(scores, k, chunks, cg):
    """rows the pre-filter lists per query: those at or above the k-th best chunk maximum"""
    n = scores.shape[1]
    pad = chunks * cg * 32 - n
    s = torch.nn.functional.pad(scores, (0, pad), value=-float("inf"))
    cmax = s.view(scores.shape[0], chunks, -1).amax(2)
    t0 = cmax.topk(k, dim=1).values[:, -1:]
    return (scores >= t0).sum(1)


def rank_scores(q, x, metric):
    q64, x64 = q.double(), x.double()
    s = q64 @ x64.t()
    return s if metric == "ip" else 2 * s - (x64 * x64).sum(1)[None, :]


# ------------------------------------------------------------------ lattice data: exact ties
def lattice(nq, ties, n_rand, seed, better=2):
    """d = 64, entries in {-2..2}/8: every fp32 (and 16-bit operand) sum is exact, whatever the
    order. Query j is a +-1/8, +-2/8 pattern on coordinates 0..15, zero elsewhere; `ties` distinct
    rows share its head and carry six +-1/8 on coordinates 16..63 at random places, so they tie
    exactly under both metrics; `better` rows double its first coordinate and beat them; the rest
    are random lattice rows, far behind. Rows are shuffled. Returns (rows, queries, tied ids [nq, ties])."""
    g = torch.Generator().manual_seed(seed)
    d = 64
    head = (torch.randint(0, 2, (nq, 16), generator=g) * 2 - 1).float() * 2 / 8
    head[:, 0] /= 2
    Q = torch.zeros(nq, d)
    Q[:, :16] = head
    rows, owner = [], []
    for j in range(nq):
        t = torch.zeros(ties, d)
        t[:, :16] = head[j]
        pos = torch.rand(ties, 48, generator=g).argsort(1)[:, :6] + 16
        t.scatter_(1, pos, (torch.randint(0, 2, (ties, 6), generator=g) * 2 - 1).float() / 8)
        b = torch.zeros(better, d)
        b[:, :16] = head[j]
        b[:, 0] *= 2
        rows += [t, b]
        owner += [torch.full((ties,), j), torch.full((better,), -1)]
    rows.append(torch.randint(-2, 3, (n_rand, d), generator=g).float() / 8)
    owner.append(torch.full((n_rand,), -1))
    X, own = torch.cat(rows), torch.cat(owner)
    perm = torch.randperm(X.shape[0], generator=g)
    X, own = X[perm], own[perm]
    tied = torch.stack([(own == j).nonzero().flatten() for j in range(nq)])
    return X.cuda(), Q.cuda(), tied.cuda()


# ------------------------------------------------------------------ search: shapes, formats, metrics
@pytest.mark.parametrize("n,nq,d,k", [(70000, 130, 768, 16), (5000, 300, 200, 64), (3000, 129, 50, 16),
                                      (257, 7, 768, 1)])
@pytest.mark.parametrize("metric", ["ip", "l2"])
@pytest.mark.parametrize("fmt", ["fp16", "bf16"])
def test_search_equals_the_fp32_reference(n, nq, d, k, metric, fmt):
    """d/4 = 50 is no multiple of 32 * 6 (the multi-row scorer's block); d = 50 takes the element
    order; n = 257 is one row past a tile. Some queries are copies of rows (L2 distance +0)."""
    x, q = unit(n, d, n + d), unit(nq, d, n + d + 1)
    q[:3] = x[:3]
    ix = build(x, metric, fmt)
    D, I, st = search(ix, q, k)
    certified(st, nq)
    Dr, Ir = fx.topk(q, x, k, metric)
    assert_bits(D, I, Dr, Ir, f"{fmt} {metric}")
    ix.set_eps_scale(EPS_ALL)                   # every query through the exact fallback
    D, I, st = search(ix, q, k)
    assert st["n_flagged"][0] == nq and st["exact_only"] == 0, st
    assert_bits(D, I, Dr, Ir, f"{fmt} {metric} fallback")


_LARGE = {}


def _large_case():
    if not _LARGE:
        x, q = unit(20000, 768, 31), unit(1408, 768, 32)
        _LARGE.update(x=x, q=q, ref64=fx.topk(q, x, 64, "ip"), ref200=fx.topk(q[:1000], x, 200, "ip"))
    return _LARGE


@pytest.mark.parametrize("env", [{}, {"KEDS_NO_PAIR": "1"}, {"KEDS_RERANK_VARIANT": "latency"},
                                 {"KEDS_RERANK_VARIANT": "throughput"}, {"KEDS_RERANK_THREADS": "32"},
                                 {"KEDS_RERANK_THREADS": "64"}, {"KEDS_RERANK_THREADS": "128"},
                                 {"KEDS_RERANK_THREADS": "256"}], ids=lambda e: ",".join(f"{a}={b}" for a, b in e.items()) or "default")
def test_large_batch_rerank_variants(env, monkeypatch):
    """1408 queries at k = 64 and 1000 at k = 200: the throughput re-rank (128-thread two-row
    variant at k >= 128, the one-row variant at every block size), the latency variant, and CTA
    pairs switched off."""
    for key, val in env.items():
        monkeypatch.setenv(key, val)
    c = _large_case()
    ix = build(c["x"], "ip")                    # the switches are read when the index first searches
    D, I, st = search(ix, c["q"], 64)
    certified(st, 1408)
    assert_bits(D, I, *c["ref64"], f"{env} k=64")
    D, I, st = search(ix, c["q"][:1000], 200)
    certified(st, 1000)
    assert_bits(D, I, *c["ref200"], f"{env} k=200")


@pytest.mark.parametrize("n,k,metric,prefilter", [(200000, 600, "ip", True), (200000, 600, "l2", True),
                                                  (60000, 1024, "ip", False), (60000, 2048, "l2", False)])
def test_exact_only_searches_and_their_selection_routes(n, k, metric, prefilter):
    """k > 512 goes to the exact kernels alone. At 200k rows the chunk maxima outnumber k = 600 and
    the pre-filter's list fits; at 60k rows k = 1024 outnumbers the chunks and k = 2048 is above the
    pre-filter's limit: the dense radix route."""
    x, q = unit(n, 768, n + k), unit(24, 768, n + k + 1)
    possible, chunks, cg = fallback_route(n, k)
    if prefilter:
        assert possible
        L = prefilter_list(rank_scores(q, x, metric), k, chunks, cg)
        assert (L <= EXACT_LIST_CAP * 0.9).all(), L    # away from the cap: fp32 rounding cannot cross it
    else:
        assert not possible
    ix = build(x, metric)
    D, I, st = search(ix, q, k)
    assert st["exact_only"] == 1, st
    assert_bits(D, I, *fx.topk(q, x, k, metric), f"n={n} k={k} {metric}")


def test_several_passes():
    """16,684 queries at d = 64: more than one pass (16,384 queries) of scratch."""
    x, q = unit(6000, 64, 41), unit(16684, 64, 42)
    ix = build(x, "l2")
    D, I, st = search(ix, q, 16)
    certified(st, 16684)
    assert_bits(D, I, *fx.topk(q, x, 16, "l2"), "two passes")


# ------------------------------------------------------------------ exact ties
@pytest.mark.parametrize("metric", ["ip", "l2"])
def test_lattice_ties_on_every_route(metric):
    """Thousands of distinct rows tie exactly at the k-th score: the lowest ids must win, on the
    certified path, in the fallback's pre-filter, in its dense id-ordered tie loop (5,000 tied rows
    at k = 5, more than EXACT_LIST_CAP rows qualify) and with eight excluded labels per query."""
    # 40 tied rows per query, k = 16: two better rows, then 14 of 40 ties
    x, q, tied = lattice(32, 40, 60000, 51)
    ix = build(x, metric)
    Dr, Ir = fx.topk(q, x, 16, metric)
    assert (Ir[:, 2:] == tied.sort(1).values[:, :14]).all()        # the reference's own tie rule
    D, I, st = search(ix, q, 16)
    certified(st, 32, most=False)
    assert_bits(D, I, Dr, Ir, "certified ties")
    n = x.shape[0]
    possible, chunks, cg = fallback_route(n, 16)
    assert possible and (prefilter_list(rank_scores(q, x, metric), 16, chunks, cg) <= EXACT_LIST_CAP).all()
    ix.set_eps_scale(EPS_ALL_LATTICE)
    D, I, st = search(ix, q, 16)
    assert st["n_flagged"][0] == 32, st
    assert_bits(D, I, Dr, Ir, "pre-filter ties")
    # exclusion: both better rows, the three lowest tied ids (one of them twice), a row id outside
    # the database and -1
    ts = tied.sort(1).values
    best = Ir[:, :2]
    ex = torch.stack([best[:, 0], best[:, 1], ts[:, 0], ts[:, 1], ts[:, 1], ts[:, 2],
                      torch.full_like(ts[:, 0], n + 5), torch.full_like(ts[:, 0], -1)], 1)
    Dre, Ire = fx.topk(q, x, 16, metric, exclude=ex)
    assert (Ire == ts[:, 3:19]).all()
    for eps in (1.0, EPS_ALL_LATTICE):
        ix.set_eps_scale(eps)
        D, I, st = search(ix, q, 16, exclude=ex)
        assert_bits(D, I, Dre, Ire, f"excluded ties eps={eps}")
    # 5,000 tied rows per query at k = 5: the dense route's id-ordered tie loop
    x, q, tied = lattice(8, 5000, 20000, 52)
    n = x.shape[0]
    possible, chunks, cg = fallback_route(n, 5)
    assert possible and (prefilter_list(rank_scores(q, x, metric), 5, chunks, cg) > EXACT_LIST_CAP).all()
    ix = build(x, metric)
    ix.set_eps_scale(EPS_ALL_LATTICE)
    Dr, Ir = fx.topk(q, x, 5, metric)
    assert (Ir[:, 2:] == tied.sort(1).values[:, :3]).all()
    D, I, st = search(ix, q, 5)
    assert st["n_flagged"][0] == 8, st
    assert_bits(D, I, Dr, Ir, "dense tie loop")
    ts = tied.sort(1).values
    ex = torch.cat([Ir[:, :2], ts[:, :6]], 1)
    Dre, Ire = fx.topk(q, x, 5, metric, exclude=ex)
    assert (Ire == ts[:, 6:11]).all()
    D, I, st = search(ix, q, 5, exclude=ex)
    assert_bits(D, I, Dre, Ire, "dense tie loop, excluded")


# ------------------------------------------------------------------ other entry points
@pytest.mark.parametrize("metric", ["ip", "l2"])
def test_search2_retrieve2_and_host_mirrors(metric):
    a, b, q = unit(9000, 768, 61), unit(9000, 768, 62), unit(70, 768, 63)
    q[:2] = a[:2]
    ia, ib = build(a, metric), build(b, metric)
    ra, rb = fx.topk(q, a, 16, metric), fx.topk(q, b, 16, metric)
    perm = torch.randperm(16, generator=torch.Generator().manual_seed(5))
    for eps in (1.0, EPS_ALL):
        ia.set_eps_scale(eps)
        (Da, Ia), (Db, Ib) = search2(ia, ib, q, 16)
        ia.sync()
        st = ia.last_stats()
        assert st["n_flagged"] == ([0, 0] if eps == 1.0 else [70, 70]), st
        assert_bits(Da, Ia, *ra, f"search2 a eps={eps}")
        assert_bits(Db, Ib, *rb, f"search2 b eps={eps}")
        o = kr.retrieve2(ia, ib, q, 16, perm_img=perm, want_feats=True, pool_mode=kr.POOL_MEAN)
        ia.sync()
        assert_bits(o["D_img"], o["I_img"], *ra, f"retrieve2 img eps={eps}")
        assert_bits(o["D_txt"], o["I_txt"], *rb, f"retrieve2 txt eps={eps}")
        ho = {"D_img": torch.zeros((70, 16)).pin_memory(), "I_img": torch.zeros((70, 16), dtype=torch.int64).pin_memory(),
              "D_txt": torch.zeros((70, 16)).pin_memory(), "I_txt": torch.zeros((70, 16), dtype=torch.int64).pin_memory()}
        kr.retrieve2(ia, ib, q.cpu().pin_memory(), 16, perm_img=perm, want_feats=True, pool_mode=kr.POOL_MEAN,
                     host_out=ho)
        ia.sync()
        assert ia.last_stats()["n_flagged"] == st["n_flagged"]
        assert_bits(ho["D_img"], ho["I_img"], *ra, f"host mirror img eps={eps}")
        assert_bits(ho["D_txt"], ho["I_txt"], *rb, f"host mirror txt eps={eps}")
    ia.set_eps_scale(1.0)


@pytest.mark.parametrize("metric", ["ip", "l2"])
@pytest.mark.parametrize("parts", [2, 3, 8])
def test_topk_merge_of_row_shards(metric, parts):
    """keds_topk_merge over shard results (each the reference's search of its rows, labels offset by
    the shard's first row): lattice ties across shards, shards with fewer rows than k."""
    x, q, _ = lattice(16, 30, 3000, 70 + parts)
    n, k = x.shape[0], 40
    cuts = [0] + sorted(torch.randperm(n - 1, generator=torch.Generator().manual_seed(parts))[:parts - 1].add(1).tolist()) + [n]
    cuts[1] = min(cuts[1], 25)                  # the first shard has fewer rows than k
    Ds, Is = [], []
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        D, I = fx.topk(q, x[lo:hi], k, metric, id_offset=lo)
        Ds.append(D)
        Is.append(I)
    Dp, Ip = torch.stack(Ds).contiguous(), torch.stack(Is).contiguous()
    D = torch.empty((16, k), dtype=torch.float32, device="cuda")
    I = torch.empty((16, k), dtype=torch.int64, device="cuda")
    lib = _capi.load()
    _capi.check(lib.keds_topk_merge(Dp.data_ptr(), Ip.data_ptr(), parts, 16, k,
                                    METRIC_L2 if metric == "l2" else METRIC_INNER_PRODUCT, D.data_ptr(), I.data_ptr(),
                                    _stream_ptr(0)))
    torch.cuda.synchronize()
    Dr, Ir = fx.merge(Ds, Is, k, metric)
    assert_bits(Dr, Ir, *fx.topk(q, x, k, metric), "reference merge vs whole search")
    assert_bits(D, I, Dr, Ir, f"merge of {parts}")


# ------------------------------------------------------------------ gallery rank
def _ranks(q, gal, tgt, ex=None):
    r = km.gallery_rank(q, gal, tgt, ex)
    torch.cuda.synchronize()
    return r


@pytest.mark.parametrize("ng,nq,d", [(50000, 1000, 768), (700, 100, 768), (250, 90, 768), (6000, 300, 50)])
def test_gallery_rank_equals_the_fp32_reference(ng, nq, d):
    """Tensor-core ranking (50k x 1000, the CIRR scale; 700 rows), the SIMT kernel (250 rows: one
    tile), the element order (d = 50); targets with copies at lower and higher ids; exclusion mixed
    with -1; an inflated bound sends every query to the exact recount; and a query tensor that
    starts 4 bytes past a 16-byte boundary ranks like its aligned copy."""
    gal = unit(ng, d, ng + d)
    g = torch.Generator().manual_seed(ng)
    tgt = torch.randint(0, ng, (nq,), generator=g).cuda()
    gal[5] = gal[ng // 2]                       # a copy below the target ...
    gal[ng - 3] = gal[ng // 2]                  # ... and one above it
    tgt[:4] = ng // 2
    q = unit(nq, d, ng + d + 1)
    q[4:8] = gal[tgt[4:8]] + 0.01 * q[4:8]      # top-ranked targets
    ex = torch.randint(-1, ng, (nq,), generator=g).cuda()
    ex[::3] = -1
    ex[0] = 5
    try:
        want = fx.target_rank(q, gal, tgt, ex)
        want_noex = fx.target_rank(q, gal, tgt)
        got = _ranks(q, gal, tgt, ex)
        assert torch.equal(got, want), (got != want).nonzero()[:5].flatten().tolist()
        assert torch.equal(_ranks(q, gal, tgt), want_noex)
        ix = km.gallery_index(gal)
        ix.set_eps_scale(200.0)
        assert torch.equal(_ranks(q, gal, tgt, ex), want)
        ix.set_eps_scale(1.0)
        flat = torch.empty(nq * d + 1, device="cuda")
        qm = flat[1:].view(nq, d)
        qm.copy_(q)
        assert qm.data_ptr() % 16 == 4
        assert torch.equal(_ranks(qm, gal, tgt, ex), want)
        assert torch.equal(_ranks(qm.clone(), gal, tgt, ex), want)
    finally:
        km.clear_gallery_cache()


# ------------------------------------------------------------------ label hits
@pytest.mark.parametrize("metric", ["ip", "l2"])
def test_label_hits_equal_the_fp32_reference(metric):
    """Cut points [1, 5, 10, 50, 100, 200] and eight up to 2048 on random rows; lattice ties
    straddling the cuts; every query through the fallback."""
    g = torch.Generator().manual_seed(81)
    x, q = unit(30000, 768, 82), unit(200, 768, 83)
    lab = torch.randint(0, 6, (30000,), generator=g).cuda()
    qlab = torch.randint(0, 6, (200,), generator=g).cuda()
    ix = build(x, metric)
    _, Ir = fx.topk(q, x, 2048, metric)
    for ks in ([1, 5, 10, 50, 100, 200], [1, 3, 16, 64, 200, 600, 1024, 2048]):
        want = fx.label_hits(Ir, lab, qlab, ks)
        for eps in (1.0, EPS_ALL):
            ix.set_eps_scale(eps)
            hits = km.index_label_hits(ix, q, lab, qlab, ks)
            ix.sync()
            st = ix.last_stats()
            assert st["err_word"] == 0, st
            if ks[-1] <= 512:
                assert st["exact_only"] == 0 and (st["n_flagged"][0] == 200 if eps > 1 else st["n_flagged"][0] <= 20), st
            else:
                assert st["exact_only"] == 1, st
            assert torch.equal(hits, want), (ks, eps, (hits != want).any(1).nonzero()[:5].flatten().tolist())
    ix.set_eps_scale(1.0)
    # lattice: 40 tied rows per query, cuts inside the tie (the two better rows come first)
    x, q, tied = lattice(32, 40, 60000, 84)
    lab = torch.randint(0, 3, (x.shape[0],), generator=g).cuda()
    qlab = torch.randint(0, 3, (32,), generator=g).cuda()
    ix = build(x, metric)
    ks = [1, 2, 3, 7, 16, 41, 42, 43]
    _, Ir = fx.topk(q, x, 43, metric)
    want = fx.label_hits(Ir, lab, qlab, ks)
    for eps in (1.0, EPS_ALL_LATTICE):
        ix.set_eps_scale(eps)
        hits = km.index_label_hits(ix, q, lab, qlab, ks)
        ix.sync()
        assert ix.last_stats()["err_word"] == 0
        if eps > 1:
            assert ix.last_stats()["n_flagged"][0] == 32
        assert torch.equal(hits, want), (eps, (hits != want).any(1).nonzero()[:5].flatten().tolist())
