"""GPU: the retrieval step's gathered neighbours and pools against oracle/pool_exact.py.

Gathers are compared bit for bit with the rows the returned I names (perm applied). Mean pools are
compared bit for bit with the emulation of the summation order of the route each query took; softmax
pools (whose __expf has no bit-exact emulation) must sit within the rigorous bound of the float64 pool
of the returned D. Each case reads the route from last_stats as tests/test_gpu_fp32_exact.py does:
no query flagged -> the re-rank's order, every query flagged or an exact-only call -> the fallback's;
a mixed call must give each query one of the two orders, and no more queries than were flagged may
match the fallback's alone.

Routes (warps, neighbours in flight per warp): the latency re-rank (8, 2) at <= 148 queries of a
two-database call, the 128-thread throughput re-rank (4, 2) at k >= 128, the one-row throughput
re-rank (T/32, 1) at KEDS_RERANK_THREADS = T, the exact fallback and exact-only calls (8, 1), the
element path (one chain over the slots) at d % 4 != 0 or a feat / pool output not 16-byte aligned."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from keds_b200 import _capi  # noqa: E402
from keds_b200 import retrieval as kr  # noqa: E402
from keds_b200.index import METRIC_INNER_PRODUCT, METRIC_L2, GpuIndexFlat  # noqa: E402
from oracle import pool_exact as pe  # noqa: E402

N = 20000
EPS_ALL = 1e4          # error-bound scale that queues every query for the exact fallback
LAT = ("latency", pe.LATENCY)
FB = ("fallback", pe.FALLBACK)


def unit(n, d, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, d, generator=g, dtype=torch.float64)
    return (x / x.norm(dim=1, keepdim=True)).float().cuda()


_ROWS = {}


def rows(d):
    if d not in _ROWS:
        _ROWS[d] = (unit(N, d, 1000 + d), unit(N, d, 2000 + d))
    return _ROWS[d]


def build(x, metric):
    ix = GpuIndexFlat(x.shape[1], METRIC_L2 if metric == "l2" else METRIC_INNER_PRODUCT, 0)
    if x.shape[0]:
        ix.add(x)
    return ix


def perms(k, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randperm(k, generator=g), torch.randperm(k, generator=g)


def throughput_route(k, threads=128):
    o = pe.THROUGHPUT_K128 if (k >= 128 and threads == 128) else pe.throughput(threads)
    return (f"throughput-T{threads}", o)


def call(ia, ib, q, k, mode, tau=50.0, pi=None, pt=None, feats=True, **kw):
    o = kr.retrieve2(ia, ib, q, k, perm_img=pi, perm_txt=pt, want_feats=feats, pool_mode=mode, tau=tau, **kw)
    ia.sync()
    st = ia.last_stats()
    assert st["err_word"] == 0, st
    return o, st


def check(o, st, xs, k, metric, mode, tau, perm, route, what, expect, vec=(True, True), fb=FB):
    """Gathers bit for bit, the pools against the orders of `route` (certified queries) and `fb`
    (flagged ones). expect: 'certified' (at least one query certified, per stream), 'fallback'
    (every query flagged) or 'exact-only'."""
    nq = o["I_img"].shape[0]
    if expect == "exact-only":
        assert st["exact_only"] == 1, (what, st)
    else:
        assert st["exact_only"] == 0, (what, st)
    for s, name in enumerate(("img", "txt")):
        x, I, D, p = xs[s], o["I_" + name], o["D_" + name], perm[s]
        nf = nq if st["exact_only"] else st["n_flagged"][s]
        if expect == "certified":
            assert nf < nq, (what, name, st)
        if expect == "fallback":
            assert nf == nq, (what, name, st)
        tag = f"{what} {name}: {route[0]} {route[1] if vec[s] else 'scalar'} / {fb[0]}, {nf} of {nq} flagged"
        if "feat_" + name in o:
            assert bool(pe.equal_rows(o["feat_" + name], pe.gather(x, I, p)).all()), f"feats {tag}"
        got = o["pool_" + name]
        if mode == 1:
            none = torch.zeros(nq, dtype=torch.bool, device=got.device)
            mc = pe.equal_rows(got, pe.mean_pool(x, I, p, *route[1], vec[s])) if nf < nq else none
            mf = pe.equal_rows(got, pe.mean_pool(x, I, p, *fb[1], vec[s])) if nf > 0 else none
            bad = ~(mc | mf)
            assert not bool(bad.any()), f"mean pool {tag}: {int(bad.sum())} queries match neither order, first {bad.nonzero()[:5].flatten().tolist()}"
            only_fb = int((mf & ~mc).sum())
            assert only_fb <= nf, f"mean pool {tag}: {only_fb} queries in the fallback's order"
        else:
            ref, bound = pe.softmax_pool_bound(x, I, D, p, tau, metric == "l2", 8)
            over = (got.double() - ref).abs() - bound
            assert not bool((over > 0).any()), f"softmax pool tau={tau} {tag}: {int((over > 0).sum())} entries outside the bound, worst {over.max().item():.3g}"


def run_route(ia, ib, xs, q, k, metric, route, what, expect, flags=0, exclude=None, vec=(True, True)):
    pi, pt = perms(k, k + q.shape[0])
    kw = dict(flags=flags, exclude=exclude)
    o, st = call(ia, ib, q, k, 1, pi=pi, pt=pt, **kw)
    check(o, st, xs, k, metric, 1, None, (pi, pt), route, what, expect, vec)
    for tau in (50.0, 0.5):
        o, st = call(ia, ib, q, k, 2, tau, pi=pi, feats=False, **kw)
        check(o, st, xs, k, metric, 2, tau, (pi, None), route, what, expect, vec)


# ------------------------------------------------------------------ every route, every shape
@pytest.mark.parametrize("metric", ["ip", "l2"])
@pytest.mark.parametrize("k", [1, 16, 64, 128, 200])
@pytest.mark.parametrize("d", [768, 1024, 200, 50, 4])
def test_pools_on_every_route(d, k, metric):
    """latency re-rank (100 queries), throughput re-rank at its default block (300 queries), the
    exact fallback (inflated bound) and exact-only calls; d = 1024 is two float4 passes per column,
    d = 50 the element path, d = 4 one float4 per row."""
    xs = rows(d)
    vec = (d % 4 == 0,) * 2
    ia, ib = build(xs[0], metric), build(xs[1], metric)
    q = unit(300, d, 3000 + d + k)
    run_route(ia, ib, xs, q[:100], k, metric, LAT, f"d={d} k={k} {metric}", "certified", vec=vec)
    run_route(ia, ib, xs, q, k, metric, throughput_route(k), f"d={d} k={k} {metric}", "certified", vec=vec)
    run_route(ia, ib, xs, q[:60], k, metric, FB, f"d={d} k={k} {metric}", "exact-only",
              flags=_capi.SEARCH_EXACT_ONLY, vec=vec)
    ia.set_eps_scale(EPS_ALL)
    run_route(ia, ib, xs, q[:100], k, metric, FB, f"d={d} k={k} {metric}", "fallback", vec=vec)


@pytest.mark.parametrize("env,nq", [
    ({"KEDS_RERANK_VARIANT": "latency"}, 300), ({"KEDS_RERANK_VARIANT": "throughput"}, 100),
    ({"KEDS_RERANK_THREADS": "32"}, 300), ({"KEDS_RERANK_THREADS": "64"}, 300),
    ({"KEDS_RERANK_THREADS": "128"}, 300), ({"KEDS_RERANK_THREADS": "256"}, 300)],
    ids=lambda v: ",".join(f"{a}={b}" for a, b in v.items()) if isinstance(v, dict) else f"nq={v}")
@pytest.mark.parametrize("k", [16, 200])
def test_rerank_variants(env, nq, k, monkeypatch):
    """The switches are read when an index first searches: a new pair per variant. At 32 threads
    the one-row re-rank sums like the element path, at 256 like the fallback."""
    for key, val in env.items():
        monkeypatch.setenv(key, val)
    xs = rows(768)
    ia, ib = build(xs[0], "ip"), build(xs[1], "ip")
    if env.get("KEDS_RERANK_VARIANT") == "latency":
        route = LAT
    else:
        route = throughput_route(k, int(env.get("KEDS_RERANK_THREADS", 128)))
    run_route(ia, ib, xs, unit(nq, 768, 4000 + k), k, "ip", route, f"{env} k={k}", "certified")


def test_d2048_matches_or_is_refused():
    """d = 2048: three float4 passes per column and 64 KB of per-warp partial pools. Either the
    pools match or the call is refused before launch with an argument error."""
    xs = (unit(6000, 2048, 5), unit(6000, 2048, 6))
    ia, ib = build(xs[0], "ip"), build(xs[1], "ip")
    q = unit(100, 2048, 7)
    try:
        run_route(ia, ib, xs, q, 16, "ip", LAT, "d=2048", "certified")
        outcome = "matches"
    except RuntimeError as e:
        assert "error -1:" in str(e), e          # KEDS_ERR_ARG
        outcome = f"refused: {e}"
    print(f"d=2048: {outcome}")


# ------------------------------------------------------------------ layouts
def test_misaligned_outputs_take_the_element_path():
    """feat_img and pool_img passed through out= as contiguous views 4 bytes past a 16-byte boundary:
    the image stream pools in the element order, into the given tensors; the text stream (aligned
    outputs) in the latency order."""
    d, k, nq = 768, 16, 100
    xs = rows(d)
    for metric in ("ip", "l2"):
        ia, ib = build(xs[0], metric), build(xs[1], metric)
        q = unit(nq, d, 11)
        pi, pt = perms(k, 12)
        ff = torch.empty(nq * k * d + 1, device="cuda")
        fp = torch.empty(nq * d + 1, device="cuda")
        out = {"feat_img": ff[1:].view(nq, k, d), "pool_img": fp[1:].view(nq, d)}
        assert out["feat_img"].data_ptr() % 16 == 4 and out["pool_img"].data_ptr() % 16 == 4
        for mode, tau in ((1, None), (2, 50.0), (2, 0.5)):
            o, st = call(ia, ib, q, k, mode, tau or 1.0, pi=pi, pt=pt, out=out)
            assert o["feat_img"].data_ptr() == ff.data_ptr() + 4 and o["pool_img"].data_ptr() == fp.data_ptr() + 4
            check(o, st, xs, k, metric, mode, tau, (pi, pt), LAT, f"misaligned {metric}", "certified", vec=(False, True))


def test_non_contiguous_out_is_replaced():
    """A column slice of a wider buffer passed as feat / pool: the call writes new tensors and leaves
    the wider buffers alone (the kernels write dense rows at data_ptr)."""
    d, k, nq = 768, 16, 100
    xs = rows(d)
    ia, ib = build(xs[0], "ip"), build(xs[1], "ip")
    q = unit(nq, d, 13)
    wide_p = torch.full((nq, 2 * d), 7.0, device="cuda")
    wide_f = torch.full((nq, k, 2 * d), 7.0, device="cuda")
    out = {"pool_txt": wide_p[:, d:], "feat_txt": wide_f[:, :, :d]}
    o, st = call(ia, ib, q, k, 1, out=out)
    assert (wide_p == 7.0).all() and (wide_f == 7.0).all()
    assert o is out and o["pool_txt"].is_contiguous() and o["feat_txt"].is_contiguous()
    check(o, st, xs, k, "ip", 1, None, (None, None), LAT, "replaced out", "certified")


def test_perm_that_is_no_permutation_is_refused():
    """A repeated or out-of-range perm entry would count one neighbour twice in the pool and drop
    another: a host perm is checked. A device perm is the caller's promise (checking it would
    synchronise): the pool then follows the slots, as the emulation says."""
    d, k = 768, 16
    xs = rows(d)
    ia, ib = build(xs[0], "ip"), build(xs[1], "ip")
    q = unit(100, d, 51)
    for bad in ([0, 0] + list(range(2, k)), list(range(k - 1)) + [k]):
        p = torch.tensor(bad)
        with pytest.raises(ValueError, match="perm_img"):
            kr.retrieve2(ia, ib, q, k, perm_img=p, pool_mode=1)
        with pytest.raises(ValueError, match="perm_txt"):
            kr.retrieve2(ia, ib, q, k, perm_txt=p, pool_mode=1)
        with pytest.raises(ValueError, match="perm_img"):
            kr.RetrievalStep(ia, ib, 100, k, perm_img=p, pool_mode=1)
    p = torch.tensor([0, 0] + list(range(2, k))).cuda()
    o, st = call(ia, ib, q, k, 1, pi=p)
    check(o, st, xs, k, "ip", 1, None, (p, None), LAT, "device perm with a repeated entry", "certified")
    for order in (pe.LATENCY, pe.FALLBACK):
        assert not bool(pe.equal_rows(o["pool_img"], pe.mean_pool(xs[0], o["I_img"], None, *order)).any())


def test_two_passes():
    """16,384 + 300 queries: the second pass's feats and pools start at its first query's rows."""
    d, k = 768, 16
    xs = rows(d)
    ia, ib = build(xs[0], "ip"), build(xs[1], "ip")
    run_route(ia, ib, xs, unit(16384 + 300, d, 15), k, "ip", throughput_route(k), "two passes", "certified")


def test_padding():
    """k > ntotal (10 rows, k = 16), and eight excluded labels on 12 rows at k = 8: -1 slots are zero
    rows; mean pools still divide by k, softmax pools give them weight 0."""
    for metric in ("ip", "l2"):
        xs = (unit(10, 64, 21), unit(10, 64, 22))
        ia, ib = build(xs[0], metric), build(xs[1], metric)
        q = unit(40, 64, 23)
        o, st = call(ia, ib, q, 16, 1)
        assert (o["I_img"][:, 10:] == -1).all() and (o["feat_img"][:, 10:] == 0).all()
        run_route(ia, ib, xs, q, 16, metric, LAT, f"k > ntotal {metric}", "exact-only" if st["exact_only"] else "certified")
        xs = (unit(12, 64, 24), unit(12, 64, 25))
        ia, ib = build(xs[0], metric), build(xs[1], metric)
        g = torch.Generator().manual_seed(26)
        ex = torch.stack([torch.randperm(12, generator=g)[:8] for _ in range(40)]).cuda()
        o, st = call(ia, ib, q, 8, 1, exclude=ex)
        assert (o["I_img"][:, 4:] == -1).all() and (o["I_txt"][:, :4] >= 0).all()
        run_route(ia, ib, xs, q, 8, metric, LAT, f"excluded E=8 {metric}", "exact-only" if st["exact_only"] else "certified",
                  exclude=ex)


def test_host_io_and_graph_replays():
    """Pinned host queries and results (keds_retrieve2's host mirrors), and RetrievalStep replays in both
    copy-node layouts: pools and feats equal to the stream path and to the emulation."""
    d, k, nq = 768, 16, 128
    xs = rows(d)
    ia, ib = build(xs[0], "l2"), build(xs[1], "l2")
    pi, _ = perms(k, 31)
    for mode in (1, 2):
        q = unit(nq, d, 32 + mode)
        o, st = call(ia, ib, q, k, mode, 50.0, pi=pi)
        check(o, st, xs, k, "l2", mode, 50.0, (pi, None), LAT, f"stream mode {mode}", "certified")
        ho = {"D_img": torch.zeros((nq, k)).pin_memory(), "I_img": torch.zeros((nq, k), dtype=torch.int64).pin_memory()}
        oh = kr.retrieve2(ia, ib, q.cpu().pin_memory(), k, perm_img=pi, want_feats=True, pool_mode=mode, tau=50.0,
                          host_out=ho)
        ia.sync()
        assert torch.equal(ho["I_img"], o["I_img"].cpu())
        for key in ("feat_img", "feat_txt", "pool_img", "pool_txt"):
            assert bool(pe.equal_rows(oh[key], o[key]).all()), ("host I/O", mode, key)
        for copy_nodes in (False, True):
            step = kr.RetrievalStep(ia, ib, nq, k, perm_img=pi, want_feats=True, pool_mode=mode, tau=50.0,
                                    copy_nodes=copy_nodes)
            for rep in range(2):
                so = step.run(q.cpu())
                for key in ("feat_img", "feat_txt", "pool_img", "pool_txt"):
                    assert bool(pe.equal_rows(so[key], o[key]).all()), ("graph", copy_nodes, mode, key, rep)


# ------------------------------------------------------------------ keds_gather_pool
def test_gather_pool_entry_point():
    """Weighted pool with H = 3, negative weights, ids -1 and >= ntotal, d = 37 (element loads);
    the gather with perm entries outside [0, k)."""
    for d in (37, 768):
        x = unit(500, d, 40 + d)
        ix = build(x, "ip")
        g = torch.Generator().manual_seed(d)
        I = torch.randint(0, 500, (64, 16), generator=g)
        I[:, 3] = -1
        I[::2, 7] = 500
        I[1::3, 9] = 10 ** 9
        I = I.cuda()
        W = (torch.randn(64, 3, 16, generator=g)).cuda()
        got = kr.weighted_pool(ix, I, W)
        torch.cuda.synchronize()
        assert bool(pe.equal_rows(got, pe.weighted_pool(x, I, W)).all()), d
        perm = torch.randperm(16, generator=g)
        perm[2], perm[5], perm[11] = -1, 16, 1000
        f = kr.gather_rows(ix, I, perm)
        torch.cuda.synchronize()
        want = pe.gather(x, I, perm)
        assert bool(pe.equal_rows(f, want).all()), d
        assert (f[:, [2, 5, 11]] == 0).all()
