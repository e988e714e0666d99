"""GPU (-m gpu): the native path, called through the C ABI, against the CPU oracle on the same
seeded inputs. Parity rule (BASELINE.json north_star): identical top-k label sets except
near-ties (exact score gap < 1e-5), distances within 1e-4 absolute."""
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from keds_b200 import _capi  # noqa: E402
from keds_b200 import faiss_compat as faiss  # noqa: E402
from keds_b200 import metrics as km  # noqa: E402
from keds_b200 import retrieval as kr  # noqa: E402
from keds_b200.index import GpuIndexFlat, search2  # noqa: E402
from oracle import knn_oracle as orc  # noqa: E402
from oracle.make_golden import load_retrieval  # noqa: E402

TIE_GAP = 1e-5   # north_star: index sets may differ only inside near-ties
D_TOL = 1e-4     # north_star: distances within 1e-4 absolute


def unit(n, d, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, d, generator=g)
    return (x / x.norm(dim=1, keepdim=True)).numpy()


def build(db, metric):
    ix = GpuIndexFlat(db.shape[1], faiss.METRIC_L2 if metric == "l2" else faiss.METRIC_INNER_PRODUCT, 0)
    ix.add(db)
    return ix


def check(ix, db, q, k, metric, flags=0):
    D, I = ix.search(q, k, flags)
    assert D.dtype == np.float32 and I.dtype == np.int64 and D.shape == (q.shape[0], k)
    Dr, Ir = orc.search(db, q, k, metric)
    c = orc.compare_topk(Dr, Ir, D, I, db, q, metric, TIE_GAP, D_TOL)
    assert c["ok"], (c, ix.last_stats())
    assert ix.last_stats()["err_word"] == 0
    return c


# ------------------------------------------------------------------ the GEMM alone
@pytest.mark.parametrize("n,b,d", [(5000, 200, 768), (300, 7, 64), (1000, 128, 200), (257, 129, 768)])
@pytest.mark.parametrize("fmt", ["fp16", "bf16"])
def test_tensor_core_scores_match_the_rounded_operand_reference(n, b, d, fmt):
    """The GEMM alone, in both operand formats: against float64 products of the operands rounded to
    that format only the fp32 accumulation differs -- and by far less than the certificate's
    allowance for it (d_pad * 2.4e-7 * |q16| * |x16|, rerank.cuh)."""
    db, q = unit(n, d, 1), unit(b, d, 2)
    ix = build(db, "ip")
    assert ix.operand_format == "fp16"     # unit-norm rows: fp16 keeps more of them than bf16
    ix.set_operand_format(fmt)
    assert ix.operand_format == fmt
    got = ix.debug_scores(torch.from_numpy(q).cuda()).cpu().double()
    dt = torch.float16 if fmt == "fp16" else torch.bfloat16
    tb = lambda a: torch.from_numpy(a).to(dt).double()
    ref = tb(q) @ tb(db).t()
    d_pad = -(-d // 64) * 64
    assert (got - ref).abs().max().item() < 0.25 * d_pad * 2.4e-7   # fp32 accumulation order only
    exact = torch.from_numpy(q).double() @ torch.from_numpy(db).double().t()
    assert (got - exact).abs().max().item() < (5e-4 if fmt == "fp16" else 4e-3)   # operand rounding, unit-norm rows
    check(ix, db, q, min(16, n), "ip")


def test_fp16_subnormal_operands_are_multiplied_not_flushed():
    """The certificate's bound is stated for the operands as rounded to fp16, subnormals included
    (|x| < 6.1e-5: about one element in 800 of a unit-norm 768-d row). If the tensor cores flushed
    them the approximate score would miss their products: check a row set made almost entirely of
    fp16 subnormals against float64 products of the rounded operands."""
    rng = np.random.default_rng(5)
    n, b, d = 512, 128, 256
    db = (rng.uniform(1e-6, 5e-5, size=(n, d)) * rng.choice([-1.0, 1.0], size=(n, d))).astype(np.float32)
    db[:, 0] = 0.5                                     # one normal element per row keeps fp16 the better format
    q = rng.uniform(0.5, 1.0, size=(b, d)).astype(np.float32)
    ix = build(db, "ip")
    ix.set_operand_format("fp16")
    got = ix.debug_scores(torch.from_numpy(q).cuda()).cpu().double()
    h = lambda a: torch.from_numpy(a).to(torch.float16).double()
    ref = h(q) @ h(db).t()
    sub = (h(q)[:, 1:] @ h(db)[:, 1:].t()).abs().mean().item()      # what the subnormal part contributes
    assert sub > 1e-4
    assert (got - ref).abs().max().item() < 2e-6, ((got - ref).abs().max().item(), sub)
    check(ix, db, q, 16, "ip")


def test_operand_format_follows_the_data():
    """fp16 for data inside its range, bf16 when a value would overflow or flush; a later add that
    breaks the fp16 assumption re-rounds the rows already held; a mixed pair of databases settles
    on bf16 for the fused search. Answers are exact throughout."""
    q = unit(64, 128, 3)
    small = unit(3000, 128, 4) * np.float32(1e-6)    # fp16 would flush most of it to subnormals
    ix = build(small, "ip")
    assert ix.operand_format == "bf16"
    check(ix, small, q, 16, "ip")
    db = unit(3000, 128, 5)
    ix = build(db, "l2")
    assert ix.operand_format == "fp16"
    big = unit(500, 128, 6) * np.float32(1e6)        # beyond fp16's range
    ix.add(big)
    assert ix.operand_format == "bf16"
    both = np.concatenate([db, big])
    check(ix, both, q, 16, "l2")
    ia, ib = build(db, "ip"), build(both, "ip")
    assert (ia.operand_format, ib.operand_format) == ("fp16", "bf16")
    (Da, Ia), (Db, Ib) = search2(ia, ib, q, 16)
    assert ia.operand_format == "bf16"
    assert orc.compare_topk(*orc.search(db, q, 16), Da, Ia, db, q)["ok"]
    assert orc.compare_topk(*orc.search(both, q, 16), Db, Ib, both, q, "ip", 1e-5 * 1e6, 1e-4 * 1e6)["ok"]
    # queries beyond fp16's range are clamped in the operand and answered by the exact path
    ix = build(db, "ip")
    qbig = q * np.float32(1e6)
    D, I = ix.search(qbig, 8)
    assert ix.last_stats()["n_flagged"][0] == 64
    Dr, Ir = orc.search(db, qbig, 8)
    assert orc.compare_topk(Dr, Ir, D, I, db, qbig, "ip", 1e-5 * 1e6, 1e-4 * 1e6)["ok"]


# ------------------------------------------------------------------ search vs oracle
SHAPES = [
    (5000, 200, 768, 16),    # several tiles, two query tiles
    (70000, 130, 768, 16),   # N not a multiple of the 256-row tile, B not a multiple of 128
    (999, 5, 768, 16),       # tiny batch
    (3000, 64, 96, 4),       # d not a multiple of 64 (zero padded k-block)
    (2297, 300, 768, 16),    # CIRR-gallery sized
    (4096, 128, 768, 1),     # k = 1
    (20000, 128, 768, 64),   # k = 64 (config 5's k)
    (300, 40, 100, 16),      # d % 4 == 0 only; two tiles
]


@pytest.mark.parametrize("metric", ["ip", "l2"])
@pytest.mark.parametrize("n,b,d,k", SHAPES)
def test_search_matches_oracle(n, b, d, k, metric):
    db, q = unit(n, d, 11), unit(b, d, 12)
    if metric == "l2":  # non-unit rows so that L2 and IP really rank differently
        db = db * np.linspace(0.8, 1.25, n, dtype=np.float32)[:, None]
    ix = build(db, metric)
    check(ix, db, q, k, metric)
    check(ix, db, q, k, metric, _capi.SEARCH_EXACT_ONLY)


def test_random_shapes_property():
    """Seeded sweep over ragged shapes: N around tile / slice boundaries, B around the 128-query
    tile, d with and without 4- / 64-alignment, k from 1 to beyond the candidate capacity, both
    metrics -- every selection path of the re-rank kernel (slice-maximum, direct, radix, n < k)
    and the exact-only planner branch must agree with the oracle."""
    rng = np.random.default_rng(2024)
    dims = [8, 50, 64, 100, 128, 200, 768]
    for trial in range(40):
        n = int(rng.choice([1, 7, 255, 256, 257, 511, 1000, 1536, 4097, 9000, 30001]))
        b = int(rng.choice([1, 2, 31, 127, 128, 129, 300]))
        d = int(rng.choice(dims))
        k = int(rng.choice([1, 2, 5, 16, 17, 33, 64, 100, 257, 300]))
        metric = "l2" if trial % 2 else "ip"
        db = unit(n, d, 5000 + trial)
        if trial % 3 == 0:   # non-unit rows
            db = db * rng.uniform(0.5, 2.0, size=(n, 1)).astype(np.float32)
        q = unit(b, d, 6000 + trial) * np.float32(rng.uniform(0.5, 3.0))
        ix = build(db, metric)
        D, I = ix.search(q, k)
        Dr, Ir = orc.search(db, q, k, metric)
        # distances scale with |q|^2 |x|^2: scale the absolute tolerance accordingly
        scale = float(np.abs(Dr[np.isfinite(Dr) & (np.abs(Dr) < 1e30)]).max()) if n else 1.0
        c = orc.compare_topk(Dr, Ir, D, I, db, q, metric, TIE_GAP * max(1.0, scale), D_TOL * max(1.0, scale))
        assert c["ok"], (trial, n, b, d, k, metric, c, ix.last_stats())


def test_config1_4096_queries_vs_50k_rows():
    """BASELINE.json configs[0]: 4,096 unit-norm queries vs 50k x 768, k = 16."""
    db, q = unit(50000, 768, 1000), unit(4096, 768, 1001)
    ix = build(db, "ip")
    c = check(ix, db, q, 16, "ip")
    assert c["rows_identical"] >= 4090
    st = ix.last_stats()
    assert st["exact_only"] == 0 and st["n_flagged"][0] < 64   # the tensor-core path answered


def test_passes_queue_without_a_host_round_trip_and_their_status_adds_up():
    """A 17,000-query call runs as two passes that queue on the stream (one status block per pass,
    read once at the end): the fused two-database retrieval with the consumer across the seam,
    flagged counts summed over the passes, and the large-batch chain on ragged batches (1000
    queries: the last CTA pair works on one tile; 2049: a tile with a single query)."""
    a, b = unit(40000, 768, 4200), unit(40000, 768, 4201)
    q = unit(17000, 768, 4202)
    ia, ib = build(a, "ip"), build(b, "ip")
    qd = torch.from_numpy(q).cuda()
    perm = torch.randperm(16, generator=torch.Generator().manual_seed(6))
    o = kr.retrieve2(ia, ib, qd, 16, perm_img=perm, want_feats=True, pool_mode=kr.POOL_SOFTMAX, tau=50.0)
    ia.sync()
    st = ia.last_stats()
    assert st["err_word"] == 0 and st["exact_only"] == 0, st
    sub = np.concatenate([np.arange(0, 17000, 173), [16383, 16384, 16385, 16999]])
    for name, db, ix_perm in (("img", a, perm.numpy()), ("txt", b, None)):
        D, I = o[f"D_{name}"].cpu().numpy()[sub], o[f"I_{name}"].cpu().numpy()[sub]
        Dr, Ir = orc.search(db, q[sub], 16, "ip")
        assert orc.compare_topk(Dr, Ir, D, I, db, q[sub], "ip", TIE_GAP, D_TOL)["ok"]
        assert np.array_equal(o[f"feat_{name}"][torch.from_numpy(sub).cuda()].cpu().numpy(), orc.gather(db, I, ix_perm))
        W = orc.softmax_weights(D, 50.0)
        assert np.abs(o[f"pool_{name}"].cpu().numpy()[sub] - orc.weighted_pool(db, I, W)[:, 0]).max() < 2e-5
    # an inflated error bound flags every query: the per-pass flag counters must add up to the batch
    ia.set_eps_scale(1e4)
    D1, I1 = ia.search(qd, 16)
    ia.sync()
    assert ia.last_stats()["n_flagged"][0] == 17000
    ia.set_eps_scale(1.0)
    assert torch.equal(I1, o["I_img"])
    for n, nb, k, metric in ((30000, 1000, 16, "l2"), (70000, 2049, 16, "ip"), (20000, 1408, 64, "l2")):
        db, qq = unit(n, 768, 4000 + n % 97), unit(nb, 768, 4100 + nb % 89)
        ix = build(db, metric)
        D, I = ix.search(torch.from_numpy(qq).cuda(), k)
        ix.sync()
        assert ix.last_stats()["exact_only"] == 0
        sub = np.linspace(0, nb - 1, 64).astype(np.int64)
        Dr, Ir = orc.search(db, qq[sub], k, metric)
        c = orc.compare_topk(Dr, Ir, D.cpu().numpy()[sub], I.cpu().numpy()[sub], db, qq[sub], metric, TIE_GAP, D_TOL)
        assert c["ok"], (n, nb, k, metric, c)


def test_more_queries_than_one_pass_holds():
    """Batches above 16,384 queries (config 3 has 65,536) are cut into passes inside one call: the
    seams must not show, for one database and for the fused two-database search."""
    db, db2 = unit(6000, 64, 301), unit(6000, 64, 302)
    q = unit(16384 + 700, 64, 303)
    ix, ix2 = build(db, "l2"), build(db2, "l2")
    check(ix, db, q, 8, "l2")
    (Da, Ia), (Db, Ib) = search2(ix, ix2, torch.from_numpy(q).cuda(), 8)
    for D, I, base in ((Da, Ia, db), (Db, Ib, db2)):
        Dr, Ir = orc.search(base, q, 8, "l2")
        c = orc.compare_topk(Dr, Ir, D.cpu().numpy(), I.cpu().numpy(), base, q, "l2", TIE_GAP, D_TOL)
        assert c["ok"], c


@pytest.mark.parametrize("flags", [0, _capi.SEARCH_EXACT_ONLY])
def test_two_indices_searched_from_two_threads_on_their_own_streams(flags):
    """One search in flight per handle, but handles are independent: two host threads, two CUDA
    streams, two indices at once (the ctypes calls release the GIL). With EXACT_ONLY both go through
    the fallback kernel, whose two phases must not depend on having the SMs to itself."""
    import threading

    dbs = [unit(30000, 256, 400 + i) for i in range(2)]
    qs = [unit(200, 256, 410 + i) for i in range(2)]
    ixs = [build(db, "ip") for db in dbs]
    res, errs = [None, None], []

    def work(i):
        try:
            s = torch.cuda.Stream()
            with torch.cuda.stream(s):
                qd = torch.from_numpy(qs[i]).cuda()
                for _ in range(8):
                    D, I = ixs[i].search(qd, 16, flags)
                s.synchronize()
            res[i] = (D.cpu().numpy(), I.cpu().numpy())
        except Exception as e:  # pragma: no cover
            errs.append(e)

    ths = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    assert not errs, errs
    for i in range(2):
        Dr, Ir = orc.search(dbs[i], qs[i], 16, "ip")
        c = orc.compare_topk(Dr, Ir, res[i][0], res[i][1], dbs[i], qs[i], "ip", TIE_GAP, D_TOL)
        assert c["ok"], c
        assert ixs[i].last_stats()["err_word"] == 0


def test_growing_batches_on_a_side_stream_and_host_arrays_there():
    """Per-call scratch is re-allocated (and its padding rows cleared) as the batch grows: on a
    non-default stream that must stay ordered with the search. numpy in / numpy out from inside a
    side-stream context goes through the pinned staging buffers and must give the same answer."""
    db = unit(20000, 128, 420)
    ix = build(db, "l2")
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        for b in (3, 130, 1100, 2500, 129):
            q = unit(b, 128, 430 + b)
            Dr, Ir = orc.search(db, q, 16, "l2")
            D, I = ix.search(torch.from_numpy(q).cuda(), 16)
            s.synchronize()
            c = orc.compare_topk(Dr, Ir, D.cpu().numpy(), I.cpu().numpy(), db, q, "l2", TIE_GAP, D_TOL)
            assert c["ok"], (b, c)
            Dh, Ih = ix.search(q, 16)
            assert np.array_equal(Ih, I.cpu().numpy()) and np.array_equal(Dh, D.cpu().numpy())
            assert ix.last_stats()["err_word"] == 0


def test_odd_dimension_and_unaligned_rows():
    db, q = unit(700, 50, 3), unit(33, 50, 4)   # d = 50: scalar fp32 path, padded k-block
    check(build(db, "ip"), db, q, 10, "ip")
    check(build(db, "l2"), db, q, 10, "l2")


def test_k_larger_than_ntotal_pads_with_minus_one():
    db, q = unit(10, 64, 5), unit(4, 64, 6)
    for metric, pad in (("ip", -orc.FLT_MAX), ("l2", orc.FLT_MAX)):
        ix = build(db, metric)
        D, I = ix.search(q, 16)
        assert (I[:, 10:] == -1).all() and (D[:, 10:] == pad).all()
        check(ix, db, q, 16, metric)
    db = unit(600, 64, 5)   # approx path with k > ntotal
    check(build(db, "ip"), db, q, 700, "ip")


def test_empty_index_and_empty_batch():
    ix = GpuIndexFlat(32, faiss.METRIC_INNER_PRODUCT, 0)
    D, I = ix.search(np.zeros((3, 32), np.float32), 4)
    assert (I == -1).all() and (D == -orc.FLT_MAX).all()
    ix.add(unit(50, 32, 1))
    D, I = ix.search(np.zeros((0, 32), np.float32), 4)
    assert D.shape == (0, 4) and I.shape == (0, 4)


def test_incremental_add_and_reset():
    db, q = unit(3000, 128, 7), unit(20, 128, 8)
    ix = GpuIndexFlat(128, faiss.METRIC_INNER_PRODUCT, 0)
    ix.add(db[:1000])
    ix.add(db[1000:1001])
    ix.add(db[1001:])
    assert ix.ntotal == 3000
    check(ix, db, q, 16, "ip")
    ix.reset()
    assert ix.ntotal == 0
    ix.add(db[:500])
    check(ix, db[:500], q, 16, "ip")


def test_exact_duplicates_follow_the_tie_policy():
    """score descending, then label ascending -- duplicates of a row are returned lowest id first."""
    base = unit(400, 768, 9)
    db = np.concatenate([base, base[:100], base[:50]])   # rows 400..499 and 500..549 are copies
    q = base[:32] + 0.01 * unit(32, 768, 10)
    for metric in ("ip", "l2"):
        ix = build(db, metric)
        D, I = ix.search(q, 8)
        Dr, Ir = orc.search(db, q, 8, metric)
        # float64 may split an fp32 tie either way: compare through the parity rule, then check
        # the deterministic order among exact fp32 ties directly
        assert orc.compare_topk(Dr, Ir, D, I, db, q, metric, TIE_GAP, D_TOL)["ok"]
        for b in range(32):
            for j in range(7):
                if D[b, j] == D[b, j + 1]:
                    assert I[b, j] < I[b, j + 1]
        assert I[0, 0] == 0 and set(I[0, :3]) == {0, 400, 500}


def test_all_equal_scores():
    db = np.tile(unit(1, 64, 1), (1000, 1))
    q = unit(3, 64, 2)
    for flags in (0, _capi.SEARCH_EXACT_ONLY):
        D, I = build(db, "ip").search(q, 5, flags)
        assert (I == np.arange(5)).all()


def clustered(n, n_cent, d, seed, noise=0.05):
    """SURVEY 8(d) stress generator: n_cent centroids + noise * unit vector, renormalised."""
    g = torch.Generator().manual_seed(seed)
    cent = unit(n_cent, d, seed + 1)
    assign = torch.randint(0, n_cent, (n,), generator=g).numpy()
    x = cent[assign] + noise * unit(n, d, seed + 2)
    return (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32), cent


def test_clustered_1024_centroids_stays_on_the_certified_path():
    """SURVEY 8(d): 1024 centroids + 0.05 * noise. A whole cluster (~200 rows here) sits inside the
    error band around the k-th score; the candidate capacity (1024) and the planner's feedback
    (more, shorter slices once a crowded band has been seen) keep such queries certified: the flag
    rate must stay below 5 % and the answers exact."""
    db, cent = clustered(200_000, 1024, 768, 700)
    qc = np.arange(128) % 1024
    q = cent[qc] + 0.05 * unit(128, 768, 703)
    q = (q / np.linalg.norm(q, axis=1, keepdims=True)).astype(np.float32)
    ix = build(db, "ip")
    qd = torch.from_numpy(q).cuda()
    for _ in range(3):            # the planner adapts from the second search on
        D, I = ix.search(qd, 16)
        ix.sync()
    st = ix.last_stats()
    assert st["exact_only"] == 0 and st["n_flagged"][0] <= 6, st     # < 5 % of 128
    Dr, Ir = orc.search(db, q, 16)
    c = orc.compare_topk(Dr, Ir, D.cpu().numpy(), I.cpu().numpy(), db, q, "ip", TIE_GAP, D_TOL)
    assert c["ok"], c
    # duplicate-heavy variant: every row 32 times, shuffled
    base = unit(4000, 768, 710)
    perm = np.random.default_rng(711).permutation(4000 * 32) % 4000
    dup = base[perm]
    qd2 = base[:96] + 0.3 * unit(96, 768, 712)
    qd2 = (qd2 / np.linalg.norm(qd2, axis=1, keepdims=True)).astype(np.float32)
    ix = build(dup, "ip")
    check(ix, dup, qd2, 16, "ip")
    assert ix.last_stats()["n_flagged"][0] <= 4


def test_anisotropic_clip_like_embeddings_stay_on_the_certified_path():
    """Embeddings shaped like a real CLIP tower's rather than i.i.d. directions: a strong common
    component (random pairs have cosine ~0.5, so all scores crowd into half the range), power-law
    sized topic clusters on top, per-row noise, plus image->text style queries that sit off the row
    manifold. Exact answers, L2 (the reference's index type), flag rate below 5 %."""
    rng = np.random.default_rng(720)
    n, d, nc = 150_000, 768, 600
    common = unit(1, d, 721)[0]
    cent = unit(nc, d, 722)
    size = rng.zipf(1.5, nc).clip(1, 2000).astype(np.float64)
    assign = rng.choice(nc, size=n, p=size / size.sum())
    db = 1.0 * common[None, :] + 0.7 * cent[assign] + 0.7 * unit(n, d, 723)
    db = (db / np.linalg.norm(db, axis=1, keepdims=True)).astype(np.float32)
    cos = float(np.mean(np.sum(db[:2000] * db[2000:4000], axis=1)))
    assert 0.35 < cos < 0.65, cos
    qa = rng.choice(nc, size=128)
    q = 0.8 * common[None, :] + 0.7 * cent[qa] + 0.9 * unit(128, d, 724)     # a modality gap: off-manifold queries
    q = (q / np.linalg.norm(q, axis=1, keepdims=True)).astype(np.float32)
    ix = build(db, "l2")
    qd = torch.from_numpy(q).cuda()
    for _ in range(3):
        D, I = ix.search(qd, 16)
        ix.sync()
    st = ix.last_stats()
    assert st["exact_only"] == 0 and st["n_flagged"][0] <= 6, st
    Dr, Ir = orc.search(db, q, 16, "l2")
    c = orc.compare_topk(Dr, Ir, D.cpu().numpy(), I.cpu().numpy(), db, q, "l2", TIE_GAP, D_TOL)
    assert c["ok"], c


def test_clustered_database_certificate_and_fallback():
    """8 tight clusters of 2,500 rows put thousands of rows inside the error band around the k-th
    score -- more than any candidate list holds -- so the certificate must hand queries to the
    exact path; answers stay exact."""
    g = torch.Generator().manual_seed(21)
    cent = unit(8, 768, 20)
    assign = torch.randint(0, 8, (20000,), generator=g).numpy()
    db = cent[assign] + 0.05 * unit(20000, 768, 22)
    db = (db / np.linalg.norm(db, axis=1, keepdims=True)).astype(np.float32)
    q = cent[np.arange(40) % 8] + 0.05 * unit(40, 768, 23)
    q = (q / np.linalg.norm(q, axis=1, keepdims=True)).astype(np.float32)
    ix = build(db, "ip")
    check(ix, db, q, 16, "ip")
    assert ix.last_stats()["n_flagged"][0] > 0


def test_inflated_error_bound_routes_everything_through_the_fallback():
    db, q = unit(6000, 768, 31), unit(150, 768, 32)
    ix = build(db, "ip")
    ix.set_eps_scale(1000.0)
    check(ix, db, q, 16, "ip")
    assert ix.last_stats()["n_flagged"][0] == 150
    ix.set_eps_scale(1.0)
    check(ix, db, q, 16, "ip")
    assert ix.last_stats()["n_flagged"][0] == 0


def test_bf16_alone_is_not_exact_but_the_certified_path_is():
    """Evidence that the re-rank matters: ranking by raw tensor-core scores disagrees with fp32 on
    some queries of config 1's shape; the library's answer does not."""
    db, q = unit(50000, 768, 1000), unit(512, 768, 1001)
    ix = build(db, "ip")
    approx = ix.debug_scores(torch.from_numpy(q).cuda())
    Ia = approx.topk(16, dim=1).indices.sort(dim=1).values.cpu().numpy()
    _, Ir = orc.search(db, q, 16)
    raw_same = int((np.sort(Ir, 1) == Ia).all(1).sum())
    c = check(ix, db, q, 16, "ip")
    assert raw_same < 512 and c["bad_rows"] == 0


def test_device_tensors_in_device_tensors_out():
    db, q = unit(9000, 768, 41), unit(100, 768, 42)
    ix = build(db, "ip")
    qd = torch.from_numpy(q).cuda()
    D, I = ix.search(qd, 16)
    assert D.is_cuda and I.is_cuda and I.dtype == torch.int64
    ix.sync()
    Dn, In = ix.search(q, 16)
    assert np.array_equal(I.cpu().numpy(), In) and np.array_equal(D.cpu().numpy(), Dn)


def test_fused_two_database_search_equals_two_searches():
    a, b, q = unit(30000, 768, 51), unit(30000, 768, 52), unit(128, 768, 53)
    ia, ib = build(a, "ip"), build(b, "ip")
    (Da, Ia), (Db, Ib) = search2(ia, ib, q, 16)
    D1, I1 = ia.search(q, 16)
    D2, I2 = ib.search(q, 16)
    assert np.array_equal(Ia, I1) and np.array_equal(Ib, I2)
    assert np.array_equal(Da, D1) and np.array_equal(Db, D2)
    q3 = unit(300, 768, 55)     # three query tiles: the CTA-pair kernel with a dangling last tile
    (Da3, Ia3), (Db3, Ib3) = search2(ia, ib, q3, 16)
    assert orc.compare_topk(*orc.search(a, q3, 16), Da3, Ia3, a, q3)["ok"]
    assert orc.compare_topk(*orc.search(b, q3, 16), Db3, Ib3, b, q3)["ok"]
    a2 = unit(12345, 768, 54)   # databases of different sizes
    ia2 = build(a2, "ip")
    (Da, Ia), (Db, Ib) = search2(ia2, ib, q, 16)
    assert orc.compare_topk(*orc.search(a2, q, 16), Da, Ia, a2, q)["ok"]
    assert np.array_equal(Ib, I2)


def test_argument_errors():
    ix = build(unit(100, 32, 1), "ip")
    with pytest.raises(AssertionError):
        ix.search(np.zeros((2, 31), np.float32), 4)
    with pytest.raises(TypeError):
        ix.search(np.zeros((2, 32), np.float64), 4)
    with pytest.raises(RuntimeError, match="exceeds"):
        ix.search(np.zeros((2, 32), np.float32), 5000)
    with pytest.raises(ValueError):
        ix.search(np.zeros((2, 32), np.float32), 0)


# ------------------------------------------------------------------ shards + merge kernel
def test_row_shards_merge_to_the_unsharded_answer():
    """size-independent property: 1, 2, 3 and 8 row shards give bit-identical (D, I)."""
    db, q = unit(40000, 768, 61), unit(96, 768, 62)
    lib = _capi.load()
    D1, I1 = build(db, "ip").search(q, 64)
    for R in (2, 3, 8):
        per = -(-len(db) // R)
        Dp = torch.empty((R, 96, 64), dtype=torch.float32, device="cuda")
        Ip = torch.empty((R, 96, 64), dtype=torch.int64, device="cuda")
        for r in range(R):
            ix = build(db[r * per:(r + 1) * per], "ip")
            ix.set_id_offset(r * per)
            D, I = ix.search(torch.from_numpy(q).cuda(), 64)
            ix.sync()
            Dp[r], Ip[r] = D, I
        D = torch.empty((96, 64), dtype=torch.float32, device="cuda")
        I = torch.empty((96, 64), dtype=torch.int64, device="cuda")
        _capi.check(lib.keds_topk_merge(Dp.data_ptr(), Ip.data_ptr(), R, 96, 64, 0, D.data_ptr(), I.data_ptr(), None))
        torch.cuda.synchronize()
        assert np.array_equal(I.cpu().numpy(), I1) and np.array_equal(D.cpu().numpy(), D1)


def test_index_shards_and_replicas_in_one_process():
    db, q = unit(5000, 64, 71), unit(50, 64, 72)
    for cls in (faiss.IndexShards, faiss.IndexReplicas):
        multi = cls(64, faiss.METRIC_L2, [0, 0])     # two handles on the one GPU of the test box
        multi.add(db)
        D, I = multi.search(q, 16)
        assert multi.ntotal == 5000
        assert orc.compare_topk(*orc.search(db, q, 16, "l2"), D, I, db, q, "l2")["ok"]


# ------------------------------------------------------------------ gather / pool
def test_gather_and_weighted_pool_match_oracle():
    db, q = unit(8000, 768, 81), unit(64, 768, 82)
    ix = build(db, "ip")
    D, I = ix.search(torch.from_numpy(q).cuda(), 16)
    perm = torch.randperm(16, generator=torch.Generator().manual_seed(3))
    got = kr.gather_rows(ix, I, perm).cpu().numpy()
    assert np.array_equal(got, orc.gather(db, I.cpu().numpy(), perm.numpy()))
    assert np.array_equal(kr.gather_rows(ix, I).cpu().numpy(), orc.gather(db, I.cpu().numpy()))
    W = torch.softmax(100.0 * D, dim=1).unsqueeze(1).repeat(1, 8, 1).contiguous()
    W[:, 1:] = torch.rand(64, 7, 16, device="cuda")
    pooled = kr.weighted_pool(ix, I, W).cpu().numpy()
    ref = orc.weighted_pool(db, I.cpu().numpy(), W.cpu().numpy())
    assert np.abs(pooled - ref).max() < 1e-5     # fp32 vs float64 accumulation of 16 terms
    Ineg = I.clone()
    Ineg[:, -1] = -1
    assert (kr.gather_rows(ix, Ineg)[:, -1] == 0).all()


@pytest.mark.parametrize("metric", ["ip", "l2"])
def test_fused_retrieve2_matches_oracle(metric):
    """one native call: two-DB search + gather (image stream permuted) + mean / softmax pool"""
    a, b, q = unit(9000, 768, 91), unit(9000, 768, 92), unit(70, 768, 93)
    ia, ib = build(a, metric), build(b, metric)
    perm = torch.randperm(16, generator=torch.Generator().manual_seed(5))
    qd = torch.from_numpy(q).cuda()
    o = kr.retrieve2(ia, ib, qd, 16, perm_img=perm, want_feats=True, pool_mode=kr.POOL_SOFTMAX, tau=50.0)
    ia.sync()
    for name, db, ix_perm in (("img", a, perm.numpy()), ("txt", b, None)):
        Dr, Ir = orc.search(db, q, 16, metric)
        D, I = o[f"D_{name}"].cpu().numpy(), o[f"I_{name}"].cpu().numpy()
        assert orc.compare_topk(Dr, Ir, D, I, db, q, metric, TIE_GAP, D_TOL)["ok"]
        assert np.array_equal(o[f"feat_{name}"].cpu().numpy(), orc.gather(db, I, ix_perm))
        W = orc.softmax_weights(D if metric == "ip" else -D, 50.0)
        ref = orc.weighted_pool(db, I, W)[:, 0]
        assert np.abs(o[f"pool_{name}"].cpu().numpy() - ref).max() < 2e-5   # fp32 softmax + 16-term sum
    o2 = kr.retrieve2(ia, ib, qd, 16, want_feats=False, pool_mode=kr.POOL_MEAN, out=o)
    ia.sync()
    ref = orc.gather(a, o2["I_img"].cpu().numpy()).astype(np.float64).mean(1)
    assert np.abs(o2["pool_img"].cpu().numpy() - ref).max() < 1e-6
    pi, pt = kr.retrieve_and_pool(qd, [None, None, None, ia, ib], 16, tau=50.0)
    assert pi.shape == (70, 1, 768) and pt.shape == (70, 1, 768)


def test_graph_captured_retrieval_step_matches_the_stream_path():
    """RetrievalStep: H2D + search + gather + pool + D2H captured in a CUDA graph; replays with new
    host queries give the same answers as the plain calls and as the oracle."""
    a, b = unit(20000, 768, 101), unit(20000, 768, 102)
    ia, ib = build(a, "ip"), build(b, "ip")
    perm = torch.randperm(16, generator=torch.Generator().manual_seed(9))
    step = kr.RetrievalStep(ia, ib, 128, 16, perm_img=perm, want_feats=True, pool_mode=kr.POOL_MEAN)
    for seed in (103, 104, 105):
        q = unit(128, 768, seed)
        out = step.run(torch.from_numpy(q))
        Dr, Ir = orc.search(a, q, 16)
        assert orc.compare_topk(Dr, Ir, step.D_img.numpy(), step.I_img.numpy(), a, q)["ok"]
        Dr, Ir = orc.search(b, q, 16)
        assert orc.compare_topk(Dr, Ir, step.D_txt.numpy(), step.I_txt.numpy(), b, q)["ok"]
        assert np.array_equal(out["feat_img"].cpu().numpy(), orc.gather(a, step.I_img.numpy(), perm.numpy()))
        ref = orc.gather(b, step.I_txt.numpy()).astype(np.float64).mean(1)
        assert np.abs(out["pool_txt"].cpu().numpy() - ref).max() < 1e-6


# ------------------------------------------------------------------ reference-shaped operators vs golden
def test_search_gather_returns_neighbours_or_their_weighted_pool():
    a, b, q = unit(7000, 768, 291), unit(7000, 768, 292), unit(50, 768, 293)
    ia, ib = build(a, "ip"), build(b, "ip")
    qd = torch.from_numpy(q).cuda()
    perm = torch.randperm(16, generator=torch.Generator().manual_seed(7))
    D, I, feats = kr.search_gather(ia, qd, 16, perm=perm)
    Dr, Ir = orc.search(a, q, 16, "ip")
    assert orc.compare_topk(Dr, Ir, D.cpu().numpy(), I.cpu().numpy(), a, q, "ip", TIE_GAP, D_TOL)["ok"]
    assert np.array_equal(feats.cpu().numpy(), orc.gather(a, I.cpu().numpy(), perm.numpy()))
    W = torch.softmax(100.0 * D, dim=1).unsqueeze(1).contiguous()
    _, I2, pooled = kr.search_gather(ia, qd, 16, bases=ib, weights=W)     # image labels, text rows
    assert torch.equal(I2, I)
    ref = orc.weighted_pool(b, I.cpu().numpy(), W.cpu().numpy())
    assert np.abs(pooled.cpu().numpy() - ref).max() < 1e-5
    with pytest.raises(ValueError):
        kr.search_gather(ia, qd, 16, bases=build(b[:100], "ip"))


def test_host_io_through_the_mapping_equals_the_copy_path():
    """keds_retrieve2 with host I/O: pinned host queries read by the first kernel through the mapping and
    (D, I) mirrored into pinned host blocks by the ranking blocks -- same answers as device queries
    + copies, for certified queries, for flagged ones (mirrored by the exact fallback), for a
    database small enough to go to the exact kernels only, and across a pass seam."""
    a, b = unit(9000, 768, 191), unit(9000, 768, 192)
    ia, ib = build(a, "l2"), build(b, "l2")
    perm = torch.randperm(16, generator=torch.Generator().manual_seed(5))

    def both(ia, ib, q, eps=1.0):
        qh = torch.from_numpy(q).pin_memory()
        B = q.shape[0]
        ho = {"D_img": torch.zeros((B, 16)).pin_memory(), "I_img": torch.zeros((B, 16), dtype=torch.int64).pin_memory(),
              "D_txt": torch.zeros((B, 16)).pin_memory(), "I_txt": torch.zeros((B, 16), dtype=torch.int64).pin_memory()}
        ia.set_eps_scale(eps)
        o = kr.retrieve2(ia, ib, qh, 16, perm_img=perm, want_feats=True, pool_mode=kr.POOL_SOFTMAX, tau=50.0, host_out=ho)
        ia.sync()
        st = ia.last_stats()
        r = kr.retrieve2(ia, ib, torch.from_numpy(q).cuda(), 16, perm_img=perm, want_feats=True, pool_mode=kr.POOL_SOFTMAX, tau=50.0)
        ia.sync()
        ia.set_eps_scale(1.0)
        for key in ("D_img", "I_img", "D_txt", "I_txt"):
            assert torch.equal(o[key], r[key]), key
            assert torch.equal(ho[key], r[key].cpu()), key
        for key in ("feat_img", "feat_txt", "pool_img", "pool_txt"):
            assert torch.equal(o[key], r[key]), key
        return st, ho

    q = unit(70, 768, 193)
    st, ho = both(ia, ib, q)
    assert st["n_flagged"] == [0, 0] and st["exact_only"] == 0
    Dr, Ir = orc.search(a, q, 16, "l2")
    assert orc.compare_topk(Dr, Ir, ho["D_img"].numpy(), ho["I_img"].numpy(), a, q, "l2", TIE_GAP, D_TOL)["ok"]
    st, _ = both(ia, ib, q, eps=1e4)              # every query flagged: the fallback mirrors the rows
    assert st["n_flagged"] == [70, 70]
    sa, sb = build(a[:200], "ip"), build(b[:200], "ip")
    st, _ = both(sa, sb, q)                       # exact kernels only (no k_prep_rows in the chain)
    assert st["exact_only"] == 1
    ca, cb = build(unit(3000, 64, 194), "ip"), build(unit(3000, 64, 195), "ip")
    both(ca, cb, unit(16384 + 300, 64, 196))      # two passes: the mirrors follow the pass offsets
    with pytest.raises(Exception):
        kr.retrieve2(ia, ib, torch.from_numpy(q), 16)   # pageable host memory is refused
    # fewer rows than k: the padding (-1, -/+FLT_MAX) reaches the host mirror as well
    ta, tb = build(a[:10], "ip"), build(b[:10], "ip")
    _, ho = both(ta, tb, q[:5])
    assert (ho["I_img"][:, 10:] == -1).all() and (ho["D_txt"][:, 10:] == -orc.FLT_MAX).all()
    assert (ho["I_img"][:, :10] >= 0).all()


def test_retrieval_pipeline_two_steps_in_flight():
    """RetrievalPipeline: batch i+1 submitted before batch i is consumed; every batch's host and
    device results equal the plain call's."""
    a, b = unit(12000, 768, 391), unit(12000, 768, 392)
    ia, ib = build(a, "l2"), build(b, "l2")
    perm = torch.randperm(16, generator=torch.Generator().manual_seed(9))
    pipe = kr.RetrievalPipeline(ia, ib, 64, topk=16, perm_img=perm, want_feats=True, pool_mode=kr.POOL_MEAN)
    qs = [torch.from_numpy(unit(64, 768, 400 + i)) for i in range(5)]
    tickets, got = [], []
    tickets.append(pipe.submit(qs[0]))
    for i in range(1, 5):
        tickets.append(pipe.submit(qs[i]))                 # batch i goes in ...
        st = pipe.wait(tickets[i - 1])                     # ... before batch i-1 is read
        got.append((st.I_img.clone(), st.D_txt.clone(), st.out["feat_img"].clone(), st.out["pool_txt"].clone()))
    st = pipe.wait(tickets[4])
    got.append((st.I_img.clone(), st.D_txt.clone(), st.out["feat_img"].clone(), st.out["pool_txt"].clone()))
    with pytest.raises(ValueError):
        pipe.wait(tickets[1])
    for i in range(5):
        r = kr.retrieve2(ia, ib, qs[i].cuda(), 16, perm_img=perm, want_feats=True, pool_mode=kr.POOL_MEAN)
        ia.sync()
        assert torch.equal(got[i][0], r["I_img"].cpu()) and torch.equal(got[i][1], r["D_txt"].cpu())
        assert torch.equal(got[i][2], r["feat_img"]) and torch.equal(got[i][3], r["pool_txt"])


def test_get_retrieved_features_matches_the_reference_outputs(golden_dir):
    z = load_retrieval(os.path.join(golden_dir, "retrieval.npz"))
    ib, tb = torch.from_numpy(z["image_base"]), torch.from_numpy(z["text_base"])
    names = [f"{i:07d}" for i in range(len(ib))]
    feature = torch.from_numpy(z["feature"]).cuda()
    for metric in (faiss.METRIC_L2, faiss.METRIC_INNER_PRODUCT):   # unit rows: same ranking
        database = kr.KnowledgeBase(ib, tb, names, 0, metric)
        torch.manual_seed(999)
        fi, ft = kr.get_retrieved_features(feature, database, None, topk=16, use_faiss=True)
        assert fi.is_cuda and fi.shape == (32, 16, 64)
        assert np.array_equal(fi.cpu().numpy(), z["faiss_branch_image"])
        assert np.array_equal(ft.cpu().numpy(), z["faiss_branch_text"])
        ti, tt = kr.get_retrieved_features(feature, database, None, topk=16, use_faiss=False)
        assert np.array_equal(ti.cpu().numpy(), z["torch_branch_image"])
        assert np.array_equal(tt.cpu().numpy(), z["torch_branch_text"])
        et, en = kr.get_extra_cap_features(feature, database, None, topk=2)
        assert np.array_equal(et.cpu().numpy(), z["extra_text"]) and en == list(z["extra_names"])


def test_reference_call_sequence_through_the_faiss_names(golden_dir):
    """src/main.py:72-83 verbatim, with `faiss` bound to keds_b200.faiss_compat."""
    z = load_retrieval(os.path.join(golden_dir, "retrieval.npz"))
    image_bases = torch.from_numpy(z["image_base"])
    image_index = faiss.IndexFlatL2(64)
    res = faiss.StandardGpuResources()
    image_gpu_index = faiss.index_cpu_to_gpu(res, 0, image_index)
    image_gpu_index.add(image_bases.numpy())
    f = z["feature"] / np.linalg.norm(z["feature"], axis=1, keepdims=True)
    _, topk = image_gpu_index.search(f, 16)
    assert np.array_equal(image_bases[topk.reshape(-1)].reshape(32, 16, -1).numpy(),
                          orc.gather(z["image_base"], orc.search(z["image_base"], f, 16, "l2")[1]))
    assert faiss.get_num_gpus() >= 1
    allg = faiss.index_cpu_to_all_gpus(image_index)
    allg.add(image_bases.numpy())
    assert np.array_equal(allg.search(f, 16)[1], topk)


def _close(got, want, tol=1e-4):
    assert set(got) == set(want)
    for k in want:
        assert float(got[k]) == pytest.approx(want[k], rel=tol, abs=tol), (k, got[k], want[k])


def test_gallery_metrics_match_the_reference_outputs(golden_dir):
    z = np.load(os.path.join(golden_dir, "metrics_inputs.npz"))
    e = json.load(open(os.path.join(golden_dir, "metrics_expected.json")))
    t = lambda a: torch.from_numpy(a).cuda()
    _close(km.get_metrics_cirr(t(z["gal"]), t(z["qf"]), e["reference_names"], e["index_names"], e["target_names"]),
           e["metrics"]["cirr"])
    ans = [e["fashion_names"][i] for i in z["tgt"]]
    _close(km.get_metrics_fashion(t(z["gal"]), t(z["qf"]), e["fashion_names"], ans), e["metrics"]["fashion"])
    _close(km.get_metrics_coco(t(z["coco_img"]), t(z["coco_ref"]), torch.tensor(100.0)), e["metrics"]["coco"])
    _close(km.get_metrics_imgnet(t(z["in_q"]), t(z["in_gal"]), torch.from_numpy(z["in_qlab"]),
                                 torch.from_numpy(z["in_glab"])), e["metrics"]["imgnet"])


def test_gallery_rank_matches_oracle_at_cirr_shape():
    """configs[3]: 4,181 queries vs 2,297 gallery rows, one excluded reference image per query."""
    gal = unit(2297, 768, 1006)
    rng = np.random.default_rng(1007)
    tgt = rng.integers(0, 2297, 4181)
    ref = (tgt + rng.integers(1, 2297, 4181)) % 2297
    q = gal[tgt] + gal[ref] + 2.0 * unit(4181, 768, 1007)
    q = (q / np.linalg.norm(q, axis=1, keepdims=True)).astype(np.float32)
    got = km.gallery_rank(torch.from_numpy(q).cuda(), torch.from_numpy(gal).cuda(), tgt, ref).cpu().numpy()
    want = orc.target_ranks(q, gal, tgt, ref)
    # fp32 vs float64 scores may flip a near-tie: ranks may differ by the number of near-ties only
    assert np.mean(got == want) > 0.999 and np.abs(got - want).max() <= 1
    for k in (1, 5, 10, 50, 100):
        assert np.mean(got < k) == pytest.approx(np.mean(want < k), abs=5e-4)


def test_gallery_rank_tensor_core_path_equals_the_exact_count():
    """keds_index_rank: the tensor-core count + exact settlement of the band rows must give the
    ranks of the plain fp32 count (keds_gallery_rank's SIMT kernel on the same inputs) bit for bit:
    mid-ranked random targets (crowded bands), a 50k-row gallery, a batch below one query tile, an
    inflated error bound that overflows the band lists (exact recount queue), no exclusions, and a
    batch of two passes (17,000 queries)."""
    lib = _capi.load()

    def simt(q, gal, tgt, ref):
        out = torch.empty(q.shape[0], dtype=torch.int64, device="cuda")
        _capi.check(lib.keds_gallery_rank(q.data_ptr(), 60, gal.data_ptr(), gal.shape[0], gal.shape[1],
                                          tgt.data_ptr(), 0 if ref is None else ref.data_ptr(), out.data_ptr(), None))
        torch.cuda.synchronize()
        return out[:60]   # below 64 queries the C entry point keeps to the fp32 SIMT kernel

    for ng, nq, seed in ((2297, 4181, 1), (50000, 1000, 2), (700, 100, 3), (2297, 17000, 4)):
        gal = torch.from_numpy(unit(ng, 768, 900 + seed)).cuda()
        q = torch.from_numpy(unit(nq, 768, 910 + seed)).cuda()
        rng = np.random.default_rng(seed)
        tgt = torch.from_numpy(rng.integers(0, ng, nq)).cuda()
        ref = (tgt + torch.from_numpy(rng.integers(1, ng, nq)).cuda()) % ng
        got = km.gallery_rank(q, gal, tgt, ref)
        want = orc.target_ranks(q.cpu().numpy(), gal.cpu().numpy(), tgt.cpu().numpy(), ref.cpu().numpy())
        # against float64: a row within fp32 rounding of the target's score may fall either side
        # (mid-ranked targets in a 50k gallery have thousands of rows per 1e-3 of score)
        assert np.abs(got.cpu().numpy() - want).max() <= 1 and np.mean(got.cpu().numpy() == want) > 0.98
        assert torch.equal(got[:60], simt(q, gal, tgt, ref))          # the exact fp32 count, bit for bit
        got2 = km.gallery_rank(q, gal, tgt)                            # cached index, no exclusion
        assert torch.equal(got2[:60], simt(q, gal, tgt, None))
        ix = km.gallery_index(gal)
        ix.set_eps_scale(200.0)                                        # bands overflow: exact recount queue
        got3 = km.gallery_rank(q, gal, tgt, ref)
        ix.set_eps_scale(1.0)
        assert torch.equal(got3, got)
    km.clear_gallery_cache()


def test_index_label_hits_equal_the_search_then_count_path():
    """keds_index_label_hits (get_metrics_imgnet's core in one call): the hit counts at every cut
    point must equal those of an exact search followed by counting -- bit for bit against the native
    search (same fp32 scores, same tie rule) and against the float64 oracle wherever no near-tie
    sits on a cut. Few classes, so that hits are plentiful; duplicated gallery rows with different
    labels, so that ties straddle the cuts; both metrics; every query through the fallback."""
    rng = np.random.default_rng(810)
    g = unit(30000, 768, 811)
    g[5000:5600] = g[:600]                       # exact duplicates: equal scores, the lower row id wins
    q = unit(700, 768, 812)
    q[:300] = g[rng.integers(0, 600, 300)] + 0.6 * q[:300]   # queries near duplicated rows
    q = (q / np.linalg.norm(q, axis=1, keepdims=True)).astype(np.float32)
    glab = torch.from_numpy(rng.integers(0, 40, 30000))
    qlab = torch.from_numpy(rng.integers(0, 40, 700))
    qd = torch.from_numpy(q).cuda()
    for metric in ("ip", "l2"):
        ix = build(g, metric)
        for ks in ([1, 5, 10, 50, 100, 200], [3], [16, 64]):
            hits = km.index_label_hits(ix, qd, glab, qlab, ks)
            ix.sync()
            st = ix.last_stats()
            assert st["exact_only"] == 0 and st["err_word"] == 0 and st["n_flagged"][0] <= 35, st
            _, I = ix.search(qd, max(ks))
            want = km.label_hits(I, glab, qlab, ks)
            assert torch.equal(hits, want), (metric, ks, (hits != want).sum().item())
        # float64 oracle: equal except where a near-tie sits on a cut point
        ks = [1, 5, 10, 50, 100, 200]
        hits = km.index_label_hits(ix, qd, glab, qlab, ks).cpu().numpy()
        Dr, Ir = orc.search(g, q, 201, metric)
        lab = glab.numpy()[Ir] == qlab.numpy()[:, None]
        for i, k in enumerate(ks):
            ref = lab[:, :k].sum(1)
            bad = np.nonzero(ref != hits[:, i])[0]
            gap = np.abs(Dr[bad, k - 1].astype(np.float64) - Dr[bad, k].astype(np.float64))
            assert (gap < TIE_GAP * (2.0 if metric == "l2" else 1.0)).all(), (metric, k, bad[:5], gap[:5])
        # every query through the exact fallback: same counts
        ix.set_eps_scale(1e4)
        h2 = km.index_label_hits(ix, qd, glab, qlab, ks)
        ix.sync()
        assert ix.last_stats()["n_flagged"][0] == 700
        ix.set_eps_scale(1.0)
        assert np.array_equal(h2.cpu().numpy(), hits)
    # more queries than one pass holds: hits, labels and status follow the pass offsets
    gm, qm = unit(6000, 64, 813), unit(16384 + 500, 64, 814)
    lm, qlm = torch.from_numpy(rng.integers(0, 20, 6000)), torch.from_numpy(rng.integers(0, 20, 16884))
    im = build(gm, "ip")
    qmd = torch.from_numpy(qm).cuda()
    hm = km.index_label_hits(im, qmd, lm, qlm, [1, 10, 100])
    im.sync()
    assert im.last_stats()["err_word"] == 0
    _, I = im.search(qmd, 100)
    assert torch.equal(hm, km.label_hits(I, lm, qlm, [1, 10, 100]))
    # a gallery too small for the tensor-core path, and cut points beyond its size
    small = build(g[:150], "ip")
    hs = km.index_label_hits(small, qd, glab[:150], qlab, [1, 100, 200])
    _, I = small.search(qd, 200)
    assert torch.equal(hs, km.label_hits(I, glab[:150], qlab, [1, 100, 200]))


def test_imgnet_shaped_recall_50k_gallery():
    """configs[3]: 50k-row gallery with labels < 7000, top-200 label hits."""
    rng = np.random.default_rng(1008)
    glab = rng.integers(0, 7000, 50000)
    qlab = rng.integers(0, 7000, 1000)
    cent = unit(7000, 256, 1008)
    gal = cent[glab] + 1.0 * unit(50000, 256, 1009)
    gal = (gal / np.linalg.norm(gal, axis=1, keepdims=True)).astype(np.float32)
    q = cent[qlab] + 1.0 * unit(1000, 256, 1010)
    q = (q / np.linalg.norm(q, axis=1, keepdims=True)).astype(np.float32)
    got = km.get_metrics_imgnet(torch.from_numpy(q), torch.from_numpy(gal), torch.from_numpy(qlab), torch.from_numpy(glab))
    want = orc.metrics_imgnet(q, gal, qlab, glab)
    _close(got, want, 2e-3)


# ------------------------------------------------------------------ full-size properties (configs[1])
def test_training_step_shape_full_size_properties():
    """128 queries vs two 0.5M x 768 databases, k = 16: too big for the float64 oracle in seconds,
    so check (a) the fused two-DB search against torch float64 on the GPU, (b) shard invariance,
    (c) invariance under a permutation of the rows, (d) L2 == IP ranking on unit rows."""
    n, d, b, k = 500000, 768, 128, 16
    dbs = []
    for s in (1002, 1003):
        g = torch.Generator(device="cuda").manual_seed(s)
        x = torch.randn(n, d, generator=g, device="cuda")
        dbs.append(x / x.norm(dim=1, keepdim=True))
    q = torch.from_numpy(unit(b, d, 1004)).cuda()
    ia = GpuIndexFlat(d, faiss.METRIC_INNER_PRODUCT, 0)
    ib = GpuIndexFlat(d, faiss.METRIC_INNER_PRODUCT, 0)
    ia.add(dbs[0])
    ib.add(dbs[1])
    (Da, Ia), (Db, Ib) = search2(ia, ib, q, k)
    ia.sync()
    assert ia.last_stats()["exact_only"] == 0 and ia.last_stats()["err_word"] == 0
    sub = np.arange(0, b, 8)    # 16 queries through the float64 numpy oracle, north_star's near-tie rule
    for dbt, D, I in ((dbs[0], Da, Ia), (dbs[1], Db, Ib)):
        s = q.double() @ dbt.double().t()
        v, i = s.topk(k, dim=1)
        assert (i == I).all(dim=1).float().mean().item() >= 0.99      # near-ties may swap
        assert (torch.sort(i, 1).values == torch.sort(I, 1).values).all(dim=1).float().mean().item() >= 0.99
        assert (v.float() - D).abs().max().item() < D_TOL
        del s
        db_host, q_host = dbt.cpu().numpy(), q.cpu().numpy()[sub]
        Dr, Ir = orc.search(db_host, q_host, k, "ip")
        c = orc.compare_topk(Dr, Ir, D.cpu().numpy()[sub], I.cpu().numpy()[sub], db_host, q_host, "ip", TIE_GAP, D_TOL)
        assert c["ok"], c
        del db_host
    # (b) two row shards + merge == whole
    lib = _capi.load()
    half = n // 2
    Dp = torch.empty((2, b, k), dtype=torch.float32, device="cuda")
    Ip = torch.empty((2, b, k), dtype=torch.int64, device="cuda")
    for r in range(2):
        sh = GpuIndexFlat(d, faiss.METRIC_INNER_PRODUCT, 0)
        sh.add(dbs[0][r * half:(r + 1) * half])
        sh.set_id_offset(r * half)
        Dp[r], Ip[r] = sh.search(q, k)
        sh.sync()
        del sh
    Dm = torch.empty((b, k), dtype=torch.float32, device="cuda")
    Im = torch.empty((b, k), dtype=torch.int64, device="cuda")
    _capi.check(lib.keds_topk_merge(Dp.data_ptr(), Ip.data_ptr(), 2, b, k, 0, Dm.data_ptr(), Im.data_ptr(), None))
    torch.cuda.synchronize()
    assert torch.equal(Im, Ia) and torch.equal(Dm, Da)
    # (c) permuting the rows permutes the labels and nothing else
    perm = torch.randperm(n, device="cuda", generator=torch.Generator(device="cuda").manual_seed(7))
    ip = GpuIndexFlat(d, faiss.METRIC_INNER_PRODUCT, 0)
    ip.add(dbs[0][perm].contiguous())
    Dq, Iq = ip.search(q, k)
    ip.sync()
    assert torch.equal(Dq, Da)
    assert (perm[Iq] == Ia).all(dim=1).float().mean().item() >= 0.99
    del ip
    # (d) squared L2 on unit rows: same ranking, D = 2 - 2 ip
    il2 = GpuIndexFlat(d, faiss.METRIC_L2, 0)
    il2.add(dbs[0])
    qn = q / q.norm(dim=1, keepdim=True)
    Dl, Il = il2.search(qn, k)
    Di, Ii = ia.search(qn, k)
    il2.sync()
    assert (Il == Ii).all(dim=1).float().mean().item() >= 0.98
    assert (Dl - (2 - 2 * Di)).abs().max().item() < 1e-5


def test_eval_scale_65536_queries_full_size():
    """BASELINE.json configs[2]: 65,536 queries vs 0.5M x 768, k = 16, issued as ONE call the way
    evaluate_* would (src/eval_utils.py:153-186): four passes of 16,384 inside the library. Checked
    against the float64 oracle on a stratified subset of 256 queries spread over all four passes
    plus the rows either side of every pass seam, with the near-tie rule."""
    n, d, nq, k = 500000, 768, 65536, 16
    g = torch.Generator(device="cuda").manual_seed(1002)
    x = torch.randn(n, d, generator=g, device="cuda")
    x = x / x.norm(dim=1, keepdim=True)
    ix = GpuIndexFlat(d, faiss.METRIC_INNER_PRODUCT, 0)
    ix.add(x)
    db_host = x.cpu().numpy()
    del x
    g = torch.Generator(device="cuda").manual_seed(1005)
    q = torch.randn(nq, d, generator=g, device="cuda")
    q = q / q.norm(dim=1, keepdim=True)
    D, I = ix.search(q, k)
    ix.sync()
    st = ix.last_stats()
    assert st["exact_only"] == 0 and st["err_word"] == 0
    seams = [s + o for s in (16384, 32768, 49152) for o in (-2, -1, 0, 1)]
    sub = np.unique(np.concatenate([np.arange(0, nq, 256), np.array(seams + [0, nq - 1])]))
    q_host = q[torch.from_numpy(sub).cuda()].cpu().numpy()
    Dr, Ir = orc.search(db_host, q_host, k, "ip")
    c = orc.compare_topk(Dr, Ir, D.cpu().numpy()[sub], I.cpu().numpy()[sub], db_host, q_host, "ip", TIE_GAP, D_TOL)
    assert c["ok"] and c["rows"] >= 256, c
    # size-independent property over ALL 65,536 rows: every answer is sorted, in range, free of repeats
    assert bool((D[:, 1:] <= D[:, :-1]).all()) and int(I.min()) >= 0 and int(I.max()) < n
    srt = torch.sort(I, dim=1).values
    assert bool((srt[:, 1:] != srt[:, :-1]).all())


def test_cirr_testoutput_matches_the_reference_output(golden_dir):
    """get_cirr_testoutput (src/eval_utils.py:1070-1087) against what the reference's own function
    produced (oracle/make_golden.py)."""
    z = np.load(os.path.join(golden_dir, "metrics_inputs.npz"))
    e = json.load(open(os.path.join(golden_dir, "metrics_expected.json")))["cirr_test"]
    got = km.get_cirr_testoutput(torch.from_numpy(z["gal"]).cuda(), torch.from_numpy(z["qf"]).cuda(),
                                 e["reference_names"], e["index_names"], torch.tensor(e["pair_ids"]))
    assert got == e["output"]
    assert got == orc.cirr_testoutput(z["gal"], z["qf"], e["reference_names"], e["index_names"], e["pair_ids"])
    with pytest.raises(IndexError):
        km.get_cirr_testoutput(torch.from_numpy(z["gal"][:40]).cuda(), torch.from_numpy(z["qf"][:3]).cuda(),
                               e["index_names"][:3], e["index_names"][:40], [1, 2, 3])


def test_real_faiss_cross_check_when_installed():
    """SURVEY 8(c): the arithmetic the reference delegates to Faiss. Runs only where `import faiss`
    works (it does not in the build image): IndexFlatIP / IndexFlatL2 of faiss-cpu on config 1's
    shape against the native index."""
    real = pytest.importorskip("faiss")
    db, q = unit(50000, 768, 1000), unit(512, 768, 1001)
    for metric, cls in (("ip", real.IndexFlatIP), ("l2", real.IndexFlatL2)):
        ref = cls(768)
        ref.add(db)
        Dr, Ir = ref.search(q, 16)
        D, I = build(db, metric).search(q, 16)
        assert orc.compare_topk(Dr, Ir, D, I, db, q, metric, TIE_GAP, D_TOL)["ok"]


def test_replicas_across_all_gpus_of_the_box():
    """index_cpu_to_all_gpus as the eval script uses it (src/eval_retrieval.py:292,295): one full
    copy per GPU, the query batch split across them from one host thread per GPU; identical to a
    single-GPU search. Needs more than one GPU (the driver's multi-GPU boxes)."""
    ngpu = faiss.get_num_gpus()
    if ngpu < 2:
        pytest.skip("one GPU on this box")
    db, q = unit(60000, 768, 1100), unit(1000, 768, 1101)
    cpu = faiss.IndexFlatL2(768)
    cpu.add(db)
    multi = faiss.index_cpu_to_all_gpus(cpu)
    assert isinstance(multi, faiss.IndexReplicas) and len(multi.subs) == ngpu
    D, I = multi.search(q, 16)
    D1, I1 = build(db, "l2").search(q, 16)
    assert np.array_equal(I, I1) and np.array_equal(D, D1)
    co = faiss.GpuMultipleClonerOptions()
    co.shard = True
    sh = faiss.index_cpu_to_all_gpus(cpu, co)
    Ds, Is = sh.search(q, 16)
    assert np.array_equal(Is, I1) and np.array_equal(Ds, D1)


def test_retrieval_step_recaptures_when_the_handle_reallocates():
    """ADVICE r1: a captured RetrievalStep bakes in the handles' scratch addresses; a later plain
    call with a larger batch moves them. run() must notice (generation counter) and re-capture
    instead of replaying over freed memory."""
    a, b = unit(20000, 768, 121), unit(20000, 768, 122)
    ia, ib = build(a, "ip"), build(b, "ip")
    step = kr.RetrievalStep(ia, ib, 64, 16, want_feats=False, pool_mode=kr.POOL_MEAN)
    q = unit(64, 768, 123)
    step.run(torch.from_numpy(q))
    want = step.I_img.clone()
    gen = ia.generation
    big = torch.from_numpy(unit(3000, 768, 124)).cuda()
    kr.retrieve2(ia, ib, big, 64, want_feats=True, pool_mode=kr.POOL_NONE)    # grows every scratch buffer
    ia.sync()
    assert ia.generation != gen
    step.run(torch.from_numpy(q))
    assert step.recaptures == 1 and torch.equal(step.I_img, want)
    assert orc.compare_topk(*orc.search(a, q, 16), step.D_img.numpy(), step.I_img.numpy(), a, q)["ok"]
    ia.add(unit(100, 768, 125))      # rows change too
    step.run(torch.from_numpy(q))
    assert step.recaptures == 2


def test_database_builder_normalises_on_the_device_and_round_trips(tmp_path):
    """§8 f1: rows are L2-normalised while they are added; the saved artefacts keep the .pt layout
    and reload into an identical database."""
    from keds_b200 import database as kdb

    g = torch.Generator().manual_seed(77)
    img = torch.randn(3000, 768, generator=g) * 3.0
    txt = torch.randn(3000, 768, generator=g) * 0.2
    names = [f"{i:07d}" for i in range(3000)]
    kb = kdb.build_knowledge_base(img, txt, names, device=0, normalize=True)
    ref = img / img.norm(dim=1, keepdim=True)                     # src/main.py:465
    assert (kb.image_bases - ref).abs().max().item() < 2e-7       # fp32 norm + divide, two roundings
    assert (kb.image_bases.norm(dim=1) - 1).abs().max().item() < 1e-6
    q = unit(40, 768, 78)
    fi, ft = kr.get_retrieved_features(torch.from_numpy(q).cuda(), kb, None, topk=16, use_faiss=False)
    want = orc.gather(kb.image_bases.numpy(), orc.search(kb.image_bases.numpy(), q, 16)[1])
    assert np.array_equal(fi.cpu().numpy(), want)
    paths = kdb.save_artefacts(kb, str(tmp_path))
    kb2 = kr.KnowledgeBase.load(*paths, device=0)
    assert torch.equal(kb2.image_bases, kb.image_bases) and kb2.basenames == names
    D1, I1 = kb.text_index.search(q, 16)
    D2, I2 = kb2.text_index.search(q, 16)
    assert np.array_equal(I1, I2) and np.array_equal(D1, D2)
