"""GPU (-m gpu): search with exclusion. Every result must equal the exact search over the rows the
query does not exclude: checked against the CPU oracle, and bit for bit against a plain search
for k + E rows with the excluded labels dropped afterwards."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from keds_b200 import _capi  # noqa: E402
from keds_b200 import retrieval as kr  # noqa: E402
from keds_b200.index import METRIC_INNER_PRODUCT, METRIC_L2, GpuIndexFlat, search2  # noqa: E402
from oracle import knn_oracle as orc  # noqa: E402

TIE_GAP = 1e-5
D_TOL = 1e-4


def unit(n, d, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, d, generator=g)
    return (x / x.norm(dim=1, keepdim=True)).numpy()


def build(db, metric, fmt=None):
    ix = GpuIndexFlat(db.shape[1], METRIC_L2 if metric == "l2" else METRIC_INNER_PRODUCT, 0)
    ix.add(db)
    if fmt is not None:
        ix.set_operand_format(fmt)
    return ix


def drop_excluded(D1, I1, ex, k):
    """A plain search for k + E rows with each query's excluded labels removed, first k kept."""
    gone = ((I1[:, :, None] == ex[:, None, :]) & (ex[:, None, :] >= 0)).any(2)
    order = np.argsort(gone, axis=1, kind="stable")[:, :k]
    return np.take_along_axis(D1, order, 1), np.take_along_axis(I1, order, 1)


def search_excluding(db, q, k, metric, ex):
    """The float64 reference over the rows each query does not exclude: the oracle's search for
    k + E rows (E >= the distinct labels a query can exclude), excluded labels dropped."""
    ex = np.asarray(ex, np.int64).reshape(q.shape[0], -1)
    D, I = orc.search(db, q, k + ex.shape[1], metric)
    return drop_excluded(D, I, ex, k)


def check(ix, db, q, k, metric, ex, flags=0, oracle_rows=300, id_offset=0):
    qd = torch.from_numpy(q).cuda()
    exd = torch.from_numpy(ex).cuda()
    D, I = ix.search(qd, k, flags, exclude=exd)
    ix.sync()  # (the flag counts of a device-tensor search are read back here)
    st = ix.last_stats()
    D, I = D.cpu().numpy(), I.cpu().numpy()
    assert st["err_word"] == 0
    E = ex.shape[1]
    D1, I1 = ix.search(qd, k + E, flags)
    Dw, Iw = drop_excluded(D1.cpu().numpy(), I1.cpu().numpy(), ex, k)
    np.testing.assert_array_equal(I, Iw)
    np.testing.assert_array_equal(D.view(np.uint32), Dw.view(np.uint32))
    assert not ((I[:, :, None] == ex[:, None, :]) & (ex[:, None, :] >= 0)).any()
    n = min(oracle_rows, q.shape[0])
    sel = np.unique(np.concatenate([np.arange(n // 2), np.arange(q.shape[0] - n // 2, q.shape[0])]))
    ex_local = np.where(ex[sel] >= 0, ex[sel] - id_offset, -1)
    Dr, Ir = search_excluding(db, q[sel], k, "ip" if (metric == "ip" or flags & _capi.SEARCH_FORCE_IP) else "l2",
                              ex_local)
    Ir = np.where(Ir >= 0, Ir + id_offset, -1)
    c = orc.compare_topk(Dr, Ir, D[sel], I[sel], None, None, metric, TIE_GAP, D_TOL)
    assert c["ok"], (c, st)
    return D, I, st


@pytest.fixture(scope="module")
def base():
    return unit(20000, 768, 7)


@pytest.mark.parametrize("metric", ["ip", "l2"])
@pytest.mark.parametrize("fmt", ["fp16", "bf16"])
@pytest.mark.parametrize("B", [7, 128, 300, 4096])
def test_self_exclusion_matches_oracle_and_plain_search(base, metric, fmt, B):
    """queries that are rows of the base leave themselves out (single-CTA and pair kernels)"""
    ix = build(base, metric, fmt)
    rows = np.random.default_rng(B).choice(base.shape[0], B, replace=False)
    q = base[rows].copy()
    D, I, st = check(ix, base, q, 16, metric, rows[:, None].astype(np.int64))
    assert st["exact_only"] == 0
    # without exclusion the row finds itself first
    D0, I0 = ix.search(torch.from_numpy(q).cuda(), 16)
    assert (I0[:, 0].cpu().numpy() == rows).all()


def test_two_passes(base):
    """more than 16,384 queries: the exclusion array is offset per pass"""
    ix = build(base, "ip")
    rows = np.random.default_rng(3).integers(0, base.shape[0], 17000)
    q = base[rows] + 0.01 * unit(17000, 768, 4)
    ex = np.stack([rows, (rows + 1) % base.shape[0]], 1).astype(np.int64)
    check(ix, base, q.astype(np.float32), 16, "ip", ex, oracle_rows=64)


def test_force_ip_on_an_l2_index(base):
    ix = build(base, "l2")
    rows = np.arange(0, 4000, 31)
    check(ix, base, base[rows].copy(), 16, "l2", rows[:, None].astype(np.int64), flags=_capi.SEARCH_FORCE_IP)


def test_unused_or_foreign_labels_change_nothing(base):
    ix = build(base, "l2")
    q = torch.from_numpy(unit(300, 768, 11)).cuda()
    D0, I0 = ix.search(q, 16)
    for ex in (np.full((300, 1), -1, np.int64), np.full((300, 8), -1, np.int64),
               np.stack([np.full(300, 20000), np.full(300, -5), np.full(300, 1 << 40)], 1).astype(np.int64)):
        D, I = ix.search(q, 16, exclude=torch.from_numpy(ex).cuda())
        assert torch.equal(I, I0) and torch.equal(D.view(torch.int32), D0.view(torch.int32))


def test_eight_labels_with_duplicated_rows():
    """the query's row repeated in the base: excluding some copies returns the others, in id order"""
    db = unit(5000, 256, 21)
    copies = np.array([3, 700, 701, 1500, 2048, 3333, 4000, 4999, 17, 2600])
    db[copies] = db[3]
    ix = build(db, "ip")
    q = db[[3, 3, 3, 10]].copy()
    ex = np.full((4, 8), -1, np.int64)
    ex[0] = copies[:8]
    ex[1, :3] = [4999, 700, 3]
    ex[2, :4] = [3, 3, 3, 3]
    ex[3, :2] = [10, 10]
    D, I, _ = check(ix, db, q, 16, "ip", ex)
    assert I[0, :2].tolist() == [17, 2600]
    assert I[1, :7].tolist() == [17, 701, 1500, 2048, 2600, 3333, 4000]
    assert I[2, :9].tolist() == [17, 700, 701, 1500, 2048, 2600, 3333, 4000, 4999]


@pytest.mark.parametrize("metric", ["ip", "l2"])
def test_fallback_and_exact_only_routes(base, metric):
    rows = np.random.default_rng(5).choice(base.shape[0], 200, replace=False)
    q = base[rows].copy()
    ex = np.stack([rows, np.full(200, -1), (rows * 7) % base.shape[0]], 1).astype(np.int64)
    ix = build(base, metric)
    ix.set_eps_scale(1e6)  # every query fails the certificate: the exact fallback answers all
    _, _, st = check(ix, base, q, 16, metric, ex)
    assert st["n_flagged"][0] == 200
    ix.set_eps_scale(1.0)
    _, _, st = check(ix, base, q, 16, metric, ex, flags=_capi.SEARCH_EXACT_ONLY)
    assert st["exact_only"] == 1
    _, _, st = check(ix, base, q, 600, metric, ex, oracle_rows=40)  # k > 512: exact only
    assert st["exact_only"] == 1


def test_small_bases_padding_and_id_offset():
    db = unit(200, 64, 31)  # smaller than one 256-row tile
    ix = build(db, "ip")
    rows = np.arange(0, 200, 3)
    _, _, st = check(ix, db, db[rows].copy(), 16, "ip", rows[:, None].astype(np.int64))
    assert st["exact_only"] == 1
    tiny = unit(16, 64, 32)  # ntotal == k: one row excluded leaves 15, then padding
    it = build(tiny, "l2")
    D, I, _ = check(it, tiny, tiny.copy(), 16, "l2", np.arange(16)[:, None].astype(np.int64))
    assert (I[:, 15] == -1).all() and (D[:, 15] == np.finfo(np.float32).max).all()
    assert (I[:, :15] >= 0).all()
    one = build(tiny[:1], "ip")  # every row excluded: padding only
    D, I = one.search(tiny[:2], 4, exclude=np.array([0, -1], np.int64))
    assert (I[0] == -1).all() and (D[0] == -np.finfo(np.float32).max).all() and I[1, 0] == 0
    big = unit(3000, 128, 33)
    ib = build(big, "ip")
    ib.set_id_offset(1000)
    rows = np.arange(0, 3000, 11)
    ex = np.stack([rows + 1000, rows], 1).astype(np.int64)  # the second label is some other row
    D, I, _ = check(ib, big, big[rows].copy(), 16, "ip", ex, id_offset=1000)
    assert not (I == (rows + 1000)[:, None]).any()


def test_numpy_path_and_argument_errors(base):
    ix = build(base, "ip")
    q = base[:5].copy()
    D, I = ix.search(q, 8, exclude=np.arange(5, dtype=np.int64))
    Dd, Id = ix.search(torch.from_numpy(q).cuda(), 8, exclude=torch.arange(5).cuda())
    assert np.array_equal(I, Id.cpu().numpy()) and np.array_equal(D, Dd.cpu().numpy())
    assert not (I == np.arange(5)[:, None]).any()
    with pytest.raises(TypeError):
        ix.search(q, 8, exclude=np.arange(5, dtype=np.int32))
    with pytest.raises(ValueError):
        ix.search(q, 8, exclude=np.zeros((5, 9), np.int64))
    with pytest.raises(ValueError):
        ix.search(q, 8, exclude=np.zeros(4, np.int64))


def test_retrieve2_feats_pools_and_hostio():
    a, b = unit(9000, 768, 41), unit(9000, 768, 42)
    ia, ib = build(a, "ip"), build(b, "ip")
    rows = np.random.default_rng(6).choice(9000, 70, replace=False)
    q = a[rows].copy()
    ex = np.stack([rows, np.full(70, -1)], 1).astype(np.int64)
    qd, exd = torch.from_numpy(q).cuda(), torch.from_numpy(ex).cuda()
    perm = torch.randperm(16, generator=torch.Generator().manual_seed(5))
    o = kr.retrieve2(ia, ib, qd, 16, perm_img=perm, want_feats=True, pool_mode=kr.POOL_SOFTMAX, tau=50.0,
                     exclude=exd)
    ia.sync()
    (Da, Ia), (Db, Ib) = search2(ia, ib, qd, 16, exclude=exd)
    assert torch.equal(o["I_img"], Ia) and torch.equal(o["I_txt"], Ib)
    assert torch.equal(o["D_img"], Da) and torch.equal(o["D_txt"], Db)
    for name, db, p in (("img", a, perm.numpy()), ("txt", b, None)):
        I = o[f"I_{name}"].cpu().numpy()
        assert not (I == rows[:, None]).any()
        Dr, Ir = search_excluding(db, q, 16, "ip", ex)
        assert orc.compare_topk(Dr, Ir, o[f"D_{name}"].cpu().numpy(), I, db, q, "ip", TIE_GAP, D_TOL)["ok"]
        assert np.array_equal(o[f"feat_{name}"].cpu().numpy(), orc.gather(db, I, p))
        W = orc.softmax_weights(o[f"D_{name}"].cpu().numpy(), 50.0)
        assert np.abs(o[f"pool_{name}"].cpu().numpy() - orc.weighted_pool(db, I, W)[:, 0]).max() < 2e-5
    # host I/O: pinned queries and pinned exclusion read through the mapping, pinned result mirrors
    qh, exh = torch.from_numpy(q).pin_memory(), torch.from_numpy(ex).pin_memory()
    host = {n: torch.empty((70, 16), dtype=t).pin_memory()
            for n, t in (("D_img", torch.float32), ("I_img", torch.int64), ("D_txt", torch.float32),
                         ("I_txt", torch.int64))}
    oh = kr.retrieve2(ia, ib, qh, 16, perm_img=perm, want_feats=True, pool_mode=kr.POOL_SOFTMAX, tau=50.0,
                      host_out=host, exclude=exh)
    ia.sync()
    for key in ("D_img", "I_img", "D_txt", "I_txt", "feat_img", "feat_txt", "pool_img", "pool_txt"):
        assert torch.equal(oh[key], o[key]), key
    for key in ("D_img", "I_img", "D_txt", "I_txt"):
        assert torch.equal(host[key], o[key].cpu()), key


@pytest.mark.parametrize("copy_nodes", [False, True])
def test_retrieval_step_reads_exclusion_on_every_replay(copy_nodes):
    a, b = unit(20000, 768, 51), unit(20000, 768, 52)
    ia, ib = build(a, "ip"), build(b, "ip")
    step = kr.RetrievalStep(ia, ib, 128, 16, want_feats=True, pool_mode=kr.POOL_MEAN, copy_nodes=copy_nodes,
                            n_exclude=1)
    rec = step.recaptures
    rows = np.random.default_rng(8).choice(20000, 128, replace=False)
    q = torch.from_numpy(a[rows].copy())
    step.run(q, exclude=torch.full((128,), -1, dtype=torch.int64))
    assert (step.I_img[:, 0].numpy() == rows).all()
    out = step.run(q, exclude=torch.from_numpy(rows))
    I = step.I_img.numpy().copy()
    assert not (I == rows[:, None]).any()
    ref = kr.retrieve2(ia, ib, q.cuda(), 16, want_feats=True, pool_mode=kr.POOL_MEAN,
                       exclude=torch.from_numpy(rows).cuda())
    ia.sync()
    assert np.array_equal(I, ref["I_img"].cpu().numpy()) and np.array_equal(step.I_txt.numpy(), ref["I_txt"].cpu().numpy())
    assert torch.equal(out["feat_img"], ref["feat_img"]) and torch.equal(out["pool_txt"], ref["pool_txt"])
    step.run(q, exclude=torch.from_numpy(np.roll(rows, 1)))
    assert (step.I_img[:, 0].numpy() == rows).all()
    assert step.recaptures == rec
    pipe = kr.RetrievalPipeline(ia, ib, 128, topk=16, copy_nodes=copy_nodes, n_exclude=1)
    t = pipe.submit(q, exclude=torch.from_numpy(rows))
    assert np.array_equal(pipe.wait(t).I_img.numpy(), I)


def test_get_retrieved_features_never_returns_excluded_rows():
    a = unit(6000, 768, 61)
    b = a + 0.05 * unit(6000, 768, 62)  # captions near their images: a pair's own caption ranks first
    b = (b / np.linalg.norm(b, axis=1, keepdims=True)).astype(np.float32)
    names = [f"{i:06d}.jpg" for i in range(6000)]
    kb = kr.KnowledgeBase(torch.from_numpy(a), torch.from_numpy(b), names, metric=METRIC_INNER_PRODUCT)
    rows = np.random.default_rng(9).choice(6000, 32, replace=False)
    batch = [names[r] for r in rows[:-1]] + ["not-in-the-base.jpg"]
    ex = kb.rows_of(batch)
    assert ex.tolist() == rows[:-1].tolist() + [-1]
    feat = torch.from_numpy(a[rows].copy()).cuda()
    torch.manual_seed(0)
    fi0, ft0 = kr.get_retrieved_features(feat, kb, topk=16)
    torch.manual_seed(0)
    fi1, ft1 = kr.get_retrieved_features(feat, kb, topk=16, exclude=None)
    assert torch.equal(fi0, fi1) and torch.equal(ft0, ft1)
    torch.manual_seed(0)
    fi, ft = kr.get_retrieved_features(feat, kb, topk=16, exclude=ex)
    own_img = torch.from_numpy(a[rows]).cuda()
    own_txt = torch.from_numpy(b[rows]).cuda()
    hit_img = (fi == own_img[:, None, :]).all(2)
    hit_txt = (ft == own_txt[:, None, :]).all(2)
    assert not hit_img[:-1].any() and not hit_txt[:-1].any()
    assert hit_img[-1].any() and hit_txt[-1].any()  # the query not in the base keeps its own row
