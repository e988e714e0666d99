"""CPU: search with exclusion -- the exclusion reference (the oracle's search for k + E rows with
the excluded labels dropped) against a brute-force argsort, the Python argument checks,
KnowledgeBase.rows_of, the exported C surface, and a spill-free sm_100a compile."""
import ctypes as C

import numpy as np
import pytest
import torch

from keds_b200 import _capi
from keds_b200.index import check_exclude
from keds_b200.retrieval import KnowledgeBase
from oracle import knn_oracle

FLT_MAX = np.finfo(np.float32).max


def search_excluding(db, q, k, metric, exclude):
    """Exact float64 search over the rows each query does not exclude, built on the unchanged
    oracle: search k + E rows, drop the excluded labels (at most E of them), keep the first k.
    Padding (-1) is never an excluded label, so short results stay padded as the search pads."""
    ex = np.asarray(exclude, np.int64).reshape(q.shape[0], -1)
    D, I = knn_oracle.search(db, q, k + ex.shape[1], metric)
    gone = ((I[:, :, None] == ex[:, None, :]) & (ex[:, None, :] >= 0)).any(2)
    order = np.argsort(gone, axis=1, kind="stable")[:, :k]
    return np.take_along_axis(D, order, 1), np.take_along_axis(I, order, 1)


def brute(db, q, k, metric, exclude):
    """Per query: drop the excluded rows, argsort everything else by (score desc, row asc)."""
    db64, q64 = db.astype(np.float64), q.astype(np.float64)
    B, N = q.shape[0], db.shape[0]
    D = np.full((B, k), -FLT_MAX if metric == "ip" else FLT_MAX, np.float32)
    I = np.full((B, k), -1, np.int64)
    for b in range(B):
        keep = np.setdiff1d(np.arange(N), exclude[b])
        if metric == "ip":
            s = db64[keep] @ q64[b]
        else:
            s = -np.maximum((q64[b] @ q64[b]) + (db64[keep] ** 2).sum(1) - 2.0 * (db64[keep] @ q64[b]), 0.0)
        order = np.lexsort((keep, -s))[:k]
        I[b, :len(order)] = keep[order]
        D[b, :len(order)] = (s[order] if metric == "ip" else -s[order]).astype(np.float32)
    return D, I


@pytest.mark.parametrize("metric", ["ip", "l2"])
@pytest.mark.parametrize("N,k", [(300, 10), (12, 10), (5, 10)])
def test_exclusion_reference_matches_bruteforce(metric, N, k):
    rng = np.random.default_rng(N + k)
    db = rng.standard_normal((N, 16)).astype(np.float32)
    db[N // 2] = db[0]  # an exact duplicate row: ties broken by the lower row
    q = np.concatenate([db[:4], rng.standard_normal((6, 16)).astype(np.float32)])
    E = 3
    ex = rng.integers(-1, N + 3, size=(q.shape[0], E)).astype(np.int64)
    ex[:4, 0] = np.arange(4)  # queries that are rows of the base leave themselves out
    ex[1, 1] = ex[1, 0]       # a repeated label
    D, I = search_excluding(db, q, k, metric, ex)
    Db, Ib = brute(db, q, k, metric, [e[(e >= 0) & (e < N)] for e in ex])
    np.testing.assert_array_equal(I, Ib)
    np.testing.assert_allclose(D, Db, rtol=1e-6, atol=1e-6)
    for b in range(q.shape[0]):
        assert not set(I[b].tolist()) & set(ex[b][ex[b] >= 0].tolist())


def test_exclusion_reference_without_labels_is_the_plain_search():
    rng = np.random.default_rng(1)
    db = rng.standard_normal((200, 8)).astype(np.float32)
    q = rng.standard_normal((7, 8)).astype(np.float32)
    for metric in ("ip", "l2"):
        D0, I0 = knn_oracle.search(db, q, 9, metric)
        D1, I1 = search_excluding(db, q, 9, metric, np.full((7, 2), -1, np.int64))
        np.testing.assert_array_equal(I0, I1)
        np.testing.assert_array_equal(D0, D1)


def test_check_exclude_shapes():
    assert check_exclude(np.arange(5, dtype=np.int64), 5).shape == (5, 1)
    assert check_exclude(np.zeros((5, 8), np.int64), 5).shape == (5, 8)
    t = check_exclude(torch.zeros(4, 3, dtype=torch.int64), 4)
    assert isinstance(t, torch.Tensor) and t.shape == (4, 3)


@pytest.mark.parametrize("bad,err", [
    (np.zeros(5, np.int32), TypeError),
    (np.zeros(5, np.float64), TypeError),
    (torch.zeros(5, dtype=torch.int32), TypeError),
    ([0, 1, 2, 3, 4], TypeError),
    (np.zeros(4, np.int64), ValueError),
    (np.zeros((5, 9), np.int64), ValueError),
    (np.zeros((5, 0), np.int64), ValueError),
    (np.zeros((5, 1, 1), np.int64), ValueError),
])
def test_check_exclude_rejects(bad, err):
    with pytest.raises(err):
        check_exclude(bad, 5)


def kb_with_names(names):
    kb = KnowledgeBase.__new__(KnowledgeBase)  # the name table needs no device index
    kb.basenames = list(names)
    return kb


def test_rows_of():
    kb = kb_with_names(["a.jpg", "b.jpg", "c.jpg", "b.jpg"])
    r = kb.rows_of(["c.jpg", "zz", "a.jpg", "b.jpg"])
    assert r.dtype == torch.int64 and r.tolist() == [2, -1, 0, 1]
    assert kb.rows_of([]).tolist() == []
    table = kb._row_table
    kb.rows_of(["a.jpg"])
    assert kb._row_table is table  # built once per basenames list
    kb.basenames = ["x", "a.jpg"]
    assert kb.rows_of(["a.jpg", "c.jpg"]).tolist() == [1, -1]


def test_search_calls_take_exclusion_arguments():
    """Every search call with exclusion is exported and takes (exclude, n_exclude) as (pointer, int)."""
    lib = _capi.load()
    for name, at in (("keds_index_search_ex", 6), ("keds_index_search2", 9), ("keds_retrieve2", 21),
                     ("keds_index_search_sharded", 7), ("keds_retrieve2_sharded", 20)):
        assert hasattr(lib, name)
        assert _capi.SIGNATURES[name][1][at:at + 2] == [C.c_void_p, C.c_int], name


def test_search_calls_refuse_bad_exclusion_without_a_gpu():
    lib = _capi.load()
    ex = np.zeros((1, 1), np.int64)
    # a null array with n_exclude != 0, or an array with n_exclude outside 1..8, is refused before anything else
    for e, n in ((None, 1), (ex.ctypes.data, 0), (ex.ctypes.data, 9)):
        assert lib.keds_index_search_ex(None, None, 1, 1, None, None, e, n, 0, None) == -1
        assert "exclude" in _capi.last_error()
        assert lib.keds_index_search2(None, None, None, 1, 1, None, None, None, None, e, n, 0, None) == -1
        assert "exclude" in _capi.last_error()
        assert lib.keds_retrieve2(None, None, None, 1, 16, None, None, 0, 1.0, None, None, None, None, None, None, None,
                                  None, None, None, None, None, e, n, 0, None) == -1
        assert "exclude" in _capi.last_error()


def test_scoring_and_fallback_kernels_do_not_spill(tmp_path):
    """sm_100a compile with -Xptxas -v: every k_score_topk instantiation (with and without
    exclusion) and k_exact_fallback keep their registers -- no spill stores or loads."""
    import re
    import subprocess

    from keds_b200 import build as kbuild

    nvcc = kbuild.find_nvcc()
    if nvcc is None:
        pytest.skip("nvcc not available")
    res = subprocess.run([nvcc, *kbuild.NVCC_FLAGS, "-Xptxas", "-v", "-o", str(tmp_path / "lib.so"), kbuild.SRC],
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-2000:]
    stats, cur = {}, None
    for line in res.stderr.splitlines():
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            cur = m.group(1)
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur and ("k_score_topk" in cur or "k_exact_fallback" in cur):
            stats[cur] = (int(m.group(1)), int(m.group(2)))
    assert sum("k_score_topk" in k for k in stats) == 6 and any("k_exact_fallback" in k for k in stats), stats
    assert all(v == (0, 0) for v in stats.values()), stats
