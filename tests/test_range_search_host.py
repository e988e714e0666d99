"""CPU: range search's host side -- the C entry points and their ctypes table, argument checks, the
index objects that refuse or split a range search, and the fp32 reference (oracle/fp32_exact.py)
against a brute-force filter of every emulated score."""
import ctypes as C

import numpy as np
import pytest
import torch

from keds_b200 import _capi
from keds_b200.index import METRIC_INNER_PRODUCT, GpuIndexFlat, IndexFlatIP, IndexFlatL2, IndexReplicas, IndexShards
from keds_b200.sharded import ShardedIndex
from oracle import fp32_exact as fx
from oracle import range_exact as rx


def test_entry_points_are_declared_and_bound():
    for name in ("keds_index_range_search", "keds_index_range_results"):
        assert name in _capi.SIGNATURES
        assert hasattr(_capi.load(), name)


def test_null_arguments_are_rejected():
    lib = _capi.load()
    lims = (C.c_int64 * 2)()
    assert lib.keds_index_range_search(None, None, 1, 0.5, lims, 0, None) == -1
    assert lib.keds_index_range_search(None, None, 0, 0.5, None, 0, None) == -1
    assert lib.keds_index_range_results(None, None, None, None) == -1


def test_cpu_index_has_no_range_search():
    for cls in (IndexFlatIP, IndexFlatL2):
        ix = cls(8)
        ix.add(np.ones((3, 8), np.float32))
        with pytest.raises(RuntimeError, match="no CPU search"):
            ix.range_search(np.ones((1, 8), np.float32), 0.5)


def test_sharded_indices_refuse():
    with pytest.raises(NotImplementedError, match="range_search"):
        IndexShards.__new__(IndexShards).range_search(np.ones((1, 8), np.float32), 0.5)
    with pytest.raises(NotImplementedError, match="range_search"):
        ShardedIndex.__new__(ShardedIndex).range_search(torch.ones(1, 8), 0.5)


class _NoLib:
    def __getattr__(self, name):
        raise AssertionError(f"{name} called for an argument that should have been refused")


def _unbound_index(d=8):
    ix = GpuIndexFlat.__new__(GpuIndexFlat)
    ix.d, ix.metric_type, ix.device, ix._lib, ix._h = d, METRIC_INNER_PRODUCT, 0, _NoLib(), None
    return ix


def test_query_validation_follows_search():
    ix = _unbound_index()
    with pytest.raises(TypeError):
        ix.range_search(np.ones((2, 8), np.float64), 0.5)
    with pytest.raises(AssertionError):
        ix.range_search(np.ones((2, 7), np.float32), 0.5)
    with pytest.raises(ValueError):
        ix.range_search(np.ones(8, np.float32), 0.5)
    with pytest.raises(ValueError, match="NaN"):
        ix.range_search(np.ones((2, 8), np.float32), float("nan"))


class _FakeReplica:
    """answers query i with i % 3 hits: labels 10 i + j, scores 1 / (j + 1)"""

    def __init__(self, first):
        self.first = first

    def range_search(self, x, radius):
        cnt = [(self.first + i) % 3 for i in range(x.shape[0])]
        lims = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64)
        I = np.array([10 * (self.first + i) + j for i, c in enumerate(cnt) for j in range(c)], np.int64)
        D = np.array([1.0 / (j + 1) for c in cnt for j in range(c)], np.float32)
        return lims, D, I


def test_replicas_concatenate_with_shifted_lims():
    rep = IndexReplicas.__new__(IndexReplicas)
    rep.d = 4
    rep.subs = [_FakeReplica(0), _FakeReplica(3)]  # the split of 7 queries over two replicas: [0, 3), [3, 7)
    lims, D, I = rep.range_search(np.zeros((7, 4), np.float32), 0.5)
    cnt = [i % 3 for i in range(7)]
    assert lims.tolist() == np.concatenate([[0], np.cumsum(cnt)]).tolist()
    assert I.tolist() == [10 * i + j for i in range(7) for j in range(cnt[i])]
    assert D.dtype == np.float32 and I.dtype == np.int64 and len(D) == lims[-1]


def brute(q, x, radius, metric, id_offset=0):
    s = fx.scores(q, x, metric).double()
    lims, Ds, Is = [0], [], []
    for i in range(q.shape[0]):
        row = s[i]
        hit = (row > radius) if metric == "ip" else (row < radius)
        ids = hit.nonzero().flatten()
        key = row[ids] if metric == "ip" else -row[ids]
        order = sorted(range(len(ids)), key=lambda t: (-float(key[t]), int(ids[t])))
        Ds += [float(row[ids[t]]) for t in order]
        Is += [int(ids[t]) + id_offset for t in order]
        lims.append(len(Is))
    return torch.tensor(lims), torch.tensor(Ds, dtype=torch.float32), torch.tensor(Is, dtype=torch.int64)


@pytest.mark.parametrize("metric", ["ip", "l2"])
@pytest.mark.parametrize("d", [64, 37])  # 37: the scalar lane order
def test_oracle_equals_brute_force(metric, d):
    g = torch.Generator().manual_seed(3)
    x = torch.randn(300, d, generator=g)
    x = x / x.norm(dim=1, keepdim=True)
    x = torch.cat([x, x[:40]])  # exact ties
    q = torch.randn(9, d, generator=g)
    q = q / q.norm(dim=1, keepdim=True)
    s = fx.scores(q, x, metric)
    for radius in (float(s[0].max()) + 1.0, float(s[0].kthvalue(300).values), float(s[1].median()),
                   float(s[2].kthvalue(5).values), -1e30 if metric == "ip" else 1e30):
        got = rx.range_search(q, x, radius, metric, id_offset=7)
        ref = brute(q, x, radius, metric, id_offset=7)
        assert torch.equal(got[0], ref[0])
        assert torch.equal(got[1].view(torch.int32), ref[1].view(torch.int32))
        assert torch.equal(got[2], ref[2])


def test_oracle_no_queries_or_rows():
    lims, D, I = rx.range_search(torch.zeros(0, 8), torch.zeros(5, 8), 0.1, "ip")
    assert lims.tolist() == [0] and D.numel() == 0 and I.numel() == 0
    lims, D, I = rx.range_search(torch.zeros(3, 8), torch.zeros(0, 8), 0.1, "l2")
    assert lims.tolist() == [0, 0, 0, 0] and D.numel() == 0


def test_range_scoring_kernel_does_not_spill(tmp_path):
    """sm_100a compile with -Xptxas -v: both k_score_range variants (the search's mainloop with the
    range epilogue) keep their registers -- no spill stores or loads."""
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
        if m and cur and "k_score_range" in cur:
            stats[cur] = (int(m.group(1)), int(m.group(2)))
    assert len(stats) == 2 and all(v == (0, 0) for v in stats.values()), stats
