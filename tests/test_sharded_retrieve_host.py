"""CPU: the row-sharded retrieval step's host side. Argument checks of ShardedKnowledgeBase.retrieve2,
the DDP block arithmetic (unequal batches), the all-gather plumbing of get_retrieved_features on a
gloo world of two with stand-ins for the local indices and the native step, the new C entry points'
refusals without a GPU, and a spill-free sm_100a compile of the kernels the step runs."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from keds_b200 import _capi
from keds_b200.sharded import ShardedKnowledgeBase, rank_block
from oracle import knn_oracle as orc

D = 16


class OracleLocal:
    def __init__(self):
        self.base = np.zeros((0, D), np.float32)

    def set_id_offset(self, off):
        pass

    def add(self, x):
        self.base = np.asarray(x, np.float32)


def search_excluding(db, q, k, metric, ex):
    """The oracle's search for k + E rows with each query's excluded labels dropped."""
    if ex is None:
        return orc.search(db, q, k, metric)
    ex = np.asarray(ex, np.int64).reshape(q.shape[0], -1)
    D1, I1 = orc.search(db, q, k + ex.shape[1], metric)
    gone = ((I1[:, :, None] == ex[:, None, :]) & (ex[:, None, :] >= 0)).any(2)
    order = np.argsort(gone, axis=1, kind="stable")[:, :k]
    return np.take_along_axis(D1, order, 1), np.take_along_axis(I1, order, 1)


def fake_step(img, txt, metric, seen):
    """Stand-in for the native sharded step: the full-base answer for the gathered queries, the
    gathered rows of the requested block only."""
    def run(q, k, perm_img, perm_txt, want_feats, pool_mode, tau, flags, ex, rows):
        seen.append((tuple(q.shape), None if ex is None else tuple(ex.shape), rows))
        lo, hi = rows
        out = {}
        for name, db, perm in (("img", img, perm_img), ("txt", txt, perm_txt)):
            _, I = search_excluding(db, q.numpy(), k, metric, None if ex is None else ex.numpy())
            f = db[I[lo:hi]]
            if perm is not None:
                f = f[:, perm.long().numpy()]
            out["feat_" + name] = torch.from_numpy(np.ascontiguousarray(f))
        return out
    return run


def _init_single(tmp_path):
    dist.init_process_group("gloo", init_method=f"file://{tmp_path}/store", rank=0, world_size=1)


def test_rank_block_arithmetic():
    assert rank_block([128, 128], 1) == (128, 128, 256)
    # unequal last batches: pad to the largest, each rank keeps its own rows of its block
    assert rank_block([5, 3], 0) == (5, 0, 5)
    assert rank_block([5, 3], 1) == (5, 5, 8)
    assert rank_block([2, 7, 0], 2) == (7, 14, 14)
    with pytest.raises(ValueError):
        rank_block([4, 4], 2)
    with pytest.raises(ValueError):
        rank_block([4, -1], 0)


def test_retrieve2_argument_checks(tmp_path):
    _init_single(tmp_path)
    try:
        with pytest.raises(ValueError, match="fused"):
            ShardedKnowledgeBase(D, 0, exchange="nccl", _local_index=OracleLocal)
        calls = []
        kb = ShardedKnowledgeBase(D, 0, _local_index=OracleLocal, _retrieve=lambda *a: calls.append(a) or {})
        q = torch.zeros(6, D)
        bad = [
            (TypeError, dict(q=q.double())),
            (TypeError, dict(q=torch.zeros(6, D + 1))),
            (TypeError, dict(q=torch.zeros(D))),
            (ValueError, dict(q=torch.zeros(0, D))),
            (ValueError, dict(k=0)),
            (ValueError, dict(k=1025)),
            (ValueError, dict(pool_mode=3)),
            (ValueError, dict(rows=(4, 2))),
            (ValueError, dict(rows=(0, 7))),
            (ValueError, dict(rows=(-1, 2))),
            (TypeError, dict(perm_img=torch.arange(5))),
            (TypeError, dict(perm_txt=torch.zeros(4, dtype=torch.float32))),
            (ValueError, dict(perm_img=torch.tensor([0, 0, 1, 2]))),     # not a permutation
            (ValueError, dict(perm_txt=torch.tensor([0, 1, 2, 4]))),
            (TypeError, dict(exclude=torch.zeros(6, dtype=torch.int32))),
            (ValueError, dict(exclude=torch.zeros(5, 1, dtype=torch.int64))),
            (ValueError, dict(exclude=torch.zeros(6, 9, dtype=torch.int64))),
        ]
        for err, kw in bad:
            args = dict(q=q, k=4)
            args.update(kw)
            with pytest.raises(err):
                kb.retrieve2(args.pop("q"), **args)
        assert not calls  # nothing reached the step
        kb.retrieve2(q, 4, perm_img=torch.tensor([3, 2, 1, 0]), exclude=torch.full((6, 2), -1, dtype=torch.int64),
                     rows=(2, 5))
        (a,) = calls
        assert a[1] == 4 and a[2].dtype == torch.int32 and a[8].shape == (6, 2) and a[9] == (2, 5)
    finally:
        dist.destroy_process_group()


def _worker(rank, world, port, metric, use_exclude, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from keds_b200.retrieval import get_retrieved_features

        rng = np.random.default_rng(11)
        img = rng.standard_normal((40, D)).astype(np.float32)
        txt = rng.standard_normal((40, D)).astype(np.float32)
        seen = []
        kb = ShardedKnowledgeBase(D, 1 if metric == "l2" else 0, _local_index=OracleLocal,
                                  _retrieve=fake_step(img, txt, metric, seen))
        kb.add(img, txt)
        B = (5, 3)[rank]  # unequal batches
        feat = torch.from_numpy(rng.standard_normal((8, D)).astype(np.float32))[rank * 5:rank * 5 + B]
        ex = None
        if use_exclude and rank == 0:  # only one rank excludes: the other's rows are padded with -1
            ex = torch.arange(B, dtype=torch.int64) + 7
        torch.manual_seed(100 + rank)
        fi, ft = get_retrieved_features(feat, (img, txt, [], kb.image, kb.text), topk=4, exclude=ex)
        torch.manual_seed(100 + rank)
        perm = torch.randperm(4).numpy()
        qn = (feat / feat.norm(dim=1, keepdim=True)).numpy()
        _, Ii = search_excluding(img, qn, 4, metric, None if ex is None else ex.numpy())
        _, It = search_excluding(txt, qn, 4, metric, None if ex is None else ex.numpy())
        ok = (tuple(fi.shape) == (B, 4, D) and np.array_equal(fi.numpy(), img[Ii][:, perm])
              and np.array_equal(ft.numpy(), txt[It]))
        lo = rank * 5
        ok = ok and seen == [((10, D), (10, 1) if use_exclude else None, (lo, lo + B))]
        ok = ok and (kb.image.lo, kb.image.hi) == ((0, 20), (20, 40))[rank]
        out[rank] = bool(ok)
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("metric,use_exclude", [("ip", False), ("l2", True)])
def test_get_retrieved_features_gathers_pads_and_returns_own_block(metric, use_exclude):
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(2, _free_port(), metric, use_exclude, out), nprocs=2, join=True)
    assert out.get(0) is True and out.get(1) is True, dict(out)


def test_sharded_calls_refuse_bad_arguments_and_exclusion_without_a_gpu():
    lib = _capi.load()
    for name in ("keds_retrieve2_sharded", "keds_index_search_sharded", "keds_index_rows_ipc",
                 "keds_exchange_attach_rows"):
        assert name in _capi.SIGNATURES and hasattr(lib, name)
    assert lib.keds_retrieve2_sharded(None, None, None, None, 1, 16, None, None, 0, 1.0, 0, 1, None, None, None, None,
                                      None, None, None, None, None, 0, 0, None) == -1
    assert lib.keds_index_search_sharded(None, None, None, 1, 1, None, None, None, 0, None) == -1
    # exclusion arrays: a null array with n_exclude != 0, or n_exclude outside 1..8, are refused first
    ex = np.zeros((1, 1), np.int64)
    for e, n in ((None, 1), (ex.ctypes.data, 0), (ex.ctypes.data, 9)):
        assert lib.keds_retrieve2_sharded(None, None, None, None, 1, 16, None, None, 0, 1.0, 0, 1, None, None, None,
                                          None, None, None, None, None, e, n, 0, None) == -1
        assert "exclude" in _capi.last_error()
        assert lib.keds_index_search_sharded(None, None, None, 1, 1, None, None, e, n, None) == -1
        assert "exclude" in _capi.last_error()
    assert lib.keds_index_rows_ipc(None, None) == -1
    assert lib.keds_exchange_attach_rows(None, 0, None, None, None) == -1


def test_shard_consume_and_rerank_fallback_do_not_spill(tmp_path):
    """sm_100a compile with -Xptxas -v: k_shard_consume, k_exact_fallback and the latency re-rank
    keep their registers. (The two throughput re-rank variants spill a few words already at the
    parent of this change: registers are capped there for four and six blocks per SM.)"""
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
        if m and cur and any(s in cur for s in ("k_shard_consume", "k_exact_fallback", "k_select_rerankILi3ELi2E")):
            stats[cur] = (int(m.group(1)), int(m.group(2)))
    assert len(stats) == 3, stats
    assert all(v == (0, 0) for v in stats.values()), stats
