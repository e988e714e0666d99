"""GPU (-m gpu): the row-sharded retrieval step (ShardedKnowledgeBase.retrieve2) on two ranks, each
against retrieval.retrieve2 on a full copy of both bases on its own GPU: D, I and the gathered rows
bit for bit, pools within 2e-6 of a float64 pool recomputed from the returned D and rows, mean pools
bit for bit against the emulation of the latency re-rank's summation order (oracle/pool_exact.py) and
softmax pools within that module's bound. Covers IP /
L2, k = 16 / 64, pool modes 0 / 1 / 2, perm_img, exclusion (own rows, E = 1; E = 8), two passes
(more than 16,384 queries), the exact fallback, an exact-only tiny shard, an empty shard, consecutive
steps, a strict sub-range of query rows, re-attachment after an add, the refusal when rows changed
without one, and ShardedIndex.search with exclusion against GpuIndexFlat.search.

With two GPUs the ranks form an NCCL group, one GPU each. With one GPU both ranks (two processes)
share it over a gloo group: every multi-rank path still runs -- both databases' peer pushes into
the other process's buffer, the cudaIpc mapping of the other rank's rows, the owner lookup over two
shards, the stand-alone push of an empty shard and the two merges on one set of flags -- only the
bytes do not cross NVLink. scripts/test_sharded_retrieve2_multigpu.py runs the same cases on every
GPU of a box."""
import os
import socket
import traceback

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu

D = 768


def unit(n, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, D, generator=g)
    return x / x.norm(dim=1, keepdim=True)


def pool_ref(Dv, Iv, feat, perm, mode, tau, l2):
    """float64 pool of rows [b] from the returned D / I and gathered (permuted) rows."""
    Dv, valid, feat = Dv.double(), Iv >= 0, feat.double()
    k = Dv.shape[1]
    if mode == 1:
        w = torch.full_like(Dv, 1.0 / k)
    else:
        z = torch.where(valid, (-tau if l2 else tau) * Dv, torch.full_like(Dv, -float("inf")))
        w = torch.nan_to_num(torch.softmax(z, dim=1), nan=0.0)
    if perm is not None:
        w = w[:, perm.long().to(w.device)]
    return (w[:, :, None] * feat).sum(1)


class Case:
    def __init__(self, rank, world, dev):
        self.rank, self.world, self.dev = rank, world, dev

    def kb(self, img, txt, metric):
        from keds_b200.index import GpuIndexFlat
        from keds_b200.sharded import ShardedKnowledgeBase

        kb = ShardedKnowledgeBase(D, metric, device=self.dev.index)
        kb.add(img, txt)
        self.rows = {"img": img.to(self.dev), "txt": txt.to(self.dev)}
        refs = []
        for x in (img, txt):
            r = GpuIndexFlat(D, metric, self.dev.index)
            if x.shape[0]:
                r.add(x)
            refs.append(r)
        return kb, refs

    def check(self, kb, refs, q, k, perm=None, pool_mode=0, ex=None, flags=0, tau=50.0, rows=None, out=None):
        from keds_b200 import retrieval as kr
        from oracle import pool_exact as pe

        Bt = q.shape[0]
        lo, hi = rows if rows is not None else (self.rank * Bt // self.world, (self.rank + 1) * Bt // self.world)
        q = q.to(self.dev)
        exd = None if ex is None else ex.to(self.dev)
        out = kb.retrieve2(q, k, perm_img=perm, pool_mode=pool_mode, tau=tau, flags=flags, exclude=exd, rows=(lo, hi),
                           out=out)
        kb.exchange_stats()  # synchronises; raises if a peer never delivered
        l2 = kb.metric_type == 1
        if refs[0].ntotal == 0:
            fmax = torch.finfo(torch.float32).max
            pad = torch.full((Bt, k), fmax if l2 else -fmax, device=self.dev)
            ref = {"D_img": pad, "D_txt": pad, "I_img": torch.full((Bt, k), -1, device=self.dev),
                   "I_txt": torch.full((Bt, k), -1, device=self.dev),
                   "feat_img": torch.zeros(Bt, k, D, device=self.dev), "feat_txt": torch.zeros(Bt, k, D, device=self.dev)}
        else:
            ref = kr.retrieve2(refs[0], refs[1], q, k, perm_img=perm, want_feats=True, pool_mode=0, flags=flags,
                               exclude=exd)
        torch.cuda.synchronize(self.dev)
        for s in ("img", "txt"):
            assert torch.equal(out["I_" + s], ref["I_" + s]), s
            assert torch.equal(out["D_" + s].view(torch.int32), ref["D_" + s].view(torch.int32)), s
            assert torch.equal(out["feat_" + s].view(torch.int32), ref["feat_" + s][lo:hi].view(torch.int32)), s
            if ex is not None:
                I = out["I_" + s].cpu()
                assert not ((I[:, :, None] == ex[:, None, :]) & (ex[:, None, :] >= 0)).any()
            if pool_mode and hi > lo:
                p = pool_ref(out["D_" + s][lo:hi], out["I_" + s][lo:hi], out["feat_" + s],
                             perm if s == "img" else None, pool_mode, tau, l2)
                err = (out["pool_" + s].double() - p).abs().max().item()
                assert err <= 2e-6, (s, err)
                # k_shard_consume sums in the latency re-rank's order (8 warps, two rows in flight), on
                # any shard count: mean pools bit for bit, softmax pools within the bound of D
                rows_s, I_s = self.rows[s], out["I_" + s][lo:hi]
                ps = perm if s == "img" else None
                if pool_mode == 1:
                    want = pe.mean_pool(rows_s, I_s, ps, *pe.SHARD)
                    assert bool(pe.equal_rows(out["pool_" + s], want).all()), ("mean pool bits", s)
                else:
                    p64, bound = pe.softmax_pool_bound(rows_s, I_s, out["D_" + s][lo:hi], ps, tau, l2, 8)
                    assert bool(((out["pool_" + s].double() - p64).abs() <= bound).all()), ("softmax bound", s)
        return out


def run_cases(rank, world, dev):
    from keds_b200.index import METRIC_INNER_PRODUCT as IP, METRIC_L2 as L2

    c = Case(rank, world, dev)
    N = 20000
    img, txt = unit(N, 1), unit(N, 2)
    g = torch.Generator().manual_seed(3)
    perm16 = torch.randperm(16, generator=g)
    for metric in (IP, L2):
        kb, refs = c.kb(img, txt, metric)
        # three consecutive steps (both exchange parities), k = 16 and 64, every pool mode
        c.check(kb, refs, unit(128 * world, 10 + metric), 16, perm=perm16, pool_mode=2)
        c.check(kb, refs, unit(128 * world, 20 + metric), 64, pool_mode=1)
        c.check(kb, refs, unit(128 * world, 30 + metric), 16, perm=perm16, pool_mode=0)
        # exclusion: queries near their own rows, E = 1 and E = 8
        sel = torch.randperm(N, generator=g)[:128 * world]
        q = img[sel] + 0.01 * unit(128 * world, 40)
        q = q / q.norm(dim=1, keepdim=True)
        c.check(kb, refs, q, 16, perm=perm16, pool_mode=2, ex=sel[:, None].clone())
        ex8 = torch.cat([sel[:, None], torch.randint(0, N, (sel.numel(), 6), generator=g),
                         torch.full((sel.numel(), 1), -1)], 1)
        c.check(kb, refs, q, 16, pool_mode=1, ex=ex8)
        # out= with column slices of wider buffers: replaced by dense tensors, the buffers untouched
        nb = 128                                # this rank's block of the 128 * world queries
        wide_p = torch.full((nb, 2 * D), 7.0, device=dev)
        wide_f = torch.full((nb, 16, 2 * D), 7.0, device=dev)
        o = {"pool_img": wide_p[:, D:], "feat_txt": wide_f[:, :, :D]}
        assert c.check(kb, refs, unit(128 * world, 44), 16, perm=perm16, pool_mode=1, out=o) is o
        assert (wide_p == 7.0).all() and (wide_f == 7.0).all() and o["pool_img"].is_contiguous()
        # a strict sub-range of rows, different on each rank
        c.check(kb, refs, unit(128 * world, 45), 16, perm=perm16, pool_mode=2, rows=(37 + 5 * rank, 101 + 3 * rank))
        # the bare sharded search with exclusion against GpuIndexFlat.search on a full copy
        for ex in (sel[:, None].clone(), ex8):
            qd, exd = q.to(dev), ex.to(dev)
            Ds, Is = kb.image.search(qd, 16, exclude=exd)
            Dr, Ir = refs[0].search(qd, 16, exclude=exd)
            torch.cuda.synchronize(dev)
            assert torch.equal(Is, Ir) and torch.equal(Ds.view(torch.int32), Dr.view(torch.int32))
        # the exact fallback answers every query
        for ix in (kb.image.local, kb.text.local):
            ix.set_eps_scale(1e4)
        c.check(kb, refs, unit(128 * world, 50), 16, perm=perm16, pool_mode=2)
        for ix in (kb.image.local, kb.text.local):
            ix.set_eps_scale(1.0)
    # more than 16,384 queries: two passes, only the last one publishes
    kb, refs = c.kb(img, txt, IP)
    c.check(kb, refs, unit(16384 + 300, 60), 16, perm=perm16, pool_mode=2, ex=torch.randint(-1, N, (16684, 2), generator=g))
    # a new set of rows after a step: add_local re-attaches; changing rows without it is refused
    img2, txt2 = unit(N // 2, 70), unit(N // 2, 71)
    for ix in (kb.image, kb.text):
        ix.local.reset()
    kb.add(img2, txt2)
    _, refs2 = c.kb(img2, txt2, IP)
    c.check(kb, refs2, unit(128 * world, 72), 16, pool_mode=2)
    kb.image.local.add(unit(10, 73).to(dev))
    with pytest.raises(RuntimeError, match="changed since"):
        kb.retrieve2(unit(128 * world, 74).to(dev), 16, rows=(0, 1))
    # an exact-only tiny shard (fewer rows than one tile) and an empty shard (N = world - 1)
    for n in (100, world - 1):
        for metric in (IP, L2):
            kb, refs = c.kb(img[:n], txt[:n], metric)
            c.check(kb, refs, unit(64 * world, 80 + n), 16, perm=perm16, pool_mode=2)
            c.check(kb, refs, unit(64 * world, 90 + n), 16, pool_mode=1)


def init_ranks(rank, world):
    """One GPU per rank over NCCL when there are enough GPUs, otherwise ranks share GPUs over gloo
    (the step itself needs no collective library; gloo carries the attach and barrier calls)."""
    n_dev = torch.cuda.device_count()
    dev = torch.device("cuda", rank % n_dev)
    torch.cuda.set_device(dev)
    if n_dev >= world:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    else:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    return dev


def _worker(rank, world, port, errs):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = init_ranks(rank, world)
    try:
        run_cases(rank, world, dev)
    except BaseException:
        errs[rank] = traceback.format_exc()
        raise
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_sharded_retrieve2_equals_unsharded():
    world = 2
    mgr = mp.Manager()
    errs = mgr.dict()
    try:
        mp.spawn(_worker, args=(world, _free_port(), errs), nprocs=world, join=True)
    finally:
        assert not dict(errs), "\n".join(dict(errs).values())
