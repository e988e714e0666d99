"""GPU (-m gpu): the neighbour consumer (NeighbourConsumer, TrainableNeighbourConsumer) on row-sharded
bases, two ranks. Every rank holds a ShardedKnowledgeBase and full GpuIndexFlat copies of both
bases, and runs the same labels through the local route (rows from its own copy) and the sharded
route (rows read from their owners through the exchange's mapping). The two must agree bit for bit:
both copy the same fp32 rows into the MLP input, and every later kernel is the same launch on the
same shapes, with the split-K reductions in a fixed order.

Covers eval tokens (IP / L2, k = 16 / 64, with and without perm, labels with -1 padding from a
12-row base at k = 16 and with E = 8 exclusions, labels outside every shard, an empty shard),
from_features on the sharded base against from_features on an unsharded KnowledgeBase (unequal
batches 48 / 37, with and without exclusion), training forward + backward in train() (dropout) and
eval() (tokens and flat.grad), a step and a search of one base that grow the knowledge base's one
exchange before a consumer call, and the refusals: rows changed without a re-attach, a mixed or
foreign index pair, a width mismatch, a base that has run no step.

The harness is that of test_gpu_sharded_retrieve.py: two GPUs over NCCL, or two processes sharing
one GPU over gloo (peer reads then go through the cudaIpc mapping of the other process, on the same
device). scripts/test_sharded_consumer_multigpu.py runs these cases on every GPU of a box. The test
took 11 s on one NVIDIA B200 at a 1000 W power limit (two processes, gloo)."""
import os
import socket
import traceback

import numpy as np
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


def raw(n, seed):
    """un-normalised query features, as img2text sees them"""
    return 3.0 * torch.randn(n, D, generator=torch.Generator().manual_seed(seed))


def same_bits(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def state_dicts(d_in=D, d_mid=512, d_tok=D, n_hidden=2, n_layers=3, heads=8, dim_head=64, seed=5):
    from oracle import consumer_oracle as corc

    sds = corc.random_state_dicts(d_in, d_mid, d_tok, n_hidden, n_layers, heads, dim_head, seed=seed)
    return [{k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in sd.items()} for sd in sds]


class Case:
    def __init__(self, rank, world, dev):
        from keds_b200.consumer import NeighbourConsumer, TrainableNeighbourConsumer

        self.rank, self.world, self.dev = rank, world, dev
        sds = state_dicts()
        self.cons_l = NeighbourConsumer(*sds, heads=8, device=dev.index)
        self.cons_s = NeighbourConsumer(*sds, heads=8, device=dev.index)
        self.train_l = TrainableNeighbourConsumer(*sds, heads=8, device=dev.index, dropout=0.1)
        self.train_s = TrainableNeighbourConsumer(*sds, heads=8, device=dev.index, dropout=0.1)

    def kb(self, img, txt, metric):
        from keds_b200.index import GpuIndexFlat
        from keds_b200.sharded import ShardedKnowledgeBase

        # the caller drops its previous base after this: no rank may still be reading its rows
        torch.cuda.synchronize(self.dev)
        dist.barrier()
        kb = ShardedKnowledgeBase(D, metric, device=self.dev.index)
        kb.add(img, txt)
        refs = []
        for x in (img, txt):
            r = GpuIndexFlat(D, metric, self.dev.index)
            if x.shape[0]:
                r.add(x)
            refs.append(r)
        return kb, refs

    def labels(self, kb, q, k, ex=None):
        """this rank's rows of the merged labels of one sharded step (no feature gathers)"""
        Bt = q.shape[0]
        lo, hi = self.rank * Bt // self.world, (self.rank + 1) * Bt // self.world
        out = kb.retrieve2(q.to(self.dev), k, want_feats=False, exclude=None if ex is None else ex.to(self.dev),
                           rows=(lo, hi))
        return out["I_img"][lo:hi], out["I_txt"][lo:hi]

    def eval_tokens(self, kb, refs, I_img, I_txt, perm, seed):
        feat = raw(I_img.shape[0], seed).to(self.dev)
        a = self.cons_l(feat, refs[0], refs[1], I_img, I_txt, perm)
        b = self.cons_s(feat, kb.image, kb.text, I_img, I_txt, perm)
        self.cons_s.check()
        torch.cuda.synchronize(self.dev)
        assert same_bits(a, b), ("eval tokens", I_img.shape, perm is not None)
        return a

    def training(self, kb, refs, I_img, I_txt, perm, seed):
        feat = raw(I_img.shape[0], seed).to(self.dev)
        for mode in (True, False):
            res = []
            for m, pair in ((self.train_l, refs), (self.train_s, (kb.image, kb.text))):
                m.train(mode)
                m.flat.grad = None
                torch.manual_seed(seed)  # the same dropout masks on both routes
                tok = m(feat, pair[0], pair[1], I_img, I_txt, perm)
                g = torch.randn(tok.shape, generator=torch.Generator().manual_seed(seed + 1)).to(self.dev)
                tok.backward(g)
                res.append((tok.detach(), m.flat.grad.clone()))
            torch.cuda.synchronize(self.dev)
            assert same_bits(res[0][0], res[1][0]), ("train tokens", mode)
            assert same_bits(res[0][1], res[1][1]), ("flat.grad", mode)

    def from_features(self, kb, img, txt, metric, exclude):
        from keds_b200.retrieval import KnowledgeBase

        sizes = [48 if r % 2 == 0 else 37 for r in range(self.world)]  # unequal batches
        B, lo = sizes[self.rank], sum(sizes[:self.rank])
        g = torch.Generator().manual_seed(200)
        sel = torch.randperm(img.shape[0], generator=g)[:sum(sizes)]
        feat = 2.0 * img[sel] + 0.05 * torch.randn(sum(sizes), D, generator=g)
        feat, own = feat[lo:lo + B].to(self.dev), sel[lo:lo + B]
        ex = own.clone() if exclude else None
        ukb = KnowledgeBase(img, txt, [str(i) for i in range(img.shape[0])], device=self.dev.index, metric=metric)
        torch.manual_seed(300 + self.rank)
        want = self.cons_l.from_features(feat, ukb, topk=16, exclude=ex)
        torch.manual_seed(300 + self.rank)
        got = self.cons_s.from_features(feat, kb, topk=16, exclude=ex)
        torch.manual_seed(300 + self.rank)
        got_seq = self.cons_s.from_features(feat, (None, None, None, kb.image, kb.text), topk=16, exclude=ex)
        torch.cuda.synchronize(self.dev)
        assert got.shape == (B, 3, D)
        assert same_bits(want, got) and same_bits(want, got_seq), ("from_features", metric, exclude)


def run_cases(rank, world, dev):
    from keds_b200.index import METRIC_INNER_PRODUCT as IP, METRIC_L2 as L2

    c = Case(rank, world, dev)
    N = 20000
    img, txt = unit(N, 1), unit(N, 2)
    g = torch.Generator().manual_seed(3)
    perm16, perm64 = torch.randperm(16, generator=g), torch.randperm(64, generator=g)
    for metric in (IP, L2):
        kb, refs = c.kb(img, txt, metric)
        for k, perm in ((16, perm16), (16, None), (64, perm64)):
            I_img, I_txt = c.labels(kb, unit(128 * world, 10 + k + metric), k)
            c.eval_tokens(kb, refs, I_img, I_txt, perm, 20 + k)
        # labels no shard holds (-1, past the end) read as zero rows on both routes
        I_any = torch.randint(-1, N + 50, (64, 16), generator=g).to(dev)
        c.eval_tokens(kb, refs, I_any, I_any.flip(0), perm16, 30)
        c.from_features(kb, img, txt, metric, exclude=False)
        c.from_features(kb, img, txt, metric, exclude=True)
    # training, forward + backward, on the IP base of the last loop's labels shape
    kb, refs = c.kb(img, txt, IP)
    I_img, I_txt = c.labels(kb, unit(64 * world, 40), 16)
    c.training(kb, refs, I_img, I_txt, perm16.to(torch.int32), 41)
    c.training(kb, refs, I_img, I_txt, None, 42)
    # a step that grows the exchange (2 * Bt * k above its 16,384 entries): new buffers, rows re-attached
    I_img, I_txt = c.labels(kb, unit(16 * world, 50), 16)
    c.eval_tokens(kb, refs, I_img, I_txt, perm16, 51)
    cap = kb._fx.capacity
    I_img, I_txt = c.labels(kb, unit(640 * world, 52), 16)
    assert kb._fx.capacity > cap
    c.eval_tokens(kb, refs, I_img, I_txt, perm16, 53)
    c.training(kb, refs, I_img[:96], I_txt[:96], perm16, 54)
    # a search of one base that outgrows the exchange grows the knowledge base's one exchange
    cap = kb._fx.capacity
    q = unit(cap // 16 + 1, 55).to(dev)
    Ds, Is = kb.image.search(q, 16)
    Dr, Ir = refs[0].search(q, 16)
    assert same_bits(Ds, Dr) and torch.equal(Is, Ir)
    assert kb._fx.capacity > cap and kb.image._fx is kb.text._fx is kb._fx
    I_img, I_txt = c.labels(kb, unit(16 * world, 56), 16)
    c.eval_tokens(kb, refs, I_img, I_txt, perm16, 57)
    # -1 padding: k above the rows of a 12-row base, and E = 8 exclusions on it; an empty shard
    for n in (12, world - 1):
        for metric in (IP, L2):
            kb, refs = c.kb(img[:n], txt[:n], metric)
            I_img, I_txt = c.labels(kb, unit(32 * world, 60 + n), 16)
            assert bool((I_img < 0).any())
            c.eval_tokens(kb, refs, I_img, I_txt, perm16, 61)
            ex8 = torch.randint(-1, n, (32 * world, 8), generator=g)
            I_img, I_txt = c.labels(kb, unit(32 * world, 62 + n), 16, ex=ex8)
            c.eval_tokens(kb, refs, I_img, I_txt, None, 63)

    # ---- refusals
    from keds_b200.consumer import NeighbourConsumer, TrainableNeighbourConsumer

    kb, refs = c.kb(img, txt, IP)
    I_img, I_txt = c.labels(kb, unit(16 * world, 70), 16)
    feat = raw(I_img.shape[0], 71).to(dev)
    kb2, _ = c.kb(img[:100], txt[:100], IP)
    with pytest.raises(RuntimeError, match="retrieve2 first"):      # no step yet: no exchange
        c.cons_s(feat, kb2.image, kb2.text, I_img, I_txt)
    c.labels(kb2, unit(16 * world, 72), 16)
    for pair in ((kb.image, refs[1]), (refs[0], kb.text), (kb.image, kb2.text), (kb.text, kb.image)):
        with pytest.raises(TypeError):
            c.cons_s(feat, pair[0], pair[1], I_img, I_txt)
        with pytest.raises(TypeError):
            c.train_s(feat, pair[0], pair[1], I_img, I_txt)
    # width: the Python check of NeighbourConsumer, the native one behind TrainableNeighbourConsumer
    sds = state_dicts(256, 128, 256, 1, 1, 4, 32, seed=9)
    narrow, narrow_t = NeighbourConsumer(*sds, heads=4, device=dev.index), TrainableNeighbourConsumer(
        *sds, heads=4, device=dev.index)
    f256 = torch.randn(I_img.shape[0], 256, device=dev)
    with pytest.raises(ValueError, match="width"):
        narrow(f256, kb.image, kb.text, I_img, I_txt)
    with pytest.raises(RuntimeError, match="d_in"):
        narrow_t(f256, kb.image, kb.text, I_img, I_txt)
    # rows changed on this rank without a re-attach (every rank changes its own)
    kb.image.local.add(unit(10, 73).to(dev))
    with pytest.raises(RuntimeError, match="changed since"):
        c.cons_s(feat, kb.image, kb.text, I_img, I_txt)
    with pytest.raises(RuntimeError, match="changed since"):
        c.train_s(feat, kb.image, kb.text, I_img, I_txt)
    torch.cuda.synchronize(dev)
    dist.barrier()


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


def test_sharded_consumer_equals_local_consumer():
    world = 2
    mgr = mp.Manager()
    errs = mgr.dict()
    try:
        mp.spawn(_worker, args=(world, _free_port(), errs), nprocs=world, join=True)
    finally:
        assert not dict(errs), "\n".join(dict(errs).values())
