"""Row-sharded knowledge database across the GPUs of one box: one process per GPU
(torch.distributed), every rank holds rows [lo_r, hi_r) and answers the full query batch locally
with exact fp32-re-ranked scores and GLOBAL labels; the [B, k] (score, label) blocks cross NVLink --
stored by the search kernels themselves into the peers' buffers (exchange="fused") or with one packed
NCCL all-gather (exchange="nccl") -- and a merge kernel gives every rank the global top-k.  The result is
bit-identical for 1, 2, 4 or 8 shards (same scores, same total order).

The reference has no such path (full replica per DDP rank: src/main.py:76,82; replicas in eval:
src/eval_retrieval.py:292,295).  The exchange is new and is the only collective on the path.

Test hooks `_local_index` / `_merge` let the CPU (gloo, world_size 2) tests drive the partition /
pack / all-gather / unpack logic with stand-ins; the product path always uses GpuIndexFlat and the
keds_topk_merge_strided kernel.
"""
from __future__ import annotations

from typing import Callable, Optional, Tuple

import numpy as np
import torch
import torch.distributed as dist

from . import _capi
from .index import GpuIndexFlat, _check_out, _exclude_arg, _exclude_ptrs, _stream_ptr
from .retrieval import _device_perm, _step_outputs, check_perm


def shard_bounds(n: int, world: int, rank: int) -> Tuple[int, int]:
    """rows [lo, hi) of shard `rank`: ceil(n / world) rows each, last shards may be short/empty."""
    per = -(-n // world) if world > 0 else n
    return min(n, rank * per), min(n, (rank + 1) * per)


def packed_layout(nq: int, k: int) -> Tuple[int, int, int]:
    """(bytes per rank, byte offset of the label block, bytes of the score block) of the exchange
    buffer: [nq*k float32 scores | pad to 8 | nq*k int64 labels]."""
    d_bytes = nq * k * 4
    off_i = (d_bytes + 7) // 8 * 8
    return off_i + nq * k * 8, off_i, d_bytes


def _exchange_name(exchange):
    return "fused" if exchange == "p2p" else exchange  # the fused exchange's former name


class _FusedExchange:
    """Symmetric (peer-mapped) receive buffers + the native exchange handle over them. The buffer
    is allocated with torch symmetric memory, so every rank holds raw pointers into every other
    rank's copy (NVLink P2P through NVSwitch); the library lays it out (flag words, two parities
    of one slot per rank) and never sees torch types. Symmetric memory needs one GPU per rank:
    ranks that share a GPU map each other's buffers with cudaIpc instead (torch's CUDA tensor
    sharing), which gives the library the same kind of peer pointers."""

    def __init__(self, world: int, rank: int, capacity: int, device: torch.device, group) -> None:
        import ctypes as C
        import torch.distributed._symmetric_memory as symm_mem

        lib = _capi.load()
        group = group if group is not None else dist.group.WORLD
        slot = -(-(12 * capacity) // 48) * 48
        total = (256 + 2 * world * slot + 255) // 256 * 256
        uuids = [None] * world
        dist.all_gather_object(uuids, str(torch.cuda.get_device_properties(device).uuid), group=group)
        self.hdl = None
        if len(set(uuids)) == world:
            self.buf = symm_mem.empty(total, dtype=torch.uint8, device=device)
            self.buf.zero_()
            torch.cuda.synchronize(device)
            self.hdl = symm_mem.rendezvous(self.buf, group)
            peers = [int(p) for p in self.hdl.buffer_ptrs]
        else:
            from torch.multiprocessing.reductions import reduce_tensor

            self.buf = torch.zeros(total, dtype=torch.uint8, device=device)
            torch.cuda.synchronize(device)
            shared = [None] * world
            dist.all_gather_object(shared, reduce_tensor(self.buf), group=group)
            self._peer_bufs = [self.buf if r == rank else fn(*args) for r, (fn, args) in enumerate(shared)]
            peers = [int(b.data_ptr()) for b in self._peer_bufs]
        assert peers[rank] == self.buf.data_ptr()
        h = C.c_void_p()
        _capi.check(lib.keds_exchange_create(world, rank, device.index, (C.c_void_p * world)(*peers), total, C.byref(h)))
        self.handle, self._lib = h, lib
        self.capacity = int(lib.keds_exchange_capacity(h))
        assert self.capacity >= capacity
        # every rank's buffer is zeroed before anyone pushes
        if self.hdl is not None:
            self.hdl.barrier()
        else:
            dist.barrier(group=group)

    def stats(self, stream_ptr: int) -> dict:
        import ctypes as C

        avg, mx, n, err = C.c_double(0), C.c_double(0), C.c_int64(0), C.c_uint32(0)
        _capi.check(self._lib.keds_exchange_stats(self.handle, stream_ptr, C.byref(avg), C.byref(mx), C.byref(n),
                                                  C.byref(err)))
        return {"wait_us_avg": float(avg.value), "wait_us_max": float(mx.value), "merges": int(n.value)}

    def __del__(self) -> None:
        h = getattr(self, "handle", None)
        if h is not None and h.value:
            try:
                self._lib.keds_exchange_free(h)
            except Exception:
                pass
            self.handle = None


def _grow_exchange(owner, need: int, floor: int) -> bool:
    """Give `owner` (a lone ShardedIndex or a ShardedKnowledgeBase) an exchange of at least `need` entries,
    at least `floor` when it allocates; True if it did. Collective: every rank grows at the same call."""
    if owner._fx is not None and owner._fx.capacity >= need:
        return False
    if owner._fx is not None:  # peers may still be using the old buffers for a step in flight
        torch.cuda.synchronize(owner.device)
        dist.barrier(group=owner.group)
    owner._fx = _FusedExchange(owner.world, owner.rank, max(need, floor), owner.device, owner.group)
    return True


class ShardedIndex:
    """exchange="fused" (default on GPUs): no collective call and no copy kernel in the step -- the
    search kernels store every finished result row straight into the peers' buffers over NVLink,
    the chain's last block publishes an epoch flag and the merge kernel waits on the peers' flags
    (keds_index_search_sharded; needs torch symmetric memory and peer access inside the box).
    exchange="nccl": one packed all-gather per search, then the merge kernel."""

    def __init__(self, d: int, metric: int, device: Optional[int] = None, group=None,
                 exchange: str = "fused", _local_index=None, _merge: Optional[Callable] = None) -> None:
        if not dist.is_initialized():
            raise RuntimeError("ShardedIndex needs an initialised torch.distributed process group")
        exchange = _exchange_name(exchange)
        if exchange not in ("nccl", "fused"):
            raise ValueError("exchange must be 'nccl' or 'fused'")
        self.group = group
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)
        self.d, self.metric_type = int(d), int(metric)
        self.exchange = exchange
        self._fx: Optional[_FusedExchange] = None
        self._merge = _merge
        if _local_index is not None:
            self.local = _local_index
            self.device = torch.device("cpu")
        else:
            dev = torch.cuda.current_device() if device is None else int(device)
            self.local = GpuIndexFlat(d, metric, dev)
            self.device = torch.device("cuda", dev)
        self.ntotal = 0
        self.lo = self.hi = 0
        self._kb: Optional["ShardedKnowledgeBase"] = None  # set when this index is a base of one
        self._db = 0

    def add_local(self, x_local, lo: int, ntotal: int) -> None:
        """This rank's rows (global row ids lo .. lo+len) of an ntotal-row database. Collective:
        every rank calls it (an index of a ShardedKnowledgeBase re-attaches the rows afterwards)."""
        kb = self._kb
        if kb is not None and kb._fx is not None and self.device.type == "cuda":
            # peers may still be reading these rows for a step in flight
            torch.cuda.synchronize(self.device)
            dist.barrier(group=self.group)
        self.lo, self.hi, self.ntotal = int(lo), int(lo) + int(x_local.shape[0]), int(ntotal)
        self.local.set_id_offset(self.lo)
        if x_local.shape[0]:
            self.local.add(x_local)
        if kb is not None:
            kb._attach_rows(self._db)

    def add(self, x) -> None:
        """Every rank passes the same full matrix and keeps its own row range."""
        lo, hi = shard_bounds(int(x.shape[0]), self.world, self.rank)
        self.add_local(x[lo:hi], lo, int(x.shape[0]))

    def range_search(self, q, radius: float):
        raise NotImplementedError("ShardedIndex.range_search is not implemented: range-search an unsharded "
                                  "GpuIndexFlat, or each rank's `local` index (its labels are global)")

    def search(self, q: torch.Tensor, k: int, out=None, exclude=None):
        """q: [nq, d] float32 on this rank's device, identical on all ranks. Returns (D, I);
        `out=(D, I)` may name preallocated contiguous device tensors to fill (fused exchange).
        exclude: int64 [nq] or [nq, E] (E <= 8) global labels each query must not get back, -1 =
        none, the same on every rank; the result is that of an unsharded search with exclusion."""
        nq = int(q.shape[0])
        total, off_i, d_bytes = packed_layout(nq, k)
        if self.exchange == "fused" and isinstance(self.local, GpuIndexFlat):
            return self._search_fused(q, nq, k, out, exclude)
        if isinstance(self.local, GpuIndexFlat):
            # the local search writes straight into the exchange buffer: no repacking copies
            send = torch.empty(total, dtype=torch.uint8, device=q.device)
            self.local.search(q, k, out=(send[:d_bytes].view(torch.float32), send[off_i:].view(torch.int64)),
                              exclude=exclude)
        else:  # CPU test stand-in
            D, I = self.local.search(q, k) if exclude is None else self.local.search(q, k, exclude=exclude)
            D, I = torch.as_tensor(D), torch.as_tensor(I)
            send = torch.empty(total, dtype=torch.uint8, device=D.device)
            send[:d_bytes].view(torch.float32).copy_(D.reshape(-1))
            send[off_i:].view(torch.int64).copy_(I.reshape(-1))
        recv = torch.empty(self.world * total, dtype=torch.uint8, device=send.device)
        dist.all_gather_into_tensor(recv, send, group=self.group)
        if self._merge is not None:  # CPU test hook
            parts = recv.view(self.world, total)
            Dp = torch.stack([parts[r, :d_bytes].view(torch.float32).view(nq, k) for r in range(self.world)])
            Ip = torch.stack([parts[r, off_i:].view(torch.int64).view(nq, k) for r in range(self.world)])
            return self._merge(Dp, Ip, k, self.metric_type)
        lib = _capi.load()
        Dg = torch.empty((nq, k), dtype=torch.float32, device=send.device)
        Ig = torch.empty((nq, k), dtype=torch.int64, device=send.device)
        base = recv.data_ptr()
        _capi.check(
            lib.keds_topk_merge_strided(base, base + off_i, total // 4, total // 8, self.world, nq, k,
                                        self.metric_type, Dg.data_ptr(), Ig.data_ptr(),
                                        _stream_ptr(self.device.index))
        )
        return Dg, Ig

    def _search_fused(self, q: torch.Tensor, nq: int, k: int, out=None, exclude=None):
        """One native call: local search with the peer stores fused into its kernels, flag
        publication by the chain's last block, merge that waits on the peers' flags. Two buffer
        parities keep a fast rank from overwriting a block a slow rank is still merging (a rank can
        only publish step t+1 after finishing its merge of step t)."""
        lib = _capi.load()
        q = self.local._check_q_tensor(q)
        ex = _exclude_arg(exclude, nq, self.device.index)
        fx = self._exchange(nq * k)
        if out is not None:
            Dg, Ig = _check_out(out, nq * k)
        else:
            Dg = torch.empty((nq, k), dtype=torch.float32, device=q.device)
            Ig = torch.empty((nq, k), dtype=torch.int64, device=q.device)
        _capi.check(lib.keds_index_search_sharded(self.local._h, fx.handle, q.data_ptr(), nq, k, Dg.data_ptr(),
                                                  Ig.data_ptr(), *_exclude_ptrs(ex), _stream_ptr(self.device.index)))
        return Dg, Ig

    def _exchange(self, need: int) -> _FusedExchange:
        """The knowledge base's exchange for one of its bases (one set of peer buffers), else its own."""
        if self._kb is not None:
            return self._kb._exchange(need)
        _grow_exchange(self, need, 8192)
        return self._fx

    def exchange_stats(self) -> dict:
        """Synchronise and report how long the merge waited for the peers (rank skew); raises if a
        peer failed to deliver within the watchdog window."""
        if self._fx is None:
            return {}
        return self._fx.stats(_stream_ptr(self.device.index))

    def check_exchange(self) -> None:
        self.exchange_stats()


def _sharded_kb(image_index, text_index,
                refusal: str = "image_index and text_index must both be GpuIndexFlat, or be the `image` and `text` "
                               "indices of one ShardedKnowledgeBase"):
    """The ShardedKnowledgeBase whose two bases are (image_index, text_index); None for two indices
    that are not sharded. A mixed pair, or the bases of two different knowledge bases, raise
    TypeError(refusal)."""
    sharded = (isinstance(image_index, ShardedIndex), isinstance(text_index, ShardedIndex))
    if not any(sharded):
        return None
    kb = image_index._kb if sharded[0] else None
    if not all(sharded) or kb is None or kb.image is not image_index or kb.text is not text_index:
        raise TypeError(refusal)
    return kb


def rank_block(batch_sizes, rank: int) -> Tuple[int, int, int]:
    """(padded batch Bmax, first row, end row) of `rank`'s queries in the all-gathered query matrix
    of a DDP step: every rank pads its batch to the largest one, so rank r owns [r*Bmax, r*Bmax + B_r)."""
    sizes = [int(b) for b in batch_sizes]
    if not sizes or min(sizes) < 0 or not 0 <= rank < len(sizes):
        raise ValueError(f"rank_block: rank {rank} of batch sizes {sizes}")
    bmax = max(sizes)
    return bmax, rank * bmax, rank * bmax + sizes[rank]


class ShardedKnowledgeBase:
    """The KEDs retrieval step over row-sharded image and text bases: two ShardedIndex (`image`,
    `text`) over one fused exchange. Every rank holds rows [lo_r, hi_r) of each base; retrieve2
    searches both bases for queries that are the same on every rank, merges the global top-k on every
    rank, and gathers / pools the neighbour rows of the query rows a rank asks for straight from the
    owners' fp32 rows over NVLink (mapped with cudaIpc, re-attached after every add). Results equal
    retrieval.retrieve2 on an unsharded index bit for bit (D, I, gathered rows); pools use the same
    weights and do not depend on the shard count.

    Test hooks: `_local_index` (a factory of stand-in local indices, as ShardedIndex takes) and
    `_retrieve` (a stand-in for the native step, called with the checked arguments) let the CPU
    (gloo) tests drive the DDP plumbing of get_retrieved_features."""

    def __init__(self, d: int, metric: int, device: Optional[int] = None, group=None, exchange: str = "fused",
                 _local_index: Optional[Callable] = None, _retrieve: Optional[Callable] = None) -> None:
        exchange = _exchange_name(exchange)
        if exchange != "fused":
            raise ValueError("ShardedKnowledgeBase: the retrieval step needs exchange='fused' (peer memory); "
                             f"got {exchange!r}")
        self.image = ShardedIndex(d, metric, device, group, exchange,
                                  _local_index=_local_index() if _local_index else None)
        self.text = ShardedIndex(d, metric, device, group, exchange,
                                 _local_index=_local_index() if _local_index else None)
        for db, ix in enumerate((self.image, self.text)):
            ix._kb, ix._db = self, db
        self.group, self.rank, self.world = group, self.image.rank, self.image.world
        self.d, self.metric_type, self.device = int(d), int(metric), self.image.device
        self._fx: Optional[_FusedExchange] = None
        self._retrieve = _retrieve

    def add(self, image_rows, text_rows) -> None:
        """Every rank passes the same full matrices and keeps its own row ranges. Collective."""
        self.image.add(image_rows)
        self.text.add(text_rows)

    def _native(self) -> bool:
        return self._retrieve is None and isinstance(self.image.local, GpuIndexFlat)

    def _attach_rows(self, db: int) -> None:
        """Tell the exchange where every rank's rows of base `db` live (collective)."""
        if self._fx is None or not self._native():
            return
        import ctypes as C

        ix = (self.image, self.text)[db]
        lib = _capi.load()
        torch.cuda.synchronize(self.device)
        h = (C.c_uint8 * 64)()
        _capi.check(lib.keds_index_rows_ipc(ix.local._h, h))
        mine = (bytes(h), ix.lo, ix.hi - ix.lo)
        every = [None] * self.world
        dist.all_gather_object(every, mine, group=self.group)
        bufs = [(C.c_uint8 * 64).from_buffer_copy(e[0]) for e in every]
        handles = (C.c_void_p * self.world)(*[C.addressof(b) for b in bufs])
        lo = (C.c_int64 * self.world)(*[e[1] for e in every])
        n = (C.c_int64 * self.world)(*[e[2] for e in every])
        _capi.check(lib.keds_exchange_attach_rows(self._fx.handle, db, handles, lo, n))

    def _exchange(self, need: int) -> _FusedExchange:
        if _grow_exchange(self, need, 16384):
            self.image._fx = self.text._fx = self._fx
            self._attach_rows(0)
            self._attach_rows(1)
        return self._fx

    def retrieve2(self, q: torch.Tensor, k: int = 16, perm_img: Optional[torch.Tensor] = None,
                  perm_txt: Optional[torch.Tensor] = None, want_feats: bool = True, pool_mode: int = 0,
                  tau: float = 100.0, flags: int = 0, exclude=None, rows: Optional[Tuple[int, int]] = None,
                  out: Optional[dict] = None) -> dict:
        """One step for queries q [Bt, d] (float32, this rank's device, identical on every rank).
        Returns D_img / I_img / D_txt / I_txt [Bt, k] for every query and, for the query rows
        rows = (lo, hi) only (default: all), feat_img / feat_txt [hi-lo, k, d] (image stream permuted
        by perm_img) and pool_img / pool_txt [hi-lo, d] (pool_mode 1 mean, 2 softmax(+-tau*D)).
        exclude: int64 [Bt] or [Bt, E] (E <= 8) global labels each query must not retrieve from
        either base, -1 = none. Collective: every rank calls it with the same q, k and exclusion.
        `out` may carry the tensors of a previous call (keys as returned); a tensor of another shape,
        dtype or device, or a non-contiguous one, is replaced in the dict.
        perm_img / perm_txt: permutations of range(k); a CPU tensor that is not one raises ValueError,
        a CUDA tensor is trusted (the pool adds, per output slot j, the neighbour perm[j] shows)."""
        if not isinstance(q, torch.Tensor) or q.dtype != torch.float32 or q.dim() != 2 or q.shape[1] != self.d:
            raise TypeError(f"retrieve2: q must be a float32 [Bt, {self.d}] tensor")
        if q.device != self.device:
            raise ValueError(f"retrieve2: q on {q.device}, the knowledge base on {self.device}")
        Bt, k = int(q.shape[0]), int(k)
        if Bt < 1:
            raise ValueError("retrieve2: empty query batch")
        if not 1 <= k <= 1024:
            raise ValueError(f"retrieve2: k must be 1..1024, got {k}")
        if pool_mode not in (0, 1, 2):
            raise ValueError(f"retrieve2: pool_mode must be 0, 1 or 2, got {pool_mode}")
        lo, hi = (0, Bt) if rows is None else (int(rows[0]), int(rows[1]))
        if not 0 <= lo <= hi <= Bt:
            raise ValueError(f"retrieve2: rows ({lo}, {hi}) outside [0, {Bt}]")
        perms = []
        for name, p in (("perm_img", perm_img), ("perm_txt", perm_txt)):
            if p is not None and (not isinstance(p, torch.Tensor) or p.dim() != 1 or p.numel() != k
                                  or p.dtype not in (torch.int32, torch.int64)):
                raise TypeError(f"retrieve2: {name} must be an integer tensor of {k} entries")
            check_perm(p, k, f"retrieve2: {name}")
            perms.append(_device_perm(p, k, self.device))
        ex = None
        if exclude is not None:
            ex = _exclude_arg(exclude, Bt, self.device.index) if self.device.type == "cuda" else \
                torch.as_tensor(_check_exclude_host(exclude, Bt))
        q = q.contiguous()
        if self._retrieve is not None:  # CPU test hook
            return self._retrieve(q, k, perms[0], perms[1], want_feats, pool_mode, tau, flags, ex, (lo, hi))
        fx = self._exchange(2 * Bt * k)
        o = out if out is not None else {}
        Di, Ii, Dt, It, fi, ft, pi, pt = _step_outputs(o, self.device, Bt, hi - lo, k, self.d, want_feats, pool_mode)
        ptr = lambda t: 0 if t is None else t.data_ptr()
        lib = _capi.load()
        _capi.check(lib.keds_retrieve2_sharded(
            self.image.local._h, self.text.local._h, fx.handle, q.data_ptr(), Bt, k, ptr(perms[0]), ptr(perms[1]),
            int(pool_mode), float(tau), lo, hi, Di.data_ptr(), Ii.data_ptr(), Dt.data_ptr(), It.data_ptr(),
            ptr(fi), ptr(ft), ptr(pi), ptr(pt), *_exclude_ptrs(ex), int(flags),
            _stream_ptr(self.device.index)))
        return o

    def retrieve2_ddp(self, q: torch.Tensor, k: int, exclude=None, **kw):
        """The DDP step: every rank passes its own queries [B_r, d] and exclusion; gather_ddp_step, then one
        retrieve2(**kw) over every rank's queries with rows = this rank's block. Returns (out, (lo, hi))."""
        q_all, ex_all, rows = gather_ddp_step(q, exclude, self.group, self.device)
        return self.retrieve2(q_all, k, exclude=ex_all, rows=rows, **kw), rows

    def exchange_stats(self) -> dict:
        """Synchronise and report how long the merges waited for the peers; raises if a peer failed
        to deliver within the watchdog window."""
        return {} if self._fx is None else self._fx.stats(_stream_ptr(self.device.index))


def _check_exclude_host(exclude, nq: int):
    from .index import check_exclude

    ex = check_exclude(exclude, nq)
    return ex if isinstance(ex, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(ex))


def gather_ddp_step(feature: torch.Tensor, exclude, group=None, device=None):
    """The all-gathers of a sharded DDP retrieval step: every rank's batch size, then the queries
    padded to the largest batch ([world * Bmax, d]) and, if any rank passes one, the exclusion arrays
    padded with -1 ([world * Bmax, E_max]). Returns (queries, exclusion or None, (lo, hi)) with
    [lo, hi) this rank's own rows."""
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    dev = feature.device if device is None else device
    B, d = int(feature.shape[0]), int(feature.shape[1])
    ex = None if exclude is None else _check_exclude_host(exclude, B)
    meta = torch.tensor([B, 0 if ex is None else int(ex.shape[1])], dtype=torch.int64, device=dev)
    # (flat receive buffers: the form every backend's all_gather_into_tensor takes)
    metas = torch.empty(world * 2, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(metas, meta, group=group)
    sizes, widths = metas[0::2].tolist(), metas[1::2].tolist()
    bmax, lo, hi = rank_block(sizes, rank)
    qp = torch.zeros((bmax, d), dtype=torch.float32, device=dev)
    qp[:B] = feature.to(device=dev, dtype=torch.float32)
    q_all = torch.empty(world * bmax * d, dtype=torch.float32, device=dev)
    dist.all_gather_into_tensor(q_all, qp.view(-1), group=group)
    q_all = q_all.view(world * bmax, d)
    e_max = max(widths)
    ex_all = None
    if e_max > 0:
        ep = torch.full((bmax, e_max), -1, dtype=torch.int64, device=dev)
        if ex is not None:
            ep[:B, :ex.shape[1]] = ex.to(dev)
        ex_all = torch.empty(world * bmax * e_max, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(ex_all, ep.view(-1), group=group)
        ex_all = ex_all.view(world * bmax, e_max)
    return q_all, ex_all, (lo, hi)
