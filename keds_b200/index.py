"""Faiss-shaped index objects over libkeds_knn.so.

Mirrors exactly the slice of the Faiss Python API that KEDs touches:

    faiss.IndexFlatL2(768) / IndexFlatIP          src/main.py:74,80  src/eval_retrieval.py:291,294
    faiss.StandardGpuResources()                   src/main.py:73
    faiss.index_cpu_to_gpu(res, gpu, index)        src/main.py:76,82
    faiss.index_cpu_to_all_gpus(index)             src/eval_retrieval.py:292,295
    faiss.get_num_gpus()                           src/eval_retrieval.py:289
    index.add(x) / index.search(x, k) / .ntotal    src/main.py:78,83  src/trainer.py:213,221,271

so that `import keds_b200.faiss_compat as faiss` leaves the reference's call sites unchanged.
numpy in -> numpy out (float32 D, int64 I) like Faiss; as an extension a CUDA torch.Tensor in gives
CUDA tensors out with no host hop, ordered on torch's current stream.

There is no CPU search: a flat index that has not been moved to a GPU can only collect rows.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _capi

try:  # torch is plumbing (device tensors, streams); numpy-only use works without it
    import torch
except Exception:  # pragma: no cover
    torch = None

METRIC_INNER_PRODUCT = _capi.METRIC_IP
METRIC_L2 = _capi.METRIC_L2


def _is_tensor(x) -> bool:
    return torch is not None and isinstance(x, torch.Tensor)


def _as_f32_matrix(x, d: int, what: str) -> np.ndarray:
    """Faiss' SWIG layer semantics: 2-D, second dim == d, coerced to C-contiguous float32."""
    a = np.asarray(x)
    if a.ndim != 2:
        raise ValueError(f"{what}: expected a 2-D array, got shape {a.shape}")
    if a.shape[1] != d:
        raise AssertionError(f"{what}: second dimension {a.shape[1]} != index dimension {d}")
    if a.dtype != np.float32:
        raise TypeError(f"{what}: expected float32, got {a.dtype}")
    return np.ascontiguousarray(a)


EXCLUDE_MAX = 8  # rows one query may leave out (include/keds_knn.h, search with exclusion)


def check_exclude(exclude, nq: int):
    """Validate a per-query exclusion array: labels as `search` returns them, -1 = unused slot.
    Accepts a numpy array or a torch tensor of int64, shaped [nq] or [nq, E] with 1 <= E <= 8.
    Returns it as [nq, E] (a view, nothing is copied or moved); raises TypeError / ValueError."""
    if _is_tensor(exclude):
        if exclude.dtype != torch.int64:
            raise TypeError(f"exclude: expected int64 labels, got {exclude.dtype}")
    elif isinstance(exclude, np.ndarray):
        if exclude.dtype != np.int64:
            raise TypeError(f"exclude: expected int64 labels, got {exclude.dtype}")
    else:
        raise TypeError(f"exclude: expected a numpy array or a torch tensor, got {type(exclude).__name__}")
    shape = tuple(exclude.shape)
    if len(shape) == 1:
        exclude = exclude.reshape(-1, 1)
    elif len(shape) != 2:
        raise ValueError(f"exclude: expected shape [nq] or [nq, E], got {shape}")
    if exclude.shape[0] != nq:
        raise ValueError(f"exclude: {exclude.shape[0]} rows for {nq} queries")
    if not 1 <= exclude.shape[1] <= EXCLUDE_MAX:
        raise ValueError(f"exclude: E = {exclude.shape[1]} labels per query, expected 1..{EXCLUDE_MAX}")
    return exclude


def _exclude_arg(exclude, nq: int, device: int, pinned_ok: bool = False):
    """None for None; else check_exclude, then a contiguous int64 tensor the native call can read:
    on `device`, or a pinned host tensor as it is when `pinned_ok` (retrieve2's host I/O reads it
    through the mapping). Keep it alive until the native call has been queued."""
    if exclude is None:
        return None
    ex = check_exclude(exclude, nq)
    if torch is None:
        raise RuntimeError("search with exclusion needs torch for the device copy of `exclude`")
    if isinstance(ex, np.ndarray):
        ex = torch.from_numpy(np.ascontiguousarray(ex))
    if ex.is_cuda:
        if ex.device.index != device:
            raise ValueError(f"exclude: on cuda:{ex.device.index}, index on cuda:{device}")
        return ex.contiguous()
    if pinned_ok and ex.is_pinned() and ex.is_contiguous():
        return ex
    return ex.to(torch.device("cuda", device), non_blocking=False).contiguous()


def _exclude_ptrs(ex) -> Tuple[int, int]:
    """The native calls' (exclude, n_exclude) for a result of _exclude_arg: (0, 0) = no exclusion."""
    return (0, 0) if ex is None else (ex.data_ptr(), int(ex.shape[1]))


def _check_out(out, n: int):
    """A caller's out=(D, I): contiguous CUDA float32 / int64 tensors of n elements each."""
    D, I = out
    assert D.is_cuda and I.is_cuda and D.is_contiguous() and I.is_contiguous()
    assert D.dtype == torch.float32 and I.dtype == torch.int64
    assert D.numel() == n and I.numel() == n
    return D, I


def _ptr(a) -> int:
    """Address of the data of a tensor or a numpy array."""
    return a.data_ptr() if _is_tensor(a) else a.ctypes.data


def _stream_ptr(device: int) -> int:
    if torch is not None and torch.cuda.is_available():
        return int(torch.cuda.current_stream(device).cuda_stream)
    return 0


class StandardGpuResources:
    """Placeholder with Faiss' name: the native handle owns its own device memory."""

    def __init__(self) -> None:
        self.temp_memory = None

    def setTempMemory(self, nbytes: int) -> None:  # noqa: N802 (Faiss spelling)
        self.temp_memory = int(nbytes)

    def noTempMemory(self) -> None:  # noqa: N802
        self.temp_memory = 0


class GpuClonerOptions:
    def __init__(self) -> None:
        self.useFloat16 = False


class GpuMultipleClonerOptions(GpuClonerOptions):
    def __init__(self) -> None:
        super().__init__()
        self.shard = False


_NO_CPU_SEARCH = ("keds_b200 has no CPU search path: move the index to a GPU with "
                  "index_cpu_to_gpu / index_cpu_to_all_gpus first")


class IndexFlat:
    """Host-side flat index: collects rows until it is cloned to a GPU (no CPU search)."""

    def __init__(self, d: int, metric: int = METRIC_L2) -> None:
        if int(d) <= 0:
            raise ValueError("dimension must be positive")
        self.d = int(d)
        self.metric_type = int(metric)
        self.is_trained = True
        self._blocks: List[np.ndarray] = []

    @property
    def ntotal(self) -> int:
        return int(sum(b.shape[0] for b in self._blocks))

    def add(self, x) -> None:
        self._blocks.append(_as_f32_matrix(x, self.d, "add").copy())

    def reset(self) -> None:
        self._blocks = []

    def search(self, x, k):
        raise RuntimeError(_NO_CPU_SEARCH)

    def range_search(self, x, radius):
        raise RuntimeError(_NO_CPU_SEARCH)


class IndexFlatIP(IndexFlat):
    def __init__(self, d: int) -> None:
        super().__init__(d, METRIC_INNER_PRODUCT)


class IndexFlatL2(IndexFlat):
    def __init__(self, d: int) -> None:
        super().__init__(d, METRIC_L2)


class GpuIndexFlat:
    """One native index on one B200. `search` == Faiss' contract (best first, -1 padding)."""

    def __init__(self, d: int, metric: int = METRIC_L2, device: int = 0) -> None:
        self._lib = _capi.load()
        self.d = int(d)
        self.metric_type = int(metric)
        self.device = int(device)
        self.is_trained = True
        h = C.c_void_p()
        _capi.check(self._lib.keds_index_create(self.d, self.metric_type, self.device, C.byref(h)))
        self._h = h

    # -- lifecycle
    def __del__(self) -> None:
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            try:
                self._lib.keds_index_free(h)
            except Exception:
                pass
            self._h = None

    @property
    def ntotal(self) -> int:
        return int(self._lib.keds_index_ntotal(self._h))

    def reset(self) -> None:
        _capi.check(self._lib.keds_index_reset(self._h))

    def set_id_offset(self, offset: int) -> None:
        _capi.check(self._lib.keds_index_set_id_offset(self._h, int(offset)))

    def set_pdl(self, enable: bool) -> None:
        _capi.check(self._lib.keds_index_set_pdl(self._h, int(bool(enable))))

    def set_eps_scale(self, scale: float) -> None:
        _capi.check(self._lib.keds_index_set_eps_scale(self._h, float(scale)))

    @property
    def operand_format(self) -> str:
        """16-bit operand format of the tensor-core pass: 'fp16' or 'bf16' (chosen from the rows)."""
        return {0: "bf16", 1: "fp16"}[int(self._lib.keds_index_operand_format(self._h))]

    def set_operand_format(self, fmt: Optional[str]) -> None:
        """Pin the operand format ('bf16' / 'fp16') or return to the automatic choice (None)."""
        code = {None: -1, "auto": -1, "bf16": 0, "fp16": 1}[fmt]
        _capi.check(self._lib.keds_index_set_operand_format(self._h, code))

    @property
    def generation(self) -> int:
        """Changes whenever a device buffer of the handle moves or its rows change; owners of a CUDA
        graph captured over a search compare it before every replay."""
        return int(self._lib.keds_index_generation(self._h))

    # -- add
    def add(self, x, normalize: bool = False) -> None:
        """index.add(x). normalize=True L2-normalises the rows on the device as they are added."""
        flags = 1 if normalize else 0
        if _is_tensor(x):
            if x.dim() != 2 or x.shape[1] != self.d:
                raise AssertionError(f"add: shape {tuple(x.shape)} does not match d={self.d}")
            if x.dtype != torch.float32:
                raise TypeError(f"add: expected float32, got {x.dtype}")
            x = x.contiguous()
            if x.is_cuda:
                torch.cuda.current_stream(x.device).synchronize()
            _capi.check(self._lib.keds_index_add_ex(self._h, x.data_ptr(), x.shape[0], flags))
            return
        a = _as_f32_matrix(x, self.d, "add")
        _capi.check(self._lib.keds_index_add_ex(self._h, a.ctypes.data, a.shape[0], flags))

    def get_rows(self, first: int = 0, n: Optional[int] = None) -> np.ndarray:
        """rows [first, first+n) of the resident fp32 master as a host array (e.g. to save a .pt)."""
        n = self.ntotal - first if n is None else int(n)
        out = np.empty((n, self.d), dtype=np.float32)
        _capi.check(self._lib.keds_index_get_rows(self._h, int(first), n, out.ctypes.data))
        return out

    # -- search
    def search(self, x, k: int, flags: int = 0, out=None, exclude=None):
        """numpy in -> numpy (D, I) out, synchronous. CUDA tensor in -> CUDA tensors out,
        stream-ordered; `out=(D, I)` may name preallocated contiguous CUDA tensors to fill.
        exclude: int64 [nq] or [nq, E] (E <= 8) labels each query must not get back (e.g. its own
        row), -1 = unused; the result is the exact search over the remaining rows."""
        k = int(k)
        if k <= 0:
            raise ValueError("k must be positive")
        if _is_tensor(x) and x.is_cuda:
            q = self._check_q_tensor(x)
            if out is not None:
                D, I = _check_out(out, q.shape[0] * k)
            else:
                D = torch.empty((q.shape[0], k), dtype=torch.float32, device=q.device)
                I = torch.empty((q.shape[0], k), dtype=torch.int64, device=q.device)
        else:
            q = _as_f32_matrix(x.numpy() if _is_tensor(x) else x, self.d, "search")
            D = np.empty((q.shape[0], k), dtype=np.float32)
            I = np.empty((q.shape[0], k), dtype=np.int64)
        ex = _exclude_arg(exclude, q.shape[0], self.device)
        _capi.check(self._lib.keds_index_search_ex(self._h, _ptr(q), q.shape[0], k, _ptr(D), _ptr(I),
                                                   *_exclude_ptrs(ex), flags, _stream_ptr(self.device)))
        return D, I

    def range_search(self, x, radius: float, flags: int = 0):
        """Faiss' index.range_search(x, radius) -> (lims, D, I): every row with score > radius (IP)
        or squared distance < radius (L2), radius rounded to float32, exact in fp32; query i owns
        [lims[i], lims[i+1]) of D and I, best first, ties by lower label. numpy in -> numpy out.
        CUDA tensor in -> CUDA tensors out; the call synchronises the stream once the search has run,
        to size D and I."""
        radius = float(radius)
        if radius != radius:
            raise ValueError("radius must not be NaN")
        stream = _stream_ptr(self.device)
        if _is_tensor(x) and x.is_cuda:
            q = self._check_q_tensor(x, "range_search")
            lims = torch.empty(q.shape[0] + 1, dtype=torch.int64, device=q.device)
            _capi.check(self._lib.keds_index_range_search(self._h, q.data_ptr(), q.shape[0], radius, lims.data_ptr(),
                                                          flags, stream))
            n = int(lims[-1].item())
            D = torch.empty(n, dtype=torch.float32, device=q.device)
            I = torch.empty(n, dtype=torch.int64, device=q.device)
            _capi.check(self._lib.keds_index_range_results(self._h, D.data_ptr(), I.data_ptr(), stream))
            return lims, D, I
        a = _as_f32_matrix(x.numpy() if _is_tensor(x) else x, self.d, "range_search")
        lims = np.empty(a.shape[0] + 1, dtype=np.int64)
        _capi.check(self._lib.keds_index_range_search(self._h, a.ctypes.data, a.shape[0], radius, lims.ctypes.data,
                                                      flags, stream))
        D = np.empty(int(lims[-1]), dtype=np.float32)
        I = np.empty(int(lims[-1]), dtype=np.int64)
        _capi.check(self._lib.keds_index_range_results(self._h, D.ctypes.data, I.ctypes.data, stream))
        return lims, D, I

    def _check_q_tensor(self, x, what: str = "search"):
        if x.dim() != 2 or x.shape[1] != self.d:
            raise AssertionError(f"{what}: shape {tuple(x.shape)} does not match d={self.d}")
        if x.dtype != torch.float32:
            raise TypeError(f"{what}: expected float32, got {x.dtype}")
        if x.device.index != self.device:
            raise ValueError(f"{what}: query on cuda:{x.device.index}, index on cuda:{self.device}")
        return x.contiguous()

    def sync(self) -> None:
        """Wait for the last asynchronous search and raise if the device reported an error."""
        _capi.check(self._lib.keds_index_sync(self._h, _stream_ptr(self.device)))

    def last_stats(self) -> dict:
        st = _capi.SearchStats()
        _capi.check(self._lib.keds_index_last_stats(self._h, C.byref(st)))
        return {
            "n_flagged": [int(st.n_flagged[0]), int(st.n_flagged[1])],
            "slices": int(st.slices),
            "items": int(st.items),
            "grid": int(st.grid),
            "exact_only": int(st.exact_only),
            "launches": int(st.launches),
            "err_word": int(st.err_word),
        }

    def set_profiling(self, mode: int) -> None:
        """0 off; 1 in-kernel timer of the scoring kernel (launch chain untouched)."""
        _capi.check(self._lib.keds_index_set_profiling(self._h, int(mode)))

    def profile(self):
        """(summed ms, launches) of the scoring kernel since set_profiling(True); waits for them."""
        ms, n = C.c_double(0.0), C.c_int64(0)
        _capi.check(self._lib.keds_index_profile(self._h, C.byref(ms), C.byref(n)))
        return float(ms.value), int(n.value)

    CHAIN = ("k_prep_rows", "k_score_topk", "k_select_rerank", "k_exact_fallback")

    def profile_chain(self) -> dict:
        """In-loop timeline of a search (mode 1): per kernel {'ms': duration, 'gap_ms': idle gap
        before it}, averaged over the searches since set_profiling(1)."""
        dur, gap, n = (C.c_double * 5)(), (C.c_double * 5)(), C.c_int64(0)
        _capi.check(self._lib.keds_index_profile_chain(self._h, dur, gap, C.byref(n), 5))
        out = {name: {"ms": float(dur[i]), "gap_ms": float(gap[i])} for i, name in enumerate(self.CHAIN)}
        out["searches"] = int(n.value)
        return out

    def rows_ptr(self) -> int:
        """Device address of the resident fp32 rows [ntotal, d]."""
        return int(self._lib.keds_index_rows(self._h) or 0)

    def debug_scores(self, q):
        """bf16 tensor-core scores of q against every row (test hook)."""
        q = self._check_q_tensor(q)
        out = torch.empty((q.shape[0], self.ntotal), dtype=torch.float32, device=q.device)
        _capi.check(
            self._lib.keds_debug_scores(self._h, q.data_ptr(), q.shape[0], out.data_ptr(),
                                        _stream_ptr(self.device))
        )
        return out


def search2(a: GpuIndexFlat, b: GpuIndexFlat, x, k: int, flags: int = 0, exclude=None):
    """Both databases against one query batch in one pass (src/trainer.py:213 + :221).
    exclude: as GpuIndexFlat.search; one array for both databases (aligned row for row)."""
    lib = _capi.load()
    k = int(k)
    if _is_tensor(x) and x.is_cuda:
        q = a._check_q_tensor(x)
        Da, Db = (torch.empty((q.shape[0], k), dtype=torch.float32, device=q.device) for _ in range(2))
        Ia, Ib = (torch.empty((q.shape[0], k), dtype=torch.int64, device=q.device) for _ in range(2))
    else:
        q = _as_f32_matrix(x.numpy() if _is_tensor(x) else x, a.d, "search2")
        Da, Db = (np.empty((q.shape[0], k), np.float32) for _ in range(2))
        Ia, Ib = (np.empty((q.shape[0], k), np.int64) for _ in range(2))
    ex = _exclude_arg(exclude, q.shape[0], a.device)
    _capi.check(lib.keds_index_search2(a._h, b._h, _ptr(q), q.shape[0], k, _ptr(Da), _ptr(Ia), _ptr(Db), _ptr(Ib),
                                       *_exclude_ptrs(ex), flags, _stream_ptr(a.device)))
    return (Da, Ia), (Db, Ib)


def _run_parallel(jobs):
    """Run the callables on one thread each and return their results in order (first error re-raised)."""
    if len(jobs) == 1:
        return [jobs[0]()]
    from concurrent.futures import ThreadPoolExecutor

    with ThreadPoolExecutor(max_workers=len(jobs)) as pool:
        futs = [pool.submit(j) for j in jobs]
        return [f.result() for f in futs]


class IndexReplicas:
    """Faiss' default for index_cpu_to_all_gpus: a full copy per GPU, queries split across them.
    Results are identical to a single-GPU search (src/eval_retrieval.py:292,295)."""

    def __init__(self, d: int, metric: int, devices: Sequence[int]) -> None:
        self.d, self.metric_type = int(d), int(metric)
        self.subs = [GpuIndexFlat(d, metric, dev) for dev in devices]
        self.is_trained = True

    @property
    def ntotal(self) -> int:
        return self.subs[0].ntotal

    def add(self, x) -> None:
        for s in self.subs:
            s.add(x)

    def reset(self) -> None:
        for s in self.subs:
            s.reset()

    def search(self, x, k: int):
        a = _as_f32_matrix(x.cpu().numpy() if _is_tensor(x) else x, self.d, "search")
        n = a.shape[0]
        bounds = np.linspace(0, n, len(self.subs) + 1).astype(np.int64)
        parts = [(s, int(lo), int(hi)) for s, lo, hi in zip(self.subs, bounds[:-1], bounds[1:]) if hi > lo]
        if not parts:
            return np.empty((0, k), np.float32), np.empty((0, k), np.int64)
        # one host thread per GPU, as Faiss' IndexReplicas does (the native call releases the GIL)
        res = _run_parallel([lambda s=s, lo=lo, hi=hi: s.search(a[lo:hi], k) for s, lo, hi in parts])
        return np.concatenate([r[0] for r in res]), np.concatenate([r[1] for r in res])

    def range_search(self, x, radius: float):
        """The queries split across the replicas as in `search`; each part's lims are shifted by the
        results of the parts before it, so the result equals one index's (numpy out)."""
        a = _as_f32_matrix(x.cpu().numpy() if _is_tensor(x) else x, self.d, "range_search")
        n = a.shape[0]
        bounds = np.linspace(0, n, len(self.subs) + 1).astype(np.int64)
        parts = [(s, int(lo), int(hi)) for s, lo, hi in zip(self.subs, bounds[:-1], bounds[1:]) if hi > lo]
        res = _run_parallel([lambda s=s, lo=lo, hi=hi: s.range_search(a[lo:hi], radius) for s, lo, hi in parts])
        lims, shift = [np.zeros(1, np.int64)], 0
        for r in res:
            lims.append(np.asarray(r[0][1:], dtype=np.int64) + shift)
            shift += int(r[0][-1])
        return (np.concatenate(lims), np.concatenate([np.zeros(0, np.float32)] + [r[1] for r in res]),
                np.concatenate([np.zeros(0, np.int64)] + [r[2] for r in res]))


class IndexShards:
    """Row shards across the GPUs of one process (GpuMultipleClonerOptions.shard=True): every GPU
    searches its rows for all queries, labels are global, a merge kernel picks the global top-k.
    The multi-process (one rank per GPU, NCCL all-gather) form is keds_b200.sharded.ShardedIndex."""

    def __init__(self, d: int, metric: int, devices: Sequence[int]) -> None:
        self.d, self.metric_type = int(d), int(metric)
        self.devices = list(devices)
        self.subs = [GpuIndexFlat(d, metric, dev) for dev in devices]
        self._ntotal = 0
        self.is_trained = True

    @property
    def ntotal(self) -> int:
        return self._ntotal

    def add(self, x) -> None:
        a = _as_f32_matrix(x.cpu().numpy() if _is_tensor(x) else x, self.d, "add")
        if self._ntotal != 0:
            raise RuntimeError("IndexShards.add: add all rows in one call (contiguous row ranges)")
        n, R = a.shape[0], len(self.subs)
        per = -(-n // R)
        for r, s in enumerate(self.subs):
            lo, hi = min(n, r * per), min(n, (r + 1) * per)
            s.set_id_offset(lo)
            if hi > lo:
                s.add(a[lo:hi])
        self._ntotal = n

    def reset(self) -> None:
        for s in self.subs:
            s.reset()
        self._ntotal = 0

    def range_search(self, x, radius: float):
        raise NotImplementedError("IndexShards.range_search is not implemented: use one GpuIndexFlat or "
                                  "IndexReplicas (index_cpu_to_all_gpus without shard=True)")

    def search(self, x, k: int):
        if torch is None:
            raise RuntimeError("IndexShards needs torch for cross-device staging")
        a = _as_f32_matrix(x.cpu().numpy() if _is_tensor(x) else x, self.d, "search")
        lib = _capi.load()
        nq, R = a.shape[0], len(self.subs)
        dev0 = torch.device("cuda", self.devices[0])
        Dp = torch.empty((R, nq, k), dtype=torch.float32, device=dev0)
        Ip = torch.empty((R, nq, k), dtype=torch.int64, device=dev0)

        def one(s):
            q = torch.from_numpy(a).to(torch.device("cuda", s.device))
            with torch.cuda.device(s.device):
                D, I = s.search(q, k)
                s.sync()
            return D, I

        # every shard searches at the same time (one host thread per GPU), then the parts meet on GPU 0
        for r, (D, I) in enumerate(_run_parallel([lambda s=s: one(s) for s in self.subs])):
            Dp[r].copy_(D)
            Ip[r].copy_(I)
        D = torch.empty((nq, k), dtype=torch.float32, device=dev0)
        I = torch.empty((nq, k), dtype=torch.int64, device=dev0)
        with torch.cuda.device(dev0):
            _capi.check(
                lib.keds_topk_merge(Dp.data_ptr(), Ip.data_ptr(), R, nq, k, self.metric_type,
                                    D.data_ptr(), I.data_ptr(), _stream_ptr(self.devices[0]))
            )
            torch.cuda.synchronize(dev0)
        return D.cpu().numpy(), I.cpu().numpy()


def get_num_gpus() -> int:
    return int(_capi.load().keds_device_count())


def index_cpu_to_gpu(res, device: int, index: IndexFlat, options=None) -> GpuIndexFlat:
    g = GpuIndexFlat(index.d, index.metric_type, int(device))
    for blk in index._blocks:
        g.add(blk)
    return g


def index_cpu_to_all_gpus(index: IndexFlat, co: Optional[GpuMultipleClonerOptions] = None, ngpu: int = -1):
    n = get_num_gpus() if ngpu is None or ngpu < 0 else int(ngpu)
    if n <= 0:
        raise RuntimeError("no CUDA device: keds_b200 has no CPU fallback")
    devices = list(range(n))
    if n == 1:
        return index_cpu_to_gpu(None, 0, index)
    cls = IndexShards if (co is not None and getattr(co, "shard", False)) else IndexReplicas
    multi = cls(index.d, index.metric_type, devices)
    if index._blocks:
        multi.add(np.concatenate(index._blocks))
    return multi


def index_gpu_to_cpu(index) -> IndexFlat:
    raise RuntimeError("keds_b200 keeps no CPU search path; rebuild the index from the .pt database")
