"""Cost of search with exclusion, and of the change on the plain entry points.

Loads two builds of libkeds_knn.so into one process (ctypes, RTLD_LOCAL: their symbols do not mix)
and times, round after round in rotating order on the same device-resident inputs:

  base     the plain entry point of a reference build (--base-lib, e.g. the parent commit's)
  plain    the plain entry point of this tree's build
  exclude  the same entry point of this tree's build with an exclusion array, E = 1: every query is
           a row of the base and leaves itself out (training without self-retrieval)

on three shapes: config 2 (retrieve2, 128 queries x 2 databases x 0.5M rows, k = 16, gathered
neighbours), config 1 (search, 4096 x 50k, k = 16) and 4096 x 0.5M; and base against plain (no
exclude variant) for gallery ranking at 4181 x 2297 (one pass) and 17,000 x 2297 (two passes) and
label hits at 10,000 x 50k (cut points 1, 5, 10, 50). Times are per call from CUDA
events around a back-to-back loop; the spread is the range over rounds, and the differences are
the median (and quartiles) of the per-round ratios of variants that ran back to back. Also checks that base and
plain return the same bits. Writes one JSON document (card name and power limit included).

    python scripts/perf_exclude.py --base-lib /path/to/parent/libkeds_knn.so --out perf.json
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from keds_b200 import _capi  # noqa: E402

D = 768
K = 16


class ParentAbi:
    """A build of the 0.1 ABI behind this build's calls. That ABI had one entry point per optional
    search input: each unified call goes to the one its arguments need (`_exclude` for an exclusion
    array, `_hostio` for retrieve2 with host mirrors), without the arguments that one lacks."""

    # unified call -> (position of exclude, n_exclude; position of retrieve2's four host mirrors)
    CALLS = {"keds_index_search_ex": (6, None), "keds_index_search2": (9, None),
             "keds_index_search_sharded": (7, None), "keds_retrieve2": (21, 13)}

    def __init__(self, lib):
        self._lib = lib
        self._twins = {}

    def _twin(self, name, exclude, hostio):
        """(the 0.1 entry point, the positions of the unified arguments it takes), set up once"""
        key = (name, exclude, hostio)
        if key not in self._twins:
            at_ex, at_mirrors = self.CALLS[name]
            drop = set() if exclude else {at_ex, at_ex + 1}
            if at_mirrors is not None and not hostio:
                drop |= set(range(at_mirrors, at_mirrors + 4))
            twin = name
            if exclude or hostio:
                twin = name.removesuffix("_ex") + ("_hostio" if hostio else "") + ("_exclude" if exclude else "")
            args = _capi.SIGNATURES[name][1]
            keep = [i for i in range(len(args)) if i not in drop]
            fn = getattr(self._lib, twin)
            fn.restype, fn.argtypes = C.c_int, [args[i] for i in keep]
            self._twins[key] = (fn, keep)
        return self._twins[key]

    def __getattr__(self, name):
        if name not in self.CALLS:
            return getattr(self._lib, name)
        at_ex, at_mirrors = self.CALLS[name]

        def call(*args):
            hostio = at_mirrors is not None and any(args[at_mirrors:at_mirrors + 4])
            fn, keep = self._twin(name, bool(args[at_ex]), hostio)
            return fn(*[args[i] for i in keep])
        return call


def load(path: str):
    """One build of the library with this tree's signatures (a build of the 0.1 ABI behind ParentAbi)."""
    lib = C.CDLL(path)
    for name, (res, args) in _capi.SIGNATURES.items():
        if hasattr(lib, name):
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
    return ParentAbi(lib) if lib.keds_version().split()[1] == b"0.1" else lib


def check(lib, rc):
    if rc != 0:
        raise RuntimeError(lib.keds_last_error().decode())


def make_index(lib, rows: torch.Tensor):
    h = C.c_void_p()
    check(lib, lib.keds_index_create(D, _capi.METRIC_IP, 0, C.byref(h)))
    check(lib, lib.keds_index_add_ex(h, rows.data_ptr(), rows.shape[0], 0))
    return h


def card() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # pragma: no cover
        return {"name": torch.cuda.get_device_name(0), "error": str(e)}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--base-lib", required=True, help="reference build of libkeds_knn.so (plain entry points)")
    ap.add_argument("--lib", default=_capi.LIB_PATH, help="this tree's build")
    ap.add_argument("--rounds", type=int, default=30)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    libs = {"base": load(os.path.abspath(args.base_lib)), "new": load(os.path.abspath(args.lib))}
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream(dev).cuda_stream
    g = torch.Generator(device=dev).manual_seed(0)

    def unit(n):
        x = torch.randn(n, D, generator=g, device=dev)
        return x / x.norm(dim=1, keepdim=True)

    big_a, big_b, small, gal = unit(500_000), unit(500_000), unit(50_000), unit(2297)
    idx = {name: {"a": make_index(lib, big_a), "b": make_index(lib, big_b), "s": make_index(lib, small),
                  "g": make_index(lib, gal)} for name, lib in libs.items()}
    torch.cuda.synchronize()

    perm = torch.randperm(K, generator=torch.Generator().manual_seed(1)).to(dev, torch.int32)
    shapes = {}
    for cfg, nq, n in (("cfg2_retrieve2_128x2x500k", 128, 500_000), ("cfg1_search_4096x50k", 4096, 50_000),
                       ("search_4096x500k", 4096, 500_000)):
        rows = torch.randperm(n, generator=torch.Generator().manual_seed(nq + n))[:nq]
        q = (big_a if n == 500_000 else small)[rows.to(dev)].contiguous()
        ex = rows.to(dev, torch.int64).reshape(nq, 1).contiguous()
        shapes[cfg] = (nq, q, ex)
    # gallery ranking: queries near random gallery rows, mid-ranked random targets, one excluded row each
    for cfg, nq in (("rank_4181x2297", 4181), ("rank_17000x2297", 17_000)):
        sel = torch.randint(0, 2297, (nq,), generator=g, device=dev)
        q = gal[sel] + 0.05 * unit(nq)
        q = (q / q.norm(dim=1, keepdim=True)).contiguous()
        tg_ex = torch.randint(0, 2297, (2, nq), generator=g, device=dev)
        shapes[cfg] = (nq, q, tg_ex)
    row_labels = torch.randint(0, 100, (50_000,), generator=g, device=dev)
    ks = np.array([1, 5, 10, 50], np.int32)  # (read on the host)
    rows = torch.randperm(50_000, generator=torch.Generator().manual_seed(7))[:10_000].to(dev)
    shapes["hits_10000x50k"] = (10_000, small[rows].contiguous(),
                                torch.randint(0, 100, (10_000,), generator=g, device=dev))

    def outputs(cfg, nq, feats):
        if cfg.startswith("rank"):
            return [torch.empty(nq, dtype=torch.int64, device=dev)]
        if cfg.startswith("hits"):
            return [torch.empty((nq, len(ks)), dtype=torch.int32, device=dev)]
        o = [torch.empty((nq, K), dtype=torch.float32, device=dev), torch.empty((nq, K), dtype=torch.int64, device=dev),
             torch.empty((nq, K), dtype=torch.float32, device=dev), torch.empty((nq, K), dtype=torch.int64, device=dev)]
        if feats:
            o += [torch.empty((nq, K, D), dtype=torch.float32, device=dev) for _ in range(2)]
        return o

    def call(cfg, variant):
        nq, q, ex = shapes[cfg]
        lib = libs["base" if variant == "base" else "new"]
        ix = idx["base" if variant == "base" else "new"]
        o = outs[(cfg, variant)]
        p = [t.data_ptr() for t in o]
        if cfg.startswith("rank"):
            return lambda: check(lib, lib.keds_index_rank(ix["g"], q.data_ptr(), nq, ex[0].data_ptr(), ex[1].data_ptr(),
                                                          p[0], st))
        if cfg.startswith("hits"):
            return lambda: check(lib, lib.keds_index_label_hits(ix["s"], q.data_ptr(), nq, row_labels.data_ptr(),
                                                                ex.data_ptr(), ks.ctypes.data, len(ks), p[0], st))
        exclusion =(ex.data_ptr(), 1) if variant == "exclude" else (None, 0)
        if cfg.startswith("cfg2"):
            return lambda: check(lib, lib.keds_retrieve2(ix["a"], ix["b"], q.data_ptr(), nq, K, perm.data_ptr(), None, 0,
                                                         100.0, p[0], p[1], p[2], p[3], None, None, None, None, p[4],
                                                         p[5], None, None, *exclusion, 0, st))
        h = ix["s"] if cfg.startswith("cfg1") else ix["a"]
        return lambda: check(lib, lib.keds_index_search_ex(h, q.data_ptr(), nq, K, p[0], p[1], *exclusion, 0, st))

    variants = {c: ("base", "plain") if c.startswith(("rank", "hits")) else ("base", "plain", "exclude")
                for c in shapes}
    outs = {(c, v): outputs(c, shapes[c][0], c.startswith("cfg2")) for c in shapes for v in variants[c]}
    fns = {(c, v): call(c, v) for c in shapes for v in variants[c]}
    iters = {"cfg2_retrieve2_128x2x500k": 50, "cfg1_search_4096x50k": 20, "search_4096x500k": 5,
             "rank_4181x2297": 20, "rank_17000x2297": 10, "hits_10000x50k": 10}
    for f in fns.values():  # warm-up: modules, scratch sizes, planner feedback
        for _ in range(5):
            f()
    torch.cuda.synchronize()

    times = {key: [] for key in fns}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for r in range(args.rounds):
        for c in shapes:
            vs = variants[c]
            order = vs[r % len(vs):] + vs[:r % len(vs)]
            for v in order:
                f = fns[(c, v)]
                f()
                e0.record()
                for _ in range(iters[c]):
                    f()
                e1.record()
                e1.synchronize()
                times[(c, v)].append(e0.elapsed_time(e1) * 1000.0 / iters[c])
    for name, lib in libs.items():
        for h in idx[name].values():
            check(lib, lib.keds_index_sync(h, st))

    result = {"card": card(), "rounds": args.rounds, "unit": "us per call", "configs": {}}
    for c in shapes:
        same = all(torch.equal(a, b) for a, b in zip(outs[(c, "base")], outs[(c, "plain")]))
        row = {"base_plain_outputs_identical": bool(same)}
        if "exclude" in variants[c]:
            I_ex = outs[(c, "exclude")][1]
            row["exclude_never_returns_self"] = bool(not (I_ex == shapes[c][2]).any().item())
        for v in variants[c]:
            t = times[(c, v)]
            row[v] = {"median": round(statistics.median(t), 2), "min": round(min(t), 2), "max": round(max(t), 2)}
        # paired within each round (the three variants ran back to back): median and range of the ratios
        for name, num, den in (("plain_vs_base_pct", "plain", "base"), ("exclude_vs_plain_pct", "exclude", "plain")):
            if num not in variants[c]:
                continue
            r = [100.0 * (a / b - 1.0) for a, b in zip(times[(c, num)], times[(c, den)])]
            row[name] = {"median": round(statistics.median(r), 2), "p25": round(statistics.quantiles(r, n=4)[0], 2),
                         "p75": round(statistics.quantiles(r, n=4)[2], 2)}
        result["configs"][c] = row
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    for name, lib in libs.items():
        for h in idx[name].values():
            lib.keds_index_free(h)


if __name__ == "__main__":
    main()
