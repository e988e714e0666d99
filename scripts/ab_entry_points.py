"""Every search entry point of two builds of libkeds_knn.so, on the same seeded inputs, bit for bit.

Loads a reference build (--base-lib, e.g. the parent commit's) and this tree's build into one
process (scripts/perf_exclude.py's loader) and runs each call on both, each build on its own
handles over the same rows: search with flags 0 / exact-only / no-fallback / force-IP, search2,
host (numpy-style) and device I/O, exclusion in search, search2 and retrieve2 (device and
page-locked host labels), retrieve2 with gathered neighbours, pools and host mirrors, label hits
(one and two passes), rank (one and two passes; misaligned queries; an inflated error bound that
sends queries to the exact recount), debug_scores and a one-rank sharded search, over
B = 7 .. 17,000, k = 16 / 200 / 600, IP and L2, fp16 and bf16. A reference build of the 0.1 ABI,
which had one entry point per optional search input, is called through the loader's ParentAbi.
Every output and every last_stats field must be identical, except launches and n_flagged of a
multi-pass rank call (summed over its passes; a reference build may report its last pass's). A
two-database search whose first database is empty is checked against the CPU oracle instead (its
status is reported differently by design). Writes one JSON document (card name and power limit
included); exits 1 on a mismatch.

    python scripts/ab_entry_points.py --base-lib /path/to/parent/libkeds_knn.so --out ab.json
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from keds_b200 import _capi  # noqa: E402
from oracle import knn_oracle as orc  # noqa: E402
from perf_exclude import card, check, load  # noqa: E402

D = 768


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--base-lib", required=True)
    ap.add_argument("--lib", default=_capi.LIB_PATH)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    libs = {"base": load(os.path.abspath(args.base_lib)), "new": load(os.path.abspath(args.lib))}
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream(dev).cuda_stream
    g = torch.Generator(device=dev).manual_seed(0)

    def unit(n, d=D):
        x = torch.randn(n, d, generator=g, device=dev)
        return x / x.norm(dim=1, keepdim=True)

    rows = {"a": unit(50_000), "b": unit(50_000), "gal": unit(2297)}
    handles = {name: {} for name in libs}

    def index(name, key, metric, fmt):
        """handle of build `name` over rows[key] (created once per metric and format)"""
        hk = (key, metric, fmt)
        if hk not in handles[name]:
            lib = libs[name]
            h = C.c_void_p()
            check(lib, lib.keds_index_create(D, metric, 0, C.byref(h)))
            if key != "empty":
                r = rows[key]
                check(lib, lib.keds_index_add_ex(h, r.data_ptr(), r.shape[0], 0))
            check(lib, lib.keds_index_set_operand_format(h, fmt))
            handles[name][hk] = h
        return handles[name][hk]

    def stats(lib, h):
        s = _capi.SearchStats()
        check(lib, lib.keds_index_last_stats(h, C.byref(s)))
        return {f: (list(getattr(s, f)) if f == "n_flagged" else getattr(s, f)) for f, _ in s._fields_}

    def queries(B, key="a"):
        src = rows[key]
        sel = torch.randint(0, src.shape[0], (B,), generator=g, device=dev)
        return (src[sel] + 0.05 * unit(B)).contiguous(), sel

    results, failures = [], []

    def compare(label, run, handle_keys, outs_of, oracle=None, loose=()):
        """run(name, lib, hs) on both builds; outs_of(name) -> list of tensors / arrays to compare;
        loose: last_stats fields the builds may report differently for this call"""
        got = {}
        for name, lib in libs.items():
            hs = [index(name, *hk) for hk in handle_keys]
            run(name, lib, hs)
            check(lib, lib.keds_index_sync(hs[0], st))
            torch.cuda.synchronize()
            got[name] = ([o.clone() if isinstance(o, torch.Tensor) else np.copy(o) for o in outs_of(name)],
                         stats(lib, hs[0]))
        (ob, sb), (on, sn) = got["base"], got["new"]
        same = all((torch.equal(x.view(torch.uint8), y.view(torch.uint8)) if isinstance(x, torch.Tensor)
                    else np.array_equal(x.view(np.uint8), y.view(np.uint8))) for x, y in zip(ob, on))
        row = {"call": label, "outputs_identical": bool(same), "stats_identical": sb == sn, "stats": sn}
        if loose:
            row["stats_base"] = sb
            row["stats_may_differ_in"] = list(loose)
        if oracle is not None:
            row["oracle_ok"] = bool(oracle(on))
            ok = row["oracle_ok"]
        else:
            ok = same and all(sb[f] == sn[f] for f in sb if f not in loose)
        results.append(row)
        if not ok:
            failures.append(row)
        print(json.dumps(row), flush=True)

    def dev_out(B, k, n=1):
        return [torch.empty((B, k), dtype=dt, device=dev) for _ in range(n) for dt in (torch.float32, torch.int64)]

    # search / search_ex over shapes, metrics, formats and flags
    for metric in (_capi.METRIC_IP, _capi.METRIC_L2):
        for fmt in (1, 0):  # fp16, bf16
            for B in (7, 128, 4096, 17000):
                for k in (16, 200, 600):
                    q, _ = queries(B)
                    outs = {n: dev_out(B, k) for n in libs}
                    compare(f"search m{metric} f{fmt} B{B} k{k}",
                            lambda n, lib, hs: check(lib, lib.keds_index_search_ex(
                                hs[0], q.data_ptr(), B, k, outs[n][0].data_ptr(), outs[n][1].data_ptr(), None, 0, 0, st)),
                            [("a", metric, fmt)], lambda n: outs[n])
    for flags in (_capi.SEARCH_EXACT_ONLY, _capi.SEARCH_NO_FALLBACK, _capi.SEARCH_FORCE_IP):
        for B in (128, 4096):
            q, _ = queries(B)
            outs = {n: dev_out(B, 16) for n in libs}
            compare(f"search flags{flags} B{B}",
                    lambda n, lib, hs: check(lib, lib.keds_index_search_ex(
                        hs[0], q.data_ptr(), B, 16, outs[n][0].data_ptr(), outs[n][1].data_ptr(), None, 0, flags, st)),
                    [("a", _capi.METRIC_L2, 1)], lambda n: outs[n])

    # host I/O (numpy-style): search and search2
    for B in (7, 128, 17000):
        qh = queries(B)[0].cpu().numpy()
        outs = {n: [np.empty((B, 16), dt) for _ in range(2) for dt in (np.float32, np.int64)] for n in libs}
        compare(f"search host B{B}",
                lambda n, lib, hs: check(lib, lib.keds_index_search_ex(
                    hs[0], qh.ctypes.data, B, 16, outs[n][0].ctypes.data, outs[n][1].ctypes.data, None, 0, 0, st)),
                [("a", _capi.METRIC_IP, 1)], lambda n: outs[n][:2])
        compare(f"search2 host B{B}",
                lambda n, lib, hs: check(lib, lib.keds_index_search2(
                    hs[0], hs[1], qh.ctypes.data, B, 16, *[o.ctypes.data for o in outs[n]], None, 0, 0, st)),
                [("a", _capi.METRIC_IP, 1), ("b", _capi.METRIC_IP, 1)], lambda n: outs[n])

    # search2 and the exclusion variants on device memory
    for B in (7, 128, 4096, 17000):
        for k in (16, 200):
            q, sel = queries(B)
            ex = torch.stack([sel, (sel + 1) % 50_000], 1).contiguous()
            outs = {n: dev_out(B, k, 2) for n in libs}
            p = lambda n: [o.data_ptr() for o in outs[n]]  # noqa: E731
            two = [("a", _capi.METRIC_IP, 1), ("b", _capi.METRIC_IP, 1)]
            compare(f"search2 B{B} k{k}", lambda n, lib, hs: check(lib, lib.keds_index_search2(
                hs[0], hs[1], q.data_ptr(), B, k, *p(n), None, 0, 0, st)), two, lambda n: outs[n])
            compare(f"search_exclude B{B} k{k}", lambda n, lib, hs: check(lib, lib.keds_index_search_ex(
                hs[0], q.data_ptr(), B, k, *p(n)[:2], ex.data_ptr(), 2, 0, st)), two[:1], lambda n: outs[n][:2])
            compare(f"search2_exclude B{B} k{k}", lambda n, lib, hs: check(lib, lib.keds_index_search2(
                hs[0], hs[1], q.data_ptr(), B, k, *p(n), ex.data_ptr(), 2, 0, st)), two, lambda n: outs[n])

    # retrieve2: gathered neighbours, pools, host mirrors, exclusion
    perm = torch.randperm(16, generator=torch.Generator().manual_seed(1)).to(dev, torch.int32)
    for B in (7, 128, 4096):
        q, sel = queries(B)
        qp = q.cpu().pin_memory()
        ex = torch.stack([sel, torch.full_like(sel, -1)], 1).contiguous()
        exp_ = ex.cpu().pin_memory()
        two = [("a", _capi.METRIC_IP, 1), ("b", _capi.METRIC_IP, 1)]
        for variant in ("plain", "exclude", "hostio", "hostio_exclude"):
            outs = {n: dev_out(B, 16, 2) + [torch.empty((B, 16, D), device=dev) for _ in range(2)]
                    + [torch.empty((B, D), device=dev) for _ in range(2)]
                    + [t.pin_memory() for t in (torch.empty(B, 16), torch.empty(B, 16, dtype=torch.int64),
                                                torch.empty(B, 16), torch.empty(B, 16, dtype=torch.int64))]
                    for n in libs}

            def run(n, lib, hs, variant=variant, outs=outs, q=q, qp=qp, ex=ex, exp_=exp_, B=B):
                o = [t.data_ptr() for t in outs[n]]
                head = (hs[0], hs[1], (qp if "hostio" in variant else q).data_ptr(), B, 16, perm.data_ptr(), None, 2,
                        100.0, *o[:4])
                mirrors = o[8:12] if "hostio" in variant else (None,) * 4
                exclusion = {"plain": (None, 0), "exclude": (ex.data_ptr(), 2), "hostio": (None, 0),
                             "hostio_exclude": (exp_.data_ptr(), 2)}[variant]
                check(lib, lib.keds_retrieve2(*head, *mirrors, o[4], o[5], o[6], o[7], *exclusion, 0, st))
            compare(f"retrieve2 {variant} B{B}", run, two,
                    lambda n, outs=outs, variant=variant: outs[n] if "hostio" in variant else outs[n][:8])

    # label hits, rank, debug_scores, one-rank sharded search
    q, sel = queries(10_000)
    row_labels = torch.randint(0, 100, (50_000,), generator=g, device=dev)
    qlabel = torch.randint(0, 100, (10_000,), generator=g, device=dev)
    ks = np.array([1, 5, 10, 50], np.int32)  # (read on the host)
    hits = {n: torch.empty((10_000, 4), dtype=torch.int32, device=dev) for n in libs}
    compare("label_hits 10000x50k", lambda n, lib, hs: check(lib, lib.keds_index_label_hits(
        hs[0], q.data_ptr(), 10_000, row_labels.data_ptr(), qlabel.data_ptr(), ks.ctypes.data, 4,
        hits[n].data_ptr(), st)), [("a", _capi.METRIC_IP, 1)], lambda n: [hits[n]])
    q, _ = queries(17_000)
    qlabel2 = torch.randint(0, 100, (17_000,), generator=g, device=dev)
    hits2 = {n: torch.empty((17_000, 4), dtype=torch.int32, device=dev) for n in libs}
    compare("label_hits 17000x50k (two passes)", lambda n, lib, hs: check(lib, lib.keds_index_label_hits(
        hs[0], q.data_ptr(), 17_000, row_labels.data_ptr(), qlabel2.data_ptr(), ks.ctypes.data, 4,
        hits2[n].data_ptr(), st)), [("a", _capi.METRIC_IP, 1)], lambda n: [hits2[n]])
    for B in (4181, 17_000):
        q, _ = queries(B, "gal")
        target = torch.randint(0, 2297, (B,), generator=g, device=dev)
        excl = torch.randint(0, 2297, (B,), generator=g, device=dev)
        flat = torch.empty(B * D + 1, device=dev)
        q_mis = flat[1:].view(B, D)  # starts 4 bytes past a 16-byte boundary: ranked from an aligned copy
        q_mis.copy_(q)
        loose = ("launches", "n_flagged") if B > 16_384 else ()
        for variant, qq, eps in (("", q, 1.0), (" misaligned q", q_mis, 1.0), (" eps x200 (recount queue)", q, 200.0)):
            ranks = {n: torch.empty(B, dtype=torch.int64, device=dev) for n in libs}

            def run(n, lib, hs, qq=qq, eps=eps, B=B, target=target, excl=excl, ranks=ranks):
                check(lib, lib.keds_index_set_eps_scale(hs[0], eps))
                check(lib, lib.keds_index_rank(hs[0], qq.data_ptr(), B, target.data_ptr(), excl.data_ptr(),
                                               ranks[n].data_ptr(), st))
                check(lib, lib.keds_index_set_eps_scale(hs[0], 1.0))
            compare(f"rank {B}x2297{variant}", run, [("gal", _capi.METRIC_IP, 1)],
                    lambda n, ranks=ranks: [ranks[n]], loose=loose)
    q, _ = queries(128)
    scores = {n: torch.empty((128, 50_000), device=dev) for n in libs}
    compare("debug_scores 128x50k", lambda n, lib, hs: check(lib, lib.keds_debug_scores(
        hs[0], q.data_ptr(), 128, scores[n].data_ptr(), st)), [("a", _capi.METRIC_IP, 1)], lambda n: [scores[n]])
    q, _ = queries(4096)
    bufs = {n: torch.zeros(32 << 20, dtype=torch.uint8, device=dev) for n in libs}
    outs = {n: dev_out(4096, 16) for n in libs}
    exch = {}
    for n, lib in libs.items():
        h = C.c_void_p()
        check(lib, lib.keds_exchange_create(1, 0, 0, (C.c_void_p * 1)(bufs[n].data_ptr()), bufs[n].numel(),
                                            C.byref(h)))
        exch[n] = h
    compare("search_sharded 1 rank 4096x50k", lambda n, lib, hs: check(lib, lib.keds_index_search_sharded(
        hs[0], exch[n], q.data_ptr(), 4096, 16, outs[n][0].data_ptr(), outs[n][1].data_ptr(), None, 0, st)),
        [("a", _capi.METRIC_IP, 1)], lambda n: outs[n])

    # the empty-database route: against the oracle (the status of the call is reported differently)
    a_np = rows["a"].cpu().numpy()
    for B in (128, 16_684):
        q, sel = queries(B)
        for excl in (False, True):
            ex = torch.stack([sel, torch.full_like(sel, -1)], 1).contiguous()
            outs = {n: dev_out(B, 16, 2) for n in libs}

            def run(n, lib, hs, outs=outs, ex=ex, excl=excl, q=q, B=B):
                p = [o.data_ptr() for o in outs[n]]
                exclusion = (ex.data_ptr(), 2) if excl else (None, 0)
                check(lib, lib.keds_index_search2(hs[0], hs[1], q.data_ptr(), B, 16, *p, *exclusion, 0, st))

            def oracle(o, q=q, ex=ex, excl=excl):
                if not (o[1] == -1).all():
                    return False
                n = 256
                qs = q[:n].cpu().numpy()
                Dr, Ir = orc.search(a_np, qs, 18 if excl else 16, "ip")
                if excl:
                    e = ex[:n].cpu().numpy()
                    gone = ((Ir[:, :, None] == e[:, None, :]) & (e[:, None, :] >= 0)).any(2)
                    order = np.argsort(gone, axis=1, kind="stable")[:, :16]
                    Dr, Ir = np.take_along_axis(Dr, order, 1), np.take_along_axis(Ir, order, 1)
                c = orc.compare_topk(Dr, Ir, o[2][:n].cpu().numpy(), o[3][:n].cpu().numpy(), None, None, "ip",
                                     1e-5, 1e-4)
                return c["ok"]
            compare(f"search2 empty-first B{B} exclude={excl}", run,
                    [("empty", _capi.METRIC_IP, 1), ("a", _capi.METRIC_IP, 1)], lambda n, outs=outs: outs[n], oracle)

    for n, lib in libs.items():
        lib.keds_exchange_free(exch[n])
        for h in handles[n].values():
            lib.keds_index_free(h)
    doc = {"card": card(), "calls": len(results), "mismatches": len(failures), "results": results}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)
    print(json.dumps({"card": doc["card"], "calls": doc["calls"], "mismatches": doc["mismatches"]}))
    sys.exit(1 if failures else 0)


if __name__ == "__main__":
    main()
