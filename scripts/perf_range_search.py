"""Cost of the range search next to the top-k search, and of the builder's near-duplicate self-join.

  1. 4096 queries x 0.5M rows (d = 768, unit rows, inner product): range_search at the radii where
     the median query gets 16 and 256 rows, against search(k = 16) on the same device-resident data
     in the same process, in rotating order round after round. Per call: a host clock around the call
     and a device synchronisation (range_search synchronises by itself: it reads its result size
     back). Reported: medians and ranges over rounds, the median of the per-round ratios, and the
     hits per query.
  2. drop_near_duplicates over 0.5M rows (batch 65536, radius 0.95, 1,000 planted near-copies),
     end to end (index build included), and the eight range-search calls of its self-join alone.

Card name and power limit are read in the same run. Writes <out_dir>/perf_range_search.json.

    python scripts/perf_range_search.py --out-dir profiles
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from keds_b200.database import drop_near_duplicates  # noqa: E402
from keds_b200.index import METRIC_INNER_PRODUCT, GpuIndexFlat  # noqa: E402

N, D, NQ = 500_000, 768, 4096


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 else f"nvidia-smi failed: {out.stderr.strip()}"


def unit(n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(n, D, generator=g, device="cuda")
    return x / x.norm(dim=1, keepdim=True)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


def summary(v):
    return {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v), "n": len(v)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", required=True)
    ap.add_argument("--rounds", type=int, default=15)
    args = ap.parse_args()
    res = {"card (name, power limit, max SM clock)": card(), "shape": {"rows": N, "d": D, "queries": NQ}}

    x, q = unit(N, 1), unit(NQ, 2)
    ix = GpuIndexFlat(D, METRIC_INNER_PRODUCT, 0)
    ix.add(x)
    Dk, _ = ix.search(q, 256)
    ix.sync()
    radii = {"16": float(Dk[:, 15].median()), "256": float(Dk[:, 255].median())}
    res["radius"] = radii

    variants = {"search_k16": lambda: ix.search(q, 16)}
    for h, r in radii.items():
        variants[f"range_{h}"] = (lambda r=r: ix.range_search(q, r))
    names = list(variants)
    for name in names:  # warm-up: every shape and buffer size the timed window uses
        for _ in range(3):
            variants[name]()
    ix.sync()
    times = {n: [] for n in names}
    for rnd in range(args.rounds):
        for name in names[rnd % len(names):] + names[:rnd % len(names)]:
            ms, _ = timed(variants[name])
            times[name].append(ms)
    ix.sync()
    res["calls"] = {n: summary(v) for n, v in times.items()}
    for h in radii:
        ratios = [a / b for a, b in zip(times[f"range_{h}"], times["search_k16"])]
        res["calls"][f"range_{h}"]["ratio_to_search_k16_median"] = statistics.median(ratios)
        lims, _, _ = ix.range_search(q, radii[h])
        per = (lims[1:] - lims[:-1]).double()
        res["calls"][f"range_{h}"]["hits_per_query"] = {"median": float(per.median()), "mean": float(per.mean()),
                                                        "max": int(per.max())}
    del ix, Dk

    # the builder's self-join: 0.5M rows with 1,000 planted near-copies
    g = torch.Generator(device="cuda").manual_seed(3)
    img = x.clone()
    src = torch.randperm(N, generator=g, device="cuda")[:2000]
    a, b = torch.minimum(src[:1000], src[1000:]), torch.maximum(src[:1000], src[1000:])
    c = img[a] + 1e-3 * torch.randn(1000, D, generator=g, device="cuda")
    img[b] = c / c.norm(dim=1, keepdim=True)
    txt = torch.zeros(N, 1, device="cuda")
    names = [str(i) for i in range(N)]
    drop_near_duplicates(img[:70000], txt[:70000], names[:70000], 0.95, batch=65536)  # warm-up
    ms, out = timed(lambda: drop_near_duplicates(img, txt, names, 0.95, batch=65536))
    join = GpuIndexFlat(D, METRIC_INNER_PRODUCT, 0)
    join.add(img, normalize=True)
    rows = torch.from_numpy(join.get_rows()).cuda()
    join_ms = []
    for _ in range(3):
        t, _ = timed(lambda: [join.range_search(rows[b0:b0 + 65536], 0.95) for b0 in range(0, N, 65536)])
        join_ms.append(t)
    res["self_join"] = {"rows": N, "radius": 0.95, "batch": 65536, "planted_pairs": 1000,
                        "dropped": int(out[3].numel()),
                        "drop_near_duplicates_ms": ms, "range_search_calls_ms": summary(join_ms)}
    os.makedirs(args.out_dir, exist_ok=True)
    path = os.path.join(args.out_dir, "perf_range_search.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
