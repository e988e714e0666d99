"""The row-sharded retrieval step on every rank of a torchrun job, against an unsharded retrieve2.

    torchrun --nproc_per_node=8 scripts/test_sharded_retrieve2_multigpu.py --out profiles/r05_sharded_retrieve2_8gpu.json

Runs the cases of tests/test_gpu_sharded_retrieve.py (IP / L2, k = 16 / 64, pool modes 0 / 1 / 2,
perm_img, exclusion with E = 1 and 8, a strict sub-range of rows, two passes, the exact fallback,
an exact-only tiny shard, an empty shard, consecutive steps, re-attachment, the refusal of changed
rows, and the bare sharded search with exclusion) on R ranks. Then, for the same rows and queries,
it checks that a one-rank ShardedKnowledgeBase on each rank's GPU returns the R-rank step's D, I,
gathered rows and pools bit for bit. Pools depend on neither the shard count nor the rank, so equality with R = 1
on every run (R = 1, 2, 8) makes them equal across shard counts. With fewer GPUs than ranks, ranks
share GPUs over gloo (the multi-rank paths run, the bytes do not cross NVLink). Rank 0 writes one
JSON document (card name and power limit included); exits 1 on a failure.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import traceback

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from test_gpu_sharded_retrieve import init_ranks, run_cases, unit  # noqa: E402


def card() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True).stdout.strip().splitlines()
        name, power = out[0].split(", ")
        return {"name": name, "power_limit": power, "gpus": len(out)}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def pools_across_shard_counts(rank, world, dev) -> dict:
    """Same rows, same queries, same block of rows: the R-rank step and a one-rank step agree."""
    from keds_b200.index import METRIC_INNER_PRODUCT as IP, METRIC_L2 as L2
    from keds_b200.sharded import ShardedKnowledgeBase

    n = 50000
    img, txt = unit(n, 101), unit(n, 102)
    q = unit(128 * world, 103).to(dev)
    perm = torch.randperm(16, generator=torch.Generator().manual_seed(104))
    lo, hi = 128 * rank, 128 * (rank + 1)
    solos = [dist.new_group([r]) for r in range(world)]  # collective: every rank creates every group
    res = {}
    for metric in (IP, L2):
        for mode in (1, 2):
            outs = []
            for group in (None, solos[rank]):
                kb = ShardedKnowledgeBase(768, metric, device=dev.index, group=group)
                kb.add(img, txt)
                o = kb.retrieve2(q, 16, perm_img=perm, pool_mode=mode, rows=(lo, hi))
                kb.exchange_stats()
                outs.append({k: v.clone() for k, v in o.items()})
            same = all(torch.equal(outs[0][k].view(torch.int32) if outs[0][k].dtype == torch.float32 else outs[0][k],
                                   outs[1][k].view(torch.int32) if outs[1][k].dtype == torch.float32 else outs[1][k])
                       for k in outs[0])
            res[f"{'l2' if metric == L2 else 'ip'}_pool{mode}"] = bool(same)
    return res


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = init_ranks(rank, world)
    result = {"ranks": world, "backend": dist.get_backend(), "card": card()}
    ok = True
    try:
        run_cases(rank, world, dev)
        result["cases_ok"] = True
    except Exception:  # noqa: BLE001
        result["cases_ok"] = False
        result["error"] = traceback.format_exc()[-3000:]
        ok = False
    if ok:
        result["bit_identical_to_one_rank"] = pools_across_shard_counts(rank, world, dev)
        ok = all(result["bit_identical_to_one_rank"].values())
    every = [None] * world
    dist.all_gather_object(every, result)
    dist.destroy_process_group()
    if rank == 0:
        doc = {"ok": all(r.get("cases_ok") and all(r.get("bit_identical_to_one_rank", {"-": False}).values())
                         for r in every), "per_rank": every}
        text = json.dumps(doc, indent=1)
        print(text)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(text + "\n")
        sys.exit(0 if doc["ok"] else 1)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
