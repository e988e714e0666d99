"""The neighbour consumer on row-sharded bases, on every rank of a torchrun job, against the local
consumer on full copies of the bases.

    torchrun --nproc_per_node=8 scripts/test_sharded_consumer_multigpu.py --out profiles/r07_sharded_consumer_8gpu.json

Runs the cases of tests/test_gpu_sharded_consumer.py (eval tokens for IP / L2, k = 16 / 64, with and
without perm, -1 padding, labels outside every shard, an empty shard; from_features on the sharded
base against an unsharded KnowledgeBase with unequal batches, with and without exclusion; training
forward + backward in train() and eval(); a step that grows the exchange; the refusals) on
R = WORLD_SIZE ranks, one GPU each, so that (R-1)/R of the neighbour rows cross NVLink. Rank 0
writes one JSON document (card name and power limit included); exits 1 on a failure.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time
import traceback

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch.distributed as dist  # noqa: E402

from test_gpu_sharded_consumer import init_ranks, run_cases  # noqa: E402


def card() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True).stdout.strip().splitlines()
        name, power = out[0].split(", ")
        return {"name": name, "power_limit": power, "gpus": len(out)}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = init_ranks(rank, world)
    result = {"rank": rank, "device": str(dev)}
    t0 = time.time()
    try:
        run_cases(rank, world, dev)
        result["cases_ok"] = True
    except Exception:  # noqa: BLE001
        result["cases_ok"] = False
        result["error"] = traceback.format_exc()[-3000:]
    result["seconds"] = round(time.time() - t0, 1)
    every = [None] * world
    dist.all_gather_object(every, result)
    backend = dist.get_backend()
    dist.destroy_process_group()
    if rank == 0:
        doc = {"ok": all(r["cases_ok"] for r in every), "ranks": world, "backend": backend, "card": card(),
               "per_rank": every}
        text = json.dumps(doc, indent=1)
        print(text)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(text + "\n")
        sys.exit(0 if doc["ok"] else 1)
    sys.exit(0 if result["cases_ok"] else 1)


if __name__ == "__main__":
    main()
