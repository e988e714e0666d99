"""Per-step time of the row-sharded DDP retrieval step against the replicated step.

    torchrun --nproc_per_node=R scripts/perf_sharded_retrieve2.py --rows 500000 --out profiles/r05_perf_sharded_R.json

Workload: 128 queries per rank, two bases of --rows rows each (768-d unit rows), k = 16, gathered
neighbours and softmax pool (tau = 100), the image stream permuted. The sharded step is one
ShardedKnowledgeBase.retrieve2 over the R * 128 queries of all ranks with rows = this rank's block. The
replicated step is retrieval.retrieve2 of this rank's 128 queries on a full copy of both bases. At
R = 1 the shard's own indices are that full copy. Both run alternately, round after round. Step times come
from CUDA events around back-to-back steps, with the median over rounds. A separate profiled pass (torch.profiler,
CUDA activities) splits the sharded step into scoring (k_score_topk + k_prep_rows), re-rank
(k_select_rerank), exact fallback, merge (k_topk_merge, including its wait for the peers) and
k_shard_consume; exchange_stats gives the merge's wait for the peers. Rank 0 writes one JSON
document with the card name and power limit.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from test_gpu_sharded_retrieve import init_ranks  # noqa: E402

D, K, B = 768, 16, 128


def card() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = out[0].split(", ")
    return {"name": name, "power_limit": power, "max_sm_clock": clock, "gpus": len(out)}


def unit_rows(n, seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    x = torch.randn(n, D, generator=g, device=dev)
    return x / x.norm(dim=1, keepdim=True)


def timed(fn, steps, dev):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) * 1000.0 / steps  # us per step


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=500000, help="rows per base")
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = init_ranks(rank, world)
    if torch.cuda.device_count() < world:
        raise SystemExit("perf_sharded_retrieve2: one GPU per rank is needed (shared GPUs time-slice)")

    from keds_b200 import retrieval as kr
    from keds_b200.index import METRIC_INNER_PRODUCT, GpuIndexFlat
    from keds_b200.sharded import ShardedKnowledgeBase, shard_bounds

    kb = ShardedKnowledgeBase(D, METRIC_INNER_PRODUCT, device=dev.index)
    full = []
    for db, seed in ((kb.image, 1), (kb.text, 2)):
        x = unit_rows(args.rows, seed, dev)  # the same matrix on every rank (same seed)
        lo, hi = shard_bounds(args.rows, world, rank)
        db.add_local(x[lo:hi], lo, args.rows)
        if world > 1:
            ix = GpuIndexFlat(D, METRIC_INNER_PRODUCT, dev.index)
            ix.add(x)
            full.append(ix)
        del x
    if world == 1:
        full = [kb.image.local, kb.text.local]
    torch.cuda.empty_cache()
    q_all = unit_rows(world * B, 3, dev)
    q_mine = q_all[rank * B:(rank + 1) * B].contiguous()
    perm = torch.randperm(K, generator=torch.Generator().manual_seed(4)).to(dev)
    rows = (rank * B, (rank + 1) * B)
    out_s, out_r = {}, {}

    def sharded():
        kb.retrieve2(q_all, K, perm_img=perm, pool_mode=2, rows=rows, out=out_s)

    def replica():
        kr.retrieve2(full[0], full[1], q_mine, K, perm_img=perm, want_feats=True, pool_mode=2, out=out_r)

    for fn in (sharded, replica):
        timed(fn, 20, dev)
    kb.exchange_stats()
    t_s, t_r = [], []
    for r in range(args.rounds):
        for name, fn in ((("sharded", sharded), ("replica", replica)) if r % 2 == 0 else
                         (("replica", replica), ("sharded", sharded))):
            dist.barrier()
            (t_s if name == "sharded" else t_r).append(timed(fn, args.steps, dev))
    wait = kb.exchange_stats()
    same = torch.equal(out_s["I_img"][rows[0]:rows[1]], out_r["I_img"]) and \
        torch.equal(out_s["feat_img"].view(torch.int32), out_r["feat_img"].view(torch.int32))

    # kernel split of the sharded step, in a profiled pass of its own
    from torch.profiler import ProfilerActivity, profile

    n_prof = 20
    dist.barrier()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n_prof):
            sharded()
        torch.cuda.synchronize(dev)
    groups = {"scoring": ("k_score_topk", "k_prep_rows"), "rerank": ("k_select_rerank",),
              "exact_fallback": ("k_exact_fallback", "k_flag_all"), "merge": ("k_topk_merge",),
              "shard_consume": ("k_shard_consume",), "push": ("k_p2p_push", "k_fill_pad")}
    split = {g: 0.0 for g in groups}
    for ev in prof.key_averages():
        for g, names in groups.items():
            if any(n in ev.key for n in names):
                split[g] += ev.device_time_total / n_prof  # us per step
    res = {"rank": rank, "sharded_us": statistics.median(t_s), "replica_us": statistics.median(t_r),
           "sharded_range_us": [min(t_s), max(t_s)], "replica_range_us": [min(t_r), max(t_r)],
           "kernel_us_per_step": {k: round(v, 2) for k, v in split.items()},
           "merge_wait_us": wait, "own_block_identical_to_replica": bool(same)}
    every = [None] * world
    dist.all_gather_object(every, res)
    dist.destroy_process_group()
    if rank == 0:
        doc = {"workload": {"queries_per_rank": B, "rows_per_base": args.rows, "k": K, "d": D,
                            "pool": "softmax(tau=100 * D)", "ranks": world, "steps": args.steps,
                            "rounds": args.rounds},
               "card": card(), "per_rank": every,
               "sharded_over_replica": statistics.median(r["sharded_us"] / r["replica_us"] for r in every)}
        text = json.dumps(doc, indent=1)
        print(text)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(text + "\n")


if __name__ == "__main__":
    main()
