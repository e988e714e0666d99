"""Time of the neighbour consumer on row-sharded bases against the local consumer and against the
route a sharded user has without it.

    torchrun --nproc_per_node=R scripts/perf_sharded_consumer.py --out profiles/r07_perf_sharded_consumer_Rgpu.json

Workload (per rank): B = 128 queries, k = 16, two bases of --rows (500,000) 768-d unit rows sharded
over the R ranks (one GPU each), the reference's consumer widths (768 / 512 / 768, 2 hidden layers,
3 cross-attention layers, 8 x 64 heads), dropout 0.1 in training. Every rank also holds full local
copies of both bases for the local route. Measured, each as the median of per-call CUDA-event times
over --calls calls after warm-up, the two routes of a pair alternating round by round:

  (a) eval forward: NeighbourConsumer over the sharded bases (rows read from their owners, (R-1)/R of
      them over NVLink) against the same call on the local copies, with the same labels;
  (b) training forward + backward: TrainableNeighbourConsumer, both routes, same labels;
  (c) the whole sharded DDP step: gather_ddp_step + ShardedKnowledgeBase.retrieve2(want_feats=False) +
      the consumer over this rank's labels (eval forward; and training forward + backward);
  (d) what a sharded user runs without the sharded consumer: retrieval.get_retrieved_features (the
      same gathers + retrieve2 with [B, k, 768] features) + IM2TEXT / CrossFormer x 2 in eager
      PyTorch (fp32 matmuls; eval forward under no_grad, and training forward + backward).

Tokens of (a) and (b) are checked bit for bit between the routes. Rank 0 writes one JSON document
with the card name, power limit and SM clock limit.
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
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from perf_consumer_train import eager_tokens  # noqa: E402
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


def per_call_us(fn, calls, dev):
    """per-call CUDA-event times (us) of `calls` back-to-back calls"""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(calls)]
    for e0, e1 in ev:
        e0.record()
        fn()
        e1.record()
    torch.cuda.synchronize(dev)
    return [e0.elapsed_time(e1) * 1000.0 for e0, e1 in ev]


def compare(pair, calls, rounds, warmup, dev):
    """median per-call time of each route of `pair` (name -> fn), routes alternating by round"""
    names = list(pair)
    for n in names:
        per_call_us(pair[n], warmup, dev)
    times = {n: [] for n in names}
    for r in range(rounds):
        for n in (names if r % 2 == 0 else names[::-1]):
            dist.barrier()
            times[n] += per_call_us(pair[n], max(1, calls // rounds), dev)
    return {n: {"median_us": round(statistics.median(t), 2), "p10_us": round(sorted(t)[len(t) // 10], 2),
                "p90_us": round(sorted(t)[len(t) * 9 // 10], 2), "calls": len(t)} for n, t in times.items()}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=500000, help="rows per base")
    ap.add_argument("--calls", type=int, default=400)
    ap.add_argument("--rounds", type=int, default=8)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = init_ranks(rank, world)
    if torch.cuda.device_count() < world:
        raise SystemExit("perf_sharded_consumer: one GPU per rank is needed (shared GPUs time-slice)")

    from keds_b200.consumer import NeighbourConsumer, TrainableNeighbourConsumer
    from keds_b200.index import METRIC_INNER_PRODUCT, GpuIndexFlat
    from keds_b200.retrieval import get_retrieved_features
    from keds_b200.sharded import ShardedKnowledgeBase, gather_ddp_step, shard_bounds
    from oracle import consumer_oracle as corc

    kb = ShardedKnowledgeBase(D, METRIC_INNER_PRODUCT, device=dev.index)
    full = []
    for db, seed in ((kb.image, 1), (kb.text, 2)):
        x = unit_rows(args.rows, seed, dev)  # the same matrix on every rank (same seed)
        lo, hi = shard_bounds(args.rows, world, rank)
        db.add_local(x[lo:hi], lo, args.rows)
        ix = GpuIndexFlat(D, METRIC_INNER_PRODUCT, dev.index)
        ix.add(x)
        full.append(ix)
        del x
    torch.cuda.empty_cache()
    sds_np = corc.random_state_dicts(768, 512, 768, 2, 3, 8, 64, seed=11)
    sds = [{k: torch.from_numpy(v) for k, v in sd.items()} for sd in sds_np]
    cons = NeighbourConsumer(*sds, heads=8, device=dev.index)
    tmod = TrainableNeighbourConsumer(*sds, heads=8, device=dev.index, dropout=0.1).train()
    feat = 3.0 * torch.randn(B, D, generator=torch.Generator(device=dev).manual_seed(10 + rank), device=dev)
    q = feat / feat.norm(dim=1, keepdim=True)
    q_all, _, (lo, hi) = gather_ddp_step(q, None, kb.group, kb.device)
    out = kb.retrieve2(q_all, K, want_feats=False, rows=(lo, hi))
    I_img, I_txt = out["I_img"][lo:hi].clone(), out["I_txt"][lo:hi].clone()
    perm = torch.randperm(K, generator=torch.Generator().manual_seed(4)).to(device=dev, dtype=torch.int32)
    dtok = torch.randn(B, 3, D, generator=torch.Generator(device=dev).manual_seed(5), device=dev)
    res = {"rank": rank}

    # (a) eval forward, same labels
    tok = {}

    def eval_route(name, a, b):
        def run():
            tok[name] = cons(feat, a, b, I_img, I_txt, perm)
        return run

    res["a_eval_forward"] = compare({"sharded": eval_route("sharded", kb.image, kb.text),
                                     "local": eval_route("local", full[0], full[1])}, args.calls, args.rounds, 20, dev)
    res["a_tokens_identical"] = bool(torch.equal(tok["sharded"].view(torch.int32), tok["local"].view(torch.int32)))

    # (b) training forward + backward, same labels and dropout masks per call pair
    grads = {}

    def train_route(name, a, b):
        def run():
            tmod.flat.grad = None
            torch.manual_seed(7)
            tmod(feat, a, b, I_img, I_txt, perm).backward(dtok)
            grads[name] = tmod.flat.grad
        return run

    res["b_train_fwd_bwd"] = compare({"sharded": train_route("sharded", kb.image, kb.text),
                                      "local": train_route("local", full[0], full[1])}, args.calls, args.rounds, 20,
                                     dev)
    res["b_grads_identical"] = bool(torch.equal(grads["sharded"].view(torch.int32), grads["local"].view(torch.int32)))

    # (c) the whole sharded step with the consumer; (d) features + eager modules
    step = {}
    params = tuple({k: v.to(dev).requires_grad_(True) for k, v in sd.items()} for sd in sds)
    rows_i = torch.arange(B * K, device=dev).view(B, K)

    def sharded_step(train):
        def run():
            qa, _, (l0, h0) = gather_ddp_step(q, None, kb.group, kb.device)
            o = kb.retrieve2(qa, K, want_feats=False, rows=(l0, h0), out=step)
            if train:
                tmod.flat.grad = None
                tmod(feat, kb.image, kb.text, o["I_img"][l0:h0], o["I_txt"][l0:h0], perm).backward(dtok)
            else:
                cons(feat, kb.image, kb.text, o["I_img"][l0:h0], o["I_txt"][l0:h0], perm)
        return run

    def eager_step(train):
        def run():
            fi, ft = get_retrieved_features(feat, (None, None, None, kb.image, kb.text), topk=K)
            # the gathered features are the bases: rows i*K + j, read by eager_tokens' own gather
            if train:
                for sd in params:
                    for t in sd.values():
                        t.grad = None
                eager_tokens(params, 8, feat, fi.view(B * K, D), ft.view(B * K, D), rows_i, rows_i, 0.1).backward(dtok)
            else:
                with torch.no_grad():
                    eager_tokens(params, 8, feat, fi.view(B * K, D), ft.view(B * K, D), rows_i, rows_i, 0.0)
        return run

    torch.backends.cuda.matmul.allow_tf32 = False
    res["cd_eval"] = compare({"c_sharded_step_consumer": sharded_step(False), "d_features_eager": eager_step(False)},
                             args.calls, args.rounds, 10, dev)
    res["cd_train"] = compare({"c_sharded_step_consumer": sharded_step(True), "d_features_eager": eager_step(True)},
                              args.calls, args.rounds, 10, dev)
    kb.exchange_stats()
    every = [None] * world
    dist.all_gather_object(every, res)
    dist.destroy_process_group()
    if rank == 0:
        med = lambda key, route: statistics.median(r[key][route]["median_us"] for r in every)  # noqa: E731
        doc = {"workload": {"queries_per_rank": B, "rows_per_base": args.rows, "k": K, "d": D, "ranks": world,
                            "consumer": "768/512/768, 2 hidden, 3 layers, 8 x 64 heads, dropout 0.1 (train)",
                            "calls_per_route": args.calls, "rounds": args.rounds,
                            "peer_row_share": (world - 1) / world,
                            "rows_read_per_forward": 2 * B * K, "bytes_read_per_forward": 2 * B * K * D * 4},
               "card": card(),
               "summary_median_over_ranks_us": {
                   "a_eval_sharded": med("a_eval_forward", "sharded"), "a_eval_local": med("a_eval_forward", "local"),
                   "b_train_sharded": med("b_train_fwd_bwd", "sharded"), "b_train_local": med("b_train_fwd_bwd", "local"),
                   "c_step_eval": med("cd_eval", "c_sharded_step_consumer"),
                   "d_step_eval": med("cd_eval", "d_features_eager"),
                   "c_step_train": med("cd_train", "c_sharded_step_consumer"),
                   "d_step_train": med("cd_train", "d_features_eager")},
               "identical": all(r["a_tokens_identical"] and r["b_grads_identical"] for r in every),
               "per_rank": every}
        text = json.dumps(doc, indent=1)
        print(text)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(text + "\n")


if __name__ == "__main__":
    main()
