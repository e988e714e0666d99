"""Same-process A/B of the end-to-end retrieval step (RetrievalStep: pinned host queries in, (D, I)
on the host out, one graph launch + one stream sync per step): copy nodes around the search vs
host I/O through the mapping (keds_retrieve2 with host mirrors), interleaved.
-> gpurun_out/ab_hostio.json"""
from __future__ import annotations

import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from keds_b200 import retrieval as kr  # noqa: E402
from keds_b200.index import METRIC_INNER_PRODUCT, GpuIndexFlat  # noqa: E402

D, N, B, K = 768, 500_000, 128, 16
dev = torch.device("cuda", 0)


def db(n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(n, D, generator=g, device="cuda")
    return x / x.norm(dim=1, keepdim=True)


ia, ib = GpuIndexFlat(D, METRIC_INNER_PRODUCT, 0), GpuIndexFlat(D, METRIC_INNER_PRODUCT, 0)
ia.add(db(N, 1))
ib.add(db(N, 2))
q_host = db(B, 3).cpu().pin_memory()
q_dev = q_host.cuda()
perm = torch.randperm(K, generator=torch.Generator().manual_seed(999)).to(dev, torch.int32)
steps = int(sys.argv[1]) if len(sys.argv) > 1 else 300


def loop(fn, n):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3


res = []
ref = None
steps_cn = {True: kr.RetrievalStep(ia, ib, B, K, perm_img=perm, want_feats=True, pool_mode=kr.POOL_SOFTMAX, tau=100.0, copy_nodes=True),
            False: kr.RetrievalStep(ia, ib, B, K, perm_img=perm, want_feats=True, pool_mode=kr.POOL_SOFTMAX, tau=100.0, copy_nodes=False)}
for st in steps_cn.values():
    st.q_host.copy_(q_host)
for rep in range(6):
    for copy_nodes in (True, False):
        st = steps_cn[copy_nodes]
        us = loop(st.run, steps)
        if ref is None:
            ref = (st.I_img.clone(), st.I_txt.clone(), st.D_img.clone(), st.D_txt.clone())
        same = all(torch.equal(a, b) for a, b in zip(ref, (st.I_img, st.I_txt, st.D_img, st.D_txt)))
        res.append({"copy_nodes": copy_nodes, "e2e_us": round(us, 2), "same": same})
        print(json.dumps(res[-1]), flush=True)
os.makedirs("gpurun_out", exist_ok=True)
json.dump(res, open("gpurun_out/ab_hostio.json", "w"), indent=1)
