"""CPU: host-side mirror of the Faiss surface (argument handling, CPU-side collection, sharding
arithmetic). No compute."""
import numpy as np
import pytest

from keds_b200 import faiss_compat as faiss
from keds_b200.sharded import packed_layout, shard_bounds


def test_flat_index_collects_rows_but_cannot_search():
    ix = faiss.IndexFlatL2(8)
    assert ix.d == 8 and ix.ntotal == 0 and ix.is_trained and ix.metric_type == faiss.METRIC_L2
    ix.add(np.zeros((3, 8), np.float32))
    ix.add(np.ones((2, 8), np.float32))
    assert ix.ntotal == 5
    with pytest.raises(RuntimeError, match="no CPU search"):
        ix.search(np.zeros((1, 8), np.float32), 1)
    ix.reset()
    assert ix.ntotal == 0
    assert faiss.IndexFlatIP(4).metric_type == faiss.METRIC_INNER_PRODUCT


def test_add_argument_checks_follow_faiss():
    ix = faiss.IndexFlatIP(8)
    with pytest.raises(AssertionError):
        ix.add(np.zeros((3, 7), np.float32))
    with pytest.raises(TypeError):
        ix.add(np.zeros((3, 8), np.float64))
    with pytest.raises(ValueError):
        ix.add(np.zeros(8, np.float32))
    ix.add(np.asfortranarray(np.zeros((3, 8), np.float32)))  # coerced to C order
    assert ix._blocks[0].flags["C_CONTIGUOUS"]


def test_cloning_to_gpu_without_a_gpu_fails_loudly():
    if faiss.get_num_gpus() > 0:
        pytest.skip("a GPU is present")
    ix = faiss.IndexFlatL2(8)
    with pytest.raises(RuntimeError):
        faiss.index_cpu_to_gpu(faiss.StandardGpuResources(), 0, ix)
    with pytest.raises(RuntimeError):
        faiss.index_cpu_to_all_gpus(ix)


@pytest.mark.parametrize("n,world", [(10, 1), (10, 2), (10, 3), (7, 8), (0, 4), (8_000_000, 8)])
def test_shard_bounds_partition_the_rows(n, world):
    spans = [shard_bounds(n, world, r) for r in range(world)]
    assert spans[0][0] == 0 and spans[-1][1] == n
    for (a, b), (c, d) in zip(spans[:-1], spans[1:]):
        assert b == c and a <= b and c <= d
    per = -(-n // world)
    assert all(hi - lo <= per for lo, hi in spans)


def test_packed_layout_is_8_byte_aligned():
    for nq, k in [(1, 1), (128, 16), (3, 5), (4096, 64)]:
        total, off_i, d_bytes = packed_layout(nq, k)
        assert off_i % 8 == 0 and total % 8 == 0 and d_bytes == nq * k * 4
        assert total == off_i + nq * k * 8


def test_database_sampling_and_pair_loading(tmp_path):
    """database.py:14-36 + LoadDataBase (src/data.py:636-671): sample names, keep complete pairs."""
    import torch
    from keds_b200 import database as kdb

    names = [f"{i:05d}.pt" for i in range(20)]
    picked = kdb.sample_pairs(names, 8, seed=3)
    assert len(picked) == 8 and len(set(picked)) == 8 and set(picked) <= set(names)
    assert picked == kdb.sample_pairs(names, 8, seed=3)
    assert len(kdb.sample_pairs(names, 100, seed=1)) == 20
    img_dir, txt_dir = tmp_path / "image_feature_database", tmp_path / "text_feature_database"
    img_dir.mkdir()
    txt_dir.mkdir()
    for i, n in enumerate(picked):
        torch.save(torch.full((1, 6), float(i)), img_dir / n)          # [1, d] like a CLIP output
        if i != 2:                                                      # one pair lacks its text half
            torch.save(torch.full((6,), -float(i)), txt_dir / n)
    img, txt, kept = kdb.load_pair_folders(str(tmp_path), picked)
    assert img.shape == (7, 6) and txt.shape == (7, 6) and picked[2] not in kept
    assert img.dtype == torch.float32 and float(img[0, 0]) == 0.0 and float(txt[1, 0]) == -1.0


# ------------------------------------------------------------------ the planner (host only)
def _plan(n_db, nq, k, n_rows, sms=148):
    import ctypes as C

    from keds_b200 import _capi
    out = (C.c_int32 * 6)()
    _capi.check(_capi.load().keds_debug_plan(n_db, nq, k, n_rows, sms, out))
    return dict(zip(("exact_only", "pair", "S", "n_qt", "items", "grid"), [int(v) for v in out]))


def test_planner_training_step_shape_fills_the_sms_with_one_item_each():
    """BASELINE.json configs[1]: 128 queries, 2 x 0.5M rows, k = 16 on 148 SMs."""
    p = _plan(2, 128, 16, 500_000)
    assert p == {"exact_only": 0, "pair": 0, "S": 73, "n_qt": 1, "items": 146, "grid": 146}


def test_planner_invariants_over_a_sweep():
    for n_db in (1, 2):
        for nq in (1, 128, 129, 1024, 4096, 16384):
            for k in (1, 16, 64, 200):
                for n in (300, 5_000, 50_000, 500_000, 1_000_000):
                    p = _plan(n_db, nq, k, n)
                    assert p["n_qt"] == -(-nq // 128)
                    if p["exact_only"]:
                        continue
                    tiles = -(-n // 256)
                    sub = 2 if p["pair"] else 1     # the pair kernel keeps a candidate list per column half of a slice
                    assert -(-6 * k // 16) <= p["S"] * sub and p["S"] <= min(tiles, 192)   # enough lists, no empty slice
                    assert p["pair"] == (1 if nq > 128 else 0)                  # CTA pairs share row tiles
                    groups = n_db * (-(-p["n_qt"] // 2) if p["pair"] else p["n_qt"])
                    assert p["items"] == groups * p["S"]
                    assert 0 < p["grid"] <= 148 and (p["grid"] % 2 == 0 or not p["pair"])


def test_planner_small_databases_and_huge_k_go_to_the_exact_kernel():
    assert _plan(1, 128, 16, 300)["exact_only"] == 1        # fewer tiles than the slices k needs
    assert _plan(1, 128, 600, 500_000)["exact_only"] == 1   # k beyond the candidate capacity


def test_planner_large_k_buys_slices_against_fallbacks():
    """k = 64 at 4096 queries x 1M rows: 37 candidate lists per query balance the SMs just as well as
    74 but leave about one query per batch to the exact fallback (a full fp32 scan); the planner must
    prefer 74 lists -- 37 slices in the CTA-pair kernel, which keeps one list per column half."""
    assert _plan(1, 4096, 64, 1_000_000)["S"] == 37
    assert _plan(1, 4096, 16, 500_000)["S"] == 23           # small k: unchanged by the fallback term
    assert _plan(1, 4096, 16, 50_000)["S"] == 9             # short database: few, long slices (two rounds of items)


def test_parallel_runner_keeps_order_and_raises_the_first_error():
    """IndexReplicas / IndexShards run one host thread per GPU: results come back in job order and a
    failing sub-search surfaces as its exception, not as a missing part."""
    import time

    from keds_b200.index import _run_parallel

    def job(i, delay):
        def f():
            time.sleep(delay)
            return i
        return f

    assert _run_parallel([job(0, 0.05), job(1, 0.0), job(2, 0.02)]) == [0, 1, 2]
    assert _run_parallel([job(7, 0.0)]) == [7]

    def boom():
        raise RuntimeError("shard 1 failed")

    with pytest.raises(RuntimeError, match="shard 1 failed"):
        _run_parallel([job(0, 0.0), boom, job(2, 0.0)])


# ------------------------------------------------------------------ the consumer's GEMM chooser (host only)
TILE128, TILE256, PERSISTENT, SPLITK2, SPLITK4 = 1, 2, 3, 4, 5


def _linear_plan(M, N, nz, sms=148):
    import ctypes as C

    from keds_b200 import _capi
    v = C.c_int32(-1)
    _capi.check(_capi.load().keds_debug_linear_plan(M, N, nz, sms, C.byref(v)))
    return v.value


@pytest.mark.parametrize("what,M,N,nz,variant", [
    # B = 128, k = 16 at the reference's widths (768 -> 512 -> 512 -> 768, inner 512, 3 layers)
    ("MLP hidden", 128 * 33, 512, 1, TILE128),
    ("fc_out", 128 * 33, 768, 1, TILE256),
    ("K/V of every layer", 128 * 16, 3072, 2, PERSISTENT),
    ("to_q", 128, 512, 2, SPLITK4),
    ("to_out", 128, 768, 2, SPLITK2),
    ("MLP dW", 512, 768, 1, SPLITK2),
    # B = 37: fewer tiles move fc_out and K/V to narrower variants
    ("fc_out B=37", 37 * 33, 768, 1, TILE128),
    ("K/V B=37", 37 * 16, 3072, 2, TILE256),
    ("to_q B=37", 37, 512, 2, SPLITK4),
    # the contrastive loss: N = 1024 logits (K = 3 x 768, nz = 2), its gradient for 256 local rows
    ("clip logits", 1024, 1024, 2, TILE128),
    ("clip gradient", 256, 768, 2, SPLITK2),
])
def test_linear_chooser_at_the_consumer_products(what, M, N, nz, variant):
    assert _linear_plan(M, N, nz) == variant, what


def test_linear_chooser_sweep_reaches_every_variant_and_respects_its_rules():
    seen = set()
    for M in (1, 37, 128, 129, 592, 1221, 2048, 4224, 20000):
        for N in (4, 32, 260, 512, 768, 1024, 3072):
            for nz in (1, 2):
                v = _linear_plan(M, N, nz)
                seen.add(v)
                mt = -(-M // 128)
                c128, c256 = mt * -(-N // 128) * nz, mt * -(-N // 256) * nz
                if c128 * 6 <= 148:
                    tiles32 = mt * -(-N // 32) * nz
                    assert v == (SPLITK4 if tiles32 * 4 <= 148 else SPLITK2), (M, N, nz)
                else:
                    assert v in (TILE128, TILE256, PERSISTENT), (M, N, nz)
                    assert (v == PERSISTENT) == (v != TILE128 and c256 > 2 * 148), (M, N, nz)
    assert seen == {TILE128, TILE256, PERSISTENT, SPLITK2, SPLITK4}


@pytest.mark.parametrize("sms", [1, 2, 3])
def test_linear_chooser_without_four_sms_never_takes_split_k(sms):
    for M, N, nz in [(1, 4, 1), (1, 32, 2), (128, 512, 2), (4224, 768, 1), (2048, 3072, 2)]:
        assert _linear_plan(M, N, nz, sms) in (TILE128, TILE256, PERSISTENT)


def test_linear_chooser_rejects_bad_arguments():
    import ctypes as C

    from keds_b200 import _capi
    v = C.c_int32(-1)
    lib = _capi.load()
    for args in [(0, 4, 1, 148), (4, 0, 1, 148), (4, 4, 3, 148), (4, 4, 1, 0)]:
        assert lib.keds_debug_linear_plan(*args, C.byref(v)) == -1
    assert lib.keds_debug_linear_plan(4, 4, 1, 148, None) == -1


@pytest.mark.parametrize("sms", [1, 4, 148])
@pytest.mark.parametrize("nz", [1, 2])
@pytest.mark.parametrize("N", [4, 16, 80, 768])
def test_linear_chooser_takes_the_persistent_kernel_past_grid_y(N, nz, sms):
    """The one-tile and split-K kernels put the 128-row tiles on grid.y, at most 65 535 of them; the
    persistent kernel walks a flat tile list. Past that edge, up to the 2^30 rows the consumer accepts,
    only the persistent kernel may be chosen; at the edge d_tok = 80 still takes 128-column tiles."""
    edge = 65535 * 128
    for M in (edge + 1, 4100 * 2049, 1 << 30):
        assert _linear_plan(M, N, nz, sms) == PERSISTENT, M
    if N == 80 and nz == 1 and sms == 148:
        assert _linear_plan(edge, N, nz, sms) == TILE128
