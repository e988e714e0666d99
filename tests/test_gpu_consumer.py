"""GPU (-m gpu): the neighbour consumer (SURVEY.md §8 f2) through the C ABI against the float64
oracle (oracle/consumer_oracle.py, itself pinned to the reference's modules by
tests/golden/consumer.npz).

Tolerance: the products run on tf32 tensor cores (10-bit mantissa operands, fp32 accumulation),
the reference runs them in fp32 (fp16 under amp autocast, src/trainer.py:462-465). Eight products
are chained; against the plain oracle the bound asserted is  max |got - oracle| <= 4e-3 * max |oracle|.
Against the oracle with tf32 operand rounding (tf32=True) only fp32 accumulation and fp32 attention
remain, and the bound is ten times tighter (TF32_TOL).
"""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from keds_b200 import faiss_compat as faiss  # noqa: E402
from keds_b200.consumer import NeighbourConsumer  # noqa: E402
from keds_b200.index import GpuIndexFlat  # noqa: E402
from oracle import consumer_oracle as corc  # noqa: E402

REL_TOL = 4e-3
# Against the tf32-faithful oracle what is left is fp32 accumulation and fp32 attention. Chains of
# sharp softmaxes over unnormalised inputs amplify such differences (an intermediate that moves by
# an fp32 unit can also round to the neighbouring tf32 number in the next product): noise of 3e-7 on
# every product output moves the float64 oracle's tokens by up to 7e-5 at 4 layers of 16 x 64, B =
# 129, k = 64. Measured on a B200 (1000 W): at most 1.1e-4 over these cases, against up to 4e-3
# without the tf32 model; rounding ties away from zero instead of to even alone costs 1.8e-4.
TF32_TOL = 4e-4


def to_torch(sd):
    return {k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in sd.items()}


def index_of(rows):
    ix = GpuIndexFlat(rows.shape[1], faiss.METRIC_INNER_PRODUCT, 0)
    ix.add(np.ascontiguousarray(rows, dtype=np.float32))
    return ix


def run_case(sds, heads, feat, base_img, base_txt, I_img, I_txt, perm=None, tf32=False):
    cons = NeighbourConsumer(to_torch(sds[0]), to_torch(sds[1]), to_torch(sds[2]), heads=heads, device=0)
    ix_i, ix_t = index_of(base_img), index_of(base_txt)
    got = cons(torch.from_numpy(feat).cuda(), ix_i, ix_t, torch.from_numpy(I_img).cuda(),
               torch.from_numpy(I_txt).cuda(), perm)
    assert cons.check() > 0
    want = corc.consumer_tokens(sds[0], sds[1], sds[2], heads, feat, base_img, base_txt, I_img, I_txt, tf32)
    got = got.cpu().numpy()
    assert got.shape == want.shape and got.dtype == np.float32
    err = np.abs(got - want).max() / np.abs(want).max()
    return err, got, want, cons


def test_reference_module_outputs_small_widths(golden_dir):
    # widths 48 / 32 / 40, 4 heads x 8: ragged k-blocks (48 = 32 + 16) and ragged output tiles
    g = np.load(os.path.join(golden_dir, "consumer.npz"))
    heads = int(g["dims"][5])
    sds = [{k.split("/", 1)[1]: g[k] for k in g.files if k.startswith(p + "/")}
           for p in ("img2text", "retrieval_fuse", "text_condition")]
    err, got, _, _ = run_case(sds, heads, g["feat"], g["base_img"], g["base_txt"], g["I_img"], g["I_txt"])
    assert err < REL_TOL, err
    # and directly against what the reference's modules produced
    assert np.abs(got - g["tokens"]).max() / np.abs(g["tokens"]).max() < REL_TOL


@pytest.mark.parametrize("B,k", [(128, 16), (37, 16), (1, 1), (130, 5)])
def test_full_width_matches_oracle(B, k):
    # the reference's sizes: 768 -> 512 -> 512 -> 768 MLP, 3 layers of 8 heads x 64 (src/main.py:147-152)
    sds = corc.random_state_dicts(768, 512, 768, 2, 3, 8, 64, seed=7 + B)
    rng = np.random.default_rng(B * 31 + k)
    n = 4000
    base_img = rng.standard_normal((n, 768)).astype(np.float32)
    base_img /= np.linalg.norm(base_img, axis=1, keepdims=True)
    base_txt = rng.standard_normal((n, 768)).astype(np.float32)
    base_txt /= np.linalg.norm(base_txt, axis=1, keepdims=True)
    feat = rng.standard_normal((B, 768)).astype(np.float32)
    feat /= np.linalg.norm(feat, axis=1, keepdims=True)
    I_img = rng.integers(0, n, (B, k)).astype(np.int64)
    I_txt = rng.integers(0, n, (B, k)).astype(np.int64)
    err, _, _, _ = run_case(sds, 8, feat, base_img, base_txt, I_img, I_txt)
    assert err < REL_TOL, err
    err, _, _, _ = run_case(sds, 8, feat, base_img, base_txt, I_img, I_txt, tf32=True)
    assert err < TF32_TOL, err


# (B, k, heads, dim_head, n_hidden, n_layers): k around one warp (one lane per neighbour: the
# neighbour loops wrap at k > 32), the generic attention kernel with dim_head > 64 and dim_head < 32,
# 32 heads (1024 threads), one head of width 4, one and four layers, one and three hidden layers
ATTENTION_SHAPES = [
    (1, 31, 16, 64, 1, 1),
    (129, 32, 32, 16, 3, 4),
    (129, 33, 6, 40, 1, 4),
    (1, 64, 2, 96, 3, 1),
    (129, 100, 1, 4, 1, 1),
    (129, 64, 16, 64, 3, 4),
    (1, 100, 32, 16, 1, 4),
    (129, 31, 2, 96, 1, 1),
]


def attention_case(B, k, heads, dim_head, n_hidden, n_layers, seed):
    sds = corc.random_state_dicts(96, 64, 80, n_hidden, n_layers, heads, dim_head, seed=seed)
    rng = np.random.default_rng(seed)
    n = 700
    base_img = rng.standard_normal((n, 96)).astype(np.float32)
    base_txt = rng.standard_normal((n, 96)).astype(np.float32)
    feat = rng.standard_normal((B, 96)).astype(np.float32)
    I_img = rng.integers(0, n, (B, k)).astype(np.int64)
    I_txt = rng.integers(0, n, (B, k)).astype(np.int64)
    return sds, feat, base_img, base_txt, I_img, I_txt


@pytest.mark.parametrize("B,k,heads,dim_head,n_hidden,n_layers", ATTENTION_SHAPES)
def test_attention_shapes_match_the_tf32_oracle(B, k, heads, dim_head, n_hidden, n_layers):
    sds, feat, base_img, base_txt, I_img, I_txt = attention_case(B, k, heads, dim_head, n_hidden, n_layers, B + k)
    err, _, _, _ = run_case(sds, heads, feat, base_img, base_txt, I_img, I_txt, tf32=True)
    print(f"B={B} k={k} heads={heads} dim_head={dim_head}: tokens {err:.2e}")
    assert err < TF32_TOL, err


def test_neighbour_order_does_not_matter_and_missing_ids_read_zero_rows():
    sds = corc.random_state_dicts(64, 32, 64, 2, 2, 4, 8, seed=3)
    rng = np.random.default_rng(5)
    base = rng.standard_normal((50, 64)).astype(np.float32)
    feat = rng.standard_normal((9, 64)).astype(np.float32)
    I = rng.integers(0, 50, (9, 8)).astype(np.int64)
    err, got, _, cons = run_case(sds, 4, feat, base, base, I, I)
    assert err < REL_TOL
    # the shared randperm (src/trainer.py:218-219) only reorders a softmax-weighted sum
    ix = index_of(base)
    perm = torch.randperm(8, generator=torch.Generator().manual_seed(1))
    got_p = cons(torch.from_numpy(feat).cuda(), ix, ix, torch.from_numpy(I).cuda(), torch.from_numpy(I).cuda(),
                 perm).cpu().numpy()
    assert np.abs(got_p - got).max() < 1e-4 * np.abs(got).max()
    # id -1 (search padding) gathers a zero row: same as a database with an appended zero row
    Ineg = I.copy()
    Ineg[:, -1] = -1
    base_z = np.concatenate([base, np.zeros((1, 64), np.float32)])
    Iz = I.copy()
    Iz[:, -1] = 50
    want = corc.consumer_tokens(sds[0], sds[1], sds[2], 4, feat, base_z, base_z, Iz, Iz)
    got_n = cons(torch.from_numpy(feat).cuda(), ix, ix, torch.from_numpy(Ineg).cuda(),
                 torch.from_numpy(Ineg).cuda()).cpu().numpy()
    assert np.abs(got_n - want).max() / np.abs(want).max() < REL_TOL


def test_consumer_argument_errors():
    sds = corc.random_state_dicts(64, 32, 64, 2, 2, 4, 8, seed=3)
    cons = NeighbourConsumer(to_torch(sds[0]), to_torch(sds[1]), to_torch(sds[2]), heads=4, device=0)
    ix = index_of(np.eye(64, dtype=np.float32))
    I = torch.zeros((2, 3), dtype=torch.int64, device="cuda")
    with pytest.raises(TypeError):
        cons(torch.zeros(2, 64), ix, ix, I, I)                       # host tensor
    with pytest.raises(ValueError):
        cons(torch.zeros(3, 64, device="cuda"), ix, ix, I, I)        # B mismatch
    bad = dict(to_torch(sds[1]))
    bad["cross_layers.0.to_q.weight"] = torch.zeros(32, 48)          # wrong in_features
    with pytest.raises(RuntimeError):
        NeighbourConsumer(to_torch(sds[0]), bad, to_torch(sds[2]), heads=4, device=0)
    with pytest.raises(ValueError):
        NeighbourConsumer(to_torch(sds[0]), to_torch(sds[1]), to_torch(sds[2]), heads=5, device=0)


def test_retrieve_and_consume_in_one_call_matches_the_oracle_pipeline():
    # src/trainer.py:53-69: normalise a copy for the search, gather, img2text, two CrossFormers
    from keds_b200 import retrieval as kr
    from oracle import knn_oracle as orc

    sds = corc.random_state_dicts(768, 512, 768, 2, 3, 8, 64, seed=21)
    rng = np.random.default_rng(77)
    n, B, k = 20000, 48, 16
    base_img = rng.standard_normal((n, 768)).astype(np.float32)
    base_img /= np.linalg.norm(base_img, axis=1, keepdims=True)
    base_txt = (0.6 * base_img + 0.4 * rng.standard_normal((n, 768)).astype(np.float32) / np.sqrt(768)).astype(np.float32)
    base_txt /= np.linalg.norm(base_txt, axis=1, keepdims=True)
    feat = (2.5 * rng.standard_normal((B, 768))).astype(np.float32)      # un-normalised on purpose
    kb = kr.KnowledgeBase(torch.from_numpy(base_img), torch.from_numpy(base_txt), [str(i) for i in range(n)], device=0)
    cons = NeighbourConsumer(to_torch(sds[0]), to_torch(sds[1]), to_torch(sds[2]), heads=8, device=0)
    got = cons.from_features(torch.from_numpy(feat).cuda(), kb, topk=k).cpu().numpy()
    assert cons.check() > 0
    qn = feat / np.linalg.norm(feat, axis=1, keepdims=True)
    _, I_img = orc.search(base_img, qn, k, "l2")
    _, I_txt = orc.search(base_txt, qn, k, "l2")
    want = corc.consumer_tokens(sds[0], sds[1], sds[2], 8, feat, base_img, base_txt, I_img, I_txt)
    assert np.abs(got - want).max() / np.abs(want).max() < REL_TOL
