"""GPU (-m gpu): the neighbour consumer in TRAINING mode (SURVEY.md §8 f2; src/trainer.py:59-69 with
the backward of :462-474) through the C ABI -- tokens and the gradient of every parameter -- against
the float64 oracle (oracle/consumer_train_oracle.py, pinned to the reference's own modules by
tests/golden/consumer_train.npz).

Tolerance: every product runs on tf32 tensor cores (10-bit mantissa operands, fp32 accumulation);
the reference trains in fp32 (fp16 under amp autocast, src/trainer.py:462-465). The native path is
compared with the oracle in its tf32 mode (every Linear product, forward and backward, with
tf32-rounded operands), with the ReLU gates of the native forward (see check_against_oracle):
tokens within TF32_TOK_TOL and every gradient within TF32_GRAD_TOL of the tensor's maximum. Against
the reference's own modules in float64 (tests/golden/consumer_train.npz), which do not round, the
bounds are TOK_TOL and GRAD_TOL.
"""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from keds_b200 import faiss_compat as faiss  # noqa: E402
from keds_b200.consumer import NeighbourConsumer, TrainableNeighbourConsumer  # noqa: E402
from keds_b200.index import GpuIndexFlat  # noqa: E402
from oracle import consumer_oracle as corc  # noqa: E402
from oracle import consumer_train_oracle as cto  # noqa: E402

TOK_TOL, GRAD_TOL = 4e-3, 1e-2
# With tf32 rounding modelled, what is left is fp32 accumulation (K up to B(1+2k) rows in dW) and
# fp32 attention and its backward, amplified by sharp softmaxes as in tests/test_gpu_consumer.py.
# A gradient is measured against the larger of its own maximum and 1e-3 of the largest gradient (the
# to_k biases have an exactly zero gradient). Measured on a B200 (1000 W): tokens at most 1.3e-4,
# gradients at most 4.1e-4, the latter in the SGD-step case on unnormalised inputs, which differs
# from the plain oracle by 5e-3: that excess is tf32 operand rounding, not a defect.
TF32_TOK_TOL, TF32_GRAD_TOL = 4e-4, 1e-3


def to_torch(sd):
    return {k: torch.from_numpy(np.ascontiguousarray(v, dtype=np.float32)) for k, v in sd.items()}


def index_of(rows):
    ix = GpuIndexFlat(rows.shape[1], faiss.METRIC_INNER_PRODUCT, 0)
    ix.add(np.ascontiguousarray(rows, dtype=np.float32))
    return ix


def rel(got, want, floor=1e-30):
    """max |got - want| relative to the tensor's own scale -- but never below `floor`: the to_k
    biases have an exactly zero gradient (a bias on every key shifts all scores of a softmax row
    alike), so their error is measured against the scale of the other gradients."""
    return float(np.abs(got - want).max() / max(np.abs(want).max(), floor))


def run(sds, heads, feat, base_img, base_txt, I_img, I_txt, dtok, masks=None, dropout=0.0):
    mod = TrainableNeighbourConsumer(to_torch(sds[0]), to_torch(sds[1]), to_torch(sds[2]), heads=heads, device=0,
                                     dropout=dropout)
    ix_i, ix_t = index_of(base_img), index_of(base_txt)
    f = torch.from_numpy(feat.astype(np.float32)).cuda()
    Ii, It = torch.from_numpy(I_img).cuda(), torch.from_numpy(I_txt).cuda()
    return mod, ix_i, ix_t, f, Ii, It


def check_against_oracle(sds, heads, feat, base_img, base_txt, I_img, I_txt, dtok, masks=None, tf32=True):
    mod, ix_i, ix_t, f, Ii, It = run(sds, heads, feat, base_img, base_txt, I_img, I_txt, dtok)
    from keds_b200.consumer import _ConsumerFn
    mk = None if masks is None else [None if m is None else torch.from_numpy(m.astype(np.float32)).cuda() for m in masks]
    tokens = _ConsumerFn.apply(mod, f, ix_i, ix_t, Ii, It, None, mk, mod.flat)
    tokens.backward(torch.from_numpy(dtok.astype(np.float32)).cuda())
    assert mod.check() > 0
    B, k = I_img.shape
    nb_i = base_img[I_img.reshape(-1)].reshape(B, k, -1)
    nb_t = base_txt[I_txt.reshape(-1)].reshape(B, k, -1)
    # The ReLU gates come from the native forward: a tf32 forward and the float64 oracle disagree on
    # the few units whose pre-activation is within rounding of zero (measured: ~4e-4 of the first
    # layer's units at full width), and one flipped gate per column already moves a bias gradient by
    # several per cent. They must agree almost everywhere, though.
    M = B * (1 + 2 * k)
    n_hidden = sum(1 for name in sds[0] if name.endswith(".0.weight"))
    gates = [(mod.debug_hidden(i, M) > 0).double().cpu().numpy() for i in range(n_hidden)]
    tok_tol, grad_tol = (TF32_TOK_TOL, TF32_GRAD_TOL) if tf32 else (TOK_TOL, GRAD_TOL)
    _, free = cto.tokens_and_grads(sds[0], sds[1], sds[2], heads, feat, nb_i, nb_t, dtok, masks, tf32=tf32)
    want_tok, want = cto.tokens_and_grads(sds[0], sds[1], sds[2], heads, feat, nb_i, nb_t, dtok, masks, gates,
                                          tf32=tf32)
    assert rel(want["img2text/fc_out.weight"], free["img2text/fc_out.weight"]) < 1e-2   # same network, same gates almost everywhere
    errs = {"tokens": rel(tokens.detach().cpu().numpy(), want_tok)}
    assert errs["tokens"] < tok_tol, errs
    gi, gf, gc = mod.state_dicts(grads=True)
    scale = 1e-3 * max(float(np.abs(v).max()) for v in want.values())
    for prefix, gsd in (("img2text", gi), ("retrieval_fuse", gf), ("text_condition", gc)):
        for name, t in gsd.items():
            errs[f"{prefix}/{name}"] = rel(t.cpu().numpy(), want[f"{prefix}/{name}"], scale)
    worst = max(errs, key=errs.get)
    assert errs[worst] < grad_tol, "\n".join(f"{v:.3e}  {k_}" for k_, v in sorted(errs.items(), key=lambda kv: -kv[1])[:14])
    return errs, mod


def test_reference_module_gradients_small_widths(golden_dir):
    """against what the reference's own modules produced in train mode (ragged widths 48 / 32 / 40)"""
    g = np.load(os.path.join(golden_dir, "consumer_train.npz"))
    heads = int(g["dims"][5])
    sds = [{k.split("/", 1)[1]: g[k] for k in g.files if k.startswith(p + "/")}
           for p in ("img2text", "retrieval_fuse", "text_condition")]
    B, k, d_in = g["topk_image"].shape
    base_img = g["topk_image"].reshape(B * k, d_in).astype(np.float32)
    base_txt = g["topk_text"].reshape(B * k, d_in).astype(np.float32)
    I = np.arange(B * k, dtype=np.int64).reshape(B, k)
    errs, mod = check_against_oracle(sds, heads, g["feat"].astype(np.float32), base_img, base_txt, I, I, g["dtokens"],
                                     tf32=False)
    check_against_oracle(sds, heads, g["feat"].astype(np.float32), base_img, base_txt, I, I, g["dtokens"])
    gi, gf, gc = mod.state_dicts(grads=True)
    scale = 1e-3 * max(float(np.abs(g[k_]).max()) for k_ in g.files if k_.startswith("grad/"))
    for prefix, gsd in (("img2text", gi), ("retrieval_fuse", gf), ("text_condition", gc)):
        for name, t in gsd.items():
            assert rel(t.cpu().numpy(), g[f"grad/{prefix}/{name}"], scale) < GRAD_TOL, (prefix, name)


@pytest.mark.parametrize("B,k,with_masks", [(128, 16, True), (37, 16, False), (130, 5, True)])
def test_full_width_gradients_match_oracle(B, k, with_masks):
    """the reference's sizes (768 -> 512 -> 512 -> 768 MLP, 3 layers of 8 heads x 64) with dropout
    masks on both hidden layers"""
    sds = corc.random_state_dicts(768, 512, 768, 2, 3, 8, 64, seed=11 + B)
    rng = np.random.default_rng(B * 7 + k)
    n = 3000
    base_img = rng.standard_normal((n, 768)).astype(np.float32)
    base_img /= np.linalg.norm(base_img, axis=1, keepdims=True)
    base_txt = rng.standard_normal((n, 768)).astype(np.float32)
    base_txt /= np.linalg.norm(base_txt, axis=1, keepdims=True)
    feat = rng.standard_normal((B, 768)).astype(np.float32)
    feat /= np.linalg.norm(feat, axis=1, keepdims=True)
    I_img = rng.integers(0, n, (B, k)).astype(np.int64)
    I_txt = rng.integers(0, n, (B, k)).astype(np.int64)
    dtok = rng.standard_normal((B, 3, 768)).astype(np.float32)
    masks = None
    if with_masks:
        M = B * (1 + 2 * k)
        masks = [((rng.random((M, 512)) < 0.9) / 0.9).astype(np.float32) for _ in range(2)]
    errs, _ = check_against_oracle(sds, 8, feat, base_img, base_txt, I_img, I_txt, dtok, masks)
    print("worst relative errors:", sorted(errs.items(), key=lambda kv: -kv[1])[:4])


def test_optimizer_updates_are_read_through_and_eval_matches_the_forward_only_consumer():
    """the flat Parameter IS the weight storage: an optimiser step changes the next forward without
    any upload, the transposed copies used by dX are refreshed, and eval() reproduces the
    forward-only consumer bit for bit on the same weights"""
    sds = corc.random_state_dicts(256, 128, 256, 2, 2, 4, 32, seed=3)
    rng = np.random.default_rng(9)
    n, B, k = 500, 40, 8
    base = rng.standard_normal((n, 256)).astype(np.float32)
    feat = rng.standard_normal((B, 256)).astype(np.float32)
    I1 = rng.integers(0, n, (B, k)).astype(np.int64)
    I2 = rng.integers(0, n, (B, k)).astype(np.int64)
    dtok = rng.standard_normal((B, 3, 256)).astype(np.float32)
    mod, ix_i, ix_t, f, Ii, It = run(sds, 4, feat, base, base, I1, I2, dtok)
    opt = torch.optim.SGD(mod.parameters(), lr=0.05)
    mod.eval()
    t0 = mod(f, ix_i, ix_t, Ii, It)
    ref = NeighbourConsumer(*mod.state_dicts(), heads=4, device=0)
    assert torch.equal(t0.detach(), ref(f, ix_i, ix_t, Ii, It))
    (t0 * torch.from_numpy(dtok).cuda()).sum().backward()
    opt.step()
    opt.zero_grad()
    # after the step: compare forward and backward with the oracle on the UPDATED weights
    new_sds = [{k_: v.cpu().numpy() for k_, v in sd.items()} for sd in mod.state_dicts()]
    t1 = mod(f, ix_i, ix_t, Ii, It)
    t1.backward(torch.from_numpy(dtok).cuda())
    nb_i = base[I1.reshape(-1)].reshape(B, k, -1)
    nb_t = base[I2.reshape(-1)].reshape(B, k, -1)
    gates = [(mod.debug_hidden(i, B * (1 + 2 * k)) > 0).double().cpu().numpy() for i in range(2)]
    want_tok, want = cto.tokens_and_grads(new_sds[0], new_sds[1], new_sds[2], 4, feat, nb_i, nb_t, dtok, None, gates,
                                          tf32=True)
    assert rel(t1.detach().cpu().numpy(), want_tok) < TF32_TOK_TOL
    assert not torch.equal(t1.detach(), t0.detach())
    gi, gf, gc = mod.state_dicts(grads=True)
    scale = 1e-3 * max(float(np.abs(v).max()) for v in want.values())
    errs = {}
    for prefix, gsd in (("img2text", gi), ("retrieval_fuse", gf), ("text_condition", gc)):
        for name, t in gsd.items():
            errs[f"{prefix}/{name}"] = rel(t.cpu().numpy(), want[f"{prefix}/{name}"], scale)
    print("after an SGD step, worst:", sorted(errs.items(), key=lambda kv: -kv[1])[:4])
    assert max(errs.values()) < TF32_GRAD_TOL, sorted(errs.items(), key=lambda kv: -kv[1])[:6]
    # train() mode draws dropout masks: outputs differ from eval, gradients still flow
    mod.train()
    mod.dropout = 0.5
    t2 = mod(f, ix_i, ix_t, Ii, It)
    assert not torch.equal(t2.detach(), t1.detach())
    t2.sum().backward()
    assert torch.isfinite(mod.flat.grad).all() and float(mod.flat.grad.abs().max()) > 0


# (B, k, heads, dim_head, n_hidden, n_layers): see tests/test_gpu_consumer.py ATTENTION_SHAPES
TRAIN_SHAPES = [
    (1, 31, 16, 64, 1, 1),
    (129, 32, 32, 16, 3, 4),
    (129, 33, 6, 40, 1, 4),
    (1, 64, 2, 96, 3, 1),
    (129, 100, 1, 4, 1, 1),
    (129, 64, 16, 64, 3, 4),
]


@pytest.mark.parametrize("B,k,heads,dim_head,n_hidden,n_layers", TRAIN_SHAPES)
def test_attention_shapes_gradients_match_the_tf32_oracle(B, k, heads, dim_head, n_hidden, n_layers):
    sds = corc.random_state_dicts(96, 64, 80, n_hidden, n_layers, heads, dim_head, seed=B * k)
    rng = np.random.default_rng(B + k)
    n = 700
    base_img = rng.standard_normal((n, 96)).astype(np.float32)
    base_txt = rng.standard_normal((n, 96)).astype(np.float32)
    feat = rng.standard_normal((B, 96)).astype(np.float32)
    I_img = rng.integers(0, n, (B, k)).astype(np.int64)
    I_txt = rng.integers(0, n, (B, k)).astype(np.int64)
    dtok = rng.standard_normal((B, 3, 80)).astype(np.float32)
    M = B * (1 + 2 * k)
    masks = [((rng.random((M, 64)) < 0.9) / 0.9).astype(np.float32) for _ in range(n_hidden)]
    errs, _ = check_against_oracle(sds, heads, feat, base_img, base_txt, I_img, I_txt, dtok, masks)
    print(f"B={B} k={k} heads={heads} dim_head={dim_head}: worst", sorted(errs.items(), key=lambda kv: -kv[1])[:3])


def test_forward_train_accepts_only_what_the_backward_can_run():
    """The attention backward needs heads (2 dim_head + 2k) floats of shared memory, twice the
    forward's. At the reference's 8 heads x 64 every k the forward accepts (up to 1024; 705 was the
    first beyond the default 48 KB) must train; at 32 heads x 64 and k = 1024 the backward needs more
    than a B200 block can have, so forward_train must refuse up front while the eval forward, which
    needs half, still runs."""
    rng = np.random.default_rng(4)
    n, B = 3000, 2
    base = rng.standard_normal((n, 64)).astype(np.float32)
    feat = rng.standard_normal((B, 64)).astype(np.float32)
    sds = corc.random_state_dicts(64, 32, 64, 1, 1, 8, 64, seed=4)
    for k in (705, 1024):
        I1 = rng.integers(0, n, (B, k)).astype(np.int64)
        I2 = rng.integers(0, n, (B, k)).astype(np.int64)
        dtok = rng.standard_normal((B, 3, 64)).astype(np.float32)
        check_against_oracle(sds, 8, feat, base, base, I1, I2, dtok)
    sds = corc.random_state_dicts(64, 32, 64, 1, 1, 32, 64, seed=5)
    I = rng.integers(0, n, (B, 1024)).astype(np.int64)
    mod, ix_i, ix_t, f, Ii, It = run(sds, 32, feat, base, base, I, I, None)
    with pytest.raises(RuntimeError, match="attention backward"):
        mod(f, ix_i, ix_t, Ii, It)
    assert mod.flat.grad is None
    ref = NeighbourConsumer(*mod.state_dicts(), heads=32, device=0)
    assert torch.isfinite(ref(f, ix_i, ix_t, Ii, It)).all()


# rows past which a 32-row-tile transpose (65 535 x 32) and a 128-row-tile GEMM (65 535 x 128) would
# need more than grid.y's 65 535 blocks
TRANSPOSE_ROWS, GEMM_ROWS = 65535 * 32, 65535 * 128


def far_queries(B, k):
    """the first and last query, and the first whose image neighbours, text neighbours or dK/dV rows
    start beyond each of the two limits (rows: queries | image neighbours | text neighbours)"""
    qs = {0, B - 1}
    for T in (TRANSPOSE_ROWS, GEMM_ROWS):
        for first_row, rows_per_query in ((B, k), (B + B * k, k), (0, k)):
            b = max(0, -(-(T - first_row) // rows_per_query))
            if b < B:
                qs.add(b)
    return sorted(qs)


@pytest.mark.parametrize("B,k", [(1100, 1024), (4100, 1024)])
def test_the_largest_batches_train(B, k):
    """forward_train accepts any B (1 + 2k) <= 2^30 rows, and the backward has to run them: its
    transposes once B (1 + 2k) > 65 535 x 32, the GEMMs' row tiles once it exceeds 65 535 x 128 (both
    past grid.y's limit). At widths of 16 (one head of 4) B = 4100, k = 1024 is 8.4M rows in about
    5 GB. dtokens are non-zero for a few queries only, the first, the last, and those whose rows lie
    beyond the two limits; every other query then contributes exact zeros, and tokens and gradients
    must match the tf32 oracle evaluated on those queries alone. The eval forward runs the same shape."""
    M = B * (1 + 2 * k)
    sds = corc.random_state_dicts(16, 16, 16, 1, 1, 1, 4, seed=B)
    rng = np.random.default_rng(B)
    n = 2000
    base_img = rng.standard_normal((n, 16)).astype(np.float32)
    base_txt = rng.standard_normal((n, 16)).astype(np.float32)
    feat = rng.standard_normal((B, 16)).astype(np.float32)
    I_img = rng.integers(0, n, (B, k)).astype(np.int64)
    I_txt = rng.integers(0, n, (B, k)).astype(np.int64)
    sel = far_queries(B, k)
    dtok = np.zeros((B, 3, 16), np.float32)
    dtok[sel] = rng.standard_normal((len(sel), 3, 16)).astype(np.float32)
    mod, ix_i, ix_t, f, Ii, It = run(sds, 1, feat, base_img, base_txt, I_img, I_txt, dtok, dropout=0.0)
    tokens = mod(f, ix_i, ix_t, Ii, It)
    tokens.backward(torch.from_numpy(dtok).cuda())
    assert mod.check() > 0
    # the oracle on the selected queries, with the native forward's ReLU gates of their rows
    rows = np.concatenate([np.array(sel)] + [B + np.arange(b * k, (b + 1) * k) for b in sel] +
                          [B + B * k + np.arange(b * k, (b + 1) * k) for b in sel])
    gate = (mod.debug_hidden(0, M)[torch.from_numpy(rows).cuda()] > 0).double().cpu().numpy()
    nb_i, nb_t = base_img[I_img[sel]], base_txt[I_txt[sel]]
    want_tok, want = cto.tokens_and_grads(sds[0], sds[1], sds[2], 1, feat[sel], nb_i, nb_t, dtok[sel], None, [gate],
                                          tf32=True)
    got_tok = tokens.detach()[torch.tensor(sel, device="cuda")].cpu().numpy()
    errs = {"tokens": rel(got_tok, want_tok)}
    gi, gf, gc = mod.state_dicts(grads=True)
    scale = 1e-3 * max(float(np.abs(v).max()) for v in want.values())
    for prefix, gsd in (("img2text", gi), ("retrieval_fuse", gf), ("text_condition", gc)):
        for name, t in gsd.items():
            errs[f"{prefix}/{name}"] = rel(t.cpu().numpy(), want[f"{prefix}/{name}"], scale)
    print(f"B={B} k={k} M={M} queries {sel}: worst", sorted(errs.items(), key=lambda kv: -kv[1])[:3])
    assert errs["tokens"] < TF32_TOK_TOL, errs
    assert max(errs.values()) < TF32_GRAD_TOL, errs
    del tokens
    mod.flat.grad = None
    ref = NeighbourConsumer(*mod.state_dicts(), heads=1, device=0)
    got_eval = ref(f, ix_i, ix_t, Ii, It)
    assert ref.check() > 0
    assert rel(got_eval[torch.tensor(sel, device="cuda")].cpu().numpy(), want_tok) < TF32_TOK_TOL
