"""CPU: the oracle restatement against outputs of the reference's own functions (tests/golden,
produced by oracle/make_golden.py from /root/reference via AST extraction)."""
import json
import os

import numpy as np
import pytest

from oracle import knn_oracle as orc
from oracle.make_golden import load_retrieval


@pytest.fixture(scope="module")
def ret(golden_dir):
    return load_retrieval(os.path.join(golden_dir, "retrieval.npz"))


def test_torch_branch_matches_reference(ret):
    # src/trainer.py:232-257: no query normalisation, no shuffle, raw inner product
    gi, gt, _, _ = orc.retrieved_features(ret["feature"], ret["image_base"], ret["text_base"], 16, None, normalize=False)
    assert np.array_equal(gi.astype(np.float32), ret["torch_branch_image"])
    assert np.array_equal(gt.astype(np.float32), ret["torch_branch_text"])


def test_faiss_branch_boundary_matches_reference(ret):
    # src/trainer.py:203-230: normalise, search, gather, shared randperm on the image stream only
    gi, gt, Ii, It = orc.retrieved_features(ret["feature"], ret["image_base"], ret["text_base"], 16, ret["perm"], True)
    assert np.array_equal(gi.astype(np.float32), ret["faiss_branch_image"])
    assert np.array_equal(gt.astype(np.float32), ret["faiss_branch_text"])
    assert Ii.dtype == np.int64 and It.shape == (32, 16)


def test_ip_and_l2_rank_identically_on_unit_rows(ret):
    f = ret["feature"] / np.linalg.norm(ret["feature"], axis=1, keepdims=True)
    _, Iip = orc.search(ret["image_base"], f, 16, "ip")
    Dl2, Il2 = orc.search(ret["image_base"], f, 16, "l2")
    Dip, _ = orc.search(ret["image_base"], f, 16, "ip")
    assert np.array_equal(Iip, Il2)
    assert np.allclose(Dl2, 2 - 2 * Dip, atol=2e-6)


def test_extra_cap_matches_reference(ret):
    f = ret["feature"] / np.linalg.norm(ret["feature"], axis=1, keepdims=True)
    _, It = orc.search(ret["text_base"], f, 2, "ip")
    assert np.array_equal(orc.gather(ret["text_base"], It), ret["extra_text"])
    assert [f"{i:07d}" for i in It.reshape(-1)] == list(ret["extra_names"])


def test_search_conventions():
    rng = np.random.default_rng(0)
    db = rng.standard_normal((5, 8)).astype(np.float32)
    q = rng.standard_normal((3, 8)).astype(np.float32)
    D, I = orc.search(db, q, 8, "ip")
    assert (I[:, 5:] == -1).all() and (D[:, 5:] == -orc.FLT_MAX).all()
    D, I = orc.search(db, q, 8, "l2")
    assert (I[:, 5:] == -1).all() and (D[:, 5:] == orc.FLT_MAX).all()
    assert (np.diff(D[:, :5], axis=1) >= 0).all()
    D, I = orc.search(np.zeros((0, 8), np.float32), q, 2)
    assert (I == -1).all()
    # ties: lower label first
    dup = np.repeat(db[:1], 4, axis=0)
    _, I = orc.search(dup, q, 3)
    assert (I == np.array([0, 1, 2])).all()


def test_blas_baseline_agrees_with_float64(ret):
    f = ret["feature"]
    D, I = orc.search_f32_blas(ret["image_base"], f, 16, chunk_rows=500)
    Dr, Ir = orc.search(ret["image_base"], f, 16)
    c = orc.compare_topk(Dr, Ir, D, I, ret["image_base"], f)
    assert c["ok"], c


@pytest.fixture(scope="module")
def met(golden_dir):
    z = np.load(os.path.join(golden_dir, "metrics_inputs.npz"))
    with open(os.path.join(golden_dir, "metrics_expected.json")) as f:
        e = json.load(f)
    return z, e


def _close(got, want):
    assert set(got) == set(want), (sorted(got), sorted(want))
    for k in want:
        assert got[k] == pytest.approx(want[k], rel=1e-5, abs=1e-5), (k, got[k], want[k])


def test_metrics_cirr(met):
    z, e = met
    _close(orc.metrics_cirr(z["gal"], z["qf"], e["reference_names"], e["index_names"], e["target_names"]), e["metrics"]["cirr"])


def test_metrics_fashion(met):
    z, e = met
    ans = [e["fashion_names"][i] for i in z["tgt"]]
    _close(orc.metrics_fashion(z["gal"], z["qf"], e["fashion_names"], ans), e["metrics"]["fashion"])


def test_metrics_coco(met):
    z, e = met
    _close(orc.metrics_coco(z["coco_img"], z["coco_ref"], 100.0), e["metrics"]["coco"])


def test_metrics_imgnet(met):
    z, e = met
    _close(orc.metrics_imgnet(z["in_q"], z["in_gal"], z["in_qlab"], z["in_glab"]), e["metrics"]["imgnet"])


# ------------------------------------------------------------------ neighbour consumer (§8 f2)
def test_consumer_oracle_matches_the_reference_modules(golden_dir):
    # tests/golden/consumer.npz: IM2TEXT / CrossFormer of src/model/model.py run unchanged
    # (oracle/make_golden_consumer.py), call sequence of src/trainer.py:59-69
    from oracle import consumer_oracle as corc

    g = np.load(os.path.join(golden_dir, "consumer.npz"))
    heads = int(g["dims"][5])
    sds = [{k.split("/", 1)[1]: g[k] for k in g.files if k.startswith(p + "/")}
           for p in ("img2text", "retrieval_fuse", "text_condition")]
    tokens = corc.consumer_tokens(sds[0], sds[1], sds[2], heads, g["feat"], g["base_img"], g["base_txt"],
                                  g["I_img"], g["I_txt"])
    assert tokens.shape == g["tokens"].shape == (5, 3, 40)
    # the reference computed in float32, the oracle in float64
    assert np.abs(tokens - g["tokens"]).max() < 2e-6 * max(1.0, np.abs(g["tokens"]).max())


# ------------------------------------------------------------------ gathered contrastive loss (§8 f3)
def test_clip_loss_oracle_matches_torch_autograd_of_the_reference_statements(golden_dir):
    from oracle import clip_loss_oracle as lorc

    g = np.load(os.path.join(golden_dir, "clip_loss.npz"))
    world, scale = int(g["world"]), float(g["scale"])
    I_all = np.concatenate([g[f"I{r}"] for r in range(world)])      # rank order (the reference: local first)
    T_all = np.concatenate([g[f"T{r}"] for r in range(world)])
    B = g["I0"].shape[0]
    for r in range(world):
        loss, dI, dT, ds = lorc.clip_loss(I_all, T_all, scale, row0=r * B, n_local=B)
        assert abs(loss - float(g[f"loss{r}"])) < 1e-12
        assert np.abs(dI - g[f"dI{r}"]).max() < 1e-12 and np.abs(dT - g[f"dT{r}"]).max() < 1e-12
        assert abs(ds - float(g[f"dscale{r}"])) < 1e-12


def test_cirr_testoutput_matches_reference(golden_dir):
    """get_cirr_testoutput (src/eval_utils.py:1070-1087), produced by the reference's own function."""
    z = np.load(os.path.join(golden_dir, "metrics_inputs.npz"))
    e = json.load(open(os.path.join(golden_dir, "metrics_expected.json")))["cirr_test"]
    got = orc.cirr_testoutput(z["gal"], z["qf"], e["reference_names"], e["index_names"], e["pair_ids"])
    assert got == e["output"]
    with pytest.raises(IndexError):   # fewer than 51 gallery images: the reference's [t] for t < 50 runs out
        orc.cirr_testoutput(z["gal"][:40], z["qf"][:3], e["index_names"][:3], e["index_names"][:40], [1, 2, 3])


def test_consumer_training_oracle_matches_reference_modules(golden_dir):
    """oracle/consumer_train_oracle.py against tokens and parameter gradients computed by the
    reference's own IM2TEXT / CrossFormer classes in train mode (oracle/make_golden_consumer_train.py)."""
    from oracle import consumer_train_oracle as cto
    g = np.load(os.path.join(golden_dir, "consumer_train.npz"))
    sds = [{k.split("/", 1)[1]: g[k] for k in g.files if k.startswith(p + "/")}
           for p in ("img2text", "retrieval_fuse", "text_condition")]
    tok, grads = cto.tokens_and_grads(sds[0], sds[1], sds[2], int(g["dims"][5]), g["feat"], g["topk_image"],
                                      g["topk_text"], g["dtokens"])
    assert np.abs(tok - g["tokens"]).max() < 1e-12
    assert len(grads) == 54
    for name, v in grads.items():
        assert np.abs(v - g["grad/" + name]).max() < 1e-12, name
    # a dropout mask of ones is no dropout; a mask of zeros on a hidden layer kills that layer's weight gradient
    M = g["feat"].shape[0] * (1 + 2 * g["topk_image"].shape[1])
    ones = [np.ones((M, int(g["dims"][1]))), None]
    tok1, grads1 = cto.tokens_and_grads(sds[0], sds[1], sds[2], int(g["dims"][5]), g["feat"], g["topk_image"],
                                        g["topk_text"], g["dtokens"], ones)
    assert np.abs(tok1 - tok).max() < 1e-12
    zeros = [np.zeros((M, int(g["dims"][1]))), None]
    _, grads0 = cto.tokens_and_grads(sds[0], sds[1], sds[2], int(g["dims"][5]), g["feat"], g["topk_image"],
                                     g["topk_text"], g["dtokens"], zeros)
    assert np.abs(grads0["img2text/layers.0.0.weight"]).max() == 0.0


# ------------------------------------------------------------------ tf32 operand rounding of the oracles
def test_round_tf32_ties_signs_subnormals_and_overflow():
    from oracle.consumer_oracle import round_tf32

    h = 2.0 ** -11                    # half a tf32 unit in the last place at 1.0
    x = np.array([1 + h, 1 + 3 * h, 1 + h * 0.999, 1 + h * 1.001, -(1 + h), -(1 + 3 * h), 0.0, -0.0])
    assert list(round_tf32(x, "rne")) == [1, 1 + 4 * h, 1, 1 + 2 * h, -1, -(1 + 4 * h), 0, 0]
    assert list(round_tf32(x, "rz")) == [1, 1 + 2 * h, 1, 1, -1, -(1 + 2 * h), 0, 0]
    assert np.signbit(round_tf32(np.float32(-0.0), "rne"))
    # subnormals round on the same 13-bit grid: 0x1000 x 2^-149 is a tie between 0 and 0x2000 x 2^-149
    sub = np.array([0x1000, 0x1001, 0x2FFF, 0x3000], np.uint32).view(np.float32)
    assert list(round_tf32(sub, "rz")) == list(2.0 ** -149 * np.array([0, 0, 0x2000, 0x2000]))
    assert list(round_tf32(sub, "rne")) == list(2.0 ** -149 * np.array([0, 0x2000, 0x2000, 0x4000]))
    # FLT_MAX lies above the largest tf32 value by more than half a unit: nearest overflows
    fmax = np.finfo(np.float32).max
    tf32_max = (2 - 2.0 ** -10) * 2.0 ** 127
    assert round_tf32(fmax, "rne") == np.inf and round_tf32(-fmax, "rne") == -np.inf
    assert round_tf32(fmax, "rz") == tf32_max and round_tf32(np.float32(tf32_max), "rne") == tf32_max
    special = round_tf32(np.array([np.inf, -np.inf, np.nan], np.float32))
    assert special[0] == np.inf and special[1] == -np.inf and np.isnan(special[2])
    # float64 input is first rounded to float32, as the native operands are stored
    assert round_tf32(1 + 2.0 ** -30, "rz") == 1.0
    with pytest.raises(ValueError):
        round_tf32(x, "up")


def test_round_tf32_matches_the_bit_masks_on_random_values():
    from oracle.consumer_oracle import round_tf32

    rng = np.random.default_rng(0)
    bits = rng.integers(0, 2 ** 32, 100_000, dtype=np.uint64).astype(np.uint32)
    x = bits.view(np.float32)
    fin = np.isfinite(x)
    for mode in ("rne", "rz"):
        r = round_tf32(x, mode).astype(np.float32)
        rb = r.view(np.uint32)
        ok = fin & np.isfinite(r)
        assert np.all(rb[ok] & 0x1FFF == 0)                                  # representable
        d = np.abs(r[ok].astype(np.float64) - x[ok].astype(np.float64))
        ulp = np.spacing(np.abs(x[ok])).astype(np.float64) * 2 ** 13         # tf32 unit of x's binade
        assert np.all(d <= (ulp if mode == "rz" else ulp / 2) * (1 + 1e-12))  # within a (half) unit
        if mode == "rz":
            assert np.all(np.abs(r[ok]) <= np.abs(x[ok]))


def test_tf32_oracles_equal_the_plain_ones_on_tf32_values():
    """Small integers are tf32 numbers and their products and sums stay exact: with such operands the
    tf32 mode changes nothing, forward (numpy oracle) and backward (the autograd Function)."""
    import torch

    from oracle import consumer_oracle as co
    from oracle import consumer_train_oracle as cto

    rng = np.random.default_rng(1)
    sd = {"layers.0.0.weight": rng.integers(-3, 4, (6, 8)), "layers.0.0.bias": rng.integers(-3, 4, 6),
          "fc_out.weight": rng.integers(-3, 4, (5, 6)), "fc_out.bias": rng.integers(-3, 4, 5)}
    x = rng.integers(-4, 5, (7, 8)).astype(np.float32)
    assert np.array_equal(co.im2text(sd, x, tf32=True), co.im2text(sd, x))
    xt = torch.from_numpy(x.astype(np.float64)).requires_grad_(True)
    W = torch.from_numpy(rng.integers(-3, 4, (5, 8)).astype(np.float64)).requires_grad_(True)
    g = torch.from_numpy(rng.integers(-3, 4, (7, 5)).astype(np.float64))
    y = cto._Tf32Linear.apply(xt, W)
    y.backward(g)
    assert torch.equal(y, xt @ W.t()) and torch.equal(xt.grad, g @ W) and torch.equal(W.grad, g.t() @ xt)
    # on general values every product of the backward sees rounded operands
    xt = torch.from_numpy(rng.standard_normal((2, 3, 8))).requires_grad_(True)
    W = torch.from_numpy(rng.standard_normal((5, 8))).requires_grad_(True)
    g = torch.from_numpy(rng.standard_normal((2, 3, 5)))
    cto._Tf32Linear.apply(xt, W).backward(g)
    r = co.round_tf32
    g2, x2 = g.numpy().reshape(6, 5), xt.detach().numpy().reshape(6, 8)
    assert np.array_equal(xt.grad.numpy(), (r(g2) @ r(W.detach().numpy())).reshape(2, 3, 8))
    assert np.array_equal(W.grad.numpy(), r(g2).T @ r(x2))
