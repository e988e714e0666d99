"""CPU oracle for the neighbour consumer (SURVEY.md §8 f2).  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py may import this module; the product
(keds_b200/) never does and has no CPU path.

A numpy float64 restatement of the reference's eval-mode forward of
  * IM2TEXT.forward          src/model/model.py:120-123  (layers = Linear -> Dropout -> ReLU, :110-116;
                                                            dropout is the identity in eval)
  * CrossAttention.forward   src/model/model.py:56-79    (to_q/to_k/to_v, heads split 'b n (h d)',
                                                            dots * dim_head**-0.5, softmax over the
                                                            neighbours, attn @ v, to_out)
  * CrossFormer.forward      src/model/model.py:98-101   (q = layer(q, k, v) for each layer; k, v fixed)
  * the call sequence        src/trainer.py:59-69, src/eval_utils.py:378-383
Weights come as state_dict-style mappings with the reference's parameter names.

PARITY PINNING: checked in tests/test_oracle_golden.py against tests/golden/consumer.npz, which
holds outputs of the reference's own classes executed unchanged from /root/reference via AST
extraction (oracle/make_golden_consumer.py).
"""
from __future__ import annotations

from typing import Mapping

import numpy as np


def _f64(a) -> np.ndarray:
    if hasattr(a, "detach"):
        a = a.detach().cpu().numpy()
    return np.asarray(a, dtype=np.float64)


# How the tensor-core products of keds_b200 see their fp32 operands: the TMA unit converts them to
# tf32 (10 explicit mantissa bits) on the way into shared memory, to nearest with ties to even,
# subnormals kept. Measured on a B200 through an identity operand (tests/test_gpu_consumer_kernels.py).
TF32_ROUNDING = "rne"


def round_tf32(x, mode: str = TF32_ROUNDING) -> np.ndarray:
    """x as float32, then rounded to tf32, as float64. mode: "rne" = to nearest, ties to even,
    "rz" = toward zero (the 13 low mantissa bits dropped). Infinities and NaNs pass unchanged; a
    finite value may round up to infinity."""
    a = np.asarray(x, dtype=np.float32)
    u = np.ascontiguousarray(a).view(np.uint32)
    if mode == "rz":
        r = u
    elif mode == "rne":
        r = u + np.uint32(0xFFF) + ((u >> np.uint32(13)) & np.uint32(1))
    else:
        raise ValueError(f"unknown tf32 rounding mode {mode!r}")
    r = np.where(np.isfinite(a), r & np.uint32(0xFFFFE000), u)
    return r.view(np.float32).astype(np.float64)


def linear(x: np.ndarray, W, b=None, tf32: bool = False) -> np.ndarray:
    """x W^T + b; tf32: both operands of the product rounded as the native GEMM rounds them (the
    bias add stays exact)."""
    y = round_tf32(x) @ round_tf32(_f64(W)).T if tf32 else x @ _f64(W).T
    return y if b is None else y + _f64(b)


def im2text(sd: Mapping[str, object], x, tf32: bool = False) -> np.ndarray:
    """src/model/model.py:120-123."""
    x = _f64(x)
    i = 0
    while f"layers.{i}.0.weight" in sd:
        x = np.maximum(linear(x, sd[f"layers.{i}.0.weight"], sd.get(f"layers.{i}.0.bias"), tf32), 0.0)
        i += 1
    return linear(x, sd["fc_out.weight"], sd.get("fc_out.bias"), tf32)


def cross_attention(sd: Mapping[str, object], prefix: str, q: np.ndarray, kv: np.ndarray, heads: int,
                    tf32: bool = False) -> np.ndarray:
    """src/model/model.py:56-79 with k = v = kv.  q: [B, nq, dq], kv: [B, n, dk] -> [B, nq, dq].
    tf32: the four projections as the native GEMM computes them; attention itself stays exact."""
    B, nq, _ = q.shape
    n = kv.shape[1]
    Q = linear(q, sd[prefix + "to_q.weight"], sd.get(prefix + "to_q.bias"), tf32)
    K = linear(kv, sd[prefix + "to_k.weight"], sd.get(prefix + "to_k.bias"), tf32)
    V = linear(kv, sd[prefix + "to_v.weight"], sd.get(prefix + "to_v.bias"), tf32)
    inner = Q.shape[-1]
    dh = inner // heads
    Q = Q.reshape(B, nq, heads, dh).transpose(0, 2, 1, 3)   # b h n d
    K = K.reshape(B, n, heads, dh).transpose(0, 2, 1, 3)
    V = V.reshape(B, n, heads, dh).transpose(0, 2, 1, 3)
    dots = np.einsum("bhid,bhjd->bhij", Q, K) * dh ** -0.5
    dots = dots - dots.max(axis=-1, keepdims=True)
    attn = np.exp(dots)
    attn = attn / attn.sum(axis=-1, keepdims=True)
    out = np.einsum("bhij,bhjd->bhid", attn, V).transpose(0, 2, 1, 3).reshape(B, nq, inner)
    return linear(out, sd[prefix + "to_out.0.weight"], sd.get(prefix + "to_out.0.bias"), tf32)


def crossformer(sd: Mapping[str, object], q: np.ndarray, kv: np.ndarray, heads: int, tf32: bool = False) -> np.ndarray:
    """src/model/model.py:98-101."""
    l = 0
    while f"cross_layers.{l}.to_q.weight" in sd:
        q = cross_attention(sd, f"cross_layers.{l}.", q, kv, heads, tf32)
        l += 1
    return q


def consumer_tokens(img2text_sd, retrieval_fuse_sd, text_condition_sd, heads: int, feature, base_img, base_txt,
                    I_img, I_txt, tf32: bool = False) -> np.ndarray:
    """tokens [B, 3, d_tok] of src/trainer.py:59-69 from neighbour ids into the two databases.
    tf32: every nn.Linear product with tf32-rounded operands (what the native path computes)."""
    I_img = np.asarray(I_img)
    I_txt = np.asarray(I_txt)
    B, k = I_img.shape
    base_img = _f64(base_img)
    base_txt = _f64(base_txt)
    mapped = im2text(img2text_sd, feature, tf32)
    nb_img = im2text(img2text_sd, base_img[I_img.reshape(-1)], tf32).reshape(B, k, -1)
    nb_txt = im2text(img2text_sd, base_txt[I_txt.reshape(-1)], tf32).reshape(B, k, -1)
    fused = crossformer(retrieval_fuse_sd, mapped[:, None, :], nb_img, heads, tf32)
    text_c = crossformer(text_condition_sd, mapped[:, None, :], nb_txt, heads, tf32)
    return np.concatenate([fused, text_c, mapped[:, None, :]], axis=1)


def random_state_dicts(d_in: int, d_mid: int, d_tok: int, n_hidden: int, n_layers: int, heads: int, dim_head: int,
                       seed: int):
    """Seeded float32 weights in the reference's parameter naming (nn.Linear-like scale), for parity
    tests at full width. Returns (img2text_sd, retrieval_fuse_sd, text_condition_sd) of numpy arrays."""
    rng = np.random.default_rng(seed)

    def lin(out_f, in_f):
        bound = 1.0 / np.sqrt(in_f)
        return (rng.uniform(-bound, bound, (out_f, in_f)).astype(np.float32),
                rng.uniform(-bound, bound, (out_f,)).astype(np.float32))

    m = {}
    w = d_in
    for i in range(n_hidden):
        m[f"layers.{i}.0.weight"], m[f"layers.{i}.0.bias"] = lin(d_mid, w)
        w = d_mid
    m["fc_out.weight"], m["fc_out.bias"] = lin(d_tok, d_mid)
    inner = heads * dim_head
    stacks = []
    for _ in range(2):
        s = {}
        for l in range(n_layers):
            p = f"cross_layers.{l}."
            s[p + "to_q.weight"], s[p + "to_q.bias"] = lin(inner, d_tok)
            s[p + "to_k.weight"], s[p + "to_k.bias"] = lin(inner, d_tok)
            s[p + "to_v.weight"], s[p + "to_v.bias"] = lin(inner, d_tok)
            s[p + "to_out.0.weight"], s[p + "to_out.0.bias"] = lin(d_tok, inner)
        stacks.append(s)
    return m, stacks[0], stacks[1]
