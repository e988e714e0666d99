"""CPU oracle for the neighbour consumer in TRAINING mode (SURVEY.md §8 f2): tokens and the
gradients of every parameter.  TEST INFRASTRUCTURE ONLY (tests/ may import it; keds_b200/ never).

A float64 restatement, written functionally on torch tensors so that torch.autograd supplies the
gradients, of what src/trainer.py:59-69 evaluates while img2text / retrieval_fuse / text_condition
are being optimised (backward at src/trainer.py:462-474):

  * IM2TEXT.forward in train mode   src/model/model.py:110-123: each hidden layer is
    nn.Sequential(Linear, Dropout, ReLU), i.e. relu(dropout(x W^T + b)); dropout multiplies by a
    mask of 0 / 1/(1-p) entries.  The mask is an INPUT here (the caller draws it), so the result is
    a deterministic function that the native path can be compared with.
  * CrossAttention / CrossFormer    src/model/model.py:56-101 (their dropout sits behind to_out
    with p = 0. in the reference's constructor calls, src/main.py:151-152).

PARITY PINNING: tests/test_oracle_golden.py checks this module against
tests/golden/consumer_train.npz = tokens and parameter gradients computed by the reference's own
module classes in train mode (AST-extracted, float64, dropout 0) through torch.autograd
(oracle/make_golden_consumer_train.py).
"""
from __future__ import annotations

from typing import Dict, Mapping, Optional, Sequence

import numpy as np
import torch

from .consumer_oracle import round_tf32


def _t(a) -> torch.Tensor:
    if isinstance(a, torch.Tensor):
        return a.detach().to(torch.float64)
    return torch.from_numpy(np.asarray(a, dtype=np.float64))


class _Tf32Linear(torch.autograd.Function):
    """x W^T with both operands rounded to tf32 in every product, as the native GEMMs compute them:
    forward x W^T, backward dX = dY W and dW = dY^T X."""

    @staticmethod
    def forward(ctx, x, W):
        ctx.save_for_backward(x, W)
        return _tf32(x) @ _tf32(W).t()

    @staticmethod
    def backward(ctx, g):
        x, W = ctx.saved_tensors
        g2 = _tf32(g.reshape(-1, g.shape[-1]))
        dx = (g2 @ _tf32(W)).reshape(x.shape)
        dW = g2.t() @ _tf32(x.reshape(-1, x.shape[-1]))
        return dx, dW


def _tf32(t: torch.Tensor) -> torch.Tensor:
    return torch.from_numpy(round_tf32(t.detach().numpy()))


def _matmul_wt(x: torch.Tensor, W: torch.Tensor, tf32: bool) -> torch.Tensor:
    return _Tf32Linear.apply(x, W) if tf32 else x @ W.t()


def _params(sd: Mapping[str, object]) -> Dict[str, torch.Tensor]:
    return {k: _t(v).clone().requires_grad_(True) for k, v in sd.items()}


def _im2text(p: Dict[str, torch.Tensor], x: torch.Tensor, masks: Optional[Sequence[Optional[torch.Tensor]]],
             gates: Optional[Sequence[torch.Tensor]] = None, tf32: bool = False) -> torch.Tensor:
    i = 0
    while f"layers.{i}.0.weight" in p:
        z = _matmul_wt(x, p[f"layers.{i}.0.weight"], tf32) + p[f"layers.{i}.0.bias"]
        if masks is not None and masks[i] is not None:
            z = z * masks[i]
        # gates: the ReLU decisions of another evaluation of the same network (0 / 1 per unit). A
        # reduced-precision forward and this float64 one disagree on units whose pre-activation is
        # within rounding of zero; each such unit passes or blocks its whole gradient, so a gradient
        # comparison takes the gates from the path under test (the forward value differs by the
        # tiny pre-activation only).
        x = torch.relu(z) if gates is None else z * gates[i]
        i += 1
    return _matmul_wt(x, p["fc_out.weight"], tf32) + p["fc_out.bias"]


def _crossformer(p: Dict[str, torch.Tensor], q: torch.Tensor, kv: torch.Tensor, heads: int,
                 tf32: bool = False) -> torch.Tensor:
    B, n, _ = kv.shape
    l = 0
    while f"cross_layers.{l}.to_q.weight" in p:
        pre = f"cross_layers.{l}."
        Q = _matmul_wt(q, p[pre + "to_q.weight"], tf32) + p[pre + "to_q.bias"]
        K = _matmul_wt(kv, p[pre + "to_k.weight"], tf32) + p[pre + "to_k.bias"]
        V = _matmul_wt(kv, p[pre + "to_v.weight"], tf32) + p[pre + "to_v.bias"]
        inner = Q.shape[-1]
        dh = inner // heads
        Qh = Q.reshape(B, 1, heads, dh).permute(0, 2, 1, 3)
        Kh = K.reshape(B, n, heads, dh).permute(0, 2, 1, 3)
        Vh = V.reshape(B, n, heads, dh).permute(0, 2, 1, 3)
        attn = torch.softmax(torch.einsum("bhid,bhjd->bhij", Qh, Kh) * dh ** -0.5, dim=-1)
        out = torch.einsum("bhij,bhjd->bhid", attn, Vh).permute(0, 2, 1, 3).reshape(B, 1, inner)
        q = _matmul_wt(out, p[pre + "to_out.0.weight"], tf32) + p[pre + "to_out.0.bias"]
        l += 1
    return q


def tokens_and_grads(img2text_sd, retrieval_fuse_sd, text_condition_sd, heads: int, feature, nb_img_rows, nb_txt_rows,
                     dtokens, masks: Optional[Sequence[Optional[object]]] = None, gates: Optional[Sequence[object]] = None,
                     tf32: bool = False):
    """feature [B, d_in]; nb_*_rows [B, k, d_in] the gathered neighbour rows; masks: per hidden layer
    None or [B(1+2k), d_mid] multipliers over the rows (queries | image neighbours | text neighbours).
    tf32: every nn.Linear product, forward and backward, with tf32-rounded operands as the native
    GEMMs compute them (attention, softmax, bias adds and bias gradients stay exact).
    Returns (tokens [B,3,d_tok] float64 numpy, {"img2text/<name>": grad, "retrieval_fuse/<name>": ...})."""
    pm, pf, pc = _params(img2text_sd), _params(retrieval_fuse_sd), _params(text_condition_sd)
    feat, ni, nt = _t(feature), _t(nb_img_rows), _t(nb_txt_rows)
    B, k, d_in = ni.shape
    x = torch.cat([feat, ni.reshape(B * k, d_in), nt.reshape(B * k, d_in)], dim=0)
    mk = None if masks is None else [None if m is None else _t(m) for m in masks]
    gt = None if gates is None else [_t(gv) for gv in gates]
    y = _im2text(pm, x, mk, gt, tf32)
    mapped = y[:B]
    nb_img = y[B:B + B * k].reshape(B, k, -1)
    nb_txt = y[B + B * k:].reshape(B, k, -1)
    fused = _crossformer(pf, mapped[:, None, :], nb_img, heads, tf32)
    text_c = _crossformer(pc, mapped[:, None, :], nb_txt, heads, tf32)
    tokens = torch.cat([fused, text_c, mapped[:, None, :]], dim=1)
    tokens.backward(_t(dtokens))
    grads = {}
    for prefix, p in (("img2text", pm), ("retrieval_fuse", pf), ("text_condition", pc)):
        for name, t in p.items():
            grads[f"{prefix}/{name}"] = t.grad.numpy()
    return tokens.detach().numpy(), grads
