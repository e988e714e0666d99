"""Forward pass of the modules that consume the retrieved neighbours, on the native path.

The reference evaluates, per batch (src/trainer.py:59-69; src/eval_utils.py:378-383, 515-519,
661-668, 806-810, 943-947):

    mapped   = img2text(image_features)                       # IM2TEXT, src/model/model.py:104-123
    nb_img   = img2text(topk_image_features)                  # [B, k, 768]
    nb_txt   = img2text(topk_text_features)
    fused    = retrieval_fuse(mapped.unsqueeze(1), nb_img, nb_img)     # CrossFormer, :81-101
    text_c   = text_condition(mapped.unsqueeze(1), nb_txt, nb_txt)
    tokens   = torch.cat([fused, text_c, mapped.unsqueeze(1)], dim=1)  # [B, 3, 768]

as ~60 small PyTorch kernels on `[B, k, 768]` tensors that first travelled GPU -> CPU -> GPU.
`NeighbourConsumer` takes the three modules' weights once and produces `tokens` from the query
features and the neighbour *ids* (the rows are gathered from the resident databases): the eval
loops.  `TrainableNeighbourConsumer` is the same block while the modules learn (src/trainer.py:59-69,
backward at :462-474): its parameters live in one flat torch Parameter that the optimiser updates
in place and the native handle reads through, forward and backward are native launch sequences
(tf32 tcgen05 GEMMs with the operand roles turned for dX and dW), and the gradients arrive through
torch.autograd like any module's.

Weights are taken from `state_dict()`s with the reference's own parameter names, so
`NeighbourConsumer.from_modules(img2text, retrieval_fuse, text_condition)` works on the reference's
module instances unchanged.
"""
from __future__ import annotations

import ctypes as C
from typing import Mapping, Optional

import torch

from . import _capi
from .index import GpuIndexFlat, _stream_ptr
from .retrieval import _device_perm
from .sharded import ShardedKnowledgeBase, _sharded_kb

KIND_MLP, KIND_TO_Q, KIND_TO_K, KIND_TO_V, KIND_TO_OUT = 0, 1, 2, 3, 4
STACK_IMAGE, STACK_TEXT = 0, 1


def _count_prefix(sd: Mapping[str, torch.Tensor], fmt: str) -> int:
    n = 0
    while fmt.format(n) in sd:
        n += 1
    return n


def _call_forward(lib, name, h, feature, image_index, text_index, tail):
    """keds_consumer_<name> with (base, n) of two local indices, or keds_consumer_<name>_sharded with
    the local shards and the exchange of a ShardedKnowledgeBase; `tail` = the arguments from I_img on."""
    kb = _sharded_kb(image_index, text_index)
    if kb is None:
        return getattr(lib, "keds_consumer_" + name)(h, feature.data_ptr(), image_index.rows_ptr(), image_index.ntotal,
                                                     text_index.rows_ptr(), text_index.ntotal, *tail)
    if kb._fx is None:
        raise RuntimeError("the ShardedKnowledgeBase has no exchange yet: run kb.retrieve2 first (its labels are "
                           "what the consumer reads)")
    return getattr(lib, "keds_consumer_" + name + "_sharded")(h, kb.image.local._h, kb.text.local._h, kb._fx.handle,
                                                              feature.data_ptr(), *tail)


class NeighbourConsumer:
    """img2text + retrieval_fuse + text_condition in one launch sequence (tf32 tensor cores)."""

    def __init__(self, img2text_sd: Mapping[str, torch.Tensor], retrieval_fuse_sd: Mapping[str, torch.Tensor],
                 text_condition_sd: Mapping[str, torch.Tensor], heads: int = 8, device: int = 0) -> None:
        self._lib = _capi.load()
        self._h = C.c_void_p()
        self.device = int(device)
        # IM2TEXT: layers.{i}.0 = Linear (+ Dropout + ReLU), fc_out (src/model/model.py:107-118)
        n_hidden = _count_prefix(img2text_sd, "layers.{}.0.weight")
        if n_hidden < 1 or "fc_out.weight" not in img2text_sd:
            raise ValueError("img2text state_dict: expected layers.<i>.0.weight and fc_out.weight")
        w0 = img2text_sd["layers.0.0.weight"]
        d_mid, d_in = int(w0.shape[0]), int(w0.shape[1])
        d_tok = int(img2text_sd["fc_out.weight"].shape[0])
        # CrossFormer: cross_layers.{l}.to_q / to_k / to_v / to_out.0 (src/model/model.py:46-55, 93)
        n_layers = _count_prefix(retrieval_fuse_sd, "cross_layers.{}.to_q.weight")
        if n_layers < 1 or _count_prefix(text_condition_sd, "cross_layers.{}.to_q.weight") != n_layers:
            raise ValueError("retrieval_fuse / text_condition state_dicts: cross_layers.<l>.to_q.weight missing "
                             "or different depths")
        inner = int(retrieval_fuse_sd["cross_layers.0.to_q.weight"].shape[0])
        if inner % heads:
            raise ValueError(f"inner width {inner} is not a multiple of heads={heads}")
        if "cross_layers.0.to_out.0.weight" not in retrieval_fuse_sd:
            raise ValueError("CrossAttention without output projection (heads == 1 and dim_head == q_dim) "
                             "is not supported")
        self.d_in, self.d_mid, self.d_tok = d_in, d_mid, d_tok
        self.n_hidden, self.n_layers, self.heads, self.dim_head = n_hidden, n_layers, heads, inner // heads
        _capi.check(self._lib.keds_consumer_create(d_in, d_mid, d_tok, n_hidden, n_layers, heads, inner // heads,
                                                   self.device, C.byref(self._h)))
        for i in range(n_hidden):
            self._set(KIND_MLP, 0, i, img2text_sd[f"layers.{i}.0.weight"], img2text_sd.get(f"layers.{i}.0.bias"))
        self._set(KIND_MLP, 0, n_hidden, img2text_sd["fc_out.weight"], img2text_sd.get("fc_out.bias"))
        for stack, sd in ((STACK_IMAGE, retrieval_fuse_sd), (STACK_TEXT, text_condition_sd)):
            for l in range(n_layers):
                p = f"cross_layers.{l}."
                self._set(KIND_TO_Q, stack, l, sd[p + "to_q.weight"], sd.get(p + "to_q.bias"))
                self._set(KIND_TO_K, stack, l, sd[p + "to_k.weight"], sd.get(p + "to_k.bias"))
                self._set(KIND_TO_V, stack, l, sd[p + "to_v.weight"], sd.get(p + "to_v.bias"))
                self._set(KIND_TO_OUT, stack, l, sd[p + "to_out.0.weight"], sd.get(p + "to_out.0.bias"))
        _capi.check(self._lib.keds_consumer_finalize(self._h))

    @classmethod
    def from_modules(cls, img2text, retrieval_fuse, text_condition, device: int = 0) -> "NeighbourConsumer":
        """Build from the reference's module instances (IM2TEXT, CrossFormer, CrossFormer)."""
        heads = int(retrieval_fuse.cross_layers[0].heads)
        return cls(img2text.state_dict(), retrieval_fuse.state_dict(), text_condition.state_dict(),
                   heads=heads, device=device)

    def _set(self, kind: int, stack: int, layer: int, W: torch.Tensor, b: Optional[torch.Tensor]) -> None:
        W = W.detach().to(dtype=torch.float32).contiguous()
        bp = 0
        if b is not None:
            b = b.detach().to(dtype=torch.float32).contiguous()
            bp = b.data_ptr()
        if W.is_cuda:  # the native copy runs on the legacy stream: finish whatever produced W / b first
            torch.cuda.current_stream(W.device).synchronize()
        _capi.check(self._lib.keds_consumer_set_linear(self._h, kind, stack, layer, W.data_ptr(), bp,
                                                       int(W.shape[0]), int(W.shape[1])))

    def __call__(self, feature: torch.Tensor, image_index: GpuIndexFlat, text_index: GpuIndexFlat,
                 I_img: torch.Tensor, I_txt: torch.Tensor, perm: Optional[torch.Tensor] = None,
                 out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """tokens [B, 3, d_tok] = cat(fused, text_conditioned, mapped) for query features [B, d_in]
        and neighbour ids I_img / I_txt [B, k] (int64, device) into the two resident databases.
        image_index / text_index may also be `kb.image, kb.text` of a ShardedKnowledgeBase after a
        kb.retrieve2: I_* are then global labels (the merged I it returns), and each neighbour row is
        read from the rank that owns it."""
        if not (feature.is_cuda and feature.dtype == torch.float32 and feature.dim() == 2
                and feature.shape[1] == self.d_in):
            raise TypeError(f"feature must be a CUDA float32 [B, {self.d_in}] tensor")
        for I in (I_img, I_txt):
            if not (I.is_cuda and I.dtype == torch.int64 and I.dim() == 2):
                raise TypeError("neighbour ids must be CUDA int64 [B, k] tensors")
        if I_img.shape != I_txt.shape or I_img.shape[0] != feature.shape[0]:
            raise ValueError("feature, I_img and I_txt disagree on B or k")
        if image_index.d != self.d_in or text_index.d != self.d_in:
            raise ValueError("database width differs from the consumer's input width")
        feature, I_img, I_txt = feature.contiguous(), I_img.contiguous(), I_txt.contiguous()
        B, k = I_img.shape
        if out is None:
            out = torch.empty((B, 3, self.d_tok), dtype=torch.float32, device=feature.device)
        perm = _device_perm(perm, k, feature.device)
        _capi.check(_call_forward(self._lib, "forward", self._h, feature, image_index, text_index,
                                  (I_img.data_ptr(), I_txt.data_ptr(), 0 if perm is None else perm.data_ptr(), B, k,
                                   out.data_ptr(), _stream_ptr(self.device))))
        return out

    def from_features(self, image_features: torch.Tensor, database, topk: int = 16,
                      shuffle: bool = True, exclude=None) -> torch.Tensor:
        """The whole block of src/trainer.py:53-69 / src/eval_utils.py:373-383 for one batch:
        retrieve the topk image / text neighbours of `image_features` from `database`
        (KnowledgeBase or the reference's 5-item sequence with native indices) and return
        tokens [B, 3, d_tok]. The search normalises its copy of the features (src/trainer.py:206);
        img2text sees them as given. shuffle: the batch-shared randperm of :218-219 (it cannot
        change the result beyond fp32 summation order). exclude: int64 [B] or [B, E] rows each query
        must not retrieve (e.g. database.rows_of(names), training without self-retrieval); None:
        the reference's search.

        A row-sharded `database` (a ShardedKnowledgeBase, or a sequence whose [3] / [4] are its
        `image` / `text`) runs the DDP step of retrieval.get_retrieved_features: every rank calls
        this with its own batch (sizes may differ), the queries and exclusions are all-gathered, one
        kb.retrieve2 without feature gathers merges the labels, and each rank runs the consumer over
        its own rows of them with its own randperm. Returns this rank's [B_r, 3, d_tok]."""
        from .index import search2

        if isinstance(database, ShardedKnowledgeBase):
            image_index, text_index = database.image, database.text
        else:
            image_index, text_index = database[3], database[4]
        kb = _sharded_kb(image_index, text_index)
        feats = image_features.detach().to(device=torch.device("cuda", self.device), dtype=torch.float32).contiguous()
        q = feats / feats.norm(dim=1, keepdim=True)
        if kb is None:
            (_, I_img), (_, I_txt) = search2(image_index, text_index, q, topk, exclude=exclude)
        else:
            res, (lo, hi) = kb.retrieve2_ddp(q, topk, exclude, want_feats=False, pool_mode=0)
            I_img, I_txt = res["I_img"][lo:hi], res["I_txt"][lo:hi]
        perm = torch.randperm(topk) if shuffle else None
        return self(feats, image_index, text_index, I_img, I_txt, perm)

    def check(self) -> int:
        """Synchronise and raise if a kernel reported a pipeline error; returns kernels launched so far."""
        n = C.c_int64(0)
        _capi.check(self._lib.keds_consumer_check(self._h, _stream_ptr(self.device), C.byref(n)))
        return int(n.value)

    def set_debug(self, on: bool) -> None:
        _capi.check(self._lib.keds_consumer_set_debug(self._h, int(bool(on))))

    def debug_timeline(self, launch: int, n_ctas: int):
        """[n_ctas, 5] uint64 ns timestamps {start, prologue, dependency, accumulator, end} of the
        `launch`-th k_linear_tf32 launch of the last forward (debug on)."""
        import numpy as np

        out = np.zeros((n_ctas, 5), dtype=np.uint64)
        _capi.check(self._lib.keds_consumer_debug_timeline(self._h, launch, out.ctypes.data, n_ctas))
        return out

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.keds_consumer_free(self._h)
            self._h = C.c_void_p()

    def __del__(self) -> None:  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass


class _ConsumerFn(torch.autograd.Function):
    """tokens = consumer(feature, ids) with the gradient of the flat parameter vector."""

    @staticmethod
    def forward(ctx, mod, feature, image_index, text_index, I_img, I_txt, perm, masks, flat):
        B, k = I_img.shape
        tokens = torch.empty((B, 3, mod.d_tok), dtype=torch.float32, device=feature.device)
        mp = None
        if masks is not None:
            mp = (C.c_void_p * mod.n_hidden)(*[0 if m is None else m.data_ptr() for m in masks])
        pp = 0 if perm is None else perm.data_ptr()
        _capi.check(_call_forward(mod._lib, "forward_train", mod._h, feature, image_index, text_index,
                                  (I_img.data_ptr(), I_txt.data_ptr(), pp, B, k, mp, tokens.data_ptr(),
                                   _stream_ptr(mod.device))))
        ctx.mod, ctx.keep = mod, (masks, feature, I_img, I_txt, perm)   # alive until the backward has run
        return tokens

    @staticmethod
    def backward(ctx, dtokens):
        mod = ctx.mod
        grads = torch.zeros_like(mod.flat)
        dt = dtokens.contiguous().to(torch.float32)
        _capi.check(mod._lib.keds_consumer_backward(mod._h, dt.data_ptr(), grads.data_ptr(), _stream_ptr(mod.device)))
        return None, None, None, None, None, None, None, None, grads


class TrainableNeighbourConsumer(torch.nn.Module):
    """img2text + retrieval_fuse + text_condition as ONE trainable module on the native path.

        consumer = TrainableNeighbourConsumer.from_modules(img2text, retrieval_fuse, text_condition, device=gpu)
        optimizer = torch.optim.AdamW(consumer.parameters(), ...)
        tokens = consumer(image_features, image_index, text_index, I_img, I_txt)      # [B, 3, d_tok], differentiable
        ...
        loss.backward(); optimizer.step()

    `flat` holds every weight and bias (layout: keds_consumer_param_offset); `state_dicts()` hands them
    back under the reference's parameter names (views), `load_state_dicts` takes them in. In train()
    mode IM2TEXT's dropout (src/model/model.py:110-116, p = `dropout`) is applied with masks drawn
    by torch's generator; eval() runs the plain forward.

    On row-sharded bases the indices are `kb.image, kb.text` of a ShardedKnowledgeBase and the ids
    global labels (neighbour rows read from their owners), e.g. per DDP rank:

        out = kb.retrieve2(q_all, 16, want_feats=False, exclude=ex_all, rows=(lo, hi))
        tokens = consumer(feature, kb.image, kb.text, out["I_img"][lo:hi], out["I_txt"][lo:hi], perm)"""

    def __init__(self, img2text_sd: Mapping[str, torch.Tensor], retrieval_fuse_sd: Mapping[str, torch.Tensor],
                 text_condition_sd: Mapping[str, torch.Tensor], heads: int = 8, device: int = 0,
                 dropout: float = 0.1) -> None:
        super().__init__()
        self._lib = _capi.load()
        self._h = C.c_void_p()
        self.device = int(device)
        self.dropout = float(dropout)
        n_hidden = _count_prefix(img2text_sd, "layers.{}.0.weight")
        n_layers = _count_prefix(retrieval_fuse_sd, "cross_layers.{}.to_q.weight")
        if n_hidden < 1 or n_layers < 1 or "fc_out.weight" not in img2text_sd:
            raise ValueError("state_dicts do not look like IM2TEXT / CrossFormer (src/model/model.py:81-123)")
        w0 = img2text_sd["layers.0.0.weight"]
        self.d_mid, self.d_in = int(w0.shape[0]), int(w0.shape[1])
        self.d_tok = int(img2text_sd["fc_out.weight"].shape[0])
        inner = int(retrieval_fuse_sd["cross_layers.0.to_q.weight"].shape[0])
        self.n_hidden, self.n_layers, self.heads, self.dim_head = n_hidden, n_layers, int(heads), inner // int(heads)
        _capi.check(self._lib.keds_consumer_create(self.d_in, self.d_mid, self.d_tok, n_hidden, n_layers, self.heads,
                                                   self.dim_head, self.device, C.byref(self._h)))
        n = int(self._lib.keds_consumer_param_count(self._h))
        self.flat = torch.nn.Parameter(torch.zeros(n, dtype=torch.float32, device=torch.device("cuda", self.device)))
        self._slots = {}   # (module prefix, reference parameter name) -> (offset, shape)
        for i in range(n_hidden + 1):
            name = f"layers.{i}.0" if i < n_hidden else "fc_out"
            self._slot("img2text", name, KIND_MLP, 0, i)
        for stack, prefix in ((STACK_IMAGE, "retrieval_fuse"), (STACK_TEXT, "text_condition")):
            for l in range(n_layers):
                for kind, nm in ((KIND_TO_Q, "to_q"), (KIND_TO_K, "to_k"), (KIND_TO_V, "to_v"), (KIND_TO_OUT, "to_out.0")):
                    self._slot(prefix, f"cross_layers.{l}.{nm}", kind, stack, l)
        self.load_state_dicts(img2text_sd, retrieval_fuse_sd, text_condition_sd)
        self._bind()

    @classmethod
    def from_modules(cls, img2text, retrieval_fuse, text_condition, device: int = 0,
                     dropout: Optional[float] = None) -> "TrainableNeighbourConsumer":
        heads = int(retrieval_fuse.cross_layers[0].heads)
        if dropout is None:  # IM2TEXT's own rate: layers[i] = Sequential(Linear, Dropout, ReLU)
            dropout = float(img2text.layers[0][1].p)
        return cls(img2text.state_dict(), retrieval_fuse.state_dict(), text_condition.state_dict(), heads=heads,
                   device=device, dropout=dropout)

    def _slot(self, prefix: str, name: str, kind: int, stack: int, layer: int) -> None:
        wo, bo, r, c_ = C.c_int64(0), C.c_int64(0), C.c_int64(0), C.c_int64(0)
        _capi.check(self._lib.keds_consumer_param_offset(self._h, kind, stack, layer, C.byref(wo), C.byref(bo),
                                                         C.byref(r), C.byref(c_)))
        self._slots[(prefix, name + ".weight")] = (int(wo.value), (int(r.value), int(c_.value)))
        self._slots[(prefix, name + ".bias")] = (int(bo.value), (int(r.value),))

    def _bind(self) -> None:
        torch.cuda.current_stream(self.flat.device).synchronize()
        _capi.check(self._lib.keds_consumer_bind_params(self._h, self.flat.data_ptr()))
        self._bound_ptr = self.flat.data_ptr()

    def _view(self, t: torch.Tensor, prefix: str, name: str) -> torch.Tensor:
        off, shape = self._slots[(prefix, name)]
        return t[off:off + int(torch.Size(shape).numel())].view(shape)

    def state_dicts(self, grads: bool = False):
        """(img2text_sd, retrieval_fuse_sd, text_condition_sd): views of `flat` (or of `flat.grad`)
        under the reference's parameter names."""
        src = self.flat.grad if grads else self.flat.detach()
        out = {"img2text": {}, "retrieval_fuse": {}, "text_condition": {}}
        for (prefix, name) in self._slots:
            out[prefix][name] = self._view(src, prefix, name)
        return out["img2text"], out["retrieval_fuse"], out["text_condition"]

    def load_state_dicts(self, img2text_sd, retrieval_fuse_sd, text_condition_sd) -> None:
        with torch.no_grad():
            for prefix, sd in (("img2text", img2text_sd), ("retrieval_fuse", retrieval_fuse_sd),
                               ("text_condition", text_condition_sd)):
                for (pf, name) in self._slots:
                    if pf != prefix:
                        continue
                    if name not in sd:
                        raise KeyError(f"{prefix}: parameter {name} missing")
                    self._view(self.flat, prefix, name).copy_(torch.as_tensor(sd[name]).to(self.flat.device, torch.float32))

    def forward(self, feature: torch.Tensor, image_index: GpuIndexFlat, text_index: GpuIndexFlat,
                I_img: torch.Tensor, I_txt: torch.Tensor, perm: Optional[torch.Tensor] = None) -> torch.Tensor:
        if self.flat.data_ptr() != self._bound_ptr:   # the parameter was re-created (.to(), load): adopt the new storage
            self._bind()
        feature = feature.detach().to(device=self.flat.device, dtype=torch.float32).contiguous()
        I_img, I_txt = I_img.contiguous(), I_txt.contiguous()
        if I_img.shape != I_txt.shape or I_img.shape[0] != feature.shape[0] or feature.shape[1] != self.d_in:
            raise ValueError("feature, I_img and I_txt disagree on B, k or d_in")
        B, k = I_img.shape
        if perm is not None:
            perm = perm.to(device=feature.device, dtype=torch.int32).contiguous()
        masks = None
        if self.training and self.dropout > 0.0:
            M = B * (1 + 2 * k)
            keep = 1.0 - self.dropout
            masks = [(torch.rand((M, self.d_mid), device=feature.device) < keep).to(torch.float32) / keep
                     for _ in range(self.n_hidden)]
        return _ConsumerFn.apply(self, feature, image_index, text_index, I_img, I_txt, perm, masks, self.flat)

    def check(self) -> int:
        n = C.c_int64(0)
        _capi.check(self._lib.keds_consumer_check(self._h, _stream_ptr(self.device), C.byref(n)))
        return int(n.value)

    def debug_hidden(self, layer: int, rows: int) -> torch.Tensor:
        """hidden activations [rows, d_mid] of IM2TEXT layer `layer` from the last forward (test hook)"""
        out = torch.empty((rows, self.d_mid), dtype=torch.float32, device=self.flat.device)
        _capi.check(self._lib.keds_consumer_debug_hidden(self._h, int(layer), out.data_ptr(), out.numel(),
                                                         _stream_ptr(self.device)))
        return out

    def __del__(self) -> None:  # pragma: no cover
        try:
            if getattr(self, "_h", None) is not None and self._h:
                self._lib.keds_consumer_free(self._h)
                self._h = C.c_void_p()
        except Exception:
            pass
