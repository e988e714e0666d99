"""GPU (-m gpu): the neighbour consumer's attention kernels ALONE (keds_consumer_debug_attend) against
the float64 reference of oracle/attention_exact.py and its per-element bound, and the backward's
column sums (k_colsum) bit for bit through the public backward.

Per shape and input kind (random, sharp softmaxes over +-80, exactly tied scores, cancelling dO):
  1. every element of O (each forward variant that applies), dQ, dK and dV lies within the bound;
  2. every float of the output and dKV buffers outside this launch's rows and this layer's key /
     value columns keeps its NaN sentinel bit for bit (KV laid out as the consumer lays it out for
     L = 3 layers, the launch at layer 1, with guard rows after each stack);
  3. three calls give bit-identical results;
  4. k_cross_attend<64> and k_cross_attend<0> agree within twice the bound, and the production
     choice (variant 0) is bit-identical to the kernel the selection rule names.
"""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from keds_b200 import _capi  # noqa: E402
from keds_b200.index import _stream_ptr  # noqa: E402
from oracle import attention_exact as ax  # noqa: E402

SENTINEL = 0x7FC0FFEE               # a quiet NaN no kernel produces
L, LAYER = 3, 1                     # KV holds three layers' keys and values; the launch reads layer 1
KINDS = ["random", "sharp", "ties", "cancel"]

# (B, k, heads, dim_head): tests/test_gpu_consumer.py's ATTENTION_SHAPES, then the reference's 8 x 64
# at k = 16 and at the shared-memory limits of the backward (705 is the first k beyond the default
# 48 KB, 1024 the largest the forward accepts), and 32 heads x 64
SHAPES = [
    (1, 31, 16, 64), (129, 32, 32, 16), (129, 33, 6, 40), (1, 64, 2, 96), (129, 100, 1, 4), (129, 64, 16, 64),
    (1, 100, 32, 16), (129, 31, 2, 96),
    (8, 16, 8, 64), (8, 705, 8, 64), (8, 1024, 8, 64), (4, 200, 32, 64),
]


class Handle:
    def __init__(self, heads, dh):
        self.lib = _capi.load()
        self.h = C.c_void_p()
        _capi.check(self.lib.keds_consumer_create(4, 4, 4, 1, 1, heads, dh, 0, C.byref(self.h)))

    def close(self):
        self.lib.keds_consumer_free(self.h)


def sentinel(n):
    return torch.full((n,), SENTINEL, dtype=torch.int32, device="cuda").view(torch.float32)


class Case:
    """Both stacks of one launch: Q, dO [2][B][inner], KV [2][B k][ld_kv] with this layer's keys at
    k_off and values at v_off, each head's inputs drawn by oracle.attention_exact.inputs."""

    def __init__(self, B, k, heads, dh, kind, seed):
        self.B, self.k, self.heads, self.dh = B, k, heads, dh
        self.inner = inner = heads * dh
        self.ld = L * 2 * inner
        self.k_off, self.v_off = 2 * LAYER * inner, (2 * LAYER + 1) * inner
        q, K, V, dO = ax.inputs(2 * B * heads, k, dh, kind, seed, device="cuda")   # [(z, b, h), ...]
        self.q, self.K, self.V, self.dO = q, K, V, dO
        g = torch.Generator(device="cuda").manual_seed(seed)
        KV = torch.randn(2, B * k, self.ld, generator=g, device="cuda")
        per_row = lambda x: x.reshape(2, B, heads, k, dh).permute(0, 1, 3, 2, 4).reshape(2, B * k, inner)  # noqa: E731
        KV[:, :, self.k_off:self.k_off + inner] = per_row(K)
        KV[:, :, self.v_off:self.v_off + inner] = per_row(V)
        self.KV = KV.contiguous()
        self.Q = q.reshape(2, B, inner).contiguous()
        self.G = dO.reshape(2, B, inner).contiguous()
        self.out_rows = B + 2                    # two guard rows after each stack's output
        self.dkv_rows = B * k + 2

    def run(self, hd, variant, backward=False):
        out = sentinel(2 * self.out_rows * self.inner)
        dkv = sentinel(2 * self.dkv_rows * self.ld)
        p = lambda t, z, rows, w: t.data_ptr() + 4 * z * rows * w  # noqa: E731
        st = _stream_ptr(0)
        _capi.check(hd.lib.keds_consumer_debug_attend(
            hd.h, variant, int(backward), self.B, self.k, p(self.Q, 0, self.B, self.inner),
            p(self.Q, 1, self.B, self.inner), p(self.KV, 0, self.B * self.k, self.ld),
            p(self.KV, 1, self.B * self.k, self.ld), self.ld, self.k_off, self.v_off,
            p(self.G, 0, self.B, self.inner), p(self.G, 1, self.B, self.inner),
            p(out, 0, self.out_rows, self.inner), p(out, 1, self.out_rows, self.inner),
            p(dkv, 0, self.dkv_rows, self.ld), p(dkv, 1, self.dkv_rows, self.ld), st))
        _capi.check(hd.lib.keds_consumer_check(hd.h, st, None))
        return out.view(2, self.out_rows, self.inner), dkv.view(2, self.dkv_rows, self.ld)

    def heads_of(self, out):
        """output rows of both stacks -> [2 B heads, dh] float64"""
        return out[:, :self.B].reshape(-1, self.dh).double()

    def rows_of(self, dkv, off):
        """dK (off = k_off) or dV (off = v_off) -> [2 B heads, k, dh] float64"""
        x = dkv[:, :self.B * self.k, off:off + self.inner].reshape(2, self.B, self.k, self.heads, self.dh)
        return x.permute(0, 1, 3, 2, 4).reshape(-1, self.k, self.dh).double()

    def untouched(self, out, dkv=None):
        """the sentinel everywhere but the rows and columns a launch may write"""
        ok = bool((out[:, self.B:].view(torch.int32) == SENTINEL).all())
        if dkv is not None:
            mask = torch.ones_like(dkv, dtype=torch.bool)
            for off in (self.k_off, self.v_off):
                mask[:, :self.B * self.k, off:off + self.inner] = False
            ok = ok and bool((dkv.view(torch.int32)[mask] == SENTINEL).all())
        return ok


def bits(t):
    return t.view(torch.int32)


def within(got, ref, bound):
    return bool(((got - ref).abs() <= bound).all())


def ratio(got, ref, bound):
    return float(((got - ref).abs() / bound).max())


@pytest.fixture(scope="module")
def report():
    worst = {}
    yield worst
    for key, v in sorted(worst.items()):
        print(f"{key}: worst error / bound " + "  ".join(f"{n} {x:.2e}" for n, x in v.items()))


@pytest.mark.parametrize("B,k,heads,dh", SHAPES)
def test_attention_kernels_within_the_bound(B, k, heads, dh, report):
    hd = Handle(heads, dh)
    try:
        worst = {}
        for i, kind in enumerate(KINDS):
            case = Case(B, k, heads, dh, kind, seed=B * 7919 + k * 31 + heads + i)
            sigma = ax.scale(dh)
            O, bo = ax.forward(case.q, case.K, case.V, sigma)
            variants = (1, 2) if dh == 64 else (1,)
            got = {}
            for v in variants:
                out, _ = case.run(hd, v)
                assert case.untouched(out), f"{kind}: variant {v} wrote outside its output rows"
                got[v] = case.heads_of(out)
                r = ratio(got[v], O, bo)
                assert r <= 1.0, f"{kind}: variant {v} O at {r:.3g} x the bound"
                worst[f"O<{64 if v == 2 else 0}>"] = max(worst.get(f"O<{64 if v == 2 else 0}>", 0.0), r)
            if len(variants) == 2:
                assert within(got[1], got[2], 2 * bo), f"{kind}: the two forward kernels disagree"
            auto, _ = case.run(hd, 0)
            for _ in range(2):
                again, _ = case.run(hd, 0)
                assert torch.equal(bits(again), bits(auto)), f"{kind}: forward not deterministic"
            ruled = 2 if dh == 64 else 1      # 16-byte aligned rows here: the rule names <64> at dim_head 64
            assert torch.equal(case.heads_of(auto), got[ruled]), f"{kind}: variant 0 is not variant {ruled}"

            ref, bb = ax.backward(case.q, case.K, case.V, case.dO, sigma)
            dq, dkv = case.run(hd, 0, backward=True)
            assert case.untouched(dq, dkv), f"{kind}: the backward wrote outside this layer's rows and columns"
            for _ in range(2):
                dq2, dkv2 = case.run(hd, 0, backward=True)
                assert torch.equal(bits(dq2), bits(dq)) and torch.equal(bits(dkv2), bits(dkv)), \
                    f"{kind}: backward not deterministic"
            for name, g in (("dQ", case.heads_of(dq)), ("dK", case.rows_of(dkv, case.k_off)),
                            ("dV", case.rows_of(dkv, case.v_off))):
                r = ratio(g, ref[name], bb[name])
                assert r <= 1.0, f"{kind}: {name} at {r:.3g} x the bound"
                worst[name] = max(worst.get(name, 0.0), r)
        report[f"B={B} k={k} heads={heads} dh={dh}"] = worst
    finally:
        hd.close()


def test_the_bound_rejects_what_a_subtly_wrong_kernel_would_compute():
    """the device results themselves, against references of a dropped neighbour, the wrong scale,
    swapped heads or stacks and the previous layer's keys (tests/test_attention_bound_host.py shows
    the same for the backward's rules on the fp32 emulation)"""
    B, k, heads, dh = 8, 1024, 8, 64
    hd = Handle(heads, dh)
    try:
        case = Case(B, k, heads, dh, "random", seed=3)
        sigma = ax.scale(dh)
        out, _ = case.run(hd, 0)
        got = case.heads_of(out)
        O, bo = ax.forward(case.q, case.K, case.V, sigma)
        assert within(got, O, bo)
        for j in (k - 1, 32):
            keep = [i for i in range(k) if i != j]
            assert not within(got, ax.forward(case.q, case.K[:, keep], case.V[:, keep], sigma)[0], bo), j
        assert not within(got, ax.forward(case.q, case.K, case.V, ax.scale(case.inner))[0], bo)
        per_head = O.reshape(2, B, heads, dh)
        assert not within(got, per_head[:, :, [1, 0] + list(range(2, heads))].reshape(-1, dh), bo)
        assert not within(got, per_head.flip(0).reshape(-1, dh), bo)
        prev = case.KV[:, :, case.k_off - 2 * case.inner:case.k_off - case.inner]
        prev = prev.reshape(2, B, k, heads, dh).permute(0, 1, 3, 2, 4).reshape(-1, k, dh)
        assert not within(got, ax.forward(case.q, prev, case.V, sigma)[0], bo)

        dq, dkv = case.run(hd, 0, backward=True)
        ref, bb = ax.backward(case.q, case.K, case.V, case.dO, sigma)
        dK, dV = case.rows_of(dkv, case.k_off), case.rows_of(dkv, case.v_off)
        assert not within(dK, ref["dV"], bb["dK"]) and not within(dV, ref["dK"], bb["dV"]), "dK and dV swapped"
        assert not within(case.heads_of(dq), ref["dQ"] / sigma, bb["dQ"]), "dQ without sigma"
    finally:
        hd.close()


def test_debug_attend_refuses_before_launching():
    hd = Handle(8, 40)
    lib = hd.lib
    try:
        Q = torch.zeros(2, 4, 320, device="cuda")
        KV = torch.zeros(2, 4 * 16, 6 * 320, device="cuda")
        host = torch.zeros(4, 320)
        p, ld = Q.data_ptr(), 6 * 320
        kv = KV.data_ptr()

        def call(variant=0, backward=0, B=4, k=16, q=p, ldkv=ld, k_off=640, v_off=960, dO=p, dkv=kv):
            return lib.keds_consumer_debug_attend(hd.h, variant, backward, B, k, q, q, kv, kv, ldkv, k_off, v_off, dO,
                                                  dO, p, p, dkv, dkv, None)
        assert call(variant=2) == -1                      # <64> needs dim_head 64
        assert call(variant=3) == -1
        assert call(variant=1, backward=1) == -1          # the forward variants are forward only
        assert call(k=0) == -1 and call(k=1025) == -1
        assert call(B=0) == -1
        assert call(q=None) == -1
        assert call(q=host.data_ptr()) == -1              # host memory
        assert call(backward=1, dO=None) == -1 and call(backward=1, dkv=None) == -1
        assert call(ldkv=960 + 319) == -1                 # values beyond ld_kv
        hd.close()
        hd = Handle(32, 64)                               # 32 x (64 + 1024) floats fit, the backward's twice not
        big = torch.zeros(2, 1024, 2 * 2048, device="cuda")
        assert lib.keds_consumer_debug_attend(hd.h, 0, 1, 1, 1024, p, p, big.data_ptr(), big.data_ptr(), 4096, 0,
                                              2048, p, p, p, p, big.data_ptr(), big.data_ptr(), None) == -1
        assert "too large" in _capi.last_error()
    finally:
        hd.close()


# ------------------------------------------------------------------------------------ through the backward
def trainable(B, k, seed):
    from keds_b200 import faiss_compat as faiss
    from keds_b200.consumer import TrainableNeighbourConsumer
    from keds_b200.index import GpuIndexFlat
    from oracle import consumer_oracle as corc

    sds = corc.random_state_dicts(96, 64, 80, 1, 2, 2, 16, seed=seed)
    mod = TrainableNeighbourConsumer(*({n: torch.from_numpy(np.ascontiguousarray(v, dtype=np.float32))
                                        for n, v in sd.items()} for sd in sds), heads=2, device=0, dropout=0.0)
    rng = np.random.default_rng(seed)
    n = 300
    ix = []
    for _ in range(2):
        i = GpuIndexFlat(96, faiss.METRIC_INNER_PRODUCT, 0)
        i.add(rng.standard_normal((n, 96)).astype(np.float32))
        ix.append(i)
    feat = torch.from_numpy(rng.standard_normal((B, 96)).astype(np.float32)).cuda()
    I = [torch.from_numpy(rng.integers(0, n, (B, k)).astype(np.int64)).cuda() for _ in range(2)]
    dtok = torch.from_numpy(rng.standard_normal((B, 3, 80)).astype(np.float32)).cuda()
    return mod, ix, feat, I, dtok


def train_step(mod, ix, feat, I, dtok):
    mod.flat.grad = None
    mod(feat, ix[0], ix[1], I[0], I[1]).backward(dtok)
    assert mod.check() > 0
    return mod.flat.grad.clone()


def colsum_order(x):
    """k_colsum's order in fp32: row r into partial r mod 8 (in row order), then partials 0..7 in order"""
    x = np.asarray(x, np.float32)
    part = np.zeros((8, x.shape[1]), np.float32)
    for r in range(x.shape[0]):
        part[r % 8] = part[r % 8] + x[r]
    t = part[0].copy()
    for i in range(1, 8):
        t = t + part[i]
    return t


@pytest.mark.parametrize("B", [1, 37, 129])
def test_last_to_out_bias_gradients_are_kcolsum_of_dtokens_bit_for_bit(B):
    """d_tok = 80: the second 32-column tile of k_colsum is full, the third holds 16 columns"""
    mod, ix, feat, I, dtok = trainable(B, 5, seed=B)
    train_step(mod, ix, feat, I, dtok)
    _, gf, gc = mod.state_dicts(grads=True)
    d = dtok.cpu().numpy()
    for z, g in ((0, gf), (1, gc)):
        got = g["cross_layers.1.to_out.0.bias"].cpu().numpy()
        want = colsum_order(d[:, z, :])
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), f"stack {z}"


def test_the_whole_backward_is_deterministic():
    mod, ix, feat, I, dtok = trainable(129, 33, seed=5)
    first = train_step(mod, ix, feat, I, dtok)
    again = train_step(mod, ix, feat, I, dtok)
    assert torch.equal(first.view(torch.int32), again.view(torch.int32))
