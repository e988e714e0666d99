"""GPU (-m gpu): the tf32 tcgen05 GEMM of the neighbour consumer ALONE, every kernel variant forced in
turn (keds_consumer_debug_linear), against a float64 reference of the same product with the operands
rounded to tf32 the way the TMA unit rounds them (oracle.consumer_oracle.round_tf32).

Per variant and shape:
  1. every element: |C - ref| <= (K + 8) 2^-23 sum_k |a~ w~| + 2^-23 |b|  (fp32 accumulation in any
     order, with rounding or truncation, plus the bias add)
  2. against the reference built with the OTHER rounding mode the max error is at least 20x larger
     (at K ~ 768 the worst-case bound of 1. cannot tell the modes apart; this ratio can)
  3. every float of C's buffer outside the two M x N results keeps its NaN sentinel bit for bit
     (padding columns up to ldc, rows after M, the gap between interleaved problems)
  4. three calls give bit-identical results (split-K reduces its partials in a fixed order)
  5. any two variants agree within twice the bound of 1.; the production choice is bit-identical
     to the variant keds_debug_linear_plan names
"""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from keds_b200 import _capi  # noqa: E402
from keds_b200.index import _stream_ptr  # noqa: E402
from oracle.consumer_oracle import TF32_ROUNDING, round_tf32  # noqa: E402

VARIANTS = (1, 2, 3, 4, 5)          # 128-col, 256-col, persistent, split-K x2, split-K x4
OTHER_MODE = "rz" if TF32_ROUNDING == "rne" else "rne"
SENTINEL = 0x7FC0FFEE               # a quiet NaN no kernel produces
U = 2.0 ** -23


@pytest.fixture(scope="module")
def handle():
    lib = _capi.load()
    h = C.c_void_p()
    _capi.check(lib.keds_consumer_create(4, 4, 4, 1, 1, 1, 4, 0, C.byref(h)))
    yield lib, h
    lib.keds_consumer_free(h)


def round4(x):
    return (x + 3) & ~3


class Problem:
    """nz independent products C[z] = act(A[z] W[z]^T + b[z]); operands padded with NaN beyond K (a
    kernel that reads the padding poisons its output), C[z] at element offsets c_off[z] of one flat
    buffer with ldc floats between rows."""

    def __init__(self, M, N, K, nz, relu=False, bias=True, lda=None, ldc=None, c_off=None, seed=0):
        rng = np.random.default_rng(seed)
        self.M, self.N, self.K, self.nz, self.relu = M, N, K, nz, relu
        self.lda = lda or round4(K)
        self.ldc = ldc or N
        self.c_off = c_off or [z * (M + 2) * self.ldc for z in range(nz)]
        A = np.full((nz, M, self.lda), np.nan, np.float32)
        W = np.full((nz, N, round4(K)), np.nan, np.float32)
        A[:, :, :K] = rng.standard_normal((nz, M, K))
        W[:, :, :K] = rng.standard_normal((nz, N, K)) / np.sqrt(K)
        self.A, self.W = A, W
        self.b = (rng.standard_normal((nz, N)) * 0.5).astype(np.float32) if bias else None
        self.total = max(self.c_off) + (M + 2) * self.ldc
        self.written = np.zeros(self.total, bool)
        for z in range(nz):
            idx = self.c_off[z] + np.arange(M)[:, None] * self.ldc + np.arange(N)[None, :]
            self.written[idx.reshape(-1)] = True
        self.dA = [torch.from_numpy(A[z]).cuda() for z in range(nz)]
        self.dW = [torch.from_numpy(W[z]).cuda() for z in range(nz)]
        self.db = None if self.b is None else [torch.from_numpy(self.b[z]).cuda() for z in range(nz)]

    def run(self, handle, variant):
        lib, h = handle
        buf = torch.full((self.total,), SENTINEL, dtype=torch.int32, device="cuda").view(torch.float32)
        ptr = lambda ts, z: ts[min(z, self.nz - 1)].data_ptr() if ts is not None and z < self.nz else None  # noqa: E731
        c_ptr = lambda z: buf.data_ptr() + 4 * self.c_off[z] if z < self.nz else None  # noqa: E731
        st = _stream_ptr(0)
        _capi.check(lib.keds_consumer_debug_linear(
            h, variant, ptr(self.dA, 0), ptr(self.dA, 1), self.lda, self.M, self.K, ptr(self.dW, 0), ptr(self.dW, 1),
            ptr(self.db, 0), ptr(self.db, 1), self.N, int(self.relu), c_ptr(0), c_ptr(1), self.ldc, self.nz, st))
        _capi.check(lib.keds_consumer_check(h, st, None))
        return buf.cpu().numpy()

    def results(self, flat):
        """[nz, M, N] float64 from the flat buffer"""
        out = []
        for z in range(self.nz):
            idx = self.c_off[z] + np.arange(self.M)[:, None] * self.ldc + np.arange(self.N)[None, :]
            out.append(flat[idx])
        return np.stack(out).astype(np.float64)

    def reference(self, mode=TF32_ROUNDING, drop_last_kblock=False):
        """float64 (ref [nz, M, N], bound [nz, M, N]) on the GPU"""
        K = self.K
        if drop_last_kblock:
            K = (K - 1) // 32 * 32
        a = torch.from_numpy(round_tf32(self.A[:, :, :K], mode)).cuda()
        w = torch.from_numpy(round_tf32(self.W[:, :, :K], mode)).cuda()
        ref = a @ w.transpose(1, 2)
        bound = (self.K + 8) * U * (a.abs() @ w.abs().transpose(1, 2))
        if self.b is not None:
            b = torch.from_numpy(self.b.astype(np.float64)).cuda()[:, None, :]
            ref = ref + b
            bound = bound + U * b.abs()
        if self.relu:
            ref = ref.clamp_min(0.0)
        return ref.cpu().numpy(), bound.cpu().numpy()


def max_err(got, ref):
    return float(np.abs(got - ref).max())


def accepts(got, ref, bound, ref_other):
    """the checks 1 and 2 of the module docstring"""
    return bool(np.all(np.abs(got - ref) <= bound)) and 20 * max_err(got, ref) <= max_err(got, ref_other)


def check_all_variants(handle, prob):
    ref, bound = prob.reference()
    ref_other, _ = prob.reference(OTHER_MODE)
    got, report = {}, {}
    for v in VARIANTS:
        flat = prob.run(handle, v)
        for _ in range(2):                                                         # 4. deterministic
            again = prob.run(handle, v)
            assert np.array_equal(flat.view(np.uint32), again.view(np.uint32)), f"variant {v}: not deterministic"
        guard = flat.view(np.uint32)[~prob.written]                                # 3. guard cells
        assert np.all(guard == SENTINEL), f"variant {v}: {int(np.sum(guard != SENTINEL))} writes outside C"
        res = prob.results(flat)
        assert np.all(np.isfinite(res)), f"variant {v}: non-finite output (padding read?)"
        over = np.abs(res - ref) / bound                                           # 1. bound
        assert np.all(over <= 1.0), f"variant {v}: error {over.max():.3g} x the bound"
        e, e_other = max_err(res, ref), max_err(res, ref_other)                    # 2. rounding mode
        assert 20 * e <= e_other, f"variant {v}: error {e:.3g} vs {e_other:.3g} against {OTHER_MODE}"
        got[v] = res
        report[v] = (float(over.max()), e_other / max(e, 1e-300))
    for i in VARIANTS:                                                             # 5. agreement
        for j in VARIANTS:
            if i < j:
                assert np.all(np.abs(got[i] - got[j]) <= 2 * bound), (i, j)
    auto = prob.run(handle, 0)
    v_auto = C.c_int32()
    _capi.check(_capi.load().keds_debug_linear_plan(prob.M, prob.N, prob.nz, torch.cuda.get_device_properties(0)
                                                    .multi_processor_count, C.byref(v_auto)))
    assert np.array_equal(prob.results(auto), got[v_auto.value]), "production choice differs from its variant"
    print(f"M={prob.M} N={prob.N} K={prob.K} nz={prob.nz}: " +
          "  ".join(f"v{v} err/bound {o:.2e} ratio {r:.0f}" for v, (o, r) in report.items()))
    return got, ref, bound, ref_other


# the consumer's products at the reference's widths (768 -> 512 -> 512 -> 768, inner 512); B(1+2k) rows
def real_products(B, k):
    M, Bk = B * (1 + 2 * k), B * k
    return [
        dict(M=M, N=512, K=768, nz=1, relu=True),                          # MLP hidden layer 0
        dict(M=M, N=512, K=512, nz=1, relu=True, bias=False),              # MLP hidden layer 1
        dict(M=M, N=768, K=512, nz=1),                                     # fc_out
        dict(M=Bk, N=3072, K=768, nz=2),                                   # K/V of three layers
        dict(M=B, N=512, K=768, nz=2),                                     # to_q
        dict(M=B, N=768, K=512, nz=2, ldc=3 * 768, c_off=[0, 768]),        # to_out -> tokens[:, 0 / 1, :]
        dict(M=B, N=512, K=768, nz=2, lda=3 * 768),                        # to_out dX from d tokens
        dict(M=512, N=768, K=M, nz=1),                                     # MLP dW (K = rows)
    ]


@pytest.mark.parametrize("B,k", [(128, 16), (37, 16)])
def test_every_variant_at_the_consumer_products(handle, B, k):
    for i, kw in enumerate(real_products(B, k)):
        check_all_variants(handle, Problem(seed=B + i, **kw))


@pytest.mark.parametrize("K", [37, 592, 1221, 4224])
def test_every_variant_at_weight_gradient_shapes(handle, K):
    """dW = dY^T X: K is the row count B(1+2k) (ragged), lda = round4(K)"""
    check_all_variants(handle, Problem(M=768, N=512, K=K, nz=2 if K < 1000 else 1, lda=round4(K), seed=K))


def test_every_variant_at_the_contrastive_loss_products(handle):
    check_all_variants(handle, Problem(M=1024, N=1024, K=2304, nz=2, seed=5))


@pytest.mark.parametrize("M", [1, 127, 128, 129])
@pytest.mark.parametrize("N", [4, 32, 36, 260])
@pytest.mark.parametrize("K", [4, 12, 36, 100])
def test_every_variant_at_edge_shapes(handle, M, N, K):
    """fewer k-blocks than splits, ragged K tails, ragged row / column tiles; ReLU and bias vary"""
    odd = (M + N + K) % 2 == 1
    ldc = N + 4 if odd else N
    check_all_variants(handle, Problem(M=M, N=N, K=K, nz=2, relu=odd, bias=not odd or M == 129, ldc=ldc,
                                       seed=M * 1000 + N * 10 + K))


def test_unaligned_output_takes_the_scalar_store_path(handle):
    """C 4-byte but not 16-byte aligned (and ldc not a multiple of 4): the epilogues' scalar stores"""
    check_all_variants(handle, Problem(M=129, N=260, K=100, nz=2, ldc=261, c_off=[1, 1 + 131 * 261], seed=3))


def test_the_checks_reject_a_subtly_wrong_product(handle):
    """The tolerance is not vacuous: references that model a kernel losing its last k-block, rounding
    the other way, swapping the two problems or shifting one row must all be rejected by 1. or 2."""
    for prob in (Problem(M=129, N=260, K=100, nz=2, seed=8), Problem(M=256, N=512, K=768, nz=2, seed=9)):
        res = prob.results(prob.run(handle, 1))
        ref, bound = prob.reference()
        ref_other, _ = prob.reference(OTHER_MODE)
        assert accepts(res, ref, bound, ref_other)
        dropped, _ = prob.reference(drop_last_kblock=True)
        assert not accepts(res, dropped, bound, ref_other), "last k-block dropped"
        assert not accepts(res, ref_other, bound, ref), "other rounding mode"
        assert not accepts(res, ref[::-1], bound, ref_other), "problems swapped"
        shifted = ref.copy()
        shifted[0, 5] = ref[0, 6]
        assert not accepts(res, shifted, bound, ref_other), "one row shifted"


def tie_patterns(rows, cols, seed):
    """fp32 values whose 13 low bits (the part tf32 drops) cover ties with even and odd kept parts,
    just-below / just-above ties, zero tails, and random tails; both signs; normal and subnormal"""
    rng = np.random.default_rng(seed)
    u = rng.integers(0, 2 ** 32, (rows, cols), dtype=np.uint64).astype(np.uint32)
    tails = np.array([0x1000, 0x1000, 0x0FFF, 0x1001, 0x0000, 0x1FFF], np.uint32)
    pick = rng.integers(0, len(tails) + 2, (rows, cols))
    tail = np.where(pick < len(tails), tails[np.minimum(pick, len(tails) - 1)], u & 0x1FFF)
    exp = rng.integers(100, 150, (rows, cols)).astype(np.uint32) << 23   # magnitudes 2^-27 .. 2^22
    sub = rng.random((rows, cols)) < 0.05
    exp[sub] = 0                                                          # subnormal
    sign = (rng.random((rows, cols)) < 0.5).astype(np.uint32) << 31
    bits = sign | exp | (u & 0x7FE000) | tail
    return bits.view(np.float32)


def test_the_tma_conversion_rounds_as_pinned(handle):
    """C = A I^T = round(A) and C = I W^T = round(W)^T, exactly (one non-zero term per sum): the
    product reads back the tf32 value each fp32 operand became, ties and subnormals included."""
    lib, h = handle
    K = 32
    for operand in ("A", "W"):
        prob = Problem(M=128, N=K, K=K, nz=1, bias=False, seed=1)
        vals = tie_patterns(128, K, seed=2 if operand == "A" else 3)
        if operand == "A":
            prob.A[0, :, :K], prob.W[0, :, :K] = vals, np.eye(K, dtype=np.float32)
        else:
            prob = Problem(M=K, N=128, K=K, nz=1, bias=False, seed=1)
            prob.A[0, :, :K], prob.W[0, :, :K] = np.eye(K, dtype=np.float32), vals
        prob.dA = [torch.from_numpy(prob.A[0]).cuda()]
        prob.dW = [torch.from_numpy(prob.W[0]).cuda()]
        for v in VARIANTS:
            got = prob.results(prob.run(handle, v))[0]
            want = vals if operand == "A" else vals.T
            match = {m: float(np.mean(got == round_tf32(want, m))) for m in ("rne", "rz")}
            sub = np.abs(want) < np.finfo(np.float32).tiny
            detail = f"operand {operand}, variant {v}: fraction matching each mode {match}; " \
                     f"subnormals -> {np.unique(got[sub])[:4]} (of {int(sub.sum())})"
            assert np.array_equal(got, round_tf32(want, TF32_ROUNDING)), detail
