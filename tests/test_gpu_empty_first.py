"""GPU (-m gpu): a two-database search whose first database is empty. The first result is padding
only, the second equals a single search on the second database, and the call reports that
database's flagged queries under its own slot, on the call's (first) handle."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from keds_b200.index import METRIC_INNER_PRODUCT, GpuIndexFlat, search2  # noqa: E402

NQ = 16384 + 300  # two passes


def unit(n, d, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, d, generator=g)
    return (x / x.norm(dim=1, keepdim=True)).numpy()


@pytest.fixture(scope="module")
def data():
    base = unit(20000, 256, 5)
    rows = np.random.default_rng(6).integers(0, base.shape[0], NQ)
    q = (base[rows] + 0.05 * unit(NQ, 256, 7)).astype(np.float32)
    ex = np.stack([rows, np.full(NQ, -1)], 1).astype(np.int64)
    return base, q, ex


def host(x):
    return x.cpu().numpy() if isinstance(x, torch.Tensor) else x


@pytest.mark.parametrize("eps_scale", [1.0, 1e4])
@pytest.mark.parametrize("exclude", [False, True])
@pytest.mark.parametrize("device_io", [False, True])
def test_empty_first_index(data, device_io, exclude, eps_scale):
    base, q, ex = data
    empty = GpuIndexFlat(base.shape[1], METRIC_INNER_PRODUCT, 0)
    full = GpuIndexFlat(base.shape[1], METRIC_INNER_PRODUCT, 0)
    full.add(base)
    for ix in (empty, full):
        ix.set_eps_scale(eps_scale)  # 1e4: the certificate passes no query, every one is flagged
    qa = torch.from_numpy(q).cuda() if device_io else q
    exa = None if not exclude else torch.from_numpy(ex).cuda() if device_io else ex
    (Da, Ia), (Db, Ib) = search2(empty, full, qa, 16, exclude=exa)
    if device_io:
        empty.sync()
    st = empty.last_stats()
    D1, I1 = full.search(qa, 16, exclude=exa)
    Da, Ia, Db, Ib, D1, I1 = map(host, (Da, Ia, Db, Ib, D1, I1))
    assert (Ia == -1).all() and (Da == -np.finfo(np.float32).max).all()
    np.testing.assert_array_equal(Ib, I1)
    np.testing.assert_array_equal(Db.view(np.uint32), D1.view(np.uint32))
    if exclude:
        assert not (Ib == ex[:, :1]).any()
    assert st["err_word"] == 0
    assert st["n_flagged"][0] == 0
    if eps_scale > 1:
        assert st["n_flagged"][1] == NQ
