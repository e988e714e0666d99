"""CPU: the host side of the neighbour consumer on row-sharded bases. The two sharded forward entry
points are declared, exported and in the ctypes table; without a GPU they refuse NULL arguments;
the Python layer refuses a mixed index pair; and an sm_100a compile keeps both instantiations of the
row-assembly kernel (local and shard row sources) and the step's shard consumer free of spills."""
import re
import subprocess

import pytest

from keds_b200 import _capi

NAMES = ("keds_consumer_forward_sharded", "keds_consumer_forward_train_sharded")


def test_sharded_consumer_symbols_are_declared_exported_and_typed():
    import os

    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include",
                            "keds_knn.h")).read()
    lib = _capi.load()
    for name in NAMES:
        assert re.search(r"\b" + name + r"\s*\(", hdr), name
        assert name in _capi.SIGNATURES and hasattr(lib, name)
    # (c, img, txt, ex, feat, I_img, I_txt, perm, B, k, [masks,] tokens, stream)
    assert len(_capi.SIGNATURES[NAMES[0]][1]) == 12
    assert len(_capi.SIGNATURES[NAMES[1]][1]) == 13


def test_sharded_consumer_entry_points_refuse_null_arguments_without_a_gpu():
    lib = _capi.load()
    assert lib.keds_consumer_forward_sharded(None, None, None, None, None, None, None, None, 4, 16, None,
                                             None) == -1
    assert lib.keds_consumer_forward_train_sharded(None, None, None, None, None, None, None, None, 4, 16, None,
                                                   None, None) == -1
    assert "NULL" in _capi.last_error()


def test_mixed_index_pair_is_a_type_error():
    from keds_b200.sharded import _sharded_kb
    from keds_b200.sharded import ShardedIndex

    local = object()
    assert _sharded_kb(local, local) is None
    sh = ShardedIndex.__new__(ShardedIndex)  # (no process group needed to tell the types apart)
    sh._kb = None
    with pytest.raises(TypeError):
        _sharded_kb(sh, local)
    with pytest.raises(TypeError):
        _sharded_kb(local, sh)
    with pytest.raises(TypeError):  # a ShardedIndex outside a ShardedKnowledgeBase
        _sharded_kb(sh, sh)


def test_consumer_rows_and_shard_consume_do_not_spill(tmp_path):
    from keds_b200 import build as kbuild

    nvcc = kbuild.find_nvcc()
    if nvcc is None:
        pytest.skip("nvcc not available")
    res = subprocess.run([nvcc, *kbuild.NVCC_FLAGS, "-Xptxas", "-v", "-o", str(tmp_path / "lib.so"), kbuild.SRC],
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-2000:]
    stats, cur = {}, None
    for line in res.stderr.splitlines():
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            cur = m.group(1)
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur and any(s in cur for s in ("k_consumer_rowsINS_17ConsumerLocalRows",
                                                "k_consumer_rowsINS_17ConsumerShardRows", "k_shard_consume")):
            stats[cur] = (int(m.group(1)), int(m.group(2)))
    assert len(stats) == 3, stats
    assert all(v == (0, 0) for v in stats.values()), stats
