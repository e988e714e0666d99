"""CPU: libkeds_knn.so loads and exports every function include/keds_knn.h declares; the ctypes
table mirrors the header; without a GPU every compute entry point refuses (no CPU fallback)."""
import ctypes as C
import os
import re

import pytest

from keds_b200 import _capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    src = open(os.path.join(ROOT, "include", "keds_knn.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(keds_[a-z0-9_]+)\s*\(", src)))


def test_header_declares_the_expected_surface():
    fns = header_functions()
    for must in ["keds_index_create", "keds_index_add", "keds_index_search", "keds_index_search2",
                 "keds_gather_pool", "keds_topk_merge", "keds_gallery_rank", "keds_last_error"]:
        assert must in fns


def test_library_exports_every_declared_symbol():
    lib = _capi.load()
    for name in header_functions():
        assert hasattr(lib, name), f"{name} declared in keds_knn.h but not exported"


def test_ctypes_table_matches_header():
    assert sorted(_capi.SIGNATURES) == header_functions()


def test_version_and_error_strings():
    lib = _capi.load()
    assert b"sm_100a" in lib.keds_version()
    assert isinstance(_capi.last_error(), str)


def test_no_gpu_means_error_not_fallback():
    lib = _capi.load()
    if lib.keds_device_count() > 0:
        pytest.skip("a GPU is present")
    h = C.c_void_p()
    rc = lib.keds_index_create(768, 0, 0, C.byref(h))
    assert rc == -3 and not h.value
    assert "no CPU fallback" in _capi.last_error()
    from keds_b200.index import GpuIndexFlat
    with pytest.raises(RuntimeError):
        GpuIndexFlat(768)


def test_bad_arguments_are_rejected_without_a_gpu():
    lib = _capi.load()
    h = C.c_void_p()
    assert lib.keds_index_create(0, 0, 0, C.byref(h)) == -1
    assert lib.keds_index_create(768, 7, 0, C.byref(h)) == -1
    assert lib.keds_index_ntotal(None) == -1
    assert lib.keds_index_search(None, None, 1, 1, None, None, None) == -1
    assert lib.keds_gather_pool(None, 0, None, None, None, 1, 1, 1, 1, None, None) == -1
    assert lib.keds_consumer_debug_attend(None, 0, 0, 1, 16, None, None, None, None, 64, 0, 32, None, None, None, None,
                                          None, None, None) == -1


def test_library_is_sm100a_tcgen05_code():
    import shutil
    import subprocess
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([cuobjdump, "-sass", _capi.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in sass
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM"):
        assert mnemonic in sass, f"{mnemonic} missing: the scoring kernel is not on tcgen05/TMA"
