"""CPU checks of the WKV7 chunk-cache entry points: the size helper, and argument validation that fails before
touching a GPU."""
import ctypes

import pytest

BOUNDED, CK64, TF32 = 1, 2, 4


@pytest.fixture(scope="module")
def lib():
    from visualrwkv_b200 import _build, _lib
    _build.build_all()
    L = _lib.lib()
    L.vrwkv_wkv7_cache_bytes.restype = ctypes.c_size_t
    L.vrwkv_last_error.restype = ctypes.c_char_p
    return L


def test_cache_bytes(lib):
    # 8 tiles of 64 x 64 bf16 per 64-step chunk of each (batch, head)
    assert lib.vrwkv_wkv7_cache_bytes(1, 64, 1) == 64 * 1024
    assert lib.vrwkv_wkv7_cache_bytes(8, 2048, 12) == 8 * 12 * 32 * 64 * 1024   # cfg2: 201 MB per layer
    assert lib.vrwkv_wkv7_cache_bytes(2, 96, 3) == 0
    assert lib.vrwkv_wkv7_cache_bytes(0, 64, 1) == 0
    from visualrwkv_b200 import wkv7 as W
    assert W.cache_bytes(3, 256, 5) == 3 * 5 * 4 * 64 * 1024


def _fwd(lib, T, cache, flags, s=0x2000):
    p = ctypes.c_void_p(0x1000)
    return lib.vrwkv_wkv7_forward_cache(1, T, 1, *[p] * 7, ctypes.c_void_p(s), p, ctypes.c_void_p(cache),
                                        ctypes.c_uint(flags), ctypes.c_void_p(0))


def _bwd(lib, T, cache, flags):
    p = ctypes.c_void_p(0x1000)
    return lib.vrwkv_wkv7_backward_cache(1, T, 1, *[p] * 9, ctypes.c_void_p(cache), *[p] * 6, ctypes.c_uint(flags),
                                         ctypes.c_void_p(0))


@pytest.mark.parametrize("call", [_fwd, _bwd], ids=["forward", "backward"])
def test_cache_calls_validate_arguments(lib, call):
    ok = BOUNDED | CK64
    assert call(lib, 96, 0x4000, ok) == -1
    assert b"multiple of 64" in lib.vrwkv_last_error()
    for flags in (BOUNDED, CK64, ok | TF32, 0):
        assert call(lib, 64, 0x4000, flags) == -1
        assert b"BOUNDED_DECAY | CHUNK_CHECKPOINTS" in lib.vrwkv_last_error()
    assert call(lib, 64, 0, ok) == -1
    assert b"required" in lib.vrwkv_last_error()
    assert call(lib, 64, 0x4040, ok) == -1
    assert b"128-byte aligned" in lib.vrwkv_last_error()


def test_forward_cache_needs_checkpoints(lib):
    assert _fwd(lib, 64, 0x4000, BOUNDED | CK64, s=0) == -1
    assert b"required" in lib.vrwkv_last_error()
