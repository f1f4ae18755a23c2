"""CPU-side checks of the fused skip-convolution backward's C ABI: exported, bound, workspace size, argument errors."""
import ctypes

import pytest

from crop2seg_b200 import _lib
from crop2seg_b200.build import LIB_PATH, build_library


@pytest.fixture(scope="module")
def lib():
    build_library()
    return _lib.load()


def test_symbols_are_exported_and_bound(lib):
    raw = ctypes.CDLL(LIB_PATH)
    for sym in ("c2s_agg_skipconv_backward_workspace_bytes", "c2s_agg_skipconv_backward"):
        assert hasattr(raw, sym) and sym in _lib.EXPORTS
    assert ctypes.sizeof(_lib.SkipConvBwdIo) == 6 * ctypes.sizeof(ctypes.c_void_p)


def test_workspace_size(lib):
    fixed = 2 * 2 * 4 * 4 * 32 * 16 + 3 * 64 * 4  # W and (alpha W)^T fragments (bf16 hi + lo), three [64] vectors
    per_cta = (64 * 64 + 2 * 64) * 4               # g_y s^T, sum g_y, sum g_y (z - mean) of one 128-pixel tile
    for b, hw in ((16, 128), (16, 64), (16, 32), (3, 16)):
        d = _lib.AggDesc(B=b, T=61, C=64, H=hw, W=hw, n_heads=16, ha=16, wa=16, mode=_lib.AGG_ATT_GROUP, dtype=_lib.BF16)
        assert lib.c2s_agg_skipconv_backward_workspace_bytes(ctypes.byref(d)) == fixed + b * (hw * hw // 128) * per_cta
    assert lib.c2s_agg_skipconv_backward_workspace_bytes(None) == 0


def test_bad_arguments_return_status_codes(lib):
    io = _lib.SkipConvBwdIo()
    assert lib.c2s_agg_skipconv_backward(None, None, None, None, None, None, None, ctypes.byref(io), None, 0, None) == 1
    assert b"desc/params/io is NULL" in lib.c2s_last_error()
    d = _lib.AggDesc(B=1, T=3, C=64, H=16, W=16, n_heads=8, ha=8, wa=8, mode=_lib.AGG_ATT_GROUP, dtype=_lib.BF16)
    p = _lib.SkipConvParams(conv_weight=16, bn_running_mean=16, bn_running_var=16, bn_eps=1e-5)
    dummy = ctypes.c_void_p(16)
    status = lib.c2s_agg_skipconv_backward(ctypes.byref(d), dummy, dummy, None, ctypes.byref(p), dummy, dummy,
                                           ctypes.byref(io), dummy, 1 << 20, None)
    assert status == 1 and b"fused backward serves" in lib.c2s_last_error()  # 8 heads: checked before any device call
