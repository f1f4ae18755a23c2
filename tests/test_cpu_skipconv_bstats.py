"""CPU-side checks of the batch-statistics skip convolution: its C ABI (exported, bound, workspace sizes, argument errors
before any device call) and the float64 reference the GPU tests compare against (vs nn.BatchNorm2d in training mode)."""
import ctypes

import numpy as np
import pytest
import torch
from torch import nn

from crop2seg_b200 import _lib
from crop2seg_b200.build import LIB_PATH, build_library
from skipconv_bstats_ref import running_update, skip_conv_bstats

SYMBOLS = ("c2s_agg_skipconv_bstats_workspace_bytes", "c2s_agg_skipconv_bstats_forward",
           "c2s_agg_skipconv_bstats_backward_workspace_bytes", "c2s_agg_skipconv_bstats_backward")


@pytest.fixture(scope="module")
def lib():
    build_library()
    return _lib.load()


def _desc(b, hw, heads=16, a=16):
    return _lib.AggDesc(B=b, T=61, C=64, H=hw, W=hw, n_heads=heads, ha=a, wa=a, mode=_lib.AGG_ATT_GROUP, dtype=_lib.BF16)


def test_symbols_are_exported_and_bound(lib):
    raw = ctypes.CDLL(LIB_PATH)
    for sym in SYMBOLS:
        assert hasattr(raw, sym) and sym in _lib.EXPORTS
        assert getattr(lib, sym).restype is not None


def test_workspace_sizes(lib):
    frags = 2 * 4 * 4 * 32 * 16  # W as bf16 hi + lo mma fragments
    for b, hw in ((16, 128), (16, 64), (16, 32), (3, 16), (64, 128)):
        ctas = b * (hw * hw // 128)
        # W fragments, scale, shift; per CTA the mean and M2 of 64 channels
        assert lib.c2s_agg_skipconv_bstats_workspace_bytes(ctypes.byref(_desc(b, hw))) == frags + 2 * 64 * 4 + ctas * 2 * 64 * 4
        # the frozen backward's fixed part, two [64] means, per CTA the weight partial (as the frozen backward) + 2 x 64 sums
        fixed = 2 * frags + 3 * 64 * 4 + 2 * 64 * 4
        assert lib.c2s_agg_skipconv_bstats_backward_workspace_bytes(ctypes.byref(_desc(b, hw))) == \
            fixed + ctas * ((64 * 64 + 2 * 64) + 2 * 64) * 4
    assert lib.c2s_agg_skipconv_bstats_workspace_bytes(None) == 0
    assert lib.c2s_agg_skipconv_bstats_backward_workspace_bytes(None) == 0


def test_bad_arguments_return_status_codes(lib):
    io = _lib.SkipConvBwdIo()
    dummy = ctypes.c_void_p(16)
    assert lib.c2s_agg_skipconv_bstats_forward(None, dummy, dummy, None, None, dummy, dummy, dummy, dummy, dummy, 0,
                                               None) == 1
    assert b"desc/params is NULL" in lib.c2s_last_error()
    p = _lib.SkipConvParams(conv_weight=16, bn_eps=1e-5)  # no running statistics: not needed with batch statistics
    d = _desc(1, 16, heads=8, a=8)
    assert lib.c2s_agg_skipconv_bstats_forward(ctypes.byref(d), dummy, dummy, None, ctypes.byref(p), None, dummy, dummy,
                                               dummy, dummy, 1 << 20, None) == 1
    assert b"is NULL" in lib.c2s_last_error()  # z missing
    status = lib.c2s_agg_skipconv_bstats_forward(ctypes.byref(d), dummy, dummy, None, ctypes.byref(p), dummy, dummy,
                                                 dummy, dummy, dummy, 1 << 20, None)
    assert status == 2 and b"fused path serves" in lib.c2s_last_error()  # 8 heads: C2S_ERR_UNSUPPORTED, no device call
    assert lib.c2s_agg_skipconv_bstats_backward(None, None, None, None, None, None, None, None, None, None,
                                                ctypes.byref(io), None, 0, None) == 1
    assert b"desc/params/io is NULL" in lib.c2s_last_error()
    status = lib.c2s_agg_skipconv_bstats_backward(ctypes.byref(d), dummy, dummy, None, ctypes.byref(p), dummy, dummy,
                                                  dummy, dummy, dummy, ctypes.byref(io), dummy, 1 << 20, None)
    assert status == 1 and b"fused backward serves" in lib.c2s_last_error()


@pytest.mark.parametrize("affine,bias,momentum", [(True, True, 0.1), (False, False, None), (True, False, 0.3)])
def test_reference_matches_batchnorm2d_in_training_mode(affine, bias, momentum):
    torch.manual_seed(0)
    conv = nn.Conv2d(64, 64, 1, bias=bias).double()
    bn = nn.BatchNorm2d(64, affine=affine, momentum=momentum).double().train()
    if affine:
        with torch.no_grad():
            bn.weight.uniform_(0.5, 1.5), bn.bias.uniform_(-0.3, 0.3)
    rm, rv, nbt = torch.zeros(64, dtype=torch.float64), torch.ones(64, dtype=torch.float64), 0
    for step in range(3):
        s = torch.randn(3, 64, 8, 16, dtype=torch.float64) + step
        s.requires_grad_(True)
        want = torch.relu(bn(conv(s)))
        got = skip_conv_bstats(s, conv.weight, conv.bias, bn.weight, bn.bias, bn.eps)
        assert torch.allclose(got["out"], want, rtol=1e-12, atol=1e-12)
        z = conv(s).detach()
        assert torch.allclose(got["mean"], z.mean(dim=(0, 2, 3)), rtol=1e-12, atol=1e-12)
        assert torch.allclose(got["var"], z.var(dim=(0, 2, 3), unbiased=False), rtol=1e-12, atol=1e-12)
        g = torch.randn_like(want)
        ref = torch.autograd.grad(want, [s] + list(conv.parameters()), g)
        mine = torch.autograd.grad(got["out"], [s] + list(conv.parameters()), g)
        for a, b in zip(mine, ref):
            assert torch.allclose(a, b, rtol=1e-10, atol=1e-12)
        if bias:  # batch statistics cancel the conv bias: its gradient is at rounding level
            assert float(mine[-1].abs().max()) < 1e-12 * float(g.abs().sum())
        nbt = running_update(rm, rv, nbt, got["mean"].detach(), got["var"].detach(), 3 * 8 * 16, momentum)
    assert nbt == int(bn.num_batches_tracked)
    assert torch.allclose(rm, bn.running_mean, rtol=1e-12, atol=1e-14)
    assert torch.allclose(rv, bn.running_var, rtol=1e-12, atol=1e-14)
