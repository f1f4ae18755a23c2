"""The 3x3 reflect convolution on 16-pixel-wide frames (``conv3x3_reflect_w16<tcgen05>``, csrc/c2s_conv.cu): the 64 and
128-channel layers of U-TAE's last down block, ``DownConvBlock(64, 128, 4, 2, 1)`` on 32 x 32 -> 16 x 16 frames.

CPU: the support predicate and the workspace size of the C ABI over the served shapes and their near misses.
GPU (``-m gpu``): the kernel against a plain fp32 torch convolution of the same bf16 operands with its GroupNorm sums,
the input normalisation on the fly, and the blocks -- down3 alone and U-TAE's four-block encoder -- with the library
convolution made to raise, against an fp32 torch stack built from the same ``state_dict``.
"""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import crop2seg_b200 as c2s
from crop2seg_b200 import _lib
from crop2seg_b200 import conv as c2s_conv
from crop2seg_b200.build import build_library

KERNEL = "conv3x3_reflect_w16<tcgen05>"


def _desc(c_in, c_out, h, w, dtype=_lib.BF16, frames=8):
    return _lib.ConvDesc(frames=frames, c_in=c_in, c_out=c_out, H=h, W=w, kernel=3, stride=1, padding=1, dtype=dtype)


@pytest.fixture(scope="module")
def lib():
    build_library()
    return _lib.load()


@pytest.mark.parametrize("c_in", [64, 128])
@pytest.mark.parametrize("c_out", [64, 128])
@pytest.mark.parametrize("h", [2, 3, 7, 16])
def test_sixteen_pixel_frames_are_served(lib, c_in, c_out, h):
    d = _desc(c_in, c_out, h, 16)
    assert lib.c2s_conv2d_supported(ctypes.byref(d)) == 1
    assert lib.c2s_conv2d_workspace_bytes(ctypes.byref(d)) == c_out * 9 * c_in * 2  # prepared bf16 weights


@pytest.mark.parametrize("c_in,c_out,h,w,dtype", [
    (64, 128, 17, 16, _lib.BF16),   # H > 16: more than one frame buffer per K chunk
    (128, 128, 32, 16, _lib.BF16),
    (64, 128, 1, 16, _lib.BF16),    # no reflect padding of one row
    (96, 128, 16, 16, _lib.BF16),
    (128, 96, 16, 16, _lib.BF16),
    (64, 256, 16, 16, _lib.BF16),
    (10, 128, 16, 16, _lib.BF16),   # c_in <= 16 at W = 16
    (128, 128, 16, 16, _lib.F32),
    (128, 128, 8, 8, _lib.BF16),    # W = 8
    (128, 64, 32, 32, _lib.BF16),   # 128 input channels at W = 32
    (64, 128, 32, 32, _lib.BF16),   # 128 output channels at W = 32
])
def test_near_misses_stay_unsupported(lib, c_in, c_out, h, w, dtype):
    d = _desc(c_in, c_out, h, w, dtype)
    assert lib.c2s_conv2d_supported(ctypes.byref(d)) == 0
    assert lib.c2s_conv2d_workspace_bytes(ctypes.byref(d)) == 0


def test_no_frames_is_unsupported(lib):
    assert lib.c2s_conv2d_supported(ctypes.byref(_desc(128, 128, 16, 16, frames=0))) == 0


def test_unsupported_forward_names_the_served_shapes(lib):
    d = _desc(128, 256, 16, 16)
    dummy = ctypes.c_void_p(256)
    assert lib.c2s_conv2d_forward(ctypes.byref(d), dummy, None, dummy, None, dummy, None, dummy, 1 << 20, None) == 2
    assert b"W = 16, H <= 16, c_in and c_out 64 or 128" in lib.c2s_last_error()


# ------------------------------------------------------------------------------------------------ GPU
def _rel(a, b):
    return (a.float() - b.float()).abs().max().item() / max(b.float().abs().max().item(), 1e-30)


def _torch_conv(x, w, b):
    xp = F.pad(x.float(), (1, 1, 1, 1), mode="reflect")
    return F.conv2d(xp, w.to(torch.bfloat16).float(), b)


# every (c_in, c_out) at every H; the frame counts rotate so that each pair sees one CTA with a single frame, several
# frames per persistent CTA and more frames than SMs
CASES = []
for i, (ci, co) in enumerate([(64, 128), (128, 128), (64, 64), (128, 64)]):
    for k, h in enumerate([2, 3, 7, 16]):
        CASES.append((ci, co, h, [1, 3, 150, 1600][(i + k) % 4], (i + k) % 2 == 0, (i + k) % 4 != 1))
CASES += [(128, 128, 16, 1600, True, True), (64, 128, 16, 1, False, False), (128, 128, 16, 150, False, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("c_in,c_out,h,frames,with_bias,with_stats", CASES)
def test_w16_convolution_matches_torch(c_in, c_out, h, frames, with_bias, with_stats):
    g = torch.Generator(device="cuda").manual_seed(frames * 131 + c_in + 7 * c_out + h)
    x = torch.randn((frames, c_in, h, 16), device="cuda", generator=g).to(torch.bfloat16)
    w = torch.randn((c_out, c_in, 3, 3), device="cuda", generator=g) * (1.0 / (3.0 * c_in ** 0.5))
    b = torch.randn(c_out, device="cuda", generator=g) * 0.1 if with_bias else None
    conv = torch.nn.Conv2d(c_in, c_out, 3, padding=1, padding_mode="reflect")
    assert c2s_conv.conv2d_supported(x, conv)
    y, stats = c2s_conv.conv2d_reflect_forward(x, w, b, with_stats=with_stats)
    torch.cuda.synchronize()
    assert _lib.load().c2s_last_kernel().decode() == KERNEL
    ref = _torch_conv(x, w, b)
    assert y.shape == ref.shape and y.dtype == torch.bfloat16
    err = _rel(y, ref)
    assert err < 6e-3, err  # bf16 rounding of the stored output; the products are exact, the sums fp32
    if not with_stats:
        assert stats is None
        return
    q = ref.view(frames, 4, -1)  # per frame and quarter of the output channels
    s1, s2 = q.sum(-1), (q * q).sum(-1)
    assert torch.allclose(stats[..., 0], s1, rtol=2e-3, atol=2e-3 * s1.abs().max().item())
    assert torch.allclose(stats[..., 1], s2, rtol=2e-3)


def _set_norms(blk, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    with torch.no_grad():
        for m in blk.modules():
            if isinstance(m, torch.nn.GroupNorm):
                m.weight.copy_(1 + 0.3 * torch.randn(m.num_channels, device="cuda", generator=g))
                m.bias.copy_(0.2 * torch.randn(m.num_channels, device="cuda", generator=g))
    return blk


@pytest.mark.gpu
@pytest.mark.parametrize("frames", [3, 400])
def test_input_normalisation_on_the_fly_equals_the_separate_pass(frames):
    """ConvBlock([64, 128, 128]) on 16 x 16 frames: its second stage normalises the raw 128-channel output of the first
    inside the producers; with the same statistics tensor that gives the same bits as c2s_group_norm_relu first."""
    blk = _set_norms(c2s.ConvBlock([64, 128, 128], pad_value=0, norm="group").cuda().eval(), 9)
    g = torch.Generator(device="cuda").manual_seed(frames)
    x = torch.randn((frames, 64, 16, 16), device="cuda", generator=g).to(torch.bfloat16)
    seq = blk.conv.conv
    with torch.no_grad():
        fused = blk(x)
        raw1, st1 = c2s_conv.conv2d_reflect_forward(x, seq[0].weight, seq[0].bias)
        a1 = c2s_conv.group_norm_relu(raw1, st1, seq[1], relu=True)
        raw2, st2 = c2s_conv.conv2d_reflect_forward(a1, seq[3].weight, seq[3].bias)
        ref = c2s_conv.group_norm_relu(raw2, st2, seq[4], relu=True)
        raw2f, _ = c2s_conv.conv2d_reflect_forward(raw1, seq[3].weight, seq[3].bias, in_norm=(st1, seq[1], True))
    torch.cuda.synchronize()
    assert _lib.load().c2s_last_kernel().decode() == KERNEL
    assert torch.equal(raw2f, raw2)
    # the GroupNorm sums are accumulated with float atomics (order-dependent last bits): compare within bf16 rounding
    assert _rel(fused, ref) < 8e-3


# ------------------------------------------------------------------------------------------------ blocks, no library conv
def _ref_layer(layer, x, residual=None):
    """fp32 nn.Conv2d(reflect) -> GroupNorm -> ReLU per stage of a ConvLayer, from its own parameters."""
    seq = layer.conv
    for ci, ni, relu in layer._plan:
        conv, norm = seq[ci], seq[ni]
        ref = torch.nn.Conv2d(conv.in_channels, conv.out_channels, conv.kernel_size, stride=conv.stride,
                              padding=conv.padding, padding_mode="reflect").cuda()
        ref.load_state_dict(conv.state_dict())
        x = F.group_norm(ref(x), norm.num_groups, norm.weight, norm.bias, norm.eps)
        if relu:
            x = torch.relu(x)
    return x if residual is None else x + residual


def _ref_block(blk, x):
    if isinstance(blk, c2s.DownConvBlock):
        out = _ref_layer(blk.conv1, _ref_layer(blk.down, x))
        return _ref_layer(blk.conv2, out, residual=out)
    return _ref_layer(blk.conv, x)


def _library_layer(layer, x, residual=None):
    """The route ConvLayer took for the 128-channel layers before they had a kernel: F.pad + F.conv2d (bf16) +
    c2s_group_stats, then c2s_group_norm_relu."""
    (ci, ni, relu), = layer._plan
    conv, norm = layer.conv[ci], layer.conv[ni]
    xp = F.pad(x, (1, 1, 1, 1), mode="reflect")
    raw = F.conv2d(xp, conv.weight.to(torch.bfloat16), conv.bias.to(torch.bfloat16))
    return c2s_conv.group_norm_relu(raw, c2s_conv.group_stats(raw, norm.num_groups), norm, relu=relu, residual=residual)


def _encoder():
    return [_set_norms(b.cuda().eval(), 40 + i) for i, b in enumerate([
        c2s.ConvBlock([10, 64, 64], pad_value=0, norm="group"),
        c2s.DownConvBlock(64, 64, 4, 2, 1, pad_value=0, norm="group"),
        c2s.DownConvBlock(64, 64, 4, 2, 1, pad_value=0, norm="group"),
        c2s.DownConvBlock(64, 128, 4, 2, 1, pad_value=0, norm="group")])]


def _no_library_conv(monkeypatch):
    def refuse(*args, **kwargs):
        raise AssertionError("library convolution called")
    monkeypatch.setattr(c2s_conv.F, "conv2d", refuse)


@pytest.mark.gpu
def test_down3_runs_without_a_library_convolution(monkeypatch):
    blk = _encoder()[3]
    g = torch.Generator(device="cuda").manual_seed(3)
    x = torch.relu(torch.randn((2, 5, 64, 32, 32), device="cuda", generator=g)).to(torch.bfloat16)
    x[0, 3] = 0
    x[1, 0] = 0
    pad = torch.zeros((2, 5), dtype=torch.bool, device="cuda")
    pad[0, 3] = pad[1, 0] = True
    flat = x.view(10, 64, 32, 32)
    with torch.no_grad():
        ref = _ref_block(blk, flat.float())
        down = blk.down(flat)
        out1 = _library_layer(blk.conv1, down)
        lib_route = _library_layer(blk.conv2, out1, residual=out1)
        with monkeypatch.context() as m:
            _no_library_conv(m)
            out = blk(flat)
            sm = blk.smart_forward(x)
    assert out.shape == (10, 128, 16, 16) and out.dtype == torch.bfloat16
    valid = ~pad.view(-1)
    assert _rel(out[valid], ref[valid]) < 2e-2
    assert _rel(out, lib_route) < 1e-2  # the library's summation order against the kernel's: bf16 rounding
    assert sm.shape == (2, 5, 128, 16, 16)
    assert torch.all(sm[0, 3] == 0) and torch.all(sm[1, 0] == 0)  # padded frames come back exactly pad_value
    assert _rel(sm.view(10, 128, 16, 16)[valid], ref[valid]) < 2e-2


@pytest.mark.gpu
def test_utae_encoder_runs_without_a_library_convolution(monkeypatch):
    blocks = _encoder()
    g = torch.Generator(device="cuda").manual_seed(4)
    x = torch.randn((1, 4, 10, 128, 128), device="cuda", generator=g).to(torch.bfloat16)
    x[0, 2] = 0
    refs, feats = [], []
    with torch.no_grad():
        r = x.view(4, 10, 128, 128).float()
        for blk in blocks:
            r = _ref_block(blk, r)
            refs.append(r)
        with monkeypatch.context() as m:
            _no_library_conv(m)
            f = x
            for blk in blocks:
                f = blk.smart_forward(f)
                feats.append(f)
    valid = torch.tensor([True, True, False, True], device="cuda")
    for got, ref in zip(feats, refs):
        got = got.view(4, *got.shape[2:])
        assert torch.all(got[2] == 0)
        assert _rel(got[valid], ref[valid]) < 2e-2
    assert feats[-1].shape == (1, 4, 128, 16, 16)
