"""Shared convolutional encoder over the (batch x time) frames (SURVEY.md section 8f, rank 4) -- inference.

Drop-ins for ``src.backbones.conv.ConvLayer`` (conv.py:29-96), ``ConvBlock`` (conv.py:164-200) and ``DownConvBlock``
(conv.py:238-296) in the configuration U-TAE / W-TAE / Time-Unet build their encoders with (``conv_type='2d'``,
``norm='group'``, ``padding_mode='reflect'``, no squeeze-and-excitation; utae.py:128-160): same constructor arguments,
same sub-module tree and therefore byte-compatible ``state_dict`` keys (``conv.conv.0.weight`` ...).

What runs where (``forward`` / ``smart_forward``, eval mode, CUDA tensors):

* frames: ``smart_forward`` packs the valid frames with the device-side frame index (no ``nonzero`` sync, no dummy
  forward; ``staging.py``), runs the block in bf16 on the packed frames and scatters the result back;
* convolution: every layer of U-TAE's spatial encoder runs as a hand-written tcgen05 implicit GEMM
  (``c2s_conv2d_forward``, ``csrc/c2s_conv.cu``): the 3x3 / stride 1 layers with 64 input (or <= 16, the model input) and
  64 output channels on rows of 128, 64 or 32 pixels, the strided 4x4 layer of ``DownConvBlock`` from rows of 128, 64 or
  32 pixels, and the 3x3 layers with 64 or 128 channels in and out on whole frames 16 pixels wide (the last block).
  A layer outside what the kernels serve (another encoder configuration: other widths or resolutions) takes the library
  branch of ``ConvLayer.forward``: ``torch.nn.functional.conv2d`` on a reflect-padded bf16 tensor -- a plain cuDNN
  convolution, NOT part of the hand-written path -- followed by ``c2s_group_stats``;
* GroupNorm + ReLU (+ the residual of ``DownConvBlock``): ``c2s_group_norm_relu``, one element-wise pass, fp32 statistics;
  between two tensor-core stages of one ``ConvLayer`` the pass is skipped: the next convolution normalises its input on
  the fly while it stages it (``c2s_conv_input_norm``).

Training mode, other norms and the experimental conv types raise ``NotImplementedError``: the reference classes remain
the training path.
"""
from __future__ import annotations

import ctypes
from typing import List, Optional

import torch
from torch import nn
import torch.nn.functional as F

from . import _lib
from .ops import _ptr, _require_cuda, _stream


def _code(dtype: torch.dtype) -> int:
    if dtype == torch.bfloat16:
        return _lib.BF16
    if dtype == torch.float32:
        return _lib.F32
    raise RuntimeError(f"crop2seg_b200: unsupported dtype {dtype}")


# ------------------------------------------------------------------------------------------------ tensor-level calls
def conv2d_supported(x: torch.Tensor, conv: nn.Conv2d) -> bool:
    """True when ``c2s_conv2d_forward`` (tcgen05 implicit GEMM) serves ``conv`` on ``x`` [frames, C, H, W]."""
    if not (x.is_cuda and x.dtype == torch.bfloat16 and conv.padding_mode == "reflect" and conv.groups == 1):
        return False
    if conv.dilation != (1, 1) or conv.kernel_size[0] != conv.kernel_size[1] or conv.stride[0] != conv.stride[1]:
        return False
    d = _lib.ConvDesc(frames=x.shape[0], c_in=conv.in_channels, c_out=conv.out_channels, H=x.shape[2], W=x.shape[3],
                      kernel=conv.kernel_size[0], stride=conv.stride[0], padding=conv.padding[0], dtype=_code(x.dtype))
    return bool(_lib.load().c2s_conv2d_supported(ctypes.byref(d)))


def conv2d_reflect_forward(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor], *, kernel: int = 3,
                           stride: int = 1, padding: int = 1, with_stats: bool = True, in_norm=None):
    """``c2s_conv2d_forward``: raw convolution output [frames, c_out, H, W] (bf16) and the GroupNorm sums
    [frames, 4, 2] (float32; per quarter of the c_out channels, i.e. one group of ``GroupNorm(4, c_out)``) of its fp32
    values.

    ``in_norm = (stats, group_norm_module, relu)``: x is the RAW output of the previous stage and the kernel reads
    ``relu(GroupNorm(x))`` on the fly (the previous stage's normalisation pass is skipped)."""
    _require_cuda(x, "x")
    x = x.contiguous()
    dev = x.device
    n, c_in, h, w = x.shape
    c_out = weight.shape[0]
    d = _lib.ConvDesc(frames=n, c_in=c_in, c_out=c_out, H=h, W=w, kernel=kernel, stride=stride, padding=padding,
                      dtype=_code(x.dtype))
    wt = weight.detach().to(device=dev, dtype=torch.float32).contiguous()
    bs = None if bias is None else bias.detach().to(device=dev, dtype=torch.float32).contiguous()
    ho, wo = (h + 2 * padding - kernel) // stride + 1, (w + 2 * padding - kernel) // stride + 1
    y = torch.empty((n, c_out, ho, wo), dtype=x.dtype, device=dev)
    stats = torch.empty((n, 4, 2), dtype=torch.float32, device=dev) if with_stats else None
    inn, keep = None, []
    if in_norm is not None:
        st, norm, relu = in_norm
        keep = [st.contiguous(), norm.weight.detach().to(device=dev, dtype=torch.float32).contiguous(),
                norm.bias.detach().to(device=dev, dtype=torch.float32).contiguous()]
        inn = ctypes.byref(_lib.ConvInputNorm(stats=keep[0].data_ptr(), gamma=keep[1].data_ptr(), beta=keep[2].data_ptr(),
                                              n_groups=norm.num_groups, n_sub=st.shape[1], relu=int(relu), eps=float(norm.eps)))
    lib = _lib.load()
    with torch.cuda.device(dev):
        ws_bytes = lib.c2s_conv2d_workspace_bytes(ctypes.byref(d))
        ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=dev)
        status = lib.c2s_conv2d_forward(ctypes.byref(d), x.data_ptr(), inn, wt.data_ptr(), _ptr(bs), y.data_ptr(), _ptr(stats),
                                        ws.data_ptr(), ws_bytes, _stream(dev))
    _lib.check(status, "c2s_conv2d_forward")
    return y, stats


def group_stats(x: torch.Tensor, n_groups: int) -> torch.Tensor:
    """``c2s_group_stats``: (sum, sum of squares) per frame and group of x [frames, C, H, W] -> float32 [frames, G, 2]."""
    _require_cuda(x, "x")
    x = x.contiguous()
    n, c, h, w = x.shape
    stats = torch.empty((n, n_groups, 2), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        status = _lib.load().c2s_group_stats(x.data_ptr(), _code(x.dtype), n, c, h * w, n_groups, stats.data_ptr(),
                                             _stream(x.device))
    _lib.check(status, "c2s_group_stats")
    return stats


def group_norm_relu(x: torch.Tensor, stats: torch.Tensor, norm: nn.GroupNorm, *, relu: bool = True,
                    residual: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``c2s_group_norm_relu``: act(GroupNorm(x)) [+ residual] with the statistics of the convolution kernel or of
    :func:`group_stats`; x [frames, C, H, W]."""
    _require_cuda(x, "x")
    x = x.contiguous()
    dev = x.device
    n, c, h, w = x.shape
    out = torch.empty_like(x) if out is None else out
    gamma = norm.weight.detach().to(device=dev, dtype=torch.float32).contiguous()
    beta = norm.bias.detach().to(device=dev, dtype=torch.float32).contiguous()
    res = None if residual is None else residual.contiguous()
    with torch.cuda.device(dev):
        status = _lib.load().c2s_group_norm_relu(x.data_ptr(), stats.data_ptr(), stats.shape[1], gamma.data_ptr(),
                                                 beta.data_ptr(), _ptr(res), out.data_ptr(), _code(x.dtype), n, c, h * w,
                                                 norm.num_groups, float(norm.eps), int(relu), _stream(dev))
    _lib.check(status, "c2s_group_norm_relu")
    return out


# ------------------------------------------------------------------------------------------------ modules
class ConvLayer(nn.Module):
    """Drop-in for ``src.backbones.conv.ConvLayer`` (conv.py:29-96): ``Conv2d -> GroupNorm -> ReLU`` per entry of
    ``nkernels``; the sub-modules sit in ``self.conv`` (an ``nn.Sequential``) exactly like in the reference."""

    def __init__(self, nkernels, norm="batch", k=3, s=1, p=1, n_groups=4, last_relu=True, padding_mode="reflect",
                 conv_type="2d", add_squeeze=False):
        super().__init__()
        if conv_type != "2d" or add_squeeze:
            raise NotImplementedError("crop2seg_b200.ConvLayer: conv_type='2d' without squeeze-and-excitation only")
        if norm != "group":
            raise NotImplementedError("crop2seg_b200.ConvLayer: norm='group' only (the encoders' setting, utae.py:133)")
        self.conv_type, self.add_squeeze = conv_type, add_squeeze
        layers: List[nn.Module] = []
        self._plan = []  # (conv index, norm index, relu?)
        for i in range(len(nkernels) - 1):
            layers.append(nn.Conv2d(nkernels[i], nkernels[i + 1], kernel_size=k, padding=p, stride=s, padding_mode=padding_mode))
            ci = len(layers) - 1
            layers.append(nn.GroupNorm(num_channels=nkernels[i + 1], num_groups=n_groups))
            relu = bool(last_relu or i < len(nkernels) - 2)
            if relu:
                layers.append(nn.ReLU())
            self._plan.append((ci, ci + 1, relu))
        self.conv = nn.Sequential(*layers)

    def forward(self, input: torch.Tensor, residual_last: bool = False) -> torch.Tensor:
        """[frames, C, H, W] -> [frames, C', H', W'] (input dtype).  ``residual_last``: add the layer's INPUT to the
        output of its last stage (``out + conv2(out)``, conv.py:291), fused into the normalisation pass."""
        if self.training:
            raise NotImplementedError("crop2seg_b200.ConvLayer is an inference path: call .eval() "
                                      "(training keeps src.backbones.conv.ConvLayer)")
        _require_cuda(input, "input")
        dtype = input.dtype
        x = input.to(torch.bfloat16).contiguous()
        first = x
        pending = None  # (raw, stats, norm, relu) of a stage whose normalisation pass has not run yet
        for n_stage, (ci, ni, relu) in enumerate(self._plan):
            conv, norm = self.conv[ci], self.conv[ni]
            last = n_stage == len(self._plan) - 1
            src = pending[0] if pending is not None else x
            if conv2d_supported(src, conv):
                # the tensor-core kernel normalises its input on the fly: the previous stage's pass never touches memory
                raw, stats = conv2d_reflect_forward(src, conv.weight, conv.bias, kernel=conv.kernel_size[0],
                                                    stride=conv.stride[0], padding=conv.padding[0],
                                                    in_norm=None if pending is None else pending[1:])
            else:  # library convolution (cuDNN through torch) for shapes no kernel serves, see the module docstring
                if pending is not None:
                    x = group_norm_relu(pending[0], pending[1], pending[2], relu=pending[3], out=pending[0])
                pad = conv.padding[0]
                xp = F.pad(x, (pad, pad, pad, pad), mode=conv.padding_mode) if pad else x
                raw = F.conv2d(xp, conv.weight.to(torch.bfloat16), None if conv.bias is None else conv.bias.to(torch.bfloat16),
                               stride=conv.stride)
                stats = group_stats(raw, norm.num_groups)
            pending = (raw, stats, norm, relu)
            if last:
                x = group_norm_relu(raw, stats, norm, relu=relu, residual=first if residual_last else None, out=raw)
        return x.to(dtype)


class _TemporallyShared(nn.Module):
    """``TemporallySharedBlock`` (temp_shared_block.py:5-47) on the device-side frame packing of ``staging.py``."""

    def __init__(self, pad_value=None):
        super().__init__()
        self.out_shape = None
        self.pad_value = pad_value

    def smart_forward(self, input: torch.Tensor, pad_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        from .staging import smart_forward
        if input.dim() == 4:
            return self.forward(input)
        return smart_forward(self.forward, input, pad_value=self.pad_value, pad_mask=pad_mask)


class ConvBlock(_TemporallyShared):
    """Drop-in for ``src.backbones.conv.ConvBlock`` (conv.py:164-200)."""

    def __init__(self, nkernels, pad_value=None, norm="batch", last_relu=True, padding_mode="reflect", conv_type="2d",
                 add_squeeze=False):
        super().__init__(pad_value=pad_value)
        self.conv = ConvLayer(nkernels=nkernels, norm=norm, last_relu=last_relu, padding_mode=padding_mode,
                              conv_type=conv_type, add_squeeze=add_squeeze)

    def forward(self, input: torch.Tensor) -> torch.Tensor:
        return self.conv(input)


class DownConvBlock(_TemporallyShared):
    """Drop-in for ``src.backbones.conv.DownConvBlock`` (conv.py:238-296): strided ``down`` layer, ``conv1``, and
    ``out + conv2(out)``."""

    def __init__(self, d_in, d_out, k, s, p, pad_value=None, norm="batch", padding_mode="reflect", conv_type="2d",
                 add_squeeze=False):
        super().__init__(pad_value=pad_value)
        if add_squeeze:
            raise NotImplementedError("crop2seg_b200.DownConvBlock: squeeze-and-excitation is not served")
        self.down = ConvLayer(nkernels=[d_in, d_in], norm=norm, k=k, s=s, p=p, padding_mode=padding_mode, conv_type=conv_type)
        self.conv1 = ConvLayer(nkernels=[d_in, d_out], norm=norm, padding_mode=padding_mode, conv_type=conv_type)
        self.conv2 = ConvLayer(nkernels=[d_out, d_out], norm=norm, padding_mode=padding_mode, conv_type=conv_type)
        self.add_squeeze = add_squeeze

    def forward(self, input: torch.Tensor) -> torch.Tensor:
        out = self.down(input)
        out = self.conv1(out)
        return self.conv2(out, residual_last=True)  # out + conv2(out), conv.py:291
