"""Tensor-level entry points over the C ABI (``include/crop2seg_b200.h``).

PyTorch is plumbing here: it owns device memory and the current stream; every arithmetic step runs
in ``libcrop2seg_b200.so``.  Inputs must live on a CUDA device -- there is no CPU path.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass
from typing import Dict, NamedTuple, Optional, Tuple

import torch

from . import _lib

_AGG_MODES = {"att_group": _lib.AGG_ATT_GROUP, "att_mean": _lib.AGG_ATT_MEAN, "mean": _lib.AGG_MEAN}
_DTYPES = {torch.float32: _lib.F32, torch.bfloat16: _lib.BF16}
_FOLDED_CACHE_MAX_BYTES = 64 << 20  # larger L-TAE workspaces are transient (their preparation is noise there)


def _require_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(
            f"crop2seg_b200: {name} is on {t.device}; the operators are CUDA (sm_100a) only and have no CPU fallback")


def _dtype_code(t: torch.Tensor, name: str) -> int:
    try:
        return _DTYPES[t.dtype]
    except KeyError:
        raise RuntimeError(f"crop2seg_b200: {name} has dtype {t.dtype}; supported: float32, bfloat16") from None


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _mask_u8(mask: Optional[torch.Tensor], shape: tuple, name: str, device) -> Optional[torch.Tensor]:
    """A pad or dropout-keep mask as uint8 on ``device`` (bool and uint8 masks are used as they are, any other dtype
    as ``mask != 0``); None stays None."""
    if mask is None:
        return None
    if tuple(mask.shape) != shape:
        raise RuntimeError(f"crop2seg_b200: {name} has shape {tuple(mask.shape)}, expected {shape}")
    m = mask.to(device=device)
    if m.dtype not in (torch.bool, torch.uint8):
        m = m != 0
    return m.contiguous().view(torch.uint8)


def _features(x: torch.Tensor) -> torch.Tensor:
    """x[B,T,C,H,W] on a CUDA device, contiguous."""
    if x.dim() != 5:
        raise RuntimeError(f"crop2seg_b200: x must be [B,T,C,H,W], got {tuple(x.shape)}")
    _require_cuda(x, "x")
    return x.contiguous()


def pad_mask_from_input(x: torch.Tensor, pad_value: float = 0.0) -> torch.Tensor:
    """``(x == pad_value).all(dim=-1).all(dim=-1).all(dim=-1)`` for x[B,T,C,H,W] (utae.py:201-203, wtae.py:221-223,
    timeunet.py:170-172): bool [B,T].  One kernel; a valid frame is left at its first non-pad value, only padded
    frames are read to the end (the reference compares and reduces the whole input three times)."""
    x = _features(x)
    b, t = x.shape[:2]
    mask = torch.empty((b, t), dtype=torch.uint8, device=x.device)
    lib = _lib.load()
    with torch.cuda.device(x.device):
        status = lib.c2s_pad_mask(x.data_ptr(), _dtype_code(x, "x"), b * t, x[0, 0].numel(), float(pad_value),
                                  mask.data_ptr(), _stream(x.device))
    _lib.check(status, "c2s_pad_mask")
    return mask.view(torch.bool)


def _agg_inputs(x: torch.Tensor, attn_mask: Optional[torch.Tensor], mode: str
                ) -> Tuple[torch.Tensor, Optional[torch.Tensor], _lib.AggDesc]:
    """Checked inputs of an aggregation: contiguous x[B,T,C,H,W], the attention map attn_mask[h,B,T,ha,wa] as float32
    on x's device (None in mode 'mean', which reads none) and the ``c2s_agg_desc`` of both."""
    if mode not in _AGG_MODES:
        raise ValueError(f"unknown aggregation mode {mode!r}")
    x = _features(x)
    b, t, c, h, w = x.shape
    desc = _lib.AggDesc(B=b, T=t, C=c, H=h, W=w, n_heads=1, ha=1, wa=1, mode=_AGG_MODES[mode],
                        dtype=_dtype_code(x, "x"))
    if mode == "mean":
        return x, None, desc
    if attn_mask is None or attn_mask.dim() != 5 or tuple(attn_mask.shape[1:3]) != (b, t):
        got = None if attn_mask is None else tuple(attn_mask.shape)
        raise RuntimeError(f"crop2seg_b200: mode {mode!r} needs attn_mask [h,{b},{t},ha,wa], got {got}")
    attn = attn_mask.to(device=x.device, dtype=torch.float32).contiguous()
    desc.n_heads, desc.ha, desc.wa = attn.shape[0], attn.shape[3], attn.shape[4]
    return x, attn, desc


def temporal_aggregate(x: torch.Tensor, pad_mask: Optional[torch.Tensor] = None,
                       attn_mask: Optional[torch.Tensor] = None, mode: str = "mean") -> torch.Tensor:
    """``TemporalAggregator(mode).forward(x, pad_mask, attn_mask)`` (temporal_aggregator.py:14-77), differentiable
    w.r.t. x and attn_mask (both directions are CUDA kernels)."""
    if torch.is_grad_enabled() and (x.requires_grad or (attn_mask is not None and attn_mask.requires_grad)):
        from .autograd import AggregateFunction
        return AggregateFunction.apply(x, attn_mask, pad_mask, mode)
    return temporal_aggregate_forward(x, pad_mask, attn_mask, mode)


def temporal_aggregate_forward(x: torch.Tensor, pad_mask: Optional[torch.Tensor] = None,
                               attn_mask: Optional[torch.Tensor] = None, mode: str = "mean") -> torch.Tensor:
    """``TemporalAggregator(mode).forward(x, pad_mask, attn_mask)`` (temporal_aggregator.py:14-77).

    x[B,T,C,H,W] float32/bfloat16, attn_mask[h,B,T,ha,wa] (float32 used as is), pad_mask[B,T] bool.
    Returns out[B,C,H,W] in x's dtype.  One kernel launch; no host synchronisation.
    """
    x, attn, desc = _agg_inputs(x, attn_mask, mode)
    b, t, c, h, w = x.shape
    pad = _mask_u8(pad_mask, (b, t), "pad_mask", x.device)
    out = torch.empty((b, c, h, w), dtype=x.dtype, device=x.device)
    lib = _lib.load()
    with torch.cuda.device(x.device):
        ws_bytes = lib.c2s_agg_workspace_bytes(ctypes.byref(desc))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device) if ws_bytes else None
        status = lib.c2s_agg_forward(ctypes.byref(desc), x.data_ptr(), _ptr(attn), _ptr(pad), out.data_ptr(),
                                     _ptr(ws), ws_bytes, _stream(x.device))
    _lib.check(status, "c2s_agg_forward")
    return out


def temporal_aggregate_skip_conv(x: torch.Tensor, pad_mask: Optional[torch.Tensor], attn_mask: torch.Tensor,
                                 conv_weight: torch.Tensor, conv_bias: Optional[torch.Tensor],
                                 bn_weight: Optional[torch.Tensor], bn_bias: Optional[torch.Tensor],
                                 bn_running_mean: torch.Tensor, bn_running_var: torch.Tensor, bn_eps: float = 1e-5
                                 ) -> torch.Tensor:
    """``relu(BatchNorm2d_eval(Conv2d_1x1(TemporalAggregator('att_group')(x, pad_mask, attn_mask))))`` in one kernel,
    differentiable w.r.t. x, attn_mask, the convolution and the BatchNorm affine (both directions are CUDA kernels;
    the BatchNorm stays frozen: running statistics)."""
    tensors = (x, attn_mask, conv_weight, conv_bias, bn_weight, bn_bias)
    if torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors):
        from .autograd import AggregateSkipConvFunction
        return AggregateSkipConvFunction.apply(x, attn_mask, pad_mask, conv_weight, conv_bias, bn_weight, bn_bias,
                                               bn_running_mean, bn_running_var, bn_eps)
    return temporal_aggregate_skip_conv_forward(x, pad_mask, attn_mask, conv_weight, conv_bias, bn_weight, bn_bias,
                                                bn_running_mean, bn_running_var, bn_eps)


def _skipconv_inputs(x, pad_mask, attn_mask, conv_weight, conv_bias, bn_weight, bn_bias, bn_running_mean, bn_running_var,
                     bn_eps, keep):
    """Checked inputs of the fused skip convolution: x, attention, uint8 pad mask, ``c2s_agg_desc`` and
    ``c2s_skipconv_params`` (the float32 parameter copies it points to are kept alive in ``keep``)."""
    x, attn, desc = _agg_inputs(x, attn_mask, "att_group")
    b, t, c, h, w = x.shape
    if tuple(conv_weight.shape[:2]) != (c, c) or conv_weight.numel() != c * c:
        raise RuntimeError(f"crop2seg_b200: skip convolution must be 1x1 {c}->{c}, got {tuple(conv_weight.shape)}")
    pad = _mask_u8(pad_mask, (b, t), "pad_mask", x.device)
    params = _lib.SkipConvParams(
        conv_weight=_f32(conv_weight, x.device, keep), conv_bias=_f32(conv_bias, x.device, keep),
        bn_weight=_f32(bn_weight, x.device, keep), bn_bias=_f32(bn_bias, x.device, keep),
        bn_running_mean=_f32(bn_running_mean, x.device, keep), bn_running_var=_f32(bn_running_var, x.device, keep),
        bn_eps=float(bn_eps))
    return x, attn, pad, desc, params


def temporal_aggregate_skip_conv_forward(x: torch.Tensor, pad_mask: Optional[torch.Tensor], attn_mask: torch.Tensor,
                                         conv_weight: torch.Tensor, conv_bias: Optional[torch.Tensor],
                                         bn_weight: Optional[torch.Tensor], bn_bias: Optional[torch.Tensor],
                                         bn_running_mean: torch.Tensor, bn_running_var: torch.Tensor, bn_eps: float = 1e-5
                                         ) -> torch.Tensor:
    """``relu(BatchNorm2d_eval(Conv2d_1x1(TemporalAggregator('att_group')(x, pad_mask, attn_mask))))`` in one kernel:
    the aggregation of utae.py:225-227 followed by ``UpConvBlock.skip_conv`` (conv.py:378-382, 408), the skip map never
    leaving the chip (``c2s_agg_skipconv_forward``).  Running statistics; bf16 x[B,T,64,H,W], 16 heads, x2/x4/x8
    up-sampling, H*W % 128 == 0 -- other shapes raise (use the two modules separately)."""
    keep = []
    x, attn, pad, desc, params = _skipconv_inputs(x, pad_mask, attn_mask, conv_weight, conv_bias, bn_weight, bn_bias,
                                                  bn_running_mean, bn_running_var, bn_eps, keep)
    b, t, c, h, w = x.shape
    out = torch.empty((b, c, h, w), dtype=x.dtype, device=x.device)
    lib = _lib.load()
    with torch.cuda.device(x.device):
        ws_bytes = lib.c2s_agg_skipconv_workspace_bytes(ctypes.byref(desc))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
        status = lib.c2s_agg_skipconv_forward(ctypes.byref(desc), x.data_ptr(), attn.data_ptr(), _ptr(pad),
                                              ctypes.byref(params), out.data_ptr(), ws.data_ptr(), ws_bytes,
                                              _stream(x.device))
    _lib.check(status, "c2s_agg_skipconv_forward")
    return out


def temporal_aggregate_skip_conv_backward(x: torch.Tensor, pad_mask: Optional[torch.Tensor], attn_mask: torch.Tensor,
                                          conv_weight: torch.Tensor, conv_bias: Optional[torch.Tensor],
                                          bn_weight: Optional[torch.Tensor], bn_bias: Optional[torch.Tensor],
                                          bn_running_mean: torch.Tensor, bn_running_var: torch.Tensor, bn_eps: float,
                                          out: torch.Tensor, grad_out: torch.Tensor, need=(True,) * 6
                                          ) -> Tuple[Optional[torch.Tensor], ...]:
    """Backward of :func:`temporal_aggregate_skip_conv_forward` (``c2s_agg_skipconv_backward``) from its output ``out``:
    ``(grad_x, grad_attn, grad_conv_weight, grad_conv_bias, grad_bn_weight, grad_bn_bias)``, each None where ``need``
    (same order) says so or the parameter is None.  grad_x is bf16 like x, the others float32; grad_attn is accumulated
    with float atomics (as in :func:`temporal_aggregate_backward`), the parameter gradients are deterministic."""
    keep = []
    x, attn, pad, desc, params = _skipconv_inputs(x, pad_mask, attn_mask, conv_weight, conv_bias, bn_weight, bn_bias,
                                                  bn_running_mean, bn_running_var, bn_eps, keep)
    b, t, c, h, w = x.shape
    if tuple(out.shape) != (b, c, h, w) or tuple(grad_out.shape) != (b, c, h, w):
        raise RuntimeError(f"crop2seg_b200: out {tuple(out.shape)} / grad_out {tuple(grad_out.shape)} must be {(b, c, h, w)}")
    o = out.to(dtype=x.dtype).contiguous()
    gout = grad_out.to(dtype=x.dtype).contiguous()
    f32 = dict(dtype=torch.float32, device=x.device)
    want = [bool(n) for n in need]
    want[3] = want[3] and conv_bias is not None
    want[4] = want[4] and bn_weight is not None
    want[5] = want[5] and bn_bias is not None
    res = [torch.empty_like(x) if want[0] else None, torch.zeros_like(attn) if want[1] else None,
           torch.empty((c, c), **f32) if want[2] else None] + [torch.empty(c, **f32) if k else None for k in want[3:]]
    io = _lib.SkipConvBwdIo(**{k: _ptr(r) for k, r in zip(_lib.SKIPCONV_BWD_IO_FIELDS, res)})
    lib = _lib.load()
    with torch.cuda.device(x.device):
        ws_bytes = lib.c2s_agg_skipconv_backward_workspace_bytes(ctypes.byref(desc))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
        status = lib.c2s_agg_skipconv_backward(ctypes.byref(desc), x.data_ptr(), attn.data_ptr(), _ptr(pad),
                                               ctypes.byref(params), o.data_ptr(), gout.data_ptr(), ctypes.byref(io),
                                               ws.data_ptr(), ws_bytes, _stream(x.device))
    _lib.check(status, "c2s_agg_skipconv_backward")
    if res[2] is not None:
        res[2] = res[2].view(conv_weight.shape)
    return tuple(res)


def temporal_aggregate_skip_conv_bstats_forward(x: torch.Tensor, pad_mask: Optional[torch.Tensor], attn_mask: torch.Tensor,
                                                conv_weight: torch.Tensor, conv_bias: Optional[torch.Tensor],
                                                bn_weight: Optional[torch.Tensor], bn_bias: Optional[torch.Tensor],
                                                bn_eps: float = 1e-5, keep_z: bool = True
                                                ) -> Tuple[torch.Tensor, Optional[torch.Tensor], torch.Tensor, torch.Tensor]:
    """``relu(BatchNorm2d_train(Conv2d_1x1(TemporalAggregator('att_group')(x, pad_mask, attn_mask))))`` with the
    BatchNorm normalising by the batch statistics of z = the bf16 convolution output (``c2s_agg_skipconv_bstats_forward``).
    Returns ``(out, z | None, batch_mean, batch_var)`` (biased variance, float32 [64]); the running statistics are the
    caller's.  ``keep_z=False`` writes z into ``out``'s memory and returns None for it.  Same shapes as
    :func:`temporal_aggregate_skip_conv_forward`."""
    keep = []
    x, attn, pad, desc, params = _skipconv_inputs(x, pad_mask, attn_mask, conv_weight, conv_bias, bn_weight, bn_bias,
                                                  None, None, bn_eps, keep)
    b, t, c, h, w = x.shape
    out = torch.empty((b, c, h, w), dtype=x.dtype, device=x.device)
    z = torch.empty_like(out) if keep_z else out
    mean = torch.empty(c, dtype=torch.float32, device=x.device)
    var = torch.empty_like(mean)
    lib = _lib.load()
    with torch.cuda.device(x.device):
        ws_bytes = lib.c2s_agg_skipconv_bstats_workspace_bytes(ctypes.byref(desc))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
        status = lib.c2s_agg_skipconv_bstats_forward(ctypes.byref(desc), x.data_ptr(), attn.data_ptr(), _ptr(pad),
                                                     ctypes.byref(params), z.data_ptr(), out.data_ptr(), mean.data_ptr(),
                                                     var.data_ptr(), ws.data_ptr(), ws_bytes, _stream(x.device))
    _lib.check(status, "c2s_agg_skipconv_bstats_forward")
    return out, (z if keep_z else None), mean, var


def temporal_aggregate_skip_conv_bstats_backward(x: torch.Tensor, pad_mask: Optional[torch.Tensor], attn_mask: torch.Tensor,
                                                 conv_weight: torch.Tensor, conv_bias: Optional[torch.Tensor],
                                                 bn_weight: Optional[torch.Tensor], bn_bias: Optional[torch.Tensor],
                                                 bn_eps: float, z: torch.Tensor, batch_mean: torch.Tensor,
                                                 batch_var: torch.Tensor, out: torch.Tensor, grad_out: torch.Tensor,
                                                 need=(True,) * 6) -> Tuple[Optional[torch.Tensor], ...]:
    """Backward of :func:`temporal_aggregate_skip_conv_bstats_forward` (``c2s_agg_skipconv_bstats_backward``) from its
    z, batch statistics and output: ``(grad_x, grad_attn, grad_conv_weight, grad_conv_bias, grad_bn_weight,
    grad_bn_bias)`` as in :func:`temporal_aggregate_skip_conv_backward`; grad_conv_bias is exactly zero."""
    keep = []
    x, attn, pad, desc, params = _skipconv_inputs(x, pad_mask, attn_mask, conv_weight, conv_bias, bn_weight, bn_bias,
                                                  None, None, bn_eps, keep)
    b, t, c, h, w = x.shape
    for name, v in (("z", z), ("out", out), ("grad_out", grad_out)):
        if tuple(v.shape) != (b, c, h, w):
            raise RuntimeError(f"crop2seg_b200: {name} {tuple(v.shape)} must be {(b, c, h, w)}")
    zz, o, gout = (v.to(dtype=x.dtype).contiguous() for v in (z, out, grad_out))
    mean, var = (v.to(device=x.device, dtype=torch.float32).contiguous() for v in (batch_mean, batch_var))
    f32 = dict(dtype=torch.float32, device=x.device)
    want = [bool(n) for n in need]
    want[3] = want[3] and conv_bias is not None
    want[4] = want[4] and bn_weight is not None
    want[5] = want[5] and bn_bias is not None
    res = [torch.empty_like(x) if want[0] else None, torch.zeros_like(attn) if want[1] else None,
           torch.empty((c, c), **f32) if want[2] else None] + [torch.empty(c, **f32) if k else None for k in want[3:]]
    io = _lib.SkipConvBwdIo(**{k: _ptr(r) for k, r in zip(_lib.SKIPCONV_BWD_IO_FIELDS, res)})
    lib = _lib.load()
    with torch.cuda.device(x.device):
        ws_bytes = lib.c2s_agg_skipconv_bstats_backward_workspace_bytes(ctypes.byref(desc))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
        status = lib.c2s_agg_skipconv_bstats_backward(ctypes.byref(desc), x.data_ptr(), attn.data_ptr(), _ptr(pad),
                                                      ctypes.byref(params), zz.data_ptr(), mean.data_ptr(),
                                                      var.data_ptr(), o.data_ptr(), gout.data_ptr(), ctypes.byref(io),
                                                      ws.data_ptr(), ws_bytes, _stream(x.device))
    _lib.check(status, "c2s_agg_skipconv_bstats_backward")
    if res[2] is not None:
        res[2] = res[2].view(conv_weight.shape)
    return tuple(res)


def temporal_aggregate_backward(x: torch.Tensor, pad_mask: Optional[torch.Tensor], attn_mask: Optional[torch.Tensor],
                                grad_out: torch.Tensor, mode: str, need_x: bool = True, need_attn: bool = True
                                ) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
    """Backward of :func:`temporal_aggregate`: ``(grad_x | None, grad_attn | None)`` (``c2s_agg_backward``).

    grad_attn is accumulated with float atomics (low bits depend on the execution order, like the reference's own
    backward, train.py:623-626)."""
    x, attn, desc = _agg_inputs(x, attn_mask, mode)
    b, t = x.shape[:2]
    gout = grad_out.to(dtype=x.dtype).contiguous()
    pad = _mask_u8(pad_mask, (b, t), "pad_mask", x.device)
    gx = torch.empty_like(x) if need_x else None
    gattn = torch.zeros_like(attn) if need_attn and attn is not None else None
    lib = _lib.load()
    with torch.cuda.device(x.device):
        ws_bytes = lib.c2s_agg_backward_workspace_bytes(ctypes.byref(desc))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device) if ws_bytes else None
        status = lib.c2s_agg_backward(ctypes.byref(desc), x.data_ptr(), _ptr(attn), _ptr(pad), gout.data_ptr(),
                                      _ptr(gx), _ptr(gattn), _ptr(ws), ws_bytes, _stream(x.device))
    _lib.check(status, "c2s_agg_backward")
    return gx, gattn


def _f32(t: Optional[torch.Tensor], device, keep) -> Optional[int]:
    """Device pointer of a float32, contiguous view of a parameter (kept alive in ``keep``)."""
    if t is None:
        return None
    v = t.detach()
    if v.device != device or v.dtype != torch.float32 or not v.is_contiguous():
        v = v.to(device=device, dtype=torch.float32).contiguous()
    keep.append(v)
    return v.data_ptr()


@dataclass(frozen=True)
class LtaeSpec:
    """What the L-TAE calls need to know about an encoder besides its tensors, for one forward (and its backward).

    ``c_out`` is mlp[-1] (0 with ``attn_only``, LTAE4WTAE); ``pe_mode`` an ``_lib.PE_*`` value; ``zero_padded``: padded
    frames of x are exactly zero and are not read; ``bn_batch_stats``: the MLP's BatchNorm normalises with the batch
    statistics (training mode); ``attn_drop_p`` / ``mlp_drop_p``: the dropout rates of the forward (0 in eval mode).
    """
    n_head: int
    d_k: int
    d_model: int
    has_inconv: bool
    c_out: int = 0
    pe_mode: int = _lib.PE_NONE
    pe_abs: bool = False
    attn_only: bool = False
    zero_padded: bool = False
    bn_batch_stats: bool = False
    gn_eps: float = 1e-5
    bn_eps: float = 1e-5
    attn_drop_p: float = 0.0
    mlp_drop_p: float = 0.0


class LtaeOutputs(NamedTuple):
    """Result of :func:`ltae_forward`."""
    out: Optional[torch.Tensor]  # [B,c_out,H,W] in x's dtype; None with attn_only
    attn: Optional[torch.Tensor]  # float32 [n_head,B,T,H,W]; None without need_attn
    stats: Optional[Tuple[torch.Tensor, torch.Tensor]]  # BatchNorm batch mean and biased variance (bn_batch_stats)
    o_rows: Optional[torch.Tensor]  # save_o: float32 [B*H*W, d_model], the rows that enter the MLP
    y_rows: Optional[torch.Tensor]  # save_y with bn_batch_stats: float32 [B*H*W, c_out], the pre-BatchNorm rows


def _ltae_desc(spec: LtaeSpec, shape, dtype: int, flags: int = 0, pos_dtype: int = 0, attn_dropout: bool = True,
               mlp_dropout: bool = True) -> _lib.LtaeDesc:
    """``c2s_ltae_desc`` of ``spec`` for x of ``shape`` [B,T,C,H,W] and dtype code ``dtype``.  ``flags`` are added to the
    spec's own (attention only, zero-padded frames); the keep scales are 1/(1-p) for the dropouts the call applies
    (``attn_dropout`` / ``mlp_dropout``) and 1 for the others."""
    b, t, c, h, w = shape
    flags |= (_lib.LTAE_ATTN_ONLY if spec.attn_only else 0) | (_lib.LTAE_ZERO_PADDED if spec.zero_padded else 0)
    return _lib.LtaeDesc(B=b, T=t, C=c, H=h, W=w, n_head=spec.n_head, d_k=spec.d_k, d_model=spec.d_model,
                         c_out=spec.c_out, has_inconv=int(spec.has_inconv), pe_mode=spec.pe_mode, pe_abs=int(spec.pe_abs),
                         pos_dtype=pos_dtype, dtype=dtype, flags=flags, gn_eps=spec.gn_eps, bn_eps=spec.bn_eps,
                         attn_keep_scale=1.0 / (1.0 - spec.attn_drop_p) if attn_dropout else 1.0,
                         mlp_keep_scale=1.0 / (1.0 - spec.mlp_drop_p) if mlp_dropout else 1.0)


def _ltae_rows_desc(spec: LtaeSpec, batch: int, height: int, width: int, dtype: int) -> _lib.LtaeDesc:
    """``c2s_ltae_desc`` of the calls on the rows after the attention (``c2s_ltae_rows_forward``,
    ``c2s_ltae_mlp_backward``): T = 1, C = n_head, d_k = 1, an in-projection, no positional encoding, and of the flags
    only the BatchNorm batch statistics."""
    desc = _ltae_desc(spec, (batch, 1, spec.n_head, height, width), dtype, attn_dropout=False)
    desc.d_k, desc.has_inconv, desc.pe_mode, desc.pe_abs = 1, 1, _lib.PE_NONE, 0
    desc.flags = _lib.LTAE_BN_BATCH_STATS if spec.bn_batch_stats else 0
    return desc


def _ltae_params(params: Dict[str, Optional[torch.Tensor]], desc: _lib.LtaeDesc, device, keep: list,
                 attn_keep: Optional[torch.Tensor] = None, mlp_keep: Optional[torch.Tensor] = None) -> _lib.LtaeParams:
    """``c2s_ltae_params`` from a dict keyed by its field names and the optional dropout keep masks ``attn_keep``
    [h,B,T,H,W] (tae.py:837) and ``mlp_keep`` [B,c_out,H,W] (after the ReLU, tae.py:448), shapes taken from ``desc``.
    The tensors it points to are kept alive in ``keep``."""
    cparams = _lib.LtaeParams(**{k: _f32(params.get(k), device, keep) for k in _lib.LTAE_PARAM_FIELDS})
    if attn_keep is not None:
        keep.append(_mask_u8(attn_keep, (desc.n_head, desc.B, desc.T, desc.H, desc.W), "attn_keep", device))
        cparams.attn_keep = keep[-1].data_ptr()
    if mlp_keep is not None:
        keep.append(_mask_u8(mlp_keep, (desc.B, desc.c_out, desc.H, desc.W), "mlp_keep", device))
        cparams.mlp_keep = keep[-1].data_ptr()
    return cparams


def _positions(positions: Optional[torch.Tensor], spec: LtaeSpec, b: int, t: int, device
               ) -> Tuple[Optional[torch.Tensor], int]:
    """``(positions, pos_dtype)`` as the kernels read them: int64 (0) or, for floating-point input, float32 (1);
    ``(None, 0)`` without positional encoding."""
    if spec.pe_mode == _lib.PE_NONE:
        return None, 0
    if positions is None:
        raise RuntimeError("crop2seg_b200: batch_positions is required when positional encoding is enabled")
    want = (b, t, 2) if spec.pe_abs else (b, t)
    if tuple(positions.shape) != want:
        raise RuntimeError(f"crop2seg_b200: batch_positions has shape {tuple(positions.shape)}, expected {want}")
    pos = positions.to(device=device)
    if pos.dtype.is_floating_point:
        return pos.to(torch.float32).contiguous(), 1
    return pos.to(torch.int64).contiguous(), 0


def ltae_forward(x: torch.Tensor, positions: Optional[torch.Tensor], pad_mask: Optional[torch.Tensor],
                 params: Dict[str, Optional[torch.Tensor]], spec: LtaeSpec, *, need_attn: bool = True,
                 attn_keep: Optional[torch.Tensor] = None, mlp_keep: Optional[torch.Tensor] = None,
                 folded_cache: Optional[dict] = None, folded_key=None, save_o: bool = False, save_y: bool = False
                 ) -> LtaeOutputs:
    """Fused ``LTAE.forward`` / ``LTAE4WTAE.forward`` (tae.py:451-504, 589-635).

    ``params`` maps the field names of ``c2s_ltae_params`` to tensors (or None); ``attn_keep`` / ``mlp_keep`` are the
    dropout keep masks of a training-mode forward (rates in ``spec``).
    ``folded_cache`` (a dict owned by the caller) with ``folded_key`` (anything that changes whenever a parameter
    does) keeps the workspace between calls: while key, shapes and flags repeat, the weight-only preparation kernels
    are skipped (``C2S_LTAE_REUSE_FOLDED``).  Workspaces above 64 MiB are never kept.
    ``save_o`` / ``save_y`` also return the rows the backward needs (see :class:`LtaeOutputs`).
    """
    x = _features(x)
    dev = x.device
    b, t, c, h, w = x.shape
    pos, pos_dtype = _positions(positions, spec, b, t, dev)
    flags = (0 if need_attn else _lib.LTAE_SKIP_ATTN_STORE) | (
        _lib.LTAE_BN_BATCH_STATS if spec.bn_batch_stats and not spec.attn_only else 0)
    desc = _ltae_desc(spec, x.shape, _dtype_code(x, "x"), flags, pos_dtype)
    keep = []
    cparams = _ltae_params(params, desc, dev, keep, attn_keep, mlp_keep)
    o_rows = y_rows = None
    if save_o and not spec.attn_only:
        o_rows = torch.empty((b * h * w, spec.d_model), dtype=torch.float32, device=dev)
        cparams.save_o = o_rows.data_ptr()
    if save_y and flags & _lib.LTAE_BN_BATCH_STATS:
        y_rows = torch.empty((b * h * w, spec.c_out), dtype=torch.float32, device=dev)
        cparams.save_y = y_rows.data_ptr()
    pad = _mask_u8(pad_mask, (b, t), "pad_mask", dev)
    out = None if spec.attn_only else torch.empty((b, spec.c_out, h, w), dtype=x.dtype, device=dev)
    attn = torch.empty((spec.n_head, b, t, h, w), dtype=torch.float32, device=dev) if need_attn else None
    stats = None
    if flags & _lib.LTAE_BN_BATCH_STATS:
        stats = (torch.empty(spec.c_out, dtype=torch.float32, device=dev),
                 torch.empty(spec.c_out, dtype=torch.float32, device=dev))
    lib = _lib.load()
    with torch.cuda.device(dev):
        ws_bytes = lib.c2s_ltae_workspace_bytes(ctypes.byref(desc))
        ws = None
        # Under CUDA-graph capture the cache is bypassed: a captured graph bakes the workspace pointer, and a cached
        # workspace can be evicted (another shape) or go stale (weights updated) while the graph lives on.  A captured
        # call allocates its workspace inside the capture (the graph's private pool keeps it alive) and folds the
        # weights on every replay.
        capturing = torch.cuda.is_current_stream_capturing()
        if folded_cache is not None and ws_bytes <= _FOLDED_CACHE_MAX_BYTES and not capturing:
            key = (folded_key, dev, bytes(desc))  # the descriptor holds every shape, flag and constant of the call
            if folded_cache.get("key") == key and folded_cache.get("ws") is not None:
                ws = folded_cache["ws"]
                desc.flags |= _lib.LTAE_REUSE_FOLDED
            else:
                ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=dev)
                folded_cache["key"], folded_cache["ws"] = key, ws
        if ws is None:
            ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=dev)
        status = lib.c2s_ltae_forward(ctypes.byref(desc), ctypes.byref(cparams), x.data_ptr(), _ptr(pos), _ptr(pad),
                                      _ptr(out), _ptr(attn), _ptr(stats[0]) if stats else None,
                                      _ptr(stats[1]) if stats else None, ws.data_ptr(), ws_bytes, _stream(dev))
    _lib.check(status, "c2s_ltae_forward")
    return LtaeOutputs(out, attn, stats, o_rows, y_rows)


def ltae_rows_forward(o_rows: torch.Tensor, params: Dict[str, Optional[torch.Tensor]], spec: LtaeSpec, *, batch: int,
                      height: int, width: int, dtype: torch.dtype) -> torch.Tensor:
    """``c2s_ltae_rows_forward``: the rows behind the attention of an encoder with n > 1 learned queries, eval mode
    (tae.py:486-499): ``o_rows`` [n, B*H*W, d_model] (float32, the ``save_o`` rows of one ``ltae_forward`` per query)
    -> ``out`` [B, n, c_out, H, W]; the output GroupNorm (eps ``spec.gn_eps``) runs over the channels of a group and
    the n queries."""
    _require_cuda(o_rows, "o_rows")
    dev = o_rows.device
    n_q = o_rows.shape[0]
    if o_rows.dim() != 3 or tuple(o_rows.shape[1:]) != (batch * height * width, spec.d_model):
        raise RuntimeError(f"crop2seg_b200: o_rows has shape {tuple(o_rows.shape)}")
    o = o_rows.to(torch.float32).contiguous()
    out = torch.empty((batch, n_q, spec.c_out, height, width), dtype=dtype, device=dev)
    desc = _ltae_rows_desc(spec, batch, height, width, _dtype_code(out, "out"))
    keep = []
    cparams = _ltae_params(params, desc, dev, keep)
    with torch.cuda.device(dev):
        status = _lib.load().c2s_ltae_rows_forward(ctypes.byref(desc), ctypes.byref(cparams), o.data_ptr(), n_q,
                                                   out.data_ptr(), _stream(dev))
    _lib.check(status, "c2s_ltae_rows_forward")
    return out


def ltae_backward(x: torch.Tensor, positions: Optional[torch.Tensor], pad_mask: Optional[torch.Tensor],
                  params: Dict[str, Optional[torch.Tensor]], grad_o: Optional[torch.Tensor],
                  grad_attn: Optional[torch.Tensor], spec: LtaeSpec, *, attn_keep: Optional[torch.Tensor] = None,
                  need_grad_pe: bool = False) -> Dict[str, Optional[torch.Tensor]]:
    """``c2s_ltae_backward``: everything of the L-TAE backward that touches the [B*H*W, T, C] features.

    ``grad_o`` [B*H*W, d_model] is the gradient w.r.t. the rows entering the MLP, ``grad_attn`` [h,B,T,H,W] the one
    w.r.t. the returned attention.  Returns ``grad_x`` and the gradients of the folded quantities (``grad_u`` [C,16],
    ``grad_cpos`` [B,T,16], ``grad_gamma`` / ``grad_beta`` [C] direct terms, ``zn_rows`` [B*H*W,h,C], ``sa_rows``
    [B*H*W,16], ``grad_pe`` [B,T,d_model] | None); see ``include/crop2seg_b200.h``."""
    x = _features(x)
    dev = x.device
    b, t, c, h, w = x.shape
    n = b * h * w
    n_head, d_model, attn_only = spec.n_head, spec.d_model, spec.attn_only
    pos, pos_dtype = _positions(positions, spec, b, t, dev)
    desc = _ltae_desc(spec, x.shape, _dtype_code(x, "x"), pos_dtype=pos_dtype, mlp_dropout=False)
    keep = []
    cparams = _ltae_params(params, desc, dev, keep, attn_keep)
    f32 = dict(dtype=torch.float32, device=dev)
    # the accumulated (atomic) outputs are slices of ONE zero-filled buffer: one memset instead of one per tensor
    want_pe = (not attn_only) and need_grad_pe and spec.pe_mode != _lib.PE_NONE
    sizes = [c * 16, b * t * 16] + ([c, c] if not attn_only else []) + ([b * t * d_model] if want_pe else [])
    offs = [0]
    for sz in sizes:
        offs.append(offs[-1] + (sz + 3) // 4 * 4)  # 16-byte aligned slices
    zeros = torch.zeros(offs[-1], dtype=torch.float32, device=dev)
    res = {
        "grad_x": torch.empty_like(x), "grad_u": zeros[offs[0]:offs[0] + c * 16].view(c, 16),
        "grad_cpos": zeros[offs[1]:offs[1] + b * t * 16].view(b, t, 16),
        "grad_gamma": None, "grad_beta": None, "zn_rows": None, "sa_rows": None, "grad_pe": None,
    }
    io = _lib.LtaeBwdIo()
    if not attn_only:
        if grad_o is None or tuple(grad_o.shape) != (n, d_model):
            raise RuntimeError(f"crop2seg_b200: grad_o must be [{n},{d_model}]")
        go = grad_o.to(**f32).contiguous()
        keep.append(go)
        io.grad_o = go.data_ptr()
        res["grad_gamma"], res["grad_beta"] = zeros[offs[2]:offs[2] + c], zeros[offs[3]:offs[3] + c]
        res["zn_rows"], res["sa_rows"] = torch.empty((n, n_head, c), **f32), torch.empty((n, 16), **f32)
        if want_pe:
            res["grad_pe"] = zeros[offs[4]:offs[4] + b * t * d_model].view(b, t, d_model)
    if grad_attn is not None:
        ga = grad_attn.to(**f32).contiguous()
        if tuple(ga.shape) != (n_head, b, t, h, w):
            raise RuntimeError(f"crop2seg_b200: grad_attn has shape {tuple(ga.shape)}")
        keep.append(ga)
        io.grad_attn = ga.data_ptr()
    for k in ("grad_x", "grad_u", "grad_cpos", "grad_gamma", "grad_beta", "zn_rows", "sa_rows", "grad_pe"):
        if res[k] is not None:
            setattr(io, k, res[k].data_ptr())
    pad = _mask_u8(pad_mask, (b, t), "pad_mask", dev)
    lib = _lib.load()
    with torch.cuda.device(dev):
        ws_bytes = lib.c2s_ltae_backward_workspace_bytes(ctypes.byref(desc))
        ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=dev)
        status = lib.c2s_ltae_backward(ctypes.byref(desc), ctypes.byref(cparams), x.data_ptr(), _ptr(pos), _ptr(pad),
                                       ctypes.byref(io), ws.data_ptr(), ws_bytes, _stream(dev))
    _lib.check(status, "c2s_ltae_backward")
    res["_fold"] = (desc, cparams, keep, ws, ws_bytes)  # c2s_ltae_fold_backward reads the folded tensors of this workspace
    return res


def ltae_fold_backward(res: Dict[str, torch.Tensor], want: Dict[str, bool], shapes: Dict[str, tuple],
                       grad_pe_through_scores: bool = False) -> Dict[str, torch.Tensor]:
    """``c2s_ltae_fold_backward`` on the result of :func:`ltae_backward`: gradients of ``in_norm_weight/bias``,
    ``inconv_weight/bias`` (folded part), ``query``, ``key_weight``, ``key_bias`` -- the ones ``want`` names --
    as float32 tensors of ``shapes``.  ``grad_pe_through_scores``: also add grad_cpos . qk to ``res['grad_pe']``."""
    desc, cparams, keep, ws, ws_bytes = res["_fold"]
    dev = res["grad_u"].device
    io = _lib.LtaeFoldBwdIo(grad_u=res["grad_u"].data_ptr(), grad_cpos=res["grad_cpos"].data_ptr(),
                            grad_gamma_direct=_ptr(res.get("grad_gamma")), grad_beta_direct=_ptr(res.get("grad_beta")))
    out = {}
    for k in ("in_norm_weight", "in_norm_bias", "inconv_weight", "inconv_bias", "query", "key_weight", "key_bias"):
        if want.get(k):
            out[k] = torch.empty(shapes[k], dtype=torch.float32, device=dev)
            setattr(io, "grad_" + k, out[k].data_ptr())
    if grad_pe_through_scores and res.get("grad_pe") is not None:
        io.grad_pe = res["grad_pe"].data_ptr()
    with torch.cuda.device(dev):
        status = _lib.load().c2s_ltae_fold_backward(ctypes.byref(desc), ctypes.byref(cparams), ctypes.byref(io), ws.data_ptr(),
                                                    ws_bytes, _stream(dev))
    _lib.check(status, "c2s_ltae_fold_backward")
    return out


def ltae_mlp_backward(o_rows: torch.Tensor, grad_out: torch.Tensor, params: Dict[str, Optional[torch.Tensor]],
                      bn_mean: torch.Tensor, bn_var: torch.Tensor, spec: LtaeSpec, *,
                      mlp_keep: Optional[torch.Tensor] = None, y_rows: Optional[torch.Tensor] = None
                      ) -> Dict[str, torch.Tensor]:
    """``c2s_ltae_mlp_backward``: backward of mlp.0 / mlp.2 / ReLU / dropout / out_norm on the pixel rows.

    ``o_rows`` [B*H*W, d_model] are the rows saved by the forward, ``grad_out`` [B, c_out, H, W] the incoming gradient,
    ``bn_mean`` / ``bn_var`` the statistics the forward normalised with, ``y_rows`` [B*H*W, c_out] the pre-BatchNorm rows
    the training-mode forward saved (``save_y``; recomputed from ``o_rows`` when None).  Returns ``grad_o`` and the
    parameter gradients keyed like ``c2s_ltae_params``."""
    _require_cuda(grad_out, "grad_out")
    dev = grad_out.device
    b, co, h, w = grad_out.shape
    n = b * h * w
    c_out, d_model = spec.c_out, spec.d_model
    if co != c_out or tuple(o_rows.shape) != (n, d_model):
        raise RuntimeError(f"crop2seg_b200: grad_out {tuple(grad_out.shape)} / o_rows {tuple(o_rows.shape)} do not match")
    g = grad_out.contiguous()
    desc = _ltae_rows_desc(spec, b, h, w, _dtype_code(g, "grad_out"))
    keep = []
    cparams = _ltae_params(params, desc, dev, keep, mlp_keep=mlp_keep)
    f32 = dict(dtype=torch.float32, device=dev)
    cpad = (c_out + 3) // 4 * 4
    zeros = torch.zeros(c_out * d_model + 5 * cpad, dtype=torch.float32, device=dev)  # one memset for the six accumulators
    res = {"grad_o": torch.empty((n, d_model), **f32), "mlp_weight": zeros[:c_out * d_model].view(c_out, d_model)}
    for i, k in enumerate(("mlp_bias", "bn_weight", "bn_bias", "out_norm_weight", "out_norm_bias")):
        res[k] = zeros[c_out * d_model + i * cpad:c_out * d_model + i * cpad + c_out]
    o = o_rows.to(**f32).contiguous()
    mean, var = bn_mean.to(**f32).contiguous(), bn_var.to(**f32).contiguous()
    yr = None
    if y_rows is not None:
        if tuple(y_rows.shape) != (n, c_out):
            raise RuntimeError(f"crop2seg_b200: y_rows has shape {tuple(y_rows.shape)}, expected {(n, c_out)}")
        yr = y_rows.to(**f32).contiguous()
    io = _lib.LtaeMlpBwdIo(o_rows=o.data_ptr(), y_rows=_ptr(yr), grad_out=g.data_ptr(), bn_mean=mean.data_ptr(), bn_var=var.data_ptr(),
                           grad_o=res["grad_o"].data_ptr(), grad_mlp_weight=res["mlp_weight"].data_ptr(),
                           grad_mlp_bias=res["mlp_bias"].data_ptr(), grad_bn_weight=res["bn_weight"].data_ptr(),
                           grad_bn_bias=res["bn_bias"].data_ptr(), grad_out_norm_weight=res["out_norm_weight"].data_ptr(),
                           grad_out_norm_bias=res["out_norm_bias"].data_ptr())
    lib = _lib.load()
    with torch.cuda.device(dev):
        ws_bytes = lib.c2s_ltae_mlp_backward_workspace_bytes(ctypes.byref(desc))
        ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=dev)
        status = lib.c2s_ltae_mlp_backward(ctypes.byref(desc), ctypes.byref(cparams), ctypes.byref(io), ws.data_ptr(),
                                           ws_bytes, _stream(dev))
    _lib.check(status, "c2s_ltae_mlp_backward")
    return res


def ltae_inconv_grad(grad_o: torch.Tensor, zn_rows: torch.Tensor, sa_rows: Optional[torch.Tensor],
                     grad_weight: torch.Tensor, grad_bias: Optional[torch.Tensor], n_head: int) -> None:
    """``c2s_ltae_inconv_grad``: add the direct term of the in-projection gradient to ``grad_weight`` [d_model, C]
    (and ``grad_bias`` [d_model]) from ``grad_o`` [N, d_model], ``zn_rows`` [N, n_head, C], ``sa_rows`` [N, 16]."""
    dev = grad_o.device
    n, d_model = grad_o.shape
    c = zn_rows.shape[-1]
    for name, t in (("grad_o", grad_o), ("zn_rows", zn_rows), ("grad_weight", grad_weight)):
        if t.dtype != torch.float32 or not t.is_contiguous() or t.device != dev:
            raise RuntimeError(f"crop2seg_b200: {name} must be a contiguous float32 tensor on {dev}")
    if grad_bias is not None and (sa_rows is None or not sa_rows.is_contiguous() or not grad_bias.is_contiguous()):
        raise RuntimeError("crop2seg_b200: the bias gradient needs contiguous sa_rows / grad_bias")
    lib = _lib.load()
    with torch.cuda.device(dev):
        status = lib.c2s_ltae_inconv_grad(grad_o.data_ptr(), zn_rows.data_ptr(), _ptr(sa_rows), grad_weight.data_ptr(),
                                          _ptr(grad_bias), n, n_head, d_model, c, _stream(dev))
    _lib.check(status, "c2s_ltae_inconv_grad")
