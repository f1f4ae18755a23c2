"""torch-CPU restatement of the reference L-TAE + TemporalAggregator.  TEST INFRASTRUCTURE ONLY.

Second oracle and the CPU baseline of ``bench.py``: it issues the ATen library calls the reference
modules make (GroupNorm, 1x1 Conv1d, Linear, matmul, softmax, bilinear Upsample -- SURVEY.md section 8c
lists the call sites) including the reference's materialising copies (one query per pixel row, head-major mask
and value copies), written functionally over a ``state_dict``-keyed parameter dict, so its speed on
the host cores is representative of the reference's own CPU path (the reference itself lives in
``/root/reference`` and cannot travel to the GPU box).  Like the numpy oracle it follows the as-written
algorithm, including the [N,T,D] activations and head-major copies the fused kernels avoid.

    LTAE.forward / LTAE4WTAE.forward    src/backbones/tae.py:451-504, 589-635
    LightweightMultiHeadAttention       src/backbones/tae.py:760-807
    ScaledDotProductAttention           src/backbones/tae.py:822-847
    PositionalEncoder / Absolute...     src/backbones/positional_encoding.py:25-43, 58-73
    TemporalAggregator.forward          src/backbones/temporal_aggregator.py:14-77

Parity status: pinned against the committed reference outputs (tests/test_oracle_golden.py).

Precision: float32 unless x is float64; then, with float64 parameters, every step runs in float64 on x's device, which
makes it the high-precision reference of the kernels' tests (tests/test_gpu_training_float64.py).
"""
from __future__ import annotations

from typing import Dict, Optional

import torch
import torch.nn.functional as F


def _t(a) -> torch.Tensor:
    return a if isinstance(a, torch.Tensor) else torch.from_numpy(a)


def _real(a) -> torch.Tensor:
    """float64 stays float64 (a high-precision reference), every other type computes in float32."""
    a = _t(a)
    return a if a.dtype == torch.float64 else a.float()


def _sinusoid(pos_rows, denom, repeat, fc_w=None, fc_b=None):
    # positional_encoding.py:29-31; the reference's denom is a float32 attribute, so the angle is a float32 quotient
    # even where the rest of the table is computed in float64
    table = (pos_rows[:, :, None] / denom[None, None, :].float()).to(denom.dtype)
    table[:, :, 0::2] = torch.sin(table[:, :, 0::2])
    table[:, :, 1::2] = torch.cos(table[:, :, 1::2])
    table = table.repeat(1, 1, repeat)  # :35-38
    return F.linear(table, fc_w, fc_b) if fc_w is not None else table  # :39-41


def _doy(pos_rows, fc_w, fc_b, repeat):
    onehot = F.one_hot(pos_rows.to(torch.int64), num_classes=365).to(fc_w.dtype)  # positional_encoding.py:63
    return F.linear(onehot, fc_w, fc_b).repeat(1, 1, repeat)  # :66-71


def ltae_forward_torch(cfg, params: Dict, x, positions=None, pad_mask=None, attn_only: bool = False,
                       training: bool = False, attn_keep=None, mlp_keep=None, attn_drop_p: float = 0.1,
                       mlp_drop_p: float = 0.2, materialise: bool = True):
    """``LTAE.forward`` (or ``LTAE4WTAE.forward`` with ``attn_only``), differentiable, on x's device and precision.

    ``cfg`` is an ``oracle.LtaeConfig``; ``params`` is keyed like the reference ``state_dict``.
    ``training``: BatchNorm1d batch statistics (tae.py:445) and the two dropouts with INJECTED keep masks (torch's
    generator cannot be matched by a kernel): ``attn_keep`` uint8/bool [n_head, B, T, H, W] applied to the attention
    before it is returned (tae.py:837), ``mlp_keep`` [B, c_out, H, W] after the ReLU (tae.py:448); a missing mask means
    no dropout.  Training mode returns ``(out, attn, (batch_mean, biased_batch_var))``.
    ``materialise``: make the copies the reference makes (``torch.stack`` of one query per pixel row, tae.py:764;
    ``pad_mask.repeat``, :772) so that the CPU timing is the reference's, not a cheaper one.
    """
    p = {k: _t(v) for k, v in params.items()}
    x = _real(x)
    b, t, c, hh, ww = x.shape
    h, dk, d = cfg.n_head, cfg.d_k, cfg.width
    rows = x.permute(0, 3, 4, 1, 2).reshape(b * hh * ww, t, c)  # tae.py:460
    n = rows.shape[0]
    pad_rows = None
    if pad_mask is not None:
        pad_rows = _t(pad_mask).to(x.device).bool()[:, None, None, :].expand(b, hh, ww, t).reshape(n, t)  # :453-457
    e = F.group_norm(rows.permute(0, 2, 1), h, p["in_norm.weight"], p["in_norm.bias"], 1e-5)  # :461  [N,C,T]
    if cfg.d_model is not None:
        e = F.conv1d(e, p["inconv.weight"], p["inconv.bias"])  # :463-464
    e = e.permute(0, 2, 1)  # [N,T,D]
    if cfg.positional_encoding:
        pos = _t(positions).to(x.device)

        def per_pixel(q):
            return q[:, None, None, :].expand(b, hh, ww, t).reshape(n, t)

        def primary(q):
            if cfg.use_doy and not cfg.add_linear:
                return _doy(q, p["positional_encoder.fc.weight"], p["positional_encoder.fc.bias"], h)
            return _sinusoid(q, p["positional_encoder.denom"], h,
                             p.get("positional_encoder.fc.weight") if cfg.add_linear else None,
                             p.get("positional_encoder.fc.bias") if cfg.add_linear else None)

        if cfg.use_abs_rel_enc:  # :467-474
            e = e + primary(per_pixel(pos[..., 0])) + _doy(per_pixel(pos[..., 1]),
                                                           p["positional_encoder_abs.fc.weight"],
                                                           p["positional_encoder_abs.fc.bias"], h)
        else:
            e = e + primary(per_pixel(pos))  # :476-479
    # LightweightMultiHeadAttention, num_queries == 1 (tae.py:760-807)
    if materialise:
        q = torch.stack([p["attention_head.Q"] for _ in range(n)], dim=1).view(-1, 1, dk)  # :764-766
    else:
        q = p["attention_head.Q"].reshape(h, 1, 1, dk).expand(h, n, 1, dk).reshape(h * n, 1, dk)
    k = F.linear(e, p["attention_head.fc1_k.weight"], p["attention_head.fc1_k.bias"]).view(n, t, h, dk)
    k = k.permute(2, 0, 1, 3).reshape(h * n, t, dk)
    v = torch.stack(e.split(d // h, dim=-1)).reshape(h * n, t, d // h)
    s = torch.matmul(q, k.transpose(1, 2)) / (dk ** 0.5)  # :827-828
    if pad_rows is not None:
        s = s.masked_fill(pad_rows.repeat(h, 1).unsqueeze(1), -1e6)  # :831
    a = torch.softmax(s, dim=2)  # :836
    if training and attn_keep is not None:  # :837 nn.Dropout(0.1): zero and rescale, BEFORE the attention is returned
        ak = _t(attn_keep).to(device=a.device, dtype=a.dtype).permute(0, 1, 3, 4, 2).reshape(h * n, 1, t)
        a = a * ak / (1.0 - attn_drop_p)
    attn = a.view(h, b, hh, ww, t).permute(0, 1, 4, 2, 3).contiguous()  # :490-493
    if attn_only:
        return attn
    o = torch.matmul(a, v).view(h, n, d // h).permute(1, 0, 2).reshape(n, d)  # :839, :796-798
    y = F.linear(o, p["mlp.0.weight"], p["mlp.0.bias"])  # :443
    stats = None
    if training:  # :445 batch statistics over all B*H*W rows (biased variance normalises)
        stats = (y.mean(dim=0).detach(), y.var(dim=0, unbiased=False).detach())
        y = F.batch_norm(y, None, None, p["mlp.2.weight"], p["mlp.2.bias"], True, 0.1, 1e-5)
    else:
        y = F.batch_norm(y, p["mlp.2.running_mean"], p["mlp.2.running_var"], p["mlp.2.weight"], p["mlp.2.bias"],
                         False, 0.1, 1e-5)  # :445 (eval)
    y = F.relu(y)  # :447
    if training and mlp_keep is not None:  # :448 nn.Dropout(0.2)
        mk = _t(mlp_keep).to(device=y.device, dtype=y.dtype).permute(0, 2, 3, 1).reshape(n, -1)
        y = y * mk / (1.0 - mlp_drop_p)
    y = F.group_norm(y[:, :, None], h, p["out_norm.weight"], p["out_norm.bias"], 1e-5)[:, :, 0]  # :488
    out = y.view(b, hh, ww, -1).permute(0, 3, 1, 2).contiguous()  # :494
    if training:
        return out, attn, stats
    return out, attn


def temporal_aggregator_torch(x, pad_mask=None, attn_mask=None, mode: str = "att_group"):
    """``TemporalAggregator(mode).forward`` (temporal_aggregator.py:14-77) on x's device and precision."""
    x = _real(x)
    b, t, c, hh, ww = x.shape
    keep = None
    if pad_mask is not None and bool(_t(pad_mask).any()):
        keep = (~_t(pad_mask).to(x.device).bool()).to(x.dtype)
    if mode == "mean":
        if keep is None:
            return x.mean(dim=1)
        return (x * keep[:, :, None, None, None]).sum(dim=1) / keep.sum(dim=1)[:, None, None, None]
    attn = _real(attn_mask)
    nh = attn.shape[0]
    if mode == "att_mean":
        a = F.interpolate(attn.mean(dim=0), size=(hh, ww), mode="bilinear", align_corners=False)
        if keep is not None:
            a = a * keep[:, :, None, None]
        return (x * a[:, :, None]).sum(dim=1)
    a = attn.reshape(nh * b, t, *attn.shape[-2:])
    if hh > attn.shape[-1]:
        a = F.interpolate(a, size=(hh, ww), mode="bilinear", align_corners=False)  # :17-19, :27
    else:
        a = F.avg_pool2d(a, kernel_size=attn.shape[-1] // hh)  # :29
    a = a.view(nh, b, t, hh, ww)
    if keep is not None:
        a = a * keep[None, :, :, None, None]  # :33
    xg = torch.stack(x.chunk(nh, dim=2))  # :35
    return torch.cat(list((a[:, :, :, None] * xg).sum(dim=2)), dim=1)  # :37-44
