"""``torch.autograd.Function``s of the hot path.

* ``AggregateFunction``: forward AND backward are CUDA kernels (``c2s_agg_forward`` / ``c2s_agg_backward``) --
  the aggregations move 97.7 % of the hot path's bytes.
* ``AggregateSkipConvFunction``: the aggregation fused with the decoder's skip convolution, BatchNorm frozen (running
  statistics); forward ``c2s_agg_skipconv_forward``, backward ``c2s_agg_skipconv_backward``, which recomputes the skip
  map on chip from x, so only the output is saved besides the inputs.
* ``LtaeFunction``: the forward is the fused CUDA kernel (train-mode BatchNorm statistics and injected dropout masks
  included).  The backward has three stages:
    M  ``c2s_ltae_mlp_backward`` (CUDA, ``csrc/c2s_ltae_mlp_bwd.cu``): the rows after the attention (MLP Linear,
       BatchNorm, ReLU, dropout mask, output GroupNorm on [N, 256] / [N, c_out] rows, N = B*H*W);
    A  ``c2s_ltae_backward`` (CUDA, ``csrc/c2s_ltae_bwd.cu``) does everything that touches the [N, T, C] features:
       it recomputes the attention, back-propagates through the value sums, the softmax, the scores and the input
       GroupNorm, writes grad_x and reduces the gradients of the folded score weights U[C,16] and cpos[B,T,16];
    F  ``c2s_ltae_fold_backward`` (CUDA, ``csrc/c2s_ltae_fold_bwd.cu``, two launches on stage A's workspace): the
       chain from (grad_U, grad_cpos) to the state_dict tensors (Q, fc1_k, inconv, in_norm) -- the adjoint of the
       weight folding of ``csrc/c2s_ltae_prep.cu`` -- plus ``c2s_ltae_inconv_grad`` for the direct in-projection
       terms.  Only LEARNABLE positional tables (use_doy / use_abs_rel_enc / add_linear) add torch autograd of the
       [B, T, 256] table construction.
  No [N, T, D] activation is ever materialised.  There is no torch fallback: encoders without ``inconv``
  (d_model=None) and output GroupNorm groups wider than 16 channels raise in training (forward-only support).
"""
from __future__ import annotations

from typing import Dict

import torch
import torch.nn.functional as F

from . import _lib, ops


class AggregateFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, attn, pad_mask, mode):
        ctx.mode = mode
        ctx.save_for_backward(x, attn, pad_mask)
        return ops.temporal_aggregate_forward(x, pad_mask, attn, mode)

    @staticmethod
    def backward(ctx, grad_out):
        x, attn, pad = ctx.saved_tensors
        gx, gattn = ops.temporal_aggregate_backward(x, pad, attn, grad_out, ctx.mode, need_x=ctx.needs_input_grad[0],
                                                    need_attn=ctx.needs_input_grad[1])
        return gx, gattn, None, None


class AggregateSkipConvFunction(torch.autograd.Function):
    """apply(x, attn, pad_mask, conv_weight, conv_bias, bn_weight, bn_bias, bn_running_mean, bn_running_var, bn_eps)"""

    @staticmethod
    def forward(ctx, x, attn, pad_mask, conv_weight, conv_bias, bn_weight, bn_bias, bn_running_mean, bn_running_var, bn_eps):
        out = ops.temporal_aggregate_skip_conv_forward(x, pad_mask, attn, conv_weight, conv_bias, bn_weight, bn_bias,
                                                       bn_running_mean, bn_running_var, bn_eps)
        ctx.bn_eps = bn_eps
        ctx.save_for_backward(x, attn, pad_mask, conv_weight, conv_bias, bn_weight, bn_bias, bn_running_mean,
                              bn_running_var, out)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        x, attn, pad, cw, cb, bw, bb, rm, rv, out = ctx.saved_tensors
        need = [ctx.needs_input_grad[i] for i in (0, 1, 3, 4, 5, 6)]
        gx, gattn, gcw, gcb, gbw, gbb = ops.temporal_aggregate_skip_conv_backward(
            x, pad, attn, cw, cb, bw, bb, rm, rv, ctx.bn_eps, out, grad_out, need=need)

        def cast(g, p):
            return None if g is None else g.to(p.dtype)
        return (gx, cast(gattn, attn), None, cast(gcw, cw), cast(gcb, cb), cast(gbw, bw), cast(gbb, bb), None, None, None)


# ------------------------------------------------------------------------------------------------------------
# positional table [B,T,D] on the device: stage F needs it (and its autograd graph for learnable tables)
# ------------------------------------------------------------------------------------------------------------
def _positional(spec: ops.LtaeSpec, P: Dict[str, torch.Tensor], positions: torch.Tensor):
    """[B,T,D] positional table (identical for every pixel of a sample; positional_encoding.py:25-73)."""
    h, d = spec.n_head, spec.d_model // spec.n_head

    def doy(pos, w, b):
        idx = pos.to(torch.int64).clamp(0, 364)
        return (w.t()[idx] + b).repeat(1, 1, h)

    def primary(pos):
        if spec.pe_mode == _lib.PE_DOY_TABLE:
            return doy(pos, P["pe_fc_weight"], P["pe_fc_bias"])
        table = pos.to(torch.float32)[:, :, None] / P["pe_denom"][None, None, :]
        enc = torch.where((torch.arange(d, device=table.device) % 2 == 0)[None, None, :], torch.sin(table), torch.cos(table))
        enc = enc.repeat(1, 1, h)
        if spec.pe_mode == _lib.PE_SINUSOID_LINEAR:
            enc = F.linear(enc, P["pe_fc_weight"], P["pe_fc_bias"])
        return enc

    if spec.pe_abs:
        return primary(positions[..., 0]) + doy(positions[..., 1], P["pe_abs_fc_weight"], P["pe_abs_fc_bias"])
    return primary(positions)


_GRAD_PARAM_ORDER = tuple(_lib.LTAE_PARAM_FIELDS)


def _cuda_backward(ctx, spec, x, positions, pad_mask, attn_keep, mlp_keep, params, g_out, g_attn):
    b, t, c, hh, ww = x.shape
    n, h, D = b * hh * ww, spec.n_head, spec.d_model
    need = dict(zip(_GRAD_PARAM_ORDER, ctx.needs_input_grad[6:]))
    raw = dict(zip(_GRAD_PARAM_ORDER, params))
    attn_only = spec.attn_only
    grads: Dict[str, torch.Tensor] = {}

    # ---- stage M: rows after the attention (c2s_ltae_mlp_backward) ---------------------------------------------
    g_o = None
    if not attn_only:
        if g_out is None:
            g_o = torch.zeros((n, D), dtype=torch.float32, device=x.device)
        else:
            if spec.c_out // h > 16:
                raise _lib.C2SError(f"crop2seg_b200: L-TAE backward supports out_norm groups of at most 16 channels "
                                    f"(mlp[-1]={spec.c_out}, n_head={h}); there is no torch fallback")
            if spec.bn_batch_stats:
                mean, var = ctx.bn_stats
            else:
                mean, var = raw["bn_running_mean"], raw["bn_running_var"]
            m_res = ops.ltae_mlp_backward(ctx.o_rows, g_out.to(x.dtype), raw, mean, var, spec, mlp_keep=mlp_keep,
                                          y_rows=ctx.y_rows)
            g_o = m_res["grad_o"]
            for k in ("mlp_weight", "mlp_bias", "bn_weight", "bn_bias", "out_norm_weight", "out_norm_bias"):
                if need[k]:
                    grads[k] = m_res[k]

    # ---- stage A: the CUDA kernel over the features ------------------------------------------------------------
    if attn_only and g_attn is None:  # LTAE4WTAE whose attention received no gradient: everything upstream is zero
        gx = torch.zeros_like(x) if ctx.needs_input_grad[0] else None
        gparams = [torch.zeros_like(p) if (p is not None and need[k]) else None for k, p in zip(_GRAD_PARAM_ORDER, params)]
        return (gx, None, None, None, None, None, *gparams)
    pe_learnable = any(need.get(k) for k in ("pe_fc_weight", "pe_fc_bias", "pe_abs_fc_weight", "pe_abs_fc_bias"))
    res = ops.ltae_backward(x, positions, pad_mask, raw, g_o, g_attn, spec, attn_keep=attn_keep,
                            need_grad_pe=pe_learnable)

    # ---- stage F: folded quantities -> state_dict tensors (the adjoint of csrc/c2s_ltae_prep.cu, written out) -----
    front = ("in_norm_weight", "in_norm_bias", "inconv_weight", "inconv_bias", "query", "key_weight", "key_bias",
             "pe_fc_weight", "pe_fc_bias", "pe_abs_fc_weight", "pe_abs_fc_bias")
    if any(need.get(k) for k in front):
        with torch.no_grad():
            # one call (two launches) on the workspace of stage A; the in-projection's direct term is added by
            # c2s_ltae_inconv_grad (one launch over the rows)
            want = {k: bool(need.get(k)) for k in front[:7]}
            shapes = {k: tuple(raw[k].shape) for k in front[:7] if raw.get(k) is not None}
            pe_learnable_now = pe_learnable and spec.pe_mode != _lib.PE_NONE
            if pe_learnable_now and res["grad_pe"] is None:  # attention-only encoders: the table acts through the scores only
                res["grad_pe"] = torch.zeros((b, t, D), dtype=torch.float32, device=x.device)
            folded = ops.ltae_fold_backward(res, want, shapes, grad_pe_through_scores=pe_learnable_now)
            g_pe = res["grad_pe"]
            if not attn_only and (need["inconv_weight"] or need["inconv_bias"]):
                g_wc = folded["inconv_weight"].view(D, c) if need["inconv_weight"] else torch.zeros((D, c), dtype=torch.float32, device=x.device)
                g_wb = folded.get("inconv_bias")
                ops.ltae_inconv_grad(g_o.contiguous(), res["zn_rows"].contiguous(), res["sa_rows"].contiguous(), g_wc,
                                     g_wb, h)
            grads.update(folded)
        pe_names = [k for k in ("pe_fc_weight", "pe_fc_bias", "pe_abs_fc_weight", "pe_abs_fc_bias")
                    if need.get(k) and raw[k] is not None]
        if pe_names and g_pe is not None:  # learnable tables / add_linear: the small table graph through autograd
            with torch.enable_grad():
                L = {k: (v.detach().float().requires_grad_(k in pe_names) if v is not None and v.is_floating_point() else v)
                     for k, v in raw.items()}
                got = torch.autograd.grad(_positional(spec, L, positions), [L[k] for k in pe_names], g_pe,
                                          allow_unused=True)
            for k, gk in zip(pe_names, got):
                if gk is not None:
                    grads[k] = gk
    gx = res["grad_x"] if ctx.needs_input_grad[0] else None
    gparams = []
    for k, p in zip(_GRAD_PARAM_ORDER, params):
        g = grads.get(k)
        gparams.append(None if g is None or p is None or not need[k] else g.to(p.dtype).reshape(p.shape))
    return (gx, None, None, None, None, None, *gparams)


class LtaeFunction(torch.autograd.Function):
    """apply(x, positions, pad_mask, attn_keep, mlp_keep, spec, *params in LTAE_PARAM_FIELDS order)
    -> (out | None, attn, bn_batch_mean | None, bn_batch_var | None)"""

    @staticmethod
    def forward(ctx, x, positions, pad_mask, attn_keep, mlp_keep, spec, *params):
        P = dict(zip(_GRAD_PARAM_ORDER, params))
        # d_model=None (tae.py:398-403: no inconv) is served in the forward only; the reference's shipped models always
        # build the in-projection (utae.py:179-189, wtae.py:196-207, timeunet.py:155-164).  backward() raises for it.
        ctx.cuda_backward = bool(spec.has_inconv)
        # with save_y the pre-BatchNorm rows of a training-mode forward are kept: the backward does not recompute them
        out, attn, stats, ctx.o_rows, ctx.y_rows = ops.ltae_forward(
            x, positions, pad_mask, P, spec, attn_keep=attn_keep, mlp_keep=mlp_keep, save_o=ctx.cuda_backward,
            save_y=ctx.cuda_backward)
        ctx.spec = spec
        # the running statistics are updated in place right after a training-mode forward and are not needed by
        # its backward (batch statistics are recomputed), so they are not saved in that case
        skip = ("bn_running_mean", "bn_running_var") if spec.bn_batch_stats else ()
        params = [None if name in skip else p for name, p in zip(_GRAD_PARAM_ORDER, params)]
        ctx.present = [p is not None for p in params]
        ctx.opt = (positions, pad_mask, attn_keep, mlp_keep)
        ctx.save_for_backward(x, *[p for p in params if p is not None])
        mean, var = stats if stats is not None else (None, None)
        ctx.bn_stats = stats  # batch statistics the forward normalised with (training mode)
        if stats is not None:
            ctx.mark_non_differentiable(mean, var)
        return out, attn, mean, var

    @staticmethod
    def backward(ctx, *grads):
        saved = ctx.saved_tensors
        x, rest = saved[0], list(saved[1:])
        positions, pad_mask, attn_keep, mlp_keep = ctx.opt
        params = [rest.pop(0) if present else None for present in ctx.present]
        g_out, g_attn = grads[0], grads[1]
        if not ctx.cuda_backward:
            raise _lib.C2SError("crop2seg_b200: the L-TAE backward needs the in-projection (d_model is not None); "
                                "there is no torch fallback for encoders without inconv")
        return _cuda_backward(ctx, ctx.spec, x, positions, pad_mask, attn_keep, mlp_keep, params, g_out, g_attn)
