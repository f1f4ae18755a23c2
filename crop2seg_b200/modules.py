"""Drop-in ``nn.Module``s for the temporal-attention bottleneck of Many98/Crop2Seg.

Same constructor arguments, ``forward`` signatures, return shapes and ``state_dict`` keys as the
reference classes (SURVEY.md section 8b):

    LTAE                src/backbones/tae.py:349-504
    LTAE4WTAE           src/backbones/tae.py:507-635
    TemporalAggregator  src/backbones/temporal_aggregator.py:6-77

The sub-modules below (``nn.Conv1d``, ``nn.Linear``, ``nn.GroupNorm``, ``nn.BatchNorm1d``) only hold
parameters, so that ``load_state_dict`` (train.py:428, prediction.py:225) and
``model.apply(weight_init)`` (train.py:450) keep working; their own ``forward`` is never called.
All arithmetic runs in the CUDA library (``ops.py``); there is no fallback.
"""
from __future__ import annotations

import copy
import dataclasses
from typing import List, Optional

import numpy as np
import torch
import torch.nn as nn

from . import _lib, ops


#: ScaledDotProductAttention(attn_dropout=0.1) -- tae.py:816-819; applied only in training mode
ATTENTION_DROPOUT = 0.1

_injected_masks = None


class injected_dropout:
    """``with injected_dropout(attn_keep, mlp_keep): module(x, ...)`` -- training-mode forwards inside the block use
    these keep masks (uint8/bool, ``attn_keep`` [n_head,B,T,H,W], ``mlp_keep`` [B,C',H,W] or None) instead of drawing
    them.  Parity tests replay the reference's own dropout realisation this way (tests/golden/make_train_golden.py)."""

    def __init__(self, attn_keep, mlp_keep=None):
        self.masks = (attn_keep, mlp_keep)

    def __enter__(self):
        global _injected_masks
        self.old, _injected_masks = _injected_masks, self.masks
        return self

    def __exit__(self, *exc):
        global _injected_masks
        _injected_masks = self.old


def _draw_keep(shape, p, device, which):
    """uint8 keep mask of a dropout with rate p (None when p == 0), or the injected one."""
    if p <= 0:
        return None
    if _injected_masks is not None and _injected_masks[which] is not None:
        m = _injected_masks[which]
        if tuple(m.shape) != tuple(shape):
            raise RuntimeError(f"crop2seg_b200: injected dropout mask has shape {tuple(m.shape)}, expected {tuple(shape)}")
        return m.to(device=device, dtype=torch.uint8)
    # one launch (Philox Bernoulli straight into the uint8 mask) instead of rand + compare + cast
    return torch.empty(shape, dtype=torch.uint8, device=device).bernoulli_(1.0 - p)


#: construction-time defaults of the encoder attributes, set by ``crop2seg_b200.install(...)``
_DEFAULTS = {"assume_zero_padded": False, "return_attention": True}


class _Placeholder(nn.Module):
    """Parameter-free stand-in for einops' ``Rearrange`` inside ``mlp`` (keeps the indices 0..5)."""

    def forward(self, x):  # pragma: no cover - never called
        return x


class PositionalEncoder(nn.Module):
    """Parameter holder for the sinusoidal encoder (positional_encoding.py:7-43)."""

    def __init__(self, d_model, T=1000, repeat=None, offset=0, add_linear=False):
        super().__init__()
        self.d = d_model
        self.T = T
        self.repeat = repeat
        # plain attribute, not a buffer: absent from the reference state_dict too (positional_encoding.py:16-18)
        self.denom = torch.pow(T, 2 * (torch.arange(offset, offset + d_model).float() // 2) / d_model)
        self.add_linear = add_linear
        if add_linear:
            width = d_model * repeat if repeat is not None else d_model
            self.fc = nn.Linear(width, width)


class AbsolutePositionalEncoder(nn.Module):
    """Parameter holder for the day-of-year encoder (positional_encoding.py:46-73)."""

    def __init__(self, d_model: int, repeat=None):
        super().__init__()
        self.d = d_model
        self.repeat = repeat
        self.fc = nn.Linear(365, d_model)


class LightweightMultiHeadAttention(nn.Module):
    """Parameter holder: learned master query ``Q`` and key projection ``fc1_k`` (tae.py:744-757)."""

    def __init__(self, n_head, d_k, d_in, n=1):
        super().__init__()
        self.n_head, self.d_k, self.d_in, self.n = n_head, d_k, d_in, n
        self.Q = nn.Parameter(torch.zeros((n_head, n, d_k))).requires_grad_(True)
        nn.init.normal_(self.Q, mean=0, std=np.sqrt(2.0 / d_k))
        self.fc1_k = nn.Linear(d_in, n_head * d_k)
        nn.init.normal_(self.fc1_k.weight, mean=0, std=np.sqrt(2.0 / d_k))


class _LTAEBase(nn.Module):
    """Shared construction of the encoder front end (tae.py:387-435 / 540-587)."""

    def _build_front(self, in_channels, n_head, d_k, d_model, positional_encoding, use_abs_rel_enc, num_queries,
                     use_doy, add_linear, T=1000):
        self.in_channels = in_channels
        self.n_head = n_head
        self.d_k = d_k
        self.num_queries = num_queries
        self.use_abs_rel_enc = use_abs_rel_enc
        self.add_linear = add_linear
        if d_model is not None:
            self.d_model = d_model
            self.inconv = nn.Conv1d(in_channels, d_model, 1)
        else:
            self.d_model = in_channels
            self.inconv = None
        if positional_encoding:
            if use_doy and not add_linear:
                self.positional_encoder = AbsolutePositionalEncoder(self.d_model // n_head, repeat=n_head)
            else:
                # the reference never forwards its own T (tae.py:409-419): the encoder's period is always 1000
                self.positional_encoder = PositionalEncoder(self.d_model // n_head, repeat=n_head,
                                                            add_linear=add_linear)
            if use_abs_rel_enc:
                self.positional_encoder_abs = AbsolutePositionalEncoder(self.d_model // n_head, repeat=n_head)
        else:
            self.positional_encoder = None
        self.attention_head = LightweightMultiHeadAttention(n_head=n_head, d_k=d_k, d_in=self.d_model, n=num_queries)
        self.in_norm = nn.GroupNorm(num_groups=n_head, num_channels=in_channels)
        #: set by the caller (``crop2seg_b200.install(assume_zero_padded=True)`` does it for every encoder it builds)
        #: when padded frames of x are exactly zero, as ``smart_forward`` guarantees with pad_value=0
        #: (temp_shared_block.py:30-40); padded frames are then not read
        self.assume_zero_padded = _DEFAULTS["assume_zero_padded"]
        #: model-level ``return_att`` (utae.py:200, timeunet.py:169) is not visible to the encoder: a caller that never
        #: consumes the attention (``TimeUNet_v1.forward`` drops it unless return_att, timeunet.py:178-205) sets this to
        #: False and ``forward`` then skips the [n_head,B,T,H,W] store and returns ``(out, None)``
        self.return_attention = _DEFAULTS["return_attention"]
        #: eval mode keeps the folded weights between calls while no parameter changes (``Tensor._version`` and
        #: ``data_ptr`` of every tensor the kernels read); writes through ``.data`` bypass the version counters -- call
        #: ``invalidate_folded_weights()`` after those, or set this to False
        self.cache_folded_weights = True
        self._folded_cache = {}

    def invalidate_folded_weights(self):
        """Forget the cached weight preparation (needed only after parameter writes that bypass autograd's version
        counters, e.g. ``p.data.copy_(...)`` between two eval-mode calls)."""
        self._folded_cache.clear()

    def _apply(self, fn, *args, **kwargs):  # .to() / .cuda() / .half(): new storages
        self._folded_cache.clear()
        return super()._apply(fn, *args, **kwargs)

    def _load_from_state_dict(self, *args, **kwargs):
        self._folded_cache.clear()
        return super()._load_from_state_dict(*args, **kwargs)

    def _folded_args(self, params):
        """kwargs for ops.ltae_forward: reuse of the weight-only preparation in eval mode, keyed on the tensors of
        ``params`` (the ones the kernels read)."""
        if self.training or not self.cache_folded_weights:
            return {}
        key = tuple((t._version, t.data_ptr()) for t in params.values() if t is not None)
        return {"folded_cache": self._folded_cache, "folded_key": key}

    # -- helpers ---------------------------------------------------------------------------------
    def _pe_mode(self) -> int:
        pe = self.positional_encoder
        if pe is None:
            return _lib.PE_NONE
        if isinstance(pe, AbsolutePositionalEncoder):
            return _lib.PE_DOY_TABLE
        return _lib.PE_SINUSOID_LINEAR if pe.add_linear else _lib.PE_SINUSOID

    def _needs_grad(self, x) -> bool:
        return torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters()))

    def _spec(self) -> ops.LtaeSpec:
        """The encoder's configuration for one forward; training mode selects BatchNorm batch statistics and dropout."""
        mlp = {}
        if isinstance(self, LTAE):
            bn = self.mlp[2]
            mlp = dict(c_out=self._widths[-1], bn_batch_stats=self.training or not bn.track_running_stats,
                       bn_eps=bn.eps, mlp_drop_p=float(self.mlp[5].p) if self.training else 0.0)
        return ops.LtaeSpec(n_head=self.n_head, d_k=self.d_k, d_model=self.d_model, has_inconv=self.inconv is not None,
                            pe_mode=self._pe_mode(), pe_abs=bool(self.use_abs_rel_enc),
                            attn_only=not isinstance(self, LTAE), zero_padded=bool(self.assume_zero_padded),
                            gn_eps=self.in_norm.eps, attn_drop_p=ATTENTION_DROPOUT if self.training else 0.0, **mlp)

    def _params(self, device):
        """The tensors of ``c2s_ltae_params``, keyed by its field names (the MLP, BatchNorm and out_norm ones for LTAE)."""
        p = {
            "in_norm_weight": self.in_norm.weight, "in_norm_bias": self.in_norm.bias,
            "query": self.attention_head.Q, "key_weight": self.attention_head.fc1_k.weight,
            "key_bias": self.attention_head.fc1_k.bias,
        }
        if self.inconv is not None:
            p["inconv_weight"] = self.inconv.weight.view(self.d_model, self.in_channels)
            p["inconv_bias"] = self.inconv.bias
        pe = self.positional_encoder
        if pe is not None:
            if isinstance(pe, PositionalEncoder):
                if pe.denom.device != device:  # lazily moved like positional_encoding.py:26-28
                    pe.denom = pe.denom.to(device)
                p["pe_denom"] = pe.denom
                if pe.add_linear:
                    p["pe_fc_weight"], p["pe_fc_bias"] = pe.fc.weight, pe.fc.bias
            else:
                p["pe_fc_weight"], p["pe_fc_bias"] = pe.fc.weight, pe.fc.bias
            if self.use_abs_rel_enc:
                p["pe_abs_fc_weight"] = self.positional_encoder_abs.fc.weight
                p["pe_abs_fc_bias"] = self.positional_encoder_abs.fc.bias
        if isinstance(self, LTAE):
            lin, bn = self.mlp[0], self.mlp[2]
            p.update({
                "mlp_weight": lin.weight, "mlp_bias": lin.bias, "bn_weight": bn.weight, "bn_bias": bn.bias,
                "bn_running_mean": bn.running_mean, "bn_running_var": bn.running_var,
                "out_norm_weight": self.out_norm.weight, "out_norm_bias": self.out_norm.bias,
            })
        return p

    def _check_inputs(self, x, batch_positions):
        if self.num_queries != 1 and (self.training or not isinstance(self, LTAE)):
            # num_queries > 1 (tae.py:495-499) is served in eval mode by one pass per query (LTAE.forward); in training
            # mode the reference's BatchNorm1d statistics run over the rows of ALL queries at once, which a per-query
            # pass cannot reproduce.  Every shipped reference model crashes for it in the aggregator anyway
            # (temporal_aggregator.py:23, SURVEY.md section 8a-v).
            raise NotImplementedError("crop2seg_b200: num_queries > 1 is supported by LTAE in eval mode only")
        if x.shape[2] != self.in_channels:
            raise RuntimeError(f"Expected {self.in_channels} input channels, got x of shape {tuple(x.shape)}")
        if self.positional_encoder is not None and batch_positions is not None:
            doy = None
            if isinstance(self.positional_encoder, AbsolutePositionalEncoder):
                doy = batch_positions[..., 0] if self.use_abs_rel_enc else batch_positions
            if self.use_abs_rel_enc:
                doy2 = batch_positions[..., 1]
                doy = doy2 if doy is None else torch.stack([doy, doy2])
            if doy is not None and not doy.is_cuda:
                # F.one_hot raises for day indices outside [0, 364] (positional_encoding.py:63); checking a
                # device tensor would force a host sync, so only host-side positions are validated here
                if doy.numel() and (int(doy.min()) < 0 or int(doy.max()) > 364):
                    raise RuntimeError("Class values must be smaller than num_classes.")


class LTAE(_LTAEBase):
    """Lightweight Temporal Attention Encoder -- drop-in for ``src.backbones.tae.LTAE`` (tae.py:349)."""

    def __init__(self, in_channels=128, n_head=16, d_k=4, mlp=[256, 128], dropout=0.2, d_model=256, T=1000,
                 positional_encoding=True, use_abs_rel_enc=False, use_doy=False, num_queries=1, add_linear=False,
                 *args, **kwargs):
        super().__init__()
        widths: List[int] = copy.deepcopy(mlp)
        # the reference never forwards its T argument to the positional encoder (tae.py:409-419): period 1000 always
        self._build_front(in_channels, n_head, d_k, d_model, positional_encoding, use_abs_rel_enc, num_queries,
                          use_doy, add_linear)
        self.T = T
        assert widths[0] == self.d_model  # tae.py:404
        self.out_norm = nn.GroupNorm(num_groups=n_head, num_channels=widths[-1])
        self.mlp = nn.Sequential(
            nn.Linear(widths[0], widths[1]),
            _Placeholder(),
            nn.BatchNorm1d(widths[1]),
            _Placeholder(),
            nn.ReLU(),
            nn.Dropout(dropout),
        )
        self._widths = widths

    def forward(self, x, batch_positions=None, pad_mask=None, return_comp=False, return_att=None):
        """x[B,T,C,H,W] -> (out[B,C',H,W], attn[n_head,B,T,H,W]); ``return_comp`` is ignored as in tae.py:451.

        ``return_att=False`` (extension; default: the module's ``return_attention`` attribute) skips the attention
        store and returns ``(out, None)``.
        Training mode follows the reference: BatchNorm1d batch statistics (+ running-stat update), dropout on the
        attention before it is returned (tae.py:837) and after the MLP's ReLU (tae.py:448); the masks are drawn with
        torch's generator here and injected into the kernel.
        """
        self._check_inputs(x, batch_positions)
        if return_att is None:
            return_att = self.return_attention
        if self.num_queries != 1:
            # tae.py:495-499: out[B, n, C', H, W], attn[n_head, B, n, T, H, W].  The queries never interact (separate
            # softmax rows, row-wise MLP, eval-mode BatchNorm): one pass of the single-query kernels per query.
            return self._forward_queries(x, batch_positions, pad_mask, return_att)
        return self._forward_one(x, batch_positions, pad_mask, return_att)

    @torch.no_grad()
    def _forward_queries(self, x, batch_positions, pad_mask, return_att):
        """num_queries = n > 1, eval mode (tae.py:486-499): out[B, n, C', H, W], attn[n_head, B, n, T, H, W].  The
        attention rows of the queries are independent: one pass of the single-query kernels per query yields its
        attention and its rows ``o``; ``out_norm`` runs over the channels of a group AND the n queries (it is applied
        to [B*H*W, C', n], tae.py:488), so the rows are finished jointly by ``c2s_ltae_rows_forward``."""
        bn = self.mlp[2]
        if not bn.track_running_stats:
            raise NotImplementedError("crop2seg_b200: num_queries > 1 needs BatchNorm running statistics")
        b, t, _, h, w = x.shape
        spec = self._spec()
        params = self._params(x.device)
        rows, attns = [], []
        for i in range(self.num_queries):
            params["query"] = self.attention_head.Q[:, i:i + 1, :]  # Q[n_head, n, d_k] -> the rows of one query
            res = ops.ltae_forward(x, batch_positions, pad_mask, params, spec, need_attn=return_att, save_o=True)
            rows.append(res.o_rows)
            attns.append(res.attn)
        # the row kernel applies out_norm alone, with out_norm's own eps
        out = ops.ltae_rows_forward(torch.stack(rows), params, dataclasses.replace(spec, gn_eps=self.out_norm.eps),
                                    batch=b, height=h, width=w, dtype=x.dtype)
        return out, (torch.stack(attns, dim=2) if return_att else None)

    def _forward_one(self, x, batch_positions, pad_mask, return_att):
        spec = self._spec()
        params = self._params(x.device)
        b, t, _, h, w = x.shape
        attn_keep = _draw_keep((self.n_head, b, t, h, w), spec.attn_drop_p, x.device, 0)
        mlp_keep = _draw_keep((b, spec.c_out, h, w), spec.mlp_drop_p, x.device, 1)
        if self._needs_grad(x):
            from .autograd import LtaeFunction
            out, attn, mean, var = LtaeFunction.apply(x, batch_positions, pad_mask, attn_keep, mlp_keep, spec,
                                                      *[params.get(k) for k in _lib.LTAE_PARAM_FIELDS])
            stats = (mean, var) if mean is not None else None
        else:
            out, attn, stats = ops.ltae_forward(x, batch_positions, pad_mask, params, spec, need_attn=return_att,
                                                attn_keep=attn_keep, mlp_keep=mlp_keep, **self._folded_args(params))[:3]
        if stats is not None and self.training and self.mlp[2].track_running_stats:
            self._update_running_stats(self.mlp[2], stats, b * h * w)
        return out, (attn if return_att else None)

    @staticmethod
    @torch.no_grad()
    def _update_running_stats(bn, stats, n_rows):
        """nn.BatchNorm1d train-mode bookkeeping (momentum, unbiased variance) -- tae.py:445."""
        mean, var = stats
        bn.num_batches_tracked += 1
        momentum = bn.momentum if bn.momentum is not None else 1.0 / float(bn.num_batches_tracked)
        unbiased = var * (n_rows / max(n_rows - 1, 1))
        bn.running_mean.mul_(1 - momentum).add_(mean.to(bn.running_mean.dtype), alpha=momentum)
        bn.running_var.mul_(1 - momentum).add_(unbiased.to(bn.running_var.dtype), alpha=momentum)


class LTAE4WTAE(_LTAEBase):
    """Attention-only L-TAE for W-TAE -- drop-in for ``src.backbones.tae.LTAE4WTAE`` (tae.py:507)."""

    def __init__(self, in_channels=128, n_head=16, d_k=4, d_model=256, positional_encoding=True,
                 use_abs_rel_enc=False, num_queries=1, use_doy=False, add_linear=False, *args, **kwargs):
        super().__init__()
        self._build_front(in_channels, n_head, d_k, d_model, positional_encoding, use_abs_rel_enc, num_queries,
                          use_doy, add_linear)

    def forward(self, x, batch_positions=None, pad_mask=None, return_comp=False):
        """x[B,T,C,H,W] -> attn[n_head,B,T,H,W] (tae.py:589-635); dropout on the attention in training mode."""
        self._check_inputs(x, batch_positions)
        spec = self._spec()
        b, t, _, h, w = x.shape
        attn_keep = _draw_keep((self.n_head, b, t, h, w), spec.attn_drop_p, x.device, 0)
        params = self._params(x.device)
        if self._needs_grad(x):
            from .autograd import LtaeFunction
            return LtaeFunction.apply(x, batch_positions, pad_mask, attn_keep, None, spec,
                                      *[params.get(k) for k in _lib.LTAE_PARAM_FIELDS])[1]
        return ops.ltae_forward(x, batch_positions, pad_mask, params, spec, attn_keep=attn_keep,
                                **self._folded_args(params)).attn


class TemporalAggregator(nn.Module):
    """Drop-in for ``src.backbones.temporal_aggregator.TemporalAggregator`` (temporal_aggregator.py:6)."""

    def __init__(self, mode="mean"):
        super().__init__()
        self.mode = mode

    def forward(self, x, pad_mask=None, attn_mask=None):
        """x[B,T,C,H,W], attn_mask[h,B,T,ha,wa] -> out[B,C,H,W].

        The reference switches between a masked and an unmasked branch on ``pad_mask.any()`` (a
        device->host sync, temporal_aggregator.py:21); both give the same result, so the fused kernel
        simply skips the padded frames and never synchronises.
        """
        if self.mode not in ("att_group", "att_mean", "mean"):
            return None  # the reference falls through its if/elif chain and returns None
        return ops.temporal_aggregate(x, pad_mask=pad_mask, attn_mask=attn_mask, mode=self.mode)

    def forward_skip_conv(self, x, pad_mask, attn_mask, skip_conv):
        """``skip_conv(self(x, pad_mask, attn_mask))`` in one kernel, for the decoder's ``UpConvBlock.skip_conv`` =
        ``Sequential(Conv2d(d, d, 1), BatchNorm2d(d), ReLU())`` (conv.py:378-382; SURVEY.md section 8f, rank 1).

        ``skip_conv`` in eval mode (running statistics); ``att_group``, bf16 features with 64 channels.  Differentiable
        w.r.t. x, attn_mask and the convolution / BatchNorm affine parameters with the BatchNorm frozen (fine-tuning
        with the decoder's BatchNorm in eval mode); batch statistics are not served.  A maintainer replaces ``self.up_blocks[i](out, skip)`` by the block's own forward with the already-convolved
        skip (INTEGRATION.md, "Fused skip convolution").
        """
        if self.mode != "att_group":
            raise NotImplementedError("forward_skip_conv: only the att_group mode has a fused kernel")
        conv, bn = skip_conv[0], skip_conv[1]
        if not (isinstance(conv, nn.Conv2d) and isinstance(bn, nn.BatchNorm2d) and isinstance(skip_conv[2], nn.ReLU)):
            raise TypeError("forward_skip_conv expects Sequential(Conv2d(d, d, 1), BatchNorm2d(d), ReLU())")
        if conv.kernel_size != (1, 1) or conv.stride != (1, 1) or conv.groups != 1:
            raise NotImplementedError("forward_skip_conv: the skip convolution must be a plain 1x1 convolution")
        if bn.training or bn.running_mean is None:
            raise RuntimeError("forward_skip_conv is an inference path: put skip_conv in eval mode (running statistics)")
        return ops.temporal_aggregate_skip_conv(x, pad_mask, attn_mask, conv.weight, conv.bias, bn.weight, bn.bias,
                                                bn.running_mean, bn.running_var, bn.eps)
