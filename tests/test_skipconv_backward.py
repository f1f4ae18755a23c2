"""Backward of the aggregation fused with the decoder's skip convolution, BatchNorm frozen (``c2s_agg_skipconv_backward``
through ``TemporalAggregator.forward_skip_conv`` / ``ops.temporal_aggregate_skip_conv_backward``) against float64 torch
autograd of the unfused composition: the oracle aggregator on the same bf16 x, the skip map rounded to bf16 as the
forward rounds it, then Conv2d -> eval BatchNorm2d -> ReLU."""
import numpy as np
import pytest
import torch
from torch import nn

from golden_util import rel_err
from oracle.torch_port import temporal_aggregator_torch

pytestmark = pytest.mark.gpu

# name: (B, T, H = W, attention size, lengths); more 128-pixel tiles than SMs at x8 (3 x 128 = 384 CTAs)
CASES = {
    "x2": (3, 9, 32, 16, [9, 4, 0]),
    "x4": (2, 13, 64, 16, [13, 0]),
    "x8": (3, 7, 128, 16, [7, 1, 0]),
}
# max |error| / max |reference| per gradient.  Measured on a B200 (largest of the three levels): x 2.6e-3 (grad_x is
# rounded to bf16), attn 3.1e-6, conv_weight 3.6e-5 and bn_weight 1.2e-5 (a bf16 skip value one ulp off where the fp32 and
# the float64 sums round to different sides), conv_bias / bn_bias 1.4e-7.  Bounds: about 3x the measurement.
TOL = {"x": 8e-3, "attn": 1e-5, "conv_weight": 1.2e-4, "conv_bias": 5e-7, "bn_weight": 4e-5, "bn_bias": 5e-7}


def _block(rng, device="cuda"):
    m = nn.Sequential(nn.Conv2d(64, 64, 1), nn.BatchNorm2d(64), nn.ReLU())
    with torch.no_grad():
        m[0].weight.copy_(torch.from_numpy(rng.standard_normal((64, 64, 1, 1)).astype(np.float32) / 8))
        m[0].bias.copy_(torch.from_numpy(0.1 * rng.standard_normal(64).astype(np.float32)))
        m[1].weight.copy_(torch.from_numpy((1.0 + 0.3 * rng.standard_normal(64)).astype(np.float32)))
        m[1].bias.copy_(torch.from_numpy((0.2 * rng.standard_normal(64)).astype(np.float32)))
        m[1].running_mean.copy_(torch.from_numpy((0.3 * rng.standard_normal(64)).astype(np.float32)))
        m[1].running_var.copy_(torch.from_numpy(rng.uniform(0.5, 2.0, 64).astype(np.float32)))
    return m.to(device).eval()


def _inputs(name):
    from c2s_testlib import bf16_round, random_attention, synth_inputs
    b, t, res, ares, lengths = CASES[name]
    rng = np.random.RandomState(100 + res + t)
    x, _, pad = synth_inputs(rng, b, t, 64, res, res, lengths)
    x = bf16_round(x)
    attn = random_attention(rng, 16, pad, ares, ares)
    gout = bf16_round(rng.standard_normal((b, 64, res, res)).astype(np.float32))
    return x, pad, attn, gout, _block(rng)


def _oracle(x, pad, attn, gout, block, relu_mask):
    """float64 autograd of the unfused composition; the ReLU takes the fused forward's decision ``relu_mask`` (its
    agreement with the float64 pre-activation is checked by the caller)."""
    from c2s_testlib import bf16_round
    conv, bn = block[0], block[1]
    xr = torch.from_numpy(x).double().requires_grad_(True)
    ar = torch.from_numpy(attn).double().requires_grad_(True)
    P = {k: v.detach().cpu().double().requires_grad_(True) for k, v in
         (("conv_weight", conv.weight), ("conv_bias", conv.bias), ("bn_weight", bn.weight), ("bn_bias", bn.bias))}
    s = temporal_aggregator_torch(xr, torch.from_numpy(pad), ar, "att_group")
    s = s + (torch.from_numpy(bf16_round(s.detach().float().numpy())).double() - s).detach()  # bf16 value, identity gradient
    z = torch.nn.functional.conv2d(s, P["conv_weight"], P["conv_bias"])
    rm, rv = bn.running_mean.cpu().double(), bn.running_var.cpu().double()
    pre = (z - rm[None, :, None, None]) / torch.sqrt(rv[None, :, None, None] + bn.eps) * P["bn_weight"][None, :, None, None] \
        + P["bn_bias"][None, :, None, None]
    (pre * torch.from_numpy(relu_mask).double()).backward(torch.from_numpy(gout).double())
    grads = {"x": xr.grad.numpy(), "attn": ar.grad.numpy()}
    grads.update({k: v.grad.numpy() for k, v in P.items()})
    return grads, pre.detach().numpy()


def _cuda(x, pad, attn, gout, block):
    import crop2seg_b200 as c2s
    from c2s_testlib import to_dev
    xd = to_dev(x, dtype=torch.bfloat16).requires_grad_(True)
    ad = to_dev(attn).requires_grad_(True)
    out = c2s.TemporalAggregator("att_group").forward_skip_conv(xd, to_dev(pad), ad, block)
    block.zero_grad(set_to_none=True)
    out.backward(to_dev(gout, dtype=torch.bfloat16))
    conv, bn = block[0], block[1]
    grads = {"x": xd.grad.float().cpu().numpy(), "attn": ad.grad.cpu().numpy(),
             "conv_weight": conv.weight.grad.cpu().numpy(), "conv_bias": conv.bias.grad.cpu().numpy(),
             "bn_weight": bn.weight.grad.cpu().numpy(), "bn_bias": bn.bias.grad.cpu().numpy()}
    return out.detach(), grads, xd.grad.dtype


@pytest.mark.parametrize("name", sorted(CASES))
def test_gradients_match_float64_autograd_of_the_unfused_composition(name):
    from crop2seg_b200 import _lib
    x, pad, attn, gout, block = _inputs(name)
    out, got, gx_dtype = _cuda(x, pad, attn, gout, block)
    assert _lib.last_kernel() == "agg_skipconv_backward<reduce>"
    mask = (out.float().cpu().numpy() > 0)
    ref, pre = _oracle(x, pad, attn, gout, block, mask)
    # the forward's ReLU decision is the float64 one except where the pre-activation is at rounding level
    flips = mask != (pre > 0)
    assert np.all(np.abs(pre[flips]) < 1e-4 * np.abs(pre).max())
    assert gx_dtype == torch.bfloat16
    for k, tol in TOL.items():
        assert np.isfinite(got[k]).all(), k
        err = rel_err(got[k], ref[k])
        assert err < tol, (k, err)
    assert np.all(got["x"][pad] == 0.0)  # padded frames receive exactly zero
    b_empty = [i for i, row in enumerate(pad) if row.all()]
    for i in b_empty:  # a series with no valid frame: its attention gradient is exactly zero too
        assert np.all(got["attn"][:, i] == 0.0)


def test_parameter_gradients_are_deterministic_and_null_outputs_are_skipped():
    from crop2seg_b200 import _lib, ops
    from c2s_testlib import to_dev
    x, pad, attn, gout, block = _inputs("x8")
    conv, bn = block[0], block[1]
    args = (to_dev(x, dtype=torch.bfloat16), to_dev(pad), to_dev(attn), conv.weight, conv.bias, bn.weight, bn.bias,
            bn.running_mean, bn.running_var, bn.eps)
    with torch.no_grad():
        out = ops.temporal_aggregate_skip_conv(*args)
        first = ops.temporal_aggregate_skip_conv_backward(*args, out, to_dev(gout, dtype=torch.bfloat16))
        second = ops.temporal_aggregate_skip_conv_backward(*args, out, to_dev(gout, dtype=torch.bfloat16))
        assert _lib.last_kernel() == "agg_skipconv_backward<reduce>"
        for a, b in zip(first[2:], second[2:]):  # fixed-order reduction: bit-identical
            assert torch.equal(a, b)
        assert torch.equal(first[0], second[0])  # grad_x has no reduction either
        only = ops.temporal_aggregate_skip_conv_backward(*args, out, to_dev(gout, dtype=torch.bfloat16),
                                                         need=(False, True, False, True, True, False))
        assert only[0] is None and only[2] is None and only[5] is None
        assert torch.equal(only[3], first[3]) and torch.equal(only[4], first[4])
        assert rel_err(only[1].cpu().numpy(), first[1].cpu().numpy()) < 1e-5  # float atomics: order-dependent low bits
        gx_only = ops.temporal_aggregate_skip_conv_backward(*args, out, to_dev(gout, dtype=torch.bfloat16),
                                                            need=(True, False, False, False, False, False))
        assert _lib.last_kernel() == "agg_skipconv_backward<x8>"  # no parameter gradient: no reduction launch
        assert gx_only[1:] == (None,) * 5 and torch.equal(gx_only[0], first[0])


@pytest.mark.parametrize("global_taps", [False, True])
@pytest.mark.parametrize("name", sorted(CASES))
def test_backward_recomputes_the_forward_skip_map_bit_for_bit(name, global_taps):
    """The weight gradient relies on the backward's skip map s being the forward's.  With an identity convolution and a
    neutral BatchNorm (eps = 0) the forward's output is exactly relu(s); a grad_out that is 1 on every channel of one
    pixel p makes grad_conv_weight[o, c] = s_bwd[c, p] exactly for every o with out[o, p] > 0 (one non-zero term,
    alpha = 1).  x has both signs, so relu(s) is zero on a part of the channels."""
    from crop2seg_b200 import _lib, ops
    from c2s_testlib import bf16_round, random_attention, synth_inputs, to_dev
    b, t, res, ares, lengths = CASES[name]
    rng = np.random.RandomState(31 + res)
    _, _, pad = synth_inputs(rng, b, t, 64, res, res, lengths)
    x = bf16_round(rng.standard_normal((b, t, 64, res, res)).astype(np.float32))
    attn = random_attention(rng, 16, pad, ares, ares)
    conv, bn = nn.Conv2d(64, 64, 1).cuda(), nn.BatchNorm2d(64, eps=0.0).cuda().eval()  # BatchNorm: weight 1, bias 0,
    with torch.no_grad():                                                                # mean 0, var 1
        conv.weight.copy_(torch.eye(64).view(64, 64, 1, 1))
        conv.bias.zero_()
    args = (to_dev(x, dtype=torch.bfloat16), to_dev(pad), to_dev(attn), conv.weight, conv.bias, bn.weight, bn.bias,
            bn.running_mean, bn.running_var, bn.eps)
    # first and last pixel of the second 128-pixel block, a right-border column and an interior pixel
    pixels = [128, 255, (res // 2) * res + res - 1, (res // 2 + 1) * res + res // 2 + 3]
    with torch.no_grad(), _lib.option(_lib.OPT_AGG_TAPS, int(global_taps)):
        out = ops.temporal_aggregate_skip_conv(*args)
        for b0 in [i for i, n in enumerate(lengths) if n > 0]:
            for p in pixels:
                gout = torch.zeros_like(out)
                gout[b0, :, p // res, p % res] = 1
                gw = ops.temporal_aggregate_skip_conv_backward(*args, out, gout)[2].view(64, 64)
                s_fwd = out[b0, :, p // res, p % res].float()
                pos = s_fwd > 0
                assert pos.any() and (~pos).any(), (b0, p)
                g = gw[pos]  # rows o with out[o, p] > 0
                assert torch.equal(g[:, pos], s_fwd[pos].expand_as(g[:, pos])), (b0, p)
                assert (g[:, ~pos] <= 0).all(), (b0, p)


def test_unsupported_shapes_raise():
    import crop2seg_b200 as c2s
    from crop2seg_b200 import ops
    from crop2seg_b200._lib import C2SError
    rng = np.random.RandomState(3)
    block = _block(rng)
    conv, bn = block[0], block[1]
    agg = c2s.TemporalAggregator("att_group")
    attn = torch.full((16, 1, 3, 8, 8), 1 / 3, device="cuda", requires_grad=True)
    x32 = torch.zeros((1, 3, 64, 16, 16), device="cuda", requires_grad=True)  # fp32 features: no fused kernel
    with pytest.raises(C2SError):
        agg.forward_skip_conv(x32, None, attn, block)
    xb = torch.zeros((1, 3, 64, 16, 16), device="cuda", dtype=torch.bfloat16)
    out = torch.zeros((1, 64, 16, 16), device="cuda", dtype=torch.bfloat16)
    params = (conv.weight, conv.bias, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.eps)
    with pytest.raises(C2SError, match="fused backward serves"):  # the backward's own check: fp32 x
        ops.temporal_aggregate_skip_conv_backward(x32.detach(), None, attn.detach(), *params, out.float(), out.float())
    with pytest.raises(C2SError, match="fused backward serves"):  # 8 heads
        ops.temporal_aggregate_skip_conv_backward(xb, None, attn.detach()[:8], *params, out, out)
    with pytest.raises(C2SError, match="fused backward serves"):  # same resolution: no up-sampling
        ops.temporal_aggregate_skip_conv_backward(xb, None, torch.ones((16, 1, 3, 16, 16), device="cuda"), *params, out, out)
    block.train()  # BatchNorm batch statistics stay unsupported
    with pytest.raises(RuntimeError, match="eval mode"):
        agg.forward_skip_conv(xb.requires_grad_(True), None, attn, block)


def test_ltae_attention_and_skip_conv_train_through_one_backward():
    """U-TAE's bottleneck with a frozen-BatchNorm skip convolution: the encoder's attention feeds the fused kernel, and one
    backward() fills the gradients of the encoder, of skip_conv and of the skip features."""
    import crop2seg_b200 as c2s
    from c2s_testlib import randomise, synth_inputs, to_dev
    rng = np.random.RandomState(21)
    enc = c2s.LTAE(in_channels=128, n_head=16, d_k=4, mlp=[256, 128], d_model=256)
    randomise(enc, rng)
    enc = enc.cuda().eval()
    block = _block(rng)
    b, t = 2, 9
    x4, pos, pad = synth_inputs(rng, b, t, 128, 8, 8, [9, 5])
    xs = synth_inputs(rng, b, t, 64, 32, 32, [9, 5])[0]
    x4d = to_dev(x4).requires_grad_(True)
    xsd = to_dev(xs, dtype=torch.bfloat16).requires_grad_(True)
    out, att = enc(x4d, batch_positions=to_dev(pos), pad_mask=to_dev(pad))
    skip = c2s.TemporalAggregator("att_group").forward_skip_conv(xsd, to_dev(pad), att, block)
    assert skip.requires_grad
    w = torch.randn(skip.shape, device="cuda", generator=torch.Generator("cuda").manual_seed(0))
    loss = out.pow(2).mean() + (skip.float() * w).mean()
    loss.backward()
    for name, p in list(enc.named_parameters()) + list(block.named_parameters()):
        assert p.grad is not None and torch.isfinite(p.grad).all(), name
    assert float(block[0].weight.grad.abs().max()) > 0 and float(enc.attention_head.Q.grad.abs().max()) > 0
    assert xsd.grad is not None and x4d.grad is not None and float(xsd.grad.float().abs().max()) > 0
