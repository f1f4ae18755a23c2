"""The aggregation fused with the decoder's skip convolution, BatchNorm with batch statistics (training mode):
``c2s_agg_skipconv_bstats_forward`` / ``c2s_agg_skipconv_bstats_backward`` through
``TemporalAggregator.forward_skip_conv(..., allow_batch_stats=True)`` and ``ops``, against float64 torch of the unfused
composition (the oracle aggregator on the same bf16 x, the skip map and z rounded to bf16 as the kernels store them,
batch-statistics BatchNorm, ReLU)."""
import copy

import numpy as np
import pytest
import torch
from torch import nn

from golden_util import rel_err
from oracle.torch_port import temporal_aggregator_torch
from skipconv_bstats_ref import bf16_value, skip_conv_bstats

pytestmark = pytest.mark.gpu

# name: (B, T, H = W, attention size, lengths): ragged, single-frame and all-padded series; more 128-pixel tiles than
# SMs at x8 (3 x 128 = 384 CTAs)
CASES = {
    "x2": (3, 9, 32, 16, [9, 4, 0]),
    "x4": (2, 13, 64, 16, [13, 0]),
    "x8": (3, 7, 128, 16, [7, 1, 0]),
}
# max |error| / max |reference| (mean: of the reference; var: per channel), bounds about 3x the largest value measured on
# a B200 over the cases below.  Forward: out against the float64 BatchNorm of the kernel's own z, measured 3.2e-3 (bf16
# output rounding); z against float64 z rounded to bf16, 4.2e-3 (one bf16 ulp where the fp32 and float64 sums round
# apart); the batch mean / variance against float64 statistics of the kernel's z, 6.1e-8 / 1.4e-7.
FWD_TOL = {"out": 1e-2, "z": 1.3e-2, "mean": 2e-7, "var": 5e-7}
# backward, all six gradients against float64 autograd with the fused forward's ReLU mask and z; measured: x 3.1e-3
# (grad_x is rounded to bf16), attn 4.7e-6, conv_weight 8.0e-5, bn_weight 2.6e-7, bn_bias 5.6e-8
BWD_TOL = {"x": 1e-2, "attn": 1.5e-5, "conv_weight": 2.4e-4, "bn_weight": 8e-7, "bn_bias": 2e-7}


def _report(what, **errs):
    print(f"[bstats] {what}: " + " ".join(f"{k}={v:.3g}" for k, v in errs.items()))


def _block(rng, affine=True, bias=True, momentum=0.1, track=True, device="cuda"):
    m = nn.Sequential(nn.Conv2d(64, 64, 1, bias=bias),
                      nn.BatchNorm2d(64, affine=affine, momentum=momentum, track_running_stats=track), nn.ReLU())
    with torch.no_grad():
        m[0].weight.copy_(torch.from_numpy(rng.standard_normal((64, 64, 1, 1)).astype(np.float32) / 8))
        if bias:
            m[0].bias.copy_(torch.from_numpy(0.1 * rng.standard_normal(64).astype(np.float32)))
        if affine:
            m[1].weight.copy_(torch.from_numpy((1.0 + 0.3 * rng.standard_normal(64)).astype(np.float32)))
            m[1].bias.copy_(torch.from_numpy((0.2 * rng.standard_normal(64)).astype(np.float32)))
        if track:
            m[1].running_mean.copy_(torch.from_numpy((0.3 * rng.standard_normal(64)).astype(np.float32)))
            m[1].running_var.copy_(torch.from_numpy(rng.uniform(0.5, 2.0, 64).astype(np.float32)))
    return m.to(device).train()


def _inputs(name, seed=0, **block_kw):
    from c2s_testlib import bf16_round, random_attention, synth_inputs
    b, t, res, ares, lengths = CASES[name]
    rng = np.random.RandomState(200 + res + t + seed)
    x, _, pad = synth_inputs(rng, b, t, 64, res, res, lengths)
    x = bf16_round(x)
    attn = random_attention(rng, 16, pad, ares, ares)
    gout = bf16_round(rng.standard_normal((b, 64, res, res)).astype(np.float32))
    return x, pad, attn, gout, _block(rng, **block_kw)


def _params(block):
    conv, bn = block[0], block[1]
    return conv.weight, conv.bias, bn.weight, bn.bias, bn.eps


def _dev(x, pad, attn):
    from c2s_testlib import to_dev
    return to_dev(x, dtype=torch.bfloat16), to_dev(pad), to_dev(attn)


def _skip64(x, pad, attn, requires_grad=False):
    """float64 skip map of the unfused route, rounded to bf16 in value (the fused kernels' s)."""
    xr = torch.from_numpy(x).double().requires_grad_(requires_grad)
    ar = torch.from_numpy(attn).double().requires_grad_(requires_grad)
    return bf16_value(temporal_aggregator_torch(xr, torch.from_numpy(pad), ar, "att_group")), xr, ar


def _p64(block, requires_grad=False):
    conv, bn = block[0], block[1]
    return [None if p is None else p.detach().cpu().double().requires_grad_(requires_grad)
            for p in (conv.weight, conv.bias, bn.weight, bn.bias)]


def _check_forward(name, x, pad, attn, block):
    from crop2seg_b200 import _lib, ops
    with torch.no_grad():
        out, z, mean, var = ops.temporal_aggregate_skip_conv_bstats_forward(*_dev(x, pad, attn), *_params(block))
    assert _lib.last_kernel() == "agg_skipconv_bstats<apply>"
    s, _, _ = _skip64(x, pad, attn)
    w, b, g, be = _p64(block)
    ref = skip_conv_bstats(s, w, b, g, be, block[1].eps, round_z=True)
    zk = z.double().cpu()
    own = skip_conv_bstats(zk, torch.eye(64, dtype=torch.float64).view(64, 64, 1, 1), None, g, be, block[1].eps)
    errs = {"out": rel_err(out.float().cpu().numpy(), own["out"].numpy()),
            "z": rel_err(z.float().cpu().numpy(), ref["z"].numpy()),
            "mean": float((mean.cpu().double() - own["mean"]).abs().max() / own["mean"].abs().max()),
            "var": float(((var.cpu().double() - own["var"]).abs() / own["var"]).max())}
    _report(f"forward {name}", **errs)
    for k, tol in FWD_TOL.items():
        assert errs[k] < tol, (k, errs[k])
    return out, z, mean, var


@pytest.mark.parametrize("name", sorted(CASES))
def test_forward_matches_float64_batch_statistics(name):
    x, pad, attn, _, block = _inputs(name)
    _check_forward(name, x, pad, attn, block)


@pytest.mark.parametrize("affine,bias", [(False, True), (True, False), (False, False)])
def test_forward_without_affine_or_conv_bias(affine, bias):
    x, pad, attn, _, block = _inputs("x4", affine=affine, bias=bias)
    _check_forward(f"x4 affine={affine} bias={bias}", x, pad, attn, block)


@pytest.mark.parametrize("momentum", [0.1, None])
def test_running_statistics_follow_batchnorm2d(momentum):
    """Several training-mode calls update running_mean / running_var / num_batches_tracked as a torch BatchNorm2d fed the
    same z does (z is deterministic, so every call sees the same one)."""
    import crop2seg_b200 as c2s
    from crop2seg_b200 import ops
    x, pad, attn, _, block = _inputs("x8", momentum=momentum)
    ref_bn = copy.deepcopy(block[1])
    xd, pd, ad = _dev(x, pad, attn)
    agg = c2s.TemporalAggregator("att_group")
    with torch.no_grad():
        _, z, _, _ = ops.temporal_aggregate_skip_conv_bstats_forward(xd, pd, ad, *_params(block))
        for _ in range(3):
            agg.forward_skip_conv(xd, pd, ad, block, allow_batch_stats=True)
            ref_bn(z.float())
    assert int(block[1].num_batches_tracked) == int(ref_bn.num_batches_tracked) == 3
    e_m = rel_err(block[1].running_mean.cpu().numpy(), ref_bn.running_mean.cpu().numpy())
    e_v = rel_err(block[1].running_var.cpu().numpy(), ref_bn.running_var.cpu().numpy())
    _report(f"running stats momentum={momentum}", mean=e_m, var=e_v)
    assert e_m < 5e-7 and e_v < 6e-7  # measured 1.1e-7 / 1.9e-7


def test_without_running_statistics_nothing_is_updated():
    import crop2seg_b200 as c2s
    from crop2seg_b200 import ops
    x, pad, attn, _, block = _inputs("x2", track=False)
    xd, pd, ad = _dev(x, pad, attn)
    agg = c2s.TemporalAggregator("att_group")
    with torch.no_grad():
        want = ops.temporal_aggregate_skip_conv_bstats_forward(xd, pd, ad, *_params(block))[0]
        for mode in (True, False):  # batch statistics in train AND eval without running statistics, as torch
            block.train(mode)
            out = agg.forward_skip_conv(xd, pd, ad, block, allow_batch_stats=True)
            assert torch.equal(out, want)
    assert block[1].running_mean is None and block[1].num_batches_tracked is None


def _backward(x, pad, attn, gout, block, need=(True,) * 6):
    from crop2seg_b200 import ops
    from c2s_testlib import to_dev
    xd, pd, ad = _dev(x, pad, attn)
    with torch.no_grad():
        out, z, mean, var = ops.temporal_aggregate_skip_conv_bstats_forward(xd, pd, ad, *_params(block))
        res = ops.temporal_aggregate_skip_conv_bstats_backward(xd, pd, ad, *_params(block), z, mean, var, out,
                                                               to_dev(gout, dtype=torch.bfloat16), need=need)
    return out, z, res


def _oracle_backward(x, pad, attn, gout, block, relu_mask, z):
    """float64 autograd with the fused forward's ReLU decision and the values of its bf16 z (which the float64 z matches
    to one bf16 ulp, checked by the forward tests): the comparison then measures the backward's own arithmetic."""
    s, xr, ar = _skip64(x, pad, attn, requires_grad=True)
    P = _p64(block, requires_grad=True)
    ref = skip_conv_bstats(s, *P, block[1].eps, relu_mask=torch.from_numpy(relu_mask).double(), z_value=z.cpu())
    ref["out"].backward(torch.from_numpy(gout).double())
    grads = {"x": xr.grad.numpy(), "attn": ar.grad.numpy()}
    grads.update({k: None if p is None else p.grad.numpy()
                  for k, p in zip(("conv_weight", "conv_bias", "bn_weight", "bn_bias"), P)})
    return grads, ref["pre"].detach().numpy()


def _check_backward(what, x, pad, attn, gout, block, tol=BWD_TOL):
    from crop2seg_b200 import _lib
    out, z, res = _backward(x, pad, attn, gout, block)
    assert _lib.last_kernel() == "agg_skipconv_bstats_backward<reduce>"
    got = dict(zip(("x", "attn", "conv_weight", "conv_bias", "bn_weight", "bn_bias"), res))
    mask = out.float().cpu().numpy() > 0
    ref, pre = _oracle_backward(x, pad, attn, gout, block, mask, z)
    flips = mask != (pre > 0)  # the fused ReLU decision is the float64 one except at rounding level
    assert np.all(np.abs(pre[flips]) < 1e-2 * np.abs(pre).max())
    assert got["x"].dtype == torch.bfloat16
    errs = {}
    for k in tol:
        if ref[k] is None:
            continue
        g = got[k].float().cpu().numpy()
        assert np.isfinite(g).all(), k
        errs[k] = rel_err(g, ref[k])
    _report(f"backward {what}", **errs)
    for k, e in errs.items():
        assert e < tol[k], (k, e)
    if ref["conv_bias"] is not None:  # batch statistics cancel the conv bias: exactly zero here, rounding level in float64
        assert torch.count_nonzero(got["conv_bias"]) == 0
        gamma = 1.0 if block[1].weight is None else np.abs(block[1].weight.detach().cpu().numpy()).max()
        scale = np.abs(gout).sum(axis=(0, 2, 3)).max() * gamma
        assert np.abs(ref["conv_bias"]).max() < 1e-9 * scale
    assert np.all(got["x"].float().cpu().numpy()[pad] == 0.0)  # padded frames receive exactly zero
    for i in [i for i, row in enumerate(pad) if row.all()]:
        assert np.all(got["attn"].cpu().numpy()[:, i] == 0.0)


@pytest.mark.parametrize("name", sorted(CASES))
def test_gradients_match_float64_autograd(name):
    x, pad, attn, gout, block = _inputs(name)
    _check_backward(name, x, pad, attn, gout, block)


@pytest.mark.parametrize("affine,bias", [(False, True), (True, False)])
def test_gradients_without_affine_or_conv_bias(affine, bias):
    x, pad, attn, gout, block = _inputs("x2", affine=affine, bias=bias)
    _check_backward(f"x2 affine={affine} bias={bias}", x, pad, attn, gout, block)


def test_gradients_when_grad_out_is_nearly_constant_per_channel():
    """grad_out = a per-channel constant + 1e-3 noise, with the BatchNorm bias opening the ReLU on every pixel so that
    g_y is that near-constant too: g_z' = g_y - mean g_y - zhat mean(g_y zhat) is then far smaller than g_y (checked on
    the test's data below), and the expanded form (alpha W)^T g_y - (.. W)^T z + const would lose it to cancellation."""
    from c2s_testlib import bf16_round
    x, pad, attn, gout, block = _inputs("x4", seed=1)
    with torch.no_grad():
        block[1].bias.fill_(8.0)  # every pixel passes the ReLU (asserted below)
    rng = np.random.RandomState(5)
    const = rng.uniform(0.5, 1.5, 64).astype(np.float32)[None, :, None, None]
    gout = bf16_round(const + 1e-3 * rng.standard_normal(gout.shape).astype(np.float32))
    # the regime this case is for, in float64: all pixels pass the ReLU and ||g_z'|| << ||g_y||
    s, _, _ = _skip64(x, pad, attn)
    ref = skip_conv_bstats(s, *_p64(block), block[1].eps, round_z=True)
    assert bool((ref["pre"] > 0).all())
    g_y = torch.from_numpy(gout).double()
    zhat = (ref["z"] - ref["mean"][None, :, None, None]) / torch.sqrt(ref["var"][None, :, None, None] + block[1].eps)
    g_z = g_y - g_y.mean(dim=(0, 2, 3), keepdim=True) - zhat * (g_y * zhat).mean(dim=(0, 2, 3), keepdim=True)
    ratio = float(g_z.norm() / g_y.norm())
    _report("x4 constant grad_out", gz_over_gy=ratio)
    assert ratio < 1e-2
    # measured: x 2.4e-3, attn 4.7e-5, conv_weight 1.6e-3, bn_weight 2.0e-3 (relative to results that cancel to 0.2 % of
    # their terms: the fp32 batch mean and the fp32 sums behind mean_N(g_y), mean_N(g_y zhat) carry ~1e-7 of the terms'
    # size).  On these inputs an fp32 emulation with the kernel's bf16 hi + lo operands (exact statistics) gives grad_s
    # errors of 4.0e-6 for the per-pixel g_z' form and 6.6e-4 for the expanded form (alpha W)^T g_y - (.. W)^T z + const,
    # which the attn bound rejects.
    _check_backward("x4 constant grad_out", x, pad, attn, gout, block,
                    tol={"x": 1e-2, "attn": 1.5e-4, "conv_weight": 5e-3, "bn_weight": 6e-3, "bn_bias": 2e-7})


def test_deterministic_and_null_outputs_are_honoured():
    import crop2seg_b200 as c2s
    from crop2seg_b200 import _lib
    x, pad, attn, gout, block = _inputs("x8")
    out1, _, r1 = _backward(x, pad, attn, gout, block)
    out2, _, r2 = _backward(x, pad, attn, gout, block)
    assert torch.equal(out1, out2)
    assert torch.equal(r1[0], r2[0])  # grad_x
    for a, b in zip(r1[2:], r2[2:]):  # fixed-order reductions: bit-identical parameter gradients
        assert torch.equal(a, b)
    assert rel_err(r1[1].cpu().numpy(), r2[1].cpu().numpy()) < 1e-5  # grad_attn: float atomics
    only = _backward(x, pad, attn, gout, block, need=(False, True, False, True, True, False))[2]
    assert only[0] is None and only[2] is None and only[5] is None
    assert torch.count_nonzero(only[3]) == 0 and torch.equal(only[4], r1[4])
    bn_only = _backward(x, pad, attn, gout, block, need=(False, False, False, False, True, True))[2]
    assert _lib.last_kernel() == "agg_skipconv_bstats_backward<means>"  # no sweep without grad_x/attn/conv_weight
    assert torch.equal(bn_only[4], r1[4]) and torch.equal(bn_only[5], r1[5])
    gx_only = _backward(x, pad, attn, gout, block, need=(True, False, False, False, False, False))[2]
    assert _lib.last_kernel() == "agg_skipconv_bstats_backward<x8>"
    assert torch.equal(gx_only[0], r1[0]) and gx_only[1:] == (None,) * 5
    # the module path: batch statistics and running statistics bit-identical over two runs
    xd, pd, ad = _dev(x, pad, attn)
    blocks = [copy.deepcopy(block) for _ in range(2)]
    agg = c2s.TemporalAggregator("att_group")
    outs = []
    for blk in blocks:
        with torch.no_grad():
            outs.append(agg.forward_skip_conv(xd, pd, ad, blk, allow_batch_stats=True))
    assert torch.equal(outs[0], outs[1])
    assert torch.equal(blocks[0][1].running_mean, blocks[1][1].running_mean)
    assert torch.equal(blocks[0][1].running_var, blocks[1][1].running_var)


def test_unsupported_shapes_raise():
    import crop2seg_b200 as c2s
    from crop2seg_b200 import ops
    from crop2seg_b200._lib import C2SError
    block = _block(np.random.RandomState(3))
    agg = c2s.TemporalAggregator("att_group")
    attn = torch.full((16, 1, 3, 8, 8), 1 / 3, device="cuda")
    x32 = torch.zeros((1, 3, 64, 16, 16), device="cuda")  # fp32 features: no fused kernel
    with pytest.raises(C2SError, match="fused path serves"):
        agg.forward_skip_conv(x32, None, attn, block, allow_batch_stats=True)
    xb = torch.zeros((1, 3, 64, 16, 16), device="cuda", dtype=torch.bfloat16)
    out = torch.zeros((1, 64, 16, 16), device="cuda", dtype=torch.bfloat16)
    st = torch.ones(64, device="cuda")
    with pytest.raises(C2SError, match="fused backward serves"):  # 8 heads
        ops.temporal_aggregate_skip_conv_bstats_backward(xb, None, attn[:8], *_params(block), out, st, st, out, out)
    with pytest.raises(RuntimeError, match="eval mode"):  # the default stays the inference path
        agg.forward_skip_conv(xb, None, attn, block)


def test_eval_block_takes_the_running_statistics_kernels_unchanged():
    import crop2seg_b200 as c2s
    from crop2seg_b200 import _lib
    x, pad, attn, _, block = _inputs("x4")
    block.eval()
    xd, pd, ad = _dev(x, pad, attn)
    agg = c2s.TemporalAggregator("att_group")
    with torch.no_grad():
        a = agg.forward_skip_conv(xd, pd, ad, block)
        ka = _lib.last_kernel()
        b = agg.forward_skip_conv(xd, pd, ad, block, allow_batch_stats=True)
        assert _lib.last_kernel() == ka == "agg_skipconv<x4>"
    assert torch.equal(a, b)
    assert int(block[1].num_batches_tracked) == 0


def test_cuda_graph_training_step_replays_eager_steps():
    """One training step (fused forward with batch statistics, backward, SGD, running statistics with momentum 0.1) is
    captured once; its replays match eager steps from the same state, bit for bit (grad_attn aside: float atomics)."""
    import crop2seg_b200 as c2s
    x, pad, attn, gout, block0 = _inputs("x4")
    xd, pd, ad = _dev(x, pad, attn)
    ad.requires_grad_(True)
    w = torch.from_numpy(gout).cuda()
    agg = c2s.TemporalAggregator("att_group")

    def make():
        blk = copy.deepcopy(block0)
        return blk, torch.optim.SGD(blk.parameters(), lr=0.1)

    def step(blk, opt):
        opt.zero_grad(set_to_none=False)
        ad.grad = None if ad.grad is None else ad.grad.zero_()
        out = agg.forward_skip_conv(xd, pd, ad, blk, allow_batch_stats=True)
        (out.float() * w).sum().backward()
        opt.step()
        return out

    eager, opt_e = make()
    eager_states, eager_attn = [], []
    for _ in range(2):
        step(eager, opt_e)
        eager_states.append({k: v.clone() for k, v in eager.state_dict().items()})
        eager_attn.append(ad.grad.clone())
    graphed, opt_g = make()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):  # warm-up (allocates .grad), then the state is reset in place
        step(graphed, opt_g)
    torch.cuda.current_stream().wait_stream(side)
    with torch.no_grad():
        for k, v in graphed.state_dict().items():
            v.copy_(block0.state_dict()[k])
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        step(graphed, opt_g)
    with torch.no_grad():  # capture ran nothing, but reset again in case the capture touched a tensor
        for k, v in graphed.state_dict().items():
            v.copy_(block0.state_dict()[k])
    for i in range(2):
        g.replay()
        torch.cuda.synchronize()
        for k, v in graphed.state_dict().items():
            assert torch.equal(v, eager_states[i][k]), (i, k)
        assert rel_err(ad.grad.cpu().numpy(), eager_attn[i].cpu().numpy()) < 1e-5


def test_ltae_attention_and_training_skip_conv_match_the_unfused_step():
    """U-TAE's bottleneck with the decoder's skip convolution in train(): the encoder's attention feeds the fused kernel;
    the gradients of the encoder, of skip_conv and of the skip features, and the updated running statistics, agree with
    the same step through TemporalAggregator + the torch block (float32).  The BatchNorm bias keeps every pre-activation
    clear of the ReLU's edge: there the two routes' z (bf16 vs float32) would flip single pixels, and one flipped pixel
    moves a sum over the random-signed grad_out by a few percent."""
    import crop2seg_b200 as c2s
    from c2s_testlib import randomise, synth_inputs, to_dev
    rng = np.random.RandomState(21)
    enc0 = c2s.LTAE(in_channels=128, n_head=16, d_k=4, mlp=[256, 128], d_model=256)
    randomise(enc0, rng)
    enc0 = enc0.cuda().eval()
    block0 = _block(rng)
    with torch.no_grad():
        block0[1].bias.fill_(8.0)  # lifts the pre-activations far above the ReLU's edge
    b, t = 2, 9
    x4, pos, pad = synth_inputs(rng, b, t, 128, 8, 8, [9, 5])
    xs = synth_inputs(rng, b, t, 64, 32, 32, [9, 5])[0]
    wgt = torch.randn((b, 64, 32, 32), device="cuda", generator=torch.Generator("cuda").manual_seed(0))
    res = {}
    for fused in (True, False):
        enc, block = copy.deepcopy(enc0), copy.deepcopy(block0)
        x4d = to_dev(x4).requires_grad_(True)
        xsd = to_dev(xs, dtype=torch.bfloat16).requires_grad_(True)
        out, att = enc(x4d, batch_positions=to_dev(pos), pad_mask=to_dev(pad))
        agg = c2s.TemporalAggregator("att_group")
        if fused:
            skip = agg.forward_skip_conv(xsd, to_dev(pad), att, block, allow_batch_stats=True).float()
        else:
            skip = block(agg(xsd, to_dev(pad), att).float())
        (out.pow(2).mean() + (skip * wgt).mean()).backward()
        res[fused] = {"enc." + n: p.grad for n, p in enc.named_parameters() if p.grad is not None}
        res[fused].update({"skip_conv." + n: p.grad for n, p in block.named_parameters()})
        res[fused].update({"x_skip": xsd.grad.float(), "running_mean": block[1].running_mean,
                           "running_var": block[1].running_var})
    worst = {}
    for k, ref in res[False].items():
        got = res[True][k]
        if k == "skip_conv.0.bias":  # zero in both up to rounding: batch statistics cancel it
            assert torch.count_nonzero(got) == 0
            continue
        if not k.startswith("enc."):
            worst[k] = rel_err(got.float().cpu().numpy(), ref.float().cpu().numpy())
    # the encoder as a whole (some of its gradients, e.g. the key bias under the softmax, are rounding noise alone)
    enc = [k for k in res[False] if k.startswith("enc.")]
    diff = torch.cat([(res[True][k] - res[False][k]).flatten() for k in enc])
    worst["enc"] = float(diff.norm() / torch.cat([res[False][k].flatten() for k in enc]).norm())
    _report("end to end", **worst)
    # measured: skip_conv and x_skip <= 6.3e-3 (the fused route's z is bf16, the torch block's float32), running
    # statistics 5.6e-5
    for k, e in worst.items():
        assert e < (2e-4 if k.startswith("running") else 2e-2), (k, e)
