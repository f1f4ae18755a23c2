"""Backward / training-mode parity on the GPU.

* TemporalAggregator: forward and backward are CUDA kernels; gradients are compared with autograd through the
  torch-CPU oracle (oracle/torch_port.py) on the same inputs.
* L-TAE: the training-mode forward kernel (BatchNorm batch statistics + injected dropout masks) is compared with the
  numpy oracle; its backward (``c2s_ltae_backward`` for everything that touches the features + autograd on the small
  rows / folded weights) is compared with autograd through the torch-CPU oracle, and, at the shipped shapes in
  training mode, with the REFERENCE's own autograd on the reference's own dropout realisation (train_*.npz).
"""
import numpy as np
import pytest
import torch

import crop2seg_b200 as c2s
from crop2seg_b200 import _lib, ops
from oracle import ltae_forward
from oracle.torch_port import ltae_forward_torch, temporal_aggregator_torch
from golden_util import rel_err
from c2s_testlib import (bf16_round, oracle_config, oracle_params, random_attention, randomise, synth_inputs,
                         to_dev)

pytestmark = pytest.mark.gpu

AGG_BWD_CASES = {
    # name: (mode, heads, (B,T,C,H,W), (ha,wa), lengths)
    "x8_128": ("att_group", 16, (2, 5, 64, 128, 128), (16, 16), [5, 3]),
    "x4_64": ("att_group", 16, (2, 5, 64, 64, 64), (16, 16), [5, 2]),
    "x2_32": ("att_group", 16, (2, 6, 64, 32, 32), (16, 16), [6, 0]),
    "x2_small": ("att_group", 4, (2, 5, 8, 8, 8), (4, 4), [5, 3]),
    "frac": ("att_group", 4, (2, 4, 8, 12, 12), (5, 5), [4, 3]),
    "rect": ("att_group", 4, (2, 4, 8, 12, 20), (4, 6), [4, 1]),
    "pool_k2": ("att_group", 4, (2, 5, 8, 8, 8), (16, 16), [5, 3]),      # AvgPool2d branch (temporal_aggregator.py:28-29)
    "pool_floor": ("att_group", 4, (2, 4, 8, 4, 4), (9, 9), [4, 2]),     # 9 // 4 = 2: the last row / column is dropped
    "same_res": ("att_group", 4, (2, 4, 8, 8, 8), (8, 8), [4, 1]),       # k = 1
    "att_mean": ("att_mean", 4, (2, 5, 8, 16, 16), (4, 4), [5, 3]),
    "mean": ("mean", 4, (2, 5, 6, 8, 8), (4, 4), [5, 3]),
}


@pytest.mark.parametrize("name", sorted(AGG_BWD_CASES))
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_aggregator_backward_matches_autograd_of_the_oracle(name, dtype):
    mode, heads, (b, t, c, h, w), (ha, wa), lengths = AGG_BWD_CASES[name]
    rng = np.random.RandomState(7000 + len(name))
    x, _, pad = synth_inputs(rng, b, t, c, h, w, lengths)
    x = x + 0.25 * rng.standard_normal(x.shape).astype(np.float32) * (~pad)[:, :, None, None, None]
    attn = random_attention(rng, heads, pad, ha, wa)
    gout = rng.standard_normal((b, c, h, w)).astype(np.float32)
    if dtype == torch.bfloat16:
        x, gout = bf16_round(x), bf16_round(gout)
    # oracle gradients (CPU autograd through the as-written algorithm)
    xr = torch.from_numpy(x).requires_grad_(True)
    ar = torch.from_numpy(attn).requires_grad_(mode != "mean")
    ref = temporal_aggregator_torch(xr, torch.from_numpy(pad), ar, mode)
    ref.backward(torch.from_numpy(gout))
    # CUDA path
    xd = to_dev(x, dtype=dtype).requires_grad_(True)
    ad = to_dev(attn).requires_grad_(mode != "mean")
    out = c2s.TemporalAggregator(mode)(xd, pad_mask=to_dev(pad), attn_mask=ad)
    out.backward(to_dev(gout, dtype=dtype))
    assert "agg_backward" in _lib.last_kernel() or "spread" in _lib.last_kernel() or "unpool" in _lib.last_kernel()
    tol = 1e-4 if dtype == torch.float32 else 1e-2
    assert rel_err(out.detach().float().cpu().numpy(), ref.detach().numpy()) < tol
    assert xd.grad.dtype == dtype and xd.grad.shape == xd.shape
    assert rel_err(xd.grad.float().cpu().numpy(), xr.grad.numpy()) < tol
    gx = xd.grad.float().cpu().numpy()
    assert np.all(gx[pad] == 0.0)  # padded frames receive exactly zero gradient
    if mode != "mean":
        assert rel_err(ad.grad.cpu().numpy(), ar.grad.numpy()) < tol


def _ltae(kw, seed, kind="ltae"):
    rng = np.random.RandomState(seed)
    m = (c2s.LTAE if kind == "ltae" else c2s.LTAE4WTAE)(**kw)
    randomise(m, rng)
    return m.cuda(), rng


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_ltae_train_mode_forward_from_a_spec_with_injected_dropout(dtype):
    """BatchNorm batch statistics + dropout masks on the attention and after the ReLU (tae.py:445-448, :837)."""
    kw = dict(in_channels=128, n_head=16, d_k=4, mlp=[256, 128], d_model=256)
    m, rng = _ltae(kw, 31)
    b, t, h, w = 2, 19, 4, 4
    x, pos, pad = synth_inputs(rng, b, t, 128, h, w, [19, 11])
    attn_keep = (rng.uniform(size=(16, b, t, h, w)) >= 0.1).astype(np.uint8)
    mlp_keep = (rng.uniform(size=(b, 128, h, w)) >= 0.2).astype(np.uint8)
    xr = x if dtype == torch.float32 else bf16_round(x)
    n = b * h * w
    ref_out, ref_attn, (rm, rv) = ltae_forward(
        oracle_config("ltae", kw), oracle_params(m), xr, pos, pad, training=True,
        attn_keep=np.ascontiguousarray(attn_keep.transpose(0, 1, 3, 4, 2)).reshape(16, n, 1, t),
        mlp_keep=np.ascontiguousarray(mlp_keep.transpose(0, 2, 3, 1)).reshape(n, 128))
    spec = ops.LtaeSpec(n_head=16, d_k=4, d_model=256, has_inconv=True, c_out=128, pe_mode=_lib.PE_SINUSOID,
                        bn_batch_stats=True, attn_drop_p=0.1, mlp_drop_p=0.2)
    out, attn, stats = ops.ltae_forward(
        to_dev(x, dtype=dtype), to_dev(pos), to_dev(pad), m._params(torch.device("cuda")), spec,
        attn_keep=to_dev(attn_keep), mlp_keep=to_dev(mlp_keep))[:3]
    tol = 1e-4 if dtype == torch.float32 else 1e-2
    assert rel_err(attn.cpu().numpy(), ref_attn) < (1e-4 if dtype == torch.float32 else 1e-3)
    assert rel_err(out.float().cpu().numpy(), ref_out) < tol
    a = attn.cpu().numpy()
    assert np.all(a[attn_keep == 0] == 0.0)


def _loss_weights(rng, out_shape, attn_shape):
    return (rng.standard_normal(out_shape).astype(np.float32), rng.standard_normal(attn_shape).astype(np.float32))


@pytest.mark.parametrize("variant", ["sinusoid", "doy", "abs_rel", "add_linear", "no_pe"])
def test_ltae_backward_matches_autograd_of_the_oracle(variant):
    extra = {"sinusoid": {}, "doy": dict(use_doy=True), "abs_rel": dict(use_abs_rel_enc=True),
             "add_linear": dict(add_linear=True), "no_pe": dict(positional_encoding=False)}[variant]
    kw = dict(in_channels=32, n_head=4, d_k=4, mlp=[64, 32], d_model=64, **extra)
    m, rng = _ltae(kw, 50 + len(variant))
    m.eval()
    b, t, h, w = 2, 7, 3, 3
    x, pos, pad = synth_inputs(rng, b, t, 32, h, w, [7, 4], doy=variant == "doy", abs_rel=variant == "abs_rel")
    x = x + 0.3 * rng.standard_normal(x.shape).astype(np.float32) * (~pad)[:, :, None, None, None]
    pos = None if variant == "no_pe" else pos
    wo, wa = _loss_weights(rng, (b, 32, h, w), (4, b, t, h, w))
    # oracle: CPU autograd through the as-written algorithm
    P = {k: torch.from_numpy(v).clone().requires_grad_(np.issubdtype(v.dtype, np.floating) and "running" not in k
                                                        and "denom" not in k)
         for k, v in oracle_params(m).items()}
    xr = torch.from_numpy(x).requires_grad_(True)
    ro, ra = ltae_forward_torch(oracle_config("ltae", kw), P, xr, None if pos is None else torch.from_numpy(pos),
                                torch.from_numpy(pad))
    ((ro * torch.from_numpy(wo)).sum() + (ra * torch.from_numpy(wa)).sum()).backward()
    # CUDA forward + backward through the module
    xd = to_dev(x).requires_grad_(True)
    out, attn = m(xd, batch_positions=to_dev(pos), pad_mask=to_dev(pad))
    assert "ltae_forward" in _lib.last_kernel()
    ((out * to_dev(wo)).sum() + (attn * to_dev(wa)).sum()).backward()
    assert _lib.last_kernel() in ("ltae_backward<general>", "ltae_inconv_grad")  # the backward ran on the CUDA kernels
    assert rel_err(xd.grad.cpu().numpy(), xr.grad.numpy()) < 1e-3
    gmax = max(float(P[name].grad.abs().max()) for name, _ in m.named_parameters())
    for name, p in m.named_parameters():
        ref = P[name].grad
        assert ref is not None, name
        assert p.grad is not None, name
        # fc1_k.bias shifts every score of a head alike, so its true gradient is zero (both sides return rounding
        # noise): the floor of the comparison is relative to the largest parameter gradient
        diff = float(np.abs(p.grad.cpu().numpy() - ref.numpy()).max())
        assert diff <= 1e-3 * max(float(ref.abs().max()), 1e-3 * gmax), (name, diff)


def test_utae_bottleneck_trains_end_to_end():
    """LTAE -> two aggregations -> loss: gradients reach x, the skip features and every encoder parameter, and one
    SGD step on the CUDA path lowers the loss (training mode: batch statistics + dropout)."""
    kw = dict(in_channels=128, n_head=16, d_k=4, mlp=[256, 128], d_model=256)
    m, rng = _ltae(kw, 91)
    m.train()
    agg = c2s.TemporalAggregator("att_group")
    b, t = 2, 9
    x4, pos, pad = synth_inputs(rng, b, t, 128, 4, 4, [9, 5])
    x3 = synth_inputs(rng, b, t, 64, 8, 8, [9, 5])[0]
    x1 = synth_inputs(rng, b, t, 64, 32, 32, [9, 5])[0]
    x4d, x3d, x1d = (to_dev(v).requires_grad_(True) for v in (x4, x3, x1))
    opt = torch.optim.SGD(m.parameters(), lr=1e-3)
    torch.manual_seed(0)
    losses = []
    for _ in range(3):
        opt.zero_grad()
        torch.manual_seed(0)  # same dropout masks every iteration so that the loss is comparable
        out, att = m(x4d, batch_positions=to_dev(pos), pad_mask=to_dev(pad))
        s3 = agg(x3d, pad_mask=to_dev(pad), attn_mask=att)
        s1 = agg(x1d, pad_mask=to_dev(pad), attn_mask=att)
        loss = out.pow(2).mean() + s3.pow(2).mean() + s1.pow(2).mean()
        loss.backward()
        losses.append(float(loss.detach()))
        opt.step()
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in m.parameters())
    assert x4d.grad is not None and x3d.grad is not None and x1d.grad is not None
    assert int(m.mlp[2].num_batches_tracked) == 3
    assert losses[-1] < losses[0]


@pytest.mark.parametrize("name", ["train_utae", "train_timeunet", "train_wtae"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_ltae_training_step_matches_the_reference_autograd(name, dtype):
    """Shipped shapes (16 heads, d_model 256) in training mode: BatchNorm batch statistics and BOTH dropouts on the
    realisation the reference itself drew (tests/golden/make_train_golden.py recorded its keep masks).  Outputs, running
    statistics, grad_x and every parameter gradient of the CUDA path against the REFERENCE's own autograd."""
    from golden_util import load, load_grads
    from c2s_testlib import module_from_fixture
    cfg, inp, params, outs = load(name)
    ref_g = load_grads(name)
    kind = cfg["kind"]
    m = module_from_fixture(cfg, params).train()
    m.assume_zero_padded = True
    x = inp["x"] if dtype == torch.float32 else bf16_round(inp["x"])
    if dtype == torch.bfloat16:
        # bf16 features: rounding x moves the reference's own answer by ~1e-2, so the comparison is with the torch-CPU
        # oracle on the rounded x (test_oracle_golden.py pins that oracle, outputs AND gradients, on these fixtures)
        outs, ref_g = _oracle_training_step(cfg, inp, params, x)
    xd = to_dev(x, dtype=dtype).requires_grad_(True)
    mk = to_dev(inp["mlp_keep"]) if kind == "ltae" else None
    with c2s.modules.injected_dropout(to_dev(inp["attn_keep"]), mk):
        res = m(xd, batch_positions=to_dev(inp["positions"]), pad_mask=to_dev(inp["pad_mask"]))
    out, attn = res if kind == "ltae" else (None, res)
    tol = 1e-4 if dtype == torch.float32 else 1e-2
    assert rel_err(attn.detach().cpu().numpy(), outs["attn"]) < (1e-4 if dtype == torch.float32 else 2e-3)
    loss = (attn * to_dev(inp["w_attn"])).sum()
    if out is not None:
        assert rel_err(out.detach().float().cpu().numpy(), outs["out"]) < tol
        assert rel_err(m.mlp[2].running_mean.cpu().numpy(), outs["running_mean"]) < 1e-3
        assert rel_err(m.mlp[2].running_var.cpu().numpy(), outs["running_var"]) < 1e-3
        loss = loss + (out.float() * to_dev(inp["w_out"])).sum()
    loss.backward()
    assert _lib.last_kernel() in ("ltae_backward<general>", "ltae_inconv_grad", "ltae_fold_backward")
    gtol = 1e-3 if dtype == torch.float32 else 2e-2
    assert rel_err(xd.grad.float().cpu().numpy(), ref_g["x"]) < gtol
    gmax = max(float(np.abs(v).max()) for k, v in ref_g.items() if k != "x")
    for pname, p in m.named_parameters():
        ref = ref_g[pname]
        assert p.grad is not None, pname
        diff = float(np.abs(p.grad.cpu().numpy() - ref).max())
        # fc1_k.bias shifts every score of a head alike (true gradient 0): floor relative to the largest gradient
        assert diff <= (2e-3 if dtype == torch.float32 else 3e-2) * max(float(np.abs(ref).max()), 1e-3 * gmax), (pname, diff)


def _oracle_training_step(cfg, inp, params, x):
    kw = dict(cfg["kwargs"])
    if cfg["kind"] != "ltae":
        kw["mlp"] = [kw["d_model"], 1]
    P = {k: torch.from_numpy(v).clone() for k, v in params.items()}
    names = [k for k in P if P[k].is_floating_point() and "running" not in k and "denom" not in k]
    for k in names:
        P[k].requires_grad_(True)
    xr = torch.from_numpy(x).requires_grad_(True)
    res = ltae_forward_torch(oracle_config(cfg["kind"], cfg["kwargs"]), P, xr, torch.from_numpy(inp["positions"]),
                             torch.from_numpy(inp["pad_mask"]), attn_only=cfg["kind"] != "ltae", training=True,
                             attn_keep=inp["attn_keep"], mlp_keep=inp.get("mlp_keep"))
    outs = {}
    if cfg["kind"] == "ltae":
        out, attn, (mean, var) = res
        n = out.shape[0] * out.shape[2] * out.shape[3]
        outs["out"] = out.detach().numpy()
        outs["running_mean"] = (0.9 * params["mlp.2.running_mean"] + 0.1 * mean.numpy()).astype(np.float32)
        outs["running_var"] = (0.9 * params["mlp.2.running_var"] + 0.1 * var.numpy() * n / (n - 1)).astype(np.float32)
        loss = (out * torch.from_numpy(inp["w_out"])).sum() + (attn * torch.from_numpy(inp["w_attn"])).sum()
    else:
        attn = res
        loss = (attn * torch.from_numpy(inp["w_attn"])).sum()
    outs["attn"] = attn.detach().numpy()
    loss.backward()
    grads = {"x": xr.grad.numpy()}
    for k in names:
        grads[k] = P[k].grad.numpy() if P[k].grad is not None else np.zeros(tuple(P[k].shape), np.float32)
    return outs, grads


def test_ltae4wtae_backward_without_attention_gradient_is_zero():
    kw = dict(in_channels=128, n_head=16, d_k=4, d_model=256)
    m, rng = _ltae(kw, 12, "ltae4wtae")
    x, pos, pad = synth_inputs(rng, 2, 7, 128, 4, 4, [7, 3])
    xd = to_dev(x).requires_grad_(True)
    attn = m(xd, batch_positions=to_dev(pos), pad_mask=to_dev(pad))
    (attn.detach().sum() + 0.0 * xd.sum()).backward()  # no gradient reaches the attention
    assert float(xd.grad.abs().max()) == 0.0


def test_encoder_without_inconv_raises_in_backward():
    m, rng = _ltae(dict(in_channels=64, n_head=4, d_k=8, mlp=[64, 48], d_model=None), 13)
    x, pos, pad = synth_inputs(rng, 2, 5, 64, 3, 2, [5, 3])
    out, attn = m(to_dev(x).requires_grad_(True), batch_positions=to_dev(pos), pad_mask=to_dev(pad))  # forward is served
    with pytest.raises(_lib.C2SError, match="no torch fallback"):
        out.sum().backward()


@pytest.mark.parametrize("c_in,variant,lengths", [
    (128, "sinusoid", [61, 27, 5]), (64, "sinusoid", [61, 33, 0]), (128, "doy", [40, 17, 40]), (64, "abs_rel", [13, 13, 2]),
    (128, "no_pe", [61, 61, 61]), (64, "sinusoid_T64", [64, 64, 1]), (128, "sinusoid", [48, 30, 1]),
    (128, "sinusoid_wide", [61, 40, 27]), (64, "sinusoid_wide", [33, 61, 27, 50])])
def test_ltae_tensor_core_backward_matches_the_general_kernel_and_the_oracle(c_in, variant, lengths):
    """Stage A on the tensor cores (``ltae_backward<tc,C=..>``: bf16 features, shipped head layout) against the fp32
    CUDA-core kernel on the same call (every output of ``c2s_ltae_backward``) and, through the module in training mode
    with an injected dropout realisation, against autograd of the torch-CPU oracle: ragged series up to T = 61 / 64,
    an all-padded series, every positional variant the kernel serves."""
    extra = {"sinusoid": {}, "sinusoid_T64": {}, "sinusoid_wide": {}, "doy": dict(use_doy=True),
             "abs_rel": dict(use_abs_rel_enc=True), "no_pe": dict(positional_encoding=False)}[variant]
    kw = dict(in_channels=c_in, n_head=16, d_k=4, mlp=[256, 64], d_model=256, **extra)
    m, rng = _ltae(kw, 7 + c_in + len(variant))
    m.train()
    m.assume_zero_padded = True
    # "wide": more pixel tiles (192 / 256) than SMs, so the persistent CTAs walk over several tiles
    b, t, (h, w) = len(lengths), max(lengths), ((32, 16) if variant == "sinusoid_wide" else (4, 4))
    x, pos, pad = synth_inputs(rng, b, t, c_in, h, w, lengths, doy=variant == "doy", abs_rel=variant == "abs_rel")
    x = bf16_round(x + 0.3 * rng.standard_normal(x.shape).astype(np.float32) * (~pad)[:, :, None, None, None])
    pos = None if variant == "no_pe" else pos
    attn_keep = (rng.uniform(size=(16, b, t, h, w)) >= 0.1).astype(np.uint8)
    mlp_keep = (rng.uniform(size=(b, 64, h, w)) >= 0.2).astype(np.uint8)
    wo, wa = _loss_weights(rng, (b, 64, h, w), (16, b, t, h, w))

    def run(general):
        for p_ in m.parameters():
            p_.grad = None
        xd = to_dev(x, dtype=torch.bfloat16).requires_grad_(True)
        with _lib.option(_lib.OPT_LTAE_BWD_KERNEL, 1 if general else 0):
            with c2s.modules.injected_dropout(to_dev(attn_keep), to_dev(mlp_keep)):
                out, attn = m(xd, batch_positions=to_dev(pos), pad_mask=to_dev(pad))
            kernels = []
            orig = ops.ltae_backward

            def spy(*a_, **k_):
                r = orig(*a_, **k_)
                kernels.append(_lib.last_kernel())
                return r
            ops.ltae_backward = spy
            try:
                ((out.float() * to_dev(wo)).sum() + (attn * to_dev(wa)).sum()).backward()
            finally:
                ops.ltae_backward = orig
        return xd.grad.float().cpu().numpy(), {n_: p_.grad.cpu().numpy().copy() for n_, p_ in m.named_parameters()}, kernels

    gx_tc, gp_tc, k_tc = run(False)
    gx_gen, gp_gen, k_gen = run(True)
    # learnable positional tables (day of year) need grad_pe, which only the CUDA-core kernel forms
    served = "ltae_backward<general>" if variant in ("doy", "abs_rel") else f"ltae_backward<tc,C={c_in}>"
    assert k_tc == [served] and k_gen == ["ltae_backward<general>"]
    assert np.isfinite(gx_tc).all()
    assert rel_err(gx_tc, gx_gen) < 1.5e-2  # both round grad_x to bf16; the tensor-core operands are bf16 (measured <= 9e-3)
    gmax = max(float(np.abs(v).max()) for v in gp_gen.values())
    for name, ref in gp_gen.items():
        diff = float(np.abs(gp_tc[name] - ref).max())
        # the outputs of the kernel itself agree to < 1e-2 (tools/experiments/bwd_tc_errors.py); stage F then takes
        # differences of them (in_norm.bias: direct term against the folded ones), hence the oracle's bf16 criterion
        assert diff <= 3e-2 * max(float(np.abs(ref).max()), 1e-3 * gmax), (name, diff)
    # the oracle's autograd on the same rounded features and the same dropout realisation
    cfg = {"kind": "ltae", "kwargs": kw}
    inp = {"positions": pos if pos is not None else np.zeros((b, t), np.int64), "pad_mask": pad, "attn_keep": attn_keep,
           "mlp_keep": mlp_keep, "w_out": wo, "w_attn": wa}
    if variant == "no_pe" or 0 in lengths:
        # _oracle_training_step always passes positions; an all-padded series is all zeros, its GroupNorm has rstd =
        # eps^-1/2 = 316 and turns the bf16 rounding of grad_x into O(1) differences: the comparison with the fp32
        # kernel above covers both
        return
    _, ref_g = _oracle_training_step(cfg, inp, {k_: v for k_, v in oracle_params(m).items()}, x)
    assert rel_err(gx_tc, ref_g["x"]) < 2e-2
    gmax = max(float(np.abs(v).max()) for k_, v in ref_g.items() if k_ != "x")
    for name, g_ in gp_tc.items():
        ref = ref_g[name]
        diff = float(np.abs(g_ - ref).max())
        assert diff <= 3e-2 * max(float(np.abs(ref).max()), 1e-3 * gmax), (name, diff)


@pytest.mark.parametrize("c_in,lengths,hw", [(128, [61, 27, 5], (4, 4)), (64, [40, 61, 33, 1], (32, 16))])
def test_attention_only_encoder_backward_on_the_tensor_cores(c_in, lengths, hw):
    """LTAE4WTAE (W-TAE, tae.py:507-635) in training mode: the attention-only variant of the tensor-core stage A against the
    fp32 CUDA-core kernel on the same call (grad_x and every parameter gradient)."""
    kw = dict(in_channels=c_in, n_head=16, d_k=4, d_model=256)
    m, rng = _ltae(kw, 11 + c_in, kind="wtae")
    m.train()
    m.assume_zero_padded = True
    b, t, (h, w) = len(lengths), max(lengths), hw
    x, pos, pad = synth_inputs(rng, b, t, c_in, h, w, lengths)
    x = bf16_round(x + 0.3 * rng.standard_normal(x.shape).astype(np.float32) * (~pad)[:, :, None, None, None])
    attn_keep = (rng.uniform(size=(16, b, t, h, w)) >= 0.1).astype(np.uint8)
    wa = rng.standard_normal((16, b, t, h, w)).astype(np.float32)

    def run(general):
        for p_ in m.parameters():
            p_.grad = None
        xd = to_dev(x, dtype=torch.bfloat16).requires_grad_(True)
        kernels = []
        orig = ops.ltae_backward

        def spy(*a_, **k_):
            r = orig(*a_, **k_)
            kernels.append(_lib.last_kernel())
            return r
        with _lib.option(_lib.OPT_LTAE_BWD_KERNEL, 1 if general else 0):
            with c2s.modules.injected_dropout(to_dev(attn_keep), None):
                attn = m(xd, batch_positions=to_dev(pos), pad_mask=to_dev(pad))
            ops.ltae_backward = spy
            try:
                (attn * to_dev(wa)).sum().backward()
            finally:
                ops.ltae_backward = orig
        return xd.grad.float().cpu().numpy(), {n_: p_.grad.cpu().numpy().copy() for n_, p_ in m.named_parameters()
                                               if p_.grad is not None}, kernels

    gx_tc, gp_tc, k_tc = run(False)
    gx_gen, gp_gen, k_gen = run(True)
    assert k_tc == [f"ltae_backward<tc,C={c_in},attention>"] and k_gen == ["ltae_backward<general>"]
    assert np.isfinite(gx_tc).all() and rel_err(gx_tc, gx_gen) < 1.5e-2
    assert set(gp_tc) == set(gp_gen)
    gmax = max(float(np.abs(v).max()) for v in gp_gen.values())
    for name, ref in gp_gen.items():
        diff = float(np.abs(gp_tc[name] - ref).max())
        assert diff <= 3e-2 * max(float(np.abs(ref).max()), 1e-3 * gmax), (name, diff)
