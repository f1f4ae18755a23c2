"""The U-TAE training step at the shapes tools/bench_training.py measures, and each backward stage at its edge shapes,
against a float64 reference.

The reference is the torch port of the reference modules (``oracle/torch_port.py``) run in float64 on the device, on the
same bf16-rounded inputs and the same dropout keep masks as the kernels; the stages of the L-TAE backward that have no
module of their own are restated here in a few lines of float64 ATen.  Errors are ``rel_err`` (max|d| / max|ref|) per
tensor, with the bounds the suite applies to the same kernels at small shapes.

What only these shapes reach: the aggregator backward split into time chunks (x2: 8 chunks of 8 frames, x4: 4 chunks of
16 at B = 16, T = 61), BatchNorm batch statistics with several rows per partial sum (N > 1024), the split-K weight GEMM
of stage M at 32 splits, group widths 3 and 16 of the output GroupNorm, every instantiation of the in-projection
gradient, and stage F on its own.
"""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import crop2seg_b200 as c2s
from bench import make_lengths, make_positions
from crop2seg_b200 import _lib, ops
from oracle.torch_port import _sinusoid, ltae_forward_torch, temporal_aggregator_torch
from golden_util import load, load_grads, rel_err
from c2s_testlib import (PAD_PATTERNS, bf16_round, oracle_config, oracle_params, pattern_masks, random_attention,
                         randomise, to_dev)

F64 = torch.float64
UTAE = dict(in_channels=128, n_head=16, d_k=4, mlp=[256, 128], d_model=256)
B, T, HEADS = 16, 61, 16
LEVELS = (32, 64, 128)  # resolutions of the three 64-channel skip features
HOLES = {3: "mid_block", 9: "lead16"}  # samples of the batch with interior / leading holes instead of a suffix pad


def _report(what, **errs):
    print("float64 max error:", what, " ".join(f"{k}={v:.3g}" for k, v in errs.items()))


@pytest.fixture(scope="module", autouse=True)
def _peak_memory():
    if torch.cuda.is_available():
        torch.cuda.reset_peak_memory_stats()
    yield
    if torch.cuda.is_available():
        print(f"float64 tests: peak device memory {torch.cuda.max_memory_allocated() / 2 ** 30:.2f} GiB")


class _MaxRel:
    """``rel_err`` of one tensor whose slices are compared one at a time on the device."""

    def __init__(self):
        self.d = self.r = 0.0

    def add(self, got, ref):
        self.d = max(self.d, float((got.to(F64) - ref).abs().max()))
        self.r = max(self.r, float(ref.abs().max()))

    @property
    def err(self):
        return self.d / max(self.r, 1e-30)


def _training_masks(seed):
    """Lengths and positions of tools/bench_training.py (rank 0), two samples with holes instead of a suffix pad."""
    lengths = make_lengths(B, seed)
    pos, pad = make_positions(lengths, seed)
    holes = pattern_masks(T, tuple(HOLES.values()))
    rng = np.random.RandomState(seed + 7)
    for row, i in zip(holes, HOLES):
        pad[i] = row
        pos[i] = np.cumsum(rng.randint(2, 11, size=T))  # a hole keeps the dates of the frames around it
    return pos, pad


def _param_errors(got, ref):
    """Per tensor ``max|d| / max(max|ref|, 1e-3 * max over params)``, the measure the bound ``tol`` of the suite's
    parameter gradients applies to; returns the largest and its tensor."""
    gmax = max(float(r.abs().max()) for r in ref.values())
    worst = (-1.0, "")
    for name, r in ref.items():
        g = got[name]
        assert g is not None and torch.isfinite(g).all(), name
        floor = max(float(r.abs().max()), 1e-3 * gmax)
        worst = max(worst, (float((g.to(F64).reshape(r.shape) - r).abs().max()) / floor, name))
    return worst


# ---- the float64 oracle ------------------------------------------------------------------------------------------------

def test_float64_oracle_matches_the_reference_training_fixture():
    """Float64 inputs keep the torch port in float64: on the reference's training fixture it meets the bounds
    tests/test_oracle_golden.py applies to the float32 port."""
    cfg, inp, params, outs = load("train_utae")
    grads = load_grads("train_utae")
    c = oracle_config(cfg["kind"], cfg["kwargs"])
    P = {k: torch.from_numpy(v).to(F64) if v.dtype.kind == "f" else torch.from_numpy(v) for k, v in params.items()}
    for k in grads:
        if k != "x":
            P[k].requires_grad_(True)
    x = torch.from_numpy(inp["x"]).to(F64).requires_grad_(True)
    out, attn, (mean, var) = ltae_forward_torch(c, P, x, torch.from_numpy(inp["positions"]),
                                                torch.from_numpy(inp["pad_mask"]), training=True,
                                                attn_keep=inp["attn_keep"], mlp_keep=inp["mlp_keep"])
    assert out.dtype == F64 and attn.dtype == F64 and mean.dtype == F64
    assert rel_err(out.detach().numpy(), outs["out"]) < 5e-5
    # the float32 port meets 2e-6 here because it rounds as the float32 reference does (1.1e-7); float64 lands 2.4e-6
    # away, the reference's own rounding of scores that span 11 in the exponent
    assert rel_err(attn.detach().numpy(), outs["attn"]) < 5e-6
    n = x.shape[0] * x.shape[3] * x.shape[4]
    rm = 0.9 * params["mlp.2.running_mean"] + 0.1 * mean.numpy()
    rv = 0.9 * params["mlp.2.running_var"] + 0.1 * var.numpy() * n / (n - 1)
    assert rel_err(rm, outs["running_mean"]) < 2e-6 and rel_err(rv, outs["running_var"]) < 2e-6, (rm, rv)
    loss = (out * torch.from_numpy(inp["w_out"])).sum() + (attn * torch.from_numpy(inp["w_attn"])).sum()
    loss.backward()
    assert x.grad.dtype == F64
    assert rel_err(x.grad.numpy(), grads["x"]) < 1e-4
    gmax = max(float(np.abs(g).max()) for k, g in grads.items() if k != "x")
    for k, g in grads.items():
        if k != "x":
            assert float(np.abs(P[k].grad.numpy() - g).max()) <= 1e-4 * max(float(np.abs(g).max()), 1e-2 * gmax), k


# ---- a. the training step at the benchmark placement -------------------------------------------------------------------

@pytest.mark.gpu
def test_training_step_at_the_benchmark_placement(monkeypatch):
    """Forward and backward of LTAE (training mode) and three att_group aggregators exactly as tools/bench_training.py
    runs them, against float64 autograd of the torch port: the L-TAE on all 16 samples at once (BatchNorm couples the
    rows), each aggregator one sample at a time, their attention gradients summed into one grad_attn."""
    monkeypatch.setattr(c2s.modules, "ATTENTION_DROPOUT", 0.1)  # the rate of tae.py:837, which the reference applies
    dev = torch.device("cuda")
    pos_np, pad_np = _training_masks(1234)
    pos, pad = to_dev(pos_np), to_dev(pad_np)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234)

    def feat(c, r):
        x = torch.randn((B, T, c, r, r), device=dev, generator=gen).clamp_(min=0)
        x[pad] = 0
        return x.to(torch.bfloat16).requires_grad_(True)

    x4 = feat(128, 16)
    xs = [feat(64, r) for r in LEVELS]
    enc = c2s.LTAE(**UTAE)
    randomise(enc, np.random.RandomState(1234))
    enc = enc.to(dev).train()
    enc.assume_zero_padded = True
    params = oracle_params(enc)  # before the step, which moves the running statistics
    attn_keep = (torch.rand((HEADS, B, T, 16, 16), device=dev, generator=gen) >= 0.1).to(torch.uint8)
    mlp_keep = (torch.rand((B, 128, 16, 16), device=dev, generator=gen) >= 0.2).to(torch.uint8)
    g_out = torch.randn((B, 128, 16, 16), device=dev, generator=gen).to(torch.bfloat16)
    g_skips = [torch.randn((B, 64, r, r), device=dev, generator=gen).to(torch.bfloat16) for r in LEVELS]

    kernels = []
    for name in ("ltae_backward", "temporal_aggregate_backward"):
        def spy(*a, _orig=getattr(ops, name), **k):
            res = _orig(*a, **k)
            kernels.append(_lib.last_kernel())
            return res
        monkeypatch.setattr(ops, name, spy)
    agg = c2s.TemporalAggregator(mode="att_group")
    with c2s.modules.injected_dropout(attn_keep, mlp_keep):
        out, attn = enc(x4, batch_positions=pos, pad_mask=pad)
    assert _lib.last_ltae_kernel() == "ltae_forward<team,C=128>", _lib.last_ltae_kernel()
    a = attn.detach()
    assert bool((a[attn_keep == 0] == 0).all())  # the injected attention dropout acted
    for b in range(B):
        if not pad_np[b].all():
            assert bool((a[:, b, pad[b]] == 0).all()), b  # padded frames
    skips = [agg(x, pad_mask=pad, attn_mask=attn) for x in xs]
    torch.autograd.backward([out] + skips, [g_out] + g_skips)
    torch.cuda.synchronize()
    assert sorted(kernels) == ["agg_backward_pipe<x2>", "agg_backward_pipe<x4>", "agg_backward_pipe<x8>",
                               "ltae_backward<tc,C=128>"], kernels

    # float64 reference on the device
    names = [k for k, _ in enc.named_parameters()]
    P = {k: torch.from_numpy(v).to(dev) for k, v in params.items()}
    P = {k: v.to(F64) if v.is_floating_point() else v for k, v in P.items()}
    for k in names:
        P[k].requires_grad_(True)
    x4r = x4.detach().to(F64).requires_grad_(True)
    ref_out, ref_attn, (mean, var) = ltae_forward_torch(oracle_config("ltae", UTAE), P, x4r, pos, pad, training=True,
                                                        attn_keep=attn_keep, mlp_keep=mlp_keep, materialise=False)
    errs = {}
    a_ref = ref_attn.detach()
    grad_attn = torch.zeros_like(a_ref)
    for li, (x, s, g) in enumerate(zip(xs, skips, g_skips)):
        e_out, e_gx = _MaxRel(), _MaxRel()
        for b in range(B):
            xb = x[b:b + 1].detach().to(F64).requires_grad_(True)
            ab = a_ref[:, b:b + 1].clone().requires_grad_(True)
            rb = temporal_aggregator_torch(xb, pad[b:b + 1], ab, "att_group")
            gxb, gab = torch.autograd.grad(rb, [xb, ab], g[b:b + 1].to(F64))
            grad_attn[:, b:b + 1] += gab
            e_out.add(s[b:b + 1].detach(), rb.detach())
            e_gx.add(x.grad[b:b + 1], gxb)
            assert bool((x.grad[b][pad[b]] == 0).all()), (li, b)  # padded frames get exactly zero gradient
            del xb, ab, rb, gxb, gab
        errs[f"skip{li}"], errs[f"skip{li}_grad_x"] = e_out.err, e_gx.err
    torch.autograd.backward([ref_out, ref_attn], [g_out.to(F64), grad_attn])

    errs["out"] = rel_err(out.detach().float().cpu().numpy(), ref_out.detach().cpu().numpy())
    errs["attn"] = rel_err(attn.detach().cpu().numpy(), a_ref.cpu().numpy())
    n = B * 16 * 16
    run_mean = 0.9 * P["mlp.2.running_mean"] + 0.1 * mean
    run_var = 0.9 * P["mlp.2.running_var"] + 0.1 * var * n / (n - 1)
    errs["running_mean"] = rel_err(enc.mlp[2].running_mean.cpu().numpy(), run_mean.cpu().numpy())
    errs["running_var"] = rel_err(enc.mlp[2].running_var.cpu().numpy(), run_var.cpu().numpy())
    errs["grad_x4"] = rel_err(x4.grad.float().cpu().numpy(), x4r.grad.cpu().numpy())
    errs["params"], worst = _param_errors({k: p.grad for k, p in enc.named_parameters()}, {k: P[k].grad for k in names})
    _report(f"training step [B=16, T=61, x4 16^2, skips 32^2/64^2/128^2] (largest parameter error: {worst})", **errs)
    assert errs["attn"] < 1e-3 and errs["out"] < 1e-2, errs
    assert all(errs[f"skip{i}"] < 1e-2 and errs[f"skip{i}_grad_x"] < 1e-2 for i in range(3)), errs
    assert errs["running_mean"] < 1e-3 and errs["running_var"] < 1e-3, errs
    assert errs["grad_x4"] < 2e-2 and errs["params"] < 3e-2, (worst, errs)


# ---- b. aggregator backward at the training shapes ---------------------------------------------------------------------

def _agg_backward_kernel(res, dtype, no_pipe):
    s = res // 16
    if dtype == torch.float32 and s == 8:
        return "agg_backward<generic>"  # fp32 vectors hold 4 pixels: no whole x8 cell per thread
    return f"agg_backward{'' if no_pipe else '_pipe'}<x{s}>"


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("res", LEVELS)
def test_aggregator_backward_at_the_training_shapes(res, dtype):
    """B = 16, T = 61, 16 heads on a 16 x 16 attention map, pipelined and register kernels; non-zero data on padded
    frames, which must never count."""
    dev = torch.device("cuda")
    _, pad_np = _training_masks(1234)
    pad = to_dev(pad_np)
    rng = np.random.RandomState(40 + res)
    attn = to_dev(random_attention(rng, HEADS, pad_np, 16, 16))
    gen = torch.Generator(device=dev)
    gen.manual_seed(res)
    x = torch.randn((B, T, 64, res, res), device=dev, generator=gen).to(dtype)
    gout = torch.randn((B, 64, res, res), device=dev, generator=gen).to(dtype)
    got = {}
    for no_pipe in (False, True):
        with _lib.option(_lib.OPT_AGG_KERNEL, int(no_pipe)):
            out = ops.temporal_aggregate_forward(x, pad, attn, "att_group")
            gx, ga = ops.temporal_aggregate_backward(x, pad, attn, gout, "att_group")
            assert _lib.last_kernel() == _agg_backward_kernel(res, dtype, no_pipe), _lib.last_kernel()
        assert gx.dtype == dtype
        got[no_pipe] = (out, gx, ga)
    torch.cuda.synchronize()
    errs = {k: [_MaxRel(), _MaxRel(), _MaxRel()] for k in got}
    for b in range(B):
        xb = x[b:b + 1].to(F64).requires_grad_(True)
        ab = attn[:, b:b + 1].to(F64).requires_grad_(True)
        rb = temporal_aggregator_torch(xb, pad[b:b + 1], ab, "att_group")
        gxb, gab = torch.autograd.grad(rb, [xb, ab], gout[b:b + 1].to(F64))
        for k, (out, gx, ga) in got.items():
            errs[k][0].add(out[b:b + 1], rb.detach())
            errs[k][1].add(gx[b:b + 1], gxb)
            errs[k][2].add(ga[:, b:b + 1], gab)
            assert bool((gx[b][pad[b]] == 0).all()), (k, b)
        del xb, ab, rb, gxb, gab
    tol = 1e-4 if dtype == torch.float32 else 1e-2
    for no_pipe, (e_out, e_gx, e_ga) in errs.items():
        _report(f"{_agg_backward_kernel(res, dtype, no_pipe)} {str(dtype)[6:]} [B=16, T=61, {res}^2]", out=e_out.err,
                grad_x=e_gx.err, grad_attn=e_ga.err)
        assert e_out.err < tol and e_gx.err < tol and e_ga.err < tol, (no_pipe, e_out.err, e_gx.err, e_ga.err)


# ---- c. stage M: c2s_ltae_mlp_backward ---------------------------------------------------------------------------------

MLP_SHAPES = [(16, 256, 128), (16, 256, 64), (16, 256, 32), (16, 256, 256), (16, 256, 48), (4, 52, 12)]
MLP_ROWS = {1: (1, 1, 1), 37: (1, 1, 37), 1587: (3, 23, 23), 4096: (16, 16, 16)}  # N: (B, H, W)
MLP_DROP = 0.2


def _mlp_reference(o, P, keep, train, n_head, bhw):
    """mlp.0 -> BatchNorm1d -> ReLU -> dropout -> out_norm on the rows, tae.py:442-449, 486-488."""
    y = o @ P["mlp_weight"].t() + P["mlp_bias"]
    if train:
        mean, var = y.mean(dim=0), y.var(dim=0, unbiased=False)
    else:
        mean, var = P["bn_running_mean"], P["bn_running_var"]
    r = torch.relu((y - mean) / torch.sqrt(var + 1e-5) * P["bn_weight"] + P["bn_bias"])
    if keep is not None:
        r = r * keep / (1.0 - MLP_DROP)
    z = F.group_norm(r[:, :, None], n_head, P["out_norm_weight"], P["out_norm_bias"], 1e-5)[:, :, 0]
    b, h, w = bhw
    return z.view(b, h, w, -1).permute(0, 3, 1, 2), y, mean, var


def _away_from_the_kink(y, mean, var, bn_w):
    """mlp.2.bias such that no row of a channel lands near the ReLU's kink: the zero crossing is put in the middle of
    the widest gap of the middle half of the sorted rows, so the fp32 kernel and the float64 reference agree on every
    ReLU decision."""
    v, _ = torch.sort((y - mean) / torch.sqrt(var + 1e-5) * bn_w, dim=0)
    n = v.shape[0]
    if n == 1:  # one row: varied distances on both sides of the kink (equal rows would make out_norm degenerate)
        step = torch.arange(v.shape[1], dtype=v.dtype, device=v.device)
        return -v[0] + (0.3 + 0.7 * torch.frac(0.618 * step)) * torch.where(step % 2 == 0, 1.0, -1.0)
    lo, hi = n // 4, max(n // 4 + 1, (3 * n) // 4)
    gaps = v[lo + 1:hi + 1] - v[lo:hi]
    k = lo + gaps.argmax(dim=0)
    return -0.5 * (v.gather(0, k[None])[0] + v.gather(0, k[None] + 1)[0])


@pytest.mark.gpu
@pytest.mark.parametrize("gdtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("with_keep", [False, True])
@pytest.mark.parametrize("mode", ["train_y_rows", "train", "eval"])
@pytest.mark.parametrize("n", sorted(MLP_ROWS))
@pytest.mark.parametrize("shape", MLP_SHAPES)
def test_mlp_backward_stage_m(shape, n, mode, with_keep, gdtype):
    """``ops.ltae_mlp_backward`` against float64 autograd of the rows' chain (training: batch statistics, with the
    pre-BatchNorm rows handed over or recomputed; eval: running statistics)."""
    if n == 1 and mode != "eval":
        pytest.skip("torch's batch norm rejects a single row in training")
    n_head, d_model, c_out = shape
    train = mode != "eval"
    dev = torch.device("cuda")
    bhw = MLP_ROWS[n]
    rng = np.random.RandomState(n + 7 * c_out + d_model)
    f32 = lambda a: torch.from_numpy(np.asarray(a, dtype=np.float32)).to(dev)  # noqa: E731
    o = f32(rng.standard_normal((n, d_model)))
    P = {"mlp_weight": f32(rng.standard_normal((c_out, d_model)) / np.sqrt(d_model)),
         "mlp_bias": f32(0.5 * rng.standard_normal(c_out)),
         "bn_weight": f32(1.0 + 0.3 * rng.standard_normal(c_out)),
         "bn_running_mean": f32(0.3 * rng.standard_normal(c_out)),
         "bn_running_var": f32(rng.uniform(0.5, 2.0, c_out)),
         "out_norm_weight": f32(1.0 + 0.3 * rng.standard_normal(c_out)),
         "out_norm_bias": f32(0.5 * rng.standard_normal(c_out))}
    P64 = {k: v.to(F64) for k, v in P.items()}
    _, y, mean, var = _mlp_reference(o.to(F64), dict(P64, bn_bias=torch.zeros_like(P64["bn_weight"])), None, train,
                                     n_head, bhw)
    P["bn_bias"] = _away_from_the_kink(y, mean, var, P64["bn_weight"]).float()
    P64["bn_bias"] = P["bn_bias"].to(F64)
    b, h, w = bhw
    keep = to_dev((rng.uniform(size=(b, c_out, h, w)) >= MLP_DROP).astype(np.uint8)) if with_keep else None
    g_out = to_dev(rng.standard_normal((b, c_out, h, w)).astype(np.float32)).to(gdtype)

    spec = ops.LtaeSpec(n_head=n_head, d_k=1, d_model=d_model, has_inconv=True, c_out=c_out, bn_batch_stats=train,
                        mlp_drop_p=MLP_DROP if with_keep else 0.0)
    res = ops.ltae_mlp_backward(o, g_out, P, mean.float(), var.float(), spec, mlp_keep=keep,
                                y_rows=y.float() if mode == "train_y_rows" else None)
    assert _lib.last_kernel() == "ltae_mlp_backward<grad_weight>", _lib.last_kernel()

    o64 = o.to(F64).requires_grad_(True)
    names = ("mlp_weight", "mlp_bias", "bn_weight", "bn_bias", "out_norm_weight", "out_norm_bias")
    for k in names:
        P64[k].requires_grad_(True)
    keep_rows = None if keep is None else keep.permute(0, 2, 3, 1).reshape(n, c_out).to(F64)
    ref, _, _, _ = _mlp_reference(o64, P64, keep_rows, train, n_head, bhw)
    got = torch.autograd.grad(ref, [o64] + [P64[k] for k in names], g_out.to(F64))
    e_o = rel_err(res["grad_o"].cpu().numpy(), got[0].cpu().numpy())
    e_p, worst = _param_errors({k: res[k] for k in names}, dict(zip(names, got[1:])))
    _report(f"ltae_mlp_backward [N={n}, (n_head, d_model, c_out)={shape}, {mode}, keep={with_keep}, "
            f"grad_out {str(gdtype)[6:]}] (largest parameter error: {worst})", grad_o=e_o, params=e_p)
    # fp32 sums over up to 4096 rows whose terms cancel (in training the gradient of mlp.0.bias is zero in exact
    # arithmetic, and a 2-channel out_norm group amplifies its rounding): up to 3.3e-4 on a B200; 30x below the
    # end-to-end parameter bound, and a dropped keep scale (x1.25) or row is far above it
    assert e_o < 1e-3 and e_p < 1e-3, (e_o, e_p, worst)


@pytest.mark.gpu
def test_mlp_backward_rejects_out_norm_groups_wider_than_16():
    dev = torch.device("cuda")
    n_head, d_model, c_out = 16, 256, 272
    P = {"mlp_weight": torch.zeros((c_out, d_model), device=dev)}
    for k in ("mlp_bias", "bn_weight", "bn_bias", "out_norm_weight", "out_norm_bias"):
        P[k] = torch.ones(c_out, device=dev)
    spec = ops.LtaeSpec(n_head=n_head, d_k=1, d_model=d_model, has_inconv=True, c_out=c_out, bn_batch_stats=True)
    _lib.reset_launch_count()
    with pytest.raises(_lib.C2SError, match="status 2.*exceed the supported 16"):
        ops.ltae_mlp_backward(torch.zeros((4, d_model), device=dev), torch.zeros((1, c_out, 2, 2), device=dev), P,
                              P["bn_bias"], P["bn_weight"], spec)
    assert _lib.launch_count() == 0


# ---- d. c2s_ltae_inconv_grad -------------------------------------------------------------------------------------------

INCONV_SHAPES = [(16, 16, 128), (16, 16, 64), (16, 16, 256), (16, 32, 256), (2, 8, 10)]  # (n_head, dh, C)


@pytest.mark.gpu
@pytest.mark.parametrize("bias", [True, False])
@pytest.mark.parametrize("n", [1, 37, 129, 4096])
@pytest.mark.parametrize("shape", INCONV_SHAPES)
def test_inconv_grad(shape, n, bias):
    """The direct term of the in-projection gradient added (+=) to prefilled outputs, against a float64 einsum.  The
    shapes run 2, 4, 8 and 16 outputs per thread and the scalar zn load (C % 4 != 0)."""
    n_head, dh, c = shape
    d_model = n_head * dh
    dev = torch.device("cuda")
    gen = torch.Generator(device=dev)
    gen.manual_seed(n + c + dh)
    g_o = torch.randn((n, d_model), device=dev, generator=gen)
    zn = torch.randn((n, n_head, c), device=dev, generator=gen)
    sa = torch.randn((n, 16), device=dev, generator=gen)
    gw0 = torch.randn((d_model, c), device=dev, generator=gen)
    gb0 = torch.randn(d_model, device=dev, generator=gen)
    gw, gb = gw0.clone(), (gb0.clone() if bias else None)
    ops.ltae_inconv_grad(g_o, zn, sa if bias else None, gw, gb, n_head)
    assert _lib.last_kernel() == "ltae_inconv_grad", _lib.last_kernel()
    g3 = g_o.to(F64).view(n, n_head, dh)
    ref_w = gw0.to(F64) + torch.einsum("nhi,nhc->hic", g3, zn.to(F64)).reshape(d_model, c)
    errs = {"weight": rel_err(gw.cpu().numpy(), ref_w.cpu().numpy())}
    if bias:
        ref_b = gb0.to(F64) + torch.einsum("nhi,nh->hi", g3, sa[:, :n_head].to(F64)).reshape(d_model)
        errs["bias"] = rel_err(gb.cpu().numpy(), ref_b.cpu().numpy())
    _report(f"ltae_inconv_grad [N={n}, (n_head, dh, C)={shape}]", **errs)
    assert all(e < 1e-5 for e in errs.values()), errs


@pytest.mark.gpu
@pytest.mark.parametrize("n_head,dh,c", [(8, 33, 64), (16, 16, 257)])
def test_inconv_grad_rejects_unsupported_shapes(n_head, dh, c):
    dev = torch.device("cuda")
    d_model = n_head * dh
    _lib.reset_launch_count()
    with pytest.raises(_lib.C2SError, match="status 2"):
        ops.ltae_inconv_grad(torch.zeros((4, d_model), device=dev), torch.zeros((4, n_head, c), device=dev), None,
                             torch.zeros((d_model, c), device=dev), None, n_head)
    assert _lib.launch_count() == 0


# ---- e. stage F: c2s_ltae_fold_backward --------------------------------------------------------------------------------

FOLD_CASES = {"c128": (128, 16, 4, 256, 128), "c64": (64, 16, 4, 256, 64), "c32": (32, 4, 8, 64, 32)}
FOLD_NAMES = ("in_norm_weight", "in_norm_bias", "inconv_weight", "inconv_bias", "query", "key_weight", "key_bias")


@pytest.mark.gpu
@pytest.mark.parametrize("bt", [(16, 61), (2, 5)])
@pytest.mark.parametrize("case", sorted(FOLD_CASES))
def test_fold_backward_stage_f(case, bt):
    """Stage F alone: the gradients of the folded score weights U and cpos (random here, written into the workspace of
    one ``ltae_backward`` call) through the folding of csrc/c2s_ltae_prep.cuh, against float64 autograd of the folding
    written out below.  The learned linear map of the positional table (add_linear) makes the kernel also return
    grad_pe through the scores."""
    c, n_head, d_k, d_model, c_out = FOLD_CASES[case]
    b, t = bt
    dev = torch.device("cuda")
    rng = np.random.RandomState(c + t)
    m = c2s.LTAE(in_channels=c, n_head=n_head, d_k=d_k, mlp=[d_model, c_out], d_model=d_model, add_linear=True)
    randomise(m, rng)
    m = m.to(dev)
    spec = ops.LtaeSpec(n_head=n_head, d_k=d_k, d_model=d_model, has_inconv=True, c_out=c_out,
                        pe_mode=_lib.PE_SINUSOID_LINEAR, bn_batch_stats=True)
    params = {k: v.detach() for k, v in m._params(dev).items()}
    h, w = 2, 2
    gen = torch.Generator(device=dev)
    gen.manual_seed(c + t)
    x = torch.randn((b, t, c, h, w), device=dev, generator=gen).to(torch.bfloat16)
    pos = to_dev(np.cumsum(rng.randint(2, 11, size=(b, t)), axis=1))
    res = ops.ltae_backward(x, pos, None, params, torch.randn((b * h * w, d_model), device=dev, generator=gen), None,
                            spec, need_grad_pe=True)
    assert res["grad_pe"] is not None
    g_u = torch.randn((c, 16), device=dev, generator=gen)
    g_u[:, n_head:] = 0  # as stage A leaves the columns of absent heads
    g_cpos = torch.randn((b, t, 16), device=dev, generator=gen)
    g_cpos[..., n_head:] = 0
    for k, v in (("grad_u", g_u), ("grad_cpos", g_cpos), ("grad_gamma", torch.randn(c, device=dev, generator=gen)),
                 ("grad_beta", torch.randn(c, device=dev, generator=gen))):
        res[k].copy_(v)
    pe0 = res["grad_pe"].clone()
    folded = ops.ltae_fold_backward(res, {k: True for k in FOLD_NAMES}, {k: tuple(params[k].shape) for k in FOLD_NAMES},
                                    grad_pe_through_scores=True)
    assert _lib.last_kernel() == "ltae_fold_backward", _lib.last_kernel()
    torch.cuda.synchronize()

    # the folding (c2s_ltae_prep.cuh, include/crop2seg_b200.h:230-231) in float64
    P = {k: params[k].to(F64).requires_grad_(True) for k in FOLD_NAMES}
    gamma, beta, wc, bc = P["in_norm_weight"], P["in_norm_bias"], P["inconv_weight"], P["inconv_bias"]
    q, bk = P["query"].reshape(n_head, d_k), P["key_bias"].view(n_head, d_k)
    wk = P["key_weight"].view(n_head, d_k, d_model)
    pe = _sinusoid(pos, params["pe_denom"].to(F64), n_head, params["pe_fc_weight"].to(F64),
                   params["pe_fc_bias"].to(F64)).requires_grad_(True)
    qk = torch.einsum("hj,hjd->hd", q, wk) / math.sqrt(d_k)
    u = gamma[:, None] * (qk @ wc).t()  # [C, h]
    cpos = torch.einsum("hd,btd->bth", qk, bc + wc @ beta + pe) + (q * bk).sum(-1) / math.sqrt(d_k)
    loss = (u * g_u[:, :n_head].to(F64)).sum() + (cpos * g_cpos[..., :n_head].to(F64)).sum() \
        + (gamma * res["grad_gamma"].to(F64)).sum() + (beta * res["grad_beta"].to(F64)).sum()
    got = torch.autograd.grad(loss, [P[k] for k in FOLD_NAMES] + [pe])
    ref = dict(zip(FOLD_NAMES, got[:-1]))
    e_p, worst = _param_errors(folded, ref)
    e_pe = rel_err(res["grad_pe"].cpu().numpy(), (pe0.to(F64) + got[-1]).cpu().numpy())
    _report(f"ltae_fold_backward [{case}, B={b}, T={t}] (largest parameter error: {worst})", params=e_p, grad_pe=e_pe)
    assert e_p < 1e-4 and e_pe < 1e-4, (e_p, e_pe, worst)


# ---- f. batch statistics of the training forward -----------------------------------------------------------------------

BN_ROWS = {1024: (4, 16, 16), 1025: (1, 25, 41), 1587: (3, 23, 23), 4096: (16, 16, 16)}  # N: (B, H, W)


@pytest.mark.gpu
@pytest.mark.parametrize("n", sorted(BN_ROWS))
def test_batch_statistics_of_the_training_forward(n):
    """``bn_batch_stats``: the statistics reduce min(N, 1024) partial sums, so N > 1024 puts several rows in a part and
    a ragged N leaves trailing parts empty.  mlp.0.bias is offset by +40: the mean is far from 0 against the spread."""
    b, h, w = BN_ROWS[n]
    t = 13
    rng = np.random.RandomState(n)
    m = c2s.LTAE(**UTAE)
    randomise(m, rng)
    with torch.no_grad():
        m.mlp[0].bias += 40.0
    m = m.cuda()
    masks = pattern_masks(t, tuple(p for p in PAD_PATTERNS if p != "all_padded"), n=b, seed=n)
    x = np.maximum(rng.standard_normal((b, t, 128, h, w)).astype(np.float32), 0)
    x = bf16_round(x * (~masks)[:, :, None, None, None])
    pos = np.cumsum(rng.randint(2, 11, size=(b, t)), axis=1)
    spec = ops.LtaeSpec(n_head=16, d_k=4, d_model=256, has_inconv=True, c_out=128, pe_mode=_lib.PE_SINUSOID,
                        zero_padded=True, bn_batch_stats=True)
    out, attn, (mean, var) = ops.ltae_forward(to_dev(x, dtype=torch.bfloat16), to_dev(pos), to_dev(masks),
                                              m._params(torch.device("cuda")), spec)[:3]
    P = {k: torch.from_numpy(v).cuda() for k, v in oracle_params(m).items()}
    P = {k: v.to(F64) if v.is_floating_point() else v for k, v in P.items()}
    ref_out, ref_attn, (ref_mean, ref_var) = ltae_forward_torch(oracle_config("ltae", UTAE), P, to_dev(x).to(F64),
                                                                to_dev(pos), to_dev(masks), training=True,
                                                                materialise=False)
    errs = {"mean": rel_err(mean.cpu().numpy(), ref_mean.cpu().numpy()),
            "var": rel_err(var.cpu().numpy(), ref_var.cpu().numpy()),
            "out": rel_err(out.float().cpu().numpy(), ref_out.cpu().numpy()),
            "attn": rel_err(attn.cpu().numpy(), ref_attn.cpu().numpy())}
    _report(f"ltae_forward batch statistics [N={n}, T={t}]", **errs)
    assert errs["mean"] < 1e-3 and errs["var"] < 1e-3 and errs["attn"] < 1e-3 and errs["out"] < 1e-2, errs
