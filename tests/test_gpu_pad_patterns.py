"""The temporal kernels on pad masks with leading, interior and scattered padded frames.

The reference derives its pad mask from the raw input (an all-zero frame anywhere in the series is padded), so a mask is
an arbitrary set of frames, and every kernel on the temporal hot path handles it as one: the L-TAE kernels build 64-bit
frame sets with two 32-frame ballots, pick 16-, 4- or 1-frame copies from them, skip dead 16-frame blocks and pivot
their GroupNorm sums on the first live frame; the aggregators build per-sample frame lists and sort the samples by
their number of valid frames.  Every case here runs one sample per named pattern (``c2s_testlib.PAD_PATTERNS``) or a
batch that cycles through them, and compares each sample with the oracles.
"""
import numpy as np
import pytest
import torch
from torch import nn

import crop2seg_b200 as c2s
from crop2seg_b200 import _lib, ops
from oracle import aggregate_skip_conv, ltae4wtae_forward, ltae_forward
from oracle.torch_port import ltae_forward_torch, temporal_aggregator_torch
from golden_util import rel_err
from c2s_testlib import (PAD_PATTERNS, bf16_round, hot_path_parity, oracle_config, oracle_params, pattern_masks,
                         random_attention, randomise, synth_inputs_masked, to_dev)

pytestmark = pytest.mark.gpu

T_VALUES = (61, 64, 33, 20)
UTAE = dict(in_channels=128, n_head=16, d_k=4, mlp=[256, 128], d_model=256)
TIMEUNET = dict(in_channels=64, n_head=16, d_k=4, mlp=[256, 64], d_model=256)
WTAE = dict(in_channels=128, n_head=16, d_k=4, d_model=256)
WTAE64 = dict(in_channels=64, n_head=16, d_k=4, d_model=256)


def _report(what, **errs):
    print("pad-pattern max error:", what, " ".join(f"{k}={v:.3g}" for k, v in errs.items()))


def _module(kind, kw, seed):
    rng = np.random.RandomState(seed)
    m = (c2s.LTAE if kind == "ltae" else c2s.LTAE4WTAE)(**kw)
    randomise(m, rng)
    return m.cuda().eval(), rng


def _oracle(kind, kw, params, x, pos, pad, chunk=64):
    """The numpy oracle, ``chunk`` samples at a time (it materialises [rows, T, 256] activations)."""
    cfg = oracle_config(kind, kw)
    outs, attns = [], []
    for s in range(0, x.shape[0], chunk):
        sl = slice(s, s + chunk)
        if kind == "ltae":
            o, a = ltae_forward(cfg, params, x[sl], pos[sl], pad[sl])
            outs.append(o)
        else:
            a = ltae4wtae_forward(cfg, params, x[sl], pos[sl], pad[sl])
        attns.append(a)
    return (np.concatenate(outs) if outs else None), np.concatenate(attns, axis=1)


def _check_per_sample(names, pad, out, ref_out, attn, ref_attn, out_tol=None):
    """Every sample against the oracle on its own: bounds of test_gpu_oracle.py (``out_tol[b]`` may raise the output
    bound of sample b, see ``_output_spread``), plus the exact zeros and the sums of the attention.  Returns the largest
    errors."""
    e_att = e_out = 0.0
    for bi in range(pad.shape[0]):
        name = names[bi]
        if attn is not None:
            a = attn[:, bi]  # [h, T, H, W]
            e = rel_err(a, ref_attn[:, bi])
            e_att = max(e_att, e)
            assert e < 1e-3, (bi, name, "attention", e)
            assert np.all(np.abs(a.sum(axis=1) - 1.0) < 1e-5), (bi, name, "attention sum")
            if not pad[bi].all():
                assert np.all(a[:, pad[bi]] == 0.0), (bi, name, "attention of padded frames")
        if out is not None:
            o = out[bi]
            assert np.isfinite(o).all(), (bi, name)
            e = rel_err(o, ref_out[bi])
            e_out = max(e_out, e)
            assert e < (1e-2 if out_tol is None else out_tol[bi]), (bi, name, "output", e)
    return e_att, e_out


def _output_spread(kind, kw, params, xr, pos, pad, ref_out, seed):
    """Per sample, how far the oracle's output moves when its features move by 1e-5 relative, about the working
    precision of the tensor-core kernels (hi/lo bf16 operands, fp32 sums).  Where a GroupNorm group of the output holds
    nearly equal values the output is ill-conditioned: in the 400-sample batch below one pixel of sample 145 moves by
    1.7e-3 for a 1e-6 perturbation (a typical sample: 1e-5), and the slab and team kernels, whose rows before the MLP
    agree to 4e-6, both land 1.5e-2 away from the oracle there."""
    noise = 1.0 + 1e-5 * np.random.RandomState(seed).standard_normal(xr.shape).astype(np.float32)
    moved, _ = _oracle(kind, kw, params, (xr * noise).astype(np.float32), pos, pad)
    return np.array([rel_err(moved[i], ref_out[i]) for i in range(xr.shape[0])])


# ---- L-TAE forward: one sample per pattern, on every kernel that serves these masks ---------------------------------

FWD_CASES = {
    # name: (kind, kwargs, kernel option, feature dtype, return_att, kernel that must serve the call)
    "team128": ("ltae", UTAE, _lib.LTAE_KERNEL_AUTO, torch.bfloat16, True, "ltae_forward<team,C=128>"),
    "team64": ("ltae", TIMEUNET, _lib.LTAE_KERNEL_AUTO, torch.bfloat16, False, "ltae_forward<team,C=64>"),
    "slab128": ("ltae", UTAE, _lib.LTAE_KERNEL_SLAB, torch.bfloat16, True, "ltae_forward<fa,C=128>"),
    "slab64": ("ltae", TIMEUNET, _lib.LTAE_KERNEL_SLAB, torch.bfloat16, True, "ltae_forward<fa,C=64>"),
    "slab128_attention": ("wtae", WTAE, _lib.LTAE_KERNEL_SLAB, torch.bfloat16, True, "ltae_forward<fa,C=128>"),
    "slab64_attention": ("wtae", WTAE64, _lib.LTAE_KERNEL_SLAB, torch.bfloat16, True, "ltae_forward<fa,C=64>"),
    "general_bf16": ("ltae", UTAE, _lib.LTAE_KERNEL_GENERAL, torch.bfloat16, True, "ltae_forward<general>"),
    "general_fp32": ("ltae", TIMEUNET, _lib.LTAE_KERNEL_GENERAL, torch.float32, True, "ltae_forward<general>"),
}


@pytest.mark.parametrize("t", T_VALUES)
@pytest.mark.parametrize("zero_padded", [False, True])
@pytest.mark.parametrize("case", sorted(FWD_CASES))
def test_ltae_forward_on_every_pad_pattern(case, zero_padded, t):
    kind, kw, choice, dtype, return_att, kernel = FWD_CASES[case]
    m, rng = _module(kind, kw, 300 + t + len(case))
    m.assume_zero_padded = zero_padded
    names = PAD_PATTERNS
    masks = pattern_masks(t, names, seed=t)
    b, h, w = len(names), 4, 4  # two 8-pixel tiles per sample
    x, pos, pad = synth_inputs_masked(rng, b, t, kw["in_channels"], h, w, masks, zero_padded)
    xr = bf16_round(x) if dtype == torch.bfloat16 else x
    ref_out, ref_attn = _oracle(kind, kw, oracle_params(m), xr, pos, pad)
    with _lib.option(_lib.OPT_LTAE_KERNEL, choice), torch.no_grad():
        if kind == "ltae":
            out, attn = m(to_dev(x, dtype=dtype), batch_positions=to_dev(pos), pad_mask=to_dev(pad), return_att=return_att)
        else:
            out, attn = None, m(to_dev(x, dtype=dtype), batch_positions=to_dev(pos), pad_mask=to_dev(pad))
        assert _lib.last_ltae_kernel() == kernel, _lib.last_ltae_kernel()
    assert (attn is None) == (not return_att)
    e_att, e_out = _check_per_sample(names, pad, None if out is None else out.float().cpu().numpy(), ref_out,
                                     None if attn is None else attn.cpu().numpy(), ref_attn)
    _report(f"{kernel} [{case}, T={t}, zero_padded={zero_padded}]", attn=e_att, out=e_out)


TRAIN_PATTERNS = ("lead17", "mid_block", "alternate", "ballot_edge", "one_mid", "sparse_random")


@pytest.mark.parametrize("t", [61, 64])
@pytest.mark.parametrize("zero_padded", [False, True])
def test_ltae_train_mode_forward_with_injected_dropout_on_pad_patterns(zero_padded, t):
    """Team kernel C = 128 with dropout (BatchNorm batch statistics over every sample, keep masks on the attention and
    after the ReLU) against the numpy oracle in training mode."""
    m, rng = _module("ltae", UTAE, 90 + t)
    masks = pattern_masks(t, TRAIN_PATTERNS)
    b, h, w = len(TRAIN_PATTERNS), 4, 4
    x, pos, pad = synth_inputs_masked(rng, b, t, 128, h, w, masks, zero_padded)
    attn_keep = (rng.uniform(size=(16, b, t, h, w)) >= 0.1).astype(np.uint8)
    mlp_keep = (rng.uniform(size=(b, 128, h, w)) >= 0.2).astype(np.uint8)
    n = b * h * w
    ref_out, ref_attn, _ = ltae_forward(
        oracle_config("ltae", UTAE), oracle_params(m), bf16_round(x), pos, pad, training=True,
        attn_keep=np.ascontiguousarray(attn_keep.transpose(0, 1, 3, 4, 2)).reshape(16, n, 1, t),
        mlp_keep=np.ascontiguousarray(mlp_keep.transpose(0, 2, 3, 1)).reshape(n, 128))
    spec = ops.LtaeSpec(n_head=16, d_k=4, d_model=256, has_inconv=True, c_out=128, pe_mode=_lib.PE_SINUSOID,
                        zero_padded=zero_padded, bn_batch_stats=True, attn_drop_p=0.1, mlp_drop_p=0.2)
    out, attn = ops.ltae_forward(to_dev(x, dtype=torch.bfloat16), to_dev(pos), to_dev(pad), m._params(torch.device("cuda")),
                                 spec, attn_keep=to_dev(attn_keep), mlp_keep=to_dev(mlp_keep))[:2]
    assert _lib.last_ltae_kernel() == "ltae_forward<team,C=128>", _lib.last_ltae_kernel()
    a, o = attn.cpu().numpy(), out.float().cpu().numpy()
    e_att, e_out = rel_err(a, ref_attn), rel_err(o, ref_out)
    assert e_att < 1e-3 and e_out < 1e-2, (e_att, e_out)
    assert np.isfinite(o).all()
    assert np.all(a[attn_keep == 0] == 0.0)
    for bi in range(b):
        assert np.all(a[:, bi, pad[bi]] == 0.0), TRAIN_PATTERNS[bi]
    _report(f"ltae_forward<team,C=128> training [T={t}, zero_padded={zero_padded}]", attn=e_att, out=e_out)


# ---- many samples per persistent CTA ---------------------------------------------------------------------------------

MANY_CASES = {
    # H*W = 16: two 8-pixel tiles per sample, 800 tiles; every CTA and every team crosses many sample boundaries
    "team128": ("ltae", UTAE, _lib.LTAE_KERNEL_AUTO, True, "ltae_forward<team,C=128>"),
    "team64": ("ltae", TIMEUNET, _lib.LTAE_KERNEL_AUTO, False, "ltae_forward<team,C=64>"),
    "slab64": ("ltae", TIMEUNET, _lib.LTAE_KERNEL_SLAB, True, "ltae_forward<fa,C=64>"),
}


@pytest.mark.parametrize("zero_padded", [False, True])
@pytest.mark.parametrize("case", sorted(MANY_CASES))
def test_ltae_forward_many_samples_per_cta_each_with_its_own_mask(case, zero_padded):
    kind, kw, choice, return_att, kernel = MANY_CASES[case]
    b, t, h, w = 400, 61, 4, 4
    m, rng = _module(kind, kw, 500 + len(case))
    m.assume_zero_padded = zero_padded
    masks = pattern_masks(t, n=b, seed=17)
    names = [(PAD_PATTERNS + ("random",))[i % (len(PAD_PATTERNS) + 1)] for i in range(b)]
    x, pos, pad = synth_inputs_masked(rng, b, t, kw["in_channels"], h, w, masks, zero_padded)
    with _lib.option(_lib.OPT_LTAE_KERNEL, choice), torch.no_grad():
        out, attn = m(to_dev(x, dtype=torch.bfloat16), batch_positions=to_dev(pos), pad_mask=to_dev(pad),
                      return_att=return_att)
        assert _lib.last_ltae_kernel() == kernel, _lib.last_ltae_kernel()
    xr, params = bf16_round(x), oracle_params(m)
    ref_out, ref_attn = _oracle(kind, kw, params, xr, pos, pad)
    # the output bound is 1e-2, or twice the oracle's own spread at the kernels' working precision where that is larger
    out_tol = np.maximum(1e-2, 2.0 * _output_spread(kind, kw, params, xr, pos, pad, ref_out, seed=b))
    e_att, e_out = _check_per_sample(names, pad, out.float().cpu().numpy(), ref_out,
                                     None if attn is None else attn.cpu().numpy(), ref_attn, out_tol)
    _report(f"{kernel} [B={b}, zero_padded={zero_padded}]", attn=e_att, out=e_out,
            samples_above_1e_2_bound=int((out_tol > 1e-2).sum()))


# ---- backward on the tensor cores ------------------------------------------------------------------------------------

def _oracle_grads(kind, kw, params, x, pos, pad, attn_keep, mlp_keep, wo, wa):
    """Autograd of the torch-CPU oracle in training mode on the same features and dropout realisation."""
    P = {k: torch.from_numpy(v).clone() for k, v in params.items()}
    names = [k for k in P if P[k].is_floating_point() and "running" not in k and "denom" not in k]
    for k in names:
        P[k].requires_grad_(True)
    xr = torch.from_numpy(x).requires_grad_(True)
    res = ltae_forward_torch(oracle_config(kind, kw), P, xr, torch.from_numpy(pos), torch.from_numpy(pad),
                             attn_only=kind != "ltae", training=True, attn_keep=attn_keep, mlp_keep=mlp_keep)
    if kind == "ltae":
        out, attn, _ = res
        loss = (out * torch.from_numpy(wo)).sum() + (attn * torch.from_numpy(wa)).sum()
    else:
        loss = (res * torch.from_numpy(wa)).sum()
    loss.backward()
    grads = {k: (P[k].grad.numpy() if P[k].grad is not None else np.zeros(tuple(P[k].shape), np.float32)) for k in names}
    return xr.grad.numpy(), grads


def _run_backward(m, kind, x, pos, pad, attn_keep, mlp_keep, wo, wa, general):
    """Training-mode forward and backward through the module; returns grad_x, the parameter gradients and the
    ``c2s_ltae_backward`` kernels that ran."""
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
        with c2s.modules.injected_dropout(to_dev(attn_keep), None if mlp_keep is None else to_dev(mlp_keep)):
            res = m(xd, batch_positions=to_dev(pos), pad_mask=to_dev(pad))
        if kind == "ltae":
            out, attn = res
            loss = (out.float() * to_dev(wo)).sum() + (attn * to_dev(wa)).sum()
        else:
            loss = (res * to_dev(wa)).sum()
        ops.ltae_backward = spy
        try:
            loss.backward()
        finally:
            ops.ltae_backward = orig
    grads = {n_: p_.grad.cpu().numpy().copy() for n_, p_ in m.named_parameters() if p_.grad is not None}
    return xd.grad.float().cpu().numpy(), grads, kernels


def _compare_grads(gx, gp, ref_gx, ref_gp, gx_tol):
    """Bounds of test_ltae_tensor_core_backward_matches_the_general_kernel_and_the_oracle; returns the largest errors."""
    assert np.isfinite(gx).all()
    e_x = rel_err(gx, ref_gx)
    assert e_x < gx_tol, e_x
    assert set(gp) <= set(ref_gp)
    gmax = max(float(np.abs(v).max()) for v in ref_gp.values())
    e_p = 0.0
    for name, g_ in gp.items():
        ref = ref_gp[name]
        floor = max(float(np.abs(ref).max()), 1e-3 * gmax)
        diff = float(np.abs(g_ - ref).max())
        e_p = max(e_p, diff / floor)
        assert diff <= 3e-2 * floor, (name, diff)
    return e_x, e_p


def _backward_case(kind, kw, b, t, h, w, masks, seed, with_oracle):
    c_in = kw["in_channels"]
    m, rng = _module(kind, kw, seed)
    m.train()
    m.assume_zero_padded = True
    x, pos, pad = synth_inputs_masked(rng, b, t, c_in, h, w, masks, zero_padded=True)
    x = bf16_round(x + 0.3 * rng.standard_normal(x.shape).astype(np.float32) * (~pad)[:, :, None, None, None])
    attn_keep = (rng.uniform(size=(16, b, t, h, w)) >= 0.1).astype(np.uint8)
    c_out = kw["mlp"][1] if kind == "ltae" else None
    mlp_keep = (rng.uniform(size=(b, c_out, h, w)) >= 0.2).astype(np.uint8) if kind == "ltae" else None
    wo = rng.standard_normal((b, c_out, h, w)).astype(np.float32) if kind == "ltae" else None
    wa = rng.standard_normal((16, b, t, h, w)).astype(np.float32)
    params = oracle_params(m)  # before any step: the training forward only moves the running statistics
    gx_tc, gp_tc, k_tc = _run_backward(m, kind, x, pos, pad, attn_keep, mlp_keep, wo, wa, general=False)
    gx_gen, gp_gen, k_gen = _run_backward(m, kind, x, pos, pad, attn_keep, mlp_keep, wo, wa, general=True)
    served = f"ltae_backward<tc,C={c_in}" + (">" if kind == "ltae" else ",attention>")
    assert k_tc == [served] and k_gen == ["ltae_backward<general>"], (k_tc, k_gen)
    assert set(gp_tc) == set(gp_gen)
    # both round grad_x to bf16; the tensor-core operands are bf16
    e_gen = _compare_grads(gx_tc, gp_tc, gx_gen, gp_gen, 1.5e-2)
    e_ora = (float("nan"), float("nan"))
    if with_oracle:
        ref_gx, ref_gp = _oracle_grads(kind, kw, params, x, pos, pad, attn_keep, mlp_keep, wo, wa)
        e_ora = _compare_grads(gx_tc, gp_tc, ref_gx, ref_gp, 2e-2)
    return served, e_gen, e_ora


BWD_CASES = {"c64": ("ltae", dict(TIMEUNET)), "c128": ("ltae", dict(UTAE, mlp=[256, 64])),
             "c128_attention": ("wtae", WTAE), "c64_attention": ("wtae", WTAE64)}


@pytest.mark.parametrize("t", T_VALUES)
@pytest.mark.parametrize("case", sorted(BWD_CASES))
def test_ltae_tensor_core_backward_on_pad_patterns(case, t, monkeypatch):
    """One sample per pattern (all but ``all_padded``: an all-zero series has rstd = eps^-1/2 and turns the bf16 rounding
    of grad_x into O(1) differences against the oracle) against the fp32 CUDA-core kernel and the oracle's autograd."""
    monkeypatch.setattr(c2s.modules, "ATTENTION_DROPOUT", 0.1)  # the rate of tae.py:837, which the oracle applies
    kind, kw = BWD_CASES[case]
    names = tuple(n_ for n_ in PAD_PATTERNS if n_ != "all_padded")
    served, e_gen, e_ora = _backward_case(kind, kw, len(names), t, 4, 4, pattern_masks(t, names), 700 + t + len(case),
                                          with_oracle=True)
    _report(f"{served} [T={t}]", grad_x_vs_general=e_gen[0], params_vs_general=e_gen[1], grad_x_vs_oracle=e_ora[0],
            params_vs_oracle=e_ora[1])


@pytest.mark.parametrize("case", ["c64", "c128"])
def test_ltae_tensor_core_backward_many_samples_per_cta(case, monkeypatch):
    """160 samples x 2 tiles: more tiles than SMs, so a persistent CTA moves from sample to sample and rebuilds its pad
    mask and positional tables each time; the masks cycle through the patterns (an all-padded series included) and
    random ones.  Against the fp32 CUDA-core kernel on the same call."""
    monkeypatch.setattr(c2s.modules, "ATTENTION_DROPOUT", 0.1)
    kind, kw = BWD_CASES[case]
    b, t = 160, 61
    served, e_gen, _ = _backward_case(kind, kw, b, t, 4, 4, pattern_masks(t, n=b, seed=5), 800 + len(case),
                                      with_oracle=False)
    _report(f"{served} [B={b}]", grad_x_vs_general=e_gen[0], params_vs_general=e_gen[1])


# ---- aggregators -------------------------------------------------------------------------------------------------------

# x2 up-sampling onto 32 x 16 pixels: 64 or more whole 16-byte vectors per plane, the shape of the pipelined kernels
# (the reference up-samples when H exceeds the attention map's width, temporal_aggregator.py:17)
AGG_HEADS, AGG_C, AGG_HW, AGG_AHW = 4, 16, (32, 16), (16, 8)
AGG_CASES = [("att_group", t) for t in T_VALUES] + [(mode, t) for mode in ("att_mean", "mean") for t in (64, 33)]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("mode,t", AGG_CASES)
def test_aggregator_on_pad_patterns(mode, t, dtype):
    """Forward and backward against autograd of the torch-CPU oracle (bounds of
    test_aggregator_backward_matches_autograd_of_the_oracle), padded frames get exactly zero gradient; for att_group the
    pipelined and register kernels, and the staged and global attention taps, agree bit for bit.  The samples have
    different valid counts and holes, so the pipelined kernels walk them in a reordered sequence."""
    names = PAD_PATTERNS if mode != "mean" else tuple(n_ for n_ in PAD_PATTERNS if n_ != "all_padded")  # mean: 0 / 0
    masks = pattern_masks(t, names)
    b = len(names)
    rng = np.random.RandomState(900 + t + len(mode))
    (h, w), (ha, wa) = AGG_HW, AGG_AHW
    x, _, pad = synth_inputs_masked(rng, b, t, AGG_C, h, w, masks, zero_padded=False)  # padded frames never count
    attn = random_attention(rng, AGG_HEADS, pad, ha, wa)
    gout = rng.standard_normal((b, AGG_C, h, w)).astype(np.float32)
    if dtype == torch.bfloat16:
        x, gout = bf16_round(x), bf16_round(gout)
    xr = torch.from_numpy(x).requires_grad_(True)
    ar = torch.from_numpy(attn).requires_grad_(mode != "mean")
    ref = temporal_aggregator_torch(xr, torch.from_numpy(pad), ar, mode)
    ref.backward(torch.from_numpy(gout))
    ref = ref.detach().numpy()
    tol = 1e-4 if dtype == torch.float32 else 1e-2
    xd, pd, ad, gd = to_dev(x, dtype=dtype), to_dev(pad), to_dev(attn), to_dev(gout, dtype=dtype)
    errs = {}
    res = {}
    for no_pipe in ((False, True) if mode == "att_group" else (False,)):
        with _lib.option(_lib.OPT_AGG_KERNEL, int(no_pipe)):
            out = ops.temporal_aggregate_forward(xd, pd, ad, mode)
            k_fwd = _lib.last_kernel()
            gx, ga = ops.temporal_aggregate_backward(xd, pd, ad, gd, mode, need_attn=mode != "mean")
            k_bwd = _lib.last_kernel()
        if mode == "att_group":
            assert ("pipe" in k_fwd) == (not no_pipe) and ("pipe" in k_bwd) == (not no_pipe), (k_fwd, k_bwd)
            assert k_fwd.startswith("agg_forward") and k_bwd.startswith("agg_backward"), (k_fwd, k_bwd)
        o, g = out.float().cpu().numpy(), gx.float().cpu().numpy()
        assert gx.dtype == dtype
        errs["out"] = max(errs.get("out", 0.0), rel_err(o, ref))
        errs["grad_x"] = max(errs.get("grad_x", 0.0), rel_err(g, xr.grad.numpy()))
        assert rel_err(o, ref) < tol, (no_pipe, rel_err(o, ref))
        assert rel_err(g, xr.grad.numpy()) < tol, (no_pipe, rel_err(g, xr.grad.numpy()))
        assert np.all(g[pad] == 0.0), no_pipe  # padded frames receive exactly zero gradient
        if mode != "mean":
            errs["grad_attn"] = max(errs.get("grad_attn", 0.0), rel_err(ga.cpu().numpy(), ar.grad.numpy()))
            assert rel_err(ga.cpu().numpy(), ar.grad.numpy()) < tol, no_pipe
        res[no_pipe] = (out, gx)
    if mode == "att_group":
        assert torch.equal(res[False][0], res[True][0])  # same taps, same accumulation order
        taps = {}
        for global_taps in (False, True):
            with _lib.option(_lib.OPT_AGG_TAPS, int(global_taps)):
                taps[global_taps] = (ops.temporal_aggregate_forward(xd, pd, ad, mode),
                                     *ops.temporal_aggregate_backward(xd, pd, ad, gd, mode))
        assert torch.equal(taps[False][0], taps[True][0])
        assert torch.equal(taps[False][1], taps[True][1])
        assert rel_err(taps[False][2].cpu().numpy(), taps[True][2].cpu().numpy()) < 1e-5  # float atomics reorder
    _report(f"aggregator {mode} {str(dtype)[6:]} [T={t}]", **errs)


def _skip_conv_block(rng):
    p = {"0.weight": (rng.standard_normal((64, 64, 1, 1)) / 8).astype(np.float32),
         "0.bias": (0.1 * rng.standard_normal(64)).astype(np.float32),
         "1.weight": (1.0 + 0.3 * rng.standard_normal(64)).astype(np.float32),
         "1.bias": (0.2 * rng.standard_normal(64)).astype(np.float32),
         "1.running_mean": (0.3 * rng.standard_normal(64)).astype(np.float32),
         "1.running_var": rng.uniform(0.5, 2.0, 64).astype(np.float32),
         "1.num_batches_tracked": np.array(3, dtype=np.int64)}
    m = nn.Sequential(nn.Conv2d(64, 64, 1), nn.BatchNorm2d(64), nn.ReLU())
    m.load_state_dict({k: torch.from_numpy(v) for k, v in p.items()}, strict=True)
    return p, m.cuda().eval()


@pytest.mark.parametrize("t", T_VALUES)
def test_aggregator_skip_conv_on_pad_patterns(t):
    rng = np.random.RandomState(950 + t)
    masks = pattern_masks(t)
    b = masks.shape[0]
    x, _, pad = synth_inputs_masked(rng, b, t, 64, 16, 16, masks, zero_padded=False)
    x = bf16_round(x)
    attn = random_attention(rng, 16, pad, 8, 8)
    params, conv = _skip_conv_block(rng)
    with torch.no_grad():
        out = c2s.TemporalAggregator("att_group").forward_skip_conv(to_dev(x, dtype=torch.bfloat16), to_dev(pad),
                                                                    to_dev(attn), conv)
    assert _lib.last_kernel() == "agg_skipconv<x2>", _lib.last_kernel()
    ref = aggregate_skip_conv(x, pad, attn, params, round_skip=bf16_round)
    o = out.float().cpu().numpy()
    worst = 0.0
    for bi in range(b):
        e = rel_err(o[bi], ref[bi])
        worst = max(worst, e)
        assert e < 1e-2, (PAD_PATTERNS[bi], e)
    _report(f"agg_skipconv<x2> [T={t}]", out=worst)


# ---- one U-TAE placement step -----------------------------------------------------------------------------------------

@pytest.mark.parametrize("t", [61, 64])
def test_utae_step_on_pad_patterns(t):
    """The L-TAE at the bottleneck, then the attention-weighted aggregation of two skip features, every sample through
    the oracles (``hot_path_parity``)."""
    masks = pattern_masks(t)
    b = masks.shape[0]
    enc, rng = _module("ltae", UTAE, 60 + t)
    enc.assume_zero_padded = True
    x4, pos, pad = synth_inputs_masked(rng, b, t, 128, 4, 4, masks, zero_padded=True)
    xs = [bf16_round(synth_inputs_masked(rng, b, t, 64, r, r, masks, zero_padded=True)[0]) for r in (8, 32)]
    x4d, posd, padd = to_dev(x4, dtype=torch.bfloat16), to_dev(pos), to_dev(pad)
    xsd = [to_dev(v, dtype=torch.bfloat16) for v in xs]
    agg = c2s.TemporalAggregator("att_group")
    with torch.no_grad():
        out, attn = enc(x4d, batch_positions=posd, pad_mask=padd)
        skips = [agg(v, pad_mask=padd, attn_mask=attn) for v in xsd]
    torch.cuda.synchronize()
    errs = hot_path_parity(enc, x4d, xsd, posd, padd, out, attn, skips, samples=range(b))
    assert errs["attn"] < 1e-3 and errs["out"] < 1e-2 and max(errs["skips"]) < 1e-2, errs
    assert errs["pad_attention_exactly_zero"]
    i = PAD_PATTERNS.index("all_padded")
    assert all(float(s[i].abs().max()) == 0.0 for s in skips)  # no valid frame: the aggregation is zero
    _report(f"U-TAE step [T={t}]", attn=errs["attn"], out=errs["out"], skips=max(errs["skips"]))
