"""GPU parity against the oracle on seeded inputs at the shapes the specialised kernels serve.

* tensor-core L-TAE (bf16, n_head=16, d_model=256, C in {64,128}, T<=64, H*W % 8 == 0)
* bulk-copy pipelined aggregator (power-of-two up-sampling, >= 64 16-byte vectors per plane)
Both are also compared with the general kernels through the library's kernel-selection options (``c2s_set_option``).
"""
import numpy as np
import pytest
import torch

import crop2seg_b200 as c2s
from crop2seg_b200 import _lib
from oracle import ltae4wtae_forward, ltae_forward
from oracle.torch_port import temporal_aggregator_torch
from golden_util import rel_err
from c2s_testlib import (bf16_round, oracle_config, oracle_params, random_attention, randomise, synth_inputs,
                         to_dev)

pytestmark = pytest.mark.gpu


LTAE_CASES = {
    # name: (kind, kwargs, (B, T, H, W), lengths, extra)
    "utae": ("ltae", dict(in_channels=128, n_head=16, d_k=4, mlp=[256, 128], d_model=256), (3, 61, 8, 8), [61, 27, 44], {}),
    "utae_short": ("ltae", dict(in_channels=128, n_head=16, d_k=4, mlp=[256, 128], d_model=256), (2, 23, 4, 4), [23, 9], {}),
    "utae_all_padded": ("ltae", dict(in_channels=128, n_head=16, d_k=4, mlp=[256, 128], d_model=256), (3, 17, 4, 4), [17, 0, 1], {}),
    "utae_nomask": ("ltae", dict(in_channels=128, n_head=16, d_k=4, mlp=[256, 128], d_model=256), (2, 30, 4, 4), [30, 30], {"no_mask": True}),
    "timeunet": ("ltae", dict(in_channels=64, n_head=16, d_k=4, mlp=[256, 64], d_model=256), (2, 61, 8, 8), [61, 33], {}),
    "utae_doy": ("ltae", dict(in_channels=128, n_head=16, d_k=4, mlp=[256, 128], d_model=256, use_doy=True), (2, 40, 4, 4), [40, 28], {"doy": True}),
    "utae_abs_rel": ("ltae", dict(in_channels=128, n_head=16, d_k=4, mlp=[256, 128], d_model=256, use_abs_rel_enc=True), (2, 40, 4, 4), [31, 40], {"abs_rel": True}),
    "utae_no_pe": ("ltae", dict(in_channels=128, n_head=16, d_k=4, mlp=[256, 128], d_model=256, positional_encoding=False), (2, 33, 4, 4), [33, 30], {"no_positions": True}),
    "utae_dk8": ("ltae", dict(in_channels=128, n_head=16, d_k=8, mlp=[256, 96], d_model=256), (2, 64, 4, 4), [64, 50], {}),
    "wtae": ("ltae4wtae", dict(in_channels=128, n_head=16, d_k=4, d_model=256), (2, 61, 8, 8), [61, 27], {}),
}


def kernel_name_ok(name):
    """The shipped shapes are served by one of the two tensor-core attention kernels, never by the general one."""
    return name.startswith("ltae_forward<fa") or name.startswith("ltae_forward<team")


def _build(kind, kw, seed):
    rng = np.random.RandomState(seed)
    m = (c2s.LTAE if kind == "ltae" else c2s.LTAE4WTAE)(**kw)
    randomise(m, rng)
    return m.cuda().eval(), rng


def _call(m, kind, x, pos, pad, general, dtype):
    choice = _lib.LTAE_KERNEL_GENERAL if general else _lib.LTAE_KERNEL_AUTO
    with _lib.option(_lib.OPT_LTAE_KERNEL, choice), torch.no_grad():
        res = m(to_dev(x, dtype=dtype), batch_positions=to_dev(pos), pad_mask=to_dev(pad))
    kernel = _lib.last_kernel()
    return (res if kind == "ltae" else (None, res)), kernel


@pytest.mark.parametrize("name", sorted(LTAE_CASES))
@pytest.mark.parametrize("zero_padded", [False, True])
def test_tensor_core_ltae_matches_oracle(name, zero_padded):
    kind, kw, (b, t, h, w), lengths, extra = LTAE_CASES[name]
    m, rng = _build(kind, kw, 4000 + len(name))
    m.assume_zero_padded = zero_padded
    x, pos, pad = synth_inputs(rng, b, t, kw["in_channels"], h, w, lengths, doy=extra.get("doy", False),
                               abs_rel=extra.get("abs_rel", False))
    pos = None if extra.get("no_positions") else pos
    pad = None if extra.get("no_mask") else pad
    xr = bf16_round(x)
    cfg, params = oracle_config(kind, kw), oracle_params(m)
    if kind == "ltae":
        ref_out, ref_attn = ltae_forward(cfg, params, xr, pos, pad)
    else:
        ref_out, ref_attn = None, ltae4wtae_forward(cfg, params, xr, pos, pad)
    (out, attn), kernel = _call(m, kind, x, pos, pad, general=False, dtype=torch.bfloat16)
    assert kernel_name_ok(_lib.last_ltae_kernel()), _lib.last_ltae_kernel()
    (out_g, attn_g), kernel_g = _call(m, kind, x, pos, pad, general=True, dtype=torch.bfloat16)
    a = attn.cpu().numpy()
    # bf16 tolerance of the north star is 1e-2; the hi/lo split keeps the tensor-core path near fp32
    assert rel_err(a, ref_attn) < 1e-3
    assert rel_err(attn_g.cpu().numpy(), ref_attn) < 1e-3
    s = a.sum(axis=2)
    assert np.all(np.abs(s - 1.0) < 1e-5)
    if pad is not None:
        for bi in np.nonzero(~pad.all(axis=1))[0]:
            assert np.all(a[:, bi, pad[bi]] == 0.0)
    if kind == "ltae":
        assert out.dtype == torch.bfloat16
        assert rel_err(out.float().cpu().numpy(), ref_out) < 1e-2
        assert rel_err(out_g.float().cpu().numpy(), ref_out) < 1e-2


def test_tensor_core_path_is_selected():
    kind, kw, (b, t, h, w), lengths, _ = LTAE_CASES["utae"]
    m, rng = _build(kind, kw, 1)
    x, pos, pad = synth_inputs(rng, b, t, 128, h, w, lengths)
    (out_tc, attn_tc), kernel = _call(m, kind, x, pos, pad, general=False, dtype=torch.bfloat16)
    # tensor-core attention kernel followed by the tcgen05 row GEMM of the MLP; the U-TAE encoder in eval mode is served
    # by the team-pipelined kernel, the whole-slab kernel on request gives the same answer
    assert kernel == "ltae_mlp<tcgen05>" and _lib.last_ltae_kernel() == "ltae_forward<team,C=128>"
    with _lib.option(_lib.OPT_LTAE_KERNEL, _lib.LTAE_KERNEL_SLAB), torch.no_grad():
        out_s, attn_s = m(to_dev(x, dtype=torch.bfloat16), batch_positions=to_dev(pos), pad_mask=to_dev(pad))
        assert _lib.last_ltae_kernel() == "ltae_forward<fa,C=128>"
    assert rel_err(attn_tc.cpu().numpy(), attn_s.cpu().numpy()) < 1e-4
    assert rel_err(out_tc.float().cpu().numpy(), out_s.float().cpu().numpy()) < 1e-2
    (out_g, attn_g), kernel = _call(m, kind, x, pos, pad, general=True, dtype=torch.bfloat16)
    assert kernel == "ltae_forward<general>"
    assert rel_err(attn_tc.cpu().numpy(), attn_g.cpu().numpy()) < 1e-3
    assert rel_err(out_tc.float().cpu().numpy(), out_g.float().cpu().numpy()) < 1e-2
    _, kernel = _call(m, kind, x, pos, pad, general=False, dtype=torch.float32)
    assert kernel == "ltae_forward<general>"  # fp32 features keep the fp32 CUDA-core kernel
    with pytest.raises(_lib.C2SError):
        _lib.check(_lib.load().c2s_set_option(99, 0), "c2s_set_option")


MULTI_TILE_CASES = {
    # more tiles than SMs: every CTA of the persistent kernel walks over several tiles (and, with C = 64, both slabs)
    "utae_many": ("ltae", dict(in_channels=128, n_head=16, d_k=4, mlp=[256, 128], d_model=256), (70, 61, 8, 8)),
    "timeunet_many": ("ltae", dict(in_channels=64, n_head=16, d_k=4, mlp=[256, 64], d_model=256), (5, 61, 16, 16)),
    "wtae_many": ("ltae4wtae", dict(in_channels=128, n_head=16, d_k=4, d_model=256), (40, 33, 8, 8)),
}


@pytest.mark.parametrize("name", sorted(MULTI_TILE_CASES))
@pytest.mark.parametrize("zero_padded", [False, True])
def test_persistent_ltae_many_tiles(name, zero_padded):
    kind, kw, (b, t, h, w) = MULTI_TILE_CASES[name]
    m, rng = _build(kind, kw, 6000 + len(name))
    m.assume_zero_padded = zero_padded
    lengths = [t] + [max(1, t - (i * 7) % (t // 2 + 1)) for i in range(1, b)]
    lengths[b // 2] = 0  # one series without a single valid frame
    x, pos, pad = synth_inputs(rng, b, t, kw["in_channels"], h, w, lengths)
    xr = bf16_round(x)
    cfg, params = oracle_config(kind, kw), oracle_params(m)
    if kind == "ltae":
        ref_out, ref_attn = ltae_forward(cfg, params, xr, pos, pad)
    else:
        ref_out, ref_attn = None, ltae4wtae_forward(cfg, params, xr, pos, pad)
    (out, attn), _ = _call(m, kind, x, pos, pad, general=False, dtype=torch.bfloat16)
    assert kernel_name_ok(_lib.last_ltae_kernel())
    a = attn.cpu().numpy()
    assert rel_err(a, ref_attn) < 1e-3
    assert np.all(np.abs(a.sum(axis=2) - 1.0) < 1e-5)
    for bi in np.nonzero(~pad.all(axis=1))[0]:
        assert np.all(a[:, bi, pad[bi]] == 0.0)
    if kind == "ltae":
        assert rel_err(out.float().cpu().numpy(), ref_out) < 1e-2


def test_tensor_core_ltae_train_mode_batch_statistics(monkeypatch):
    kind, kw, (b, t, h, w), lengths, _ = LTAE_CASES["utae"]
    m, rng = _build(kind, kw, 77)
    x, pos, pad = synth_inputs(rng, b, t, 128, h, w, lengths)
    params = oracle_params(m)
    m.train()
    m.mlp[5].p = 0.0
    monkeypatch.setattr(c2s.modules, "ATTENTION_DROPOUT", 0.0)  # restored behind the test: later tests train with 0.1
    with torch.no_grad():
        out, attn = m(to_dev(x, dtype=torch.bfloat16), batch_positions=to_dev(pos), pad_mask=to_dev(pad))
    ref_out, ref_attn, (rm, rv) = ltae_forward(oracle_config(kind, kw), params, bf16_round(x), pos, pad, training=True)
    assert rel_err(out.float().cpu().numpy(), ref_out) < 1e-2
    assert rel_err(m.mlp[2].running_mean.cpu().numpy(), rm) < 1e-3
    assert rel_err(m.mlp[2].running_var.cpu().numpy(), rv) < 1e-3


AGG_CASES = {
    # name: (heads, (B, T, C, H, W), (ha, wa), lengths)
    "x8_128": (16, (2, 7, 64, 128, 128), (16, 16), [7, 4]),
    "x4_64": (16, (2, 7, 64, 64, 64), (16, 16), [7, 3]),
    "x2_32": (16, (3, 9, 64, 32, 32), (16, 16), [9, 0, 5]),
    "x8_rect": (4, (2, 5, 16, 64, 128), (8, 16), [5, 2]),
    "x2_heads8": (8, (2, 6, 64, 32, 32), (16, 16), [6, 6]),
}


@pytest.mark.parametrize("name", sorted(AGG_CASES))
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_pipelined_aggregator_matches_oracle(name, dtype):
    heads, (b, t, c, h, w), (ha, wa), lengths = AGG_CASES[name]
    rng = np.random.RandomState(5000 + len(name))
    x, _, pad = synth_inputs(rng, b, t, c, h, w, lengths)
    attn = random_attention(rng, heads, pad, ha, wa)
    xr = x if dtype == torch.float32 else bf16_round(x)
    ref = temporal_aggregator_torch(xr, pad, attn, "att_group").numpy()
    agg = c2s.TemporalAggregator("att_group")
    outs = {}
    for no_pipe in (False, True):
        with _lib.option(_lib.OPT_AGG_KERNEL, int(no_pipe)):
            outs[no_pipe] = agg(to_dev(x, dtype=dtype), pad_mask=to_dev(pad), attn_mask=to_dev(attn))
            kernel = _lib.last_kernel()
        assert ("pipe" in kernel) == (not no_pipe), kernel
        assert rel_err(outs[no_pipe].float().cpu().numpy(), ref) < (1e-5 if dtype == torch.float32 else 1e-2)
    # same taps, same accumulation order: the two kernels agree bit for bit
    assert torch.equal(outs[False], outs[True])


@pytest.mark.parametrize("name", sorted(AGG_CASES))
def test_staged_attention_rows_equal_global_taps(name):
    """The attention rows that ride in the stage (default) give the same bits as per-thread global loads of the taps
    (option OPT_AGG_TAPS): forward, both gradients' kernels, bf16."""
    from crop2seg_b200 import ops
    heads, (b, t, c, h, w), (ha, wa), lengths = AGG_CASES[name]
    rng = np.random.RandomState(6000 + len(name))
    x, _, pad = synth_inputs(rng, b, t, c, h, w, lengths)
    attn = random_attention(rng, heads, pad, ha, wa)
    go = rng.standard_normal((b, c, h, w)).astype(np.float32)
    xd, pd, ad, gd = to_dev(x, dtype=torch.bfloat16), to_dev(pad), to_dev(attn), to_dev(go, dtype=torch.bfloat16)
    res = {}
    for global_taps in (False, True):
        with _lib.option(_lib.OPT_AGG_TAPS, int(global_taps)):
            out = ops.temporal_aggregate_forward(xd, pd, ad, "att_group")
            gx, ga = ops.temporal_aggregate_backward(xd, pd, ad, gd, "att_group")
        res[global_taps] = (out, gx, ga)
    assert torch.equal(res[False][0], res[True][0])
    assert torch.equal(res[False][1], res[True][1])
    assert rel_err(res[False][2].cpu().numpy(), res[True][2].cpu().numpy()) < 1e-5  # float atomics reorder


def test_folded_weights_are_reused_until_a_parameter_changes():
    kind, kw, (b, t, h, w), lengths, _ = LTAE_CASES["utae"]
    m, rng = _build(kind, kw, 31)
    x, pos, pad = synth_inputs(rng, b, t, 128, h, w, lengths)
    args = (to_dev(x, dtype=torch.bfloat16),)
    kwargs = dict(batch_positions=to_dev(pos), pad_mask=to_dev(pad))
    with torch.no_grad():
        _lib.reset_launch_count()
        out0, attn0 = m(*args, **kwargs)
        first = _lib.launch_count()
        _lib.reset_launch_count()
        out1, attn1 = m(*args, **kwargs)
        second = _lib.launch_count()
        assert second < first, (first, second)          # the weight-only preparation kernels were skipped
        assert torch.equal(out0, out1) and torch.equal(attn0, attn1)
        m.attention_head.Q.mul_(1.5)                     # in-place update: the version counter moves
        m.mlp[0].weight.add_(0.01)
        _lib.reset_launch_count()
        out2, attn2 = m(*args, **kwargs)
        assert _lib.launch_count() == first
    ref_out, ref_attn = ltae_forward(oracle_config(kind, kw), oracle_params(m), bf16_round(x), pos, pad)
    assert rel_err(attn2.cpu().numpy(), ref_attn) < 1e-3
    assert rel_err(out2.float().cpu().numpy(), ref_out) < 1e-2
    assert not torch.equal(attn2, attn0)
    m.cache_folded_weights = False
    with torch.no_grad():
        _lib.reset_launch_count()
        out3, attn3 = m(*args, **kwargs)
        assert _lib.launch_count() == first
    assert torch.equal(out3, out2) and torch.equal(attn3, attn2)


@pytest.mark.parametrize("name", ["utae", "timeunet"])
def test_ltae_without_attention_store(name):
    """``return_att=False`` (model-level flag of the reference, timeunet.py:205): same output, no attention tensor."""
    kind, kw, (b, t, h, w), lengths, _ = LTAE_CASES[name]
    m, rng = _build(kind, kw, 77 + len(name))
    x, pos, pad = synth_inputs(rng, b, t, kw["in_channels"], h, w, lengths)
    for dtype in (torch.bfloat16, torch.float32):
        with torch.no_grad():
            out, attn = m(to_dev(x, dtype=dtype), batch_positions=to_dev(pos), pad_mask=to_dev(pad))
            out2, none = m(to_dev(x, dtype=dtype), batch_positions=to_dev(pos), pad_mask=to_dev(pad), return_att=False)
        assert none is None and attn is not None
        if dtype == torch.float32 or name == "utae":
            assert torch.equal(out, out2)
        else:  # Time-Unet shape in bf16: without the attention store the team-pipelined kernel serves the call
            assert _lib.last_ltae_kernel().startswith("ltae_forward<team")
            ref_out, _ = ltae_forward(oracle_config(kind, kw), oracle_params(m), bf16_round(x), pos, pad)
            assert rel_err(out2.float().cpu().numpy(), ref_out) < 1e-2
            assert rel_err(out2.float().cpu().numpy(), out.float().cpu().numpy()) < 1e-2


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs in one process")
def test_one_process_two_devices():
    """Kernel attributes (dynamic shared memory) are per device: the same process drives cuda:0 and then cuda:1."""
    heads, (b, t, c, h, w), (ha, wa), lengths = AGG_CASES["x4_64"]
    rng = np.random.RandomState(99)
    x, pos, pad = synth_inputs(rng, b, t, c, h, w, lengths)
    attn = random_attention(rng, heads, pad, ha, wa)
    kind, kw, (lb, lt, lh, lw), llen, _ = LTAE_CASES["utae"]
    m, rng2 = _build(kind, kw, 98)
    lx, lpos, lpad = synth_inputs(rng2, lb, lt, 128, lh, lw, llen)
    res = []
    for dev in ("cuda:0", "cuda:1"):
        with torch.cuda.device(dev), torch.no_grad():
            out = c2s.TemporalAggregator("att_group")(to_dev(x, dev, torch.bfloat16), pad_mask=to_dev(pad, dev),
                                                      attn_mask=to_dev(attn, dev))
            lo, la = m.to(dev)(to_dev(lx, dev, torch.bfloat16), batch_positions=to_dev(lpos, dev), pad_mask=to_dev(lpad, dev))
            res.append((out.cpu(), lo.cpu(), la.cpu()))
    for a, b_ in zip(res[0], res[1]):
        assert torch.equal(a, b_)


TEAM_CASES = {
    # name: (kwargs extra, (B, T, H, W), lengths or None = ragged incl. an all-padded series, synth extra)
    "full": ({}, (3, 61, 16, 16), [61, 61, 61], {}),
    "ragged": ({}, (6, 61, 16, 16), [61, 27, 0, 44, 1, 16], {}),
    "many_tiles": ({}, (5, 61, 32, 32), None, {}),           # 640 tiles: every team walks over several
    "t64": ({}, (2, 64, 8, 8), [64, 33], {}),
    "t20": ({}, (3, 20, 8, 8), [20, 7, 16], {}),            # whole 16-frame blocks behind T
    "no_mask": ({}, (2, 33, 8, 8), [33, 33], {"no_mask": True}),
    "no_pe": (dict(positional_encoding=False), (2, 40, 8, 8), [40, 21], {"no_positions": True}),
    "doy": (dict(use_doy=True), (2, 61, 8, 8), [61, 30], {"doy": True}),
    "abs_rel": (dict(use_abs_rel_enc=True), (2, 40, 8, 8), [31, 40], {"abs_rel": True}),
    "c_out32": (dict(mlp=[256, 32]), (2, 61, 8, 8), [61, 45], {}),
}


@pytest.mark.parametrize("name", sorted(TEAM_CASES))
@pytest.mark.parametrize("zero_padded", [False, True])
def test_team_kernel_matches_oracle_and_the_slab_kernel(name, zero_padded):
    """The team-pipelined kernel (c2s_ltae_team.cu: C = 64, attention not stored) against the oracle and against the
    whole-slab kernel on the same call."""
    extra_kw, (b, t, h, w), lengths, extra = TEAM_CASES[name]
    kw = dict(in_channels=64, n_head=16, d_k=4, mlp=[256, 64], d_model=256)
    kw.update(extra_kw)
    m, rng = _build("ltae", kw, 8100 + len(name))
    m.assume_zero_padded = zero_padded
    if lengths is None:
        lengths = [t] + [max(1, t - (i * 7) % (t // 2 + 1)) for i in range(1, b)]
        lengths[b // 2] = 0
    x, pos, pad = synth_inputs(rng, b, t, 64, h, w, lengths, doy=extra.get("doy", False), abs_rel=extra.get("abs_rel", False))
    if not zero_padded and pad.any():  # padded frames that are NOT zero: they count in the statistics, not in the attention
        x = x + 0.3 * pad[:, :, None, None, None] * rng.standard_normal(x.shape).astype(np.float32)
    pos = None if extra.get("no_positions") else pos
    pad = None if extra.get("no_mask") else pad
    xr = bf16_round(x)
    ref_out, _ = ltae_forward(oracle_config("ltae", kw), oracle_params(m), xr, pos, pad)
    args = (to_dev(x, dtype=torch.bfloat16),)
    kwargs = dict(batch_positions=None if pos is None else to_dev(pos), pad_mask=None if pad is None else to_dev(pad), return_att=False)
    with torch.no_grad():
        out, none = m(*args, **kwargs)
        assert none is None and _lib.last_ltae_kernel() == "ltae_forward<team,C=64>", _lib.last_ltae_kernel()
        with _lib.option(_lib.OPT_LTAE_KERNEL, _lib.LTAE_KERNEL_SLAB):
            out_s, _ = m(*args, **kwargs)
            assert _lib.last_ltae_kernel().startswith("ltae_forward<fa")
    o = out.float().cpu().numpy()
    assert np.isfinite(o).all()
    assert rel_err(o, ref_out) < 1e-2, rel_err(o, ref_out)
    assert rel_err(o, out_s.float().cpu().numpy()) < 1e-2
