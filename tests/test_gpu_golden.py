"""GPU parity against the committed reference outputs (tests/golden/*.npz) and the numpy oracle.

Every call goes through the drop-in modules -> ctypes -> C ABI -> CUDA kernels.  Tolerances are the
north-star ones: 1e-4 relative (max|d| / max|ref|) in fp32, 1e-2 with bf16 I/O.
"""
import numpy as np
import pytest
import torch

import crop2seg_b200 as c2s
from oracle import ltae4wtae_forward, ltae_forward, temporal_aggregator
from golden_util import fixture_names, load, rel_err
from c2s_testlib import bf16_round, module_from_fixture, oracle_config, to_dev

pytestmark = pytest.mark.gpu

TOL_F32 = 1e-4
TOL_BF16 = 1e-2
UNSUPPORTED = {"ltae_two_queries"}  # num_queries > 1: crashes in every shipped reference model (SURVEY 8a-v)


def _run_ltae(cfg, inp, params, dtype=torch.float32, zero_padded=False):
    m = module_from_fixture(cfg, params)
    m.assume_zero_padded = zero_padded
    rate = c2s.modules.ATTENTION_DROPOUT
    if cfg["train"]:
        m.train()
        c2s.modules.ATTENTION_DROPOUT = 0.0
        m.mlp[5].p = 0.0
    else:
        m.eval()
    try:
        with torch.no_grad():
            res = m(to_dev(inp["x"], dtype=dtype), batch_positions=to_dev(inp.get("positions")),
                    pad_mask=to_dev(inp.get("pad_mask")))
    finally:
        c2s.modules.ATTENTION_DROPOUT = rate  # a process-wide rate: later training-mode tests apply 0.1
    return m, res


@pytest.mark.parametrize("name", [n for n in fixture_names(["ltae_"]) if n not in UNSUPPORTED])
@pytest.mark.parametrize("zero_padded", [False, True])
def test_ltae_fp32_matches_reference(name, zero_padded):
    cfg, inp, params, outs = load(name)
    m, (out, attn) = _run_ltae(cfg, inp, params, zero_padded=zero_padded)
    assert out.shape == outs["out"].shape and attn.shape == outs["attn"].shape
    assert out.dtype == torch.float32 and attn.dtype == torch.float32
    assert rel_err(attn.cpu().numpy(), outs["attn"]) < TOL_F32
    assert rel_err(out.cpu().numpy(), outs["out"]) < TOL_F32
    if cfg["train"]:
        assert rel_err(m.mlp[2].running_mean.cpu().numpy(), outs["running_mean"]) < TOL_F32
        assert rel_err(m.mlp[2].running_var.cpu().numpy(), outs["running_var"]) < TOL_F32
        assert int(m.mlp[2].num_batches_tracked) == 1
    if "pad_mask" in inp:  # identical pad handling: exactly zero attention on padded frames
        pad = inp["pad_mask"]
        a = attn.cpu().numpy()
        for b in np.nonzero(~pad.all(axis=1))[0]:
            assert np.all(a[:, b, pad[b]] == 0.0)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_two_queries_match_reference(dtype):
    """num_queries = 2 (tae.py:495-499): out[B, n, C', H, W], attn[n_head, B, n, T, H, W], one kernel pass per query."""
    cfg, inp, params, outs = load("ltae_two_queries")
    m = module_from_fixture(cfg, params).eval()
    x = inp["x"] if dtype == torch.float32 else bf16_round(inp["x"])
    with torch.no_grad():
        out, attn = m(to_dev(x, dtype=dtype), batch_positions=to_dev(inp["positions"]), pad_mask=to_dev(inp["pad_mask"]))
    assert out.shape == outs["out"].shape and attn.shape == outs["attn"].shape
    tol = TOL_F32 if dtype == torch.float32 else TOL_BF16
    assert rel_err(attn.cpu().numpy(), outs["attn"]) < tol
    assert rel_err(out.float().cpu().numpy(), outs["out"]) < tol
    pad = inp["pad_mask"]
    a = attn.cpu().numpy()
    for b in np.nonzero(~pad.all(axis=1))[0]:
        assert np.all(a[:, b, :, pad[b]] == 0.0)


def test_two_queries_in_training_mode_are_rejected_loudly():
    """BatchNorm1d batch statistics run over the rows of all queries at once in the reference: not served per query."""
    cfg, inp, params, _ = load("ltae_two_queries")
    m = module_from_fixture(cfg, params).train()
    with pytest.raises(NotImplementedError):
        m(to_dev(inp["x"]), batch_positions=to_dev(inp["positions"]), pad_mask=to_dev(inp["pad_mask"]))


@pytest.mark.parametrize("name", fixture_names(["wtae_"]))
def test_ltae4wtae_fp32_matches_reference(name):
    cfg, inp, params, outs = load(name)
    _, attn = _run_ltae(cfg, inp, params)
    assert attn.shape == outs["attn"].shape
    assert rel_err(attn.cpu().numpy(), outs["attn"]) < TOL_F32


@pytest.mark.parametrize("name", [n for n in fixture_names(["ltae_", "wtae_"]) if n not in UNSUPPORTED
                                  and n != "ltae_train_bn"])
def test_ltae_bf16_io_matches_oracle(name):
    """bf16 feature maps in, bf16 out, fp32 attention: compared with the fp32 oracle on the same rounded x."""
    cfg, inp, params, _ = load(name)
    xr = bf16_round(inp["x"])
    ocfg = oracle_config(cfg["kind"], cfg["kwargs"])
    _, res = _run_ltae(cfg, inp, params, dtype=torch.bfloat16)
    if cfg["kind"] == "ltae":
        ref_out, ref_attn = ltae_forward(ocfg, params, xr, inp.get("positions"), inp.get("pad_mask"))
        out, attn = res
        assert out.dtype == torch.bfloat16
        assert rel_err(out.float().cpu().numpy(), ref_out) < TOL_BF16
    else:
        ref_attn = ltae4wtae_forward(ocfg, params, xr, inp.get("positions"), inp.get("pad_mask"))
        attn = res
    assert attn.dtype == torch.float32
    assert rel_err(attn.cpu().numpy(), ref_attn) < TOL_BF16


@pytest.mark.parametrize("name", fixture_names(["agg_"]))
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_aggregator_matches_reference(name, dtype):
    cfg, inp, _, outs = load(name)
    agg = c2s.TemporalAggregator(mode=cfg["mode"])
    x = to_dev(inp["x"], dtype=dtype)
    out = agg(x, pad_mask=to_dev(inp.get("pad_mask")), attn_mask=to_dev(inp["attn"]))
    assert out.shape == outs["out"].shape and out.dtype == dtype
    if dtype == torch.float32:
        ref, tol = outs["out"], TOL_F32
    else:
        ref, tol = temporal_aggregator(bf16_round(inp["x"]), inp.get("pad_mask"), inp["attn"], cfg["mode"]), TOL_BF16
    got = out.float().cpu().numpy()
    if np.isnan(ref).any():  # 'mean' over a series with no valid frame is 0/0 in the reference too
        assert np.array_equal(np.isnan(got), np.isnan(ref))
        got, ref = np.nan_to_num(got), np.nan_to_num(ref)
    assert rel_err(got, ref) < tol
