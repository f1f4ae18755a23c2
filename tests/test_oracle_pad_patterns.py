"""The numpy and torch-CPU oracles agree with each other on pad masks with leading, interior and scattered padded frames.

Both are pinned against the reference on suffix masks only (test_oracle_golden.py); the GPU tests of
test_gpu_pad_patterns.py rely on them for every pattern of ``c2s_testlib.PAD_PATTERNS``."""
import numpy as np
import pytest
import torch

from oracle import LtaeConfig, ltae_forward, temporal_aggregator
from oracle.torch_port import ltae_forward_torch, temporal_aggregator_torch
from golden_util import rel_err
from c2s_testlib import PAD_PATTERNS, pattern_masks, random_attention, synth_inputs_masked


def _params(cfg, rng):
    c, d, dk, h = cfg.in_channels, cfg.width, cfg.d_k, cfg.n_head
    c_out = cfg.mlp[1]  # mlp.0: Linear(d_model, c_out), then BatchNorm1d(c_out)
    p = {"in_norm.weight": 1.0 + 0.3 * rng.standard_normal(c), "in_norm.bias": 0.5 * rng.standard_normal(c),
         "inconv.weight": rng.standard_normal((d, c, 1)) / np.sqrt(c), "inconv.bias": 0.5 * rng.standard_normal(d),
         "attention_head.Q": rng.standard_normal((h, 1, dk)),
         "attention_head.fc1_k.weight": rng.standard_normal((h * dk, d)) / np.sqrt(d),
         "attention_head.fc1_k.bias": 0.5 * rng.standard_normal(h * dk),
         "mlp.0.weight": rng.standard_normal((c_out, d)) / np.sqrt(d), "mlp.0.bias": 0.5 * rng.standard_normal(c_out),
         "mlp.2.weight": 1.0 + 0.3 * rng.standard_normal(c_out), "mlp.2.bias": 0.5 * rng.standard_normal(c_out),
         "mlp.2.running_mean": 0.3 * rng.standard_normal(c_out), "mlp.2.running_var": rng.uniform(0.5, 2.0, c_out),
         "out_norm.weight": 1.0 + 0.3 * rng.standard_normal(c_out), "out_norm.bias": 0.5 * rng.standard_normal(c_out)}
    p = {k: np.asarray(v, dtype=np.float32) for k, v in p.items()}
    p["positional_encoder.denom"] = np.power(np.float64(cfg.T), 2.0 * (np.arange(d // h) // 2) / (d // h)).astype(np.float32)
    return p


@pytest.mark.parametrize("t", [61, 64, 33, 20])
@pytest.mark.parametrize("zero_padded", [False, True])
def test_numpy_and_torch_oracles_agree_on_pad_patterns(t, zero_padded):
    rng = np.random.RandomState(40 + t)
    cfg = LtaeConfig(in_channels=32, n_head=4, d_k=4, mlp=[64, 32], d_model=64)
    params = _params(cfg, rng)
    masks = pattern_masks(t)
    b = masks.shape[0]
    x, pos, pad = synth_inputs_masked(rng, b, t, 32, 2, 3, masks, zero_padded)
    out, attn = ltae_forward(cfg, params, x, pos, pad)
    with torch.no_grad():
        out_t, attn_t = ltae_forward_torch(cfg, params, x, pos, pad)
    for bi, name in enumerate(PAD_PATTERNS):
        assert rel_err(out_t[bi].numpy(), out[bi]) < 1e-4, name
        assert rel_err(attn_t[:, bi].numpy(), attn[:, bi]) < 1e-5, name
        if name != "all_padded":
            assert np.all(attn[:, bi, pad[bi]] == 0.0), name
    for mode, (h, w), (ha, wa) in [("att_group", (8, 8), (4, 4)), ("att_group", (4, 4), (8, 8)), ("att_mean", (8, 8), (4, 4)),
                                   ("mean", (8, 8), (4, 4))]:
        xa = synth_inputs_masked(rng, b, t, 8, h, w, masks, zero_padded)[0]
        a = random_attention(rng, 4, pad, ha, wa)
        keep = slice(None) if mode != "mean" else ~pad.all(axis=1)  # mean over no valid frame is 0 / 0 in both
        ref = temporal_aggregator(xa[keep], pad[keep], a[:, keep], mode)
        with torch.no_grad():
            got = temporal_aggregator_torch(xa[keep], pad[keep], a[:, keep], mode).numpy()
        assert np.isfinite(ref).all()
        assert rel_err(got, ref) < 1e-5, mode
