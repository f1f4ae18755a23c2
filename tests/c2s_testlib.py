"""Shared helpers for the parity tests: build the fused modules from a golden fixture, seeded inputs."""
import numpy as np
import torch

import crop2seg_b200 as c2s
from oracle import LtaeConfig


def synth_inputs(rng, b, t, c, h, w, lengths, doy=False, abs_rel=False):
    """Same generator as tests/golden/make_golden.py: relu(N(0,1)) features, padded frames exactly zero."""
    x = np.maximum(rng.standard_normal((b, t, c, h, w)).astype(np.float32), 0)
    pad = np.zeros((b, t), dtype=bool)
    pos = np.zeros((b, t), dtype=np.int64)
    for i, L in enumerate(lengths):
        pad[i, L:] = True
        x[i, L:] = 0
        if L == 0:
            continue
        gaps = rng.randint(2, 11, size=L)
        gaps[0] = rng.randint(0, 11)
        pos[i, :L] = np.cumsum(gaps)
    if abs_rel:
        positions = np.stack([pos, np.where(pad, 0, (pos + 243) % 365)], axis=-1)
    elif doy:
        positions = np.where(pad, 0, (pos + 243) % 365)
    else:
        positions = pos
    return x, positions, pad


PAD_PATTERNS = ("suffix", "lead1", "lead16", "lead17", "mid_block", "ballot_edge", "alternate", "one_last", "one_mid",
                "sparse_random", "all_padded")


def pad_pattern(name, t, seed=0):
    """[T] bool pad mask (True = padded) of one named pattern.  The kernels handle the mask as a set of frames in
    16-frame blocks, 4-frame groups and two 32-frame ballot halves; each pattern puts its holes where one of those
    decisions changes."""
    pad = np.zeros(t, dtype=bool)
    if name == "suffix":
        pad[max(1, (2 * t) // 3):] = True
    elif name.startswith("lead"):
        pad[:int(name[4:])] = True         # lead16: the first 16-frame block holds no live frame
    elif name == "mid_block":
        pad[16:32] = True                  # live frames on both sides of a dead block (T > 32)
    elif name == "ballot_edge":
        pad[31:33] = True                  # the last frame of the low ballot half and the first of the high one
        if t == 64:
            pad[32:63] = True              # only frame 63 is live in the high half
    elif name == "alternate":
        pad[0::2] = True                   # every 4-frame group is partial, the first live frame is frame 1
    elif name == "one_last":
        pad[:t - 1] = True
    elif name == "one_mid":
        pad[:] = True
        pad[t // 2] = False
    elif name == "sparse_random":
        pad = np.random.RandomState(1000 * seed + t).uniform(size=t) < 0.4
        if pad.all():
            pad[t // 3] = False
    elif name == "all_padded":
        pad[:] = True
    else:
        raise KeyError(name)
    return pad


def pattern_masks(t, names=PAD_PATTERNS, n=None, seed=0):
    """[B, T] bool, one row per sample.  Without ``n``: the named patterns in order.  With ``n``: sample i takes pattern
    i mod (len(names) + 1), the extra slot being a seeded random mask of random density, so that neighbouring samples
    never share a mask."""
    if n is None:
        return np.stack([pad_pattern(name, t) for name in names])
    rng = np.random.RandomState(seed + t)
    rows = []
    for i in range(n):
        k = i % (len(names) + 1)
        rows.append(pad_pattern(names[k], t) if k < len(names) else rng.uniform(size=t) < rng.uniform(0.0, 0.9))
    return np.stack(rows)


def synth_inputs_masked(rng, b, t, c, h, w, masks, zero_padded):
    """Like ``synth_inputs`` but with an explicit [B, T] pad mask.  Positions increase over every frame, so a padded frame
    keeps a plausible date, as a hole in a real series does.  ``zero_padded``: padded frames are exactly zero; otherwise
    they carry non-zero data, which the reference counts in the input GroupNorm but never in the attention."""
    pad = np.asarray(masks, dtype=bool).reshape(b, t)
    x = np.maximum(rng.standard_normal((b, t, c, h, w)).astype(np.float32), 0)
    if zero_padded:
        x[pad] = 0
    else:
        x[pad] = 0.3 * rng.standard_normal(x[pad].shape).astype(np.float32)
    gaps = rng.randint(2, 11, size=(b, t))
    gaps[:, 0] = rng.randint(0, 11, size=b)
    return x, np.cumsum(gaps, axis=1).astype(np.int64), pad


def random_attention(rng, heads, pad, ha, wa):
    b, t = pad.shape
    logits = rng.standard_normal((heads, b, t, ha, wa)).astype(np.float32)
    logits = np.where(pad[None, :, :, None, None], -1e6, logits)
    e = np.exp(logits - logits.max(axis=2, keepdims=True))
    return (e / e.sum(axis=2, keepdims=True)).astype(np.float32)


def randomise(module, rng):
    """Non-trivial parameters everywhere (BN running statistics included)."""
    with torch.no_grad():
        for name, p in module.named_parameters():
            scale = 1.0 / np.sqrt(max(p.shape[-1], 1)) if p.dim() > 1 else 0.5
            vals = rng.standard_normal(tuple(p.shape)).astype(np.float32) * scale
            if name.endswith("norm.weight") or name == "mlp.2.weight":
                vals = 1.0 + 0.3 * vals
            p.copy_(torch.from_numpy(vals))
        for name, buf in module.named_buffers():
            if name.endswith("running_mean"):
                buf.copy_(torch.from_numpy(rng.standard_normal(tuple(buf.shape)).astype(np.float32) * 0.3))
            elif name.endswith("running_var"):
                buf.copy_(torch.from_numpy(rng.uniform(0.5, 2.0, tuple(buf.shape)).astype(np.float32)))


def module_from_fixture(cfg, params, device="cuda"):
    """The fused module with the fixture's constructor kwargs and state_dict."""
    kw = dict(cfg["kwargs"])
    cls = c2s.LTAE if cfg["kind"] == "ltae" else c2s.LTAE4WTAE
    m = cls(**kw)
    sd = {k: torch.from_numpy(np.asarray(v)) for k, v in params.items() if k != "positional_encoder.denom"}
    missing, unexpected = m.load_state_dict(sd, strict=True)
    assert not missing and not unexpected
    if "positional_encoder.denom" in params:
        assert np.array_equal(m.positional_encoder.denom.numpy(), params["positional_encoder.denom"])
    return m.to(device)


def oracle_params(module):
    """numpy state_dict (+ the denom attribute) of a fused module, keyed as the oracle expects."""
    p = {k: v.detach().cpu().numpy() for k, v in module.state_dict().items()}
    pe = getattr(module, "positional_encoder", None)
    if pe is not None and hasattr(pe, "denom"):
        p["positional_encoder.denom"] = pe.denom.cpu().numpy()
    return p


def oracle_config(kind, kw):
    kw = dict(kw)
    if kind != "ltae":
        kw["mlp"] = [kw.get("d_model") or kw["in_channels"], 1]
    kw.setdefault("mlp", [256, 128])
    kw.pop("dropout", None)
    return LtaeConfig(**kw)


def to_dev(a, device="cuda", dtype=None):
    if a is None:
        return None
    t = torch.from_numpy(np.ascontiguousarray(a)).to(device)
    if dtype is not None and t.is_floating_point():
        t = t.to(dtype)
    return t


def bf16_round(a):
    """float32 array rounded to bfloat16 and back (what a bf16 tensor of the same values holds)."""
    return torch.from_numpy(np.ascontiguousarray(a)).to(torch.bfloat16).to(torch.float32).numpy()


def hot_path_parity(enc, x4, xs, pos, pad, out, attn, skips, samples):
    """Oracle check of one U-TAE-placement step at its REAL shapes, per sample: the device tensors of the samples in
    ``samples`` are copied to the host and pushed through the numpy / torch-CPU oracles.  ``x4`` [B,T,C,h,w] and ``xs``
    (list of [B,T,c,H,W]) are the device inputs, ``out`` / ``attn`` [heads,B,T,h,w] / ``skips`` the device outputs.
    Returns max relative errors (max|d| / max|ref| per tensor and sample) and the pad-handling check."""
    from oracle import ltae_forward
    from oracle.torch_port import temporal_aggregator_torch
    params = oracle_params(enc)
    kw = dict(in_channels=enc.in_channels, n_head=enc.n_head, d_k=enc.d_k, mlp=list(enc._widths), d_model=enc.d_model)
    cfg = LtaeConfig(**kw)
    errs = {"attn": 0.0, "out": 0.0, "skips": [0.0] * len(xs), "pad_attention_exactly_zero": True, "samples": list(samples)}

    def rel(a, r):
        return float(np.abs(a - r).max() / max(np.abs(r).max(), 1e-30))

    for b in samples:
        xb = x4[b:b + 1].float().cpu().numpy()
        pb, mb = pos[b:b + 1].cpu().numpy(), pad[b:b + 1].cpu().numpy()
        ref_out, ref_attn = ltae_forward(cfg, params, xb, pb, mb)
        a = attn[:, b:b + 1].float().cpu().numpy()
        errs["attn"] = max(errs["attn"], rel(a, ref_attn))
        errs["out"] = max(errs["out"], rel(out[b:b + 1].float().cpu().numpy(), ref_out))
        if not mb.all():
            errs["pad_attention_exactly_zero"] &= bool(np.all(a[:, 0, mb[0]] == 0.0))
        for i, x in enumerate(xs):
            ref = temporal_aggregator_torch(x[b:b + 1].float().cpu(), mb, ref_attn, "att_group").numpy()
            errs["skips"][i] = max(errs["skips"][i], rel(skips[i][b:b + 1].float().cpu().numpy(), ref))
    return errs
