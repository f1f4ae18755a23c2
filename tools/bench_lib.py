"""Sub-benchmarks that ride in bench.py's JSON line next to the headline (BASELINE.json configs[2], [3], [4]).

Every function returns a dict; timing is CUDA events on the current stream, barrier + synchronize on both sides, MAX
over ranks, and each timed region lasts at least ``min_seconds`` (the step count is calibrated from a short probe) so
that the clock sampler sees the load.  The stand-alone scripts tools/bench_placements.py, bench_training.py and
bench_tile.py print the same records one per line.
"""
import json
import math
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
import crop2seg_b200 as c2s  # noqa: E402
from crop2seg_b200 import _lib  # noqa: E402
from c2s_testlib import randomise  # noqa: E402

T_FRAMES = 61
N_HEAD = 16
LEVELS = ((64, 32), (64, 64), (64, 128))
LTAE_C, LTAE_RES = 128, 16


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    return 6650.0, "B200_PROFILING.md fallback"


def _world():
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


def _barrier():
    if _world() > 1:
        dist.barrier()
    torch.cuda.synchronize()


def _max_over_ranks(ms, dev):
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if _world() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def timed(fn, dev, min_seconds=1.0, warmup=3, max_steps=20000):
    """(ms per call, calls timed, library launches per call): at least ``min_seconds`` of device time, max over ranks."""
    for _ in range(warmup):
        fn()
    _barrier()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(3):
        fn()
    e.record()
    _barrier()
    probe = _max_over_ranks(s.elapsed_time(e) / 3, dev)
    steps = int(min(max_steps, max(5, math.ceil(min_seconds * 1e3 / max(probe, 1e-3)))))
    _lib.reset_launch_count()
    s.record()
    for _ in range(steps):
        fn()
    e.record()
    _barrier()
    launches = _lib.launch_count() / steps
    return _max_over_ranks(s.elapsed_time(e), dev) / steps, steps, launches


def _features(B, T, c, r, pad, dev, gen, requires_grad=False):
    x = torch.empty((B, T, c, r, r), dtype=torch.bfloat16, device=dev)
    for i in range(B):  # per sample: bounds the fp32 temporaries
        v = torch.randn((T, c, r, r), device=dev, generator=gen).clamp_(min=0)
        if pad is not None:
            v[pad[i]] = 0  # padded frames are exactly zero (temp_shared_block.py:30-40)
        x[i] = v.to(torch.bfloat16)
    return x.requires_grad_(True) if requires_grad else x


def _positions(lengths, seed, T=T_FRAMES):
    rng = np.random.RandomState(seed + 1)
    b = len(lengths)
    pos = np.zeros((b, T), dtype=np.int64)
    pad = np.zeros((b, T), dtype=bool)
    for i, L in enumerate(lengths):
        gaps = rng.randint(2, 11, size=L)
        gaps[0] = rng.randint(0, 11)
        pos[i, :L] = np.cumsum(gaps)
        pad[i, L:] = True
    return pos, pad


def _record(name, ms, steps, launches, B, alg_bytes, note, extra=None):
    peak, src = hbm_peak()
    world = _world()
    gbs = alg_bytes / (ms * 1e-3) / 1e9
    rec = {"workload": name, "value": world * B / (ms * 1e-3), "unit": "patches/s", "n_gpus": world, "ms_per_step": ms,
           "steps": steps, "timed_s": ms * steps * 1e-3, "batch_per_gpu": B, "dtype": "bf16",
           "roofline": {"bound": "hbm", "algorithmic_bytes": alg_bytes, "achieved": gbs, "peak": peak, "unit": "GB/s",
                        "frac": gbs / peak, "peak_source": src},
           "gpu_launches_per_step": launches, "note": note}
    if extra:
        rec.update(extra)
    return rec


# ------------------------------------------------------------------------------------------------ configs[2]
def placements(dev, B=64, min_seconds=1.0, only=("wtae", "timeunet", "timeunet_att"), seed=1234):
    """W-TAE and Time-Unet placements (BASELINE configs[2]: B=64, T=61, every series full length)."""
    rank = dist.get_rank() if _world() > 1 else 0
    lengths = np.full(B, T_FRAMES)
    pos_np, pad_np = _positions(lengths, seed + rank)
    pos, pad = torch.from_numpy(pos_np).to(dev), torch.from_numpy(pad_np).to(dev)
    n_valid = int(lengths.sum())
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed + rank)
    agg = c2s.TemporalAggregator("att_group")
    out = {}
    if "wtae" in only:
        enc = c2s.LTAE4WTAE(in_channels=128, n_head=16, d_k=4, d_model=256)
        randomise(enc, np.random.RandomState(1))
        enc = enc.to(dev).eval()
        enc.assume_zero_padded = True
        x4, x1 = _features(B, T_FRAMES, 128, 16, pad, dev, gen), _features(B, T_FRAMES, 64, 128, pad, dev, gen)

        def wtae():
            with torch.no_grad():
                att = enc(x4, batch_positions=pos, pad_mask=pad)
                return agg(x1, pad_mask=pad, attn_mask=att)
        ms, steps, n = timed(wtae, dev, min_seconds)
        alg = 2 * n_valid * (128 * 256 + 64 * 16384) + 2 * B * 64 * 16384 + 4 * 16 * T_FRAMES * 256 * B
        out["wtae"] = _record("W-TAE placement", ms, steps, n, B, alg,
                              "LTAE4WTAE[B,61,128,16,16] + TemporalAggregator x8 on [B,61,64,128,128] (wtae.py:237-242)")
        del x4, x1
    if "timeunet" in only or "timeunet_att" in only:
        enc = c2s.LTAE(in_channels=64, n_head=16, d_k=4, mlp=[256, 64], d_model=256)
        randomise(enc, np.random.RandomState(2))
        enc = enc.to(dev).eval()
        enc.assume_zero_padded = True
        x = _features(B, T_FRAMES, 64, 128, pad, dev, gen)
        for name, need_att in (("timeunet", False), ("timeunet_att", True)):
            if name not in only:
                continue

            def tu():
                with torch.no_grad():
                    return enc(x, batch_positions=pos, pad_mask=pad, return_att=need_att)
            ms, steps, n = timed(tu, dev, min_seconds)
            alg = 2 * n_valid * 64 * 16384 + 2 * B * 64 * 16384 + (4 * 16 * T_FRAMES * 16384 * B if need_att else 0)
            out[name] = _record("Time-Unet placement" + (", attention returned" if need_att else ""), ms, steps, n, B, alg,
                                "LTAE(C=64, mlp=[256,64]) on [B,61,64,128,128] (timeunet.py:178-180), attention "
                                + ("returned" if need_att else "not materialised (return_att=False)"),
                                {"kernel": _lib.last_ltae_kernel()})
        del x
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------ configs[3]
def training(dev, local_rank, B=16, min_seconds=1.0, seed=1234, ddp=False):
    """U-TAE hot path, forward + backward + Adam, DDP gradient all-reduce over the ranks (BASELINE configs[3])."""
    world = _world()
    rank = dist.get_rank() if world > 1 else 0
    rng = np.random.RandomState(seed + rank)
    lengths = rng.randint(27, T_FRAMES + 1, size=B)
    lengths[0] = T_FRAMES
    pos_np, pad_np = _positions(lengths, seed + rank)
    pos, pad = torch.from_numpy(pos_np).to(dev), torch.from_numpy(pad_np).to(dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed + rank)
    x4 = _features(B, T_FRAMES, LTAE_C, LTAE_RES, pad, dev, gen, True)
    xs = [_features(B, T_FRAMES, c, r, pad, dev, gen, True) for c, r in LEVELS]
    enc = c2s.LTAE(in_channels=LTAE_C, n_head=N_HEAD, d_k=4, mlp=[256, 128], d_model=256)
    randomise(enc, np.random.RandomState(seed))
    enc = enc.to(dev).train()
    enc.assume_zero_padded = True
    # data parallelism: ONE flat gradient buffer, ONE NCCL all-reduce per step (crop2seg_b200.GradientBucket); `ddp=True`
    # wraps the encoder in DistributedDataParallel instead (per-bucket hooks), for comparison
    bucket = None if ddp else c2s.GradientBucket(enc.parameters())
    model = torch.nn.parallel.DistributedDataParallel(enc, device_ids=[local_rank]) if (ddp and world > 1) else enc
    agg = c2s.TemporalAggregator(mode="att_group")
    # train.py: Adam, lr 1e-3; `fused=True` is torch's single-kernel implementation of the same update (the default
    # `foreach` one is ~8 element-wise launches, 0.08 ms of a 2 ms step)
    opt = torch.optim.Adam(enc.parameters(), lr=1e-3, fused=True)
    projs = [torch.randn((B, 128, LTAE_RES, LTAE_RES), device=dev, generator=gen).to(torch.bfloat16)] + \
            [torch.randn((B, c, r, r), device=dev, generator=gen).to(torch.bfloat16) for c, r in LEVELS]

    def step():
        if bucket is None:
            opt.zero_grad(set_to_none=True)
        else:
            bucket.zero()
        for x in [x4] + xs:
            x.grad = None
        out, att = model(x4, batch_positions=pos, pad_mask=pad)
        outs = [out] + [agg(x, pad_mask=pad, attn_mask=att) for x in xs]
        # the decoder and the loss are outside the path: its backward hands these four gradients over (fixed tensors here)
        torch.autograd.backward(outs, projs)
        if bucket is not None:
            bucket.all_reduce()
        opt.step()
        return outs[0]

    ms, steps, n = timed(step, dev, min_seconds, warmup=5)
    e_in = LTAE_C * LTAE_RES ** 2 + sum(c * r * r for c, r in LEVELS)
    n_valid = int(lengths.sum())
    attn_bytes = 4 * N_HEAD * T_FRAMES * LTAE_RES ** 2 * B
    fwd = 2 * n_valid * e_in + 2 * B * e_in + attn_bytes
    bwd = 2 * n_valid * e_in + 2 * B * T_FRAMES * e_in + 2 * B * e_in + 2 * attn_bytes  # x again, grad_x, grad_out, attn + grad_attn
    rec = _record("U-TAE placement training step", ms, steps, n, B, fwd + bwd,
                  "BASELINE configs[3] hot path: LTAE(train: batch statistics, both dropouts) + 3x TemporalAggregator "
                  "forward + backward, Adam step (torch.optim.Adam(fused=True))" + ((", DistributedDataParallel" if ddp else ", one NCCL all-reduce of one flat "
                                                      "gradient buffer (GradientBucket)") if world > 1 else "")
                  + "; the gradients of the four outputs are supplied as fixed tensors (what the decoder's backward hands over: "
                  "the decoder and the loss are outside the path)",
                  {"mean_valid_frames": float(np.mean(lengths))})
    del x4, xs, projs
    torch.cuda.empty_cache()
    return rec


# ------------------------------------------------------------------------------------------------ section 8f rank 4
def encoder(dev, frames=1024, min_seconds=1.0, seed=1234):
    """Shared conv encoder slice (SURVEY.md section 8f, rank 4): U-TAE's ``in_conv`` = ConvBlock([10, 64, 64], GroupNorm)
    on ``frames`` packed valid frames of [10, 128, 128] (bf16), both convolutions on the tcgen05 implicit-GEMM kernel, and
    the 64 -> 64 convolution alone against the measured dense bf16 tensor-core peak."""
    from crop2seg_b200 import conv as cc
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed)
    blk = c2s.ConvBlock([10, 64, 64], pad_value=0, norm="group").to(dev).eval()
    x = torch.randn((frames, 10, 128, 128), device=dev, generator=gen).to(torch.bfloat16)
    with torch.no_grad():
        ms, steps, launches = timed(lambda: blk(x), dev, min_seconds)
    world = _world()
    flops = 2.0 * frames * 128 * 128 * 64 * (10 + 64) * 9
    peaks = {}
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        peaks = json.load(open(path))
    tpeak = float(peaks.get("bf16_tflops", 1637.8))
    rec = {"workload": "in_conv = ConvBlock([10,64,64], norm='group') on packed frames (utae.py:128-136)",
           "value": world * frames / (ms * 1e-3), "unit": "frames/s", "n_gpus": world, "ms_per_step": ms, "steps": steps,
           "timed_s": ms * steps * 1e-3, "frames_per_gpu": frames, "dtype": "bf16", "tflops": flops / ms * 1e-9,
           "gpu_launches_per_step": launches,
           "note": "two 3x3 reflect convolutions (tcgen05 implicit GEMM, raw bf16 output + GroupNorm sums) and two "
                   "normalisation passes; forward only"}
    x64 = torch.randn((frames, 64, 128, 128), device=dev, generator=gen).to(torch.bfloat16)
    conv = blk.conv.conv[3]
    ms2, steps2, _ = timed(lambda: cc.conv2d_reflect_forward(x64, conv.weight, conv.bias), dev, min_seconds)
    f2 = 2.0 * frames * 128 * 128 * 64 * 64 * 9
    rec["conv64"] = {"kernel": "conv3x3_reflect<tcgen05> 64 -> 64 at 128^2", "ms": ms2, "steps": steps2,
                     "roofline": {"bound": "tensor", "achieved": f2 / ms2 * 1e-9, "peak": tpeak, "unit": "TFLOP/s",
                                  "frac": f2 / ms2 * 1e-9 / tpeak,
                                  "peak_source": "MEASURED_PEAKS.json bf16_tflops (cuBLAS burst)" if peaks else "fallback",
                                  "note": "M 128 x N 64 x K 16 products read 6 KB of shared memory each: 48 cycles against "
                                          "a 32-cycle tensor floor (tools/ubench/umma_rowshift.cu), i.e. at most 0.67 of "
                                          "the nominal rate with 64 output channels"}}
    del x, x64
    # the four blocks of the spatial encoder one after the other (utae.py:128-149): every layer runs on the tensor-core
    # kernels (3x3 with 128 / 64 / 32-pixel rows, strided 4x4 with parity-split rows, 3x3 on whole 16 x 16 frames for the
    # 128-channel layers of the last block); the share of the multiply-adds they serve is read from conv2d_supported
    blocks = [("in_conv", blk, (10, 128)),
              ("down1", c2s.DownConvBlock(64, 64, 4, 2, 1, pad_value=0, norm="group").to(dev).eval(), (64, 128)),
              ("down2", c2s.DownConvBlock(64, 64, 4, 2, 1, pad_value=0, norm="group").to(dev).eval(), (64, 64)),
              ("down3", c2s.DownConvBlock(64, 128, 4, 2, 1, pad_value=0, norm="group").to(dev).eval(), (64, 32))]
    per, total = {}, 0.0
    for name, b, (c, r) in blocks:
        xb = torch.randn((frames, c, r, r), device=dev, generator=gen).to(torch.bfloat16)
        with torch.no_grad():
            m, _, _ = timed(lambda: b(xb), dev, min_seconds / 4)
        per[name] = m
        total += m
        del xb
    macs = 128 * 128 * 64 * 9 * 74 + 64 * 64 * 64 * 64 * 34 + 32 * 32 * 64 * 64 * 34 + 16 * 16 * (64 * 64 * 16 + 9 * 64 * 128 + 9 * 128 * 128)
    rec["spatial_encoder"] = {"workload": "U-TAE spatial encoder (in_conv + 3 DownConvBlock, widths [64,64,64,128]) on packed frames, "
                                          "block by block", "ms_per_block": per, "ms": total,
                              "frames_per_s": world * frames / (total * 1e-3), "tflops": 2.0 * frames * macs / total * 1e-9,
                              "hand_written_share_of_macs": _hand_written_share(blocks, dev)}
    torch.cuda.empty_cache()
    return rec


def _hand_written_share(blocks, dev):
    """Share of the convolution multiply-adds of ``blocks`` that ``conv2d_supported`` routes to the hand-written kernels."""
    from crop2seg_b200 import conv as cc
    total = hand = 0
    for _, b, (c, r) in blocks:
        h = r
        for layer in ([b.conv] if isinstance(b, c2s.ConvBlock) else [b.down, b.conv1, b.conv2]):
            for ci, _, _ in layer._plan:
                conv = layer.conv[ci]
                k, st, p = conv.kernel_size[0], conv.stride[0], conv.padding[0]
                ho = (h + 2 * p - k) // st + 1
                macs = ho * ho * conv.out_channels * conv.in_channels * k * k
                total += macs
                if cc.conv2d_supported(torch.empty((1, conv.in_channels, h, h), device=dev, dtype=torch.bfloat16), conv):
                    hand += macs
                h = ho
    return hand / total


# ------------------------------------------------------------------------------------------------ configs[4]
def tile(dev, placement="timeunet", B=64, tiles=1, seed=1234, with_edges=True):
    """Webapp-style full Sentinel-2 tile (BASELINE configs[4]): 10980^2 -> zero-pad to 11008^2 -> 86 x 86 = 7396 patches of
    128^2, T = 60, contiguous shards over the ranks (strong scaling), batches of B.  ``placement``: "timeunet" is what
    the reference webapp runs (src/webapp/prediction.py:201); "utae" the U-TAE hot path.  ``with_edges``: every batch
    also goes through the tile-edge kernels (raw int16 tile -> normalised model inputs; class scores -> class map),
    section 8f rank 3, on a device-resident synthetic tile strip."""
    world = _world()
    rank = dist.get_rank() if world > 1 else 0
    T, n_patches = 60, 86 * 86
    lo, hi = c2s.shard_bounds(n_patches, rank, world)
    lengths = np.full(B, T)
    pos_np, pad_np = _positions(lengths, seed, T)
    pos, pad = torch.from_numpy(pos_np).to(dev), torch.from_numpy(pad_np).to(dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed + rank)
    agg = c2s.TemporalAggregator("att_group")
    if placement == "timeunet":
        enc = c2s.LTAE(in_channels=64, n_head=16, d_k=4, mlp=[256, 64], d_model=256)
        feats = [_features(B, T, 64, 128, None, dev, gen)]
        e_in, e_out, attn = 64 * 16384, 64 * 16384, 0
    else:
        enc = c2s.LTAE(in_channels=LTAE_C, n_head=N_HEAD, d_k=4, mlp=[256, 128], d_model=256)
        feats = [_features(B, T, LTAE_C, LTAE_RES, None, dev, gen)] + [_features(B, T, c, r, None, dev, gen) for c, r in LEVELS]
        e_in = e_out = LTAE_C * LTAE_RES ** 2 + sum(c * r * r for c, r in LEVELS)
        attn = 4 * N_HEAD * T * LTAE_RES ** 2
    randomise(enc, np.random.RandomState(seed))
    enc = enc.to(dev).eval()
    enc.assume_zero_padded = True
    edges = None
    if with_edges:  # one row of 86 patches of the raw tile lives on the device; the batches walk along it
        strip = torch.randint(0, 6000, (T, 10, 128, 11008), dtype=torch.int16, device=dev, generator=gen)
        pat = c2s.TilePatchifier(strip, [1000.0] * 10, [500.0] * 10, t_pad=T_FRAMES, dtype=torch.bfloat16)
        raw_in = torch.empty((B, T_FRAMES, 10, 128, 128), dtype=torch.bfloat16, device=dev)
        logits = torch.randn((B, 15, 128, 128), device=dev, generator=gen).to(torch.bfloat16)
        cmap = c2s.ClassMap(128, 11008, 15, dev, with_proba=False)
        edges = (pat, raw_in, logits, cmap)

    def run_tile():
        done = lo
        while done < hi:
            n = min(B, hi - done)
            if edges is not None:
                pat, raw_in, logits, cmap = edges
                begin = (done - lo) % (86 - B + 1) if B <= 86 else 0
                pat.patches(begin, min(n, 86), out=raw_in[:min(n, 86)])
            with torch.no_grad():
                if placement == "timeunet":
                    enc(feats[0][:n], batch_positions=pos[:n], pad_mask=pad[:n], return_att=False)
                else:
                    _, att = enc(feats[0][:n], batch_positions=pos[:n], pad_mask=pad[:n])
                    for x in feats[1:]:
                        agg(x[:n], pad_mask=pad[:n], attn_mask=att)
            if edges is not None:
                cmap.put(logits[:min(n, 86)], begin)
            done += n

    run_tile()
    _barrier()
    _lib.reset_launch_count()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(tiles):
        run_tile()
    e.record()
    _barrier()
    sec = _max_over_ranks(s.elapsed_time(e), dev) * 1e-3 / tiles
    per_patch = 2 * T * e_in + 2 * e_out + attn
    if with_edges:
        per_patch += 2 * T * 10 * 16384 + 2 * T_FRAMES * 10 * 16384 + 2 * 15 * 16384 + 16384  # raw in, inputs out, scores in, classes out
    peak, src = hbm_peak()
    gbs = per_patch * n_patches / sec / 1e9 / world
    rec = {"workload": f"BASELINE configs[4]: full Sentinel-2 tile, {placement} placement", "value": n_patches / sec,
           "unit": "patches/s", "seconds_per_tile": sec, "n_gpus": world, "scaling": "strong", "patches": n_patches,
           "batch": B, "frames": T, "tile_edges": bool(with_edges),
           "roofline": {"bound": "hbm", "algorithmic_bytes": per_patch * n_patches, "achieved": gbs, "peak": peak,
                        "unit": "GB/s per GPU", "frac": gbs / peak, "peak_source": src},
           "gpu_launches_per_tile_rank0": _lib.launch_count() / tiles,
           "note": "src/webapp/prediction.py:201 runs Time-Unet; patches sharded contiguously over the ranks, no collective"}
    del feats, edges
    torch.cuda.empty_cache()
    return rec


# ------------------------------------------------------------------------------------------------ host link
def pcie_ceiling(dev, n_bytes=1 << 30, repeats=4):
    """Plain pinned cudaMemcpyAsync host->device and device->host of ``n_bytes`` on every rank at the same time: the
    ceiling the end-to-end number is compared with (GB/s of this rank, max-time over ranks)."""
    h = torch.empty(n_bytes, dtype=torch.uint8).pin_memory()
    d = torch.empty(n_bytes, dtype=torch.uint8, device=dev)
    res = {}
    for name, (dst, src) in (("h2d", (d, h)), ("d2h", (h, d))):
        dst.copy_(src, non_blocking=True)
        _barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(repeats):
            dst.copy_(src, non_blocking=True)
        e.record()
        _barrier()
        ms = _max_over_ranks(s.elapsed_time(e), dev) / repeats
        res[name + "_gbs"] = n_bytes / (ms * 1e-3) / 1e9
    del h, d
    return res


def topology():
    import subprocess
    out = {}
    for key, cmd in (("nvidia_smi_topo", ["nvidia-smi", "topo", "-m"]), ("lspci_tree", ["lspci", "-t"])):
        try:
            out[key] = subprocess.run(cmd, capture_output=True, text=True, timeout=20).stdout[-6000:]
        except Exception as exc:  # pragma: no cover
            out[key] = f"unavailable: {exc}"
    return out
