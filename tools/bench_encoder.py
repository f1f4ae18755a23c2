#!/usr/bin/env python
"""Throughput of the shared conv encoder slice (SURVEY.md section 8f, rank 4): the tcgen05 3x3 reflect convolution at
the full resolution, the normalisation pass, and U-TAE's ``in_conv`` block on packed frames.  One JSON line per record.

    python tools/bench_encoder.py [--frames 1024] [--seconds 0.5] [--last-block]

``--last-block`` runs only the records of U-TAE's last down block (the 16 x 16 kernel against the library route it
replaced, alternated in one run) and the four-block encoder total.

``cudnn_*`` lines time ``torch.nn.functional.conv2d`` on the same bf16 tensors (reflect padding done beforehand, outside
the timed region for the NCHW line) -- a library yardstick, not part of the product path.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import crop2seg_b200 as c2s  # noqa: E402
from crop2seg_b200 import conv as cc  # noqa: E402


def timed(fn, seconds, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n, total = 0, 0.0
    while total < seconds * 1e3:
        s.record()
        for _ in range(20):
            fn()
        e.record()
        torch.cuda.synchronize()
        total += s.elapsed_time(e)
        n += 20
    return total / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1024)
    ap.add_argument("--seconds", type=float, default=0.5)
    ap.add_argument("--last-block", action="store_true")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    print(json.dumps(card()), flush=True)
    if args.last_block:
        last_block(args.frames, args.seconds)
        full_encoder(args.frames, args.seconds)
        return
    n, H, W = args.frames, 128, 128
    peaks = {}
    p = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")
    if os.path.exists(p):
        peaks = json.load(open(p))
    for c_in in (64, 10):
        x = torch.randn((n, c_in, H, W), device=dev).to(torch.bfloat16)
        conv = torch.nn.Conv2d(c_in, 64, 3, padding=1, padding_mode="reflect").to(dev)
        flops = 2.0 * n * H * W * 64 * c_in * 9
        ms = timed(lambda: cc.conv2d_reflect_forward(x, conv.weight, conv.bias), args.seconds)
        byts = 2.0 * n * H * W * (c_in + 64)
        rec = {"record": f"conv3x3_reflect<tcgen05> c_in={c_in}", "frames": n, "ms": ms, "tflops": flops / ms * 1e-9,
               "gbs": byts / ms * 1e-6, "hbm_frac": byts / ms * 1e-6 / float(peaks.get("hbm_gbs", 6551.0)),
               "note": "raw bf16 output + GroupNorm sums; algorithmic bytes = input + output once"}
        if "bf16_tflops" in peaks:
            rec["tensor_frac"] = rec["tflops"] / float(peaks["bf16_tflops"])
        print(json.dumps(rec), flush=True)
        wb, bb = conv.weight.to(torch.bfloat16), conv.bias.to(torch.bfloat16)
        xp = F.pad(x, (1, 1, 1, 1), mode="reflect")
        ms = timed(lambda: F.conv2d(xp, wb, bb), args.seconds)
        print(json.dumps({"record": f"cudnn_nchw c_in={c_in} (padding outside the timed region)", "ms": ms,
                          "tflops": flops / ms * 1e-9}), flush=True)
        xcl = xp.contiguous(memory_format=torch.channels_last)
        wcl = wb.contiguous(memory_format=torch.channels_last)
        ms = timed(lambda: F.conv2d(xcl, wcl, bb), args.seconds)
        print(json.dumps({"record": f"cudnn_channels_last c_in={c_in} (padding and layout change outside the timed region)",
                          "ms": ms, "tflops": flops / ms * 1e-9}), flush=True)
        ms = timed(lambda: F.conv2d(F.pad(x, (1, 1, 1, 1), mode="reflect"), wb, bb), args.seconds)
        print(json.dumps({"record": f"cudnn_nchw c_in={c_in} with the reflect padding", "ms": ms, "tflops": flops / ms * 1e-9}),
              flush=True)
        del x, xp, xcl
    raw = torch.randn((n, 64, H, W), device=dev).to(torch.bfloat16)
    norm = torch.nn.GroupNorm(4, 64).to(dev)
    stats = cc.group_stats(raw, 4)
    out = torch.empty_like(raw)
    ms = timed(lambda: cc.group_norm_relu(raw, stats, norm, out=out), args.seconds)
    byts = 2.0 * raw.numel() * 2
    print(json.dumps({"record": "group_norm_relu", "ms": ms, "gbs": byts / ms * 1e-6,
                      "hbm_frac": byts / ms * 1e-6 / float(peaks.get("hbm_gbs", 6551.0))}), flush=True)
    ms = timed(lambda: cc.group_stats(raw, 4), args.seconds)
    print(json.dumps({"record": "group_stats", "ms": ms, "gbs": raw.numel() * 2 / ms * 1e-6}), flush=True)
    del raw, out
    blk = c2s.ConvBlock([10, 64, 64], pad_value=0, norm="group").to(dev).eval()
    x = torch.randn((n, 10, H, W), device=dev).to(torch.bfloat16)
    with torch.no_grad():
        ms = timed(lambda: blk(x), args.seconds)
    flops = 2.0 * n * H * W * 64 * (10 + 64) * 9
    print(json.dumps({"record": "in_conv block ConvBlock([10,64,64]) on packed frames", "frames": n, "ms": ms,
                      "frames_per_s": n / ms * 1e3, "tflops": flops / ms * 1e-9}), flush=True)
    ref = torch.nn.Sequential(torch.nn.Conv2d(10, 64, 3, padding=1, padding_mode="reflect"), torch.nn.GroupNorm(4, 64), torch.nn.ReLU(),
                              torch.nn.Conv2d(64, 64, 3, padding=1, padding_mode="reflect"), torch.nn.GroupNorm(4, 64), torch.nn.ReLU()).to(dev).eval()
    xf = x.float()
    with torch.no_grad():
        ms = timed(lambda: ref(xf), args.seconds)
    print(json.dumps({"record": "the same layers as the reference runs them (torch eager, fp32, cuDNN)", "ms": ms,
                      "frames_per_s": n / ms * 1e3, "tflops": flops / ms * 1e-9}), flush=True)
    refb = ref.to(torch.bfloat16)
    with torch.no_grad():
        ms = timed(lambda: refb(x), args.seconds)
    print(json.dumps({"record": "the same layers, torch eager bf16 (cuDNN)", "ms": ms, "frames_per_s": n / ms * 1e3,
                      "tflops": flops / ms * 1e-9}), flush=True)
    del x, xf
    # first down block of U-TAE (utae.py:137-149): 4x4 / stride 2 layer 128^2 -> 64^2, then two 3x3 layers at 64^2
    x64 = torch.randn((n, 64, 64, 64), device=dev).to(torch.bfloat16)
    conv = torch.nn.Conv2d(64, 64, 3, padding=1, padding_mode="reflect").to(dev)
    flops = 2.0 * n * 64 * 64 * 64 * 64 * 9
    ms = timed(lambda: cc.conv2d_reflect_forward(x64, conv.weight, conv.bias), args.seconds)
    print(json.dumps({"record": "conv3x3_reflect<tcgen05> c_in=64 at 64^2 (M = 64 products)", "frames": n, "ms": ms,
                      "tflops": flops / ms * 1e-9, "tensor_frac": flops / ms * 1e-9 / float(peaks.get("bf16_tflops", 1637.8))}),
          flush=True)
    del x64
    down = c2s.DownConvBlock(64, 64, 4, 2, 1, pad_value=0, norm="group").to(dev).eval()
    x = torch.randn((n, 64, H, W), device=dev).to(torch.bfloat16)
    with torch.no_grad():
        ms = timed(lambda: down(x), args.seconds)
        ms_down = timed(lambda: down.down(x), args.seconds)
    flops = 2.0 * n * 64 * 64 * 64 * 64 * (16 + 9 + 9)
    print(json.dumps({"record": "DownConvBlock(64, 64, 4, 2, 1) on packed frames 128^2 -> 64^2", "frames": n, "ms": ms,
                      "ms_strided_layer": ms_down, "frames_per_s": n / ms * 1e3, "tflops": flops / ms * 1e-9}), flush=True)
    del x
    full_encoder(n, args.seconds)


def card():
    """The device the numbers below were taken on: name and power limit (nvidia-smi, read only)."""
    rec = {"record": "card", "name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        rec["power_limit_and_max_sm_clock"] = q.stdout.strip() if q.returncode == 0 else "unknown"
    except (OSError, subprocess.TimeoutExpired):
        rec["power_limit_and_max_sm_clock"] = "unknown"
    return rec


def library_conv(x, conv, n_groups):
    """The route ConvLayer took for these layers before conv3x3_reflect_w16 served them: F.pad + cuDNN F.conv2d + group_stats."""
    wb, bb = conv.weight.to(torch.bfloat16), conv.bias.to(torch.bfloat16)
    raw = F.conv2d(F.pad(x, (1, 1, 1, 1), mode="reflect"), wb, bb)
    return raw, cc.group_stats(raw, n_groups)


def last_block(n, seconds, rounds=5):
    """U-TAE's last down block (64 -> 128 channels, 32^2 -> 16^2): its two 128-channel layers on the 16-pixel-wide kernel
    and on the library route, and the whole block, alternated round by round; the median of the rounds is reported."""
    dev = torch.device("cuda", 0)
    blk = c2s.DownConvBlock(64, 128, 4, 2, 1, pad_value=0, norm="group").to(dev).eval()
    x32 = torch.randn((n, 64, 32, 32), device=dev).to(torch.bfloat16)
    x1 = torch.randn((n, 64, 16, 16), device=dev).to(torch.bfloat16)
    x2 = torch.randn((n, 128, 16, 16), device=dev).to(torch.bfloat16)
    c1, c2 = blk.conv1.conv[0], blk.conv2.conv[0]
    cases = {
        "conv1 64->128 @16 conv3x3_reflect_w16<tcgen05>": (lambda: cc.conv2d_reflect_forward(x1, c1.weight, c1.bias), 64),
        "conv1 64->128 @16 library route (F.pad + F.conv2d + group_stats)": (lambda: library_conv(x1, c1, 4), 64),
        "conv2 128->128 @16 conv3x3_reflect_w16<tcgen05>": (lambda: cc.conv2d_reflect_forward(x2, c2.weight, c2.bias), 128),
        "conv2 128->128 @16 library route (F.pad + F.conv2d + group_stats)": (lambda: library_conv(x2, c2, 4), 128),
        "down3 block DownConvBlock(64, 128, 4, 2, 1) 32^2 -> 16^2": (lambda: blk(x32), None),
    }
    times = {k: [] for k in cases}
    with torch.no_grad():
        for _ in range(rounds):
            for k, (fn, _c) in cases.items():
                times[k].append(timed(fn, seconds / rounds))
    for k, (fn, c_in) in cases.items():
        ms = statistics.median(times[k])
        rec = {"record": k, "frames": n, "ms": ms, "ms_rounds": [round(t, 4) for t in times[k]]}
        if c_in is not None:
            rec["tflops"] = 2.0 * n * 16 * 16 * 128 * c_in * 9 / ms * 1e-9
        print(json.dumps(rec), flush=True)


def full_encoder(n, seconds):
    """U-TAE's spatial encoder (utae.py:128-149, widths [64, 64, 64, 128]) block by block on n packed frames."""
    dev = torch.device("cuda", 0)
    blocks = [("in_conv 10->64->64 @128", c2s.ConvBlock([10, 64, 64], pad_value=0, norm="group"), (10, 128)),
              ("down1 64->64 @128->64", c2s.DownConvBlock(64, 64, 4, 2, 1, pad_value=0, norm="group"), (64, 128)),
              ("down2 64->64 @64->32", c2s.DownConvBlock(64, 64, 4, 2, 1, pad_value=0, norm="group"), (64, 64)),
              ("down3 64->128 @32->16", c2s.DownConvBlock(64, 128, 4, 2, 1, pad_value=0, norm="group"), (64, 32))]
    total = 0.0
    for name, blk, (c, r) in blocks:
        blk = blk.to(dev).eval()
        x = torch.randn((n, c, r, r), device=dev).to(torch.bfloat16)
        with torch.no_grad():
            ms = timed(lambda: blk(x), seconds)
        total += ms
        print(json.dumps({"record": "encoder block " + name, "frames": n, "ms": ms}), flush=True)
        del x
    macs = 128 * 128 * 64 * 9 * 74 + 64 * 64 * 64 * 64 * 34 + 32 * 32 * 64 * 64 * 34 + 16 * 16 * (64 * 64 * 16 + 9 * 64 * 128 + 9 * 128 * 128)
    print(json.dumps({"record": "U-TAE spatial encoder, four blocks", "frames": n, "ms": total, "frames_per_s": n / total * 1e3,
                      "tflops": 2.0 * n * macs / total * 1e-9}), flush=True)


if __name__ == "__main__":
    main()
