"""Backward of the aggregation + skip convolution with the BatchNorm frozen: fused kernel (c2s_agg_skipconv_backward) vs
the unfused route (skip map materialised by the aggregator kernel, torch autograd of Conv2d/BatchNorm2d(eval)/ReLU in
bf16, then c2s_agg_backward), at U-TAE's three skip levels.

    python tools/bench_skipconv_backward.py [--batch 16] [--rounds 10] [--steps 10] [--out FILE]
One JSON line per level (and a header line with the card name and power limit).  The two routes alternate, round by
round, in one process; times are medians over the rounds of CUDA-event means over --steps calls.  x is larger than L2 at
every level but 32 x 32 (B = 16: 64 MB, read from L2 after the first pass there).  The HBM bytes are the ones the fused
kernel needs: x on the valid frames read once, grad_x written on every frame, out and grad_out read, the attention read
and its gradient written once."""
import argparse, json, os, statistics, subprocess, sys
import numpy as np, torch
from torch import nn
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import crop2seg_b200 as c2s
from crop2seg_b200 import _lib, ops
from bench import LEVELS, T_FRAMES, make_lengths, make_positions
from c2s_testlib import random_attention

HBM_GBS = 7700.0  # HGX B200 data sheet, one GPU

ap = argparse.ArgumentParser()
ap.add_argument("--batch", type=int, default=16); ap.add_argument("--rounds", type=int, default=10)
ap.add_argument("--steps", type=int, default=10); ap.add_argument("--out", default=None)
args = ap.parse_args()
if not torch.cuda.is_available():
    raise SystemExit("bench_skipconv_backward: no CUDA device")
dev = torch.device("cuda", 0); B = args.batch
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
lines = [{"card": card or torch.cuda.get_device_name(0), "batch": B, "frames": T_FRAMES}]
lengths = make_lengths(B, 1234); _, pad_np = make_positions(lengths, 1234)
pad = torch.from_numpy(pad_np).to(dev)
attn = torch.from_numpy(random_attention(np.random.RandomState(1), 16, pad_np, 16, 16)).to(dev)
agg = c2s.TemporalAggregator("att_group")


def timed(fn):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(args.steps):
        fn()
    e.record(); torch.cuda.synchronize()
    return s.elapsed_time(e) / args.steps


for c, r in LEVELS:
    x = torch.empty((B, T_FRAMES, c, r, r), dtype=torch.bfloat16, device=dev)
    for i in range(B):
        v = torch.randn((T_FRAMES, c, r, r), device=dev).clamp_(min=0); v[pad[i]] = 0; x[i] = v.to(torch.bfloat16)
    block = nn.Sequential(nn.Conv2d(c, c, 1), nn.BatchNorm2d(c), nn.ReLU()).to(dev).eval()
    with torch.no_grad():
        block[1].running_mean.normal_(0, 0.3); block[1].running_var.uniform_(0.5, 2.0)
    block_bf16 = nn.Sequential(nn.Conv2d(c, c, 1), nn.BatchNorm2d(c), nn.ReLU()).to(dev).eval()
    block_bf16.load_state_dict(block.state_dict()); block_bf16 = block_bf16.to(torch.bfloat16)
    conv, bn = block[0], block[1]
    params = (conv.weight, conv.bias, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.eps)
    gout = torch.randn((B, c, r, r), device=dev).to(torch.bfloat16)
    with torch.no_grad():
        out = ops.temporal_aggregate_skip_conv(x, pad, attn, *params)
    # unfused: the skip map is materialised and kept with the graph of the torch block, as autograd keeps it
    skip = agg(x, pad_mask=pad, attn_mask=attn).requires_grad_(True)
    y = block_bf16(skip)
    wrt = [skip] + list(block_bf16.parameters())

    def fused():
        ops.temporal_aggregate_skip_conv_backward(x, pad, attn, *params, out, gout)

    def unfused():
        g = torch.autograd.grad(y, wrt, gout, retain_graph=True)
        ops.temporal_aggregate_backward(x, pad, attn, g[0], "att_group")

    for fn in (fused, unfused, fused, unfused):  # warm-up: module loads, cuDNN algorithm choice
        fn()
    torch.cuda.synchronize()
    t_f, t_u = [], []
    for _ in range(args.rounds):
        t_f.append(timed(fused)); t_u.append(timed(unfused))
    fused(); kname = _lib.last_kernel()
    tf, tu = statistics.median(t_f), statistics.median(t_u)
    n_valid = int(sum(lengths))
    nbytes = (2 * n_valid * c * r * r + 2 * B * T_FRAMES * c * r * r + 2 * 2 * B * c * r * r
              + 2 * 4 * 16 * B * T_FRAMES * 256)
    lines.append({"level": f"{c}x{r}x{r}", "batch": B, "fused_ms": round(tf, 4), "unfused_ms": round(tu, 4),
                  "speedup": round(tu / tf, 3), "fused_gbs": round(nbytes / tf / 1e6, 1),
                  "fused_frac_of_hbm_roofline": round(nbytes / tf / 1e6 / HBM_GBS, 3),
                  "fused_ms_spread": [round(min(t_f), 4), round(max(t_f), 4)],
                  "unfused_ms_spread": [round(min(t_u), 4), round(max(t_u), 4)], "kernel": kname})
    del x, skip, y
    torch.cuda.empty_cache()

for line in lines:
    print(json.dumps(line))
if args.out:
    with open(args.out, "w") as f:
        f.write("".join(json.dumps(line) + "\n" for line in lines))
