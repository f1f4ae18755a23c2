"""Training step of the aggregation + skip convolution with its BatchNorm in training mode (batch statistics): fused
kernels (c2s_agg_skipconv_bstats_forward + c2s_agg_skipconv_bstats_backward) vs the unfused route (skip map materialised
by c2s_agg_forward, torch autograd of Conv2d/BatchNorm2d(train)/ReLU in bf16, then c2s_agg_backward), at U-TAE's three
skip levels.  For reference it also times the fused kernels with the BatchNorm frozen (running statistics).  The three
routes are timed as a training loop calls them: the fused ones through TemporalAggregator.forward_skip_conv and
torch.autograd.grad w.r.t. x, the attention and the block's parameters (so the fused batch-statistics route includes its
running-statistics update, as torch's BatchNorm does in the unfused route).  The *_fwd / *_bwd parts are the ops-level
calls alone (no autograd, no running-statistics update), for the ratios against the frozen kernels.

    python tools/bench_skipconv_bstats.py [--batch 16] [--rounds 10] [--steps 10] [--out FILE]
One JSON line per level (and a header line with the card name and power limit).  The routes alternate, round by round,
in one process; times are medians over the rounds of CUDA-event means over --steps calls.  x is larger than L2 at every
level but 32 x 32 (B = 16: 64 MB, read from L2 after the first pass there).  The HBM bytes are the ones the fused step
needs: x on the valid frames read twice (forward and backward), grad_x written on every frame, the attention read twice
and its gradient written once, and nine [B,64,H,W] bf16 maps (forward: z written, read, out written; backward: grad_out,
out and z read by the statistics pre-pass and again by the main kernel)."""
import argparse, copy, json, os, statistics, subprocess, sys
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
    raise SystemExit("bench_skipconv_bstats: no CUDA device")
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
    block = nn.Sequential(nn.Conv2d(c, c, 1), nn.BatchNorm2d(c), nn.ReLU()).to(dev)
    with torch.no_grad():
        block[1].running_mean.normal_(0, 0.3); block[1].running_var.uniform_(0.5, 2.0)
    block_bf16 = nn.Sequential(nn.Conv2d(c, c, 1), nn.BatchNorm2d(c), nn.ReLU()).to(dev)
    block_bf16.load_state_dict(block.state_dict()); block_bf16 = block_bf16.to(torch.bfloat16).train()
    conv, bn = block[0], block[1]
    train_params = (conv.weight, conv.bias, bn.weight, bn.bias, bn.eps)
    frozen_params = (conv.weight, conv.bias, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.eps)
    gout = torch.randn((B, c, r, r), device=dev).to(torch.bfloat16)
    wrt = list(block_bf16.parameters())

    xg, ag = x.detach().requires_grad_(True), attn.detach().requires_grad_(True)
    block.train()
    block_eval = copy.deepcopy(block).eval()

    def fused():
        out = agg.forward_skip_conv(xg, pad, ag, block, allow_batch_stats=True)
        torch.autograd.grad(out, [xg, ag] + list(block.parameters()), gout)

    def unfused():
        skip = agg(x, pad_mask=pad, attn_mask=attn).requires_grad_(True)
        y = block_bf16(skip)
        g = torch.autograd.grad(y, [skip] + wrt, gout)
        ops.temporal_aggregate_backward(x, pad, attn, g[0], "att_group")

    def frozen():
        out = agg.forward_skip_conv(xg, pad, ag, block_eval)
        torch.autograd.grad(out, [xg, ag] + list(block_eval.parameters()), gout)

    with torch.no_grad():
        out, z, mean, var = ops.temporal_aggregate_skip_conv_bstats_forward(x, pad, attn, *train_params)
        out_e = ops.temporal_aggregate_skip_conv_forward(x, pad, attn, *frozen_params)
    parts = {"fused_fwd": lambda: ops.temporal_aggregate_skip_conv_bstats_forward(x, pad, attn, *train_params),
             "fused_bwd": lambda: ops.temporal_aggregate_skip_conv_bstats_backward(x, pad, attn, *train_params, z, mean,
                                                                                   var, out, gout),
             "frozen_fwd": lambda: ops.temporal_aggregate_skip_conv_forward(x, pad, attn, *frozen_params),
             "frozen_bwd": lambda: ops.temporal_aggregate_skip_conv_backward(x, pad, attn, *frozen_params, out_e, gout)}
    routes = {"fused": fused, "unfused": unfused, "frozen": frozen, **parts}
    for fn in list(routes.values()) * 2:  # warm-up: module loads, cuDNN algorithm choice
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in routes}
    for _ in range(args.rounds):
        for k, fn in routes.items():
            times[k].append(timed(fn))
    fused(); kname = _lib.last_kernel()
    med = {k: statistics.median(v) for k, v in times.items()}
    n_valid = int(sum(lengths))
    nbytes = (2 * 2 * n_valid * c * r * r + 2 * B * T_FRAMES * c * r * r + 3 * 4 * 16 * B * T_FRAMES * 256
              + 9 * 2 * B * c * r * r)
    line = {"level": f"{c}x{r}x{r}", "batch": B, "fused_ms": round(med["fused"], 4), "unfused_ms": round(med["unfused"], 4),
            "speedup": round(med["unfused"] / med["fused"], 3), "fused_gbs": round(nbytes / med["fused"] / 1e6, 1),
            "fused_frac_of_hbm_roofline": round(nbytes / med["fused"] / 1e6 / HBM_GBS, 3),
            "fused_ms_spread": [round(min(times["fused"]), 4), round(max(times["fused"]), 4)],
            "unfused_ms_spread": [round(min(times["unfused"]), 4), round(max(times["unfused"]), 4)],
            "frozen_bn_ms": round(med["frozen"], 4)}
    for k in parts:
        line[k + "_ms"] = round(med[k], 4)
    line["fwd_over_frozen"] = round(med["fused_fwd"] / med["frozen_fwd"], 3)
    line["bwd_over_frozen"] = round(med["fused_bwd"] / med["frozen_bwd"], 3)
    line["kernel"] = kname
    lines.append(line)
    del x, xg, ag, out, z, out_e
    torch.cuda.empty_cache()

for line in lines:
    print(json.dumps(line))
if args.out:
    with open(args.out, "w") as f:
        f.write("".join(json.dumps(line) + "\n" for line in lines))
