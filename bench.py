#!/usr/bin/env python
"""Benchmark of the L-TAE + TemporalAggregator hot path (BASELINE.json metric: patches/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

One "step" = one pass of the U-TAE temporal bottleneck over a batch of B synthetic patches
(BASELINE.json configs[1]: bf16, B=64, T=61 with irregular lengths 27..61 and pad masks):
``LTAE`` on x[B,61,128,16,16] followed by three ``TemporalAggregator('att_group')`` calls on
x[B,61,64,{32,64,128}^2].  Inputs are 11 GB per batch (> L2), so no L2 flush is needed.

* ``value``  : patches/s with the inputs resident in HBM, CUDA-event timed, max over ranks.
* ``e2e``    : same metric through the public modules with HOST (pinned) buffers: every step copies the
               step's inputs host->device and the outputs device->host inside the timed region.
* ``roofline``: achieved algorithmic GB/s of the dominant kernel (the 128x128 aggregation) against the
               measured HBM copy bandwidth in MEASURED_PEAKS.json.
* ``cpu_baseline`` / ``--impl reference``: the torch-CPU port of the reference modules (``oracle/torch_port.py``) timed
               on the host cores on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "patches/sec (T=61,C=10,128^2) LTAE+aggregator fwd"
UNIT = "patches/s"
T_FRAMES = 61
LEVELS = ((64, 32), (64, 64), (64, 128))  # (channels, resolution) of the three skip feature maps
LTAE_C, LTAE_RES = 128, 16
N_HEAD = 16
DUMP_PATCHES = 8  # 6.6 MB of float32 outputs per patch: 8 patches keep a dump under 64 MB at any batch size
FALLBACK_HBM_GBS = 6650.0  # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="patches per GPU per step")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "f32"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle check of one step's outputs")
    ap.add_argument("--cpu-patches", type=int, default=2, help="patches in the CPU-baseline sample")
    ap.add_argument("--no-sub", action="store_true", help="skip the sub-records (placements, training, tile, sustained)")
    ap.add_argument("--sub-seconds", type=float, default=1.0, help="minimum timed seconds of every sub-record")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a fixed sample of the last timed step's outputs to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path; it does not apply to --impl reference")
    return args


# ------------------------------------------------------------------------------------------------
# workload
# ------------------------------------------------------------------------------------------------
def make_lengths(batch, seed):
    import numpy as np
    rng = np.random.RandomState(seed)
    lengths = rng.randint(27, T_FRAMES + 1, size=batch)
    lengths[0] = T_FRAMES  # at least one full-length series (SURVEY.md section 8d)
    return lengths


def make_positions(lengths, seed):
    import numpy as np
    rng = np.random.RandomState(seed + 1)
    b = len(lengths)
    pos = np.zeros((b, T_FRAMES), dtype=np.int64)
    pad = np.zeros((b, T_FRAMES), dtype=bool)
    for i, L in enumerate(lengths):
        gaps = rng.randint(2, 11, size=L)
        gaps[0] = rng.randint(0, 11)
        pos[i, :L] = np.cumsum(gaps)
        pad[i, L:] = True
    return pos, pad


def algorithmic_bytes(lengths, elem):
    """SURVEY.md section 8d: x read once (valid frames only), outputs written once, fp32 attention once."""
    n_valid = int(sum(lengths))
    b = len(lengths)
    e_in = LTAE_C * LTAE_RES ** 2 + sum(c * r * r for c, r in LEVELS)
    e_out = e_in
    return elem * n_valid * e_in + elem * b * e_out + 4 * N_HEAD * T_FRAMES * LTAE_RES ** 2 * b


def agg128_bytes(lengths, elem):
    """Algorithmic bytes of the dominant launch: the 128x128 aggregation (x valid frames + out + attention read)."""
    c, r = LEVELS[-1]
    n_valid = int(sum(lengths))
    b = len(lengths)
    return elem * n_valid * c * r * r + elem * b * c * r * r + 4 * N_HEAD * n_valid * LTAE_RES ** 2


def dump_outputs(dump_dir, out, att, skips):
    """Write what one step returned -- the encoder's output and attention and the three aggregations -- for a fixed,
    seeded sample of the batch's patches as float32 ``dump_dir/<name>.npy``, so that two builds of the project can be
    compared output for output.  Returns a description of the files for the result line."""
    import numpy as np
    import torch
    batch = out.shape[0]
    patches = np.sort(np.random.RandomState(0).choice(batch, min(batch, DUMP_PATCHES), replace=False))
    idx = torch.from_numpy(patches).to(out.device)
    arrays = {"ltae_out": out.index_select(0, idx), "ltae_attn": att.index_select(1, idx)}
    for (_, r), s in zip(LEVELS, skips):
        arrays[f"agg_{r}"] = s.index_select(0, idx)
    os.makedirs(dump_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(dump_dir, name + ".npy"), t.float().cpu().numpy())
    return {"dir": dump_dir, "patches": patches.tolist(), "arrays": {n: list(t.shape) for n, t in arrays.items()}}


class ClockSampler:
    """SM clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md): NVML every 5 ms when
    pynvml is importable, else the recipe's nvidia-smi query."""
    QUERY = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.index, self._stop, self._thr = index, threading.Event(), None
        self.sm, self.max_sm, self.reasons, self.source = [], [], set(), "nvidia-smi"
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[index]) if visible and visible.split(",")[index].isdigit() else index
            self._handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self._nvml, self.source = pynvml, "nvml"
        except Exception:
            self._nvml = None

    def _sample_nvml(self):
        n = self._nvml
        self.sm.append(float(n.nvmlDeviceGetClockInfo(self._handle, n.NVML_CLOCK_SM)))
        self.max_sm.append(float(n.nvmlDeviceGetMaxClockInfo(self._handle, n.NVML_CLOCK_SM)))
        get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        bits = get(self._handle)
        for name, const in (("hw_slowdown", "nvmlClocksThrottleReasonHwSlowdown"),
                            ("hw_thermal_slowdown", "nvmlClocksThrottleReasonHwThermalSlowdown"),
                            ("sw_thermal_slowdown", "nvmlClocksThrottleReasonSwThermalSlowdown"),
                            ("sw_power_cap", "nvmlClocksThrottleReasonSwPowerCap")):
            if bits & getattr(n, const, 0):
                self.reasons.add(name)

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                              "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
        if not out.strip():
            return
        r = [f.strip() for f in out.strip().splitlines()[0].split(",")]
        self.sm.append(float(r[0]))
        self.max_sm.append(float(r[1]))
        for name, v in zip(self.NAMES, r[2:6]):
            if v.lower().startswith("active"):
                self.reasons.add(name)

    def _run(self):
        while not self._stop.is_set():
            try:
                if self._nvml is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            self._stop.wait(0.001 if self._nvml is not None else 0.1)

    def __enter__(self):
        # the launching thread holds the GIL almost all the time: hand it over every 0.5 ms instead of every 5 ms so
        # that a 30 ms timed region still yields a few dozen samples (the steps are GPU-bound, not launch-bound)
        self._switch = sys.getswitchinterval()
        sys.setswitchinterval(5e-4)
        self._thr = threading.Thread(target=self._run, daemon=True)
        self._thr.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._thr.join(timeout=10)
        sys.setswitchinterval(self._switch)

    def summary(self):
        import statistics
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None,
                "sm_max_mhz": max(self.max_sm) if self.max_sm else None,
                "reasons": sorted(self.reasons), "samples": len(self.sm), "source": self.source}


# ------------------------------------------------------------------------------------------------
# CPU leg: the numpy port of the reference algorithm (oracle/) on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_leg(n_patches, repeats, seed=1234):
    import numpy as np
    import torch
    import crop2seg_b200 as c2s
    from oracle import LtaeConfig
    from oracle.torch_port import ltae_forward_torch, temporal_aggregator_torch
    from c2s_testlib import oracle_params, randomise

    torch.set_num_threads(os.cpu_count() or 1)
    rng = np.random.RandomState(seed)
    enc = c2s.LTAE(in_channels=LTAE_C, n_head=N_HEAD, d_k=4, mlp=[256, 128], d_model=256)
    randomise(enc, rng)
    params = oracle_params(enc)
    cfg = LtaeConfig(in_channels=LTAE_C, n_head=N_HEAD, d_k=4, mlp=[256, 128], d_model=256)
    lengths = [T_FRAMES] + [27] * (n_patches - 1)  # BASELINE configs[0]: one series of length 27
    pos, pad = make_positions(lengths, seed)

    def feat(c, r):
        x = np.maximum(rng.standard_normal((n_patches, T_FRAMES, c, r, r)).astype(np.float32), 0)
        x[pad] = 0
        return x

    x4 = torch.from_numpy(feat(LTAE_C, LTAE_RES))
    xs = [torch.from_numpy(feat(c, r)) for c, r in LEVELS]
    params = {k: torch.from_numpy(v) for k, v in params.items()}
    pos, pad = torch.from_numpy(pos), torch.from_numpy(pad)
    best = float("inf")
    with torch.no_grad():
        for _ in range(repeats):
            t0 = time.perf_counter()
            _, att = ltae_forward_torch(cfg, params, x4, pos, pad)
            for x in xs:
                temporal_aggregator_torch(x, pad, att, "att_group")
            best = min(best, time.perf_counter() - t0)
    return n_patches / best, best


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    times = []
    for _ in range(args.warmup):
        cpu_leg(args.cpu_patches, 1)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        v, dt = cpu_leg(args.cpu_patches, 1)
        times.append(dt)
    total = time.perf_counter() - t0
    value = args.cpu_patches * args.steps / sum(times)
    sample = (f"{args.cpu_patches} patches/step (U-TAE placement fp32, T=61, one full series + series of length 27), "
              f"torch-CPU port of the reference modules (oracle/torch_port.py: the reference's ATen calls and materialising copies, pinned on the reference's outputs; the reference itself cannot travel to the GPU box)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "U-TAE placement: LTAE[B,61,128,16,16] + 3x TemporalAggregator[B,61,64,{32,64,128}^2]",
                   "batch_per_step": args.cpu_patches, "wall_s": total},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU leg
# ------------------------------------------------------------------------------------------------
def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import crop2seg_b200 as c2s
    from crop2seg_b200 import _lib
    from c2s_testlib import randomise

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: crop2seg_b200 has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()

    dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float32
    elem = 2 if args.dtype == "bf16" else 4
    B = args.batch
    seed = 1234 + rank  # every rank owns its own shard of patches (weak scaling, no collective on the data path)
    lengths = make_lengths(B, seed)
    pos_np, pad_np = make_positions(lengths, seed)
    pos = torch.from_numpy(pos_np).to(dev)
    pad = torch.from_numpy(pad_np).to(dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed)

    def feat(c, r):
        x = torch.empty((B, T_FRAMES, c, r, r), dtype=dtype, device=dev)
        for i in range(B):  # generated per sample to bound the fp32 temporaries
            v = torch.randn((T_FRAMES, c, r, r), device=dev, generator=gen).clamp_(min=0)
            v[pad[i]] = 0  # padded frames are exactly zero (temp_shared_block.py:30-40)
            x[i] = v.to(dtype)
        return x

    x4 = feat(LTAE_C, LTAE_RES)
    xs = [feat(c, r) for c, r in LEVELS]
    enc = c2s.LTAE(in_channels=LTAE_C, n_head=N_HEAD, d_k=4, mlp=[256, 128], d_model=256)
    randomise(enc, np.random.RandomState(1234))
    enc = enc.to(dev).eval()
    enc.assume_zero_padded = True
    agg = c2s.TemporalAggregator(mode="att_group")

    def step(x4_, xs_, timers=None):
        def mark():
            if timers is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                timers.append(ev)
        with torch.no_grad():
            mark()
            out, att = enc(x4_, batch_positions=pos, pad_mask=pad)
            mark()
            skips = []
            for x in xs_:
                skips.append(agg(x, pad_mask=pad, attn_mask=att))
                mark()
        return out, att, skips

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- resident-input throughput -----------------------------------------------------------
    for _ in range(args.warmup):
        step(x4, xs)
    barrier()
    _lib.reset_launch_count()
    timers = []
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        start.record()
        for _ in range(args.steps - 1):
            step(x4, xs, timers)
        last = step(x4, xs, timers)  # kept for --dump-outputs; no step runs while it is held
        stop.record()
        barrier()
    launches = _lib.launch_count()
    dumped = dump_outputs(args.dump_outputs, *last) if args.dump_outputs and rank == 0 else None
    del last
    elapsed_ms = start.elapsed_time(stop)
    t = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())
    value = world * B * args.steps / (elapsed_ms * 1e-3)

    # per-kernel durations (events recorded on the launching stream inside the timed region)
    per = [0.0] * 4
    for s in range(args.steps):
        evs = timers[s * 5:(s + 1) * 5]
        for k in range(4):
            per[k] += evs[k].elapsed_time(evs[k + 1])
    per = [p / args.steps for p in per]  # ms: [ltae(+prep), agg32, agg64, agg128]

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    else:
        peak, peak_src = FALLBACK_HBM_GBS, "B200_PROFILING.md fallback"
    a128 = agg128_bytes(lengths, elem) / (per[3] * 1e-3) / 1e9
    traffic = None  # DRAM bytes per launch of the same kernel from the committed ncu --set full capture
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath) and B == 64 and args.dtype == "bf16":
        traffic = json.load(open(tpath)).get("agg_pipe_x8_b64_bf16_dram_bytes")
    step_bytes = algorithmic_bytes(lengths, elem)
    roofline = {
        "bound": "hbm", "kernel": "agg_forward<x8> (TemporalAggregator att_group, x[B,61,64,128,128])",
        "achieved": a128, "peak": peak, "unit": "GB/s", "frac": a128 / peak, "traffic": traffic,
        "algorithmic_bytes": agg128_bytes(lengths, elem),
        "peak_source": peak_src, "kernel_ms": per[3],
        "peak_note": "the measured peak is a COPY bandwidth (half reads, half writes); this kernel is 98 percent reads, so "
                     f"a fraction above 1 is possible ({a128 / 7700.0:.2f} of the 7.7 TB/s HBM3e figure of the hardware guide)",
        "step": {"algorithmic_bytes": step_bytes, "achieved_gbs": step_bytes / (elapsed_ms / args.steps * 1e-3) / 1e9,
                 "frac": step_bytes / (elapsed_ms / args.steps * 1e-3) / 1e9 / peak,
                 "kernel_ms": {"ltae": per[0], "agg32": per[1], "agg64": per[2], "agg128": per[3]}},
    }

    # ---- parity of one step at the benchmarked shapes (outside every timed region): first, middle and LAST sample
    #      of the batch against the oracle on the host (offsets beyond 2^32 elements are exercised by the last one) ----
    parity = None
    if not args.no_parity:
        from c2s_testlib import hot_path_parity
        out_p, att_p = None, None
        with torch.no_grad():
            out_p, att_p = enc(x4, batch_positions=pos, pad_mask=pad)
            skips_p = [agg(x, pad_mask=pad, attn_mask=att_p) for x in xs]
        torch.cuda.synchronize()
        parity = hot_path_parity(enc, x4, xs, pos, pad, out_p, att_p, skips_p, samples=sorted({0, B // 2, B - 1}))
        parity["tolerance"] = 1e-2 if args.dtype == "bf16" else 1e-4
        parity["ok"] = bool(parity["attn"] < parity["tolerance"] and parity["out"] < parity["tolerance"]
                            and max(parity["skips"]) < parity["tolerance"] and parity["pad_attention_exactly_zero"])
        del out_p, att_p, skips_p

    # ---- end to end through the modules with host buffers -------------------------------------
    e2e = None
    if not args.no_e2e:
        chunk = min(8, B)
        n_chunks = B // chunk
        host_in = [x.cpu().pin_memory() for x in [x4] + xs]
        host_out = [torch.empty((B, c, r, r), dtype=dtype).pin_memory() for c, r in [(128, LTAE_RES)] + list(LEVELS)]
        dev_in = [[torch.empty((chunk,) + tuple(h.shape[1:]), dtype=dtype, device=dev) for h in host_in] for _ in range(2)]
        copy_s = torch.cuda.Stream(device=dev)
        comp_s = torch.cuda.current_stream(dev)
        # only the valid frames of every series cross PCIe (crop2seg_b200.copy_valid_frames_): the kernels never read
        # a padded frame, so the device buffers may keep stale data there
        frame_bytes = sum(h[0, 0].numel() * h.element_size() for h in host_in)
        h2d = int(lengths.sum()) * frame_bytes + pos.numel() * 8 + pad.numel()
        len_list = [int(v) for v in lengths]
        d2h = sum(h.numel() * h.element_size() for h in host_out)
        pos_h, pad_h = pos.cpu().pin_memory(), pad.cpu().pin_memory()

        def e2e_step():
            loaded = [torch.cuda.Event() for _ in range(n_chunks)]
            freed = [None, None]
            for ci in range(n_chunks):
                sl = slice(ci * chunk, (ci + 1) * chunk)
                buf = dev_in[ci % 2]
                with torch.cuda.stream(copy_s):
                    if freed[ci % 2] is not None:
                        copy_s.wait_event(freed[ci % 2])
                    for d, h in zip(buf, host_in):
                        c2s.copy_valid_frames_(d, h[sl], len_list[sl])
                    p_d = pos_h[sl].to(dev, non_blocking=True)
                    m_d = pad_h[sl].to(dev, non_blocking=True)
                    loaded[ci].record(copy_s)
                comp_s.wait_event(loaded[ci])
                with torch.no_grad():
                    out, att = enc(buf[0], batch_positions=p_d, pad_mask=m_d)
                    outs = [out] + [agg(x, pad_mask=m_d, attn_mask=att) for x in buf[1:]]
                for o, h in zip(outs, host_out):
                    h[sl].copy_(o, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(comp_s)
                freed[ci % 2] = ev
                p_d.record_stream(comp_s), m_d.record_stream(comp_s)

        e_steps = max(2, min(args.steps, 5))
        for _ in range(2):
            e2e_step()
        barrier()
        s2, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s2.record()
        for _ in range(e_steps):
            e2e_step()
        e2.record()
        barrier()
        t2 = torch.tensor([s2.elapsed_time(e2)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        e2e_s = float(t2.item()) * 1e-3
        e2e = {"value": world * B * e_steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "steps": e_steps,
               "note": "pinned host buffers, 8-patch chunks double-buffered on a copy stream, padded frames are not copied; "
                       "PCIe-bound"}
        del host_in, host_out, dev_in
        # the ceiling beside it: a plain pinned cudaMemcpyAsync of 1 GiB in each direction, all ranks at the same time
        from tools.bench_lib import pcie_ceiling
        link = pcie_ceiling(dev)
        e2e["h2d_gbs_achieved"] = h2d * e_steps / e2e_s / 1e9
        e2e["pcie_gbs_measured"] = link["h2d_gbs"]
        e2e["pcie_d2h_gbs_measured"] = link["d2h_gbs"]
        e2e["frac"] = e2e["h2d_gbs_achieved"] / link["h2d_gbs"]
        e2e["frac_note"] = ("host->device bytes per second of the e2e steps over the measured rate of one plain pinned "
                            "host->device copy per rank, all ranks concurrently (max time over ranks)")

    # ---- sub-records: every placement, the training step and the full tile, each timed for >= --sub-seconds ----
    sub = {}
    if not args.no_sub:
        from tools import bench_lib
        del x4, xs
        torch.cuda.empty_cache()
        with ClockSampler(local_rank) as sub_clocks:
            sub["placements"] = bench_lib.placements(dev, B=B, min_seconds=args.sub_seconds)
            sub["training"] = bench_lib.training(dev, local_rank, B=16, min_seconds=args.sub_seconds)
            sub["tile"] = bench_lib.tile(dev, "timeunet", B=B)
            sub["tile_utae"] = bench_lib.tile(dev, "utae", B=B)
            sub["encoder"] = bench_lib.encoder(dev, frames=1024, min_seconds=args.sub_seconds)
        sub["sub_clocks"] = sub_clocks.summary()  # sampled over the sub-records (several seconds of load)
        if rank == 0 and world > 1:
            sub["topology"] = bench_lib.topology()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        v, dt = cpu_leg(args.cpu_patches, 3)
        cpu = {"value": v, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
               "sample": f"{args.cpu_patches} patches (fp32, T=61, one series of length 27), best of 3, "
                         f"torch-CPU port of the reference modules (oracle/torch_port.py), {dt:.2f} s per pass"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": "BASELINE configs[1]: U-TAE placement, LTAE[B,61,128,16,16] + 3x TemporalAggregator"
                                   "[B,61,64,{32,64,128}^2], irregular T 27..61 with pad masks",
                       "batch_per_gpu": B, "mean_valid_frames": float(np.mean(lengths)),
                       "l2": "inputs (11 GB/step) exceed L2; no flush", "sharding": f"{world} x independent patch shards"},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "parity": parity, "gpu_launches": int(launches),
            "clocks": clocks.summary(),
        }
        if dumped is not None:
            line["dump"] = dumped
        line.update(sub)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
