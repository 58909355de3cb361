#!/usr/bin/env python
"""Benchmark of the PPN output-parsing path (decode + NMS + limb arg-max + tree parse).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config cfg2] [--impl ours|reference] [--dump-outputs DIR]

One step = one pass of the whole path over one batch of synthetic head tensors per GPU
(BASELINE.json configs[1]: MPII 16-part, 384x384, 12x12 grid, 9x9 window, batch 512).  N > 1 is
launched by torchrun, one rank per GPU; every rank parses its own batch (weak scaling, images are
independent) and the poses are gathered at rank 0 inside the timed region: the parse kernel stores its
dense records straight into rank 0's peer-mapped buffer over NVLink, NCCL carries the 8-byte "landed"
notifications and the timings (sharded.PeerPoseGatherer; --gather selects the alternatives).
`--config cfg5` is BASELINE.json configs[4]: 8 192 images in contiguous blocks per rank, streamed in
chunks of 512, poses gathered (strong scaling: the job is fixed).
Rank 0 prints ONE JSON line (see README / DESIGN.md for the keys).

`--impl reference` times the reference's CPU algorithm (the numpy port in oracle/, which follows
datatest.py line by line and is checked against the reference's own outputs) on all host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH = {"cfg1": 1, "cfg2": 512, "cfg3": 1024, "cfg4": 256, "native": 64, "cfg5": 512}
DIST = {"cfg1": "U", "cfg2": "U", "cfg3": "D", "cfg4": "U", "native": "U", "cfg5": "U"}
PRESET = {"cfg5": "cfg2"}                     # cfg5 streams cfg2-shaped images
CFG5_IMAGES = 8192
WORKLOAD = {
    "cfg1": "MPII 16-part PPN, 384x384 (12x12 grid, 9x9 limb window), batch 1 (latency)",
    "cfg2": "MPII 16-part PPN, 384x384 (12x12 grid, 9x9 limb window), batch 512 synthetic head tensors per GPU",
    "cfg3": "COCO 18-part PPN, 512x512 (16x16 grid, 9x9 window), batch 1024, dense crowd",
    "cfg4": "18-part PPN, 768x768 (24x24 grid, 11x11 window), batch 256",
    "native": "reference-native 18-part PPN, 384x384 (24x24 grid, 21x21 window), batch 64",
    "cfg5": "streaming image-sharded decode: 8192 MPII 16-part images (12x12 grid, 9x9 window) in contiguous blocks per GPU, "
            "chunks of 512, poses gathered at rank 0",
}
METRIC = "PPN decode+NMS+parse images/s"


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


# ----------------------------------------------------------------------------------------------
# clocks: sampled DURING the run with NVML (falls back to nvidia-smi)
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, cuda_index: int, period_s: float = 0.01):
        self.period = period_s
        self.samples = []          # (t, sm_mhz, reasons_bits, power_w)
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None
        self.h = None
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            self.nv = pynvml
            uuid = str(torch.cuda.get_device_properties(cuda_index).uuid)
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
            except Exception:
                try:
                    self.h = pynvml.nvmlDeviceGetHandleByUUID("GPU-" + uuid)
                except Exception:
                    self.h = pynvml.nvmlDeviceGetHandleByIndex(cuda_index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:                                     # pragma: no cover
            self.err = repr(e)
            self.h = None

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    bits = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                try:
                    pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                except Exception:
                    pw = None
                self.samples.append((time.perf_counter(), float(mhz), int(bits), pw))
            except Exception:
                pass
            self._stop.wait(self.period)

    def start(self):
        if self.h is not None:
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()
        return self

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=2)

    def summary(self, t0=None, t1=None):
        if self.h is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "NVML unavailable: " + getattr(self, "err", "")}
        sel = [s for s in self.samples if (t0 is None or s[0] >= t0) and (t1 is None or s[0] <= t1)]
        window = "timed region"
        if len(sel) < 3:                       # a short timed region: use every sample taken under load
            sel, window = self.samples, "warm-up + timed region"
        reasons = set()
        for _, _, bits, _ in sel:
            for bit, name in self.REASONS.items():
                if bits & bit:
                    reasons.add(name)
        mhz = [s[1] for s in sel]
        pw = [s[3] for s in sel if s[3] is not None]
        return {"sm_mhz": statistics.median(mhz) if mhz else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(reasons), "samples": len(sel), "window": window,
                "power_w_max": max(pw) if pw else None}


def preset_of(name):
    from pytorch_pose_proposal_network_b200.config import PRESETS
    return PRESETS[PRESET.get(name, name)]()


def images_per_step(args, world=1):
    if args.config == "cfg5":
        return CFG5_IMAGES                    # the whole job, whatever the number of GPUs
    return (args.batch or BATCH[args.config]) * world


# ----------------------------------------------------------------------------------------------
# reference arm: the CPU algorithm on all host cores
# ----------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    if rank != 0:
        return 0
    from oracle import cpu_bench, ppn_oracle as O
    cfg = preset_of(args.config)
    g = O.Geometry.of(cfg)
    cores = cpu_bench.host_cores()
    per_step = images_per_step(args, 1)              # the same images per step as one GPU of our arm parses
    sample = min(per_step, 32)
    pool = cpu_bench.CpuPool(g, dist=DIST[args.config], seed=0, n_images=per_step, cores=cores, sample_images=sample)
    try:
        for _ in range(max(min(args.warmup, 2), 1)):
            pool.one_pass()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            pool.one_pass()
        dt = time.perf_counter() - t0
    finally:
        pool.close()
    value = per_step * args.steps / dt
    sample_txt = (f"{per_step} images per step, cycling a {sample}-image synthetic sample ({DIST[args.config]}, seed 0) held by every "
                  f"worker, through the numpy port of datatest.py (oracle/ppn_oracle.parse_head_like_reference), process pool over "
                  f"{cores} cores")
    B = args.batch or BATCH[args.config]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "strong" if args.config == "cfg5" else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD[args.config], "preset": args.config, "images_per_gpu_per_step": B,
                   "K": cfg.K, "E": cfg.E, "grid": [cfg.H, cfg.W], "window": [cfg.sH, cfg.sW],
                   "bytes_per_image": cfg.C * cfg.HW * 4, "head_dtype": "f32", "input_distribution": DIST[args.config]},
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample_txt},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ----------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------
def make_batches(torch, cfg, B, dist_name, dev, head_dtype, n_buf, seed):
    """n_buf distinct input batches generated on the device (SURVEY §8d distributions)."""
    gen = torch.Generator(device=dev).manual_seed(seed)
    bufs = []
    for _ in range(n_buf):
        t = torch.rand(B, cfg.C, cfg.H, cfg.W, device=dev, generator=gen)
        if dist_name == "D":
            t[:, :2 * cfg.K] = 0.4 + 0.6 * t[:, :2 * cfg.K]
            t[:, 4 * cfg.K:6 * cfg.K] *= 0.08
        bufs.append(t.to(head_dtype))               # a 16-bit head: same values rounded once, widened exactly by the kernels
        del t
    return bufs


def timed_loop(torch, dev, fn, K, pre_sync=None):
    """K calls of fn(i) between two events on torch's current stream -> ms per call."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    (pre_sync or (lambda: torch.cuda.synchronize(dev)))()
    a.record()
    for i in range(K):
        fn(i)
    b.record()
    torch.cuda.synchronize(dev)
    return a.elapsed_time(b) / K


def measure_other_config(torch, name, dev, steps=30, warmup=5):
    """One compact record for a BASELINE config that is not the headline one (1 GPU)."""
    from pytorch_pose_proposal_network_b200.parser import PoseParser
    cfg = preset_of(name)
    B = BATCH[name]
    parser = PoseParser(cfg, device=dev)
    batch_bytes = B * cfg.C * cfg.HW * 4
    n_buf = max(2, min(4, -(-(1 << 29) // batch_bytes)))
    bufs = make_batches(torch, cfg, B, DIST[name], dev, torch.float32, n_buf, seed=4000)
    outs = [parser.alloc_output(B) for _ in range(2)]
    step = lambda i: parser.parse(bufs[i % n_buf], out=outs[i % 2], input_complete=True)
    for i in range(warmup):
        step(i)
    ms = timed_loop(torch, dev, step, steps)
    counts = outs[(steps - 1) % 2].count.float().mean().item()
    plan = parser.parse_plan(B)
    del bufs, outs, parser
    torch.cuda.empty_cache()
    return {"images_per_step": B, "ms_per_step": ms, "value": B / (ms * 1e-3), "gbs": batch_bytes / (ms * 1e-3) / 1e9,
            "launches_per_step": plan["launches"], "humans_per_image": counts, "steps": steps,
            "l2": "inputs rotate over %d batches of %.0f MB%s" % (n_buf, batch_bytes / 1e6, "" if batch_bytes * n_buf > (126 << 20)
                                                                   else " (smaller than L2: a latency figure, not a bandwidth one)")}


def measure_fused_head(torch, dev, peaks, name="cfg2", B=512, Cin=512, iters=20):
    """The widened path of SURVEY §8f row 1 on the same preset: conv3 (1x1, model.py:85) + sigmoid + the whole parse from
    the last layer's INPUT (PoseParser.parse_features -> ppn_head_parse_opt), beside cuDNN's convolution alone.
    FLOPs against the measured bf16 tensor peak (TF32 runs at half of it)."""
    from pytorch_pose_proposal_network_b200.config import PRESETS
    from pytorch_pose_proposal_network_b200.parser import PoseParser
    cfg = PRESETS[name]()
    gen = torch.Generator(device=dev).manual_seed(5)
    feats = [torch.randn(B, Cin, cfg.H, cfg.W, device=dev, generator=gen) for _ in range(3)]
    weight = (torch.randn(cfg.C, Cin, device=dev, generator=gen) * (2.0 / (1.01 * Cin)) ** 0.5).contiguous()
    bias = torch.randn(cfg.C, device=dev, generator=gen) * 0.5
    bias[:2 * cfg.K] += 1.0
    parser = PoseParser(cfg, device=dev)
    outs = [parser.alloc_output(B) for _ in range(2)]
    flops = 2.0 * B * cfg.HW * cfg.C * Cin

    def timed(fn):
        for i in range(3):
            fn(i)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        a.record()
        for i in range(iters):
            fn(i)
        b.record()
        torch.cuda.synchronize(dev)
        return a.elapsed_time(b) / iters

    bf16_peak = peaks.get("bf16_tflops") or 1590.0
    rec = {"preset": name, "images_per_call": B, "Cin": Cin, "gflop_per_call": flops / 1e9, "calls": iters,
           "api": "PoseParser.parse_features(feat, conv3.weight, conv3.bias, operand=...) -> ppn_head_parse_opt: memset, [pack,] "
                  "tcgen05 GEMM + arg-max epilogue, finalize, fused parse; inputs resident, 3 feature batches rotated"}
    ms = timed(lambda i: parser.parse_features(feats[i % 3], weight, bias, out=outs[i % 2]))
    rec["tf32_nchw_in_place"] = {"ms_per_call": ms, "images_per_s": B / ms * 1e3, "tflops": flops / ms / 1e9,
                                 "frac_of_tensor_peak": flops / ms / 1e9 / (bf16_peak / 2), "peak_tflops": bf16_peak / 2}
    ms = timed(lambda i: parser.parse_features(feats[i % 3], weight, bias, out=outs[i % 2], operand="f16"))
    rec["f16_nchw_packed"] = {"ms_per_call": ms, "images_per_s": B / ms * 1e3, "tflops": flops / ms / 1e9,
                              "frac_of_tensor_peak": flops / ms / 1e9 / bf16_peak, "peak_tflops": bf16_peak}
    cl = [f.half().contiguous(memory_format=torch.channels_last) for f in feats]
    ms = timed(lambda i: parser.parse_features(cl[i % 3], weight, bias, out=outs[i % 2], operand="f16"))
    rec["f16_channels_last_in_place"] = {"ms_per_call": ms, "images_per_s": B / ms * 1e3, "tflops": flops / ms / 1e9,
                                         "frac_of_tensor_peak": flops / ms / 1e9 / bf16_peak, "peak_tflops": bf16_peak}
    w4 = weight[:, :, None, None].contiguous()
    torch.backends.cudnn.allow_tf32 = True
    ms = timed(lambda i: torch.nn.functional.conv2d(feats[i % 3], w4, bias))
    rec["cudnn_conv_tf32_alone_ms"] = ms
    head = torch.sigmoid(torch.nn.functional.conv2d(feats[0], w4, bias))
    ms = timed(lambda i: parser.parse(torch.sigmoid(torch.nn.functional.conv2d(feats[i % 3], w4, bias)), out=outs[i % 2]))
    rec["cudnn_conv_sigmoid_then_ppn_parse_ms"] = ms
    rec["humans_per_image"] = float(parser.parse(head, out=outs[0]).count.float().mean())
    del feats, cl, outs, head, parser
    torch.cuda.empty_cache()
    return rec


def measure_compat(torch, dev, calls=20):
    """Wall time of the reference-signature call (datatest.get_humans_by_feature: numpy arrays in, lists of dicts out)
    at the reference's native shape — what rt_test.py:109-133 costs per frame with the drop-in."""
    import numpy as np
    from pytorch_pose_proposal_network_b200 import datatest as D
    from pytorch_pose_proposal_network_b200.config import PPNConfig
    cfg = PPNConfig.reference_native()
    rng = np.random.default_rng(7)
    K, E, H, W, sH, sW = cfg.K, cfg.E, cfg.H, cfg.W, cfg.sH, cfg.sW
    resp, conf = rng.random((K, H, W), dtype=np.float32), rng.random((K, H, W), dtype=np.float32)
    x, y, w, h = (rng.random((K, H, W), dtype=np.float32) for _ in range(4))
    e = rng.random((E, sH, sW, H, W), dtype=np.float32)
    delta = resp * conf
    for _ in range(3):
        humans, _ = D.get_humans_by_feature(delta, x, y, w, h, e, detection_thresh=0.15)
    ts = []
    for _ in range(calls):
        t0 = time.perf_counter()
        humans, scores = D.get_humans_by_feature(delta, x, y, w, h, e, detection_thresh=0.15)
        ts.append((time.perf_counter() - t0) * 1e3)
    return {"api": "datatest.get_humans_by_feature(numpy [K,H,W] x5, [E,sH,sW,H,W]) -> (humans, scores) dicts",
            "shape": "native: K=18, 24x24 grid, 21x21 window (17.5 MB per call, pageable host arrays)",
            "ms_per_call_median": statistics.median(ts), "ms_per_call_min": min(ts), "calls": calls,
            "humans": len(humans), "reference_cpu_ms_per_call": 7.8,
            "note": "reference figure: SURVEY §6 probe of the unmodified datatest.get_humans_by_feature on one host core"}


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from pytorch_pose_proposal_network_b200 import _lib
    from pytorch_pose_proposal_network_b200.parser import PoseParser
    from pytorch_pose_proposal_network_b200.sharded import PeerPoseGatherer, PoseGatherer, shard_range

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    cfg = preset_of(args.config)
    B = args.batch or BATCH[args.config]
    K, W = args.steps, max(args.warmup, 3)
    job = args.config == "cfg5"
    for kv in args.tune:
        k, v = kv.split("=")
        _lib.tune(**{k.replace(".", "_"): int(v)})

    parser = PoseParser(cfg, device=dev, max_humans=args.max_humans or None)
    per_image = args.gather_entries or 6 * cfg.K   # (human, part) entries per image the gather buffers hold on average (overflow is checked)
    cap_entries = B * per_image

    # ---- inputs --------------------------------------------------------------------------------
    head_dtype = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}[args.head_dtype]
    elem = 4 if args.head_dtype == "f32" else 2
    batch_bytes = B * cfg.C * cfg.HW * elem
    if job:
        # the job's images in global order are chunks 0..15 of 512, chunk c generated from seed 9000 + c wherever it is
        # parsed, so that every GPU count parses the same 8 192 images; rank r owns a contiguous block of chunks
        lo, hi = shard_range(CFG5_IMAGES, world, rank)
        assert lo % B == 0 and (hi - lo) % B == 0, "cfg5 shards must be whole chunks"
        chunk_ids = list(range(lo // B, hi // B))
        bufs = [make_batches(torch, cfg, B, "U", dev, head_dtype, 1, seed=9000 + c)[0] for c in chunk_ids]
        n_buf = len(bufs)
        steps_per_pass = n_buf
    else:
        n_buf = max(2, min(6, -(-(1 << 30) // batch_bytes)))
        bufs = make_batches(torch, cfg, B, DIST[args.config], dev, head_dtype, n_buf, seed=1000 + rank)
        steps_per_pass = 1
    outs = [parser.alloc_output(B) for _ in range(2)]

    # ---- the pose gather (N > 1) ------------------------------------------------------------------
    def make_gatherer(kind):
        if world == 1 or kind == "none":
            return None
        if kind == "nccl":                      # one async all_gather per group of steps; the group sized from the run
            return PoseGatherer(parser, B, cap_entries, group_steps=max(1, min(args.gather_every, (K * steps_per_pass) // 4 or 1)))
        return PeerPoseGatherer(parser, B, cap_entries, slots=args.gather_slots, notify_every=args.notify_every,
                                mode="store" if kind == "peer_store" else "copy", control=args.gather_control)
    gatherer = make_gatherer(args.gather)

    def make_step(g):
        def step(i):
            # the inputs have been resident in HBM since before the timed region: the parser may overlap
            # consecutive steps (PPN_FLAG_INPUT_COMPLETE); results still complete in step order
            if g is not None:                   # poses leave as dense records written by the parse kernel itself
                return g.parse(bufs[i % n_buf], out=outs[i % 2], input_complete=not args.no_step_overlap)
            return parser.parse(bufs[i % n_buf], out=outs[i % 2], input_complete=not args.no_step_overlap)
        return step
    step = make_step(gatherer)

    def drain(g=None):
        g = gatherer if g is None else g
        if g is not None:
            g.finish()

    align = torch.zeros(1, device=dev)

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)
            dist.all_reduce(align)              # stream-ordered: the ranks' device timelines start together (host skew
                                                # after a barrier is tens of microseconds, a third of a step here)

    n_steps = K * steps_per_pass                # kernel-level steps in the timed region

    def timed_region(step_fn, drain_fn):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        t0 = time.perf_counter()
        ev0.record()
        last = None
        for i in range(n_steps):
            last = step_fn(i)
        drain_fn()                              # the timed region ends when every rank's poses have landed at rank 0
        ev1.record()
        host_ms = (time.perf_counter() - t0) * 1e3 / n_steps
        torch.cuda.synchronize(dev)
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            tm = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            ms = float(tm.item())
        return ms, host_ms, last, t0

    sampler = ClockSampler(local_rank).start()
    # warm-up: W steps, then keep the GPU under the same load for ~0.4 s so that the clock
    # sampler sees loaded clocks even when the timed region is only milliseconds long
    t_w = time.perf_counter()
    for i in range(W * steps_per_pass):
        step(i)
    drain()
    torch.cuda.synchronize(dev)
    # the number of extra steps must be the SAME on every rank (each submits collectives): rank 0
    # sizes it from its own warm-up time and broadcasts it
    per_step = max((time.perf_counter() - t_w) / (W * steps_per_pass), 1e-5)
    n_extra = torch.tensor([min(20000, int(args.settle_s / per_step) + 1)], device=dev, dtype=torch.int64)
    if world > 1:
        dist.broadcast(n_extra, src=0)
    extra = int(n_extra.item())
    for i in range(extra):
        step(i)
    drain()
    torch.cuda.synchronize(dev)

    # optional: replay the steps from a CUDA graph (one graph = `group` consecutive steps, so that the
    # rotation of input and output buffers is part of it); the remainder of K runs eagerly
    graph, group = None, 0
    if args.cuda_graph and world == 1 and not job:
        group = 2 * n_buf                           # a multiple of both rotations
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=side):
                for i in range(group):
                    step(i)
        torch.cuda.current_stream(dev).wait_stream(side)
        for _ in range(3):
            graph.replay()
        torch.cuda.synchronize(dev)

    if graph is not None:
        def graph_steps(i):
            if i % group == 0 and i + group <= n_steps:
                graph.replay()
                return None
            return step(i) if i >= n_steps - n_steps % group else None
        elapsed_ms, host_issue_ms, last, t0 = timed_region(graph_steps, drain)
        last = outs[(n_steps - 1) % 2] if last is None else last
    else:
        elapsed_ms, host_issue_ms, last, t0 = timed_region(step, drain)
    if args.dump_outputs:
        dump_outputs(last, args.dump_outputs)

    # Spread of the measurement (SURVEY §8d asks for median and min): the same region four more times.
    # `value` stays the FIRST region's (exactly K steps after the warm-up); these are reported beside it.
    repeat_ms = [elapsed_ms / n_steps]
    if graph is None:
        for _ in range(4):
            r_ms, _, _, _ = timed_region(step, drain)
            repeat_ms.append(r_ms / n_steps)
    t1 = time.perf_counter()
    total_images = images_per_step(args, world) * K
    value = total_images / (elapsed_ms * 1e-3)

    # ---- what was produced (outside the timed region) ---------------------------------------------
    counts = last.count.cpu()
    humans_per_image = float(counts.float().mean())
    gather_note, pose_checksum = "none (1 GPU)", None
    if gatherer is not None:
        if isinstance(gatherer, PeerPoseGatherer):
            if rank == 0:
                tot = 0
                for r in range(world):
                    rec = gatherer.records_of(r)
                    if rec["overflow"]:
                        raise SystemExit(f"bench.py: rank {r} produced more pose entries than the {cap_entries} its slot holds; raise --gather-entries")
                    if r == 0:
                        assert int(rec["count"].sum()) == int(counts.sum()), "gathered humans differ from the local result"
                    tot += int(rec["total"])
                gather_note = (f"{args.gather}: every step's dense (human, part) records "
                               + ("are stored by the parse kernel straight into rank 0's peer-mapped buffer over NVLink (exactly the bytes produced, "
                                  if args.gather == "peer_store" else
                                  f"go to a local slot; one cudaMemcpyAsync (copy engine) per {args.notify_every} steps ships them to rank 0 (slot capacity, ")
                               + f"{tot / world * 24 / 1e6:.2f} MB per rank and step); "
                               + ("'landed' = a 64-bit counter per rank in rank 0's buffer, stored (release.sys) behind every "
                                  f"{args.notify_every} steps and at the end; rank 0's stream waits for all of them inside the timed region — no collective"
                                  if args.gather_control == "flags" else
                                  f"NCCL: one 8-byte all_gather of step counters per {args.notify_every} "
                                  "steps + one at the end of the timed region ('landed' notification)"))
                gatherer.check_landed()
        else:
            for r in range(world):
                rec = gatherer.records_of(r)
                if rec["overflow"]:
                    raise SystemExit(f"bench.py: rank {r} produced {rec['total']} pose entries, more than the {cap_entries} shipped per step")
            mine = gatherer.records_of(rank)
            assert int(mine["count"].sum()) == int(counts.sum()), "gathered humans differ from the local result"
            gather_note = (f"nccl: dense records written by the parse kernel; one async all_gather per {gatherer.gs} steps "
                           f"({gatherer.gs * gatherer.nbytes / 1e6:.2f} MB per rank), overlapped with the following steps")

    # ---- cfg5: checksum of the whole job's poses as rank 0 holds them --------------------------------
    if job:
        pose_checksum = job_checksum(torch, dist, args, parser, gatherer, bufs, outs, B, world, rank, dev)

    # ---- alternatives of the gather, same K steps each (N > 1) ---------------------------------------
    gather_variants = None
    if world > 1 and not args.no_gather_compare:
        gather_variants = {args.gather: {"ms_per_step": elapsed_ms / n_steps, "min_ms_per_step": min(repeat_ms)}}
        for kind in ("peer_store", "peer_copy", "nccl", "none"):
            if kind == args.gather:
                continue
            g2 = make_gatherer(kind)
            s2 = make_step(g2)
            d2 = (lambda g=g2: drain(g)) if g2 is not None else (lambda: None)
            for i in range(3 * steps_per_pass):
                s2(i)
            d2()
            runs = [timed_region(s2, d2)[0] / n_steps for _ in range(3)]
            gather_variants[kind] = {"ms_per_step": runs[0], "min_ms_per_step": min(runs)}
            if isinstance(g2, PeerPoseGatherer):
                g2.close()
        gather_variants["note"] = ("the timed region (K steps + drain, max over ranks) run with each way of gathering the poses; "
                                   "'none' = no gather at all (the floor); first region after 3 warm-up steps, and the best of 3")

    # ---- per-kernel durations ---------------------------------------------------------------------
    # The same steps again with the library recording CUDA events around every kernel on its stream
    # (ppn_profile_*).  Bracketing a kernel with events forbids the overlapped launch chain the timed
    # region uses, so this pass runs the kernels back to back; its step time is NOT the headline value.
    plain = make_step(None)
    _lib.profile_enable(True)
    Kp = min(n_steps, 4096)
    profiled_ms_per_step = timed_loop(torch, dev, plain, Kp)
    stage_ms, n_prof = _lib.profile_read()
    _lib.profile_enable(False)
    # the arg-max kernel alone, K launches back to back (no events in between, no parse kernel beside it): its
    # steady-state launch time, i.e. without the ramp-up and tail an isolated launch pays
    plan = parser.parse_plan(B)
    parser.limb_argmax_into(bufs[0])                 # (allocates the map it writes: not inside a timed loop)
    parser.limb_stream_probe(bufs[0])
    k3_stream_ms = timed_loop(torch, dev, lambda i: parser.limb_argmax_into(bufs[i % n_buf]), n_steps)
    # the read ceiling of the same bulk-copy ring on this GPU: same bytes, no compares, nothing written —
    # with all of shared memory, and capped as ppn_parse caps it to leave room for the parse CTAs
    probe_ms = timed_loop(torch, dev, lambda i: parser.limb_stream_probe(bufs[i % n_buf]), n_steps)
    probe_cap_ms = (timed_loop(torch, dev, lambda i: parser.limb_stream_probe(bufs[i % n_buf], plan["ring_cap"]), n_steps)
                    if plan["ring_cap"] else probe_ms)
    clocks = sampler.summary(t0, t1)

    # ---- end to end through the public host-buffer call: H2D + kernels + D2H every step ------------
    host_in = torch.empty(B, cfg.C, cfg.H, cfg.W, dtype=head_dtype, pin_memory=True)
    host_in.copy_(bufs[0])
    host_out = parser.alloc_output(B, device="cpu", pin=True)
    Ke = max(1, min(K, args.e2e_steps))
    for _ in range(2):
        parser.parse_host(host_in, out=host_out)
    sync_all()
    te0 = time.perf_counter()
    for _ in range(Ke):
        parser.parse_host(host_in, out=host_out)      # synchronous: returns with results on the host
    torch.cuda.synchronize(dev)
    e2e_s = time.perf_counter() - te0
    # the host-memory ceiling of that call on this box: the same pinned batch copied to the device, nothing else
    stage = torch.empty_like(bufs[0])
    sync_all()
    th0 = time.perf_counter()
    for _ in range(Ke):
        stage.copy_(host_in, non_blocking=True)
    torch.cuda.synchronize(dev)
    h2d_s = time.perf_counter() - th0
    del stage
    if world > 1:
        tmax = torch.tensor([e2e_s, h2d_s], device=dev, dtype=torch.float64)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        e2e_s, h2d_s = float(tmax[0].item()), float(tmax[1].item())
    m_slots = int(min(int(host_out.count.max()), parser.R))
    d2h = B * 4 + B * m_slots * (4 + cfg.K * 24)
    e2e = {"value": world * B * Ke / e2e_s, "unit": "images/s", "h2d_bytes_per_step": batch_bytes,
           "d2h_bytes_per_step": d2h, "steps": Ke, "api": "PoseParser.parse_host -> ppn_parse_host (pinned host buffers)",
           "d2h": f"counts, then the first {m_slots} of {parser.R} slots per image (the largest count in the batch)",
           "h2d_gbs_per_rank": batch_bytes * Ke / e2e_s / 1e9,
           "h2d_only_gbs_per_rank": batch_bytes * Ke / h2d_s / 1e9,
           "h2d_only_note": "the same pinned batch copied host->device with nothing else running, all ranks at once (max over ranks): "
                            "the host-memory / PCIe ceiling of the end-to-end call on this box"}
    sampler.stop()

    # ---- roofline of the dominant kernel (limb arg-max) -----------------------------------------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    else:
        peak, peak_src = 6650.0, "B200_PROFILING.md fallback (of fallback)"
    limb_bytes = B * cfg.E * cfg.S * cfg.HW * elem + B * cfg.E * cfg.HW * 2    # read once + uint16 map written
    traffic = None                                   # DRAM bytes per launch from the committed ncu capture
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        rec = json.load(open(tpath)).get(PRESET.get(args.config, args.config))
        if rec and rec.get("images") == B and args.head_dtype == "f32":
            traffic = rec["dram_bytes_read"] + rec["dram_bytes_write"]
    k3_iso_ms = stage_ms["limb_argmax"] / max(n_prof, 1)
    gbs = lambda nbytes, ms: nbytes / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
    achieved = gbs(limb_bytes, k3_stream_ms)
    step_ms = elapsed_ms / n_steps
    read_peak = gbs(limb_bytes, probe_ms)
    two_kernel = plan["launches"] == 2 * plan["sub_batches"]
    roofline = {"bound": "hbm", "kernel": "limb_argmax", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": limb_bytes, "avg_launch_ms": k3_stream_ms,
                "timing": f"the dominant kernel launched {n_steps} times back to back over the rotating inputs on the launching stream, one "
                          "pair of CUDA events around all launches: its average launch duration over a timed region.  (Events BETWEEN "
                          "launches forbid the programmatic overlap of consecutive launches that the product path uses; that figure is "
                          "isolated_launch_ms.)",
                # one launch between two events (the library brackets every kernel of a step: ppn_profile_*): plus the ramp-up
                # and the half-empty last wave of a launch on an idle GPU, which the call chain hides
                "isolated_launch_ms": k3_iso_ms, "isolated_gbs": gbs(limb_bytes, k3_iso_ms), "isolated_frac": gbs(limb_bytes, k3_iso_ms) / peak,
                "isolated_note": f"CUDA events around each kernel on its stream, {n_prof} steps run right after the timed region with the "
                                 "kernels back to back instead of overlapped",
                "stage_ms_per_step": ({"limb_argmax": k3_iso_ms, "parse_fused": stage_ms["tree_parse"] / max(n_prof, 1)} if two_kernel else
                                      {"limb_argmax": k3_iso_ms, "decode_nms": stage_ms["nms"] / max(n_prof, 1),
                                       "tree_parse": stage_ms["tree_parse"] / max(n_prof, 1)}),
                "serial_ms_per_step": profiled_ms_per_step,
                # the read-only ceiling of this ring on this GPU (a copy is half writes; this path is 99 % reads)
                "read_peak_gbs": read_peak, "read_peak_capped_gbs": gbs(limb_bytes, probe_cap_ms), "ring_cap_bytes": plan["ring_cap"],
                "frac_of_read_peak": achieved / read_peak if read_peak else None,
                "read_peak_note": "ppn_limb_stream_probe: the same bulk-copy ring moving the same bytes through shared memory without "
                                  "compares or stores, launched back to back like avg_launch_ms; 'capped' = ring limited to the "
                                  "shared memory ppn_parse leaves it beside the parse CTAs",
                "pipeline_gbs": gbs(batch_bytes, step_ms), "pipeline_frac": gbs(batch_bytes, step_ms) / peak,
                "pipeline_frac_of_read_peak": gbs(batch_bytes, step_ms) / read_peak if read_peak else None}

    # kernels of the library launched in the timed region besides the parse kernels: the peer gather's landing counters
    # (one one-thread store kernel per `notify_every` steps and at the end; on rank 0 one polling warp at the end)
    gather_launches = 0
    if isinstance(gatherer, PeerPoseGatherer) and gatherer.control == "flags":
        gather_launches = -(-n_steps // gatherer.ne) + (1 if rank == gatherer.root else 0)
    line = {
        "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": elapsed_ms / K, "higher_is_better": True, "scaling": "strong" if job else "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD[args.config], "preset": args.config, "images_per_gpu_per_step": B,
                   "K": cfg.K, "E": cfg.E, "grid": [cfg.H, cfg.W], "window": [cfg.sH, cfg.sW],
                   "bytes_per_image": cfg.C * cfg.HW * elem, "head_dtype": args.head_dtype,
                   "input_distribution": DIST[args.config],
                   "l2": (f"{n_buf} distinct input batches of {batch_bytes / 1e6:.0f} MB rotated (each larger than L2)" if not job else
                          f"every image is read once per pass: {n_buf} chunks of {batch_bytes / 1e6:.0f} MB per rank"),
                   "humans_per_image": humans_per_image, "extra_warmup_steps": extra,
                   "warmup_note": f"{W} warm-up steps as asked, then {extra} more (~{args.settle_s} s) so that the clock sampler sees the "
                                  "GPU under load before a timed region of a few milliseconds",
                   "host_issue_ms_per_step": host_issue_ms, "cuda_graph": bool(graph is not None),
                   "step_overlap": "off" if args.no_step_overlap else
                   "PPN_FLAG_INPUT_COMPLETE: inputs resident before the timed region, so step i+1's arg-max may start while "
                   "step i's tree parse finishes; steps complete in order",
                   "pose_gather": gather_note},
        "roofline": roofline, "e2e": e2e, "clocks": clocks,
        "gpu_launches": plan["launches"] * n_steps + gather_launches,
        "repeats": {"ms_per_step": repeat_ms, "median_ms_per_step": sorted(repeat_ms)[len(repeat_ms) // 2],
                    "min_ms_per_step": min(repeat_ms), "note": "the timed region run five times; `value` is the first"},
    }
    if job:
        line["config"]["job"] = {"images": CFG5_IMAGES, "chunk_images": B, "chunks_per_rank": n_buf, "passes": K,
                                 "pose_checksum": pose_checksum,
                                 "checksum_note": "sha256 over the job's poses in global image order as rank 0 holds them after the "
                                                  "gather; the same string for every GPU count = sharded result == single-GPU result"}
        line["ms_per_step"] = elapsed_ms / K
    if gather_variants is not None:
        line["config"]["gather_variants"] = gather_variants

    if isinstance(gatherer, PeerPoseGatherer):
        gatherer.close()
    del bufs, outs
    torch.cuda.empty_cache()
    if rank == 0 and world == 1 and not args.no_other_configs and not job:
        others = {}
        for name in ("cfg1", "cfg3", "cfg4", "native"):
            if name == args.config:
                continue
            rec = measure_other_config(torch, name, dev)
            rec["pipeline_frac"] = rec["gbs"] / peak
            others[name] = rec
        others["note"] = ("the other BASELINE.json configurations on this GPU, 30 timed steps each after 5 warm-up steps, inputs resident; "
                          "pipeline_frac = whole head tensor / step time / the measured copy peak; cfg1 is one image per call: a latency")
        line["other_configs"] = others
        line["compat_e2e"] = measure_compat(torch, dev)
        if args.config == "cfg2" and args.head_dtype == "f32":
            line["fused_head"] = measure_fused_head(torch, dev, json.load(open(peaks_path)) if os.path.exists(peaks_path) else {})
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(cfg, args)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def job_checksum(torch, dist, args, parser, gatherer, bufs, outs, B, world, rank, dev):
    """cfg5: one more pass over this rank's chunks with the gather, then rank 0 hashes all ranks' records in global
    image order (count, then per human its (part, cell, score bits, box bits) entries)."""
    import hashlib
    import numpy as np
    from pytorch_pose_proposal_network_b200.parser import entries_to_packed, unpack_entries
    from pytorch_pose_proposal_network_b200.sharded import PeerPoseGatherer
    n_chunks = len(bufs)
    h = hashlib.sha256()
    if world == 1:
        cap = B * (args.gather_entries or 6 * parser.cfg.K)
        nbytes, offs = parser.packed_layout(B, cap)
        dense = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
        recs = []
        for c in range(n_chunks):
            parser.parse(bufs[c], out=outs[0], dense=dense, cap_entries=cap)
            torch.cuda.synchronize(dev)
            recs.append(unpack_entries(dense.cpu(), B, cap, offs))
        per_rank = [recs]
    else:
        if not isinstance(gatherer, PeerPoseGatherer):
            return None
        if n_chunks > gatherer.slots - 2 * gatherer.ne:
            return None                                   # the ring would wrap inside one pass
        for c in range(n_chunks):
            gatherer.parse(bufs[c], out=outs[c % 2])
        gatherer.finish()
        torch.cuda.synchronize(dev)
        dist.barrier()
        if rank != 0:
            return None
        per_rank = [[gatherer.records_of(r, step_back=n_chunks - 1 - c) for c in range(n_chunks)] for r in range(world)]
    for recs in per_rank:
        for rec in recs:
            assert not rec["overflow"], "pose records overflowed their slot"
            for b in range(B):
                pc, ps, pb = entries_to_packed(rec, b, parser.cfg.K)
                h.update(np.int32(pc.shape[0]).tobytes())
                h.update(pc.tobytes()); h.update(ps.tobytes()); h.update(pb.tobytes())
    return h.hexdigest()


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(out, directory):
    """Write the PackedHumans of one step as float32 DIR/<name>.npy, so that two builds can be compared output for
    output.  Slots past count[b] keep whatever the buffer held before (the parse does not write them), so they are
    reset to -1 / 0 here as PPN_FLAG_CLEAR_UNUSED would.  `count` covers the whole batch; the per-slot arrays cover
    every image, or a fixed seeded sample of images (listed in images.npy) when the whole batch exceeds DUMP_BYTES."""
    import numpy as np
    a = out.numpy()
    count = a["count"]
    B, R = a["root_cell"].shape
    used = np.arange(R)[None, :] < count[:, None]
    slots = {"root_cell": np.where(used, a["root_cell"], -1),
             "part_cell": np.where(used[..., None], a["part_cell"], -1),
             "part_score": np.where(used[..., None], a["part_score"], 0),
             "part_box": np.where(used[..., None, None], a["part_box"], 0)}
    per_image = sum(v[0].size for v in slots.values()) * 4
    n = min(B, (DUMP_BYTES - 8 * B - 4096) // per_image)      # count and images are 4 bytes an image; 4096 for headers
    images = np.arange(B) if n == B else np.sort(np.random.default_rng(0).choice(B, n, replace=False))
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "count.npy"), count.astype(np.float32))
    np.save(os.path.join(directory, "images.npy"), images.astype(np.float32))
    for name, v in slots.items():
        np.save(os.path.join(directory, f"{name}.npy"), v[images].astype(np.float32))


def cpu_baseline(cfg, args):
    """The reference-shaped numpy port on all host cores, bounded to ~args.cpu_budget_s seconds."""
    from oracle import cpu_bench, ppn_oracle as O
    g = O.Geometry.of(cfg)
    cores = cpu_bench.host_cores()
    dist = DIST[args.config]
    one_core_ips, one_core_ms, n1 = cpu_bench.time_single_core(g, dist, seed=0, n_images=16, budget_s=min(4.0, args.cpu_budget_s / 3))
    per_pass = max(4 * cores, 16)
    pool = cpu_bench.CpuPool(g, dist=dist, seed=0, n_images=per_pass, cores=cores)
    try:
        pool.one_pass()
        n, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < args.cpu_budget_s * 0.6:
            pool.one_pass()
            n += per_pass
        dt = time.perf_counter() - t0
    finally:
        pool.close()
    c_ips = cpu_bench.time_c_port(g, dist, seed=0, n_images=max(2 * cores, 16), threads=cores, budget_s=min(3.0, args.cpu_budget_s / 4))
    return {"value": n / dt, "unit": "images/s", "cores": cores, "kind": "port",
            "sample": f"{n} images ({per_pass}-image synthetic sample, dist {dist}, repeated for {dt:.1f} s) through the numpy port "
                      f"of datatest.get_humans_by_feature, one process per core",
            "one_core_images_per_s": one_core_ips, "one_core_ms_per_image": one_core_ms,
            "c_port_images_per_s": c_ips, "c_port_threads": cores,
            "c_port_note": "the C restatement (oracle/ppn_oracle.c, pthreads) on the same cores: what a compiled CPU implementation "
                           "of the same algorithm does; the end-to-end advantage over it is e2e.value / c_port_images_per_s"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(BATCH))
    ap.add_argument("--batch", type=int, default=0, help="images per GPU per step (default: the config's)")
    ap.add_argument("--max-humans", type=int, default=0, help="slots per image in the packed output (default H*W)")
    ap.add_argument("--gather", default="peer_store", choices=["peer_store", "peer_copy", "nccl", "none"],
                    help="how the poses of N > 1 GPUs reach rank 0 (see sharded.py)")
    ap.add_argument("--gather-control", default="flags", choices=["flags", "nccl"],
                    help="peer gather: how rank 0 learns that the records have landed (counters in its buffer, or an 8-byte NCCL all_gather)")
    ap.add_argument("--gather-entries", type=int, default=0,
                    help="average (human, part) entries per image a gather slot holds (default 6*K; overflow is detected)")
    ap.add_argument("--gather-every", type=int, default=32, help="--gather nccl: steps per all_gather (at most a quarter of the run)")
    ap.add_argument("--gather-slots", type=int, default=32, help="peer gather: slots of the ring at rank 0 per rank")
    ap.add_argument("--notify-every", type=int, default=8, help="peer gather: steps per 'landed' notification")
    ap.add_argument("--no-gather-compare", action="store_true", help="N > 1: do not also time the other gather variants")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--settle-s", type=float, default=0.4)
    ap.add_argument("--cpu-budget-s", type=float, default=15.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the compact records of the other BASELINE configs")
    ap.add_argument("--head-dtype", default="f32", choices=["f32", "f16", "bf16"],
                    help="element type of the head tensor (the reference's is f32; the arithmetic is fp32 either way)")
    ap.add_argument("--cuda-graph", action="store_true", help="replay the timed steps from a CUDA graph (1 GPU)")
    ap.add_argument("--no-step-overlap", action="store_true",
                    help="do not pass PPN_FLAG_INPUT_COMPLETE (each step's kernels wait for the previous step's)")
    ap.add_argument("--tune", action="append", default=[], help="library knob, e.g. argmax.stages=6")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the poses of the last one as DIR/<name>.npy (float32, at most 64 MB; "
                         "one GPU, --impl ours)")
    args = ap.parse_args()
    if args.config == "cfg5" and "--steps" not in " ".join(sys.argv):
        args.steps = 10                         # passes over the 8 192-image job
    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if args.dump_outputs and (args.impl == "reference" or world > 1):
        # with N > 1 the parse leaves the fixed-stride arrays unwritten and the poses exist only as gathered records
        ap.error("--dump-outputs writes the one-GPU result of --impl ours")
    if args.impl == "reference":
        return run_reference(args, rank, world)
    return run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    sys.exit(main())
