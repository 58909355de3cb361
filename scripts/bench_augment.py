"""Batch augmentation (Augmenter.images / ppn_augment_images) on seeded synthetic images, beside two other routes.

    python scripts/bench_augment.py [--calls 20] [--out profiles/bench_augment.txt]

Per workload (output geometry, batch, source sizes, output dtype and layout):
  * device time per batch: CUDA events around each call, the 126 MB L2 flushed (a 256 MB buffer overwritten) before
    every call, median over --calls calls, sampled parameters (scale 0.75-1.25, +-30 deg, +-0.1 shift, flips);
    with the default (every tap gathered through L1) and with the staging budget at 16, 32 and 48 KB;
  * the bytes bound: the whole sources plus the output over 7.7 TB/s (arithmetic, not a measurement), and the same
    with only the source pixels some tap reads;
  * the pinned host-to-device upload of the same batch (one copy, CUDA events, median);
  * torch route: per image affine_grid + grid_sample(align_corners=False) after a float conversion, then the
    normalisation, on the same parameters (device time of the loop over the batch, CUDA events);
  * host route: the numpy restatement (oracle/augment.py) over the batch on all host cores (process pool, wall clock).
Every GPU result is checked against the restatement on a few images first.
"""
import argparse
import multiprocessing as mp
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.nn.functional as Fn

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import augment as OA                                        # noqa: E402
from pytorch_pose_proposal_network_b200 import _lib                     # noqa: E402
from pytorch_pose_proposal_network_b200.augment import Augmenter, ImageBatch   # noqa: E402
from pytorch_pose_proposal_network_b200.config import PRESETS           # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--calls", type=int, default=20)
ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "profiles", "bench_augment.txt"))
a = ap.parse_args()
assert torch.cuda.is_available(), "bench_augment measures on the GPU; there is nothing to measure without one"

HBM = 7.7e12
lines = []


def say(s=""):
    print(s, flush=True)
    lines.append(s)


def sizes_of(kind, B, rng):
    if kind != "mixed":
        w, h = (int(v) for v in kind.split("x"))
        return [(h, w)] * B
    return [(int(h), int(w)) for h, w in zip(rng.integers(240, 1081, B), rng.integers(320, 1921, B))]   # mixed


def median_ms(fn, calls, flush):
    ts = []
    for _ in range(calls):
        flush.zero_()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        e.synchronize()
        ts.append(s.elapsed_time(e))
    return float(np.median(ts))


def tapped_bytes(batch, M, insize):
    """Distinct source pixels some bilinear tap of the output reads, x 3 bytes (restated taps, on the device)."""
    inW, inH = insize
    u = torch.arange(inW, device="cuda", dtype=torch.float32) + 0.5
    v = torch.arange(inH, device="cuda", dtype=torch.float32) + 0.5
    total = 0
    for b in range(batch.B):
        h, w = (int(x) for x in batch.hw_host[b])
        m = M[b]
        sx = (m[0, 0] * u[None, :] + m[0, 1] * v[:, None] + m[0, 2]) - 0.5
        sy = (m[1, 0] * u[None, :] + m[1, 1] * v[:, None] + m[1, 2]) - 0.5
        ix, iy = torch.floor(sx).long(), torch.floor(sy).long()
        seen = torch.zeros(h * w, dtype=torch.bool, device="cuda")
        for dx in (0, 1):
            for dy in (0, 1):
                x, y = ix + dx, iy + dy
                ok = (x >= 0) & (x < w) & (y >= 0) & (y < h)
                seen[(y * w + x)[ok]] = True
        total += int(seen.sum()) * 3
    return total


def torch_route(batch, M, insize, out, mean, std):
    """affine_grid + grid_sample per image on the same parameters: theta = N_src M N_out^-1 (normalised coordinates)."""
    inW, inH = insize
    Md = M.double()
    for b in range(batch.B):
        h, w = (int(x) for x in batch.hw_host[b])
        o = int(batch.offset_host[b])
        img = batch.pixels[o:o + 3 * h * w].view(1, h, w, 3).permute(0, 3, 1, 2).float()
        n_src = torch.tensor([[2.0 / w, 0, -1], [0, 2.0 / h, -1], [0, 0, 1]], dtype=torch.float64, device="cuda")
        n_out_inv = torch.tensor([[inW / 2.0, 0, inW / 2.0], [0, inH / 2.0, inH / 2.0], [0, 0, 1]], dtype=torch.float64, device="cuda")
        full = torch.cat([Md[b], torch.tensor([[0, 0, 1]], dtype=torch.float64, device="cuda")])
        theta = (n_src @ full @ n_out_inv)[:2].float()[None]
        grid = Fn.affine_grid(theta, [1, 3, inH, inW], align_corners=False)
        val = Fn.grid_sample(img, grid, mode="bilinear", padding_mode="zeros", align_corners=False)
        out[b] = (val[0] * (1.0 / 255.0) - mean) / std


def host_one(args):
    img, M, insize = args
    return OA.warp_image(img, M, insize)


try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
except Exception as ex:
    q = f"{torch.cuda.get_device_name()} (nvidia-smi unavailable: {ex})"
say(f"# GPU (name, power limit, SM clock, max SM clock): {q}")
say(f"# torch {torch.__version__}, CUDA {torch.version.cuda}; host route on {os.cpu_count()} host processes")
say(f"# device time per batch: median of {a.calls} calls, L2 flushed (256 MB overwritten) before each; "
    f"bound = bytes / 7.7 TB/s (arithmetic)")
say("# workload                              | kernel us | bound us whole src (tapped) | % of bound | "
    "H2D us (GB/s)    | torch us | host ms")

WORKLOADS = [("native", 64, "1280x720", torch.float32, False), ("native", 64, "1280x720", torch.bfloat16, True),
             ("native", 64, "mixed", torch.float32, False), ("cfg2", 512, "1280x720", torch.float32, False),
             ("cfg2", 512, "1280x720", torch.bfloat16, True), ("native", 64, "320x240", torch.float32, False),
             ("cfg3", 256, "640x480", torch.bfloat16, True)]
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
default_stage = _lib.tune_get("augment.stage_bytes")
pool = mp.get_context("fork").Pool(os.cpu_count())
for preset, B, kind, dtype, cl in WORKLOADS:
    cfg = PRESETS[preset]()
    rng = np.random.default_rng(B)
    imgs = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in sizes_of(kind, B, rng)]
    batch = ImageBatch.from_arrays(imgs)
    aug = Augmenter(cfg, dtype=dtype, channels_last=cl)
    params = aug.sample(batch, torch.Generator(device="cuda").manual_seed(1))
    out = aug.images(batch, params)
    torch.cuda.synchronize()
    M = params.M.cpu().numpy()
    for b in (0, B // 2, B - 1):                                   # the result before any timing
        want = OA.warp_image(imgs[b], M[b], cfg.insize, dtype={torch.float32: "float32", torch.bfloat16: "bfloat16"}[dtype])
        got = out[b].cpu().contiguous()
        got = got.view(torch.int16).numpy().view(np.uint16) if dtype == torch.bfloat16 else got.numpy()
        assert np.array_equal(got.view(np.uint16 if dtype == torch.bfloat16 else np.uint32),
                              want.view(np.uint16 if dtype == torch.bfloat16 else np.uint32)), b
    src_bytes = int(sum(i.nbytes for i in imgs))
    out_bytes = out.numel() * out.element_size()
    tapped = tapped_bytes(batch, params.M, cfg.insize)
    ms = {}
    for stage in (default_stage, 16 * 1024, 32 * 1024, 48 * 1024):
        _lib.tune(augment_stage_bytes=stage)
        aug.images(batch, params, out=out)
        ms[stage] = median_ms(lambda: aug.images(batch, params, out=out), a.calls, flush)
    _lib.tune(augment_stage_bytes=default_stage)
    # the upload: one pinned buffer of the same bytes, one copy
    host = torch.empty(batch.pixels.numel() + 16 * B, dtype=torch.uint8, pin_memory=True)
    dev = torch.empty_like(host, device="cuda")
    h2d = median_ms(lambda: dev.copy_(host, non_blocking=True), a.calls, flush)
    # torch route (fp32 NCHW) on the same parameters
    mean = torch.tensor(OA.IMAGENET_MEAN, device="cuda").view(3, 1, 1)
    std = torch.tensor(OA.IMAGENET_STD, device="cuda").view(3, 1, 1)
    tout = torch.empty(B, 3, cfg.inH, cfg.inW, device="cuda")
    torch_route(batch, params.M, cfg.insize, tout, mean, std)
    tms = median_ms(lambda: torch_route(batch, params.M, cfg.insize, tout, mean, std), max(3, a.calls // 4), flush)
    diff = float((tout - out.float()).abs().max())
    # host route: the restatement over the whole batch on all cores
    t0 = time.perf_counter()
    pool.map(host_one, [(imgs[b], M[b], cfg.insize) for b in range(B)])
    host_ms = (time.perf_counter() - t0) * 1e3
    bound = (src_bytes + out_bytes) / HBM * 1e6
    bound_t = (tapped + out_bytes) / HBM * 1e6
    name = f"{preset:6s} B={B:<4d} {kind:8s} {str(dtype)[6:]:8s} {'NHWC' if cl else 'NCHW'}"
    say(f"{name:38s}  | {ms[default_stage] * 1e3:9.1f} | {bound:8.1f} ({bound_t:8.1f})        | "
        f"{100 * bound / (ms[default_stage] * 1e3):5.1f}      | {h2d * 1e3:7.1f} ({src_bytes / (h2d * 1e-3) / 1e9:5.1f}) | "
        f"{tms * 1e3:8.1f} | {host_ms:8.1f}")
    say(f"#   source {src_bytes / 1e6:.1f} MB (tapped {tapped / 1e6:.1f} MB), output {out_bytes / 1e6:.1f} MB; torch route "
        f"max |diff| {diff:.3g} vs the kernel; kernel us with a 16 / 32 / 48 KB staging "
        f"budget: {ms[16 * 1024] * 1e3:.1f} / {ms[32 * 1024] * 1e3:.1f} / {ms[48 * 1024] * 1e3:.1f}")
pool.close()
pool.join()
os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
with open(a.out, "w") as f:
    f.write("\n".join(lines) + "\n")
