"""The flip test's merge (FlipMerge / ppn_flip_merge) on seeded synthetic heads, beside a copy and a torch composite.

    python scripts/bench_flip.py [--calls 20] [--out profiles/bench_flip.txt]

Per workload (preset, batch, head dtype); every head is larger than the 126 MB L2, so each call streams from HBM:
  * merge: device time per call, CUDA events around each call, median of --calls calls after a warm-up;
  * bound: 3 x head bytes (A and Bf read, out written) over 7.7 TB/s: arithmetic, not a measurement;
  * copy: a device-to-device copy_ of a head-sized tensor in the same run (2 x head bytes moved, median), and the
    merge's bytes/s as a fraction of the copy's;
  * torch: the same rule as index_select + flip + arithmetic on the same inputs (median);
  * the merge in front of each parser: merge + parse against parse alone, merge + parse_proposals against
    parse_proposals alone (medians of whole chains).
The merge is checked bit for bit against the torch composite (fp32) or its restatement (16-bit) first.
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import flip_merge as FM, ppn_oracle as O                    # noqa: E402
from pytorch_pose_proposal_network_b200.config import PRESETS           # noqa: E402
from pytorch_pose_proposal_network_b200.flip import FlipMerge           # noqa: E402
from pytorch_pose_proposal_network_b200.parser import PoseParser        # noqa: E402
from tests.gpu_inputs import device_head                                # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--calls", type=int, default=20)
ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "profiles", "bench_flip.txt"))
a = ap.parse_args()
assert torch.cuda.is_available(), "bench_flip measures on the GPU; there is nothing to measure without one"

HBM = 7.7e12
L2 = 126e6
WORKLOADS = [("cfg2", 512, torch.float32), ("cfg2", 512, torch.float16), ("native", 64, torch.float32),
             ("native", 64, torch.bfloat16), ("cfg3", 1024, torch.float32), ("cfg4", 256, torch.float32)]
lines = []


def say(s=""):
    print(s, flush=True)
    lines.append(s)


def median_us(fn, calls):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(calls):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        e.synchronize()
        ts.append(s.elapsed_time(e) * 1e3)
    return float(np.median(ts))


def composite(A, Bf, src, K):
    m = Bf.index_select(1, src).flip(-1)
    m[:, 2 * K:3 * K] = 1 - m[:, 2 * K:3 * K]
    return (A + m) * 0.5


gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()[0]
say(f"# GPU (name, power limit, SM clock, max SM clock): {gpu}")
say(f"# torch {torch.__version__}, CUDA {torch.version.cuda}")
say(f"# device time per call: CUDA events, median of {a.calls} calls after warm-up; every head is larger than the "
    f"126 MB L2")
say("# bound = 3 x head bytes / 7.7 TB/s (arithmetic); copy = head-sized copy_ in the same run, 2 x head bytes moved")
say("# workload                  | head MB | merge us | bound us | copy us (GB/s) | merge / copy rate | torch us | "
    "parse us: alone / +merge | proposals us: alone / +merge")
for preset, B, dt in WORKLOADS:
    cfg = PRESETS[preset]()
    g = O.Geometry.of(cfg)
    A, hostA = device_head(g, "U", 1, B, dtype=dt, distinct=False)
    Bf, hostB = device_head(g, "R", 2, B, dtype=dt, distinct=False)
    fm = FlipMerge(cfg)
    parser = PoseParser(cfg)
    nbytes = A.numel() * A.element_size()
    assert nbytes > L2
    out = torch.empty_like(A)
    fm(A, Bf, out=out)
    src = torch.from_numpy(FM.source_planes(cfg.K, cfg.E, cfg.sH, cfg.sW, fm.part_mirror, fm.limb_mirror)).cuda()
    if dt == torch.float32:
        assert torch.equal(out.view(torch.int32), composite(A, Bf, src, cfg.K).view(torch.int32))
    else:
        name = {torch.float16: "float16", torch.bfloat16: "bfloat16"}[dt]
        n = min(B, 8)
        ref = FM.flip_merge(hostA[:n], hostB[:n], g, fm.part_mirror, fm.limb_mirror, name)
        assert np.array_equal(out[:n].cpu().view(torch.int16).numpy().view(np.uint16), ref.view(np.uint16))
    del hostA, hostB
    t_merge = median_us(lambda: fm(A, Bf, out=out), a.calls)
    dst = torch.empty_like(A)
    t_copy = median_us(lambda: dst.copy_(A), a.calls)
    del dst
    t_torch = median_us(lambda: composite(A, Bf, src, cfg.K), a.calls)
    t_parse = median_us(lambda: parser.parse(A), a.calls)
    t_parse_m = median_us(lambda: parser.parse(fm(A, Bf, out=out)), a.calls)
    t_prop = median_us(lambda: parser.parse_proposals(A), a.calls)
    t_prop_m = median_us(lambda: parser.parse_proposals(fm(A, Bf, out=out)), a.calls)
    bound = 3 * nbytes / HBM * 1e6
    copy_rate = 2 * nbytes / (t_copy * 1e-6)
    merge_rate = 3 * nbytes / (t_merge * 1e-6)
    tag = f"{preset:<6} B={B:<5} {str(dt).replace('torch.', ''):<8}"
    say(f"{tag} | {nbytes / 1e6:7.1f} | {t_merge:8.1f} | {bound:8.1f} | {t_copy:7.1f} ({copy_rate / 1e9:5.0f}) | "
        f"{merge_rate / copy_rate:17.3f} | {t_torch:8.1f} | {t_parse:8.1f} / {t_parse_m:8.1f}   | "
        f"{t_prop:9.1f} / {t_prop_m:9.1f}")
    del A, Bf, out, src
    torch.cuda.empty_cache()

os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
with open(a.out, "w") as f:
    f.write("\n".join(lines) + "\n")
