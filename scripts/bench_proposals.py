"""The proposal-pair parse (PoseParser.parse_proposals) on the BASELINE workloads, beside ppn_parse on the same batch.

    python scripts/bench_proposals.py [--calls 30] [--out profiles/bench_proposals.txt]

Per workload (preset, input distribution, batch):
  * device time per call from CUDA events around --calls back-to-back calls after warm-up, the input alternating
    between two batches (every batch but cfg1's single image is larger than the 126 MB L2); parse_proposals and
    parse are timed in alternating blocks, the median block is reported;
  * the split between the two kernels (decode + NMS of every part, pair scoring + matching) from torch.profiler, in a
    separate run;
  * the C twin of the specification (oracle/proposal_parse.c) on all host cores, one pass over the batch, from a host clock;
  * proposals per part and candidate pairs per limb, counted by the C restatement (mean over images and parts /
    limbs, and the largest per-limb count of any image);
  * the GPU result is checked against the C restatement on every image before anything is timed.
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import c_proposal_parse, ppn_oracle as O                    # noqa: E402
from pytorch_pose_proposal_network_b200.config import PRESETS           # noqa: E402
from pytorch_pose_proposal_network_b200.parser import PoseParser        # noqa: E402
from tests.gpu_inputs import device_head                                # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--calls", type=int, default=30)
ap.add_argument("--blocks", type=int, default=3)
ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "profiles", "bench_proposals.txt"))
a = ap.parse_args()
assert torch.cuda.is_available(), "bench_proposals measures on the GPU; there is nothing to measure without one"

WORKLOADS = [("cfg2", "U", 512), ("cfg2", "R", 512), ("cfg2", "S", 512), ("cfg3", "D", 1024), ("cfg4", "U", 256),
             ("native", "U", 64), ("native", "S", 64), ("cfg1", "U", 1)]
lines = []


def say(s=""):
    print(s, flush=True)
    lines.append(s)


try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
except Exception as ex:
    q = f"{torch.cuda.get_device_name()} (nvidia-smi unavailable: {ex})"
say(f"# GPU (name, power limit, SM clock, max SM clock): {q}")
say(f"# torch {torch.__version__}, CUDA {torch.version.cuda}; C restatement on {os.cpu_count()} host threads")
say(f"# device time per call: median of {a.blocks} blocks of {a.calls} back-to-back calls, two input batches alternating")
say("# workload            props/part  pairs/limb (max)  | proposals us  (nms us + pairs us) | ppn_parse us | C all cores ms")


def timed(fn, heads, calls):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for c in range(calls):
        fn(heads[c & 1])
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) * 1e3 / calls


def kernel_split(parser, head, out, calls=10):
    """us per call of decode+NMS and of the pair kernel, from a profiler run of its own."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            parser.parse_proposals(head, out=out)
        torch.cuda.synchronize()
    tot = {"decode_nms": 0.0, "proposal_pairs": 0.0}
    for ev in prof.key_averages():
        for k in tot:
            if k + "_kernel" in ev.key:
                tot[k] += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
    return tot["decode_nms"] / calls, tot["proposal_pairs"] / calls


for preset, dist, B in WORKLOADS:
    cfg = PRESETS[preset]()
    g = O.Geometry.of(cfg)
    h0, host0 = device_head(g, dist, 100 + B, B, distinct=False)
    h1, _ = device_head(g, dist, 200 + B, B, distinct=False)
    heads = (h0, h1)
    parser = PoseParser(cfg)
    out_p, out_r = parser.alloc_output(B), parser.alloc_output(B)
    got = parser.parse_proposals(h0, out=out_p).numpy()
    t0 = time.perf_counter()
    ref = c_proposal_parse.proposal_parse_batch(host0, g, n_threads=os.cpu_count(), stats=True)
    t_c = (time.perf_counter() - t0) * 1e3
    assert np.array_equal(got["count"], ref["count"]), f"{preset}-{dist}: GPU and C restatement differ"
    for w in range(2):
        for h in heads:
            parser.parse_proposals(h, out=out_p)
            parser.parse(h, out=out_r)
    torch.cuda.synchronize()
    tp, tr = [], []
    for _ in range(a.blocks):
        tp.append(timed(lambda h: parser.parse_proposals(h, out=out_p), heads, a.calls))
        tr.append(timed(lambda h: parser.parse(h, out=out_r), heads, a.calls))
    t_nms, t_pairs = kernel_split(parser, h0, out_p)
    props = ref["n_prop"].mean()
    tree_limbs = sorted({e for eis, _ in g.graphs for e in eis})
    pairs = ref["n_pairs"][:, tree_limbs]
    say(f"{preset:6s} {dist} B={B:<5d}   {props:8.1f}  {pairs.mean():9.0f} ({pairs.max():6d})  | "
        f"{np.median(tp):10.1f}  ({t_nms:8.1f} + {t_pairs:9.1f}) | {np.median(tr):10.1f} | {t_c:10.1f}")
    say(f"#   humans/image {ref['count'].mean():.1f}; per image: proposals {np.median(tp) / B:.2f} us, ppn_parse "
        f"{np.median(tr) / B:.2f} us, C restatement {t_c * 1e3 / B:.1f} us; blocks {['%.1f' % v for v in tp]}")
    del h0, h1, heads, out_p, out_r, parser
    torch.cuda.empty_cache()

os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
with open(a.out, "w") as f:
    f.write("\n".join(lines) + "\n")
print(f"wrote {a.out}")
