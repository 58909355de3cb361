"""Throughput of the GPU target encoder (ppn_encode_targets) next to the CPU restatement of dataset.py:98-185.

    python scripts/bench_encode.py [--config cfg2] [--batch 512] [--people 4] [--limb-dtype float16] > encode.txt

--limb-dtype float16 / bfloat16 writes te and weight_ij in 16 bits (TargetEncoder(cfg, limb_dtype=...)); bytes are
counted with their element size.
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import encode_gt  # noqa: E402  (CPU baseline only)
from pytorch_pose_proposal_network_b200 import config as pcfg  # noqa: E402
from pytorch_pose_proposal_network_b200.config import PRESETS  # noqa: E402
from pytorch_pose_proposal_network_b200.dataset import TargetEncoder, flatten_samples  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--config", default="cfg2")
ap.add_argument("--batch", type=int, default=512)
ap.add_argument("--people", type=int, default=4)
ap.add_argument("--iters", type=int, default=50)
ap.add_argument("--sweep", type=int, default=1)
ap.add_argument("--ctas", type=int, default=6)
ap.add_argument("--limb-dtype", default="float32", choices=("float32", "float16", "bfloat16"))
a = ap.parse_args()
cfg = PRESETS[a.config]()
K, B = cfg.K, a.batch
rng = np.random.default_rng(0)
raw = [encode_gt.random_people(rng, a.people, K, cfg.insize) for _ in range(B)]
samples = [dict(keypoints=kp, bbox=bb, is_visible=vis, size=size) for kp, bb, vis, size in raw]
from pytorch_pose_proposal_network_b200 import _lib  # noqa: E402
_lib.tune(encode_sweep=a.sweep, encode_ctas_per_sm=a.ctas)
limb_dtype = getattr(torch, a.limb_dtype)
limb_bytes = torch.empty(0, dtype=limb_dtype).element_size()
enc = TargetEncoder(cfg, limb_dtype=limb_dtype)
flat = [torch.from_numpy(x).cuda() for x in flatten_samples(samples, K)]
outs = [enc.alloc(B) for _ in range(3)]                       # rotate: each set is larger than L2 at the default size
for o in outs:
    enc.encode_flat(*flat, out=o)
torch.cuda.synchronize()
ev = [torch.cuda.Event(enable_timing=True) for _ in range(a.iters + 1)]
ev[0].record()
for i in range(a.iters):
    enc.encode_flat(*flat, out=outs[i % 3])
    ev[i + 1].record()
torch.cuda.synchronize()
ts = sorted(ev[i].elapsed_time(ev[i + 1]) for i in range(a.iters))
med = ts[len(ts) // 2]
# plain fills of the two big tensors, for scale: what writing these bytes costs without any logic
evf = [torch.cuda.Event(enable_timing=True) for _ in range(a.iters + 1)]
evf[0].record()
for i in range(a.iters):
    outs[i % 3].te.zero_()
    outs[i % 3].weight_ij.fill_(0.0005)
    evf[i + 1].record()
torch.cuda.synchronize()
fill_ms = sorted(evf[i].elapsed_time(evf[i + 1]) for i in range(a.iters))[a.iters // 2]
bytes_out = B * (2 * cfg.E * cfg.S * cfg.HW * limb_bytes + 8 * cfg.K * cfg.HW * 4)
peak = 6553.0
p = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")
if os.path.exists(p):
    peak = float(json.load(open(p))["hbm_gbs"])
edges = pcfg.EDGES if K == 18 else pcfg.EDGES_16
n_cpu = min(B, 24)
t0 = time.perf_counter()
for kp, bb, vis, size in raw[:n_cpu]:
    encode_gt.encode_targets(kp, bb, vis, size, K, edges, cfg.insize, cfg.outsize, cfg.local_grid_size)
cpu_ms = (time.perf_counter() - t0) * 1e3 / n_cpu
print(json.dumps({"op": "ppn_encode_targets", "config": a.config, "images": B, "people_per_image": a.people, "sweep": a.sweep, "ctas_per_sm": a.ctas,
                  "limb_dtype": a.limb_dtype,
                  "ms_per_batch": med, "images_per_s": B / (med * 1e-3), "bytes_written": bytes_out,
                  "achieved_gbs": bytes_out / (med * 1e-3) / 1e9, "peak_gbs": peak, "torch_fill_of_the_two_limb_tensors_ms": fill_ms,
                  "torch_fill_gbs": B * 2 * cfg.E * cfg.S * cfg.HW * limb_bytes / (fill_ms * 1e-3) / 1e9, "frac_of_copy_peak": bytes_out / (med * 1e-3) / 1e9 / peak,
                  "cpu_restatement_ms_per_image_1core": cpu_ms, "cpu_images_per_s_1core": 1e3 / cpu_ms}))
