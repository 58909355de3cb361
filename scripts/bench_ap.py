"""Scoring a validation pass: APEvaluator on the GPU against pred_frames + the float64 restatement of poseval's
assignGTmulti / computeMetrics on frames (oracle/pose_ap.py) on one host core.

    python scripts/bench_ap.py [--images 3000] [--cpu-images 96] [--out profiles/bench_ap.txt]

Two passes of about --images images each:
  native  B = 64 per update, the S head distribution (a few to a few dozen humans per image), 1-8 synthetic GT
          people per image, most of them placed near a predicted human;
  cfg3    B = 1024 per update, the dense D distribution (about 226 humans per image): a stress shape.
The heads are generated and parsed before the timed region; the GT frames are built on the host from the parse.
Reported, from CUDA events: the device time of one update (ppn_ap_match on a batch, GT already on the device) and of
compute() (ppn_ap_finalize and the copy of its results); from a host clock: the whole pass through update() on host GT
frames + compute().  The restatement arm (pred_frames + restated assignGTmulti / computeMetrics) runs on the first
--cpu-images images of the first batch only (an eighth of that at cfg3), since it takes up to seconds per image at
the dense shape; its time per image and that rate scaled to the pass are reported as such.  The GPU result on those images is checked against the restatement.
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import pose_ap as P, ppn_oracle as O                        # noqa: E402
from pytorch_pose_proposal_network_b200.config import PRESETS           # noqa: E402
from pytorch_pose_proposal_network_b200.evaluation import APEvaluator, gt_from_frames, pred_frames   # noqa: E402
from pytorch_pose_proposal_network_b200.parser import PoseParser        # noqa: E402
from tests.gpu_inputs import device_head                                # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--images", type=int, default=3000)
ap.add_argument("--cpu-images", type=int, default=96)
ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "profiles", "bench_ap.txt"))
a = ap.parse_args()
assert torch.cuda.is_available(), "bench_ap measures on the GPU; there is nothing to measure without one"
torch.set_num_threads(1)

lines = []


def say(s=""):
    print(s, flush=True)
    lines.append(s)


try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
except Exception as ex:
    q = f"{torch.cuda.get_device_name()} (nvidia-smi unavailable: {ex})"
say(f"# GPU: {q}")
say(f"# torch {torch.__version__}, CUDA {torch.version.cuda}; host arm on one core: {os.cpu_count()} cores visible")


def gt_near(rng, a_np, c_np, R, J):
    """1-8 GT people per image, 85 % of them on a predicted human (joints jittered by ~12 px, 20 % missing)."""
    frames = []
    for b in range(a_np["count"].shape[0]):
        n_pred = min(int(a_np["count"][b]), R)
        rects = []
        for _ in range(int(rng.integers(1, 9))):
            x0, y0 = (float(v) for v in rng.integers(0, 300, 2))
            rect = {"x1": [x0], "y1": [y0], "x2": [x0 + 30.0], "y2": [y0 + 40.0]}
            i = int(rng.integers(n_pred)) if n_pred and rng.random() < 0.85 else -1
            pts = []
            for j in range(c_np.shape[2] - 1):
                if rng.random() < 0.2:
                    continue
                if i >= 0:
                    x, y = c_np[b, i, j + 1, 1] + rng.normal(0, 12), c_np[b, i, j + 1, 0] + rng.normal(0, 12)
                else:
                    x, y = rng.uniform(0, 400, 2)
                pts.append({"id": [j], "x": [float(x)], "y": [float(y)]})
            rect["annopoints"] = [{"point": pts}]
            rects.append(rect)
        frames.append({"image": [f"{b}.jpg"], "annorect": rects})
    return frames


def run(preset, dist, B, cpu_images):
    cfg = PRESETS[preset]()
    J = cfg.K - 1
    n_batches = max(1, round(a.images / B))
    parser = PoseParser(cfg)
    rng = np.random.default_rng(0)
    batches = []
    for i in range(n_batches):
        head, _ = device_head(O.Geometry.of(cfg), dist, seed=100 + i, B=B, distinct=False)
        packed = parser.parse(head, out=parser.alloc_output(B))
        centres = parser.part_centres(packed)
        del head
        frames = gt_near(rng, packed.numpy(), centres.cpu().numpy(), packed.R, J)
        flat = [torch.from_numpy(x).cuda() for x in gt_from_frames(frames, J)]
        batches.append((packed, centres, frames, flat))
    torch.cuda.synchronize()
    N = n_batches * B
    humans = sum(int(p.count.sum()) for p, *_ in batches)
    gt_people = sum(len(f["annorect"]) for *_, fr, _ in batches for f in fr)
    tag = f"{preset} B={B} {dist}"
    say(f"{tag:<18} {N} images in {n_batches} updates: {humans / N:.1f} humans and {gt_people / N:.2f} GT people per image")

    def device_pass(ev):
        st = torch.cuda.current_stream()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in batches]
        for (packed, _, _, flat), (e0, e1) in zip(batches, evs):
            e0.record(st)
            ev.update_flat(packed, *flat)
            e1.record(st)
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record(st)
        res = ev.compute()
        c1.record(st)
        c1.synchronize()
        return res, [e0.elapsed_time(e1) for e0, e1 in evs], c0.elapsed_time(c1)

    ev = APEvaluator(cfg)
    device_pass(ev)                                                      # warm-up: module load, allocator
    times = []
    for _ in range(3):
        ev.reset()
        res, upd, comp = device_pass(ev)
        times.append((float(np.median(upd)), comp))
    upd_ms = float(np.median([t[0] for t in times]))
    comp_ms = float(np.median([t[1] for t in times]))
    say(f"{tag:<18} device: update (ppn_ap_match, {B} images) {upd_ms:.4f} ms = {upd_ms / B * 1e3:.2f} us per image; "
        f"compute() {comp_ms:.3f} ms")

    walls = []
    for _ in range(3):
        ev.reset()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for packed, _, frames, _ in batches:
            ev.update(packed, frames)
        host_res = ev.compute()
        walls.append(time.perf_counter() - t0)
    wall = float(np.median(walls))
    assert all(np.array_equal(host_res[k].view(np.uint64), res[k].view(np.uint64)) for k in res)
    say(f"{tag:<18} GPU pass from host GT frames (gt_from_frames + upload + update, compute): {wall * 1e3:.1f} ms "
        f"= {wall / N * 1e6:.1f} us per image")

    # the restatement arm on the first images of the pass
    n_cpu = min(cpu_images, B)
    packed, centres, frames, _ = batches[0]
    sub_packed = type(packed)(cfg, *(t[:n_cpu] for t in (packed.count, packed.root_cell, packed.part_cell,
                                                         packed.part_score, packed.part_box)))
    ev_sub = APEvaluator(cfg)
    ev_sub.update(sub_packed, frames[:n_cpu])
    gpu_sub = ev_sub.compute()
    t0 = time.perf_counter()
    preds = pred_frames([f"{b}.jpg" for b in range(n_cpu)], sub_packed, centres[:n_cpu])
    t1 = time.perf_counter()
    want = P.evaluate(frames[:n_cpu], preds, J)
    t2 = time.perf_counter()
    for k in want:
        np.testing.assert_allclose(gpu_sub[k], want[k], rtol=0, atol=1e-9, equal_nan=True)
    per_img = (t2 - t0) / n_cpu
    say(f"{tag:<18} restatement arm on {n_cpu} images: pred_frames {(t1 - t0) * 1e3:.1f} ms + restated poseval "
        f"{(t2 - t1) * 1e3:.1f} ms = {per_img * 1e3:.2f} ms per image; at that rate the pass takes {per_img * N:.1f} s "
        f"(scaled, not run): {per_img * N / wall:.0f}x the GPU pass; results on those images agree within 1e-9")
    say(f"{tag:<18} mean AP {res['ap'][-1]:.3f}, precision {res['precision'][-1]:.3f}, recall {res['recall'][-1]:.3f}")
    say()


run("native", "S", 64, a.cpu_images)
run("cfg3", "D", 1024, max(1, a.cpu_images // 8))
os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
with open(a.out, "w") as f:
    f.write("\n".join(lines) + "\n")
