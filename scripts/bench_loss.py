"""PPNLoss: the fused kernel pair (ppn_loss_forward / ppn_loss_backward) against the torch composite, as a share of
the copy bandwidth measured in the same run.

    python scripts/bench_loss.py [--iters 30] > profiles/bench_loss.txt
    python scripts/bench_loss.py --amp [--iters 30] > profiles/bench_loss_amp.txt
    python scripts/bench_loss.py --logits [--iters 30] > profiles/bench_loss_logits.txt

--amp adds, per shape, the mixed-precision rows: fp16 and bf16 heads, each with fp32 and with 16-bit te / weight_ij
(ppn_loss_forward_opt / ppn_loss_backward_opt); the upcast route an AMP user has without them (crit(head.float(), ...)
under autograd, the fp32 gradient cast back to the head's dtype by autograd); and the torch composite on the 16-bit
head.  Algorithmic bytes are counted per dtype: a 16-bit element is 2 bytes.  The upcast route also counts its two
casts (read the 16-bit head, write it in fp32; read the fp32 gradient, write it in 16 bits).

--logits adds, per shape, the loss on logits (PPNLoss(cfg, from_logits=True): ppn_loss_forward_logits /
ppn_loss_backward_logits) with fp32 logits and targets and with fp16 logits and fp16 te / weight_ij, against today's
route on the same logits: torch.sigmoid, the sigmoid-input loss, autograd's sigmoid backward.  Its bytes add the
sigmoid's read and write of the head and the sigmoid backward's two reads and one write.  The logits are randn * 3.

Shapes: cfg2 (mpii16: K16 / E15, 12x12 grid, 9x9 window) at B = 512 and the reference's native shape (K18 / E17,
24x24, 21x21) at B = 64; targets from TargetEncoder on random annotation sets, heads sigmoid(randn).  Every input
set is several times the 126 MB L2.  Times are means over back-to-back calls between two CUDA events, after warm-up; the fused rows call the C
exports with prebuilt arguments, so no Python checking sits in the window.
Algorithmic bytes: forward = head + te + weight_ij + the eight [B, K, H, W] targets; backward = the same plus the
gradient write.  The composite is the float32 restatement (oracle/ppn_loss.py loss_terms) under autograd.
"""
import argparse
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import encode_gt  # noqa: E402  (inputs and the composite baseline)
from oracle import ppn_loss as L  # noqa: E402
from pytorch_pose_proposal_network_b200 import PPNLoss, _lib  # noqa: E402
from pytorch_pose_proposal_network_b200.config import PRESETS  # noqa: E402
from pytorch_pose_proposal_network_b200.dataset import TargetEncoder  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--iters", type=int, default=30)
ap.add_argument("--warmup", type=int, default=3)
ap.add_argument("--amp", action="store_true", help="also the fp16 / bf16 rows")
ap.add_argument("--logits", action="store_true", help="also the loss-on-logits rows")
a = ap.parse_args()
assert torch.cuda.is_available(), "bench_loss measures on the GPU; there is nothing to measure without one"


def timed(fn, iters=a.iters, warmup=a.warmup):
    """Mean ms per call over `iters` back-to-back calls between two CUDA events (after warm-up): the host only
    enqueues, so as long as it stays ahead of the GPU the window holds device time alone."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(iters):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / iters


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as ex:                                           # the name from torch is still recorded
        q = f"{torch.cuda.get_device_name()} (nvidia-smi unavailable: {ex})"
    return q


print(f"# GPU: {gpu_info()}")
print(f"# torch {torch.__version__}, CUDA {torch.version.cuda}")

# copy bandwidth: one 4 GB device-to-device cudaMemcpyAsync (tensor.copy_), read + write counted
n = (4 << 30) // 4
src = torch.ones(n, device="cuda")
dst = torch.empty_like(src)
copy_ms = timed(lambda: dst.copy_(src), iters=20)
copy_gbs = 2 * n * 4 / copy_ms / 1e6
del src, dst
torch.cuda.empty_cache()
print(f"copy: 4 GiB device-to-device in {copy_ms:.3f} ms = {copy_gbs:.0f} GB/s (read + write)")


def inputs(cfg, B, seed=0):
    rng = np.random.default_rng(seed)
    samples = []
    for _ in range(B):
        kp, bb, vis, size = encode_gt.random_people(rng, int(rng.integers(0, 9)), cfg.K, cfg.insize)
        samples.append(dict(keypoints=kp, bbox=np.asarray(bb).reshape(-1, 4), is_visible=vis, size=size))
    t = TargetEncoder(cfg).encode(samples)
    head = torch.sigmoid(torch.randn(B, cfg.C, cfg.H, cfg.W, device="cuda"))
    return head, [getattr(t, nme) for nme in L.ARG_ORDER]


def peak_extra(fn):
    """Peak bytes allocated by fn beyond what was live before it."""
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def amp_rows(tag, cfg, B, crit, head32, targets32, ws, loss, g, lam):
    """The mixed-precision rows of one shape (see the module docstring)."""
    i_wij, i_te = L.ARG_ORDER.index("weight_ij"), L.ARG_ORDER.index("te")
    codes = {torch.float32: _lib.HEAD_F32, torch.float16: _lib.HEAD_F16, torch.bfloat16: _lib.HEAD_BF16}
    name = {torch.float32: "f32", torch.float16: "f16", torch.bfloat16: "bf16"}
    L_el, C_el, S_el = cfg.E * cfg.S * cfg.HW, cfg.C * cfg.HW, 8 * cfg.K * cfg.HW

    def per_img(hb, lb):                                              # forward, backward bytes per image
        fwd = C_el * hb + 2 * L_el * lb + S_el * 4
        return fwd, fwd + C_el * hb

    for hd in (torch.float16, torch.bfloat16):
        head = head32.to(hd)
        res, mem = {}, {}
        for ld in (torch.float32, hd):
            targets = list(targets32)
            targets[i_wij], targets[i_te] = targets32[i_wij].to(ld), targets32[i_te].to(ld)
            lb = 4 if ld == torch.float32 else 2
            fb, bb = per_img(2, lb)
            shape, tg = crit._shape(B, codes[hd]), crit._targets_struct(targets)
            opt = _lib.PPNLossOptions(codes[ld])
            grad = torch.empty_like(head)
            stream = crit._stream()
            fwd_args = (C.c_void_p(head.data_ptr()), C.byref(shape), C.byref(tg), C.byref(opt), C.c_void_p(loss.data_ptr()),
                        C.c_void_p(ws.data_ptr()), C.c_size_t(ws.numel()), stream)
            bwd_args = (C.c_void_p(head.data_ptr()), C.byref(shape), C.byref(tg), C.byref(opt), C.c_void_p(g.data_ptr()),
                        C.c_void_p(grad.data_ptr()), stream)
            assert crit.lib.ppn_loss_forward_opt(*fwd_args) == 0 and crit.lib.ppn_loss_backward_opt(*bwd_args) == 0
            fm = head.clone().requires_grad_(True)

            def fused_fb():
                fm.grad = None
                sum(l * t for l, t in zip(lam, crit(fm, *targets))).backward()

            lt = f"{name[hd]} head, {name[ld]} limb"
            res[f"{lt} forward"] = (timed(lambda: crit.lib.ppn_loss_forward_opt(*fwd_args)), fb)
            res[f"{lt} backward"] = (timed(lambda: crit.lib.ppn_loss_backward_opt(*bwd_args)), bb)
            res[f"{lt} fwd+bwd"] = (timed(fused_fb), fb + bb)
            fm.grad = None
            mem[lt] = peak_extra(fused_fb)
            if ld == hd:
                def composite_fb():
                    fm.grad = None
                    sum(l * t for l, t in zip(lam, L.loss_terms(fm, *targets, cfg))).backward()
                res[f"composite on {name[hd]} fwd+bwd"] = (timed(composite_fb), fb + bb)
            del grad, fm
        # the upcast route: an fp32 copy of the head, the fp32 loss on it (fp32 limb targets), the gradient cast back
        fm = head.clone().requires_grad_(True)

        def upcast_fb():
            fm.grad = None
            sum(l * t for l, t in zip(lam, crit(fm.float(), *targets32))).backward()

        fb, bb = per_img(4, 4)
        res[f"upcast {name[hd]} -> f32 fwd+bwd"] = (timed(upcast_fb), fb + bb + C_el * (2 + 4) + C_el * (4 + 2))
        fm.grad = None
        mem["upcast"] = peak_extra(upcast_fb)
        del fm, head
        for path, (ms, pi) in res.items():
            gbs = B * pi / ms / 1e6
            print(f"{tag:<18}{path:<32}{ms:>9.3f}{gbs:>9.0f}{gbs / copy_gbs:>8.2f}")
        for k, (fb, bb) in ((f"{name[hd]} head, f32 limb", per_img(2, 4)), (f"{name[hd]} head, {name[hd]} limb", per_img(2, 2))):
            print(f"{tag:<18}{k}: algorithmic bytes per image: forward {fb / 1e6:.2f} MB, backward {bb / 1e6:.2f} MB, "
                  f"peak memory fwd+bwd {mem[k] / 1e9:.2f} GB")
        up = res[f"upcast {name[hd]} -> f32 fwd+bwd"][0]
        print(f"{tag:<18}upcast route peak memory fwd+bwd {mem['upcast'] / 1e9:.2f} GB; fused fwd+bwd speed-up over it: "
              f"{name[hd]} limb {up / res[f'{name[hd]} head, {name[hd]} limb fwd+bwd'][0]:.2f}x, "
              f"f32 limb {up / res[f'{name[hd]} head, f32 limb fwd+bwd'][0]:.2f}x")
        torch.cuda.empty_cache()


def logits_rows(tag, cfg, B, targets32, ws, loss, g, lam):
    """The loss-on-logits rows of one shape (see the module docstring)."""
    i_wij, i_te = L.ARG_ORDER.index("weight_ij"), L.ARG_ORDER.index("te")
    codes = {torch.float32: _lib.HEAD_F32, torch.float16: _lib.HEAD_F16}
    name = {torch.float32: "f32", torch.float16: "f16"}
    L_el, C_el, S_el = cfg.E * cfg.S * cfg.HW, cfg.C * cfg.HW, 8 * cfg.K * cfg.HW
    crit, crit_l = PPNLoss(cfg), PPNLoss(cfg, from_logits=True)
    gen = torch.Generator(device="cuda").manual_seed(1)
    x32 = torch.randn(B, cfg.C, cfg.H, cfg.W, device="cuda", generator=gen) * 3
    for hd in (torch.float32, torch.float16):
        x = x32.to(hd)
        targets = list(targets32)
        targets[i_wij], targets[i_te] = targets32[i_wij].to(hd), targets32[i_te].to(hd)
        eb = 4 if hd == torch.float32 else 2
        fb = C_el * eb + 2 * L_el * eb + S_el * 4                     # forward bytes per image
        bb = fb + C_el * eb                                           # backward: the same plus the gradient write
        shape, tg = crit_l._shape(B, codes[hd]), crit_l._targets_struct(targets)
        opt = _lib.PPNLossOptions(codes[hd])
        grad = torch.empty_like(x)
        stream = crit_l._stream()
        fwd_args = (C.c_void_p(x.data_ptr()), C.byref(shape), C.byref(tg), C.byref(opt), C.c_void_p(loss.data_ptr()),
                    C.c_void_p(ws.data_ptr()), C.c_size_t(ws.numel()), stream)
        bwd_args = (C.c_void_p(x.data_ptr()), C.byref(shape), C.byref(tg), C.byref(opt), C.c_void_p(g.data_ptr()),
                    C.c_void_p(grad.data_ptr()), stream)
        assert crit_l.lib.ppn_loss_forward_logits(*fwd_args) == 0 and crit_l.lib.ppn_loss_backward_logits(*bwd_args) == 0
        fm = x.clone().requires_grad_(True)

        def fused_fb():
            fm.grad = None
            sum(l * t for l, t in zip(lam, crit_l(fm, *targets))).backward()

        def today_fb():
            fm.grad = None
            sum(l * t for l, t in zip(lam, crit(torch.sigmoid(fm), *targets))).backward()

        lt = f"{name[hd]} logits, {name[hd]} limb"
        res = {
            f"{lt} forward": (timed(lambda: crit_l.lib.ppn_loss_forward_logits(*fwd_args)), fb),
            f"{lt} backward": (timed(lambda: crit_l.lib.ppn_loss_backward_logits(*bwd_args)), bb),
            f"{lt} fwd+bwd": (timed(fused_fb), fb + bb),
            f"{name[hd]} sigmoid route fwd+bwd": (timed(today_fb), fb + bb + 2 * C_el * eb + 3 * C_el * eb),
        }
        fm.grad = None
        mem_fused = peak_extra(fused_fb)
        fm.grad = None
        mem_today = peak_extra(today_fb)
        for path, (ms, pi) in res.items():
            gbs = B * pi / ms / 1e6
            print(f"{tag:<18}{path:<32}{ms:>9.3f}{gbs:>9.0f}{gbs / copy_gbs:>8.2f}")
        print(f"{tag:<18}{name[hd]}: algorithmic bytes per image: logits forward {fb / 1e6:.2f} MB, backward {bb / 1e6:.2f} MB, "
              f"fwd+bwd {(fb + bb) / 1e6:.2f} MB; sigmoid route fwd+bwd {(fb + bb + 5 * C_el * eb) / 1e6:.2f} MB")
        print(f"{tag:<18}{name[hd]}: peak memory beyond the inputs (gradient included), fwd+bwd: logits {mem_fused / 1e9:.2f} GB, "
              f"sigmoid route {mem_today / 1e9:.2f} GB; speed-up over the sigmoid route: "
              f"{res[f'{name[hd]} sigmoid route fwd+bwd'][0] / res[f'{lt} fwd+bwd'][0]:.2f}x")
        del x, fm, grad
        torch.cuda.empty_cache()


print()
print(f"{'shape':<18}{'path':<32}{'ms':>9}{'GB/s':>9}{'/copy':>8}")
for name, B in (("cfg2", 512), ("native", 64)):
    cfg = PRESETS[name]()
    head, targets = inputs(cfg, B)
    crit = PPNLoss(cfg)
    L_el = cfg.E * cfg.S * cfg.HW
    per_img_fwd = (cfg.C * cfg.HW + 2 * L_el + 8 * cfg.K * cfg.HW) * 4
    per_img_bwd = per_img_fwd + cfg.C * cfg.HW * 4
    g = torch.tensor([0.7, 1.9, 1.3, 0.4, 2.2], device="cuda")
    grad = torch.empty_like(head)
    lam = [0.7, 1.9, 1.3, 0.4, 2.2]
    fm = head.clone().requires_grad_(True)

    def fused_fb():
        fm.grad = None
        sum(l * t for l, t in zip(lam, crit(fm, *targets))).backward()

    def composite_f():
        with torch.no_grad():
            L.loss_terms(head, *targets, cfg)

    def composite_fb():
        fm.grad = None
        sum(l * t for l, t in zip(lam, L.loss_terms(fm, *targets, cfg))).backward()

    # the two exports with their ctypes arguments built once
    lib, shape, tg = crit.lib, crit._shape(B), crit._targets_struct(targets)
    ws = crit._workspace(B)
    loss = torch.empty(5, device="cuda")
    stream = crit._stream()
    fwd_args = (C.c_void_p(head.data_ptr()), C.byref(shape), C.byref(tg), C.c_void_p(loss.data_ptr()),
                C.c_void_p(ws.data_ptr()), C.c_size_t(ws.numel()), stream)
    bwd_args = (C.c_void_p(head.data_ptr()), C.byref(shape), C.byref(tg), C.c_void_p(g.data_ptr()),
                C.c_void_p(grad.data_ptr()), stream)
    assert lib.ppn_loss_forward(*fwd_args) == 0 and lib.ppn_loss_backward(*bwd_args) == 0
    res = {
        "fused forward": (timed(lambda: lib.ppn_loss_forward(*fwd_args)), per_img_fwd),
        "fused backward": (timed(lambda: lib.ppn_loss_backward(*bwd_args)), per_img_bwd),
        "fused fwd+bwd (autograd)": (timed(fused_fb), per_img_fwd + per_img_bwd),
        "composite forward": (timed(composite_f), per_img_fwd),
        "composite fwd+bwd": (timed(composite_fb), per_img_fwd + per_img_bwd),
    }
    tag = f"{name} B={B}"
    # the host's cost per fused call, against which the device times above are safe only if it is far smaller
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(a.iters):
        lib.ppn_loss_forward(*fwd_args)
        lib.ppn_loss_backward(*bwd_args)
    host_us = (time.perf_counter() - t0) / (2 * a.iters) * 1e6
    torch.cuda.synchronize()
    for path, (ms, per_img) in res.items():
        gbs = B * per_img / ms / 1e6
        print(f"{tag:<18}{path:<32}{ms:>9.3f}{gbs:>9.0f}{gbs / copy_gbs:>8.2f}")
    print(f"{tag:<18}host enqueue per fused call: {host_us:.1f} us")
    fm.grad = None                                                    # the gradient counts in each path's peak
    mem_fused = peak_extra(fused_fb)
    fm.grad = None
    mem_comp = peak_extra(composite_fb)
    print(f"{tag:<18}algorithmic bytes per image: forward {per_img_fwd / 1e6:.2f} MB, backward {per_img_bwd / 1e6:.2f} MB")
    print(f"{tag:<18}peak memory beyond the inputs (gradient included), fwd+bwd: fused {mem_fused / 1e9:.2f} GB, composite {mem_comp / 1e9:.2f} GB")
    print(f"{tag:<18}fwd+bwd speed-up over the composite: {res['composite fwd+bwd'][0] / res['fused fwd+bwd (autograd)'][0]:.1f}x")
    if a.amp:
        amp_rows(tag, cfg, B, crit, head, targets, ws, loss, g, lam)
    if a.logits:
        logits_rows(tag, cfg, B, targets, ws, loss, g, lam)
    del head, targets, crit, grad, fm, ws, loss
    torch.cuda.empty_cache()
