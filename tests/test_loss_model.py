"""The training loss's float32 gradient model against torch autograd of the float64 restatement (CPU only).

oracle/ppn_loss.py restates the reference's PPNLoss (main.py:125-216) in torch and models, in numpy float32, the
closed-form per-element gradient that csrc/ppn_loss.cu computes.  Here the model is held to autograd — on random
heads, and on cases built to sit exactly on the kinks (equal predicted and target edges: ties in min / max; boxes
that only touch: relu at 0) — and the restatement is held to its defining property: a head that reproduces its
targets has zero loss in every term but the IoU's eps residual.
"""
import numpy as np
import pytest
import torch

from oracle import encode_gt
from oracle import ppn_loss as L
from pytorch_pose_proposal_network_b200.config import EDGES, EDGES_16, PPNConfig

# float32 model vs float64 autograd: each element within RTOL of the reference value, plus ATOL_REL times the
# largest magnitude of its channel group (the IoU part of d/dx and d/dw can cancel the coordinate / size part, so an
# element's own magnitude is no scale for the rounding it carries; single-precision rounding of the summands is ~1e-7
# of the group's scale)
RTOL, ATOL_REL = 1e-4, 1e-6


def geometries():
    return {"mpii16": PPNConfig.mpii16(), "k18_13x13": PPNConfig.reference_native(insize=(416, 416), outsize=(13, 13),
                                                                                  local_grid_size=(7, 7))}


def encoded_targets(cfg, B, rng, people=(0, 9)):
    edges = EDGES_16 if cfg.K == 16 else EDGES
    per = []
    for _ in range(B):
        kp, bb, vis, size = encode_gt.random_people(rng, int(rng.integers(*people)), cfg.K, cfg.insize)
        per.append(encode_gt.encode_targets(kp, bb, vis, size, cfg.K, edges, cfg.insize, cfg.outsize,
                                            cfg.local_grid_size))
    names = ("delta", "weight", "weight_ij", "tx", "ty", "tx_half", "ty_half", "tw", "th", "te")   # __getitem__ order
    by_name = {n: np.stack([p[i] for p in per]) for i, n in enumerate(names)}
    return [by_name[n] for n in L.ARG_ORDER]                                                       # criterion order


def check_against_autograd(cfg, head, targets, grad_loss):
    got = L.grad_model_f32(head, *targets, cfg, grad_loss)
    want = L.autograd_grad(torch.from_numpy(head), [torch.from_numpy(t) for t in targets], cfg, grad_loss).numpy()
    assert np.isfinite(got).all()
    K = cfg.K
    groups = [slice(i * K, (i + 1) * K) for i in range(6)] + [slice(6 * K, cfg.C)]
    for gi, sl in enumerate(groups):
        g, w = got[:, sl].astype(np.float64), want[:, sl]
        tol = RTOL * np.abs(w) + ATOL_REL * max(np.abs(w).max(), 1e-30)
        bad = np.abs(g - w) > tol
        assert not bad.any(), (gi, int(bad.sum()), np.abs(g - w).max())
    return got, want


@pytest.mark.parametrize("geo", list(geometries()))
@pytest.mark.parametrize("seed", range(3))
def test_grad_model_matches_autograd_random(geo, seed):
    cfg = geometries()[geo]
    rng = np.random.default_rng(seed)
    B = 2
    targets = encoded_targets(cfg, B, rng)
    head = (1.0 / (1.0 + np.exp(-rng.standard_normal((B, cfg.C, cfg.H, cfg.W))))).astype(np.float32)
    grad_loss = rng.uniform(0.2, 3.0, 5).astype(np.float32)          # GradNorm-like weights
    check_against_autograd(cfg, head, targets, grad_loss)


def kink_case(cfg, rng, B=2):
    """Targets and a head whose boxes sit exactly on the kinks, in dyadic values (exact in float32 and float64):
    equal edges (min / max ties), boxes that only touch (relu at 0), partial overlaps, zero-area boxes, and a
    random 0/1 delta with its weight and half-offset targets."""
    K, H, W = cfg.K, cfg.H, cfg.W
    gW, gH = cfg.gridsize
    shape = (B, K, H, W)
    delta = (rng.random(shape) < 0.5).astype(np.float32)
    tx = rng.integers(0, 16, shape).astype(np.float32) / 16
    ty = rng.integers(0, 16, shape).astype(np.float32) / 16
    tw = rng.integers(0, 8, shape).astype(np.float32) / 64
    th = rng.integers(0, 8, shape).astype(np.float32) / 64
    kind = rng.integers(0, 5, shape)
    x, y, w, h = tx.copy(), ty.copy(), tw.copy(), th.copy()              # kind 0: identical boxes (ties everywhere)
    # kind 1: touching in x (predicted left edge = target right edge), overlapping in y
    w1 = rng.integers(1, 8, shape).astype(np.float32) / 64
    x = np.where(kind == 1, tx + (cfg.inW * (tw + w1) / 2) / gW, x)
    w = np.where(kind == 1, w1, w)
    # kind 2: shared left edge, different widths (a max tie, no min tie); y shifted by a dyadic amount
    w2 = tw + 1.0 / 64
    x = np.where(kind == 2, tx + (cfg.inW * (w2 - tw) / 2) / gW, x)
    w = np.where(kind == 2, w2, w)
    y = np.where(kind == 2, ty + 1.0 / 8, y)
    # kind 3: zero-area prediction
    w = np.where(kind == 3, 0.0, w)
    h = np.where(kind == 3, 0.0, h)
    # kind 4: touching in y (predicted top edge = target bottom edge)
    h4 = rng.integers(1, 8, shape).astype(np.float32) / 64
    y = np.where(kind == 4, ty + (cfg.inH * (th + h4) / 2) / gH, y)
    h = np.where(kind == 4, h4, h)
    resp = rng.integers(0, 16, shape) / 16
    conf = rng.integers(0, 16, shape) / 16
    small = np.stack([resp, conf, x, y, w, h], 1).reshape(B, 6 * K, H, W)
    e = rng.integers(0, 16, (B, cfg.E * cfg.S, H, W)) / 16
    head = np.concatenate([small, e], 1).astype(np.float32)
    weight = np.where(delta < 0.5, np.float32(0.0005), np.float32(1)).astype(np.float32)
    half = np.where(delta < 0.5, np.float32(0.5), np.float32(0)).astype(np.float32)
    big = (B, cfg.E, cfg.sH, cfg.sW, H, W)
    weight_ij = np.where(rng.random(big) < 0.3, np.float32(1), np.float32(0.0005)).astype(np.float32)
    te = (rng.random(big) < 0.01).astype(np.float32)
    targets = [delta, weight, weight_ij, (tx + half).astype(np.float32), (ty + half).astype(np.float32),
               tx, ty, tw, th, te]
    return head, [np.ascontiguousarray(t, np.float32) for t in targets], kind


@pytest.mark.parametrize("geo", list(geometries()))
def test_grad_model_matches_autograd_on_kinks(geo):
    cfg = geometries()[geo]
    rng = np.random.default_rng(7)
    head, targets, kind = kink_case(cfg, rng)
    K = cfg.K
    x = head[:, 2 * K:3 * K]
    for k in range(5):
        assert (kind == k).sum() > 50                                    # every kind of kink is present
    # the constructed edges really are equal in float32 (the model's arithmetic) where they should be
    gW = np.float32(cfg.gridsize[0])
    X = np.arange(cfg.W, dtype=np.float32)
    tx, tw = targets[5], targets[7]
    w = head[:, 4 * K:5 * K]
    p1 = (x + X) * gW - np.float32(cfg.inW) * w * np.float32(0.5)
    q2 = (tx + X) * gW + np.float32(cfg.inW) * tw * np.float32(0.5)
    assert np.array_equal(p1[kind == 1], q2[kind == 1])
    got, want = check_against_autograd(cfg, head, targets, np.array([0.7, 1.9, 1.3, 0.4, 2.2], np.float32))
    # zero-area predictions where delta = 0 (and elsewhere): finite, as eps in the union guarantees
    assert np.isfinite(want).all()


def perfect_head(cfg, targets):
    """The head that reproduces its targets: resp = delta, conf = 1, x = tx_half, y = ty_half, w = tw, h = th, e = te."""
    t = dict(zip(L.ARG_ORDER, targets))
    B = t["delta"].shape[0]
    return np.concatenate([t["delta"], np.ones_like(t["delta"]), t["tx_half"], t["ty_half"], t["tw"], t["th"],
                           t["te"].reshape(B, -1, cfg.H, cfg.W)], 1).astype(np.float32)


@pytest.mark.parametrize("geo", list(geometries()))
def test_perfect_prediction(geo):
    cfg = geometries()[geo]
    rng = np.random.default_rng(11)
    targets = encoded_targets(cfg, 3, rng, people=(2, 9))
    head = perfect_head(cfg, targets)
    tt = [torch.from_numpy(t).double() for t in targets]
    terms = [float(v) for v in L.loss_terms(torch.from_numpy(head).double(), *tt, cfg)]
    assert terms[0] == 0.0 and terms[2] == 0.0 and terms[3] == 0.0 and terms[4] == 0.0, terms
    # L_iou: where delta = 1 the boxes coincide, iou = A / (A + eps), the residual is sum (eps / (A + eps))^2 / B
    t = dict(zip(L.ARG_ORDER, targets))
    on = t["delta"] == 1
    A = (cfg.inW * t["tw"].astype(np.float64)) * (cfg.inH * t["th"].astype(np.float64))
    want = float(np.sum((L.EPSILON / (A[on] + L.EPSILON)) ** 2)) / 3
    assert on.sum() > 10 and 0 < want < 1e-12
    assert terms[1] == pytest.approx(want, rel=1e-4)
    # the gradient of the four exact terms vanishes in the float32 model too
    g = L.grad_model_f32(head, *targets, cfg, np.array([1, 0, 1, 1, 1], np.float32))
    assert not np.any(g)
    # the order trap: tx / ty passed where tx_half / ty_half belong (TargetBatch.as_list() order) is not a zero loss
    swapped = list(tt)
    swapped[3], swapped[4], swapped[5], swapped[6] = tt[5], tt[6], tt[3], tt[4]
    assert float(L.loss_terms(torch.from_numpy(head).double(), *swapped, cfg)[2]) > 0


def test_loss_abi_argument_checks_without_gpu():
    """Host-side validation of the three loss exports: every rejection happens before anything is enqueued."""
    import ctypes as C
    from pytorch_pose_proposal_network_b200 import _lib
    from pytorch_pose_proposal_network_b200.parser import _CConfig
    lib = _lib.lib()
    cfg = PPNConfig.mpii16()
    shape = _CConfig(cfg).shape(512)
    need = C.c_size_t()
    assert lib.ppn_loss_workspace_bytes(C.byref(shape), C.byref(need)) == 0
    assert 8 * 5 <= need.value <= 2048 * 5 * 8                       # one fp64 partial set per CTA, at most 2048 CTAs
    assert lib.ppn_loss_workspace_bytes(None, C.byref(need)) == -1
    assert lib.ppn_loss_workspace_bytes(C.byref(_CConfig(cfg).shape(0)), C.byref(need)) == -1
    assert lib.ppn_loss_workspace_bytes(C.byref(_CConfig(cfg).shape(4, _lib.HEAD_BF16)), C.byref(need)) == -2
    fake = 1 << 20                                                     # aligned, never dereferenced: rejected first
    tg = _lib.PPNTargets(*[fake] * 10)
    fwd = lambda head, t=tg, s=shape, ws=fake, n=need.value: lib.ppn_loss_forward(head, C.byref(s), C.byref(t), fake, ws, n, None)
    assert fwd(None) == -1
    assert fwd(fake + 2) == -1
    assert fwd(fake, n=need.value - 1) == -3
    assert fwd(fake, ws=fake + 4) == -1
    assert fwd(fake, t=_lib.PPNTargets(*([fake] * 9 + [0]))) == -1
    assert fwd(fake, s=_CConfig(cfg).shape(512, _lib.HEAD_F16)) == -2
    assert lib.ppn_loss_backward(fake, C.byref(shape), C.byref(tg), None, fake, None) == -1
    assert lib.ppn_loss_backward(fake, C.byref(shape), C.byref(tg), fake, fake + 1, None) == -1
    assert lib.ppn_loss_backward(fake, C.byref(_CConfig(cfg).shape(512, _lib.HEAD_F16)), C.byref(tg), fake, fake, None) == -2
