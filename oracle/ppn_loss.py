"""The training loss, restated.  TEST INFRASTRUCTURE.

The reference's criterion ``PPNLoss`` (main.py:125-216) is not in this tree.  This file is its specification,
reconstructed from what is pinned here: the argument order of its call site (INTEGRATION.md), the exact semantics of
the ten targets (encode_gt.encode_targets: weight = min(delta + 0.0005 [delta < 0.5], 1), tx_half = tx + 0.5
[delta < 0.5], ...), config.EPSILON, and the loss of the paper (Sekii, Pose Proposal Networks, ECCV 2018) in the
form of the Chainer original the reference ports.  Three points rest on the reconstruction:

1. the IoU is differentiable: gradient flows into x, y, w and h;
2. eps appears in the IoU denominator;
3. L_resp is unweighted.

``loss_terms`` is plain torch (any device, any float dtype: the tests run it in float64, under autograd for the
gradient).  ``grad_model_f32`` is numpy float32 with the closed-form per-element gradient in the operation order
csrc/ppn_loss.cu documents, so that the kernel's output can be compared bit for bit.
"""
from __future__ import annotations

import numpy as np
import torch

EPSILON = 1e-6
ARG_ORDER = ("delta", "weight", "weight_ij", "tx_half", "ty_half", "tx", "ty", "tw", "th", "te")


def _grid(cfg, like):
    X = torch.arange(cfg.W, dtype=like.dtype, device=like.device).view(1, 1, 1, cfg.W)
    Y = torch.arange(cfg.H, dtype=like.dtype, device=like.device).view(1, 1, cfg.H, 1)
    return X, Y


def iou_terms(x, y, w, h, tx, ty, tw, th, cfg, eps=EPSILON):
    """IoU of the predicted and the target box of every cell, in pixels (centre / size boxes)."""
    gW, gH = cfg.gridsize
    X, Y = _grid(cfg, x)
    px, py = (x + X) * gW, (y + Y) * gH
    pw, ph = cfg.inW * w, cfg.inH * h
    qx, qy = (tx + X) * gW, (ty + Y) * gH
    qw, qh = cfg.inW * tw, cfg.inH * th
    iw = torch.relu(torch.minimum(px + pw * 0.5, qx + qw * 0.5) - torch.maximum(px - pw * 0.5, qx - qw * 0.5))
    ih = torch.relu(torch.minimum(py + ph * 0.5, qy + qh * 0.5) - torch.maximum(py - ph * 0.5, qy - qh * 0.5))
    inter = iw * ih
    return inter / (pw * ph + qw * qh - inter + eps)


def loss_terms(feature_map, delta, weight, weight_ij, tx_half, ty_half, tx, ty, tw, th, te, cfg, eps=EPSILON):
    """(L_resp, L_iou, L_coor, L_size, L_limb): each summed over every element of an image, averaged over the batch.
    Arguments in the criterion's order; feature_map [B, 6K + E*sH*sW, H, W]."""
    B, K = feature_map.shape[0], cfg.K
    resp, conf, x, y, w, h = feature_map[:, :6 * K].reshape(B, 6, K, cfg.H, cfg.W).unbind(1)
    e = feature_map[:, 6 * K:].reshape(B, cfg.E, cfg.sH, cfg.sW, cfg.H, cfg.W)
    iou = iou_terms(x, y, w, h, tx, ty, tw, th, cfg, eps)
    l_resp = ((resp - delta) ** 2).sum()
    l_iou = (delta * (conf - iou) ** 2).sum()
    l_coor = (weight * ((x - tx_half) ** 2 + (y - ty_half) ** 2)).sum()
    l_size = (weight * ((torch.sqrt(w + eps) - torch.sqrt(tw + eps)) ** 2 +
                        (torch.sqrt(h + eps) - torch.sqrt(th + eps)) ** 2)).sum()
    l_limb = (weight_ij * (e - te) ** 2).sum()
    return tuple(t / B for t in (l_resp, l_iou, l_coor, l_size, l_limb))


def grad_model_f32(feature_map, delta, weight, weight_ij, tx_half, ty_half, tx, ty, tw, th, te, cfg, grad_loss,
                   eps=EPSILON, batch=None):
    """d(sum_t grad_loss[t] * L_t)/d(feature_map) in numpy float32, one rounding per operation, in the order of
    csrc/ppn_loss.cu.  Arrays (numpy) in the criterion's order; returns [B, C, H, W] float32.  `batch`: the size of
    the batch the loss averages over, when the arrays are a sample of its images (default: all of them)."""
    f = np.float32
    fm = np.asarray(feature_map, f)
    B, K, H, W = fm.shape[0], cfg.K, cfg.H, cfg.W
    g = np.asarray(grad_loss, f).reshape(5)
    Bf, two, half, epsf = f(B if batch is None else batch), f(2), f(0.5), f(eps)
    cr, ci, cc, cl = (two * g[i] / Bf for i in (0, 1, 2, 4))
    cs = g[3] / Bf
    d, wt, txh, tyh, tx_, ty_, tw_, th_ = (np.asarray(a, f) for a in (delta, weight, tx_half, ty_half, tx, ty, tw, th))
    resp, conf, x, y, w, h = fm[:, :6 * K].reshape(B, 6, K, H, W).transpose(1, 0, 2, 3, 4)
    e = fm[:, 6 * K:].reshape(B, cfg.E, cfg.sH, cfg.sW, H, W)
    gW, gH = (f(v) for v in cfg.gridsize)
    inW, inH = f(cfg.inW), f(cfg.inH)
    X = np.arange(W, dtype=f).reshape(1, 1, 1, W)
    Y = np.arange(H, dtype=f).reshape(1, 1, H, 1)

    def axis(v, t, sz, tsz, pos, grid, size_in):
        p, q = (v + pos) * grid, (t + pos) * grid
        ps, qs = size_in * sz, size_in * tsz
        hp, hq = ps * half, qs * half
        p1, p2, q1, q2 = p - hp, p + hp, q - hq, q + hq
        r = np.minimum(p2, q2) - np.maximum(p1, q1)
        return dict(p1=p1, p2=p2, q1=q1, q2=q2, size=ps, qsize=qs, r=r, i=np.where(r > 0, r, f(0)))

    bx = axis(x, tx_, w, tw_, X, gW, inW)
    by = axis(y, ty_, h, th_, Y, gH, inH)
    inter = bx["i"] * by["i"]
    union = ((bx["size"] * by["size"] + bx["qsize"] * by["qsize"]) - inter) + epsf
    iou = inter / union

    def axis_grad(b, gi):
        s2 = np.where(b["p2"] < b["q2"], f(1), np.where(b["p2"] == b["q2"], half, f(0)))
        s1 = np.where(b["p1"] > b["q1"], f(1), np.where(b["p1"] == b["q1"], half, f(0)))
        d2 = gi * s2
        d1 = -(gi * s1)
        return d2 + d1, (d2 - d1) * half

    out = np.empty_like(fm)
    grp = out[:, :6 * K].reshape(B, 6, K, H, W)
    grp[:, 0] = cr * (resp - d)
    a = ci * (d * (conf - iou))
    grp[:, 1] = a
    r = (-a) / union
    ri = r * iou
    dI = r + ri
    giw = np.where(bx["r"] > 0, dI * by["i"], f(0))
    gih = np.where(by["r"] > 0, dI * bx["i"], f(0))
    dpx, dpw = axis_grad(bx, giw)
    dpy, dph = axis_grad(by, gih)
    dpw = dpw - ri * by["size"]
    dph = dph - ri * bx["size"]
    grp[:, 2] = cc * (wt * (x - txh)) + dpx * gW
    grp[:, 3] = cc * (wt * (y - tyh)) + dpy * gH
    sw, st = np.sqrt(w + epsf), np.sqrt(tw_ + epsf)
    sh, sth = np.sqrt(h + epsf), np.sqrt(th_ + epsf)
    grp[:, 4] = cs * (wt * ((sw - st) / sw)) + dpw * inW
    grp[:, 5] = cs * (wt * ((sh - sth) / sh)) + dph * inH
    wij, te_ = np.asarray(weight_ij, f), np.asarray(te, f)
    out[:, 6 * K:] = (cl * (wij * (e - te_))).reshape(B, -1, H, W)
    return out


def autograd_grad(feature_map, targets, cfg, grad_loss, dtype=torch.float64):
    """torch autograd of loss_terms in `dtype`: d(sum_t grad_loss[t] * L_t)/d(feature_map).  targets: the ten
    tensors in the criterion's order."""
    fm = feature_map.detach().to(dtype).requires_grad_(True)
    terms = loss_terms(fm, *[t.to(dtype) for t in targets], cfg)
    gl = torch.as_tensor(grad_loss, dtype=dtype, device=fm.device)
    sum(gl[i] * terms[i] for i in range(5)).backward()
    return fm.grad
