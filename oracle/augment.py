"""Batch augmentation restated in numpy.  TEST INFRASTRUCTURE (the specification of ppn_augment_*).

The reference's aug.py (imgaug affine / crop / resize of the image, keypoints and boxes, then ToNormalizedTensor) is
not part of this tree, so, as for the loss and AP, this restatement is the specification; DESIGN.md §14 lists its
reconstruction points.  Exactness starts at the parameters: per image a forward affine A (float64 [2, 3], source
pixel coordinates -> output coordinates, pixel (row i, col j) centred at (j + .5, i + .5)), M = A^-1 rounded once to
fp32, and a flip flag.  Images in fp32 with one rounding per operation (no fused multiply-add), annotations in fp64.
"""
from __future__ import annotations

import math

import numpy as np

f32, f64 = np.float32, np.float64
COORD_LIMIT = f32(2.0 ** 30)
IMAGENET_MEAN = (0.485, 0.456, 0.406)
IMAGENET_STD = (0.229, 0.224, 0.225)
IN_SCALE = f32(1.0 / 255.0)


def bf16_bits(x: np.ndarray) -> np.ndarray:
    """fp32 -> bfloat16 bit patterns (uint16), rounded to nearest even; NaN stays a (quiet) NaN."""
    u = np.ascontiguousarray(x, f32).view(np.uint32).astype(np.uint64)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)
    nan = np.isnan(x)
    r[nan] = ((u[nan] >> 16) | 0x40).astype(np.uint16)
    return r


def to_dtype(x: np.ndarray, dtype: str) -> np.ndarray:
    """The fp32 result rounded once to the output dtype ('float32', 'float16'; 'bfloat16' as uint16 bits)."""
    if dtype == "float32":
        return x.astype(f32)
    if dtype == "float16":
        return x.astype(np.float16)
    if dtype == "bfloat16":
        return bf16_bits(x)
    raise ValueError(dtype)


def warp_image(img: np.ndarray, M, insize, mean=IMAGENET_MEAN, std=IMAGENET_STD, fill=(0.0, 0.0, 0.0),
               in_scale=IN_SCALE, dtype="float32") -> np.ndarray:
    """One image [h, w, 3] uint8 -> [3, inH, inW] of `dtype`, for fp32 M [2, 3]:
    sx = ((m00 pcx + m01 pcy) + m02) - .5 at the output pixel centre (pcx, pcy) = (u + .5, v + .5), sy likewise;
    bilinear taps at floor(s) and floor(s) + 1, val = (p00 (1 - ax) + p01 ax) (1 - ay) + (p10 (1 - ax) + p11 ax) ay;
    out = (val * in_scale - mean[c]) / std[c].  A tap outside the source reads fill[c]; a pixel whose four taps are
    all outside, or whose sx or sy is non-finite or beyond +-2^30, takes val = fill[c]."""
    h, w = img.shape[:2]
    inW, inH = int(insize[0]), int(insize[1])
    m = np.asarray(M, f32).reshape(2, 3)
    with np.errstate(all="ignore"):
        pcx = (np.arange(inW, dtype=f32) + f32(0.5))[None, :]
        pcy = (np.arange(inH, dtype=f32) + f32(0.5))[:, None]
        sx = ((m[0, 0] * pcx + m[0, 1] * pcy) + m[0, 2]) - f32(0.5)
        sy = ((m[1, 0] * pcx + m[1, 1] * pcy) + m[1, 2]) - f32(0.5)
        ok = (np.abs(sx) <= COORD_LIMIT) & (np.abs(sy) <= COORD_LIMIT)
        fx, fy = np.floor(np.where(ok, sx, f32(0))), np.floor(np.where(ok, sy, f32(0)))
        ix, iy = fx.astype(np.int64), fy.astype(np.int64)
        ok &= (ix + 1 >= 0) & (ix < w) & (iy + 1 >= 0) & (iy < h)
        ax, ay = (sx - fx).astype(f32), (sy - fy).astype(f32)
        bx, by = f32(1) - ax, f32(1) - ay
        out = np.empty((3, inH, inW), f32)
        src = img.astype(f32)
        for c in range(3):
            fc = f32(fill[c])

            def tap(x, y):
                inside = (x >= 0) & (x < w) & (y >= 0) & (y < h)
                return np.where(inside, src[np.clip(y, 0, h - 1), np.clip(x, 0, w - 1), c], fc)

            p00, p01, p10, p11 = tap(ix, iy), tap(ix + 1, iy), tap(ix, iy + 1), tap(ix + 1, iy + 1)
            val = (p00 * bx + p01 * ax) * by + (p10 * bx + p11 * ax) * ay
            val = np.where(ok, val, fc).astype(f32)
            out[c] = (val * f32(in_scale) - f32(mean[c])) / f32(std[c])
    return to_dtype(out, dtype)


def flip_permutation(keypoint_names) -> np.ndarray:
    """[K - 1]: column i of a mirrored image takes column perm[i] (left_* <-> right_*, others fixed)."""
    names = list(keypoint_names)[1:]
    perm = []
    for n in names:
        if n.startswith("left_"):
            n = "right_" + n[5:]
        elif n.startswith("right_"):
            n = "left_" + n[6:]
        perm.append(names.index(n))
    return np.asarray(perm, np.int32)


def _apply(A, x, y):
    return (A[0, 0] * x + A[0, 1] * y) + A[0, 2], (A[1, 0] * x + A[1, 1] * y) + A[1, 2]


def transform_people(person_off, bbox, keypoints, visible, size, A, flip, perm):
    """Flat annotations of B images through A [B, 2, 3] float64 (see ppn_augment_people):
    keypoints by A in fp64 rounded once to fp32; on a flipped image column i takes column perm[i] (also `visible`,
    otherwise unchanged); a box with w > 0 and h > 0 becomes the bounds of its four transformed corners, any other
    keeps w = h = 0 around its transformed centre; size times sqrt|det A|."""
    off = np.asarray(person_off, np.int64)
    bbox = np.asarray(bbox, f64).reshape(-1, 4)
    kp = np.asarray(keypoints, f32)
    vis = np.asarray(visible, np.uint8)
    size = np.asarray(size, f64)
    A = np.asarray(A, f64).reshape(-1, 2, 3)
    bo, ko, vo, so = np.empty_like(bbox), np.empty_like(kp), np.empty_like(vis), np.empty_like(size)
    for b in range(len(off) - 1):
        a = A[b]
        rows = slice(off[b], off[b + 1])
        cols = np.asarray(perm) if flip[b] else np.arange(kp.shape[1])
        k = kp[rows][:, cols].astype(f64)
        X, Y = _apply(a, k[..., 0], k[..., 1])
        ko[rows] = np.stack([X, Y], axis=-1).astype(f32)
        vo[rows] = vis[rows][:, cols]
        for p in range(off[b], off[b + 1]):
            cx, cy, bw, bh = bbox[p]
            if bw > 0 and bh > 0:
                hw, hh = bw * 0.5, bh * 0.5
                xs, ys = (cx - hw, cx + hw), (cy - hh, cy + hh)
                X, Y = zip(*[_apply(a, xs[i & 1], ys[i >> 1]) for i in range(4)])
                lx, hx, ly, hy = X[0], X[0], Y[0], Y[0]
                for i in range(1, 4):
                    lx = X[i] if X[i] < lx else lx
                    hx = X[i] if X[i] > hx else hx
                    ly = Y[i] if Y[i] < ly else ly
                    hy = Y[i] if Y[i] > hy else hy
                bo[p] = ((lx + hx) * 0.5, (ly + hy) * 0.5, hx - lx, hy - ly)
            else:
                X, Y = _apply(a, cx, cy)
                bo[p] = (X, Y, 0.0, 0.0)
            so[p] = size[p] * math.sqrt(abs(a[0, 0] * a[1, 1] - a[0, 1] * a[1, 0]))
    return off.astype(np.int32), bo, ko, vo, so


def compose(w, h, insize, scale=1.0, theta=0.0, tx=0.0, ty=0.0, flip=False) -> np.ndarray:
    """The sampler's A = T(c_out + t insize) . R(theta) . S(scale s0) . F . T(-c_src) for one w x h source, float64,
    as a product of 3x3 homogeneous matrices (s0 = min(inW / w, inH / h), c_src = (w/2, h/2), c_out = (inW/2, inH/2))."""
    inW, inH = insize
    s0 = min(inW / w, inH / h)
    T = lambda x, y: np.array([[1, 0, x], [0, 1, y], [0, 0, 1]], f64)
    R = np.array([[math.cos(theta), -math.sin(theta), 0], [math.sin(theta), math.cos(theta), 0], [0, 0, 1]], f64)
    S = np.diag([scale * s0, scale * s0, 1.0])
    F = np.diag([-1.0 if flip else 1.0, 1.0, 1.0])
    return (T(inW / 2 + tx * inW, inH / 2 + ty * inH) @ R @ S @ F @ T(-w / 2, -h / 2))[:2]


def inverse_f32(A) -> np.ndarray:
    """M = A^-1 (2 x 3), computed in float64 and rounded once to fp32."""
    full = np.vstack([np.asarray(A, f64).reshape(2, 3), [0, 0, 1]])
    return np.linalg.inv(full)[:2].astype(f32)
