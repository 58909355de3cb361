"""The flip test's merge restated in numpy.  TEST INFRASTRUCTURE (the specification of ppn_flip_merge).

The reference has no flip test, so, as for the loss, AP and augmentation, this restatement is the specification;
DESIGN.md §15 lists its reconstruction points.  For one image, A is the head of the network input x and Bf the head
of x.flip(-1), both [C, H, W].  The merge mirrors Bf back into A's frame and averages the two:

  part mirror   p[K]: p[0] = 0, p[k] = flip_permutation(names)[k - 1] + 1   (left_* <-> right_*)
  limb mirror   q[E]: q[e] is the limb whose edge is (p[s], p[t]) for edges[e] = (s, t), in the same direction
                (both tables are inputs here; flip.part_mirror / flip.limb_mirror build them, the tests check them
                against hand-written ones)
  source plane  part group g, part k: g*K + p[k];  limb plane (e, a, b) of [E, sH, sW]: (q[e], a, sW - 1 - b)
  source cell   (i, j) reads Bf at (i, W - 1 - j)
  value         fp32, one rounding per operation: b' = 1 - b in the x group (b otherwise), out = (a + b') * 0.5,
                rounded once to the head's dtype

The cell mirror is exact only for inW == W * gridW, the window mirror only for 2 * off_w == sW - 1.
"""
from __future__ import annotations

import numpy as np

from oracle.augment import to_dtype

f32 = np.float32


def source_planes(K: int, E: int, sH: int, sW: int, p: np.ndarray, q: np.ndarray) -> np.ndarray:
    """int64 [C]: the plane of Bf that output plane c reads."""
    parts = [g * K + p[k] for g in range(6) for k in range(K)]
    limbs = [6 * K + (q[e] * sH + a) * sW + (sW - 1 - b) for e in range(E) for a in range(sH) for b in range(sW)]
    return np.asarray(parts + limbs, np.int64)


def check_geometry(g) -> None:
    """ValueError where the mirror is not exact (g: anything with K, E, inW, W, sW, ow / off_w as ppn_oracle's
    Geometry)."""
    if g.inW != g.W * g.gridW:
        raise ValueError(f"the cell mirror needs inW == W * gridW, got inW = {g.inW}, W = {g.W}, gridW = {g.gridW}")
    if 2 * g.ow != g.sW - 1:
        raise ValueError(f"the window mirror needs 2 * off_w == sW - 1, got off_w = {g.ow}, sW = {g.sW}")


def merge_values(a: np.ndarray, b: np.ndarray, is_x, dtype: str = "float32") -> np.ndarray:
    """The elementwise rule on fp32 a (the head) and b (Bf's mirrored element): b' = 1 - b where is_x, out =
    (a + b') * 0.5, each operation rounded once in fp32, the result rounded once to `dtype`."""
    a, b = np.asarray(a, f32), np.asarray(b, f32)
    with np.errstate(all="ignore"):
        bp = np.where(is_x, f32(1.0) - b, b).astype(f32)
        out = ((a + bp).astype(f32) * f32(0.5)).astype(f32)
    return to_dtype(out, dtype)


def flip_merge(A: np.ndarray, Bf: np.ndarray, g, p: np.ndarray, q: np.ndarray, dtype: str = "float32") -> np.ndarray:
    """A, Bf: [B, C, H, W] or [C, H, W], fp32 (16-bit heads widened exactly) -> the merged head, rounded to `dtype`
    ('bfloat16' as uint16 bits)."""
    check_geometry(g)
    src = source_planes(g.K, g.E, g.sH, g.sW, p, q)
    mirrored = np.asarray(Bf, f32)[..., src, :, ::-1]
    is_x = np.zeros(g.C, bool)
    is_x[2 * g.K:3 * g.K] = True
    return merge_values(A, mirrored, is_x[:, None, None], dtype)
