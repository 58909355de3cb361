"""The flip test on the GPU: merge a head with the mirrored head of its horizontally flipped input.

The standard test-time step of a bottom-up pose estimator: the image and its mirror go through the network, the
mirror's head is mirrored back and averaged with the first head, and the parse reads the average.  For a PPN head
that is more than a ``torch.flip``: the part channels swap ``left_*`` <-> ``right_*``, the x offset inside a cell
becomes ``1 - x``, each limb's channels move to the mirrored limb, and inside each limb's displacement window the
columns reverse.  ``ppn_flip_merge`` does all of it in one pass over the two heads (DESIGN.md §15).

    fm = FlipMerge(cfg)                                  # part / limb mirror tables of cfg's skeleton
    head2 = model(torch.cat([x, x.flip(-1)]))            # one network call on both views
    head = fm(head2[:B], head2[B:], out=head2[:B])       # in place into the first half (or out=None: a new tensor)
    packed = parser.parse(head)                          # or parser.parse_proposals(head)
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from .augment import OUT_DTYPES as HEAD_DTYPES, flip_permutation
from .config import PPNConfig, default_skeleton
from .parser import _CConfig


def part_mirror(keypoint_names: Sequence[str]) -> np.ndarray:
    """int32 [K]: part k of the mirrored image is part p[k] of the image; p[0] = 0 (the instance)."""
    return np.concatenate([[0], flip_permutation(keypoint_names) + 1]).astype(np.int32)


def limb_mirror(p: np.ndarray, edges) -> np.ndarray:
    """int32 [E]: for edges[e] = (s, t), the limb q[e] whose edge is (p[s], p[t]).  ValueError where the skeleton has
    no such limb, or has it only in the other direction: then the skeleton has no flip test."""
    e = [tuple(int(v) for v in st) for st in np.asarray(edges, np.int64).reshape(-1, 2)]
    index = {st: i for i, st in enumerate(e)}
    q = np.zeros(len(e), np.int32)
    for i, (s, t) in enumerate(e):
        m = (int(p[s]), int(p[t]))
        if m not in index:
            how = "only reversed" if m[::-1] in index else "missing"
            raise ValueError(f"limb {i} {(s, t)} has no mirror limb {m} ({how}): the skeleton has no flip test")
        q[i] = index[m]
    if not np.array_equal(q[q], np.arange(len(e))):
        raise ValueError("the limb mirror is not an involution (a limb listed twice?)")
    return q


class FlipMerge:
    """``fm(head, head_flipped, out=None)``: ``head`` is the network's head on the input ``x``, ``head_flipped`` its
    head on ``x.flip(-1)`` (the exact pixel mirror, in either memory format), both contiguous ``[B, C, H, W]`` fp32,
    fp16 or bf16 of one dtype on the object's device.  Returns the merged head in that dtype, asynchronously on the
    current stream; ``out`` may be ``head``.  ``keypoint_names`` (K names, the instance first) and ``edges`` ([E][2]
    part ids) define the mirror; config.py's two skeletons are the defaults."""

    def __init__(self, cfg: PPNConfig, keypoint_names=None, edges=None, device=None):
        keypoint_names, edges = default_skeleton(cfg, keypoint_names, edges)
        if len(keypoint_names) != cfg.K:
            raise ValueError(f"{len(keypoint_names)} keypoint names for a configuration with K = {cfg.K}")
        if np.asarray(edges).reshape(-1, 2).shape[0] != cfg.E:
            raise ValueError(f"{np.asarray(edges).reshape(-1, 2).shape[0]} edges for a configuration with E = {cfg.E}")
        gW, _ = cfg.gridsize
        if cfg.inW != cfg.W * gW:
            raise ValueError(f"the flip test needs inW == W * gridW (an exact cell mirror), got inW = {cfg.inW}, "
                             f"W = {cfg.W}, gridW = {gW}")
        if 2 * cfg.off_w != cfg.sW - 1:
            raise ValueError(f"the flip test needs 2 * off_w == sW - 1 (an exact window mirror), got off_w = "
                             f"{cfg.off_w}, sW = {cfg.sW}")
        self.cfg = cfg
        self.part_mirror = part_mirror(keypoint_names)
        self.limb_mirror = limb_mirror(self.part_mirror, edges)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.c = _CConfig(cfg)
        self.lib = _lib.lib()

    def __call__(self, head: torch.Tensor, head_flipped: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        cfg = self.cfg
        if head.dtype not in HEAD_DTYPES:
            raise ValueError(f"the head must be float32, float16 or bfloat16, got {head.dtype}")
        B = int(head.shape[0]) if head.dim() == 4 else 0
        want = (B, cfg.C, cfg.H, cfg.W)
        if out is None:
            out = torch.empty_like(head, memory_format=torch.contiguous_format)
        for name, t in (("head", head), ("head_flipped", head_flipped), ("out", out)):
            if (t.dtype != head.dtype or tuple(t.shape) != want or t.device != self.device or not t.is_contiguous()):
                raise ValueError(f"{name} must be a contiguous {head.dtype} [B, {cfg.C}, {cfg.H}, {cfg.W}] tensor with "
                                 f"the head's B on {self.device}, got {t.dtype} {tuple(t.shape)} on {t.device}")
        if B < 1:
            raise ValueError("the heads need B >= 1 images")
        shape = self.c.shape(B, HEAD_DTYPES[head.dtype])
        stream = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ppn_flip_merge(head.data_ptr(), head_flipped.data_ptr(), out.data_ptr(), C.byref(shape),
                                               self.part_mirror.ctypes.data_as(_lib.i32p),
                                               self.limb_mirror.ctypes.data_as(_lib.i32p), stream),
                       "ppn_flip_merge")
        return out
