"""Training targets on the GPU — the encoder half of the reference's ``dataset.py``.

The reference builds its loss targets inside ``KeypointsDataset.__getitem__`` (dataset.py:89-198):
per image ~70 lines of Python over numpy grids, the O(E*H*W) window loop of dataset.py:155-168 among
them, run by DataLoader workers, then stacked by ``CustomBatch`` (dataset.py:233-246).  Here the whole
batch is encoded by one kernel launch (``ppn_encode_targets``): the annotations of the batch — a few
KB — go to the device, the grids (whose two limb tensors are as large as the head's limb block) are
written there once, where the loss reads them.  Same arithmetic, same overwrite order, same ten
tensors; checked bit for bit against outputs of the reference's own ``__getitem__``
(``tests/golden/encode``).

    enc = TargetEncoder(cfg)                       # geometry + EDGES of a PPNConfig
    batch = enc.encode(samples)                    # samples: what the reference's transforms return
    batch.delta, batch.weight, batch.weight_ij, batch.tx, ... batch.te      # like CustomBatch, on the GPU

For mixed-precision training, ``TargetEncoder(cfg, limb_dtype=torch.float16)`` (or bfloat16) writes the two limb
tensors — most of the bytes — in 16 bits: te in {0, 1} is exact, weight_ij stores 0.0005 rounded to the type
(fp16 0.000500202..., bf16 0.000499725...).  The eight [B, K, H, W] grids stay fp32.

Image loading and augmentation (aug.py) stay where they are: they are not on this path.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from .config import PPNConfig
from .parser import _CConfig


class TargetBatch:
    """The reference's ``CustomBatch`` (dataset.py:233-246) without the image: ten device tensors."""

    __slots__ = _lib.TARGET_NAMES

    def __init__(self, **tensors):
        for name in _lib.TARGET_NAMES:
            setattr(self, name, tensors[name])

    def as_list(self):
        """In the order ``__getitem__`` returns them after the image (dataset.py:198)."""
        return [getattr(self, n) for n in _lib.TARGET_NAMES]


def flatten_samples(samples: Sequence[dict], K: int):
    """Samples as the reference's transform pipeline returns them (aug.py:138-160: 'keypoints' fp32
    [n, K-1, 2], 'bbox' float64 [n, 4] (cx, cy, w, h), 'is_visible' n arrays of K-1 bools, 'size' n
    floats) -> flat host arrays (person_off, bbox, keypoints, visible, size).  People are what the
    reference's encoder loop zips over (dataset.py:108): min over the four lists' lengths."""
    offs, bbs, kps, vis, sizes = [0], [], [], [], []
    for s in samples:
        bb = np.asarray(s["bbox"], np.float64).reshape(-1, 4)
        kp = np.asarray(s["keypoints"], np.float32).reshape(-1, K - 1, 2)
        n = min(len(bb), len(kp), len(s["is_visible"]), len(s["size"]))
        bbs.append(bb[:n])
        kps.append(kp[:n])
        vis.append(np.asarray([np.asarray(v, bool) for v in s["is_visible"][:n]], bool).reshape(n, K - 1))
        sizes.append(np.asarray(s["size"][:n], np.float64).reshape(n))
        offs.append(offs[-1] + n)
    cat = lambda parts, shape, dt: (np.concatenate(parts).astype(dt) if parts else np.zeros(shape, dt))
    return (np.asarray(offs, np.int32), cat(bbs, (0, 4), np.float64), cat(kps, (0, K - 1, 2), np.float32),
            cat(vis, (0, K - 1), np.uint8), cat(sizes, (0,), np.float64))


LIMB_DTYPES = {torch.float32: _lib.HEAD_F32, torch.float16: _lib.HEAD_F16, torch.bfloat16: _lib.HEAD_BF16}


class TargetEncoder:
    """Batched GPU replacement of the encode half of ``KeypointsDataset.__getitem__``.  ``limb_dtype``: the
    element type of te and weight_ij (float32, float16 or bfloat16)."""

    def __init__(self, cfg: PPNConfig, edges=None, device=None, limb_dtype=torch.float32):
        if not torch.cuda.is_available():
            raise RuntimeError("TargetEncoder needs a CUDA device: there is no CPU path")
        if limb_dtype not in LIMB_DTYPES:
            raise ValueError(f"limb_dtype must be torch.float32, float16 or bfloat16, got {limb_dtype}")
        self.cfg = cfg
        self.limb_dtype = limb_dtype
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.lib = _lib.lib()
        self.c = _CConfig(cfg)
        if edges is None:                                      # the skeletons config.py knows (config.py:65 EDGES)
            from . import config as pcfg
            edges = {(18, 17): pcfg.EDGES, (16, 15): pcfg.EDGES_16}.get((cfg.K, cfg.E))
            if edges is None:
                raise ValueError("pass `edges` ([E][2] part ids) for a skeleton that is not one of config.py's")
        e = np.asarray(edges, np.int32).reshape(-1, 2)
        if e.shape[0] != cfg.E:
            raise ValueError(f"{e.shape[0]} edges for a configuration with E = {cfg.E}")
        self.edges = np.ascontiguousarray(e)

    def alloc(self, B: int) -> TargetBatch:
        cfg = self.cfg
        small = lambda: torch.empty(B, cfg.K, cfg.H, cfg.W, dtype=torch.float32, device=self.device)
        big = lambda: torch.empty(B, cfg.E, cfg.sH, cfg.sW, cfg.H, cfg.W, dtype=self.limb_dtype, device=self.device)
        return TargetBatch(**{n: (big() if n in ("weight_ij", "te") else small()) for n in _lib.TARGET_NAMES})

    @staticmethod
    def check_offsets(person_off, n: int) -> None:
        """person_off must be the running count of people per image: starts at 0, never decreases, ends at n.
        (The kernel trusts it: a bad table reads outside the annotation arrays.)"""
        off = np.asarray(person_off.cpu() if isinstance(person_off, torch.Tensor) else person_off, np.int64)
        if off.ndim != 1 or off.size < 1 or off[0] != 0 or off[-1] != n or (np.diff(off) < 0).any():
            raise ValueError(f"person_off must rise from 0 to the number of people ({n}) without decreasing")

    def encode_flat(self, person_off, bbox, keypoints, visible, size, out: Optional[TargetBatch] = None,
                    validate: bool = False) -> TargetBatch:
        """Device tensors in (int32 [B+1], float64 [n,4], fp32 [n,K-1,2], uint8 [n,K-1], float64 [n]),
        targets out; asynchronous on torch's current stream.  ``validate`` checks `person_off` first (it copies
        the table to the host, i.e. synchronises; :meth:`encode` checks its host copy for free)."""
        B = int(person_off.numel()) - 1
        n = int(bbox.shape[0])
        if validate:
            self.check_offsets(person_off, n)
        want = ((person_off, torch.int32, (B + 1,)), (bbox, torch.float64, (n, 4)), (keypoints, torch.float32, (n, self.cfg.K - 1, 2)),
                (visible, torch.uint8, (n, self.cfg.K - 1)), (size, torch.float64, (n,)))
        for t, dt, shp in want:
            if t.dtype != dt or tuple(t.shape) != shp or t.device != self.device or not t.is_contiguous():
                raise ValueError(f"expected a contiguous {dt} tensor of shape {shp} on {self.device}, got {t.dtype} {tuple(t.shape)} on {t.device}")
        if out is None:
            out = self.alloc(B)
        elif out.te.dtype != self.limb_dtype or out.weight_ij.dtype != self.limb_dtype:
            raise ValueError(f"out.te and out.weight_ij must be {self.limb_dtype}, got {out.te.dtype} and {out.weight_ij.dtype}")
        people = _lib.PPNPeople(person_off.data_ptr(), bbox.data_ptr(), keypoints.data_ptr(), visible.data_ptr(), size.data_ptr())
        targets = _lib.PPNTargets(*[getattr(out, nme).data_ptr() for nme in _lib.TARGET_NAMES])
        shape = self.c.shape(B)
        stream = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        edges = self.edges.ctypes.data_as(_lib.i32p)
        with torch.cuda.device(self.device):
            if self.limb_dtype == torch.float32:
                _lib.check(self.lib.ppn_encode_targets(C.byref(people), C.byref(shape), edges, C.byref(targets), stream),
                           "ppn_encode_targets")
            else:
                _lib.check(self.lib.ppn_encode_targets_opt(C.byref(people), C.byref(shape), edges, C.byref(targets),
                                                           LIMB_DTYPES[self.limb_dtype], stream),
                           "ppn_encode_targets_opt")
        return out

    def encode(self, samples: Sequence[dict], out: Optional[TargetBatch] = None) -> TargetBatch:
        """samples: the dicts the reference's transforms return (see :func:`flatten_samples`)."""
        flat = flatten_samples(samples, self.cfg.K)
        self.check_offsets(flat[0], int(flat[1].shape[0]))
        dev = [torch.from_numpy(a).to(self.device, non_blocking=True) for a in flat]
        return self.encode_flat(*dev, out=out)
