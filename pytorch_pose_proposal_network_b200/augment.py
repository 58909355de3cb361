"""Batch augmentation on the GPU — the reference's per-image transform (aug.py) for a whole batch.

The reference warps each image, its keypoints and boxes with imgaug inside the DataLoader workers, then converts the
image with ``ToNormalizedTensor``.  Here the workers only decode; the decoded uint8 images of a batch travel to the
device as one ragged buffer (:class:`ImageBatch`), and two launches do the rest: ``ppn_augment_images`` warps, flips
and normalises every image into ``[B, 3, inH, inW]`` (fp32, fp16 or bf16, NCHW or channels_last), and
``ppn_augment_people`` moves the annotations into the flat layout :meth:`dataset.TargetEncoder.encode_flat` takes.

    batch = ImageBatch.from_arrays(images)              # list of HWC uint8 RGB arrays, any sizes
    aug = Augmenter(cfg)                                # random affine + flip (training)
    x, flat, params = aug(batch, samples)               # samples: annotation dicts (dataset.flatten_samples)
    targets = TargetEncoder(cfg).encode_flat(*flat)

The per-image parameters are a forward affine ``A`` (float64, source pixel coordinates -> output coordinates, pixel
(row i, col j) centred at (j + 0.5, i + 0.5)), ``M = A^-1`` rounded to fp32 and a flip flag.  The kernels are exact
functions of them (DESIGN.md §14); :meth:`Augmenter.sample` draws them with torch on the device.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import NamedTuple, Optional, Sequence

import numpy as np
import torch

from . import _lib
from .config import PPNConfig, default_skeleton

IMAGENET_MEAN = (0.485, 0.456, 0.406)
IMAGENET_STD = (0.229, 0.224, 0.225)
IN_SCALE = float(np.float32(1.0 / 255.0))          # ToNormalizedTensor's /255 as one fp32 multiply
OUT_DTYPES = {torch.float32: _lib.HEAD_F32, torch.float16: _lib.HEAD_F16, torch.bfloat16: _lib.HEAD_BF16}


def flip_permutation(keypoint_names: Sequence[str]) -> np.ndarray:
    """int32 [K - 1]: on a mirrored image, part column i (part i + 1) takes column perm[i]: ``left_*`` <-> ``right_*``,
    every other part stays.  ``keypoint_names[0]`` is the instance (part 0), which has no column."""
    names = list(keypoint_names)
    perm = np.arange(len(names) - 1, dtype=np.int32)
    for i, n in enumerate(names[1:]):
        for a, b in (("left_", "right_"), ("right_", "left_")):
            if n.startswith(a):
                partner = b + n[len(a):]
                if partner not in names[1:]:
                    raise ValueError(f"part {n!r} has no mirror part {partner!r}")
                perm[i] = names.index(partner) - 1
    return perm


def compose(src_w, src_h, insize, scale, theta, tx, ty, flip) -> torch.Tensor:
    """A = T(c_out + t * insize) . R(theta) . S(scale * s0) . F . T(-c_src), float64 [B, 2, 3].
    s0 = min(inW / w, inH / h) letterboxes the source into the output; c_src = (w / 2, h / 2), c_out = (inW / 2,
    inH / 2); F mirrors x where `flip` is true; theta in radians; t = (tx, ty) in fractions of the output size."""
    inW, inH = float(insize[0]), float(insize[1])
    w, h = src_w.to(torch.float64), src_h.to(torch.float64)
    k = scale.to(torch.float64) * torch.minimum(inW / w, inH / h)
    c, s = torch.cos(theta.to(torch.float64)), torch.sin(theta.to(torch.float64))
    f = 1.0 - 2.0 * flip.to(torch.float64)
    a00, a01, a10, a11 = c * k * f, -s * k, s * k * f, c * k
    a02 = (inW / 2 + tx.to(torch.float64) * inW) - (a00 * (w / 2) + a01 * (h / 2))
    a12 = (inH / 2 + ty.to(torch.float64) * inH) - (a10 * (w / 2) + a11 * (h / 2))
    return torch.stack([a00, a01, a02, a10, a11, a12], dim=-1).reshape(-1, 2, 3)


def invert(A: torch.Tensor) -> torch.Tensor:
    """The inverse affine of each [2, 3] matrix, float64."""
    a00, a01, a02, a10, a11, a12 = A.reshape(-1, 6).unbind(-1)
    det = a00 * a11 - a01 * a10
    i00, i01, i10, i11 = a11 / det, -a01 / det, -a10 / det, a00 / det
    return torch.stack([i00, i01, -(i00 * a02 + i01 * a12), i10, i11, -(i10 * a02 + i11 * a12)], dim=-1).reshape(-1, 2, 3)


class AugParams(NamedTuple):
    A: torch.Tensor         # float64 [B, 2, 3] source -> output (annotations)
    M: torch.Tensor         # fp32 [B, 2, 3] output pixel centre -> source (images)
    flip: torch.Tensor      # uint8 [B]


def params_from(A: torch.Tensor, flip: torch.Tensor) -> AugParams:
    return AugParams(A.contiguous(), invert(A).to(torch.float32).contiguous(), flip.to(torch.uint8).contiguous())


def draw(hw: torch.Tensor, insize, scale=(0.75, 1.25), rotation=30.0, shift=0.1, p_flip=0.5, generator=None) -> AugParams:
    """Random parameters for images of sizes hw (int [B, 2] (h, w)), drawn on hw's device: scale uniform in `scale`,
    rotation uniform in +-`rotation` degrees, shift uniform in +-`shift` per axis, a mirror with probability p_flip."""
    u = torch.rand(hw.shape[0], 5, dtype=torch.float64, device=hw.device, generator=generator)
    s = scale[0] + (scale[1] - scale[0]) * u[:, 0]
    theta = (2.0 * u[:, 1] - 1.0) * math.radians(rotation)
    tx, ty = (2.0 * u[:, 2] - 1.0) * shift, (2.0 * u[:, 3] - 1.0) * shift
    flip = u[:, 4] < p_flip
    return params_from(compose(hw[:, 1], hw[:, 0], insize, s, theta, tx, ty, flip), flip)


class ImageBatch:
    """A ragged batch of HWC uint8 RGB images in one device buffer: image b is ``hw[b]`` = (h, w) at byte
    ``offset[b]`` of ``pixels``.  ``offset_host`` / ``hw_host`` are host copies of the same table (the C entry
    checks them without reading the device).  ``pixels`` must be readable up to the next 16-byte boundary after the
    last image byte (:meth:`from_arrays` pads it)."""

    def __init__(self, pixels: torch.Tensor, offset: torch.Tensor, hw: torch.Tensor, offset_host, hw_host, host=None):
        self.pixels, self.offset, self.hw = pixels, offset, hw
        self.offset_host = np.ascontiguousarray(offset_host, np.int64)
        self.hw_host = np.ascontiguousarray(hw_host, np.int32).reshape(-1, 2)
        self._host = host                     # the pinned staging buffer of from_arrays, alive until the copy is done
        B = self.offset_host.shape[0]
        if B < 1 or self.hw_host.shape[0] != B:
            raise ValueError(f"need a table of B >= 1 images, got {B} offsets and {self.hw_host.shape[0]} sizes")
        if pixels.dtype != torch.uint8 or pixels.dim() != 1 or offset.dtype != torch.int64 or hw.dtype != torch.int32:
            raise ValueError("pixels must be a flat uint8 tensor, offset int64 [B], hw int32 [B, 2]")
        if tuple(offset.shape) != (B,) or tuple(hw.shape) != (B, 2):
            raise ValueError(f"offset must be [{B}] and hw [{B}, 2], got {tuple(offset.shape)} and {tuple(hw.shape)}")

    @property
    def B(self) -> int:
        return int(self.offset_host.shape[0])

    @property
    def device(self) -> torch.device:
        return self.pixels.device

    @classmethod
    def from_arrays(cls, arrays: Sequence[np.ndarray], device=None) -> "ImageBatch":
        """Pack decoded images ([h, w, 3] uint8 each) and their table into one pinned host buffer and upload it with
        one asynchronous copy on the current stream."""
        arrays = [np.asarray(a) for a in arrays]
        if not arrays:
            raise ValueError("an ImageBatch needs at least one image")
        for a in arrays:
            if a.dtype != np.uint8 or a.ndim != 3 or a.shape[2] != 3:
                raise ValueError(f"images must be [h, w, 3] uint8 arrays, got {a.dtype} {a.shape}")
        B = len(arrays)
        hw = np.asarray([a.shape[:2] for a in arrays], np.int32).reshape(B, 2)
        nbytes = np.asarray([a.nbytes for a in arrays], np.int64)
        offset = np.concatenate([[0], np.cumsum(nbytes)[:-1]]).astype(np.int64)
        table = 16 * B                                         # offsets then (h, w) pairs: 16 bytes per image
        total = table + ((int(nbytes.sum()) + 15) & ~15)
        host = torch.empty(total, dtype=torch.uint8, pin_memory=True)
        buf = host.numpy()
        buf[:8 * B] = offset.view(np.uint8)
        buf[8 * B:table] = hw.reshape(-1).view(np.uint8)
        for a, o in zip(arrays, offset):
            buf[table + o:table + o + a.nbytes] = np.ascontiguousarray(a).reshape(-1)
        buf[table + int(nbytes.sum()):] = 0
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        gpu = torch.empty(total, dtype=torch.uint8, device=dev)
        gpu.copy_(host, non_blocking=True)
        return cls(gpu[table:], gpu[:8 * B].view(torch.int64), gpu[8 * B:table].view(torch.int32).view(B, 2),
                   offset, hw, host=host)

    def c_struct(self) -> _lib.PPNImageBatch:
        return _lib.PPNImageBatch(self.pixels.data_ptr(), self.offset.data_ptr(), self.hw.data_ptr(),
                                  self.offset_host.ctypes.data, self.hw_host.ctypes.data,
                                  self.pixels.numel(), self.B)


def collate(items):
    """DataLoader ``collate_fn`` for workers that return (decoded image array, annotation dict): the two lists as
    they are, for :meth:`ImageBatch.from_arrays` and :meth:`Augmenter.__call__`."""
    items = list(items)
    return [it[0] for it in items], [it[1] for it in items]


class Augmenter:
    """Random affine + flip + normalisation of an :class:`ImageBatch` and its annotations, on the GPU.

    scale: (lo, hi) of the uniform zoom on top of the letterbox fit; rotation: degrees (uniform in +-);
    shift: fraction of the output size per axis (uniform in +-); p_flip: probability of a horizontal mirror.
    out = (pixel * in_scale - mean) / std per channel, `fill` (uint8 units) outside the source.  ``in_scale = 1``
    reproduces rt_test.py's ImageNet statistics applied to 0-255 pixels.  ``keypoint_names`` (K names, the instance
    first) defines the left/right mirror of the parts; config.py's two skeletons are the default."""

    def __init__(self, cfg: PPNConfig, keypoint_names=None, scale=(0.75, 1.25), rotation=30.0, shift=0.1, p_flip=0.5,
                 mean=IMAGENET_MEAN, std=IMAGENET_STD, in_scale=IN_SCALE, fill=(0.0, 0.0, 0.0), dtype=torch.float32,
                 channels_last=False, device=None):
        if dtype not in OUT_DTYPES:
            raise ValueError(f"dtype must be torch.float32, float16 or bfloat16, got {dtype}")
        keypoint_names, _ = default_skeleton(cfg, keypoint_names, need=("names",))
        if len(keypoint_names) != cfg.K:
            raise ValueError(f"{len(keypoint_names)} keypoint names for a configuration with K = {cfg.K}")
        lo, hi = (float(v) for v in scale)
        if not 0 < lo <= hi or not rotation >= 0 or not shift >= 0 or not 0 <= p_flip <= 1:
            raise ValueError("need 0 < scale[0] <= scale[1], rotation >= 0, shift >= 0 and 0 <= p_flip <= 1")
        for name, v in (("mean", mean), ("std", std), ("fill", fill)):
            if len(v) != 3:
                raise ValueError(f"{name} needs one value per channel, got {v}")
        if not all(s > 0 for s in std):
            raise ValueError(f"std must be positive, got {std}")
        self.cfg, self.dtype, self.channels_last = cfg, dtype, bool(channels_last)
        self.scale, self.rotation, self.shift, self.p_flip = (lo, hi), float(rotation), float(shift), float(p_flip)
        self.perm = flip_permutation(keypoint_names)
        self.norm = _lib.PPNImageNorm((C.c_float * 3)(*mean), (C.c_float * 3)(*std), (C.c_float * 3)(*fill),
                                      float(in_scale))
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.lib = _lib.lib()

    # ---- parameters ------------------------------------------------------------------------------------------- #
    def sample(self, batch: ImageBatch, generator: Optional[torch.Generator] = None) -> AugParams:
        """Random parameters for the batch's source sizes, drawn on the device from `generator` (a generator of
        that device; torch's default one if None).  No host synchronisation."""
        self._check_batch(batch)
        return draw(batch.hw, self.cfg.insize, self.scale, self.rotation, self.shift, self.p_flip, generator)

    def fit(self, batch: ImageBatch) -> AugParams:
        """The deterministic validation transform: the letterbox fit alone (scale 1, no rotation, shift or flip)."""
        self._check_batch(batch)
        zero = torch.zeros(batch.B, dtype=torch.float64, device=batch.device)
        A = compose(batch.hw[:, 1], batch.hw[:, 0], self.cfg.insize, zero + 1.0, zero, zero, zero, zero)
        return params_from(A, zero.to(torch.uint8))

    # ---- the two launches ------------------------------------------------------------------------------------- #
    def images(self, batch: ImageBatch, params: AugParams, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """[B, 3, inH, inW] of `dtype` (channels_last memory if so configured), asynchronous on the current stream."""
        self._check_batch(batch)
        B, inW, inH = batch.B, self.cfg.inW, self.cfg.inH
        M = params.M
        if M.dtype != torch.float32 or tuple(M.shape) != (B, 2, 3) or M.device != self.device or not M.is_contiguous():
            raise ValueError(f"params.M must be a contiguous float32 [{B}, 2, 3] tensor on {self.device}")
        fmt = torch.channels_last if self.channels_last else torch.contiguous_format
        if out is None:
            out = torch.empty(B, 3, inH, inW, dtype=self.dtype, device=self.device, memory_format=fmt)
        elif (out.dtype != self.dtype or tuple(out.shape) != (B, 3, inH, inW) or out.device != self.device
              or not out.is_contiguous(memory_format=fmt)):
            raise ValueError(f"out must be a {self.dtype} [{B}, 3, {inH}, {inW}] tensor on {self.device} in "
                             f"{'channels_last' if self.channels_last else 'contiguous'} memory format")
        layout = _lib.LAYOUT_NHWC if self.channels_last else _lib.LAYOUT_NCHW
        stream = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ppn_augment_images(C.byref(batch.c_struct()), M.data_ptr(), C.byref(self.norm), inH, inW,
                                                   OUT_DTYPES[self.dtype], layout, out.data_ptr(),
                                                   out.numel() * out.element_size(), stream), "ppn_augment_images")
        return out

    def people(self, person_off, bbox, keypoints, visible, size, params: AugParams):
        """The flat annotations (int32 [B+1], float64 [n,4], fp32 [n,K-1,2], uint8 [n,K-1], float64 [n], device
        tensors) moved by the batch's parameters: the five arrays ``TargetEncoder.encode_flat`` takes."""
        J = self.cfg.K - 1
        B = int(person_off.numel()) - 1
        n = int(bbox.shape[0])
        want = ((person_off, torch.int32, (B + 1,)), (bbox, torch.float64, (n, 4)), (keypoints, torch.float32, (n, J, 2)),
                (visible, torch.uint8, (n, J)), (size, torch.float64, (n,)),
                (params.A, torch.float64, (B, 2, 3)), (params.flip, torch.uint8, (B,)))
        for t, dt, shp in want:
            if t.dtype != dt or tuple(t.shape) != shp or t.device != self.device or not t.is_contiguous():
                raise ValueError(f"expected a contiguous {dt} tensor of shape {shp} on {self.device}, got {t.dtype} "
                                 f"{tuple(t.shape)} on {t.device}")
        if B < 1:
            raise ValueError("person_off needs B + 1 >= 2 entries")
        out = (torch.empty_like(bbox), torch.empty_like(keypoints), torch.empty_like(visible), torch.empty_like(size))
        src = _lib.PPNPeople(person_off.data_ptr(), bbox.data_ptr(), keypoints.data_ptr(), visible.data_ptr(), size.data_ptr())
        dst = _lib.PPNPeopleOut(*[t.data_ptr() for t in out])
        stream = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ppn_augment_people(C.byref(src), B, n, self.cfg.K, params.A.data_ptr(), params.flip.data_ptr(),
                                                   self.perm.ctypes.data_as(_lib.i32p), C.byref(dst), stream),
                       "ppn_augment_people")
        return (person_off,) + out

    def __call__(self, batch: ImageBatch, samples_or_flat, generator: Optional[torch.Generator] = None):
        """sample + images + people: -> (images, the five flat annotation arrays, params).  `samples_or_flat`: the
        annotation dicts of the batch's images (see dataset.flatten_samples) or the five flat device tensors."""
        if len(samples_or_flat) == 5 and all(isinstance(t, torch.Tensor) for t in samples_or_flat):
            flat = tuple(samples_or_flat)
        else:
            from .dataset import flatten_samples
            if len(samples_or_flat) != batch.B:
                raise ValueError(f"{len(samples_or_flat)} annotation dicts for {batch.B} images")
            flat = tuple(torch.from_numpy(a).to(self.device, non_blocking=True)
                         for a in flatten_samples(samples_or_flat, self.cfg.K))
        params = self.sample(batch, generator)
        return self.images(batch, params), self.people(*flat, params), params

    def _check_batch(self, batch: ImageBatch):
        if batch.device != self.device:
            raise ValueError(f"the batch is on {batch.device}, the augmenter on {self.device}")
