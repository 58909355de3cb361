"""Prediction records for the reference's AP evaluation, built from the packed GPU result.

``datatest.evaluation`` (/root/reference/datatest.py:278-369) first turns every image's
``(humans, scores)`` into an MPII-style frame ``{"image": [fname], "annorect": [...]}``
(datatest.py:298-328) — one dict per person with the root box, the root score and, for each of the
K-1 joints, the centre of its box and its score (zeros when absent) — and then hands the frames to
the poseval fork.  :func:`pred_frame` builds exactly that frame from :class:`..parser.PackedHumans`
and the centres computed on the GPU (``PoseParser.part_centres`` -> ``ppn_part_centres``), without
going through per-human dicts.

The scoring of those frames -- the poseval fork's ``assignGTmulti`` and ``computeMetrics`` -- runs on the GPU as
well: :class:`APEvaluator` reads the packed result and the ground truth on the device and returns AP, precision and
recall per joint without building any frame (``ppn_ap_match`` / ``ppn_ap_finalize``, DESIGN.md §12).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np
import torch

from . import _lib


def pred_frame(fname, packed_np, centres_np, b: int):
    """packed_np: ``PackedHumans.numpy()``; centres_np: ``part_centres(...).cpu().numpy()``.

    Value types follow the reference: numpy fp32 scalars for present parts, Python ints 0 for
    absent ones, joint ids ``num - 1``."""
    n = int(packed_np["count"][b])
    cell, score, box = packed_np["part_cell"][b], packed_np["part_score"][b], packed_np["part_box"][b]
    K = cell.shape[1]
    rects = []
    for i in range(n):
        y1, x1, y2, x2 = box[i, 0]
        pp = {"x1": [x1], "y1": [y1], "x2": [x2], "y2": [y2], "score": [score[i, 0]], "annopoints": [{"point": []}]}
        points = pp["annopoints"][0]["point"]
        for num in range(1, K):
            if cell[i, num] >= 0:
                y, x, s = centres_np[b, i, num, 0], centres_np[b, i, num, 1], score[i, num]
            else:
                y, x, s = 0, 0, 0
            points.append({"id": [num - 1], "x": [x], "y": [y], "score": [s]})
        rects.append(pp)
    return {"image": [fname], "annorect": rects}


def pred_frames(fnames, packed, centres):
    """One frame per image of the batch, ready for ``eval_helpers.load_data`` (datatest.py:350)."""
    packed_np = packed.numpy()
    centres_np = centres.cpu().numpy() if hasattr(centres, "cpu") else np.asarray(centres)
    return [pred_frame(f, packed_np, centres_np, b) for b, f in enumerate(fnames)]


# ---- scoring: multi-person pose AP on the GPU ----------------------------------------------------------------------
def _first(v):
    return v[0] if isinstance(v, (list, tuple, np.ndarray)) else v


def gt_from_frames(frames, n_joints: int):
    """MPII / poseval-style GT frames -> flat host arrays (person_off int32 [B+1], head_box float64 [n, 4] (x1, y1,
    x2, y2), joint_xy float64 [n, J, 2], joint_valid uint8 [n, J]), what :meth:`APEvaluator.update_flat` takes.

    Every ``annorect`` is one person.  Its joints are the points of ``annopoints[0]["point"]`` with ids below J, the
    first point of each id (poseval's ``getPointGTbyID``); a rect without ``annopoints`` has no joint, so it can never
    be matched, as in poseval."""
    J = int(n_joints)
    offs, boxes, xy, valid = [0], [], [], []
    for fr in frames:
        rects = fr["annorect"]
        for r in rects:
            boxes.append([float(_first(r[k])) for k in ("x1", "y1", "x2", "y2")])
            p_xy = np.zeros((J, 2), np.float64)
            p_ok = np.zeros(J, np.uint8)
            pts = r["annopoints"][0]["point"] if len(r.get("annopoints") or []) > 0 else []
            for p in pts:
                if p["id"] is None:
                    continue
                j = int(_first(p["id"]))
                if 0 <= j < J and not p_ok[j]:
                    p_xy[j] = (float(_first(p["x"])), float(_first(p["y"])))
                    p_ok[j] = 1
            xy.append(p_xy)
            valid.append(p_ok)
        offs.append(offs[-1] + len(rects))
    n = len(boxes)
    return (np.asarray(offs, np.int32), np.asarray(boxes, np.float64).reshape(n, 4),
            np.asarray(xy, np.float64).reshape(n, J, 2), np.asarray(valid, np.uint8).reshape(n, J))


class APEvaluator:
    """AP, precision and recall per joint over a validation pass, in percent: what the poseval fork's
    ``assignGTmulti`` + ``computeMetrics`` return for the frames :func:`pred_frames` builds (DESIGN.md §12).

        ev = APEvaluator(cfg)                          # J = cfg.K - 1 joints, PCKh 0.5, head size 0.6 * diagonal
        for images, gt_frames in val_loader:
            ev.update(parser.parse(model(images)), gt_frames)
        res = ev.compute()                             # {"ap", "precision", "recall"}: float64 [J + 1], last = mean

    ``update`` / ``update_flat`` run the per-image matching (``ppn_ap_match``, one CTA per image) on torch's current
    stream and keep its small per-slot result on the device, so the parser may reuse its output buffers for the next
    batch.  ``compute`` ranks the entries of the whole pass and scores them (``ppn_ap_finalize``) with one host
    synchronisation.  Images are appended in update order; the ranking of equal scores depends on it."""

    def __init__(self, cfg, n_joints: Optional[int] = None, dist_thresh: float = 0.5, head_scale: float = 0.6,
                 device=None):
        J = cfg.K - 1 if n_joints is None else int(n_joints)
        if not 1 <= J <= _lib.AP_MAX_JOINTS:
            raise ValueError(f"n_joints must be in [1, {_lib.AP_MAX_JOINTS}], got {J}")
        if not (dist_thresh > 0 and head_scale > 0):
            raise ValueError("dist_thresh and head_scale must be positive")
        if not torch.cuda.is_available():
            raise RuntimeError("APEvaluator needs a CUDA device: there is no CPU path")
        self.cfg, self.J = cfg, J
        self.lib = _lib.lib()
        self.params = _lib.PPNAPParams(J, float(dist_thresh), float(head_scale))
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.reset()

    def reset(self) -> None:
        self._batches = []            # per update: (B, R, score, label, used, flags, n_gt) on the device

    @property
    def n_images(self) -> int:
        return sum(b[0] for b in self._batches)

    def _check_packed(self, packed) -> int:
        if packed.count.device != self.device:
            raise ValueError(f"packed result must be on {self.device} (PoseParser.parse), not {packed.count.device}")
        if packed.part_cell.shape[2] != self.cfg.K:
            raise ValueError(f"packed result has {packed.part_cell.shape[2]} parts, the configuration {self.cfg.K}")
        return int(packed.count.shape[0])

    def update(self, packed, gt_frames) -> None:
        """``packed``: device :class:`..parser.PackedHumans` of B images; ``gt_frames``: their B GT frames."""
        B = self._check_packed(packed)
        if len(gt_frames) != B:
            raise ValueError(f"{len(gt_frames)} GT frames for {B} images")
        flat = gt_from_frames(gt_frames, self.J)
        if B and int(np.diff(flat[0]).max()) > _lib.AP_MAX_GT:
            raise ValueError(f"an image has more than {_lib.AP_MAX_GT} GT people")
        self.update_flat(packed, *[torch.from_numpy(a).to(self.device) for a in flat])

    def update_flat(self, packed, person_off, head_box, joint_xy, joint_valid) -> None:
        """GT as device tensors: person_off int32 [B+1], head_box float64 [n, 4] (x1, y1, x2, y2), joint_xy float64
        [n, J, 2], joint_valid uint8 or bool [n, J].  Asynchronous: never synchronises the host."""
        B = self._check_packed(packed)
        n, J = int(head_box.shape[0]), self.J
        want = ((person_off, (torch.int32,), (B + 1,)), (head_box, (torch.float64,), (n, 4)),
                (joint_xy, (torch.float64,), (n, J, 2)), (joint_valid, (torch.uint8, torch.bool), (n, J)))
        for t, dts, shp in want:
            if t.dtype not in dts or tuple(t.shape) != shp or t.device != self.device or not t.is_contiguous():
                raise ValueError(f"expected a contiguous {dts[0]} tensor of shape {shp} on {self.device}, "
                                 f"got {t.dtype} {tuple(t.shape)} on {t.device}")
        R = packed.R
        kw = dict(device=self.device)
        out = (torch.empty(B, R, J, dtype=torch.float32, **kw), torch.empty(B, R, J, dtype=torch.uint8, **kw),
               torch.empty(B, dtype=torch.int32, **kw), torch.empty(B, dtype=torch.int32, **kw),
               torch.empty(B, J, dtype=torch.int32, **kw))
        hs = _lib.PPNHumans(packed.count.data_ptr(), packed.root_cell.data_ptr(), packed.part_cell.data_ptr(),
                            packed.part_score.data_ptr(), packed.part_box.data_ptr(), R)
        gt = _lib.PPNPoseGT(person_off.data_ptr(), head_box.data_ptr(), joint_xy.data_ptr(), joint_valid.data_ptr(), n)
        m = _lib.PPNAPMatch(*[t.data_ptr() for t in out], R)
        with torch.cuda.device(self.device):
            st = torch.cuda.current_stream(self.device).cuda_stream
            _lib.check(self.lib.ppn_ap_match(C.byref(hs), B, self.cfg.K, C.byref(gt), C.byref(self.params), C.byref(m), st),
                       "ppn_ap_match")
        self._batches.append((B, R) + out)

    def _gathered(self):
        """The match results of every update as one [N, R, ...] set (a copy when there were several updates)."""
        if len(self._batches) == 1:
            return self._batches[0][1:]
        N, R, J = self.n_images, max(b[1] for b in self._batches), self.J
        kw = dict(device=self.device)
        score, label = torch.empty(N, R, J, dtype=torch.float32, **kw), torch.empty(N, R, J, dtype=torch.uint8, **kw)
        used, flags, n_gt = (torch.empty(N, dtype=torch.int32, **kw), torch.empty(N, dtype=torch.int32, **kw),
                             torch.empty(N, J, dtype=torch.int32, **kw))
        b0 = 0
        for B, Rb, s, l, u, f, g in self._batches:
            score[b0:b0 + B, :Rb].copy_(s)
            label[b0:b0 + B, :Rb].copy_(l)
            used[b0:b0 + B].copy_(u)
            flags[b0:b0 + B].copy_(f)
            n_gt[b0:b0 + B].copy_(g)
            b0 += B
        return R, score, label, used, flags, n_gt

    def compute(self) -> dict:
        """{"ap", "precision", "recall"}: float64 numpy [J + 1] in percent, the last entry the mean over the joints.
        Raises if an image had more humans than the packed result's slots (the reference would have scored them) or
        unusable GT rows."""
        J, N = self.J, self.n_images
        if N == 0:
            return {k: np.zeros(J + 1) for k in ("ap", "precision", "recall")}
        R = max(b[1] for b in self._batches)
        if N * R * J > 0x7fffffff:
            raise ValueError(f"{N} images x {R} slots x {J} joints: the entry ordinal would exceed its 31 bits; "
                             "score the pass in parts or parse with a smaller max_humans")
        R, score, label, used, flags, n_gt = self._gathered()
        need = C.c_size_t()
        _lib.check(self.lib.ppn_ap_workspace_bytes(N, R, J, C.byref(need)), "ppn_ap_workspace_bytes")
        ws = torch.empty(need.value, dtype=torch.uint8, device=self.device)
        res = torch.empty(3, J + 1, dtype=torch.float64, device=self.device)
        status = torch.empty(3, dtype=torch.int32, device=self.device)
        m = _lib.PPNAPMatch(score.data_ptr(), label.data_ptr(), used.data_ptr(), flags.data_ptr(), n_gt.data_ptr(), R)
        res_h = torch.empty(3, J + 1, dtype=torch.float64, pin_memory=True)
        status_h = torch.empty(3, dtype=torch.int32, pin_memory=True)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device)
            _lib.check(self.lib.ppn_ap_finalize(C.byref(m), N, self.cfg.K, J, res[0].data_ptr(), res[1].data_ptr(),
                                                res[2].data_ptr(), status.data_ptr(), ws.data_ptr(), ws.numel(),
                                                stream.cuda_stream), "ppn_ap_finalize")
            res_h.copy_(res, non_blocking=True)
            status_h.copy_(status, non_blocking=True)
            stream.synchronize()
        n_over, n_bad = int(status_h[0]), int(status_h[1])
        if n_over:
            raise RuntimeError(f"{n_over} image(s) had more humans than the packed result's {R} slots: "
                               "parse with a larger max_humans")
        if n_bad:
            raise RuntimeError(f"{n_bad} image(s) had more than {_lib.AP_MAX_GT} GT people or person_off outside "
                               "the GT rows")
        r = res_h.numpy().copy()
        return {"ap": r[0], "precision": r[1], "recall": r[2]}
