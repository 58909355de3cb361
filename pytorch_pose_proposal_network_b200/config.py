"""Skeleton (parts, limbs, track orders) and the explicit parser geometry.

The reference keeps the skeleton in ``config.py`` (/root/reference/config.py:3-80)
and the parser geometry in module globals of ``datatest.py``
(/root/reference/datatest.py:53-60) with the thresholds written as literals at the
call sites (0.15 at rt_test.py:133 / main.py:972,1141; NMS 0.3 at datatest.py:94;
``min_num_keypoints=1`` at datatest.py:74).  Here all of that is one explicit,
immutable :class:`PPNConfig`; the module-level names ``KEYPOINT_NAMES``, ``EDGES``,
``EDGES_BY_NAME``, ``TRACK_ORDERS``, ``DIRECTED_GRAPHS``, ``COLOR_MAP`` and ``EPSILON`` keep the
reference's spelling and values so ``from config import *`` call sites still work.
"""
from __future__ import annotations

from dataclasses import dataclass, field, replace
from typing import List, Sequence, Tuple

import numpy as np

from .utils import pairwise

# --------------------------------------------------------------------------- #
# 18-part skeleton of the reference (config.py:3-21, 44-65): 'instance' + 17.
# --------------------------------------------------------------------------- #
_SIDES = ("left", "right")
_ARM = ("shoulder", "elbow", "wrist")
_LEG = ("hip", "knee", "ankle")

name_list = (
    [f"{s}_{j}" for j in _ARM for s in _SIDES]
    + [f"{s}_{j}" for j in _LEG for s in _SIDES]
    + ["thorax", "pelvis", "neck", "top", "stomach"]
)
KEYPOINT_NAMES = ["instance"] + name_list


def _limb_chain(*names):
    return [[a, b] for a, b in pairwise(names)]


EDGES_BY_NAME = (
    _limb_chain("instance", "neck", "thorax", "left_shoulder", "left_elbow", "left_wrist")
    + _limb_chain("thorax", "right_shoulder", "right_elbow", "right_wrist")
    + _limb_chain("thorax", "stomach", "pelvis")
    + [["pelvis", "left_hip"], ["pelvis", "right_hip"],
       ["left_hip", "left_knee"], ["right_hip", "right_knee"],
       ["left_knee", "left_ankle"], ["right_knee", "right_ankle"],
       ["instance", "top"]]
)
EDGES = [[KEYPOINT_NAMES.index(s), KEYPOINT_NAMES.index(d)] for s, d in EDGES_BY_NAME]

_TRUNK = ["instance", "neck", "thorax"]
TRACK_ORDERS = [
    _TRUNK + [f"left_{j}" for j in _ARM],
    _TRUNK + [f"right_{j}" for j in _ARM],
    _TRUNK + ["stomach", "pelvis"] + [f"left_{j}" for j in _LEG],
    _TRUNK + ["stomach", "pelvis"] + [f"right_{j}" for j in _LEG],
    ["instance", "top"],
]


def directed_graphs(track_orders, edges_by_name, keypoint_names):
    """[[limb indices], [target part indices]] per track order (config.py:75-80)."""
    graphs = []
    for order in track_orders:
        eis = [edges_by_name.index([a, b]) for a, b in pairwise(order)]
        ts = [keypoint_names.index(b) for _, b in pairwise(order)]
        graphs.append([eis, ts])
    return graphs


DIRECTED_GRAPHS = directed_graphs(TRACK_ORDERS, EDGES_BY_NAME, KEYPOINT_NAMES)
EPSILON = 1e-6

# Drawing colours of the parts (config.py:23-42): the consumers of the parser's output (datatest.draw_humans,
# datatest.py:170-221) look parts up here.  One RGB triple per entry of KEYPOINT_NAMES, in that order; the dict
# keeps the reference's key order (instance, right arm, left arm, right leg, left leg, trunk).
_PALETTE = ("8f2323 0040ff 4f8f23 0095ff 6aff00 00eaff bfff00 6b238f 23628f aa00ff b9d7ed dcb9ed b9ede0 "
            "ffff00 ff00aa edb9b9 ff0000 4f2323").split()
_RGB = {n: tuple(int(h[i:i + 2], 16) for i in (0, 2, 4)) for n, h in zip(KEYPOINT_NAMES, _PALETTE)}
COLOR_MAP = {n: _RGB[n] for n in (["instance"] + [f"{s}_{j}" for s in ("right", "left") for j in _ARM]
                                  + [f"{s}_{j}" for s in ("right", "left") for j in _LEG]
                                  + ["thorax", "pelvis", "neck", "top", "stomach"])}

# --------------------------------------------------------------------------- #
# 16-part skeleton used by BASELINE.json configs[0:2] ("MPII 16-part PPN"):
# 'instance' + 15 joints, 15 limbs.  The reference has no such preset (its K is
# fixed at 18); this one drops 'top' and 'stomach' and hangs the pelvis off the
# thorax, so that K=16 / E=15 as BASELINE.md §3 requires.
# --------------------------------------------------------------------------- #
KEYPOINT_NAMES_16 = ["instance"] + [n for n in name_list if n not in ("top", "stomach")]
EDGES_BY_NAME_16 = (
    _limb_chain("instance", "neck", "thorax", "left_shoulder", "left_elbow", "left_wrist")
    + _limb_chain("thorax", "right_shoulder", "right_elbow", "right_wrist")
    + [["thorax", "pelvis"]]
    + _limb_chain("pelvis", "left_hip", "left_knee", "left_ankle")
    + _limb_chain("pelvis", "right_hip", "right_knee", "right_ankle")
)
EDGES_16 = [[KEYPOINT_NAMES_16.index(s), KEYPOINT_NAMES_16.index(d)] for s, d in EDGES_BY_NAME_16]
TRACK_ORDERS_16 = [
    _TRUNK + [f"left_{j}" for j in _ARM],
    _TRUNK + [f"right_{j}" for j in _ARM],
    _TRUNK + ["pelvis"] + [f"left_{j}" for j in _LEG],
    _TRUNK + ["pelvis"] + [f"right_{j}" for j in _LEG],
]
DIRECTED_GRAPHS_16 = directed_graphs(TRACK_ORDERS_16, EDGES_BY_NAME_16, KEYPOINT_NAMES_16)


def default_skeleton(cfg, keypoint_names=None, edges=None, need=("names", "edges")):
    """(keypoint_names, edges) of `cfg`'s skeleton, each given one passed through and a missing one of those `need`
    names taken from config.py's two skeletons: the part names by K, the edges by (K, E).  ValueError where K (or
    (K, E)) matches neither."""
    if keypoint_names is None and "names" in need:
        keypoint_names = {len(KEYPOINT_NAMES): KEYPOINT_NAMES, len(KEYPOINT_NAMES_16): KEYPOINT_NAMES_16}.get(cfg.K)
        if keypoint_names is None:
            raise ValueError("pass `keypoint_names` (K part names) for a skeleton that is not one of config.py's")
    if edges is None and "edges" in need:
        edges = {(len(KEYPOINT_NAMES), len(EDGES)): EDGES, (len(KEYPOINT_NAMES_16), len(EDGES_16)): EDGES_16}.get(
            (cfg.K, cfg.E))
        if edges is None:
            raise ValueError("pass `edges` ([E][2] part ids) for a skeleton that is not one of config.py's")
    return keypoint_names, edges


def _freeze_graphs(graphs) -> Tuple[Tuple[Tuple[int, ...], Tuple[int, ...]], ...]:
    return tuple((tuple(int(v) for v in eis), tuple(int(v) for v in ts)) for eis, ts in graphs)


@dataclass(frozen=True)
class PPNConfig:
    """Everything the parser needs to know about one head-tensor layout.

    ``insize``/``outsize``/``local_grid_size`` are (W, H) pairs exactly as in the
    reference (datatest.py:53-59, model.py:52-64).  The head tensor is
    ``[B, 6K + sH*sW*E, outH, outW]`` fp32 with channel groups
    ``resp, conf, x, y, w, h`` (K channels each) followed by the limb block viewed
    as ``[E, sH, sW, outH, outW]`` (rt_test.py:109-120).
    """

    K: int = len(KEYPOINT_NAMES)
    E: int = len(EDGES)
    insize: Tuple[int, int] = (384, 384)            # (inW, inH)
    outsize: Tuple[int, int] = (24, 24)             # (outW, outH)
    local_grid_size: Tuple[int, int] = (21, 21)     # (sW, sH)
    directed_graphs: tuple = field(default_factory=lambda: _freeze_graphs(DIRECTED_GRAPHS))
    detection_thresh: float = 0.15                  # rt_test.py:133
    nms_thresh: float = 0.3                         # datatest.py:94
    min_num_keypoints: int = 1                      # datatest.py:74
    # Which half-window is subtracted along h and along w.  The reference subtracts
    # local_grid_size[0]//2 (= sW//2) from the ROW and local_grid_size[1]//2 (= sH//2)
    # from the COLUMN (datatest.py:115-116); for square windows they coincide.  The
    # stale copy in test.py:211-212 does it the other way round.
    swap_window_offsets: bool = False

    def __post_init__(self):
        object.__setattr__(self, "directed_graphs", _freeze_graphs(self.directed_graphs))
        if self.K < 1 or self.E < 0:
            raise ValueError("K >= 1 and E >= 0 required")
        for eis, ts in self.directed_graphs:
            if len(eis) != len(ts):
                raise ValueError("each directed graph needs as many limbs as targets")
            if any(not 0 <= e < self.E for e in eis) or any(not 0 <= t < self.K for t in ts):
                raise ValueError("directed graph indexes a limb/part outside E/K")

    # ---- geometry -------------------------------------------------------- #
    @property
    def inW(self): return int(self.insize[0])
    @property
    def inH(self): return int(self.insize[1])
    @property
    def W(self): return int(self.outsize[0])
    @property
    def H(self): return int(self.outsize[1])
    @property
    def sW(self): return int(self.local_grid_size[0])
    @property
    def sH(self): return int(self.local_grid_size[1])
    @property
    def S(self): return self.sH * self.sW
    @property
    def HW(self): return self.H * self.W
    @property
    def gridsize(self):
        """(gridW, gridH) = (int(inW/outW), int(inH/outH))  (datatest.py:60)."""
        return (int(self.inW / self.W), int(self.inH / self.H))
    @property
    def C(self):
        """Channel count of the head tensor, ``lastsize`` in model.py:64."""
        return 6 * self.K + self.S * self.E
    @property
    def off_h(self):
        """Half-window subtracted from the row index (datatest.py:115)."""
        return (self.sH if self.swap_window_offsets else self.sW) // 2
    @property
    def off_w(self):
        """Half-window subtracted from the column index (datatest.py:116)."""
        return (self.sW if self.swap_window_offsets else self.sH) // 2
    @property
    def bytes_per_image(self):
        return self.C * self.HW * 4

    # ---- flattened track orders, the form the kernels take ---------------- #
    def chains(self):
        """(chain_off[n+1], chain_limb[L], chain_part[L]) int32 arrays."""
        off, limbs, parts = [0], [], []
        for eis, ts in self.directed_graphs:
            limbs += list(eis)
            parts += list(ts)
            off.append(len(limbs))
        return (np.asarray(off, np.int32), np.asarray(limbs, np.int32), np.asarray(parts, np.int32))

    def key_order(self) -> List[int]:
        """Part ids in the order a complete human's dict receives them (datatest.py:104-125)."""
        seen = [0]
        for _, ts in self.directed_graphs:
            for t in ts:
                if t not in seen:
                    seen.append(t)
        return seen

    def with_(self, **kw) -> "PPNConfig":
        return replace(self, **kw)

    # ---- presets ---------------------------------------------------------- #
    @classmethod
    def reference_native(cls, **kw):
        """The reference's hard-coded shape: K=18, E=17, 384², 24×24 grid, 21×21 window."""
        return cls(**kw)

    @classmethod
    def mpii16(cls, insize=(384, 384), outsize=(12, 12), local_grid_size=(9, 9), **kw):
        """BASELINE.json configs[0:2]: 16 parts, 15 limbs, 12×12 grid, 9×9 window."""
        return cls(K=16, E=15, insize=insize, outsize=outsize, local_grid_size=local_grid_size,
                   directed_graphs=_freeze_graphs(DIRECTED_GRAPHS_16), **kw)

    @classmethod
    def coco18(cls, insize=(512, 512), outsize=(16, 16), local_grid_size=(9, 9), **kw):
        """BASELINE.json configs[2]: 18 parts / 17 limbs (reference tree), 16×16 grid."""
        return cls(insize=insize, outsize=outsize, local_grid_size=local_grid_size, **kw)

    @classmethod
    def highres(cls, **kw):
        """BASELINE.json configs[3]: 768², 24×24 grid, 11×11 window."""
        return cls(insize=(768, 768), outsize=(24, 24), local_grid_size=(11, 11), **kw)


PRESETS = {
    "cfg1": PPNConfig.mpii16,
    "cfg2": PPNConfig.mpii16,
    "cfg3": PPNConfig.coco18,
    "cfg4": PPNConfig.highres,
    "native": PPNConfig.reference_native,
}
