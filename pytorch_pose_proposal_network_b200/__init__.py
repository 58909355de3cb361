"""B200-native Pose Proposal Network output parsing (decode + NMS + limb arg-max + tree parse).

Public surface:

* :class:`PPNConfig` — skeleton, head-tensor geometry and thresholds (config.py / datatest.py globals
  of the reference made explicit);
* :class:`PoseParser` — batched device entry: ``parser.parse(out)`` on the raw head tensor;
* :mod:`.datatest` — drop-in ``get_humans_by_feature`` / ``non_maximum_suppression`` /
  ``restore_xy`` / ``restore_size`` with the reference's signatures;
* :mod:`.sharded` — image-sharded multi-GPU driver (one process per GPU, NCCL gather of poses);
* :mod:`.dataset` — :class:`TargetEncoder`: the reference's training-target encoder (dataset.py:89-198) as one
  kernel launch per batch;
* :class:`PPNLoss` — the reference's criterion (main.py:125-216) over the head tensor and those targets, a fused
  forward and backward kernel pair behind ``torch.autograd``.

All compute happens in ``libppn_decode.so`` (hand-written sm_100a CUDA behind a C ABI, see
``include/ppn_decode.h``); there is no CPU or PyTorch fallback.
"""
from .config import (DIRECTED_GRAPHS, EDGES, EDGES_BY_NAME, EPSILON, KEYPOINT_NAMES, PPNConfig, TRACK_ORDERS)
from .utils import pairwise

__all__ = ["PPNConfig", "PoseParser", "PackedHumans", "PPNLoss", "pairwise", "KEYPOINT_NAMES", "EDGES", "EDGES_BY_NAME",
           "TRACK_ORDERS", "DIRECTED_GRAPHS", "EPSILON"]


def __getattr__(name):
    # torch and the CUDA library are only needed by the parser itself; keep `import package`
    # (config, skeleton) usable in tooling that has neither
    if name in ("PoseParser", "PackedHumans"):
        from . import parser
        return getattr(parser, name)
    if name == "PPNLoss":
        from . import loss
        return loss.PPNLoss
    raise AttributeError(name)
