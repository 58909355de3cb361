"""ctypes binding of libppn_decode.so — the only way the package reaches its kernels.

There is no fallback of any kind: if the shared library is missing or does not export every
symbol declared in include/ppn_decode.h, importing this module's :func:`lib` raises.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

ABI_VERSION = 7
HEAD_F32, HEAD_F16, HEAD_BF16 = 0, 1, 2
GEMM_TF32, GEMM_F16, GEMM_BF16 = 0, 1, 2
FEAT_NCHW_F32, FEAT_NHWC_16 = 0, 1
FLAG_INPUT_COMPLETE = 1
FLAG_CLEAR_UNUSED = 2
MAX_CELLS = 1024
MAX_CHAINS = 32
MAX_CHAIN_STEPS = 192
PROPOSAL_MAX_PARTS = 64
IPC_HANDLE_BYTES = 64

i32p = C.POINTER(C.c_int32)
f32p = C.POINTER(C.c_float)
u16p = C.POINTER(C.c_uint16)


class PPNShape(C.Structure):
    _fields_ = [(n, C.c_int32) for n in
                ("B", "K", "E", "H", "W", "sH", "sW", "inW", "inH", "gridW", "gridH", "off_h", "off_w", "head_dtype")]


class PPNParams(C.Structure):
    _fields_ = [("det_thresh", C.c_float), ("nms_thresh", C.c_float), ("min_num_keypoints", C.c_int32),
                ("n_nms_parts", C.c_int32), ("n_chains", C.c_int32), ("flags", C.c_int32),
                ("chain_off", i32p), ("chain_limb", i32p), ("chain_part", i32p)]


class PPNHumans(C.Structure):
    _fields_ = [("count", C.c_void_p), ("root_cell", C.c_void_p), ("part_cell", C.c_void_p),
                ("part_score", C.c_void_p), ("part_box", C.c_void_p), ("R", C.c_int32)]


class PPNHeadOptions(C.Structure):
    _fields_ = [("operand", C.c_int32), ("feat_layout", C.c_int32)]


class PPNPeople(C.Structure):
    _fields_ = [("person_off", C.c_void_p), ("bbox", C.c_void_p), ("keypoints", C.c_void_p),
                ("visible", C.c_void_p), ("size", C.c_void_p)]


TARGET_NAMES = ("delta", "weight", "weight_ij", "tx", "ty", "tx_half", "ty_half", "tw", "th", "te")


class PPNTargets(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in TARGET_NAMES]


class PPNLossOptions(C.Structure):
    _fields_ = [("limb_dtype", C.c_int32)]


class PPNPoseGT(C.Structure):
    _fields_ = [("person_off", C.c_void_p), ("head_box", C.c_void_p), ("joint_xy", C.c_void_p),
                ("joint_valid", C.c_void_p), ("n", C.c_int32)]


class PPNAPParams(C.Structure):
    _fields_ = [("n_joints", C.c_int32), ("dist_thresh", C.c_double), ("head_scale", C.c_double)]


class PPNAPMatch(C.Structure):
    _fields_ = [("score", C.c_void_p), ("label", C.c_void_p), ("used", C.c_void_p), ("flags", C.c_void_p),
                ("n_gt", C.c_void_p), ("R", C.c_int32)]


AP_MAX_JOINTS = 32
AP_MAX_GT = 64


class PPNImageBatch(C.Structure):
    _fields_ = [("pixels", C.c_void_p), ("offset", C.c_void_p), ("hw", C.c_void_p), ("offset_host", C.c_void_p),
                ("hw_host", C.c_void_p), ("bytes", C.c_size_t), ("B", C.c_int32)]


class PPNImageNorm(C.Structure):
    _fields_ = [("mean", C.c_float * 3), ("std", C.c_float * 3), ("fill", C.c_float * 3), ("in_scale", C.c_float)]


class PPNPeopleOut(C.Structure):
    _fields_ = [("bbox", C.c_void_p), ("keypoints", C.c_void_p), ("visible", C.c_void_p), ("size", C.c_void_p)]


LAYOUT_NCHW, LAYOUT_NHWC = 0, 1


# name -> (restype, argtypes); must list every function of include/ppn_decode.h
EXPORTS = {
    "ppn_abi_version": (C.c_int, []),
    "ppn_strerror": (C.c_char_p, [C.c_int]),
    "ppn_workspace_bytes": (C.c_int, [C.POINTER(PPNShape), C.POINTER(PPNParams), C.POINTER(C.c_size_t)]),
    "ppn_parse_launches": (C.c_int, [C.POINTER(PPNShape), C.POINTER(PPNParams)]),
    "ppn_parse_plan": (C.c_int, [C.POINTER(PPNShape), C.POINTER(PPNParams), i32p]),
    "ppn_limb_argmax": (C.c_int, [C.c_void_p, C.POINTER(PPNShape), C.c_void_p, C.c_void_p]),
    "ppn_limb_stream_probe": (C.c_int, [C.c_void_p, C.POINTER(PPNShape), C.c_void_p, C.c_int32, C.c_void_p]),
    "ppn_decode_candidates": (C.c_int, [C.c_void_p, C.POINTER(PPNShape), C.c_int32, C.c_float,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ppn_restore_xy": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(PPNShape), C.c_void_p]),
    "ppn_restore_size": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(PPNShape), C.c_void_p]),
    "ppn_nms": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_int32,
                          C.c_void_p, C.c_void_p, C.c_void_p]),
    "ppn_tree_parse": (C.c_int, [C.c_void_p, C.POINTER(PPNShape), C.POINTER(PPNParams), C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.POINTER(PPNHumans), C.c_void_p]),
    "ppn_parse": (C.c_int, [C.c_void_p, C.POINTER(PPNShape), C.POINTER(PPNParams), C.POINTER(PPNHumans),
                            C.c_void_p, C.c_size_t, C.c_void_p]),
    "ppn_parse_proposals_workspace_bytes": (C.c_int, [C.POINTER(PPNShape), C.POINTER(PPNParams), C.POINTER(C.c_size_t)]),
    "ppn_parse_proposals": (C.c_int, [C.c_void_p, C.POINTER(PPNShape), C.POINTER(PPNParams), C.POINTER(PPNHumans),
                                      C.c_void_p, C.c_size_t, C.c_void_p]),
    "ppn_parse_host_scratch_bytes": (C.c_int, [C.POINTER(PPNShape), C.POINTER(PPNParams), C.c_int32,
                                               C.POINTER(C.c_size_t)]),
    "ppn_parse_host": (C.c_int, [C.c_void_p, C.POINTER(PPNShape), C.POINTER(PPNParams), C.POINTER(PPNHumans),
                                 C.c_void_p, C.c_size_t]),
    "ppn_part_centres": (C.c_int, [C.POINTER(PPNHumans), C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "ppn_skeleton": (C.c_int, [C.POINTER(PPNHumans), C.c_int32, C.c_int32, C.c_int32, i32p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ppn_packed_bytes": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "ppn_pack_humans": (C.c_int, [C.POINTER(PPNHumans), C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ppn_parse_dense": (C.c_int, [C.c_void_p, C.POINTER(PPNShape), C.POINTER(PPNParams), C.POINTER(PPNHumans),
                                  C.c_void_p, C.c_size_t, C.c_int32, C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ppn_parse_dense_remote": (C.c_int, [C.c_void_p, C.POINTER(PPNShape), C.POINTER(PPNParams), C.POINTER(PPNHumans),
                                         C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int32, C.c_int32,
                                         C.c_void_p, C.c_size_t, C.c_void_p]),
    "ppn_peer_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p), C.c_char_p]),
    "ppn_peer_open": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "ppn_peer_close": (C.c_int, [C.c_void_p]),
    "ppn_peer_free": (C.c_int, [C.c_void_p]),
    "ppn_peer_copy": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ppn_peer_post": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p]),
    "ppn_peer_wait": (C.c_int, [C.c_void_p, C.c_int32, C.c_longlong, C.c_uint32, C.c_void_p, C.c_void_p]),
    "ppn_head_workspace_bytes": (C.c_int, [C.POINTER(PPNShape), C.POINTER(C.c_size_t)]),
    "ppn_head_gemm_argmax": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(PPNShape), C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p]),
    "ppn_head_parse": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(PPNShape), C.POINTER(PPNParams),
                                 C.POINTER(PPNHumans), C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ppn_head_workspace_bytes_opt": (C.c_int, [C.POINTER(PPNShape), C.c_int32, C.POINTER(PPNHeadOptions), C.POINTER(C.c_size_t)]),
    "ppn_head_gemm_argmax_opt": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(PPNShape), C.POINTER(PPNHeadOptions),
                                           C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ppn_head_parse_opt": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(PPNShape), C.POINTER(PPNParams),
                                     C.POINTER(PPNHeadOptions), C.POINTER(PPNHumans), C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                     C.c_void_p]),
    "ppn_encode_targets": (C.c_int, [C.POINTER(PPNPeople), C.POINTER(PPNShape), i32p, C.POINTER(PPNTargets), C.c_void_p]),
    "ppn_loss_workspace_bytes": (C.c_int, [C.POINTER(PPNShape), C.POINTER(C.c_size_t)]),
    "ppn_loss_forward": (C.c_int, [C.c_void_p, C.POINTER(PPNShape), C.POINTER(PPNTargets), C.c_void_p, C.c_void_p,
                                   C.c_size_t, C.c_void_p]),
    "ppn_loss_backward": (C.c_int, [C.c_void_p, C.POINTER(PPNShape), C.POINTER(PPNTargets), C.c_void_p, C.c_void_p,
                                    C.c_void_p]),
    "ppn_loss_workspace_bytes_opt": (C.c_int, [C.POINTER(PPNShape), C.POINTER(PPNLossOptions), C.POINTER(C.c_size_t)]),
    "ppn_loss_forward_opt": (C.c_int, [C.c_void_p, C.POINTER(PPNShape), C.POINTER(PPNTargets), C.POINTER(PPNLossOptions),
                                       C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ppn_loss_backward_opt": (C.c_int, [C.c_void_p, C.POINTER(PPNShape), C.POINTER(PPNTargets), C.POINTER(PPNLossOptions),
                                        C.c_void_p, C.c_void_p, C.c_void_p]),
    "ppn_encode_targets_opt": (C.c_int, [C.POINTER(PPNPeople), C.POINTER(PPNShape), i32p, C.POINTER(PPNTargets), C.c_int32,
                                         C.c_void_p]),
    "ppn_loss_forward_logits": (C.c_int, [C.c_void_p, C.POINTER(PPNShape), C.POINTER(PPNTargets), C.POINTER(PPNLossOptions),
                                          C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ppn_loss_backward_logits": (C.c_int, [C.c_void_p, C.POINTER(PPNShape), C.POINTER(PPNTargets), C.POINTER(PPNLossOptions),
                                           C.c_void_p, C.c_void_p, C.c_void_p]),
    "ppn_sigmoid": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ppn_ap_match": (C.c_int, [C.POINTER(PPNHumans), C.c_int32, C.c_int32, C.POINTER(PPNPoseGT), C.POINTER(PPNAPParams),
                               C.POINTER(PPNAPMatch), C.c_void_p]),
    "ppn_ap_workspace_bytes": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_size_t)]),
    "ppn_ap_finalize": (C.c_int, [C.POINTER(PPNAPMatch), C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ppn_augment_images": (C.c_int, [C.POINTER(PPNImageBatch), C.c_void_p, C.POINTER(PPNImageNorm), C.c_int32, C.c_int32,
                                     C.c_int32, C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ppn_augment_people": (C.c_int, [C.POINTER(PPNPeople), C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, i32p,
                                     C.POINTER(PPNPeopleOut), C.c_void_p]),
    "ppn_flip_merge": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(PPNShape), i32p, i32p, C.c_void_p]),
    "ppn_debug_argmax_items": (C.c_int, [C.POINTER(PPNShape), C.c_int32, i32p, i32p, i32p, C.c_int32]),
    "ppn_timeline": (C.c_int, [C.c_void_p, C.c_int32]),
    "ppn_profile_enable": (C.c_int, [C.c_int32]),
    "ppn_profile_read": (C.c_int, [f32p, i32p]),
    "ppn_tune": (C.c_int, [C.c_char_p, C.c_int32]),
    "ppn_tune_get": (C.c_int, [C.c_char_p, i32p]),
}

_lib = None


class PPNError(RuntimeError):
    def __init__(self, code: int, where: str):
        self.code = code
        msg = lib().ppn_strerror(code)
        super().__init__(f"{where}: {msg.decode() if msg else 'error'} (code {code})")


def lib_path() -> str:
    return os.environ.get("PPN_DECODE_LIB", _build.LIB_PATH)


def lib():
    """Load (once) and return the CDLL; raises if it is absent or incomplete."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise ImportError(
            f"{path} not found: build it with `python -m pytorch_pose_proposal_network_b200.build` "
            "(needs nvcc); this package has no CPU or PyTorch fallback")
    handle = C.CDLL(path)
    for name, (restype, argtypes) in EXPORTS.items():
        try:
            fn = getattr(handle, name)
        except AttributeError as e:
            raise ImportError(f"{path} does not export {name}") from e
        fn.restype = restype
        fn.argtypes = argtypes
    if handle.ppn_abi_version() != ABI_VERSION:
        raise ImportError(f"{path}: ABI version {handle.ppn_abi_version()} != {ABI_VERSION}")
    _lib = handle
    return _lib


def check(code: int, where: str):
    if code != 0:
        raise PPNError(code, where)


def tune(**knobs):
    """tune(argmax_variant=0, argmax_stage_bytes=..., ...) — benchmark knobs (ppn_tune)."""
    for k, v in knobs.items():
        check(lib().ppn_tune(k.replace("_", ".", 1).encode(), int(v)), f"ppn_tune({k})")


def tune_get(key: str) -> int:
    v = C.c_int32()
    check(lib().ppn_tune_get(key.encode(), C.byref(v)), f"ppn_tune_get({key})")
    return v.value


STAGES = ("limb_argmax", "decode_candidates", "nms", "tree_parse")


def profile_enable(on: bool = True):
    check(lib().ppn_profile_enable(1 if on else 0), "ppn_profile_enable")


def profile_read():
    """-> ({stage: total ms}, n_calls) since the last read; waits for the recorded events."""
    ms = (C.c_float * 4)()
    n = C.c_int32()
    check(lib().ppn_profile_read(ms, C.byref(n)), "ppn_profile_read")
    return dict(zip(STAGES, (float(v) for v in ms))), n.value
