"""Host-side checks of ppn_augment_images and ppn_augment_people without a GPU.

Every rejection happens before anything touches a device, so the device pointers are aligned fakes that are never
dereferenced; ppn_augment_people with n = 0 is a checked no-op.
"""
import ctypes as C

import numpy as np
import pytest

FAKE = 1 << 20                                                       # 256-byte aligned, never dereferenced


@pytest.fixture(scope="module")
def abi():
    from pytorch_pose_proposal_network_b200 import _lib
    return _lib, _lib.lib()


def norm(_lib, std=(0.229, 0.224, 0.225)):
    return _lib.PPNImageNorm((C.c_float * 3)(0.485, 0.456, 0.406), (C.c_float * 3)(*std), (C.c_float * 3)(0, 0, 0),
                             1 / 255)


def test_augment_images_rejections(abi):
    _lib, lib = abi
    B, H, W = 3, 16, 24
    hw = np.array([[5, 7], [1, 1], [9, 3]], np.int32)
    off = np.array([0, 105, 108], np.int64)
    nbytes = 108 + 81

    def call(hw=hw, off=off, nbytes=nbytes, B=B, M=FAKE, std=(0.229, 0.224, 0.225), h=H, w=W, dtype=0, layout=0, out=FAKE,
             out_bytes=None, null=()):
        hw = np.ascontiguousarray(hw, np.int32)
        off = np.ascontiguousarray(off, np.int64)
        f = dict(pixels=FAKE + 3, offset=FAKE, hw=FAKE, offset_host=off.ctypes.data, hw_host=hw.ctypes.data)
        for k in null:
            f[k] = None
        batch = _lib.PPNImageBatch(f["pixels"], f["offset"], f["hw"], f["offset_host"], f["hw_host"], nbytes, B)
        elem = 4 if dtype == 0 else 2
        ob = B * 3 * h * w * elem if out_bytes is None else out_bytes
        return lib.ppn_augment_images(None if "batch" in null else C.byref(batch), M,
                                      None if "norm" in null else C.byref(norm(_lib, std)), h, w, dtype, layout, out, ob, None)

    for k in ("pixels", "offset", "hw", "offset_host", "hw_host", "batch", "norm"):
        assert call(null=(k,)) == -1, k
    assert call(M=None) == -1 and call(out=None) == -1
    assert call(M=FAKE + 2) == -1                                    # fp32 parameters
    assert call(out=FAKE + 2) == -1                                  # fp32 output needs 4-byte alignment
    assert call(dtype=1, out=FAKE + 1) == -1                         # 16-bit output needs 2-byte alignment
    assert call(B=0) == -1 and call(B=-1) == -1
    for bad in ([0, 7], [5, 0], [65536, 1], [1, 65536], [-1, 4]):
        h2 = hw.copy()
        h2[1] = bad
        assert call(hw=h2, nbytes=1 << 40) == -1, bad
    assert call(nbytes=nbytes - 1) == -1                             # the last image ends past the buffer
    assert call(off=np.array([0, 105, -1], np.int64)) == -1
    assert call(dtype=3) == -1 and call(dtype=-1) == -1
    assert call(layout=2) == -1 and call(layout=-1) == -1
    for std in ((0.2, 0.0, 0.2), (0.2, 0.2, -1.0), (float("nan"), 0.2, 0.2)):
        assert call(std=std) == -1, std
    for h, w in ((0, W), (H, 0), (65536, W), (H, 65536)):
        assert call(h=h, w=w, out_bytes=4 * B * 3 * max(h, 1) * max(w, 1)) == -1
    assert call(out_bytes=B * 3 * H * W * 4 - 4) == -1
    assert call(out_bytes=B * 3 * H * W * 4 + 4) == -1
    assert call(dtype=1, out_bytes=B * 3 * H * W * 4) == -1          # fp32 bytes for a 16-bit output


def test_augment_people_rejections(abi):
    _lib, lib = abi
    K = 4
    perm = np.array([1, 0, 2], np.int32)

    def call(B=2, n=5, K=K, perm=perm, A=FAKE, flip=FAKE, src=None, dst=None, null=()):
        src = src or dict(person_off=FAKE, bbox=FAKE, keypoints=FAKE, visible=FAKE, size=FAKE)
        dst = dst or dict(bbox=FAKE, keypoints=FAKE, visible=FAKE, size=FAKE)
        s = _lib.PPNPeople(*[src[k] for k in ("person_off", "bbox", "keypoints", "visible", "size")])
        d = _lib.PPNPeopleOut(*[dst[k] for k in ("bbox", "keypoints", "visible", "size")])
        p = None if perm is None else np.ascontiguousarray(perm, np.int32).ctypes.data_as(_lib.i32p)
        return lib.ppn_augment_people(None if "in" in null else C.byref(s), B, n, K, A, flip, p,
                                      None if "out" in null else C.byref(d), None)

    assert call(n=0) == 0                                            # checked, nothing to do
    assert call(null=("in",)) == -1 and call(null=("out",)) == -1
    assert call(perm=None) == -1 and call(A=None) == -1 and call(flip=None) == -1
    assert call(A=FAKE + 4) == -1                                    # float64 parameters
    assert call(B=0) == -1 and call(n=-1) == -1
    assert call(K=0) == -1 and call(K=257) == -1
    for bad in ([1, 1, 2], [0, 1, 3], [-1, 0, 2]):
        assert call(perm=bad) == -1, bad
    for k in ("person_off", "bbox", "keypoints", "visible", "size"):
        src = dict(person_off=FAKE, bbox=FAKE, keypoints=FAKE, visible=FAKE, size=FAKE)
        src[k] = None
        assert call(src=src) == -1, k
    for k in ("bbox", "keypoints", "visible", "size"):
        dst = dict(bbox=FAKE, keypoints=FAKE, visible=FAKE, size=FAKE)
        dst[k] = None
        assert call(dst=dst) == -1, k
    dst = dict(bbox=FAKE + 4, keypoints=FAKE, visible=FAKE, size=FAKE)
    assert call(dst=dst) == -1                                       # float64 boxes need 8-byte alignment
    assert call(K=1, perm=np.zeros(0, np.int32), n=0) == 0           # no parts: only the boxes and sizes move


def test_python_checks_without_a_device(abi):
    import torch
    from pytorch_pose_proposal_network_b200.augment import Augmenter, ImageBatch
    from pytorch_pose_proposal_network_b200.config import PPNConfig
    cfg = PPNConfig.mpii16()
    for kw in (dict(dtype=torch.float64), dict(scale=(1.2, 0.8)), dict(scale=(0, 1)), dict(rotation=-1), dict(shift=-0.1),
               dict(p_flip=1.5), dict(std=(0.2, 0.0, 0.2)), dict(mean=(0.1, 0.2)), dict(keypoint_names=["instance"])):
        with pytest.raises(ValueError):
            Augmenter(cfg, device="cpu", **kw)
    with pytest.raises(ValueError):
        Augmenter(PPNConfig(K=5, E=1, directed_graphs=(((0,), (1,)),)), device="cpu")
    a = Augmenter(PPNConfig(K=3, E=1, directed_graphs=(((0,), (1,)),)), keypoint_names=["i", "left_x", "right_x"], device="cpu")
    assert a.perm.tolist() == [1, 0]
    px, off, hw = torch.zeros(64, dtype=torch.uint8), torch.zeros(2, dtype=torch.int64), torch.ones(2, 2, dtype=torch.int32)
    ImageBatch(px, off, hw, np.zeros(2), np.ones((2, 2)))
    for bad in ((px.float(), off, hw), (px, off.int(), hw), (px, off, hw.long()), (px, off[:1], hw)):
        with pytest.raises(ValueError):
            ImageBatch(*bad, np.zeros(2), np.ones((2, 2)))
    with pytest.raises(ValueError):
        ImageBatch.from_arrays([np.zeros((4, 4), np.uint8)])
    with pytest.raises(ValueError):
        ImageBatch.from_arrays([])
