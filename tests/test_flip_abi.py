"""Host-side checks of ppn_flip_merge without a GPU.

Every call here is rejected before anything touches a device, so the device pointers are aligned fakes that are
never dereferenced.
"""
import ctypes as C

import numpy as np
import pytest

FAKE = 1 << 30                                                       # 256-byte aligned, never dereferenced


@pytest.fixture(scope="module")
def abi():
    from pytorch_pose_proposal_network_b200 import _lib
    return _lib, _lib.lib()


def shape_of(_lib, cfg, B=2, dtype=0, **over):
    gW, gH = cfg.gridsize
    f = dict(B=B, K=cfg.K, E=cfg.E, H=cfg.H, W=cfg.W, sH=cfg.sH, sW=cfg.sW, inW=cfg.inW, inH=cfg.inH, gridW=gW,
             gridH=gH, off_h=cfg.off_h, off_w=cfg.off_w, head_dtype=dtype)
    f.update(over)
    return _lib.PPNShape(**f)


def test_flip_merge_rejections(abi):
    _lib, lib = abi
    from pytorch_pose_proposal_network_b200.config import PPNConfig
    from pytorch_pose_proposal_network_b200.flip import limb_mirror, part_mirror
    from pytorch_pose_proposal_network_b200 import config as pcfg
    cfg = PPNConfig.mpii16()
    P = part_mirror(pcfg.KEYPOINT_NAMES_16)
    Q = limb_mirror(P, pcfg.EDGES_16)
    nbytes = 2 * cfg.C * cfg.H * cfg.W * 4
    BF = FAKE + 4 * nbytes                                           # apart from head and out

    def call(head=FAKE, flipped=BF, out=FAKE + 2 * nbytes, p=P, q=Q, shape=None, **over):
        s = shape if shape is not None else shape_of(_lib, cfg, **over)
        pp = None if p is None else np.ascontiguousarray(p, np.int32).ctypes.data_as(_lib.i32p)
        qq = None if q is None else np.ascontiguousarray(q, np.int32).ctypes.data_as(_lib.i32p)
        return lib.ppn_flip_merge(head, flipped, out, None if shape is False else C.byref(s), pp, qq, None)

    # NULL pointers, B < 1, an unknown dtype
    assert call(head=None) == -1 and call(flipped=None) == -1 and call(out=None) == -1
    assert call(p=None) == -1 and call(q=None) == -1
    assert lib.ppn_flip_merge(FAKE, BF, FAKE, None, P.ctypes.data_as(_lib.i32p), Q.ctypes.data_as(_lib.i32p), None) == -1
    assert call(B=0) == -1 and call(B=-3) == -1
    assert call(dtype=3) == -1 and call(dtype=-1) == -1
    # alignment to the element size
    assert call(head=FAKE + 2) == -1 and call(flipped=BF + 1) == -1 and call(out=FAKE + 2 * nbytes + 2) == -1
    assert call(dtype=1, head=FAKE + 1) == -1 and call(dtype=2, out=FAKE + 2 * nbytes + 1) == -1
    # mirror tables: self-inverse permutations, part 0 fixed
    bad_p = P.copy(); bad_p[[0, 1]] = bad_p[[1, 0]]
    assert call(p=bad_p) == -1                                       # part_mirror[0] != 0 (an involution otherwise)
    bad_p = P.copy(); bad_p[1] = 1                                   # 1 -> 1 but 2 -> 1: not a permutation
    assert call(p=bad_p) == -1
    bad_p = P.copy(); bad_p[[1, 3, 2, 4]] = [3, 2, 4, 1]             # a permutation, not self-inverse
    assert call(p=bad_p) == -1
    bad_p = P.copy(); bad_p[5] = 16
    assert call(p=bad_p) == -1 and call(p=np.where(P == 5, -1, P)) == -1
    bad_q = Q.copy(); bad_q[[2, 3, 4]] = [3, 4, 2]
    assert call(q=bad_q) == -1
    bad_q = Q.copy(); bad_q[0] = 15
    assert call(q=bad_q) == -1
    # out overlapping head_flipped (any overlap, equal included), or overlapping head without being it
    assert call(out=BF) == -1 and call(out=BF + nbytes - 4) == -1 and call(out=BF - nbytes + 4) == -1
    assert call(head=BF, out=BF) == -1                               # in place into the flipped view
    assert call(out=FAKE + 4) == -1 and call(out=FAKE - nbytes + 4) == -1
    # geometry whose mirror is not exact, and the kernel's limits
    assert call(inW=cfg.inW + 1) == -2
    assert call(off_w=cfg.off_w - 1) == -2 and call(sW=cfg.sW + 1, E=cfg.E) == -2
    P70 = np.arange(70, dtype=np.int32)
    assert call(shape=shape_of(_lib, cfg, K=70, E=0, H=12, W=12), p=P70, q=None) == -2
    assert call(shape=shape_of(_lib, cfg, E=0, H=33, W=33, inW=33 * 32)) == -2   # H * W > PPN_MAX_CELLS
