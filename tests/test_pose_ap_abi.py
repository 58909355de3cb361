"""Host-side checks of ppn_ap_match, ppn_ap_workspace_bytes and ppn_ap_finalize without a GPU.

Every rejection happens before anything touches a device, so the pointers are aligned fakes that are never
dereferenced; a B = 0 match with valid arguments is a no-op.
"""
import ctypes as C

import pytest

FAKE = 1 << 20                                                       # 256-byte aligned, never dereferenced


@pytest.fixture(scope="module")
def abi():
    from pytorch_pose_proposal_network_b200 import _lib
    return _lib, _lib.lib()


def humans(_lib, R=8, **moved):
    f = dict(count=FAKE, root_cell=FAKE, part_cell=FAKE, part_score=FAKE, part_box=FAKE)
    f.update(moved)
    return _lib.PPNHumans(f["count"], f["root_cell"], f["part_cell"], f["part_score"], f["part_box"], R)


def match(_lib, R=8, **moved):
    f = dict(score=FAKE, label=FAKE, used=FAKE, flags=FAKE, n_gt=FAKE)
    f.update(moved)
    return _lib.PPNAPMatch(f["score"], f["label"], f["used"], f["flags"], f["n_gt"], R)


def gt(_lib, n=4, **moved):
    f = dict(person_off=FAKE, head_box=FAKE, joint_xy=FAKE, joint_valid=FAKE)
    f.update(moved)
    return _lib.PPNPoseGT(f["person_off"], f["head_box"], f["joint_xy"], f["joint_valid"], n)


def test_match_checks(abi):
    _lib, lib = abi

    def call(h=None, g=None, p=None, m=None, B=0, K=16, null=()):
        h = h or humans(_lib)
        g = g or gt(_lib)
        p = p or _lib.PPNAPParams(15, 0.5, 0.6)
        m = m or match(_lib)
        args = {"h": C.byref(h), "g": C.byref(g), "p": C.byref(p), "m": C.byref(m)}
        for k in null:
            args[k] = None
        return lib.ppn_ap_match(args["h"], B, K, args["g"], args["p"], args["m"], None)

    assert call() == 0                                                # B = 0: checked, nothing to do
    for k in ("h", "g", "p", "m"):
        assert call(null=(k,)) == -1
    assert call(B=-1) == -1 and call(K=0) == -1
    for J, rc in ((0, -1), (-3, -1), (33, -2), (64, -2), (32, 0), (1, 0)):
        assert call(p=_lib.PPNAPParams(J, 0.5, 0.6)) == rc, J
    for thr in (0.0, -0.5, float("nan")):
        assert call(p=_lib.PPNAPParams(15, thr, 0.6)) == -1
        assert call(p=_lib.PPNAPParams(15, 0.5, thr)) == -1
    assert call(p=_lib.PPNAPParams(15, float("inf"), 0.6)) == 0      # every finite distance matches: allowed
    for name in ("count", "part_cell", "part_score", "part_box"):
        assert call(h=humans(_lib, **{name: 0})) == -1
    assert call(h=humans(_lib, part_box=FAKE + 4)) == -1             # boxes are read as float4
    for name in ("score", "label", "used", "flags", "n_gt"):
        assert call(m=match(_lib, **{name: 0})) == -1
    assert call(m=match(_lib, score=FAKE + 2)) == -1
    assert call(m=match(_lib, R=4)) == -1                            # slot stride below the result's R
    assert call(m=match(_lib, R=16)) == 0
    assert call(g=gt(_lib, person_off=0)) == -1
    assert call(g=gt(_lib, n=-1)) == -1
    for name in ("head_box", "joint_xy", "joint_valid"):
        assert call(g=gt(_lib, **{name: 0})) == -1
        assert call(g=gt(_lib, n=0, **{name: 0})) == 0               # no GT rows: the arrays are never read
    assert call(g=gt(_lib, head_box=FAKE + 4)) == -1                 # float64


def test_workspace_and_finalize_checks(abi):
    _lib, lib = abi
    need = C.c_size_t()
    assert lib.ppn_ap_workspace_bytes(3000, 576, 17, C.byref(need)) == 0
    assert need.value >= 2 * 3000 * 576 * 17 * 8
    assert lib.ppn_ap_workspace_bytes(0, 576, 17, C.byref(need)) == -1
    assert lib.ppn_ap_workspace_bytes(8, 0, 17, C.byref(need)) == -1
    assert lib.ppn_ap_workspace_bytes(8, 8, 0, C.byref(need)) == -1
    assert lib.ppn_ap_workspace_bytes(8, 8, 33, C.byref(need)) == -2
    assert lib.ppn_ap_workspace_bytes(8, 8, 17, None) == -1
    assert lib.ppn_ap_workspace_bytes(1 << 20, 1024, 17, C.byref(need)) == -2   # the 31-bit entry ordinal
    N, R, J = 64, 8, 15
    assert lib.ppn_ap_workspace_bytes(N, R, J, C.byref(need)) == 0

    def fin(m=None, N=N, K=16, J=J, ap=FAKE, pre=FAKE, rec=FAKE, st=FAKE, ws=FAKE, n=need.value, null_m=False):
        m = m or match(_lib, R=R)
        return lib.ppn_ap_finalize(None if null_m else C.byref(m), N, K, J, ap, pre, rec, st, ws, n, None)

    assert fin(n=need.value - 1) == -3
    assert fin(n=0) == -3
    assert fin(null_m=True) == -1
    assert fin(m=match(_lib, R=R, label=0)) == -1
    assert fin(N=0) == -1 and fin(K=0) == -1
    assert fin(J=0) == -1 and fin(J=33) == -2
    for kw in ({"ap": None}, {"pre": FAKE + 4}, {"rec": None}, {"st": None}, {"ws": None}, {"ws": FAKE + 16}):
        assert fin(**kw) == -1, kw
