"""Host-side validation of the mixed-precision loss and encoder exports (ppn_loss_*_opt, ppn_encode_targets_opt).

Every rejection happens before anything touches a device, so the pointers are aligned fakes that are never
dereferenced and no GPU is needed.
"""
import ctypes as C

import pytest

from pytorch_pose_proposal_network_b200.config import PPNConfig

FAKE = 1 << 20                                                       # 256-byte aligned, never dereferenced


@pytest.fixture(scope="module")
def abi():
    from pytorch_pose_proposal_network_b200 import _lib
    from pytorch_pose_proposal_network_b200.parser import _CConfig
    return _lib, _lib.lib(), _CConfig(PPNConfig.mpii16())


def opt(_lib, limb):
    return _lib.PPNLossOptions(limb)


def test_workspace_is_the_fp32_workspace(abi):
    _lib, lib, cc = abi
    want = C.c_size_t()
    assert lib.ppn_loss_workspace_bytes(C.byref(cc.shape(512)), C.byref(want)) == 0
    for head, limb in ((_lib.HEAD_F32, _lib.HEAD_F32), (_lib.HEAD_F16, _lib.HEAD_F32), (_lib.HEAD_F16, _lib.HEAD_F16),
                       (_lib.HEAD_BF16, _lib.HEAD_F32), (_lib.HEAD_BF16, _lib.HEAD_BF16)):
        got = C.c_size_t()
        assert lib.ppn_loss_workspace_bytes_opt(C.byref(cc.shape(512, head)), C.byref(opt(_lib, limb)), C.byref(got)) == 0
        assert got.value == want.value


def test_unsupported_pairs_and_bad_options(abi):
    _lib, lib, cc = abi
    n = C.c_size_t()
    ws = lambda head, o: lib.ppn_loss_workspace_bytes_opt(C.byref(cc.shape(8, head)), o, C.byref(n))
    assert ws(_lib.HEAD_F32, C.byref(opt(_lib, _lib.HEAD_F16))) == -2           # fp32 head, 16-bit limb targets
    assert ws(_lib.HEAD_F32, C.byref(opt(_lib, _lib.HEAD_BF16))) == -2
    assert ws(_lib.HEAD_F16, C.byref(opt(_lib, _lib.HEAD_BF16))) == -2          # limb targets in the other 16-bit type
    assert ws(_lib.HEAD_BF16, C.byref(opt(_lib, _lib.HEAD_F16))) == -2
    assert ws(_lib.HEAD_F16, None) == -1
    assert ws(_lib.HEAD_F16, C.byref(opt(_lib, 3))) == -1
    assert ws(_lib.HEAD_F16, C.byref(opt(_lib, -1))) == -1
    assert lib.ppn_loss_workspace_bytes_opt(C.byref(cc.shape(0, _lib.HEAD_F16)), C.byref(opt(_lib, _lib.HEAD_F16)),
                                            C.byref(n)) == -1
    tg = _lib.PPNTargets(*[FAKE] * 10)
    fwd = lambda head, limb: lib.ppn_loss_forward_opt(FAKE, C.byref(cc.shape(8, head)), C.byref(tg), C.byref(opt(_lib, limb)),
                                                      FAKE, FAKE, 1 << 20, None)
    bwd = lambda head, limb: lib.ppn_loss_backward_opt(FAKE, C.byref(cc.shape(8, head)), C.byref(tg), C.byref(opt(_lib, limb)),
                                                       FAKE, FAKE, None)
    for f in (fwd, bwd):
        assert f(_lib.HEAD_F32, _lib.HEAD_F16) == -2
        assert f(_lib.HEAD_F16, _lib.HEAD_BF16) == -2
        assert f(_lib.HEAD_BF16, _lib.HEAD_F16) == -2
        assert f(_lib.HEAD_F16, 7) == -1


@pytest.mark.parametrize("head,limb", [("HEAD_F16", "HEAD_F16"), ("HEAD_BF16", "HEAD_F32")])
def test_pointer_checks(abi, head, limb):
    _lib, lib, cc = abi
    head, limb = getattr(_lib, head), getattr(_lib, limb)
    shape, o = cc.shape(64, head), opt(_lib, limb)
    need = C.c_size_t()
    assert lib.ppn_loss_workspace_bytes_opt(C.byref(shape), C.byref(o), C.byref(need)) == 0
    limb_step = 4 if limb == _lib.HEAD_F32 else 2                    # bytes per limb-target element

    def fwd(h=FAKE, t=None, ws=FAKE, n=need.value, loss=FAKE, op=o):
        t = t or _lib.PPNTargets(*[FAKE] * 10)
        return lib.ppn_loss_forward_opt(h, C.byref(shape), C.byref(t), C.byref(op) if op is not None else None, loss, ws, n, None)

    def bwd(h=FAKE, t=None, gl=FAKE, g=FAKE):
        t = t or _lib.PPNTargets(*[FAKE] * 10)
        return lib.ppn_loss_backward_opt(h, C.byref(shape), C.byref(t), C.byref(o), gl, g, None)

    def targets(**moved):
        return _lib.PPNTargets(*[moved.get(n, FAKE) for n in _lib.TARGET_NAMES])

    for f in (fwd, bwd):
        assert f(h=None) == -1
        assert f(h=FAKE + 1) == -1                                   # odd: no 16-bit head is there
        assert f(t=targets(te=0)) == -1
        assert f(t=targets(weight_ij=FAKE + 1)) == -1
        assert f(t=targets(te=FAKE + limb_step // 2)) == -1              # half an element off
        assert f(t=targets(delta=FAKE + 2)) == -1                    # the small targets are fp32
        assert f(t=targets(tx_half=0)) == -1
    assert fwd(op=None) == -1
    assert fwd(n=need.value - 1) == -3
    assert fwd(ws=FAKE + 4) == -1
    assert fwd(ws=None) == -1
    assert fwd(loss=FAKE + 2) == -1
    assert bwd(gl=None) == -1
    assert bwd(g=FAKE + 1) == -1                                     # the gradient has the head's type
    assert bwd(g=None) == -1


def test_fp32_exports_unchanged_for_16bit_shapes(abi):
    """The fp32 exports keep refusing 16-bit shapes; the 16-bit path is only reached through the _opt exports."""
    _lib, lib, cc = abi
    n = C.c_size_t()
    tg = _lib.PPNTargets(*[FAKE] * 10)
    for head in (_lib.HEAD_F16, _lib.HEAD_BF16):
        s = cc.shape(8, head)
        assert lib.ppn_loss_workspace_bytes(C.byref(s), C.byref(n)) == -2
        assert lib.ppn_loss_forward(FAKE, C.byref(s), C.byref(tg), FAKE, FAKE, 1 << 20, None) == -2
        assert lib.ppn_loss_backward(FAKE, C.byref(s), C.byref(tg), FAKE, FAKE, None) == -2


def test_encode_opt_argument_checks(abi):
    _lib, lib, cc = abi
    people = _lib.PPNPeople(FAKE, FAKE, FAKE, FAKE, FAKE)
    edges = (C.c_int32 * 30)(*([0, 1] * 15))
    tg = _lib.PPNTargets(*[FAKE] * 10)
    enc = lambda dtype, t=tg, s=cc.shape(4): lib.ppn_encode_targets_opt(C.byref(people), C.byref(s), edges, C.byref(t), dtype, None)
    assert enc(3) == -1
    assert enc(-1) == -1
    for dtype in (_lib.HEAD_F16, _lib.HEAD_BF16):
        assert enc(dtype, t=_lib.PPNTargets(*[0 if n == "te" else FAKE for n in _lib.TARGET_NAMES])) == -1
        assert enc(dtype, t=_lib.PPNTargets(*[FAKE + 8 if n == "weight_ij" else FAKE for n in _lib.TARGET_NAMES])) == -1
        assert enc(dtype, s=cc.shape(0)) == 0                         # an empty batch is a no-op
