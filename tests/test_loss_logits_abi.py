"""The loss on logits without a GPU: the host-side checks of ppn_loss_forward_logits, ppn_loss_backward_logits and
ppn_sigmoid, and the float64 restatement of the loss on logits against torch autograd through torch.sigmoid.

Every rejection happens before anything touches a device, so the pointers are aligned fakes that are never
dereferenced.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import ppn_loss as L
from pytorch_pose_proposal_network_b200.config import PPNConfig
from tests import loss_logits_ref as R
from tests.test_loss_model import encoded_targets, geometries

FAKE = 1 << 20                                                       # 256-byte aligned, never dereferenced


@pytest.fixture(scope="module")
def abi():
    from pytorch_pose_proposal_network_b200 import _lib
    from pytorch_pose_proposal_network_b200.parser import _CConfig
    return _lib, _lib.lib(), _CConfig(PPNConfig.mpii16())


def test_dtype_pairs_and_options(abi):
    _lib, lib, cc = abi
    tg = _lib.PPNTargets(*[FAKE] * 10)

    def fwd(head, o, B=8):
        return lib.ppn_loss_forward_logits(FAKE, C.byref(cc.shape(B, head)), C.byref(tg), o, FAKE, FAKE, 1 << 20, None)

    def bwd(head, o, B=8):
        return lib.ppn_loss_backward_logits(FAKE, C.byref(cc.shape(B, head)), C.byref(tg), o, FAKE, FAKE, None)

    opt = lambda limb: C.byref(_lib.PPNLossOptions(limb))
    for f in (fwd, bwd):
        assert f(_lib.HEAD_F32, opt(_lib.HEAD_F16)) == -2               # fp32 logits, 16-bit limb targets
        assert f(_lib.HEAD_F32, opt(_lib.HEAD_BF16)) == -2
        assert f(_lib.HEAD_F16, opt(_lib.HEAD_BF16)) == -2              # limb targets in the other 16-bit type
        assert f(_lib.HEAD_BF16, opt(_lib.HEAD_F16)) == -2
        assert f(_lib.HEAD_F16, opt(3)) == -1
        assert f(_lib.HEAD_F16, opt(-1)) == -1
        assert f(_lib.HEAD_F32, None) == -1                             # no options
        assert f(_lib.HEAD_F16, opt(_lib.HEAD_F16), B=0) == -1          # the batch mean needs an image
        assert f(_lib.HEAD_F32, opt(_lib.HEAD_F32), B=0) == -1


@pytest.mark.parametrize("head,limb", [("HEAD_F32", "HEAD_F32"), ("HEAD_F16", "HEAD_F16"), ("HEAD_BF16", "HEAD_F32")])
def test_pointer_checks(abi, head, limb):
    _lib, lib, cc = abi
    head, limb = getattr(_lib, head), getattr(_lib, limb)
    shape, o = cc.shape(64, head), _lib.PPNLossOptions(limb)
    need = C.c_size_t()
    assert lib.ppn_loss_workspace_bytes_opt(C.byref(shape), C.byref(o), C.byref(need)) == 0
    head_step = 4 if head == _lib.HEAD_F32 else 2
    limb_step = 4 if limb == _lib.HEAD_F32 else 2

    def targets(**moved):
        return _lib.PPNTargets(*[moved.get(n, FAKE) for n in _lib.TARGET_NAMES])

    def fwd(h=FAKE, t=None, ws=FAKE, n=need.value, loss=FAKE, null_targets=False):
        t = t or targets()
        return lib.ppn_loss_forward_logits(h, C.byref(shape), None if null_targets else C.byref(t), C.byref(o), loss, ws, n,
                                           None)

    def bwd(h=FAKE, t=None, gl=FAKE, g=FAKE, null_targets=False):
        t = t or targets()
        return lib.ppn_loss_backward_logits(h, C.byref(shape), None if null_targets else C.byref(t), C.byref(o), gl, g, None)

    for f in (fwd, bwd):
        assert f(h=None) == -1
        assert f(h=FAKE + head_step // 2) == -1                       # half an element off
        assert f(null_targets=True) == -1
        assert f(t=targets(te=0)) == -1
        assert f(t=targets(weight_ij=FAKE + limb_step // 2)) == -1
        assert f(t=targets(delta=FAKE + 2)) == -1                     # the small targets are fp32
        assert f(t=targets(th=0)) == -1
    assert fwd(loss=None) == -1
    assert fwd(loss=FAKE + 2) == -1
    assert fwd(n=need.value - 1) == -3
    assert fwd(ws=FAKE + 4) == -1
    assert fwd(ws=None) == -1
    assert bwd(gl=None) == -1
    assert bwd(gl=FAKE + 2) == -1
    assert bwd(g=None) == -1
    assert bwd(g=FAKE + head_step // 2) == -1                        # the gradient has the logits' type


def test_sigmoid_checks(abi):
    _lib, lib, _ = abi
    for dtype in (3, -1, 7):
        assert lib.ppn_sigmoid(FAKE, dtype, FAKE, 16, None) == -1      # unknown dtype, checked first
        assert lib.ppn_sigmoid(FAKE, dtype, FAKE, 0, None) == -1
    for dtype, step in ((_lib.HEAD_F32, 4), (_lib.HEAD_F16, 2), (_lib.HEAD_BF16, 2)):
        assert lib.ppn_sigmoid(None, dtype, FAKE, 16, None) == -1
        assert lib.ppn_sigmoid(FAKE, dtype, None, 16, None) == -1
        assert lib.ppn_sigmoid(FAKE + step // 2, dtype, FAKE, 16, None) == -1
        assert lib.ppn_sigmoid(FAKE, dtype, FAKE + 2, 16, None) == -1  # y is fp32
        assert lib.ppn_sigmoid(None, dtype, None, 0, None) == 0       # nothing to do: a no-op


@pytest.mark.parametrize("geo", list(geometries()))
@pytest.mark.parametrize("seed", range(2))
def test_restatement_on_logits_matches_autograd(geo, seed):
    """grad_logits (the chain rule written out as the kernels apply it) equals float64 autograd through torch.sigmoid;
    loss_terms is the restated loss of torch.sigmoid(logits)."""
    cfg = geometries()[geo]
    rng = np.random.default_rng(seed)
    B = 2
    targets = [torch.from_numpy(t) for t in encoded_targets(cfg, B, rng)]
    x = torch.from_numpy(rng.standard_normal((B, cfg.C, cfg.H, cfg.W)) * 4)
    x[0, :, 0, 0] = 40.0                                              # saturated cells: s = 1 - 4e-18, s' ~ 4e-18
    x[1, :, 1, 1] = -40.0
    g = rng.uniform(0.2, 3.0, 5)
    got = R.grad_logits(x, targets, cfg, g)
    xa = x.clone().requires_grad_(True)
    terms = L.loss_terms(torch.sigmoid(xa), *[t.double() for t in targets], cfg)
    sum(float(g[i]) * terms[i] for i in range(5)).backward()
    assert got.dtype == torch.float64
    torch.testing.assert_close(got, xa.grad, rtol=1e-12, atol=1e-15)
    np.testing.assert_array_equal(torch.stack(R.loss_terms(x, *targets, cfg=cfg)).numpy(),
                                  torch.stack(terms).detach().numpy())
