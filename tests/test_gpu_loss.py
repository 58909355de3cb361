"""PPNLoss on the GPU (ppn_loss_forward / ppn_loss_backward) against the restatement of oracle/ppn_loss.py.

Targets come from TargetEncoder on encode_gt.random_people, heads are sigmoid(randn).  Tolerances:
* terms: relative 1e-5 of the float64 restatement (fp32 elements, fp64 accumulation in the kernel);
* gradient: the limb block and the resp channels bit for bit against the float32 model (grad_model_f32: the same
  operation order); every channel within RTOL of float64 autograd plus ATOL_REL times the channel group's largest
  magnitude (the IoU part of d/dx, d/dw can cancel the coordinate / size part, so an element's own magnitude is no
  scale for the fp32 rounding it carries; that rounding is ~1e-7 of the group's scale).
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import encode_gt
from oracle import ppn_loss as L

gpu = pytest.mark.gpu
RTOL, ATOL_REL = 1e-4, 1e-6
TERM_RTOL = 1e-5


def geometry(name):
    from pytorch_pose_proposal_network_b200.config import PPNConfig
    return {"mpii16": PPNConfig.mpii16(), "native": PPNConfig.reference_native(),
            "k18_13x13": PPNConfig.reference_native(insize=(416, 416), outsize=(13, 13), local_grid_size=(7, 7))}[name]


def make_batch(cfg, B, seed, people=(0, 9)):
    """(head, targets in the criterion's order) on cuda:0."""
    from pytorch_pose_proposal_network_b200.dataset import TargetEncoder
    rng = np.random.default_rng(seed)
    samples = []
    for _ in range(B):
        kp, bb, vis, size = encode_gt.random_people(rng, int(rng.integers(*people)), cfg.K, cfg.insize)
        samples.append(dict(keypoints=kp, bbox=np.asarray(bb).reshape(-1, 4), is_visible=vis, size=size))
    batch = TargetEncoder(cfg).encode(samples)
    gen = torch.Generator(device="cuda").manual_seed(seed)
    head = torch.sigmoid(torch.randn(B, cfg.C, cfg.H, cfg.W, device="cuda", generator=gen))
    return head, [getattr(batch, n) for n in L.ARG_ORDER]


def criterion(cfg):
    from pytorch_pose_proposal_network_b200 import PPNLoss
    return PPNLoss(cfg)


def bits(t):
    a = t.cpu().numpy() if isinstance(t, torch.Tensor) else t
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def f64_terms(cfg, head, targets, chunk=None):
    """The restatement in float64 on the GPU, chunk-wise over the batch (sum of chunk means * chunk size / B)."""
    B = head.shape[0]
    chunk = chunk or B
    acc = torch.zeros(5, dtype=torch.float64, device=head.device)
    for b0 in range(0, B, chunk):
        sl = slice(b0, min(B, b0 + chunk))
        t = L.loss_terms(head[sl].double(), *[x[sl].double() for x in targets], cfg)
        acc += torch.stack(t) * (sl.stop - sl.start)
    return (acc / B).cpu().numpy()


def check_grad(cfg, head, targets, grad_loss, got, batch=None):
    """got: the kernel's gradient of the images in `head` (a sample of a batch of `batch` images)."""
    K = cfg.K
    B = batch or head.shape[0]
    model = L.grad_model_f32(head.cpu().numpy(), *[t.cpu().numpy() for t in targets], cfg, grad_loss.cpu().numpy(),
                             batch=B)
    g = got.cpu().numpy()
    assert np.array_equal(bits(g[:, 6 * K:]), bits(model[:, 6 * K:])), "limb block"
    assert np.array_equal(bits(g[:, :K]), bits(model[:, :K])), "resp"
    want = L.autograd_grad(head, targets, cfg, grad_loss).cpu().numpy() * (head.shape[0] / B)
    groups = [slice(i * K, (i + 1) * K) for i in range(6)] + [slice(6 * K, cfg.C)]
    for gi, sl in enumerate(groups):
        a, w = g[:, sl].astype(np.float64), want[:, sl]
        bad = np.abs(a - w) > RTOL * np.abs(w) + ATOL_REL * max(np.abs(w).max(), 1e-30)
        assert not bad.any(), (gi, int(bad.sum()), float(np.abs(a - w).max()))


def gradnorm_weights(seed):
    return torch.from_numpy(np.random.default_rng(seed).uniform(0.2, 3.0, 5).astype(np.float32)).cuda()


@gpu
@pytest.mark.parametrize("geo,B", [("mpii16", 1), ("mpii16", 7), ("mpii16", 512), ("native", 1), ("native", 16),
                                   ("k18_13x13", 5)])
def test_terms_match_restatement(geo, B):
    cfg = geometry(geo)
    head, targets = make_batch(cfg, B, seed=B)
    got = criterion(cfg).forward_raw(head, *targets).cpu().numpy().astype(np.float64)
    want = f64_terms(cfg, head, targets, chunk=64)
    assert np.all(want > 0)
    np.testing.assert_allclose(got, want, rtol=TERM_RTOL, atol=0)


@gpu
@pytest.mark.parametrize("geo,B", [("mpii16", 7), ("native", 2), ("k18_13x13", 5)])
def test_gradient(geo, B):
    cfg = geometry(geo)
    head, targets = make_batch(cfg, B, seed=100 + B)
    g = gradnorm_weights(B)
    out = torch.full_like(head, float("nan"))                         # every element must be written
    criterion(cfg).backward_raw(head, *targets, grad_loss=g, out=out)
    assert not torch.isnan(out).any()
    check_grad(cfg, head, targets, g, out)


def shifted(t, off):
    """A contiguous copy of t whose storage starts `off` floats past a 16-byte boundary."""
    buf = torch.empty(t.numel() + 4, dtype=t.dtype, device=t.device)
    v = buf[off:off + t.numel()].view(t.shape)
    v.copy_(t)
    return v


@gpu
@pytest.mark.parametrize("geo", ["mpii16", "k18_13x13"])
def test_mixed_alignment_phases(geo):
    """Every combination of the four streams' phases within 16 bytes (head, weight_ij, te, gradient: 4^4): vectors
    where the phases agree, element-wise where they differ — the same gradient bits and terms every time."""
    cfg = geometry(geo)
    B = 3
    head, targets = make_batch(cfg, B, seed=31)
    crit = criterion(cfg)
    g = gradnorm_weights(31)
    ref_loss = crit.forward_raw(head, *targets)
    ref_grad = crit.backward_raw(head, *targets, grad_loss=g)
    i_wij, i_te = L.ARG_ORDER.index("weight_ij"), L.ARG_ORDER.index("te")
    heads = [shifted(head, o) for o in range(4)]
    wijs = [shifted(targets[i_wij], o) for o in range(4)]
    tes = [shifted(targets[i_te], o) for o in range(4)]
    outs = [shifted(torch.empty_like(head), o) for o in range(4)]
    deltas = [shifted(targets[0], o) for o in range(4)]               # the small planes are read element-wise anyway
    losses = []
    for oh in range(4):
        for ow in range(4):
            for ot in range(4):
                t2 = list(targets)
                t2[0], t2[i_wij], t2[i_te] = deltas[(oh + ot) % 4], wijs[ow], tes[ot]
                losses.append(crit.forward_raw(heads[oh], *t2))
                for og in range(4):
                    outs[og].fill_(float("nan"))
                    crit.backward_raw(heads[oh], *t2, grad_loss=g, out=outs[og])
                    assert torch.equal(outs[og].view(torch.int32), ref_grad.view(torch.int32)), (oh, ow, ot, og)
    np.testing.assert_allclose(torch.stack(losses).cpu().numpy(), np.tile(ref_loss.cpu().numpy(), (64, 1)), rtol=1e-6)
    check_grad(cfg, head, targets, g, ref_grad)
    np.testing.assert_allclose(ref_loss.cpu().numpy(), f64_terms(cfg, head, targets), rtol=TERM_RTOL)


@gpu
@pytest.mark.parametrize("geo", ["mpii16", "k18_13x13"])
def test_gradient_on_kinks(geo):
    """The kernel's IoU branches at their kinks: equal predicted and target edges (min / max ties split evenly),
    boxes that only touch (relu'(0) = 0), zero-area boxes, a random 0/1 delta — the CPU test's dyadic case, exact in
    float32 and float64, with a non-zero IoU weight so that those branches carry gradient."""
    from tests.test_loss_model import kink_case
    cfg = geometry(geo)
    head_np, targets_np, kind = kink_case(cfg, np.random.default_rng(7))
    head = torch.from_numpy(head_np).cuda()
    targets = [torch.from_numpy(t).cuda() for t in targets_np]
    g = torch.tensor([0.7, 1.9, 1.3, 0.4, 2.2], device="cuda")
    out = torch.full_like(head, float("nan"))
    criterion(cfg).backward_raw(head, *targets, grad_loss=g, out=out)
    K = cfg.K
    dw = out[:, 4 * K:5 * K].cpu().numpy()
    on = targets_np[0] == 1
    # boxes sharing their left edge (kind 2, a max tie): d/dw is carried by the IoU chain through the tie
    assert np.count_nonzero(dw[(kind == 2) & on]) > 100
    check_grad(cfg, head, targets, g, out)
    np.testing.assert_allclose(criterion(cfg).forward_raw(head, *targets).cpu().numpy(), f64_terms(cfg, head, targets),
                               rtol=TERM_RTOL)


@gpu
def test_device_argument_and_from_batch():
    """PPNLoss(cfg, device="cuda") means the current device; from_batch takes the targets by name, so it equals the
    call in the criterion's order (and not the TargetBatch.as_list() order)."""
    from pytorch_pose_proposal_network_b200 import PPNLoss
    from pytorch_pose_proposal_network_b200.dataset import TargetEncoder
    cfg = geometry("mpii16")
    crit = PPNLoss(cfg, device="cuda")
    assert crit.device == torch.device("cuda", torch.cuda.current_device())
    with pytest.raises(ValueError):
        PPNLoss(cfg, device="cpu")
    rng = np.random.default_rng(4)
    samples = []
    for _ in range(5):
        kp, bb, vis, size = encode_gt.random_people(rng, 4, cfg.K, cfg.insize)
        samples.append(dict(keypoints=kp, bbox=np.asarray(bb).reshape(-1, 4), is_visible=vis, size=size))
    batch = TargetEncoder(cfg).encode(samples)
    head = torch.sigmoid(torch.randn(5, cfg.C, cfg.H, cfg.W, device="cuda"))
    by_name = torch.stack(crit.from_batch(head, batch))
    ordered = torch.stack(crit(head, *[getattr(batch, n) for n in L.ARG_ORDER]))
    as_list = torch.stack(crit(head, *batch.as_list()))
    assert torch.equal(by_name, ordered)
    assert not torch.equal(by_name, as_list)


@gpu
def test_deterministic():
    cfg = geometry("mpii16")
    head, targets = make_batch(cfg, 512, seed=5)
    crit = criterion(cfg)
    g = gradnorm_weights(5)
    a, b = crit.forward_raw(head, *targets), crit.forward_raw(head, *targets)
    ga, gb = crit.backward_raw(head, *targets, grad_loss=g), crit.backward_raw(head, *targets, grad_loss=g)
    assert np.array_equal(bits(a), bits(b))
    assert np.array_equal(bits(ga), bits(gb))


@gpu
def test_autograd():
    cfg = geometry("mpii16")
    head, targets = make_batch(cfg, 7, seed=9)
    crit = criterion(cfg)
    lam = [0.7, 1.9, 1.3, 0.4, 2.2]
    fm = head.clone().requires_grad_(True)
    targets = [t.clone().requires_grad_(True) for t in targets]
    terms = crit(fm, *targets)
    assert len(terms) == 5 and all(t.dim() == 0 for t in terms)
    sum(l * t for l, t in zip(lam, terms)).backward()
    direct = crit.backward_raw(head, *[t.detach() for t in targets], grad_loss=torch.tensor(lam, device="cuda"))
    assert np.array_equal(bits(fm.grad), bits(direct))
    assert all(t.grad is None for t in targets)                       # the targets get no gradient
    # only one term used: the others' upstream gradients are None, i.e. zero
    fm2 = head.clone().requires_grad_(True)
    crit(fm2, *targets)[4].backward()
    limb_only = crit.backward_raw(head, *[t.detach() for t in targets],
                                  grad_loss=torch.tensor([0, 0, 0, 0, 1.0], device="cuda"))
    assert np.array_equal(bits(fm2.grad), bits(limb_only))
    assert torch.count_nonzero(fm2.grad[:, :6 * cfg.K]) == 0
    # the terms as tensors: same values as the raw export
    raw = crit.forward_raw(head, *[t.detach() for t in targets])
    assert np.array_equal(bits(torch.stack([t.detach() for t in terms])), bits(raw))


@gpu
def test_no_host_synchronisation():
    cfg = geometry("mpii16")
    head, targets = make_batch(cfg, 64, seed=3)
    crit = criterion(cfg)
    fm = head.clone().requires_grad_(True)
    sum(crit(fm, *targets)).backward()                                # warm-up: workspace, lazy CUDA state
    torch.cuda.synchronize()
    fm.grad = None
    torch.cuda.set_sync_debug_mode("error")
    try:
        terms = crit(fm, *targets)
        (0.5 * terms[0] + terms[1] + 2.0 * terms[4]).backward()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert torch.isfinite(fm.grad).all()


@gpu
@pytest.mark.parametrize("geo", ["mpii16", "native"])
def test_perfect_prediction(geo):
    """encoder -> the head that reproduces its targets, assembled on the device -> four terms and their gradient
    exactly zero; L_iou only the eps residual.  The targets passed in TargetBatch.as_list() order (tx, ty before
    tx_half, ty_half) is caught: then L_coor is not zero."""
    cfg = geometry(geo)
    B = 16
    _, targets = make_batch(cfg, B, seed=77, people=(2, 9))
    t = dict(zip(L.ARG_ORDER, targets))
    head = torch.cat([t["delta"], torch.ones_like(t["delta"]), t["tx_half"], t["ty_half"], t["tw"], t["th"],
                      t["te"].reshape(B, -1, cfg.H, cfg.W)], 1).contiguous()
    crit = criterion(cfg)
    terms = crit.forward_raw(head, *targets).cpu().numpy()
    assert terms[0] == 0 and terms[2] == 0 and terms[3] == 0 and terms[4] == 0, terms
    want_iou = f64_terms(cfg, head, targets)[1]
    # float64: the eps residual alone (< 1e-12); float32 adds the rounding of the box edges (|1 - iou| ~ 1e-7 at
    # most per cell), still negligible next to any training loss
    assert want_iou <= 1e-12 and 0 <= terms[1] < 1e-6
    grad = crit.backward_raw(head, *targets, grad_loss=torch.tensor([1.0, 0, 1.0, 1.0, 1.0], device="cuda"))
    assert torch.count_nonzero(grad) == 0
    swapped = [t[n] for n in ("delta", "weight", "weight_ij", "tx", "ty", "tx_half", "ty_half", "tw", "th", "te")]
    assert crit.forward_raw(head, *swapped)[2].item() > 0


@gpu
def test_native_batch_512_beyond_32_bit_offsets():
    """2.2e9 elements per tensor: terms against the chunk-wise float64 restatement, the gradient of a sample of
    images (the last one among them: its offsets do not fit 32 bits) against the model and autograd."""
    cfg = geometry("native")
    B = 512
    head, targets = make_batch(cfg, B, seed=512, people=(0, 5))
    assert head.numel() > 2 ** 31
    crit = criterion(cfg)
    got = crit.forward_raw(head, *targets).cpu().numpy().astype(np.float64)
    np.testing.assert_allclose(got, f64_terms(cfg, head, targets, chunk=16), rtol=TERM_RTOL, atol=0)
    g = gradnorm_weights(512)
    grad = torch.full_like(head, float("nan"))
    crit.backward_raw(head, *targets, grad_loss=g, out=grad)
    idx = torch.tensor([0, 255, 511], device="cuda")
    assert not torch.isnan(grad[idx]).any()
    check_grad(cfg, head[idx].contiguous(), [t[idx].contiguous() for t in targets], g, grad[idx], batch=B)


@gpu
def test_bad_input():
    from pytorch_pose_proposal_network_b200 import _lib
    cfg = geometry("mpii16")
    head, targets = make_batch(cfg, 3, seed=1)
    crit = criterion(cfg)
    bad = [
        (head.double(), targets),
        (head[:, :-1], targets),
        (head.cpu(), targets),
        (head.transpose(2, 3), targets),
        (head, targets[:-1]),
        (head, [t.half() if i == 0 else t for i, t in enumerate(targets)]),
        (head, [t[:2] if i == 2 else t for i, t in enumerate(targets)]),
        (head, [t.cpu() if i == 9 else t for i, t in enumerate(targets)]),
        (head, [t.transpose(2, 3) if i == 5 else t for i, t in enumerate(targets)]),
    ]
    for h, ts in bad:
        with pytest.raises(ValueError):
            crit.forward_raw(h, *ts)
    with pytest.raises(ValueError):
        crit.backward_raw(head, *targets, grad_loss=torch.ones(4, device="cuda"))
    # the C ABI
    lib = _lib.lib()
    shape = crit._shape(3)
    tg = crit._targets_struct(targets)
    need = C.c_size_t()
    assert lib.ppn_loss_workspace_bytes(C.byref(shape), C.byref(need)) == 0
    ws = torch.empty(need.value, dtype=torch.uint8, device="cuda")
    loss = torch.empty(5, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    fwd = lambda h, s=shape, t=tg, w=ws.data_ptr(), n=need.value: lib.ppn_loss_forward(h, C.byref(s), C.byref(t),
                                                                                       loss.data_ptr(), w, n, st)
    assert fwd(head.data_ptr()) == 0
    assert fwd(None) == -1
    assert fwd(head.data_ptr() + 2) == -1                              # misaligned
    assert fwd(head.data_ptr(), n=need.value - 8) == -3
    assert fwd(head.data_ptr(), w=None) == -1
    t_null = _lib.PPNTargets(*[0 if n == "tx_half" else getattr(tg, n) for n in _lib.TARGET_NAMES])
    assert fwd(head.data_ptr(), t=t_null) == -1
    half = crit.c.shape(3, _lib.HEAD_F16)
    assert fwd(head.data_ptr(), s=half) == -2
    grad = torch.empty_like(head)
    gl = torch.ones(5, device="cuda")
    assert lib.ppn_loss_backward(head.data_ptr(), C.byref(shape), C.byref(tg), gl.data_ptr(), grad.data_ptr(), st) == 0
    assert lib.ppn_loss_backward(head.data_ptr(), C.byref(half), C.byref(tg), gl.data_ptr(), grad.data_ptr(), st) == -2
    assert lib.ppn_loss_backward(head.data_ptr(), C.byref(shape), C.byref(tg), None, grad.data_ptr(), st) == -1
    assert lib.ppn_loss_backward(head.data_ptr(), C.byref(shape), C.byref(tg), gl.data_ptr(), grad.data_ptr() + 1, st) == -1
    torch.cuda.synchronize()
