"""PPNLoss on logits (from_logits=True, ppn_loss_*_logits, ppn_sigmoid): the network's final sigmoid fused into the
loss kernels.

The contract under test: every logit x is widened exactly and replaced by s = sigmoid_f32(x) (fp32, never narrowed);
the existing loss runs on s; the gradient is (g_s * (1 - s)) * s, one rounding per operation, rounded once to the
logits' dtype.  So:
* loss.sigmoid (the library's s) is within 1 ulp of torch.sigmoid;
* in fp32 the gradient equals, bit for bit, the sigmoid-input kernels on s = loss.sigmoid(x) followed by torch's
  sigmoid backward in fp32, and the terms equal theirs up to the order of the fp64 sums;
* a 16-bit call equals the fp32 call on the widened inputs, the gradient converted to the head's dtype;
* the terms are held to the float64 restatement on logits (tests/loss_logits_ref.py) as the sigmoid-input terms are.
"""
import numpy as np
import pytest
import torch

from oracle import ppn_loss as L
from tests import loss_logits_ref as R
from tests.test_gpu_loss import geometry, gradnorm_weights, make_batch
from tests.test_gpu_loss_amp import mixed, same_bits, samples_for, shifted, widened

gpu = pytest.mark.gpu
I_WIJ, I_TE = L.ARG_ORDER.index("weight_ij"), L.ARG_ORDER.index("te")
F16, BF16, F32 = torch.float16, torch.bfloat16, torch.float32
COMBOS = [pytest.param(F16, F32, id="f16-limb32"), pytest.param(F16, F16, id="f16-limb16"),
          pytest.param(BF16, F32, id="bf16-limb32"), pytest.param(BF16, BF16, id="bf16-limb16")]


def crits(cfg):
    from pytorch_pose_proposal_network_b200 import PPNLoss
    return PPNLoss(cfg), PPNLoss(cfg, from_logits=True)


def sig(x):
    from pytorch_pose_proposal_network_b200 import loss
    return loss.sigmoid(x)


def logits_batch(cfg, B, seed, scale=3.0):
    """(fp32 logits, targets in the criterion's order) on cuda:0; the logits span the sigmoid's curved range and its
    tails."""
    _, targets = make_batch(cfg, B, seed)
    gen = torch.Generator(device="cuda").manual_seed(10_000 + seed)
    return torch.randn(B, cfg.C, cfg.H, cfg.W, device="cuda", generator=gen) * scale, targets


def via_sigmoid(crit, x, targets, g):
    """Today's route on fp32 logits: the sigmoid-input kernels on s = loss.sigmoid(x), then torch's sigmoid
    backward expression in fp32 (a * (1 - b) * b)."""
    s = sig(x)
    return (crit.backward_raw(s, *targets, grad_loss=g) * (1 - s)) * s


def ulp_diff(a, b):
    """|a - b| in units in the last place, for fp32 tensors of one sign (the sigmoid's range is [0, 1])."""
    return (a.view(torch.int32).long() - b.view(torch.int32).long()).abs()


@gpu
@pytest.mark.parametrize("dtype", [F32, F16, BF16])
def test_sigmoid_matches_torch(dtype):
    gen = torch.Generator(device="cuda").manual_seed(7)
    edges = torch.tensor([-88.7, -88.72, -88.73, -87.3, -103.0, -104.0, 16.6, 16.63, 17.0, 17.33, 17.34, 200.0, -200.0,
                          float("inf"), float("-inf"), 0.0, -0.0], device="cuda")
    near = torch.cat([edges + d for d in (-1e-3, 1e-3)] + [edges, torch.nextafter(edges, edges + 1),
                                                             torch.nextafter(edges, edges - 1)])
    x = torch.cat([torch.randn(1 << 22, device="cuda", generator=gen) * 8, near]).to(dtype)
    got = sig(x)
    assert got.dtype == F32 and got.shape == x.shape
    want = torch.sigmoid(x.float())
    d = ulp_diff(got, want)
    n_diff = int((d > 0).sum())
    print(f"\n{dtype}: {n_diff} of {x.numel()} elements differ from torch.sigmoid, at most {int(d.max())} ulp")
    assert int(d.max()) <= 1
    xf = x.float()
    assert torch.equal(got[xf == float("inf")], torch.ones_like(got[xf == float("inf")]))
    assert torch.equal(got[xf == float("-inf")], torch.zeros_like(got[xf == float("-inf")]))
    assert torch.equal(got[xf == 0], torch.full_like(got[xf == 0], 0.5))
    assert not torch.isnan(got).any()
    y2 = sig(x[:1 << 22].view(64, -1)[:, ::2])                        # a strided view is read as a copy
    assert torch.equal(y2, got[:1 << 22].view(64, -1)[:, ::2])
    assert sig(x[:0]).numel() == 0
    with pytest.raises(ValueError):
        sig(x.double())
    with pytest.raises(ValueError):
        sig(x.cpu())


@gpu
@pytest.mark.parametrize("geo,B", [("mpii16", 7), ("native", 2), ("k18_13x13", 5)])
def test_fp32_equals_sigmoid_route(geo, B):
    cfg = geometry(geo)
    x, targets = logits_batch(cfg, B, seed=400 + B)
    crit, crit_l = crits(cfg)
    g = gradnorm_weights(B)
    out = torch.full_like(x, float("nan"))                            # every element must be written
    crit_l.backward_raw(x, *targets, grad_loss=g, out=out)
    assert same_bits(out, via_sigmoid(crit, x, targets, g))
    terms = crit_l.forward_raw(x, *targets).cpu().numpy().astype(np.float64)
    np.testing.assert_allclose(terms, crit.forward_raw(sig(x), *targets).cpu().numpy(), rtol=1e-6, atol=0)
    want = R.terms_chunked(cfg, x, targets)
    assert np.all(want > 0)
    np.testing.assert_allclose(terms, want, rtol=1e-5, atol=0)


@gpu
@pytest.mark.parametrize("hd,ld", COMBOS)
@pytest.mark.parametrize("geo,B", [("mpii16", 7), ("native", 2), ("k18_13x13", 5)])
def test_16bit_equals_fp32_on_widened_inputs(geo, B, hd, ld):
    cfg = geometry(geo)
    x, targets = mixed(*logits_batch(cfg, B, seed=500 + B), hd, ld)
    wx, wt = widened(x, targets)
    _, crit_l = crits(cfg)
    g = gradnorm_weights(B)
    out = torch.full_like(x, float("nan"))
    crit_l.backward_raw(x, *targets, grad_loss=g, out=out)
    assert out.dtype == hd
    assert same_bits(out, crit_l.backward_raw(wx, *wt, grad_loss=g).to(hd))
    terms = crit_l.forward_raw(x, *targets).cpu().numpy().astype(np.float64)
    np.testing.assert_allclose(terms, crit_l.forward_raw(wx, *wt).cpu().numpy(), rtol=1e-6, atol=0)
    np.testing.assert_allclose(terms, R.terms_chunked(cfg, wx, wt), rtol=1e-5, atol=0)


@gpu
@pytest.mark.parametrize("scale", [65536.0, 2.0 ** 22])
@pytest.mark.parametrize("ld", [F32, F16])
def test_fp16_overflow_is_inf_as_torch_rounds_it(ld, scale):
    """GradScaler's initial scale (65536), and a larger one that must overflow, on every term at B = 1: gradient
    elements beyond fp16's range become +-inf exactly where rounding the fp32 gradient does, never NaN."""
    cfg = geometry("mpii16")
    x, targets = mixed(*logits_batch(cfg, 1, seed=65), F16, ld)
    _, crit_l = crits(cfg)
    g = torch.full((5,), scale, device="cuda")
    got = crit_l.backward_raw(x, *targets, grad_loss=g)
    wx, wt = widened(x, targets)
    want32 = crit_l.backward_raw(wx, *wt, grad_loss=g)
    assert torch.isfinite(want32).all()
    assert same_bits(got, want32.to(F16))
    assert not torch.isnan(got).any()
    assert torch.equal(torch.isinf(got), want32.abs() >= 65520)       # fp16's rounding boundary to inf
    if scale > 65536:
        assert torch.isinf(got).any()


@gpu
@pytest.mark.parametrize("hd,ld", [pytest.param(F32, F32, id="f32"), pytest.param(F16, F16, id="f16-limb16")])
@pytest.mark.parametrize("geo", ["mpii16", "k18_13x13"])
def test_alignment_phases(geo, hd, ld):
    """Every element offset within 16 bytes of logits, weight_ij, te and gradient, in every combination: the same
    gradient bits and terms every time."""
    cfg = geometry(geo)
    x, targets = mixed(*logits_batch(cfg, 3, seed=34), hd, ld)
    _, crit_l = crits(cfg)
    g = gradnorm_weights(34)
    ref_loss = crit_l.forward_raw(x, *targets)
    ref_grad = crit_l.backward_raw(x, *targets, grad_loss=g)
    ph, pl = 16 // x.element_size(), 16 // targets[I_TE].element_size()
    xs = [shifted(x, o) for o in range(ph)]
    wijs = [shifted(targets[I_WIJ], o) for o in range(pl)]
    tes = [shifted(targets[I_TE], o) for o in range(pl)]
    outs = [shifted(torch.empty_like(x), o) for o in range(ph)]
    losses = []
    for ox in range(ph):
        for ow in range(pl):
            for ot in range(pl):
                t2 = list(targets)
                t2[I_WIJ], t2[I_TE] = wijs[ow], tes[ot]
                losses.append(crit_l.forward_raw(xs[ox], *t2))
                for og in range(ph):
                    outs[og].fill_(float("nan"))
                    crit_l.backward_raw(xs[ox], *t2, grad_loss=g, out=outs[og])
                    assert same_bits(outs[og], ref_grad), (ox, ow, ot, og)
    np.testing.assert_allclose(torch.stack(losses).cpu().numpy(), np.tile(ref_loss.cpu().numpy(), (len(losses), 1)), rtol=1e-6)


@gpu
@pytest.mark.parametrize("hd", [F32, F16, BF16])
def test_saturated_logits(hd):
    """Logits whose sigmoid is exactly 0 or 1 (+-inf among them), in every channel of some cells and scattered over
    the limb block: finite terms, a zero gradient at exactly those elements, no NaN anywhere."""
    cfg = geometry("mpii16")
    x, targets = logits_batch(cfg, 4, seed=9)
    gen = torch.Generator(device="cuda").manual_seed(9)
    sat = torch.tensor([float("inf"), float("-inf"), 200.0, -200.0, 30.0, -100.0], device="cuda")
    x[0, :, 0, :] = sat[torch.randint(0, 6, (cfg.C, cfg.W), device="cuda", generator=gen)]       # whole rows of cells
    x[3] = sat[torch.randint(0, 6, x[3].shape, device="cuda", generator=gen)]                    # a whole image
    pick = torch.rand(x.shape, device="cuda", generator=gen) < 0.05
    x[pick] = sat[torch.randint(0, 6, (int(pick.sum()),), device="cuda", generator=gen)]
    x = x.to(hd)
    s = sig(x)
    saturated = (s == 0) | (s == 1)
    assert torch.equal(saturated, torch.isin(x.float(), sat.to(hd).float()))
    _, crit_l = crits(cfg)
    if hd != F32:
        targets = mixed(x, targets, hd, hd)[1]
    terms = crit_l.forward_raw(x, *targets)
    assert torch.isfinite(terms).all()
    grad = crit_l.backward_raw(x, *targets, grad_loss=gradnorm_weights(9))
    assert not torch.isnan(grad).any() and torch.isfinite(grad).all()
    assert (grad[saturated] == 0).all()
    assert (grad[~saturated] != 0).any()


@gpu
def test_native_batch_512_beyond_32_bit_offsets():
    """fp32 logits at native B = 512 (more than 2^31 elements per tensor): the gradient of a sample of images, the
    last among them, bit for bit against the sigmoid route on the whole batch; the terms against it and the float64
    restatement on logits."""
    from pytorch_pose_proposal_network_b200.dataset import TargetEncoder
    cfg = geometry("native")
    B = 512
    batch = TargetEncoder(cfg).encode(samples_for(cfg, B, seed=513, people=(0, 5)))
    targets = [getattr(batch, n) for n in L.ARG_ORDER]
    gen = torch.Generator(device="cuda").manual_seed(513)
    x = torch.empty(B, cfg.C, cfg.H, cfg.W, device="cuda")
    for b0 in range(0, B, 64):
        x[b0:b0 + 64] = torch.randn(64, cfg.C, cfg.H, cfg.W, device="cuda", generator=gen) * 3
    assert x.numel() > 2 ** 31 and targets[I_TE].numel() > 2 ** 31
    crit, crit_l = crits(cfg)
    g = gradnorm_weights(513)
    terms = crit_l.forward_raw(x, *targets).cpu().numpy().astype(np.float64)
    grad = torch.full_like(x, float("nan"))
    crit_l.backward_raw(x, *targets, grad_loss=g, out=grad)
    idx = torch.tensor([0, 255, 511], device="cuda")
    s = sig(x)
    np.testing.assert_allclose(terms, crit.forward_raw(s, *targets).cpu().numpy(), rtol=1e-6, atol=0)
    gs = crit.backward_raw(s, *targets, grad_loss=g)[idx]
    si = s[idx]
    assert same_bits(grad[idx], (gs * (1 - si)) * si)
    assert not torch.isnan(grad[-1]).any()
    del s, gs, grad
    np.testing.assert_allclose(terms, R.terms_chunked(cfg, x, targets, chunk=16), rtol=1e-5, atol=0)


def agreeing(x, cfg):
    """Elements whose gradient depends only on logits at which the library's sigmoid equals torch.sigmoid: a limb
    element on itself, a cell's six box channels on all six (the IoU couples them)."""
    a = sig(x) == torch.sigmoid(x.float())
    B, K = x.shape[0], cfg.K
    cells = a[:, :6 * K].view(B, 6, K, cfg.H, cfg.W).all(1, keepdim=True).expand(B, 6, K, cfg.H, cfg.W)
    return torch.cat([cells.reshape(B, 6 * K, cfg.H, cfg.W), a[:, 6 * K:]], 1)


def conv_setup(cfg, B, seed):
    torch.manual_seed(seed)
    conv = torch.nn.Conv2d(64, cfg.C, 1).cuda()
    feat = torch.randn(B, 64, cfg.H, cfg.W, device="cuda")
    return conv, feat


@gpu
def test_autograd_step_fp32():
    """conv -> PPNLoss(from_logits=True) against conv -> torch.sigmoid -> PPNLoss(cfg): the logits' gradient agrees
    bit for bit wherever it depends only on logits at which torch.sigmoid equals the library's sigmoid, the conv
    weight gradients to rtol 1e-5."""
    cfg = geometry("mpii16")
    B = 8
    targets = make_batch(cfg, B, seed=81)[1]
    conv, feat = conv_setup(cfg, B, 0)
    crit, crit_l = crits(cfg)
    lam = [0.3, 0.9, 0.6, 0.2, 0.25]

    def step(fused):
        conv.zero_grad(set_to_none=True)
        seen = {}
        logits = conv(feat)
        logits.register_hook(lambda grad: seen.setdefault("g", grad))
        terms = crit_l(logits, *targets) if fused else crit(torch.sigmoid(logits), *targets)
        loss = sum(l * t for l, t in zip(lam, terms))
        loss.backward()
        return logits.detach(), seen["g"], conv.weight.grad.clone(), conv.bias.grad.clone(), loss.detach()

    x, g_f, w_f, b_f, l_f = step(True)
    _, g_t, w_t, b_t, l_t = step(False)
    agree = agreeing(x, cfg)
    assert agree.float().mean().item() > 0.9
    assert torch.equal(g_f[agree], g_t[agree])
    for a, b in ((w_f, w_t), (b_f, b_t)):
        scale = b.abs().max().item()
        torch.testing.assert_close(a, b, rtol=1e-5, atol=1e-6 * scale)
    torch.testing.assert_close(l_f, l_t, rtol=1e-6, atol=0)


@gpu
@pytest.mark.parametrize("dtype", [F16, BF16])
def test_autograd_step_amp(dtype):
    """The same under autocast (fp16 with a GradScaler, bf16 without): the logits are 16-bit, and the fused route is
    compared with the upcast-logits route, crit(torch.sigmoid(logits.float()), ...) on the widened targets, whose
    gradient autograd rounds to the logits' dtype once, as the kernel does.  Tolerances: the logits' gradient bit for
    bit wherever the two sigmoids agree; the conv weight gradient, itself computed in 16 bits by autocast, to rtol
    1e-2 (fp16) / 3e-2 (bf16) of its largest element."""
    cfg = geometry("mpii16")
    B = 8
    targets = mixed(*make_batch(cfg, B, seed=89), dtype, dtype)[1]
    targets_wide = [t.float() for t in targets]
    conv, feat = conv_setup(cfg, B, 1)
    crit, crit_l = crits(cfg)
    lam = [0.3, 0.9, 0.6, 0.2, 0.25]

    def step(fused):
        conv.zero_grad(set_to_none=True)
        seen = {}
        scaler = torch.amp.GradScaler("cuda", init_scale=1024.0) if dtype == F16 else None
        with torch.autocast("cuda", dtype=dtype):
            logits = conv(feat)
            assert logits.dtype == dtype
            logits.register_hook(lambda grad: seen.setdefault("g", grad))
            terms = crit_l(logits, *targets) if fused else crit(torch.sigmoid(logits.float()), *targets_wide)
            loss = sum(l * t for l, t in zip(lam, terms))
        (scaler.scale(loss) if scaler is not None else loss).backward()
        return logits.detach(), seen["g"], conv.weight.grad.clone(), conv.bias.grad.clone(), loss.detach()

    x, g_f, w_f, b_f, l_f = step(True)
    _, g_u, w_u, b_u, l_u = step(False)
    assert g_f.dtype == dtype and torch.isfinite(g_f).all() and torch.isfinite(w_f).all()
    agree = agreeing(x, cfg)
    assert agree.float().mean().item() > 0.9
    assert same_bits(g_f[agree], g_u[agree])
    tol = dict(rtol=1e-2, atol=1e-3) if dtype == F16 else dict(rtol=3e-2, atol=1e-2)
    scale = max(w_u.abs().max().item(), 1e-30)
    torch.testing.assert_close(w_f / scale, w_u / scale, **tol)
    torch.testing.assert_close(b_f / scale, b_u / scale, **tol)
    torch.testing.assert_close(l_f, l_u, rtol=1e-6, atol=0)


@gpu
@pytest.mark.parametrize("hd", [F32, F16])
def test_peak_memory_below_the_sigmoid_route(hd):
    """The fused step allocates one gradient and nothing else head-sized; today's route (torch.sigmoid, the loss,
    autograd's sigmoid backward) holds at least one head-sized buffer more at its peak."""
    cfg = geometry("native")
    B = 8
    x, targets = mixed(*logits_batch(cfg, B, seed=8), hd, hd)
    crit, crit_l = crits(cfg)
    fm = x.clone().requires_grad_(True)

    def fused():
        fm.grad = None
        sum(crit_l(fm, *targets)).backward()

    def today():
        fm.grad = None
        sum(crit(torch.sigmoid(fm), *targets)).backward()

    def peak(fn):
        fn()                                                          # warm-up: workspace, lazy CUDA state
        fm.grad = None
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        fn()
        torch.cuda.synchronize()
        return torch.cuda.max_memory_allocated() - base

    head_bytes = fm.numel() * fm.element_size()
    m_fused, m_today = peak(fused), peak(today)
    assert fm.grad.dtype == hd
    assert head_bytes <= m_fused <= head_bytes + (1 << 20), (m_fused, head_bytes)
    assert m_today - m_fused >= head_bytes, (m_today, m_fused, head_bytes)


@gpu
def test_no_host_synchronisation_and_deterministic():
    cfg = geometry("mpii16")
    x, targets = mixed(*logits_batch(cfg, 64, seed=4), F16, F16)
    _, crit_l = crits(cfg)
    fm = x.clone().requires_grad_(True)
    sum(crit_l(fm, *targets)).backward()
    torch.cuda.synchronize()
    first = fm.grad.clone()
    fm.grad = None
    torch.cuda.set_sync_debug_mode("error")
    try:
        terms = crit_l(fm, *targets)
        sum(terms).backward()
        sig(x)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert same_bits(fm.grad, first)
    g = gradnorm_weights(4)
    a, b = crit_l.forward_raw(x, *targets), crit_l.forward_raw(x, *targets)
    assert same_bits(a, b) and same_bits(torch.stack(terms).detach(), a)
    assert same_bits(crit_l.backward_raw(x, *targets, grad_loss=g), crit_l.backward_raw(x, *targets, grad_loss=g))
    x32, t32 = logits_batch(cfg, 16, seed=5)
    assert same_bits(crit_l.backward_raw(x32, *t32, grad_loss=g), crit_l.backward_raw(x32, *t32, grad_loss=g))


@gpu
def test_from_batch_and_checks():
    """from_batch routes to the logits kernels too; the checks are those of the sigmoid-input loss."""
    from pytorch_pose_proposal_network_b200.dataset import TargetEncoder
    cfg = geometry("mpii16")
    batch = TargetEncoder(cfg).encode(samples_for(cfg, 3, seed=6))
    targets = [getattr(batch, n) for n in L.ARG_ORDER]
    gen = torch.Generator(device="cuda").manual_seed(6)
    x = torch.randn(3, cfg.C, cfg.H, cfg.W, device="cuda", generator=gen)
    crit, crit_l = crits(cfg)
    assert crit_l.from_logits and not crit.from_logits
    got = torch.stack(crit_l.from_batch(x, batch))
    assert same_bits(got, crit_l.forward_raw(x, *targets))
    np.testing.assert_allclose(got.cpu().numpy(), crit.forward_raw(sig(x), *targets).cpu().numpy(), rtol=1e-6)
    for bad in (x.double(), x[:, :-1].contiguous(), x.transpose(2, 3), x.cpu()):
        with pytest.raises(ValueError):
            crit_l.forward_raw(bad, *targets)
    with pytest.raises(ValueError):                                   # fp32 logits, 16-bit limb targets
        crit_l.forward_raw(x, *mixed(x, targets, F32, F16)[1])
    torch.cuda.synchronize()
