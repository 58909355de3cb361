"""Mixed-precision PPNLoss: fp16 / bf16 heads, gradients in the head's dtype, 16-bit te / weight_ij from the encoder.

The rule under test: a 16-bit input is the fp32 loss applied to the exactly widened inputs, and the gradient is that
fp32 gradient rounded once (round to nearest even) to the head's dtype.  So every check is against the existing fp32
kernels on `.float()` copies: the gradient bit for bit after `.to(head.dtype)`, the terms to 1e-6 (only the order of
the fp64 sums may differ), and the terms also against the float64 restatement.
"""
import numpy as np
import pytest
import torch

from oracle import encode_gt
from oracle import ppn_loss as L
from tests.test_gpu_loss import criterion, f64_terms, geometry, gradnorm_weights, make_batch

gpu = pytest.mark.gpu
I_WIJ, I_TE = L.ARG_ORDER.index("weight_ij"), L.ARG_ORDER.index("te")
F16, BF16, F32 = torch.float16, torch.bfloat16, torch.float32
COMBOS = [pytest.param(F16, F32, id="f16-limb32"), pytest.param(F16, F16, id="f16-limb16"),
          pytest.param(BF16, F32, id="bf16-limb32"), pytest.param(BF16, BF16, id="bf16-limb16")]


def mixed(head, targets, hd, ld):
    """The head in hd, te and weight_ij in ld, the eight small targets as they are (fp32)."""
    t = list(targets)
    t[I_WIJ], t[I_TE] = t[I_WIJ].to(ld), t[I_TE].to(ld)
    return head.to(hd), t


def widened(head, targets):
    return head.float(), [t.float() for t in targets]


def same_bits(a, b):
    assert a.dtype == b.dtype and a.shape == b.shape
    iv = {2: torch.int16, 4: torch.int32}[a.element_size()]
    return torch.equal(a.view(iv), b.view(iv))


def samples_for(cfg, B, seed, people=(0, 9)):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(B):
        kp, bb, vis, size = encode_gt.random_people(rng, int(rng.integers(*people)), cfg.K, cfg.insize)
        out.append(dict(keypoints=kp, bbox=np.asarray(bb).reshape(-1, 4), is_visible=vis, size=size))
    return out


@gpu
@pytest.mark.parametrize("hd,ld", COMBOS)
@pytest.mark.parametrize("geo,B", [("mpii16", 7), ("native", 2), ("k18_13x13", 5)])
def test_equals_fp32_kernels_on_widened_inputs(geo, B, hd, ld):
    cfg = geometry(geo)
    head, targets = mixed(*make_batch(cfg, B, seed=300 + B), hd, ld)
    wh, wt = widened(head, targets)
    crit = criterion(cfg)
    g = gradnorm_weights(B)
    out = torch.full_like(head, float("nan"))                         # every element must be written
    crit.backward_raw(head, *targets, grad_loss=g, out=out)
    assert same_bits(out, crit.backward_raw(wh, *wt, grad_loss=g).to(hd))
    terms = crit.forward_raw(head, *targets).cpu().numpy().astype(np.float64)
    np.testing.assert_allclose(terms, crit.forward_raw(wh, *wt).cpu().numpy(), rtol=1e-6, atol=0)
    want = f64_terms(cfg, wh, wt)
    assert np.all(want > 0)
    np.testing.assert_allclose(terms, want, rtol=1e-5, atol=0)


def shifted(t, off):
    """A contiguous copy of t whose storage starts `off` elements past a 16-byte boundary."""
    buf = torch.empty(t.numel() + 16 // t.element_size(), dtype=t.dtype, device=t.device)
    v = buf[off:off + t.numel()].view(t.shape)
    v.copy_(t)
    return v


@gpu
@pytest.mark.parametrize("hd,ld", [pytest.param(F16, F16, id="f16-limb16"), pytest.param(BF16, F32, id="bf16-limb32")])
@pytest.mark.parametrize("geo", ["mpii16", "k18_13x13"])
def test_alignment_phases(geo, hd, ld):
    """Every element offset within 16 bytes of head, weight_ij, te and gradient (8 for a 16-bit stream, 4 for an fp32
    one), in every combination: vectors from the first element where all streams are aligned, element-wise where there
    is none — the same gradient bits and terms every time."""
    cfg = geometry(geo)
    head, targets = mixed(*make_batch(cfg, 3, seed=33), hd, ld)
    crit = criterion(cfg)
    g = gradnorm_weights(33)
    ref_loss = crit.forward_raw(head, *targets)
    ref_grad = crit.backward_raw(head, *targets, grad_loss=g)
    wh, wt = widened(head, targets)
    assert same_bits(ref_grad, crit.backward_raw(wh, *wt, grad_loss=g).to(hd))
    ph, pl = 16 // head.element_size(), 16 // targets[I_TE].element_size()
    heads = [shifted(head, o) for o in range(ph)]
    wijs = [shifted(targets[I_WIJ], o) for o in range(pl)]
    tes = [shifted(targets[I_TE], o) for o in range(pl)]
    outs = [shifted(torch.empty_like(head), o) for o in range(ph)]
    losses = []
    for oh in range(ph):
        for ow in range(pl):
            for ot in range(pl):
                t2 = list(targets)
                t2[I_WIJ], t2[I_TE] = wijs[ow], tes[ot]
                losses.append(crit.forward_raw(heads[oh], *t2))
                for og in range(ph):
                    outs[og].fill_(float("nan"))
                    crit.backward_raw(heads[oh], *t2, grad_loss=g, out=outs[og])
                    assert same_bits(outs[og], ref_grad), (oh, ow, ot, og)
    np.testing.assert_allclose(torch.stack(losses).cpu().numpy(), np.tile(ref_loss.cpu().numpy(), (len(losses), 1)), rtol=1e-6)


@gpu
@pytest.mark.parametrize("ld", [F32, F16])
def test_fp16_overflow_is_inf_as_torch_rounds_it(ld):
    """GradScaler's initial scale (65536) on every term at B = 1: gradients beyond fp16's range become +-inf exactly
    where rounding the fp32 gradient does, never NaN."""
    cfg = geometry("mpii16")
    head, targets = mixed(*make_batch(cfg, 1, seed=65), F16, ld)
    crit = criterion(cfg)
    g = torch.full((5,), 65536.0, device="cuda")
    got = crit.backward_raw(head, *targets, grad_loss=g)
    wh, wt = widened(head, targets)
    want32 = crit.backward_raw(wh, *wt, grad_loss=g)
    assert torch.isfinite(want32).all()
    assert same_bits(got, want32.to(F16))
    assert torch.isinf(got).any() and not torch.isnan(got).any()
    assert torch.equal(torch.isinf(got), want32.abs() >= 65520)       # fp16's rounding boundary to inf


@gpu
@pytest.mark.parametrize("dtype", [F16, BF16])
def test_amp_training_step(dtype):
    """A 1x1 Conv2d(64 -> C) + sigmoid under autocast (fp16 with a GradScaler, bf16 without): the head is 16-bit, the
    gradient the loss hands to it equals bit for bit the one the upcast route (criterion(head.float(), ...)) delivers,
    and the weight gradients of the two routes agree."""
    cfg = geometry("mpii16")
    B = 8
    targets = mixed(*make_batch(cfg, B, seed=88), dtype, dtype)[1]
    targets_wide = [t.float() for t in targets]                       # what the upcast route sees: the same values
    torch.manual_seed(0)
    conv = torch.nn.Conv2d(64, cfg.C, 1).cuda()
    x = torch.randn(B, 64, cfg.H, cfg.W, device="cuda")
    crit = criterion(cfg)
    lam = [0.3, 0.9, 0.6, 0.2, 0.25]

    def step(upcast):
        conv.zero_grad(set_to_none=True)
        seen = {}
        # a scale at which the fp16 convolution's weight gradient does not overflow either (at the default 65536 it
        # does, in both routes alike: the step GradScaler would skip); overflow at 65536 has its own test above
        scaler = torch.amp.GradScaler("cuda", init_scale=1024.0) if dtype == F16 else None
        with torch.autocast("cuda", dtype=dtype):
            out = torch.sigmoid(conv(x))
            assert out.dtype == dtype
            out.register_hook(lambda grad: seen.setdefault("g", grad))
            terms = crit(out.float(), *targets_wide) if upcast else crit(out, *targets)
            loss = sum(l * t for l, t in zip(lam, terms))
        (scaler.scale(loss) if scaler is not None else loss).backward()
        return seen["g"], conv.weight.grad.clone(), conv.bias.grad.clone(), loss.detach()

    g_fused, w_fused, b_fused, l_fused = step(upcast=False)
    g_up, w_up, b_up, l_up = step(upcast=True)
    assert g_fused.dtype == dtype and torch.isfinite(g_fused).all()
    assert torch.isfinite(w_fused).all() and torch.isfinite(w_up).all()
    assert same_bits(g_fused, g_up)
    tol = dict(rtol=1e-2, atol=1e-3) if dtype == F16 else dict(rtol=3e-2, atol=1e-2)
    scale = max(w_up.abs().max().item(), 1e-30)
    torch.testing.assert_close(w_fused / scale, w_up / scale, **tol)
    torch.testing.assert_close(b_fused / scale, b_up / scale, **tol)
    torch.testing.assert_close(l_fused, l_up, rtol=1e-6, atol=0)


@gpu
@pytest.mark.parametrize("hd", [F16, BF16])
def test_memory_is_one_16bit_gradient(hd):
    """Forward + backward on a 16-bit head allocates the gradient in the head's dtype and nothing head-sized besides
    (the workspace exists from the warm-up call)."""
    cfg = geometry("native")
    B = 8
    head, targets = mixed(*make_batch(cfg, B, seed=8), hd, hd)
    crit = criterion(cfg)
    fm = head.clone().requires_grad_(True)
    sum(crit(fm, *targets)).backward()                               # warm-up: workspace, lazy CUDA state
    fm.grad = None
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    sum(crit(fm, *targets)).backward()
    torch.cuda.synchronize()
    extra = torch.cuda.max_memory_allocated() - base
    grad_bytes = fm.numel() * fm.element_size()
    assert fm.grad.dtype == hd
    assert grad_bytes <= extra <= grad_bytes + (1 << 20), (extra, grad_bytes)
    assert extra < fm.numel() * 4                                    # no fp32 head-sized buffer


@gpu
def test_no_host_synchronisation_and_deterministic():
    cfg = geometry("mpii16")
    head, targets = mixed(*make_batch(cfg, 64, seed=3), F16, F16)
    crit = criterion(cfg)
    fm = head.clone().requires_grad_(True)
    sum(crit(fm, *targets)).backward()
    torch.cuda.synchronize()
    first = fm.grad.clone()
    fm.grad = None
    torch.cuda.set_sync_debug_mode("error")
    try:
        terms = crit(fm, *targets)
        sum(terms).backward()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert same_bits(fm.grad, first)
    g = gradnorm_weights(3)
    a, b = crit.forward_raw(head, *targets), crit.forward_raw(head, *targets)
    assert same_bits(a, b) and same_bits(torch.stack(terms).detach(), a)
    assert same_bits(crit.backward_raw(head, *targets, grad_loss=g), crit.backward_raw(head, *targets, grad_loss=g))


@gpu
def test_native_batch_512_beyond_32_bit_offsets():
    """fp16 head and limb targets at native B = 512 (more than 2^31 elements per tensor), the targets from the 16-bit
    encoder: the gradient of a sample of images, the last among them, bit for bit against the fp32 kernels on the
    widened batch; the terms against them and the float64 restatement."""
    from pytorch_pose_proposal_network_b200.dataset import TargetEncoder
    cfg = geometry("native")
    B = 512
    batch = TargetEncoder(cfg, limb_dtype=F16).encode(samples_for(cfg, B, seed=512, people=(0, 5)))
    targets = [getattr(batch, n) for n in L.ARG_ORDER]
    gen = torch.Generator(device="cuda").manual_seed(512)
    head = torch.empty(B, cfg.C, cfg.H, cfg.W, dtype=F16, device="cuda")
    for b0 in range(0, B, 64):
        head[b0:b0 + 64] = torch.sigmoid(torch.randn(64, cfg.C, cfg.H, cfg.W, device="cuda", generator=gen))
    assert head.numel() > 2 ** 31 and targets[I_TE].numel() > 2 ** 31
    crit = criterion(cfg)
    g = gradnorm_weights(512)
    terms = crit.forward_raw(head, *targets).cpu().numpy().astype(np.float64)
    grad = torch.full_like(head, float("nan"))
    crit.backward_raw(head, *targets, grad_loss=g, out=grad)
    idx = torch.tensor([0, 255, 511], device="cuda")
    wh, wt = widened(head, targets)
    np.testing.assert_allclose(terms, crit.forward_raw(wh, *wt).cpu().numpy(), rtol=1e-6, atol=0)
    want = crit.backward_raw(wh, *wt, grad_loss=g)
    assert same_bits(grad[idx], want[idx].to(F16))
    del want, wh, wt
    np.testing.assert_allclose(terms, f64_terms(cfg, head, targets, chunk=16), rtol=1e-5, atol=0)


@gpu
@pytest.mark.parametrize("ld", [F16, BF16])
@pytest.mark.parametrize("sweep", [0, 1])
@pytest.mark.parametrize("geo", ["mpii16", "k18_13x13"])
def test_encoder_16bit_limb_targets(geo, sweep, ld):
    """te and weight_ij written in 16 bits equal the fp32 encoder's .to(dtype) bit for bit, the eight small targets
    are identical; both kernels (the address-order sweep and the per-image kernel), and H*W = 169, which is not a
    multiple of 4 (element-wise stores)."""
    from pytorch_pose_proposal_network_b200 import _lib
    from pytorch_pose_proposal_network_b200.dataset import TargetEncoder
    cfg = geometry(geo)
    samples = samples_for(cfg, 9, seed=17 + sweep, people=(0, 12))
    before = _lib.tune_get("encode.sweep")
    _lib.tune(encode_sweep=sweep)
    try:
        ref = TargetEncoder(cfg).encode(samples)
        got = TargetEncoder(cfg, limb_dtype=ld).encode(samples)
        torch.cuda.synchronize()
    finally:
        _lib.tune(encode_sweep=before)
    for n in _lib.TARGET_NAMES:
        a, b = getattr(got, n), getattr(ref, n)
        if n in ("te", "weight_ij"):
            assert a.dtype == ld and same_bits(a, b.to(ld)), n
        else:
            assert same_bits(a, b), n
    assert (ref.te == 1).any() and (ref.weight_ij == 1).any()
    low = torch.tensor(0.0005, dtype=torch.float32).to(ld).item()
    assert set(got.weight_ij.unique().float().tolist()) == {low, 1.0}
    assert low == {F16: 0.0005002021789550781, BF16: 0.000499725341796875}[ld]


@gpu
def test_bad_input():
    from pytorch_pose_proposal_network_b200.dataset import TargetEncoder
    cfg = geometry("mpii16")
    head32, targets32 = make_batch(cfg, 3, seed=1)
    head, targets = mixed(head32, targets32, F16, F16)
    crit = criterion(cfg)
    crit.forward_raw(head, *targets)                                  # the valid call
    bad = [
        (head, [t.half() if i == 0 else t for i, t in enumerate(targets)]),               # a 16-bit small target
        (head, [t.to(BF16) if i in (I_WIJ, I_TE) else t for i, t in enumerate(targets)]),  # the other 16-bit type
        (head, [t.float() if i == I_WIJ else t for i, t in enumerate(targets)]),          # mixed limb dtypes
        (head, [t.float() if i == I_TE else t for i, t in enumerate(targets)]),
        (head32, targets),                                                                 # fp32 head, 16-bit limbs
        (head.to(BF16), targets),
    ]
    for h, ts in bad:
        with pytest.raises(ValueError):
            crit.forward_raw(h, *ts)
        with pytest.raises(ValueError):
            crit(h, *ts)
    g = torch.ones(5, device="cuda")
    with pytest.raises(ValueError):
        crit.backward_raw(head, *targets, grad_loss=g, out=torch.empty_like(head32))
    with pytest.raises(ValueError):
        crit.backward_raw(head, *targets, grad_loss=g, out=torch.empty_like(head, dtype=BF16))
    with pytest.raises(ValueError):
        TargetEncoder(cfg, limb_dtype=torch.float64)
    enc = TargetEncoder(cfg, limb_dtype=F16)
    with pytest.raises(ValueError):                                   # an fp32 batch handed to a 16-bit encoder
        enc.encode(samples_for(cfg, 2, seed=2), out=TargetEncoder(cfg).alloc(2))
    torch.cuda.synchronize()
