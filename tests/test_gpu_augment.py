"""ppn_augment_images / ppn_augment_people on the GPU against oracle/augment.py, bit for bit, on the parameters the
sampler produced (read back from the device)."""
import numpy as np
import pytest
import torch

from oracle import augment as OA, encode_gt

pytestmark = pytest.mark.gpu

DTYPES = {torch.float32: "float32", torch.float16: "float16", torch.bfloat16: "bfloat16"}
NAMES = ("delta", "weight", "weight_ij", "tx", "ty", "tx_half", "ty_half", "tw", "th", "te")


def cfg_of(preset):
    from pytorch_pose_proposal_network_b200.config import PRESETS
    return PRESETS[preset]()


def images_of(sizes, seed):
    rng = np.random.default_rng(seed)
    return [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in sizes]


def ragged_sizes(B, seed, big=True):
    """Mixed sources: 1 x 1, odd widths, 320 x 240 up to 1920 x 1080."""
    rng = np.random.default_rng(seed)
    fixed = [(1, 1), (1080, 1920), (240, 320), (719, 1281), (7, 3), (2, 1)] if big else [(1, 1), (37, 3), (2, 1)]
    hi = 1081 if big else 300
    sizes = [(int(rng.integers(1, hi)), int(rng.integers(1, hi)) | 1) for _ in range(B)]
    sizes[:len(fixed)] = fixed[:B]
    return sizes


def host_out(t, dtype):
    """[B, 3, H, W] device tensor -> numpy in the oracle's representation (bf16 as uint16 bits)."""
    t = t.detach().cpu().contiguous()
    if dtype == torch.bfloat16:
        return t.view(torch.int16).numpy().view(np.uint16)
    return t.numpy()


def check_images(aug, imgs, params, out, where, every=1):
    M = params.M.cpu().numpy()
    got = host_out(out, aug.dtype)
    for b in range(0, len(imgs), every):
        want = OA.warp_image(imgs[b], M[b], aug.cfg.insize, fill=tuple(aug.norm.fill), in_scale=aug.norm.in_scale,
                             mean=tuple(aug.norm.mean), std=tuple(aug.norm.std), dtype=DTYPES[aug.dtype])
        g = got[b]
        if g.dtype != np.uint16:                                   # compare bit patterns
            bits = np.uint32 if g.dtype == np.float32 else np.uint16
            g, want = g.view(bits), want.view(bits)
        bad = np.flatnonzero(g != want)
        assert bad.size == 0, f"{where}: image {b} ({imgs[b].shape}) differs in {bad.size} elements, first {np.unravel_index(bad[0], g.shape)}"


def augmenter(cfg, **kw):
    from pytorch_pose_proposal_network_b200.augment import Augmenter
    return Augmenter(cfg, **kw)


def batch_of(imgs):
    from pytorch_pose_proposal_network_b200.augment import ImageBatch
    return ImageBatch.from_arrays(imgs)


@pytest.mark.parametrize("channels_last", [False, True])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16])
def test_ragged_batch_bit_exact(dtype, channels_last):
    cfg = cfg_of("native")
    imgs = images_of(ragged_sizes(64, 1), 2)
    batch = batch_of(imgs)
    assert (batch.offset_host % 16 != 0).sum() > 30                 # unaligned image offsets
    aug = augmenter(cfg, dtype=dtype, channels_last=channels_last, fill=(12.0, 0.0, 255.0))
    params = aug.sample(batch, torch.Generator(device="cuda").manual_seed(5))
    out = aug.images(batch, params)
    assert out.shape == (64, 3, 384, 384) and out.dtype == dtype
    assert out.is_contiguous(memory_format=torch.channels_last if channels_last else torch.contiguous_format)
    check_images(aug, imgs, params, out, f"{dtype} channels_last={channels_last}")


@pytest.mark.parametrize("B,preset,dtype,channels_last", [(1, "cfg2", torch.float32, False), (512, "cfg2", torch.float32, False),
                                                           (512, "cfg2", torch.bfloat16, True), (7, "cfg3", torch.float16, True)])
def test_batch_sizes(B, preset, dtype, channels_last):
    cfg = cfg_of(preset)
    imgs = images_of(ragged_sizes(B, 10 + B, big=B < 100), 11)
    batch = batch_of(imgs)
    aug = augmenter(cfg, dtype=dtype, channels_last=channels_last)
    params = aug.sample(batch, torch.Generator(device="cuda").manual_seed(B))
    out = aug.images(batch, params)
    check_images(aug, imgs, params, out, f"B={B}", every=1 if B < 100 else 7)


@pytest.mark.parametrize("scale", [(0.2, 0.3), (3.0, 6.0)])
def test_minification_and_magnification(scale):
    """Strong minification (always gathered) and magnification (staged when a staging budget is set); the budget never
    changes a result."""
    from pytorch_pose_proposal_network_b200 import _lib
    cfg = cfg_of("native")
    sizes = [(1080, 1920), (720, 1280), (1, 1), (33, 47), (480, 641)] * 3
    imgs = images_of(sizes, 3)
    batch = batch_of(imgs)
    aug = augmenter(cfg, scale=scale, dtype=torch.float16)
    params = aug.sample(batch, torch.Generator(device="cuda").manual_seed(9))
    default = _lib.tune_get("augment.stage_bytes")
    outs = []
    try:
        for stage in (16 * 1024, 48 * 1024, default):
            _lib.tune(augment_stage_bytes=stage)
            outs.append(aug.images(batch, params))
    finally:
        _lib.tune(augment_stage_bytes=default)
    assert torch.equal(outs[0].view(torch.int16), outs[1].view(torch.int16))
    assert torch.equal(outs[0].view(torch.int16), outs[2].view(torch.int16))
    check_images(aug, imgs, params, outs[2], f"scale {scale}")


def test_every_corner_outside_and_special_parameters():
    from pytorch_pose_proposal_network_b200.augment import compose, params_from
    cfg = cfg_of("cfg2")
    sizes = [(300, 200), (64, 64), (1, 1), (500, 333), (80, 90)]
    imgs = images_of(sizes, 4)
    batch = batch_of(imgs)
    aug = augmenter(cfg, fill=(100.0, 50.0, 3.0))
    d = lambda *v: torch.tensor(v, dtype=torch.float64, device="cuda")
    hw = batch.hw
    A = compose(hw[:, 1], hw[:, 0], cfg.insize, d(1.0, 0.5, 1.0, 1.0, 0.1), d(0.7, 3.0, -0.5, 1.2, 0.0),
                d(2.0, -1.6, 0.0, 0.4, 0.0), d(0.0, 1.7, -3.0, 0.5, 0.0), d(1, 0, 1, 0, 0) > 0)
    params = params_from(A, torch.tensor([1, 0, 1, 0, 0], dtype=torch.uint8, device="cuda"))
    params.M[4, 0, 2] = float("nan")                                # a non-finite parameter: the fill
    out = aug.images(batch, params)
    check_images(aug, imgs, params, out, "outside")
    fill = OA.warp_image(imgs[0], [[1, 0, 1e6], [0, 1, 0]], cfg.insize, fill=(100.0, 50.0, 3.0))
    got = out.cpu().numpy()
    for b in (0, 1, 2, 4):                                         # wholly outside the source
        assert np.array_equal(got[b].view(np.uint32), fill.view(np.uint32)), b


def people_of(sizes, K, seed, crowd=6):
    rng = np.random.default_rng(seed)
    samples = []
    for h, w in sizes:
        n = int(rng.integers(0, crowd))
        kp, bb, vis, size = encode_gt.random_people(rng, n, K, (w, h), spread=1.3)
        samples.append(dict(keypoints=kp, bbox=np.asarray(bb).reshape(-1, 4), is_visible=vis, size=size))
    return samples


def flat_on_device(samples, K):
    from pytorch_pose_proposal_network_b200.dataset import flatten_samples
    return tuple(torch.from_numpy(a).cuda() for a in flatten_samples(samples, K))


@pytest.mark.parametrize("preset", ["native", "cfg2"])
def test_people_bit_exact_with_flip(preset):
    cfg = cfg_of(preset)
    sizes = ragged_sizes(96, 7)
    imgs = images_of(sizes, 8)
    batch = batch_of(imgs)
    aug = augmenter(cfg)
    samples = people_of(sizes, cfg.K, 9)
    flat = flat_on_device(samples, cfg.K)
    params = aug.sample(batch, torch.Generator(device="cuda").manual_seed(10))
    got = aug.people(*flat, params)
    assert got[0] is flat[0]
    flip = params.flip.cpu().numpy()
    assert 20 < flip.sum() < 76
    want = OA.transform_people(*[t.cpu().numpy() for t in flat], params.A.cpu().numpy(), flip, aug.perm)
    for g, w, nm in zip(got[1:], want[1:], ("bbox", "keypoints", "visible", "size")):
        g = g.cpu().numpy()
        assert g.dtype == w.dtype and g.shape == w.shape, nm
        assert np.array_equal(g.view(np.uint8), np.ascontiguousarray(w).view(np.uint8)), nm


@pytest.mark.parametrize("preset", ["native", "cfg2"])
def test_augment_then_encode_matches_the_restated_encoder(preset):
    from pytorch_pose_proposal_network_b200.dataset import TargetEncoder
    cfg = cfg_of(preset)
    sizes = ragged_sizes(40, 12)
    imgs = images_of(sizes, 13)
    batch = batch_of(imgs)
    aug = augmenter(cfg)
    samples = people_of(sizes, cfg.K, 14, crowd=12)
    x, flat, params = aug(batch, samples, generator=torch.Generator(device="cuda").manual_seed(15))
    enc = TargetEncoder(cfg)
    targets = enc.encode_flat(*flat)
    host = [t.cpu().numpy() for t in flat_on_device(samples, cfg.K)]
    off, bb, kp, vis, size = OA.transform_people(*host, params.A.cpu().numpy(), params.flip.cpu().numpy(), aug.perm)
    got = {nm: getattr(targets, nm).cpu().numpy() for nm in NAMES}
    labelled = 0
    for b in range(batch.B):
        r = slice(off[b], off[b + 1])
        want = encode_gt.encode_targets(kp[r], bb[r], vis[r].astype(bool), size[r], cfg.K, enc.edges.tolist(), cfg.insize,
                                        cfg.outsize, cfg.local_grid_size)
        labelled += int(want[0].sum())
        for nm, w in zip(NAMES, want):
            assert np.array_equal(got[nm][b].view(np.uint32), w.view(np.uint32)), (b, nm)
    assert labelled > 50


def test_whole_chain_runs_forward_and_backward():
    from pytorch_pose_proposal_network_b200.dataset import TargetEncoder
    from pytorch_pose_proposal_network_b200.loss import PPNLoss
    cfg = cfg_of("cfg2")
    sizes = ragged_sizes(16, 20)
    batch = batch_of(images_of(sizes, 21))
    samples = people_of(sizes, cfg.K, 22, crowd=4)
    aug = augmenter(cfg, dtype=torch.bfloat16, channels_last=True)
    x, flat, _ = aug(batch, samples, generator=torch.Generator(device="cuda").manual_seed(23))
    t = TargetEncoder(cfg).encode_flat(*flat)
    conv = torch.nn.Conv2d(3, cfg.C, 1).cuda()
    pool = torch.nn.functional.avg_pool2d(x.float(), cfg.gridsize[0])
    head = torch.sigmoid(conv(pool)).contiguous()
    terms = PPNLoss(cfg)(head, t.delta, t.weight, t.weight_ij, t.tx_half, t.ty_half, t.tx, t.ty, t.tw, t.th, t.te)
    total = sum(terms)
    total.backward()
    assert torch.isfinite(total).item() and total.item() > 0
    assert conv.weight.grad is not None and torch.isfinite(conv.weight.grad).all().item()
    assert conv.weight.grad.abs().sum().item() > 0


def test_sample_is_deterministic_and_fit_is_the_letterbox():
    cfg = cfg_of("native")
    sizes = ragged_sizes(32, 30)
    batch = batch_of(images_of(sizes, 31))
    aug = augmenter(cfg)
    p1 = aug.sample(batch, torch.Generator(device="cuda").manual_seed(77))
    p2 = aug.sample(batch, torch.Generator(device="cuda").manual_seed(77))
    p3 = aug.sample(batch, torch.Generator(device="cuda").manual_seed(78))
    assert torch.equal(p1.A, p2.A) and torch.equal(p1.M, p2.M) and torch.equal(p1.flip, p2.flip)
    assert not torch.equal(p1.A, p3.A)
    fit = aug.fit(batch)
    assert not fit.flip.any().item()
    for b, (h, w) in enumerate(sizes):
        want = OA.compose(w, h, cfg.insize)
        assert np.allclose(fit.A[b].cpu().numpy(), want, rtol=0, atol=1e-12 * max(1.0, np.abs(want).max())), b
    out = aug.images(batch, fit)
    check_images(aug, images_of(sizes, 31), fit, out, "fit", every=3)


def test_calls_do_not_synchronise():
    cfg = cfg_of("cfg2")
    sizes = ragged_sizes(24, 40)
    imgs = images_of(sizes, 41)
    batch = batch_of(imgs)
    flat = flat_on_device(people_of(sizes, cfg.K, 42), cfg.K)
    aug = augmenter(cfg, dtype=torch.float16, channels_last=True)
    gen = torch.Generator(device="cuda").manual_seed(43)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        params = aug.sample(batch, gen)
        out = aug.images(batch, params)
        moved = aug.people(*flat, params)
        x, moved2, params2 = aug(batch, flat, generator=gen)
        fit = aug.fit(batch)
        out_fit = aug.images(batch, fit)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    check_images(aug, imgs, params, out, "no sync", every=5)
    check_images(aug, imgs, params2, x, "no sync call", every=5)


def test_graph_capture_and_replay_with_fresh_parameters():
    cfg = cfg_of("cfg2")
    sizes = ragged_sizes(20, 50)
    imgs = images_of(sizes, 51)
    batch = batch_of(imgs)
    flat = flat_on_device(people_of(sizes, cfg.K, 52), cfg.K)
    aug = augmenter(cfg, dtype=torch.bfloat16)
    gen = torch.Generator(device="cuda").manual_seed(53)
    static = aug.sample(batch, gen)
    out = torch.empty(batch.B, 3, cfg.inH, cfg.inW, dtype=torch.bfloat16, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):                                     # warm-up outside the capture
        aug.images(batch, static, out=out)
        aug.people(*flat, static)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        aug.images(batch, static, out=out)
        moved = aug.people(*flat, static)
    for seed in (54, 55):
        fresh = aug.sample(batch, torch.Generator(device="cuda").manual_seed(seed))
        for dst, src in zip(static, fresh):
            dst.copy_(src)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(out.view(torch.int16), aug.images(batch, fresh).view(torch.int16)), seed
        direct = aug.people(*flat, fresh)
        for a, b in zip(moved[1:], direct[1:]):
            assert torch.equal(a, b), seed
        check_images(aug, imgs, fresh, out, f"replay {seed}", every=4)
