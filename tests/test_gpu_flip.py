"""FlipMerge (ppn_flip_merge) on the GPU against the numpy restatement oracle/flip_merge.py, bit for bit.

Also the whole flip-test chain: annotations mirrored by Augmenter.people and encoded by TargetEncoder must merge back
into the unmirrored encoding, so that both parsers read the same humans and APEvaluator scores 100; a merged random
head must parse to the C oracle's humans on the restated merge; and the call must be graph-capturable,
synchronisation-free and deterministic.
"""
import numpy as np
import pytest
import torch

from oracle import c_oracle, flip_merge as FM, ppn_oracle as O
from tests.gpu_inputs import device_head

pytestmark = pytest.mark.gpu

F32, F16, BF16 = torch.float32, torch.float16, torch.bfloat16
NAMES = {F32: "float32", F16: "float16", BF16: "bfloat16"}


def cfg_of(preset, **kw):
    from pytorch_pose_proposal_network_b200.config import PRESETS
    return PRESETS[preset](**kw)


def merger(cfg, **kw):
    from pytorch_pose_proposal_network_b200.flip import FlipMerge
    return FlipMerge(cfg, **kw)


def gpu_bits(t):
    t = t.cpu()
    return (t.view(torch.int32) if t.dtype == F32 else t.view(torch.int16)).numpy().view(
        np.uint32 if t.dtype == F32 else np.uint16)


def ref_bits(r):
    r = np.ascontiguousarray(r)
    return r.view(np.uint32) if r.dtype == np.float32 else r.view(np.uint16)


def assert_merge_equals_restatement(got, hostA, hostB, g, fm, dtype, where, chunk=64):
    """Bit for bit, in chunks of images (the largest heads are GBs on the host).  NaN results compare as NaN: the
    device's canonical NaN and numpy's propagated payload differ in their bits, never in being NaN."""
    got = got.cpu()
    for b0 in range(0, hostA.shape[0], chunk):
        ref = FM.flip_merge(hostA[b0:b0 + chunk], hostB[b0:b0 + chunk], g, fm.part_mirror, fm.limb_mirror, NAMES[dtype])
        gb = gpu_bits(got[b0:b0 + chunk])
        rb = ref_bits(ref)
        gnan = got[b0:b0 + chunk].float().isnan().numpy()
        rnan = np.isnan(ref.astype(np.float32)) if dtype != BF16 else (
            np.isnan((rb.astype(np.uint32) << 16).view(np.float32)))
        assert np.array_equal(gnan, rnan), f"{where}: NaN positions differ"
        diff = (gb != rb) & ~rnan
        if diff.any():
            idx = np.argwhere(diff)[:5]
            raise AssertionError(f"{where}: {int(diff.sum())} elements differ, first at {idx.tolist()}")


WORKLOADS = [("cfg2", 512, F32), ("cfg3", 1024, F32), ("cfg4", 256, F32), ("native", 64, F32), ("cfg1", 1, F32),
             ("cfg2", 512, F16), ("cfg2", 512, BF16), ("native", 64, F16), ("native", 64, BF16)]


@pytest.mark.parametrize("preset,B,dtype", WORKLOADS, ids=[f"{p}-B{b}-{NAMES[d]}" for p, b, d in WORKLOADS])
def test_presets_bit_exact(preset, B, dtype):
    cfg = cfg_of(preset)
    g = O.Geometry.of(cfg)
    A, hostA = device_head(g, "U", 100 + B, B, dtype=dtype, distinct=False)
    Bf, hostB = device_head(g, "R", 200 + B, B, dtype=dtype, distinct=False)
    fm = merger(cfg)
    got = fm(A, Bf)
    assert got.dtype == dtype and got.shape == A.shape
    assert_merge_equals_restatement(got, hostA, hostB, g, fm, dtype, f"{preset}-B{B}-{dtype}")


def odd_configs():
    from pytorch_pose_proposal_network_b200.config import PPNConfig
    return {
        "grid13-win7": (PPNConfig(insize=(13 * 32, 13 * 32), outsize=(13, 13), local_grid_size=(7, 7)), {}),
        "grid13x8": (PPNConfig.mpii16(insize=(13 * 32, 8 * 32), outsize=(13, 8), local_grid_size=(5, 5)), {}),
        "grid1": (PPNConfig.mpii16(insize=(32, 32), outsize=(1, 1), local_grid_size=(1, 1)), {}),
        "E0": (PPNConfig(E=0, directed_graphs=()), dict(edges=[])),
        "K1": (PPNConfig(K=1, E=1, insize=(96, 96), outsize=(3, 3), local_grid_size=(3, 3), directed_graphs=()),
               dict(keypoint_names=["instance"], edges=[[0, 0]])),
    }


@pytest.mark.parametrize("name", ["grid13-win7", "grid13x8", "grid1", "E0", "K1"])
@pytest.mark.parametrize("dtype", [F32, F16, BF16], ids=["float32", "float16", "bfloat16"])
def test_geometries_the_presets_do_not_reach(name, dtype):
    """13 x 13 and 1 x 1 take the scalar path; 13 x 8 the vector path with units that straddle rows of odd W."""
    cfg, kw = odd_configs()[name]
    g = O.Geometry.of(cfg)
    A, hostA = device_head(g, "U", 7, 9, dtype=dtype, distinct=False)
    Bf, hostB = device_head(g, "U", 8, 9, dtype=dtype, distinct=False)
    fm = merger(cfg, **kw)
    assert_merge_equals_restatement(fm(A, Bf), hostA, hostB, g, fm, dtype, name)


@pytest.mark.parametrize("dtype", [F32, F16], ids=["float32", "float16"])
def test_element_aligned_heads_take_the_scalar_path(dtype):
    """Heads that are aligned to their element but not to 16 bytes (a view one element into its storage)."""
    cfg = cfg_of("cfg2")
    g = O.Geometry.of(cfg)
    A, hostA = device_head(g, "U", 3, 16, dtype=dtype, distinct=False)
    Bf, hostB = device_head(g, "U", 4, 16, dtype=dtype, distinct=False)
    store = torch.empty(2 * A.numel() + 2, dtype=dtype, device="cuda")
    a1 = store[1:1 + A.numel()].view(A.shape)
    b1 = store[1 + A.numel():1 + 2 * A.numel()].view(A.shape)
    a1.copy_(A)
    b1.copy_(Bf)
    fm = merger(cfg)
    assert_merge_equals_restatement(fm(a1, b1), hostA, hostB, g, fm, dtype, "element-aligned")


def test_special_values():
    cfg = cfg_of("cfg2")
    g = O.Geometry.of(cfg)
    A, hostA = device_head(g, "U", 5, 8, distinct=False)
    Bf, hostB = device_head(g, "U", 6, 8, distinct=False)
    rng = np.random.default_rng(0)
    specials = np.array([np.nan, np.inf, -np.inf, -0.0, 0.0, 2.0 ** -149, 3 * 2.0 ** -149, 2.0 ** -127, -2.0 ** -130,
                         3.4e38, -3.4e38, 1.0], np.float32)
    for host in (hostA, hostB):
        mask = rng.random(host.shape) < 0.3
        host[mask] = rng.choice(specials, int(mask.sum()))
    A.copy_(torch.from_numpy(hostA))
    Bf.copy_(torch.from_numpy(hostB))
    fm = merger(cfg)
    assert_merge_equals_restatement(fm(A, Bf), hostA, hostB, g, fm, F32, "specials")


@pytest.mark.parametrize("dtype", [F32, BF16], ids=["float32", "bfloat16"])
def test_in_place_and_halves_of_one_batch(dtype):
    cfg = cfg_of("native")
    g = O.Geometry.of(cfg)
    both, host = device_head(g, "U", 9, 2 * 24, dtype=dtype, distinct=False)
    fm = merger(cfg)
    apart = fm(both[:24], both[24:])
    assert_merge_equals_restatement(apart, host[:24], host[24:], g, fm, dtype, "halves")
    ret = fm(both[:24], both[24:], out=both[:24])
    assert ret.data_ptr() == both.data_ptr()
    assert torch.equal(both[:24].view(torch.int16 if dtype != F32 else torch.int32),
                       apart.view(torch.int16 if dtype != F32 else torch.int32))
    assert torch.equal(both[24:].float().cpu(), torch.from_numpy(host[24:]))          # the flipped half is untouched


def test_rejections():
    from pytorch_pose_proposal_network_b200 import _lib
    cfg = cfg_of("cfg2")
    fm = merger(cfg)
    h = torch.zeros(4, cfg.C, cfg.H, cfg.W, device="cuda")
    with pytest.raises(ValueError):
        fm(h, h.half())
    with pytest.raises(ValueError):
        fm(h, h[:2])
    with pytest.raises(ValueError):
        fm(h.double(), h.double())
    with pytest.raises(ValueError):
        fm(h, h, out=torch.zeros(4, cfg.C, cfg.H, cfg.W + 1, device="cuda")[..., :cfg.W])
    with pytest.raises(_lib.PPNError, match="code -1"):
        fm(h, h, out=h)                                                    # out overlaps the flipped head


# ---- the whole chain: Augmenter.people mirrors, TargetEncoder encodes, FlipMerge merges --------------------------
def flat_of(people, K):
    """people: per image a list of (box (cx, cy, w, h), {part: (x, y)}, size) -> the five flat device tensors."""
    offs, bbs, kps, vis, sizes = [0], [], [], [], []
    for img in people:
        for box, pts, size in img:
            kp = np.zeros((K - 1, 2), np.float32)
            v = np.zeros(K - 1, np.uint8)
            for k, xy in pts.items():
                kp[k - 1], v[k - 1] = xy, 1
            bbs.append(box), kps.append(kp), vis.append(v), sizes.append(size)
        offs.append(len(bbs))
    arrays = (np.asarray(offs, np.int32), np.asarray(bbs, np.float64).reshape(-1, 4),
              np.asarray(kps, np.float32).reshape(-1, K - 1, 2), np.asarray(vis, np.uint8).reshape(-1, K - 1),
              np.asarray(sizes, np.float64))
    return tuple(torch.from_numpy(a).cuda() for a in arrays)


def mirror_and_encode(cfg, flat):
    """(head form of the encoding, head form of the encoding of the mirrored annotations)."""
    from pytorch_pose_proposal_network_b200.augment import Augmenter, params_from
    from pytorch_pose_proposal_network_b200.dataset import TargetEncoder
    B = int(flat[0].numel()) - 1
    A = torch.tensor([[-1.0, 0.0, float(cfg.inW)], [0.0, 1.0, 0.0]], dtype=torch.float64, device="cuda")
    params = params_from(A.expand(B, 2, 3).contiguous(), torch.ones(B, dtype=torch.uint8, device="cuda"))
    mirrored = Augmenter(cfg).people(*flat, params)
    enc = TargetEncoder(cfg)

    def head(t):
        return torch.cat([t.delta, t.delta, t.tx, t.ty, t.tw, t.th, t.te.reshape(B, -1, cfg.H, cfg.W)], 1).contiguous()
    return head(enc.encode_flat(*flat)), head(enc.encode_flat(*mirrored))


def quadrant_people(cfg, rng, B):
    """Up to four people per image, one per quadrant of the grid, every labelled point at (cell + m / 64) pixels of
    a cell, 1 <= m <= 63 (exact in fp32 and under the mirror), and their PCKh ground truth frames."""
    cell = cfg.inW // cfg.W
    half = cfg.W // 2
    people, frames = [], []
    for b in range(B):
        img, rects = [], []
        for qd in range(4):
            qy, qx = divmod(qd, 2)
            if rng.random() < 0.2:
                continue
            pts = {}
            for k in range(1, cfg.K):
                r, c = half * qy + 1 + 2 * ((k - 1) // 6), half * qx + 1 + 2 * ((k - 1) % 6)
                pts[k] = ((c + rng.integers(13, 51) / 64) * cell, (r + rng.integers(13, 51) / 64) * cell)
            box = ((half * qx + 6.5) * cell, (half * qy + 8.5) * cell, 150.0, 150.0)
            img.append((box, pts, 18.75))
            hx, hy = pts[1]
            rects.append({"x1": [hx - 15.0], "y1": [hy - 20.0], "x2": [hx + 15.0], "y2": [hy + 20.0],
                          "annopoints": [{"point": [{"id": [k - 1], "x": [p[0]], "y": [p[1]]} for k, p in pts.items()]}]})
        people.append(img)
        frames.append({"image": [f"{b}.jpg"], "annorect": rects})
    return people, frames


def random_people(cfg, rng, B):
    from tests.test_flip_restatement import dyadic_people
    people = []
    for _ in range(B):
        kp, bb, vis, size = dyadic_people(rng, cfg, int(rng.integers(0, 12)))
        people.append([(tuple(bb[i]), {k + 1: tuple(kp[i, k]) for k in range(cfg.K - 1) if vis[i, k]}, float(size[i]))
                       for i in range(bb.shape[0])])
    return people


def packed_equal(a, b):
    a, b = a.numpy(), b.numpy()
    assert np.array_equal(a["count"], b["count"])
    for k in ("root_cell", "part_cell", "part_score", "part_box"):
        for i, n in enumerate(a["count"]):
            x, y = a[k][i, :n], b[k][i, :n]
            assert np.array_equal(x.view(np.uint32) if x.dtype == np.float32 else x,
                                  y.view(np.uint32) if y.dtype == np.float32 else y), (k, i)


@pytest.mark.parametrize("preset", ["cfg2", "cfg3", "cfg4", "native"])
def test_encoder_chain_merges_back_and_parses_alike(preset):
    from pytorch_pose_proposal_network_b200.parser import PoseParser
    cfg = cfg_of(preset)
    rng = np.random.default_rng(len(preset))
    B = 64
    T, Tm = mirror_and_encode(cfg, flat_of(random_people(cfg, rng, B), cfg.K))
    assert not torch.equal(T, Tm)
    merged = merger(cfg)(T, Tm)
    want = T.clone()
    K = cfg.K
    x = want[:, 2 * K:3 * K]
    x[T[:, :K] == 0] = 0.5                                                 # x where the part is unlabelled
    assert torch.equal(merged.view(torch.int32), want.view(torch.int32))
    parser = PoseParser(cfg)
    packed_equal(parser.parse(merged), parser.parse(T))
    packed_equal(parser.parse_proposals(merged), parser.parse_proposals(T))


def test_encoder_chain_scores_ap_100():
    from pytorch_pose_proposal_network_b200.evaluation import APEvaluator
    from pytorch_pose_proposal_network_b200.parser import PoseParser
    cfg = cfg_of("native")
    people, frames = quadrant_people(cfg, np.random.default_rng(4), 8)
    T, Tm = mirror_and_encode(cfg, flat_of(people, cfg.K))
    merged = torch.empty_like(T)
    merger(cfg)(T, Tm, out=merged)
    parser = PoseParser(cfg)
    for packed in (parser.parse(merged), parser.parse_proposals(merged)):
        assert packed.count.cpu().tolist() == [len(f["annorect"]) for f in frames]
        ev = APEvaluator(cfg)
        ev.update(packed, frames)
        got = ev.compute()
        np.testing.assert_allclose(got["ap"], 100.0, rtol=0, atol=1e-9)


def test_parse_of_a_merged_random_head_equals_the_c_oracle():
    from pytorch_pose_proposal_network_b200.parser import PoseParser
    cfg = cfg_of("cfg2")
    g = O.Geometry.of(cfg)
    B = 512
    A, hostA = device_head(g, "U", 41, B, distinct=False)
    Bf, hostB = device_head(g, "S", 42, B, distinct=False)
    fm = merger(cfg)
    packed = PoseParser(cfg).parse(fm(A, Bf)).numpy()
    ref = c_oracle.parse_batch(FM.flip_merge(hostA, hostB, g, fm.part_mirror, fm.limb_mirror), g, n_threads=8)
    assert np.array_equal(packed["count"], ref["counts"][:, 2])
    assert packed["count"].sum() > B
    for b in range(B):
        n = int(ref["counts"][b, 2])
        assert np.array_equal(packed["root_cell"][b, :n], ref["root_cell"][b, :n]), b
        assert np.array_equal(packed["part_cell"][b, :n], ref["part_cell"][b, :n]), b
        assert np.array_equal(packed["part_score"][b, :n].view(np.uint32), ref["part_score"][b, :n].view(np.uint32)), b
        assert np.array_equal(packed["part_box"][b, :n].view(np.uint32), ref["part_box"][b, :n].view(np.uint32)), b


# ---- stream behaviour ------------------------------------------------------------------------------------------
def test_graph_replay_on_refilled_inputs():
    from pytorch_pose_proposal_network_b200.parser import PoseParser
    cfg = cfg_of("cfg2")
    g = O.Geometry.of(cfg)
    B = 32
    A, _ = device_head(g, "U", 51, B, distinct=False)
    Bf, _ = device_head(g, "U", 52, B, distinct=False)
    A2, _ = device_head(g, "S", 53, B, distinct=False)
    Bf2, _ = device_head(g, "R", 54, B, distinct=False)
    fm, parser = merger(cfg), PoseParser(cfg)
    merged = torch.empty_like(A)
    out = parser.alloc_output(B)
    fm(A, Bf, out=merged)                                                 # warm-up outside capture
    parser.parse(merged, out=out)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.graph(graph, stream=side):
        fm(A, Bf, out=merged)
        parser.parse(merged, out=out)
    torch.cuda.current_stream().wait_stream(side)
    for a, b in ((A2, Bf2), (A.clone(), Bf.clone())):
        want_head = fm(a, b)
        want = parser.parse(want_head).numpy()
        A.copy_(a), Bf.copy_(b)
        out.count.zero_()
        graph.replay()
        assert torch.equal(merged.view(torch.int32), want_head.view(torch.int32))
        got = out.numpy()
        assert np.array_equal(got["count"], want["count"])
        for b_ in range(B):
            n = int(want["count"][b_])
            assert np.array_equal(got["part_cell"][b_, :n], want["part_cell"][b_, :n])


def test_no_host_synchronisation_and_deterministic():
    cfg = cfg_of("native")
    g = O.Geometry.of(cfg)
    A, _ = device_head(g, "U", 61, 16, distinct=False)
    Bf, _ = device_head(g, "U", 62, 16, distinct=False)
    fm = merger(cfg)
    first = fm(A, Bf)
    out = torch.empty_like(A)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        fm(A, Bf, out=out)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert torch.equal(first.view(torch.int32), out.view(torch.int32))
