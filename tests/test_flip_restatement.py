"""The flip test's merge (oracle/flip_merge.py, DESIGN.md §15) against hand-derived answers, without a GPU.

The mirror tables are checked against hand-written ones for both skeletons; the merge against single elements worked
out by hand on a tiny configuration; the fp32 rule on special values; and the whole channel and window mapping
against the encoder: encoding mirrored annotations and merging must give back the encoding of the originals.
"""
import numpy as np
import pytest

from oracle import encode_gt, flip_merge as FM, ppn_oracle as O
from pytorch_pose_proposal_network_b200 import config as pcfg
from pytorch_pose_proposal_network_b200.augment import flip_permutation
from pytorch_pose_proposal_network_b200.config import PPNConfig, PRESETS
from pytorch_pose_proposal_network_b200.flip import limb_mirror, part_mirror

f32 = np.float32

# KEYPOINT_NAMES: instance, (left, right) x (shoulder, elbow, wrist, hip, knee, ankle), thorax, pelvis, neck, top, stomach
P18 = [0, 2, 1, 4, 3, 6, 5, 8, 7, 10, 9, 12, 11, 13, 14, 15, 16, 17]
# EDGES: 0 instance-neck, 1 neck-thorax, 2-4 thorax-l_shoulder-l_elbow-l_wrist, 5-7 thorax-r_shoulder-r_elbow-r_wrist,
# 8 thorax-stomach, 9 stomach-pelvis, 10/11 pelvis-l/r_hip, 12/13 l/r_hip-knee, 14/15 l/r_knee-ankle, 16 instance-top
Q18 = [0, 1, 5, 6, 7, 2, 3, 4, 8, 9, 11, 10, 13, 12, 15, 14, 16]
# KEYPOINT_NAMES_16: the same without top and stomach
P16 = [0, 2, 1, 4, 3, 6, 5, 8, 7, 10, 9, 12, 11, 13, 14, 15]
# EDGES_16: 0 instance-neck, 1 neck-thorax, 2-4 left arm, 5-7 right arm, 8 thorax-pelvis, 9-11 pelvis-l_hip-l_knee-
# l_ankle, 12-14 pelvis-r_hip-r_knee-r_ankle
Q16 = [0, 1, 5, 6, 7, 2, 3, 4, 8, 12, 13, 14, 9, 10, 11]


@pytest.mark.parametrize("names,edges,p_want,q_want", [(pcfg.KEYPOINT_NAMES, pcfg.EDGES, P18, Q18),
                                                       (pcfg.KEYPOINT_NAMES_16, pcfg.EDGES_16, P16, Q16)],
                         ids=["18", "16"])
def test_mirror_tables_by_hand(names, edges, p_want, q_want):
    p = part_mirror(names)
    q = limb_mirror(p, edges)
    assert p.dtype == np.int32 and q.dtype == np.int32
    assert p.tolist() == p_want and q.tolist() == q_want
    assert np.array_equal(p[p], np.arange(len(p))) and np.array_equal(q[q], np.arange(len(q)))
    i = names.index
    assert p[i("left_shoulder")] == i("right_shoulder") and p[i("thorax")] == i("thorax")
    e = [tuple(x) for x in edges]
    assert q[e.index((i("thorax"), i("left_shoulder")))] == e.index((i("thorax"), i("right_shoulder")))


def test_skeletons_without_a_mirror_raise():
    names = ["instance", "left_a", "right_a"]
    p = part_mirror(names)
    assert p.tolist() == [0, 2, 1]
    assert limb_mirror(p, [[0, 1], [0, 2]]).tolist() == [1, 0]
    with pytest.raises(ValueError, match="missing"):
        limb_mirror(p, [[0, 1]])                                        # instance->right_a is not a limb
    with pytest.raises(ValueError, match="reversed"):
        limb_mirror(p, [[0, 1], [2, 0]])                                # only right_a->instance
    with pytest.raises(ValueError, match="mirror part"):
        part_mirror(["instance", "left_a"])


def test_flipmerge_checks_its_configuration():
    from pytorch_pose_proposal_network_b200.flip import FlipMerge
    with pytest.raises(ValueError, match="keypoint_names"):
        FlipMerge(PPNConfig(K=5, E=0, directed_graphs=()), device="cuda:0")
    with pytest.raises(ValueError, match="inW == W"):
        FlipMerge(PPNConfig.mpii16(insize=(390, 384)), device="cuda:0")
    with pytest.raises(ValueError, match="off_w"):
        FlipMerge(PPNConfig.mpii16(local_grid_size=(9, 7)), device="cuda:0")
    with pytest.raises(ValueError, match="reversed"):
        FlipMerge(PPNConfig(K=3, E=2, directed_graphs=()), keypoint_names=["instance", "left_a", "right_a"],
                  edges=[[0, 1], [2, 0]], device="cuda:0")
    for preset in PRESETS.values():
        fm = FlipMerge(preset(), device="cuda:0")                         # every preset has a flip test
        assert fm.part_mirror.dtype == np.int32 and fm.limb_mirror.dtype == np.int32


def tiny():
    """Parts instance, left_a, right_a; limbs instance->left_a, instance->right_a; a 2 x 3 grid of 8 x 8 cells, a
    3 x 3 window.  C = 6 * 3 + 9 * 2 = 36: resp 0-2, conf 3-5, x 6-8, y 9-11, w 12-14, h 15-17, limb 0 at 18 + 3a + b,
    limb 1 at 27 + 3a + b."""
    cfg = PPNConfig(K=3, E=2, insize=(24, 16), outsize=(3, 2), local_grid_size=(3, 3), directed_graphs=())
    return O.Geometry.of(cfg), np.array([0, 2, 1], np.int32), np.array([1, 0], np.int32)


def test_hand_derived_elements():
    g, p, q = tiny()
    assert g.C == 36 and g.gridW == 8
    A = np.zeros((36, 2, 3), f32)
    Bf = np.zeros((36, 2, 3), f32)
    A[1, 0, 0], Bf[2, 0, 2] = 0.25, 0.75              # resp of left_a at (0, 0) <- resp of right_a at (0, 2)
    A[7, 1, 1], Bf[8, 1, 1] = 0.25, 0.125             # x of left_a on the mirror axis (column 1 of 3): 1 - 0.125
    A[21, 1, 2], Bf[32, 1, 0] = 0.5, 1.0              # limb 0 (1, 0) at (1, 2) <- limb 1 (1, 2) at (1, 0)
    A[9, 0, 1], Bf[9, 0, 1] = 0.5, 0.25               # y of the instance on the mirror axis: itself
    A[30, 0, 0], Bf[23, 0, 2] = 0.0, 0.5              # limb 1 (1, 0) at (0, 0) <- limb 0 (1, 2) at (0, 2)
    out = FM.flip_merge(A, Bf, g, p, q)
    assert out[1, 0, 0] == f32(0.5)
    assert out[7, 1, 1] == f32((0.25 + 0.875) * 0.5)
    assert out[21, 1, 2] == f32(0.75)
    assert out[9, 0, 1] == f32(0.375)
    assert out[30, 0, 0] == f32(0.25)
    assert out[6, 0, 0] == f32(0.5) and out[8, 1, 2] == f32(0.5)      # x planes where neither view has the part
    src = FM.source_planes(3, 2, 3, 3, p, q)
    assert src[:18].tolist() == [0, 2, 1, 3, 5, 4, 6, 8, 7, 9, 11, 10, 12, 14, 13, 15, 17, 16]
    assert src[18:21].tolist() == [29, 28, 27] and src[27:30].tolist() == [20, 19, 18]


def test_geometry_rule():
    with pytest.raises(ValueError, match="inW == W"):
        FM.check_geometry(O.Geometry.of(PPNConfig(K=3, E=0, insize=(25, 16), outsize=(3, 2), directed_graphs=())))
    with pytest.raises(ValueError, match="off_w"):
        FM.check_geometry(O.Geometry.of(PPNConfig(K=3, E=0, insize=(24, 16), outsize=(3, 2), local_grid_size=(4, 4),
                                                  directed_graphs=())))
    for preset in PRESETS.values():
        FM.check_geometry(O.Geometry.of(preset()))


def bits(a):
    return np.ascontiguousarray(a, f32).view(np.uint32)


def test_special_values_through_the_fp32_rule():
    inf, nan, tiny_ = np.inf, np.nan, f32(2.0 ** -149)
    a = np.array([nan, 1.0, inf, inf, -0.0, -0.0, tiny_, 3 * tiny_, f32(2.0 ** -126), -inf, 1.0], f32)
    b = np.array([0.5, nan, 1.0, -inf, -0.0, -0.0, 0.0, 0.0, 0.0, inf, 2.0 ** -11], f32)
    is_x = np.array([0, 0, 0, 0, 0, 1, 0, 0, 0, 1, 0], bool)
    out = FM.merge_values(a, b, is_x)
    assert np.isnan(out[:2]).all() and out[2] == inf and np.isnan(out[3])   # inf + -inf
    assert bits(out[4]) == 0x80000000                    # -0 + -0 = -0, times 0.5
    assert out[5] == f32(0.5)                              # x group: 1 - (-0) = 1
    assert bits(out[6]) == 0                               # 2^-150 is a tie: to even, 0
    assert out[7] == f32(2 * tiny_)                        # 1.5 * 2^-149: to even, 2^-148
    assert out[8] == f32(2.0 ** -127)                      # a denormal result, exact
    assert out[9] == -inf                                  # x group: 1 - inf = -inf, then -inf + -inf
    assert out[10] == f32(0.5 + 2.0 ** -12)
    h = FM.merge_values(a[10:], b[10:], is_x[10:], "float16")
    assert h[0] == np.float16(0.5)                         # 0.5 + 2^-12 is a tie in fp16: to even
    bf = FM.merge_values(np.array([1.0], f32), np.array([2.0 ** -8], f32), [False], "bfloat16")
    assert bf[0] == 0x3F00                                 # 0.5 + 2^-9 (bf16 ulp 2^-8 at 0.5): a tie, to even, 0.5


def dyadic_people(rng, cfg, n):
    """People whose labelled points sit at (j + m / 64) cells, 1 <= m <= 63, inside the image: every coordinate and
    its mirror inW - x is exact in fp32, and the mirror lands in column W - 1 - j at offset 1 - m / 64.  (Points left
    of the image would not do: the reference's int() truncation puts x in (-gridW, 0) into column 0, but the mirror of
    such a point lies right of the grid, so the identity below does not hold there.)"""
    gW, gH = cfg.gridsize
    K = cfg.K

    def coord(cells, g, size):
        return ((rng.integers(0, cells, size) + rng.integers(1, 64, size) / 64.0) * g)

    keypoints = np.stack([coord(cfg.W, gW, (n, K - 1)), coord(cfg.H, gH, (n, K - 1))], axis=-1).astype(f32)
    bbox = np.stack([coord(cfg.W, gW, n), coord(cfg.H, gH, n), rng.integers(1, 12, n) * 8.0,
                     rng.integers(1, 12, n) * 8.0], axis=1)
    bbox[rng.random(n) < 0.2, 2] = 0.0
    visible = rng.random((n, K - 1)) < 0.7
    size = rng.integers(1, 40, n).astype(np.float64)
    return keypoints, bbox, visible, size


def head_form(t, cfg):
    delta, _, _, tx, ty, _, _, tw, th, te = t
    return np.concatenate([delta, delta, tx, ty, tw, th, te.reshape(-1, cfg.H, cfg.W)], axis=0)


@pytest.mark.parametrize("preset", ["cfg2", "cfg3", "cfg4", "native"])
def test_encoder_mirror_identity(preset):
    cfg = PRESETS[preset]()
    names, edges = pcfg.default_skeleton(cfg)
    g = O.Geometry.of(cfg)
    p = part_mirror(names)
    q = limb_mirror(p, edges)
    perm = flip_permutation(names)
    rng = np.random.default_rng(len(preset) * 100 + cfg.K)
    for _ in range(3):
        kp, bb, vis, size = dyadic_people(rng, cfg, int(rng.integers(1, 9)))
        enc = lambda k, b, v: head_form(encode_gt.encode_targets(k, b, v, size, cfg.K, edges, cfg.insize, cfg.outsize,
                                                                 cfg.local_grid_size), cfg)
        T = enc(kp, bb, vis)
        kpm = kp[:, perm].copy()
        kpm[..., 0] = (cfg.inW - kpm[..., 0].astype(np.float64)).astype(f32)
        bbm = bb.copy()
        bbm[:, 0] = cfg.inW - bbm[:, 0]
        Tm = enc(kpm, bbm, vis[:, perm])
        assert not np.array_equal(T, Tm)
        got = FM.flip_merge(T, Tm, g, p, q)
        want = T.copy()
        xs = slice(2 * cfg.K, 3 * cfg.K)
        want[xs][T[:cfg.K] == 0] = f32(0.5)                       # x where the part is unlabelled: (0 + (1 - 0)) / 2
        assert np.array_equal(bits(got), bits(want))
        assert (T[:cfg.K] != 0).any() and (T[6 * cfg.K:] != 0).any()
