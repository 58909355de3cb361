"""oracle/augment.py (the specification of ppn_augment_*) against answers derived by hand, and the package's sampler
composition against a hand-built matrix product.  No GPU."""
import math

import numpy as np
import pytest
import torch

from oracle import augment as OA

f32 = np.float32


def norm(img, mean=OA.IMAGENET_MEAN, std=OA.IMAGENET_STD, in_scale=OA.IN_SCALE):
    """[h, w, 3] values (already the bilinear result) -> [3, h, w] normalised, fp32 one rounding per operation."""
    v = np.asarray(img, f32).transpose(2, 0, 1)
    return np.stack([(v[c] * f32(in_scale) - f32(mean[c])) / f32(std[c]) for c in range(3)]).astype(f32)


def image(h, w, seed=0):
    return np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)


def bits_equal(a, b):
    return np.array_equal(np.asarray(a, f32).view(np.uint32), np.asarray(b, f32).view(np.uint32))


def test_identity_reproduces_the_normalised_input():
    img = image(12, 16)
    out = OA.warp_image(img, [[1, 0, 0], [0, 1, 0]], (16, 12))
    assert bits_equal(out, norm(img))


@pytest.mark.parametrize("dx,dy", [(3, 0), (0, -2), (-5, 4), (16, 0)])
def test_integer_translation_shifts(dx, dy):
    h, w = 10, 16
    img = image(h, w, 1)
    out = OA.warp_image(img, [[1, 0, dx], [0, 1, dy]], (w, h))          # sx = u + dx
    want = np.zeros((h, w, 3), f32)                                      # fill 0
    for v in range(h):
        for u in range(w):
            if 0 <= u + dx < w and 0 <= v + dy < h:
                want[v, u] = img[v + dy, u + dx]
    assert bits_equal(out, norm(want))


def test_flip_mirrors():
    img = image(7, 9, 2)
    out = OA.warp_image(img, [[-1, 0, 9], [0, 1, 0]], (9, 7))           # sx = 9 - (u + .5) - .5 = 8 - u
    assert bits_equal(out, norm(img[:, ::-1]))


def test_quarter_turns_permute():
    h, w = 6, 11
    img = image(h, w, 3)
    # output w_out = h, h_out = w: sx = v, sy = h - 1 - u  (a quarter turn)
    out = OA.warp_image(img, [[0, 1, 0], [-1, 0, h]], (h, w))
    want = np.empty((w, h, 3), np.uint8)
    for v in range(w):
        for u in range(h):
            want[v, u] = img[h - 1 - u, v]
    assert bits_equal(out, norm(want))
    # and the other way: sx = w - 1 - v, sy = u
    out = OA.warp_image(img, [[0, -1, w], [1, 0, 0]], (h, w))
    for v in range(w):
        for u in range(h):
            want[v, u] = img[u, w - 1 - v]
    assert bits_equal(out, norm(want))
    # half turn
    out = OA.warp_image(img, [[-1, 0, w], [0, -1, h]], (w, h))
    assert bits_equal(out, norm(img[::-1, ::-1]))


def test_taps_on_pixel_boundaries():
    h, w = 5, 8
    img = image(h, w, 4)
    src = img.astype(f32)
    pad = np.concatenate([src, np.zeros((h, 1, 3), f32)], axis=1)     # the fill beyond the right edge
    out = OA.warp_image(img, [[1, 0, 0.5], [0, 1, 0]], (w, h))          # sx = u + .5: halfway between two centres
    assert bits_equal(out, norm(pad[:, :-1] * f32(0.5) + pad[:, 1:] * f32(0.5)))
    left = np.concatenate([np.zeros((h, 1, 3), f32), src], axis=1)
    out = OA.warp_image(img, [[1, 0, -0.5], [0, 1, 0]], (w, h))         # sx = u - .5: at u = 0 half the fill
    assert bits_equal(out, norm(left[:, :-1] * f32(0.5) + left[:, 1:] * f32(0.5)))


@pytest.mark.parametrize("M", [[[1, 0, 1000], [0, 1, 0]], [[1, 0, -2], [0, 1, 0]], [[0.5, 0, 0], [0, 0.5, -40]],
                               [[np.nan, 0, 0], [0, 1, 0]], [[1, 0, np.inf], [0, 1, 0]], [[1, 0, 3e9], [0, 1, 0]]])
def test_outside_gives_the_fill(M):
    img = image(4, 2, 5)
    fill = (10.0, 20.0, 30.0)
    out = OA.warp_image(img, M, (3, 4), fill=fill)
    if M[0][2] == -2:                                   # sx = u - 2: columns 0 and 1 are outside, column 2 maps to 0
        out = out[:, :, :1]
    want = norm(np.broadcast_to(np.asarray(fill, f32), (4, out.shape[2], 3)))
    assert bits_equal(out, want)


def test_one_by_one_source():
    p = np.array([[[200, 7, 99]]], np.uint8)
    assert bits_equal(OA.warp_image(p, [[1, 0, 0], [0, 1, 0]], (1, 1)), norm(p))
    # the letterbox fit into 4 x 4: A = 4x, M = x / 4; sx = (u + .5) / 4 - .5 -> taps weighted 5/8, 7/8, 7/8, 5/8
    A = OA.compose(1, 1, (4, 4))
    assert np.allclose(A, [[4, 0, 0], [0, 4, 0]], rtol=0, atol=1e-15)
    M = OA.inverse_f32(A)
    wgt = np.array([0.625, 0.875, 0.875, 0.625])
    want = (p[0, 0].astype(np.float64)[None, None, :] * wgt[None, :, None] * wgt[:, None, None]).astype(f32)
    assert bits_equal(OA.warp_image(p, M, (4, 4)), norm(want))


def test_output_dtypes_round_once():
    img = image(9, 13, 6)
    M = OA.inverse_f32(OA.compose(13, 9, (8, 8), 1.1, 0.3, 0.05, -0.02, True))
    o32 = OA.warp_image(img, M, (8, 8))
    assert np.array_equal(OA.warp_image(img, M, (8, 8), dtype="float16"), o32.astype(np.float16))
    bf = OA.warp_image(img, M, (8, 8), dtype="bfloat16")
    assert np.array_equal(bf, torch.from_numpy(o32).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16))


def test_flip_permutation_both_skeletons():
    from pytorch_pose_proposal_network_b200 import config
    from pytorch_pose_proposal_network_b200.augment import flip_permutation
    pairs = list(range(12))
    want18 = [p ^ 1 for p in pairs] + [12, 13, 14, 15, 16]
    want16 = [p ^ 1 for p in pairs] + [12, 13, 14]
    for names, want, edges in ((config.KEYPOINT_NAMES, want18, config.EDGES), (config.KEYPOINT_NAMES_16, want16, config.EDGES_16)):
        assert OA.flip_permutation(names).tolist() == want
        assert flip_permutation(names).tolist() == want
        for i, j in enumerate(want):                    # pairs really are left/right twins
            a, b = names[i + 1], names[j + 1]
            assert a == b or a.split("_", 1)[1] == b.split("_", 1)[1]
        part = lambda k: 0 if k == 0 else want[k - 1] + 1
        assert {tuple(e) for e in edges} == {(part(s), part(t)) for s, t in edges}   # the limbs map onto limbs
    with pytest.raises(ValueError):
        flip_permutation(["instance", "left_eye", "nose"])


def test_people_flip_and_rotation_by_hand():
    names = ["instance", "left_a", "right_a", "mid"]
    perm = OA.flip_permutation(names)
    assert perm.tolist() == [1, 0, 2]
    off = np.array([0, 2], np.int32)
    bbox = np.array([[10.0, 20.0, 4.0, 6.0], [5.0, 5.0, 0.0, 3.0]])
    kp = np.array([[[1, 2], [3, 4], [5, 6]], [[7, 8], [9, 10], [11, 12]]], f32)
    vis = np.array([[1, 0, 1], [0, 1, 1]], np.uint8)
    size = np.array([8.0, 2.0])
    # quarter turn about the origin then a shift: (x, y) -> (-y + 100, x); a mirror flag
    A = np.array([[[0.0, -1.0, 100.0], [1.0, 0.0, 0.0]]])
    _, bo, ko, vo, so = OA.transform_people(off, bbox, kp, vis, size, A, [1], perm)
    assert ko[0].tolist() == [[96, 3], [98, 1], [94, 5]]
    assert ko[1].tolist() == [[90, 9], [92, 7], [88, 11]]
    assert vo.tolist() == [[0, 1, 1], [1, 0, 1]]
    assert bo[0].tolist() == [80.0, 10.0, 6.0, 4.0]                 # w and h swap under the quarter turn
    assert bo[1].tolist() == [95.0, 5.0, 0.0, 0.0]                  # rule (c): an empty box stays empty
    assert so.tolist() == [8.0, 2.0]                                # |det| = 1
    _, bo, _, _, so = OA.transform_people(off, bbox, kp, vis, size, A * 2.0, [0], perm)
    assert bo[1].tolist() == [190.0, 10.0, 0.0, 0.0] and so.tolist() == [16.0, 4.0]


def test_rotated_box_is_the_bounds_of_its_corners():
    A = OA.compose(100, 100, (100, 100), theta=math.pi / 4)
    _, bo, _, _, _ = OA.transform_people([0, 1], [[50.0, 50.0, 20.0, 20.0]], np.zeros((1, 1, 2), f32), np.ones((1, 1), np.uint8),
                                         [1.0], A[None], [0], [0])
    assert np.allclose(bo[0], [50, 50, 20 * math.sqrt(2), 20 * math.sqrt(2)], rtol=0, atol=1e-12)


def test_sampler_composition_against_hand_built_matrices():
    from pytorch_pose_proposal_network_b200.augment import compose, invert
    rng = np.random.default_rng(7)
    for _ in range(50):
        w, h = int(rng.integers(1, 2000)), int(rng.integers(1, 2000))
        insize = (int(rng.integers(8, 800)), int(rng.integers(8, 800)))
        s, th, tx, ty, fl = rng.uniform(0.5, 1.5), rng.uniform(-3, 3), rng.uniform(-.3, .3), rng.uniform(-.3, .3), bool(rng.integers(2))
        t = lambda v: torch.tensor([v], dtype=torch.float64)
        got = compose(torch.tensor([w]), torch.tensor([h]), insize, t(s), t(th), t(tx), t(ty), torch.tensor([fl]))[0].numpy()
        want = OA.compose(w, h, insize, s, th, tx, ty, fl)
        assert np.allclose(got, want, rtol=0, atol=1e-12 * max(1.0, np.abs(want).max())), (got, want)
        full = np.vstack([got, [0, 0, 1]])
        inv = invert(torch.from_numpy(got)[None])[0].numpy()
        assert np.allclose(np.vstack([inv, [0, 0, 1]]) @ full, np.eye(3), rtol=0, atol=1e-9)


def test_sampler_ranges():
    from pytorch_pose_proposal_network_b200.augment import draw
    B = 4000
    hw = torch.stack([torch.randint(1, 1500, (B,)), torch.randint(1, 1500, (B,))], 1).to(torch.int32)
    g = torch.Generator().manual_seed(3)
    p = draw(hw, (384, 256), scale=(0.8, 1.2), rotation=20.0, shift=0.1, p_flip=0.3, generator=g)
    A, h, w = p.A.numpy(), hw[:, 0].double().numpy(), hw[:, 1].double().numpy()
    s0 = np.minimum(384 / w, 256 / h)
    k = np.sqrt(np.abs(A[:, 0, 0] * A[:, 1, 1] - A[:, 0, 1] * A[:, 1, 0])) / s0
    assert k.min() >= 0.8 - 1e-12 and k.max() <= 1.2 + 1e-12 and k.max() - k.min() > 0.35
    flip = p.flip.numpy().astype(bool)
    assert np.array_equal(np.linalg.det(A[:, :, :2]) < 0, flip)
    assert 0.25 < flip.mean() < 0.35
    theta = np.degrees(np.arctan2(A[:, 1, 0] * np.where(flip, -1, 1), A[:, 0, 0] * np.where(flip, -1, 1)))
    assert np.abs(theta).max() <= 20 + 1e-9 and np.abs(theta).max() > 19
    centre = np.einsum("bij,bj->bi", A[:, :, :2], np.stack([w / 2, h / 2], 1)) + A[:, :, 2]
    t = (centre - [192, 128]) / [384, 256]
    assert np.abs(t).max() <= 0.1 + 1e-9 and np.abs(t).max() > 0.099
    assert p.M.dtype == torch.float32 and p.flip.dtype == torch.uint8
    again = draw(hw, (384, 256), scale=(0.8, 1.2), rotation=20.0, shift=0.1, p_flip=0.3, generator=torch.Generator().manual_seed(3))
    assert torch.equal(again.A, p.A) and torch.equal(again.M, p.M) and torch.equal(again.flip, p.flip)
