"""The proposal-pair parse restatement (oracle/proposal_parse.py) against hand-derived answers, and its C twin
(oracle/proposal_parse.c) against it.  No GPU.

Hand-built heads: every delta is resp * 1 with resp exact in fp32; x = y = 0.5 and w = h = 0.01 give 3.84-pixel boxes
16 pixels apart, so NMS keeps every candidate unless a test widens a box on purpose.
"""
import multiprocessing
import os
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import pytest

from oracle import c_proposal_parse, ppn_oracle as O, proposal_parse as PP, synth

CHAIN = (((0, 1), (1, 2)),)                      # instance -> part 1 -> part 2, limbs 0 and 1


def geom(K=3, E=2, graphs=CHAIN, H=5, W=6, sH=3, sW=3, **kw):
    return O.Geometry(K=K, E=E, inW=16 * W, inH=16 * H, W=W, H=H, sW=sW, sH=sH, graphs=graphs, **kw)


def blank(g):
    out = np.zeros((g.C, g.H, g.W), np.float32)
    K = g.K
    out[K:2 * K] = 1.0                           # conf: delta = resp
    out[2 * K:4 * K] = 0.5                       # x, y
    out[4 * K:6 * K] = 0.01                      # w, h
    return out


def part(out, g, k, cell, d):
    out[k].flat[cell] = d


def limb(out, g, e, a, b, v):
    """The limb value of pair (source cell a, target cell b) for limb e."""
    (ih, iw), (jh, jw) = divmod(a, g.W), divmod(b, g.W)
    dy, dx = jh - ih + g.oh, jw - iw + g.ow
    assert 0 <= dy < g.sH and 0 <= dx < g.sW
    out[6 * g.K + (e * g.sH + dy) * g.sW + dx].flat[a] = v


def parse(out, g):
    """numpy restatement, checked against the C twin on the same image."""
    p = PP.parse_image(out, g)
    c = c_proposal_parse.proposal_parse_batch(out[None], g)
    n = p.root_cell.size
    assert c["count"][0] == n
    assert np.array_equal(c["part_cell"][0, :n], p.part_cell)
    assert np.array_equal(c["part_score"][0, :n].view(np.uint32), p.part_score.view(np.uint32))
    assert np.array_equal(c["part_box"][0, :n].view(np.uint32), p.part_box.view(np.uint32))
    return p


def test_competing_roots_take_distinct_cells():
    """Both roots' reference walks land on the same part-1 cell; here the better pair keeps it and the other human
    takes its next proposal, or nothing when it has none."""
    g = geom(min_kp=0)
    out = blank(g)
    r0, r1, c, c2 = 7, 9, 8, 14                  # roots at (1,1) and (1,3); c = (1,2) between them; c2 = (2,2)
    part(out, g, 0, r0, 0.9); part(out, g, 0, r1, 0.8)
    part(out, g, 1, c, 0.75); part(out, g, 1, c2, 0.5)
    limb(out, g, 0, r0, c, 0.9); limb(out, g, 0, r1, c, 0.95)
    limb(out, g, 0, r1, c2, 0.6)
    ref = O.parse_image(out, g)
    assert list(ref.part_cell[:, 1]) == [c, c]                           # the reference walk: both claim c
    p = parse(out, g)
    # (0.9 * 0.9) * 0.75 > (0.8 * 0.95) * 0.75: human 0 keeps c, human 1 falls back to c2
    assert list(p.root_cell) == [r0, r1] and list(p.part_cell[:, 1]) == [c, c2]
    limb(out, g, 0, r1, c2, 0.0)                                          # remove r1's second option
    p = parse(out, g)
    assert list(p.part_cell[:, 1]) == [c, -1]
    # a better pair wins against root order: human 1's pair now outscores human 0's
    limb(out, g, 0, r1, c, 1.0); limb(out, g, 0, r0, c, 0.5); limb(out, g, 0, r0, 1, 0.4)
    part(out, g, 1, 1, 0.5)
    p = parse(out, g)
    assert list(p.part_cell[:, 1]) == [1, c]


def test_both_tie_levels():
    g = geom(min_kp=0)
    out = blank(g)
    r0, r1, c = 7, 9, 8
    part(out, g, 0, r0, 0.75); part(out, g, 0, r1, 0.5)
    part(out, g, 1, c, 0.5)
    limb(out, g, 0, r0, c, 0.5); limb(out, g, 0, r1, c, 0.75)            # 0.75 * 0.5 == 0.5 * 0.75: equal scores
    p = parse(out, g)
    assert list(p.part_cell[:, 1]) == [c, -1]                            # equal scores: the smaller human index
    g = geom(min_kp=0)
    out = blank(g)
    part(out, g, 0, r0, 0.5)
    for b in (2, 14, 13):                                                 # three cells of one window, equal scores
        part(out, g, 1, b, 0.5)
        limb(out, g, 0, r0, b, 0.5)
    p = parse(out, g)
    assert list(p.part_cell[:, 1]) == [2]                                 # equal scores: the smaller cell


@pytest.mark.parametrize("v", [np.nan, 0.0, -0.0, -0.5])
def test_nonpositive_and_nan_limb_values_never_connect(v):
    g = geom(min_kp=0)
    out = blank(g)
    part(out, g, 0, 7, 0.9)
    part(out, g, 1, 8, 0.9)
    limb(out, g, 0, 7, 8, v)
    assert list(parse(out, g).part_cell[:, 1]) == [-1]


def test_nan_delta_is_not_a_proposal():
    g = geom(min_kp=0)
    out = blank(g)
    part(out, g, 0, 7, 0.9)
    part(out, g, 1, 8, np.nan)
    part(out, g, 1, 13, 0.2)
    limb(out, g, 0, 7, 8, 1.0); limb(out, g, 0, 7, 13, 0.1)
    p = parse(out, g)
    assert list(p.part_cell[:, 1]) == [13]
    assert [int(x) for x in p.proposals[1]] == [13]


def test_at_threshold_cell_is_not_a_proposal():
    g = geom(min_kp=0, det_thresh=0.25)
    out = blank(g)
    part(out, g, 0, 7, 0.9)
    part(out, g, 1, 8, 0.25)                                              # == thr: the reference would accept it
    limb(out, g, 0, 7, 8, 1.0)
    assert list(parse(out, g).part_cell[:, 1]) == [-1]


def test_target_outside_the_window():
    g = geom(min_kp=0)
    out = blank(g)
    part(out, g, 0, 7, 0.9)
    part(out, g, 1, 10, 0.9)                                              # (1,4): in the grid, 3 columns away
    out[6 * g.K:6 * g.K + g.S].reshape(g.S, -1)[:, 7] = 1.0               # every window value of the root
    assert list(parse(out, g).part_cell[:, 1]) == [-1]


def test_target_suppressed_by_nms():
    g = geom(min_kp=0)
    out = blank(g)
    part(out, g, 0, 7, 0.9)
    part(out, g, 1, 8, 0.8); part(out, g, 1, 14, 0.6)
    out[4 * g.K + 1].flat[[8, 14]] = 0.5                                  # 48-pixel boxes one cell apart: IoU >= 0.3
    out[5 * g.K + 1].flat[[8, 14]] = 0.5
    limb(out, g, 0, 7, 14, 1.0); limb(out, g, 0, 7, 8, 0.1)
    p = parse(out, g)
    assert [int(x) for x in p.proposals[1]] == [8]
    assert list(p.part_cell[:, 1]) == [8]


def test_unattached_parent_forms_no_orphan():
    g = geom(min_kp=0)
    out = blank(g)
    part(out, g, 0, 7, 0.9)
    part(out, g, 1, 22, 0.9)                                              # a part-1 proposal no root reaches
    part(out, g, 2, 23, 0.9)
    limb(out, g, 1, 22, 23, 1.0)
    p = parse(out, g)
    assert p.part_cell.tolist() == [[7, -1, -1]]


def test_min_kp_filters_after_matching():
    """Human 0 wins part 1 and is then dropped (min_kp = 2); the part does not go to human 1."""
    g = geom()
    out = blank(g)
    r0, r1, c = 7, 9, 8
    part(out, g, 0, r0, 0.9); part(out, g, 0, r1, 0.8)
    part(out, g, 1, c, 0.9)
    limb(out, g, 0, r0, c, 0.9); limb(out, g, 0, r1, c, 0.5)
    part(out, g, 2, 3, 0.9)                                               # human 1 only gets part 2 through part 1
    limb(out, g, 1, c, 3, 0.9)
    full = parse(out, geom(min_kp=-1))
    assert full.part_cell.tolist() == [[r0, c, 3], [r1, -1, -1]]
    assert parse(out, geom(min_kp=3)).root_cell.size == 0
    p = parse(out, geom(min_kp=2))
    assert p.part_cell.tolist() == [[r0, c, 3]]
    p = parse(out, geom(min_kp=1))
    assert p.part_cell.tolist() == [[r0, c, 3]]
    part(out, g, 2, 3, 0.1)                                               # below the threshold: human 0 keeps 1 part
    assert parse(out, geom(min_kp=2)).root_cell.size == 0                # dropped, and human 1 still gets nothing
    assert parse(out, geom(min_kp=0)).part_cell.tolist() == [[r0, c, -1], [r1, -1, -1]]


def test_swap_window_offsets():
    from pytorch_pose_proposal_network_b200.config import PPNConfig
    cfg = PPNConfig(K=3, E=2, insize=(96, 80), outsize=(6, 5), local_grid_size=(5, 3), directed_graphs=CHAIN,
                    min_num_keypoints=0)
    for swap, want in ((False, [1]), (True, [-1])):
        g = O.Geometry.of(cfg.with_(swap_window_offsets=swap))
        assert (g.oh, g.ow) == ((2, 1) if not swap else (1, 2))
        out = blank(g)
        part(out, g, 0, 19, 0.9)                                          # (3,1)
        part(out, g, 1, 7, 0.9)                                           # (1,1): two rows up
        dy, dx = 1 - 3 + g.oh, 0 + g.ow
        if 0 <= dy < g.sH:
            out[6 * g.K + (0 * g.sH + dy) * g.sW + dx].flat[19] = 1.0
        else:                                                             # out of the window: every value of the root
            out[6 * g.K:6 * g.K + g.S].reshape(g.S, -1)[:, 19] = 1.0
        assert [c >= 0 for c in parse(out, g).part_cell[:, 1]] == [w >= 0 for w in want]


def test_sixteen_part_tree_order():
    from pytorch_pose_proposal_network_b200.config import PPNConfig
    cfg = PPNConfig.mpii16()
    tree = PP.limb_tree(O.Geometry.of(cfg))
    assert len(tree) == 15 and sorted(t for _, _, t in tree) == list(range(1, 16))
    assert [t for _, _, t in tree] == cfg.key_order()[1:]
    from pytorch_pose_proposal_network_b200.config import EDGES_16
    edges = {tuple(e) for e in EDGES_16}
    for e, s, t in tree:
        assert (s, t) in edges
    g = O.Geometry.of(cfg)
    for dist in "US":
        head = synth.make_head(g, dist, 5, 3)
        for img in head:
            p = parse(img, g)
            for e, s, t in tree:
                assert ((p.part_cell[:, t] < 0) | (p.part_cell[:, s] >= 0)).all()


@pytest.mark.parametrize("graphs", [(((0, 1), (1, 0)),), (((0,), (1,)), ((1,), (1,))), (((0, 1), (1, 2)), ((0,), (2,)))],
                         ids=["back-to-root", "two-limbs", "two-parents"])
def test_non_tree_chains_rejected(graphs):
    g = geom(graphs=graphs)
    with pytest.raises(ValueError):
        PP.limb_tree(g)
    with pytest.raises(ValueError):
        c_proposal_parse.proposal_parse_batch(blank(g)[None], g)


def _numpy_batch(args):
    head, g = args
    return PP.parse_batch(head, g)


PRESET_NAMES = ["cfg1", "cfg2", "cfg3", "cfg4", "native"]


@pytest.mark.parametrize("preset", PRESET_NAMES)
def test_numpy_equals_c_on_seeded_images(preset):
    """40 seeded images per distribution U, R, D, S, every array bit for bit."""
    from pytorch_pose_proposal_network_b200.config import PRESETS
    g = O.Geometry.of(PRESETS[preset]())
    heads = {d: synth.make_head(g, d, 100 + i, 40) for i, d in enumerate("URDS")}
    jobs = [(d, q) for d in "URDS" for q in range(0, 40, 5)]
    with ProcessPoolExecutor(min(8, os.cpu_count() or 1), mp_context=multiprocessing.get_context("spawn")) as ex:
        parts = dict(zip(jobs, ex.map(_numpy_batch, [(heads[d][q:q + 5], g) for d, q in jobs])))
    for d in "URDS":
        c = c_proposal_parse.proposal_parse_batch(heads[d], g, n_threads=8)
        assert c["count"].sum() > 0
        for k, v in c.items():
            n = np.concatenate([parts[(d, q)][k] for q in range(0, 40, 5)])
            bits = (lambda a: a.view(np.uint32)) if v.dtype == np.float32 else (lambda a: a)
            assert np.array_equal(bits(v), bits(n)), (preset, d, k)


@pytest.mark.parametrize("name", ["roundtrip_cfg2_s21", "roundtrip_native_s22"])
def test_round_trip_fixtures_give_the_reference_humans(name):
    from tests.golden_util import load_case
    g, out, fx = load_case(name)
    p = parse(out, g)
    assert np.array_equal(p.root_cell, fx["root_cell"])
    assert np.array_equal(p.part_cell, fx["part_cell"])
    present = fx["part_cell"] >= 0
    assert np.array_equal(p.part_score.view(np.uint32)[present], fx["ref_score"].view(np.uint32)[present])
    assert np.array_equal(p.part_box.view(np.uint32)[present], fx["ref_box"].view(np.uint32)[present])
