"""PoseParser.parse_proposals (ppn_parse_proposals) on the GPU against the C twin of oracle/proposal_parse.py.

Bar: the packed result bit for bit on every image (counts exact; slots below min(count, R) identical), plus the
invariants the rule guarantees: no (part, cell) in two humans, every present part's parent present, every part cell
a survivor of that part's ppn_nms, humans in root NMS order.
"""
import numpy as np
import pytest
import torch

from oracle import c_proposal_parse, encode_gt, ppn_oracle as O, proposal_parse as PP
from tests.gpu_inputs import device_head

pytestmark = pytest.mark.gpu

F32, F16, BF16 = torch.float32, torch.float16, torch.bfloat16
SENT_I = 0x5A5A5A5A
SENT_F_BITS = 0x7FC5A5A5


def cfg_of(preset):
    from pytorch_pose_proposal_network_b200.config import PRESETS
    return PRESETS[preset]()


def parser_of(cfg, **kw):
    from pytorch_pose_proposal_network_b200.parser import PoseParser
    return PoseParser(cfg, **kw)


def ibits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32) if a.dtype == np.float32 else a


def check_against(got, ref, R, where):
    cnt = ref["count"]
    bad = np.flatnonzero(got["count"] != cnt)
    assert bad.size == 0, f"{where}: counts differ at images {bad[:8]} ({got['count'][bad[:8]]} vs {cnt[bad[:8]]})"
    used = np.arange(R)[None, :] < np.minimum(cnt, R)[:, None]
    for k in ("root_cell", "part_cell", "part_score", "part_box"):
        g, w = got[k][:, :R], ref[k][:, :R]
        m = np.broadcast_to(used.reshape(used.shape + (1,) * (w.ndim - 2)), w.shape)
        diff = (ibits(g) != ibits(w)) & m
        if diff.any():
            imgs = np.flatnonzero(diff.reshape(diff.shape[0], -1).any(1))[:8]
            raise AssertionError(f"{where}: {k} differs in {int(diff.sum())} elements, images {imgs}")


def survivors(parser, head):
    """Per (image, part): the cells ppn_nms keeps, in visiting order (decode_candidates + nms with n_parts = K)."""
    cfg = parser.cfg
    cell, score, box, count = parser.decode_candidates(head, n_parts=cfg.K)
    B, K, HW = cell.shape
    keep, kcount = parser.nms(box.reshape(B * K, HW, 4), score.reshape(B * K, HW), count.reshape(-1), cfg.nms_thresh)
    cell, keep, kcount = cell.cpu().numpy(), keep.cpu().numpy(), kcount.cpu().numpy()
    return [[cell[b, k][keep[b * K + k, :kcount[b * K + k]]] for k in range(K)] for b in range(B)]


def check_invariants(got, cfg, surv, where):
    g = O.Geometry.of(cfg)
    parent = {t: s for _, s, t in PP.limb_tree(g)}
    for b, n in enumerate(got["count"]):
        n = min(int(n), got["root_cell"].shape[1])
        pc = got["part_cell"][b, :n]
        assert np.array_equal(pc[:, 0], got["root_cell"][b, :n]), where
        for k in range(cfg.K):
            col = pc[:, k][pc[:, k] >= 0]
            assert np.unique(col).size == col.size, f"{where}: image {b} part {k}: a cell held by two humans"
            assert np.isin(col, surv[b][k]).all(), f"{where}: image {b} part {k}: a cell that is not an NMS survivor"
            if k in parent:
                assert ((pc[:, k] < 0) | (pc[:, parent[k]] >= 0)).all(), f"{where}: image {b} part {k} without parent"
        pos = {int(c): i for i, c in enumerate(surv[b][0])}
        order = [pos[int(c)] for c in pc[:, 0]]
        assert order == sorted(order), f"{where}: image {b}: humans not in root NMS order"


WORKLOADS = [("cfg2", "U", 512), ("cfg2", "R", 512), ("cfg2", "S", 512), ("cfg3", "D", 1024), ("cfg4", "U", 256),
             ("native", "U", 64), ("native", "S", 64), ("cfg1", "U", 1)]


@pytest.mark.parametrize("preset,dist,B", WORKLOADS, ids=[f"{p}-{d}-B{b}" for p, d, b in WORKLOADS])
def test_every_image_matches_c_restatement(preset, dist, B):
    cfg = cfg_of(preset)
    g = O.Geometry.of(cfg)
    head, host = device_head(g, dist, 7000 + B, B, distinct=False)
    parser = parser_of(cfg)
    got = parser.parse_proposals(head).numpy()
    ref = c_proposal_parse.proposal_parse_batch(host, g, n_threads=8)
    check_against(got, ref, parser.R, f"{preset}-{dist}-B{B}")
    check_invariants(got, cfg, survivors(parser, head), f"{preset}-{dist}")
    if preset == "cfg3":
        assert got["count"].mean() > 200                                # the dense crowd really is dense


@pytest.mark.parametrize("preset,B", [("cfg2", 512), ("native", 64)])
@pytest.mark.parametrize("dtype", [F16, BF16], ids=["f16", "bf16"])
@pytest.mark.parametrize("dist", ["U", "D"])
def test_16bit_heads_equal_the_widened_head(preset, B, dtype, dist):
    """A 16-bit head is widened exactly: the result is the C restatement's on head.float(); 16-bit values are full
    of equal scores and equal limb values, so both tie levels and the NMS tie rule are exercised."""
    cfg = cfg_of(preset)
    g = O.Geometry.of(cfg)
    head, host = device_head(g, dist, 11 + B, B if dist == "U" else B // 4, dtype=dtype, distinct=False)
    parser = parser_of(cfg)
    got = parser.parse_proposals(head).numpy()
    ref = c_proposal_parse.proposal_parse_batch(host, g, n_threads=8)
    check_against(got, ref, parser.R, f"{preset}-{dist}-{dtype}")
    check_invariants(got, cfg, survivors(parser, head.float()), f"{preset}-{dtype}")


@pytest.mark.parametrize("name", ["roundtrip_cfg2_s21", "roundtrip_native_s22"])
def test_golden_round_trip_gives_the_reference_humans(name):
    """When people do not compete, the two parsers agree: the fixture's humans are the live reference's own."""
    from tests.golden_util import load_case
    g, out, fx = load_case(name)
    cfg = cfg_of("cfg2" if g.K == 16 else "native")
    assert (cfg.K, cfg.H, cfg.sH) == (g.K, g.H, g.sH)
    parser = parser_of(cfg)
    got = parser.parse_proposals(torch.from_numpy(out[None]).cuda()).numpy()
    n = int(got["count"][0])
    assert n == fx["root_cell"].size
    assert np.array_equal(got["root_cell"][0, :n], fx["root_cell"])
    assert np.array_equal(got["part_cell"][0, :n], fx["part_cell"])
    present = fx["part_cell"] >= 0
    assert np.array_equal(ibits(got["part_score"][0, :n])[present], ibits(fx["ref_score"])[present])
    assert np.array_equal(ibits(got["part_box"][0, :n])[present], ibits(fx["ref_box"])[present])


def test_encoder_round_trip_scores_ap_100():
    from pytorch_pose_proposal_network_b200 import config as pcfg
    from pytorch_pose_proposal_network_b200.evaluation import APEvaluator
    cfg = cfg_of("native")
    g = O.Geometry.of(cfg)
    cell = cfg.inW // cfg.W
    heads, frames = [], []
    rng = np.random.default_rng(3)
    for b in range(6):
        people, rects = [], []
        for q in range(4):
            qy, qx = divmod(q, 2)
            if rng.random() < 0.2:
                continue
            ry, rx = 12 * qy + 8, 12 * qx + 6
            pts = {}
            for k in range(1, cfg.K):
                r, c = 12 * qy + 1 + 2 * ((k - 1) // 6), 12 * qx + 1 + 2 * ((k - 1) % 6)
                pts[k] = ((c + rng.uniform(0.2, 0.8)) * cell, (r + rng.uniform(0.2, 0.8)) * cell)
            people.append({"box": ((rx + 0.5) * cell, (ry + 0.5) * cell, 150.0, 150.0), "points": pts})
            hx, hy = pts[1]
            rects.append({"x1": [hx - 15.0], "y1": [hy - 20.0], "x2": [hx + 15.0], "y2": [hy + 20.0],
                          "annopoints": [{"point": [{"id": [k - 1], "x": [p[0]], "y": [p[1]]} for k, p in pts.items()]}]})
        heads.append(encode_gt.encode_people(people, g, pcfg.EDGES))
        frames.append({"image": [f"{b}.jpg"], "annorect": rects})
    head = torch.from_numpy(np.stack(heads)).cuda()
    packed = parser_of(cfg).parse_proposals(head)
    assert packed.count.cpu().tolist() == [len(f["annorect"]) for f in frames]
    ev = APEvaluator(cfg)
    ev.update(packed, frames)
    got = ev.compute()
    assert (got["recall"] == 100.0).all() and (got["precision"] == 100.0).all()
    np.testing.assert_allclose(got["ap"], 100.0, rtol=0, atol=1e-9)
    lists = packed.to_lists()                                           # present parts always form a rooted subtree
    assert [len(h) for h, _ in lists] == [len(f["annorect"]) for f in frames]


def test_clear_unused_and_small_R():
    cfg = cfg_of("cfg2")
    g = O.Geometry.of(cfg)
    head, host = device_head(g, "U", 5, 64, distinct=False)
    ref = c_proposal_parse.proposal_parse_batch(host, g, n_threads=8)
    R = int(np.median(ref["count"]))                                   # some images overflow R
    assert (ref["count"] > R).any() and (ref["count"] < R).any()
    parser = parser_of(cfg, max_humans=R)
    for clear in (False, True):
        out = parser.alloc_output(64)
        for t in (out.count, out.root_cell, out.part_cell):
            t.fill_(SENT_I)
        for t in (out.part_score, out.part_box):
            t.view(torch.int32).fill_(SENT_F_BITS)
        got = parser.parse_proposals(head, out=out, clear_unused=clear).numpy()
        check_against(got, ref, R, f"clear={clear}")
        used = np.arange(R)[None, :] < np.minimum(ref["count"], R)[:, None]
        tail_i = -1 if clear else SENT_I
        tail_f = 0 if clear else SENT_F_BITS
        assert (got["root_cell"][~used] == tail_i).all()
        assert (got["part_cell"][~used] == tail_i).all()
        assert (ibits(got["part_score"])[~used] == tail_f).all()
        assert (ibits(got["part_box"])[~used] == tail_f).all()


def test_cuda_graph_replay_equals_eager():
    cfg = cfg_of("native")
    g = O.Geometry.of(cfg)
    head, _ = device_head(g, "U", 21, 16, distinct=False)
    other, host2 = device_head(g, "S", 22, 16, distinct=False)
    parser = parser_of(cfg)
    eager = parser.parse_proposals(head).numpy()
    out = parser.alloc_output(16)
    parser.parse_proposals(head, out=out)                                # workspace and attributes outside capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.graph(graph, stream=side):
        parser.parse_proposals(head, out=out)
    torch.cuda.current_stream().wait_stream(side)
    out.count.zero_()
    graph.replay()
    check_against(out.numpy(), eager, parser.R, "replay")
    head.copy_(other)                                                    # refill the captured input, replay again
    graph.replay()
    check_against(out.numpy(), c_proposal_parse.proposal_parse_batch(host2, g, n_threads=8), parser.R, "replay on new input")


def test_no_host_synchronisation():
    cfg = cfg_of("cfg2")
    g = O.Geometry.of(cfg)
    head, host = device_head(g, "U", 31, 32, distinct=False)
    parser = parser_of(cfg)
    out = parser.alloc_output(32)
    parser.parse_proposals(head, out=out)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        parser.parse_proposals(head, out=out, clear_unused=True)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    check_against(out.numpy(), c_proposal_parse.proposal_parse_batch(host, g, n_threads=8), parser.R, "sync-debug")


def test_unsupported_shapes_raise():
    from pytorch_pose_proposal_network_b200 import _lib
    cfg = cfg_of("cfg2")
    bad = cfg.with_(directed_graphs=(((0,), (1,)), ((1,), (1,))))       # part 1 reached by two limbs
    head = torch.zeros(1, bad.C, bad.H, bad.W, device="cuda")
    with pytest.raises(_lib.PPNError, match="code -4"):
        parser_of(bad).parse_proposals(head)
