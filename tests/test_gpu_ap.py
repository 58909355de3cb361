"""APEvaluator (ppn_ap_match + ppn_ap_finalize) against the float64 restatement of poseval's assignGTmulti and
computeMetrics (oracle/pose_ap.py), on parser outputs.

Per-(image, slot, joint) scores and labels and the GT joint counts must equal the restatement bit for bit; AP,
precision and recall within 1e-9 (in percent; the kernel sums VOCap's terms in its own fixed order).
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import encode_gt, pose_ap as P, ppn_oracle as O
from tests.gpu_inputs import device_head

pytestmark = pytest.mark.gpu


def cfg_of(name):
    from pytorch_pose_proposal_network_b200.config import PRESETS
    return PRESETS[name]()


def parse(cfg, head, max_humans=None):
    from pytorch_pose_proposal_network_b200.parser import PoseParser
    parser = PoseParser(cfg, max_humans=max_humans)
    out = parser.alloc_output(head.shape[0])
    packed = parser.parse(head, out=out)
    return parser, packed


def gt_frames_near(rng, packed, centres, J, max_people=8, p_empty=0.1, crowd_image=None):
    """Synthetic GT frames: 1..max_people people per image, most placed near a predicted human (each joint jittered
    by up to about one head size, so that some match and some do not), some with missing joints, some without any
    annotation, some joints exactly at the threshold (offset 0.5 * headSize = 15 px along x from the prediction),
    and images without GT.  crowd_image: that image gets 64 people."""
    a = packed.numpy()
    c = centres.cpu().numpy()
    frames = []
    for b in range(a["count"].shape[0]):
        n_pred = min(int(a["count"][b]), packed.R)
        n = 0 if rng.random() < p_empty else int(rng.integers(1, max_people + 1))
        if b == crowd_image:
            n = 64
        rects = []
        for _ in range(n):
            x0, y0 = (float(v) for v in rng.integers(0, 300, 2))                     # x2 - x1 = 30 exactly
            rect = {"x1": [x0], "y1": [y0], "x2": [x0 + 30.0], "y2": [y0 + 40.0]}     # headSize 30
            if rng.random() < 0.08:
                rects.append(rect)                                                  # no annotation at all
                continue
            i = int(rng.integers(n_pred)) if n_pred and rng.random() < 0.85 else -1
            pts = []
            for j in range(J):
                if rng.random() < 0.2:
                    continue
                if i >= 0:
                    y, x = float(c[b, i, j + 1, 0]), float(c[b, i, j + 1, 1])
                    u = rng.random()
                    if u < 0.1:
                        x += 15.0                                                   # exactly at the threshold
                    elif u < 0.15:
                        x += 15.0000001                                             # just beyond it
                    else:
                        x, y = x + rng.normal(0, 12), y + rng.normal(0, 12)
                else:
                    x, y = rng.uniform(0, 400, 2)
                pts.append({"id": [j], "x": [x], "y": [y]})
            if rng.random() < 0.1 and pts:
                pts.append(dict(pts[0], x=[-1000.0]))                               # a duplicate id: the first counts
            rect["annopoints"] = [{"point": pts}]
            rects.append(rect)
        frames.append({"image": [f"{b}.jpg"], "annorect": rects})
    return frames


def run_match(cfg, packed, gt_frames, J):
    """ppn_ap_match on one batch -> host (score, label, used, flags, n_gt)."""
    from pytorch_pose_proposal_network_b200 import _lib
    from pytorch_pose_proposal_network_b200.evaluation import gt_from_frames
    lib = _lib.lib()
    B, R = packed.count.shape[0], packed.R
    off, box, xy, valid = [torch.from_numpy(x).cuda() for x in gt_from_frames(gt_frames, J)]
    out = (torch.full((B, R, J), -1.0, device="cuda"), torch.full((B, R, J), 7, dtype=torch.uint8, device="cuda"),
           torch.empty(B, dtype=torch.int32, device="cuda"), torch.empty(B, dtype=torch.int32, device="cuda"),
           torch.empty(B, J, dtype=torch.int32, device="cuda"))
    hs = _lib.PPNHumans(*[t.data_ptr() for t in (packed.count, packed.root_cell, packed.part_cell, packed.part_score,
                                                   packed.part_box)], R)
    gt = _lib.PPNPoseGT(off.data_ptr(), box.data_ptr(), xy.data_ptr(), valid.data_ptr(), box.shape[0])
    m = _lib.PPNAPMatch(*[t.data_ptr() for t in out], R)
    _lib.check(lib.ppn_ap_match(C.byref(hs), B, cfg.K, C.byref(gt), C.byref(_lib.PPNAPParams(J, 0.5, 0.6)), C.byref(m),
                                torch.cuda.current_stream().cuda_stream), "ppn_ap_match")
    return [t.cpu().numpy() for t in out]


CASES = [("cfg2", 512, "U", torch.float32, 24), ("cfg2", 512, "S", torch.float16, 24), ("native", 64, "S", torch.float32, 64),
         ("native", 64, "R", torch.float16, 16), ("cfg3", 1024, "D", torch.float32, 6), ("cfg3", 1024, "D", torch.float16, 6)]


@pytest.mark.parametrize("preset,B,dist,dtype,n_check", CASES)
def test_match_equals_restatement(preset, B, dist, dtype, n_check):
    from pytorch_pose_proposal_network_b200.evaluation import pred_frames
    cfg = cfg_of(preset)
    J = cfg.K - 1
    head, _ = device_head(O.Geometry.of(cfg), dist, seed=B + len(dist), B=B, dtype=dtype, distinct=False)
    parser, packed = parse(cfg, head)
    centres = parser.part_centres(packed)
    rng = np.random.default_rng(B)
    gts = gt_frames_near(rng, packed, centres, J, crowd_image=1)
    score, label, used, flags, n_gt = run_match(cfg, packed, gts, J)
    counts = packed.count.cpu().numpy()
    assert (used == np.minimum(counts, packed.R)).all() and (flags == 0).all()
    check = sorted(set(rng.choice(B, n_check, replace=False).tolist()) | {0, 1})       # 1 holds 64 GT people
    preds = pred_frames([f"{b}.jpg" for b in range(B)], packed, centres)
    s_all, l_all, n_all = P.assign_gt_multi([gts[b] for b in check], [preds[b] for b in check], J)
    n_tp = 0
    for k, b in enumerate(check):
        u = used[b]
        assert n_gt[b].tolist() == n_all[:, k].astype(int).tolist(), b
        for j in range(J):
            want_s = np.asarray(s_all[j][k], np.float32).reshape(u)
            assert np.array_equal(score[b, :u, j].view(np.uint32), want_s.view(np.uint32)), (b, j)
            assert label[b, :u, j].tolist() == l_all[j][k], (b, j)
            n_tp += sum(l_all[j][k])
        assert (label[b, u:] == 7).all() and (score[b, u:] == -1.0).all()       # slots past the count untouched
    assert n_tp > 0


def evaluator(cfg, **kw):
    from pytorch_pose_proposal_network_b200.evaluation import APEvaluator
    return APEvaluator(cfg, **kw)


def assert_results_close(got, want):
    for k in ("ap", "precision", "recall"):
        assert got[k].dtype == np.float64 and got[k].shape == want[k].shape
        np.testing.assert_allclose(got[k], want[k], rtol=0, atol=1e-9, equal_nan=True, err_msg=k)


def bit_equal(r1, r2):
    return all(np.array_equal(r1[k].view(np.uint64), r2[k].view(np.uint64)) for k in ("ap", "precision", "recall"))


def pass_inputs(preset, dist, dtype, B, n_batches, seed, **gt_kw):
    """Parsed batches (re-parsed into fresh buffers each time) with their pred and GT frames."""
    from pytorch_pose_proposal_network_b200.evaluation import pred_frames
    cfg = cfg_of(preset)
    batches = []
    rng = np.random.default_rng(seed)
    for i in range(n_batches):
        head, _ = device_head(O.Geometry.of(cfg), dist, seed=seed + i, B=B, dtype=dtype, distinct=False)
        parser, packed = parse(cfg, head)
        centres = parser.part_centres(packed)
        gts = gt_frames_near(rng, packed, centres, cfg.K - 1, **gt_kw)
        batches.append((head, packed, pred_frames([f"{i}_{b}.jpg" for b in range(B)], packed, centres), gts))
    return cfg, batches


@pytest.mark.parametrize("preset,dist,dtype,B,n_batches", [("native", "S", torch.float32, 16, 3),
                                                          ("cfg2", "S", torch.float16, 24, 2),
                                                          ("cfg3", "D", torch.float16, 4, 2)])
def test_ap_values_match_restatement(preset, dist, dtype, B, n_batches):
    cfg, batches = pass_inputs(preset, dist, dtype, B, n_batches, seed=11)
    ev = evaluator(cfg)
    for _, packed, _, gts in batches:
        ev.update(packed, gts)
    got = ev.compute()
    want = P.evaluate([g for *_, gts in batches for g in gts], [p for _, _, preds, _ in batches for p in preds], cfg.K - 1)
    assert_results_close(got, want)
    assert np.isfinite(got["ap"]).all() and got["ap"][-1] > 0
    ev.reset()
    assert (ev.compute()["ap"] == 0).all()


def test_score_ties_and_joint_count():
    """fp16 heads make many equal part scores; absent parts add score-0 ties; J below and above K - 1."""
    cfg, batches = pass_inputs("cfg2", "R", torch.float16, 16, 2, seed=5)
    for J in (4, cfg.K - 1, cfg.K + 3):
        ev = evaluator(cfg, n_joints=J)
        for _, packed, _, gts in batches:
            ev.update(packed, gts)
        got = ev.compute()
        want = P.evaluate([g for *_, gts in batches for g in gts], [p for _, _, preds, _ in batches for p in preds], J)
        assert_results_close(got, want)
    used = [(a["part_score"][b, :n, 1:]).ravel() for a in (bt[1].numpy() for bt in batches)
            for b, n in enumerate(a["count"])]
    scores = np.concatenate(used)
    assert np.unique(scores).size < scores.size // 4


def test_nan_for_joints_without_gt():
    cfg, batches = pass_inputs("native", "S", torch.float32, 8, 1, seed=3)
    _, packed, preds, gts = batches[0]
    for fr in gts:
        for r in fr["annorect"]:
            if "annopoints" in r:
                r["annopoints"][0]["point"] = [p for p in r["annopoints"][0]["point"] if p["id"][0] != 2]
    ev = evaluator(cfg)
    ev.update(packed, gts)
    got = ev.compute()
    assert np.isnan(got["ap"][2]) and np.isnan(got["recall"][2]) and got["precision"][2] == 0.0
    assert np.isnan(got["ap"][-1])
    assert_results_close(got, P.evaluate(gts, preds, cfg.K - 1))


def test_batch_split_max_humans_and_repeat_invariance():
    from pytorch_pose_proposal_network_b200.evaluation import gt_from_frames
    cfg, batches = pass_inputs("native", "S", torch.float32, 48, 1, seed=21)
    head, packed, _, gts = batches[0]
    ev = evaluator(cfg)
    ev.update(packed, gts)
    ref = ev.compute()
    assert bit_equal(ref, ev.compute())                                      # compute twice
    ev2 = evaluator(cfg)
    ev2.update(packed, gts)
    assert bit_equal(ref, ev2.compute())                                     # a second run
    for split in ((7, 41), (16, 16, 16), (1, 46, 1)):
        ev = evaluator(cfg)
        b0 = 0
        for n in split:
            _, p = parse(cfg, head[b0:b0 + n].contiguous())
            ev.update(p, gts[b0:b0 + n])
            b0 += n
        assert bit_equal(ref, ev.compute()), split
    need = int(packed.count.max())
    for R in (need, need + 3):
        _, p = parse(cfg, head, max_humans=R)
        ev = evaluator(cfg)
        ev.update(p, gts)
        assert bit_equal(ref, ev.compute()), R
    # mixed slot counts in one pass, and update_flat with device GT
    ev = evaluator(cfg)
    _, p1 = parse(cfg, head[:20].contiguous(), max_humans=need)
    _, p2 = parse(cfg, head[20:].contiguous())
    ev.update(p1, gts[:20])
    ev.update_flat(p2, *[torch.from_numpy(a).cuda() for a in gt_from_frames(gts[20:], cfg.K - 1)])
    assert bit_equal(ref, ev.compute())


def test_encoder_round_trip_scores_100():
    """People encoded into a head tensor and parsed back are scored against themselves: AP 100 for every joint."""
    from pytorch_pose_proposal_network_b200 import config as pcfg
    cfg = cfg_of("native")
    g = O.Geometry.of(cfg)
    cell = cfg.inW // cfg.W
    heads, frames = [], []
    rng = np.random.default_rng(0)
    for b in range(6):
        people, rects = [], []
        for q in range(4):
            qy, qx = divmod(q, 2)
            if rng.random() < 0.2:
                continue
            ry, rx = 12 * qy + 8, 12 * qx + 6                                  # root cell of the quadrant
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
    parser, packed = parse(cfg, head)
    assert packed.count.cpu().tolist() == [len(f["annorect"]) for f in frames]
    ev = evaluator(cfg)
    ev.update(packed, frames)
    got = ev.compute()
    assert (got["recall"] == 100.0).all() and (got["precision"] == 100.0).all()
    np.testing.assert_allclose(got["ap"], 100.0, rtol=0, atol=1e-9)         # VOCap's sum of recall steps


def test_overflow_and_bad_gt_raise():
    from pytorch_pose_proposal_network_b200.evaluation import gt_from_frames
    cfg, batches = pass_inputs("native", "S", torch.float32, 8, 1, seed=9)
    head, packed, _, gts = batches[0]
    assert int(packed.count.max()) > 1
    _, small = parse(cfg, head, max_humans=1)
    ev = evaluator(cfg)
    ev.update(small, gts)
    with pytest.raises(RuntimeError, match="max_humans"):
        ev.compute()
    crowd = [{"image": ["c.jpg"], "annorect": [{"x1": [0.0], "y1": [0.0], "x2": [3.0], "y2": [4.0]}] * 65}] + gts[1:]
    ev = evaluator(cfg)
    with pytest.raises(ValueError, match="64"):
        ev.update(packed, crowd)
    ev.update_flat(packed, *[torch.from_numpy(a).cuda() for a in gt_from_frames(crowd, cfg.K - 1)])   # flagged on the device
    with pytest.raises(RuntimeError, match="GT people"):
        ev.compute()
    with pytest.raises(ValueError):
        ev.update(packed.cpu(), gts)


def test_update_flat_does_not_synchronise():
    from pytorch_pose_proposal_network_b200.evaluation import gt_from_frames
    cfg, batches = pass_inputs("native", "S", torch.float32, 16, 1, seed=2)
    _, packed, _, gts = batches[0]
    flat = [torch.from_numpy(a).cuda() for a in gt_from_frames(gts, cfg.K - 1)]
    ev = evaluator(cfg)
    ev.update_flat(packed, *flat)                                            # first call: library load etc.
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        ev.update_flat(packed, *flat)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    res = ev.compute()
    ev1 = evaluator(cfg)
    ev1.update(packed, gts)
    ev1.update(packed, gts)
    assert bit_equal(res, ev1.compute())
