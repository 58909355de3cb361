"""Known answers for the float64 restatement of poseval's assignGTmulti / computeMetrics (oracle/pose_ap.py), worked
out by hand so that the restatement the GPU tests compare against cannot merely confirm itself.  No GPU."""
import math

import numpy as np
import pytest

from oracle import pose_ap as P


def gt_rect(points, box=(0.0, 0.0, 30.0, 40.0)):
    """points: {joint: (x, y)}; the default head box has headSize 0.6 * |(30, 40)| = 30."""
    x1, y1, x2, y2 = box
    rect = {"x1": [x1], "y1": [y1], "x2": [x2], "y2": [y2]}
    if points is not None:
        rect["annopoints"] = [{"point": [{"id": [j], "x": [x], "y": [y]} for j, (x, y) in points.items()]}]
    return rect


def pr_rect(points, score=0.5):
    """points: {joint: (x, y)} or {joint: (x, y, score)}."""
    pts = []
    for j, p in points.items():
        pts.append({"id": [j], "x": [p[0]], "y": [p[1]], "score": [p[2] if len(p) > 2 else score]})
    return {"annopoints": [{"point": pts}]}


def frame(rects):
    return {"image": ["x.jpg"], "annorect": rects}


def labels(gt_rects, pr_rects, J):
    s, l, n = P.assign_gt_multi([frame(gt_rects)], [frame(pr_rects)], J)
    return [l[j][0] for j in range(J)], [s[j][0] for j in range(J)], n[:, 0]


def test_head_size_and_threshold():
    assert P.head_size(0.0, 0.0, 30.0, 40.0) == 30.0
    gt = [gt_rect({0: (100.0, 100.0)})]
    lab, _, n_gt = labels(gt, [pr_rect({0: (115.0, 100.0)})], 1)     # exactly 0.5 * headSize away
    assert lab == [[1]] and list(n_gt) == [1]
    lab, _, _ = labels(gt, [pr_rect({0: (100.0, 85.0)})], 1)
    assert lab == [[1]]
    lab, _, _ = labels(gt, [pr_rect({0: (115.00001, 100.0)})], 1)    # slightly over
    assert lab == [[0]]
    lab, _, _ = labels(gt, [pr_rect({0: (109.0, 112.0)})], 1)        # |(9, 12)| = 15
    assert lab == [[1]]


def test_higher_pck_wins_and_first_index_on_ties():
    g = {j: (50.0 * j, 10.0) for j in range(4)}
    near = lambda js: {j: (g[j][0] if j in js else g[j][0] + 100.0, 10.0) for j in range(4)}
    gt = [gt_rect(g)]
    lab, _, _ = labels(gt, [pr_rect(near({0, 1})), pr_rect(near({1, 2, 3}))], 4)
    assert [lab[j][0] for j in range(4)] == [0, 0, 0, 0]            # pck 2/4 loses
    assert [lab[j][1] for j in range(4)] == [0, 1, 1, 1]            # pck 3/4 takes the GT person
    lab, _, _ = labels(gt, [pr_rect(near({0, 1})), pr_rect(near({2, 3}))], 4)
    assert [lab[j][0] for j in range(4)] == [1, 1, 0, 0]            # equal pck: the first prediction
    assert [lab[j][1] for j in range(4)] == [0, 0, 0, 0]


def test_prediction_preferring_a_taken_gt_stays_unmatched():
    gt = [gt_rect({0: (10.0, 10.0), 1: (60.0, 10.0)}), gt_rect({0: (300.0, 10.0), 1: (400.0, 10.0)})]
    p0 = pr_rect({0: (10.0, 10.0), 1: (60.0, 10.0)})                # GT 0 with pck 1
    p1 = pr_rect({0: (10.0, 10.0), 1: (400.0, 10.0)})               # GT 0 with 1/2 (its best), GT 1 with 1/2
    lab, _, n_gt = labels(gt, [p0, p1], 2)
    assert [lab[j][0] for j in range(2)] == [1, 1]
    assert [lab[j][1] for j in range(2)] == [0, 0]                  # GT 1 is free but p1's best was GT 0
    assert list(n_gt) == [2, 2]


def test_gt_without_joints_never_matches():
    gt = [gt_rect(None), gt_rect({})]
    lab, _, n_gt = labels(gt, [pr_rect({0: (0.0, 0.0), 1: (5.0, 5.0)})], 2)
    assert lab == [[0], [0]] and list(n_gt) == [0, 0]


def test_image_without_gt_labels_its_predictions_zero():
    lab, sc, n_gt = labels([], [pr_rect({0: (1.0, 1.0)}, 0.9), pr_rect({0: (2.0, 2.0)}, 0.8)], 1)
    assert lab == [[0, 0]] and sc == [[0.9, 0.8]] and list(n_gt) == [0]


def test_absent_parts_are_score_zero_entries():
    from pytorch_pose_proposal_network_b200.evaluation import pred_frame
    K, R = 4, 3
    cell = np.full((1, R, K), -1, np.int32)
    cell[0, 0, [0, 1, 3]] = [5, 6, 7]                               # part 2 (joint 1) absent
    score = np.zeros((1, R, K), np.float32)
    score[0, 0, [0, 1, 3]] = [0.9, 0.75, 0.5]
    box = np.zeros((1, R, K, 4), np.float32)
    box[0, 0, 1] = (10, 20, 30, 40)                                 # centre (y, x) = (20, 30)
    centres = np.zeros((1, R, K, 2), np.float32)
    centres[0, 0, 1] = (20, 30)
    packed = {"count": np.array([1], np.int32), "part_cell": cell, "part_score": score, "part_box": box}
    pr = pred_frame("a.jpg", packed, centres, 0)
    gt = gt_rect({0: (30.0, 20.0), 1: (0.0, 0.0)})                 # joint 1 annotated exactly at (0, 0)
    s, l, n = P.assign_gt_multi([frame([gt])], [pr], 3)
    assert [s[j][0] for j in range(3)] == [[np.float32(0.75)], [0], [np.float32(0.5)]]
    assert [l[j][0] for j in range(3)] == [[1], [1], [0]]            # the absent part still sits at (0, 0)
    assert list(n[:, 0]) == [1, 1, 0]


def metrics(scores, labels, n_gt):
    """one joint, one image per list entry"""
    return P.compute_metrics([[list(scores)]], [[list(labels)]], np.array([[float(n_gt)]]))


def test_tie_rule_later_entry_first():
    ap, pre, rec = metrics([0.5, 0.5], [1, 0], 1)
    assert ap[0] == 50.0 and pre[0] == 50.0 and rec[0] == 100.0
    ap, _, _ = metrics([0.5, 0.5], [0, 1], 1)
    assert ap[0] == 100.0
    ap, _, _ = metrics([-0.0, 0.0], [1, 0], 1)                      # -0 ties with +0
    assert ap[0] == 50.0
    ap, _, _ = metrics([0.9, float("nan")], [1, 0], 1)              # NaN ranks first
    assert ap[0] == 50.0


def test_precision_envelope():
    ap, pre, rec = metrics([0.9, 0.8, 0.7], [0, 1, 1], 4)
    assert math.isclose(ap[0], 100.0 / 3.0, rel_tol=1e-15)
    assert math.isclose(pre[0], 200.0 / 3.0, rel_tol=1e-15) and rec[0] == 50.0
    assert ap[1] == ap[0] and pre[1] == pre[0] and rec[1] == rec[0]  # one joint: the mean is that joint


def test_no_gt_is_nan_and_no_entries_is_zero():
    scores_all = [[[0.9, 0.5]], [[]], [[0.4]]]
    labels_all = [[[0, 0]], [[]], [[1]]]
    ap, pre, rec = P.compute_metrics(scores_all, labels_all, np.array([[0.0], [3.0], [1.0]]))
    assert math.isnan(ap[0]) and math.isnan(rec[0]) and pre[0] == 0.0
    assert ap[1] == 0.0 and pre[1] == 0.0 and rec[1] == 0.0
    assert ap[2] == 100.0 and pre[2] == 100.0 and rec[2] == 100.0
    assert math.isnan(ap[3]) and math.isnan(rec[3]) and math.isclose(pre[3], 100.0 / 3.0)


def test_gt_from_frames():
    from pytorch_pose_proposal_network_b200.evaluation import gt_from_frames
    frames = [frame([gt_rect({1: (5.0, 6.0), 0: (1.0, 2.0), 7: (9.0, 9.0)}), gt_rect(None, (1, 2, 3, 4))]), frame([])]
    frames[0]["annorect"][0]["annopoints"][0]["point"].append({"id": [1], "x": [50.0], "y": [60.0]})   # not the first
    off, box, xy, valid = gt_from_frames(frames, 3)
    assert off.tolist() == [0, 2, 2] and off.dtype == np.int32
    assert box.tolist() == [[0, 0, 30, 40], [1, 2, 3, 4]] and box.dtype == np.float64
    assert valid.tolist() == [[1, 1, 0], [0, 0, 0]] and valid.dtype == np.uint8
    assert xy[0, :2].tolist() == [[1.0, 2.0], [5.0, 6.0]] and xy.shape == (2, 3, 2)
