"""Multi-person pose AP, restated in float64.  TEST INFRASTRUCTURE (the specification of csrc/ppn_eval.cu).

The reference scores its validation pass with the poseval fork: ``eval_helpers.assignGTmulti`` matches the
predicted people of every image to the ground truth by PCKh, and ``evaluateAP.computeMetrics`` turns the labelled
joint detections of the whole pass into AP, precision and recall per joint.  The fork is not part of this tree, so
this module restates those functions loop for loop, on the same frames (``{"image": ..., "annorect": [...]}``):
predictions as ``evaluation.pred_frame`` builds them, ground truth with ``x1, y1, x2, y2`` head boxes and
``annopoints[0]["point"]`` entries ``{"id": [j], "x": [..], "y": [..]}``.  It is also the CPU arm of
``scripts/bench_ap.py``.

Reconstruction points (DESIGN.md §12):
  1. ties: ``np.argsort(scores, kind="stable")[::-1]`` -- descending score, the later-appended entry first among
     equal scores, NaN first; numpy's default quicksort leaves the order of ties unpinned;
  2. distances are ``sqrt(dx*dx + dy*dy)`` in float64, one rounding per operation, in place of ``np.linalg.norm``;
  3. no ``cleanupData`` / ``removeIgnoredPoints``: images without GT people keep their predictions as false
     positives, which is what ``assignGTmulti`` itself does;
  4. the number of joints J is a parameter (the fork's ``Joint().count`` is not known here).
"""
from __future__ import annotations

import numpy as np


def get_point(points, pidx):
    """poseval's getPointGTbyID: the first point whose id is ``pidx``, or [] if there is none."""
    for p in points:
        if p["id"] is not None and p["id"][0] == pidx:
            return p
    return []


def head_size(x1, y1, x2, y2, head_scale=0.6):
    hx = np.float64(x2) - np.float64(x1)
    hy = np.float64(y2) - np.float64(y1)
    return np.float64(head_scale) * np.sqrt(hx * hx + hy * hy)


def _points(rect):
    if "annopoints" in rect and len(rect["annopoints"]) > 0:
        return rect["annopoints"][0]["point"]
    return []


def assign_gt_multi(gt_frames, pr_frames, n_joints, dist_thresh=0.5, head_scale=0.6):
    """assignGTmulti: -> (scores_all, labels_all, n_gt_all) with scores_all[j][img] / labels_all[j][img] the entries
    of joint j appended by image img (in prediction order) and n_gt_all [J, n_images] the annotated GT joints."""
    assert len(gt_frames) == len(pr_frames)
    J = n_joints
    scores_all = [[[] for _ in gt_frames] for _ in range(J)]
    labels_all = [[[] for _ in gt_frames] for _ in range(J)]
    n_gt_all = np.zeros((J, len(gt_frames)))
    for img, (gtf, prf) in enumerate(zip(gt_frames, pr_frames)):
        gts, prs = gtf["annorect"], prf["annorect"]
        dist = np.full((len(prs), len(gts), J), np.inf)
        score = np.full((len(prs), J), np.nan)
        has_pr = np.zeros((len(prs), J), dtype=bool)
        has_gt = np.zeros((len(gts), J), dtype=bool)
        for g, rect in enumerate(gts):
            pts = _points(rect)
            for j in range(J):
                if len(get_point(pts, j)) > 0:
                    has_gt[g, j] = True
        for i, rect in enumerate(prs):
            pts = _points(rect)
            for j in range(J):
                pp = get_point(pts, j)
                if len(pp) > 0:
                    score[i, j] = pp["score"][0]
                    has_pr[i, j] = True
        pr_to_gt = np.zeros(0, dtype=np.int64)
        match = np.zeros((len(prs), len(gts), J), dtype=bool)
        if len(prs) and len(gts):
            with np.errstate(divide="ignore", invalid="ignore"):
                for g, rect in enumerate(gts):
                    hs = head_size(rect["x1"][0], rect["y1"][0], rect["x2"][0], rect["y2"][0], head_scale)
                    pts_gt = _points(rect)
                    for i, prect in enumerate(prs):
                        pts_pr = _points(prect)
                        for j in range(J):
                            if has_pr[i, j] and has_gt[g, j]:
                                pg, pp = get_point(pts_gt, j), get_point(pts_pr, j)
                                dx = np.float64(pp["x"][0]) - np.float64(pg["x"][0])
                                dy = np.float64(pp["y"][0]) - np.float64(pg["y"][0])
                                dist[i, g, j] = np.sqrt(dx * dx + dy * dy) / hs
                match = dist <= dist_thresh
            n_gtp = np.sum(has_gt, axis=1)
            pck = 1.0 * np.sum(match, axis=2)
            for i in range(has_pr.shape[0]):
                for g in range(has_gt.shape[0]):
                    if n_gtp[g] > 0:
                        pck[i, g] = pck[i, g] / n_gtp[g]
            idx = np.argmax(pck, axis=1)                       # best GT of every prediction ...
            for i in range(pck.shape[0]):
                for g in range(pck.shape[1]):
                    if g != idx[i]:
                        pck[i, g] = 0
            pr_to_gt = np.argmax(pck, axis=0)                  # ... and the best of those for every GT
            val = np.max(pck, axis=0)
            pr_to_gt[val == 0] = -1
        for i in range(has_pr.shape[0]):
            if i in pr_to_gt:
                g = np.argwhere(pr_to_gt == i)
                assert g.size == 1
                m = match[i, g[0, 0], :]
            else:
                m = np.zeros(J, dtype=bool)
            for j in range(J):
                if has_pr[i, j]:
                    scores_all[j][img].append(score[i, j])
                    labels_all[j][img].append(int(m[j]))
        for g in range(has_gt.shape[0]):
            for j in range(J):
                n_gt_all[j, img] += has_gt[g, j]
    return scores_all, labels_all, n_gt_all


def compute_rpc(scores, labels, total_pos):
    """computeRPC, with the tie order pinned (reconstruction point 1)."""
    precision = np.zeros(len(scores))
    recall = np.zeros(len(scores))
    npos = 0
    idxs = np.asarray(scores, np.float64).argsort(kind="stable")[::-1]
    labels_sorted = np.asarray(labels)[idxs]
    with np.errstate(divide="ignore", invalid="ignore"):
        for s in range(len(idxs)):
            if labels_sorted[s] == 1:
                npos += 1
            recall[s] = np.float64(npos) / np.float64(total_pos)
            precision[s] = np.float64(npos) / np.float64(s + 1)
    return precision, recall, idxs


def voc_ap(rec, prec):
    """VOCap: area under the precision envelope at the recall steps."""
    mpre = np.zeros([1, 2 + len(prec)])
    mpre[0, 1:len(prec) + 1] = prec
    mrec = np.zeros([1, 2 + len(rec)])
    mrec[0, 1:len(rec) + 1] = rec
    mrec[0, len(rec) + 1] = 1.0
    for i in range(len(prec) + 1, 0, -1):
        mpre[0, i - 1] = max(mpre[0, i - 1], mpre[0, i])
    i = np.argwhere(~np.equal(mrec[0, 1:], mrec[0, :mrec.shape[1] - 1])) + 1
    i = i.flatten()
    return np.sum(np.multiply(np.subtract(mrec[0, i], mrec[0, i - 1]), mpre[0, i]))


def compute_metrics(scores_all, labels_all, n_gt_all):
    """computeMetrics -> (ap, precision, recall), float64 [J + 1] in percent, the last entry the mean over joints.
    A joint without entries keeps 0; a joint with entries and no GT joint gets NaN recall and AP (0 / 0), and so
    does the mean."""
    J = n_gt_all.shape[0]
    ap, pre, rec = np.zeros(J + 1), np.zeros(J + 1), np.zeros(J + 1)
    for j in range(J):
        scores = [s for img in scores_all[j] for s in img]
        labels = [l for img in labels_all[j] for l in img]
        n_gt = np.sum(n_gt_all[j, :])
        precision, recall, _ = compute_rpc(scores, labels, n_gt)
        if len(precision) > 0:
            with np.errstate(invalid="ignore"):
                ap[j] = voc_ap(recall, precision) * 100
            pre[j] = precision[len(precision) - 1] * 100
            rec[j] = recall[len(recall) - 1] * 100
    ap[J], pre[J], rec[J] = np.mean(ap[:J]), np.mean(pre[:J]), np.mean(rec[:J])
    return ap, pre, rec


def evaluate(gt_frames, pr_frames, n_joints, dist_thresh=0.5, head_scale=0.6):
    """The whole scoring stage: {"ap", "precision", "recall"}, float64 [J + 1] each."""
    ap, pre, rec = compute_metrics(*assign_gt_multi(gt_frames, pr_frames, n_joints, dist_thresh, head_scale))
    return {"ap": ap, "precision": pre, "recall": rec}
