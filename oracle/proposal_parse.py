"""Proposal-pair parse restated in numpy: the specification of ``ppn_parse_proposals``.  TEST INFRASTRUCTURE ONLY.

The reference parser (``oracle/ppn_oracle.py``) runs NMS on part 0 only and walks the arg-max of each limb window
from every root, so several humans may claim the same part cell.  This is the parse the paper describes instead:
every part gets NMS-filtered proposals, limbs score candidate pairs of proposals, and a greedy parse down the
skeleton tree lets humans compete for parts.  The reference has no code for it; this file is its specification
(DESIGN.md §13).  ``oracle/proposal_parse.c`` (binding: ``oracle/c_proposal_parse.py``) is its C twin.

Arithmetic is fp32 with one rounding per written operation (numpy never fuses); thresholds are demoted to fp32.
For one image [C, H, W]:

1. Proposals.  delta = resp * conf and the boxes are ``ppn_oracle``'s.  For EVERY part k the candidates are the
   cells with delta[k] > det_thresh (strict), suppressed by ``ppn_oracle.nms`` (IoU >= nms_thresh; equal scores:
   larger cell first).  The survivors P_k keep NMS order.
2. Humans.  Human i is the i-th proposal of P_0; its root is that cell.
3. Tree.  Every target part of the track orders must be reached by one limb from one predecessor, and part 0 must
   never be a target (``ValueError`` otherwise).  Non-root parts are processed in first-reach order.
4. Pairs of limb e = (s -> t).  Sources: the cell a of part s of every human that has part s.  Targets: every
   b in P_t.  With (ih, iw) = divmod(a, W), (jh, jw) = divmod(b, W), dy = jh - ih + off_h, dx = jw - iw + off_w,
   the pair exists iff 0 <= dy < sH and 0 <= dx < sW (the reference's displacement, datatest.py:115-116).
   Its score is sc = (delta[s, a] * lv) * delta[t, b], left to right, lv = e[e, dy, dx, ih, iw].  It is a
   candidate iff sc > 0 (so NaN, zero and negative limb values never connect).
5. Matching.  Candidates in order of score descending, then smaller human index, then smaller target cell (a strict
   total order); a pair is accepted if its human has no part t yet and b is unused by this limb.
6. Output.  Humans in root NMS order; those with at least min_kp non-root parts are kept (after matching: the
   parts of a dropped human go to no one).  part_score = delta[t, cell], part_box = box(t, cell).

Reconstruction points (the paper leaves them open; DESIGN.md §13 states them too):
  (a) the connection score (delta_s * limb) * delta_t — the paper combines limb and part confidences, this exact
      form is a choice made here;
  (b) sc > 0 is the only limb test, no separate limb threshold (the reference has none either);
  (c) the tie rule of step 5;
  (d) an at-threshold cell is not a proposal: every part needs delta > thr, while the reference accepts a walked
      limb target at delta == thr (datatest.py:121);
  (e) top-down matching: only sources attached to a human compete, so orphan subtrees are never formed.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Tuple

import numpy as np

from . import ppn_oracle as O

f32 = np.float32


def limb_tree(g: O.Geometry) -> List[Tuple[int, int, int]]:
    """(limb, source part, target part) of every non-root part in first-reach order over the track orders.

    Raises ValueError unless the track orders form a tree rooted at part 0 (the ``parallel_ok`` test of the C ABI's
    chain check): a part reached twice must be reached by the same limb from the same predecessor."""
    how = {}
    order = []
    for eis, ts in g.graphs:
        pred = 0
        for e, t in zip(eis, ts):
            e, t = int(e), int(t)
            if t == 0:
                raise ValueError("track orders lead back to part 0: not a tree")
            if t not in how:
                how[t] = (e, pred)
                order.append((e, pred, t))
            elif how[t] != (e, pred):
                raise ValueError(f"part {t} is reached by two different limbs or predecessors: not a tree")
            pred = t
    return order


def proposals(out: np.ndarray, g: O.Geometry):
    """Step 1 -> (delta [K, HW], boxes [K, HW, 4], [P_k cells in NMS order for every part])."""
    resp, conf, x, y, w, h, _ = O.split_head(out, g)
    delta = (resp * conf).reshape(g.K, -1)
    bbox = O.boxes(x, y, w, h, g).reshape(g.K, -1, 4)
    P = []
    for k in range(g.K):
        cand = O.root_candidates(delta[k], g.det_thresh)
        keep = O.nms(bbox[k][cand], g.nms_thresh, score=delta[k][cand])
        P.append(cand[keep].astype(np.int32))
    return delta, bbox, P


def limb_pairs(e_img: np.ndarray, delta: np.ndarray, cell: np.ndarray, P_t: np.ndarray, limb: Tuple[int, int, int],
               g: O.Geometry):
    """Step 4 for one limb -> (score, human, target cell) of every candidate pair, unsorted.  e_img: [E, sH, sW, H, W]."""
    e, s, t = limb
    jh, jw = np.divmod(P_t.astype(np.int64), g.W)
    sc_l, hum_l, tgt_l = [], [], []
    for i in range(cell.shape[0]):                   # one source at a time, all targets of P_t at once
        a = int(cell[i, s])
        if a < 0:
            continue
        ih, iw = divmod(a, g.W)
        dy, dx = jh - ih + g.oh, jw - iw + g.ow
        inside = (dy >= 0) & (dy < g.sH) & (dx >= 0) & (dx < g.sW)
        b = P_t[inside]
        lv = e_img[e, dy[inside], dx[inside], ih, iw]
        sc = (delta[s, a] * lv) * delta[t, b]           # two fp32 products, left to right
        ok = sc > f32(0)
        sc_l.append(sc[ok]); hum_l.append(np.full(int(ok.sum()), i, np.int64)); tgt_l.append(b[ok].astype(np.int64))
    if not sc_l:
        return np.zeros(0, f32), np.zeros(0, np.int64), np.zeros(0, np.int64)
    return np.concatenate(sc_l).astype(f32), np.concatenate(hum_l), np.concatenate(tgt_l)


def match_limb(sc, hum, tgt, cell: np.ndarray, t: int) -> None:
    """Step 5 for one limb, in place on cell[:, t]."""
    order = np.lexsort((tgt, hum, -sc.astype(np.float64)))     # score descending, then human, then cell
    used = set()
    for q in order:
        i, b = int(hum[q]), int(tgt[q])
        if cell[i, t] < 0 and b not in used:
            cell[i, t] = b
            used.add(b)


@dataclass
class ProposalParsed:
    """One image's result in the packed layout (include/ppn_decode.h, PPNHumans) plus the stage counts."""
    root_cell: np.ndarray     # [n] int32
    part_cell: np.ndarray     # [n, K] int32, -1 = absent
    part_score: np.ndarray    # [n, K] fp32 (0 where absent)
    part_box: np.ndarray      # [n, K, 4] fp32 (0 where absent)
    proposals: list           # P_k, cells in NMS order
    n_pairs: np.ndarray       # [E] candidate pairs (sc > 0) per limb, 0 for limbs outside the tree


def parse_image(out: np.ndarray, g: O.Geometry) -> ProposalParsed:
    """Steps 1-6 for one image [C, H, W] fp32."""
    tree = limb_tree(g)
    delta, bbox, P = proposals(out, g)
    e_img = out[6 * g.K:].reshape(g.E, g.sH, g.sW, g.H, g.W)
    n0 = P[0].size
    cell = np.full((n0, g.K), -1, np.int32)
    cell[:, 0] = P[0]
    n_pairs = np.zeros(g.E, np.int64)
    for limb in tree:
        sc, hum, tgt = limb_pairs(e_img, delta, cell, P[limb[2]], limb, g)
        n_pairs[limb[0]] = sc.size
        match_limb(sc, hum, tgt, cell, limb[2])
    keep = [i for i in range(n0) if int((cell[i, 1:] >= 0).sum()) >= g.min_kp]
    cell = cell[keep] if keep else np.zeros((0, g.K), np.int32)
    n = cell.shape[0]
    score = np.zeros((n, g.K), f32)
    box = np.zeros((n, g.K, 4), f32)
    for i in range(n):
        for t in np.flatnonzero(cell[i] >= 0):
            score[i, t] = delta[t, cell[i, t]]
            box[i, t] = bbox[t, cell[i, t]]
    return ProposalParsed(cell[:, 0].copy(), cell, score, box, P, n_pairs)


def parse_batch(head: np.ndarray, g: O.Geometry):
    """[B, C, H, W] -> dict(count [B], root_cell [B, HW], part_cell [B, HW, K], part_score, part_box), the layout of
    ``c_proposal_parse.proposal_parse_batch`` (slots past count: -1 / 0)."""
    B, HW, K = head.shape[0], g.H * g.W, g.K
    r = dict(count=np.zeros(B, np.int32), root_cell=np.full((B, HW), -1, np.int32),
             part_cell=np.full((B, HW, K), -1, np.int32), part_score=np.zeros((B, HW, K), f32),
             part_box=np.zeros((B, HW, K, 4), f32))
    for b in range(B):
        p = parse_image(np.ascontiguousarray(head[b], f32), g)
        n = p.root_cell.size
        r["count"][b] = n
        r["root_cell"][b, :n] = p.root_cell
        r["part_cell"][b, :n] = p.part_cell
        r["part_score"][b, :n] = p.part_score
        r["part_box"][b, :n] = p.part_box
    return r
