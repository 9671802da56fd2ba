"""TEST INFRASTRUCTURE: CPU restatements for the class-agnostic box mAP (torchmetrics
``MeanAveragePrecision(average="micro")``) and for the third table of pycocotools ``COCOeval.accumulate``, ``scores``.

* ``micro_records`` -- COCOeval.evaluateImg on one image of an ``oracle.run_pipeline`` output with every label set to 0:
  ``oracle.coco_match`` on all kept detections (descending score) against all GT boxes of the image.  With the records'
  labels at 0, ``oracle.accumulate_ap(..., nc=1)`` cuts maxDets per image, as torchmetrics does under "micro".
* ``score_table`` -- the numpy restatement of the score table (the layout of ``precision``: [T, R, nc, A, M]),
  written the way ``oracle.accumulate_ap`` restates precision.
* ``pycocotools_score_table`` -- an independent, loop-for-loop restatement of pycocotools' accumulate for that table
  (``inds = searchsorted(rc, recThrs, 'left')``, ``ss[ri] = dtScoresSorted[pi]`` until the IndexError), used to
  cross-check ``score_table``.
"""
from __future__ import annotations

import numpy as np

from oracle import oracle

REC_THRS = np.linspace(0.0, 1.0, 101)


def micro_records(out, b, thrs):
    """(record dict for accumulate_ap with labels 0, dt_match [A, T, k], dt_ignore [A, T, k], gt_ignore [A, g]) of image
    `b` of an oracle output, matched with the labels ignored."""
    k, g = int(out["det_count"][b]), int(out["gt_count"][b])
    dm, di, gi = oracle.coco_match(out["dets"][b, :k, :4], out["gt_boxes"][b, :g], thrs)
    rec = dict(labels=np.zeros(k, np.int64), scores=out["dets"][b, :k, 4], matched=dm > 0, ignored=di > 0)
    return rec, dm, di, gi


def micro_ap(outs, thrs, max_dets=(1, 10, 100), drop=False):
    """oracle.accumulate_ap(nc=1) over the class-agnostic records of a list of oracle outputs (images in global order),
    and the NPIG counts [4, 1] (GTs of every class; v2's `drop` rule removes an image without candidates)."""
    recs, npig = [], np.zeros((4, 1), np.int64)
    for out in outs:
        for b in range(len(out["det_count"])):
            rec, _, _, gi = micro_records(out, b, thrs)
            recs.append(rec)
            if not (drop and int(out["n_cand"][b]) == 0):
                npig[:, 0] += (gi == 0).sum(1)
    return oracle.accumulate_ap(recs, npig, thrs, max_dets, 1), npig, recs


def _sequence(records, c, a, md):
    """The (class, area range, maxDet) sequence in the accumulate's order: scores, matched [T, n], ignored [T, n]."""
    sc, mt, ig = [], [], []
    for r in records:
        sel = np.nonzero(r["labels"] == c)[0][:md]
        sc.append(r["scores"][sel]); mt.append(r["matched"][a][:, sel]); ig.append(r["ignored"][a][:, sel])
    sc = np.concatenate(sc) if sc else np.zeros(0, np.float32)
    T = records[0]["matched"].shape[1] if records else 0
    mt = np.concatenate(mt, 1) if mt else np.zeros((T, 0), bool)
    ig = np.concatenate(ig, 1) if ig else np.zeros((T, 0), bool)
    order = np.argsort(-sc, kind="mergesort")
    return sc[order], mt[:, order], ig[:, order]


def score_table(records, n_gt_valid, thrs, max_dets=(1, 10, 100), nc=3):
    """COCOeval.accumulate's `scores` [T, R, nc, A, M]: the score of the first position whose recall reaches each recall
    threshold; 0 past the last recall reached (or for an empty sequence), -1 where npig == 0."""
    T, A, M = len(thrs), 4, len(max_dets)
    scores = -np.ones((T, len(REC_THRS), nc, A, M))
    for c in range(nc):
        for a in range(A):
            npig = int(n_gt_valid[a][c])
            if npig == 0:
                continue
            for mi, md in enumerate(max_dets):
                sc, mt, ig = _sequence(records, c, a, md)
                nd = len(sc)
                rc = np.cumsum(mt & ~ig, 1).astype(np.float64) / npig          # [T, nd]
                for t in range(T):
                    pos = np.searchsorted(rc[t], REC_THRS, side="left")
                    scores[t, :, c, a, mi] = np.where(pos < nd, sc[np.minimum(pos, max(nd - 1, 0))] if nd else 0.0, 0.0)
    return scores


def pycocotools_score_table(records, n_gt_valid, thrs, max_dets=(1, 10, 100), nc=3):
    """The same table, restated statement by statement from pycocotools' COCOeval.accumulate."""
    T, A, M, R = len(thrs), 4, len(max_dets), len(REC_THRS)
    scores = -np.ones((T, R, nc, A, M))
    for k0 in range(nc):
        for a0 in range(A):
            for m, maxDet in enumerate(max_dets):
                E = [dict(dtScores=r["scores"][r["labels"] == k0][0:maxDet],
                          dtMatches=r["matched"][a0][:, r["labels"] == k0][:, 0:maxDet],
                          dtIgnore=r["ignored"][a0][:, r["labels"] == k0][:, 0:maxDet]) for r in records]
                if len(E) == 0:
                    continue
                dtScores = np.concatenate([e["dtScores"] for e in E])
                inds = np.argsort(-dtScores, kind="mergesort")
                dtScoresSorted = dtScores[inds]
                dtm = np.concatenate([e["dtMatches"] for e in E], axis=1)[:, inds]
                dtIg = np.concatenate([e["dtIgnore"] for e in E], axis=1)[:, inds]
                npig = int(n_gt_valid[a0][k0])
                if npig == 0:
                    continue
                tps = np.logical_and(dtm, np.logical_not(dtIg))
                tp_sum = np.cumsum(tps, axis=1).astype(dtype=np.float64)
                for t, tp in enumerate(tp_sum):
                    tp = np.array(tp)
                    rc = tp / npig
                    ss = np.zeros((R,))
                    inds2 = np.searchsorted(rc, REC_THRS, side="left")
                    try:
                        for ri, pi in enumerate(inds2):
                            ss[ri] = dtScoresSorted[pi]
                    except IndexError:
                        pass
                    scores[t, :, k0, a0, m] = np.array(ss)
    return scores


def records_from_ring(rec):
    """decode_records() output -> per-image record dicts in image order, each in rank order (the layout accumulate_ap
    and score_table take)."""
    out = []
    for img in np.unique(rec["image"]):
        sel = np.nonzero(rec["image"] == img)[0]
        sel = sel[np.argsort(rec["rank"][sel], kind="stable")]
        out.append(dict(labels=rec["label"][sel], scores=rec["score"][sel], matched=np.moveaxis(rec["matched"][sel], 0, 2),
                        ignored=np.moveaxis(rec["ignored"][sel], 0, 2)))
    return out
