"""Oracle of the device VID evaluator's ranking rule: calc_detection_vid_prec_rec (the host path of
mega_core/data/datasets/evaluation/vid/vid_eval.py) restated with numpy's STABLE sorts, `argsort(kind="stable")[::-1]`
both inside each (image, class) and over each class. Matching is the host's own native call. On data without equal scores
inside a class this is the host path element for element (tests/test_vid_eval_device_cpu.py checks it); with ties it is
the order the device evaluator documents. Also builds BoxLists from arrays."""
from collections import defaultdict

import numpy as np
import torch


def boxlists(preds, gts, size=(640, 360)):
    """(boxes, labels, scores) / (boxes, labels) numpy tuples per image -> (pred BoxLists, gt BoxLists)"""
    from mega_core.structures.bounding_box import BoxList
    pl, gl = [], []
    for (b, l, s), (gb, glab) in zip(preds, gts):
        p = BoxList(torch.as_tensor(np.asarray(b, dtype=np.float32)).reshape(-1, 4), size, mode="xyxy")
        p.add_field("labels", torch.as_tensor(np.asarray(l, dtype=np.int64)))
        p.add_field("scores", torch.as_tensor(np.asarray(s, dtype=np.float32)))
        g = BoxList(torch.as_tensor(np.asarray(gb, dtype=np.float32)).reshape(-1, 4), size, mode="xyxy")
        g.add_field("labels", torch.as_tensor(np.asarray(glab, dtype=np.int64)))
        pl.append(p)
        gl.append(g)
    return pl, gl


def prec_rec_stable(gt_boxlists, pred_boxlists, motion_ious, iou_thresh=0.5, motion_range=(0.0, 1.0)):
    from mega_core.data.datasets.evaluation.vid.vid_eval import _empty_weight, _match
    lo, hi = motion_range
    empty_weight = _empty_weight(motion_ious, motion_range)
    if motion_ious is None:
        motion_ious = [None] * len(gt_boxlists)
    n_pos = defaultdict(int)
    scores, matches, ignores = defaultdict(list), defaultdict(list), defaultdict(list)
    for gt, pred, motion in zip(gt_boxlists, pred_boxlists, motion_ious):
        pb, pl, ps = pred.bbox.numpy(), pred.get_field("labels").numpy(), pred.get_field("scores").numpy()
        gb, gl = gt.bbox.numpy(), gt.get_field("labels").numpy()
        g_ign = np.zeros(len(gb))
        if motion is not None and len(motion) > 0:
            m = np.asarray(motion, dtype=np.float64)[:len(gb)]
            g_ign[:len(m)] = ((m < lo) | (m > hi)).astype(np.float64)
        for l in np.unique(np.concatenate((pl, gl)).astype(int)):
            sel = pl == l
            order = ps[sel].argsort(kind="stable")[::-1]
            pb_l, ps_l = pb[sel][order], ps[sel][order]
            gsel = gl == l
            gb_l, gi_l = gb[gsel], g_ign[gsel]
            n_pos[l] += gb_l.shape[0] - gi_l.sum()
            scores[l].append(ps_l)
            if pb_l.shape[0] == 0:
                continue
            m_l, i_l = _match(pb_l, gb_l, gi_l, iou_thresh, empty_weight)
            matches[l].append(m_l)
            ignores[l].append(i_l)
    n_fg_class = max(n_pos.keys()) + 1
    prec, rec = [None] * n_fg_class, [None] * n_fg_class
    for l in n_pos.keys():
        cat = lambda parts, dt: np.concatenate(parts).astype(dt) if parts else np.zeros(0, dtype=dt)   # noqa: E731
        score_l, match_l, ign_l = cat(scores[l], np.float32), cat(matches[l], np.int8), cat(ignores[l], np.float64)
        order = score_l.argsort(kind="stable")[::-1]
        match_l, ign_l = match_l[order], ign_l[order]
        counted = ign_l != 1
        tps = (match_l == 1) & counted
        fps = ((match_l == 0) & counted) * np.where(ign_l == 0, 1.0, ign_l)
        tp, fp = np.cumsum(tps), np.cumsum(fps)
        prec[l] = tp / (fp + tp + np.spacing(1))
        if n_pos[l] > 0:
            rec[l] = tp / n_pos[l]
    return prec, rec
