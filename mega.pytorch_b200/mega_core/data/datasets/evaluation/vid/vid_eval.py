"""ImageNet-VID detection evaluation with the reference's function names and results
(data/datasets/evaluation/vid/vid_eval.py:14-343; SURVEY.md section 8f row 2).

Same protocol: per image and class the detections, sorted by score, are matched greedily against that class's
ground-truth boxes (IoU on integer-typed "+1" boxes, ignore flags from the motion-IoU range), the per-class match /
ignore lists are concatenated over the dataset, sorted by score, and turned into precision / recall and the
area-under-curve AP. What differs is where the time goes: the matching loops, which the reference runs in Python for every
(image, class, detection, box), are one native call per (image, class) (`mega_vid_match_host` in libmega_b200.so), and
the per-image bookkeeping is array code. Precision / recall / AP arrays equal the reference's element for element
(tests/test_vid_eval_cpu.py runs both on the same synthetic detections).

`device="cuda"` scores the whole run on the GPU instead (libmega_b200.so's mega_vid_eval_* kernels, every motion range
in one pass; mega_core.b200.ops.vid_eval): the same structures come back. It ranks equal scores by one rule, the order of
numpy's `argsort(kind="stable")[::-1]`, where the host path keeps the reference's plain `argsort()[::-1]`, whose order
among equal scores is numpy's unstable sort; without ties both give the same order. Cumulative false positives of the
motion ranges (fractional weights) are summed in a parallel order, so they agree with the host's to ~1e-15 relative.
`do_vid_evaluation` uses the device path when the environment variable MEGA_B200_EVAL_DEVICE is "cuda"."""
import os
from collections import defaultdict

import numpy as np

from ..... import _lib


def _match(pred_boxes, gt_boxes, gt_ignore, iou_thresh, empty_weight):
    p, g = pred_boxes.shape[0], gt_boxes.shape[0]
    match = np.zeros(p, dtype=np.int8)
    ignore = np.zeros(p, dtype=np.float64)
    pb = np.ascontiguousarray(pred_boxes, dtype=np.float32)
    gb = np.ascontiguousarray(gt_boxes, dtype=np.float32)
    gi = np.ascontiguousarray(gt_ignore != 0, dtype=np.uint8)
    _lib.check(_lib.lib.mega_vid_match_host(pb.ctypes.data, p, gb.ctypes.data, gi.ctypes.data, g, float(iou_thresh),
                                            float(empty_weight), match.ctypes.data, ignore.ctypes.data),
               "mega_vid_match_host")
    return match, ignore


def _empty_weight(motion_ious, motion_range):
    """ignore weight of detections of a class without GT in their image (vid_eval.py:160-169)"""
    if motion_ious is None:
        return 0
    lo, hi = motion_range
    flat = np.concatenate(motion_ious, axis=0)
    empty_weight = np.count_nonzero((flat >= lo) & (flat <= hi)) / float(len(flat))
    return 0 if empty_weight == 1 else empty_weight


def _device_eval(gt_boxlists, pred_boxlists, motion_ious, iou_thresh, motion_ranges, want_prec_rec, device):
    """-> per range (prec, rec, ap) from the GPU evaluator, ranges in passes of up to four"""
    from .....b200 import ops
    packed = ops.vid_eval_pack(pred_boxlists, gt_boxlists, motion_ious)
    out = []
    step = ops.VID_EVAL_MAX_RANGES
    for first in range(0, len(motion_ranges), step):
        ranges = [tuple(rng) for rng in motion_ranges[first:first + step]]
        res = ops.vid_eval(packed, ranges, [_empty_weight(motion_ious, rng) for rng in ranges], iou_thresh,
                           want_prec_rec, device)
        host = {k: (v.cpu().numpy() if v is not None and k not in ("match", "ignore", "order") else None)
                for k, v in res.items()}
        seen, count, n_pos = host["seen"], host["det_count"].astype(np.int64), host["n_pos"]
        start = np.concatenate(([0], np.cumsum(count)))
        for i in range(len(ranges)):
            prec = rec = None
            if want_prec_rec:
                prec = [host["prec"][i, start[l]:start[l + 1]].copy() if seen[l] else None for l in range(len(seen))]
                rec = [host["rec"][i, start[l]:start[l + 1]].copy() if seen[l] and n_pos[i, l] > 0 else None
                       for l in range(len(seen))]
            out.append((prec, rec, host["ap"][i].copy()))
    return out


def calc_detection_vid_prec_rec(gt_boxlists, pred_boxlists, motion_ious, iou_thresh=0.5, motion_range=(0., 1.),
                                device=None):
    """-> (prec, rec): lists indexed by class id (None where a class never occurs), as vid_eval.py:156-284.
    device="cuda": computed by the GPU evaluator (module docstring)"""
    if device is not None and str(device) != "cpu":
        prec, rec, _ = _device_eval(gt_boxlists, pred_boxlists, motion_ious, iou_thresh, [motion_range], True, device)[0]
        return prec, rec
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
            order = ps[sel].argsort()[::-1]                    # the reference's (unstable) sort call: same tie order
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
        order = score_l.argsort()[::-1]
        match_l, ign_l = match_l[order], ign_l[order]
        counted = ign_l != 1
        tps = (match_l == 1) & counted
        fps = ((match_l == 0) & counted) * np.where(ign_l == 0, 1.0, ign_l)      # fractional weight of "mixed" misses
        tp, fp = np.cumsum(tps), np.cumsum(fps)
        prec[l] = tp / (fp + tp + np.spacing(1))
        if n_pos[l] > 0:
            rec[l] = tp / n_pos[l]
    return prec, rec


def calc_detection_vid_ap(prec, rec, use_07_metric=False):
    """per-class average precision from precision / recall (vid_eval.py:287-343): area under the monotone envelope of the
    PR curve, or the 11-point VOC07 metric; NaN for classes without ground truth"""
    ap = np.full(len(prec), np.nan)
    for l, (p, r) in enumerate(zip(prec, rec)):
        if p is None or r is None:
            continue
        p = np.nan_to_num(p)
        if use_07_metric:
            ap[l] = sum((p[r >= t].max() if np.any(r >= t) else 0.0) / 11 for t in np.arange(0.0, 1.1, 0.1))
            continue
        mpre = np.concatenate(([0], p, [0]))
        mrec = np.concatenate(([0], r, [1]))
        mpre = np.maximum.accumulate(mpre[::-1])[::-1]
        step = np.where(mrec[1:] != mrec[:-1])[0]
        ap[l] = np.sum((mrec[step + 1] - mrec[step]) * mpre[step + 1])
    return ap


def eval_detection_vid(pred_boxlists, gt_boxlists, iou_thresh=0.5, motion_ranges=((0.0, 0.7), (0.7, 0.9), (0.9, 1.0)),
                       motion_specific=False, use_07_metric=False, motion_ious=None, device=None):
    """vid_eval.py:120-153; motion_specific reads the reference's vid_groundtruth_motion_iou.mat (from the working
    directory, like the reference) unless `motion_ious` is given. device="cuda": every range in one GPU pass (module
    docstring); only the per-class APs come back to the host, or prec / rec for the 11-point metric."""
    assert len(gt_boxlists) == len(pred_boxlists), "Length of gt and pred lists need to be same."
    if motion_specific and motion_ious is None:
        import scipy.io as sio
        mat = sio.loadmat(os.path.join("mega_core", "data", "datasets", "evaluation", "vid",
                                       "vid_groundtruth_motion_iou.mat"))["motion_iou"]
        motion_ious = [[mat[i][0][j][0] if len(mat[i][0][j]) != 0 else 0 for j in range(len(mat[i][0]))]
                       for i in range(len(mat))]
    result = {}
    if device is not None and str(device) != "cpu":
        scored = _device_eval(gt_boxlists, pred_boxlists, motion_ious if motion_specific else None, iou_thresh,
                              motion_ranges, use_07_metric, device)
        for index, (prec, rec, ap) in enumerate(scored):
            if use_07_metric:
                ap = calc_detection_vid_ap(prec, rec, True)
            result[index] = {"ap": ap, "map": np.nanmean(ap)}
        return result
    for index, rng in enumerate(motion_ranges):
        prec, rec = calc_detection_vid_prec_rec(gt_boxlists, pred_boxlists, motion_ious if motion_specific else None,
                                                iou_thresh, rng)
        ap = calc_detection_vid_ap(prec, rec, use_07_metric)
        result[index] = {"ap": ap, "map": np.nanmean(ap)}
    return result


def do_vid_evaluation(dataset, predictions, output_folder, box_only, motion_specific, logger):
    """vid_eval.py:14-69 (detection branch; proposal recall -- box_only -- is outside the inference path).
    MEGA_B200_EVAL_DEVICE=cuda scores on the GPU (eval_detection_vid's device path); unset or "cpu": on the host"""
    if box_only:
        raise NotImplementedError("proposal-recall evaluation is not part of the B200 build")
    device = os.environ.get("MEGA_B200_EVAL_DEVICE", "cpu") or "cpu"
    if device != "cpu" and not device.startswith("cuda"):
        raise ValueError("MEGA_B200_EVAL_DEVICE must be 'cpu' or 'cuda', not %r" % device)
    preds, gts = [], []
    for image_id, prediction in enumerate(predictions):
        info = dataset.get_img_info(image_id)
        preds.append(prediction.resize((info["width"], info["height"])))
        gts.append(dataset.get_groundtruth(image_id))
    ranges = [[0.0, 1.0], [0.0, 0.7], [0.7, 0.9], [0.9, 1.0]] if motion_specific else [[0.0, 1.0]]
    names = ["all", "fast", "medium", "slow"][:len(ranges)]
    result = eval_detection_vid(preds, gts, 0.5, ranges, motion_specific, False,
                                device=None if device == "cpu" else device)
    text = "".join("AP50 | motion={:>6s} = {:0.4f}\n".format(n, result[i]["map"]) for i, n in enumerate(names))
    text += "Category AP:\n"
    for i, ap in enumerate(result[0]["ap"]):
        if i:                                          # class 0 is the background
            text += "{:<16}: {:.4f}\n".format(dataset.map_class_id_to_class_name(i), ap)
    logger.info("\n" + text)
    if output_folder:
        with open(os.path.join(output_folder, "result.txt"), "w") as fid:
            fid.write(text)
    return result
