"""CPU checks of the device VID evaluator (csrc/vid_eval.cu, vid_eval.cuh; mega_core.b200.ops.vid_eval):
  1. the per-(image, class) segment body the matching kernel runs, compiled for the host by g++ with -ffp-contract=off
     (tests/native/vid_eval_host.cpp: one lane, the warp's 32-lane argmax tree emulated), returns the match flags and
     ignore weights of mega_vid_match_host -- on every segment of tests/golden/vid_eval.pt and on 20 k seeded segments
     full of tied IoUs (between ignored and non-ignored GT too), IoUs exactly at the threshold, zero-area boxes, tied
     scores and empty sides, with the segment's detections and GT listed in shuffled order;
  2. the stable-tie restatement of the host evaluator (tests/vid_eval_restatement.py), the device's ranking rule, equals
     the host path element for element on data without equal scores;
  3. the library exports the new entry points, the ABI version is still 6, and the device path refuses CPU tensors."""
import ctypes
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import vid_eval_restatement as vr  # noqa: E402

RANGES = [(0.0, 1.0), (0.0, 0.7), (0.7, 0.9), (0.9, 1.0)]
_host = None


def host_lib():
    """g++ build of the segment body (into a temporary directory: the tree may be read-only)"""
    global _host
    if _host is None:
        out = os.path.join(tempfile.mkdtemp(prefix="vid_eval_host_"), "libvid_eval_host.so")
        subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-std=c++17", "-I",
                               os.path.join(ROOT, "mega.pytorch_b200", "csrc"), "-o", out,
                               os.path.join(ROOT, "tests", "native", "vid_eval_host.cpp")])
        _host = ctypes.CDLL(out)
        _host.vid_match_segment_host.restype = ctypes.c_int
        _host.vid_match_segment_host.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_int] + [ctypes.c_void_p] * 3 + [
            ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_float] + [ctypes.c_void_p] * 4
        _host.vid_score_key_host.restype = ctypes.c_uint
        _host.vid_score_key_host.argtypes = [ctypes.c_float]
    return _host


def _p(a):
    return a.ctypes.data if a is not None else None


def segment_body(boxes, scores, gt_boxes, motion, ranges, empties, thr, det_idx, gt_idx):
    n, g, r = len(scores), len(gt_boxes), len(ranges)
    boxes = np.ascontiguousarray(boxes, dtype=np.float32).reshape(-1, 4)
    scores = np.ascontiguousarray(scores, dtype=np.float32)
    gt_boxes = np.ascontiguousarray(gt_boxes, dtype=np.float32).reshape(-1, 4)
    motion = None if motion is None else np.ascontiguousarray(motion, dtype=np.float64)
    det_idx, gt_idx = np.ascontiguousarray(det_idx, dtype=np.int32), np.ascontiguousarray(gt_idx, dtype=np.int32)
    rng = np.ascontiguousarray(ranges, dtype=np.float64).reshape(-1)
    emp = np.ascontiguousarray(empties, dtype=np.float64)
    order = np.zeros(max(n, 1), dtype=np.int32)
    sel = np.zeros(max(g * r, 1), dtype=np.uint8)
    match = np.full((r, max(n, 1)), -7, dtype=np.int8)
    ign = np.full((r, max(n, 1)), -7.0)
    assert host_lib().vid_match_segment_host(_p(boxes), _p(scores), _p(det_idx), n, _p(gt_boxes), _p(motion),
                                             _p(gt_idx), g, r, _p(rng), _p(emp), thr, _p(order), _p(sel), _p(match),
                                             _p(ign)) == 0
    return match[:, :n], ign[:, :n]


def segment_host(boxes, scores, gt_boxes, motion, ranges, empties, thr):
    """mega_vid_match_host per range on the detections in stable descending score order"""
    from mega_core.data.datasets.evaluation.vid.vid_eval import _match
    n = len(scores)
    order = np.asarray(scores, dtype=np.float32).argsort(kind="stable")[::-1]
    match = np.zeros((len(ranges), n), dtype=np.int8)
    ign = np.zeros((len(ranges), n))
    for r, (lo, hi) in enumerate(ranges):
        gi = np.zeros(len(gt_boxes)) if motion is None else ((motion < lo) | (motion > hi)).astype(np.float64)
        if n:
            m, w = _match(np.asarray(boxes, dtype=np.float32).reshape(-1, 4)[order],
                          np.asarray(gt_boxes, dtype=np.float32).reshape(-1, 4), gi, thr, empties[r])
            match[r, order], ign[r, order] = m, w
    return match, ign


def _check_segment(boxes, scores, gt_boxes, motion, ranges, empties, thr, rs):
    mh, ih = segment_host(boxes, scores, gt_boxes, motion, ranges, empties, thr)
    mb, ib = segment_body(boxes, scores, gt_boxes, motion, ranges, empties, thr, rs.permutation(len(scores)),
                          rs.permutation(len(gt_boxes)))
    assert np.array_equal(mh, mb) and np.array_equal(ih.view(np.int64), ib.view(np.int64)), (boxes, scores, gt_boxes,
                                                                                              motion, mh, mb, ih, ib)


def test_segment_body_equals_native_matching_on_the_golden_fixture():
    from mega_core.data.datasets.evaluation.vid.vid_eval import _empty_weight
    cases = torch.load(os.path.join(ROOT, "tests", "golden", "vid_eval.pt"), weights_only=False)
    rs = np.random.RandomState(0)
    n_seg = 0
    for case in cases:
        motions = [im["motion"] for im in case["images"]]
        empties = [_empty_weight(motions, rng) for rng in RANGES]
        for im in case["images"]:
            pl, gl = im["labels"].numpy(), im["gt_labels"].numpy()
            m = np.full(len(gl), np.nan)
            mm = np.asarray(im["motion"], dtype=np.float64)[:len(gl)]
            m[:len(mm)] = mm
            for l in np.unique(np.concatenate((pl, gl))):
                d, g = pl == l, gl == l
                args = (im["boxes"].numpy()[d], im["scores"].numpy()[d], im["gt"].numpy()[g])
                _check_segment(*args, m[g], RANGES, empties, 0.5, rs)
                _check_segment(*args, None, RANGES[:1], [0.0], 0.5, rs)
                n_seg += 1
    assert n_seg > 300


def _iou_f32(p, g):
    """the IoU of mega_vid_match_host in numpy float32 (same operation order, no contraction)"""
    one = np.float32(1)
    px2, py2, gx2, gy2 = p[:, None, 2] + one, p[:, None, 3] + one, g[None, :, 2] + one, g[None, :, 3] + one
    pa = (px2 - p[:, None, 0] + one) * (py2 - p[:, None, 1] + one)
    ga = (gx2 - g[None, :, 0] + one) * (gy2 - g[None, :, 1] + one)
    w = np.maximum(np.minimum(px2, gx2) - np.maximum(p[:, None, 0], g[None, :, 0]) + one, np.float32(0))
    h = np.maximum(np.minimum(py2, gy2) - np.maximum(p[:, None, 1], g[None, :, 1]) + one, np.float32(0))
    inter = w * h
    return inter / (pa + ga - inter)


def test_segment_body_equals_native_matching_on_seeded_hard_segments():
    rs = np.random.RandomState(1)
    motion_values = np.array([0.3, 0.65, 0.7, 0.8, 0.9, 0.95, 1.0, np.nan])
    empties = [0.0, 0.3, 0.25, 0.4]
    stats = dict(at_thresh=0, tied_max=0, tied_mixed=0, zero_area=0, no_gt=0, no_det=0)

    def box(k):
        x1, y1 = rs.randint(0, 8, k), rs.randint(0, 8, k)
        x2, y2 = x1 + rs.randint(-1, 5, k), y1 + rs.randint(-1, 5, k)
        return np.stack([x1, y1, x2, y2], 1).astype(np.float32)

    for _ in range(20000):
        n, g = rs.randint(0, 10), rs.randint(0, 6)
        boxes, gt = box(n), box(g)
        if g and rs.rand() < 0.5:                                   # duplicated GT boxes: tied IoUs
            gt = np.concatenate([gt, gt[rs.randint(0, g, rs.randint(1, 4))]])
        motion = motion_values[rs.randint(0, len(motion_values), len(gt))]
        scores = (rs.randint(1, 6, n) / 10.0).astype(np.float32)    # tied scores
        if len(gt) and n:
            iou = _iou_f32(boxes, gt)
            stats["at_thresh"] += int((iou == np.float32(0.5)).sum())
            mx = iou.max(1, keepdims=True)
            tied = (iou == mx) & (mx >= 0.5)
            stats["tied_max"] += int((tied.sum(1) > 1).sum())
            ign = (motion < 0.7) | (motion > 0.9)
            stats["tied_mixed"] += int(((tied & ign[None]).any(1) & (tied & ~ign[None]).any(1)).sum())
        stats["zero_area"] += int(((boxes[:, 2] <= boxes[:, 0]) | (boxes[:, 3] <= boxes[:, 1])).sum())
        stats["no_gt"] += len(gt) == 0
        stats["no_det"] += n == 0
        thr = 0.5 if rs.rand() < 0.8 else float(rs.choice([0.3, 0.7]))
        _check_segment(boxes, scores, gt, motion, RANGES, empties, thr, rs)
        _check_segment(boxes, scores, gt, None, RANGES[:1], [0.0], thr, rs)
    assert min(stats.values()) > 100, stats


def test_score_key_orders_like_the_floats():
    lib = host_lib()
    vals = np.array([-np.inf, -3.5, -1e-30, -0.0, 0.0, 1e-38, 1e-3, 0.5, 0.5000001, 1.0, np.inf], dtype=np.float32)
    keys = [lib.vid_score_key_host(float(v)) for v in vals]
    assert keys[3] == keys[4]
    assert all(a < b for a, b in zip(keys[:3] + keys[4:], keys[1:3] + keys[4:][1:] + [2 ** 32])) and keys[2] < keys[3]


def test_stable_restatement_equals_host_path_without_ties():
    from mega_core.b200 import synth
    from mega_core.data.datasets.evaluation.vid import calc_detection_vid_prec_rec
    preds, gts, motions = synth.vid_eval_set(400, seed=5, max_dets=40, tie_free=True)
    pl, gl = vr.boxlists(preds, gts)
    for motion, rng in [(None, (0.0, 1.0))] + [(motions, r) for r in RANGES]:
        hp, hr = calc_detection_vid_prec_rec(gl, pl, motion, 0.5, rng)
        sp, sr = vr.prec_rec_stable(gl, pl, motion, 0.5, rng)
        assert len(hp) == len(sp) == 31
        for a, b in zip(hp + hr, sp + sr):
            assert (a is None) == (b is None)
            if a is not None:
                assert np.array_equal(a, b)


def test_stable_restatement_differs_from_host_only_in_tie_order_on_the_fixture():
    """the golden fixture has tied scores inside classes; the restatement orders them one documented way, and the APs it
    gives stay close to the reference's own (their difference is the tie order alone)"""
    from mega_core.data.datasets.evaluation.vid import calc_detection_vid_ap
    cases = torch.load(os.path.join(ROOT, "tests", "golden", "vid_eval.pt"), weights_only=False)
    for case in cases:
        pl, gl = vr.boxlists([(im["boxes"], im["labels"], im["scores"]) for im in case["images"]],
                             [(im["gt"], im["gt_labels"]) for im in case["images"]])
        sp, sr = vr.prec_rec_stable(gl, pl, None, 0.5, (0.0, 1.0))
        ap = calc_detection_vid_ap(sp, sr)
        assert np.nanmax(np.abs(ap - case["reference"]["all"]["ap"])) < 0.05


def test_library_exports_the_device_evaluator():
    from mega_core import _lib
    lib = _lib.lib
    for s in ("mega_vid_eval_workspace_bytes", "mega_vid_eval_match", "mega_vid_eval_rank", "mega_vid_eval_scan_ap"):
        assert hasattr(lib, s) and s in _lib.EXPORTS
    assert lib.mega_abi_version() == 6
    assert lib.mega_vid_eval_workspace_bytes(1000, 100, 31, 4) > 1000 * 24
    assert lib.mega_vid_eval_workspace_bytes(0, 0, 31, 1) >= 0
    assert lib.mega_vid_eval_workspace_bytes(1000, 100, 513, 4) == -1
    assert lib.mega_vid_eval_workspace_bytes(1000, 100, 31, 5) == -1
    assert lib.mega_vid_eval_workspace_bytes(2 ** 31, 100, 31, 1) == -1


def test_device_path_has_no_cpu_fallback():
    from mega_core import _lib
    from mega_core.b200 import ops
    preds = [(np.array([[0, 0, 10, 10]]), np.array([1]), np.array([0.9]))]
    gts = [(np.array([[0, 0, 10, 10]]), np.array([1]))]
    pl, gl = vr.boxlists(preds, gts)
    packed = ops.vid_eval_pack(pl, gl, None)
    assert packed["num_classes"] == 2 and packed["det_off"].tolist() == [0, 1]
    with pytest.raises(_lib.MegaError):
        ops.vid_eval(packed, [(0.0, 1.0)], [0.0], device="cpu")
    with pytest.raises(ValueError):
        ops.vid_eval_pack(vr.boxlists([(np.zeros((0, 4)), [], [])], [(np.zeros((0, 4)), [])])[0],
                          vr.boxlists([(np.zeros((0, 4)), [], [])], [(np.zeros((0, 4)), [])])[1])
