"""The device VID evaluator (mega_core.b200.ops.vid_eval; eval_detection_vid(..., device="cuda")) against the host path
on the B200: per-detection match flags / ignore weights, precision / recall and AP for the plain protocol and the three
motion ranges; the golden fixture (tied scores) against the stable-tie restatement; edge cases; determinism; and
do_vid_evaluation's result.txt with MEGA_B200_EVAL_DEVICE=cuda."""
import logging
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import vid_eval_restatement as vr  # noqa: E402

RANGES = [(0.0, 1.0), (0.0, 0.7), (0.7, 0.9), (0.9, 1.0)]
MOTION_RANGES = RANGES[1:]


def _host_matches(pl, gl, motions, ranges):
    """per-detection match / ignore of the host matching ([R, N], detections packed image after image)"""
    from mega_core.data.datasets.evaluation.vid.vid_eval import _empty_weight, _match
    n = sum(len(p) for p in pl)
    match = np.zeros((len(ranges), n), dtype=np.int8)
    ign = np.zeros((len(ranges), n))
    empties = [_empty_weight(motions, r) for r in ranges]
    base = 0
    for i, (p, g) in enumerate(zip(pl, gl)):
        pb, lab, sc = p.bbox.numpy(), p.get_field("labels").numpy(), p.get_field("scores").numpy()
        gb, glab = g.bbox.numpy(), g.get_field("labels").numpy()
        m = np.full(len(gb), np.nan)
        if motions is not None and len(motions[i]):
            mm = np.asarray(motions[i], dtype=np.float64)[:len(gb)]
            m[:len(mm)] = mm
        for l in np.unique(lab):
            idx = np.nonzero(lab == l)[0]
            idx = idx[sc[idx].argsort(kind="stable")[::-1]]
            gsel = glab == l
            for r, (lo, hi) in enumerate(ranges):
                gi = ((m[gsel] < lo) | (m[gsel] > hi)).astype(np.float64)
                mt, w = _match(pb[idx], gb[gsel], gi, 0.5, empties[r])
                match[r, base + idx], ign[r, base + idx] = mt, w
        base += len(pb)
    return match, ign


def _same_bits(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert (x is None) == (y is None)
        if x is not None:
            assert x.shape == y.shape and np.array_equal(x, y), np.abs(x - y).max()


def _close(a, b, rel=1e-12):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert (x is None) == (y is None)
        if x is not None:
            assert x.shape == y.shape
            assert np.all(np.abs(x - y) <= rel * np.abs(y)), np.max(np.abs(x - y) / np.maximum(np.abs(y), 1e-300))


def _ap_close(a, b, tol=1e-12):
    assert a.shape == b.shape and np.array_equal(np.isnan(a), np.isnan(b))
    assert np.nanmax(np.abs(a - b)) <= tol if np.any(~np.isnan(a)) else True


@pytest.fixture(scope="module")
def tie_free():
    from mega_core.b200 import synth
    preds, gts, motions = synth.vid_eval_set(20000, seed=11, max_dets=20, tie_free=True)
    pl, gl = vr.boxlists(preds, gts)
    return pl, gl, motions


def test_match_flags_and_ignore_weights_are_bit_identical(tie_free):
    from mega_core.b200 import ops
    from mega_core.data.datasets.evaluation.vid.vid_eval import _empty_weight
    pl, gl, motions = tie_free
    packed = ops.vid_eval_pack(pl, gl, motions)
    out = ops.vid_eval(packed, RANGES, [_empty_weight(motions, r) for r in RANGES])
    mh, ih = _host_matches(pl, gl, motions, RANGES)
    assert np.array_equal(out["match"].cpu().numpy(), mh)
    assert np.array_equal(out["ignore"].cpu().numpy().view(np.int64), ih.view(np.int64))
    # the ranking: every class block, read backwards, in descending score
    order = out["order"].cpu().numpy()
    labels, scores = packed["det_labels"].numpy()[order], packed["det_scores"].numpy()[order]
    assert np.all(np.diff(labels) >= 0) and sorted(order.tolist()) == list(range(len(order)))
    same = np.diff(labels) == 0
    assert np.all(np.diff(scores)[same] > 0)


def test_prec_rec_ap_equal_the_host_path(tie_free):
    from mega_core.data.datasets.evaluation.vid import calc_detection_vid_ap, calc_detection_vid_prec_rec, eval_detection_vid
    pl, gl, motions = tie_free
    hp, hr = calc_detection_vid_prec_rec(gl, pl, None, 0.5, (0.0, 1.0))
    dp, dr = calc_detection_vid_prec_rec(gl, pl, None, 0.5, (0.0, 1.0), device="cuda")
    _same_bits(dp, hp)                               # every fp is 0 or 1: integer sums, exact in any order
    _same_bits(dr, hr)
    host_ap = {None: calc_detection_vid_ap(hp, hr)}
    for rng in MOTION_RANGES:
        hp, hr = calc_detection_vid_prec_rec(gl, pl, motions, 0.5, rng)
        dp, dr = calc_detection_vid_prec_rec(gl, pl, motions, 0.5, rng, device="cuda")
        _close(dp, hp)
        _close(dr, hr)
        host_ap[rng] = calc_detection_vid_ap(hp, hr)
    res = eval_detection_vid(pl, gl, 0.5, [(0.0, 1.0)], motion_specific=False, device="cuda")
    _ap_close(res[0]["ap"], host_ap[None])
    assert abs(res[0]["map"] - np.nanmean(host_ap[None])) <= 1e-12
    res = eval_detection_vid(pl, gl, 0.5, MOTION_RANGES, motion_specific=True, motion_ious=motions, device="cuda")
    for i, rng in enumerate(MOTION_RANGES):
        _ap_close(res[i]["ap"], host_ap[rng])
        assert abs(res[i]["map"] - np.nanmean(host_ap[rng])) <= 1e-12
    res07 = eval_detection_vid(pl, gl, 0.5, MOTION_RANGES, motion_specific=True, motion_ious=motions, use_07_metric=True,
                               device="cuda")
    host07 = eval_detection_vid(pl, gl, 0.5, MOTION_RANGES, motion_specific=True, motion_ious=motions, use_07_metric=True)
    for i in range(len(MOTION_RANGES)):
        _ap_close(res07[i]["ap"], host07[i]["ap"])


def test_golden_fixture_equals_the_stable_tie_restatement():
    from mega_core.data.datasets.evaluation.vid import calc_detection_vid_ap, calc_detection_vid_prec_rec
    cases = torch.load(os.path.join(ROOT, "tests", "golden", "vid_eval.pt"), weights_only=False)
    for case in cases:
        pl, gl = vr.boxlists([(im["boxes"], im["labels"], im["scores"]) for im in case["images"]],
                             [(im["gt"], im["gt_labels"]) for im in case["images"]])
        motions = [im["motion"] for im in case["images"]]
        for name, motion, rng in [("all", None, (0.0, 1.0))] + [(n, motions, r) for n, r in
                                                                 zip(("fast", "medium", "slow"), MOTION_RANGES)]:
            sp, sr = vr.prec_rec_stable(gl, pl, motion, 0.5, rng)
            dp, dr = calc_detection_vid_prec_rec(gl, pl, motion, 0.5, rng, device="cuda")
            if motion is None:
                _same_bits(dp, sp)
                _same_bits(dr, sr)
            else:
                _close(dp, sp)
                _close(dr, sr)
            ap = calc_detection_vid_ap(dp, dr)
            _ap_close(ap, calc_detection_vid_ap(sp, sr))
            print("golden seed %s %s: |AP - reference AP| max %.3e (tie order)" % (
                case["seed"], name, np.nanmax(np.abs(ap - case["reference"][name]["ap"]))))


def test_edge_cases():
    from mega_core.b200 import ops
    from mega_core.data.datasets.evaluation.vid import calc_detection_vid_ap, calc_detection_vid_prec_rec
    rs = np.random.RandomState(3)

    def boxes(k, scale=300):
        xy = rs.uniform(0, scale, (k, 2))
        return np.concatenate([xy, xy + rs.uniform(5, 80, (k, 2))], 1).astype(np.float32)

    gts = [(boxes(3), np.array([30, 2, 2])), (boxes(200), rs.randint(1, 21, 200)), (boxes(2), np.array([25, 25])),
           (boxes(0), np.zeros(0, int))]
    big = np.concatenate([gts[1][0][rs.randint(0, 200, 700)] + rs.normal(0, 2, (700, 4)).astype(np.float32),
                          boxes(900)])
    preds = [(np.concatenate([gts[0][0], boxes(4)]), np.array([30, 2, 2, 30, 30, 5, 9]),
              rs.uniform(0, 1, 7).astype(np.float32)),
             (big, rs.randint(1, 21, 1600), rs.uniform(0, 1, 1600).astype(np.float32)),     # > the shared-memory stage
             (np.zeros((0, 4), np.float32), np.zeros(0, int), np.zeros(0, np.float32)),     # class 25: GT, no detections
             (boxes(3), np.array([28, 28, 30]), rs.uniform(0, 1, 3).astype(np.float32))]   # class 28: no GT anywhere
    motions = [[0.3, 0.9, 1.0], list(rs.choice([0.3, 0.7, 0.8, 0.95], 200)), [0.65], []]
    pl, gl = vr.boxlists(preds, gts)
    for motion, rng in [(None, (0.0, 1.0))] + [(motions, r) for r in MOTION_RANGES]:
        sp, sr = vr.prec_rec_stable(gl, pl, motion, 0.5, rng)
        dp, dr = calc_detection_vid_prec_rec(gl, pl, motion, 0.5, rng, device="cuda")
        (_same_bits if motion is None else _close)(dp, sp)
        (_same_bits if motion is None else _close)(dr, sr)
        assert len(dp) == 31 and dp[25] is not None and len(dp[25]) == 0 and dp[28] is not None and dr[28] is None
        _ap_close(calc_detection_vid_ap(dp, dr), calc_detection_vid_ap(sp, sr))
    # no predictions at all: every class with GT scores AP 0
    empty = [(np.zeros((0, 4), np.float32), np.zeros(0, int), np.zeros(0, np.float32))] * len(gts)
    pl0, gl0 = vr.boxlists(empty, gts)
    sp, sr = vr.prec_rec_stable(gl0, pl0, None)
    dp, dr = calc_detection_vid_prec_rec(gl0, pl0, None, device="cuda")
    _same_bits(dp, sp)
    _same_bits(dr, sr)
    ap = calc_detection_vid_ap(dp, dr)
    assert np.array_equal(ap, calc_detection_vid_ap(sp, sr), equal_nan=True) and np.nanmax(ap) == 0.0
    assert ops.vid_eval(ops.vid_eval_pack(pl0, gl0, None), [(0.0, 1.0)], [0.0])["order"].numel() == 0


def test_two_calls_give_the_same_bits(tie_free):
    from mega_core.b200 import ops
    from mega_core.data.datasets.evaluation.vid.vid_eval import _empty_weight
    pl, gl, motions = tie_free
    packed = ops.vid_eval_pack(pl[:5000], gl[:5000], motions[:5000])
    emp = [_empty_weight(motions[:5000], r) for r in RANGES]
    a = ops.vid_eval(packed, RANGES, emp, want_prec_rec=True)
    b = ops.vid_eval(packed, RANGES, emp, want_prec_rec=True)
    for k in ("match", "ignore", "order", "n_pos", "ap", "prec", "rec", "det_count", "seen"):
        x, y = a[k].cpu(), b[k].cpu()
        assert torch.equal(x.view(torch.uint8) if x.is_floating_point() else x,
                           y.view(torch.uint8) if y.is_floating_point() else y), k


class _Dataset:
    def __init__(self, gl):
        self.gl = gl

    def get_img_info(self, i):
        return {"width": 640, "height": 360}

    def get_groundtruth(self, i):
        return self.gl[i]

    def map_class_id_to_class_name(self, i):
        return "class%02d" % i


def test_do_vid_evaluation_writes_the_same_result_txt(tie_free, tmp_path, monkeypatch):
    from mega_core.data.datasets.evaluation.vid import vid_eval
    pl, gl, motions = tie_free
    pl, gl = pl[:4000], gl[:4000]
    texts = []
    for dev in ("cpu", "cuda"):
        out = tmp_path / dev
        out.mkdir()
        monkeypatch.setenv("MEGA_B200_EVAL_DEVICE", dev)
        vid_eval.do_vid_evaluation(_Dataset(gl), pl, str(out), False, False, logging.getLogger("vid_eval_test"))
        texts.append((out / "result.txt").read_text())
    assert texts[0] == texts[1] and "AP50 | motion=   all" in texts[0]
