"""Times the VID evaluator's host path against its device path on a seeded synthetic set of ImageNet VID validation size
(176,126 images, 30 classes, up to 300 detections and 0-5 GT per image, motion IoUs drawn from the values of
tests/golden/vid_eval.pt), all four motion ranges, in one process, and checks that both give the same mAPs.

  host    eval_detection_vid(..., motion_specific=True) with the four ranges of do_vid_evaluation (perf_counter)
  pack    ops.vid_eval_pack: the BoxLists -> flat arrays (perf_counter; not part of the device time)
  device  CUDA events around H2D of the packed arrays + kernels + D2H of the per-class APs, one pass for all ranges
  loop    do_vid_evaluation's per-image prediction.resize / get_groundtruth loop, which stays on the host (ground truth
          from memory: parsing annotation files is not included)

Usage: python tools/vid_eval_timing.py [--images 176126] [--classes 30] [--max-dets 300] [--seed 0] [--repeat 5]
                                       [--json PATH]
Prints the card's name and power limit beside the numbers. Without a CUDA device it stops with an error where the device
path begins."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "mega.pytorch_b200"))

RANGES = [(0.0, 1.0), (0.0, 0.7), (0.7, 0.9), (0.9, 1.0)]


def _card():
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit or "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=176126)
    ap.add_argument("--classes", type=int, default=30)
    ap.add_argument("--max-dets", type=int, default=300)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--repeat", type=int, default=5)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()

    from mega_core.b200 import ops, synth
    from mega_core.data.datasets.evaluation.vid.vid_eval import _empty_weight, eval_detection_vid
    from mega_core.structures.bounding_box import BoxList

    golden = torch.load(os.path.join(ROOT, "tests", "golden", "vid_eval.pt"), weights_only=False)
    motion_values = np.unique(np.concatenate([np.asarray(im["motion"], dtype=np.float64)
                                              for case in golden for im in case["images"]]))
    t0 = time.perf_counter()
    preds, gts, motions = synth.vid_eval_set(args.images, args.seed, args.classes, args.max_dets,
                                             motion_values=tuple(motion_values.tolist()))
    pl, gl = [], []
    for (b, l, s), (gb, glab) in zip(preds, gts):
        p = BoxList(torch.from_numpy(b), (640, 360), mode="xyxy")
        p.add_field("labels", torch.from_numpy(l))
        p.add_field("scores", torch.from_numpy(s))
        g = BoxList(torch.from_numpy(gb), (640, 360), mode="xyxy")
        g.add_field("labels", torch.from_numpy(glab))
        pl.append(p)
        gl.append(g)
    n_det = sum(len(p) for p in pl)
    print("synthetic set: %d images, %d detections, %d GT, %d classes (%.1f s to make)" % (
        args.images, n_det, sum(len(g) for g in gl), args.classes, time.perf_counter() - t0), flush=True)

    t0 = time.perf_counter()
    for i, p in enumerate(pl):                      # do_vid_evaluation's per-image loop (ground truth from memory)
        p.resize((640, 360))
        gl[i]
    loop_s = time.perf_counter() - t0

    t0 = time.perf_counter()
    packed = ops.vid_eval_pack(pl, gl, motions)
    pack_s = time.perf_counter() - t0
    empties = [_empty_weight(motions, r) for r in RANGES]
    print("pack %.2f s, per-image resize / get_groundtruth loop %.2f s" % (pack_s, loop_s), flush=True)

    if not torch.cuda.is_available():
        raise SystemExit("vid_eval_timing: the device path needs a CUDA device (there is no fallback)")
    card, power = _card()
    packed = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in packed.items()}
    times = []
    for it in range(args.repeat + 1):               # the first pass warms up (module load, allocator)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = ops.vid_eval(packed, RANGES, empties)
        ap_dev = out["ap"].cpu().numpy()
        e1.record()
        torch.cuda.synchronize()
        if it:
            times.append(e0.elapsed_time(e1) / 1e3)
        del out
    dev_s = statistics.median(times)
    seen = ops.vid_eval(packed, RANGES, empties)["seen"].cpu().numpy().astype(bool)
    ap_dev[:, ~seen] = np.nan
    map_dev = [float(np.nanmean(a)) for a in ap_dev]
    print("device %.4f s (median of %d; min %.4f, max %.4f) on %s, power limit %s" % (
        dev_s, len(times), min(times), max(times), card, power), flush=True)

    t0 = time.perf_counter()
    res = eval_detection_vid(pl, gl, 0.5, RANGES, motion_specific=True, motion_ious=motions)
    host_s = time.perf_counter() - t0
    map_host = [float(res[i]["map"]) for i in range(len(RANGES))]
    diff = max(abs(a - b) for a, b in zip(map_dev, map_host))
    print("host %.1f s" % host_s)
    print("mAP host   " + " ".join("%.6f" % m for m in map_host))
    print("mAP device " + " ".join("%.6f" % m for m in map_dev))
    result = {"images": args.images, "detections": n_det, "classes": args.classes, "ranges": RANGES,
              "host_s": host_s, "device_s": dev_s, "device_s_all": times, "pack_s": pack_s, "resize_gt_loop_s": loop_s,
              "map_host": map_host, "map_device": map_dev, "max_map_diff": diff, "gpu": card, "power_limit": power}
    print(json.dumps(result))
    if args.json:
        with open(args.json, "w") as fh:
            json.dump(result, fh, indent=1)
    if diff > 1e-4:                                  # tied scores are ranked differently (module docstring of vid_eval)
        raise SystemExit("vid_eval_timing: host and device mAPs differ by %.3e" % diff)


if __name__ == "__main__":
    main()
