#!/usr/bin/env python
"""bench.py -- frames/sec of MEGA R-101 inference (1000x600) on B200, with parity, roofline and CPU baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--arch mega_r101|rdn_r101|fgfa_r101]
                    [--dump-outputs DIR]

A "step" of the default workload (configs[1] of BASELINE.json) is one pass of the MEGA R-101 hot path at 600x1000 in
steady state: the new look-ahead local frame and the new global frame of every key frame of the step go through
backbone -> RPN -> res5 -> ROIAlign -> l_fcs[0], then each key frame (position 12 of the 25-frame local window) is
aggregated against 25 local / 10 global / 25 memory frames and post-processed. `config.key_frames_per_step` says how
many key frames a step carries (--frames-per-step: the per-frame branch of n consecutive key frames runs as one batch of
2n images, the n aggregations in order; value counts key frames, not steps). Weights are the seeded synthetic
initialisation of mega_core.b200.synth (no checkpoints offline); frames are synthetic.

Arithmetic modes and the headline. The engine has a throughput mode ("f16": fp16 operands / fp32 accumulate) and a
strict mode ("fp32x3": every product as three tensor-core products on operands split hi + lo -- 22 mantissa bits -- with
round-to-nearest accumulator folds: near-fp32. Since round 2 the split operands are stored as fp16 pairs, DESIGN.md section 4). Both are timed in full at N = 1 and both are replayed over the
committed 600x1000 / 42-key-frame fixture of the UNMODIFIED reference (tests/golden/mega_r101_600x1000.pt) inside this
run: the `parity` block reports, per mode, the distance of the class logits from the reference's and whether the mode
meets the bar (PARITY_BAR below; the floor it sits on -- the reference's own fp32 vs fp64 vs other-thread-count
distances -- is profiles/r02_parity_floor.json). The top-level `value` / `e2e` / `roofline` belong to the FASTEST MODE
THAT MEETS THE BAR (`config.precision`); every measured mode is listed under `modes`.

Output: ONE JSON line (driver contract): `value` = key frames/s with inputs resident in HBM (CUDA events, max over ranks),
`e2e` = the same through the public model API with pinned-host inputs and a host read of the detections, `roofline` for
the tensor-core kernels, `cpu_baseline` = the reference path on this box's host cores on a bounded sample.

--dump-outputs DIR: after the timed steps, the detections the last device-resident step returned (what a caller of
that step receives) go to DIR as float32 .npy files, one set per timed mode and key frame of the step:
<precision>_frame<g>_{boxes,scores,labels}.npy. Inputs and weights are seeded, so the same arguments give the same
inputs on every run and two builds can be compared output for output.

N > 1 (torchrun): ONE video stream, frame-parallel (SURVEY.md section 8e): per step every rank runs the per-frame branch
of its own (local, global) frame pair, NCCL all-gathers exchange the fixed-size ROI-feature payloads (and, in the
wavefront schedule, the per-stage memory increments) in frame order; a step produces N key frames:
value = N * steps / max-over-ranks time. Per-GPU work per step is fixed -> "weak".
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "mega.pytorch_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

METRIC = "frames/sec MEGA R-101 inference (1000x600)"
H, W = 600, 1000
# algorithmic GFLOP per key frame, minimal exact form (SURVEY.md section 8a / 8d)
ALGO_GFLOP = {"mega_r101": 734.0,
              # RDN: 1 backbone + RPN head + 1 res5 + fcs[0] on 300 rows + attention (minimal form, section 8a row a18)
              "rdn_r101": 166.1 + 45.5 + 71.5 + 61.7 + 2 * 17.4 + 22.3 + 4.0 + 2 * 1.3,
              # FGFA: FlowNetS on 19 pairs + backbone + embednet + RPN head + res5 + fc6/fc7 (section 8a row a19)
              "fgfa_r101": 472.0 + 166.1 + 18.8 + 45.5 + 71.5 + 61.7 + 0.6}
FIXTURE = os.path.join(ROOT, "tests", "golden", "mega_r101_600x1000.pt")
# The bar a mode must meet on EVERY check frame of the fixture to carry the headline (DESIGN.md section 2): every proposal
# of the reference reproduced, the same number of detections, and the 99th percentile of |class logit - reference| within
# the north star's 1e-3. Why a percentile: two evaluations of the UNMODIFIED reference that differ only in rounding (fp32
# vs fp64, profiles/r02_parity_floor.json) agree to 8e-5 at the 99th percentile, but single logits move by up to 1.1e-2
# (a proposal pair crossing the relu gate of the position bias, roi_box_feature_extractors.py:593-633): on 2 of 42 key
# frames the reference is further than 1e-3 from itself, so "max <= 1e-3" is not a property any arithmetic can have.
PARITY_BAR = {"min_matched_frac": 1.0, "logits_p99": 1e-3, "frames_with_equal_det_count": "all"}
MODES = ("f16", "fp32x3")            # fastest first
PRECISION_DTYPE = {"f16": "f16 operands / f32 accumulate", "tf32": "tf32 operands / f32 accumulate",
                   "fp32x3": "f16 hi + f16 lo split operands, 3 products (near-f32) / f32 accumulate"}
KERNEL_NOTE = {"f16": "conv_chain_kernel + conv_gemm_kernel<.., kModeF16> (tcgen05 kind::f16, fp16 operands; same dense peak as "
                      "bf16): all tensor-core launches of the step",
               "tf32": "conv_gemm_kernel<.., kModeTf32> (tcgen05 kind::tf32; TF32 dense peak is half the bf16 figure)",
               "fp32x3": "conv_gemm_kernel<.., kModeF16x3> (3 tcgen05 kind::f16 MMAs per product on split-fp16 operands; the stem "
                         "runs kModeSplit3 = 3 kind::tf32 MMAs). The bf16 dense peak is the denominator of the ALGORITHMIC "
                         "FLOP/s, so frac <= 1/3 by construction"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--arch", default="mega_r101", choices=sorted(ALGO_GFLOP))
    ap.add_argument("--height", type=int, default=H)
    ap.add_argument("--width", type=int, default=W)
    ap.add_argument("--precision", default="auto", choices=["auto", "f16", "tf32", "fp32x3"],
                    help="auto: time f16 and fp32x3, replay the reference fixture through both, headline = fastest mode "
                         "that meets PARITY_BAR; a mode name: time (and check) that mode only")
    ap.add_argument("--no-parity", action="store_true", help="skip the in-run fixture replay")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--wave", action="store_true",
                    help="N > 1: force the wavefront schedule (MegaEngine.dist_step_wave) without the self-check")
    ap.add_argument("--no-wave", action="store_true",
                    help="N > 1: keep the replicated-state schedule (dist_step). Default: every rank replays "
                         "parallel.wave_selfcheck on its own GPU and the run uses the wavefront schedule only if ALL pass")
    ap.add_argument("--pipeline", type=int, default=-1, choices=[-1, 0, 1],
                    help="N = 1, frames-per-step > 1: overlap the aggregation of a batch of key frames with the per-frame branch of "
                         "the next batch (MegaEngine.stepn_pipelined / model.forward_frames(prefetch=)); -1 = the build's default")
    ap.add_argument("--frames-per-step", type=int, default=0, choices=[0, 1, 2, 3, 4, 5, 6, 7, 8],
                    help="N = 1: key frames per step (MegaEngine.stepn_batched); 0 = the default of the build (DEFAULT_FPS)")
    ap.add_argument("--prime", type=int, default=-1, help="untimed steady frames before timing (default: fill the memory)")
    ap.add_argument("--cpu-sample-frames", type=int, default=3)
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-roofline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the detections of the last timed step to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


def detection_arrays(prefix, dets):
    """{name: float32 array} of one step's detections (a Detections or a list of them, one per key frame)"""
    import numpy as np
    out = {}
    for g, det in enumerate(dets if isinstance(dets, list) else [dets]):
        for field, t in zip(("boxes", "scores", "labels"), det.to_host()):
            out["%s_frame%d_%s" % (prefix, g, field)] = t.numpy().astype(np.float32)
    return out


def dump_outputs(path, arrays):
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, a in sorted(arrays.items()):
        np.save(os.path.join(path, name + ".npy"), a)


DEFAULT_PIPELINE = 0   # --pipeline 1 (N = 1, strict mode): the aggregation of a batch overlaps the per-frame branch of the next one
                       # (stepn_pipelined): 214 -> 223 key frames/s. Off by default so that the N = 1 line runs the same schedule
                       # per GPU as the N > 1 lines (whose wavefront step is not pipelined) and the scaling figures compare like
                       # with like
DEFAULT_FPS = 4      # key frames per step at N = 1 (the per-frame branch of 4 key frames = one batch of 8 images)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"hbm_gbs": d["hbm_gbs"], "tflops": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "src": "MEASURED_PEAKS.json (bf16 dense sustained)"}
    return {"hbm_gbs": 6650.0, "tflops": 1400.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """samples nvidia-smi clocks / throttle reasons of ONE GPU during the timed regions. Started before the warm-up
    (nvidia-smi needs ~1 s to come up on an 8-GPU box; round 1 started 8 of them at the first timed step of an 8-rank
    run, got no sample and perturbed the region) and only on rank 0; `mark()` brackets the timed regions."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc, self.marks = index, [], None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def mark(self):
        self.marks.append(time.time())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        spans = list(zip(self.marks[0::2], self.marks[1::2]))
        rows = [r for (ts, r) in self.rows if len(r) >= 6 and any(a - 0.06 <= ts <= b + 0.06 for a, b in spans)]
        if not rows:                                  # regions shorter than the sampling period: nearest samples
            rows = [r for (_, r) in self.rows if len(r) >= 6][-4:]
        sm = sorted(float(r[0]) for r in rows if r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in rows for i in range(4) if r[2 + i] == "Active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx[0] if mx else None,
                "reasons": reasons, "samples": len(sm), "gpu_index": self.index}


def workload(args, fps=1):
    if args.arch == "mega_r101":
        return ("MEGA R-101 C4 steady-state key frame, %dx%d, 25 local / 10 global / 25 memory frames, "
                "1 new local + 1 new global frame per key frame" % (args.width, args.height))
    if args.arch == "rdn_r101":
        return "RDN R-101 C4 steady-state key frame, %dx%d, 37-frame window, 1 new frame per key frame" % (args.width, args.height)
    return "FGFA R-101 C4 steady-state key frame, %dx%d, 19-frame window (FlowNetS on 19 pairs), 1 new frame per key frame" % (
        args.width, args.height)


def frame_pool(n, h, w):
    from mega_core.b200 import synth
    return [synth.synthetic_frame(i, h, w) for i in range(n)]


def meets_bar(summary, n_check):
    if summary is None:
        return False
    return (summary["all_finite"] and summary["min_matched_frac"] >= PARITY_BAR["min_matched_frac"]
            and summary["logits_p99"] <= PARITY_BAR["logits_p99"] and summary["frames_with_equal_det_count"] == n_check)


# ------------------------------------------------------------------------------------------ B200 arm, MEGA
class MegaBench:
    """everything that is shared by the modes of one run: frames, state dict, fixture"""

    def __init__(self, args, rank, world):
        from mega_core.b200 import synth
        self.args, self.rank, self.world = args, rank, world
        self.dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
        torch.cuda.set_device(self.dev)
        self.h, self.w = args.height, args.width
        self.sd = synth.make_state_dict(args.arch, seed=0)
        pool = frame_pool(16, self.h, self.w)
        self.pool_pinned = [f.pin_memory() for f in pool]
        self.pool_dev = [f.to(self.dev) for f in pool]
        self.pairs_dev = [torch.cat([self.pool_dev[(i + 12) % 16], self.pool_dev[(5 * i + 3) % 16]], 0) for i in range(16)]
        self.pairs_pinned = [torch.cat([pool[(i + 12) % 16], pool[(5 * i + 3) % 16]], 0).pin_memory() for i in range(16)]
        self.fps = args.frames_per_step or DEFAULT_FPS      # N > 1: per rank (wavefront schedule), see measure()
        self.gold = None
        if not args.no_parity and os.path.exists(FIXTURE) and (self.h, self.w) == (H, W):
            self.gold = torch.load(FIXTURE)
        self.gold_frames = None
        self.sampler = None

    def infos_first(self):
        pp = self.pool_pinned
        return {"cur": pp[0], "ref_l": [], "ref_g": [pp[(3 * j + 1) % 16] for j in range(10)],
                "frame_category": 0, "seg_len": 10 ** 6, "pattern": "%06d", "img_dir": "%s",
                "lookahead": [pp[(j + 1) % 16] for j in range(12)]}

    def infos_next(self, t):
        pp = self.pool_pinned
        return {"cur": pp[t % 16], "ref_l": [pp[(t + 12) % 16]], "ref_g": [pp[(5 * t + 3) % 16]],
                "frame_category": 1, "seg_len": 10 ** 6, "pattern": "%06d", "img_dir": "%s"}

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize(self.dev)

    def parity(self, eng):
        """replay the reference fixture through `eng` (its per-video state is reset by start_video)"""
        if self.gold is None:
            return None
        from mega_core.b200 import parity, synth
        if self.gold_frames is None:
            g = self.gold
            self.gold_frames = [synth.synthetic_frame(i, g["h"], g["w"]).to(self.dev) for i in range(g["total"])]
        graphs, eng._graphs = eng._graphs, {}
        flag, eng.use_graph = eng.use_graph, False
        try:
            with torch.no_grad():
                rows = parity.replay(eng, self.gold, self.dev, frames=self.gold_frames)
        finally:
            eng._graphs, eng.use_graph = graphs, flag
        s = parity.summarize(rows)
        s["meets_bar"] = meets_bar(s, len(rows))
        s["key_frames_replayed"] = len(self.gold["frames"])
        return s

    def measure(self, precision, timed=True):
        """build the model in `precision`, prime it, time the device-resident and the end-to-end regions"""
        import torch.distributed as dist
        from mega_core.b200 import engine, ops
        from mega_core.modeling.detector import build_detection_model_from_state_dict
        args, rank, world, dev, h, w, fps = self.args, self.rank, self.world, self.dev, self.h, self.w, self.fps
        model = build_detection_model_from_state_dict(self.sd, method="mega", device=dev, precision=precision)
        eng = model.engine
        eng.use_graph = not args.no_graph
        res = {"precision": precision, "model": model, "eng": eng}
        if not timed:
            return res
        pairs_dev, pairs_pinned = self.pairs_dev, self.pairs_pinned
        # ---- prime: first frame of the video, then fill the long-range memory (25 key frames)
        t = 1
        with torch.no_grad():
            model(self.infos_first())
            n_prime = eng.MEMF + 2 if args.prime < 0 else args.prime
            if world == 1:
                for _ in range(n_prime):
                    model(self.infos_next(t))
                    t += 1
            else:
                for i in range(-(-n_prime // world)):
                    eng.dist_step(pairs_dev[(i * world + rank) % 16], w, h)
        torch.cuda.synchronize(dev)

        wave = world > 1 and (args.wave or os.environ.get("MEGA_B200_WAVE", "0") == "1")
        wave_note = "forced" if wave else None
        if world > 1 and not wave and not args.no_wave:
            # each rank proves the wavefront schedule on its own device first (no communication inside the check, one MIN
            # all-reduce of the verdicts after it)
            from mega_core.b200 import parallel
            ok, wave_note = False, ""
            try:
                with torch.no_grad():
                    ok, wave_note = parallel.wave_selfcheck(lambda: engine.MegaEngine(self.sd, eng.cfg, dev), w, h, world=2,
                                                            groups=3, use_graph=not args.no_graph)
            except Exception as e:                      # any surprise keeps the proven schedule
                ok, wave_note = False, "self-check raised %s: %s" % (type(e).__name__, str(e)[:200])
            verdict = torch.tensor([1 if ok else 0], device=dev, dtype=torch.int32)
            dist.all_reduce(verdict, op=dist.ReduceOp.MIN)
            wave = int(verdict.item()) == 1
            if not wave and ok:
                wave_note = "another rank failed the self-check"
            torch.cuda.empty_cache()

        if world > 1 and not wave:
            fps = 1          # the replicated-state fallback schedule runs one key frame per rank and step

        def dstep(pair):
            return eng.dist_step_wave(pair, w, h) if wave else eng.dist_step(pair, w, h)[rank]

        def pair_index(i, g):
            """pool index of the frame pair of step i, round g on this rank (key frame (i * fps + g) * world + rank)"""
            return ((i * fps + g) * world + rank) % 16

        batches = {}

        def batch_dev(i):
            key = tuple(pair_index(i, g) for g in range(fps))
            if key not in batches:
                batches[key] = torch.cat([pairs_dev[k] for k in key], 0) if fps > 1 else pairs_dev[key[0]]
            return batches[key]

        def step_dev(i):
            if world > 1 and fps == 1:
                return dstep(pairs_dev[pair_index(i, 0)])
            batch = batch_dev(i)
            if world > 1:
                return eng.dist_stepn_wave(batch, w, h)
            if fps > 1 and pipelined:
                return eng.stepn_pipelined(batch_dev(i + 1), w, h)      # aggregates batch i, starts the branch of batch i + 1
            if fps > 1:
                return eng.stepn_batched(batch, w, h)
            return eng.step_batched(batch, w, h)

        # (default: the strict mode only -- the fp16 mode's chain kernels must run on capped, disjoint SM budgets side by side,
        #  which measured slower than the sequential step: 252 vs 383 key frames/s)
        pipelined = world == 1 and fps > 1 and (args.pipeline == 1 or (args.pipeline < 0 and DEFAULT_PIPELINE and not eng.chained))
        res["pipelined"] = bool(pipelined)
        static_in = eng.static_input((2 * fps, 3, h, w))
        state = {"t": t}

        def step_e2e():
            """pinned host frames -> device, one step, detections of this rank's key frame(s) back on the host"""
            t0 = state["t"]
            if world == 1 and fps > 1:
                nxt = [self.infos_next(t0 + fps + j) for j in range(fps)] if pipelined else None
                outs = model.forward_frames([self.infos_next(t0 + j) for j in range(fps)], prefetch=nxt)
                state["t"] = t0 + fps
                return sum(len(o[0].to("cpu")) for o in outs)
            state["t"] = t0 + 1
            if world == 1:
                # the call a user of the reference makes, followed by the .to(cpu) of engine/inference.py:43
                return len(model(self.infos_next(t0))[0].to("cpu"))
            for g in range(fps):
                static_in[2 * g:2 * g + 2].copy_(pairs_pinned[pair_index(t0, g)], non_blocking=True)
            if fps == 1:
                return len(dstep(static_in).to_host()[0])
            return sum(len(d.to_host()[0]) for d in eng.dist_stepn_wave(static_in, w, h))

        with torch.no_grad():
            # ---- settle: every CUDA graph of the schedule captured AND replayed, every collective size seen, before the
            #      W warm-up steps (a graph key runs eagerly once, is captured on its second use and replays from the third)
            for i in range(4 if world > 1 or fps > 1 else 2):
                step_dev(i)
            launches0 = ops.LAUNCHES[0]
            for i in range(args.warmup):
                step_dev(i)
            launches_per_step = (ops.LAUNCHES[0] - launches0) / max(args.warmup, 1)
            if eng._graphs:
                launches_per_step = float(eng.launches_per_frame)
            # ---- timed region A: device-resident inputs, engine-level step (no host transfers)
            self.barrier()
            if self.sampler is not None:
                self.sampler.mark()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(args.steps):
                last = step_dev(i)
            e1.record()
            self.barrier()
            if self.sampler is not None:
                self.sampler.mark()
            dev_ms = e0.elapsed_time(e1)
            if args.dump_outputs:          # read before the next step overwrites the engine's static detection buffers
                res["outputs"] = detection_arrays(precision, last)
            # ---- timed region B: end to end: pinned host inputs -> detections on the host (the public model API at N=1)
            for i in range(max(args.warmup, 3)):
                step_e2e()
            self.barrier()
            if self.sampler is not None:
                self.sampler.mark()
            e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e2.record()
            ndet = 0
            for i in range(args.steps):
                ndet += step_e2e()
            e3.record()
            self.barrier()
            if self.sampler is not None:
                self.sampler.mark()
            e2e_ms = e2.elapsed_time(e3)
            # ---- N > 1: where a step's time goes on this rank (instrumented pass, not part of the timed regions)
            comm = None
            if world > 1:
                from mega_core.b200 import parallel
                rec = []
                parallel.COMM_EVENTS[0] = rec
                s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s0.record()
                for i in range(6):
                    step_dev(i)
                s1.record()
                torch.cuda.synchronize(dev)
                parallel.COMM_EVENTS[0] = None
                comm = {"collectives_per_step": len(rec) / 6.0,
                        "collective_ms_per_step": sum(a.elapsed_time(b) for a, b in rec) / 6.0,
                        "step_ms_instrumented": s0.elapsed_time(s1) / 6.0}
        # ---- N > 1: the hand-off that follows the path in tools/test_net.py (engine/inference.py:50-69): every rank's
        #      detections of its last key frames to rank 0 through mega_core.utils.comm.gather_predictions over NCCL,
        #      checked on rank 0 against the count every rank reports (SURVEY section 8f row 2; outside the timed regions)
        handoff = None
        if world > 1:
            from mega_core.structures.bounding_box import BoxList
            from mega_core.utils import comm as comm_utils
            with torch.no_grad():
                dets = step_dev(0)
            dets = dets if isinstance(dets, list) else [dets]
            preds, mine = {}, 0
            for g, det in enumerate(dets):
                b, sc, lb = det.to_host()
                bl = BoxList(b, (w, h), mode="xyxy")
                bl.add_field("scores", sc)
                bl.add_field("labels", lb)
                preds[g * world + rank] = bl
                mine += len(bl)
            t0 = time.time()
            merged = comm_utils.gather_predictions(preds)
            dt = time.time() - t0
            tot = torch.tensor([mine], device=dev, dtype=torch.int64)
            dist.all_reduce(tot)
            if rank == 0:
                handoff = {"images": len(merged), "detections": int(sum(len(m) for m in merged)),
                           "expected_images": world * len(dets), "expected_detections": int(tot.item()),
                           "ok": len(merged) == world * len(dets) and sum(len(m) for m in merged) == int(tot.item()),
                           "backend": dist.get_backend(), "seconds": round(dt, 4)}
        h2d = fps * 2 * 3 * h * w * 4 + eng.tab_h.numel() * 4 * world * fps
        d2h = (model.d2h_bytes_per_frame if world == 1 else 4 + 300 * 28) * fps
        times = torch.tensor([dev_ms, e2e_ms, comm["collective_ms_per_step"] if comm else 0.0,
                              comm["step_ms_instrumented"] if comm else 0.0], device=dev, dtype=torch.float64)
        per_rank = None
        if world > 1:
            allt = [torch.zeros_like(times) for _ in range(world)]
            dist.all_gather(allt, times)
            per_rank = {"device_ms_per_step": [round(x[0].item() / args.steps, 4) for x in allt],
                        "e2e_ms_per_step": [round(x[1].item() / args.steps, 4) for x in allt],
                        "collective_ms_per_step": [round(x[2].item(), 4) for x in allt],
                        "instrumented_step_ms": [round(x[3].item(), 4) for x in allt]}
            dist.all_reduce(times, op=dist.ReduceOp.MAX)
        dev_ms, e2e_ms = times[0].item(), times[1].item()
        kf = world * fps
        res.update({"fps": fps, "dev_ms": dev_ms, "e2e_ms": e2e_ms, "value": kf * args.steps / (dev_ms * 1e-3),
                    "e2e_value": kf * args.steps / (e2e_ms * 1e-3), "ms_per_step": dev_ms / args.steps,
                    "launches_per_step": launches_per_step, "h2d": h2d, "d2h": d2h,
                    "detections_per_frame": ndet / float(args.steps * fps), "wave": wave, "wave_note": wave_note,
                    "per_rank": per_rank, "comm": comm, "cuda_graph": bool(eng._graphs), "handoff": handoff})
        return res


def roofline_pass(eng, step, reps=3):
    """sum of the tensor-core kernel durations of one step (CUDA events on the launching stream, eager launches)"""
    from mega_core.b200 import ops
    has_graphs = hasattr(eng, "_graphs")         # the windowed engines replay CUDA graphs; FGFA / DFF / base launch eagerly
    if has_graphs:
        saved_graphs, eng._graphs = eng._graphs, {}
        saved_flag, eng.use_graph = eng.use_graph, False
    rec = []

    def hook(run, flops, info):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        run()
        b.record()
        rec.append((a, b, flops, info))

    ops.TIMING_HOOK[0] = hook
    try:
        with torch.no_grad():
            step(0)   # warm
            rec.clear()
            for i in range(reps):
                # park the GPU behind a ~15 ms spin so the whole step is queued before it starts executing:
                # the event pairs then bracket kernel execution only, not host launch latency
                torch.cuda._sleep(30_000_000)
                step(i + 1)
                torch.cuda.synchronize()
    finally:
        ops.TIMING_HOOK[0] = None
        if has_graphs:
            eng._graphs, eng.use_graph = saved_graphs, saved_flag
    ms = sum(r[0].elapsed_time(r[1]) for r in rec) / reps
    fl = sum(r[2] for r in rec) / reps
    n = max(len(rec) // reps, 1)
    # the dominant launch = the one with the largest share of the step's tensor-core time
    dom, best = None, -1.0
    for i in range(n):
        t = sum(q[0].elapsed_time(q[1]) for q in rec[i::n]) / reps
        if t > best:
            r = rec[i]
            info = r[3] if isinstance(r[3], dict) else {}
            name = ("conv_chain_kernel (%d layers, grid %d)" % (info["chain_layers"], info["grid"]) if "chain_layers" in info
                    else "conv_gemm_kernel (m %s, cout %s, k %s x %s taps, block_n %s)" % (
                        info.get("m"), info.get("cout"), info.get("k"), info.get("taps"), info.get("bn")))
            dom, best = {"name": name, "executed_gflop": r[2] / 1e9, "ms": t,
                         "executed_tflops": r[2] / (t * 1e-3) / 1e12}, t
    return {"kernel_ms": ms, "exec_gflop": fl / 1e9, "exec_tflops": fl / (ms * 1e-3) / 1e12, "launches": len(rec) / reps,
            "dominant": dom}


def traffic_bytes(precision):
    """DRAM bytes per launch of the dominant kernel of `precision` from the committed ncu capture (null when that mode's
    dominant kernel has no capture): profiles/r02_traffic.json = {"<precision>": {"traffic_bytes_per_launch": ..,
    "kernel": .., "capture": ..}}"""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json"))).get(precision)
        if d:
            return d["traffic_bytes_per_launch"], "profiles/r02_traffic.json: %s, %s" % (d.get("kernel"), d.get("capture"))
    except Exception:
        pass
    return None, None


def roofline_block(args, roof, step_ms, key_frames_per_step, precision):
    pk = peaks()
    algo_tflops = ALGO_GFLOP[args.arch] * key_frames_per_step * 1e9 / (roof["kernel_ms"] * 1e-3) / 1e12
    traffic, tname = traffic_bytes(precision)
    return {"bound": "tensor", "achieved": algo_tflops, "peak": pk["tflops"], "unit": "TFLOP/s",
            "frac": algo_tflops / pk["tflops"], "traffic": traffic, "peak_source": pk["src"],
            "traffic_note": ("dram__bytes_read.sum + dram__bytes_write.sum per launch, one ncu --set full capture (%s)" % tname)
                            if tname else "no ncu --set full capture of this mode's dominant kernel is committed",
            "dominant_kernel": roof["dominant"], "kernel": KERNEL_NOTE.get(precision),
            "algorithmic_gflop_per_key_frame": ALGO_GFLOP[args.arch],
            "executed_gflop_per_step": roof["exec_gflop"], "kernel_ms_per_step": roof["kernel_ms"],
            "launches_per_step": roof["launches"], "executed_tflops": roof["exec_tflops"],
            "kernel_share_of_step": roof["kernel_ms"] / step_ms if step_ms else None,
            "whole_step": {"achieved": ALGO_GFLOP[args.arch] * key_frames_per_step / step_ms,     # GFLOP / ms = TFLOP/s
                           "frac": ALGO_GFLOP[args.arch] * key_frames_per_step / step_ms / pk["tflops"],
                           "note": "algorithmic GFLOP of the step / device-timed ms_per_step (everything included)"}
            if step_ms else None}


def run_mega(args, rank, world):
    mb = MegaBench(args, rank, world)
    if rank == 0:
        mb.sampler = ClockSampler(mb.dev.index or 0)
        mb.sampler.start()
    modes = list(MODES) if args.precision == "auto" else [args.precision]
    results, parity = {}, {}
    for p in modes:
        r = mb.measure(p)
        results[p] = r
        parity[p] = mb.parity(r["eng"]) if (rank == 0 or world == 1) else None
    # headline: the fastest mode that meets the bar (rank 0 decides; N > 1 broadcasts the decision)
    passing = [p for p in modes if parity[p] is not None and parity[p]["meets_bar"]]
    if mb.gold is None:
        head, why = modes[0], "no fixture replay in this run (parity unchecked)"
    elif passing:
        head = max(passing, key=lambda p: results[p]["value"])
        why = "fastest measured mode that meets PARITY_BAR on every check frame of the fixture"
    else:
        head = max(modes, key=lambda p: results[p]["value"])
        why = "NO measured mode meets PARITY_BAR: the fastest mode is printed, parity unqualified"
    if world > 1:
        import torch.distributed as dist
        idx = torch.tensor([modes.index(head)], device=mb.dev, dtype=torch.int32)
        dist.broadcast(idx, src=0)
        head = modes[int(idx.item())]
    R = results[head]
    eng, fps, kf = R["eng"], R["fps"], world * R["fps"]
    clocks = mb.sampler.stop() if mb.sampler is not None else None
    # ---- roofline of the tensor-core kernels: eager steps with an event pair per launch (rank 0)
    roofs = {}
    if rank == 0 and not args.skip_roofline:
        for p in modes:
            e = results[p]["eng"]
            if fps > 1:
                nb = 16 // fps
                md = [torch.cat([mb.pairs_dev[(fps * i + j) % 16] for j in range(fps)], 0) for i in range(nb)]
                roofs[p] = roofline_pass(e, lambda i, e=e, md=md, nb=nb: e.stepn_batched(md[i % nb], mb.w, mb.h))
            else:
                roofs[p] = roofline_pass(e, lambda i, e=e: e.step_batched(mb.pairs_dev[i % 16], mb.w, mb.h))
    if rank != 0:
        return None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: v for p in modes for k, v in results[p]["outputs"].items()})
    kf_step_roof = fps                      # the roofline pass runs the single-GPU step
    line = {
        "metric": METRIC, "value": R["value"], "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": R["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": PRECISION_DTYPE[head], "data": "synthetic",
        "config": {"workload": workload(args, fps), "arch": args.arch,
                   "weights": "seeded synthetic init (mega_core.b200.synth)",
                   "parallelism": ("frame-parallel over %d GPUs: per-frame branch on the frame's owner, NCCL all-gather of "
                                   "ROI-feature payloads, memory-feeding rows of the aggregation replicated, key-frame "
                                   "rows / predictor / post-processing on the owner" % world) if world > 1 and not R["wave"] else
                                  ("frame-parallel over %d GPUs, wavefront schedule: per-frame branch and the whole aggregation "
                                   "of a key frame on its owner, NCCL all-gather of the ROI-feature payloads + one all-gather of "
                                   "the memory increments per relation stage" % world) if R["wave"] else "single GPU",
                   "key_frames_per_step": kf,
                   "pipelined": ("aggregation of batch i concurrently with the per-frame branch of batch i + 1 (two streams, "
                                 "MegaEngine.stepn_pipelined; SM caps branch / aggregation: %s)" % (list(R["eng"].PIPE_SMS),))
                                if R.get("pipelined") else False,
                   "schedule": ("wavefront" if R["wave"] else "replicated-state") if world > 1 else None,
                   "wave_selfcheck": R["wave_note"], "cuda_graph": R["cuda_graph"], "precision": head,
                   "headline_rule": why,
                   "l2": "per-step working set (>= 0.35 GB fp16 weights + > 0.5 GB activations) exceeds the 126 MB L2; no flush"},
        "clocks": clocks,
        "e2e": {"value": R["e2e_value"], "unit": "frames/s", "h2d_bytes_per_step": R["h2d"], "d2h_bytes_per_step": R["d2h"],
                "ms_per_step": R["e2e_ms"] / args.steps, "detections_per_frame": R["detections_per_frame"],
                "api": "model(images) per key frame" if fps == 1 and world == 1 else
                       ("model.forward_frames([images] * %d%s)" % (fps, ", prefetch=next" if R.get("pipelined") else "") if world == 1 else
                        "MegaEngine.dist_step%s (one video stream)" % ("n_wave" if R["fps"] > 1 else "_wave" if R["wave"] else ""))},
        "gpu_launches": int(round(R["launches_per_step"] * args.steps)),
        "parity": {"fixture": "tests/golden/mega_r101_600x1000.pt (unmodified reference, %s key frames)" % (
                       len(mb.gold["frames"]) if mb.gold else "n/a"),
                   "bar": PARITY_BAR, "floor": "profiles/r02_parity_floor.json",
                   "modes": {p: parity[p] for p in modes}},
        "modes": {p: {"value": results[p]["value"], "ms_per_step": results[p]["ms_per_step"],
                      "e2e": results[p]["e2e_value"], "meets_parity_bar": bool(parity[p] and parity[p]["meets_bar"]),
                      "roofline_frac": (roofline_block(args, roofs[p], None, kf_step_roof, p)["frac"] if p in roofs else None)}
                  for p in modes},
    }
    if head in roofs:
        line["roofline"] = roofline_block(args, roofs[head], R["ms_per_step"] if world == 1 else None, kf_step_roof, head)
        if world > 1:
            line["roofline"]["note"] = "kernel timing pass = the single-GPU step of rank 0 (the per-GPU kernels are the same at any N)"
    if R["per_rank"] is not None:
        line["per_rank"] = R["per_rank"]
        line["comm"] = R["comm"]
        line["prediction_handoff"] = R["handoff"]
    return line


# ------------------------------------------------------------------------------------------ B200 arm, RDN / FGFA (N = 1)
def run_windowed(args, rank, world):
    """BASELINE configs[3] / configs[4]: one new frame per key frame; replicas only at N > 1 (no exchange step)"""
    from mega_core.b200 import ops, synth
    from mega_core.modeling.detector import build_detection_model_from_state_dict
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(dev)
    h, w = args.height, args.width
    method = args.arch.split("_")[0]
    precision = "f16" if args.precision == "auto" else args.precision
    sd = synth.make_state_dict(args.arch, seed={"rdn": 4, "fgfa": 5}[method])
    model = build_detection_model_from_state_dict(sd, method=method, device=dev, precision=precision)
    eng = model.engine
    if hasattr(eng, "use_graph"):
        eng.use_graph = not args.no_graph
    pool = frame_pool(16, h, w)
    pinned = [f.pin_memory() for f in pool]
    pdev = [f.to(dev) for f in pool]
    look = eng.L - eng.cfg.key_frame_location - 1
    sampler = ClockSampler(dev.index or 0) if rank == 0 else None
    if sampler:
        sampler.start()

    def infos(t, first=False):
        d = {"cur": pinned[t % 16], "ref": [] if first else [pinned[(t + look) % 16]], "frame_category": 0 if first else 1,
             "seg_len": 10 ** 6, "pattern": "%06d", "img_dir": "%s"}
        if first:
            d["lookahead"] = [pinned[(j + 1) % 16] for j in range(look)]
        return d

    with torch.no_grad():
        model(infos(0, True))
        t = 1
        for _ in range(3):
            model(infos(t))
            t += 1
        l0 = ops.LAUNCHES[0]
        for i in range(args.warmup):
            eng.step(pdev[i % 16], w, h)
        lps = (ops.LAUNCHES[0] - l0) / max(args.warmup, 1)
        torch.cuda.synchronize(dev)
        if sampler:
            sampler.mark()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(args.steps):
            last = eng.step(pdev[i % 16], w, h)
        e1.record()
        torch.cuda.synchronize(dev)
        dev_ms = e0.elapsed_time(e1)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, detection_arrays(precision, last))
        for i in range(3):
            model(infos(t))[0].to("cpu")
            t += 1
        torch.cuda.synchronize(dev)
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e2.record()
        ndet = 0
        for i in range(args.steps):
            ndet += len(model(infos(t))[0].to("cpu"))
            t += 1
        e3.record()
        torch.cuda.synchronize(dev)
        e2e_ms = e2.elapsed_time(e3)
        if sampler:
            sampler.mark()
    clocks = sampler.stop() if sampler else None
    roof = None if args.skip_roofline else roofline_pass(eng, lambda i: eng.step(pdev[i % 16], w, h))
    if rank != 0:
        return None
    line = {"metric": METRIC.replace("MEGA", method.upper()), "value": args.steps / (dev_ms * 1e-3), "unit": "frames/s",
            "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": PRECISION_DTYPE[precision],
            "data": "synthetic",
            "config": {"workload": workload(args), "arch": args.arch, "weights": "seeded synthetic init (mega_core.b200.synth)",
                       "parallelism": "single GPU", "key_frames_per_step": 1, "cuda_graph": bool(getattr(eng, "_graphs", None)),
                       "precision": precision, "l2": "per-step working set exceeds the 126 MB L2; no flush"},
            "clocks": clocks,
            "e2e": {"value": args.steps / (e2e_ms * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": 3 * h * w * 4,
                    "d2h_bytes_per_step": model.d2h_bytes_per_frame, "ms_per_step": e2e_ms / args.steps,
                    "detections_per_frame": ndet / float(args.steps), "api": "model(images) per key frame"},
            "gpu_launches": int(round((eng.launches_per_frame if getattr(eng, "_graphs", None) else lps) * args.steps)),
            "parity": {"note": "tests/test_engine_gpu.py replays the reference's 192x320 %s fixture through this engine in the "
                               "exact-fp32 shadow / fp32x3 / f16 modes; no full-size fixture for this arch" % method.upper()}}
    if roof is not None:
        line["roofline"] = roofline_block(args, roof, dev_ms / args.steps, 1, precision)
    return line


# ------------------------------------------------------------------------------------------ CPU arm
def host_threads():
    """the fixed thread policy of both CPU legs: one thread per physical core, at most 32 (one NUMA node of the pool's
    2 x 32-core hosts: torch's intra-op pool does not scale across the socket boundary on convolutions of this size)"""
    logical = os.cpu_count() or 1
    physical = logical
    try:
        import psutil
        physical = psutil.cpu_count(logical=False) or logical
    except Exception:
        physical = max(logical // 2, 1)
    return min(physical, 32), physical, logical


def cpu_frames(args, warm, timed):
    """`warm` + `timed` steady-state frames of the hot path on the host cores -> the cpu_baseline block.
    MEGA: the unmodified reference's model when /root/reference is importable (this container), else the oracle port
    (oracle/mega_oracle.py -- pinned bit-for-bit to the reference, oracle/make_golden.py). The 25-frame window, the global
    pool and the long-range memory are pre-filled with synthetic rows (building them for real costs 23 backbone passes);
    every timed frame runs 2 backbone / RPN / res5 / ROIAlign / FC passes + the full 25 / 10 / 25 aggregation."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import mega_oracle as mo
    from collections import deque
    from mega_core.b200 import synth
    nt, physical, logical = host_threads()
    torch.set_num_threads(nt)
    h, w = args.height, args.width
    method = args.arch.split("_")[0]
    sd = synth.make_state_dict(args.arch, seed={"mega": 0, "rdn": 4, "fgfa": 5}[method])
    pool = frame_pool(4, h, w)
    g = torch.Generator().manual_seed(1)
    kind = "port"
    if method == "mega":
        orc = mo.MegaOracle(sd)
        c = orc.cfg
        L, R, A = c.all_frame_interval, c.ref_post_nms_top_n, c.advanced_num

        def boxes(n):
            xy = torch.rand(n, 2, generator=g) * torch.tensor([w * 0.8, h * 0.8])
            return torch.cat([xy, xy + torch.rand(n, 2, generator=g) * 150 + 8], 1)

        fh, fw = (h - 1) // 16 + 1, (w - 1) // 16 + 1
        orc.q_feats = deque([torch.randn(1, 1024, fh, fw, generator=g).relu() for _ in range(L)], maxlen=L)
        orc.q_boxes = deque([boxes(R) for _ in range(L)], maxlen=L)
        orc.q_boxes_dis = deque([b[:A] for b in orc.q_boxes], maxlen=L)
        orc.q_pfeat = deque([torch.randn(R, 1024, generator=g).relu() * 0.3 for _ in range(L)], maxlen=L)
        orc.q_pfeat_dis = deque([p[:A] for p in orc.q_pfeat], maxlen=L)
        orc.mem_q = []
        for i in range(c.stage):
            n = R if i == 0 else A
            orc.mem_q.append({"rois": deque([boxes(n) for _ in range(L)], maxlen=L),
                              "feats": deque([torch.randn(n, 1024, generator=g).relu() * 0.3 for _ in range(L)], maxlen=L)})
        orc.mem = [{"rois": torch.cat(list(q["rois"])), "feats": torch.cat(list(q["feats"]))} for q in orc.mem_q]
        orc.global_q = deque([torch.randn(R, 1024, generator=g).relu() * 0.3 for _ in range(c.global_size)], maxlen=c.global_size)

        def frame(i):
            orc.forward(pool[i % 4], {"frame_category": 1, "ref_l": [pool[(i + 1) % 4]], "ref_g": [pool[(i + 2) % 4]]})
        what = "2 backbone passes + full 25/10/25 aggregation each; window/global/memory pre-filled with synthetic rows"
    else:
        orc = (mo.RdnOracle if method == "rdn" else mo.FgfaOracle)(sd)
        look = 18 if method == "rdn" else 9
        with torch.no_grad():
            orc.forward(pool[0], {"frame_category": 0, "ref": [pool[(j + 1) % 4] for j in range(look)]})

        def frame(i):
            orc.forward(pool[i % 4], {"frame_category": 1, "ref": [pool[(i + 1) % 4]]})
        what = "1 new frame per key frame after a real first frame (window filled by %d look-ahead frames)" % look
    with torch.no_grad():
        for i in range(warm):
            frame(i)
        t0 = time.time()
        for i in range(timed):
            frame(warm + i)
        dt = time.time() - t0
    return {"value": timed / dt, "unit": "frames/s", "cores": nt, "host_physical_cores": physical, "host_logical_cores": logical,
            "kind": kind,
            "sample": "%d timed (+%d untimed) steady-state %s R-101 frames at %dx%d (%s); oracle/mega_oracle.py (CPU port "
                      "pinned bit-for-bit to the unmodified reference, whose Python cannot travel to the GPU box), torch fp32, "
                      "%d threads = min(physical cores, 32)" % (timed, warm, method.upper(), w, h, what, nt),
            "seconds": dt, "frames_timed": timed}


def run_reference(args, rank, world):
    """`--impl reference`: the reference path on the host cores. EXACTLY `steps` frames are timed after `warmup` untimed
    ones, each a full steady-state frame of the workload (~5 s on 32 threads: 25 frames ~ 2 min)."""
    if rank != 0:
        return None
    base = cpu_frames(args, args.warmup, args.steps)
    v = base["value"]
    return {"impl": "reference", "metric": METRIC if args.arch == "mega_r101" else METRIC.replace("MEGA", args.arch.split("_")[0].upper()),
            "value": v, "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 / v, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload(args), "arch": args.arch,
                       "weights": "seeded synthetic init (mega_core.b200.synth)", "key_frames_per_step": 1,
                       "implementation": "CPU port of the reference path (oracle/mega_oracle.py), %d timed frames on %d threads"
                                         % (args.steps, base["cores"])},
            "cpu_baseline": base,
            "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}


def main():
    args = parse()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        line = run_reference(args, rank, world)
        if line is not None:
            print(json.dumps(line))
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
        dist.init_process_group("nccl")
    if args.arch == "mega_r101":
        line = run_mega(args, rank, world)
    elif world == 1 or rank == 0:
        line = run_windowed(args, rank, 1)
    else:
        line = None
    if rank == 0:
        if not args.skip_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_frames(args, 1, args.cpu_sample_frames)
        elif world == 1:
            line["cpu_baseline"] = None
        print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
