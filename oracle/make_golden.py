"""Generate tests/golden/*.pt by running the UNMODIFIED reference in this container, and check the
oracle restatement (oracle/mega_oracle.py, oracle/csrc/oracle_ops.c) against it on the way.

Run here (needs /root/reference):   python oracle/make_golden.py
The fixtures are small (inputs are regenerated from seeds; only outputs are stored) and are
what the GPU-side tests and the CPU oracle tests compare against on a box without the
reference.
"""
import importlib.util
import json
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
GOLD = os.path.join(ROOT, "tests", "golden")

import ref_import  # noqa: E402
import mega_oracle as mo  # noqa: E402


def load_synth():
    spec = importlib.util.spec_from_file_location(
        "mega_synth", os.path.join(ROOT, "mega.pytorch_b200", "mega_core", "b200", "synth.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


synth = load_synth()


def close(a, b, tol, what):
    a, b = a.double(), b.double()
    err = (a - b).abs().max().item() if a.numel() else 0.0
    scale = max(b.abs().max().item() if b.numel() else 0.0, 1e-12)
    print("  %-38s max|diff| %.3e (rel %.2e)" % (what, err, err / scale))
    assert err <= tol * max(scale, 1.0), (what, err)


# ------------------------------------------------------------------ 1. reference unit-test vectors
def golden_from_reference_tests():
    """replays the reference's tests/test_nms.py and tests/test_box_coder.py with recording wrappers"""
    pkg = ref_import.setup()
    import mega_core.layers as layers
    rec = {"nms": [], "decode": []}
    ref_nms = layers.nms

    def rec_nms(boxes, scores, thresh):
        keep = ref_nms(boxes, scores, thresh)
        rec["nms"].append({"boxes": boxes.clone(), "scores": scores.clone(), "thresh": float(thresh),
                           "keep": keep.clone()})
        return keep

    layers.nms = rec_nms
    spec = importlib.util.spec_from_file_location("ref_test_nms", os.path.join(ref_import.REFERENCE, "tests/test_nms.py"))
    tm = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tm)
    tm.box_nms = rec_nms
    import unittest
    expected = []
    orig_eq = np.testing.assert_array_equal

    def cap_eq(a, b, *k, **kw):
        expected.append(np.asarray(b).copy())
        return orig_eq(a, b, *k, **kw)

    np.testing.assert_array_equal = cap_eq
    res = unittest.TextTestRunner(verbosity=0).run(unittest.defaultTestLoader.loadTestsFromModule(tm))
    np.testing.assert_array_equal = orig_eq
    layers.nms = ref_nms
    assert res.wasSuccessful(), "reference tests/test_nms.py failed under the compiled reference op"
    assert len(rec["nms"]) == len(expected) == 6
    for r, e in zip(rec["nms"], expected):
        r["expected"] = torch.from_numpy(np.asarray(e)).long()

    from mega_core.modeling import box_coder as bc
    spec = importlib.util.spec_from_file_location("ref_test_bc", os.path.join(ref_import.REFERENCE, "tests/test_box_coder.py"))
    tb = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tb)
    orig_dec = bc.BoxCoder.decode
    cap = {}

    def rec_dec(self, rel, boxes):
        out = orig_dec(self, rel, boxes)
        cap.update({"deltas": rel.clone(), "boxes": boxes.clone(), "weights": tuple(self.weights), "out": out.clone()})
        return out

    bc.BoxCoder.decode = rec_dec
    orig_close = np.testing.assert_allclose

    def cap_close(a, b, *k, **kw):
        cap["expected"] = torch.from_numpy(np.asarray(b).copy())
        return orig_close(a, b, *k, **kw)

    np.testing.assert_allclose = cap_close
    res = unittest.TextTestRunner(verbosity=0).run(unittest.defaultTestLoader.loadTestsFromModule(tb))
    np.testing.assert_allclose = orig_close
    bc.BoxCoder.decode = orig_dec
    assert res.wasSuccessful()
    rec["decode"] = cap

    # oracle vs golden
    for r in rec["nms"]:
        for cuda_sem in (False, True):
            keep = mo.nms(r["boxes"], r["scores"], r["thresh"], cuda_sem)
            assert keep.tolist() == sorted(r["expected"].tolist()), ("oracle nms", r["thresh"], cuda_sem)
    out = mo.decode_boxes(cap["deltas"], cap["boxes"], cap["weights"])
    close(out, cap["expected"], 1e-4, "decode vs test_box_coder golden")
    assert torch.equal(out, cap["out"]), "oracle decode != reference decode bitwise"
    print("  reference NMS / box-coder golden vectors: oracle matches (6 + 1 cases)")
    return rec


# ------------------------------------------------------------------ 2. op-level outputs of the reference
def golden_ops():
    ref_import.setup()
    out = {}
    from mega_core.modeling.rpn.anchor_generator import generate_anchors
    ref_anchors = generate_anchors(16, (64, 128, 256, 512), (0.5, 1.0, 2.0)).float()
    assert torch.equal(ref_anchors, mo.cell_anchors(16, (64, 128, 256, 512), (0.5, 1.0, 2.0)))
    # the table in the reference's comments (anchor_generator.py:199-217) is for sizes 32..512 @ stride 16
    out["cell_anchors"] = ref_anchors
    _C = sys.modules["mega_core._C"]
    g = torch.Generator().manual_seed(11)
    cases = []
    for (c, h, w, k, sr) in ((8, 20, 30, 24, 0), (5, 13, 17, 9, 2), (16, 38, 63, 40, 0)):
        feat = torch.randn(2, c, h, w, generator=g)
        x1 = torch.rand(k, generator=g) * w * 16 * 0.8 - 20
        y1 = torch.rand(k, generator=g) * h * 16 * 0.8 - 20
        bw = torch.rand(k, generator=g) * w * 8 + 1
        bh = torch.rand(k, generator=g) * h * 8 + 1
        rois = torch.stack([torch.randint(0, 2, (k,), generator=g).float(), x1, y1, x1 + bw, y1 + bh], 1)
        rois[0, 1:] = torch.tensor([5.0, 5.0, 5.0, 5.0])        # degenerate roi -> forced 1x1
        rois[1, 1:] = torch.tensor([-50.0, -60.0, 3000.0, 2000.0])  # far out of bounds
        ref = _C.roi_align_forward(feat, rois, 1.0 / 16, 7, 7, sr)
        got = mo.roi_align(feat, rois, 1.0 / 16, 7, 7, sr)
        close(got, ref, 2e-6, "roi_align C oracle vs reference (c=%d)" % c)
        cases.append({"seed_case": (c, h, w, k, sr), "feat": feat, "rois": rois, "out": ref})
    out["roi_align"] = cases

    # random NMS at RPN scale, both semantics
    nms_cases = []
    for n, thr in ((300, 0.5), (2000, 0.7), (6000, 0.7)):
        xy = torch.rand(n, 2, generator=g) * torch.tensor([900.0, 500.0])
        wh = torch.rand(n, 2, generator=g) * 200 + 4
        boxes = torch.cat([xy, xy + wh], 1)
        scores = torch.rand(n, generator=g)
        ref = _C.nms(boxes, scores, thr)
        got = mo.nms(boxes, scores, thr, False)
        assert torch.equal(ref, got), "oracle nms != reference nms_cpu (n=%d)" % n
        nms_cases.append({"n": n, "thr": thr, "seed": 11, "keep_cpu": ref, "keep_cuda_sem": mo.nms(boxes, scores, thr, True),
                          "boxes": boxes if n <= 2000 else None, "scores": scores if n <= 2000 else None})
    out["nms_random"] = nms_cases
    print("  roi_align / nms / anchors: oracle matches the compiled reference ops")
    return out


# ------------------------------------------------------------------ 3. end-to-end reference runs
class _FakeImage:
    def __init__(self, idx):
        self.idx = idx

    def convert(self, mode):
        return self


def run_reference_mega(sd, frames, globals_per_frame, n_frames):
    cfg = ref_import.build_cfg("configs/MEGA/vid_R_101_C4_MEGA_1x.yaml")
    from mega_core.modeling.detector import build_detection_model
    from mega_core.structures.image_list import to_image_list
    import mega_core.modeling.detector.generalized_rcnn_mega as gm
    model = build_detection_model(cfg).eval()
    full = dict(sd)
    full["rpn.anchor_generator.cell_anchors.0"] = model.state_dict()["rpn.anchor_generator.cell_anchors.0"]
    model.load_state_dict(full, strict=True)

    gm.Image = types.SimpleNamespace(open=lambda path: _FakeImage(int(os.path.basename(path).split(".")[0])))
    outs = []
    hooks = {}
    pred = model.roi_heads.box.predictor
    orig_pred = pred.forward

    def pred_fwd(x):
        r = orig_pred(x)
        hooks["class_logits"], hooks["box_regression"], hooks["x_final"] = r[0].clone(), r[1].clone(), x.clone()
        return r

    pred.forward = pred_fwd
    with torch.no_grad():
        for t in range(n_frames):
            images = {"cur": frames[t][0].clone(),
                      "ref_l": [] if t == 0 else [to_image_list(frames[min(t + 12, len(frames) - 1)][0].clone())],
                      "ref_g": [to_image_list(frames[j][0].clone()) for j in globals_per_frame[t]],
                      "frame_category": 0 if t == 0 else 1, "seg_len": len(frames), "pattern": "%06d",
                      "img_dir": "/nonexistent/%s.JPEG", "transforms": lambda im: frames[im.idx][0].clone()}
            res = model(images)[0]
            outs.append({"boxes": res.bbox.clone(), "scores": res.get_field("scores").clone(),
                         "labels": res.get_field("labels").clone(), **{k: v for k, v in hooks.items()}})
    return outs


def golden_mega(h=192, w=320, n_frames=4, total=40):
    print("  MEGA R-101 @%dx%d: reference vs oracle, %d frames" % (h, w, n_frames))
    sd = synth.make_state_dict("mega_r101", seed=0)
    frames = [synth.synthetic_frame(i, h, w) for i in range(total)]
    gidx = synth.global_frame_indices(total, seed=0)
    globals_per_frame = [gidx[:10]] + [[gidx[(10 + t - 1) % total]] for t in range(1, n_frames)]
    ref = run_reference_mega(sd, frames, globals_per_frame, n_frames)
    orc = mo.MegaOracle(sd, record=True)
    gold = []
    for t in range(n_frames):
        infos = {"frame_category": 0 if t == 0 else 1,
                 "ref_l": frames[1:13] if t == 0 else [frames[min(t + 12, total - 1)]],
                 "ref_g": [frames[j] for j in globals_per_frame[t]]}
        b, s, l = orc.forward(frames[t], infos)
        r = ref[t]
        assert r["class_logits"].shape == orc.trace["class_logits"].shape, "proposal count differs"
        close(orc.trace["class_logits"], r["class_logits"], 2e-5, "frame %d class_logits" % t)
        close(orc.trace["box_regression"], r["box_regression"], 2e-5, "frame %d box_regression" % t)
        assert torch.equal(l, r["labels"]) and b.shape == r["boxes"].shape, "detections differ (frame %d)" % t
        close(b, r["boxes"], 1e-4, "frame %d det boxes" % t)
        close(s, r["scores"], 1e-5, "frame %d det scores" % t)
        gold.append({"class_logits": r["class_logits"], "box_regression": r["box_regression"],
                     "proposals": orc.trace["proposals"], "boxes": r["boxes"], "scores": r["scores"],
                     "labels": r["labels"]})
    return {"arch": "mega_r101", "seed": 0, "h": h, "w": w, "total": total, "globals_per_frame": globals_per_frame,
            "frames": gold}


def run_reference_rdn(sd, frames, n_frames):
    cfg = ref_import.build_cfg("configs/RDN/vid_R_101_C4_RDN_1x.yaml")
    from mega_core.modeling.detector import build_detection_model
    from mega_core.structures.image_list import to_image_list
    import mega_core.modeling.detector.generalized_rcnn_rdn as gr
    model = build_detection_model(cfg).eval()
    full = dict(sd)
    full["rpn.anchor_generator.cell_anchors.0"] = model.state_dict()["rpn.anchor_generator.cell_anchors.0"]
    model.load_state_dict(full, strict=True)
    gr.Image = types.SimpleNamespace(open=lambda path: _FakeImage(int(os.path.basename(path).split(".")[0])))
    outs, hooks = [], {}
    pred = model.roi_heads.box.predictor
    orig_pred = pred.forward

    def pred_fwd(x):
        r = orig_pred(x)
        hooks["class_logits"], hooks["box_regression"] = r[0].clone(), r[1].clone()
        return r

    pred.forward = pred_fwd
    with torch.no_grad():
        for t in range(n_frames):
            images = {"cur": frames[t][0].clone(),
                      "ref": [] if t == 0 else [to_image_list(frames[min(t + 18, len(frames) - 1)][0].clone())],
                      "frame_category": 0 if t == 0 else 1, "seg_len": len(frames), "pattern": "%06d",
                      "img_dir": "/nonexistent/%s.JPEG", "transforms": lambda im: frames[im.idx][0].clone()}
            res = model(images)[0]
            outs.append({"boxes": res.bbox.clone(), "scores": res.get_field("scores").clone(),
                         "labels": res.get_field("labels").clone(), **{k: v for k, v in hooks.items()}})
    return outs


def golden_rdn(h=192, w=320, n_frames=3, total=40):
    print("  RDN R-101 @%dx%d: reference vs oracle, %d frames" % (h, w, n_frames))
    sd = synth.make_state_dict("rdn_r101", seed=4)
    frames = [synth.synthetic_frame(i, h, w) for i in range(total)]
    ref = run_reference_rdn(sd, frames, n_frames)
    orc = mo.RdnOracle(sd, record=True)
    gold = []
    for t in range(n_frames):
        infos = {"frame_category": 0 if t == 0 else 1, "ref": frames[1:19] if t == 0 else [frames[min(t + 18, total - 1)]]}
        b, s, l = orc.forward(frames[t], infos)
        r = ref[t]
        assert r["class_logits"].shape == orc.trace["class_logits"].shape, "proposal count differs"
        close(orc.trace["class_logits"], r["class_logits"], 2e-5, "frame %d class_logits" % t)
        close(orc.trace["box_regression"], r["box_regression"], 2e-5, "frame %d box_regression" % t)
        assert torch.equal(l, r["labels"]) and b.shape == r["boxes"].shape, "detections differ (frame %d)" % t
        close(b, r["boxes"], 1e-4, "frame %d det boxes" % t)
        close(s, r["scores"], 1e-5, "frame %d det scores" % t)
        gold.append({"class_logits": r["class_logits"], "box_regression": r["box_regression"],
                     "proposals": orc.trace["proposals"], "boxes": r["boxes"], "scores": r["scores"],
                     "labels": r["labels"]})
    return {"arch": "rdn_r101", "seed": 4, "h": h, "w": w, "total": total, "frames": gold}


def run_reference_fgfa(sd, frames, n_frames):
    cfg = ref_import.build_cfg("configs/FGFA/vid_R_101_C4_FGFA_1x.yaml")
    from mega_core.modeling.detector import build_detection_model
    from mega_core.structures.image_list import to_image_list
    import mega_core.modeling.detector.generalized_rcnn_fgfa as gf
    model = build_detection_model(cfg).eval()
    full = dict(sd)
    full["rpn.anchor_generator.cell_anchors.0"] = model.state_dict()["rpn.anchor_generator.cell_anchors.0"]
    model.load_state_dict(full, strict=True)
    gf.Image = types.SimpleNamespace(open=lambda path: _FakeImage(int(os.path.basename(path).split(".")[0])))
    outs, hooks = [], {}
    pred = model.roi_heads.box.predictor
    orig_pred = pred.forward

    def pred_fwd(x):
        r = orig_pred(x)
        hooks["class_logits"], hooks["box_regression"] = r[0].clone(), r[1].clone()
        return r

    pred.forward = pred_fwd
    orig_flow = model.flownet.forward

    def flow_fwd(x):
        r = orig_flow(x)
        hooks["flow"] = r.clone()
        return r

    model.flownet.forward = flow_fwd
    orig_rpn = model.rpn.forward

    def rpn_fwd(images, features, targets=None):
        hooks["feats"] = features[0].clone()
        return orig_rpn(images, features, targets)

    model.rpn.forward = rpn_fwd
    with torch.no_grad():
        for t in range(n_frames):
            images = {"cur": frames[t][0].clone(),
                      "ref": [] if t == 0 else [to_image_list(frames[min(t + 9, len(frames) - 1)][0].clone())],
                      "frame_category": 0 if t == 0 else 1, "seg_len": len(frames), "pattern": "%06d",
                      "img_dir": "/nonexistent/%s.JPEG", "transforms": lambda im: frames[im.idx][0].clone()}
            res = model(images)[0]
            outs.append({"boxes": res.bbox.clone(), "scores": res.get_field("scores").clone(),
                         "labels": res.get_field("labels").clone(), **{k: v for k, v in hooks.items()}})
    return outs


def golden_fgfa(h=192, w=320, n_frames=3, total=30):
    print("  FGFA R-101 @%dx%d: reference vs oracle, %d frames" % (h, w, n_frames))
    sd = synth.make_state_dict("fgfa_r101", seed=5)
    frames = [synth.synthetic_frame(i, h, w) for i in range(total)]
    ref = run_reference_fgfa(sd, frames, n_frames)
    orc = mo.FgfaOracle(sd, record=True)
    gold = []
    for t in range(n_frames):
        infos = {"frame_category": 0 if t == 0 else 1, "ref": frames[1:10] if t == 0 else [frames[min(t + 9, total - 1)]]}
        b, s, l = orc.forward(frames[t], infos)
        r = ref[t]
        close(orc.trace["flow"], r["flow"], 2e-5, "frame %d flow" % t)
        close(orc.trace["feats"], r["feats"], 2e-5, "frame %d aggregated feats" % t)
        assert r["class_logits"].shape == orc.trace["class_logits"].shape, "proposal count differs"
        close(orc.trace["class_logits"], r["class_logits"], 2e-5, "frame %d class_logits" % t)
        close(orc.trace["box_regression"], r["box_regression"], 2e-5, "frame %d box_regression" % t)
        assert torch.equal(l, r["labels"]) and b.shape == r["boxes"].shape, "detections differ (frame %d)" % t
        close(b, r["boxes"], 1e-4, "frame %d det boxes" % t)
        print("    flow rms %.3f max %.3f" % (r["flow"].pow(2).mean().sqrt().item(), r["flow"].abs().max().item()))
        gold.append({"class_logits": r["class_logits"], "box_regression": r["box_regression"],
                     "proposals": orc.trace["proposals"], "boxes": r["boxes"], "scores": r["scores"],
                     "labels": r["labels"], "flow": r["flow"], "feats_sample": r["feats"][:, ::64].clone(),
                     "feats_rms": r["feats"].pow(2).mean().sqrt().item()})
    return {"arch": "fgfa_r101", "seed": 5, "h": h, "w": w, "total": total, "frames": gold}


def run_reference_dff(sd, frames, key_flags):
    cfg = ref_import.build_cfg("configs/DFF/vid_R_101_C4_DFF_1x.yaml")
    from mega_core.modeling.detector import build_detection_model
    model = build_detection_model(cfg).eval()
    full = dict(sd)
    full["rpn.anchor_generator.cell_anchors.0"] = model.state_dict()["rpn.anchor_generator.cell_anchors.0"]
    model.load_state_dict(full, strict=True)
    outs, hooks = [], {}
    pred = model.roi_heads.box.predictor
    orig_pred = pred.forward

    def pred_fwd(x):
        r = orig_pred(x)
        hooks["class_logits"], hooks["box_regression"] = r[0].clone(), r[1].clone()
        return r

    pred.forward = pred_fwd
    orig_flow = model.flownet.forward

    def flow_fwd(x):
        r = orig_flow(x)
        hooks["flow"], hooks["scale"] = r[0].clone(), r[1].clone()
        return r

    model.flownet.forward = flow_fwd
    orig_rpn = model.rpn.forward

    def rpn_fwd(images, features, targets=None):
        hooks["feats"] = features[0].clone()
        return orig_rpn(images, features, targets)

    model.rpn.forward = rpn_fwd
    with torch.no_grad():
        for t, key in enumerate(key_flags):
            res = model({"cur": frames[t][0].clone(), "is_key_frame": key})[0]      # vid_dff.py test-time dict
            outs.append({"boxes": res.bbox.clone(), "scores": res.get_field("scores").clone(),
                         "labels": res.get_field("labels").clone(), **{k: v for k, v in hooks.items()}})
    return outs


def golden_dff(h=192, w=320, key_flags=(True, False, False, True, False)):
    print("  DFF R-101 @%dx%d: reference vs oracle, %d frames" % (h, w, len(key_flags)))
    sd = synth.make_state_dict("dff_r101", seed=6)
    frames = [synth.synthetic_frame(3 * i, h, w) for i in range(len(key_flags))]       # 3-frame stride: visible motion
    ref = run_reference_dff(sd, frames, key_flags)
    orc = mo.DffOracle(sd, record=True)
    gold = []
    for t, key in enumerate(key_flags):
        b, s, l = orc.forward(frames[t], key)
        r = ref[t]
        close(orc.trace["flow"], r["flow"], 2e-5, "frame %d flow" % t)
        close(orc.trace["scale"], r["scale"], 2e-5, "frame %d scale map" % t)
        close(orc.trace["feats"], r["feats"], 2e-5, "frame %d warped feats" % t)
        assert r["class_logits"].shape == orc.trace["class_logits"].shape, "proposal count differs"
        close(orc.trace["class_logits"], r["class_logits"], 2e-5, "frame %d class_logits" % t)
        close(orc.trace["box_regression"], r["box_regression"], 2e-5, "frame %d box_regression" % t)
        assert torch.equal(l, r["labels"]) and b.shape == r["boxes"].shape, "detections differ (frame %d)" % t
        close(b, r["boxes"], 1e-4, "frame %d det boxes" % t)
        print("    flow rms %.3f, scale in [%.2f, %.2f]" % (r["flow"].pow(2).mean().sqrt().item(), r["scale"].min().item(),
                                                          r["scale"].max().item()))
        gold.append({"class_logits": r["class_logits"], "box_regression": r["box_regression"],
                     "proposals": orc.trace["proposals"], "boxes": r["boxes"], "scores": r["scores"],
                     "labels": r["labels"], "flow": r["flow"], "scale_sample": r["scale"][:, ::64].clone(),
                     "feats_sample": r["feats"][:, ::64].clone(), "feats_rms": r["feats"].pow(2).mean().sqrt().item()})
    return {"arch": "dff_r101", "seed": 6, "h": h, "w": w, "key_flags": list(key_flags), "frame_stride": 3, "frames": gold}


def golden_base(h=192, w=320):
    print("  single-frame R-50-C4 @%dx%d: reference vs oracle" % (h, w))
    cfg = ref_import.build_cfg("configs/vid_R_50_C4_1x.yaml")
    from mega_core.modeling.detector import build_detection_model
    model = build_detection_model(cfg).eval()
    sd = synth.make_state_dict("base_r50", seed=1)
    full = dict(sd)
    full["rpn.anchor_generator.cell_anchors.0"] = model.state_dict()["rpn.anchor_generator.cell_anchors.0"]
    model.load_state_dict(full, strict=True)
    img = synth.synthetic_frame(3, h, w)
    hooks = {}
    pred = model.roi_heads.box.predictor
    orig = pred.forward

    def pf(x):
        r = orig(x)
        hooks["class_logits"], hooks["box_regression"] = r[0].clone(), r[1].clone()
        return r

    pred.forward = pf
    with torch.no_grad():
        res = model([img[0].clone()])[0]
    orc = mo.BaseOracle(sd, record=True)
    b, s, l = orc.forward(img)
    close(orc.trace["class_logits"], hooks["class_logits"], 2e-5, "base class_logits")
    assert torch.equal(l, res.get_field("labels"))
    close(b, res.bbox, 1e-4, "base det boxes")
    return {"arch": "base_r50", "seed": 1, "h": h, "w": w, "frame_index": 3,
            "class_logits": hooks["class_logits"], "box_regression": hooks["box_regression"],
            "proposals": orc.trace["proposals"], "boxes": res.bbox.clone(),
            "scores": res.get_field("scores").clone(), "labels": res.get_field("labels").clone()}


# ------------------------------------------------------------------ 4. the YAML configs tools/test_net.py is run with
CONFIGS = ("configs/BASE_RCNN_1gpu.yaml", "configs/MEGA/vid_R_101_C4_MEGA_1x.yaml", "configs/RDN/vid_R_101_C4_RDN_1x.yaml",
           "configs/FGFA/vid_R_101_C4_FGFA_1x.yaml", "configs/DFF/vid_R_101_C4_DFF_1x.yaml", "configs/vid_R_50_C4_1x.yaml")


def golden_configs():
    """the settings of each config, by path, as yaml.safe_load reads them (what cfg.merge_from_file merges)"""
    import yaml
    out = {}
    for rel in CONFIGS:
        with open(os.path.join(ref_import.REFERENCE, rel)) as fh:
            out[rel] = yaml.safe_load(fh)
    return out


def write_golden_configs():
    with open(os.path.join(GOLD, "reference_configs.json"), "w") as fh:
        json.dump(golden_configs(), fh, indent=1, sort_keys=True)
        fh.write("\n")


def main():
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(8)
    only = set(sys.argv[1:])
    if "rdn" in only:
        torch.save(golden_rdn(), os.path.join(GOLD, "rdn_r101_192x320.pt"))
        return
    if "fgfa" in only:
        torch.save(golden_fgfa(), os.path.join(GOLD, "fgfa_r101_192x320.pt"))
        return
    if "dff" in only:
        torch.save(golden_dff(), os.path.join(GOLD, "dff_r101_192x320.pt"))
        return
    if "configs" in only:
        write_golden_configs()
        return
    print("[1] reference unit-test vectors")
    torch.save(golden_from_reference_tests(), os.path.join(GOLD, "reference_unit_vectors.pt"))
    print("[2] op-level reference outputs")
    torch.save(golden_ops(), os.path.join(GOLD, "reference_ops.pt"))
    print("[3] end-to-end")
    torch.save(golden_base(), os.path.join(GOLD, "base_r50_192x320.pt"))
    torch.save(golden_mega(), os.path.join(GOLD, "mega_r101_192x320.pt"))
    torch.save(golden_rdn(), os.path.join(GOLD, "rdn_r101_192x320.pt"))
    torch.save(golden_fgfa(), os.path.join(GOLD, "fgfa_r101_192x320.pt"))
    torch.save(golden_dff(), os.path.join(GOLD, "dff_r101_192x320.pt"))
    print("[4] configs")
    write_golden_configs()
    for f in sorted(os.listdir(GOLD)):
        print("  wrote", f, os.path.getsize(os.path.join(GOLD, f)), "bytes")


if __name__ == "__main__":
    main()
