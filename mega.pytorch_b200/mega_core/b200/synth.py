"""Synthetic video frames and a deterministic, calibration-free random initialisation.

There is no network for datasets or checkpoints, so benchmarks and parity tests use seeded
synthetic inputs. The stock initialisers of the reference give activations of O(1e2..1e3) on
0-255 inputs and NaN logits in the reference itself (SURVEY.md section 7, "hard parts"), so
this routine keeps the reference's parameter *shapes and names* but picks values analytically
so that every layer's output is O(1) -- like a trained net -- without any data-dependent
calibration (both the oracle and the CUDA path regenerate the identical state_dict from a seed;
the 690 MB of weights are never stored).
"""
import math

import torch

PIXEL_MEAN = (102.9801, 115.9465, 122.7717)  # config/defaults.py:51-55 (BGR, 0-255 domain)


def synthetic_frame(index, height=600, width=1000, seed=1000, boxes=4):
    """fp32 [1,3,H,W] frame in the reference's post-transform domain (BGR*255 - mean):
    low-amplitude noise background with a few moving bright rectangles so that RPN scores are
    spread out (few exact ties) and detections move coherently."""
    g = torch.Generator().manual_seed(seed + index)
    img = torch.rand(3, height, width, generator=g) * 64.0 + 64.0
    gb = torch.Generator().manual_seed(seed)  # rectangle layout fixed per video, moves with index
    for b in range(boxes):
        bw = int(torch.randint(width // 10, width // 3, (1,), generator=gb))
        bh = int(torch.randint(height // 8, height // 2, (1,), generator=gb))
        x0 = int(torch.randint(0, width - bw, (1,), generator=gb))
        y0 = int(torch.randint(0, height - bh, (1,), generator=gb))
        vx = int(torch.randint(-6, 7, (1,), generator=gb))
        vy = int(torch.randint(-4, 5, (1,), generator=gb))
        col = torch.rand(3, 1, 1, generator=gb) * 200.0 + 30.0
        x = min(max(x0 + vx * index, 0), width - bw)
        y = min(max(y0 + vy * index, 0), height - bh)
        img[:, y:y + bh, x:x + bw] = col + torch.rand(3, bh, bw, generator=g) * 16.0
    img = img - torch.tensor(PIXEL_MEAN).view(3, 1, 1)
    return img.unsqueeze(0).contiguous()


def _kaiming(shape, gen, gain=math.sqrt(2.0)):
    fan_in = 1
    for d in shape[1:]:
        fan_in *= d
    return torch.randn(*shape, generator=gen) * (gain / math.sqrt(fan_in))


def _bn(sd, p, n, gen, out_scale=1.0, in_var=1.0):
    """FrozenBatchNorm2d buffers (layers/batch_norm.py:15-18). scale = weight * rsqrt(var)."""
    sd[p + "weight"] = (torch.rand(n, generator=gen) * 0.2 + 0.9) * out_scale
    sd[p + "bias"] = torch.randn(n, generator=gen) * 0.1
    sd[p + "running_mean"] = torch.randn(n, generator=gen) * 0.1 * math.sqrt(in_var)
    sd[p + "running_var"] = (torch.rand(n, generator=gen) * 0.2 + 0.9) * in_var


def _stage(sd, prefix, gen, cin, mid, cout, blocks):
    for b in range(blocks):
        p = prefix + "%d." % b
        if b == 0:
            sd[p + "downsample.0.weight"] = _kaiming((cout, cin, 1, 1), gen, gain=1.0)
            _bn(sd, p + "downsample.1.", cout, gen)
        sd[p + "conv1.weight"] = _kaiming((mid, cin if b == 0 else cout, 1, 1), gen)
        _bn(sd, p + "bn1.", mid, gen)
        sd[p + "conv2.weight"] = _kaiming((mid, mid, 3, 3), gen)
        _bn(sd, p + "bn2.", mid, gen)
        sd[p + "conv3.weight"] = _kaiming((cout, mid, 1, 1), gen)
        _bn(sd, p + "bn3.", cout, gen, out_scale=0.25)   # damp the residual branch
    return cout


def _linear(sd, p, nout, nin, gen, std=None, gain=1.0):
    std = std if std is not None else gain / math.sqrt(nin)
    sd[p + "weight"] = torch.randn(nout, nin, generator=gen) * std
    sd[p + "bias"] = torch.randn(nout, generator=gen) * 0.01


def make_state_dict(arch="mega_r101", seed=0, num_classes=31):
    """state_dict with the reference's key names/shapes for
    arch in {"mega_r101", "mega_r50", "rdn_r101", "fgfa_r101", "dff_r101", "base_r50", "base_r101"} (+ "_tiny" suffix: 1 block per stage,
    for fast CPU tests)."""
    gen = torch.Generator().manual_seed(seed)
    tiny = arch.endswith("_tiny")
    base = arch.replace("_tiny", "")
    method, depth = base.split("_")
    blocks = {"r50": (3, 4, 6, 3), "r101": (3, 4, 23, 3)}[depth]
    if tiny:
        blocks = (1, 1, 2, 1)
    sd = {}
    # stem: input std ~ 50 (0-255 domain); conv output variance ~ 2 * E[x^2]
    sd["backbone.body.stem.conv1.weight"] = _kaiming((64, 3, 7, 7), gen)
    _bn(sd, "backbone.body.stem.bn1.", 64, gen, in_var=2.0 * 70.0 ** 2)
    c = _stage(sd, "backbone.body.layer1.", gen, 64, 64, 256, blocks[0])
    c = _stage(sd, "backbone.body.layer2.", gen, c, 128, 512, blocks[1])
    c = _stage(sd, "backbone.body.layer3.", gen, c, 256, 1024, blocks[2])
    sd["rpn.anchor_generator.cell_anchors.0"] = None  # filled by the module / oracle (12 x 4)
    sd["rpn.head.conv.weight"] = _kaiming((1024, 1024, 3, 3), gen, gain=1.0)
    sd["rpn.head.conv.bias"] = torch.zeros(1024)
    sd["rpn.head.cls_logits.weight"] = torch.randn(12, 1024, 1, 1, generator=gen) * (2.0 / 32)
    sd["rpn.head.cls_logits.bias"] = torch.zeros(12)
    sd["rpn.head.bbox_pred.weight"] = torch.randn(48, 1024, 1, 1, generator=gen) * (0.25 / 32)
    sd["rpn.head.bbox_pred.bias"] = torch.zeros(48)
    fe = "roi_heads.box.feature_extractor."
    _stage(sd, fe + "head.layer4.", gen, 1024, 512, 2048, blocks[3])
    if method == "base":
        sd[fe + "conv.weight"] = _kaiming((256, 2048, 1, 1), gen, gain=1.0)
        sd[fe + "conv.bias"] = torch.zeros(256)
        _linear(sd, fe + "fc6.", 1024, 256 * 49, gen)
        _linear(sd, fe + "fc7.", 1024, 1024, gen)
    elif method in ("fgfa", "dff"):
        # GeneralizedRCNNFGFA / GeneralizedRCNNDFF: FlowNetS (+ EmbedNet for FGFA) next to the backbone
        # (backbone/flownet.py, embednet.py), box head = ResNetConv52MLPFeatureExtractor without the channel reduction
        # (configs/FGFA/vid_R_101_C4_FGFA_1x.yaml, configs/DFF/vid_R_101_C4_DFF_1x.yaml)
        _linear(sd, fe + "fc6.", 1024, 2048 * 49, gen)
        _linear(sd, fe + "fc7.", 1024, 1024, gen)

        def conv(name, cout, cin, k, gain=math.sqrt(2.0 / 1.01), bias=0.01):
            sd[name + ".weight"] = _kaiming((cout, cin, k, k), gen, gain=gain)
            sd[name + ".bias"] = torch.randn(cout, generator=gen) * bias

        conv("flownet.flow_conv1", 64, 6, 7)
        conv("flownet.conv2", 128, 64, 5)
        conv("flownet.conv3", 256, 128, 5)
        conv("flownet.conv3_1", 256, 256, 3)
        conv("flownet.conv4", 512, 256, 3)
        conv("flownet.conv4_1", 512, 512, 3)
        conv("flownet.conv5", 512, 512, 3)
        conv("flownet.conv5_1", 512, 512, 3)
        conv("flownet.conv6", 1024, 512, 3)
        conv("flownet.conv6_1", 1024, 1024, 3)
        for i, cin in zip(range(1, 6), (1024, 1026, 770, 386, 194)):
            conv("flownet.Convolution%d" % i, 2, cin, 3, gain=0.5)
        for name, cin, cout in (("deconv5", 1024, 512), ("deconv4", 1026, 256), ("deconv3", 770, 128), ("deconv2", 386, 64)):
            # ConvTranspose2d weight [cin, cout, 4, 4]; every output pixel sums 4 taps x cin inputs
            sd["flownet.%s.weight" % name] = torch.randn(cin, cout, 4, 4, generator=gen) * (1.4 / math.sqrt(4.0 * cin))
            sd["flownet.%s.bias" % name] = torch.randn(cout, generator=gen) * 0.01
        for name in ("upsample_flow6to5", "upsample_flow5to4", "upsample_flow4to3", "upsample_flow3to2"):
            sd["flownet.%s.weight" % name] = torch.randn(2, 2, 4, 4, generator=gen) * 0.25
            sd["flownet.%s.bias" % name] = torch.zeros(2)
        if method == "fgfa":
            conv("embednet.embed_conv1", 512, 1024, 1)
            conv("embednet.embed_conv2", 512, 512, 3)
            conv("embednet.embed_conv3", 2048, 512, 1, gain=1.0)
        else:
            # the reference zero-initialises the scale head (flownet.py:36-38: scale map == 1); a trained one is not
            # zero, so give it a spread of about +-0.3 around 1 to make the parity test see the branch
            sd["flownet.Convolution5_scale.weight"] = _kaiming((1024, 194, 1, 1), gen, gain=0.3)
    elif method == "rdn":
        # RDNFeatureExtractor with ATTENTION.STAGE = 2, ADVANCED_STAGE = 1 (configs/RDN/vid_R_101_C4_RDN_1x.yaml):
        # fcs[0..2], Wgs/Wqs/Wks/Wvs[0..3] (roi_box_feature_extractors.py:305-328)
        _linear(sd, fe + "fcs.0.", 1024, 2048 * 49, gen)
        for i in (1, 2):
            _linear(sd, fe + "fcs.%d." % i, 1024, 1024, gen)
        for i in range(4):
            sd[fe + "Wgs.%d.weight" % i] = torch.randn(16, 64, 1, 1, generator=gen) * 0.2
            sd[fe + "Wgs.%d.bias" % i] = torch.rand(16, generator=gen) * 0.5
            _linear(sd, fe + "Wqs.%d." % i, 1024, 1024, gen)
            _linear(sd, fe + "Wks.%d." % i, 1024, 1024, gen)
            sd[fe + "Wvs.%d.weight" % i] = torch.randn(1024, 1024, 1, 1, generator=gen) * (0.5 / 32)
            sd[fe + "Wvs.%d.bias" % i] = torch.randn(1024, generator=gen) * 0.01
    else:
        _linear(sd, fe + "l_fcs.0.", 1024, 2048 * 49, gen)
        for i in (1, 2):
            _linear(sd, fe + "l_fcs.%d." % i, 1024, 1024, gen)
        for i in range(3):
            sd[fe + "l_Wgs.%d.weight" % i] = torch.randn(16, 64, 1, 1, generator=gen) * 0.2
            sd[fe + "l_Wgs.%d.bias" % i] = torch.rand(16, generator=gen) * 0.5
            _linear(sd, fe + "l_Wqs.%d." % i, 1024, 1024, gen)
            _linear(sd, fe + "l_Wks.%d." % i, 1024, 1024, gen)
            sd[fe + "l_Wvs.%d.weight" % i] = torch.randn(1024, 1024, 1, 1, generator=gen) * (0.5 / 32)
            sd[fe + "l_Wvs.%d.bias" % i] = torch.randn(1024, generator=gen) * 0.01
        for i in range(3):
            sd[fe + "l_us.%d" % i] = torch.randn(16, 1, 64, generator=gen) * 0.1
        for i in range(2):
            _linear(sd, fe + "g_Wqs.%d." % i, 1024, 1024, gen)
            _linear(sd, fe + "g_Wks.%d." % i, 1024, 1024, gen)
            sd[fe + "g_Wvs.%d.weight" % i] = torch.randn(1024, 1024, 1, 1, generator=gen) * (0.5 / 32)
            sd[fe + "g_Wvs.%d.bias" % i] = torch.randn(1024, generator=gen) * 0.01
        for i in range(2):
            sd[fe + "g_us.%d" % i] = torch.randn(16, 1, 64, generator=gen) * 0.1
    _linear(sd, "roi_heads.box.predictor.cls_score.", num_classes, 1024, gen, std=0.03)
    _linear(sd, "roi_heads.box.predictor.bbox_pred.", num_classes * 4, 1024, gen, std=0.01)
    sd.pop("rpn.anchor_generator.cell_anchors.0")
    return sd


def global_frame_indices(seg_len, size=10, seed=0):
    """shuffled global-frame order per video, like datasets/vid_mega.py:112-120 (np.random there;
    a seeded torch permutation here -- only determinism matters for synthetic video)."""
    g = torch.Generator().manual_seed(seed)
    return torch.randperm(seg_len, generator=g).tolist()


VID_MOTION_VALUES = (0.3, 0.65, 0.7, 0.8, 0.9, 0.95, 1.0)   # the motion IoUs of tests/golden/vid_eval.pt


def vid_eval_set(n_images, seed=0, num_classes=30, max_dets=300, max_gt=5, tie_free=False,
                 motion_values=VID_MOTION_VALUES, width=640, height=360):
    """Seeded detections + ground truth for the VID evaluator, vectorised so that validation size (176,126 images) is
    quick to make. Per image 0..max_gt GT boxes (labels 1..num_classes, motion IoU drawn from motion_values) and
    0..max_dets detections: jittered copies of GT boxes with high scores and random boxes with the low, long-tailed scores
    a detector emits after its 1e-3 threshold. tie_free: every score distinct (nudged by ulps).
    -> (preds, gts, motions): numpy arrays per image, (boxes f32 [n,4], labels i64, scores f32) / (boxes, labels) / list"""
    import numpy as np
    rng = np.random.default_rng(seed)
    n_gt = rng.integers(0, max_gt + 1, n_images)
    n_det = rng.integers(0, max_dets + 1, n_images)
    G, N = int(n_gt.sum()), int(n_det.sum())
    wh = rng.uniform(16, 300, (G, 2))
    xy = rng.uniform(0, 1, (G, 2)) * (np.array([width, height]) - wh)
    gt_boxes = np.round(np.concatenate([xy, xy + wh], 1)).astype(np.float32)
    gt_labels = rng.integers(1, num_classes + 1, G)
    motion = rng.choice(np.asarray(motion_values, dtype=np.float64), G)
    gt_img = np.repeat(np.arange(n_images), n_gt)
    det_img = np.repeat(np.arange(n_images), n_det)
    gt_first = np.concatenate(([0], np.cumsum(n_gt)))
    # a detection copies one of its image's GT (jittered) with probability 0.3 when the image has any
    has_gt = n_gt[det_img] > 0
    copy = has_gt & (rng.uniform(0, 1, N) < 0.3)
    src = gt_first[det_img] + (rng.uniform(0, 1, N) * np.maximum(n_gt[det_img], 1)).astype(np.int64)
    src = np.where(copy, src, 0)
    wh_d = rng.uniform(8, 300, (N, 2))
    xy_d = rng.uniform(0, 1, (N, 2)) * (np.array([width, height]) - wh_d)
    rand_boxes = np.concatenate([xy_d, xy_d + wh_d], 1)
    g = gt_boxes[src].astype(np.float64) if G else np.zeros((N, 4))
    jit = rng.normal(0, 0.06, (N, 4)) * (g[:, 2:] - g[:, :2] + 1)[:, [0, 1, 0, 1]]
    boxes = np.where(copy[:, None], g + jit, rand_boxes)
    boxes[:, 2:] = np.maximum(boxes[:, 2:], boxes[:, :2])
    det_boxes = np.clip(boxes, 0, [width - 1, height - 1, width - 1, height - 1]).astype(np.float32)
    det_labels = np.where(copy & (rng.uniform(0, 1, N) < 0.85), gt_labels[src] if G else 0,
                          rng.integers(1, num_classes + 1, N))
    scores = np.where(copy, rng.beta(4.0, 1.5, N), rng.beta(0.4, 6.0, N) * 0.999 + 1e-3).astype(np.float32)
    if tie_free and N:
        order = np.argsort(scores, kind="stable")
        bits = scores[order].view(np.int32).astype(np.int64)
        ramp = np.arange(N, dtype=np.int64)
        bits = np.maximum.accumulate(bits - ramp) + ramp
        scores = np.empty(N, dtype=np.float32)
        scores[order] = bits.astype(np.int32).view(np.float32)
    det_first = np.concatenate(([0], np.cumsum(n_det)))
    preds, gts, motions = [], [], []
    for i in range(n_images):
        a, b = det_first[i], det_first[i + 1]
        c, d = gt_first[i], gt_first[i + 1]
        preds.append((det_boxes[a:b], det_labels[a:b], scores[a:b]))
        gts.append((gt_boxes[c:d], gt_labels[c:d]))
        motions.append(motion[c:d].tolist())
    return preds, gts, motions
