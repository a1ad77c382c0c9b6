"""GPU parity of the `_C` ops that no VID config reaches but the north star names: sigmoid focal loss, deformable
convolution v1/v2, deformable PSROI pooling. Oracles: the reference's own Python focal-loss formula
(layers/sigmoid_focal_loss.py:40-50, restated in the oracle); torchvision.ops.deform_conv2d (same mmdet lineage
as csrc/cuda/deform_conv_kernel_cuda.cu; the reference has no CPU implementation, deform_conv.h:41 -- parity
otherwise unpinned); a plain-Python restatement of the PSROI kernel."""
import os
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))


@pytest.mark.parametrize("c", [30, 32])       # 32: the 128-bit path (four logits of a row per thread), 30: the scalar path
def test_sigmoid_focal_loss_forward_backward(cuda_dev, c):
    import mega_oracle as mo
    from mega_core import _C
    g = torch.Generator().manual_seed(1)
    n = 257
    logits = torch.randn(n, c, generator=g) * 1.5   # the reference's two formulas (stable CUDA vs naive CPU) agree to ~1e-4 here
    targets = torch.randint(-1, c + 1, (n,), generator=g, dtype=torch.int32)
    ref = mo.sigmoid_focal_loss(logits, targets.long(), 2.0, 0.25)
    got = _C.sigmoid_focalloss_forward(logits.to(cuda_dev), targets.to(cuda_dev), c, 2.0, 0.25).cpu()
    assert torch.allclose(got, ref, rtol=2e-3, atol=1e-6)
    lg = logits.clone().requires_grad_(True)
    mo.sigmoid_focal_loss(lg, targets.long(), 2.0, 0.25).sum().backward()
    d = _C.sigmoid_focalloss_backward(logits.to(cuda_dev), targets.to(cuda_dev), torch.ones(n, c, device=cuda_dev), c,
                                      2.0, 0.25).cpu()
    assert torch.allclose(d, lg.grad, rtol=5e-3, atol=1e-5)


@pytest.mark.parametrize("modulated,groups,dg", [(False, 1, 1), (True, 1, 1), (True, 2, 2)])
def test_deform_conv_matches_torchvision(cuda_dev, modulated, groups, dg):
    import torchvision
    from mega_core import _C
    from mega_core.b200 import ops
    g = torch.Generator().manual_seed(5 + groups)
    b, c, h, w, cout, k = 2, 32, 19, 23, 48, 3
    x = torch.randn(b, c, h, w, generator=g)
    wt = torch.randn(cout, c // groups, k, k, generator=g) / (c * 9 / groups) ** 0.5
    bias = torch.randn(cout, generator=g)
    off = torch.randn(b, dg * 2 * k * k, h, w, generator=g) * 2.0
    mask = torch.rand(b, dg * k * k, h, w, generator=g) if modulated else None
    ref = torchvision.ops.deform_conv2d(x.to(cuda_dev), off.to(cuda_dev), wt.to(cuda_dev),
                                        bias.to(cuda_dev) if modulated else None, stride=1, padding=1, dilation=1,
                                        mask=mask.to(cuda_dev) if modulated else None).cpu()
    out = torch.zeros(b, cout, h, w, device=cuda_dev)
    with ops.precision("fp32x3"):
        if modulated:
            _C.modulated_deform_conv_forward(x.to(cuda_dev), wt.to(cuda_dev), bias.to(cuda_dev), None, off.to(cuda_dev),
                                             mask.to(cuda_dev), out, None, k, k, 1, 1, 1, 1, 1, 1, groups, dg, True)
        else:
            _C.deform_conv_forward(x.to(cuda_dev), wt.to(cuda_dev), off.to(cuda_dev), out, None, None, k, k, 1, 1, 1, 1, 1,
                                   1, groups, dg, 64)
    torch.cuda.synchronize()
    err = ((out.cpu() - ref).abs().max() / ref.pow(2).mean().sqrt()).item()
    assert err < 1e-4, err


def test_deform_psroi_pooling(cuda_dev):
    import mega_oracle as mo
    from mega_core import _C
    g = torch.Generator().manual_seed(3)
    gs, ps, od, ncls = 3, 3, 4, 2
    data = torch.randn(1, od * gs * gs, 11, 13, generator=g)
    rois = torch.tensor([[0, 8.0, 10.0, 120.0, 90.0], [0, 40.2, 33.7, 150.9, 160.1], [0, -10.0, -5.0, 30.0, 20.0]])
    trans = torch.randn(3, 2 * ncls, ps, ps, generator=g) * 0.5
    for no_trans in (True, False):
        ref, rc = mo.deform_psroi_pool(data, rois, trans, no_trans, 1 / 16.0, od, gs, ps, ps, 4, 0.1)
        out = torch.zeros(3, od, ps, ps, device=cuda_dev)
        cnt = torch.zeros(3, od, ps, ps, device=cuda_dev)
        _C.deform_psroi_pooling_forward(data.to(cuda_dev), rois.to(cuda_dev), trans.to(cuda_dev), out, cnt, no_trans,
                                        1 / 16.0, od, gs, ps, ps, 4, 0.1)
        assert torch.equal(cnt.cpu(), rc)
        assert torch.allclose(out.cpu(), ref, rtol=1e-5, atol=1e-5)


def test_callable_submodules_match_the_oracle_pieces(cuda_dev):
    """model.backbone(x), model.rpn(images, (feats,), version=...), feature_extractor(feats, proposals, pre_calculate=True),
    feature_extractor.init_memory / init_global / update_global -- the calls GeneralizedRCNNMEGA._forward_test makes on its
    parts (generalized_rcnn_mega.py:145-158, :173-175, :208; rpn/rpn.py:213-243; extractors :657-676, :885-896) -- served
    by the detector's engine, against the oracle's functions of the same steps on the same inputs."""
    import mega_oracle as mo
    from mega_core.b200 import ops, synth
    from mega_core.modeling.detector import build_detection_model_from_state_dict
    from mega_core.structures.image_list import to_image_list
    sd = synth.make_state_dict("mega_r101_tiny", seed=3)
    model = build_detection_model_from_state_dict(sd, method="mega", device=cuda_dev, precision="fp32x3")
    h, w = 96, 160
    img = synth.synthetic_frame(2, h, w)
    images = to_image_list(img[0])
    feats = model.backbone(img.to(cuda_dev))[0]
    ref_feats = mo.resnet_c4_body(img, sd)
    assert feats.shape == ref_feats.shape and feats.dtype == torch.float32
    assert ((feats.cpu() - ref_feats).abs().max() / ref_feats.pow(2).mean().sqrt()).item() < 1e-3
    # proposals on the ORACLE's map (identical inputs): the key set, and the ref set as its prefix
    dfeats = ref_feats.to(cuda_dev)
    key = model.rpn(images, (dfeats,), version="key")
    ref = model.rpn(images, (dfeats,), version="ref")
    assert len(key) == 1 and len(ref) == 1 and len(ref[0]) == 75 and len(key[0]) <= 300
    logits, deltas = mo.rpn_head(ref_feats, sd)
    ob, osc = mo.rpn_select(logits, deltas, w, h, post_nms_top_n=300, cuda_semantics=True)[:2]
    kb = key[0].bbox.cpu()
    assert kb.shape == ob.shape
    d = (kb[:, None, :] - ob[None, :, :]).abs().amax(2)            # a near-tied NMS decision may flip: match by box
    val, idx = d.min(0)
    m = val < 0.05
    assert m.float().mean().item() >= 0.97, m.float().mean().item()
    assert (key[0].get_field("objectness").cpu()[idx[m]] - osc[m]).abs().max().item() < 1e-4
    assert torch.equal(ref[0].bbox, key[0].bbox[:75])
    # ROI features of the ref proposals
    fe = model.roi_heads.box.feature_extractor
    x = fe((dfeats,), ref, pre_calculate=True)
    r5 = mo.res5_head(ref_feats, sd, "roi_heads.box.feature_extractor.head.")
    rois = torch.cat([torch.zeros(75, 1), ref[0].bbox.cpu()], 1)
    pooled = mo.roi_align(r5, rois, 1.0 / 16, 7, 7, 0).flatten(1)
    want = torch.relu(pooled @ sd["roi_heads.box.feature_extractor.l_fcs.0.weight"].t()
                      + sd["roi_heads.box.feature_extractor.l_fcs.0.bias"])
    assert x.shape == want.shape and ((x.cpu() - want).abs().max() / want.pow(2).mean().sqrt()).item() < 2e-3
    # global pool: init + push lands in ring slot 0
    fe.init_memory()
    fe.init_global()
    x_in = x.clone()
    fe.update_global(x)
    eng = model.engine
    assert eng.glob_pushed == 1 and eng.mem_pushed == 0
    assert torch.equal(x, x_in)                                      # the caller's rows are left as they were
    pushed = eng.glob_x[:75].float()
    if ops.is_split16(eng.glob_x):                                   # strict mode stores the pool as split-fp16 pairs
        pushed = ops.unpack_split16(pushed, torch.empty_like(pushed))
    assert torch.allclose(pushed, x, atol=1e-6)
    with pytest.raises(NotImplementedError):
        fe((dfeats,), [key[0]], pre_calculate=False)
