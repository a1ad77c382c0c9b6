"""The reference's OWN evaluation script, unmodified -- tools/test_net.py of the reference checkout the oracle
imports (oracle/ref_import.py) -- executed against this package: its imports (`mega_core.config / data /
engine.inference / modeling.detector / utils.*`) resolve here, the reference's YAML configs drive it, a synthetic
ImageNet-VID tree in the reference layout stands in for the dataset, a checkpoint saved the way the reference's trainer
saves it is loaded through DetectronCheckpointer, every frame goes through `model(images)` (MEGA R-101: window / global
/ memory state machine, look-ahead frames read from disk inside the model) and the VID evaluator writes result.txt. The
device ops run on the CPU stand-ins of tests/cpu_ops.py and the device check of the module is lifted (both test-only),
so no GPU is needed; on a B200 the same script runs as is."""
import os
import runpy
import sys
import types

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
from ref_import import REFERENCE as REF  # noqa: E402  (the checkout the oracle imports; MEGA_REFERENCE overrides it)


@pytest.mark.skipif(not os.path.isfile(os.path.join(REF, "tools", "test_net.py")),
                    reason="reference checkout not present (MEGA_REFERENCE names it)")
def test_unmodified_tools_test_net_runs_on_this_package(tmp_path, monkeypatch):
    from cpu_ops import cpu_ops
    from test_datasets_cpu import CpuTransform, make_tree
    from mega_core.b200 import synth
    from mega_core.data import build as data_build
    from mega_core.modeling.detector import generalized_rcnn as G
    work = str(tmp_path)
    os.symlink(os.path.join(REF, "configs"), os.path.join(work, "configs"))
    make_tree(os.path.join(work, "datasets"), videos=(("val/vidA", 5, 160, 96), ("val/vidB", 3, 160, 96)))
    sd = synth.make_state_dict("mega_r101", seed=0)
    torch.save({"model": {"module." + k: v for k, v in sd.items()}, "iteration": 1}, os.path.join(work, "model_final.pth"))
    out_dir = os.path.join(work, "out")
    # test-only environment: an `apex` import for the script, CPU transform instead of the device one, no device check
    apex = types.ModuleType("apex")
    apex.amp = types.SimpleNamespace(init=lambda **k: None)
    monkeypatch.setitem(sys.modules, "apex", apex)
    monkeypatch.setattr(data_build, "build_transforms", lambda cfg, is_train=False: CpuTransform(96, 160))

    def engine(self):
        if self._engine is None:
            from mega_core.modeling.nets import engine_config_from
            sd_ = self._sd_override if self._sd_override is not None else self.state_dict()
            self._engine = self.engine_cls(sd_, engine_config_from(self.cfg), self.device)
        return self._engine
    monkeypatch.setattr(G._EngineBacked, "engine", property(engine))
    monkeypatch.chdir(work)
    monkeypatch.setattr(sys, "argv", ["test_net.py", "--config-file", "configs/MEGA/vid_R_101_C4_MEGA_1x.yaml",
                                      "--ckpt", os.path.join(work, "model_final.pth"), "MODEL.DEVICE", "cpu",
                                      "OUTPUT_DIR", out_dir, "DATALOADER.NUM_WORKERS", "0", "INPUT.MIN_SIZE_TEST", "96",
                                      "INPUT.MAX_SIZE_TEST", "160", "MODEL.B200.PRECISION", "tf32"])
    np.random.seed(0)
    from mega_core.config import cfg
    saved = cfg.clone()                      # the script merges into and freezes the package's GLOBAL cfg: put it back
    try:
        with cpu_ops():
            runpy.run_path(os.path.join(REF, "tools", "test_net.py"), run_name="__main__")
    finally:
        cfg.defrost()
        dict.clear(cfg)
        dict.update(cfg, saved)
    folder = os.path.join(out_dir, "inference", "VID_val_videos")
    text = open(os.path.join(folder, "result.txt")).read()
    assert "AP50 | motion=   all" in text and "Category AP" in text
    preds = torch.load(os.path.join(folder, "predictions.pth"), weights_only=False)
    assert len(preds) == 8 and all(p.has_field("scores") and p.has_field("labels") for p in preds)
    assert sum(len(p) for p in preds) > 0
