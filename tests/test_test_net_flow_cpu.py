"""What tools/test_net.py of the reference imports from `mega_core` (test_net.py:4-19) resolves in this package, the
reference's YAML configs merge into its config tree, and the steps of test_net.main that do not need a GPU -- config,
logger, checkpointer, data loader over a synthetic ImageNet-VID tree with the reference dataset layout -- run. The
configs' settings are stored in tests/golden/reference_configs.json (oracle/make_golden.py) and written back as YAML."""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))


def test_imports_of_tools_test_net_resolve():
    from mega_core.utils.env import setup_environment  # noqa: F401
    from mega_core.utils.dist_env import init_dist  # noqa: F401
    from mega_core.config import cfg  # noqa: F401
    from mega_core.data import make_data_loader  # noqa: F401
    from mega_core.engine.inference import inference  # noqa: F401
    from mega_core.modeling.detector import build_detection_model  # noqa: F401
    from mega_core.utils.checkpoint import DetectronCheckpointer  # noqa: F401
    from mega_core.utils.collect_env import collect_env_info
    from mega_core.utils.comm import synchronize, get_rank
    from mega_core.utils.logger import setup_logger
    from mega_core.utils.miscellaneous import mkdir  # noqa: F401
    assert get_rank() == 0 and "libmega_b200" in collect_env_info()
    synchronize()
    assert setup_logger("mega_core.test", "", 1) is not None


def write_reference_configs(root):
    """the reference's configs as YAML files under `root`, at their paths in the reference checkout"""
    import yaml
    with open(os.path.join(ROOT, "tests", "golden", "reference_configs.json")) as fh:
        configs = json.load(fh)
    for rel, settings in configs.items():
        os.makedirs(os.path.dirname(os.path.join(root, rel)), exist_ok=True)
        with open(os.path.join(root, rel), "w") as fh:
            yaml.safe_dump(settings, fh)
    return root


def test_reference_yaml_configs_merge_and_drive_the_loader(tmp_path):
    from mega_core.config import cfg as base
    from mega_core.config.paths_catalog import DatasetCatalog
    from mega_core.data import make_data_loader
    from mega_core.modeling.detector import build_detection_model
    from test_datasets_cpu import CpuTransform, make_tree
    ref = write_reference_configs(str(tmp_path / "reference"))
    for method, yaml, arch in (("mega", "configs/MEGA/vid_R_101_C4_MEGA_1x.yaml", "GeneralizedRCNNMEGA"),
                               ("rdn", "configs/RDN/vid_R_101_C4_RDN_1x.yaml", "GeneralizedRCNNRDN"),
                               ("fgfa", "configs/FGFA/vid_R_101_C4_FGFA_1x.yaml", "GeneralizedRCNNFGFA"),
                               ("dff", "configs/DFF/vid_R_101_C4_DFF_1x.yaml", "GeneralizedRCNNDFF"),
                               ("base", "configs/vid_R_50_C4_1x.yaml", "GeneralizedRCNN")):
        cfg = base.clone()
        cfg.merge_from_file(os.path.join(ref, "configs/BASE_RCNN_1gpu.yaml"))          # test_net.py:75-78
        cfg.merge_from_file(os.path.join(ref, yaml))
        cfg.merge_from_list(["MODEL.DEVICE", "cpu", "DATALOADER.NUM_WORKERS", 0])
        cfg.freeze()
        assert cfg.MODEL.VID.METHOD == method and cfg.MODEL.META_ARCHITECTURE == arch and cfg.TEST.IMS_PER_BATCH == 1
        model = build_detection_model(cfg)
        assert type(model).__name__ == arch
    # the MEGA config drives the loader over a tree laid out like datasets/ILSVRC2015
    make_tree(str(tmp_path))

    class Catalog(DatasetCatalog):
        DATA_DIR = str(tmp_path)

    cfg = base.clone()
    cfg.merge_from_file(os.path.join(ref, "configs/BASE_RCNN_1gpu.yaml"))
    cfg.merge_from_file(os.path.join(ref, "configs/MEGA/vid_R_101_C4_MEGA_1x.yaml"))
    cfg.merge_from_list(["DATALOADER.NUM_WORKERS", 0])
    assert tuple(cfg.DATASETS.TEST) == ("VID_val_videos",)
    np.random.seed(0)
    (loader,) = make_data_loader(cfg, is_train=False, is_distributed=False, transforms=CpuTransform(), dataset_catalog=Catalog)
    images, targets, ids = next(iter(loader))
    assert images["frame_category"] == 0 and len(images["ref_g"]) == 10 and images["cur"].tensors.shape[:2] == (1, 3)
    assert torch.is_tensor(targets[0].bbox) and ids == (0,)
