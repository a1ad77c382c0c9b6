"""Runs the UNMODIFIED reference dataset classes (mega_core/data/datasets/vid*.py) with the reference's CPU transforms on
the synthetic ImageNet-VID tree of tests/test_datasets_cpu.make_tree and writes every test item as the fixture the
checker of mega_core.data.datasets in tests/test_datasets_cpu.py compares with: image tensors as fingerprints (dtype,
shape, SHA-256 of the bytes), paths relative to the tree. TEST INFRASTRUCTURE; separate process (it imports the
reference's `mega_core`).
Usage (needs the reference checkout, see ref_import.py):
    python oracle/run_ref_datasets.py tests/golden/reference_datasets.pt"""
import importlib.util
import os
import sys
import tempfile
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tests"))
import ref_import  # noqa: E402
from test_datasets_cpu import fingerprint, make_tree  # noqa: E402


def load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def main(out_path):
    with tempfile.TemporaryDirectory() as data_dir:
        make_tree(data_dir)
        out = run(data_dir)
    torch.save(out, out_path)


def run(data_dir):
    ref_import.setup()
    ref = os.path.join(ref_import.REFERENCE, "mega_core")
    # the dataset files, by path: the package __init__ chain pulls in COCO / Cityscapes helpers that are not installed
    for pkg in ("mega_core.data", "mega_core.data.datasets", "mega_core.data.transforms"):
        m = types.ModuleType(pkg)
        m.__path__ = []
        sys.modules[pkg] = m
    if "cv2" not in sys.modules:
        try:
            import cv2  # noqa: F401
        except Exception:
            sys.modules["cv2"] = types.ModuleType("cv2")
    T = load("mega_core.data.transforms.transforms", os.path.join(ref, "data", "transforms", "transforms.py"))
    sys.modules["mega_core.data.transforms"].transforms = T
    build = load("mega_core.data.transforms.build", os.path.join(ref, "data", "transforms", "build.py"))
    mods = {}
    for name in ("vid", "vid_rdn", "vid_mega", "vid_fgfa", "vid_dff"):
        mods[name] = load("mega_core.data.datasets." + name, os.path.join(ref, "data", "datasets", name + ".py"))
    from mega_core.config import cfg
    cfg.merge_from_list(["INPUT.MIN_SIZE_TEST", 60, "INPUT.MAX_SIZE_TEST", 100])
    transforms = build.build_transforms(cfg, is_train=False)
    root = os.path.join(data_dir, "ILSVRC2015")
    args = dict(image_set="VID_val_videos", data_dir=data_dir, img_dir=os.path.join(root, "Data", "VID"),
                anno_path=os.path.join(root, "Annotations", "VID"), img_index=os.path.join(root, "ImageSets", "VID_val_videos.txt"),
                transforms=transforms, is_train=False)
    out = {}
    for key, cls in (("base", mods["vid"].VIDDataset), ("rdn", mods["vid_rdn"].VIDRDNDataset),
                     ("mega", mods["vid_mega"].VIDMEGADataset), ("fgfa", mods["vid_fgfa"].VIDFGFADataset),
                     ("dff", mods["vid_dff"].VIDDFFDataset)):
        np.random.seed(0)
        ds = cls(**args)
        items = []
        for i in range(len(ds)):
            images, target, idx = ds[i]
            items.append({"images": fingerprint(images, data_dir), "boxes": target.bbox.clone(),
                          "labels": target.get_field("labels").clone(), "size": target.size, "idx": idx})
        out[key] = {"items": items, "img_info": [ds.get_img_info(i) for i in range(len(ds))],
                    "start_index": getattr(ds, "start_index", None)}
        os.remove(os.path.join(data_dir, "cache", "VID_val_videos_anno.pkl"))
    return out


if __name__ == "__main__":
    main(sys.argv[1])
