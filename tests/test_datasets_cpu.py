"""mega_core.data.datasets / collate / sampler / make_data_loader (test-time side; SURVEY.md section 8f row 1: the step
in front of the hot path) on a synthetic ImageNet-VID tree. Every item of all five dataset classes is compared with what
the UNMODIFIED reference classes produced on the same tree (tests/golden/reference_datasets.pt, written by
oracle/run_ref_datasets.py) -- tensors bit for bit, targets, the scalar fields, including the reference's `cur` /
last-global-frame aliasing in VIDMEGADataset."""
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import image_oracle as io_  # noqa: E402

WNIDS = ["n02691156", "n02084071", "n02958343"]
MEAN, STD = [102.9801, 115.9465, 122.7717], [1.0, 1.0, 1.0]


def make_tree(root, videos=(("val/vidA", 14, 160, 96), ("val/vidB", 9, 128, 80))):
    from PIL import Image
    g = np.random.default_rng(0)
    ils = os.path.join(root, "ILSVRC2015")
    os.makedirs(os.path.join(ils, "ImageSets"), exist_ok=True)
    lines, fid = [], 1
    for vdir, n, w, h in videos:
        os.makedirs(os.path.join(ils, "Data", "VID", vdir), exist_ok=True)
        os.makedirs(os.path.join(ils, "Annotations", "VID", vdir), exist_ok=True)
        for i in range(n):
            img = g.integers(0, 256, (h, w, 3), dtype=np.uint8)
            Image.fromarray(img, "RGB").save(os.path.join(ils, "Data", "VID", vdir, "%06d.JPEG" % i), quality=95)
            objs = ""
            for _ in range(int(g.integers(0, 3))):
                x1, y1 = int(g.integers(0, w - 30)), int(g.integers(0, h - 30))
                objs += ("<object><name>%s</name><bndbox><xmin>%d</xmin><ymin>%d</ymin><xmax>%d</xmax><ymax>%d</ymax></bndbox>"
                         "</object>" % (WNIDS[int(g.integers(0, 3))], x1, y1, x1 + int(g.integers(8, 29)), y1 + int(g.integers(8, 29))))
            with open(os.path.join(ils, "Annotations", "VID", vdir, "%06d.xml" % i), "w") as f:
                f.write("<annotation><size><width>%d</width><height>%d</height></size>%s</annotation>" % (w, h, objs))
            lines.append("%s %d %d %d" % (vdir, fid, i, n))
            fid += 1
    with open(os.path.join(ils, "ImageSets", "VID_val_videos.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")
    return len(lines)


def fingerprint(x, root):
    """what the comparison with the reference keeps of an item's images: tensors as (dtype, shape, SHA-256 of the
    bytes), paths relative to the tree's `root`, everything else as is"""
    if hasattr(x, "tensors"):
        x = x.tensors
    if torch.is_tensor(x):
        return (str(x.dtype), tuple(x.shape), hashlib.sha256(x.contiguous().numpy().tobytes()).hexdigest())
    if isinstance(x, dict):
        return {k: fingerprint(v, root) for k, v in x.items() if k != "transforms"}
    if isinstance(x, (list, tuple)):
        return [fingerprint(v, root) for v in x]
    if isinstance(x, str):
        return x.replace(root, "<root>")
    return x


class CpuTransform(object):
    """the reference's test-time transform (PIL pipeline) with its (image, target) -> (tensor, target) signature"""

    def __init__(self, min_size=60, max_size=100):
        self.min_size, self.max_size = min_size, max_size

    def __call__(self, image, target=None):
        t = io_.reference_pipeline(np.asarray(image), self.min_size, self.max_size, MEAN, STD, True)
        if target is not None:
            target = target.resize((t.shape[2], t.shape[1]))
        return t, target


def _datasets(root):
    from mega_core.data import datasets as D
    ils = os.path.join(root, "ILSVRC2015")
    args = dict(image_set="VID_val_videos", data_dir=root, img_dir=os.path.join(ils, "Data", "VID"),
                anno_path=os.path.join(ils, "Annotations", "VID"), img_index=os.path.join(ils, "ImageSets", "VID_val_videos.txt"),
                transforms=CpuTransform(), is_train=False)
    out = {}
    for key, cls in (("base", D.VIDDataset), ("rdn", D.VIDRDNDataset), ("mega", D.VIDMEGADataset),
                     ("fgfa", D.VIDFGFADataset), ("dff", D.VIDDFFDataset)):
        np.random.seed(0)
        out[key] = cls(**args)
    return out


def test_datasets_collate_sampler_loader(tmp_path):
    from mega_core.config import cfg
    from mega_core.data.collate_batch import BatchCollator
    from mega_core.data.samplers import VIDTestDistributedSampler
    n = make_tree(str(tmp_path))
    ds = _datasets(str(tmp_path))
    assert all(len(d) == n for d in ds.values()) and ds["mega"].start_index == [0, 14]
    images, target, idx = ds["mega"][0]
    assert images["frame_category"] == 0 and len(images["ref_g"]) == cfg.MODEL.VID.MEGA.GLOBAL.SIZE and len(images["ref_l"]) == 1
    assert torch.equal(images["cur"], images["ref_g"][-1])                 # the reference's aliasing, kept
    images, _, _ = ds["mega"][5]
    assert images["frame_category"] == 1 and len(images["ref_g"]) == 1 and images["seg_len"] == 14
    assert ds["dff"][10][0]["is_key_frame"] and not ds["dff"][11][0]["is_key_frame"]
    assert ds["rdn"][0][0]["pattern"] == "val/vidA/%06d" and ds["base"].get_img_info(20) == {"height": 80, "width": 128}
    batch = BatchCollator(0, "mega", False)([ds["mega"][3]])
    assert batch[0]["cur"].tensors.shape[0] == 1 and batch[0]["ref_l"][0].tensors.dim() == 4 and batch[2] == (3,)
    base = BatchCollator(0, "base", False)([ds["base"][1], ds["base"][2]])
    assert base[0].tensors.shape[0] == 2
    parts = [list(VIDTestDistributedSampler(ds["mega"], num_replicas=2, rank=r)) for r in range(2)]
    assert parts[0] == list(range(0, 14)) and parts[1] == list(range(14, 23))      # whole videos per rank
    # make_data_loader with an explicit CPU transform and catalog
    from mega_core.config.paths_catalog import DatasetCatalog
    from mega_core.data import make_data_loader

    class Catalog(DatasetCatalog):
        DATA_DIR = str(tmp_path)

    c = cfg.clone()
    c.merge_from_dict({"DATASETS": {"TEST": ("VID_val_videos",)}, "TEST": {"IMS_PER_BATCH": 1},
                       "MODEL": {"VID": {"METHOD": "rdn"}}, "DATALOADER": {"NUM_WORKERS": 0}})
    np.random.seed(0)
    (loader,) = make_data_loader(c, is_train=False, transforms=CpuTransform(), dataset_catalog=Catalog)
    first = next(iter(loader))
    assert first[0]["frame_category"] == 0 and first[2] == (0,) and len(loader) == n


def test_datasets_equal_the_reference_classes(tmp_path):
    make_tree(str(tmp_path))
    ref = torch.load(os.path.join(ROOT, "tests", "golden", "reference_datasets.pt"), weights_only=False)
    mine = _datasets(str(tmp_path))
    for key, ds in mine.items():
        assert ref[key]["start_index"] == getattr(ds, "start_index", None)
        assert len(ds) == len(ref[key]["items"]), key
        for i, want in enumerate(ref[key]["items"]):
            images, target, idx = ds[i]
            assert idx == want["idx"] and torch.equal(target.bbox, want["boxes"]) and target.size == tuple(want["size"])
            assert torch.equal(target.get_field("labels"), want["labels"])
            assert ds.get_img_info(i) == ref[key]["img_info"][i]
            assert fingerprint(images, str(tmp_path)) == want["images"], (key, i)
