"""bench.py --impl reference (the CPU arm of the benchmark contract: the oracle port of the reference path timed on the
host cores) runs without a GPU and prints ONE JSON line with the contract's keys; the b200 arm's flags parse."""
import json
import os
import subprocess
import sys
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--height", "96", "--width", "160"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True and d["n_gpus"] == 1
    assert d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 1 and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_b200_arm_flags():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True, timeout=120)
    for flag in ("--gpus", "--steps", "--warmup", "--impl", "--wave", "--no-wave", "--precision", "--dump-outputs"):
        assert flag in out.stdout
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True,
                         text=True, timeout=120)
    assert out.returncode != 0 and "--steps" in out.stderr


def test_dump_outputs_writes_every_key_frame_as_float32(tmp_path):
    """--dump-outputs: <precision>_frame<g>_{boxes,scores,labels}.npy for each key frame of the last step"""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench

    def det(n):
        return types.SimpleNamespace(to_host=lambda: (torch.rand(n, 4) * 100, torch.rand(n), torch.randint(1, 31, (n,))))

    arrays = bench.detection_arrays("fp32x3", [det(3), det(0)])
    bench.dump_outputs(str(tmp_path / "out"), arrays)
    names = sorted(os.listdir(tmp_path / "out"))
    assert names == sorted("fp32x3_frame%d_%s.npy" % (g, f) for g in range(2) for f in ("boxes", "scores", "labels"))
    for name in names:
        a = np.load(tmp_path / "out" / name)
        assert a.dtype == np.float32 and np.array_equal(a, arrays[name[:-4]])
    assert arrays["fp32x3_frame0_boxes"].shape == (3, 4) and arrays["fp32x3_frame1_labels"].shape == (0,)
