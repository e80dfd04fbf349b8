"""bench.py contract checks: the reference arm (the unmodified reference / the oracle port on the host cores) prints one
JSON line with the agreed keys; our arm refuses to run without a CUDA device (no CPU fallback); with --dump-outputs both
arms write the image of their last timed step, which in the bit-exact modes is the reference's frame."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from test_oracle import image_hash, parity_render

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LAST_STEP = "stock_1280x720_t0.0_flags0_frames4+1"       # --warmup 3 --steps 2: frames 3 and 4 are timed


def test_reference_arm_json_line(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "3",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "Mray/s" and line["higher_is_better"] is True
    assert line["metric"].startswith("Mray/s on 46-sphere scene") and line["steps"] == 2
    assert line["value"] > 1.0 and line["ms_per_step"] > 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "Mray/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and "model" not in line["config"]
    assert os.listdir(tmp_path) == ["image.npy"]
    img = np.load(tmp_path / "image.npy")
    assert img.dtype == np.float32 and img.shape == (720, 1280, 4)
    assert image_hash(img, []) == parity_render(LAST_STEP)["sha256_pads_zeroed"]


def test_our_arm_needs_a_gpu():
    import toypathtracer_b200 as tpt
    if tpt.device_count() > 0:
        pytest.skip("a CUDA device is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "3", "--no-cpu-baseline"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0          # fails loudly: nothing is rendered on the CPU
    assert not r.stdout.strip()


@pytest.mark.gpu
def test_our_arm_dumps_its_last_step(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--mode", "exact", "--steps", "2", "--warmup", "3",
                        "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["n_gpus"] == 1
    assert os.listdir(tmp_path) == ["image.npy"]
    img = np.load(tmp_path / "image.npy")
    assert img.dtype == np.float32 and img.shape == (720, 1280, 4)
    assert image_hash(img, []) == parity_render(LAST_STEP)["sha256_pads_zeroed"]
