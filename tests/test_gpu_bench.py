"""bench.py on the GPU: --dump-outputs writes the image its last timed step assembled, and --steps is the number of
timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

BENCH = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py")


def test_bench_dumps_the_image_of_its_last_timed_step(gpu_ok, tmp_path):
    out = subprocess.run([sys.executable, BENCH, "--gpus", "1", "--steps", "3", "--warmup", "1", "--spp", "4",
                          "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(tmp_path / "dump")],
                         capture_output=True, text=True, check=True)
    line = json.loads(out.stdout)
    assert line["steps"] == 3 and line["gpu_launches"] % 3 == 0
    assert sorted(os.listdir(tmp_path / "dump")) == ["image.npy"]
    img = np.load(tmp_path / "dump" / "image.npy")
    assert img.dtype == np.float32 and img.shape == (800, 800, 3) and np.isfinite(img).all()
    assert img.mean(dtype=np.float64) == pytest.approx(line["image_mean"], rel=1e-4)
    assert img.max() > 0.0
