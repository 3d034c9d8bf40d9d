"""bench.py --dump-outputs on the device: the frame the last timed step rendered, as the render call returns it."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_timed_frame(tmp_path):
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                        "--no-cpu-baseline", "--no-fp32-tier", "--no-torch-gpu", "--no-finetune", "--dump-outputs", str(out)],
                       capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
    assert sorted(os.listdir(out)) == ["depth.npy", "rgb.npy"]
    rgb, depth = np.load(out / "rgb.npy"), np.load(out / "depth.npy")
    assert rgb.dtype == depth.dtype == np.float32
    assert rgb.shape == (512 * 640, 3) and depth.shape == (512 * 640,)
    assert np.isfinite(rgb).all() and rgb.min() >= 0 and rgb.max() <= 1 and rgb.std() > 0
    assert np.isfinite(depth).all() and depth.std() > 0
