"""bench.py on the GPU: --steps sets the number of timed steps, and --dump-outputs writes the last timed step's outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu


def test_bench_steps_and_dump_outputs(tmp_path):
    out_dir = tmp_path / "outputs"
    steps = 3
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
                          "--no-e2e", "--no-cpu", "--no-nms", "--no-pipelined", "--no-extra", "--dump-outputs", str(out_dir)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["steps"] == steps and line["gpu_launches"] == 3 * steps      # preprocess, detect, align per timed step
    d = {f[:-4]: np.load(out_dir / f) for f in os.listdir(out_dir)}
    assert set(d) == {"counts", "det_scale", "det", "lmk", "tensor_sample", "tensor_sample_index", "crops_sample", "crops_sample_index"}
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    assert sum(a.nbytes for a in d.values()) <= 64 << 20
    B = line["config"]["frames_per_gpu_per_step"]
    n = int(d["counts"].sum())
    assert d["counts"].shape == d["det_scale"].shape == (B,) and n == line["faces_per_step"] > 0
    assert d["det"].shape == (n, 5) and d["lmk"].shape == (n, 5, 2)
    assert d["crops_sample"].shape == (len(d["crops_sample_index"]), 112, 112, 3) and d["crops_sample"].max() > 0
    assert d["tensor_sample"].shape == d["tensor_sample_index"].shape and d["tensor_sample_index"].max() < B * 3 * 640 * 640
