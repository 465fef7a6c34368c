"""`bench.py --dump-outputs` on a B200: the last timed step's outputs land as float32 .npy files, within 64 MB, and the
JSON line reports exactly the --steps timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_of_the_last_timed_step(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--no-cpu-baseline",
                          "--dump-outputs", str(tmp_path)], cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["steps"] == 2 and "sustained" not in d
    files = sorted(os.listdir(tmp_path))
    assert files == ["logits.npy", "loss.npy", "params_sample.npy"]
    a = {f[:-4]: np.load(tmp_path / f) for f in files}
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in a.values())
    assert a["loss"].shape == (1,) and a["loss"][0] == np.float32(d["loss"])
    assert a["logits"].shape == (d["config"]["per_gpu_batch"], 14)
    assert a["params_sample"].shape == (1 << 22,) and a["params_sample"].std() > 0
    assert sum(os.path.getsize(tmp_path / f) for f in files) <= 64 << 20
