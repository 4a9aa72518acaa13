"""bench.py --dump-outputs on the GPU, at a small batch: the files hold what the last timed step computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_of_the_last_step(tmp_path):
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                        "--batch", "4", "--prototypes", "1024", "--no-cpu-baseline", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=900, cwd=tmp_path)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["steps"] == 2
    arrays = {name[:-4]: np.load(out / name) for name in os.listdir(out)}
    assert sorted(arrays) == ["loss", "params", "teacher"]
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    for name, a in arrays.items():
        assert a.dtype == np.float32 and np.isfinite(a).all(), name
    assert np.allclose(arrays["loss"][:6], d["loss"], rtol=0, atol=1e-5)   # the loss vector the bench line reports
    assert np.abs(arrays["params"]).max() > 0 and np.abs(arrays["teacher"]).max() > 0
