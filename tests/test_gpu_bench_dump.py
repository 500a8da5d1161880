"""bench.py --dump-outputs: the flagship step's outputs land as float .npy files within 64 MB, next to one JSON line."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_dump_outputs_writes_the_timed_step_tables(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0", "--blocks", "none",
                        "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, cwd=tmp_path, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
    files = sorted(p.name for p in tmp_path.iterdir())
    assert files == ["item_bias.npy", "item_factors.npy", "loss_sum.npy", "user_factors_every16th_row.npy"], files
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= 64 << 20
    arrays = {p.stem: np.load(p) for p in tmp_path.iterdir()}
    assert arrays["item_factors"].shape == (100_000, 64) and arrays["user_factors_every16th_row"].shape == (62_500, 64)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64) and np.isfinite(a).all(), name
    assert arrays["loss_sum"][0] > 0
