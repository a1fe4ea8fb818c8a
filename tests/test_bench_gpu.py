"""bench.py end to end at a small size: one JSON line, --steps timed steps, and --dump-outputs writing what the last
timed step returned, from inputs that are the same on every run with the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, steps):
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "3",
           "--batch", "2", "--size", "64", "--no-cpu-baseline", "--no-other-configs", "--dump-outputs", str(out_dir)]
    res = subprocess.run(cmd, capture_output=True, text=True, cwd=out_dir.parent)
    assert res.returncode == 0, res.stderr[-4000:]
    lines = res.stdout.strip().splitlines()
    assert len(lines) == 1, res.stdout
    assert os.listdir(out_dir) == ["losses.npy"]
    return json.loads(lines[0]), np.load(out_dir / "losses.npy")


def test_bench_steps_and_dumped_losses(tmp_path):
    line, losses = _bench(tmp_path / "a", 2)
    assert line["steps"] == 2 and line["e2e"]["steps"] == 2
    assert losses.dtype == np.float64 and losses.shape == (3,)
    np.testing.assert_array_equal(losses, np.array(line["losses_last_step"]))

    # same arguments, same inputs: the losses agree within the fast-mode loss tolerance (reordered sums are the only
    # difference; up to 3e-3 apart on a B200)
    _, again = _bench(tmp_path / "b", 2)
    spread = float(np.abs(again / losses - 1).max())
    assert spread < 1e-2, spread

    # one more timed step is one more Adam update before the last loss is taken (the style loss drops ~7 % here)
    _, more = _bench(tmp_path / "c", 3)
    moved = float(np.abs(more / losses - 1).max())
    assert moved > 3e-2, (moved, spread)
    print(f"run-to-run loss spread {spread:.2e}, one extra step {moved:.2e}")
