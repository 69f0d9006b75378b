"""bench.py on the GPU: --dump-outputs writes the final latents of the last timed step of both timed paths, and --steps sets the number
of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_dump_outputs(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny", "--steps", "2", "--warmup", "1", "--no-cpu",
                        "--no-eager", "--no-profile", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == 2 and d["finite_output"] is True
    assert sorted(os.listdir(tmp_path)) == ["tiny_e2e_latents.npy", "tiny_latents.npy"]
    resident, e2e = np.load(tmp_path / "tiny_latents.npy"), np.load(tmp_path / "tiny_e2e_latents.npy")
    assert resident.dtype == e2e.dtype == np.float32 and resident.shape == e2e.shape == (2, 4, 32, 32)
    assert np.isfinite(resident).all() and np.abs(resident).max() > 0
    # same seeded inputs through the same captured graphs: the two paths agree up to 16-bit rounding
    assert np.abs(resident - e2e).max() <= 2e-2 * max(1.0, np.abs(resident).max())
