"""bench.py --dump-outputs on the GPU: what the timed path returned for its last step is written as float32 / float64 .npy files,
64 MB at most, and two runs with the same arguments write the same arrays (so two builds can be compared output for output)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def _bench(out_dir):
    args = ["--config", "1", "--frames", "512", "--steps", "2", "--warmup", "3", "--skip-cpu", "--skip-e2e", "--dump-outputs", str(out_dir)]
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [line for line in p.stdout.splitlines() if line.startswith("{")]
    assert len(lines) == 1
    assert json.loads(lines[0])["steps"] == 2
    return {f[: -len(".npy")]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


@pytest.mark.gpu
def test_dump_outputs_are_reproducible(tmp_path):
    a, b = _bench(tmp_path / "a"), _bench(tmp_path / "b")
    names = ("result_counts", "transmissions", "signals", "spectrogram_times_ms", "spectrogram_rows", "averager_db", "noise_threshold_db")
    assert sorted(a) == sorted(b) == sorted(f"band0_{n}" for n in names)
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    assert a["band0_averager_db"].shape == a["band0_noise_threshold_db"].shape == (4096,)
    assert a["band0_result_counts"].shape == (4,) and a["band0_transmissions"].shape[1] == 4
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        assert np.array_equal(a[k], b[k]), k
