"""bench.py --dump-outputs: what the timed path computed in its last step, written as .npy, is the library's
spectrogram of the benchmark's seeded input (the flagship workload, shortened to 30 s of signal)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from glfer_b200 import synth
from parity import assert_psd_close

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_hold_the_rows_of_the_timed_path(gpu_api, tmp_path):
    out = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
           "--seconds", "30", "--no-e2e", "--no-cpu", "--no-configs", "--dump-outputs", str(out)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-4000:]
    assert sorted(os.listdir(out)) == ["psd.npy"]
    got = np.load(out / "psd.npy")
    hop = 2048
    x = synth.tiled_stream(30 * 48000 // hop * hop, fs=48000, block_s=20.0, seed=0x5EED)
    want = gpu_api.GramPlan(n=4096, window_type=0, overlap=0.5, sub_mean=True).run(x)["psd"]
    assert got.dtype == np.float32 and got.shape == want.shape
    assert_psd_close(got, want, "bench --dump-outputs")
