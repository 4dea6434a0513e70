"""GPU: bench.py --dump-outputs writes the last timed step's search result, and two runs with the same arguments write
the same arrays (sizes shrunk so that each run takes seconds)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, nq, k):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1", "--corpus", "20000",
           "--nq", str(nq), "--k", str(k), "--skip-encode", "--skip-cpu", "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["parity"]["ok"]
    return np.load(out_dir / "D.npy"), np.load(out_dir / "I.npy")


@pytest.mark.parametrize("nq,k,rows", [(300, 100, 300), (6000, 1000, 5332)])  # 6000 x 1000 exceeds 64 MB: sampled rows
def test_dump_outputs_are_reproducible(tmp_path, nq, k, rows):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    D, I = _bench(tmp_path / "a", nq, k)
    assert D.dtype == np.float32 and I.dtype == np.float64 and D.shape == I.shape == (rows, k)
    assert D.nbytes + I.nbytes <= 64 * 10 ** 6
    assert (np.diff(D, axis=1) <= 0).all() and (I >= 0).all() and (I < 20000).all() and (I == np.round(I)).all()
    D2, I2 = _bench(tmp_path / "b", nq, k)
    np.testing.assert_array_equal(D, D2)
    np.testing.assert_array_equal(I, I2)
