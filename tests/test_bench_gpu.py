"""bench.py --dump-outputs on a GPU: what it writes is the sorted input, the same for both algorithms."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_is_a_sample_of_the_sorted_input(tmp_path):
    import torch
    sys.path.insert(0, ROOT)
    import bench
    log2n = 23                                       # above bench.DUMP_KEYS: the sampled form
    n = 1 << log2n
    want = np.sort(bench._make_device_keys(torch, n, "uniform", 1, "cuda").cpu().numpy())[bench.dump_positions(n)]
    for algo in ("radix", "merge"):
        d = tmp_path / algo
        r = subprocess.run([sys.executable, "bench.py", "--algo", algo, "--log2n", str(log2n), "--steps", "2",
                            "--warmup", "1", "--e2e-steps", "1", "--no-cpu-baseline", "--no-configs",
                            "--dump-outputs", str(d)], cwd=ROOT, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        assert os.listdir(d) == ["sorted_keys.npy"]
        got = np.load(d / "sorted_keys.npy")
        assert got.dtype == np.float64 and got.shape == (bench.DUMP_KEYS,)
        assert os.path.getsize(d / "sorted_keys.npy") <= 64 << 20
        assert np.array_equal(got, want.astype(np.float64)), algo
