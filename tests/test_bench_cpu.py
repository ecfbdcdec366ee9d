"""bench.py's reference arm runs on CPU and prints the contract's JSON line."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ)
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--log2n", "20"], cwd=ROOT, capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    j = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in j, key
    assert j["impl"] == "reference" and j["unit"] == "keys/s" and j["value"] > 0
    assert j["cpu_baseline"]["kind"] in ("reference", "port") and j["cpu_baseline"]["cores"] == 1
    assert j["e2e"]["h2d_bytes_per_step"] == 0 and j["e2e"]["value"] == j["value"]
    assert "workload" in j["config"]


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       cwd=ROOT, capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_arguments_it_cannot_honour_are_rejected():
    for extra in (["--steps", "0"], ["--impl", "reference", "--steps", "0"], ["--gpus", "2", "--dump-outputs", "d"]):
        r = subprocess.run([sys.executable, "bench.py", *extra], cwd=ROOT, capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and r.stdout == "" and "error:" in r.stderr, extra


def test_reference_arm_dumps_the_sorted_sample_it_timed(tmp_path):
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from b200sort import datagen
    d = tmp_path / "dump"
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--dump-outputs", str(d)], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    m = 1 << 24                                      # the arm's host sample at this step count
    assert os.listdir(d) == ["sorted_keys.npy"]
    got = np.load(d / "sorted_keys.npy")
    assert got.dtype == np.float64 and got.shape == (bench.DUMP_KEYS,)
    assert np.array_equal(got, np.sort(datagen.make("uniform", m, 1))[bench.dump_positions(m)].astype(np.float64))


def test_roofline_traffic_comes_from_the_committed_ncu_summary():
    sys.path.insert(0, ROOT)
    import bench
    t = bench._ncu_traffic("radix_onesweep")
    assert t is None or (t["bytes"] > 2.0e9 and t["source"].startswith("profiles/"))
