"""bench.py's reference arm (the CPU port of the path) needs no GPU: run it on a small sample and check the
JSON contract the driver relies on."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "view1m",
                        "--cpu-sample", "20000", "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "points/s" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "crop" in d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and d["config"]["workload"].startswith("synthetic 1M-point")


def test_dumped_outputs_are_finite_and_bounded(tmp_path):
    """--dump-outputs: unscored points (NaN from the library) are dumped as -1, non-finite values are refused, indices
    become float64, and an output beyond the 64 MB budget is cut to a seeded sample, the same on every run."""
    import numpy as np
    import pytest
    import bench
    sc = np.linspace(0, 1, 20_000_000, dtype=np.float32)
    sc[::1000] = np.nan
    out = bench.dump_scores(sc)
    assert np.isfinite(out).all() and (out[::1000] == -1.0).all() and np.array_equal(out[1::1000], sc[1::1000])
    with pytest.raises(ValueError):
        bench.dump_outputs(str(tmp_path / "bad"), {"scores": sc})
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"scores": out, "keypoints": np.arange(7, dtype=np.int32)})
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["keypoints.npy", "scores.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64_000_000
    a, b = np.load(tmp_path / "a" / "scores.npy"), np.load(tmp_path / "b" / "scores.npy")
    assert a.dtype == np.float32 and 0 < len(a) < len(out) and np.array_equal(a, b)
    kp = np.load(tmp_path / "a" / "keypoints.npy")
    assert kp.dtype == np.float64 and np.array_equal(kp, np.arange(7))


def test_non_zero_ranks_of_the_reference_arm_do_nothing():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True, text=True,
                       timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""
