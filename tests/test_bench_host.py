"""Host-side pieces of bench.py that need no GPU."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_watchdog_reports_stage_and_exits():
    """A run that stops making progress prints one JSON line naming the stage it was in (rank 0) and exits non-zero."""
    code = ("import sys, time; sys.path.insert(0, %r); import bench; bench.stage('unit test stage'); "
            "bench.start_watchdog(1, 0, 2); time.sleep(30)" % ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=25)
    assert r.returncode == 4
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["value"] == 0.0 and line["n_gpus"] == 2 and "unit test stage" in line["error"]
    # other ranks exit silently
    code2 = code.replace("start_watchdog(1, 0, 2)", "start_watchdog(1, 1, 2)")
    r2 = subprocess.run([sys.executable, "-c", code2], capture_output=True, text=True, timeout=25)
    assert r2.returncode == 4 and r2.stdout.strip() == ""


def test_dump_outputs_fixed_sample(tmp_path):
    """--dump-outputs: float32 I/Q of the caller's complex64 output, the whole array when small, else a sample that is
    the same on every run and within the size cap."""
    sys.path.insert(0, ROOT)
    import numpy as np
    import bench
    small = (np.arange(12) + 1j * -np.arange(12)).astype(np.complex64).reshape(3, 4)
    bench.dump_outputs(str(tmp_path / "a"), small)
    got = np.load(tmp_path / "a" / "baseband.npy")
    assert got.dtype == np.float32 and np.array_equal(got[:, 0] + 1j * got[:, 1], small.reshape(-1))
    big = np.random.default_rng(1).standard_normal((2, 2 * bench.DUMP_SAMPLES + 6)).astype(np.float32).view(np.complex64)
    for d in ("b", "c"):
        bench.dump_outputs(str(tmp_path / d), big)
    idx = np.load(tmp_path / "b" / "baseband_index.npy")
    iq = np.load(tmp_path / "b" / "baseband.npy")
    assert idx.dtype == np.float64 and iq.shape == (bench.DUMP_SAMPLES, 2)
    assert np.array_equal(idx, np.load(tmp_path / "c" / "baseband_index.npy"))
    assert np.array_equal(iq.view(np.complex64)[:, 0], big.reshape(-1)[idx.astype(np.int64)])
    assert sum(f.stat().st_size for f in (tmp_path / "b").iterdir()) <= 64 << 20
