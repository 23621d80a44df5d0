"""bench.py's CPU-only pieces: the C1 record (examples/pitch_detection.rs as shipped, timed on the oracle) must work with and
without --steps, and --dump-outputs writes a bounded, reproducible sample of a step's outputs.  The GPU test runs bench.py
itself with --steps and --dump-outputs."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_c1_record_without_and_with_steps():
    for steps in (None, 3):
        rec = bench.c1_record(argparse.Namespace(steps=steps))
        assert rec["unit"] == "frames/s" and rec["value"] > 0 and rec["higher_is_better"] is True
        assert rec["steps"] == (20 if steps is None else 3)
        case = rec["cases"]["sine_150hz_2048"] if "sine_150hz_2048" in rec["cases"] else next(iter(rec["cases"].values()))
        assert isinstance(case, dict)


def test_dump_outputs_writes_a_seeded_sample_of_large_outputs(tmp_path):
    n = bench.DUMP_ROWS + 1000
    arrays = {"tracks": np.arange(n * 8, dtype=np.float32).reshape(n, 4, 2), "n_cand": np.arange(300, dtype=np.int32),
              "r": np.linspace(0, 1, 26).reshape(2, 13)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), "cx", arrays)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["cx_n_cand.npy", "cx_r.npy", "cx_tracks.npy", "cx_tracks_rows.npy"]
    for name in names:
        a, b = np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), name
    rows = np.load(tmp_path / "a" / "cx_tracks_rows.npy").astype(np.int64)
    assert rows.size == bench.DUMP_ROWS and np.all(np.diff(rows) > 0) and rows[-1] < n
    assert np.array_equal(np.load(tmp_path / "a" / "cx_tracks.npy"), arrays["tracks"][rows])
    assert np.array_equal(np.load(tmp_path / "a" / "cx_n_cand.npy"), np.arange(300, dtype=np.float32))
    assert np.load(tmp_path / "a" / "cx_r.npy").dtype == np.float64


def test_dump_outputs_of_every_config_stay_below_64_mb(tmp_path):
    """The outputs of Workload's four configs, each longer than DUMP_ROWS: --config all writes them all into one directory."""
    F = 2 * bench.DUMP_ROWS
    f32 = lambda *s: np.zeros(s, dtype=np.float32)  # noqa: E731
    outs = {"c2": {"r": f32(F, 13), "lpc": f32(F, 13)}, "c3": {"tracks": f32(F, 4, 2), "estimates": f32(F, 4, 2)},
            "c4": {"candidates": f32(F, 16, 2), "n_cand": np.zeros(F, np.int32), "status": np.zeros(F, np.uint8)},
            "c5": {"mfcc": f32(F, 13)}}
    for key, arrays in outs.items():
        bench.dump_outputs(str(tmp_path), key, arrays)
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) < 64 << 20


@pytest.mark.gpu
def test_bench_steps_and_dump_outputs(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "c2", "--utts", "4", "--steps", "3",
                          "--warmup", "1", "--no-cpu", "--dump-outputs", str(tmp_path)],
                         cwd=str(tmp_path), capture_output=True, text=True, check=True).stdout
    rec = json.loads(out.strip().splitlines()[-1])
    F = rec["config"]["frames_per_gpu"]
    assert rec["steps"] == 3 and F == 4 * bench.n_frames_of(160000, 400, 160)
    assert sorted(os.listdir(tmp_path)) == ["c2_lpc.npy", "c2_r.npy"]
    r, lpc = np.load(tmp_path / "c2_r.npy"), np.load(tmp_path / "c2_lpc.npy")
    assert r.shape == lpc.shape == (F, 13) and r.dtype == lpc.dtype == np.float32
    assert np.all(np.isfinite(lpc)) and np.all(r[:, 0] > 0) and np.all(lpc[:, 0] == 1.0)
