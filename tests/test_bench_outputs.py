"""bench.py --dump-outputs: the state of the timed path written as .npy files.  Host logic against a stand-in engine (no
GPU), and on the GPU two runs with the same arguments, which must write the same files with the same contents."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load_bench():
    spec = importlib.util.spec_from_file_location("kta_bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


class FakeEngine:
    """Answers every read-back getter with a value derived from its arguments."""

    def counter(self, i, p):
        return 1000 * p + i

    def hist(self, which, p):
        return np.arange(32, dtype=np.uint64) + 100 * p + which

    def global_(self, i):
        return [2**64 - 1, 0, 7, 8][i]

    def timestamps(self):
        return 1500000000, 5000000, 1500000001000

    def alive_keys(self):
        return 12345

    def hll_registers(self):
        return np.arange(1 << 12, dtype=np.uint8) % 30

    def alive_keys_hll(self):
        return 12001.5


def test_dump_files_dtypes_and_values(tmp_path):
    bench = load_bench()
    bench.dump_outputs(FakeEngine(), 8, "fused", str(tmp_path), "x_")
    names = sorted(os.listdir(tmp_path))
    assert names == ["x_%s.npy" % n for n in ("alive_keys", "alive_keys_hll", "counters", "globals", "hll_registers",
                                               "key_size_hist", "partitions", "timestamps", "value_size_hist")]
    load = lambda n: np.load(tmp_path / ("x_%s.npy" % n))
    assert load("hll_registers").dtype == np.float32
    assert all(load(n).dtype == np.float64 for n in ("counters", "key_size_hist", "globals", "alive_keys"))
    assert load("counters").shape == (8, 7) and load("counters")[3, 2] == 3002
    assert load("value_size_hist").shape == (8, 32) and load("value_size_hist")[2, 5] == 206
    assert list(load("timestamps")) == [1500000000, 5000000, 1500000001000]
    assert load("alive_keys")[0] == 12345 and load("alive_keys_hll")[0] == 12001.5
    assert np.array_equal(load("hll_registers"), FakeEngine().hll_registers())


def test_dump_modes_and_partition_sample(tmp_path):
    """counters mode has no alive-key outputs; a topic with more partitions than DUMP_PARTITIONS is dumped for a fixed
    sample of them, the same one on every run, within the 64 MB budget."""
    bench = load_bench()
    P = 100_000
    for run in ("a", "b"):
        bench.dump_outputs(FakeEngine(), P, "counters", str(tmp_path / run))
    assert sorted(os.listdir(tmp_path / "a")) == ["counters.npy", "globals.npy", "key_size_hist.npy", "partitions.npy",
                                                  "timestamps.npy", "value_size_hist.npy"]
    parts = np.load(tmp_path / "a" / "partitions.npy")
    assert parts.shape == (bench.DUMP_PARTITIONS,) and len(set(parts.tolist())) == parts.size and parts.max() < P
    for name in os.listdir(tmp_path / "a"):
        assert np.array_equal(np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name))
    assert np.array_equal(np.load(tmp_path / "a" / "counters.npy")[:, 0], parts * 1000)
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in os.listdir(tmp_path / "a")) < 64 << 20


def test_steps_below_one_are_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True)
    assert r.returncode == 2 and "--steps" in r.stderr


@pytest.mark.gpu
def test_dump_is_reproducible_and_matches_the_timed_steps(tmp_path):
    n, steps = 64 * 10_000, 3
    args = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
            "--n", str(n), "--distinct-keys", "50000", "--no-cpu", "--no-e2e", "--no-extra"]
    for run in ("a", "b"):
        r = subprocess.run(args + ["--dump-outputs", str(tmp_path / run)], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
        assert line["steps"] == steps
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b")) and "hll_registers.npy" in names
    for name in names:
        assert np.array_equal(np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)), name
    counters = np.load(tmp_path / "a" / "counters.npy")
    assert counters.shape == (64, 7) and counters[:, 0].sum() == n * steps       # every timed step was counted once
    assert np.load(tmp_path / "a" / "globals.npy")[3] == n * steps
    assert np.load(tmp_path / "a" / "hll_registers.npy").max() > 0
