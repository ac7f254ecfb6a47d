"""bench.py --dump-outputs: the outputs of the last timed wave, exact and reproducible from the arguments."""

import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.conftest import ROOT

BENCH = os.path.join(ROOT, "bench.py")


def test_bench_rejects_zero_steps_and_a_dump_of_the_reference_arm():
    for args, msg in ((["--steps", "0"], "--steps must be at least 1"),
                      (["--impl", "reference", "--dump-outputs", "x"], "--dump-outputs needs --impl b200")):
        r = subprocess.run([sys.executable, BENCH, *args], capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and msg in r.stderr, r.stderr


def test_dump_is_exact_and_a_fixed_sample_above_the_size_limit(tmp_path, monkeypatch):
    import bench

    n = 1000
    g = torch.Generator().manual_seed(3)
    states = torch.randint(-2**31, 2**31 - 1, (n, 32), dtype=torch.int32, generator=g)
    steps = torch.randint(0, 80, (n,), dtype=torch.int32, generator=g)
    bench.dump_outputs(str(tmp_path / "all"), states, steps)
    words = states.numpy().view(np.uint32)
    got = np.load(tmp_path / "all" / "states.npy")
    assert got.dtype == np.float64 and np.array_equal(got.astype(np.uint32), words)
    assert np.array_equal(np.load(tmp_path / "all" / "steps.npy"), steps.numpy())
    assert np.load(tmp_path / "all" / "total_steps.npy").tolist() == [int(steps.sum())]
    assert not (tmp_path / "all" / "rows.npy").exists()

    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 100_000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), states, steps)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["rows.npy", "states.npy", "steps.npy", "total_steps.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 100_000
    rows = np.load(tmp_path / "a" / "rows.npy").astype(np.int64)
    assert 0 < len(rows) < n and np.all(np.diff(rows) > 0)
    assert np.array_equal(np.load(tmp_path / "a" / "states.npy").astype(np.uint32), words[rows])
    assert np.array_equal(np.load(tmp_path / "a" / "steps.npy"), steps.numpy()[rows])
    assert np.load(tmp_path / "a" / "total_steps.npy").tolist() == [int(steps.sum())]
    for f in files:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_wave(tmp_path, oracle):
    """--steps K times K waves; the last one plays the games of seed 1000 + K - 1 (bench.py fresh())"""
    n, k = 2048, 3
    r = subprocess.run([sys.executable, BENCH, "--gpus", "1", "--steps", str(k), "--warmup", "1", "--games", str(n), "--no-mcts",
                        "--no-cpu-baseline", "--no-python-reference", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    ref, ref_steps, ref_total = oracle.playout(oracle.init_states(n, seed=1000 + k - 1), n_threads=4)
    assert np.array_equal(np.load(tmp_path / "states.npy").astype(np.uint32), ref)
    assert np.array_equal(np.load(tmp_path / "steps.npy").astype(np.uint32), ref_steps)
    assert np.load(tmp_path / "total_steps.npy").tolist() == [ref_total]
