"""bench.py --dump-outputs: the samples of the last timed move as float32 / float64 .npy files, capped in size by a
fixed seeded subset of the games, identical from run to run with the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ("boards", "acts", "pi", "counts", "moves", "over", "flags")


def _sample(g, seed=1):
    rng = np.random.default_rng(seed)
    return {"boards": rng.integers(0, 256, (g, 96), dtype=np.uint8),
            "acts": rng.integers(-1, 2086, (g, 128), dtype=np.int16),
            "pi": rng.random((g, 128)),
            "counts": rng.integers(1, 120, g, dtype=np.int16),
            "moves": rng.integers(0, 2086, g, dtype=np.int16),
            "over": rng.integers(0, 2, g, dtype=np.uint8),
            "flags": rng.integers(0, 32, g, dtype=np.uint8)}


def _load(d):
    return {k: np.load(os.path.join(d, f"{k}.npy")) for k in KEYS + ("game_index",)}


def test_dump_keeps_every_game_under_the_limit(tmp_path):
    sample = _sample(300)
    bench.dump_outputs(str(tmp_path), sample)
    got = _load(tmp_path)
    assert np.array_equal(got["game_index"], np.arange(300))
    for k in KEYS:
        assert got[k].dtype == (np.float64 if k == "pi" else np.float32)
        assert np.array_equal(got[k], sample[k])


def test_dump_samples_a_fixed_subset_above_the_limit(tmp_path):
    sample, limit = _sample(1000), 400_000
    bench.dump_outputs(str(tmp_path / "a"), sample, limit=limit)
    bench.dump_outputs(str(tmp_path / "b"), sample, limit=limit)
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= limit
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    idx = a["game_index"].astype(np.int64)
    assert 100 < len(idx) < 1000 and np.array_equal(idx, np.unique(idx)) and np.array_equal(idx, b["game_index"])
    for k in KEYS:
        assert np.array_equal(a[k], sample[k][idx]) and np.array_equal(a[k], b[k])


def test_steps_below_one_are_rejected():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       timeout=120)
    assert p.returncode == 2 and "--steps" in p.stderr


@pytest.mark.gpu
def test_dump_is_reproducible_and_steps_are_timed(tmp_path):
    """Two runs with the same arguments dump the same arrays; --steps 4 fills the 4-move sample ring with the last
    timed move, so the dump comes from the ring drained inside that move."""
    games, steps = 32, 4
    dumps = []
    for run in ("a", "b"):
        out = tmp_path / run
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--games", str(games), "--playouts", "16",
                            "--steps", str(steps), "--warmup", "1", "--no-replay", "--no-movegen", "--no-train",
                            "--no-cpu-baseline", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900)
        assert p.returncode == 0, p.stderr[-3000:]
        line = json.loads(p.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps
        assert line["config"]["resident_samples_drained_in_timed_region"] == steps * games
        dumps.append(_load(out))
    a, b = dumps
    assert np.array_equal(a["game_index"], np.arange(games))
    assert a["boards"].shape == (games, 96) and a["pi"].shape == (games, 128)
    counts = a["counts"].astype(np.int64)
    assert (counts > 0).all() and np.allclose(a["pi"].sum(1), 1.0)
    # the move played is one of the root's children
    assert all(a["moves"][g] in a["acts"][g, : counts[g]] for g in range(games))
    for k in KEYS:
        assert np.array_equal(a[k], b[k]), k
