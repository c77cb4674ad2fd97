"""bench.py --dump-outputs: what the last timed step returned is written as float .npy files, exactly, and a larger result
is sampled the same way every time so that two builds can be compared output for output."""
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench as B  # noqa: E402
from hyperqueue_b200 import _lib as L  # noqa: E402


def _result(n, seed=0):
    rng = np.random.default_rng(seed)
    a = np.zeros(n, dtype=L.assignment_dtype)
    a["task"] = rng.permutation(n).astype(np.uint32) + np.uint32(4_000_000_000 - n)     # beyond float32's exact range
    a["worker"] = rng.integers(0, 1024, n)
    a["variant"] = rng.integers(0, 8, n)
    a["kind"] = rng.integers(0, 3, n)
    free = rng.integers(0, 1 << 40, (256, 4)).astype(np.uint64)
    return a, free


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_is_exact_and_float(tmp_path):
    a, free = _result(5000)
    B.dump_outputs(str(tmp_path), 0, 1, a, free)
    got = _load(tmp_path)
    assert sorted(got) == ["assignment_kind", "assignment_task", "assignment_variant", "assignment_worker", "free_after"]
    assert all(v.dtype in (np.float32, np.float64) for v in got.values())
    for f in ("task", "worker", "variant", "kind"):
        assert np.array_equal(got[f"assignment_{f}"], a[f].astype(np.float64))
    assert np.array_equal(got["free_after"], free.astype(np.float64))


def test_larger_results_are_sampled_the_same_way_within_the_budget(tmp_path, monkeypatch):
    monkeypatch.setattr(B, "DUMP_BYTES", 400_000)
    a, free = _result(100_000)
    for world in (1, 3):
        dirs = [tmp_path / f"w{world}_{k}" for k in range(2)]
        for d in dirs:
            for r in range(world):
                B.dump_outputs(str(d), r, world, a, free)
        first, second = _load(dirs[0]), _load(dirs[1])
        assert first.keys() == second.keys() and all(np.array_equal(first[k], second[k]) for k in first)
        assert sum(os.path.getsize(os.path.join(dirs[0], f)) for f in os.listdir(dirs[0])) <= B.DUMP_BYTES
        sfx = ".rank0" if world > 1 else ""
        rows = first["assignment_row" + sfx].astype(np.int64)
        assert 0 < rows.size < a.size and (np.diff(rows) > 0).all()
        assert np.array_equal(first["assignment_task" + sfx], a["task"][rows].astype(np.float64))


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True)
    assert r.returncode == 2 and "--steps" in r.stderr
