"""bench.py --dump-outputs: what lands on disk for a small and for an over-budget set of output planes (CPU only)."""
import os

import numpy as np

import bench


def planes(h, w):
    rng = np.random.default_rng(5)
    return {"output_1_y": rng.integers(0, 256, (h, w), dtype=np.uint8),
            "output_1_uv": rng.integers(0, 256, (h // 2, w // 2, 2), dtype=np.uint8)}


def written(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_small_set_is_written_whole(tmp_path):
    p = planes(36, 64)
    bench.dump_outputs(str(tmp_path), p)
    got = written(str(tmp_path))
    assert sorted(got) == sorted(p)
    for name, a in p.items():
        assert got[name].dtype == np.float32 and np.array_equal(got[name], a.astype(np.float32))


def test_large_set_keeps_the_same_seeded_rows_within_budget(tmp_path):
    p = planes(360, 640)
    budget = 200_000   # the whole set as float32 is 1.38 MB
    runs = []
    for k in range(2):
        d = tmp_path / str(k)
        bench.dump_outputs(str(d), p, budget)
        assert sum(os.path.getsize(d / f) for f in os.listdir(d)) <= budget
        runs.append(written(str(d)))
    a, b = runs
    assert sorted(a) == sorted(b) == sorted(list(p) + [f"{n}_rows" for n in p])
    for name, src in p.items():
        rows = a[f"{name}_rows"].astype(np.int64)
        assert 0 < len(rows) < len(src) and np.all(np.diff(rows) > 0)
        assert np.array_equal(a[name], src[rows].astype(np.float32))
        assert np.array_equal(a[name], b[name]) and np.array_equal(a[f"{name}_rows"], b[f"{name}_rows"])
