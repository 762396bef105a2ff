"""bench.py --dump-outputs: the arrays of the last timed step, as float32 / float64 .npy files within 64 MiB."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _sizes(d):
    return sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d))


def test_dump_writes_every_row_when_it_fits(tmp_path):
    rng = np.random.default_rng(0)
    pts, ind = rng.standard_normal((1000, 3)), rng.integers(1, 4097, (1000, 8)).astype(np.float32)
    bench.dump_outputs(str(tmp_path), {"points": pts, "indices": ind})
    assert sorted(os.listdir(tmp_path)) == ["indices.npy", "points.npy"]
    assert np.array_equal(np.load(tmp_path / "points.npy"), pts)
    got = np.load(tmp_path / "indices.npy")
    assert got.dtype == np.float32 and np.array_equal(got, ind)


def test_dump_samples_the_same_seeded_rows_when_too_large(tmp_path):
    n, limit = 20_000, 200_000
    pts = np.arange(3 * n, dtype=np.float64).reshape(n, 3)
    ind = np.arange(8 * n, dtype=np.float32).reshape(n, 8)
    for sub in ("a", "b"):
        bench.dump_outputs(str(tmp_path / sub), {"points": pts, "indices": ind}, limit=limit)
        assert _sizes(tmp_path / sub) <= limit
    rows = np.load(tmp_path / "a" / "rows.npy")
    assert rows.dtype == np.float64 and len(rows) > 0.9 * limit / 64 and np.all(np.diff(rows) > 0)
    r = rows.astype(np.int64)
    assert np.array_equal(np.load(tmp_path / "a" / "points.npy"), pts[r])
    assert np.array_equal(np.load(tmp_path / "a" / "indices.npy"), ind[r])
    for f in ("rows.npy", "points.npy", "indices.npy"):
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))


def test_dump_refuses_integer_arrays(tmp_path):
    with pytest.raises(ValueError):
        bench.dump_outputs(str(tmp_path), {"points": np.ones((4, 3)), "indices": np.ones((4, 8), dtype=np.int64)})
    assert os.listdir(tmp_path) == []


@pytest.mark.gpu
def test_bench_dump_is_the_product_of_the_timed_path(tmp_path):
    n = 4096
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--samples", str(n),
                        "--no-secondary", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["gpu_launches"] == 2
    import kde_b200 as K
    K.init(0)
    trees = [K.kde(p, bench.silverman(p)) for p in (bench.synth_points(j) for j in range(bench.NDENS))]
    p, i = K.prodAppxMSGibbsS(None, trees, None, None, Niter=bench.NITER, Np=n, seed=bench.SEED)
    got_p, got_i = np.load(tmp_path / "points.npy"), np.load(tmp_path / "indices.npy")
    assert got_p.dtype == np.float64 and got_p.shape == (n, bench.DIM)
    assert got_i.dtype == np.float32 and got_i.shape == (n, bench.NDENS)
    assert np.array_equal(got_i.astype(np.int64), i.T) and np.array_equal(got_p, p.T)
