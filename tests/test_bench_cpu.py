"""CPU: bench.py --dump-outputs writes the last step's token ids and lengths exactly (float32), within its size limit."""
import os

import numpy as np

import bench


def test_dump_outputs_exact(tmp_path):
    toks = np.random.default_rng(1).integers(0, 51866, size=(5, 7), dtype=np.int32)
    lens = np.array([7, 3, 0, 7, 1], np.int32)
    out = tmp_path / "out"
    bench.dump_outputs(str(out), {"tokens": toks, "lengths": lens})
    assert sorted(os.listdir(out)) == ["lengths.npy", "tokens.npy"]
    t, n = np.load(out / "tokens.npy"), np.load(out / "lengths.npy")
    assert t.dtype == np.float32 and np.array_equal(t, toks)
    assert n.dtype == np.float32 and np.array_equal(n, lens)


def test_dump_outputs_seeded_sample_within_limit(tmp_path):
    toks = np.arange(1000 * 252, dtype=np.int32).reshape(1000, 252)
    lens = np.arange(1000, dtype=np.int32)
    limit = 100_000
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"tokens": toks, "lengths": lens}, limit=limit)
        assert sum(f.stat().st_size for f in (tmp_path / d).iterdir()) <= limit
    rows = np.load(tmp_path / "a" / "rows.npy")
    assert rows.dtype == np.float64 and len(rows) > 50 and np.all(np.diff(rows) > 0)
    r = rows.astype(np.int64)
    assert np.array_equal(np.load(tmp_path / "a" / "tokens.npy"), toks[r])
    assert np.array_equal(np.load(tmp_path / "a" / "lengths.npy"), lens[r])
    for f in ("rows.npy", "tokens.npy", "lengths.npy"):          # the same rows from run to run
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))
