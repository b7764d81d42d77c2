"""bench.py --dump-outputs: what is written for an output-for-output comparison of two builds."""
import numpy as np

from bench import DUMP_BYTES, dump_outputs


def test_small_outputs_are_written_whole(tmp_path):
    ids = np.arange(40, dtype=np.int32).reshape(4, 10)
    ids[3, 9] = -1                                           # a padded slot
    dist = np.linspace(0, 1, 40, dtype=np.float32).reshape(4, 10)
    dump_outputs(str(tmp_path), {"ids": ids, "distances": dist})
    got_i, got_d = np.load(tmp_path / "ids.npy"), np.load(tmp_path / "distances.npy")
    assert got_i.dtype == np.float64 and np.array_equal(got_i, ids)
    assert got_d.dtype == np.float32 and np.array_equal(got_d, dist)
    assert sorted(p.name for p in tmp_path.iterdir()) == ["distances.npy", "ids.npy"]


def test_large_outputs_are_one_fixed_sample(tmp_path):
    n = 1 << 24                                              # the scores of PageRank at RMAT scale 24: 64 MiB
    scores = np.arange(n, dtype=np.float32)
    for d in ("a", "b"):
        dump_outputs(str(tmp_path / d), {"scores": scores})
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= DUMP_BYTES
    rows = np.load(tmp_path / "a" / "sample_rows.npy")
    assert np.array_equal(rows, np.load(tmp_path / "b" / "sample_rows.npy"))
    assert np.all(np.diff(rows) > 0) and rows.size > n // 4
    assert np.array_equal(np.load(tmp_path / "a" / "scores.npy"), scores[rows.astype(np.int64)])
