"""bench.py --dump-outputs: one float64 .npy per output array, and above the size cap the same fixed,
seeded sample of rows in every array and every run.  CPU only."""
import numpy as np

import bench


def test_dump_outputs_writes_float64_arrays_whole(tmp_path):
    mu = np.linspace(0.5, 7.0, 11)
    tr = mu.astype(np.float32)
    bench.dump_outputs(str(tmp_path / "out"), {"mu": mu, "trace_last_step": tr})
    a, b = np.load(tmp_path / "out" / "mu.npy"), np.load(tmp_path / "out" / "trace_last_step.npy")
    assert a.dtype == b.dtype == np.float64
    assert np.array_equal(a, mu) and np.array_equal(b, tr.astype(np.float64))


def test_dump_outputs_samples_the_same_rows_above_the_cap(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 8000)
    mu = np.arange(10000, dtype=np.float64)
    got = []
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {"mu": mu, "trace_last_step": -mu})
        got.append((np.load(tmp_path / run / "mu.npy"), np.load(tmp_path / run / "trace_last_step.npy")))
    (a, ta), (b, tb) = got
    assert 0 < a.nbytes + ta.nbytes <= 8000
    assert np.array_equal(ta, -a)                        # the same rows of every array
    assert np.all(np.diff(a) > 0)                         # distinct rows, in order
    assert np.array_equal(a, b) and np.array_equal(ta, tb)
