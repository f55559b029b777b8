"""bench.py --dump-outputs: what it writes for one result (CPU only)."""
import os

import numpy as np
import pytest

import bench


@pytest.mark.parametrize("n", [10, 3 * bench.DUMP_SAMPLE + 5])
def test_dump_outputs_fixed_sample_within_bounds(tmp_path, n):
    ms = np.random.default_rng(n).choice(np.frombuffer(b"ACGTacgt", dtype=np.uint8), n).tobytes()
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), ms, 123)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["result.npy", "superstring_sample.npy", "superstring_sample_positions.npy"]
    out = {}
    for f in files:
        a = np.load(tmp_path / "a" / f)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, np.load(tmp_path / "b" / f))
        out[f[:-4]] = a
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 << 20
    assert out["result"].tolist() == [n, 123]
    pos = out["superstring_sample_positions"].astype(np.int64)
    assert len(pos) == min(n, bench.DUMP_SAMPLE) and pos[0] >= 0 and pos[-1] < n and np.all(np.diff(pos) > 0)
    assert np.array_equal(out["superstring_sample"], np.frombuffer(ms, dtype=np.uint8)[pos])
