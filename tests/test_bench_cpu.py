"""CPU tier: bench.py --dump-outputs writes float32 / float64 .npy files within its size cap, sampling the same seeded images
from every array when the outputs are larger."""
import os

import numpy as np


def _outputs(n=6000):
    rng = np.random.default_rng(1)
    return {"beam3_seq": rng.integers(0, 10000, (n, 3, 16), dtype=np.int32),
            "beam3_logprobs": -rng.random((n, 3, 16), dtype=np.float32)}


def _read(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_outputs_under_the_cap_is_exact(tmp_path):
    import bench
    arrays = _outputs()
    arrays["loss"] = np.array([2.5])
    bench.write_outputs(str(tmp_path), arrays)
    got = _read(tmp_path)
    assert set(got) == set(arrays)
    assert got["beam3_seq"].dtype == np.float32 and np.array_equal(got["beam3_seq"], arrays["beam3_seq"])
    assert got["beam3_logprobs"].dtype == np.float32 and np.array_equal(got["beam3_logprobs"], arrays["beam3_logprobs"])
    assert got["loss"].dtype == np.float64 and got["loss"][0] == 2.5


def test_dump_outputs_above_the_cap_keeps_a_fixed_sample_of_images(tmp_path):
    import bench
    arrays, cap = _outputs(), 200_000
    for d in ("a", "b"):
        bench.write_outputs(str(tmp_path / d), arrays, cap=cap)
    a, b = _read(tmp_path / "a"), _read(tmp_path / "b")
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= cap + 3 * 128   # (+ .npy headers)
    rows = a["rows"].astype(np.int64)
    assert a["rows"].dtype == np.float64 and 0 < len(rows) < 6000 and np.all(np.diff(rows) > 0)
    for k in arrays:
        assert a[k].dtype == np.float32 and np.array_equal(a[k], arrays[k][rows])
        assert np.array_equal(a[k], b[k])
