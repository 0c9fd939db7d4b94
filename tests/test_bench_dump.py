"""bench.py --dump-outputs: the writer keeps every array whole and in float64 below the size cap, and above it takes the
same seeded sample of GP rows from every array (CPU only: it calls the writer, it does not run the bench)."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def _outputs(B=400, P=28, m=100):
    rng = np.random.default_rng(1)
    return {"mll": np.arange(B, dtype=np.float64), "grad": rng.standard_normal((B, P)), "info": np.arange(B, dtype=np.int32) % 3,
            "predict_mu": rng.standard_normal((B, m)), "predict_var": rng.random((B, m))}


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_whole_outputs_in_float64(tmp_path):
    want = _outputs()
    bench.dump_outputs(str(tmp_path), want)
    got = _load(tmp_path)
    assert sorted(got) == sorted(want)
    for k, a in want.items():
        assert got[k].dtype == np.float64 and np.array_equal(got[k], a)


def test_seeded_sample_above_the_cap(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 200_000)
    want = _outputs()
    bench.dump_outputs(str(tmp_path / "a"), want)
    bench.dump_outputs(str(tmp_path / "b"), want)
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 200_000
    idx = a["gp_index"].astype(np.int64)
    assert 0 < idx.size < 400 and np.all(np.diff(idx) > 0)
    for k, v in want.items():
        assert np.array_equal(a[k], v[idx]) and np.array_equal(a[k], b[k])
