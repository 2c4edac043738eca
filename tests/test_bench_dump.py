"""bench.py --dump-outputs: the per-read results of the timed step as float npy files, a fixed seeded sample of
them when the batch is larger than DUMP_SAMPLE, within 64 MB."""
import os
import subprocess
import sys

import numpy as np

import bdx_b200 as bdx
import bench


def _results(n):
    rng = np.random.default_rng(9)
    res = np.zeros(n, bdx.RESULT_DTYPE)
    for f in res.dtype.names:
        res[f] = rng.integers(-1, 151, n)
    return res


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_dump_is_a_fixed_sample_of_the_results(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 1000)
    res = _results(5000)
    bench.dump_outputs(str(tmp_path / "a"), res)
    bench.dump_outputs(str(tmp_path / "b"), res.copy())
    a, b = _load(str(tmp_path / "a")), _load(str(tmp_path / "b"))
    assert sorted(a) == sorted(list(res.dtype.names) + ["read_index"])
    idx = a["read_index"]
    assert idx.dtype == np.float64 and len(idx) == 1000 and (np.diff(idx) > 0).all() and idx[-1] < 5000
    # spread over the whole batch, not its first reads: every fifth of it holds about a fifth of the sample
    assert (np.bincount((idx // 1000).astype(np.int64), minlength=5) > 150).all()
    for f in res.dtype.names:
        assert a[f].dtype == np.float32 and (a[f] == res[f][idx.astype(np.int64)]).all()
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def test_small_batch_is_dumped_whole(tmp_path):
    res = _results(300)
    bench.dump_outputs(str(tmp_path), res)
    got = _load(str(tmp_path))
    assert (got["read_index"] == np.arange(300)).all()
    assert all((got[f] == res[f]).all() for f in res.dtype.names)


def test_dump_size_bound():
    n_fields = len(bdx.RESULT_DTYPE.names)
    assert bench.DUMP_SAMPLE * (4 * n_fields + 8) <= 64 * 2**20


def test_bad_arguments_are_refused(tmp_path):
    """Refused while parsing, before any device is touched: no timed step, and a dump of a path that does not run."""
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "d")]):
        r = subprocess.run([sys.executable, bench.__file__, *extra], capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and "error" in r.stderr, (extra, r.stderr)
    assert not os.path.exists(tmp_path / "d")
