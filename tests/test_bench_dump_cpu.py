"""bench.py --dump-outputs: the filtered URLs come back exactly from the .npy files, as all rows or as a seeded sample that
keeps the files under the byte cap. No GPU needed."""
import os

import numpy as np
import pyarrow as pa
import pytest

import bench


def _load(d):
    rows, offs, data = (np.load(os.path.join(d, f"url_{k}.npy")) for k in ("rows", "offsets", "bytes"))
    assert rows.dtype == offs.dtype == np.float64 and data.dtype == np.float32
    raw, offs = data.astype(np.uint8).tobytes(), offs.astype(np.int64)
    strs = [raw[offs[i]:offs[i + 1]].decode() for i in range(len(offs) - 1)]
    return rows.astype(np.int64), strs, sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d))


@pytest.mark.parametrize("cap", [64 << 20, 50_000])
def test_dumped_urls_are_the_rows_they_name(tmp_path, monkeypatch, cap):
    monkeypatch.setattr(bench, "DUMP_BYTES", cap)
    rng = np.random.default_rng(1)
    urls = pa.array([f"http://{'x' * int(rng.integers(0, 40))}é/{i}" for i in range(5000)])
    arr = pa.concat_arrays([urls.slice(7, 3000), urls.slice(4000, 1000)])  # parts, as the gathered ranks arrive
    bench.dump_strings(str(tmp_path / "a"), "url", arr)
    rows, strs, nbytes = _load(tmp_path / "a")
    assert nbytes <= cap
    assert np.all(np.diff(rows) > 0) and strs == arr.take(pa.array(rows)).to_pylist()
    assert len(rows) == len(arr) if cap == 64 << 20 else 0 < len(rows) < len(arr)
    bench.dump_strings(str(tmp_path / "b"), "url", arr)
    for k in ("rows", "offsets", "bytes"):
        assert np.array_equal(np.load(tmp_path / "a" / f"url_{k}.npy"), np.load(tmp_path / "b" / f"url_{k}.npy"))


def test_no_matching_rows_dumps_empty_arrays(tmp_path):
    bench.dump_strings(str(tmp_path), "url", pa.array([], pa.string()))
    rows, strs, _ = _load(tmp_path)
    assert len(rows) == 0 and strs == []
