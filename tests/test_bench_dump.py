"""CPU: bench.py --dump-outputs writes the deflate call's result record and a fixed sample of its stream as float .npy
files that stay under 64 MB."""
import os
import zlib

import numpy as np

import bench
import zlibts_b200 as z


def _dump(path, n, rank=0, world=1):
    stream = np.random.default_rng(3).integers(0, 256, n, dtype=np.uint8)
    results = np.zeros(1, dtype=z.RESULT_DTYPE)
    results["out_len"], results["in_used"], results["blocks"] = n, 5 * n, 7
    bench.dump_outputs(str(path), stream, results, rank, world)
    return stream, results, {f: np.load(os.path.join(path, f)) for f in sorted(os.listdir(path))}


def test_short_stream_is_dumped_whole(tmp_path):
    stream, results, files = _dump(tmp_path, 1000)
    assert files["deflate_stream_index.npy"].tolist() == list(range(1000))
    assert np.array_equal(files["deflate_stream.npy"], stream.astype(np.float32))
    assert files["deflate_stream_crc32.npy"].tolist() == [zlib.crc32(stream)]
    for f in results.dtype.names:
        assert files["deflate_%s.npy" % f].tolist() == results[f].tolist(), f
    assert all(a.dtype in (np.float32, np.float64) for a in files.values())


def test_long_stream_is_sampled_the_same_way_every_time(tmp_path):
    n = bench.DUMP_SAMPLE + 654321
    stream, _, a = _dump(tmp_path / "a", n)
    _, _, b = _dump(tmp_path / "b", n)
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)
    idx = a["deflate_stream_index.npy"].astype(np.int64)
    assert idx.size == bench.DUMP_SAMPLE and idx[0] >= 0 and idx[-1] < n and np.all(np.diff(idx) > 0)
    assert np.array_equal(a["deflate_stream.npy"], stream[idx].astype(np.float32))
    assert sum(os.path.getsize(os.path.join(tmp_path, "a", f)) for f in a) <= 64 << 20


def test_ranks_write_their_own_smaller_samples(tmp_path):
    _dump(tmp_path, bench.DUMP_SAMPLE, rank=1, world=4)
    names = os.listdir(tmp_path)
    assert names and all(f.endswith("_rank1.npy") for f in names)
    assert np.load(os.path.join(tmp_path, "deflate_stream_rank1.npy")).size == bench.DUMP_SAMPLE // 4
