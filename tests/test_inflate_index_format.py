"""CPU: the serialized form of an InflateIndex (versioned header, points, windows) and the checks that need no GPU."""
import numpy as np
import pytest


def _index():
    import zlibts_b200 as Z
    pts = np.zeros(3, dtype=Z.POINT_DTYPE)
    pts["in_bit"] = [0, 80003, 160101]
    pts["out_pos"] = [0, 1 << 20, 2 << 20]
    pts["win_off"] = [0, 0, 32768]
    wins = (np.arange(65536) * 7 % 251).astype(np.uint8)
    return Z.InflateIndex("gzip", 10, 123456, 123438, 3 << 20, 1 << 20, pts, wins)


def test_round_trip():
    import zlibts_b200 as Z
    idx = _index()
    b = idx.to_bytes()
    assert len(b) == idx.nbytes == 72 + 3 * 24 + 65536
    back = Z.InflateIndex.from_bytes(b)
    assert back.to_bytes() == b
    assert (back.kind, back.start, back.data_len, back.deflate_len, back.size, back.spacing) == \
        ("gzip", 10, 123456, 123438, 3 << 20, 1 << 20)
    assert back.points.tobytes() == idx.points.tobytes() and back.windows.tobytes() == idx.windows.tobytes()
    assert len(back) == 3


def test_refusals():
    import zlibts_b200 as Z
    b = _index().to_bytes()
    with pytest.raises(Z.ZlibError, match="not an inflate index"):
        Z.InflateIndex.from_bytes(b"x" + b[1:])
    with pytest.raises(Z.ZlibError, match="not an inflate index"):
        Z.InflateIndex.from_bytes(b[:20])
    with pytest.raises(Z.ZlibError, match="unsupported inflate index version: 2"):
        Z.InflateIndex.from_bytes(b[:8] + b"\x02" + b[9:])
    with pytest.raises(Z.ZlibError, match="corrupt"):
        Z.InflateIndex.from_bytes(b[:-1])
    with pytest.raises(Z.ZlibError, match="unknown index kind"):
        Z.inflate_index(b"", "zip")
    # data of another length is refused before anything reaches the GPU
    with pytest.raises(Z.ZlibError, match="does not belong to this index"):
        _index().read(bytes(100), 0, 10)
    with pytest.raises(Z.ZlibError, match="negative"):
        _index().read(bytes(123456), -1, 10)
