"""GPU: zlb_inflate_size_batch[_host] -- decompressed sizes without writing the bytes. Every size result must equal,
field by field (status, out_len, in_used, blocks), what the decoder returns for the same item, flags and dictionary
with out_cap = that size, on both routes (with and without ZLB_INFLATE_SPLIT); the sizes are exact slots (size - 1
overflows); the profile slots tell which kernels a size call ran."""
import json
import os
import zlib

import numpy as np
import pytest

import oracle
from helpers import _BitWriter, pack, rand_bytes, zlib_raw
from test_dictionary_gpu import _expand, _fixed_block, _hand_stream
from test_split_window_gpu import _gpu_deflate, _stored, _stored_pieces, _sync_flushed, _sync_marker

pytestmark = pytest.mark.gpu

FIELDS = ("status", "out_len", "in_used", "blocks")
WINDOW_KERNELS = ("inflate_warp_kernel_window", "window_run_kernel", "window_scan_kernel", "window_resolve_kernel")


def _dict_blob(dicts):
    import zlibts_b200 as z
    table = z.make_dicts(len(dicts))
    parts, at = [], 0
    for i, d in enumerate(dicts):
        if d:
            table[i] = (at, len(d))
            parts.append(d)
            at += len(d)
    return np.frombuffer(b"".join(parts) or b"\0", dtype=np.uint8).copy(), table


def _profiled(engine, fn):
    engine.profile_enable(True)
    engine.profile_reset()
    try:
        out = fn()
        prof = engine.profile_read()
    finally:
        engine.profile_enable(False)
    return out, {k: v["launches"] for k, v in prof.items()}


def _check(engine, streams, dicts=None, flags=0, trailer=b"\0\0\0\0"):
    """Size calls with and without ZLB_INFLATE_SPLIT against the decoder on both routes with out_cap = the size; then
    size - 1 for every valid non-empty item. Returns (size results, launches of the split size call)."""
    import torch
    import zlibts_b200 as z
    blob, offs, lens = pack([bytes(s) + trailer for s in streams])
    n = len(streams)
    items = z.make_items(n)
    items["in_off"], items["in_len"] = offs, lens
    items["out_off"], items["out_cap"] = 12345, 1            # ignored by a size call
    table, d_dict = None, None
    if dicts is not None:
        dblob, table = _dict_blob(dicts)
        d_dict = torch.from_numpy(dblob).cuda()
    d_in = torch.from_numpy(blob).cuda()
    sizes, launches = _profiled(engine, lambda: engine.inflate_size_batch(d_in, items, flags | z.INFLATE_SPLIT, table))
    sizes0 = engine.inflate_size_batch(d_in, items, flags, table)
    assert sizes.tobytes() == sizes0.tobytes()
    assert int(sizes["crc32"].max(initial=0)) == 0 and int(sizes["adler32"].max(initial=0)) == 0
    assert not any(int(s) == z.ST_OUT_OVERFLOW for s in sizes["status"])
    caps = sizes["out_len"].astype(np.uint64)
    ooffs = np.concatenate([[0], np.cumsum(caps)]).astype(np.uint64)
    items["out_off"], items["out_cap"] = ooffs[:-1], caps
    d_out = torch.zeros(max(int(ooffs[-1]), 1), dtype=torch.uint8, device="cuda")
    for route in (0, z.INFLATE_SPLIT):
        res = engine.inflate_batch(d_in, d_out, items, flags | route, d_dict, table)
        for i in range(n):
            for f in FIELDS:
                assert int(sizes[i][f]) == int(res[i][f]), (i, route, f, int(sizes[i][f]), int(res[i][f]))
    short = [i for i in range(n) if int(sizes["status"][i]) == 0 and int(caps[i]) > 0]
    if short:
        items["out_cap"][short] -= 1
        res = engine.inflate_batch(d_in, d_out, items, flags, d_dict, table)
        assert all(int(res["status"][i]) == z.ST_OUT_OVERFLOW for i in short)
    return sizes, launches


def test_reference_and_zlib_streams(engine):
    from zlibts_b200 import synth
    rng = np.random.default_rng(101)
    datas = [b"", b"a", b"abcabcabcabc", bytes(range(256)), synth.text(65536, 1).tobytes(), synth.mixed(65536, 2).tobytes()]
    streams = [oracle.raw_deflate(d, ct) for ct in (oracle.DYNAMIC, oracle.FIXED, oracle.NONE) for d in datas if d]
    for _ in range(400):
        d = rand_bytes(rng, int(rng.integers(0, 4000)), int(rng.choice([1, 3, 16, 256]))).tobytes()
        level = int(rng.choice([0, 1, 6, 9]))
        strategy = int(rng.choice([zlib.Z_DEFAULT_STRATEGY, zlib.Z_FIXED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE]))
        streams.append(zlib_raw(d, level, strategy))
    streams += [zlib_raw(synth.mixed(1 << 20, 3).tobytes(), 6), zlib_raw(b"0123456789abcdef" * 40000, 1)]
    sizes, _ = _check(engine, streams)
    assert int(sizes["status"].max()) == 0


def test_every_status_with_and_without_check_nlen(engine):
    import zlibts_b200 as z
    vec = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "truncation_vectors.json")))["vectors"]
    streams = [bytes.fromhex(v["stream"])[:cut] for v in vec for cut in range(len(v["cuts"]))]
    good = zlib_raw(b"hello hello hello hello hello", 6)
    streams += [b"\x07\x00\x00",                                  # BTYPE 3
                bytes([0b00000011, 0b00000010, 0, 0]),            # a distance before the start of the output
                b"\x01\x05\x00\x00\x00abcde",                     # stored block, NLEN != ~LEN
                b"\x01\x05\x00\xfa",                              # stored block cut inside NLEN
                good[:3], good]
    for flags in (0, z.INFLATE_CHECK_NLEN):
        sizes, _ = _check(engine, streams, flags=flags, trailer=b"")
        seen = {int(s) & 0xFF for s in sizes["status"]} | {int(s) for s in sizes["status"]}
        for st in (z.ST_OK, z.ST_INPUT_BROKEN, z.ST_BTYPE, z.ST_CODE_LENGTH, z.ST_STORED_LEN, z.ST_STORED_LEN | 1 << 8,
                   z.ST_BAD_CODE):
            assert st in seen, (flags, st)
        assert any((int(s) & 0xFF) == z.ST_CODE_LENGTH and int(s) >> 8 for s in sizes["status"])
        nlen = int(sizes["status"][len(streams) - 4])
        assert nlen == (z.ST_STORED_LEN if flags else z.ST_OK), nlen


def test_gpu_streams_in_every_mode_and_sync_flushes(engine):
    import zlibts_b200 as z
    from zlibts_b200 import synth
    streams = []
    for k, (mode, chunk) in enumerate(((z.MODE_COMPAT, 0), (z.mode_fast(), 0), (z.MODE_PRIMED, 32768),
                                       (z.MODE_PRIMED, 4096), (z.mode_fast() | z.MODE_PRIMED, 1500),
                                       (z.MODE_SMALLEST, 0), (z.MODE_PRIMED | z.MODE_SMALLEST, 32768))):
        d = (synth.text if k % 2 else synth.mixed)((3 << 20) + 1000 * k, 200 + k).tobytes()
        streams.append(_gpu_deflate(engine, d, mode, chunk))
    text = synth.text(4 << 20, 210).tobytes()
    for interval, level, strategy in ((5000, 1, zlib.Z_DEFAULT_STRATEGY), (32768, 6, zlib.Z_DEFAULT_STRATEGY),
                                      (100000, 9, zlib.Z_DEFAULT_STRATEGY), (40000, 6, zlib.Z_RLE)):
        streams.append(_sync_flushed(text, interval, level, strategy))
    streams.append(_sync_flushed(text, 40000, modes=(zlib.Z_SYNC_FLUSH, zlib.Z_FULL_FLUSH)))
    streams.append(_sync_flushed(text, 1 << 20))                  # pieces larger than the decode split's slots
    assert all(len(s) >= 256 << 10 for s in streams)
    sizes, launches = _check(engine, streams)
    assert int(sizes["status"].max()) == 0
    assert launches["marker_scan_kernel"] > 0 and not any(launches[k] for k in WINDOW_KERNELS)
    assert launches["segment_gather_kernel"] == 0 and launches["inflate_warp_kernel"] == 0
    assert launches["inflate_warp_kernel_size"] == 1                # every item settled by the split


def test_dictionaries_on_both_routes(engine):
    import torch
    import zlibts_b200 as z
    from zlibts_b200 import synth
    rng = np.random.default_rng(102)
    zd = synth.text(32768, 103).tobytes()
    dd = rand_bytes(rng, 1000).tobytes()
    tail = rand_bytes(rng, 300000).tobytes()
    streams, dicts = [], []
    # CPython zdict streams, small and sync-flushed ones the split cuts
    for k in range(40):
        d = synth.text(int(rng.integers(1, 5000)), 110 + k).tobytes()
        co = zlib.compressobj(6, zlib.DEFLATED, -15, 9, zlib.Z_DEFAULT_STRATEGY, zd)
        streams.append(co.compress(d) + co.flush())
        dicts.append(zd)
    big = synth.text(3 << 20, 104).tobytes()
    for interval in (30000, 100000):
        co = zlib.compressobj(6, zlib.DEFLATED, -15, 9, zlib.Z_DEFAULT_STRATEGY, zd)
        streams.append(b"".join(co.compress(big[k:k + interval]) + co.flush(zlib.Z_SYNC_FLUSH)
                                for k in range(0, len(big), interval)) + co.flush())
        dicts.append(zd)
    # hand-built: a distance exactly at the dictionary's first usable byte, and one beyond it; 32768 at byte 0
    for toks, dic in (([1, 2, 3, 4, 5, (10, 1005)], dd), ([1, 2, 3, 4, 5, (10, 1006)], dd),
                      ([(258, 32768), (258, 32768)], zd), ([(3, 32768)] + [(258, 1)] * 3 + [(7, 32768)], zd)):
        for t in (None, tail):
            streams.append(_hand_stream(toks, t))
            dicts.append(dic)
    # GPU dictionary deflate, primed and not
    for mode in (z.MODE_COMPAT, z.MODE_PRIMED):
        d = synth.mixed(2 << 20, 105 + mode).tobytes()
        dblob, table = _dict_blob([zd])
        cap = z.deflate_bound(len(d), 0, z.DYNAMIC, mode, True)
        items = z.make_items(1)
        items["in_len"], items["out_cap"] = len(d), cap
        d_z = torch.zeros(cap, dtype=torch.uint8, device="cuda")
        r = engine.deflate_batch(torch.from_numpy(np.frombuffer(d, dtype=np.uint8).copy()).cuda(), d_z, items,
                                 mode=mode, d_dict=torch.from_numpy(dblob).cuda(), dicts=table)
        streams.append(d_z[:int(r["out_len"][0])].cpu().numpy().tobytes())
        dicts.append(zd)
    streams.append(zlib_raw(tail, 6))                              # an item without a dictionary in the same call
    dicts.append(None)
    sizes, _ = _check(engine, streams, dicts)
    st = [int(s) for s in sizes["status"]]
    h = 42                                                         # first hand-built stream
    assert st[h] == st[h + 1] == 0 and st[h + 2] == st[h + 3] == z.ST_BAD_CODE
    assert int(sizes["out_len"][h + 2]) == int(sizes["out_len"][h + 3]) == 5
    assert st[:h] == [0] * h and st[h + 4:] == [0] * (len(st) - h - 4)
    assert int(sizes["out_len"][h + 1]) == len(_expand(dd, [1, 2, 3, 4, 5, (10, 1005)])) + len(tail)


def test_invalid_split_cases_fall_back(engine):
    """A false marker, a later piece that reaches before the stream, one that reaches exactly to byte 0, truncations:
    each equals the decoder."""
    import zlibts_b200 as z
    from zlibts_b200 import synth
    rng = np.random.default_rng(106)
    streams = []
    hist = rand_bytes(rng, 1000).tobytes()
    lits = [65 + k % 26 for k in range(40)]
    for dist in (1040, 1041, 24577):
        w = _BitWriter()
        _stored(w, hist)
        _sync_marker(w)
        _fixed_block(w, lits + [(258, dist)], False)
        _sync_marker(w)
        _stored_pieces(w, rand_bytes(rng, 300000).tobytes(), final=True)
        streams.append(w.bytes())
    d = synth.text(2 << 20, 107).tobytes()
    s = _gpu_deflate(engine, d, z.MODE_PRIMED)
    m = s.find(b"\x00\x00\xff\xff", len(s) // 2)
    streams += [s[:len(s) // 2], s[:m + 2], s[:-1]]
    parts = []
    for k in range(48):
        if k % 3 == 2:
            parts.append(b"".join(rand_bytes(rng, 3000).tobytes() + b"\x00\x00\xff\xff" for _ in range(5)))
        else:
            parts.append(synth.text(20000, 130 + k).tobytes())
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    streams.append(b"".join(co.compress(p) + co.flush(zlib.Z_SYNC_FLUSH) for p in parts) + co.flush())
    sizes, launches = _check(engine, streams)
    st = [int(x) for x in sizes["status"]]
    assert st[0] == 0 and st[1] == st[2] == z.ST_BAD_CODE and st[-1] == 0 and all(st[3:6])
    assert int(sizes["out_len"][1]) == 1040 and int(sizes["out_len"][-1]) == len(b"".join(parts))
    assert launches["inflate_warp_kernel_size"] == 2              # the pieces, then the items that fell back


def test_mixed_batch_large_invalid_and_many_small(engine):
    import zlibts_b200 as z
    from zlibts_b200 import synth
    rng = np.random.default_rng(108)
    big = [synth.mixed(3 << 20, 109).tobytes(), synth.text(3 << 20, 110).tobytes()]
    streams = [_gpu_deflate(engine, big[0], z.MODE_PRIMED), _gpu_deflate(engine, big[1], z.MODE_COMPAT),
               _sync_flushed(big[1], 50000)]
    streams.append(streams[0][:len(streams[0]) // 2])
    for k in range(3000):
        d = synth.text(int(rng.integers(0, 3000)), 2000 + k).tobytes()
        streams.append(zlib_raw(d, int(rng.choice([1, 6, 9]))))
    streams.insert(100, b"\x07\x00\x00")
    sizes, launches = _check(engine, streams)
    st = [int(x) for x in sizes["status"]]
    assert st[:3] == [0, 0, 0] and st[3] != 0 and st[100] == z.ST_BTYPE
    assert sum(1 for x in st if x) == 2
    assert int(sizes["out_len"][0]) == len(big[0]) and int(sizes["out_len"][2]) == len(big[1])


def test_route_of_a_256_mib_primed_stream(engine):
    import torch
    import zlibts_b200 as z
    from zlibts_b200 import synth
    d_in = torch.from_numpy(synth.mixed(256 << 20, 1)).cuda()
    cap = z.deflate_bound(d_in.numel(), 0, z.DYNAMIC, z.MODE_PRIMED)
    items = z.make_items(1)
    items["in_len"], items["out_cap"] = d_in.numel(), cap
    d_z = torch.empty(cap, dtype=torch.uint8, device="cuda")
    r = engine.deflate_batch(d_in, d_z, items, mode=z.MODE_PRIMED)
    items["in_len"] = int(r["out_len"][0])
    res, launches = _profiled(engine, lambda: engine.inflate_size_batch(d_z, items, z.INFLATE_SPLIT))
    assert int(res["status"][0]) == 0 and int(res["out_len"][0]) == 256 << 20
    assert int(res["in_used"][0]) == int(r["out_len"][0])
    assert launches["marker_scan_kernel"] > 0 and launches["inflate_warp_kernel_size"] == 1
    assert not any(launches[k] for k in WINDOW_KERNELS + ("segment_gather_kernel", "inflate_warp_kernel"))
    d_out = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    items["out_cap"] = 256 << 20
    ref = engine.inflate_batch(d_z, d_out, items, z.INFLATE_SPLIT)
    assert all(int(res[0][f]) == int(ref[0][f]) for f in FIELDS) and torch.equal(d_out, d_in)


@pytest.mark.parametrize("pinned", [False, True])
def test_host_entry_point(engine, pinned):
    import torch
    import zlibts_b200 as z
    from zlibts_b200 import synth
    zd = synth.text(20000, 111).tobytes()
    big = synth.mixed(3 << 20, 112).tobytes()
    co = zlib.compressobj(6, zlib.DEFLATED, -15, 9, zlib.Z_DEFAULT_STRATEGY, zd)
    sync = b"".join(co.compress(big[k:k + 50000]) + co.flush(zlib.Z_SYNC_FLUSH) for k in range(0, len(big), 50000))
    sync += co.flush()
    streams = [_gpu_deflate(engine, big, z.MODE_PRIMED), sync, sync[:len(sync) // 3]]
    streams += [zlib_raw(synth.text(1000 + k, 300 + k).tobytes()) for k in range(500)]
    blob, offs, lens = pack(streams)
    items = z.make_items(len(streams))
    items["in_off"], items["in_len"] = offs, lens
    table = z.make_dicts(len(streams))
    table["len"][1:3] = len(zd)
    if pinned:
        h_in = z.host_alloc(blob.size)
        h_in[:] = blob
    else:
        h_in = blob.copy()
    try:
        for flags in (z.INFLATE_SPLIT, 0):
            for dicts in (table, None):
                host = engine.inflate_size_batch_host(h_in, items, flags, dicts)
                dev = engine.inflate_size_batch(torch.from_numpy(blob).cuda(), items, flags, dicts)
                assert host.tobytes() == dev.tobytes()
                st = [int(s) for s in host["status"]]
                assert st[0] == 0 and st[2] != 0 and (st[1] == 0 or dicts is None)
    finally:
        if pinned:
            z.host_free(h_in)
    _check(engine, streams, [None, zd, zd] + [None] * 500)


def test_refusals(engine):
    import torch
    import zlibts_b200 as z
    items = z.make_items(1)
    items["in_len"] = 10
    d_in = torch.zeros(16, dtype=torch.uint8, device="cuda")
    for flags in (z.INFLATE_WANT_CRC32, z.INFLATE_WANT_ADLER32 | z.INFLATE_SPLIT):
        with pytest.raises(z.EngineError, match="checksum"):
            engine.inflate_size_batch(d_in, items, flags)
        with pytest.raises(z.EngineError, match="checksum"):
            engine.inflate_size_batch_host(np.zeros(16, dtype=np.uint8), items, flags)
    with pytest.raises(z.EngineError, match="NULL"):
        engine.inflate_size_batch(None, items)
    with pytest.raises(z.EngineError, match="NULL"):
        engine.inflate_size_batch_host(None, items)
    with pytest.raises(z.EngineError, match="out of range"):
        engine.inflate_size_batch_host(np.zeros(9, dtype=np.uint8), items)
    assert len(engine.inflate_size_batch(None, z.make_items(0))) == 0


def test_api_sizes_make_one_decode_call(engine):
    import zlibts_b200 as Z
    from zlibts_b200 import synth
    Z.api.set_engine(engine)
    zd = synth.text(4096, 113).tobytes()
    recs = [(synth.text(200, 400 + k).tobytes() * 40) for k in range(300)]   # ratio >= 20: 4 x the input overflows
    bufs = [zlib_raw(r, 9) for r in recs]
    co = zlib.compressobj(6, zlib.DEFLATED, -15, 9, zlib.Z_DEFAULT_STRATEGY, zd)
    bufs.append(b"\xaa" * 3 + co.compress(recs[0]) + co.flush())
    sizes = Z.inflate_sizes(bufs, indices=[0] * 300 + [3], dictionary=[None] * 300 + [zd])
    assert sizes.dtype == np.uint64 and list(sizes) == [len(r) for r in recs] + [len(recs[0])]
    calls = []
    real = engine.inflate_batch_host
    engine.inflate_batch_host = lambda *a, **k: calls.append(1) or real(*a, **k)
    try:
        outs, _ = Z.inflate_many(bufs, [0] * 300 + [3], size_hints=sizes, dictionary=[None] * 300 + [zd])
    finally:
        del engine.inflate_batch_host
    assert len(calls) == 1 and [o.tobytes() for o in outs] == recs + [recs[0]]
    bad = [bufs[0], b"\x07\x00\x00"]
    with pytest.raises(Z.ZlibError) as want:
        Z.inflate_many(bad)
    with pytest.raises(Z.ZlibError) as got:
        Z.inflate_sizes(bad)
    assert str(got.value) == str(want.value) == "unknown BTYPE: 3"
