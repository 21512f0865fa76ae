"""GPU: ZLB_INFLATE_SPLIT on streams whose pieces share history (primed mode, zlib's Z_SYNC_FLUSH): the pieces are
decoded side by side in window mode and their windows resolved by a scan. Every case is compared with the one-warp
decoder (the same call without INFLATE_SPLIT) and with CPython's zlib; the profile slots tell which route ran."""
import zlib

import numpy as np
import pytest

from helpers import _BitWriter, pack, rand_bytes, zlib_raw

pytestmark = pytest.mark.gpu

WINDOW_KERNELS = ("inflate_warp_kernel_window", "window_run_kernel", "window_scan_kernel", "window_resolve_kernel")
FIELDS = ("status", "out_len", "in_used", "blocks", "crc32", "adler32")


def _inflate(engine, streams, caps, flags, trailer=b"\0\0\0\0"):
    """(whole output buffer, output offsets, results, kernel launches by name) of one call; the output buffer starts
    out filled with 0xA5, so whatever a route writes beyond what it reports shows."""
    import torch
    import zlibts_b200 as z
    blob, offs, lens = pack([bytes(s) + trailer for s in streams])
    ooffs = np.concatenate([[0], np.cumsum(caps)]).astype(np.uint64)
    items = z.make_items(len(streams))
    items["in_off"], items["in_len"] = offs, lens
    items["out_off"], items["out_cap"] = ooffs[:-1], caps
    d_in = torch.from_numpy(blob).cuda()
    d_out = torch.full((max(int(ooffs[-1]), 1),), 0xA5, dtype=torch.uint8, device="cuda")
    engine.profile_enable(True)
    engine.profile_reset()
    try:
        res = engine.inflate_batch(d_in, d_out, items, flags)
        prof = engine.profile_read()
    finally:
        engine.profile_enable(False)
    return d_out.cpu().numpy().tobytes(), ooffs, res, {k: v["launches"] for k, v in prof.items()}


def _compare(engine, streams, datas, caps=None, window=True):
    """Split route vs one-warp route (and CPython zlib for the valid streams); `window`: True = the window kernels
    must have run, False = they must not have, None = either. Returns the split route's results."""
    import zlibts_b200 as z
    caps = [len(d) for d in datas] if caps is None else caps
    flags = z.INFLATE_WANT_CRC32 | z.INFLATE_WANT_ADLER32
    buf1, ooffs, res1, launches = _inflate(engine, streams, caps, flags | z.INFLATE_SPLIT)
    buf0, _, res0, launches0 = _inflate(engine, streams, caps, flags)
    assert not any(launches0[k] for k in WINDOW_KERNELS)
    for i, (s, d) in enumerate(zip(streams, datas)):
        r0, r1 = res0[i], res1[i]
        if int(r0["status"]) == z.ST_OUT_OVERFLOW:   # the split route writes nothing then (out_len 0)
            assert int(r1["status"]) == z.ST_OUT_OVERFLOW, i
            continue
        for f in FIELDS:
            assert int(r1[f]) == int(r0[f]), (i, f, int(r1[f]), int(r0[f]))
        lo, hi = int(ooffs[i]), int(ooffs[i + 1])
        assert buf1[lo:hi] == buf0[lo:hi], i                         # incl. the bytes behind out_len
        if d is not None and int(r1["status"]) == 0:
            o = buf1[lo:lo + int(r1["out_len"])]
            assert o == d and zlib.decompressobj(-15).decompress(bytes(s)) == d, i
            assert int(r1["in_used"]) == len(s) and int(r1["crc32"]) == zlib.crc32(d), i
            assert int(r1["adler32"]) == zlib.adler32(d), i
    if window is not None:
        ran = [launches[k] > 0 for k in WINDOW_KERNELS]
        assert all(ran) if window else not any(ran), launches
    return res1


def _gpu_deflate(engine, data, mode, chunk_bytes=0):
    import torch
    import zlibts_b200 as z
    cap = z.deflate_bound(len(data), chunk_bytes, z.DYNAMIC, mode)
    items = z.make_items(1)
    items["in_len"], items["out_cap"] = len(data), cap
    d_z = torch.zeros(cap, dtype=torch.uint8, device="cuda")
    d_in = torch.from_numpy(np.frombuffer(data, dtype=np.uint8).copy()).cuda()
    r = engine.deflate_batch(d_in, d_z, items, chunk_bytes=chunk_bytes, mode=mode)
    assert int(r["status"][0]) == 0
    return d_z[:int(r["out_len"][0])].cpu().numpy().tobytes()


def _sync_flushed(data, interval, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, modes=(zlib.Z_SYNC_FLUSH,)):
    co = zlib.compressobj(level, zlib.DEFLATED, -15, 9, strategy)
    out = []
    for n, k in enumerate(range(0, len(data), interval)):
        out.append(co.compress(data[k:k + interval]) + co.flush(modes[n % len(modes)]))
    return b"".join(out) + co.flush()


def test_gpu_primed_streams(engine):
    import zlibts_b200 as z
    from zlibts_b200 import synth
    datas, streams = [], []
    for k, (mode, chunk, gen, size) in enumerate((
            (z.MODE_PRIMED, 32768, synth.text, 8 << 20),
            (z.MODE_PRIMED, 4096, synth.mixed, 4 << 20),
            (z.mode_fast() | z.MODE_PRIMED, 32768, synth.mixed, 16 << 20),
            (z.mode_fast() | z.MODE_PRIMED, 1500, synth.text, 4 << 20),
            (z.MODE_PRIMED | z.MODE_SMALLEST, 32768, synth.mixed, 6 << 20),
            (z.MODE_PRIMED | z.MODE_SMALLEST, 4096, synth.text, 4 << 20 | 12345))):
        d = gen(size, 700 + k).tobytes()
        datas.append(d)
        streams.append(_gpu_deflate(engine, d, mode, chunk))
    for d, s in zip(datas, streams):
        _compare(engine, [s], [d])
    _compare(engine, streams, datas)   # all in one call


def test_zlib_sync_flush_streams(engine):
    from zlibts_b200 import synth
    text = synth.text(4 << 20, 801).tobytes()
    mixed = synth.mixed(4 << 20, 802).tobytes()
    datas, streams = [], []
    for interval in (5000, 32768, 100000):
        for level, strategy in ((1, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_DEFAULT_STRATEGY), (9, zlib.Z_DEFAULT_STRATEGY),
                                (6, zlib.Z_RLE)):
            d = text if (interval + level) % 2 else mixed
            datas.append(d)
            streams.append(_sync_flushed(d, interval, level, strategy))
    _compare(engine, streams, datas)
    # full and sync flushes in one stream: independent pieces and pieces with history side by side
    d = synth.mixed(3 << 20, 803).tobytes()
    _compare(engine, [_sync_flushed(d, 40000, modes=(zlib.Z_SYNC_FLUSH, zlib.Z_FULL_FLUSH, zlib.Z_SYNC_FLUSH))], [d])
    # pieces whose output overflows the slot (128 KiB): the one-warp decoder does them, with the same results
    for interval in (200000, 1 << 20):
        _compare(engine, [_sync_flushed(text, interval)], [text], window=None)


def test_longest_chains(engine):
    """Nearly every byte of every piece comes from the previous piece: one repeated byte, and a period of 3. The split
    looks at items of at least 256 KiB of compressed input; such data compresses ~500:1 in primed mode (64 MiB of one
    byte to ~140 KiB, which one warp decodes), so the chains are 256 MiB long."""
    import zlibts_b200 as z
    for d in (b"\x61" * (256 << 20), b"xyz" * ((256 << 20) // 3)):
        s = _gpu_deflate(engine, d, z.MODE_PRIMED)
        assert len(s) >= 256 << 10, len(s)
        _compare(engine, [s], [d])


def _stored(w, data, final=False):
    for at in range(0, len(data), 65535):
        piece = data[at:at + 65535]
        w.bits(1 if final and at + 65535 >= len(data) else 0, 1)
        w.bits(0, 2)
        w.align()
        w.bits(len(piece), 16)
        w.bits(len(piece) ^ 0xFFFF, 16)
        w.buf.extend(piece)


def _stored_pieces(w, data, final=False):
    """`data` as stored blocks of at most 60 000 bytes, each followed by a sync marker (but a final last one): pieces
    that fit the split's 128 KiB slots"""
    for at in range(0, len(data), 60000):
        last = at + 60000 >= len(data)
        _stored(w, data[at:at + 60000], final=final and last)
        if not (final and last):
            _sync_marker(w)


def _sync_marker(w):
    """an empty stored block: `00 00 FF FF` after the byte alignment"""
    w.bits(0, 3)
    w.align()
    w.bits(0, 16)
    w.bits(0xFFFF, 16)


def _fixed_lit(w, v):
    if v < 144:
        w.code(0x30 + v, 8)
    elif v < 256:
        w.code(0x190 + v - 144, 9)
    elif v < 280:
        w.code(v - 256, 7)
    else:
        w.code(0xC0 + v - 280, 8)


def _fixed_match(w, out, length, dist):
    """length 3 (symbol 257) or 258 (285); distances 1..4 (codes 0..3) or 24577..32768 (code 29)."""
    assert length in (3, 258)
    _fixed_lit(w, 257 if length == 3 else 285)
    if dist <= 4:
        w.code(dist - 1, 5)
    else:
        w.code(29, 5)
        w.bits(dist - 24577, 13)
    for _ in range(length):
        out.append(out[-dist])


def _wrap(w, out, tail_bytes=0, seed=0):
    """Ends a hand-built stream: a sync marker, `tail_bytes` stored bytes, then a final empty fixed block."""
    rng = np.random.default_rng(seed)
    _sync_marker(w)
    if tail_bytes:
        t = rand_bytes(rng, tail_bytes).tobytes()
        _stored(w, t)
        out.extend(t)
    w.bits(1, 1)
    w.bits(1, 2)
    _fixed_lit(w, 256)
    return w.bytes(), bytes(out)


def test_exact_distance_at_the_first_byte(engine):
    """Stored history, a sync marker, then a block whose very first symbols copy from exactly 32768 bytes back."""
    rng = np.random.default_rng(21)
    hist = rand_bytes(rng, 300000).tobytes()
    w, out = _BitWriter(), bytearray(hist)
    _stored_pieces(w, hist)
    w.bits(0, 1)
    w.bits(1, 2)
    for k in range(300):
        _fixed_match(w, out, 258 if k % 3 else 3, 32768)
        if k % 7 == 0:
            _fixed_lit(w, k % 256)
            out.append(k % 256)
    _fixed_match(w, out, 258, 1)
    _fixed_lit(w, 256)
    s, d = _wrap(w, out)
    assert zlib.decompressobj(-15).decompress(s) == d
    _compare(engine, [s], [d])


def test_invalid_streams_fall_back(engine):
    """Each gives the one-warp decoder's status, out_len and bytes, and nothing else is written."""
    import zlibts_b200 as z
    from zlibts_b200 import synth
    rng = np.random.default_rng(22)
    streams, datas = [], []
    # a later piece reaches before the start of the stream (1000 bytes, then a match 24577 back): its pieces pass the
    # chain checks in window mode, the resolve pass finds the byte before the stream
    w, out = _BitWriter(), bytearray(rand_bytes(rng, 1000).tobytes())
    _stored(w, bytes(out))
    _sync_marker(w)
    w.bits(0, 1)
    w.bits(1, 2)
    for k in range(40):
        _fixed_lit(w, 65 + k % 26)
    _fixed_lit(w, 285)
    w.code(29, 5)
    w.bits(0, 13)
    _fixed_lit(w, 256)
    _sync_marker(w)
    _stored_pieces(w, rand_bytes(rng, 300000).tobytes(), final=True)
    streams.append(w.bytes())
    datas.append(None)
    # truncations of a primed stream (inside a piece, inside a marker, the last byte)
    d = synth.text(2 << 20, 23).tobytes()
    s = _gpu_deflate(engine, d, z.MODE_PRIMED)
    m = s.find(b"\x00\x00\xff\xff", len(s) // 2)
    for cut in (len(s) // 2, m + 2, len(s) - 1):
        streams.append(s[:cut])
        datas.append(None)
    # false markers inside stored payload, between pieces that share history
    parts = []
    for k in range(48):
        if k % 3 == 2:
            parts.append(b"".join(rand_bytes(rng, 3000).tobytes() + b"\x00\x00\xff\xff" for _ in range(5)))
        else:
            parts.append(synth.text(20000, 30 + k).tobytes())
    d = b"".join(parts)
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    streams.append(b"".join(co.compress(p) + co.flush(zlib.Z_SYNC_FLUSH) for p in parts) + co.flush())
    datas.append(d)
    res = _compare(engine, streams, datas, caps=[4 << 20] * len(streams), window=True)
    assert int(res["status"][0]) == z.ST_BAD_CODE and int(res["out_len"][0]) == 1040
    assert int(res["status"][4]) == 0


def test_mixed_batch_with_one_undersized_slot(engine):
    import zlibts_b200 as z
    from zlibts_b200 import synth
    rng = np.random.default_rng(24)
    datas, streams = [], []
    for k in range(8):
        d = synth.mixed(400000 + 50000 * k, 900 + k).tobytes()
        kind = k % 4
        if kind == 0:
            s = _gpu_deflate(engine, d, z.MODE_PRIMED)
        elif kind == 1:
            s = _sync_flushed(d, 30000)
        elif kind == 2:
            s = _gpu_deflate(engine, d, z.MODE_COMPAT)
        else:
            d = rand_bytes(rng, 3000, 5).tobytes()
            s = zlib_raw(d)
        datas.append(d)
        streams.append(s)
    _compare(engine, streams, datas)
    caps = [len(d) for d in datas]
    caps[4] -= 1                          # a primed item (window route)
    res = _compare(engine, streams, datas, caps=caps)
    assert [int(r["status"]) for r in res] == [z.ST_OUT_OVERFLOW if k == 4 else 0 for k in range(len(datas))]


def test_compat_streams_keep_todays_route(engine):
    import zlibts_b200 as z
    from zlibts_b200 import synth
    d = synth.mixed(6 << 20, 31).tobytes()
    full = _sync_flushed(d, 65536, modes=(zlib.Z_FULL_FLUSH,))
    _compare(engine, [_gpu_deflate(engine, d, z.MODE_COMPAT), full], [d, d], window=False)


def test_host_entry_point_pinned_and_pageable(engine):
    """The host entry point on a mixed batch -- large primed, compat, Z_SYNC_FLUSH and invalid items beside a few
    thousand small streams -- without and with dictionaries, through page-locked and pageable buffers: the same results
    and the same bytes, the slack included, as the call without INFLATE_SPLIT."""
    import zlibts_b200 as z
    from zlibts_b200 import synth
    rng = np.random.default_rng(43)
    zd = synth.text(32768, 40).tobytes()
    big = [synth.text(3 << 20, 41).tobytes(), synth.mixed(4 << 20, 44).tobytes(), synth.mixed(5 << 20, 42).tobytes()]
    small = [synth.text(int(n), 1000 + k).tobytes() for k, n in enumerate(rng.integers(1, 3000, 3000))]
    fixed = [_gpu_deflate(engine, big[0], z.MODE_PRIMED), _gpu_deflate(engine, big[1], z.MODE_COMPAT)]
    base = z.INFLATE_WANT_CRC32 | z.INFLATE_WANT_ADLER32
    for with_dicts in (False, True):
        # with dictionaries: the zlib streams (the Z_SYNC_FLUSH one, the invalid one and every other small one) have one
        has = [False, False, with_dicts, with_dicts] + [with_dicts and k % 2 == 0 for k in range(len(small))]
        co = zlib.compressobj(6, zlib.DEFLATED, -15, 9, zlib.Z_DEFAULT_STRATEGY, *([zd] if with_dicts else []))
        sync = b"".join(co.compress(big[2][k:k + 50000]) + co.flush(zlib.Z_SYNC_FLUSH)
                        for k in range(0, len(big[2]), 50000)) + co.flush()
        streams = fixed + [sync, sync[:len(sync) // 2]]
        for d, h in zip(small, has[4:]):
            co = zlib.compressobj(6, zlib.DEFLATED, -15, 9, zlib.Z_DEFAULT_STRATEGY, *([zd] if h else []))
            streams.append(co.compress(d) + co.flush())
        datas = big + [None] + small
        assert all(len(s) >= 256 << 10 for s in streams[:4])
        blob, offs, lens = pack(streams)
        caps = [len(big[0]) + 100, len(big[1]) + 100, len(big[2]) + 100, len(big[2])]
        caps += [len(d) + (5 if k % 500 == 0 else 0) for k, d in enumerate(small)]
        ooffs = np.concatenate([[0], np.cumsum(caps)]).astype(np.uint64)
        items = z.make_items(len(streams))
        items["in_off"], items["in_len"], items["out_off"], items["out_cap"] = offs, lens, ooffs[:-1], caps
        h_dict, table = np.frombuffer(zd, dtype=np.uint8).copy(), z.make_dicts(len(streams))
        table["len"] = [len(zd) if h else 0 for h in has]
        for pinned in (True, False):
            runs = []
            for flags in (base | z.INFLATE_SPLIT, base):
                if pinned:
                    h_in, h_out = z.host_alloc(blob.size), z.host_alloc(int(ooffs[-1]))
                    h_in[:] = blob
                else:
                    h_in, h_out = blob.copy(), np.empty(int(ooffs[-1]), dtype=np.uint8)
                h_out[:] = 0xA5
                engine.profile_enable(True)
                engine.profile_reset()
                try:
                    res = engine.inflate_batch_host(h_in, h_out, items, flags, *((h_dict, table) if with_dicts else ()))
                    prof = engine.profile_read()
                finally:
                    engine.profile_enable(False)
                runs.append((res, h_out.tobytes(), prof))
                if pinned:
                    z.host_free(h_in)
                    z.host_free(h_out)
            (res, out, prof), (res0, out0, prof0) = runs
            assert all(prof[k]["launches"] > 0 for k in WINDOW_KERNELS), prof
            assert not any(prof0[k]["launches"] for k in WINDOW_KERNELS), prof0
            assert res.tobytes() == res0.tobytes() and out == out0
            assert int(res["status"][3]) != 0
            for i, (d, s, r) in enumerate(zip(datas, streams, res)):
                if d is None:
                    continue
                assert int(r["status"]) == 0 and int(r["out_len"]) == len(d) and int(r["in_used"]) == len(s), i
                assert out[int(ooffs[i]):int(ooffs[i]) + len(d)] == d, i
                assert int(r["crc32"]) == zlib.crc32(d) and int(r["adler32"]) == zlib.adler32(d), i


def test_host_api_primed_round_trips(engine):
    import gzip
    import zlibts_b200 as Z
    from zlibts_b200 import synth
    Z.api.set_engine(engine)
    d = synth.text(6 << 20, 51).tobytes()
    engine.profile_enable(True)
    try:
        engine.profile_reset()
        g = Z.GZip(d, {"deflateOptions": {"b200": {"mode": "primed"}}}).compress().tobytes()
        assert gzip.decompress(g) == d
        engine.profile_reset()
        assert Z.GUnzip(g).decompress().tobytes() == d
        prof = engine.profile_read()
        assert all(prof[k]["launches"] > 0 for k in WINDOW_KERNELS), prof
        c = Z.Deflate(d, {"b200": {"mode": "primed"}}).compress().tobytes()
        assert zlib.decompress(c) == d
        engine.profile_reset()
        assert Z.Inflate(c, {"verify": True}).decompress().tobytes() == d
        prof = engine.profile_read()
        assert all(prof[k]["launches"] > 0 for k in WINDOW_KERNELS), prof
    finally:
        engine.profile_enable(False)


def test_repeats_are_identical_and_scratch_is_bounded(engine):
    import torch
    import zlibts_b200 as z
    from zlibts_b200 import synth
    d = synth.mixed(8 << 20, 61).tobytes()
    s = _gpu_deflate(engine, d, z.mode_fast() | z.MODE_PRIMED)
    runs = [_inflate(engine, [s], [len(d)], z.INFLATE_SPLIT | z.INFLATE_WANT_CRC32) for _ in range(3)]
    for buf, _, res, launches in runs:
        assert buf == runs[0][0] and buf == d and launches["window_resolve_kernel"] > 0
        assert res.tobytes() == runs[0][2].tobytes()
    # many short pieces that each reach into their predecessors: the scratch stays within its bound (byte slots:
    # 2048 x the input; window mode: 3 x that), it does not grow with the number of pieces alone
    t = synth.text(2 << 20, 62).tobytes()
    s = _sync_flushed(t, 300)
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info()
    _compare(engine, [s], [t], window=None)
    free1, _ = torch.cuda.mem_get_info()
    assert free0 - free1 < 4 * 2048 * len(s) + (256 << 20), (free0 - free1, len(s))
