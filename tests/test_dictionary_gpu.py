"""GPU: preset dictionaries (zlb_deflate_batch_dict / zlb_inflate_batch_dict and their host forms, RFC 1950 FDICT in
Deflate / Inflate). Deflate blocks are compared with the oracle's block construction run with the dictionary as
history (zo_raw_deflate_dict); every stream is read back by CPython's zlib with the same zdict and by the GPU; streams
CPython writes with a zdict are decoded on both inflate routes, which must agree with each other field by field."""
import zlib

import numpy as np
import pytest

from helpers import _BitWriter, pack, rand_bytes

pytestmark = pytest.mark.gpu

FIELDS = ("status", "out_len", "in_used", "blocks", "crc32", "adler32")
WINDOW_KERNELS = ("inflate_warp_kernel_window", "window_run_kernel", "window_scan_kernel", "window_resolve_kernel")


def _dict_blob(dicts):
    """(blob, zlb_dict table) of a list of dictionaries (bytes; None or b'' = none)."""
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


def _deflate(engine, datas, dicts, btype=2, mode=0, chunk=0, flags=0):
    """Device entry point; returns (outputs, results, kernel launches)."""
    import torch
    import zlibts_b200 as z
    blob, offs, lens = pack(datas)
    dblob, table = _dict_blob(dicts)
    caps = [z.deflate_bound(len(d), chunk, btype, mode, True) for d in datas]
    ooffs = np.concatenate([[0], np.cumsum(caps)]).astype(np.uint64)
    items = z.make_items(len(datas))
    items["in_off"], items["in_len"], items["out_off"], items["out_cap"] = offs, lens, ooffs[:-1], caps
    d_out = torch.zeros(int(ooffs[-1]), dtype=torch.uint8, device="cuda")
    d_in, d_dict = torch.from_numpy(blob).cuda(), torch.from_numpy(dblob).cuda()
    res, launches = _profiled(engine, lambda: engine.deflate_batch(d_in, d_out, items, btype, chunk, flags, mode,
                                                                   d_dict, table))
    h = d_out.cpu().numpy()
    outs = [h[int(o):int(o) + int(r["out_len"])].tobytes() for o, r in zip(ooffs[:-1], res)]
    assert int(res["status"].max()) == 0
    return outs, res, launches


def _inflate(engine, streams, caps, dicts, flags=0, trailer=b"\0\0\0\0"):
    """Device entry point; the output starts out filled with 0xA5. Returns (buffer, offsets, results, launches)."""
    import torch
    import zlibts_b200 as z
    blob, offs, lens = pack([bytes(s) + trailer for s in streams])
    dblob, table = _dict_blob(dicts)
    ooffs = np.concatenate([[0], np.cumsum(caps)]).astype(np.uint64)
    items = z.make_items(len(streams))
    items["in_off"], items["in_len"], items["out_off"], items["out_cap"] = offs, lens, ooffs[:-1], caps
    d_in, d_dict = torch.from_numpy(blob).cuda(), torch.from_numpy(dblob).cuda()
    d_out = torch.full((max(int(ooffs[-1]), 1),), 0xA5, dtype=torch.uint8, device="cuda")
    res, launches = _profiled(engine, lambda: engine.inflate_batch(d_in, d_out, items, flags, d_dict, table))
    return d_out.cpu().numpy().tobytes(), ooffs, res, launches


def _roundtrip(engine, streams, datas, dicts):
    """Every stream decodes with CPython (same zdict) and with the GPU dictionary inflate."""
    import zlibts_b200 as z
    for s, d, dd in zip(streams, datas, dicts):
        do = zlib.decompressobj(-15, zdict=dd) if dd else zlib.decompressobj(-15)
        assert do.decompress(s) == d
    buf, ooffs, res, launches = _inflate(engine, streams, [len(d) + 8 for d in datas], dicts,
                                         z.INFLATE_WANT_CRC32 | z.INFLATE_WANT_ADLER32)
    for i, (s, d) in enumerate(zip(streams, datas)):
        r = res[i]
        assert int(r["status"]) == 0 and int(r["out_len"]) == len(d) and int(r["in_used"]) == len(s), i
        assert buf[int(ooffs[i]):int(ooffs[i]) + len(d)] == d, i
        assert int(r["crc32"]) == zlib.crc32(d) and int(r["adler32"]) == zlib.adler32(d), i
    assert launches["inflate_warp_kernel_dict"] > 0


def _walk(o, blocks):
    """o = the blocks in order, joined by the byte-aligning empty stored block."""
    pos = 0
    for k, want in enumerate(blocks):
        assert o[pos:pos + len(want)] == want, ("block", k)
        pos += len(want)
        if k + 1 < len(blocks):
            if o[pos:pos + 4] == b"\x00\x00\xff\xff":
                pos += 4
            else:
                assert o[pos:pos + 5] == b"\x00\x00\x00\xff\xff", ("join", k)
                pos += 5
    assert pos == len(o)


def _expected_blocks(d, dd, cb, primed, btype):
    """The oracle's blocks: chunk k searches the last min(32768, .) bytes of dictionary || item in front of it (only
    the first chunk without primed mode)."""
    import oracle
    if not d and btype == oracle.FIXED:
        return [b"\x03\x00"]   # the engine's empty FIXED block keeps its end-of-block symbol (api.py deviations)
    v = (dd or b"") + d
    base = len(dd or b"")
    n_chunks = max(1, -(-len(d) // cb))
    out = []
    for k in range(n_chunks):
        lo, hi = k * cb, min(len(d), (k + 1) * cb)
        if primed or k == 0:
            h = min(32768, base + lo) if d else 0
        else:
            h = 0
        out.append(oracle.raw_deflate_dict(v[base + lo - h:base + hi], h, k + 1 == n_chunks, btype))
    return out


def _synth_text(n, seed):
    from zlibts_b200 import synth
    return synth.text(n, seed).tobytes()


def test_compat_blocks_equal_the_oracle_with_the_dictionary(engine):
    import oracle
    sizes = (0, 1, 3, 257, 32767, 32768, 32769, 100000)
    dict_sizes = (0, 1, 100, 4096, 32768, 40000)
    src = _synth_text(200000 + 40000, 11)
    datas, dicts = [], []
    for i, ds in enumerate(dict_sizes):
        for j, n in enumerate(sizes):
            at = (i * 7919 + j * 104729) % 100000
            dicts.append(src[at:at + ds])               # text the item shares with its dictionary
            datas.append(src[at + ds // 2:at + ds // 2 + n] if j % 2 else _synth_text(n, 100 + j))
    for btype in (oracle.DYNAMIC, oracle.FIXED):
        outs, res, launches = _deflate(engine, datas, dicts, btype)
        assert launches["dict_stage_kernel"] > 0
        for i, (o, d, dd) in enumerate(zip(outs, datas, dicts)):
            try:
                _walk(o, _expected_blocks(d, dd, 32768, False, btype))
            except AssertionError as e:
                raise AssertionError((btype, len(dd), len(d), e.args))
        _roundtrip(engine, outs, datas, dicts)


def test_primed_blocks_search_dictionary_and_item(engine):
    import zlibts_b200 as z
    src = _synth_text(400000, 12)
    datas = [src[5000:5000 + n] for n in (1, 1499, 1500, 20000, 70001)] + [src[100000:200000]]
    dicts = [src[:4096], src[:40000], src[1000:33768], src[:1], src[4000:8000], src[60000:100000]]
    for chunk in (1500, 8192, 32768):
        outs, res, _ = _deflate(engine, datas, dicts, 2, z.MODE_PRIMED, chunk)
        for o, d, dd in zip(outs, datas, dicts):
            try:
                _walk(o, _expected_blocks(d, dd, chunk, True, 2))
            except AssertionError as e:
                raise AssertionError((chunk, len(dd), len(d), e.args))
        _roundtrip(engine, outs, datas, dicts)


def test_other_modes_round_trip(engine):
    import zlibts_b200 as z
    src = _synth_text(300000, 13)
    datas = [src[1000:1000 + n] for n in (0, 5, 600, 4000, 40000, 150000)]
    dicts = [src[:32768], src[:4096], src[500:1500], src[:32768], b"", src[100000:140000]]
    for mode in (z.mode_fast(), z.mode_fast() | z.MODE_LAZY, z.MODE_SMALLEST, z.mode_fast() | z.MODE_PRIMED,
                 z.MODE_PRIMED | z.MODE_SMALLEST):
        for chunk in (0, 3000):
            outs, res, _ = _deflate(engine, datas, dicts, 2, mode, chunk)
            _roundtrip(engine, outs, datas, dicts)
    # stored blocks do not change with a dictionary
    outs, res, _ = _deflate(engine, datas, dicts, z.NONE)
    plain, _, _ = _deflate(engine, datas, [None] * len(datas), z.NONE)
    assert outs == plain


def test_adversarial_dictionaries(engine):
    import oracle
    rng = np.random.default_rng(14)
    r = rand_bytes(rng, 32768).tobytes()
    t = _synth_text(20000, 15)
    datas = [r, t, b"a" * 100000, b"a" * 3, b"ab" * 40000, r[:100]]
    dicts = [r, t, b"a" * 32768, b"a" * 32768, b"b" + b"ab" * 16383, r]
    for btype in (oracle.DYNAMIC, oracle.FIXED):
        outs, res, _ = _deflate(engine, datas, dicts, btype)
        for o, d, dd in zip(outs, datas, dicts):
            _walk(o, _expected_blocks(d, dd, 32768, False, btype))
        # the item equal to its dictionary is 128 matches of up to 258 bytes (~26 bits each with the fixed codes), where
        # 32 KiB of random bytes without a dictionary take ~32 KiB
        assert len(outs[0]) < 1024
        _roundtrip(engine, outs, datas, dicts)


def test_mixed_batches_and_many_small_records(engine):
    src = _synth_text(1 << 20, 16)
    rng = np.random.default_rng(17)
    datas, dicts = [], []
    for i in range(300):
        n = int(rng.integers(0, 3)) and int(rng.integers(1, 5000))   # a third of them empty
        at = int(rng.integers(0, len(src) - 40000))
        datas.append(src[at:at + n])
        choices = (None, src[max(0, at - 3000):at], src[at + 1:at + 1 + 37000], src[7:8])
        dicts.append(choices[i % 4])
    for mode in (0, 2):
        outs, res, _ = _deflate(engine, datas, dicts, 2, mode)
        _roundtrip(engine, outs, datas, dicts)
    # 65 536 records of 256 B .. 4 KiB sharing one 4 KiB dictionary; smaller than without it
    shared = src[:4096]
    lens = rng.integers(256, 4097, 65536)
    offs = rng.integers(4096, len(src) - 4096, 65536)
    recs = [src[int(o):int(o) + int(n)] for o, n in zip(offs, lens)]
    outs, res, _ = _deflate(engine, recs, [shared] * len(recs))
    plain, _, _ = _deflate(engine, recs, [None] * len(recs))
    assert sum(map(len, outs)) < 0.95 * sum(map(len, plain))
    _roundtrip(engine, outs, recs, [shared] * len(recs))


def test_dict_entry_points_with_a_null_table_equal_the_old_ones(engine):
    import torch
    import zlibts_b200 as z
    datas = [_synth_text(n, 18 + n) for n in (0, 100, 70000, 200000)]
    blob, offs, lens = pack(datas)
    caps = [z.deflate_bound(len(d)) for d in datas]
    ooffs = np.concatenate([[0], np.cumsum(caps)]).astype(np.uint64)
    items = z.make_items(len(datas))
    items["in_off"], items["in_len"], items["out_off"], items["out_cap"] = offs, lens, ooffs[:-1], caps
    d_in = torch.from_numpy(blob).cuda()
    outs = []
    for use_dict in (False, True):
        d_out = torch.zeros(int(ooffs[-1]), dtype=torch.uint8, device="cuda")
        res = np.zeros(len(datas), dtype=z.RESULT_DTYPE)
        if use_dict:
            rc = engine.lib.zlb_deflate_batch_dict(engine.h, d_in.data_ptr(), d_out.data_ptr(), None, None,
                                                   items.ctypes.data, res.ctypes.data, len(datas), 0, 2, 0, 3)
        else:
            rc = engine.lib.zlb_deflate_batch(engine.h, d_in.data_ptr(), d_out.data_ptr(), items.ctypes.data,
                                              res.ctypes.data, len(datas), 0, 2, 0, 3)
        assert rc == 0
        outs.append((d_out.cpu().numpy().tobytes(), res.tobytes()))
    assert outs[0] == outs[1]
    comp = d_out.cpu().numpy()
    iitems = z.make_items(len(datas))
    iitems["in_off"], iitems["in_len"] = ooffs[:-1], np.frombuffer(outs[0][1], dtype=z.RESULT_DTYPE)["out_len"]
    icaps = [len(d) + 1 for d in datas]
    iitems["out_off"], iitems["out_cap"] = np.concatenate([[0], np.cumsum(icaps)[:-1]]), icaps
    d_c = torch.from_numpy(comp.copy()).cuda()
    got = []
    for use_dict in (False, True):
        d_o = torch.zeros(int(sum(len(d) + 1 for d in datas)) + 8, dtype=torch.uint8, device="cuda")
        res = np.zeros(len(datas), dtype=z.RESULT_DTYPE)
        fn = engine.lib.zlb_inflate_batch_dict if use_dict else engine.lib.zlb_inflate_batch
        args = (None, None) if use_dict else ()
        rc = fn(engine.h, d_c.data_ptr(), d_o.data_ptr(), *args, iitems.ctypes.data, res.ctypes.data, len(datas), 3)
        assert rc == 0
        got.append((d_o.cpu().numpy().tobytes(), res.tobytes()))
    assert got[0] == got[1]


def test_invalid_dictionary_tables_are_refused(engine):
    import zlibts_b200 as z
    data = np.frombuffer(b"hello hello hello", dtype=np.uint8).copy()
    out = np.zeros(256, dtype=np.uint8)
    items = z.make_items(1)
    items["in_len"], items["out_cap"] = data.size, 256
    table = z.make_dicts(1)
    table[0] = (10, 20)
    with pytest.raises(z.EngineError):     # span beyond the 16-byte blob
        engine.deflate_batch_host(data, out, items, h_dict=np.zeros(16, dtype=np.uint8), dicts=table)
    with pytest.raises(z.EngineError):     # a dictionary without a blob
        engine.inflate_batch_host(data, out, items, h_dict=None, dicts=table)


def _zdict_stream(data, zdict, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, interval=None):
    co = zlib.compressobj(level, zlib.DEFLATED, -15, 9, strategy, zdict=zdict)
    if interval is None:
        return co.compress(data) + co.flush()
    parts = [co.compress(data[k:k + interval]) + co.flush(zlib.Z_SYNC_FLUSH) for k in range(0, len(data), interval)]
    return b"".join(parts) + co.flush()


def _compare_routes(engine, streams, datas, dicts, caps=None, window=True):
    """ZLB_INFLATE_SPLIT vs the one-warp dictionary decoder: the same fields, the same bytes (0xA5 behind out_len)."""
    import zlibts_b200 as z
    caps = [len(d) for d in datas] if caps is None else caps
    flags = z.INFLATE_WANT_CRC32 | z.INFLATE_WANT_ADLER32
    buf1, ooffs, res1, l1 = _inflate(engine, streams, caps, dicts, flags | z.INFLATE_SPLIT)
    buf0, _, res0, l0 = _inflate(engine, streams, caps, dicts, flags)
    assert not any(l0[k] for k in WINDOW_KERNELS) and l0["inflate_warp_kernel_dict"] > 0
    for i in range(len(streams)):
        for f in FIELDS:
            assert int(res1[i][f]) == int(res0[i][f]), (i, f, int(res1[i][f]), int(res0[i][f]))
        lo, hi = int(ooffs[i]), int(ooffs[i + 1])
        assert buf1[lo:hi] == buf0[lo:hi], i
        if datas[i] is not None:
            assert int(res1[i]["status"]) == 0 and buf1[lo:lo + len(datas[i])] == datas[i], i
    if window is not None:
        ran = [l1[k] > 0 for k in WINDOW_KERNELS]
        assert all(ran) if window else not any(ran), l1
    return res1


def test_inflate_cpython_zdict_streams(engine):
    src = _synth_text(3 << 20, 19)
    zd = src[:32768]
    datas, streams, dicts = [], [], []
    for k, (level, strategy) in enumerate(((1, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_DEFAULT_STRATEGY),
                                           (9, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_RLE), (6, zlib.Z_HUFFMAN_ONLY))):
        for n in (1, 1000, 50000):
            d = src[40000 + 977 * k:40000 + 977 * k + n]
            for dd in (zd, zd[-500:]):
                datas.append(d)
                dicts.append(dd)
                streams.append(_zdict_stream(d, dd, level, strategy))
    _roundtrip(engine, streams, datas, dicts)
    _compare_routes(engine, streams, datas, dicts, window=None)


def test_inflate_sync_flushed_zdict_streams_take_the_window_route(engine):
    src = _synth_text(6 << 20, 20)
    datas, streams, dicts = [], [], []
    for k, (level, strategy, interval, dl) in enumerate(((1, zlib.Z_DEFAULT_STRATEGY, 5000, 32768),
                                                         (6, zlib.Z_DEFAULT_STRATEGY, 32768, 4096),
                                                         (9, zlib.Z_DEFAULT_STRATEGY, 60000, 40000),
                                                         (6, zlib.Z_RLE, 20000, 32768))):
        d = src[(1 << 20) + k * 100000:(1 << 20) + k * 100000 + (2 << 20)]
        dd = src[(1 << 20) + k * 100000 - dl:(1 << 20) + k * 100000]      # the text right in front of the item
        datas.append(d)
        dicts.append(dd)
        streams.append(_zdict_stream(d, dd, level, strategy, interval))
        assert len(streams[-1]) >= 256 << 10
    _compare_routes(engine, streams, datas, dicts)
    _roundtrip(engine, streams, datas, dicts)


# ---- hand-built streams ------------------------------------------------------------------------------------------
_LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195,
             227, 258]
_LEN_EXTRA = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
_DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073,
              4097, 6145, 8193, 12289, 16385, 24577]
_DIST_EXTRA = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13]


def _fixed_sym(w, sym):
    if sym < 144:
        w.code(0x30 + sym, 8)
    elif sym < 256:
        w.code(0x190 + sym - 144, 9)
    elif sym < 280:
        w.code(sym - 256, 7)
    else:
        w.code(0xC0 + sym - 280, 8)


def _fixed_block(w, tokens, final):
    """One fixed-Huffman block: tokens are literal bytes (int) or (length, distance)."""
    w.bits(1 if final else 0, 1)
    w.bits(1, 2)
    for t in tokens:
        if isinstance(t, int):
            _fixed_sym(w, t)
            continue
        length, dist = t
        li = max(i for i, b in enumerate(_LEN_BASE) if b <= length) if length < 258 else 28
        _fixed_sym(w, 257 + li)
        w.bits(length - _LEN_BASE[li], _LEN_EXTRA[li])
        di = max(i for i, b in enumerate(_DIST_BASE) if b <= dist)
        w.code(di, 5)
        w.bits(dist - _DIST_BASE[di], _DIST_EXTRA[di])
    _fixed_sym(w, 256)


def _expand(dictionary, tokens):
    out = bytearray()
    for t in tokens:
        if isinstance(t, int):
            out.append(t)
            continue
        length, dist = t
        for _ in range(length):
            v = dictionary + bytes(out)
            out.append(v[len(v) - dist])
    return bytes(out)


def _hand_stream(tokens, tail=None):
    """The tokens as one fixed block; with `tail`, behind a sync-flush marker, stored blocks of `tail` (> 256 KiB, so
    that ZLB_INFLATE_SPLIT cuts the stream) joined by markers."""
    w = _BitWriter()
    _fixed_block(w, tokens, tail is None)
    if tail is not None:
        for at in range(0, len(tail), 60000):
            w.bits(0, 3)             # empty stored block: the marker
            w.align()
            w.bits(0, 16)
            w.bits(0xFFFF, 16)
            piece = tail[at:at + 60000]
            w.bits(1 if at + 60000 >= len(tail) else 0, 1)
            w.bits(0, 2)
            w.align()
            w.bits(len(piece), 16)
            w.bits(len(piece) ^ 0xFFFF, 16)
            w.buf.extend(piece)
    return w.bytes()


def test_hand_built_matches_into_the_dictionary(engine):
    rng = np.random.default_rng(21)
    d32 = rand_bytes(rng, 32768).tobytes()
    tail = rand_bytes(rng, 300000).tobytes()
    cases = [
        (d32, [(258, 32768), (258, 32768)]),                              # distance 32768 at output byte 0
        (d32[:1000], [65, 66, 67] + [(50, 30)] + [(40, 60)]),             # a match straddling the dictionary's end
        (d32[:1000], [(100, 3), (20, 1), (258, 7)]),                      # periodic, source in the dictionary
        (d32, [(3, 32768)] + [(258, 1)] * 3 + [(7, 32768)]),
    ]
    streams, datas, dicts = [], [], []
    for dd, toks in cases:
        for with_tail in (False, True):
            out = _expand(dd, toks)
            streams.append(_hand_stream(toks, tail if with_tail else None))
            datas.append(out + (tail if with_tail else b""))
            dicts.append(dd)
    _roundtrip(engine, streams, datas, dicts)
    _compare_routes(engine, streams, datas, dicts)


def test_distance_beyond_the_dictionary_is_bad_code_on_both_routes(engine):
    import zlibts_b200 as z
    rng = np.random.default_rng(22)
    dd = rand_bytes(rng, 1000).tobytes()
    tail = rand_bytes(rng, 300000).tobytes()
    toks = [1, 2, 3, 4, 5, (10, 1006)]                      # one byte in front of the dictionary
    streams = [_hand_stream(toks), _hand_stream(toks, tail)]
    caps = [len(tail) + 64] * 2
    res = _compare_routes(engine, streams, [None, None], [dd, dd], caps, window=None)
    for r in res:
        assert int(r["status"]) == z.ST_BAD_CODE and int(r["out_len"]) == 5
    buf, ooffs, _, _ = _inflate(engine, streams, caps, [dd, dd], z.INFLATE_SPLIT)
    for i in range(2):
        lo = int(ooffs[i])
        assert buf[lo:lo + 5] == bytes([1, 2, 3, 4, 5]) and set(buf[lo + 5:int(ooffs[i + 1])]) == {0xA5}
    # the same streams with the distance inside the dictionary decode
    ok = [1, 2, 3, 4, 5, (10, 1005)]
    datas = [_expand(dd, ok), _expand(dd, ok) + tail]
    _compare_routes(engine, [_hand_stream(ok), _hand_stream(ok, tail)], datas, [dd, dd], caps, window=None)


# ---- host entry points and the host API ---------------------------------------------------------------------------
@pytest.mark.parametrize("pinned", [False, True])
def test_host_entry_points(engine, pinned):
    import zlibts_b200 as z
    src = _synth_text(2 << 20, 23)
    datas = [src[(k + 1) * 50000:(k + 1) * 50000 + n] for k, n in enumerate((0, 10, 3000, 33000, 500000))]
    dicts = [src[:32768], None, src[40000:50000], src[100:200], src[:40000]]
    blob, offs, lens = pack(datas)
    dblob, table = _dict_blob(dicts)
    caps = [z.deflate_bound(len(d), 0, z.DYNAMIC, 0, True) for d in datas]
    ooffs = np.concatenate([[0], np.cumsum(caps)]).astype(np.uint64)

    def host(a):
        if not pinned:
            return a
        p = z.host_alloc(a.size)
        p[:] = a
        return p
    items = z.make_items(len(datas))
    items["in_off"], items["in_len"], items["out_off"], items["out_cap"] = offs, lens, ooffs[:-1], caps
    h_in, h_dict, h_out = host(blob), host(dblob), host(np.zeros(int(ooffs[-1]), dtype=np.uint8))
    assert z.host_is_pinned(h_in) == pinned
    res = engine.deflate_batch_host(h_in, h_out, items, z.DYNAMIC, 0, z.DEFLATE_WANT_CRC32, 0, h_dict, table)
    assert int(res["status"].max()) == 0
    streams = [bytes(h_out[int(o):int(o) + int(r["out_len"])]) for o, r in zip(ooffs[:-1], res)]
    dev, dres, _ = _deflate(engine, datas, dicts)
    assert streams == dev and [int(c) for c in res["crc32"]] == [zlib.crc32(d) for d in datas]
    cblob, coffs, clens = pack(streams)
    icaps = [len(d) + 3 for d in datas]
    iooffs = np.concatenate([[0], np.cumsum(icaps)]).astype(np.uint64)
    it = z.make_items(len(datas))
    it["in_off"], it["in_len"], it["out_off"], it["out_cap"] = coffs, clens, iooffs[:-1], icaps
    h_c, h_o = host(cblob), host(np.zeros(int(iooffs[-1]), dtype=np.uint8))
    r2 = engine.inflate_batch_host(h_c, h_o, it, z.INFLATE_WANT_ADLER32 | z.INFLATE_SPLIT, h_dict, table)
    for i, d in enumerate(datas):
        assert int(r2["status"][i]) == 0 and bytes(h_o[int(iooffs[i]):int(iooffs[i]) + len(d)]) == d
        assert int(r2["adler32"][i]) == zlib.adler32(d)


def test_host_api_zlib_fdict(engine):
    import zlibts_b200 as z
    z.api.set_engine(engine)
    src = _synth_text(300000, 24)
    zd, data = src[:20000], src[20000:120000]
    for opts in ({}, {"compressionType": z.CompressionType.FIXED}, {"b200": {"mode": "primed"}}):
        o = dict(opts)
        o["b200"] = dict(o.get("b200", {}), dictionary=zd)
        s = z.Deflate(data, o).compress().tobytes()
        assert s[1] & 0x20 and int.from_bytes(s[2:6], "big") == zlib.adler32(zd) and ((s[0] << 8) | s[1]) % 31 == 0
        assert zlib.decompressobj(zdict=zd).decompress(s) == data
        inf = z.Inflate(s, {"verify": True, "b200": {"dictionary": zd}})
        assert inf.decompress().tobytes() == data and inf.ip == len(s) - 4
    co = zlib.compressobj(9, zdict=zd)
    s = co.compress(data) + co.flush()
    assert z.Inflate(s, {"b200": {"dictionary": zd}}).decompress().tobytes() == data
    with pytest.raises(z.ZlibError, match="invalid dictionary"):
        z.Inflate(s, {"b200": {"dictionary": zd[1:]}})
    with pytest.raises(z.ZlibError, match="^fdict flag is not supported$"):
        z.Inflate(s)
    # a dictionary given for a stream without FDICT is ignored
    s2 = zlib.compress(data)
    assert z.Inflate(s2, {"b200": {"dictionary": zd}}).decompress().tobytes() == data
    # raw streams
    r = z.RawDeflate(data, {"b200": {"dictionary": zd}}).compress().tobytes()
    assert zlib.decompressobj(-15, zdict=zd).decompress(r) == data
    assert z.RawInflate(r, {"b200": {"dictionary": zd}}).decompress().tobytes() == data
    outs, _ = z.deflate_many([data[:100], data[:5000], b""], dictionary=[zd, None, zd])
    back, _ = z.inflate_many(outs, dictionary=[zd, None, zd])
    assert [b.tobytes() for b in back] == [data[:100], data[:5000], b""]
