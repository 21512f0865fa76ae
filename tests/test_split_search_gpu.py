"""GPU: ZLB_INFLATE_SPLIT on streams without sync-flush markers (CPython zlib, gzip): the split searches block starts
on the device, sizes the pieces, repairs broken chains and decodes the pieces in window mode. Every case is compared
with the one-warp decoder (the same call without INFLATE_SPLIT) field by field and byte by byte, and with CPython's
zlib where the stream is valid; the profile slots tell which route ran. The finder's proposals are checked against
the block starts a reference walker (below) reads from the streams."""
import gzip
import zlib

import numpy as np
import pytest

from helpers import pack, rand_bytes

pytestmark = pytest.mark.gpu

WINDOW_KERNELS = ("inflate_warp_kernel_window", "window_run_kernel", "window_scan_kernel", "window_resolve_kernel")
FIELDS = ("status", "out_len", "in_used", "blocks", "crc32", "adler32")
SIZE_FIELDS = ("status", "out_len", "in_used", "blocks")
MIB = 1 << 20


def _raw(data, level=6, mem=8, strategy=zlib.Z_DEFAULT_STRATEGY, zdict=None):
    co = zlib.compressobj(level, zlib.DEFLATED, -15, mem, strategy, *([zdict] if zdict else []))
    return co.compress(data) + co.flush()


def _profiled(engine, fn):
    engine.profile_enable(True)
    engine.profile_reset()
    try:
        res = fn()
        prof = engine.profile_read()
    finally:
        engine.profile_enable(False)
    return res, {k: v["launches"] for k, v in prof.items()}


def _inflate(engine, streams, caps, flags, zdicts=None):
    """(whole output buffer, output offsets, results, launches by kernel) of one call; the output buffer starts out
    filled with 0xA5, so whatever a route writes beyond what it reports shows."""
    import torch
    import zlibts_b200 as z
    blob, offs, lens = pack([bytes(s) for s in streams])
    ooffs = np.concatenate([[0], np.cumsum(caps)]).astype(np.uint64)
    items = z.make_items(len(streams))
    items["in_off"], items["in_len"] = offs, lens
    items["out_off"], items["out_cap"] = ooffs[:-1], caps
    d_in = torch.from_numpy(blob).cuda()
    d_out = torch.full((max(int(ooffs[-1]), 1),), 0xA5, dtype=torch.uint8, device="cuda")
    kw = {}
    if zdicts is not None:
        dblob, doffs, dlens = pack([d or b"" for d in zdicts])
        table = z.make_dicts(len(streams))
        table["off"], table["len"] = doffs, dlens
        kw = {"d_dict": torch.from_numpy(dblob).cuda(), "dicts": table}
    res, launches = _profiled(engine, lambda: engine.inflate_batch(d_in, d_out, items, flags, **kw))
    return d_out.cpu().numpy().tobytes(), ooffs, res, launches


def _compare(engine, streams, datas, caps=None, route="search", zdicts=None):
    """Split route vs one-warp route (and CPython zlib for the valid streams). route: "search" = the finder and the
    window kernels ran and inflate_warp_kernel did not; "mixed" = the finder and the window kernels ran (a batch with
    marker or small items, which inflate_warp_kernel decodes); "one_warp" = inflate_warp_kernel ran; None = either.
    Returns (results, launches) of the split route."""
    import zlibts_b200 as z
    caps = [len(d) if d is not None else 8 * MIB for d in datas] if caps is None else caps
    flags = z.INFLATE_WANT_CRC32 | z.INFLATE_WANT_ADLER32
    buf1, ooffs, res1, launches = _inflate(engine, streams, caps, flags | z.INFLATE_SPLIT, zdicts)
    buf0, _, res0, launches0 = _inflate(engine, streams, caps, flags, zdicts)
    assert not launches0["block_find_kernel"] and not any(launches0[k] for k in WINDOW_KERNELS)
    for i, (s, d) in enumerate(zip(streams, datas)):
        r0, r1 = res0[i], res1[i]
        if int(r0["status"]) == z.ST_OUT_OVERFLOW:   # the split route writes nothing then (out_len 0)
            assert int(r1["status"]) == z.ST_OUT_OVERFLOW, i
            continue
        for f in FIELDS:
            assert int(r1[f]) == int(r0[f]), (i, f, int(r1[f]), int(r0[f]))
        lo, hi = int(ooffs[i]), int(ooffs[i + 1])
        assert buf1[lo:hi] == buf0[lo:hi], i                         # incl. the bytes behind out_len
        if d is not None:
            assert int(r1["status"]) == 0, i
            o = buf1[lo:lo + int(r1["out_len"])]
            zd = zdicts[i] if zdicts else None
            ref = zlib.decompressobj(-15, *([zd] if zd else [])).decompress(bytes(s))
            assert o == d and ref == d, i
            assert int(r1["crc32"]) == zlib.crc32(d) and int(r1["adler32"]) == zlib.adler32(d), i
    if route in ("search", "mixed"):
        assert launches["block_find_kernel"] > 0 and all(launches[k] > 0 for k in WINDOW_KERNELS), launches
    if route == "search":
        assert launches["inflate_warp_kernel"] == 0, launches
    elif route == "one_warp":
        assert launches["inflate_warp_kernel"] > 0, launches
    _compare_sizes(engine, streams, res0, zdicts, launches if route == "search" else None)
    return res1, launches


def _compare_sizes(engine, streams, res0, zdicts=None, settled=None):
    """zlb_inflate_size_batch with SPLIT: the decoder's status / out_len / in_used / blocks (out_cap large enough), with
    no window kernel, no gather and no inflate_warp_kernel launch. settled: the launches of a decode call that the split
    settled alone; the size call then runs the same size passes and no one-warp size launch behind them (which reports
    under the same slot)."""
    import torch
    import zlibts_b200 as z
    blob, offs, lens = pack([bytes(s) for s in streams])
    items = z.make_items(len(streams))
    items["in_off"], items["in_len"] = offs, lens
    table = None
    if zdicts is not None:
        table = z.make_dicts(len(streams))
        table["len"] = [len(d or b"") for d in zdicts]
    d_in = torch.from_numpy(blob).cuda()
    res, launches = _profiled(engine, lambda: engine.inflate_size_batch(d_in, items, z.INFLATE_SPLIT, table))
    assert not any(launches[k] for k in WINDOW_KERNELS + ("segment_gather_kernel", "inflate_warp_kernel")), launches
    if settled is not None:
        assert launches["inflate_warp_kernel_size"] == settled["inflate_warp_kernel_size"], (launches, settled)
    for i in range(len(streams)):
        if int(res0[i]["status"]) == z.ST_OUT_OVERFLOW:
            continue
        for f in SIZE_FIELDS:
            assert int(res[i][f]) == int(res0[i][f]), (i, f, int(res[i][f]), int(res0[i][f]))


def test_zlib_streams_without_markers(engine):
    from zlibts_b200 import synth
    text = synth.text(4 * MIB, 101).tobytes()
    mixed = synth.mixed(4 * MIB + 777, 102).tobytes()
    cases = [(1, 8, zlib.Z_DEFAULT_STRATEGY), (6, 8, zlib.Z_DEFAULT_STRATEGY), (9, 8, zlib.Z_DEFAULT_STRATEGY),
             (6, 1, zlib.Z_DEFAULT_STRATEGY), (6, 9, zlib.Z_DEFAULT_STRATEGY), (6, 8, zlib.Z_FILTERED),
             (6, 8, zlib.Z_HUFFMAN_ONLY), (6, 8, zlib.Z_RLE)]
    for d in (text, mixed):
        streams = [_raw(d, *c) for c in cases]
        for s in streams[:2]:
            _compare(engine, [s], [d])
        _compare(engine, streams, [d] * len(streams))
    big = synth.text(16 * MIB, 103).tobytes()
    _compare(engine, [_raw(big, 6)], [big])


def test_random_data_stored_blocks(engine):
    rng = np.random.default_rng(7)
    d = rand_bytes(rng, 6 * MIB).tobytes()
    s = _raw(d, 6)
    assert s[0] & 7 == 0    # stored blocks
    _compare(engine, [s], [d])


def test_fixed_blocks_take_the_one_warp_route(engine):
    from zlibts_b200 import synth
    d = synth.text(4 * MIB, 104).tobytes()
    _compare(engine, [_raw(d, 6, 8, zlib.Z_FIXED)], [d], route="one_warp")


def test_false_candidates_are_repaired(engine):
    """Stored blocks whose payload is zlib output: it holds real dynamic block headers at arbitrary bit offsets, which
    pass the finder's test but are no block starts of this stream. Results are identical; the size pass ran again on
    merged pieces."""
    from zlibts_b200 import synth
    payload = b"".join(_raw(synth.text(600000, 110 + k).tobytes(), 6) for k in range(8))
    streams = [_raw(payload, 0), _raw(payload, 0) + b"junk" * 5]
    res, launches = _compare(engine, streams, [payload, payload], route=None)
    assert launches["inflate_warp_kernel_size"] >= 2, launches   # at least one repair round


def test_robustness(engine):
    import zlibts_b200 as z
    from zlibts_b200 import synth
    d = synth.mixed(4 * MIB, 120).tobytes()
    s = _raw(d, 6)
    bad = bytearray(s)
    bad[len(s) // 2] ^= 0x5A
    streams = [s[:len(s) // 2], s[:-1], bytes(bad)]
    _compare(engine, streams, [None] * 3, caps=[len(d)] * 3, route=None)
    # a gzip member with its trailer and junk behind it: the item ends where the stream ends plus 64 bytes
    g = gzip.compress(d, 6)
    hdr = 10
    _compare(engine, [g[hdr:] + b"\xA7" * 64], [d])
    # markers and long stretches without (more than the 1 MiB the split searches): a Z_SYNC_FLUSH every 4 MiB of input
    m = synth.mixed(14 * MIB, 125).tobytes()
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    sync = b"".join(co.compress(m[k:k + 4 * MIB]) + co.flush(zlib.Z_SYNC_FLUSH) for k in range(0, len(m), 4 * MIB))
    sync += co.flush()
    assert sync.count(b"\x00\x00\xff\xff") >= 3
    _compare(engine, [sync], [m])
    # one batch: searched, marker (a GPU stream), small and one undersized searched item
    rng = np.random.default_rng(121)
    datas = [synth.text(4 * MIB, 122).tobytes(), synth.mixed(3 * MIB, 123).tobytes(),
             rand_bytes(rng, 5000, 7).tobytes(), synth.mixed(5 * MIB, 124).tobytes()]
    streams = [_raw(datas[0], 6), _gpu_deflate(engine, datas[1], z.MODE_PRIMED), _raw(datas[2], 6), _raw(datas[3], 9)]
    _compare(engine, streams, datas, route="mixed")
    caps = [len(x) for x in datas]
    caps[3] -= 1
    res, _ = _compare(engine, streams, datas, caps=caps, route=None)
    assert [int(r["status"]) for r in res] == [0, 0, 0, z.ST_OUT_OVERFLOW]


def _gpu_deflate(engine, data, mode):
    import torch
    import zlibts_b200 as z
    cap = z.deflate_bound(len(data), 0, z.DYNAMIC, mode)
    items = z.make_items(1)
    items["in_len"], items["out_cap"] = len(data), cap
    d_z = torch.zeros(cap, dtype=torch.uint8, device="cuda")
    d_in = torch.from_numpy(np.frombuffer(data, dtype=np.uint8).copy()).cuda()
    r = engine.deflate_batch(d_in, d_z, items, mode=mode)
    assert int(r["status"][0]) == 0
    return d_z[:int(r["out_len"][0])].cpu().numpy().tobytes()


def test_stream_followed_by_another(engine):
    """A stream with a second one behind it in the same item: the finder proposes block starts of the second, whose
    pieces decode cleanly; the chain is kept up to the piece that reaches BFINAL, where the one-warp decoder stops."""
    from zlibts_b200 import synth
    d1, d2 = synth.text(4 * MIB, 133).tobytes(), synth.mixed(3 * MIB, 134).tobytes()
    s1 = _raw(d1, 6)
    res, _ = _compare(engine, [s1 + _raw(d2, 6)], [d1])
    assert int(res["in_used"][0]) == len(s1)


def test_reach_before_the_stream_with_a_small_slot(engine):
    """A stream written with a dictionary, decoded without it: its first distances reach before the stream. The one-warp
    decoder stops there with ZLB_ST_BAD_CODE, also when the slot is too small for the whole output, so the split may
    not answer ZLB_ST_OUT_OVERFLOW from the sizes alone."""
    import zlibts_b200 as z
    from zlibts_b200 import synth
    zd = synth.text(32768, 135).tobytes()
    d = synth.text(4 * MIB, 136).tobytes()
    s = _raw(d, 6, zdict=zd)
    for cap in (len(d) - 1, len(d)):
        res, _ = _compare(engine, [s], [None], caps=[cap], route=None)
        assert int(res["status"][0]) == z.ST_BAD_CODE


def test_preset_dictionary_without_markers(engine):
    from zlibts_b200 import synth
    zd = synth.text(32768, 130).tobytes()
    d = synth.text(4 * MIB, 131).tobytes()
    m = synth.mixed(3 * MIB, 132).tobytes()
    _compare(engine, [_raw(d, 6, zdict=zd), _raw(m, 6)], [d, m], zdicts=[zd, None])
    assert len(_raw(m, 6)) > MIB


def test_public_surface(engine):
    import zlibts_b200 as Z
    from zlibts_b200 import synth
    Z.api.set_engine(engine)
    d = synth.mixed(6 * MIB, 140).tobytes()
    g = gzip.compress(d, 6)
    out, launches = _profiled(engine, lambda: Z.GUnzip(g).decompress().tobytes())
    assert out == d and all(launches[k] > 0 for k in WINDOW_KERNELS), launches
    c = zlib.compress(d)
    out, launches = _profiled(engine, lambda: Z.Inflate(c, {"verify": True}).decompress().tobytes())
    assert out == d and all(launches[k] > 0 for k in WINDOW_KERNELS), launches


def test_gunzip_with_a_signature_inside_the_body(engine):
    """A `1F 8B 08` that parses as a member header inside the compressed body (a large file holds a few by chance)
    sends GUnzip down its member-candidate path; the first member still decodes through the split."""
    import zlibts_b200 as Z
    from zlibts_b200 import synth
    Z.api.set_engine(engine)
    rng = np.random.default_rng(180)
    decoy = gzip.compress(b"decoy", mtime=0)
    noise = b"".join(rand_bytes(rng, 16384).tobytes() + decoy for _ in range(16))   # stored blocks keep it verbatim
    d = synth.text(3 * MIB, 181).tobytes() + noise + synth.mixed(2 * MIB, 182).tobytes()
    g = gzip.compress(d, 6)
    assert g.find(decoy[:10], 10) > 0
    gu = Z.GUnzip(g)
    out, launches = _profiled(engine, lambda: gu.decompress().tobytes())
    assert out == d and len(gu.getMembers()) == 1
    assert launches["block_find_kernel"] > 0 and all(launches[k] > 0 for k in WINDOW_KERNELS), launches


def test_host_entry_points_pinned_and_pageable(engine):
    import zlibts_b200 as z
    from zlibts_b200 import synth
    rng = np.random.default_rng(150)
    big = [synth.text(4 * MIB, 151).tobytes(), synth.mixed(4 * MIB, 152).tobytes()]
    small = [synth.text(int(n), 1500 + k).tobytes() for k, n in enumerate(rng.integers(1, 3000, 1000))]
    datas = big + small
    streams = [_raw(x, 6) for x in datas]
    blob, offs, lens = pack(streams)
    caps = [len(x) + 50 for x in datas]
    ooffs = np.concatenate([[0], np.cumsum(caps)]).astype(np.uint64)
    items = z.make_items(len(streams))
    items["in_off"], items["in_len"], items["out_off"], items["out_cap"] = offs, lens, ooffs[:-1], caps
    base = z.INFLATE_WANT_CRC32 | z.INFLATE_WANT_ADLER32
    for pinned in (True, False):
        runs = []
        for flags in (base | z.INFLATE_SPLIT, base):
            if pinned:
                h_in, h_out = z.host_alloc(blob.size), z.host_alloc(int(ooffs[-1]))
                h_in[:] = blob
            else:
                h_in, h_out = blob.copy(), np.empty(int(ooffs[-1]), dtype=np.uint8)
            h_out[:] = 0xA5
            res, launches = _profiled(engine, lambda: engine.inflate_batch_host(h_in, h_out, items, flags))
            sizes, slaunch = _profiled(engine, lambda: engine.inflate_size_batch_host(h_in, items, flags & z.INFLATE_SPLIT))
            runs.append((res, h_out.tobytes(), launches, sizes, slaunch))
            if pinned:
                z.host_free(h_in)
                z.host_free(h_out)
        (res, out, launches, sizes, slaunch), (res0, out0, launches0, sizes0, _) = runs
        assert launches["block_find_kernel"] > 0 and all(launches[k] > 0 for k in WINDOW_KERNELS), launches
        assert slaunch["block_find_kernel"] > 0 and not slaunch["inflate_warp_kernel_window"], slaunch
        assert res.tobytes() == res0.tobytes() and out == out0
        for f in SIZE_FIELDS:
            assert (sizes[f] == sizes0[f]).all() and (sizes[f] == res0[f]).all(), f
        for i, (x, r) in enumerate(zip(datas, res)):
            assert int(r["status"]) == 0 and out[int(ooffs[i]):int(ooffs[i]) + len(x)] == x, i


# ---- finder quality ------------------------------------------------------------------------------------------------
_ORDER = (16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15)
_LBASE = (3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227,
          258)
_LEXTRA = (0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0)
_DEXTRA = (0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13)


def _table(lens):
    """LSB-first lookup table of a canonical code: entry = symbol << 4 | length, indexed by the next max-length bits"""
    mx = max(lens)
    tab = [0] * (1 << mx)
    code = 0
    for length in range(1, mx + 1):
        for sym, l in enumerate(lens):
            if l != length:
                continue
            r = int(format(code, "0%db" % length)[::-1], 2)
            for j in range(r, 1 << mx, 1 << length):
                tab[j] = sym << 4 | length
            code += 1
        code <<= 1
    return tab, (1 << mx) - 1


def block_starts(s):
    """(bit offset, BTYPE) of every block of the raw deflate stream s, read by walking its symbols"""
    buf = bytes(s) + b"\0" * 8
    pos = 0
    out = []

    def peek(p):
        return int.from_bytes(buf[p >> 3:(p >> 3) + 5], "little") >> (p & 7)

    fixed = _table([8] * 144 + [9] * 112 + [7] * 24 + [8] * 8), _table([5] * 30)
    while True:
        h = peek(pos)
        final, btype = h & 1, (h >> 1) & 3
        out.append((pos, btype))
        pos += 3
        if btype == 0:
            pos = (pos + 7) & ~7
            n = peek(pos) & 0xFFFF
            pos += 32 + 8 * n
        else:
            if btype == 1:
                (lt, lm), (dt, dm) = fixed
            else:
                hlit, hdist, hclen = (h >> 3 & 31) + 257, (h >> 8 & 31) + 1, (h >> 13 & 15) + 4
                pos += 14
                cl = [0] * 19
                for i in range(hclen):
                    cl[_ORDER[i]] = peek(pos + 3 * i) & 7
                pos += 3 * hclen
                ct, cm = _table(cl)
                lens = []
                while len(lens) < hlit + hdist:
                    e = ct[peek(pos) & cm]
                    sym = e >> 4
                    pos += e & 15
                    if sym < 16:
                        lens.append(sym)
                    elif sym == 16:
                        lens += [lens[-1]] * (3 + (peek(pos) & 3))
                        pos += 2
                    elif sym == 17:
                        lens += [0] * (3 + (peek(pos) & 7))
                        pos += 3
                    else:
                        lens += [0] * (11 + (peek(pos) & 127))
                        pos += 7
                (lt, lm), (dt, dm) = _table(lens[:hlit]), _table(lens[hlit:] if any(lens[hlit:]) else [1])
            while True:
                e = lt[peek(pos) & lm]
                sym = e >> 4
                pos += e & 15
                if sym < 256:
                    continue
                if sym == 256:
                    break
                pos += _LEXTRA[sym - 257]
                e = dt[peek(pos) & dm]
                pos += (e & 15) + _DEXTRA[e >> 4]
        if final:
            return out


def test_finder_quality(engine):
    """Where a span holds a dynamic block start first, the finder returns it; where it holds a stored block first, the
    start of the block behind that one (a stored block is proposed by where it ends). Never an offset that is no block
    start."""
    import torch
    from zlibts_b200 import synth
    rng = np.random.default_rng(162)
    for d, kind in ((synth.text(2 * MIB, 160).tobytes(), 2), (synth.mixed(2 * MIB, 161).tobytes(), 2),
                    (rand_bytes(rng, 2 * MIB).tobytes(), 0)):
        s = _raw(d, 6)
        starts = block_starts(s)
        assert len(starts) > 10
        truth = {b for b, t in starts}
        after = {b: starts[i + 1][0] for i, (b, t) in enumerate(starts[:-1])}
        step, span = 4096, 8 * 16384
        cuts = np.arange(1, len(s) - 64, step, dtype=np.uint64)
        got = engine.debug_block_starts(torch.from_numpy(np.frombuffer(s, dtype=np.uint8).copy()).cuda(), cuts, span)
        hits = tries = 0
        for c, g in zip(cuts, got):
            lo = 8 * int(c)
            inside = [(b, t) for b, t in starts[:-2] if lo <= b < lo + span and t in (0, 2)]
            assert g == -1 or int(g) in truth, (int(c), int(g))     # never an offset that is no block start
            if inside and inside[0][1] == kind:
                tries += 1
                hits += int(g) == (inside[0][0] if kind == 2 else after[inside[0][0]])
        assert tries > 20 and hits >= 0.9 * tries, (kind, hits, tries)


def test_repeats_are_identical_and_scratch_is_bounded(engine):
    import torch
    import zlibts_b200 as z
    from zlibts_b200 import synth
    d = synth.mixed(8 * MIB, 170).tobytes()
    s = _raw(d, 6)
    runs = [_inflate(engine, [s], [len(d)], z.INFLATE_SPLIT | z.INFLATE_WANT_CRC32) for _ in range(3)]
    for buf, _, res, launches in runs:
        assert buf == runs[0][0] and buf == d and launches["window_resolve_kernel"] > 0
        assert res.tobytes() == runs[0][2].tobytes()
    # small blocks (memLevel 1: 128 symbols each): many short pieces, the scratch stays within its bound
    t = synth.text(4 * MIB, 171).tobytes()
    s = _raw(t, 6, 1)
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info()
    _compare(engine, [s], [t], route=None)
    free1, _ = torch.cuda.mem_get_info()
    assert free0 - free1 < 4 * 2048 * len(s) + (256 << 20), (free0 - free1, len(s))
