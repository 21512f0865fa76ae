"""GPU: random access through an index of access points (zlb_inflate_index / zlb_inflate_ranges). The build is
compared with zlb_inflate_batch + ZLB_INFLATE_SPLIT field by field and byte by byte on every route the split takes;
its points are checked against the block starts a reference walker (below) reads from the streams; reads are
compared with CPython's zlib output."""
import gzip
import json
import os
import zlib

import numpy as np
import pytest

from helpers import pack, rand_bytes

pytestmark = pytest.mark.gpu

FIELDS = ("status", "out_len", "in_used", "blocks", "crc32", "adler32")
MIB = 1 << 20


def _raw(data, level=6, mem=8, strategy=zlib.Z_DEFAULT_STRATEGY):
    co = zlib.compressobj(level, zlib.DEFLATED, -15, mem, strategy)
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


class Built:
    """One index build over streams (device entry point) and the plain SPLIT decode of the same items."""

    def __init__(self, engine, streams, caps, spacing, slots=None, flags=None):
        import torch
        import zlibts_b200 as z
        self.streams = [bytes(s) for s in streams]
        blob, offs, lens = pack(self.streams)
        self.caps = list(caps)
        self.ooffs = np.concatenate([[0], np.cumsum(self.caps)]).astype(np.uint64)
        items = z.make_items(len(streams))
        items["in_off"], items["in_len"] = offs, lens
        items["out_off"], items["out_cap"] = self.ooffs[:-1], self.caps
        self.items = items
        flags = z.INFLATE_WANT_CRC32 | z.INFLATE_WANT_ADLER32 if flags is None else flags
        self.d_in = torch.from_numpy(blob).cuda()
        self.d_out = torch.full((max(int(self.ooffs[-1]), 1),), 0xA5, dtype=torch.uint8, device="cuda")
        slots = [max(c // spacing, 1) + 2 for c in self.caps] if slots is None else slots
        self.first = np.concatenate([[0], np.cumsum(slots)]).astype(np.uint64)
        (self.res, self.points, self.counts), self.launches = _profiled(
            engine, lambda: engine.inflate_index(self.d_in, self.d_out, items, self.first, spacing, flags))
        d_ref = torch.full_like(self.d_out, 0xA5)
        self.ref, self.ref_launches = _profiled(engine, lambda: engine.inflate_batch(self.d_in, d_ref, items,
                                                                                     flags | z.INFLATE_SPLIT))
        self.out = self.d_out.cpu().numpy().tobytes()
        self.ref_out = d_ref.cpu().numpy().tobytes()

    def pts(self, i):
        a = int(self.first[i])
        return self.points[a:a + int(self.counts[i])]

    def check_equal_to_split(self):
        for i in range(len(self.streams)):
            for f in FIELDS:
                assert int(self.res[i][f]) == int(self.ref[i][f]), (i, f, int(self.res[i][f]), int(self.ref[i][f]))
            if int(self.res[i]["status"]) != 0:
                assert int(self.counts[i]) == 0, i
        assert self.out == self.ref_out
        for k in ("block_find_kernel", "marker_scan_kernel", "inflate_warp_kernel_window", "segment_gather_kernel"):
            assert self.launches.get(k, 0) == self.ref_launches.get(k, 0), (k, self.launches, self.ref_launches)
        # the one-warp launch behind the split is the points instantiation; the marker route's own launches stay
        assert self.ref_launches["inflate_warp_kernel_points"] == 0 and self.launches["inflate_warp_kernel_points"] <= 1
        assert (self.launches["inflate_warp_kernel"] + self.launches["inflate_warp_kernel_points"] ==
                self.ref_launches["inflate_warp_kernel"])

    def check_points(self, spacing):
        for i in range(len(self.streams)):
            p = self.pts(i)
            if int(self.res[i]["status"]) != 0:
                continue
            assert len(p) >= 1 and int(p[0]["in_bit"]) == 0 and int(p[0]["out_pos"]) == 0, i
            assert (np.diff(p["in_bit"].astype(np.int64)) > 0).all() and (np.diff(p["out_pos"].astype(np.int64)) >= spacing).all()
            wl = np.minimum(p["out_pos"], 32768)
            assert (p["win_off"] == self.ooffs[i] + p["out_pos"] - wl).all(), i


# ---- reference walker: block starts and the output in front of each --------------------------------------------
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
    """(bit offset, BTYPE, output bytes in front) of every block of the raw deflate stream s, read by walking its
    symbols"""
    buf = bytes(s) + b"\0" * 8
    pos = op = 0
    out = []

    def peek(p):
        return int.from_bytes(buf[p >> 3:(p >> 3) + 5], "little") >> (p & 7)

    fixed = _table([8] * 144 + [9] * 112 + [7] * 24 + [8] * 8), _table([5] * 30)
    while True:
        h = peek(pos)
        final, btype = h & 1, (h >> 1) & 3
        out.append((pos, btype, op))
        pos += 3
        if btype == 0:
            pos = (pos + 7) & ~7
            n = peek(pos) & 0xFFFF
            pos += 32 + 8 * n
            op += n
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
                    op += 1
                    continue
                if sym == 256:
                    break
                op += _LBASE[sym - 257] + (peek(pos) & ((1 << _LEXTRA[sym - 257]) - 1))
                pos += _LEXTRA[sym - 257]
                e = dt[peek(pos) & dm]
                pos += (e & 15) + _DEXTRA[e >> 4]
        if final:
            return out


def _greedy(starts, spacing):
    taken, due = [], 0
    for b, _, op in starts:
        if op >= due:
            taken.append((b, op))
            due = op + spacing
    return taken


def _assert_block_starts(points, starts):
    truth = {(b, op) for b, _, op in starts}
    for p in points:
        assert (int(p["in_bit"]), int(p["out_pos"])) in truth, (int(p["in_bit"]), int(p["out_pos"]))


# ---- build = decode ----------------------------------------------------------------------------------------------
def test_marker_route_64_mib_gpu_stream(engine):
    import zlibts_b200 as z
    from zlibts_b200 import synth
    d = synth.mixed(64 * MIB, 201).tobytes()
    s = _gpu_deflate(engine, d, z.MODE_COMPAT)
    b = Built(engine, [s], [len(d)], MIB)
    b.check_equal_to_split()
    b.check_points(MIB)
    p = b.pts(0)
    assert len(p) >= 16 and b.launches["inflate_warp_kernel_points"] == 0 and b.launches["block_find_kernel"] == 0
    assert b.out[:len(d)] == d
    # every point is a chunk start of this engine's stream: behind a sync-flush marker, at a multiple of 64 KiB
    for q in p[1:]:
        assert int(q["in_bit"]) % 8 == 0 and s[int(q["in_bit"]) // 8 - 4:int(q["in_bit"]) // 8] == b"\0\0\xff\xff"
        assert int(q["out_pos"]) % 65536 == 0
    _check_reads(engine, b, 0, d, np.random.default_rng(202), 24)


def test_primed_and_searched_routes(engine):
    import zlibts_b200 as z
    from zlibts_b200 import synth
    text = synth.text(4 * MIB, 211).tobytes()
    mixed = synth.mixed(4 * MIB + 333, 212).tobytes()
    datas = [mixed, text, text, mixed, text]
    streams = [_gpu_deflate(engine, mixed, z.MODE_PRIMED), _raw(text, 1), _raw(text, 6), _raw(mixed, 9),
               _raw(text, 6, 1)]
    spacing = 256 << 10
    b = Built(engine, streams, [len(x) for x in datas], spacing)
    b.check_equal_to_split()
    b.check_points(spacing)
    assert b.launches["inflate_warp_kernel_window"] > 0 and b.launches["block_find_kernel"] > 0
    assert b.launches["inflate_warp_kernel_points"] == 0
    rng = np.random.default_rng(213)
    for i, (s, d) in enumerate(zip(streams, datas)):
        assert b.out[int(b.ooffs[i]):int(b.ooffs[i]) + len(d)] == d
        assert len(b.pts(i)) >= 8, (i, len(b.pts(i)))
        if 0 < i < 4:   # (the primed stream's piece starts are checked by the reads; memLevel 1 is slow to walk)
            _assert_block_starts(b.pts(i), block_starts(s))
        _check_reads(engine, b, i, d, rng, 12)


def test_one_warp_route(engine):
    """Z_FIXED (the split finds no block to cut at) and items under 256 KiB: every block header is a candidate; the
    points are the greedy choice over the walker's block starts."""
    from zlibts_b200 import synth
    rng = np.random.default_rng(221)
    datas = [synth.text(2 * MIB, 222).tobytes(), synth.mixed(200000, 223).tobytes(), synth.text(100000, 224).tobytes(),
             rand_bytes(rng, 150000).tobytes()]
    streams = [_raw(datas[0], 6, 8, zlib.Z_FIXED), _raw(datas[1], 6, 1), _raw(datas[2], 9, 1), _raw(datas[3], 6)]
    starts = [block_starts(s) for s in streams]
    for spacing in (16384, 65536):
        b = Built(engine, streams, [len(x) for x in datas], spacing)
        b.check_equal_to_split()
        b.check_points(spacing)
        assert b.launches["inflate_warp_kernel_points"] == 1
        for i, s in enumerate(streams):
            want = _greedy(starts[i], spacing)
            got = [(int(p["in_bit"]), int(p["out_pos"])) for p in b.pts(i)]
            assert got == want, (spacing, i, got[:5], want[:5])
        for i, d in enumerate(datas):
            _check_reads(engine, b, i, d, rng, 8)
    # slots that run out: the first points only, the rest dropped
    b = Built(engine, streams[:1], [len(datas[0])], 16384, slots=[3])
    assert int(b.counts[0]) == 3
    assert [(int(p["in_bit"]), int(p["out_pos"])) for p in b.pts(0)] == _greedy(starts[0], 16384)[:3]


def test_stored_sync_flush_empty_and_corrupt_streams(engine):
    from zlibts_b200 import synth
    rng = np.random.default_rng(231)
    rnd = rand_bytes(rng, 6 * MIB).tobytes()
    m = synth.mixed(6 * MIB, 232).tobytes()
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    sync = b"".join(co.compress(m[k:k + 512 * 1024]) + co.flush(zlib.Z_SYNC_FLUSH) for k in range(0, len(m), 512 * 1024))
    sync += co.flush()
    vec = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "truncation_vectors.json")))["vectors"]
    bad = [bytes.fromhex(v["stream"])[:cut] for v in vec for cut in range(len(v["cuts"]))]
    big_bad = bytearray(_raw(m, 6))
    big_bad[len(big_bad) // 2] ^= 0x5A
    streams = [_raw(rnd, 6), sync, _raw(b""), bytes(big_bad), _raw(m, 6)[:len(big_bad) // 2]] + bad
    datas = [rnd, m, b"", None, None] + [None] * len(bad)
    caps = [len(rnd), len(m), 0, len(m), len(m)] + [4096] * len(bad)
    b = Built(engine, streams, caps, MIB)
    b.check_equal_to_split()
    b.check_points(MIB)
    assert int(b.counts[2]) == 1 and int(b.res[4]["status"]) != 0 and int(b.counts[4]) == 0
    assert any(int(b.res[i]["status"]) != 0 for i in range(5, len(streams)))
    for i in (0, 1):
        assert len(b.pts(i)) >= 4
        _assert_block_starts(b.pts(i), block_starts(streams[i]))
        _check_reads(engine, b, i, datas[i], rng, 10)


# ---- reads -------------------------------------------------------------------------------------------------------
def _ranges_for(b, i, spans, out_gap=17):
    import zlibts_b200 as z
    p = b.pts(i)
    rg = z.make_ranges(len(spans))
    caps = [l for _, l in spans]
    offs = np.concatenate([[0], np.cumsum(np.array(caps, dtype=np.int64) + out_gap)]).astype(np.uint64)
    rg["in_off"], rg["in_len"] = b.items["in_off"][i], b.items["in_len"][i]
    rg["pt_first"], rg["pt_count"] = 0, len(p)
    rg["pos"] = [pp for pp, _ in spans]
    rg["out_off"], rg["out_cap"] = offs[:-1] + out_gap, caps
    return rg, int(offs[-1]) + out_gap


def _spans(rng, p, size, n):
    """random (pos, len): around points, across many of them, the whole stream, past the end, at the end"""
    pos = [int(x) for x in p["out_pos"]]
    spans = [(0, size), (size, 100), (size + 5, 10), (max(size - 7, 0), 100), (0, 0)]
    for _ in range(n):
        k = int(rng.integers(0, len(pos)))
        at = max(0, pos[k] + int(rng.integers(-1, 2)))
        far = pos[min(len(pos) - 1, k + int(rng.integers(1, 4)))] - at + int(rng.integers(0, 5000))
        spans += [(at, int(rng.integers(1, 70000))), (at, max(far, 1)), (int(rng.integers(0, size + 1)), int(rng.integers(0, 300000)))]
    return spans


def _read(engine, b, i, rg, total, flags=0, points=None):
    import torch
    d_out = torch.full((total,), 0xA5, dtype=torch.uint8, device="cuda")
    res = engine.inflate_ranges(b.d_in, b.d_out, d_out, b.pts(i) if points is None else points, rg, flags)
    return res, d_out.cpu().numpy().tobytes()


def _check_reads(engine, b, i, d, rng, n):
    import zlibts_b200 as z
    p = b.pts(i)
    spans = _spans(rng, p, len(d), n)
    rg, total = _ranges_for(b, i, spans)
    flags = z.INFLATE_WANT_CRC32 | z.INFLATE_WANT_ADLER32
    res, out = _read(engine, b, i, rg, total, flags)
    untouched = bytearray(b"\xA5" * total)
    for r, g, (pos, ln) in zip(res, rg, spans):
        want = d[pos:pos + ln]
        o = int(g["out_off"])
        assert int(r["status"]) == 0 and int(r["out_len"]) == len(want), (pos, ln, int(r["status"]), int(r["out_len"]))
        assert out[o:o + len(want)] == want, (pos, ln)
        assert int(r["crc32"]) == zlib.crc32(want) and int(r["adler32"]) == zlib.adler32(want), (pos, ln)
        assert int(r["in_used"]) == 0 and int(r["blocks"]) == 0
        untouched[o:o + len(want)] = want
    assert out == bytes(untouched)   # nothing behind a read's bytes, nothing between the slots
    # the same reads with only the first point and with every other point: the same bytes
    for sub in (p[:1], p[::2]):
        rg2 = rg.copy()
        rg2["pt_count"] = len(sub)
        res2, out2 = _read(engine, b, i, rg2, total, 0, sub)
        assert out2 == out and (res2["out_len"] == res["out_len"]).all() and (res2["status"] == 0).all()
    # windows from a compacted blob
    import torch
    wl = np.minimum(p["out_pos"], 32768)
    wins = b"".join(b.out[int(w):int(w) + int(n)] for w, n in zip(p["win_off"], wl))
    q = p.copy()
    q["win_off"] = np.concatenate([[0], np.cumsum(wl)[:-1]]).astype(np.uint64)
    d_out = torch.full((total,), 0xA5, dtype=torch.uint8, device="cuda")
    d_win = torch.from_numpy(np.frombuffer(wins + b"\0", dtype=np.uint8).copy()).cuda()
    res3 = engine.inflate_ranges(b.d_in, d_win, d_out, q, rg, 0)
    assert d_out.cpu().numpy().tobytes() == out and (res3["out_len"] == res["out_len"]).all()


def test_ranges_of_several_streams_in_one_call_and_host_entry_points(engine):
    import zlibts_b200 as z
    from zlibts_b200 import synth
    datas = [synth.text(3 * MIB, 241).tobytes(), synth.mixed(3 * MIB, 242).tobytes(), synth.text(500000, 243).tobytes()]
    streams = [_raw(datas[0], 6), _raw(datas[1], 6, 8, zlib.Z_FIXED), _raw(datas[2], 6)]
    b = Built(engine, streams, [len(x) for x in datas], 128 << 10)
    b.check_equal_to_split()
    rng = np.random.default_rng(244)
    # every stream's points in one table, windows in the build's output blob; ranges interleaved
    allp = np.concatenate([b.pts(i) for i in range(3)])
    base = np.concatenate([[0], np.cumsum([len(b.pts(i)) for i in range(3)])])
    spans = []
    for k in range(300):
        i = k % 3
        pos = int(rng.integers(0, len(datas[i]) + 10))
        spans.append((i, pos, int(rng.integers(0, 400000))))
    rg = z.make_ranges(len(spans))
    caps = np.array([ln for _, _, ln in spans], dtype=np.uint64)
    offs = np.concatenate([[0], np.cumsum(caps)]).astype(np.uint64)
    for k, (i, pos, ln) in enumerate(spans):
        rg[k] = (b.items["in_off"][i], b.items["in_len"][i], base[i], len(b.pts(i)), pos, offs[k], ln)
    flags = z.INFLATE_WANT_CRC32
    outs = []
    h_in = b.d_in.cpu().numpy()
    for mode in ("device", "pinned", "pageable"):
        if mode == "device":
            import torch
            d_out = torch.full((int(offs[-1]) + 1,), 0xA5, dtype=torch.uint8, device="cuda")
            res = engine.inflate_ranges(b.d_in, b.d_out, d_out, allp, rg, flags)
            out = d_out.cpu().numpy()
        else:
            win = np.frombuffer(b.out, dtype=np.uint8)
            if mode == "pinned":
                hi, hw, out = z.host_alloc(h_in.size), z.host_alloc(win.size), z.host_alloc(int(offs[-1]) + 1)
                hi[:], hw[:] = h_in, win
            else:
                hi, hw, out = h_in.copy(), win.copy(), np.empty(int(offs[-1]) + 1, dtype=np.uint8)
            out[:] = 0xA5
            res = engine.inflate_ranges_host(hi, hw, out, allp, rg, flags)
            out = out.copy()
        for k, (i, pos, ln) in enumerate(spans):
            want = datas[i][pos:pos + ln]
            assert int(res[k]["status"]) == 0 and int(res[k]["out_len"]) == len(want), (mode, k)
            assert out[int(offs[k]):int(offs[k]) + len(want)].tobytes() == want, (mode, k)
            assert int(res[k]["crc32"]) == zlib.crc32(want)
        outs.append((res.tobytes(), out.tobytes()))
    assert outs[0] == outs[1] == outs[2]
    # the index build's own _host entry point: the device call's results, bytes and points
    h_out = np.full(len(b.out), 0xA5, dtype=np.uint8)
    res, points, counts = engine.inflate_index_host(h_in, h_out, b.items, b.first, 128 << 10,
                                                    z.INFLATE_WANT_CRC32 | z.INFLATE_WANT_ADLER32)
    assert res.tobytes() == b.res.tobytes() and (counts == b.counts).all()
    for i in range(3):
        a = int(b.first[i])
        assert points[a:a + int(counts[i])].tobytes() == b.pts(i).tobytes()
        lo = int(b.ooffs[i])
        assert h_out[lo:lo + len(datas[i])].tobytes() == datas[i]


def test_first_piece_scratch_beyond_the_budget_runs_in_waves(engine):
    """Reads far behind their only point: each decodes ~15 MiB into scratch; 1200 of them need more than the 16 GiB a
    call's scratch may take, so they run in more than one wave."""
    import torch
    from zlibts_b200 import synth
    d = synth.text(16 * MIB, 251).tobytes()
    s = _raw(d, 6, 8, zlib.Z_FIXED)
    b = Built(engine, [s], [len(d)], MIB)
    n = 1200
    spans = [(15 * MIB + 700 * k, 4096) for k in range(n)]   # (all inside the stream: every piece gathers)
    rg, total = _ranges_for(b, 0, spans, 0)
    rg["pt_count"] = 1
    d_out = torch.full((total,), 0xA5, dtype=torch.uint8, device="cuda")
    res, launches = _profiled(engine, lambda: engine.inflate_ranges(b.d_in, b.d_out, d_out, b.pts(0)[:1], rg, 0))
    assert launches["inflate_warp_kernel_range"] >= 2 and launches["segment_gather_kernel"] >= 2, launches
    out = d_out.cpu().numpy().tobytes()
    for k, (pos, ln) in enumerate(spans):
        assert int(res[k]["status"]) == 0 and out[4096 * k:4096 * (k + 1)] == d[pos:pos + ln], k


def test_refusals(engine):
    import torch
    import zlibts_b200 as z
    from zlibts_b200 import synth
    d = synth.text(600000, 261).tobytes()
    b = Built(engine, [_raw(d, 6, 1)], [len(d)], 65536)
    p = b.pts(0)
    assert len(p) > 3

    def ranges(**kw):
        rg, total = _ranges_for(b, 0, [(1000, 100)])
        for k, v in kw.items():
            rg[k] = v
        return rg

    d_out = torch.zeros(1 << 16, dtype=torch.uint8, device="cuda")
    cases = [(p, ranges(pt_count=0), 0, "no access points"),
             (p, ranges(pt_first=1, pt_count=len(p) - 1), 0, "first point is not {0, 0}"),
             (p[[0, 2, 1]], ranges(pt_count=3), 0, "do not ascend"),
             (p, ranges(in_len=int(p[-1]["in_bit"]) // 8), 0, "behind the stream"),
             (p, ranges(pt_count=len(p) + 1), 0, "outside the point table"),
             (p, ranges(), z.INFLATE_SPLIT, "takes ZLB_INFLATE_WANT_CRC32")]
    for pts, rg, flags, text in cases:
        with pytest.raises(z.EngineError, match=text):
            engine.inflate_ranges(b.d_in, b.d_out, d_out, pts, rg, flags)
    h_in, h_win = b.d_in.cpu().numpy(), np.frombuffer(b.out, dtype=np.uint8)
    h_out = np.zeros(1 << 16, dtype=np.uint8)
    for pts, rg, flags, text in cases:
        with pytest.raises(z.EngineError, match=text):
            engine.inflate_ranges_host(h_in, h_win, h_out, pts, rg, flags)
    with pytest.raises(z.EngineError, match="window of point"):
        engine.inflate_ranges_host(h_in, h_win[:int(p[-1]["win_off"]) + 100], h_out, p, ranges(), 0)
    with pytest.raises(z.EngineError, match="slot lies outside the output"):
        engine.inflate_ranges_host(h_in, h_win, h_out[:50], p, ranges(), 0)
    with pytest.raises(z.EngineError, match="an index build takes"):
        engine.inflate_index(b.d_in, b.d_out, b.items, b.first, 0, z.INFLATE_SPLIT)
    # pos + out_cap beyond 2^64; windows named with a NULL window blob
    for call, win in ((lambda rg, w: engine.inflate_ranges(b.d_in, w, d_out, p, rg, 0), b.d_out),
                      (lambda rg, w: engine.inflate_ranges_host(h_in, w, h_out, p, rg, 0), h_win)):
        with pytest.raises(z.EngineError, match="pos \\+ out_cap overflows"):
            call(ranges(pos=2**64 - 100, out_cap=101), win)
        with pytest.raises(z.EngineError, match="window blob is NULL"):
            call(ranges(), None)
    res = engine.inflate_ranges(b.d_in, None, d_out, p[:1], ranges(pt_count=1), 0)   # (no window needed: point {0, 0})
    assert int(res["status"][0]) == 0 and int(res["out_len"][0]) == 100


def test_reads_far_past_the_end(engine):
    """A pos beyond what the stream can give from the point in front of it is a read past the end: out_len 0, nothing
    decoded and no scratch taken, whatever pos is (the stream's input bounds its output: 258 bytes per bit). A first
    piece whose scratch alone exceeds what a call may take is refused with ZLB_E_NOMEM and a text."""
    import torch
    import zlibts_b200 as z
    from zlibts_b200 import synth
    d = synth.text(300000, 291).tobytes()
    b = Built(engine, [_raw(d, 6)], [len(d)], MIB)
    assert len(b.pts(0)) == 1
    spans = [(2**64 - 100, 99), (2**63, 4096), (len(d) + 1000, 50), (len(d) - 10, 50), (5, 20)]
    rg, total = _ranges_for(b, 0, spans)
    d_out = torch.full((total,), 0xA5, dtype=torch.uint8, device="cuda")
    res, launches = _profiled(engine, lambda: engine.inflate_ranges(b.d_in, b.d_out, d_out, b.pts(0), rg, 0))
    assert [int(r["out_len"]) for r in res] == [0, 0, 0, 10, 20] and (res["status"] == 0).all()
    assert launches["inflate_warp_kernel_range"] == 1 and launches["segment_gather_kernel"] == 1, launches
    out = d_out.cpu().numpy().tobytes()
    assert out[int(rg[3]["out_off"]):int(rg[3]["out_off"]) + 10] == d[-10:]
    assert out.count(0xA5) == total - 30
    # 10 MB of stored blocks can give 20 GB as far as the host knows: a read 17 GiB in asks for more scratch than a
    # call may take (at most 16 GiB)
    rnd = rand_bytes(np.random.default_rng(292), 10 << 20).tobytes()
    b = Built(engine, [_raw(rnd, 0)], [len(rnd)], 64 * MIB)
    rg, total = _ranges_for(b, 0, [(17 << 30, 1)])
    d_out = torch.zeros(total, dtype=torch.uint8, device="cuda")
    with pytest.raises(z.EngineError, match="into scratch, more than"):
        engine.inflate_ranges(b.d_in, b.d_out, d_out, b.pts(0), rg, 0)


# ---- the Python surface ------------------------------------------------------------------------------------------
def test_api_round_trips(engine):
    import zlibts_b200 as Z
    from zlibts_b200 import synth
    Z.api.set_engine(engine)
    d = synth.mixed(5 * MIB, 271).tobytes()
    rng = np.random.default_rng(272)
    for kind, data in (("raw", _raw(d, 6)), ("zlib", zlib.compress(d, 6)), ("gzip", gzip.compress(d, 6))):
        out, idx = Z.inflate_index(data, kind, spacing=256 << 10)
        assert out.tobytes() == d and len(idx) >= 10 and idx.size == len(d)
        idx2 = Z.InflateIndex.from_bytes(idx.to_bytes())
        assert idx2.to_bytes() == idx.to_bytes() and len(idx.to_bytes()) == idx.nbytes
        spans = [(int(rng.integers(0, len(d))), int(rng.integers(0, 1 << 20))) for _ in range(40)] + [(len(d) - 3, 10)]
        for got, (pos, ln) in zip(idx2.read_many(data, spans), spans):
            assert got.tobytes() == d[pos:pos + ln], (kind, pos, ln)
        assert idx.read(data, 12345, 777).tobytes() == d[12345:12345 + 777]
        with pytest.raises(Z.ZlibError, match="does not belong to this index"):
            idx.read(data + b"\0", 0, 10)
    # reads of several streams in one call
    e = synth.text(2 * MIB, 273).tobytes()
    ze = zlib.compress(e, 9)
    _, ie = Z.inflate_index(ze, "zlib", spacing=65536)
    g = gzip.compress(d, 6)
    _, ig = Z.inflate_index(g, "gzip", spacing=MIB)
    reads = [(ze, ie, 1000, 5000), (g, ig, 3 * MIB, 70000), (ze, ie, len(e) - 10, 100)]
    got, res = Z.read_ranges(reads, want_crc32=True)
    for o, r, (_, _, pos, ln), src in zip(got, res, reads, (e, d, e)):
        assert o.tobytes() == src[pos:pos + ln] and int(r["crc32"]) == zlib.crc32(src[pos:pos + ln])


def test_api_refusals(engine):
    import zlibts_b200 as Z
    from zlibts_b200 import synth
    Z.api.set_engine(engine)
    d = synth.text(MIB, 281).tobytes()
    g = bytearray(gzip.compress(d, 6))
    g[-6] ^= 1   # CRC-32
    with pytest.raises(Z.ZlibError, match="invalid CRC-32 checksum"):
        Z.inflate_index(bytes(g), "gzip")
    with pytest.raises(Z.ZlibError, match="multi-member"):
        Z.inflate_index(gzip.compress(d[:1000]) + gzip.compress(d[1000:]), "gzip")
    c = bytearray(zlib.compress(d))
    c[-1] ^= 1
    with pytest.raises(Z.ZlibError, match="invalid adler-32 checksum"):
        Z.inflate_index(bytes(c), "zlib")
    with pytest.raises(Z.ZlibError, match="invalid file signature"):
        Z.inflate_index(b"\x1f\x8c" + bytes(20), "gzip")
    with pytest.raises(Z.ZlibError, match="unsupported compression method"):
        Z.inflate_index(b"\x79\x9c" + bytes(20), "zlib")
