"""Host-side mirror of the zlib.ts public surface over the C-ABI engine.

The reference is TypeScript (`window.Zlib = {GZip, GUnzip, Zip, Unzip, Deflate, Inflate}`, src/index.ts:8-12) and
no Node toolchain exists in this image, so the glue that stays on the host -- container headers and trailers,
option handling, error texts -- is restated here in Python with the reference's class names, option names and
thrown messages, and every call that the reference makes into RawDeflate / RawInflate / CRC32 / Adler32 goes to
the GPU through zlibts_b200._native.Engine (no CPU fallback). napi/ holds the same glue as the N-API addon +
TypeScript shim a maintainer would ship (INTEGRATION.md).

Deviations from the reference, all deliberate (SURVEY.md Appendix B):
  * inputs larger than one chunk (64 KiB) are emitted as several blocks joined by sync-flush markers instead of
    one block; the result is a valid stream that the reference's own Inflate / GUnzip / Unzip decodes.
  * Deflate.compress does not raise the reference's RangeError for outputs > 32 KiB (B-1): it returns header +
    body + Adler-32 as evidently intended.
  * `lazy` > 0 is refused: the reference corrupts data with it (B-2).
  * `b200: {mode: "fast" | "primed" | "fast-primed"}` selects the engine's other modes (valid streams, not the
    reference's bytes; default is the reference-compatible mode).
  * an empty input with compressionType FIXED gets its end-of-block symbol ("03 00"); upstream drops it ("03",
    which no inflater accepts) because LZ77's output array has length 0 there (src/LZ77.ts:122,278).
  * corrupt streams that make the reference loop or emit zeros (B-8) raise ZlibError instead.
  * ZipCrypto (password) is out of scope (SURVEY section 2: serial byte cipher, broken upstream).
  * preset dictionaries (zlib's deflateSetDictionary / inflateSetDictionary): `b200: {dictionary}` on RawDeflate,
    RawInflate, Deflate and Inflate, `dictionary=` on the batch functions. Deflate then writes FLG.FDICT and DICTID
    (RFC 1950); Inflate reads FDICT streams when given the dictionary whose Adler-32 is DICTID, where the reference
    always throws "fdict flag is not supported" (it still does here without a dictionary). A dictionary given for a
    stream without FDICT is ignored, as zlib does. Only a dictionary's last 32 KiB can be reached.
  * decompressed sizes without decoding the bytes: `inflate_sizes` (zlb_inflate_size_batch) returns what each stream
    inflates to, so that the output slots of `inflate_many(..., size_hints=sizes)` or RawInflate's `bufferSize` are
    exact and that call needs no retry. The reference has no such query (its buffer grows while it decodes).
  * random access (zlb_inflate_index / zlb_inflate_ranges): `inflate_index` decodes a raw, zlib or gzip stream once and
    keeps access points -- proven block starts with the 32 KiB window in front of each -- in an `InflateIndex`, whose
    `read` / `read_many` (and `read_ranges` across streams) decode only from the last point in front of a range. What
    zlib's zran.c and indexed_gzip offer; the reference has nothing of the kind.
"""
import datetime
import struct

import numpy as np

from . import _native as N


class ZlibError(Exception):
    """`throw new Error(msg)` of the reference; str(e) is the reference's message text."""


class CompressionType:  # src/RawDeflate.ts:12-17
    NONE, FIXED, DYNAMIC, RESERVED = 0, 1, 2, 3


class BufferType:  # src/RawInflate.ts:5-8 (accepted, irrelevant on the GPU: output slots are sized up front)
    BLOCK, ADAPTIVE = 0, 1


class ZipCompressionMethod:  # src/Zip.ts:7-10
    STORE, DEFLATE = 0, 8


_STATUS_TEXT = {  # zlb_result.status -> reference message (include/zlibts_b200.h)
    N.ST_INPUT_BROKEN: "input buffer is broken",
    N.ST_BTYPE: "unknown BTYPE: 3",
    N.ST_STORED_LEN: "invalid uncompressed block header: LEN",
    N.ST_BAD_CODE: "invalid deflate stream: undefined code or distance",
    N.ST_BAD_LENGTHS: "invalid deflate stream: over-subscribed code lengths",
}


def status_text(st):
    """The reference's message for a zlb_result.status (src/RawInflate.ts:168,188,238,266,272)."""
    st = int(st)
    if (st & 0xFF) == N.ST_CODE_LENGTH:
        return "invalid code length: %d" % (st >> 8)
    if (st & 0xFF) == N.ST_STORED_LEN and (st >> 8):
        return "invalid uncompressed block header: NLEN"
    return _STATUS_TEXT.get(st & 0xFF, "inflate failed with status %d" % st)


_engine = None


def set_engine(engine):
    """Use this Engine for every call made through this module (default: one engine on device 0)."""
    global _engine
    _engine = engine


def engine():
    global _engine
    if _engine is None:
        _engine = N.default_engine(0)
    return _engine


def _u8(data):
    if isinstance(data, np.ndarray):
        return np.ascontiguousarray(data, dtype=np.uint8).reshape(-1)
    if isinstance(data, (bytes, bytearray, memoryview)):
        return np.frombuffer(data, dtype=np.uint8)
    return np.asarray(list(data), dtype=np.uint8)  # number[]


def _opt(opts, key, default):
    v = (opts or {}).get(key)
    return default if v is None else v  # the reference's `??`


def _b200(opts):
    return (opts or {}).get("b200") or {}


# ------------------------------------------------------------------------------------------------------------
# batch entry points (what the N-API addon exposes below the classes)
# ------------------------------------------------------------------------------------------------------------
def _mode_of(opts):
    """engine-only knob `b200: {mode: 'compat' | 'fast' | 'primed' | 'fast-primed', depth: N, lazy: bool}` (default:
    reference-compatible bytes). 'primed' = every chunk also searches the 32 KiB in front of it (better ratio,
    still one stream the reference inflates, no longer RawDeflate(chunk) per chunk)."""
    b = _b200(opts)
    name = b.get("mode", "compat")
    if name not in ("compat", "fast", "primed", "fast-primed"):
        raise ZlibError("unknown b200 mode: %s" % name)
    mode = N.mode_fast(int(b.get("depth", 0))) if name.startswith("fast") else N.MODE_COMPAT
    # `lazy: true` (fast modes only): one-step lazy evaluation that is actually correct -- what src/LZ77.ts:243-256 meant
    # to do; the reference's own `lazy` option corrupts data and stays refused
    if b.get("lazy"):
        if not name.startswith("fast"):
            raise ZlibError("b200.lazy needs a fast mode: the compat mode is the reference's greedy parse")
        mode |= N.MODE_LAZY
    # `smallest: true` lets every chunk fall back to a fixed or stored block when that is shorter
    return mode | (N.MODE_PRIMED if name.endswith("primed") else 0) | (N.MODE_SMALLEST if b.get("smallest") else 0)


def _dict_table(dictionary, n):
    """(dictionary blob, zlb_dict table) for `dictionary` = None | bytes-like (every item) | list (one entry per
    item, None = no dictionary); (None, None) when no item has one. Equal dictionaries are stored once."""
    if dictionary is None:
        return None, None
    per_item = [dictionary] * n if not isinstance(dictionary, (list, tuple)) else list(dictionary)
    if len(per_item) != n:
        raise ZlibError("dictionary list must have one entry per input")
    table = N.make_dicts(n)
    parts, at, where = [], 0, {}
    for i, d in enumerate(per_item):
        if d is None:
            continue
        key = _u8(d).tobytes()
        if not key:
            continue
        if key not in where:
            where[key] = at
            parts.append(key)
            at += len(key)
        table[i] = (where[key], len(key))
    if not parts:
        return None, None
    return np.frombuffer(b"".join(parts), dtype=np.uint8), table


def deflate_many(inputs, compression_type=CompressionType.DYNAMIC, chunk_bytes=0, want_crc32=False,
                 want_adler32=False, prefixes=None, mode=N.MODE_COMPAT, dictionary=None):
    """Raw-deflates every input in one GPU batch. Returns (list of uint8 arrays, results table). With `prefixes`
    each output starts with its prefix bytes (RawDeflate's outputBuffer / outputIndex contract). `dictionary`: a
    preset dictionary for every input (bytes-like) or one per input (a list; None entries have none)."""
    arrs = [_u8(x) for x in inputs]
    n = len(arrs)
    if n == 0:
        return [], np.zeros(0, dtype=N.RESULT_DTYPE)
    if compression_type not in (0, 1, 2):
        raise ZlibError("invalid compression type")  # src/RawDeflate.ts:110 (a thrown string there)
    dblob, dicts = _dict_table(dictionary, n)
    lens = np.array([a.size for a in arrs], dtype=np.uint64)
    in_off = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.uint64)
    blob = np.concatenate(arrs) if int(lens.sum()) else np.zeros(1, dtype=np.uint8)
    caps = np.array([N.deflate_bound(int(l), chunk_bytes, compression_type, mode, dicts is not None) for l in lens],
                    dtype=np.uint64)
    out_off = np.concatenate([[0], np.cumsum(caps)[:-1]]).astype(np.uint64)
    out = np.zeros(int(caps.sum()), dtype=np.uint8)
    items = N.make_items(n)
    items["in_off"], items["in_len"], items["out_off"], items["out_cap"] = in_off, lens, out_off, caps
    flags = (N.DEFLATE_WANT_CRC32 if want_crc32 else 0) | (N.DEFLATE_WANT_ADLER32 if want_adler32 else 0)
    res = engine().deflate_batch_host(blob, out, items, compression_type, chunk_bytes, flags, mode, dblob, dicts)
    outs = []
    for i in range(n):
        if int(res["status"][i]) != N.ST_OK:
            raise ZlibError("deflate failed with status %d" % int(res["status"][i]))
        body = out[int(out_off[i]):int(out_off[i]) + int(res["out_len"][i])]
        if prefixes is not None and len(prefixes[i]):
            body = np.concatenate([_u8(prefixes[i]), body])
        outs.append(body)
    return outs, res


def inflate_blob(blob, offs, lens, size_hints=None, want_crc32=False, want_adler32=False, split=True, tolerant=False,
                 dictionary=None):
    """Raw-inflates the streams blob[offs[i] : offs[i] + lens[i]] in one GPU batch; output slots that turn out
    too small are retried larger (the reference grows its buffer instead, src/RawInflate.ts:550-581).
    Returns (list of uint8 arrays, results table); raises ZlibError with the reference's text on corrupt input.
    `tolerant`: nothing is raised or retried -- a stream that fails or overflows its slot comes back as None with its
    status in the table (speculative decoding of gzip member candidates). `dictionary`: as for deflate_many."""
    blob = _u8(blob)
    n = len(offs)
    if n == 0:
        return [], np.zeros(0, dtype=N.RESULT_DTYPE)
    dblob, dicts = _dict_table(dictionary, n)
    offs = np.asarray(offs, dtype=np.uint64)
    lens = np.asarray(lens, dtype=np.uint64)
    caps = np.zeros(n, dtype=np.uint64)
    for i in range(n):
        hint = None if size_hints is None else size_hints[i]
        caps[i] = int(hint) if hint is not None else max(0x8000, 4 * int(lens[i]))  # DefaultInflateBufferSize
    # large streams decode piecewise wherever the engine can prove a block boundary: at sync-flush markers, and in any
    # other stream (gzip, zlib.compress, ...) at block starts found on the device (same result, see the header)
    flags = ((N.INFLATE_WANT_CRC32 if want_crc32 else 0) | (N.INFLATE_WANT_ADLER32 if want_adler32 else 0) |
             (N.INFLATE_SPLIT if split else 0))
    if blob.size == 0:
        blob = np.zeros(1, dtype=np.uint8)
    outs = [None] * n
    final = np.zeros(n, dtype=N.RESULT_DTYPE)
    todo = np.arange(n)
    for _ in range(12):
        m = len(todo)
        out_off = np.concatenate([[0], np.cumsum(caps[todo])[:-1]]).astype(np.uint64)
        out = np.zeros(max(1, int(caps[todo].sum())), dtype=np.uint8)
        items = N.make_items(m)
        items["in_off"], items["in_len"] = offs[todo], lens[todo]
        items["out_off"], items["out_cap"] = out_off, caps[todo]
        res = engine().inflate_batch_host(blob, out, items, flags, dblob, None if dicts is None else dicts[todo])
        again = []
        for k, i in enumerate(todo):
            st = int(res["status"][k])
            if tolerant and st != N.ST_OK:
                final[i] = res[k]
                continue
            if st == N.ST_OUT_OVERFLOW:
                caps[i] = max(int(caps[i]) * 4, 1 << 16)
                again.append(i)
                continue
            if st != N.ST_OK:
                raise ZlibError(status_text(st))
            outs[i] = out[int(out_off[k]):int(out_off[k]) + int(res["out_len"][k])]
            final[i] = res[k]
        if not again:
            return outs, final
        todo = np.array(again)
    raise ZlibError("inflate output does not fit")


def inflate_many(buffers, indices=None, size_hints=None, want_crc32=False, want_adler32=False, dictionary=None):
    """One stream per buffer, starting at indices[i] (RawInflate's `index` option); `dictionary` as for
    deflate_many."""
    arrs = [_u8(x) for x in buffers]
    n = len(arrs)
    if n == 0:
        return [], np.zeros(0, dtype=N.RESULT_DTYPE)
    idx = np.zeros(n, dtype=np.uint64) if indices is None else np.asarray(indices, dtype=np.uint64)
    lens = np.array([a.size for a in arrs], dtype=np.uint64)
    base = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.uint64)
    blob = np.concatenate(arrs) if int(lens.sum()) else np.zeros(1, dtype=np.uint8)
    idx = np.minimum(idx, lens)
    return inflate_blob(blob, base + idx, lens - idx, size_hints, want_crc32, want_adler32, dictionary=dictionary)


def inflate_sizes(buffers, indices=None, dictionary=None):
    """Decompressed size of the stream in every buffer (starting at indices[i]) as a uint64 array, from one size-only
    GPU call that writes no output (ZLB_INFLATE_SPLIT, as inflate_many); `dictionary` as for deflate_many (only its
    length matters). Raises ZlibError with the text inflate_many would raise for a corrupt stream."""
    arrs = [_u8(x) for x in buffers]
    n = len(arrs)
    if n == 0:
        return np.zeros(0, dtype=np.uint64)
    idx = np.zeros(n, dtype=np.uint64) if indices is None else np.asarray(indices, dtype=np.uint64)
    lens = np.array([a.size for a in arrs], dtype=np.uint64)
    base = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.uint64)
    blob = np.concatenate(arrs) if int(lens.sum()) else np.zeros(1, dtype=np.uint8)
    idx = np.minimum(idx, lens)
    _, dicts = _dict_table(dictionary, n)
    items = N.make_items(n)
    items["in_off"], items["in_len"] = base + idx, lens - idx
    res = engine().inflate_size_batch_host(blob, items, N.INFLATE_SPLIT, dicts)
    for st in res["status"]:
        if int(st) != N.ST_OK:
            raise ZlibError(status_text(st))
    return res["out_len"].astype(np.uint64)


def checksum_many(buffers, crc32=True, adler32=True):
    arrs = [_u8(x) for x in buffers]
    n = len(arrs)
    if n == 0:
        return np.zeros(0, dtype=N.RESULT_DTYPE)
    lens = np.array([a.size for a in arrs], dtype=np.uint64)
    off = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.uint64)
    blob = np.concatenate(arrs) if int(lens.sum()) else np.zeros(1, dtype=np.uint8)
    items = N.make_items(n)
    items["in_off"], items["in_len"] = off, lens
    return engine().checksum_batch_host(blob, items, (N.SUM_CRC32 if crc32 else 0) | (N.SUM_ADLER32 if adler32 else 0))


def archive_many(kind, inputs, heads, compression_type=CompressionType.DYNAMIC, chunk_bytes=0, mode=N.MODE_COMPAT,
                 methods=None, cdirs=None, tail=b""):
    """Checksums, deflates and frames every input on the device (zlb_archive_host): entry i becomes
    heads[i] | body | trailer, packed back to back; for FRAME_ZIP the central directory (cdirs) and the end
    record (tail) follow. Returns (archive as one uint8 array, results table: crc32 / adler32, out_len = framed
    bytes of the entry, in_used = its offset in the archive)."""
    arrs = [_u8(x) for x in inputs]
    n = len(arrs)
    if compression_type not in (0, 1, 2):
        raise ZlibError("invalid compression type")  # src/RawDeflate.ts:110
    lens = np.array([a.size for a in arrs], dtype=np.uint64)
    blob = np.concatenate(arrs) if n and int(lens.sum()) else np.zeros(1, dtype=np.uint8)
    parts = [bytes(h) for h in heads] + [bytes(c) for c in (cdirs or [])] + [bytes(tail)]
    plens = np.array([len(p) for p in parts], dtype=np.uint64)
    poffs = np.concatenate([[0], np.cumsum(plens)[:-1]]).astype(np.uint64)
    meta = np.frombuffer(b"".join(parts) or b"\0", dtype=np.uint8)
    ent = N.make_entries(n)
    if n:
        ent["in_off"] = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.uint64)
        ent["in_len"] = lens
        ent["head_off"], ent["head_len"] = poffs[:n], plens[:n]
        ent["method"] = 8 if methods is None else np.asarray(methods, dtype=np.uint32)
        if cdirs:
            ent["cdir_off"], ent["cdir_len"] = poffs[n:2 * n], plens[n:2 * n]
    out, res = engine().archive_host(kind, blob, meta, ent, (int(poffs[-1]), int(plens[-1])), compression_type,
                                     chunk_bytes, mode)
    return out, res


def zlib_many(inputs, compression_type=CompressionType.DYNAMIC, chunk_bytes=0, mode=N.MODE_COMPAT):
    """Every input as a zlib stream (what Deflate.compress returns), back to back in one buffer; stream i is
    archive[res['in_used'][i] : + res['out_len'][i]]."""
    return archive_many(N.FRAME_ZLIB, inputs, [_zlib_header(compression_type)] * len(inputs), compression_type,
                        chunk_bytes, mode)


def gzip_many(inputs, compression_type=CompressionType.DYNAMIC, chunk_bytes=0, mode=N.MODE_COMPAT, mtime=0):
    """Every input as one gzip member; the members back to back are one multi-member gzip file that
    GUnzip.decompress (src/GUnzip.ts:56-58) and gzip(1) read as the concatenation of the inputs."""
    hdr = b"\x1f\x8b\x08\x00" + struct.pack("<I", int(mtime) & 0xFFFFFFFF) + b"\x00\x03"
    return archive_many(N.FRAME_GZIP, inputs, [hdr] * len(inputs), compression_type, chunk_bytes, mode)


# ------------------------------------------------------------------------------------------------------------
# CRC32 / Adler32 (src/CRC32.ts, src/Adler32.ts)
# ------------------------------------------------------------------------------------------------------------
class CRC32:
    @staticmethod
    def create(data, pos=None, length=None):  # src/CRC32.ts:13
        return CRC32.update(data, 0, pos, length)

    @staticmethod
    def update(data, crc, pos=None, length=None):  # src/CRC32.ts:25: CRC of data[pos, pos+length) continued from crc
        a = _u8(data)
        pos = 0 if pos is None else pos
        length = a.size if length is None else length  # `length ?? data.length`, exactly as the reference
        piece = a[pos:pos + length]
        c = int(checksum_many([piece], True, False)["crc32"][0])
        return N.crc32_combine(crc & 0xFFFFFFFF, c, piece.size) if crc else c


class Adler32:
    @staticmethod
    def create(array):  # src/Adler32.ts:13
        if isinstance(array, str):
            array = bytes(ord(c) & 0xFF for c in array)  # stringToByteArray, src/Util.ts:5
        return Adler32.update(1, array)

    @staticmethod
    def update(adler, array, length=None, pos=0):  # src/Adler32.ts:28
        a = _u8(array)
        length = a.size if length is None else length
        piece = a[pos:pos + length]
        c = int(checksum_many([piece], False, True)["adler32"][0])
        return c if adler == 1 else N.adler32_combine(adler & 0xFFFFFFFF, c, piece.size)


# ------------------------------------------------------------------------------------------------------------
# RawDeflate / RawInflate (src/RawDeflate.ts:50-114, src/RawInflate.ts:70-140)
# ------------------------------------------------------------------------------------------------------------
class RawDeflate:
    def __init__(self, input, opts=None):
        self.input = _u8(input)
        self.lazy = _opt(opts, "lazy", 0)
        self.compressionType = _opt(opts, "compressionType", CompressionType.DYNAMIC)
        ob = (opts or {}).get("outputBuffer")
        self.output = _u8(ob) if ob is not None else np.zeros(0, dtype=np.uint8)
        self.op = _opt(opts, "outputIndex", 0)
        self.chunkBytes = _b200(opts).get("chunkBytes", 0)
        self.mode = _mode_of(opts)
        self.dictionary = _b200(opts).get("dictionary")  # preset dictionary (engine extension)
        if self.lazy:
            raise ZlibError("lazy matching is not supported: the reference corrupts data with lazy > 0")

    def compress(self):
        prefix = self.output[:self.op]
        if prefix.size < self.op:  # outputIndex beyond the given buffer: the reference doubles it, zero filled
            prefix = np.concatenate([prefix, np.zeros(self.op - prefix.size, dtype=np.uint8)])
        outs, _ = deflate_many([self.input], self.compressionType, self.chunkBytes, prefixes=[prefix], mode=self.mode,
                               dictionary=self.dictionary)
        self.output = outs[0]
        self.op = int(self.output.size)
        return self.output


class RawInflate:
    def __init__(self, input, opts=None):
        self.input = _u8(input)
        self.ip = _opt(opts, "index", 0)
        self.bufferSize = (opts or {}).get("bufferSize")
        self.bufferType = _opt(opts, "bufferType", BufferType.ADAPTIVE)
        self.resize = _opt(opts, "resize", False)
        self.dictionary = _b200(opts).get("dictionary")  # preset dictionary (engine extension)
        self.buffer = None
        self.op = 0

    def decompress(self):
        outs, res = inflate_many([self.input], [self.ip], [self.bufferSize], dictionary=self.dictionary)
        self.ip += int(res["in_used"][0])  # first byte after the deflate data (src/RawInflate.ts:511-514)
        self.buffer = outs[0]
        self.op = int(outs[0].size)
        return self.buffer


# ------------------------------------------------------------------------------------------------------------
# zlib container (src/Deflate.ts, src/Inflate.ts)
# ------------------------------------------------------------------------------------------------------------
def _zlib_header(compression_type, fdict=False):  # src/Deflate.ts:67-78 (FDICT: RFC 1950)
    cmf = 120
    flg = (compression_type << 6) | ((1 if fdict else 0) << 5)
    flg |= 31 - ((cmf << 8) + flg) % 31
    return bytes([cmf, flg & 0xFF])


def _dictid(dictionary):
    """DICTID of a preset dictionary: its Adler-32 (RFC 1950), computed on the GPU."""
    return int(checksum_many([_u8(dictionary)], False, True)["adler32"][0])


class Deflate:
    def __init__(self, input, opts=None):
        self.input = _u8(input)
        self.compressionType = _opt(opts, "compressionType", CompressionType.DYNAMIC)
        self.opts = dict(opts or {})
        self.adler32 = None
        self.output = None
        if _opt(opts, "lazy", 0):
            raise ZlibError("lazy matching is not supported: the reference corrupts data with lazy > 0")

    @staticmethod
    def compress_static(input, opts=None):  # `Deflate.compress(input, opts)`, src/Deflate.ts:52
        return Deflate(input, opts).compress()

    def compress(self):
        dictionary = _b200(self.opts).get("dictionary")
        if dictionary is not None and _u8(dictionary).size:
            # preset dictionary: header with FDICT, DICTID, the dictionary deflate, Adler-32 of the input (zlb_archive
            # has no dictionary, so this stream is framed here)
            outs, res = deflate_many([self.input], self.compressionType, _b200(self.opts).get("chunkBytes", 0),
                                     want_adler32=True, mode=_mode_of(self.opts), dictionary=dictionary)
            self.adler32 = int(res["adler32"][0])
            head = _zlib_header(self.compressionType, fdict=True) + struct.pack(">I", _dictid(dictionary))
            self.output = np.concatenate([_u8(head), outs[0], _u8(struct.pack(">I", self.adler32))])
            return self.output
        # header (:67-78), raw stream (:84-85) and Adler-32 big endian (:95) are put together on the device
        self.output, res = archive_many(N.FRAME_ZLIB, [self.input], [_zlib_header(self.compressionType)],
                                        self.compressionType, _b200(self.opts).get("chunkBytes", 0), _mode_of(self.opts))
        self.adler32 = int(res["adler32"][0])
        return self.output


class Inflate:
    def __init__(self, input, opts=None):
        self.input = _u8(input)
        self.ip = _opt(opts, "index", 0)
        self.verify = _opt(opts, "verify", False)
        self.adler32 = None
        cmf, flg = int(self.input[self.ip]), int(self.input[self.ip + 1])
        self.ip += 2
        if (cmf & 0x0F) != 8:
            raise ZlibError("unsupported compression method")  # src/Inflate.ts:47
        if ((cmf << 8) + flg) % 31 != 0:
            raise ZlibError("invalid fcheck flag:%d" % (((cmf << 8) + flg) % 31))  # :52
        # a preset dictionary (engine extension) is used for FDICT streams only; other streams ignore it, like zlib
        dictionary = _b200(opts).get("dictionary") if flg & 0x20 else None
        if flg & 0x20:
            if dictionary is None:
                raise ZlibError("fdict flag is not supported")  # :57
            dictid = struct.unpack(">I", self.input[self.ip:self.ip + 4].tobytes().ljust(4, b"\0"))[0]
            have = _dictid(dictionary)
            if have != dictid:
                raise ZlibError("invalid dictionary: adler-32 0x%08x, DICTID 0x%08x" % (have, dictid))
            self.ip += 4
        self.rawinflate = RawInflate(self.input, {"index": self.ip, "bufferSize": (opts or {}).get("bufferSize"),
                                                  "bufferType": (opts or {}).get("bufferType"),
                                                  "resize": (opts or {}).get("resize"),
                                                  "b200": {"dictionary": dictionary}})

    def decompress(self):
        r = self.rawinflate
        outs, res = inflate_many([r.input], [r.ip], [r.bufferSize], want_adler32=self.verify, dictionary=r.dictionary)
        r.ip += int(res["in_used"][0])
        self.ip = r.ip
        buf = outs[0]
        if self.verify:  # src/Inflate.ts:81-90
            self.adler32 = int(res["adler32"][0])
            stored = struct.unpack(">I", self.input[self.ip:self.ip + 4].tobytes().ljust(4, b"\0"))[0]
            if self.adler32 != stored:
                raise ZlibError("invalid adler-32 checksum")
        return buf


# ------------------------------------------------------------------------------------------------------------
# gzip container (src/GZip.ts, src/GUnzip.ts)
# ------------------------------------------------------------------------------------------------------------
def _gzip_string(s):  # src/GZip.ts:133-150: chars > 0xFF are written as two bytes, NUL terminated
    out = bytearray()
    for ch in s:
        c = ord(ch)
        out += struct.pack("<H", c & 0xFFFF) if c > 0xFF else bytes([c])
    return bytes(out) + b"\0"


class GZip:
    def __init__(self, input, opts=None):
        self.input = _u8(input)
        self.filename = _opt(opts, "filename", "")
        self.comment = _opt(opts, "comment", "")
        self.flags = {"fname": bool(self.filename), "fcomment": bool(self.comment), "fhcrc": bool(_opt(opts, "hcrc", False))}
        self.deflateOptions = dict(_opt(opts, "deflateOptions", {}))
        self.mtime = _b200(opts).get("mtime")  # engine-only knob: fixed MTIME for reproducible output
        self.crc32 = None
        self.output = None

    def header(self):
        flg = (0x08 if self.flags["fname"] else 0) | (0x10 if self.flags["fcomment"] else 0) | (0x02 if self.flags["fhcrc"] else 0)
        mtime = int(datetime.datetime.now().timestamp()) if self.mtime is None else int(self.mtime)  # Date.now()/1000, :121
        h = b"\x1f\x8b\x08" + bytes([flg]) + struct.pack("<I", mtime & 0xFFFFFFFF) + b"\x00\x03"  # XFL 0, OS Unix
        if self.flags["fname"]:
            h += _gzip_string(self.filename)
        if self.flags["fcomment"]:
            h += _gzip_string(self.comment)
        if self.flags["fhcrc"]:
            h += struct.pack("<H", CRC32.create(h) & 0xFFFF)  # :153-156
        return h

    def compress(self):
        hdr = self.header()
        ctype = _opt(self.deflateOptions, "compressionType", CompressionType.DYNAMIC)
        if _opt(self.deflateOptions, "lazy", 0):
            raise ZlibError("lazy matching is not supported: the reference corrupts data with lazy > 0")
        # member header, raw stream (:159-166), CRC-32 and ISIZE (:180-185) are put together on the device
        self.output, res = archive_many(N.FRAME_GZIP, [self.input], [hdr], ctype,
                                        _b200(self.deflateOptions).get("chunkBytes", 0), _mode_of(self.deflateOptions))
        self.crc32 = int(res["crc32"][0])
        return self.output


class GUnzip:
    """Multi-member files are decoded as ONE GPU batch: every `1F 8B 08` signature in the buffer is a candidate
    member, all candidates are inflated speculatively side by side, and the chain of true members is then walked on
    the host exactly as the reference's loop would (src/GUnzip.ts:56-58): member k + 1 begins where member k's trailer
    ends; candidates that lie inside compressed data are never reached. Results, checks and error texts are those of
    the member-by-member loop."""

    BATCH_MIN_CANDIDATES = 2

    def __init__(self, input):
        self.input = _u8(input)
        self.ip = 0
        self.members = []
        self.decompressed = False
        self.crc32 = None

    def getMembers(self):
        if not self.decompressed:
            self.decompress()
        return list(self.members)

    def decompress(self):
        if self.ip == 0 and not self.members:
            self._decode_all_members()
        while self.ip < self.input.size:  # src/GUnzip.ts:56-58 (multi-member)
            self.decodeMember()
        self.decompressed = True
        return np.concatenate([m["data"] for m in self.members]) if self.members else np.zeros(0, dtype=np.uint8)

    def _parse_header(self, p):  # src/GUnzip.ts:66-133; returns (member fields, offset of the deflate data)
        inp = self.input
        m = {"id1": int(inp[p]), "id2": int(inp[p + 1])}
        if m["id1"] != 0x1F or m["id2"] != 0x8B:
            raise ZlibError("invalid file signature:%d,%d" % (m["id1"], m["id2"]))
        m["cm"] = int(inp[p + 2])
        if m["cm"] != 8:
            raise ZlibError("unknown compression method: %d" % m["cm"])
        flg = m["flg"] = int(inp[p + 3])
        m["mtime"] = struct.unpack("<I", inp[p + 4:p + 8].tobytes())[0]
        m["xfl"], m["os"] = int(inp[p + 8]), int(inp[p + 9])
        p += 10
        if flg & 0x04:
            m["xlen"] = int(inp[p]) | (int(inp[p + 1]) << 8)
            p += 2 + m["xlen"]
        for bit, key in ((0x08, "name"), (0x10, "comment")):
            if flg & bit:
                e = p
                while int(inp[e]) != 0:
                    e += 1
                m[key] = "".join(chr(c) for c in inp[p:e])
                p = e + 1
        if flg & 0x02:
            m["crc16"] = CRC32.create(inp, 0, p) & 0xFFFF  # from offset 0, as the reference does (:128)
            if m["crc16"] != (int(inp[p]) | (int(inp[p + 1]) << 8)):
                raise ZlibError("invalid header crc16")
            p += 2
        return m, p

    def _finish_member(self, m, p, data, res_row):  # src/GUnzip.ts:151-183: trailer checks, member record
        inp = self.input
        m["data"] = data
        p += int(res_row["in_used"])
        crc32, isize2 = struct.unpack("<II", inp[p:p + 8].tobytes().ljust(8, b"\0"))
        self.crc32 = int(res_row["crc32"])
        if self.crc32 != crc32:
            raise ZlibError("invalid CRC-32 checksum: 0x%x / 0x%x" % (self.crc32, crc32))
        if (data.size & 0xFFFFFFFF) != isize2:
            raise ZlibError("invalid input size: %d / %d" % (data.size & 0xFFFFFFFF, isize2))
        m["crc32"], m["isize"] = crc32, isize2
        self.members.append(m)
        self.ip = p + 8

    def decodeMember(self):  # src/GUnzip.ts:66-183
        inp = self.input
        m, p = self._parse_header(self.ip)
        isize = struct.unpack("<I", inp[-4:].tobytes())[0]  # size hint from the last 4 bytes of the buffer (:135-149)
        hint = isize if inp.size - p - 8 < isize * 512 else None
        # only this member's bytes and what follows it travel; the marker split is for one large member, not for a
        # tail of further members (they are decoded by the batch path above)
        outs, res = inflate_many([inp[p:]], [0], [hint], want_crc32=True)
        self._finish_member(m, p, outs[0], res[0])

    def _decode_all_members(self):
        """Batch path. Leaves self.ip at the first member it could not settle (the member loop carries on there and
        reports whatever is wrong in the reference's words)."""
        inp = self.input
        if inp.size < 36:
            return
        sig = np.flatnonzero((inp[:-2] == 0x1F) & (inp[1:-1] == 0x8B) & (inp[2:] == 0x08))
        if sig.size < self.BATCH_MIN_CANDIDATES or sig[0] != 0:
            return
        heads = {}
        for c in sig.tolist():
            try:
                heads[c] = self._parse_header(c)
            except (ZlibError, IndexError):
                pass  # not a member start (or a broken one: the member loop will say so if the chain gets there)
        starts = sorted(heads)
        if len(starts) < self.BATCH_MIN_CANDIDATES:
            return
        offs = np.array([heads[c][1] for c in starts], dtype=np.uint64)
        lens = np.uint64(inp.size) - offs
        nxt = np.array(starts[1:] + [inp.size], dtype=np.int64)
        gaps = np.maximum(nxt - offs.astype(np.int64), 0)
        caps = np.maximum(0x8000, 4 * gaps)
        index_of = {c: i for i, c in enumerate(starts)}
        outs, res = [None] * len(starts), np.zeros(len(starts), dtype=N.RESULT_DTYPE)

        def decode(idx):
            """inflates the candidates idx (ascending). The first member (candidate 0, at offset 0) goes through the
            split, which decodes one large stream in parallel from whatever wrote it (its item reaches to the end of the
            buffer, the split stops where its stream does); the other candidates' items reach to the end as well, so
            they are inflated in one call without the split, which would scan the rest of the buffer once per candidate."""
            idx = list(idx)
            if idx and idx[0] == 0:
                o, r = inflate_blob(inp, offs[:1], lens[:1], [int(caps[0])], want_crc32=True, tolerant=True)
                outs[0], res[0] = o[0], r[0]
                idx = idx[1:]
            if idx:
                o, r = inflate_blob(inp, offs[idx], lens[idx], list(caps[idx]), want_crc32=True, split=False,
                                    tolerant=True)
                for k, i in enumerate(idx):
                    outs[i], res[i] = o[k], r[k]

        g0 = 0
        while g0 < len(starts):  # groups of candidates whose output slots stay below 2 GiB together
            g1, tot = g0, 0
            while g1 < len(starts) and (g1 == g0 or tot + int(caps[g1]) <= (2 << 30)):
                tot += int(caps[g1])
                g1 += 1
            decode(range(g0, g1))
            g0 = g1
        for _ in range(6):  # candidates on the chain whose slot was too small are decoded again, larger
            pos, retry = 0, None
            while pos < inp.size and pos in index_of:
                i = index_of[pos]
                st = int(res["status"][i])
                if st == N.ST_OUT_OVERFLOW:
                    retry = i
                    break
                if st != N.ST_OK:
                    break
                pos = int(offs[i]) + int(res["in_used"][i]) + 8
            if retry is None:
                break
            again = [i for i in range(retry, len(starts)) if int(res["status"][i]) == N.ST_OUT_OVERFLOW]
            caps[again] *= 4
            decode(again)
        while self.ip < inp.size and self.ip in index_of:
            i = index_of[self.ip]
            if int(res["status"][i]) != N.ST_OK:
                return
            m, p = heads[self.ip]
            self._finish_member(dict(m), p, outs[i], res[i])


# ------------------------------------------------------------------------------------------------------------
# random access: an index of access points (zlb_inflate_index / zlb_inflate_ranges)
# ------------------------------------------------------------------------------------------------------------
_INDEX_KINDS = ("raw", "zlib", "gzip")
_INDEX_MAGIC = b"ZLBINDEX"
_INDEX_VERSION = 1
# magic, version, kind, deflate start, container bytes, deflate bytes, decompressed bytes, spacing, points, window bytes
_INDEX_HEAD = struct.Struct("<8sIIQQQQQQQ")


class InflateIndex:
    """Access points into one raw deflate, zlib or gzip stream (made by inflate_index). A read of any decompressed
    range decodes from the last point at or before it, not from the start of the stream; a long one is cut at every
    point inside it and its pieces are decoded side by side. Holds the points and, compacted, the window of each (the
    up to 32 KiB of output in front of it): about 32 KiB per point. The compressed data is not part of it: every read
    is given the same bytes the index was built over."""

    def __init__(self, kind, start, data_len, deflate_len, size, spacing, points, windows):
        if kind not in _INDEX_KINDS:
            raise ZlibError("unknown index kind: %s" % kind)
        self.kind, self.start, self.data_len, self.deflate_len = kind, int(start), int(data_len), int(deflate_len)
        self.size, self.spacing = int(size), int(spacing)
        self.points = np.ascontiguousarray(points, dtype=N.POINT_DTYPE)
        self.windows = np.ascontiguousarray(windows, dtype=np.uint8).reshape(-1)

    def __len__(self):
        return len(self.points)

    @property
    def nbytes(self):
        """bytes of the serialized index"""
        return _INDEX_HEAD.size + self.points.nbytes + self.windows.nbytes

    def read(self, data, pos, length):
        """data[...] decompressed, bytes [pos, pos + length) (fewer at the end of the stream) as a uint8 array."""
        return read_ranges([(data, self, pos, length)])[0]

    def read_many(self, data, spans):
        """read() of every (pos, length) in spans, in one GPU call."""
        return read_ranges([(data, self, pos, length) for pos, length in spans])

    def to_bytes(self):
        head = _INDEX_HEAD.pack(_INDEX_MAGIC, _INDEX_VERSION, _INDEX_KINDS.index(self.kind), self.start, self.data_len,
                                self.deflate_len, self.size, self.spacing, len(self.points), self.windows.size)
        return head + self.points.tobytes() + self.windows.tobytes()

    @classmethod
    def from_bytes(cls, blob):
        b = bytes(blob)
        if len(b) < _INDEX_HEAD.size or b[:8] != _INDEX_MAGIC:
            raise ZlibError("not an inflate index")
        magic, version, kind, start, data_len, deflate_len, size, spacing, n, wbytes = _INDEX_HEAD.unpack_from(b)
        if version != _INDEX_VERSION:
            raise ZlibError("unsupported inflate index version: %d" % version)
        if kind >= len(_INDEX_KINDS) or len(b) != _INDEX_HEAD.size + n * N.POINT_DTYPE.itemsize + wbytes:
            raise ZlibError("inflate index is corrupt")
        at = _INDEX_HEAD.size
        points = np.frombuffer(b, dtype=N.POINT_DTYPE, count=n, offset=at).copy()
        windows = np.frombuffer(b, dtype=np.uint8, count=wbytes, offset=at + points.nbytes).copy()
        return cls(_INDEX_KINDS[kind], start, data_len, deflate_len, size, spacing, points, windows)

    def _deflate(self, data):
        """the stream's deflate bytes in data, which must be as long as what the index was built over"""
        a = _u8(data)
        if a.size != self.data_len:
            raise ZlibError("data of %d bytes does not belong to this index (built over %d bytes)" % (a.size, self.data_len))
        return a[self.start:self.start + self.deflate_len]


def inflate_index(data, kind="raw", spacing=N.INDEX_DEFAULT_SPACING):
    """Decompresses one raw deflate, zlib or gzip stream and indexes it: returns (output, InflateIndex) with an access
    point about every `spacing` decompressed bytes. zlib and gzip headers are read as Inflate / GUnzip read them, with
    their error texts, and the Adler-32, or CRC-32 and ISIZE, are always checked. Preset dictionaries (FDICT) and
    multi-member gzip files are refused."""
    if kind not in _INDEX_KINDS:
        raise ZlibError("unknown index kind: %s" % kind)
    a = _u8(data)
    start = 0
    if kind == "zlib":
        cmf, flg = int(a[0]), int(a[1])
        if (cmf & 0x0F) != 8:
            raise ZlibError("unsupported compression method")  # src/Inflate.ts:47
        if ((cmf << 8) + flg) % 31 != 0:
            raise ZlibError("invalid fcheck flag:%d" % (((cmf << 8) + flg) % 31))  # :52
        if flg & 0x20:
            raise ZlibError("fdict flag is not supported")  # :57
        start = 2
    elif kind == "gzip":
        _, start = GUnzip(a)._parse_header(0)
    body = a[start:]
    size = int(inflate_sizes([body])[0])  # exact slot: no retry
    out = np.zeros(max(size, 1), dtype=np.uint8)
    items = N.make_items(1)
    items["in_len"], items["out_cap"] = body.size, size
    slots = size // max(int(spacing), 1) + 2
    flags = {"raw": 0, "zlib": N.INFLATE_WANT_ADLER32, "gzip": N.INFLATE_WANT_CRC32}[kind]
    res, points, counts = engine().inflate_index_host(body if body.size else np.zeros(1, dtype=np.uint8), out, items,
                                                      [0, slots], int(spacing), flags)
    if int(res["status"][0]) != N.ST_OK:
        raise ZlibError(status_text(res["status"][0]))
    out = out[:int(res["out_len"][0])]
    used = int(res["in_used"][0])
    p = start + used
    if kind == "zlib":
        stored = struct.unpack(">I", a[p:p + 4].tobytes().ljust(4, b"\0"))[0]
        if int(res["adler32"][0]) != stored:
            raise ZlibError("invalid adler-32 checksum")  # src/Inflate.ts:88
    elif kind == "gzip":  # src/GUnzip.ts:160-176
        crc32, isize = struct.unpack("<II", a[p:p + 8].tobytes().ljust(8, b"\0"))
        if int(res["crc32"][0]) != crc32:
            raise ZlibError("invalid CRC-32 checksum: 0x%x / 0x%x" % (int(res["crc32"][0]), crc32))
        if (out.size & 0xFFFFFFFF) != isize:
            raise ZlibError("invalid input size: %d / %d" % (out.size & 0xFFFFFFFF, isize))
        if p + 8 < a.size:
            raise ZlibError("multi-member gzip files cannot be indexed")
    points = points[:int(counts[0])].copy()
    # keep only the windows, back to back
    wl = np.minimum(points["out_pos"], 32768)
    windows = np.concatenate([out[int(q) - int(w):int(q)] for q, w in zip(points["out_pos"], wl)] or [out[:0]])
    points["win_off"] = np.concatenate([[0], np.cumsum(wl)[:-1]]).astype(np.uint64)
    return out, InflateIndex(kind, start, a.size, used, out.size, spacing, points, windows)


def read_ranges(reads, want_crc32=False, want_adler32=False):
    """Reads of (data, InflateIndex, pos, length) -- any streams, any number of each -- in one GPU call
    (zlb_inflate_ranges_host). Returns a uint8 array per read: bytes [pos, pos + length) of the decompressed stream,
    fewer where it ends. With want_crc32 / want_adler32, (arrays, results table) with the checksums of each read."""
    reads = list(reads)
    if not reads:
        return ([], np.zeros(0, dtype=N.RESULT_DTYPE)) if want_crc32 or want_adler32 else []
    blobs, where, pts, wins, pbase = [], {}, [], [], {}
    at = wat = pat = out_at = 0
    ranges = N.make_ranges(len(reads))
    for i, (data, idx, pos, length) in enumerate(reads):
        pos, length = int(pos), int(length)
        if pos < 0 or length < 0:
            raise ZlibError("negative position or length")
        key = (id(data), id(idx))
        if key not in where:
            blobs.append(idx._deflate(data))
            where[key] = at
            at += idx.deflate_len
        if id(idx) not in pbase:
            p = idx.points.copy()
            p["win_off"] += np.uint64(wat)
            pts.append(p)
            wins.append(idx.windows)
            pbase[id(idx)] = pat
            pat += len(p)
            wat += idx.windows.size
        cap = max(0, min(length, idx.size - pos))
        ranges[i] = (where[key], idx.deflate_len, pbase[id(idx)], len(idx.points), pos, out_at, cap)
        out_at += cap
    blob = np.concatenate(blobs + [np.zeros(1, dtype=np.uint8)])
    win = np.concatenate(wins + [np.zeros(1, dtype=np.uint8)])
    out = np.zeros(max(out_at, 1), dtype=np.uint8)
    flags = (N.INFLATE_WANT_CRC32 if want_crc32 else 0) | (N.INFLATE_WANT_ADLER32 if want_adler32 else 0)
    res = engine().inflate_ranges_host(blob, win, out, np.concatenate(pts), ranges, flags)
    outs = []
    for r, rg in zip(res, ranges):
        if int(r["status"]) != N.ST_OK:
            raise ZlibError(status_text(r["status"]))
        if int(r["out_len"]) != int(rg["out_cap"]):
            raise ZlibError("input buffer is broken")  # the stream ended before the index said it would
        outs.append(out[int(rg["out_off"]):int(rg["out_off"]) + int(rg["out_cap"])])
    return (outs, res) if flags else outs


# ------------------------------------------------------------------------------------------------------------
# PKZIP container (src/Zip.ts, src/Unzip.ts)
# ------------------------------------------------------------------------------------------------------------
def _dos_time(date):  # src/Zip.ts:129-139
    return bytes([((date.minute & 0x7) << 5) | (date.second >> 1), (date.hour << 3) | (date.minute >> 3),
                  (((date.month) & 0x7) << 5) | date.day, (((date.year - 1980) & 0x7F) << 1) | (date.month >> 3)])


class Zip:
    """addFile() only queues; compress() deflates and checksums every queued entry in ONE GPU batch (the
    reference compresses inside addFile, one file at a time, src/Zip.ts:92-96 -- same bytes, different schedule)."""

    def __init__(self, comment=b""):
        self.files = []
        self.comment = _u8(comment)
        self.password = None

    def addFile(self, input, filename="", opts=None):
        opts = dict(opts or {})
        self.files.append({"filename": filename, "buffer": _u8(input), "option": opts, "size": _u8(input).size,
                           "compressionMethod": _opt(opts, "compressionMethod", ZipCompressionMethod.DEFLATE),
                           "compressed": False, "crc32": 0})

    def setPassword(self, password):
        self.password = password

    def compress(self):
        files = self.files
        if self.password is not None or any(f["option"].get("password") is not None for f in files):
            raise NotImplementedError("ZipCrypto is out of scope (SURVEY.md section 2)")
        if len(files) > 0xFFFF:
            raise ZlibError("too many entries for a ZIP32 end-of-central-directory record")
        # one batch per compression type used by the entries (normally one)
        # (`compress: false` only defers the work from addFile to here in the reference, src/Zip.ts:92,142-149)
        todo = [i for i, f in enumerate(files) if not f["compressed"] and f["compressionMethod"] == ZipCompressionMethod.DEFLATE]
        by_type = {}
        for i in todo:
            do = files[i]["option"].get("deflateOptions") or {}
            if _opt(do, "lazy", 0):
                raise ZlibError("lazy matching is not supported: the reference corrupts data with lazy > 0")
            by_type.setdefault((_opt(do, "compressionType", CompressionType.DYNAMIC), _b200(do).get("chunkBytes", 0),
                                _mode_of(do)), []).append(i)
        if len(by_type) <= 1 and not any(f["compressed"] for f in files):
            return self._compress_on_device(next(iter(by_type), (CompressionType.DYNAMIC, 0, N.MODE_COMPAT)))
        for (ctype, chunk, mode), idxs in by_type.items():
            outs, res = deflate_many([files[i]["buffer"] for i in idxs], ctype, chunk, want_crc32=True, mode=mode)
            for i, o, r in zip(idxs, outs, res):
                files[i]["crc32"], files[i]["buffer"], files[i]["compressed"] = int(r["crc32"]), o, True
        rest = [i for i, f in enumerate(files) if not f["compressed"]]
        if rest:  # stored entries: CRC-32 only (src/Zip.ts:144)
            res = checksum_many([files[i]["buffer"] for i in rest], True, False)
            for i, r in zip(rest, res):
                files[i]["crc32"] = int(r["crc32"])
        local, central = [], []
        offset = 0
        for f in files:
            name = bytes(ord(c) & 0xFF for c in f["filename"])  # stringToByteArray
            comment = bytes(ord(c) & 0xFF for c in (f["option"].get("comment") or ""))
            date = f["option"].get("date") or datetime.datetime.now()
            mt = _dos_time(date)
            body = f["buffer"]
            common = struct.pack("<HHH", 20, 0, f["compressionMethod"]) + mt + struct.pack(
                "<IIIHH", f["crc32"], body.size, f["size"], len(name), 0)
            local.append(b"PK\x03\x04" + common + name)
            local.append(body)
            central.append(b"PK\x01\x02" + bytes([20, _opt(f["option"], "os", 0)]) + common +
                           struct.pack("<HHHII", len(comment), 0, 0, 0, offset) + name + comment)
            offset += 30 + len(name) + body.size
        cd = b"".join(central)
        eocd = b"PK\x05\x06" + struct.pack("<HHHHIIH", 0, 0, len(files), len(files), len(cd), offset, self.comment.size)
        parts = [(_u8(p) if not isinstance(p, np.ndarray) else p) for p in local] + [_u8(cd), _u8(eocd), self.comment]
        return np.concatenate(parts) if parts else np.zeros(0, dtype=np.uint8)


    def _compress_on_device(self, settings):
        """All entries share one deflate setting and none is compressed yet (the usual case): header templates
        go to the device with the data, and local headers, bodies, central directory and end record are laid
        out there (zlb_archive_host) -- the same bytes as the loop below produces."""
        ctype, chunk, mode = settings
        files = self.files
        heads, cdirs, methods = [], [], []
        for f in files:
            name = bytes(ord(c) & 0xFF for c in f["filename"])  # stringToByteArray
            comment = bytes(ord(c) & 0xFF for c in (f["option"].get("comment") or ""))
            mt = _dos_time(f["option"].get("date") or datetime.datetime.now())
            deflated = f["compressionMethod"] == ZipCompressionMethod.DEFLATE
            # CRC-32 and compressed size (0 here) are filled in by the engine
            common = struct.pack("<HHH", 20, 0, f["compressionMethod"]) + mt + struct.pack(
                "<IIIHH", 0, 0, f["size"], len(name), 0)
            heads.append(b"PK\x03\x04" + common + name)
            cdirs.append(b"PK\x01\x02" + bytes([20, _opt(f["option"], "os", 0)]) + common +
                         struct.pack("<HHHII", len(comment), 0, 0, 0, 0) + name + comment)
            methods.append(8 if deflated else 0)
        eocd = b"PK\x05\x06" + struct.pack("<HHHHIIH", 0, 0, len(files), len(files), 0, 0, self.comment.size)
        out, res = archive_many(N.FRAME_ZIP, [f["buffer"] for f in files], heads, ctype, chunk, mode, methods, cdirs,
                                eocd + self.comment.tobytes())
        for f, h, r in zip(files, heads, res):  # what the reference leaves in its file table (src/Zip.ts:144-149)
            f["crc32"] = int(r["crc32"])
            if f["compressionMethod"] == ZipCompressionMethod.DEFLATE:
                a = int(r["in_used"]) + len(h)
                f["buffer"], f["compressed"] = out[a:int(r["in_used"]) + int(r["out_len"])], True
        return out


class Unzip:
    def __init__(self, input, opts=None):
        self.input = _u8(input)
        self.verify = _opt(opts, "verify", False)
        self.password = (opts or {}).get("password")
        self.EOCD = None
        self.fileHeaderList = None
        self.filenameToIndex = None

    def setPassword(self, password):
        self.password = password

    def _search_eocd(self):  # src/Unzip.ts:150-161
        inp = self.input
        for ip in range(inp.size - 12, 0, -1):
            if inp[ip] == 0x50 and inp[ip + 1] == 0x4B and inp[ip + 2] == 0x05 and inp[ip + 3] == 0x06:
                return ip
        raise ZlibError("End of Central Directory Record not found")

    def parseFileHeader(self):  # src/Unzip.ts:220-246
        if self.fileHeaderList is not None:
            return
        inp = self.input
        p = self._search_eocd()
        f = struct.unpack("<HHHHIIH", inp[p + 4:p + 22].tobytes())
        eocd = dict(zip(["numberOfThisDisk", "startDisk", "totalEntriesThisDisk", "totalEntries", "centralDirectorySize",
                         "centralDirectoryOffset", "commentLength"], f))
        eocd["comment"] = inp[p + 22:p + 22 + eocd["commentLength"]]
        lst, tab = [], {}
        q = eocd["centralDirectoryOffset"]
        for i in range(eocd["totalEntries"]):
            if inp[q:q + 4].tobytes() != b"PK\x01\x02":
                raise ZlibError("invalid file header signature")
            v = struct.unpack("<BBHHHHHIIIHHHHHII", inp[q + 4:q + 46].tobytes())
            fh = dict(zip(["version", "os", "needVersion", "flags", "compression", "time", "date", "crc32", "compressedSize",
                           "plainSize", "fileNameLength", "extraFieldLength", "fileCommentLength", "diskNumberStart",
                           "internalFileAttributes", "externalFileAttributes", "relativeOffset"], v))
            q += 46
            fh["filename"] = inp[q:q + fh["fileNameLength"]].tobytes().decode("utf-8", "replace")  # TextDecoder, readString
            q += fh["fileNameLength"]
            fh["extraField"] = inp[q:q + fh["extraFieldLength"]]
            q += fh["extraFieldLength"]
            fh["comment"] = inp[q:q + fh["fileCommentLength"]]
            q += fh["fileCommentLength"]
            lst.append(fh)
            tab[fh["filename"]] = i
        if eocd["centralDirectorySize"] < q - eocd["centralDirectoryOffset"]:
            raise ZlibError("invalid file header size")
        self.EOCD, self.fileHeaderList, self.filenameToIndex = eocd, lst, tab

    def getFilenames(self):
        self.parseFileHeader()
        return [fh["filename"] for fh in self.fileHeaderList]

    def _local(self, index):  # src/Unzip.ts:28-62
        self.parseFileHeader()
        if index is None or index < 0 or index >= len(self.fileHeaderList):
            raise ZlibError("wrong index")
        inp = self.input
        off = self.fileHeaderList[index]["relativeOffset"]
        if inp[off:off + 4].tobytes() != b"PK\x03\x04":
            raise ZlibError("invalid local file header signature")
        v = struct.unpack("<HHHHHIIIHH", inp[off + 4:off + 30].tobytes())
        lh = dict(zip(["needVersion", "flags", "compression", "time", "date", "crc32", "compressedSize", "plainSize",
                       "fileNameLength", "extraFieldLength"], v))
        lh["dataOffset"] = off + 30 + lh["fileNameLength"] + lh["extraFieldLength"]
        if lh["flags"] & 0x0001:
            raise NotImplementedError("ZipCrypto is out of scope (SURVEY.md section 2)")
        return lh

    def getFileData(self, index, opts=None):  # src/Unzip.ts:248-307
        return self.getFilesData([index])[0]

    def getFilesData(self, indices):
        """Batch form of getFileData: every deflated entry of `indices` is inflated (and CRC-checked when
        verify is set) in one GPU batch."""
        lhs = [self._local(i) for i in indices]
        out = [None] * len(lhs)
        defl = [k for k, lh in enumerate(lhs) if lh["compression"] == ZipCompressionMethod.DEFLATE]
        if defl:
            outs, res = inflate_blob(self.input, [lhs[k]["dataOffset"] for k in defl],
                                     [lhs[k]["compressedSize"] for k in defl], [lhs[k]["plainSize"] for k in defl],
                                     want_crc32=self.verify)
            for k, o, r in zip(defl, outs, res):
                out[k] = o
                if self.verify and lhs[k]["crc32"] != int(r["crc32"]):
                    raise ZlibError("Incorrect crc: file=0x%x, data=0x%x" % (lhs[k]["crc32"], int(r["crc32"])))
        stored = [k for k, lh in enumerate(lhs) if lh["compression"] != ZipCompressionMethod.DEFLATE]
        for k in stored:
            out[k] = self.input[lhs[k]["dataOffset"]:lhs[k]["dataOffset"] + lhs[k]["compressedSize"]]
        if self.verify and stored:
            res = checksum_many([out[k] for k in stored], True, False)
            for k, r in zip(stored, res):
                if lhs[k]["crc32"] != int(r["crc32"]):
                    raise ZlibError("Incorrect crc: file=0x%x, data=0x%x" % (lhs[k]["crc32"], int(r["crc32"])))
        return out

    def decompress(self, filename, opts=None):  # src/Unzip.ts:327-334
        self.parseFileHeader()
        index = self.filenameToIndex.get(filename)
        if index is None:
            raise ZlibError(filename + " not found")
        return self.getFileData(index, opts)

    def decompressAll(self):
        """{filename: data} of every entry, one GPU batch (engine-side extension for the C4 workload)."""
        names = self.getFilenames()
        return dict(zip(names, self.getFilesData(list(range(len(names))))))


Zlib = {"GZip": GZip, "GUnzip": GUnzip, "Zip": Zip, "Unzip": Unzip, "Deflate": Deflate, "Inflate": Inflate}  # src/index.ts:8-12
