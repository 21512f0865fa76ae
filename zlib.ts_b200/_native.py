"""ctypes binding of libzlibts_b200.so (include/zlibts_b200.h) -- the only way Python reaches the kernels.

There is no CPU fallback: if the shared library is missing, or no B200-class GPU is visible,
construction of an Engine raises.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ZLB_LIB_OVERRIDE") or os.path.join(_HERE, "libzlibts_b200.so")  # override: kernel-variant experiments (tools/build_variants.sh)

ITEM_DTYPE = np.dtype([("in_off", "<u8"), ("in_len", "<u8"), ("out_off", "<u8"), ("out_cap", "<u8")])
RESULT_DTYPE = np.dtype([("status", "<u4"), ("crc32", "<u4"), ("adler32", "<u4"), ("blocks", "<u4"),
                         ("out_len", "<u8"), ("in_used", "<u8")])
ENTRY_DTYPE = np.dtype([("in_off", "<u8"), ("in_len", "<u8"), ("head_off", "<u8"), ("head_len", "<u4"),
                        ("method", "<u4"), ("cdir_off", "<u8"), ("cdir_len", "<u4"), ("reserved", "<u4")])
DICT_DTYPE = np.dtype([("off", "<u8"), ("len", "<u8")])   # zlb_dict: an item's preset dictionary in the dictionary blob
POINT_DTYPE = np.dtype([("in_bit", "<u8"), ("out_pos", "<u8"), ("win_off", "<u8")])   # zlb_point: an access point
RANGE_DTYPE = np.dtype([("in_off", "<u8"), ("in_len", "<u8"), ("pt_first", "<u8"), ("pt_count", "<u8"), ("pos", "<u8"),
                        ("out_off", "<u8"), ("out_cap", "<u8")])                     # zlb_range: one read
assert ITEM_DTYPE.itemsize == 32 and RESULT_DTYPE.itemsize == 32 and ENTRY_DTYPE.itemsize == 48 and DICT_DTYPE.itemsize == 16
assert POINT_DTYPE.itemsize == 24 and RANGE_DTYPE.itemsize == 56
INDEX_DEFAULT_SPACING = 1 << 20

# CompressionType (src/RawDeflate.ts:12-17)
NONE, FIXED, DYNAMIC = 0, 1, 2
MODE_COMPAT, MODE_FAST, MODE_PRIMED, MODE_SMALLEST, MODE_LAZY = 0, 1, 2, 4, 8   # PRIMED / SMALLEST / LAZY are flags (or-ed in)
PRIMED_CHUNK = 32768


def mode_fast(depth=0):
    """ZLB_MODE_FAST_DEPTH(depth); 0 = the library default (16 candidates)."""
    return MODE_FAST | (int(depth) << 8)

DEFLATE_WANT_CRC32, DEFLATE_WANT_ADLER32, DEFLATE_NOT_FINAL = 1, 2, 4
INFLATE_WANT_CRC32, INFLATE_WANT_ADLER32, INFLATE_CHECK_NLEN, INFLATE_SPLIT = 1, 2, 4, 8
SUM_CRC32, SUM_ADLER32 = 1, 2
FRAME_ZLIB, FRAME_GZIP, FRAME_ZIP = 1, 2, 3

ST_OK, ST_INPUT_BROKEN, ST_BTYPE, ST_CODE_LENGTH, ST_OUT_OVERFLOW, ST_STORED_LEN, ST_BAD_CODE, ST_BAD_LENGTHS = range(8)

EXPORTS = [
    "zlb_create", "zlb_destroy", "zlb_last_error", "zlb_abi_version", "zlb_stream",
    "zlb_deflate_batch", "zlb_deflate_batch_host", "zlb_deflate_bound",
    "zlb_inflate_batch", "zlb_inflate_batch_host",
    "zlb_checksum_batch", "zlb_checksum_batch_host", "zlb_crc32_combine", "zlb_adler32_combine",
    "zlb_archive", "zlb_archive_host", "zlb_archive_bound",
    "zlb_profile_enable", "zlb_profile_read", "zlb_profile_reset", "zlb_launch_count",
    "zlb_debug_lz77", "zlb_debug_code_lengths", "zlb_debug_block_starts",
    "zlb_host_alloc", "zlb_host_free", "zlb_host_is_pinned",
    "zlb_deflate_batch_dict", "zlb_deflate_batch_dict_host", "zlb_inflate_batch_dict", "zlb_inflate_batch_dict_host",
    "zlb_inflate_size_batch", "zlb_inflate_size_batch_host",
    "zlb_inflate_index", "zlb_inflate_index_host", "zlb_inflate_ranges", "zlb_inflate_ranges_host",
]

_lib = None


def load_library():
    """Loads the C-ABI library and declares every signature. Raises if it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing -- the CUDA extension was not built "
            "(run `python -c 'import __graft_entry__ as g; g.build()'`); there is no CPU fallback")
    lib = ctypes.CDLL(LIB_PATH)
    vp, sz, u32, u64, i32 = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint32, ctypes.c_uint64, ctypes.c_int
    lib.zlb_create.argtypes = [i32, vp, ctypes.POINTER(vp)]
    lib.zlb_create.restype = i32
    lib.zlb_destroy.argtypes = [vp]
    lib.zlb_destroy.restype = None
    lib.zlb_last_error.argtypes = [vp]
    lib.zlb_last_error.restype = ctypes.c_char_p
    lib.zlb_abi_version.restype = i32
    lib.zlb_stream.argtypes = [vp]
    lib.zlb_stream.restype = vp
    lib.zlb_deflate_batch.argtypes = [vp, vp, vp, vp, vp, sz, i32, i32, u32, u32]
    lib.zlb_deflate_batch.restype = i32
    lib.zlb_deflate_batch_host.argtypes = [vp, vp, sz, vp, sz, vp, vp, sz, i32, i32, u32, u32]
    lib.zlb_deflate_batch_host.restype = i32
    lib.zlb_deflate_bound.argtypes = [u64, u32, i32]
    lib.zlb_deflate_bound.restype = u64
    lib.zlb_inflate_batch.argtypes = [vp, vp, vp, vp, vp, sz, u32]
    lib.zlb_inflate_batch.restype = i32
    lib.zlb_inflate_batch_host.argtypes = [vp, vp, sz, vp, sz, vp, vp, sz, u32]
    lib.zlb_inflate_batch_host.restype = i32
    lib.zlb_deflate_batch_dict.argtypes = [vp, vp, vp, vp, vp, vp, vp, sz, i32, i32, u32, u32]
    lib.zlb_deflate_batch_dict.restype = i32
    lib.zlb_deflate_batch_dict_host.argtypes = [vp, vp, sz, vp, sz, vp, sz, vp, vp, vp, sz, i32, i32, u32, u32]
    lib.zlb_deflate_batch_dict_host.restype = i32
    lib.zlb_inflate_batch_dict.argtypes = [vp, vp, vp, vp, vp, vp, vp, sz, u32]
    lib.zlb_inflate_batch_dict.restype = i32
    lib.zlb_inflate_batch_dict_host.argtypes = [vp, vp, sz, vp, sz, vp, sz, vp, vp, vp, sz, u32]
    lib.zlb_inflate_batch_dict_host.restype = i32
    lib.zlb_inflate_size_batch.argtypes = [vp, vp, vp, vp, vp, sz, u32]
    lib.zlb_inflate_size_batch.restype = i32
    lib.zlb_inflate_size_batch_host.argtypes = [vp, vp, sz, vp, vp, vp, sz, u32]
    lib.zlb_inflate_size_batch_host.restype = i32
    lib.zlb_inflate_index.argtypes = [vp, vp, vp, vp, vp, sz, u32, u64, vp, vp, vp]
    lib.zlb_inflate_index.restype = i32
    lib.zlb_inflate_index_host.argtypes = [vp, vp, sz, vp, sz, vp, vp, sz, u32, u64, vp, vp, vp]
    lib.zlb_inflate_index_host.restype = i32
    lib.zlb_inflate_ranges.argtypes = [vp, vp, vp, vp, vp, sz, vp, vp, sz, u32]
    lib.zlb_inflate_ranges.restype = i32
    lib.zlb_inflate_ranges_host.argtypes = [vp, vp, sz, vp, sz, vp, sz, vp, sz, vp, vp, sz, u32]
    lib.zlb_inflate_ranges_host.restype = i32
    lib.zlb_checksum_batch.argtypes = [vp, vp, vp, vp, sz, u32]
    lib.zlb_checksum_batch.restype = i32
    lib.zlb_checksum_batch_host.argtypes = [vp, vp, sz, vp, vp, sz, u32]
    lib.zlb_checksum_batch_host.restype = i32
    lib.zlb_crc32_combine.argtypes = [u32, u32, u64]
    lib.zlb_crc32_combine.restype = u32
    lib.zlb_adler32_combine.argtypes = [u32, u32, u64]
    lib.zlb_adler32_combine.restype = u32
    lib.zlb_archive_bound.argtypes = [i32, vp, sz, u64, u32, i32]
    lib.zlb_archive_bound.restype = u64
    lib.zlb_archive.argtypes = [vp, i32, vp, vp, vp, sz, u64, u64, vp, u64, ctypes.POINTER(u64), vp, i32, i32, u32]
    lib.zlb_archive.restype = i32
    lib.zlb_archive_host.argtypes = [vp, i32, vp, sz, vp, sz, vp, sz, u64, u64, vp, u64, ctypes.POINTER(u64), vp,
                                     i32, i32, u32]
    lib.zlb_archive_host.restype = i32
    lib.zlb_profile_enable.argtypes = [vp, i32]
    lib.zlb_profile_enable.restype = i32
    lib.zlb_profile_read.argtypes = [vp, ctypes.POINTER(i32), vp, vp, vp]
    lib.zlb_profile_read.restype = i32
    lib.zlb_profile_reset.argtypes = [vp]
    lib.zlb_profile_reset.restype = i32
    lib.zlb_launch_count.argtypes = [vp]
    lib.zlb_launch_count.restype = u64
    lib.zlb_debug_lz77.argtypes = [vp, vp, u32, vp, ctypes.POINTER(u32), vp]
    lib.zlb_debug_lz77.restype = i32
    lib.zlb_debug_code_lengths.argtypes = [vp, vp, i32, i32, vp]
    lib.zlb_debug_code_lengths.restype = i32
    lib.zlb_debug_block_starts.argtypes = [vp, vp, u64, vp, sz, u64, vp]
    lib.zlb_debug_block_starts.restype = i32
    lib.zlb_host_alloc.argtypes = [sz, ctypes.POINTER(vp)]
    lib.zlb_host_alloc.restype = i32
    lib.zlb_host_free.argtypes = [vp]
    lib.zlb_host_free.restype = None
    lib.zlb_host_is_pinned.argtypes = [vp]
    lib.zlb_host_is_pinned.restype = i32
    _lib = lib
    return lib


class _Pinned:
    """Owner of one zlb_host_alloc block; the numpy views made over it keep it alive."""

    def __init__(self, nbytes):
        lib = load_library()
        p = ctypes.c_void_p()
        rc = lib.zlb_host_alloc(nbytes, ctypes.byref(p))
        if rc != 0 or not p.value:
            raise MemoryError(f"zlb_host_alloc({nbytes}) failed ({rc})")
        self.ptr, self.nbytes = p.value, nbytes

    def __del__(self):
        if getattr(self, "ptr", None) and _lib is not None:
            _lib.zlb_host_free(self.ptr)
            self.ptr = None


def host_alloc(nbytes):
    """uint8 numpy array over page-locked memory from zlb_host_alloc (what an addon hands out as external ArrayBuffers)."""
    owner = _Pinned(max(1, int(nbytes)))
    buf = (ctypes.c_uint8 * owner.nbytes).from_address(owner.ptr)
    arr = np.frombuffer(buf, dtype=np.uint8)[:int(nbytes)]
    _PIN_OWNERS[owner.ptr] = owner   # freed by host_free() or at interpreter exit
    return arr


_PIN_OWNERS = {}


def host_free(arr):
    owner = _PIN_OWNERS.pop(arr.ctypes.data, None)
    if owner is not None:
        del owner


def host_is_pinned(arr):
    return bool(load_library().zlb_host_is_pinned(arr.ctypes.data))


def crc32_combine(crc_a, crc_b, len_b):
    return load_library().zlb_crc32_combine(crc_a, crc_b, len_b)


def adler32_combine(adler_a, adler_b, len_b):
    return load_library().zlb_adler32_combine(adler_a, adler_b, len_b)


def deflate_bound(in_len, chunk_bytes=0, block_type=DYNAMIC, mode=MODE_COMPAT, dictionary=False):
    """Output bytes that always suffice for an item; `dictionary`: some item of the call has a preset dictionary."""
    return int(load_library().zlb_deflate_bound(in_len, mode_chunk(mode, chunk_bytes, dictionary), block_type))


def mode_chunk(mode, chunk_bytes=0, dictionary=False):
    """The chunk size a deflate call with this mode really uses (primed modes, and calls in which some item has a
    preset dictionary: at most 32 KiB)."""
    if (mode & MODE_PRIMED or dictionary) and (chunk_bytes == 0 or chunk_bytes > PRIMED_CHUNK):
        return PRIMED_CHUNK
    return chunk_bytes


def make_dicts(n):
    return np.zeros(n, dtype=DICT_DTYPE)


def make_items(n):
    return np.zeros(n, dtype=ITEM_DTYPE)


def make_ranges(n):
    return np.zeros(n, dtype=RANGE_DTYPE)


def make_entries(n):
    return np.zeros(n, dtype=ENTRY_DTYPE)


def archive_bound(kind, entries, tail_len=0, chunk_bytes=0, block_type=DYNAMIC):
    entries = np.ascontiguousarray(entries, dtype=ENTRY_DTYPE)
    return int(load_library().zlb_archive_bound(kind, entries.ctypes.data, len(entries), tail_len, chunk_bytes,
                                                block_type))


class EngineError(RuntimeError):
    pass


class Engine:
    """One zlb_ctx: one GPU, one stream. Data buffers are torch uint8 CUDA tensors (device entry
    points) or numpy / bytes-like host buffers (host entry points)."""

    def __init__(self, device=0, stream=None):
        self.lib = load_library()
        handle = ctypes.c_void_p()
        rc = self.lib.zlb_create(int(device), ctypes.c_void_p(stream) if stream else None, ctypes.byref(handle))
        if rc != 0 or not handle:
            raise EngineError(f"zlb_create(device={device}) failed with {rc}: no usable sm_100 GPU (no CPU fallback)")
        self.h = handle
        self.device = int(device)

    def close(self):
        if getattr(self, "h", None):
            self.lib.zlb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise EngineError(f"{what} failed ({rc}): {self.lib.zlb_last_error(self.h).decode()}")

    @property
    def stream(self):
        return self.lib.zlb_stream(self.h)

    @property
    def launch_count(self):
        return int(self.lib.zlb_launch_count(self.h))

    # ---- instrumentation -----------------------------------------------------------------
    def profile_enable(self, on=True):
        self._check(self.lib.zlb_profile_enable(self.h, 1 if on else 0), "zlb_profile_enable")

    def profile_reset(self):
        self._check(self.lib.zlb_profile_reset(self.h), "zlb_profile_reset")

    def profile_read(self):
        n = ctypes.c_int(0)
        self._check(self.lib.zlb_profile_read(self.h, ctypes.byref(n), None, None, None), "zlb_profile_read")
        names = (ctypes.c_char_p * n.value)()
        ms = (ctypes.c_double * n.value)()
        cnt = (ctypes.c_uint64 * n.value)()
        self._check(self.lib.zlb_profile_read(self.h, ctypes.byref(n), names, ms, cnt), "zlb_profile_read")
        return {names[i].decode(): {"ms": ms[i], "launches": int(cnt[i])} for i in range(n.value)}

    # ---- device entry points ------------------------------------------------------------------
    @staticmethod
    def _tables(items):
        items = np.ascontiguousarray(items, dtype=ITEM_DTYPE)
        results = np.zeros(len(items), dtype=RESULT_DTYPE)
        return items, results

    @staticmethod
    def _dicts(dicts):
        """The zlb_dict table as an array (None: no dictionaries, a NULL table)."""
        return None if dicts is None else np.ascontiguousarray(dicts, dtype=DICT_DTYPE)

    def deflate_batch(self, d_in, d_out, items, block_type=DYNAMIC, chunk_bytes=0, flags=0, mode=MODE_COMPAT,
                      d_dict=None, dicts=None):
        """zlb_deflate_batch; with `dicts` (a DICT_DTYPE table, one entry per item, spans of the device blob d_dict)
        zlb_deflate_batch_dict."""
        items, results = self._tables(items)
        dicts = self._dicts(dicts)
        if dicts is None:
            rc = self.lib.zlb_deflate_batch(self.h, d_in.data_ptr(), d_out.data_ptr(), items.ctypes.data,
                                            results.ctypes.data, len(items), mode, block_type, chunk_bytes, flags)
        else:
            rc = self.lib.zlb_deflate_batch_dict(self.h, d_in.data_ptr(), d_out.data_ptr(),
                                                 d_dict.data_ptr() if d_dict is not None else None, dicts.ctypes.data,
                                                 items.ctypes.data, results.ctypes.data, len(items), mode, block_type,
                                                 chunk_bytes, flags)
        self._check(rc, "zlb_deflate_batch")
        return results

    def inflate_batch(self, d_in, d_out, items, flags=0, d_dict=None, dicts=None):
        """zlb_inflate_batch; with `dicts` zlb_inflate_batch_dict (see deflate_batch)."""
        items, results = self._tables(items)
        dicts = self._dicts(dicts)
        if dicts is None:
            rc = self.lib.zlb_inflate_batch(self.h, d_in.data_ptr(), d_out.data_ptr(), items.ctypes.data,
                                            results.ctypes.data, len(items), flags)
        else:
            rc = self.lib.zlb_inflate_batch_dict(self.h, d_in.data_ptr(), d_out.data_ptr(),
                                                 d_dict.data_ptr() if d_dict is not None else None, dicts.ctypes.data,
                                                 items.ctypes.data, results.ctypes.data, len(items), flags)
        self._check(rc, "zlb_inflate_batch")
        return results

    def inflate_size_batch(self, d_in, items, flags=0, dicts=None):
        """zlb_inflate_size_batch: the decompressed size of every item (results' out_len), nothing written; `dicts`
        (DICT_DTYPE) is read for its lengths only."""
        items, results = self._tables(items)
        dicts = self._dicts(dicts)
        rc = self.lib.zlb_inflate_size_batch(self.h, d_in.data_ptr() if d_in is not None else None,
                                             None if dicts is None else dicts.ctypes.data, items.ctypes.data,
                                             results.ctypes.data, len(items), flags)
        self._check(rc, "zlb_inflate_size_batch")
        return results

    @staticmethod
    def _index_tables(n, point_first):
        """(point_first as uint64 with n + 1 entries, point table, point counts) of an index build."""
        first = np.ascontiguousarray(point_first, dtype=np.uint64)
        if first.size != n + 1:
            raise ValueError("point_first needs n_items + 1 entries")
        return first, np.zeros(max(int(first[-1]), 1), dtype=POINT_DTYPE), np.zeros(n, dtype=np.uint64)

    def inflate_index(self, d_in, d_out, items, point_first, spacing=0, flags=0):
        """zlb_inflate_index: the decode of inflate_batch(..., flags | INFLATE_SPLIT) that also reports access points.
        Item i's points are points[point_first[i] : point_first[i] + counts[i]]. Returns (results, points, counts)."""
        items, results = self._tables(items)
        first, points, counts = self._index_tables(len(items), point_first)
        rc = self.lib.zlb_inflate_index(self.h, d_in.data_ptr(), d_out.data_ptr(), items.ctypes.data, results.ctypes.data,
                                        len(items), flags, spacing, points.ctypes.data, first.ctypes.data,
                                        counts.ctypes.data)
        self._check(rc, "zlb_inflate_index")
        return results, points, counts

    def inflate_ranges(self, d_in, d_win, d_out, points, ranges, flags=0):
        """zlb_inflate_ranges: reads through access points (RANGE_DTYPE table; device blobs d_in, d_win, d_out)."""
        points = np.ascontiguousarray(points, dtype=POINT_DTYPE)
        ranges = np.ascontiguousarray(ranges, dtype=RANGE_DTYPE)
        results = np.zeros(len(ranges), dtype=RESULT_DTYPE)
        rc = self.lib.zlb_inflate_ranges(self.h, d_in.data_ptr(), d_win.data_ptr() if d_win is not None else None,
                                         d_out.data_ptr(), points.ctypes.data, len(points), ranges.ctypes.data,
                                         results.ctypes.data, len(ranges), flags)
        self._check(rc, "zlb_inflate_ranges")
        return results

    def checksum_batch(self, d_in, items, kinds=SUM_CRC32 | SUM_ADLER32):
        items, results = self._tables(items)
        rc = self.lib.zlb_checksum_batch(self.h, d_in.data_ptr(), items.ctypes.data, results.ctypes.data,
                                         len(items), kinds)
        self._check(rc, "zlb_checksum_batch")
        return results

    # ---- host entry points ----------------------------------------------------------------------
    @staticmethod
    def _host_ptr(buf):
        """(address, nbytes, keepalive) of a host buffer: numpy array, torch CPU tensor, bytes-like."""
        if hasattr(buf, "data_ptr"):
            return buf.data_ptr(), buf.numel() * buf.element_size(), buf
        arr = buf if isinstance(buf, np.ndarray) else np.frombuffer(buf, dtype=np.uint8)
        arr = np.ascontiguousarray(arr)
        return arr.ctypes.data, arr.nbytes, arr

    def deflate_batch_host(self, h_in, h_out, items, block_type=DYNAMIC, chunk_bytes=0, flags=0, mode=MODE_COMPAT,
                           h_dict=None, dicts=None):
        """zlb_deflate_batch_host; with `dicts` (spans of the host blob h_dict) zlb_deflate_batch_dict_host."""
        items, results = self._tables(items)
        pi, ni, ki = self._host_ptr(h_in)
        po, no, ko = self._host_ptr(h_out)
        dicts = self._dicts(dicts)
        if dicts is None:
            rc = self.lib.zlb_deflate_batch_host(self.h, pi, ni, po, no, items.ctypes.data, results.ctypes.data,
                                                 len(items), mode, block_type, chunk_bytes, flags)
        else:
            pd, nd, kd = self._host_ptr(h_dict) if h_dict is not None else (None, 0, None)
            rc = self.lib.zlb_deflate_batch_dict_host(self.h, pi, ni, po, no, pd, nd, dicts.ctypes.data,
                                                      items.ctypes.data, results.ctypes.data, len(items), mode,
                                                      block_type, chunk_bytes, flags)
        self._check(rc, "zlb_deflate_batch_host")
        return results

    def inflate_batch_host(self, h_in, h_out, items, flags=0, h_dict=None, dicts=None):
        """zlb_inflate_batch_host; with `dicts` zlb_inflate_batch_dict_host (see deflate_batch_host)."""
        items, results = self._tables(items)
        pi, ni, ki = self._host_ptr(h_in)
        po, no, ko = self._host_ptr(h_out)
        dicts = self._dicts(dicts)
        if dicts is None:
            rc = self.lib.zlb_inflate_batch_host(self.h, pi, ni, po, no, items.ctypes.data, results.ctypes.data,
                                                 len(items), flags)
        else:
            pd, nd, kd = self._host_ptr(h_dict) if h_dict is not None else (None, 0, None)
            rc = self.lib.zlb_inflate_batch_dict_host(self.h, pi, ni, po, no, pd, nd, dicts.ctypes.data,
                                                      items.ctypes.data, results.ctypes.data, len(items), flags)
        self._check(rc, "zlb_inflate_batch_host")
        return results

    def inflate_size_batch_host(self, h_in, items, flags=0, dicts=None):
        """zlb_inflate_size_batch_host (see inflate_size_batch)."""
        items, results = self._tables(items)
        pi, ni, ki = self._host_ptr(h_in) if h_in is not None else (None, 0, None)
        dicts = self._dicts(dicts)
        rc = self.lib.zlb_inflate_size_batch_host(self.h, pi, ni, None if dicts is None else dicts.ctypes.data,
                                                  items.ctypes.data, results.ctypes.data, len(items), flags)
        self._check(rc, "zlb_inflate_size_batch_host")
        return results

    def inflate_index_host(self, h_in, h_out, items, point_first, spacing=0, flags=0):
        """zlb_inflate_index_host (see inflate_index)."""
        items, results = self._tables(items)
        first, points, counts = self._index_tables(len(items), point_first)
        pi, ni, ki = self._host_ptr(h_in)
        po, no, ko = self._host_ptr(h_out)
        rc = self.lib.zlb_inflate_index_host(self.h, pi, ni, po, no, items.ctypes.data, results.ctypes.data, len(items),
                                             flags, spacing, points.ctypes.data, first.ctypes.data, counts.ctypes.data)
        self._check(rc, "zlb_inflate_index_host")
        return results, points, counts

    def inflate_ranges_host(self, h_in, h_win, h_out, points, ranges, flags=0):
        """zlb_inflate_ranges_host (see inflate_ranges)."""
        points = np.ascontiguousarray(points, dtype=POINT_DTYPE)
        ranges = np.ascontiguousarray(ranges, dtype=RANGE_DTYPE)
        results = np.zeros(len(ranges), dtype=RESULT_DTYPE)
        pi, ni, ki = self._host_ptr(h_in)
        pw, nw, kw = self._host_ptr(h_win) if h_win is not None else (None, 0, None)
        po, no, ko = self._host_ptr(h_out)
        rc = self.lib.zlb_inflate_ranges_host(self.h, pi, ni, pw, nw, po, no, points.ctypes.data, len(points),
                                              ranges.ctypes.data, results.ctypes.data, len(ranges), flags)
        self._check(rc, "zlb_inflate_ranges_host")
        return results

    def checksum_batch_host(self, h_in, items, kinds=SUM_CRC32 | SUM_ADLER32):
        items, results = self._tables(items)
        pi, ni, ki = self._host_ptr(h_in)
        rc = self.lib.zlb_checksum_batch_host(self.h, pi, ni, items.ctypes.data, results.ctypes.data, len(items), kinds)
        self._check(rc, "zlb_checksum_batch_host")
        return results

    # ---- container assembly -------------------------------------------------------------------
    def archive(self, kind, d_in, d_meta, entries, d_out, tail=(0, 0), block_type=DYNAMIC, chunk_bytes=0,
                mode=MODE_COMPAT):
        """zlb_archive on device tensors; returns (archive bytes written, results)."""
        entries = np.ascontiguousarray(entries, dtype=ENTRY_DTYPE)
        results = np.zeros(len(entries), dtype=RESULT_DTYPE)
        total = ctypes.c_uint64(0)
        rc = self.lib.zlb_archive(self.h, kind, d_in.data_ptr(), d_meta.data_ptr(), entries.ctypes.data, len(entries),
                                  tail[0], tail[1], d_out.data_ptr(), d_out.numel(), ctypes.byref(total),
                                  results.ctypes.data, mode, block_type, chunk_bytes)
        self._check(rc, "zlb_archive")
        return int(total.value), results

    def archive_host(self, kind, h_in, h_meta, entries, tail=(0, 0), block_type=DYNAMIC, chunk_bytes=0,
                     mode=MODE_COMPAT, h_out=None):
        """zlb_archive_host; returns (archive as a uint8 array, results)."""
        entries = np.ascontiguousarray(entries, dtype=ENTRY_DTYPE)
        results = np.zeros(len(entries), dtype=RESULT_DTYPE)
        pi, ni, ki = self._host_ptr(h_in)
        pm, nm, km = self._host_ptr(h_meta)
        if h_out is None:
            h_out = np.empty(max(1, archive_bound(kind, entries, tail[1], mode_chunk(mode, chunk_bytes), block_type)),
                             dtype=np.uint8)
        po, no, ko = self._host_ptr(h_out)
        total = ctypes.c_uint64(0)
        rc = self.lib.zlb_archive_host(self.h, kind, pi, ni, pm, nm, entries.ctypes.data, len(entries), tail[0],
                                       tail[1], po, no, ctypes.byref(total), results.ctypes.data, mode, block_type,
                                       chunk_bytes)
        self._check(rc, "zlb_archive_host")
        return h_out[:int(total.value)], results

    # ---- test hooks ---------------------------------------------------------------------------
    def debug_lz77(self, d_in, n):
        tokens = np.zeros(n + 1, dtype=np.uint32)
        hist = np.zeros(316, dtype=np.uint32)
        ntok = ctypes.c_uint32(0)
        rc = self.lib.zlb_debug_lz77(self.h, d_in.data_ptr(), n, tokens.ctypes.data, ctypes.byref(ntok), hist.ctypes.data)
        self._check(rc, "zlb_debug_lz77")
        return tokens[:ntok.value], hist

    def debug_code_lengths(self, freqs, limit):
        freqs = np.ascontiguousarray(freqs, dtype=np.uint32)
        lengths = np.zeros(len(freqs), dtype=np.uint8)
        rc = self.lib.zlb_debug_code_lengths(self.h, freqs.ctypes.data, len(freqs), limit, lengths.ctypes.data)
        self._check(rc, "zlb_debug_code_lengths")
        return lengths

    def debug_block_starts(self, d_in, cuts, span):
        """The split's block finder on the bytes of d_in (a CUDA uint8 tensor) as one item: per byte position in
        `cuts`, the first candidate bit offset in [8 cut, 8 cut + span) (a stored block: where it ends), or -1."""
        cuts = np.ascontiguousarray(cuts, dtype=np.uint64)
        out = np.zeros(len(cuts), dtype=np.uint64)
        rc = self.lib.zlb_debug_block_starts(self.h, d_in.data_ptr(), d_in.numel(), cuts.ctypes.data, len(cuts), span,
                                             out.ctypes.data)
        self._check(rc, "zlb_debug_block_starts")
        return np.where(out == np.uint64(2**64 - 1), -1, out.astype(np.int64))


_default_engines = {}


def default_engine(device=0):
    """Process-wide engine per device, created on first use (raises without a GPU)."""
    eng = _default_engines.get(device)
    if eng is None:
        eng = _default_engines[device] = Engine(device)
    return eng
