"""zlib.ts on B200: CUDA DEFLATE engine behind the zlib.ts API (host mirror + C-ABI binding)."""
from ._native import (  # noqa: F401
    Engine, EngineError, load_library, default_engine, make_items, make_entries, deflate_bound, archive_bound,
    crc32_combine, adler32_combine, host_alloc, host_free, host_is_pinned, ITEM_DTYPE, RESULT_DTYPE, ENTRY_DTYPE, EXPORTS, LIB_PATH,
    DICT_DTYPE, make_dicts, POINT_DTYPE, RANGE_DTYPE, make_ranges, INDEX_DEFAULT_SPACING,
    FRAME_ZLIB, FRAME_GZIP, FRAME_ZIP,
    NONE, FIXED, DYNAMIC, MODE_COMPAT, MODE_FAST, MODE_PRIMED, MODE_SMALLEST, MODE_LAZY, PRIMED_CHUNK, mode_fast, mode_chunk,
    DEFLATE_WANT_CRC32, DEFLATE_WANT_ADLER32, DEFLATE_NOT_FINAL,
    INFLATE_WANT_CRC32, INFLATE_WANT_ADLER32, INFLATE_CHECK_NLEN, INFLATE_SPLIT, SUM_CRC32, SUM_ADLER32,
    ST_OK, ST_INPUT_BROKEN, ST_BTYPE, ST_CODE_LENGTH, ST_OUT_OVERFLOW, ST_STORED_LEN, ST_BAD_CODE, ST_BAD_LENGTHS,
)
from . import synth  # noqa: F401
from . import api  # noqa: F401,E402
from .api import (  # noqa: F401,E402
    Zlib, Deflate, Inflate, GZip, GUnzip, Zip, Unzip, RawDeflate, RawInflate, CRC32, Adler32, ZlibError,
    CompressionType, BufferType, ZipCompressionMethod, deflate_many, inflate_many, inflate_blob, inflate_sizes, checksum_many,
    archive_many, zlib_many, gzip_many, inflate_index, InflateIndex, read_ranges,
)
