/*
 * zlibts_b200.h -- C ABI of the B200-native DEFLATE engine behind the zlib.ts API.
 *
 * The reference (ExaGraphica/zlib.ts) has no FFI: its container classes construct the codec
 * classes directly. The entry points below are what a Node N-API addon binds at exactly those
 * seams (INTEGRATION.md shows the binding):
 *
 *   raw deflate  new RawDeflate(input, opts).compress()   src/Deflate.ts:43,84-85  src/GZip.ts:159-166
 *                                                         src/Zip.ts:379-382       -> zlb_deflate_batch[_host]
 *   raw inflate  new RawInflate(input, {index,...})       src/Inflate.ts:61-66,77-78  src/GUnzip.ts:152-156
 *                  .decompress()                          src/Unzip.ts:285-288     -> zlb_inflate_batch[_host]
 *   CRC-32       CRC32.create / update                    src/GZip.ts:154,180  src/GUnzip.ts:128,160
 *                                                         src/Zip.ts:93,144    src/Unzip.ts:294
 *   Adler-32     Adler32.create / update                  src/Deflate.ts:81    src/Inflate.ts:84
 *                                                                                  -> zlb_checksum_batch[_host]
 *   preset dictionaries (zlib's deflateSetDictionary / inflateSetDictionary; the reference's Inflate refuses FDICT,
 *   src/Inflate.ts:56-57)                                 -> zlb_deflate_batch_dict[_host], zlb_inflate_batch_dict[_host]
 *
 * Conventions
 *   - plain pointers and sizes only; no exceptions cross the ABI.
 *   - return value: 0 = ok, < 0 = API / CUDA failure (zlb_last_error() has the text).
 *   - per-item data errors (corrupt stream, output too small) are reported in zlb_result.status;
 *     the TS shim turns them into `throw new Error(<reference text>)` (texts listed below).
 *   - a ctx is single-owner (not internally locked); one ctx per GPU for multi-GPU work.
 *   - "device" entry points take DEVICE pointers for data and HOST pointers for the item/result
 *     tables; "_host" entry points take HOST pointers for everything and do the copies themselves.
 *   - there is no CPU fallback: without a usable CUDA device zlb_create() fails.
 */
#ifndef ZLIBTS_B200_H
#define ZLIBTS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ZLB_ABI_VERSION 1

typedef struct zlb_ctx zlb_ctx;

/* API-level return codes */
enum {
    ZLB_OK = 0,
    ZLB_E_ARG = -1,
    ZLB_E_CUDA = -2,
    ZLB_E_NOMEM = -3,
    ZLB_E_UNSUPPORTED = -4
};

/* per-item status (zlb_result.status); reference message each one maps to */
enum {
    ZLB_ST_OK = 0,
    ZLB_ST_INPUT_BROKEN = 1,  /* 'input buffer is broken'                    src/RawInflate.ts:188,282 */
    ZLB_ST_BTYPE = 2,         /* 'unknown BTYPE: 3'                          src/RawInflate.ts:168 */
    ZLB_ST_CODE_LENGTH = 3,   /* 'invalid code length: N'                    src/RawInflate.ts:238; the input ends inside a
                                 Huffman code of N bits: status = ZLB_ST_CODE_LENGTH | N << 8 (compare (status & 0xFF):
                                 this status and ZLB_ST_STORED_LEN carry a detail above bit 7) */
    ZLB_ST_OUT_OVERFLOW = 4,  /* caller's out_cap too small (the reference grows its buffer instead) */
    ZLB_ST_STORED_LEN = 5,    /* 'invalid uncompressed block header: LEN'    src/RawInflate.ts:266; | 1 << 8: '... NLEN' (:272) */
    ZLB_ST_BAD_CODE = 6,      /* undefined Huffman code / distance beyond output start / bad symbol:
                                 the reference loops or emits zeros here (SURVEY App. B-8); we stop */
    ZLB_ST_BAD_LENGTHS = 7    /* over-subscribed code-length set in a dynamic header */
};

/* CompressionType, src/RawDeflate.ts:12-17 */
enum { ZLB_NONE = 0, ZLB_FIXED = 1, ZLB_DYNAMIC = 2 };

/* deflate mode. COMPAT: every chunk's bytes equal the reference's RawDeflate run on that chunk
 * (lazy = 0, src/LZ77.ts:196-283 exhaustive longest/nearest match, src/RawDeflate.ts:484-571 code
 * lengths). */
enum { ZLB_MODE_COMPAT = 0, ZLB_MODE_FAST = 1, ZLB_MODE_PRIMED = 2, ZLB_MODE_SMALLEST = 4, ZLB_MODE_LAZY = 8 };
/* FAST: same kernels and the same exact Huffman construction, but a match search looks only at the `depth` nearest
 * entries of the position's hash bucket (default ZLB_FAST_DEFAULT_DEPTH, at most 64): still the greedy parse and a
 * valid stream for the reference's Inflate, no longer byte-identical; the size stays within 3 % of the
 * reference-compatible mode on the benchmark data (bench.py reports it). A depth is passed as ZLB_MODE_FAST_DEPTH(d).
 * LAZY (a flag for FAST): one-step lazy evaluation -- a match shorter than 32 is only taken if the next position
 * has no longer one, otherwise the position becomes a literal (what src/LZ77.ts:243-256 meant to do; the reference's
 * own `lazy` option corrupts data, SURVEY B-2, and is refused by the host mirror). */
/* PRIMED (SURVEY 8(f)-1, pigz-style dictionary priming; may be or-ed with FAST): the match search of a chunk also
 * reaches into the 32 KiB of the same item in front of it, which recovers the ratio independent chunks lose. History
 * and chunk share the 64 KiB a CTA indexes, so chunks are at most ZLB_PRIMED_CHUNK bytes (chunk_bytes 0 = that; pass
 * the same value to zlb_deflate_bound). Blocks are still one per chunk with their own codes, joined by the
 * byte-aligning empty stored block, so the item remains one RFC-1951 stream for the reference's RawInflate; what is
 * given up is per-chunk byte identity with RawDeflate(chunk). ZLB_INFLATE_SPLIT still decodes the chunks side by side
 * (its window mode resolves the back references across the markers). Without FAST the search is the reference's exhaustive one, and
 * every block equals the reference's block construction run with that history (oracle: zo_raw_deflate_dict). */
/* SMALLEST (SURVEY 8(f)-4; a flag for block_type DYNAMIC, may be or-ed with the others): each chunk is written as the
 * shortest of the reference's three block constructions over the chunk's tokens -- dynamic, fixed, or stored
 * (stored only if strictly shorter than both, fixed only if strictly shorter than dynamic; sizes compared in whole
 * bytes of the block alone). The reference never falls back (src/RawDeflate.ts:105-108), so incompressible data grows
 * by a code table per chunk there; here it grows by 5 bytes per 65535. results[i].blocks counts chunks. */
#define ZLB_PRIMED_CHUNK 32768u
#define ZLB_FAST_DEFAULT_DEPTH 16
#define ZLB_MODE_FAST_DEPTH(d) (ZLB_MODE_FAST | ((int)(d) << 8))

/* flags for zlb_deflate_batch */
enum {
    ZLB_DEFLATE_WANT_CRC32 = 1u << 0,   /* results[i].crc32   = CRC-32 of item input  */
    ZLB_DEFLATE_WANT_ADLER32 = 1u << 1, /* results[i].adler32 = Adler-32 of item input */
    ZLB_DEFLATE_NOT_FINAL = 1u << 2     /* the last chunk of every item is not final either (BFINAL = 0 + join
                                           marker): the item is a shard whose successor follows, e.g. on the next GPU */
};

/* flags for zlb_inflate_batch */
enum {
    ZLB_INFLATE_WANT_CRC32 = 1u << 0,   /* results[i].crc32   = CRC-32 of item output  */
    ZLB_INFLATE_WANT_ADLER32 = 1u << 1, /* results[i].adler32 = Adler-32 of item output */
    ZLB_INFLATE_CHECK_NLEN = 1u << 2,   /* verify NLEN == ~LEN in stored blocks (the reference
                                           never does: src/RawInflate.ts:277 is always false) */
    ZLB_INFLATE_SPLIT = 1u << 3,        /* large items are cut where the engine can prove a block boundary and
                                           their pieces decoded side by side: at sync-flush markers (empty stored
                                           blocks, `00 00 FF FF`), and in any stream -- gzip, zlib.compress, any
                                           encoder -- at block starts found on the device in stretches of more than
                                           1 MiB without markers. Independent pieces (what zlb_deflate_batch
                                           emits) are decoded directly, pieces that reach up to 32 KiB into the ones
                                           before (ZLB_MODE_PRIMED, zlib's Z_SYNC_FLUSH, found block starts) in
                                           window mode; a cut is used only once the piece in front of it ended
                                           exactly there, anything else falls back to the one-warp decoder. Results
                                           are identical. */
    ZLB_INFLATE_SEGMENT = 1u << 4       /* internal: an item may end at a block boundary without BFINAL */
};

/* flags for zlb_checksum_batch */
enum { ZLB_SUM_CRC32 = 1u << 0, ZLB_SUM_ADLER32 = 1u << 1 };

/* one unit of work: offsets into the caller's input / output buffers */
typedef struct {
    uint64_t in_off;   /* first input byte of this item                                  */
    uint64_t in_len;   /* deflate: bytes to compress; inflate: bytes available from in_off */
    uint64_t out_off;  /* where this item's output starts                                */
    uint64_t out_cap;  /* bytes available at out_off                                     */
} zlb_item;

typedef struct {
    uint32_t status;   /* ZLB_ST_*                                                        */
    uint32_t crc32;    /* when requested                                                  */
    uint32_t adler32;  /* when requested                                                  */
    uint32_t blocks;   /* deflate: blocks written; inflate: blocks parsed                 */
    uint64_t out_len;  /* bytes written at out_off  (deflate: == reference `.op - outputIndex`) */
    uint64_t in_used;  /* inflate: deflate bytes consumed, so reference `.ip` = index + in_used */
} zlb_result;

/* ---- context ---------------------------------------------------------------------------- */
/* `stream` is a cudaStream_t to launch on (NULL = the ctx creates its own non-blocking stream). */
int zlb_create(int device, void* stream, zlb_ctx** out);
void zlb_destroy(zlb_ctx* ctx);
const char* zlb_last_error(const zlb_ctx* ctx);
int zlb_abi_version(void);
/* the cudaStream_t all work of this ctx is ordered on */
void* zlb_stream(const zlb_ctx* ctx);

/* ---- page-locked host memory ----------------------------------------------------------------
 * The "_host" entry points run at full speed on page-locked buffers (their copies overlap the kernels wave by wave).
 * A caller that owns its allocations -- an N-API addon handing out external ArrayBuffers (napi/addon.cc), a C
 * program -- gets such buffers here. Buffers that are NOT page-locked (a JS-heap Uint8Array, malloc) are accepted
 * just the same: the library then goes through page-locked shadows of its own, filled and drained by a few copy
 * threads while the pipeline runs (one more memcpy per byte; blobs above 4 GiB take the driver's pageable path).
 * Replaces nothing in the reference -- `new Uint8Array(n)` (src/RawDeflate.ts:58, src/RawInflate.ts:100-106) is what
 * a binding would swap for it. */
int zlb_host_alloc(size_t bytes, void** out);
void zlb_host_free(void* p);
int zlb_host_is_pinned(const void* p);  /* 1 when the "_host" entry points can copy from / to p directly */

/* ---- raw deflate (replaces RawDeflate.compress, src/RawDeflate.ts:87-114) -------------------
 * Each item is cut into chunks of `chunk_bytes` (<= 65536; 0 = 65536); every chunk becomes one
 * block of `block_type`. Chunks of an item are joined with an empty stored block that byte-aligns
 * (sync-flush marker, SURVEY App. A.7) and the last one carries BFINAL=1, so the item's output is
 * one RFC-1951 stream that the reference's RawInflate decodes (src/RawInflate.ts:128-130).
 * An item of at most chunk_bytes bytes is byte-identical to the reference's output.              */
int zlb_deflate_batch(zlb_ctx* ctx, const void* d_in, void* d_out, const zlb_item* items,
                      zlb_result* results, size_t n_items, int mode, int block_type,
                      uint32_t chunk_bytes, uint32_t flags);
int zlb_deflate_batch_host(zlb_ctx* ctx, const void* h_in, size_t in_bytes, void* h_out, size_t out_bytes,
                           const zlb_item* items, zlb_result* results, size_t n_items, int mode,
                           int block_type, uint32_t chunk_bytes, uint32_t flags);
/* output bytes that always suffice for an item of in_len bytes */
uint64_t zlb_deflate_bound(uint64_t in_len, uint32_t chunk_bytes, int block_type);

/* ---- preset dictionaries (zlib's deflateSetDictionary / inflateSetDictionary, RFC 1950 FDICT) ----------------
 * An engine extension: the reference's Inflate refuses FDICT streams (src/Inflate.ts:56-57). dicts[i] names item i's
 * dictionary as a span of one dictionary blob (d_dict: device pointer; h_dict: host pointer); a shared dictionary is
 * every entry naming the same span. dicts == NULL, or len == 0, means no dictionary; zlb_deflate_batch[_host] and
 * zlb_inflate_batch[_host] are these calls with dicts == NULL. Only the last 32768 bytes of a dictionary can be
 * reached (the DEFLATE window). Results keep their meaning: CRC-32 / Adler-32 cover the item's own bytes.
 * ZLB_E_ARG: a span outside dict_bytes (host entry points), or len > 0 with a NULL blob.                        */
typedef struct {
    uint64_t off;   /* first byte of this item's dictionary in the dictionary blob                    */
    uint64_t len;   /* 0 = no dictionary; only the last 32768 bytes are used (the DEFLATE window)      */
} zlb_dict;

/* Deflate with a dictionary: a chunk's match search also reaches into the last min(32768, ...) bytes of
 * dictionary || the item's bytes in front of the chunk. Without ZLB_MODE_PRIMED only an item's first chunk has the
 * dictionary as history (later chunks stay independent); with it every chunk searches its 32 KiB of dictionary || item.
 * When any item of the call has a dictionary, chunks are at most ZLB_PRIMED_CHUNK bytes (history and chunk share
 * the 64 KiB a CTA indexes; size slots with zlb_deflate_bound(in_len, ZLB_PRIMED_CHUNK, ...)). In the compat mode the
 * first chunk's block is the reference's block construction run with that history; block_type ZLB_NONE ignores the
 * dictionary.                                                                                                    */
int zlb_deflate_batch_dict(zlb_ctx* ctx, const void* d_in, void* d_out, const void* d_dict, const zlb_dict* dicts,
                           const zlb_item* items, zlb_result* results, size_t n_items, int mode, int block_type,
                           uint32_t chunk_bytes, uint32_t flags);
int zlb_deflate_batch_dict_host(zlb_ctx* ctx, const void* h_in, size_t in_bytes, void* h_out, size_t out_bytes,
                                const void* h_dict, size_t dict_bytes, const zlb_dict* dicts, const zlb_item* items,
                                zlb_result* results, size_t n_items, int mode, int block_type, uint32_t chunk_bytes,
                                uint32_t flags);

/* ---- raw inflate (replaces RawInflate.decompress, src/RawInflate.ts:127-140) ----------------
 * One warp per item. in_off points at the first deflate byte (the caller has applied the
 * reference's `index` option); trailing container bytes may follow the stream.               */
int zlb_inflate_batch(zlb_ctx* ctx, const void* d_in, void* d_out, const zlb_item* items,
                      zlb_result* results, size_t n_items, uint32_t flags);
int zlb_inflate_batch_host(zlb_ctx* ctx, const void* h_in, size_t in_bytes, void* h_out, size_t out_bytes,
                           const zlb_item* items, zlb_result* results, size_t n_items, uint32_t flags);
/* Inflate with a dictionary (zlb_dict above): a distance may reach up to the dictionary's first usable byte in
 * front of the output; one beyond it is ZLB_ST_BAD_CODE as before. ZLB_INFLATE_SPLIT takes the same routes, the
 * window in front of an item's first piece being the dictionary.                                                */
int zlb_inflate_batch_dict(zlb_ctx* ctx, const void* d_in, void* d_out, const void* d_dict, const zlb_dict* dicts,
                           const zlb_item* items, zlb_result* results, size_t n_items, uint32_t flags);
int zlb_inflate_batch_dict_host(zlb_ctx* ctx, const void* h_in, size_t in_bytes, void* h_out, size_t out_bytes,
                                const void* h_dict, size_t dict_bytes, const zlb_dict* dicts, const zlb_item* items,
                                zlb_result* results, size_t n_items, uint32_t flags);
/* Decompressed size of every item without writing it (an engine extension: no format carries a usable size -- zlib
 * none, gzip's ISIZE only mod 2^32, raw deflate none -- so callers can allocate exact output slots). items[i].in_off /
 * in_len as for zlb_inflate_batch; out_off / out_cap are ignored. dicts (may be NULL): as for zlb_inflate_batch_dict,
 * but only .len is read -- a dictionary decides how far a distance may reach, never a size -- so no dictionary blob is
 * passed. flags: ZLB_INFLATE_SPLIT, ZLB_INFLATE_CHECK_NLEN; ZLB_INFLATE_WANT_CRC32 / _ADLER32 are ZLB_E_ARG (there are
 * no bytes to sum), as is a NULL input with items. results[i].status / out_len / in_used / blocks equal those
 * zlb_inflate_batch_dict returns for the same item, flags and dictionary with out_cap >= the item's size (never
 * ZLB_ST_OUT_OVERFLOW); crc32 = adler32 = 0. A size-only decode stores nothing and skips stored data; with
 * ZLB_INFLATE_SPLIT every stream the split can cut, primed, Z_SYNC_FLUSH and marker-less ones included, is sized
 * piecewise without scratch for its bytes.                                                                                 */
int zlb_inflate_size_batch(zlb_ctx* ctx, const void* d_in, const zlb_dict* dicts, const zlb_item* items,
                           zlb_result* results, size_t n_items, uint32_t flags);
int zlb_inflate_size_batch_host(zlb_ctx* ctx, const void* h_in, size_t in_bytes, const zlb_dict* dicts,
                                const zlb_item* items, zlb_result* results, size_t n_items, uint32_t flags);

/* ---- random access through an index of access points (what zlib's zran.c, indexed_gzip and rapidgzip offer) -----
 * An access point is a block start of a stream that a decode proved: its bit offset from the stream's first byte
 * (items[i].in_off), the decompressed bytes in front of it, and where its window -- the min(out_pos, 32768) bytes in
 * front of it -- lies in a window blob. A read of [pos, pos + len) starts at the last point at or before pos instead
 * of the start of the stream, and a long read is cut at every point inside it, each piece decoded by its own warp.
 *
 * zlb_inflate_index[_host]: a decode that also reports access points. Output bytes and results are those of
 * zlb_inflate_batch[_host] with flags | ZLB_INFLATE_SPLIT (flags: ZLB_INFLATE_WANT_CRC32 / _ADLER32 / _CHECK_NLEN;
 * no preset dictionaries). Item i's points go to points[point_first[i] .. point_first[i + 1]) (point_first has
 * n_items + 1 nondecreasing entries; when the slots run out later points are dropped: the index is only sparser) and
 * their number to point_count[i]; an item that failed gets 0. Points ascend in in_bit and out_pos, the first is
 * {0, 0}. The candidates are the block starts the decode proved: the split's piece starts, or every block header
 * when one warp decodes the item. The choice is greedy: the first candidate whose out_pos is at least the previous
 * point's out_pos + spacing (0 = ZLB_INDEX_DEFAULT_SPACING). win_off = items[i].out_off + out_pos -
 * min(out_pos, 32768): the call's output blob is the window blob (a caller that keeps only the windows compacts them
 * and rewrites win_off).
 *
 * zlb_inflate_ranges[_host]: batched reads. Range i wants out_cap bytes from decompressed position pos of the stream
 * at in_off / in_len of the input, whose points are points[pt_first .. pt_first + pt_count). The range is cut at the
 * points inside [pos, pos + out_cap); every piece is decoded by one warp from its point with that point's window (in
 * d_win / h_win). results[i].out_len = min(out_cap, size - pos) (0 at or past the end: a short read is ZLB_ST_OK),
 * status = the decoder's status for a data error inside the stretch decoded, crc32 / adler32 of the bytes written
 * when requested (flags: ZLB_INFLATE_WANT_CRC32 / _ADLER32 / _CHECK_NLEN), in_used = blocks = 0. Nothing is written
 * outside [out_off, out_off + out_cap), whatever the windows hold: a wrong window gives wrong bytes or
 * ZLB_ST_BAD_CODE (zlib's inflateSetDictionary contract). The bytes do not depend on which of a stream's points are
 * passed as long as the first one is; only the speed does. ZLB_E_ARG: pt_count == 0, a first point that is not
 * {0, 0}, points that do not ascend, a point behind 8 * in_len, pos + out_cap beyond 2^64, a point with a window and
 * a NULL window blob, a window span outside win_bytes or a range slot outside out_bytes (_host), any other flag.
 * A range's first piece decodes the bytes between its point and pos into scratch (at most what the rest of the
 * stream can give: 258 bytes per bit); ZLB_E_NOMEM when that alone exceeds what a call may take -- pass the points
 * between. A pos beyond what the stream can give from its point is a read past the end (out_len 0), decoded not at
 * all.                                                                                                           */
#define ZLB_INDEX_DEFAULT_SPACING (1u << 20)
typedef struct {
    uint64_t in_bit;   /* a block start: bit offset from the stream's first byte; 0 for the first point           */
    uint64_t out_pos;  /* decompressed bytes in front of it                                                        */
    uint64_t win_off;  /* its window, the min(out_pos, 32768) decompressed bytes in front of it, in the window blob */
} zlb_point;

typedef struct {
    uint64_t in_off, in_len;     /* the stream, as the index build saw it                                  */
    uint64_t pt_first, pt_count; /* its points: points[pt_first .. pt_first + pt_count)                    */
    uint64_t pos;                /* first decompressed byte wanted                                          */
    uint64_t out_off, out_cap;   /* where the bytes go; out_cap bytes are wanted                            */
} zlb_range;

int zlb_inflate_index(zlb_ctx* ctx, const void* d_in, void* d_out, const zlb_item* items, zlb_result* results,
                      size_t n_items, uint32_t flags, uint64_t spacing, zlb_point* points, const uint64_t* point_first,
                      uint64_t* point_count);
int zlb_inflate_index_host(zlb_ctx* ctx, const void* h_in, size_t in_bytes, void* h_out, size_t out_bytes,
                           const zlb_item* items, zlb_result* results, size_t n_items, uint32_t flags, uint64_t spacing,
                           zlb_point* points, const uint64_t* point_first, uint64_t* point_count);
int zlb_inflate_ranges(zlb_ctx* ctx, const void* d_in, const void* d_win, void* d_out, const zlb_point* points,
                       size_t n_points, const zlb_range* ranges, zlb_result* results, size_t n_ranges, uint32_t flags);
int zlb_inflate_ranges_host(zlb_ctx* ctx, const void* h_in, size_t in_bytes, const void* h_win, size_t win_bytes,
                            void* h_out, size_t out_bytes, const zlb_point* points, size_t n_points,
                            const zlb_range* ranges, zlb_result* results, size_t n_ranges, uint32_t flags);

/* ---- checksums (replace CRC32.create src/CRC32.ts:13, Adler32.create src/Adler32.ts:13) ----- */
int zlb_checksum_batch(zlb_ctx* ctx, const void* d_in, const zlb_item* items, zlb_result* results,
                       size_t n_items, uint32_t kinds);
int zlb_checksum_batch_host(zlb_ctx* ctx, const void* h_in, size_t in_bytes, const zlb_item* items,
                            zlb_result* results, size_t n_items, uint32_t kinds);
/* checksum of A||B from checksum(A), checksum(B), len(B); used to stitch shards / GPUs */
uint32_t zlb_crc32_combine(uint32_t crc_a, uint32_t crc_b, uint64_t len_b);
uint32_t zlb_adler32_combine(uint32_t adler_a, uint32_t adler_b, uint64_t len_b);

/* ---- container assembly on the device (SURVEY 8(f)-2) ---------------------------------------
 * Replaces the byte shuffling around the codec in Deflate.compress (src/Deflate.ts:60-99: 2-byte header, raw
 * stream, Adler-32 big endian), GZip.compress (src/GZip.ts:96-194: member header, raw stream, CRC-32 and ISIZE
 * little endian) and Zip.compress (src/Zip.ts:117-372: local header + data per entry, central directory, end
 * record): every entry is checksummed and deflated in ONE batch, then framed and packed back to back by kernels,
 * so the archive leaves the GPU as one contiguous buffer and the host never touches an entry's bytes.
 *
 * The caller supplies the parts that do not depend on the data as byte templates in a `meta` blob:
 *   ZLB_FRAME_ZLIB  head = CMF, FLG (src/Deflate.ts:67-78)
 *   ZLB_FRAME_GZIP  head = the member header incl. name / comment / header CRC (src/GZip.ts:108-156)
 *   ZLB_FRAME_ZIP   head = local file header, 30 bytes + name (src/Zip.ts:228-312); cdir = the entry's central
 *                   directory header, 46 bytes + name + comment (src/Zip.ts:234-326); tail = end record,
 *                   22 bytes + comment (src/Zip.ts:340-369). The engine fills in what only it knows: CRC-32 and
 *                   compressed size (local +14, +18; central +16, +20), the local header offset (central +42),
 *                   directory size and offset (end record +12, +16).
 * Archive layout: entries in order, each head | body | trailer; for ZIP the central directory and the end record
 * follow the last entry (ZIP32 only, like the reference: more than 65 535 entries or 4 GiB are refused). results[i]: status, crc32 / adler32, out_len = bytes of the framed entry,
 * in_used = offset of its first header byte in the archive.                                               */
enum { ZLB_FRAME_ZLIB = 1, ZLB_FRAME_GZIP = 2, ZLB_FRAME_ZIP = 3 };

typedef struct {
    uint64_t in_off;    /* the entry's plain bytes in the input blob                          */
    uint64_t in_len;
    uint64_t head_off;  /* header template in the meta blob                                   */
    uint32_t head_len;
    uint32_t method;    /* ZIP: 0 = stored, 8 = deflate (src/Zip.ts:7-10); otherwise ignored  */
    uint64_t cdir_off;  /* ZIP: central directory header template in the meta blob            */
    uint32_t cdir_len;
    uint32_t reserved;
} zlb_entry;

/* archive bytes that always suffice for these entries */
uint64_t zlb_archive_bound(int kind, const zlb_entry* entries, size_t n_entries, uint64_t tail_len,
                           uint32_t chunk_bytes, int block_type);
/* device buffers: d_in (plain bytes), d_meta (templates), d_out (archive, out_cap bytes). *out_len = archive size;
 * when out_cap is too small nothing is written, *out_len is the size needed and ZLB_E_ARG is returned. */
int zlb_archive(zlb_ctx* ctx, int kind, const void* d_in, const void* d_meta, const zlb_entry* entries,
                size_t n_entries, uint64_t tail_off, uint64_t tail_len, void* d_out, uint64_t out_cap,
                uint64_t* out_len, zlb_result* results, int mode, int block_type, uint32_t chunk_bytes);
int zlb_archive_host(zlb_ctx* ctx, int kind, const void* h_in, size_t in_bytes, const void* h_meta,
                     size_t meta_bytes, const zlb_entry* entries, size_t n_entries, uint64_t tail_off,
                     uint64_t tail_len, void* h_out, uint64_t out_cap, uint64_t* out_len, zlb_result* results,
                     int mode, int block_type, uint32_t chunk_bytes);

/* ---- instrumentation ----------------------------------------------------------------------- */
/* When enabled every kernel launch is bracketed by CUDA events on the ctx stream.            */
int zlb_profile_enable(zlb_ctx* ctx, int on);
/* Resolves pending events (synchronises the stream) and reports, for kernel slot k < *n:
 * names[k], total milliseconds, launch count since the last reset. Pass NULL arrays to query n. */
int zlb_profile_read(zlb_ctx* ctx, int* n, const char** names, double* total_ms, uint64_t* launches);
int zlb_profile_reset(zlb_ctx* ctx);
/* kernels launched by this ctx since creation (all entry points) */
uint64_t zlb_launch_count(const zlb_ctx* ctx);

/* ---- test hooks (used by tests/ only): expose intermediate results of the deflate pipeline -- */
/* LZ77 tokens of ONE chunk (<= 65536 bytes at d_in): tokens_out[k] = literal byte, or
 * 0x80000000 | (len-3) << 16 | (dist-1); *n_tokens excludes the end-of-block symbol.
 * hist_out: 286 litlen + 30 dist counters exactly as src/LZ77.ts:126-128,279 leaves them.     */
int zlb_debug_lz77(zlb_ctx* ctx, const void* d_in, uint32_t n, uint32_t* h_tokens_out,
                   uint32_t* n_tokens, uint32_t* h_hist_out);
/* code lengths for one histogram (src/RawDeflate.ts:440-474): freqs[nsym] -> lengths[nsym]     */
int zlb_debug_code_lengths(zlb_ctx* ctx, const uint32_t* h_freqs, int nsym, int limit, uint8_t* h_lengths);
/* the block finder of ZLB_INFLATE_SPLIT on the n input bytes at d_in, taken as one item: for each byte position
 * h_cuts[c] (< n), h_bits_out[c] = the first candidate bit offset b in [8 h_cuts[c], 8 h_cuts[c] + span) -- a dynamic
 * block header as an encoder writes it (the offset itself), or a stored block with LEN == ~NLEN (the offset of the
 * block behind it) -- or UINT64_MAX when there is none. One kernel launch; synchronises.                         */
int zlb_debug_block_starts(zlb_ctx* ctx, const void* d_in, uint64_t n, const uint64_t* h_cuts, size_t n_cuts,
                           uint64_t span, uint64_t* h_bits_out);

#ifdef __cplusplus
}
#endif
#endif
