// zts_container.cu -- container assembly on the device (SURVEY 8(f)-2).
//
// The reference frames the raw stream on the host, entry by entry: Deflate.compress writes CMF/FLG, the stream and
// the Adler-32 (src/Deflate.ts:60-99); GZip.compress the member header, the stream, CRC-32 and ISIZE
// (src/GZip.ts:96-194); Zip.compress sizes one buffer and walks the files with two cursors, local header + data
// through one, central directory through the other, end record last (src/Zip.ts:117-372). Here every entry of a
// call is checksummed and deflated in one batch into scratch slots, the host turns the resulting sizes into
// final offsets (a prefix sum over at most 65 535 numbers), and two kernels write the archive: one copies the
// bodies to their final place in 64 KiB pieces, one writes and patches the headers, trailers, central directory
// and end record. The archive is contiguous in device memory and leaves in one copy.
#include "zts_common.cuh"

#define FRAME_PIECE 65536u

struct ZtsFrame {        // host-built after compression, one per entry
    uint64_t dst_off;    // first header byte in the archive
    uint64_t body_src;   // the body in the scratch slots (or in the input blob when the entry is stored)
    uint64_t body_len;
    uint64_t head_off;   // template in the meta blob
    uint64_t cdir_dst;   // ZIP: where the central directory header goes
    uint64_t cdir_off;   // ZIP: its template
    uint64_t plain_len;
    uint32_t head_len, cdir_len;
    uint32_t crc32, adler32;
    uint32_t stored;     // body = the plain bytes
    uint32_t piece_first;  // index of the entry's first body piece
};

__device__ __forceinline__ void put_u32le(uint8_t* p, uint32_t v)  // ByteStream.writeUint, src/ByteStream.ts
{
    p[0] = (uint8_t)v;
    p[1] = (uint8_t)(v >> 8);
    p[2] = (uint8_t)(v >> 16);
    p[3] = (uint8_t)(v >> 24);
}

// headers, trailers, central directory; block n_entries writes the tail (end record)
__global__ void __launch_bounds__(128)
frame_header_kernel(const uint8_t* __restrict__ meta, const ZtsFrame* __restrict__ frames, uint32_t n, int kind,
                    uint8_t* __restrict__ out, uint64_t tail_off, uint32_t tail_len, uint64_t tail_dst,
                    uint32_t cd_size, uint32_t cd_off)
{
    const uint32_t e = blockIdx.x, tid = threadIdx.x;
    if (e == n) {
        for (uint32_t i = tid; i < tail_len; i += 128) out[tail_dst + i] = meta[tail_off + i];
        __syncthreads();
        if (tid == 0 && kind == ZLB_FRAME_ZIP && tail_len >= 22) {
            put_u32le(out + tail_dst + 12, cd_size);  // src/Zip.ts:357
            put_u32le(out + tail_dst + 16, cd_off);   // src/Zip.ts:360
        }
        return;
    }
    const ZtsFrame f = frames[e];
    uint8_t* d = out + f.dst_off;
    for (uint32_t i = tid; i < f.head_len; i += 128) d[i] = meta[f.head_off + i];
    if (kind == ZLB_FRAME_ZIP)
        for (uint32_t i = tid; i < f.cdir_len; i += 128) out[f.cdir_dst + i] = meta[f.cdir_off + i];
    __syncthreads();
    if (tid != 0) return;
    uint8_t* t = d + f.head_len + f.body_len;
    if (kind == ZLB_FRAME_ZIP) {
        if (f.head_len >= 30) {
            put_u32le(d + 14, f.crc32);                // src/Zip.ts:265
            put_u32le(d + 18, (uint32_t)f.body_len);   // src/Zip.ts:270
        }
        if (f.cdir_len >= 46) {
            uint8_t* c = out + f.cdir_dst;
            put_u32le(c + 16, f.crc32);                // src/Zip.ts:266
            put_u32le(c + 20, (uint32_t)f.body_len);   // src/Zip.ts:271
            put_u32le(c + 42, (uint32_t)f.dst_off);    // src/Zip.ts:304
        }
    } else if (kind == ZLB_FRAME_ZLIB) {
        t[0] = (uint8_t)(f.adler32 >> 24);             // writeUintBE, src/Deflate.ts:95
        t[1] = (uint8_t)(f.adler32 >> 16);
        t[2] = (uint8_t)(f.adler32 >> 8);
        t[3] = (uint8_t)f.adler32;
    } else {
        put_u32le(t, f.crc32);                         // src/GZip.ts:180-181
        put_u32le(t + 4, (uint32_t)f.plain_len);       // ISIZE, src/GZip.ts:184-185
    }
}

// one 64 KiB piece of one body per CTA
__global__ void __launch_bounds__(256)
frame_body_kernel(const uint8_t* __restrict__ in, const uint8_t* __restrict__ body,
                  const ZtsFrame* __restrict__ frames, uint32_t n, uint8_t* __restrict__ out)
{
    __shared__ uint32_t s_entry;
    const uint32_t tid = threadIdx.x;
    if (tid == 0) {  // last entry whose first piece is at or before this one
        uint32_t lo = 0, hi = n;
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (frames[mid].piece_first <= blockIdx.x)
                lo = mid;
            else
                hi = mid;
        }
        s_entry = lo;
    }
    __syncthreads();
    const ZtsFrame f = frames[s_entry];
    const uint64_t begin = (uint64_t)(blockIdx.x - f.piece_first) * FRAME_PIECE;
    if (begin >= f.body_len) return;
    const uint32_t len = (uint32_t)min((uint64_t)FRAME_PIECE, f.body_len - begin);
    const uint8_t* src = (f.stored ? in : body) + f.body_src + begin;
    uint8_t* dst = out + f.dst_off + f.head_len + begin;
    zts_block_copy(dst, src, len, tid, 256);
}

static uint32_t trailer_bytes(int kind) { return kind == ZLB_FRAME_ZLIB ? 4u : kind == ZLB_FRAME_GZIP ? 8u : 0u; }

static bool entry_is_stored(int kind, const zlb_entry& e) { return kind == ZLB_FRAME_ZIP && e.method != 8u; }

extern "C" uint64_t zlb_archive_bound(int kind, const zlb_entry* entries, size_t n, uint64_t tail_len,
                                      uint32_t chunk_bytes, int block_type)
{
    uint64_t total = tail_len;
    for (size_t i = 0; i < n; ++i) {
        const zlb_entry& e = entries[i];
        total += e.head_len + trailer_bytes(kind) + (kind == ZLB_FRAME_ZIP ? e.cdir_len : 0u);
        total += entry_is_stored(kind, e) ? e.in_len : zlb_deflate_bound(e.in_len, chunk_bytes, block_type);
    }
    return total;
}

// Everything up to the final layout: compresses / checksums, fills `frames` and the results, returns the archive size.
struct ArchivePlan {
    std::vector<ZtsFrame> frames;
    uint64_t total = 0, tail_dst = 0, cd_off = 0, cd_size = 0;
    size_t n_pieces = 0;
};

static int archive_compress(zlb_ctx* ctx, int kind, const uint8_t* d_in, const zlb_entry* entries, size_t n,
                            uint64_t tail_len, zlb_result* results, int mode, int block_type, uint32_t chunk_bytes,
                            ArchivePlan& plan)
{
    if (kind != ZLB_FRAME_ZLIB && kind != ZLB_FRAME_GZIP && kind != ZLB_FRAME_ZIP)
        return zts_fail(ctx, ZLB_E_ARG, "unknown container kind %d", kind);
    if (n > 0x7FFFFFFFull) return zts_fail(ctx, ZLB_E_ARG, "too many entries");
    if ((mode & ZLB_MODE_PRIMED) && (chunk_bytes == 0 || chunk_bytes > ZLB_PRIMED_CHUNK)) chunk_bytes = ZLB_PRIMED_CHUNK;
    std::vector<zlb_item> items;
    std::vector<uint32_t> defl, stor;
    uint64_t slot = 0;
    for (size_t i = 0; i < n; ++i) {
        const zlb_entry& e = entries[i];
        zlb_item it = {e.in_off, e.in_len, 0, 0};
        if (entry_is_stored(kind, e)) {
            stor.push_back((uint32_t)i);
        } else {
            it.out_off = slot;
            it.out_cap = zlb_deflate_bound(e.in_len, chunk_bytes, block_type);
            slot += (it.out_cap + 15) & ~15ull;
            defl.push_back((uint32_t)i);
            items.push_back(it);
        }
    }
    memset(results, 0, n * sizeof(zlb_result));
    std::vector<zlb_result> res(defl.size() > stor.size() ? defl.size() : stor.size());
    if (!defl.empty()) {
        int rc = zts_reserve(ctx, &ctx->d_body, slot + 256);
        if (rc) return rc;
        const uint32_t flags = kind == ZLB_FRAME_ZLIB ? ZLB_DEFLATE_WANT_ADLER32 : ZLB_DEFLATE_WANT_CRC32;
        rc = zlb_deflate_batch(ctx, d_in, ctx->d_body.p, items.data(), res.data(), defl.size(), mode, block_type,
                               chunk_bytes, flags);
        if (rc) return rc;
        for (size_t k = 0; k < defl.size(); ++k) results[defl[k]] = res[k];
    }
    if (!stor.empty()) {
        std::vector<zlb_item> sitems(stor.size());
        for (size_t k = 0; k < stor.size(); ++k) sitems[k] = {entries[stor[k]].in_off, entries[stor[k]].in_len, 0, 0};
        int rc = zlb_checksum_batch(ctx, d_in, sitems.data(), res.data(), stor.size(), ZLB_SUM_CRC32);  // src/Zip.ts:144
        if (rc) return rc;
        for (size_t k = 0; k < stor.size(); ++k) {
            results[stor[k]] = res[k];
            results[stor[k]].out_len = entries[stor[k]].in_len;
        }
    }
    // final layout (what src/Zip.ts:190-209 sizes up front after compressing every file)
    plan.frames.resize(n);
    uint64_t off = 0, pieces = 0;
    size_t kd = 0;
    for (size_t i = 0; i < n; ++i) {
        const zlb_entry& e = entries[i];
        ZtsFrame& f = plan.frames[i];
        memset(&f, 0, sizeof f);
        if (results[i].status != ZLB_ST_OK) return zts_fail(ctx, ZLB_E_CUDA, "entry %zu: deflate status %u", i, results[i].status);
        f.stored = entry_is_stored(kind, e) ? 1u : 0u;
        f.body_src = f.stored ? e.in_off : items[kd++].out_off;
        f.body_len = results[i].out_len;
        f.dst_off = off;
        f.head_off = e.head_off;
        f.head_len = e.head_len;
        f.cdir_off = e.cdir_off;
        f.cdir_len = kind == ZLB_FRAME_ZIP ? e.cdir_len : 0u;
        f.plain_len = e.in_len;
        f.crc32 = results[i].crc32;
        f.adler32 = results[i].adler32;
        if (pieces > 0xFFFFFFFFull) return zts_fail(ctx, ZLB_E_ARG, "archive too large");
        f.piece_first = (uint32_t)pieces;
        pieces += (f.body_len + FRAME_PIECE - 1) / FRAME_PIECE;
        const uint64_t framed = (uint64_t)f.head_len + f.body_len + trailer_bytes(kind);
        results[i].out_len = framed;
        results[i].in_used = off;
        off += framed;
    }
    plan.cd_off = off;
    for (size_t i = 0; i < n; ++i) {
        plan.frames[i].cdir_dst = off;
        off += plan.frames[i].cdir_len;
    }
    plan.cd_size = off - plan.cd_off;
    plan.tail_dst = off;
    plan.total = off + tail_len;
    plan.n_pieces = (size_t)pieces;
    if (plan.n_pieces > 0x7FFFFFFFull) return zts_fail(ctx, ZLB_E_ARG, "archive too large");
    if (kind == ZLB_FRAME_ZIP) {
        // the reference writes 32-bit sizes / offsets and a 16-bit entry count (src/Zip.ts:265-304,351-360) and has no
        // ZIP64 records: refuse what would not fit instead of wrapping around
        if (plan.tail_dst > 0xFFFFFFFFull || n > 0xFFFFull)
            return zts_fail(ctx, ZLB_E_ARG, "archive does not fit ZIP32 (%zu entries, %llu bytes before the end record)", n,
                            (unsigned long long)plan.tail_dst);
        for (size_t i = 0; i < n; ++i)
            if (entries[i].in_len > 0xFFFFFFFFull) return zts_fail(ctx, ZLB_E_ARG, "entry %zu does not fit ZIP32", i);
    }
    return ZLB_OK;
}

static int archive_assemble(zlb_ctx* ctx, int kind, const uint8_t* d_in, const uint8_t* d_meta, size_t n,
                            uint64_t tail_off, uint64_t tail_len, uint8_t* d_out, const ArchivePlan& plan)
{
    const size_t bytes = n * sizeof(ZtsFrame);
    int rc = zts_reserve(ctx, &ctx->d_frames, bytes + 64);
    if (rc) return rc;
    rc = zts_reserve_pinned(ctx, &ctx->h_pin, bytes + 64);
    if (rc) return rc;
    if (n) memcpy(ctx->h_pin.p, plan.frames.data(), bytes);
    ZtsFrame* d_frames = (ZtsFrame*)ctx->d_frames.p;
    if (n) ZTS_CUDA(ctx, cudaMemcpyAsync(d_frames, ctx->h_pin.p, bytes, cudaMemcpyHostToDevice, ctx->stream));
    ctx->work = ctx->stream;
    if (plan.n_pieces)
        ZTS_LAUNCH(ctx, ZK_FRAME_BODY,
                   frame_body_kernel<<<(unsigned)plan.n_pieces, 256, 0, ctx->stream>>>(
                       d_in, (const uint8_t*)ctx->d_body.p, d_frames, (uint32_t)n, d_out));
    ZTS_LAUNCH(ctx, ZK_FRAME_HEADER,
               frame_header_kernel<<<(unsigned)n + 1u, 128, 0, ctx->stream>>>(
                   d_meta, d_frames, (uint32_t)n, kind, d_out, tail_off, (uint32_t)tail_len, plan.tail_dst,
                   (uint32_t)plan.cd_size, (uint32_t)plan.cd_off));
    return ZLB_OK;
}

extern "C" int zlb_archive(zlb_ctx* ctx, int kind, const void* d_in, const void* d_meta, const zlb_entry* entries,
                           size_t n, uint64_t tail_off, uint64_t tail_len, void* d_out, uint64_t out_cap,
                           uint64_t* out_len, zlb_result* results, int mode, int block_type, uint32_t chunk_bytes)
{
    if (!ctx || !out_len || (!entries && n) || (!results && n) || (!d_out && out_cap)) return ZLB_E_ARG;
    ZTS_CUDA(ctx, cudaSetDevice(ctx->device));
    ArchivePlan plan;
    int rc = archive_compress(ctx, kind, (const uint8_t*)d_in, entries, n, tail_len, results, mode, block_type,
                              chunk_bytes, plan);
    if (rc) return rc;
    *out_len = plan.total;
    if (plan.total > out_cap) return zts_fail(ctx, ZLB_E_ARG, "archive needs %llu bytes, %llu given",
                                              (unsigned long long)plan.total, (unsigned long long)out_cap);
    rc = archive_assemble(ctx, kind, (const uint8_t*)d_in, (const uint8_t*)d_meta, n, tail_off, tail_len,
                          (uint8_t*)d_out, plan);
    if (rc) return rc;
    ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ZLB_OK;
}

extern "C" int zlb_archive_host(zlb_ctx* ctx, int kind, const void* h_in, size_t in_bytes, const void* h_meta,
                                size_t meta_bytes, const zlb_entry* entries, size_t n, uint64_t tail_off,
                                uint64_t tail_len, void* h_out, uint64_t out_cap, uint64_t* out_len,
                                zlb_result* results, int mode, int block_type, uint32_t chunk_bytes)
{
    if (!ctx || !out_len || (!entries && n) || (!results && n) || (!h_in && in_bytes) || (!h_meta && meta_bytes) ||
        (!h_out && out_cap))
        return ZLB_E_ARG;
    ZTS_CUDA(ctx, cudaSetDevice(ctx->device));
    for (size_t i = 0; i < n; ++i) {
        const zlb_entry& e = entries[i];
        if (e.in_off + e.in_len > in_bytes || e.head_off + e.head_len > meta_bytes ||
            (kind == ZLB_FRAME_ZIP && e.cdir_off + e.cdir_len > meta_bytes))
            return zts_fail(ctx, ZLB_E_ARG, "entry %zu out of range", i);
    }
    if (tail_off + tail_len > meta_bytes) return zts_fail(ctx, ZLB_E_ARG, "tail out of range");
    // input blob and templates share the staging buffer
    const size_t meta_at = (in_bytes + 255) & ~(size_t)255;
    int rc = zts_reserve(ctx, &ctx->d_stage_in, meta_at + meta_bytes + 256);
    if (rc) return rc;
    uint8_t* d_in = (uint8_t*)ctx->d_stage_in.p;
    if (in_bytes) ZTS_CUDA(ctx, cudaMemcpyAsync(d_in, h_in, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    if (meta_bytes)
        ZTS_CUDA(ctx, cudaMemcpyAsync(d_in + meta_at, h_meta, meta_bytes, cudaMemcpyHostToDevice, ctx->stream));
    ArchivePlan plan;
    rc = archive_compress(ctx, kind, d_in, entries, n, tail_len, results, mode, block_type, chunk_bytes, plan);
    if (rc) return rc;
    *out_len = plan.total;
    if (plan.total > out_cap) return zts_fail(ctx, ZLB_E_ARG, "archive needs %llu bytes, %llu given",
                                              (unsigned long long)plan.total, (unsigned long long)out_cap);
    rc = zts_reserve(ctx, &ctx->d_stage_out, plan.total + 256);
    if (rc) return rc;
    rc = archive_assemble(ctx, kind, d_in, d_in + meta_at, n, tail_off, tail_len, (uint8_t*)ctx->d_stage_out.p, plan);
    if (rc) return rc;
    if (plan.total)
        ZTS_CUDA(ctx, cudaMemcpyAsync(h_out, ctx->d_stage_out.p, plan.total, cudaMemcpyDeviceToHost, ctx->stream));
    ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ZLB_OK;
}
