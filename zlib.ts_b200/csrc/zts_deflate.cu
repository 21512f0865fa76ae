// zts_deflate.cu -- chunk-parallel raw deflate: output-offset scan, bit packing, stored blocks, host
// orchestration (replaces RawDeflate.compress / dynamicHuffman / fixedHuffman / makeNocompressBlock,
// src/RawDeflate.ts:87-173,262-330, and BitStream.writeBits / finish, src/Bitstream.ts:62-130).
//
// Pipeline per wave of chunks (all on ctx->stream, no host round trip in between):
//   lz77_chunk_kernel    tokens + histograms                      (zts_lz77.cu)
//   huffman_build_kernel code tables, header bits, exact block size (zts_huffman.cu)
//   chunk_scan_kernel    exclusive scan of block sizes -> byte offset of every chunk in its item
//   bitpack_kernel       prefix sum over code lengths, bits OR-ed into a shared-memory image of the
//                        block, image copied out with aligned word stores (byte stores at the edges)
// Chunks of one item are joined by an empty stored block that byte-aligns (SURVEY App. A.7); the
// reference's RawInflate accepts this (src/RawInflate.ts:128-130,261-262,311).
#include <stdint.h>
#include <stdlib.h>
#include "zts_deflate.cuh"

size_t zts_lz77_smem_bytes();
size_t zts_lz77_scratch_bytes(int sm_count);   // per-CTA tile token scratch of the reference-compatible kernel
int zts_lz77_launch(zlb_ctx* ctx, const uint8_t* d_in, const ZtsChunk* d_chunks, uint32_t n_chunks,
                    ZtsChunkInfo* d_info, uint32_t* d_tile_tok, uint32_t* d_list, uint32_t* d_hist, uint32_t* d_sortT,
                    uint32_t* d_counter, uint32_t grid, uint32_t depth, uint32_t lazy);
int zts_huffman_launch(zlb_ctx* ctx, const ZtsChunk* d_chunks, uint32_t n_chunks, const uint32_t* d_hist,
                       ZtsChunkInfo* d_info, ZtsChunkCodes* d_codes, int block_type, int smallest);
int zts_huffman_lengths_debug(zlb_ctx* ctx, const uint32_t* d_freqs, int nsym, int limit, uint8_t* d_lengths);

#define WAVE_CHUNKS 8192u
#define PACK_THREADS 512
#define PACK_STAGE_WORDS 31744u  // 124 KiB image: 64 Ki literals * 15 bits + header + join marker

// ---- exclusive scan of chunk sizes (single CTA; a wave has <= 2048 chunks) --------------------------
__global__ void __launch_bounds__(1024)
chunk_scan_kernel(const ZtsChunk* __restrict__ chunks, ZtsChunkInfo* __restrict__ info, uint32_t n_chunks,
                  const zlb_item* __restrict__ items, unsigned long long* __restrict__ item_running,
                  unsigned long long* __restrict__ gpos)
{
    __shared__ uint32_t warp_tot[32];
    __shared__ uint32_t tile_total;
    const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    unsigned long long carry = 0;
    for (uint32_t base = 0; base < n_chunks; base += 1024) {
        const uint32_t c = base + tid;
        const uint32_t v = c < n_chunks ? info[c].out_bytes : 0u;
        uint32_t inc = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, d);
            if (lane >= (unsigned)d) inc += t;
        }
        if (lane == 31) warp_tot[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            uint32_t w = warp_tot[lane], winc = w;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                uint32_t t = __shfl_up_sync(0xFFFFFFFFu, winc, d);
                if (lane >= (unsigned)d) winc += t;
            }
            warp_tot[lane] = winc - w;
            if (lane == 31) tile_total = winc;
        }
        __syncthreads();
        if (c < n_chunks) gpos[c] = carry + warp_tot[warp] + inc - v;
        carry += tile_total;
        __syncthreads();
    }
    __threadfence_block();
    __syncthreads();
    // offset inside the item = running total of earlier waves + distance from the item's first chunk
    for (uint32_t c = tid; c < n_chunks; c += 1024) {
        const ZtsChunk ch = chunks[c];
        const unsigned long long rel = item_running[ch.item] + (gpos[c] - gpos[ch.seg_first]);
        info[c].out_off = items[ch.item].out_off + rel;
    }
    __syncthreads();
    for (uint32_t c = tid; c < n_chunks; c += 1024) {
        const ZtsChunk ch = chunks[c];
        const bool last_in_wave = (c + 1 == n_chunks) || (chunks[c + 1].item != ch.item);
        if (last_in_wave)
            item_running[ch.item] = (info[c].out_off - items[ch.item].out_off) + info[c].out_bytes;
    }
}

__global__ void deflate_finalize_kernel(const zlb_item* __restrict__ items, zlb_result* __restrict__ results,
                                        const unsigned long long* __restrict__ item_running,
                                        const uint32_t* __restrict__ item_blocks, uint32_t n_items)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_items) return;
    const unsigned long long total = item_running[i];
    results[i].out_len = total;
    results[i].blocks = item_blocks[i];
    results[i].in_used = items[i].in_len;
    results[i].status = total > items[i].out_cap ? ZLB_ST_OUT_OVERFLOW : ZLB_ST_OK;
}

__global__ void running_snapshot_kernel(unsigned long long* __restrict__ h_dst, const unsigned long long* __restrict__ src, uint32_t n)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) h_dst[i] = src[i];  // h_dst is page-locked host memory (cudaMallocHost: device-accessible)
}

// ---- bit packer: one CTA per chunk ------------------------------------------------------------------------
// The chunk's tokens are one contiguous list (both LZ77 kernels write it). Every warp owns a contiguous range of
// it. Pass 1 adds up the bits of each range, a 16-entry scan gives every range its first bit, pass 2 re-derives the
// codes and ORs them into a shared-memory image of the block with warp-level prefix sums only (no block barrier per
// batch of tokens). Launched twice per wave with two image sizes: a CTA whose block fits the small image runs in the
// small launch (4 CTAs per SM), the others in the large one; the CTA of the other class exits at once.
#define PACK_WARPS (PACK_THREADS / 32)
#define PACK_SMALL_WORDS 13312u  // 52 KiB image: 4 CTAs per SM

struct PackTok {
    unsigned long long bits;
    uint32_t nb;
};

// Token g of the chunk (g == n_tok is the end-of-block symbol, g >= g_end nothing). Loads are issued two batches
// ahead of their use (the loop bodies are short next to a trip to L2 / DRAM).
#define PACK_TOK_EOB 0x7F000000u   // bits 24..30 are zero in every real token
#define PACK_TOK_NONE 0x7E000000u
__device__ __forceinline__ uint32_t fetch_token(uint32_t g, uint32_t g_end, uint32_t n_tok, const uint32_t* __restrict__ list)
{
    if (g >= g_end) return PACK_TOK_NONE;
    if (g >= n_tok) return PACK_TOK_EOB;
    return __ldg(list + g);
}

// code bits of a token
__device__ __forceinline__ PackTok encode_token(uint32_t tok, const uint32_t* s_ll, const uint32_t* s_d)
{
    PackTok r = {0ull, 0u};
    if (tok & TOK_MATCH) {
        uint32_t ls, lb, lv, ds, db, dv;
        zts_len_code(((tok >> 16) & 0xFF) + 3, ls, lb, lv);
        zts_dist_code((tok & 0xFFFF) + 1, ds, db, dv);
        const uint32_t le = s_ll[257 + ls], de = s_d[ds];
        // litlen code, length extra, distance code, distance extra (src/RawDeflate.ts:279-289)
        r.bits = le & 0xFFFF;
        r.nb = le >> 16;
        r.bits |= (unsigned long long)lv << r.nb;
        r.nb += lb;
        r.bits |= (unsigned long long)(de & 0xFFFF) << r.nb;
        r.nb += de >> 16;
        r.bits |= (unsigned long long)dv << r.nb;
        r.nb += db;
    } else if (tok != PACK_TOK_NONE) {
        const uint32_t le = s_ll[tok == PACK_TOK_EOB ? 256u : (tok & 0xFFu)];
        r.bits = le & 0xFFFF;
        r.nb = le >> 16;
    }
    return r;
}

__global__ void __launch_bounds__(PACK_THREADS)
bitpack_kernel(const ZtsChunk* __restrict__ chunks, const ZtsChunkInfo* __restrict__ info,
               const ZtsChunkCodes* __restrict__ codes, const uint32_t* __restrict__ tok_list,
               const zlb_item* __restrict__ items, uint8_t* __restrict__ out,
               uint32_t stage_words, uint32_t min_words, const uint8_t* __restrict__ in)
{
    extern __shared__ __align__(16) uint32_t stage[];  // stage_words
    __shared__ uint32_t s_ll[286];
    __shared__ uint32_t s_d[30];
    __shared__ unsigned long long range_bits[PACK_WARPS];

    const uint32_t c = blockIdx.x;
    const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const ZtsChunk ch = chunks[c];
    const ZtsChunkInfo* ci = info + c;
    const zlb_item it = items[ch.item];
    const uint32_t out_bytes = ci->out_bytes;
    const unsigned long long rel = ci->out_off - it.out_off;
    if (rel + out_bytes > it.out_cap) return;  // item overflows its slot: status is set by the finalize kernel
    uint8_t* dst = out + ci->out_off;
    const uint32_t shift = (uint32_t)((uintptr_t)dst & 15u);  // image byte j <-> byte j of the 16-byte aligned block dst sits in
    const uint32_t n_words = ((shift + out_bytes + 15) >> 4) << 2;  // whole 16-byte groups: the image leaves in 128-bit stores
    if (n_words > stage_words || n_words <= min_words) return;  // the other launch's size class

    if (ci->hdr_bits == ZTS_HDR_STORED) {
        // ZLB_MODE_SMALLEST chose stored blocks for this chunk (makeNocompressBlock, src/RawDeflate.ts:122-153):
        // pieces of at most 65535 bytes, each header byte | LEN | NLEN | bytes; the chunk starts byte-aligned
        const uint8_t* src = in + ch.in_off;
        uint32_t o = 0;
        for (uint32_t pos = 0; pos < ch.len;) {
            const uint32_t len = min(0xFFFFu, ch.len - pos);
            if (tid == 0) {
                dst[o] = ((ch.flags & CHUNK_LAST) && pos + len == ch.len) ? 1 : 0;  // bfinal | btype(0) << 1
                dst[o + 1] = len & 0xFF;
                dst[o + 2] = len >> 8;
                dst[o + 3] = (len ^ 0xFFFFu) & 0xFF;
                dst[o + 4] = (len ^ 0xFFFFu) >> 8;
            }
            zts_block_copy(dst + o + 5, src + pos, len, tid, PACK_THREADS);
            o += 5 + len;
            pos += len;
        }
        if (tid == 0 && !(ch.flags & CHUNK_LAST)) {  // join marker behind a byte-aligned block: 00 | 00 00 FF FF
            dst[o] = dst[o + 1] = dst[o + 2] = 0;
            dst[o + 3] = dst[o + 4] = 0xFF;
        }
        return;
    }

    for (uint32_t i = tid; i < n_words; i += PACK_THREADS) stage[i] = 0;
    for (uint32_t i = tid; i < 286; i += PACK_THREADS) s_ll[i] = codes[c].ll[i];
    if (tid < 30) s_d[tid] = codes[c].d[tid];
    const uint32_t n_tok = ci->n_tokens;
    __syncthreads();
    // header bits
    const uint32_t hdr_bits = ci->hdr_bits;
    const uint32_t base_bit = shift * 8;
    for (uint32_t i = tid; i < (hdr_bits + 7) / 8; i += PACK_THREADS) {
        const uint32_t b = codes[c].hdr[i];
        const uint32_t bit = base_bit + i * 8;
        ZTS_ASSERT((bit >> 5) < stage_words);
        if (b) atomicOr(&stage[bit >> 5], b << (bit & 31));  // byte-aligned inside a word: never straddles
    }
    const uint32_t* list = tok_list + (size_t)c * LZ_LIST_PER_CHUNK;

    // tokens 0 .. n_tok-1, then the end-of-block symbol: warp w owns [w * per, (w + 1) * per)
    const uint32_t per = (((n_tok + 1 + PACK_WARPS - 1) / PACK_WARPS) + 31u) & ~31u;
    const uint32_t g_begin = warp * per, g_end = min(n_tok + 1, g_begin + per);
    {
        unsigned long long tot = 0;
        uint32_t t0 = fetch_token(g_begin + lane, g_end, n_tok, list);
        uint32_t t1 = fetch_token(g_begin + 32 + lane, g_end, n_tok, list);
        for (uint32_t g0 = g_begin; g0 < g_end; g0 += 32) {
            const uint32_t t2 = fetch_token(g0 + 64 + lane, g_end, n_tok, list);
            tot += encode_token(t0, s_ll, s_d).nb;
            t0 = t1;
            t1 = t2;
        }
#pragma unroll
        for (int d = 16; d; d >>= 1) tot += __shfl_xor_sync(0xFFFFFFFFu, tot, d);
        if (lane == 0) range_bits[warp] = tot;
    }
    __syncthreads();
    unsigned long long bitpos = (unsigned long long)base_bit + hdr_bits;
    for (uint32_t w = 0; w < warp; ++w) bitpos += range_bits[w];
    {
        uint32_t t0 = fetch_token(g_begin + lane, g_end, n_tok, list);
        uint32_t t1 = fetch_token(g_begin + 32 + lane, g_end, n_tok, list);
        for (uint32_t g0 = g_begin; g0 < g_end; g0 += 32) {
            const uint32_t t2 = fetch_token(g0 + 64 + lane, g_end, n_tok, list);
            const PackTok t = encode_token(t0, s_ll, s_d);
            t0 = t1;
            t1 = t2;
            uint32_t inc = t.nb;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                uint32_t u = __shfl_up_sync(0xFFFFFFFFu, inc, d);
                if (lane >= (unsigned)d) inc += u;
            }
            if (t.nb) {
                const unsigned long long bp = bitpos + inc - t.nb;
                const uint32_t w0 = (uint32_t)(bp >> 5), sh = (uint32_t)(bp & 31);
                // up to 48 + 31 bits -> three words
                const unsigned long long lo64 = t.bits << sh;
                ZTS_ASSERT(w0 + 2u < stage_words + 2u && w0 < stage_words);
                atomicOr(&stage[w0], (uint32_t)lo64);
                const uint32_t mid = (uint32_t)(lo64 >> 32);
                if (mid) atomicOr(&stage[w0 + 1], mid);
                if (sh && t.nb + sh > 64) {
                    const uint32_t hi32 = (uint32_t)(t.bits >> (64 - sh));
                    if (hi32) atomicOr(&stage[w0 + 2], hi32);
                }
            }
            bitpos += __shfl_sync(0xFFFFFFFFu, inc, 31);
        }
    }
    // join marker: (byte align incl. the 3 header bits of an empty stored block) 00 00 FF FF
    if (tid == 0 && !(ch.flags & CHUNK_LAST)) {
        const uint32_t b0 = shift + out_bytes - 2;  // the two 0xFF bytes are the last two of the chunk
        atomicOr(&stage[b0 >> 2], 0xFFu << ((b0 & 3) * 8));
        atomicOr(&stage[(b0 + 1) >> 2], 0xFFu << (((b0 + 1) & 3) * 8));
    }
    __syncthreads();
    // copy the image out: 128-bit stores for the 16-byte groups that lie inside the chunk's bytes (coalesced, 512
    // bytes per warp instruction), own bytes only in the two edge groups
    uint4* g4 = reinterpret_cast<uint4*>(dst - shift);
    const uint4* s4 = reinterpret_cast<const uint4*>(stage);
    const uint32_t end_byte = shift + out_bytes;
    for (uint32_t j = tid; j < (n_words >> 2); j += PACK_THREADS) {
        const uint4 q = s4[j];
        const uint32_t b_lo = j * 16, b_hi = b_lo + 16;
        if (b_lo >= shift && b_hi <= end_byte) {
            g4[j] = q;
        } else {
            uint8_t* gb = reinterpret_cast<uint8_t*>(g4 + j);
            const uint32_t w[4] = {q.x, q.y, q.z, q.w};
            for (uint32_t k = 0; k < 16; ++k)
                if (b_lo + k >= shift && b_lo + k < end_byte) gb[k] = (uint8_t)(w[k >> 2] >> (8 * (k & 3)));
        }
    }
}

// ---- preset dictionaries: the window of every chunk whose history reaches into its item's dictionary ---------------
// The window of a chunk at byte `pos` of its item is the last dict_len bytes of dictionary || item[0, pos), then the
// chunk: its first dict_len - pos bytes are the dictionary's last ones. It is written to the chunk's place in the
// staging arena (16-byte aligned, like the input the LZ77 kernel otherwise stages from), which that kernel reads
// instead of the input (CHUNK_STAGED): its own chunk table names the window by an in_off taken relative to the input
// (deflate_device). Only chunks that start in the first 32 KiB of their item have such a window.
__global__ void __launch_bounds__(256)
dict_stage_kernel(const uint8_t* __restrict__ in, const uint8_t* __restrict__ dict, const zlb_dict* __restrict__ dicts,
                  const zlb_item* __restrict__ items, const ZtsChunk* __restrict__ chunks, uint8_t* __restrict__ stage)
{
    const ZtsChunk ch = chunks[blockIdx.x];
    if (!(ch.flags & CHUNK_STAGED)) return;
    const zlb_dict d = dicts[ch.item];
    const zlb_item it = items[ch.item];
    const uint32_t pos = (uint32_t)(ch.in_off - it.in_off);  // < 32768
    const uint32_t from_dict = ch.dict_len - pos;             // > 0, <= d.len
    uint8_t* dst = stage + 16ull * ch.stage_off;
    zts_block_copy(dst, dict + d.off + d.len - from_dict, from_dict, threadIdx.x, 256);
    zts_block_copy(dst + from_dict, in + it.in_off, pos + ch.len, threadIdx.x, 256);
}

// ---- stored blocks (CompressionType.NONE, src/RawDeflate.ts:93-100,122-153): 65535-byte pieces ----------
__global__ void __launch_bounds__(256)
stored_block_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, const zlb_item* __restrict__ items,
                    const uint32_t* __restrict__ blk_item, const uint32_t* __restrict__ blk_index)
{
    const uint32_t b = blockIdx.x;
    const zlb_item it = items[blk_item[b]];
    const uint64_t k = blk_index[b];
    const uint64_t n_blocks = (it.in_len + 0xFFFEull) / 0xFFFFull;
    const uint64_t o = k * (0xFFFFull + 5ull);
    const uint64_t pos = k * 0xFFFFull;
    const uint32_t len = (uint32_t)min((uint64_t)0xFFFF, it.in_len - pos);
    if (o + 5 + len > it.out_cap) return;
    const uint8_t* s = in + it.in_off + pos;
    uint8_t* d = out + it.out_off + o;
    if (threadIdx.x == 0) {
        d[0] = (k + 1 == n_blocks) ? 1 : 0;  // bfinal | btype(0) << 1
        d[1] = len & 0xFF;
        d[2] = len >> 8;
        d[3] = (len ^ 0xFFFFu) & 0xFF;
        d[4] = (len ^ 0xFFFFu) >> 8;
    }
    for (uint32_t i = threadIdx.x; i < len; i += 256) d[5 + i] = s[i];
}

extern "C" uint64_t zlb_deflate_bound(uint64_t in_len, uint32_t chunk_bytes, int block_type)
{
    if (block_type == ZLB_NONE) return in_len + 5 * ((in_len + 0xFFFE) / 0xFFFF) + 8;
    uint64_t cb = (chunk_bytes == 0 || chunk_bytes > LZ_MAX_CHUNK) ? LZ_MAX_CHUNK : chunk_bytes;
    uint64_t n_chunks = in_len ? (in_len + cb - 1) / cb : 1;
    // <= 15 bits per literal, <= 4498 header bits, end-of-block, join marker
    return (in_len * 15 + 7) / 8 + n_chunks * (ZTS_HDR_BYTES + 8) + 16;
}

static int deflate_stored(zlb_ctx* ctx, const uint8_t* d_in, uint8_t* d_out, const zlb_item* h_items,
                          zlb_result* h_results, size_t n, zlb_item* d_items)
{
    size_t n_blocks = 0;
    for (size_t i = 0; i < n; ++i) n_blocks += (h_items[i].in_len + 0xFFFE) / 0xFFFF;
    for (size_t i = 0; i < n; ++i) {
        uint64_t nb = (h_items[i].in_len + 0xFFFE) / 0xFFFF;
        uint64_t total = h_items[i].in_len + 5 * nb;
        h_results[i].status = total > h_items[i].out_cap ? ZLB_ST_OUT_OVERFLOW : ZLB_ST_OK;
        h_results[i].out_len = total;
        h_results[i].in_used = h_items[i].in_len;
        h_results[i].blocks = (uint32_t)nb;
    }
    if (n_blocks == 0) return ZLB_OK;
    if (n_blocks > 0x7FFFFFFFull) return zts_fail(ctx, ZLB_E_ARG, "too many stored blocks");
    int rc = zts_reserve_pinned(ctx, n_blocks * 8);
    if (rc) return rc;
    uint32_t* h_bi = (uint32_t*)ctx->h_pin;
    uint32_t* h_bk = h_bi + n_blocks;
    size_t k = 0;
    for (size_t i = 0; i < n; ++i) {
        uint64_t nb = (h_items[i].in_len + 0xFFFE) / 0xFFFF;
        for (uint64_t j = 0; j < nb; ++j) {
            h_bi[k] = (uint32_t)i;
            h_bk[k] = (uint32_t)j;
            ++k;
        }
    }
    rc = zts_reserve(ctx, &ctx->d_misc, n_blocks * 8 + 64);
    if (rc) return rc;
    ZTS_CUDA(ctx, cudaMemcpyAsync(ctx->d_misc.p, h_bi, n_blocks * 8, cudaMemcpyHostToDevice, ctx->stream));
    uint32_t* d_bi = (uint32_t*)ctx->d_misc.p;
    ZTS_LAUNCH(ctx, ZK_STORED,
               stored_block_kernel<<<(unsigned)n_blocks, 256, 0, ctx->stream>>>(d_in, d_out, d_items, d_bi,
                                                                                d_bi + n_blocks));
    ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ZLB_OK;
}

#define HOST_DELTA_MAX_ITEMS 256u  // per-wave output read-back is done item by item up to this many items

// Runs the pipeline on device buffers. Results land in h_results after the final synchronise.
// d_dict / h_dicts: the preset dictionaries (h_dicts == NULL: none; checked by the caller)
// hio: the host buffers of a "_host" call. The device path then also moves the data: the input of wave k+1 travels
// while wave k is compressed, and with few items what wave k produced travels while wave k+1 runs (hio->out_done).
static int deflate_device(zlb_ctx* ctx, const uint8_t* d_in, uint8_t* d_out, const uint8_t* d_dict,
                          const zlb_dict* h_dicts, const zlb_item* h_items, zlb_result* h_results, size_t n, int mode,
                          int block_type, uint32_t chunk_bytes, uint32_t flags, ZtsHostIO* hio)
{
    if ((mode & 0xFF) & ~(ZLB_MODE_FAST | ZLB_MODE_PRIMED | ZLB_MODE_SMALLEST | ZLB_MODE_LAZY))
        return zts_fail(ctx, ZLB_E_UNSUPPORTED, "unknown deflate mode %d", mode);
    uint32_t depth = 0xFFFFFFFFu;  // compat: every candidate, like the reference
    // fast mode: the same kernel, but a search looks at the `depth` nearest entries of the position's bucket only
    const bool fast = (mode & ZLB_MODE_FAST) != 0;
    const bool primed = (mode & ZLB_MODE_PRIMED) != 0 && block_type != ZLB_NONE;
    const bool smallest = (mode & ZLB_MODE_SMALLEST) != 0 && block_type == ZLB_DYNAMIC;
    if (fast) depth = ((uint32_t)mode >> 8) ? ((uint32_t)mode >> 8) : ZLB_FAST_DEFAULT_DEPTH;
    if (fast && depth > 64u) depth = 64u;  // (the lane-private search; longer lists belong to the exact mode)
    const bool lazy = fast && (mode & ZLB_MODE_LAZY) != 0;  // a fast-mode option: the exact mode is the reference's greedy parse
    if (block_type != ZLB_NONE && block_type != ZLB_FIXED && block_type != ZLB_DYNAMIC)
        return zts_fail(ctx, ZLB_E_ARG, "invalid compression type");  // src/RawDeflate.ts:110
    bool any_dict = false;  // some item has a dictionary
    for (size_t i = 0; h_dicts && i < n && !any_dict; ++i) any_dict = h_dicts[i].len != 0;
    // primed or a dictionary: history + chunk share the 64 KiB a CTA stages and indexes, so a chunk is at most 32 KiB
    const uint32_t cb_max = (primed || any_dict) ? ZLB_PRIMED_CHUNK : LZ_MAX_CHUNK;
    const uint32_t cb = (chunk_bytes == 0 || chunk_bytes > cb_max) ? cb_max : chunk_bytes;
    if (n > 0x7FFFFFFFull) return zts_fail(ctx, ZLB_E_ARG, "too many items");
    ctx->work = ctx->stream;

    int rc = zts_reserve(ctx, &ctx->d_items, n * sizeof(zlb_item) + 64);
    if (rc) return rc;
    rc = zts_reserve(ctx, &ctx->d_results, n * sizeof(zlb_result) + 64);
    if (rc) return rc;
    zlb_item* d_items = (zlb_item*)ctx->d_items.p;
    zlb_result* d_results = (zlb_result*)ctx->d_results.p;
    ZTS_CUDA(ctx, cudaMemcpyAsync(d_items, h_items, n * sizeof(zlb_item), cudaMemcpyHostToDevice, ctx->stream));
    ZTS_CUDA(ctx, cudaMemsetAsync(d_results, 0, n * sizeof(zlb_result), ctx->stream));
    memset(h_results, 0, n * sizeof(zlb_result));

    uint32_t kinds = 0;
    if (flags & ZLB_DEFLATE_WANT_CRC32) kinds |= ZLB_SUM_CRC32;
    if (flags & ZLB_DEFLATE_WANT_ADLER32) kinds |= ZLB_SUM_ADLER32;

    if (hio && block_type == ZLB_NONE) {
        zts_stage_wait_in(hio->stage, 0, hio->in_bytes);
        ZTS_CUDA(ctx, cudaMemcpyAsync((void*)d_in, hio->h_in, hio->in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    if (block_type == ZLB_NONE) {
        rc = deflate_stored(ctx, d_in, d_out, h_items, h_results, n, d_items);
        if (rc) return rc;
        if (kinds) {
            rc = zts_checksum_device(ctx, d_in, d_items, d_results, h_items, n, kinds, 0);
            if (rc) return rc;
            zlb_result* tmp = nullptr;
            rc = zts_reserve_pinned(ctx, n * sizeof(zlb_result));
            if (rc) return rc;
            tmp = (zlb_result*)ctx->h_pin;
            ZTS_CUDA(ctx, cudaMemcpyAsync(tmp, d_results, n * sizeof(zlb_result), cudaMemcpyDeviceToHost, ctx->stream));
            ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            for (size_t i = 0; i < n; ++i) {
                h_results[i].crc32 = tmp[i].crc32;
                h_results[i].adler32 = tmp[i].adler32;
            }
        }
        return ZLB_OK;
    }

    // ---- chunk table
    size_t n_chunks = 0;
    for (size_t i = 0; i < n; ++i) n_chunks += h_items[i].in_len ? (h_items[i].in_len + cb - 1) / cb : 1;
    if (n_chunks > 0x7FFFFFFFull) return zts_fail(ctx, ZLB_E_ARG, "too many chunks");
    // ---- wave plan: wstart[k] = first chunk of wave k, wstart[n_waves] = n_chunks
    std::vector<size_t> wstart;
    {
        const size_t sm = (size_t)ctx->sm_count;
        if (hio && n_chunks >= 16u * sm) {
            // host path, large job: the first wave's input and the last wave's small kernels + output are the
            // transfers nothing hides, so the waves ramp up (one, then two chunks per SM), cruise in about four
            // large waves (every wave costs ~0.15 ms of launches and tails) and end with a small one; consecutive
            // waves overlap on two streams, so even a small wave keeps every SM busy
            wstart.push_back(0);
            wstart.push_back(sm);
            wstart.push_back(3u * sm);
            const size_t rest = n_chunks - 5u * sm;  // minus the ramp (3 sm) and the last wave (2 sm)
            size_t cruise = (rest + 3) / 4;
            if (cruise > WAVE_CHUNKS) cruise = WAVE_CHUNKS;
            for (size_t at = 3u * sm; at + cruise < n_chunks - 2u * sm; at += cruise) wstart.push_back(at + cruise);
            if (wstart.back() < n_chunks - 2u * sm) wstart.push_back(n_chunks - 2u * sm);
            wstart.push_back(n_chunks);
        } else {
            size_t wave = n_chunks < WAVE_CHUNKS ? n_chunks : WAVE_CHUNKS;
            if (hio && n_chunks > 4u * sm) {  // host path, medium job: about eight equal waves of at least two chunks per SM
                size_t w8 = (n_chunks + 7) / 8;
                if (w8 < 2u * sm) w8 = 2u * sm;
                if (w8 < wave) wave = w8;
            }
            for (size_t at = 0; at < n_chunks; at += wave) wstart.push_back(at);
            wstart.push_back(n_chunks);
        }
    }
    const size_t n_waves = wstart.size() - 1;
    size_t wave = 0;  // the largest wave sizes the scratch sets
    for (size_t k = 0; k < n_waves; ++k)
        if (wstart[k + 1] - wstart[k] > wave) wave = wstart[k + 1] - wstart[k];
    // table upload: chunks | with dictionaries: the LZ77 kernel's view of the chunks and the dictionary table |
    // blocks per item
    const size_t view_b = any_dict ? n_chunks * sizeof(ZtsChunk) : 0;
    const size_t dicts_b = any_dict ? n * sizeof(zlb_dict) : 0;
    const size_t tables_b = n_chunks * sizeof(ZtsChunk) + view_b + dicts_b + n * sizeof(uint32_t);
    rc = zts_reserve_pinned(ctx, tables_b);
    if (rc) return rc;
    ZtsChunk* h_chunks = (ZtsChunk*)ctx->h_pin;
    ZtsChunk* h_view = h_chunks + n_chunks;
    if (any_dict) memcpy((uint8_t*)h_view + view_b, h_dicts, dicts_b);
    uint32_t* h_blocks = (uint32_t*)((uint8_t*)h_view + view_b + dicts_b);
    size_t stage_b = 0;  // staging arena of the largest wave (dictionaries)
    {
        size_t k = 0, wk = 0, stage_at = 0;  // stage_at: 16-byte units used by the chunk's wave so far
        for (size_t i = 0; i < n; ++i) {
            const uint64_t len = h_items[i].in_len;
            const uint64_t nc = len ? (len + cb - 1) / cb : 1;
            // dictionary bytes a chunk can reach (an empty item has nothing to search for)
            const uint32_t dl = (any_dict && len) ? (uint32_t)(h_dicts[i].len < LZ_WINDOW ? h_dicts[i].len : LZ_WINDOW) : 0u;
            h_blocks[i] = (uint32_t)nc;
            for (uint64_t j = 0; j < nc; ++j, ++k) {
                ZtsChunk& c = h_chunks[k];
                c.in_off = h_items[i].in_off + j * cb;
                c.len = (uint32_t)(len - j * cb < cb ? len - j * cb : cb);
                c.item = (uint32_t)i;
                c.flags = (j + 1 == nc && !(flags & ZLB_DEFLATE_NOT_FINAL)) ? CHUNK_LAST : 0u;
                c.dict_len = primed ? (uint32_t)(j * cb < LZ_WINDOW ? j * cb : LZ_WINDOW) : 0u;
                c.stage_off = 0;
                if (k >= wstart[wk + 1]) stage_at = 0;  // a new wave (the loop below moves wk on)
                // history from the dictionary: an item's first chunk, and in primed mode every chunk in its first 32 KiB
                if (dl && (primed || j == 0) && j * cb < LZ_WINDOW) {
                    const uint32_t pos = (uint32_t)(j * cb);
                    c.dict_len = dl + pos < LZ_WINDOW ? dl + pos : LZ_WINDOW;
                    c.flags |= CHUNK_STAGED;
                    c.stage_off = (uint32_t)stage_at;
                    stage_at += (c.dict_len + c.len + 15u) / 16u;
                    if (16 * stage_at > stage_b) stage_b = 16 * stage_at;
                }
                // first chunk of this item inside the chunk's wave
                while (k >= wstart[wk + 1]) ++wk;
                const size_t wave_base = wstart[wk];
                const size_t item_first = k - j;
                c.seg_first = (uint32_t)((item_first > wave_base ? item_first : wave_base) - wave_base);
            }
        }
    }
    const uint32_t grid = (uint32_t)(wave < (size_t)ctx->sm_count ? wave : (size_t)ctx->sm_count);
    // Host path with several waves: consecutive waves run on two streams with a scratch set each, so that the next
    // wave's LZ77 CTAs take over the SMs as the previous wave's drain (no idle tail per wave) and its small kernels
    // overlap too; only the offset scan is chained from wave to wave.
    const int n_sets = (hio && n_waves > 1) ? 2 : 1;
    rc = zts_reserve(ctx, &ctx->d_chunks, tables_b + 64);
    if (rc) return rc;
    stage_b = (stage_b + 255) & ~(size_t)255;
    if (stage_b && (rc = zts_reserve(ctx, &ctx->d_dict_stage, n_sets * stage_b + 64))) return rc;
    if (any_dict) {
        // The LZ77 kernel stages `in + in_off - dict_len` (the history in front of the chunk, then the chunk). Its view
        // of a staged chunk names the chunk's place in the staging arena of the chunk's wave that way, so that the
        // kernel itself reads windows from the arena unchanged; the other kernels keep the chunk's place in the input.
        for (size_t k = 0, wk = 0; k < n_chunks; ++k) {
            while (k >= wstart[wk + 1]) ++wk;
            h_view[k] = h_chunks[k];
            if (h_chunks[k].flags & CHUNK_STAGED) {
                const uint64_t arena = (uint64_t)(uintptr_t)ctx->d_dict_stage.p + (n_sets == 2 ? (wk & 1) : 0) * stage_b;
                h_view[k].in_off = arena + 16ull * h_chunks[k].stage_off + h_chunks[k].dict_len - (uint64_t)(uintptr_t)d_in;
            }
        }
    }
    const size_t info_b = (wave * sizeof(ZtsChunkInfo) + 255) & ~(size_t)255;
    const size_t list_b = (wave * (size_t)LZ_LIST_PER_CHUNK * 4 + 255) & ~(size_t)255;   // token list of every chunk
    const size_t tile_b = (zts_lz77_scratch_bytes(ctx->sm_count) + 255) & ~(size_t)255;  // per-CTA tile token scratch
    const size_t hist_b = (wave * 316 * 4 + 255) & ~(size_t)255;
    const size_t codes_b = (wave * sizeof(ZtsChunkCodes) + 255) & ~(size_t)255;
    const size_t sort_b = ((size_t)ctx->sm_count * LZ_MAX_CHUNK * 4 + 255) & ~(size_t)255;
    const size_t gpos_b = (wave * 8 + 256 + 255) & ~(size_t)255;  // chunk offsets of the wave + the work counter
    rc = zts_reserve(ctx, &ctx->d_chunk_info, n_sets * info_b + 64);
    if (rc) return rc;
    rc = zts_reserve(ctx, &ctx->d_tokens, n_sets * list_b + 64);
    if (rc) return rc;
    if ((rc = zts_reserve(ctx, &ctx->d_spec, n_sets * tile_b + 64))) return rc;
    rc = zts_reserve(ctx, &ctx->d_hist, n_sets * hist_b + 64);
    if (rc) return rc;
    rc = zts_reserve(ctx, &ctx->d_codes, n_sets * codes_b + 64);
    if (rc) return rc;
    rc = zts_reserve(ctx, &ctx->d_sortT, n_sets * sort_b + 64);
    if (rc) return rc;
    rc = zts_reserve(ctx, &ctx->d_misc, n * 8 + n_sets * gpos_b + 256);
    if (rc) return rc;
    ZtsChunk* d_chunks = (ZtsChunk*)ctx->d_chunks.p;
    const ZtsChunk* d_lz_chunks = any_dict ? d_chunks + n_chunks : d_chunks;  // what the LZ77 kernel reads
    const zlb_dict* d_dicts = (const zlb_dict*)((uint8_t*)(d_chunks + n_chunks) + view_b);
    uint32_t* d_blocks = (uint32_t*)((uint8_t*)d_dicts + dicts_b);
    unsigned long long* d_running = (unsigned long long*)ctx->d_misc.p;
    struct Set {
        ZtsChunkInfo* info;
        uint32_t *list, *tile_tok, *hist, *sortT, *counter;
        ZtsChunkCodes* codes;
        unsigned long long* gpos;
        uint8_t* stage;
    } sets[2];
    for (int b = 0; b < n_sets; ++b) {
        sets[b].info = (ZtsChunkInfo*)((uint8_t*)ctx->d_chunk_info.p + b * info_b);
        sets[b].list = (uint32_t*)((uint8_t*)ctx->d_tokens.p + b * list_b);
        sets[b].tile_tok = (uint32_t*)((uint8_t*)ctx->d_spec.p + b * tile_b);
        sets[b].hist = (uint32_t*)((uint8_t*)ctx->d_hist.p + b * hist_b);
        sets[b].codes = (ZtsChunkCodes*)((uint8_t*)ctx->d_codes.p + b * codes_b);
        sets[b].sortT = (uint32_t*)((uint8_t*)ctx->d_sortT.p + b * sort_b);
        sets[b].gpos = (unsigned long long*)((uint8_t*)(d_running + n) + b * gpos_b);
        sets[b].counter = (uint32_t*)(sets[b].gpos + wave);
        sets[b].stage = stage_b ? (uint8_t*)ctx->d_dict_stage.p + b * stage_b : nullptr;
    }
    ZTS_CUDA(ctx, cudaMemcpyAsync(d_chunks, h_chunks, tables_b, cudaMemcpyHostToDevice, ctx->stream));
    ZTS_CUDA(ctx, cudaMemsetAsync(d_running, 0, n * 8, ctx->stream));
    ZTS_CUDA(ctx, cudaFuncSetAttribute(bitpack_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)(PACK_STAGE_WORDS * 4)));

    // ---- host path: copy plan
    bool pipe_in = false, delta_out = false;
    unsigned long long* h_run = nullptr;      // [n_waves][n] running totals read back after each wave
    std::vector<unsigned long long> copied;   // bytes of every item already copied to the host
    if (hio) {
        rc = zts_host_streams(ctx);
        if (rc) return rc;
        pipe_in = n_waves > 1;
        for (size_t k = 1; k < n_chunks && pipe_in; ++k)
            if (h_chunks[k].in_off < h_chunks[k - 1].in_off + h_chunks[k - 1].len) pipe_in = false;  // not laid out in order
        delta_out = n <= HOST_DELTA_MAX_ITEMS;
        if (delta_out) {
            rc = zts_reserve_pinned2(ctx, n_waves * n * sizeof(unsigned long long));
            if (rc) return rc;
            h_run = (unsigned long long*)ctx->h_pin2;
            copied.assign(n, 0ull);
        }
        if (!pipe_in) {
            zts_stage_wait_in(hio->stage, 0, hio->in_bytes);
            ZTS_CUDA(ctx, cudaMemcpyAsync((void*)d_in, hio->h_in, hio->in_bytes, cudaMemcpyHostToDevice, ctx->stream));
        }
    }
    // Everything the second stream reads must be on the device before it starts: the tables uploaded above and, when
    // the input is not pipelined wave by wave (items not laid out in ascending order), the whole-input copy just
    // queued on ctx->stream. The event is recorded behind both.
    if (n_sets == 2) ZTS_CUDA(ctx, cudaEventRecord(zts_sync_event(ctx, 4 * n_waves), ctx->stream));
    auto wave_in_copy = [&](size_t k) -> int {  // input bytes of wave k: one contiguous hull (chunks are in order)
        const size_t a = wstart[k], b = wstart[k + 1] - 1;
        const uint64_t lo = h_chunks[a].in_off, hi = h_chunks[b].in_off + h_chunks[b].len;
        if (hi > lo) {
            zts_stage_wait_in(hio->stage, lo, hi);  // pageable caller buffer: its copy threads have filled the shadow up to here
            ZTS_CUDA(ctx, cudaMemcpyAsync((void*)(d_in + lo), hio->h_in + lo, hi - lo, cudaMemcpyHostToDevice, ctx->s_in));
        }
        ZTS_CUDA(ctx, cudaEventRecord(zts_sync_event(ctx, 2 * k), ctx->s_in));
        return ZLB_OK;
    };
    auto wave_out_copy = [&](size_t k) -> int {  // what wave k appended to the items it touched
        ZTS_CUDA(ctx, cudaEventSynchronize(zts_sync_event(ctx, 2 * k + 1)));
        const size_t a = wstart[k], b = wstart[k + 1] - 1;
        for (uint32_t i = h_chunks[a].item; i <= h_chunks[b].item; ++i) {
            unsigned long long now = h_run[k * n + i];
            if (now > h_items[i].out_cap) now = copied[i];  // overflowed item: nothing more was written
            if (now > copied[i]) {
                const uint64_t off = h_items[i].out_off + copied[i];
                ZTS_CUDA(ctx, cudaMemcpyAsync(hio->h_out + off, d_out + off, now - copied[i], cudaMemcpyDeviceToHost,
                                              ctx->s_out));
                int rc2 = zts_stage_out_ready(ctx, hio->stage, ctx->s_out, off, now - copied[i]);
                if (rc2) return rc2;
                copied[i] = now;
            }
        }
        return ZLB_OK;
    };
    if (pipe_in && (rc = wave_in_copy(0))) return rc;

    // events: 2k = input of wave k arrived, 2k+1 = wave k done; 2 n_waves + k = offset scan of wave k done
    for (size_t k = 0; k < n_waves; ++k) {
        const size_t w0 = wstart[k];
        const uint32_t wn = (uint32_t)(wstart[k + 1] - w0);
        const uint32_t g = wn < grid ? wn : grid;
        const Set& S = sets[n_sets == 2 ? (k & 1) : 0];
        cudaStream_t st = (n_sets == 2 && (k & 1)) ? ctx->s_aux[0] : ctx->stream;
        ctx->work = st;
        if (n_sets == 2 && k == 1)  // the tables uploaded on ctx->stream must be there before the second stream starts
            ZTS_CUDA(ctx, cudaStreamWaitEvent(st, zts_sync_event(ctx, 4 * n_waves), 0));
        if (pipe_in) ZTS_CUDA(ctx, cudaStreamWaitEvent(st, zts_sync_event(ctx, 2 * k), 0));
        if (stage_b)
            ZTS_LAUNCH(ctx, ZK_DICT_STAGE,
                       dict_stage_kernel<<<wn, 256, 0, st>>>(d_in, d_dict, d_dicts, d_items, d_chunks + w0, S.stage));
        rc = zts_lz77_launch(ctx, d_in, d_lz_chunks + w0, wn, S.info, S.tile_tok, S.list, S.hist, S.sortT, S.counter, g, depth,
                             lazy ? 1u : 0u);
        if (rc) return rc;
        rc = zts_huffman_launch(ctx, d_chunks + w0, wn, S.hist, S.info, S.codes, block_type, smallest ? 1 : 0);
        if (rc) return rc;
        if (n_sets == 2 && k > 0)  // item_running is handed from wave to wave
            ZTS_CUDA(ctx, cudaStreamWaitEvent(st, zts_sync_event(ctx, 2 * n_waves + k - 1), 0));
        ZTS_LAUNCH(ctx, ZK_SCAN,
                   chunk_scan_kernel<<<1, 1024, 0, st>>>(d_chunks + w0, S.info, wn, d_items, d_running, S.gpos));
        if (delta_out) {
            // snapshot of the running totals before the next wave's scan moves them on: written straight into the
            // page-locked table by a kernel. (A device-to-host copy queued here, behind kernels that are still
            // running, would hold up the output copy of the wave before -- the copy engine serves its queue in order.)
            running_snapshot_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(h_run + k * n, d_running, (uint32_t)n);
            ZTS_CUDA(ctx, cudaGetLastError());
        }
        if (n_sets == 2) ZTS_CUDA(ctx, cudaEventRecord(zts_sync_event(ctx, 2 * n_waves + k), st));
        ZTS_LAUNCH(ctx, ZK_BITPACK,
                   bitpack_kernel<<<wn, PACK_THREADS, PACK_SMALL_WORDS * 4, st>>>(
                       d_chunks + w0, S.info, S.codes, S.list, d_items, d_out, PACK_SMALL_WORDS, 0u, d_in));
        ZTS_LAUNCH(ctx, ZK_BITPACK,
                   bitpack_kernel<<<wn, PACK_THREADS, PACK_STAGE_WORDS * 4, st>>>(
                       d_chunks + w0, S.info, S.codes, S.list, d_items, d_out, PACK_STAGE_WORDS, PACK_SMALL_WORDS,
                       d_in));
        // wave k is queued: the input of wave k+1 follows (with a pageable caller buffer this waits for the copy
        // threads, so it comes behind the launches), then the output of wave k-1
        if (pipe_in && k + 1 < n_waves && (rc = wave_in_copy(k + 1))) return rc;
        if (delta_out) {
            ZTS_CUDA(ctx, cudaEventRecord(zts_sync_event(ctx, 2 * k + 1), st));
            if (k > 0 && (rc = wave_out_copy(k - 1))) return rc;
        }
    }
    ctx->work = ctx->stream;
    if (n_sets == 2) {  // everything that follows on ctx->stream comes after the second stream's last wave
        ZTS_CUDA(ctx, cudaEventRecord(zts_sync_event(ctx, 4 * n_waves + 1), ctx->s_aux[0]));
        ZTS_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, zts_sync_event(ctx, 4 * n_waves + 1), 0));
    }
    if (delta_out) {
        if ((rc = wave_out_copy(n_waves - 1))) return rc;
        hio->out_done = true;
    }
    ZTS_LAUNCH(ctx, ZK_FINALIZE,
               deflate_finalize_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(d_items, d_results,
                                                                                             d_running, d_blocks,
                                                                                             (uint32_t)n));
    if (kinds) {
        rc = zts_checksum_device(ctx, d_in, d_items, d_results, h_items, n, kinds, 0);
        if (rc) return rc;
    }
    ZTS_CUDA(ctx, cudaMemcpyAsync(h_results, d_results, n * sizeof(zlb_result), cudaMemcpyDeviceToHost, ctx->stream));
    ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (delta_out) ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->s_out));
    return ZLB_OK;
}

extern "C" int zlb_deflate_batch_dict(zlb_ctx* ctx, const void* d_in, void* d_out, const void* d_dict,
                                      const zlb_dict* dicts, const zlb_item* items, zlb_result* results, size_t n,
                                      int mode, int block_type, uint32_t chunk_bytes, uint32_t flags)
{
    bool any = false;
    int rc = zts_entry_begin(ctx, d_out || !n, items, results, n, SIZE_MAX, d_dict, SIZE_MAX, dicts, &any);
    if (rc) return rc > 0 ? ZLB_OK : rc;
    return deflate_device(ctx, (const uint8_t*)d_in, (uint8_t*)d_out, (const uint8_t*)d_dict, any ? dicts : nullptr,
                          items, results, n, mode, block_type, chunk_bytes, flags, nullptr);
}

extern "C" int zlb_deflate_batch(zlb_ctx* ctx, const void* d_in, void* d_out, const zlb_item* items,
                                 zlb_result* results, size_t n, int mode, int block_type, uint32_t chunk_bytes,
                                 uint32_t flags)
{
    return zlb_deflate_batch_dict(ctx, d_in, d_out, nullptr, nullptr, items, results, n, mode, block_type, chunk_bytes,
                                  flags);
}

extern "C" int zlb_deflate_batch_dict_host(zlb_ctx* ctx, const void* h_in, size_t in_bytes, void* h_out,
                                           size_t out_bytes, const void* h_dict, size_t dict_bytes,
                                           const zlb_dict* dicts, const zlb_item* items, zlb_result* results, size_t n,
                                           int mode, int block_type, uint32_t chunk_bytes, uint32_t flags)
{
    return zts_host_call(ctx, h_in, in_bytes, h_out, out_bytes, h_dict, dict_bytes, dicts, items, results, n, SIZE_MAX,
                         [&](ZtsHostIO& io, const zlb_dict* d) {
        const uint8_t* d_out = (const uint8_t*)ctx->d_stage_out.p;
        int rc = deflate_device(ctx, (const uint8_t*)ctx->d_stage_in.p, (uint8_t*)d_out, (const uint8_t*)ctx->d_dict.p, d,
                                items, results, n, mode, block_type, chunk_bytes, flags, &io);
        if (rc || io.out_done) return rc;
        // many items: what each of them wrote, adjacent ranges merged
        return zts_copy_back(ctx, io.stage, ctx->stream, d_out, io.h_out, items, results, (const zlb_item*)ctx->d_items.p,
                             (const zlb_result*)ctx->d_results.p, 0, n);
    });
}

extern "C" int zlb_deflate_batch_host(zlb_ctx* ctx, const void* h_in, size_t in_bytes, void* h_out, size_t out_bytes,
                                      const zlb_item* items, zlb_result* results, size_t n, int mode, int block_type,
                                      uint32_t chunk_bytes, uint32_t flags)
{
    return zlb_deflate_batch_dict_host(ctx, h_in, in_bytes, h_out, out_bytes, nullptr, 0, nullptr, items, results, n, mode,
                                       block_type, chunk_bytes, flags);
}

// ---- test hooks ---------------------------------------------------------------------------------------
extern "C" int zlb_debug_lz77(zlb_ctx* ctx, const void* d_in, uint32_t n, uint32_t* h_tokens_out, uint32_t* n_tokens,
                              uint32_t* h_hist_out)
{
    if (!ctx || !h_tokens_out || !n_tokens || !h_hist_out || n > LZ_MAX_CHUNK) return ZLB_E_ARG;
    ZTS_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc;
    if ((rc = zts_reserve(ctx, &ctx->d_chunks, sizeof(ZtsChunk) + 64))) return rc;
    if ((rc = zts_reserve(ctx, &ctx->d_chunk_info, sizeof(ZtsChunkInfo) + 64))) return rc;
    if ((rc = zts_reserve(ctx, &ctx->d_tokens, (size_t)LZ_LIST_PER_CHUNK * 4 + 64))) return rc;
    if ((rc = zts_reserve(ctx, &ctx->d_spec, zts_lz77_scratch_bytes(ctx->sm_count) + 64))) return rc;
    if ((rc = zts_reserve(ctx, &ctx->d_hist, 316 * 4 + 64))) return rc;
    if ((rc = zts_reserve(ctx, &ctx->d_sortT, (size_t)ctx->sm_count * LZ_MAX_CHUNK * 4 + 64))) return rc;
    if ((rc = zts_reserve(ctx, &ctx->d_misc, 256))) return rc;
    ZtsChunk ch = {0, n, 0, 0, CHUNK_LAST, 0, 0};  // no history
    ZTS_CUDA(ctx, cudaMemcpyAsync(ctx->d_chunks.p, &ch, sizeof ch, cudaMemcpyHostToDevice, ctx->stream));
    ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    rc = zts_lz77_launch(ctx, (const uint8_t*)d_in, (const ZtsChunk*)ctx->d_chunks.p, 1, (ZtsChunkInfo*)ctx->d_chunk_info.p,
                         (uint32_t*)ctx->d_spec.p, (uint32_t*)ctx->d_tokens.p, (uint32_t*)ctx->d_hist.p,
                         (uint32_t*)ctx->d_sortT.p, (uint32_t*)ctx->d_misc.p, 1, 0xFFFFFFFFu, 0u);
    if (rc) return rc;
    ZtsChunkInfo ci;
    ZTS_CUDA(ctx, cudaMemcpyAsync(&ci, ctx->d_chunk_info.p, sizeof ci, cudaMemcpyDeviceToHost, ctx->stream));
    ZTS_CUDA(ctx, cudaMemcpyAsync(h_hist_out, ctx->d_hist.p, 316 * 4, cudaMemcpyDeviceToHost, ctx->stream));
    ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (ci.n_tokens > n) return zts_fail(ctx, ZLB_E_CUDA, "token count %u for %u bytes", ci.n_tokens, n);
    ZTS_CUDA(ctx, cudaMemcpyAsync(h_tokens_out, ctx->d_tokens.p, (size_t)ci.n_tokens * 4, cudaMemcpyDeviceToHost, ctx->stream));
    ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *n_tokens = ci.n_tokens;
    return ZLB_OK;
}

extern "C" int zlb_debug_code_lengths(zlb_ctx* ctx, const uint32_t* h_freqs, int nsym, int limit, uint8_t* h_lengths)
{
    if (!ctx || !h_freqs || !h_lengths || nsym < 1 || nsym > 286 || limit < 1 || limit > 15) return ZLB_E_ARG;
    ZTS_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = zts_reserve(ctx, &ctx->d_hist, 316 * 4 + 64);
    if (rc) return rc;
    rc = zts_reserve(ctx, &ctx->d_misc, 1024);
    if (rc) return rc;
    ZTS_CUDA(ctx, cudaMemcpyAsync(ctx->d_hist.p, h_freqs, (size_t)nsym * 4, cudaMemcpyHostToDevice, ctx->stream));
    rc = zts_huffman_lengths_debug(ctx, (const uint32_t*)ctx->d_hist.p, nsym, limit, (uint8_t*)ctx->d_misc.p);
    if (rc) return rc;
    ZTS_CUDA(ctx, cudaMemcpyAsync(h_lengths, ctx->d_misc.p, (size_t)nsym, cudaMemcpyDeviceToHost, ctx->stream));
    ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ZLB_OK;
}
