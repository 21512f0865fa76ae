// zts_deflate.cuh -- shared definitions of the chunk-parallel deflate pipeline.
#pragma once
#include "zts_common.cuh"

#define LZ_THREADS 1024
#define LZ_WARPS 32
#define LZ_MAX_CHUNK 65536u
// Speculative parse tiles: the chunk is cut into 1024 tiles of 64 positions and every thread of the CTA owns one
// (see zts_lz77.cu): it parses its tile from the tile's start, then carries on into the next tile until it meets
// that tile's own parse.
#define LZ_TILE_POS 64u
#define LZ_NTILES (LZ_MAX_CHUNK / LZ_TILE_POS)
#define LZ_SORT_TILE 2048u              // positions ranked by one warp in a radix pass
#define LZ_HASH_BITS 16                 // positions are grouped by a 16-bit hash of their 3-byte key
#define LZ_WINDOW 32768u                // WindowSize, src/LZ77.ts:8
#define LZ_MAXLEN 258u                  // LZ77MaxLength, src/LZ77.ts:5
#define LZ_TOK_PER_CHUNK (LZ_MAX_CHUNK + 8u * LZ_NTILES + 8u)  // token slots of the per-CTA spec / fix scratch (tile t at lz_tok_off(t))
#define LZ_LIST_PER_CHUNK (LZ_MAX_CHUNK + 8u)                  // token slots per chunk in the token list both LZ77 kernels write

#define TOK_MATCH 0x80000000u           // literal: byte ; match: TOK_MATCH | (len-3) << 16 | (dist-1)

#define ZTS_HDR_BYTES 576               // 3 + 14 + 19*3 + 316*14 bits = 4498 bits = 563 bytes

#define ZTS_HDR_STORED 0xFFFFFFFFu       // ZtsChunkInfo.hdr_bits of a chunk written as stored block(s)

#define CHUNK_LAST 1u                   // last chunk of its item: BFINAL = 1, no join marker
#define CHUNK_STAGED 2u                 // history || chunk is put together in the staging arena (dict_stage_kernel)

struct ZtsChunk {      // host-built, one per chunk
    uint64_t in_off;   // absolute offset of the chunk in d_in
    uint32_t len;      // <= 65536
    uint32_t item;
    uint32_t seg_first;  // index (within the wave) of the first chunk of the same item
    uint32_t flags;
    uint32_t dict_len;   // bytes of history in front of the chunk (<= 32768) the match search may reach into: the same
                         // item's (primed mode) and / or a preset dictionary's
    uint32_t stage_off;  // CHUNK_STAGED: the window's offset in the staging arena, in 16-byte units
};

// first position of tile t (t == LZ_NTILES gives the chunk size)
__host__ __device__ __forceinline__ uint32_t lz_tile_begin(uint32_t t) { return t * LZ_TILE_POS; }
// tiles that a chunk of n bytes has
__host__ __device__ __forceinline__ uint32_t lz_tile_count(uint32_t n) { return (n + LZ_TILE_POS - 1u) / LZ_TILE_POS; }
// tile that holds position pos
__host__ __device__ __forceinline__ uint32_t lz_tile_of(uint32_t pos) { return pos / LZ_TILE_POS; }
// first token slot of tile t: a tile never holds more tokens than positions
__host__ __device__ __forceinline__ uint32_t lz_tok_off(uint32_t t) { return lz_tile_begin(t) + 8u * t; }

struct ZtsChunkInfo {  // device-produced, one per chunk
    uint32_t n_tokens;   // tokens of the parse (without end-of-block), contiguous at the start of the chunk's list
    uint32_t hdr_bits;   // block header bits incl. BFINAL/BTYPE
    unsigned long long body_bits;  // token bits incl. end-of-block
    uint32_t out_bytes;  // bytes this chunk contributes (incl. the join marker)
    uint32_t pad;
    unsigned long long out_off;    // absolute offset in d_out
};

struct ZtsChunkCodes {  // device-produced by the Huffman kernel
    uint32_t ll[286];   // (bit-reversed code) | len << 16
    uint32_t d[30];
    uint8_t hdr[ZTS_HDR_BYTES];
};

// length (3..258) -> litlen symbol index (0..28), extra bit count and value  (src/LZ77.ts:20-53)
__host__ __device__ __forceinline__ void zts_len_code(uint32_t len, uint32_t& sym, uint32_t& ebits, uint32_t& eval)
{
    uint32_t l = len - 3;
    if (l < 8) {
        sym = l;
        ebits = 0;
        eval = 0;
    } else if (l == 255) {
        sym = 28;
        ebits = 0;
        eval = 0;
    } else {
#ifdef __CUDA_ARCH__
        uint32_t nb = (31 - __clz(l)) - 2;
#else
        uint32_t nb = (31 - __builtin_clz(l)) - 2;
#endif
        sym = 4 * nb + 4 + ((l >> nb) & 3);
        ebits = nb;
        eval = l & ((1u << nb) - 1);
    }
}

// distance (1..32768) -> distance symbol (0..29), extra bit count and value  (src/LZ77.ts:56-90)
__host__ __device__ __forceinline__ void zts_dist_code(uint32_t dist, uint32_t& sym, uint32_t& ebits, uint32_t& eval)
{
    uint32_t d = dist - 1;
    if (d < 4) {
        sym = d;
        ebits = 0;
        eval = 0;
    } else {
#ifdef __CUDA_ARCH__
        uint32_t nb = (31 - __clz(d)) - 1;
#else
        uint32_t nb = (31 - __builtin_clz(d)) - 1;
#endif
        sym = 2 * nb + 2 + ((d >> nb) & 1);
        ebits = nb;
        eval = d & ((1u << nb) - 1);
    }
}
