// zts_inflate.cu -- batched RFC-1951 decoder, one warp per independent stream
// (replaces RawInflate.decompress / parseBlock / parseDynamicHuffmanBlock / decodeHuffmanAdaptive,
//  src/RawInflate.ts:127-516, and buildHuffmanTable, src/Huffman.ts:8-68).
//
// Design (B200): the decode state is warp-uniform -- every lane tracks the same bit buffer and
// output cursor, so table look-ups are shared-memory broadcasts and there is no divergence; the
// lanes differ only where they cooperate:
//   * input: the warp keeps a 128-byte window of the stream in registers (one coalesced 4-byte
//     load per lane), words are handed to the bit reader with a shuffle;
//   * decode and copy are split: up to 32 symbols are decoded back to back into one token per lane
//     without touching the output (the serial part is then only bit-buffer arithmetic and shared-
//     memory look-ups), then the batch is written: all literals with one store, all short matches
//     side by side (one per lane), long matches cooperatively (lane k copies byte k, k+32, ...).
//     A match that reads bytes produced inside the same batch cuts the batch into sub-batches that
//     run one after the other, so memory latency is paid per sub-batch, not per symbol;
//   * overlapping matches (dist < len, src/RawInflate.ts:506-508) read the periodic source
//     out[op - dist + k mod dist], which lies entirely before the match;
//   * table construction: canonical code assignment with ballots, no atomics.
// Tables per warp in shared memory: a 10-bit root for literal/length codes and an 8-bit root for
// distance codes (entry = base << 16 | kind << 8 | extra_bits << 4 | code_bits); codes longer than
// the root are resolved canonically (first_code / count per length + symbols sorted by code), which
// replaces the reference's 2^15-entry single-level table.
//
// Algorithmic bytes per stream: C (compressed, read once) + N (output, written once).
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <array>
#include <climits>
#include <cstddef>
#include <set>
#include <chrono>
#include <type_traits>

#include "zts_common.cuh"

#ifndef INF_WARPS_PER_CTA
#define INF_WARPS_PER_CTA 1  // a CTA holds its shared memory until its slowest stream is done: one stream per CTA wastes none
#endif
#define LIT_ROOT_BITS 10
#ifndef DIST_ROOT_BITS
#define DIST_ROOT_BITS 7
#endif
#ifndef INF_MIN_CTAS
#define INF_MIN_CTAS 32  // 64 registers; 32 one-warp CTAs per SM (6272 B of tables + 1 KB the system reserves per CTA)
#endif
#define CL_ROOT_BITS 7

#define KIND_LITERAL 0u
#define KIND_BASE 1u   // length or distance base + extra bits
#define KIND_EOB 2u
#define KIND_INVALID 3u
#define INF_TOK_MATCH 0x80000000u  // token of a match: INF_TOK_MATCH | len << 16 | dist; a literal: byte << 16 | (ignored) < 256
#define ROOT_UNRESOLVED (KIND_INVALID << 8)  // root-table entry of a bit pattern whose code is longer than the root (0 bits)

struct HuffTab {
    uint16_t first_code[16];  // canonical (MSB-first) first code of each length
    uint16_t first_idx[16];   // index into sorted[] of the first symbol of each length
    uint16_t count[16];
};

// 6272 bytes per stream: with the 1 KB the system reserves per CTA, 32 one-warp CTAs fill the 228 KB of an SM. What a
// dynamic block header needs only while it is read lives where the tables it leads to are built afterwards: the
// code-length code's root table in the distance root, its sorted symbols and counts in the distance code's, its 19
// lengths in the first bytes of the literal / length code's sorted symbols.
struct InfWarpSmem {
    uint32_t lit_root[1 << LIT_ROOT_BITS];
    uint32_t dist_root[1 << DIST_ROOT_BITS];  // (+ the code-length code's root table)
    uint16_t lit_sorted[288];                  // (+ the code-length code's lengths, 32 bytes)
    uint16_t dist_sorted[32];                  // (+ the code-length code's sorted symbols)
    HuffTab lit, dist;                         // (dist: + the code-length code's)
    uint8_t stage[320];                        // litlen ++ dist code lengths of a header; the token slots of a batch
    uint32_t ring[128];                        // input words on their way into the bit buffer (BitReader)
};
static_assert(CL_ROOT_BITS <= DIST_ROOT_BITS, "the code-length root table lives in the distance root table");
static_assert(sizeof(InfWarpSmem) == 6272, "32 x (sizeof + 1 KB) fills an SM");
static_assert(offsetof(InfWarpSmem, stage) % 4 == 0 && sizeof(InfWarpSmem::stage) >= 128,
              "the token slots of a batch alias the code-length staging area");

// LengthCodeTable / LengthExtraTable (src/RawInflate.ts:17-28; symbols 286/287 decode as 258 there)
__constant__ uint16_t c_len_base[31] = {3,  4,  5,  6,  7,  8,  9,  10, 11,  13,  15,  17,  19,  23,  27, 31,
                                        35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258, 258, 258};
__constant__ uint8_t c_len_extra[31] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2,
                                        3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0, 0, 0};
// DistCodeTable / DistExtraTable (src/RawInflate.ts:31-42)
__constant__ uint16_t c_dist_base[30] = {1,    2,    3,    4,    5,    7,    9,    13,    17,    25,
                                         33,   49,   65,   97,   129,  193,  257,  385,   513,   769,
                                         1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
__constant__ uint8_t c_dist_extra[30] = {0, 0, 0, 0, 1, 1, 2, 2,  3,  3,  4,  4,  5,  5,  6,
                                         6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
// HuffmanOrder (src/RawInflate.ts:14)
__constant__ uint8_t c_huff_order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

enum { TAB_LITLEN = 0, TAB_DIST = 1, TAB_CL = 2 };

__device__ __forceinline__ uint32_t make_entry(int which, uint32_t sym, uint32_t nbits)
{
    if (which == TAB_LITLEN) {
        if (sym < 256) return (sym << 16) | (KIND_LITERAL << 8) | nbits;
        if (sym == 256) return (KIND_EOB << 8) | nbits;
        // (bit 31 marks a match token: it travels with the length base into `len << 16 | dist`, so that a literal's
        // token is its table entry as it is -- byte << 16, code length below -- without a mask in the symbol loop)
        if (sym < 288) return INF_TOK_MATCH | ((uint32_t)c_len_base[sym - 257] << 16) | (KIND_BASE << 8) |
                              ((uint32_t)c_len_extra[sym - 257] << 4) | nbits;
        return (KIND_INVALID << 8) | nbits;
    }
    if (which == TAB_DIST) {
        if (sym < 30) return ((uint32_t)c_dist_base[sym] << 16) | (KIND_BASE << 8) |
                             ((uint32_t)c_dist_extra[sym] << 4) | nbits;
        return (KIND_INVALID << 8) | nbits;  // DistCodeTable[30..31] is undefined in the reference
    }
    return (sym << 16) | (KIND_LITERAL << 8) | nbits;
}

// Canonical decoder construction for one code (warp-cooperative, all lanes call it).
// Mirrors what buildHuffmanTable (src/Huffman.ts:8-68) produces for complete or incomplete codes:
// shorter lengths first, ascending symbol order inside a length. Returns false when the lengths
// are over-subscribed (the reference would silently overwrite table slots).
__device__ bool build_table(int which, const uint8_t* lens, int n, int root_bits, uint32_t* root,
                            uint16_t* sorted, HuffTab* tab)
{
    const unsigned lane = zts_lane();
    const unsigned lt = zts_lanemask_lt();
    // count per length: lane L accumulates count[L]
    uint32_t mycount = 0;
    for (int base = 0; base < n; base += 32) {
        int s = base + (int)lane;
        uint32_t l = s < n ? lens[s] : 0;
#pragma unroll
        for (uint32_t L = 1; L <= 15; ++L) {
            unsigned m = __ballot_sync(0xFFFFFFFFu, l == L);
            if (lane == L) mycount += __popc(m);
        }
    }
    if (lane < 16) tab->count[lane] = (uint16_t)(lane ? mycount : 0);
    __syncwarp();
    // first codes / first indices, Kraft check (every lane computes the same values)
    uint32_t code = 0, idx = 0, kraft = 0;
#pragma unroll
    for (uint32_t L = 1; L <= 15; ++L) {
        uint32_t c = tab->count[L];
        if (lane == L) {
            tab->first_code[L] = (uint16_t)code;
            tab->first_idx[L] = (uint16_t)idx;
        }
        code = (code + c) << 1;
        idx += c;
        kraft += c << (15 - L);
    }
    if (kraft > (1u << 15)) return false;
    // root table: 0 bits = "not resolved here" (long code or unused pattern); the kind field of such an entry says
    // "not a literal", so the symbol loop meets it behind the one test it makes anyway
    for (int i = (int)lane; i < (1 << root_bits); i += 32) root[i] = ROOT_UNRESOLVED;
    __syncwarp();
    // assign codes in (length, symbol) order; running offset per length kept uniformly in registers
    uint32_t offs[16];
#pragma unroll
    for (int L = 0; L < 16; ++L) offs[L] = 0;
    for (int base = 0; base < n; base += 32) {
        int s = base + (int)lane;
        uint32_t l = s < n ? lens[s] : 0;
        uint32_t my_rank = 0;
#pragma unroll
        for (uint32_t L = 1; L <= 15; ++L) {
            unsigned m = __ballot_sync(0xFFFFFFFFu, l == L);
            if (l == L) my_rank = offs[L] + __popc(m & lt);
            offs[L] += __popc(m);
        }
        if (l) {
            uint32_t slot = tab->first_idx[l] + my_rank;
            sorted[slot] = (uint16_t)s;
            uint32_t c = tab->first_code[l] + my_rank;  // MSB-first canonical code
            if ((int)l <= root_bits) {
                uint32_t r = __brev(c) >> (32 - l);  // as it appears in the LSB-first bit buffer
                uint32_t e = make_entry(which, (uint32_t)s, l);
                for (uint32_t j = r; j < (1u << root_bits); j += (1u << l)) root[j] = e;
            }
        }
    }
    __syncwarp();
    return true;
}

// canonical resolution of a code that the root table did not resolve; `bits` = bit buffer (LSB first)
__device__ __forceinline__ uint32_t slow_decode(int which, uint32_t bits, int root_bits, const uint16_t* sorted,
                                                const HuffTab* tab)
{
    uint32_t v = __brev(bits) >> 17;  // first 15 stream bits, MSB-first
    for (int L = root_bits + 1; L <= 15; ++L) {
        uint32_t c = v >> (15 - L);
        uint32_t d = c - tab->first_code[L];
        if (d < tab->count[L]) return make_entry(which, sorted[tab->first_idx[L] + d], (uint32_t)L);
    }
    return 0;  // undefined code
}

// Input words reach the bit buffer through a ring of 128 words in shared memory: a window of 32 words (one per lane,
// requested a window ahead) is appended whenever fewer than INF_RING_MIN unread words are left, which the symbol loop
// checks once per batch -- a batch of 32 symbols takes at most 32 x 48 bits, i.e. at most 50 words -- so that its refills are one shared-memory
// load at a running address.
#define INF_RING_WORDS 128u
#define INF_RING_MIN 52u
struct BitReader {
    const uint32_t* next_base;  // aligned address of the window behind the prefetched one
    const uint8_t* end;         // one past the last readable input byte
    uint32_t win_next;          // this lane's word of the next window to append (prefetched)
    uint32_t ring_s;            // shared-window address of this warp's ring
    uint32_t rd, wr;            // words consumed / appended since the last (re)start
    unsigned long long buf;
    int cnt;                    // valid bits in buf
    unsigned long long base_bits;    // stream bits consumed before the last (re)start
    uint32_t skip_bits;         // bits of the first word that precede the (re)start point
};

__device__ __forceinline__ uint32_t br_fetch(const BitReader& br, const uint32_t* base)
{
    const uint32_t* p = base + zts_lane();
    // a word is readable if it overlaps [.., end); bytes past `end` inside that word are never
    // consumed as data because every consumer checks the consumed-bit count against the item length
    return ((const uint8_t*)p < br.end) ? __ldg(p) : 0u;
}

// appends the prefetched window and requests the one behind it (all lanes; the slots it overwrites were read at
// least INF_RING_WORDS - 32 - INF_RING_MIN words ago)
__device__ __forceinline__ void br_append(BitReader& br)
{
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(br.ring_s + (((br.wr + zts_lane()) & (INF_RING_WORDS - 1u)) << 2)), "r"(br.win_next)
                 : "memory");
    br.wr += 32u;
    br.win_next = br_fetch(br, br.next_base);
    br.next_base += 32;
    __syncwarp();
}

__device__ __forceinline__ uint32_t br_ring_word(const BitReader& br, uint32_t i)
{
    uint32_t w;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w) : "r"(br.ring_s + ((i & (INF_RING_WORDS - 1u)) << 2)) : "memory");
    return w;
}

__device__ __forceinline__ void br_init(BitReader& br, const uint8_t* src, const uint8_t* end,
                                        unsigned long long base_bits)
{
    uintptr_t a = (uintptr_t)src;
    const uint32_t* base = (const uint32_t*)(a & ~(uintptr_t)3);
    br.end = end;
    br.base_bits = base_bits;
    br.skip_bits = (uint32_t)(a & 3) * 8;
    br.rd = br.wr = 0;
    __syncwarp();  // (a restart: every lane is done with the ring)
    br.win_next = br_fetch(br, base);
    br.next_base = base + 32;
    br_append(br);
    br_append(br);
    // first word: drop the bytes before the stream
    const uint32_t w = br_ring_word(br, 0);
    br.rd = 1;
    br.buf = (unsigned long long)(w >> br.skip_bits);
    br.cnt = 32 - (int)br.skip_bits;
}

__device__ __forceinline__ void br_refill(BitReader& br)
{
    if (br.cnt <= 32) {
        if (br.rd == br.wr) br_append(br);
        const uint32_t w = br_ring_word(br, br.rd);
        br.rd++;
        br.buf |= (unsigned long long)w << br.cnt;
        br.cnt += 32;
    }
}

__device__ __forceinline__ uint32_t br_take(BitReader& br, int n)
{
    uint32_t v = (uint32_t)br.buf & ((1u << n) - 1u);
    br.buf >>= n;
    br.cnt -= n;
    return v;
}

// stream bits consumed so far
__device__ __forceinline__ unsigned long long br_bits_used(const BitReader& br)
{
    return br.base_bits + (unsigned long long)br.rd * 32ull - br.skip_bits - (unsigned long long)br.cnt;
}

// ---- which error does the reference raise when the input ends early? ---------------------------------------------
// readBits throws 'input buffer is broken' (src/RawInflate.ts:188), readCodeByTable looks the code up in what is left
// (zero padded) and throws 'invalid code length: N' when the N bits of that code are not all there (:238). The decode
// loops only notice that a batch ran past the end; these helpers replay from a known bit position, one symbol at a
// time, and tell the two cases apart. Rare path, every lane computes the same.
// 32 bits of the stream at bit position `pos`, zero padded behind the end of the input
__device__ uint32_t inf_peek(const uint8_t* src, unsigned long long in_len, unsigned long long pos)
{
    const unsigned long long byte = pos >> 3;
    unsigned long long v = 0;
    for (uint32_t k = 0; k < 6; ++k)
        if (byte + k < in_len) v |= (unsigned long long)src[byte + k] << (8u * k);
    return (uint32_t)(v >> (pos & 7u));
}
// status of a Huffman code of the code-length alphabet read at `pos` (dynamic block header)
__device__ uint32_t inf_classify_cl(const InfWarpSmem* S, const uint8_t* src, unsigned long long in_len, unsigned long long pos)
{
    const uint32_t e = S->dist_root[inf_peek(src, in_len, pos) & ((1u << CL_ROOT_BITS) - 1u)];
    const uint32_t nb = e & 15u;
    if (nb && pos + nb > in_len * 8ull) return ZLB_ST_CODE_LENGTH | (nb << 8);
    return ZLB_ST_INPUT_BROKEN;  // the code was there: its repeat count was not
}
// replays the symbols of a block from `pos` until the input runs out
__device__ uint32_t inf_classify_symbols(const InfWarpSmem* S, const uint8_t* src, unsigned long long in_len, unsigned long long pos)
{
    const unsigned long long in_bits = in_len * 8ull;
    for (uint32_t k = 0; k < 64 && pos < in_bits + 64; ++k) {
        uint32_t bits = inf_peek(src, in_len, pos);
        uint32_t e = S->lit_root[bits & ((1u << LIT_ROOT_BITS) - 1u)];
        if ((e & 15u) == 0) e = slow_decode(TAB_LITLEN, bits, LIT_ROOT_BITS, S->lit_sorted, &S->lit);
        if (e == 0) return ZLB_ST_BAD_CODE;
        if (pos + (e & 15u) > in_bits) return ZLB_ST_CODE_LENGTH | ((e & 15u) << 8);
        pos += e & 15u;
        if (!(e & 0x300u)) continue;              // literal
        if ((e & 0x300u) != (KIND_BASE << 8)) break;  // end of block / invalid symbol: not an input problem
        pos += (e >> 4) & 15u;                    // length extra bits (readBits)
        if (pos > in_bits) return ZLB_ST_INPUT_BROKEN;
        bits = inf_peek(src, in_len, pos);
        uint32_t d = S->dist_root[bits & ((1u << DIST_ROOT_BITS) - 1u)];
        if ((d & 15u) == 0) d = slow_decode(TAB_DIST, bits, DIST_ROOT_BITS, S->dist_sorted, &S->dist);
        if (d == 0) return ZLB_ST_BAD_CODE;
        if (pos + (d & 15u) > in_bits) return ZLB_ST_CODE_LENGTH | ((d & 15u) << 8);
        pos += d & 15u;
        pos += (d >> 4) & 15u;                    // distance extra bits (readBits)
        if (pos > in_bits) return ZLB_ST_INPUT_BROKEN;
    }
    return ZLB_ST_INPUT_BROKEN;
}

// INF_BYTES: the decoder. INF_WINDOW: the window mode of the marker split (see there): the output is one 16-bit word per
// byte, out_off / out_cap count bytes / words, and the 32768 words in front of out_off belong to the item as well -- the
// kernel fills them with 0x8000 | w, "byte w of the window" (the 32 KiB of output in front of the piece), so that the
// copy code below is the same for both: a match that reaches before the piece copies window words. INF_DICT: the
// decoder with a preset dictionary (dicts[item] in the blob `dict`, zlb_inflate_batch_dict): a match may reach up to
// the dictionary's last 32768 bytes in front of the output; one whose source starts there takes a path of its own.
// The dictionary arguments are read by INF_DICT only. INF_SIZE: the decoder without an output (zlb_inflate_size_batch):
// it decodes and checks exactly like INF_BYTES but stores no byte, copies no match, skips stored data after its LEN
// check and has no capacity; only the dictionary's length is read (dicts may be NULL). In segment mode a distance that
// reaches before the piece's first byte does not fail it: results[item].crc32 tells how far in front the piece
// reached, at most 32768 (the marker split compares that with the output of the pieces in front). INF_SIZE and
// INF_WINDOW read ZLB_INFLATE_BITS (the searched split): in_off / in_len / in_used count bits. Positions then count
// from the piece's first byte, its first bits consumed at the start, so that a stored block's byte alignment holds.
// INF_POINTS (zlb_inflate_index): INF_BYTES that also records access points into `sink` (ZtsPointSink). INF_RANGE
// (zlb_inflate_ranges): INF_DICT -- the window of an access point is the dictionary -- that starts at a bit offset
// (ZLB_INFLATE_BITS) and stops, without an error, once out_cap bytes are written: a match or stored copy that crosses
// the cap is clamped, so exactly the bytes up to the cap are written and nothing behind it.
#define WIN_WORDS 32768u
enum { INF_BYTES = 0, INF_WINDOW = 1, INF_DICT = 2, INF_SIZE = 3, INF_POINTS = 4, INF_RANGE = 5 };
// Where INF_POINTS puts the access points of item i: slots points[first[i] .. first[i + 1]), its count in count[i]. A
// block start becomes a point when its output position is at least the last point's plus `spacing` (the first block
// always): the greedy rule of zlb_inflate_index, the same as the host applies to the split's piece starts.
struct ZtsPointSink {
    zlb_point* points;
    const unsigned long long* first;
    unsigned long long* count;
    unsigned long long spacing;
};
// `out`: the output base of items[*].out_off. INF_RANGE is launched with out == NULL and device addresses in out_off
// (a range's pieces write into the caller's slots and into scratch in one launch): the slot address is only ever
// out + out_off, never compared with or offset from `out` otherwise.
template <int MODE>
__global__ void __launch_bounds__(INF_WARPS_PER_CTA * 32, INF_MIN_CTAS)
inflate_warp_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, const zlb_item* __restrict__ items,
                    zlb_result* __restrict__ results, uint32_t n_items, uint32_t flags,
                    const zlb_dict* __restrict__ dicts, const uint8_t* __restrict__ dict, ZtsPointSink sink)
{
    using T = typename std::conditional<MODE == INF_WINDOW, uint16_t, uint8_t>::type;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const unsigned lane = zts_lane();
    const unsigned warp = threadIdx.x >> 5;
    InfWarpSmem* S = reinterpret_cast<InfWarpSmem*>(smem_raw) + warp;
    const uint32_t item = blockIdx.x * INF_WARPS_PER_CTA + warp;
    if (item >= n_items) return;

    const zlb_item it = items[item];
    constexpr bool BITS_OK = MODE == INF_SIZE || MODE == INF_WINDOW || MODE == INF_RANGE;
    constexpr bool DICT = MODE == INF_DICT || MODE == INF_RANGE;  // a window in front of the output, from the blob
    const bool bits = BITS_OK && (flags & ZLB_INFLATE_BITS);
    const uint32_t sb = bits ? (uint32_t)(it.in_off & 7u) : 0u;  // bits of the first byte in front of the piece
    const uint8_t* src = in + (bits ? it.in_off >> 3 : it.in_off);
    const unsigned long long in_len = bits ? (sb + it.in_len + 7) >> 3 : it.in_len;  // bytes the piece touches
    T* dst = reinterpret_cast<T*>(out + it.out_off);
    uint32_t reach = MODE == INF_WINDOW ? WIN_WORDS : 0u;  // how far a distance may reach in front of the output
    const uint8_t* dtail = nullptr;                       // INF_DICT: the `reach` bytes in front of the output
    if constexpr (DICT) {
        const zlb_dict d = dicts[item];
        reach = d.len < WIN_WORDS ? (uint32_t)d.len : WIN_WORDS;
        dtail = dict + d.off + d.len - reach;
    }
    if constexpr (MODE == INF_SIZE) {
        if (flags & ZLB_INFLATE_SEGMENT) {
            reach = WIN_WORDS;  // (every distance: how far it went is recorded instead)
        } else if (dicts) {
            const unsigned long long l = dicts[item].len;
            reach = l < WIN_WORDS ? (uint32_t)l : WIN_WORDS;
        }
    }
    uint32_t reached = 0;  // INF_SIZE: the farthest a match reached in front of the output
    if constexpr (MODE == INF_WINDOW) {
        uint4* w = reinterpret_cast<uint4*>(dst - WIN_WORDS);  // (slots are 256-byte aligned)
        for (uint32_t i = lane; i < WIN_WORDS / 8; i += 32) {
            const uint32_t a = 0x80008000u | (8u * i) | ((8u * i + 1u) << 16);
            w[i] = make_uint4(a, a + 0x00020002u, a + 0x00040004u, a + 0x00060006u);
        }
        __syncwarp();
    }
    const unsigned long long in_bits = bits ? sb + it.in_len : it.in_len * 8ull;
    const unsigned long long cap = it.out_cap;

    BitReader br;
    br.ring_s = (uint32_t)__cvta_generic_to_shared(S->ring);
    br_init(br, src, src + in_len, 0);
    if constexpr (BITS_OK)
        if (sb) br_take(br, (int)sb);

    unsigned long long op = 0;
    uint32_t status = ZLB_ST_OK;
    uint32_t blocks = 0;
    int have_fixed = 0;
    bool bfinal = false;
    bool full = false;  // INF_RANGE: out_cap bytes written
    // INF_POINTS: the item's next slot, its end, and the output position the next point needs at least
    unsigned long long pt_next = 0, pt_end = 0, pt_due = 0;
    if constexpr (MODE == INF_POINTS) {
        pt_next = sink.first[item];
        pt_end = sink.first[item + 1];
    }

    while (!bfinal && status == ZLB_ST_OK && !full) {
        // segment mode: a piece of a larger stream ends cleanly where a block ends and its input is used up
        if ((flags & ZLB_INFLATE_SEGMENT) && blocks > 0 && br_bits_used(br) == in_bits) break;
        br_refill(br);
        if (br_bits_used(br) + 3 > in_bits) {
            status = ZLB_ST_INPUT_BROKEN;
            break;
        }
        if constexpr (MODE == INF_POINTS) {
            if (op >= pt_due) {
                if (lane == 0 && pt_next < pt_end) sink.points[pt_next] = {br_bits_used(br), op, 0};
                pt_next++;
                pt_due = op + sink.spacing;
            }
        }
        uint32_t hdr = br_take(br, 3);  // src/RawInflate.ts:146-152
        bfinal = hdr & 1u;
        uint32_t btype = hdr >> 1;
        blocks++;

        if (btype == 0) {
            // ---- stored block (src/RawInflate.ts:251-318): drop to the byte boundary, LEN, NLEN
            unsigned long long used = br_bits_used(br);
            unsigned long long byte_pos = (used + 7) >> 3;
            if (byte_pos + 4 > in_len) {
                // src/RawInflate.ts:266 (LEN) / :272 (NLEN): which of the two 16-bit fields is cut short
                status = byte_pos + 2 > in_len ? ZLB_ST_STORED_LEN : (ZLB_ST_STORED_LEN | (1u << 8));
                break;
            }
            const uint8_t* p = src + byte_pos;
            uint32_t len = (uint32_t)p[0] | ((uint32_t)p[1] << 8);
            uint32_t nlen = (uint32_t)p[2] | ((uint32_t)p[3] << 8);
            if ((flags & ZLB_INFLATE_CHECK_NLEN) && ((len ^ nlen) != 0xFFFFu)) {
                status = ZLB_ST_STORED_LEN;
                break;
            }
            byte_pos += 4;
            if (byte_pos + len > in_len) {
                status = ZLB_ST_INPUT_BROKEN;
                break;
            }
            if (MODE == INF_RANGE && op + len >= cap) {
                len = (uint32_t)(cap - op);  // (the cap is reached: what is left of the block is not wanted)
                full = true;
            }
            if (MODE != INF_SIZE && op + len > cap) {
                status = ZLB_ST_OUT_OVERFLOW;
                break;
            }
            if constexpr (MODE != INF_SIZE)
                for (uint32_t k = lane; k < len; k += 32) dst[op + k] = src[byte_pos + k];
            op += len;
            br_init(br, src + byte_pos + len, src + in_len, (byte_pos + len) * 8ull);
            __syncwarp();
            continue;
        }
        if (btype == 3) {
            status = ZLB_ST_BTYPE;  // src/RawInflate.ts:168
            break;
        }

        if (btype == 1) {
            // ---- fixed Huffman tables (src/RawInflate.ts:45-61)
            if (have_fixed != 1) {
                for (int i = (int)lane; i < 288; i += 32) S->stage[i] = i <= 143 ? 8 : i <= 255 ? 9 : i <= 279 ? 7 : 8;
                for (int i = (int)lane; i < 30; i += 32) S->stage[288 + i] = 5;
                __syncwarp();
                build_table(TAB_LITLEN, S->stage, 288, LIT_ROOT_BITS, S->lit_root, S->lit_sorted, &S->lit);
                build_table(TAB_DIST, S->stage + 288, 30, DIST_ROOT_BITS, S->dist_root, S->dist_sorted, &S->dist);
                have_fixed = 1;
            }
        } else {
            // ---- dynamic Huffman header (src/RawInflate.ts:345-388)
            have_fixed = 0;
            br_refill(br);
            uint32_t hlit = br_take(br, 5) + 257;
            uint32_t hdist = br_take(br, 5) + 1;
            uint32_t hclen = br_take(br, 4) + 4;
            uint8_t* const cl_lens = reinterpret_cast<uint8_t*>(S->lit_sorted);  // (dead before that table is built)
            if (lane < 19) cl_lens[lane] = 0;
            __syncwarp();
            for (uint32_t i = 0; i < hclen; ++i) {
                br_refill(br);
                uint32_t v = br_take(br, 3);
                if (lane == 0) cl_lens[c_huff_order[i]] = (uint8_t)v;
            }
            __syncwarp();
            if (br_bits_used(br) > in_bits) {
                status = ZLB_ST_INPUT_BROKEN;
                break;
            }
            if (!build_table(TAB_CL, cl_lens, 19, CL_ROOT_BITS, S->dist_root, S->dist_sorted, &S->dist)) {
                status = ZLB_ST_BAD_LENGTHS;
                break;
            }
            // code lengths with repeat codes 16/17/18 (:361-383); over-long repeats are clipped like
            // the reference's out-of-range typed-array stores
            const uint32_t total = hlit + hdist;
            uint32_t i = 0, prev = 0;
            while (i < total && status == ZLB_ST_OK) {
                br_refill(br);
                const unsigned long long cl_pos = br_bits_used(br);
                uint32_t e = S->dist_root[(uint32_t)br.buf & ((1u << CL_ROOT_BITS) - 1u)];  // (the code-length code's table)
                uint32_t nb = e & 15u;
                if (nb == 0) {
                    status = ZLB_ST_BAD_CODE;
                    break;
                }
                br_take(br, (int)nb);
                uint32_t sym = e >> 16;
                uint32_t rep = 1, val = sym;
                if (sym == 16) {
                    rep = 3 + br_take(br, 2);
                    val = prev;
                } else if (sym == 17) {
                    rep = 3 + br_take(br, 3);
                    val = 0;
                } else if (sym == 18) {
                    rep = 11 + br_take(br, 7);
                    val = 0;
                }
                // lanes store the run cooperatively (rep <= 138)
                for (uint32_t k = lane; k < rep; k += 32)
                    if (i + k < total) S->stage[i + k] = (uint8_t)val;
                i += rep;
                prev = val;
                if (br_bits_used(br) > in_bits) status = inf_classify_cl(S, src, in_len, cl_pos);
            }
            if (status != ZLB_ST_OK) break;
            __syncwarp();
            // stage[0 .. total) holds litlen then dist lengths
            if (!build_table(TAB_LITLEN, S->stage, (int)hlit, LIT_ROOT_BITS, S->lit_root, S->lit_sorted, &S->lit) ||
                !build_table(TAB_DIST, S->stage + hlit, (int)hdist, DIST_ROOT_BITS, S->dist_root, S->dist_sorted,
                             &S->dist)) {
                status = ZLB_ST_BAD_LENGTHS;
                break;
            }
        }

        // ---- symbol loop (src/RawInflate.ts:466-516), 32 symbols per batch
        bool eob = false;
        while (!eob && status == ZLB_ST_OK && !full) {
            // -- decode: token of symbol i ends up in lane i: literal = byte << 16 | junk < 256, match = INF_TOK_MATCH | len << 16 | dist.
            //    The tables are addressed through 32-bit shared-window addresses held in registers (a generic
            //    pointer to the per-warp slice gets rematerialised from %tid on every look-up otherwise).
            uint32_t mytok = 0, ntok = 0;
            uint32_t stop = 0;  // 1 = end of block, 2 = undefined code / symbol
            const unsigned long long batch_pos = br_bits_used(br);  // (only looked at when the input ends inside the batch)
            {
                // the address of the warp's slice is warp-uniform; routing it through a shuffle keeps it in a register
                // (ptxas otherwise recomputes it from %tid and %cluster_ctaid in front of every look-up: 9 instructions),
                // and everything in the slice is that register plus a constant
                const uint32_t smem_s = __shfl_sync(0xFFFFFFFFu, (uint32_t)__cvta_generic_to_shared(S), 0);
                const uint32_t lit_s = smem_s + (uint32_t)offsetof(InfWarpSmem, lit_root);
                const uint32_t dist_s = smem_s + (uint32_t)offsetof(InfWarpSmem, dist_root);
                // same for the end-of-input pointer of the bit reader (recomputed from the item table otherwise)
                br.end = reinterpret_cast<const uint8_t*>(__shfl_sync(0xFFFFFFFFu, (unsigned long long)br.end, 0));
                // with a whole batch worth of words in the ring the refills below need no test
                while (br.wr - br.rd < INF_RING_MIN) br_append(br);
                unsigned long long buf = br.buf;
                int cnt = br.cnt;
                const uint32_t ring_s = smem_s + (uint32_t)offsetof(InfWarpSmem, ring), ring_e = ring_s + 4u * INF_RING_WORDS;
                const uint32_t ra0 = ring_s + ((br.rd & (INF_RING_WORDS - 1u)) << 2);
                uint32_t ra = ra0;  // address of the next word
                // the batch's tokens go through shared memory (one store per symbol instead of a compare + select into the
                // lane that owns the slot); the code-length staging area is dead while symbols are decoded
                const uint32_t tok_s = smem_s + (uint32_t)offsetof(InfWarpSmem, stage);
                uint32_t ta = tok_s;
                const uint32_t tok_e = tok_s + 128u;
                // a word from the ring if 32 more bits fit (a length code: before it reads on, which is enough for its
                // extra bits and the distance, 5 + 15 + 13 bits)
#define INF_TAKE_WORD()                                                                       \
    if (cnt <= 32) {                                                                          \
        uint32_t w_;                                                                          \
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w_) : "r"(ra) : "memory");              \
        ra += 4u;                                                                             \
        ra = ra == ring_e ? ring_s : ra;                                                      \
        buf |= (unsigned long long)w_ << cnt;                                                 \
        cnt += 32;                                                                            \
    }
#define INF_SYMBOL(SLOT, TOP, TAIL) { \
                    if (TOP) INF_TAKE_WORD() \
                    uint32_t e; \
                    asm volatile("{\n\t.reg .b32 a;\n\tmad.lo.u32 a, %1, 4, %2;\n\tld.shared.u32 %0, [a];\n\t}" /* (index * 4 + base in one instruction) */ \
                                 : "=r"(e) : "r"((uint32_t)buf & ((1u << LIT_ROOT_BITS) - 1u)), "r"(lit_s) : "memory"); \
                    buf >>= (e & 15u); \
                    cnt -= (int)(e & 15u); \
                    uint32_t tokv = e; /* (a literal's entry is its token) */ \
                    if (e & 0x300u) { \
                        bool is_match = (e & 0x300u) == (KIND_BASE << 8); \
                        if (!is_match) { /* unresolved by the root table, end of block or an undefined symbol */ \
                            if ((e & 15u) == 0) { \
                                e = slow_decode(TAB_LITLEN, (uint32_t)buf, LIT_ROOT_BITS, S->lit_sorted, &S->lit); \
                                if (e == 0) { \
                                    stop = 2; \
                                    { ta += 4u * (SLOT); break; } \
                                } \
                                buf >>= (e & 15u); \
                                cnt -= (int)(e & 15u); \
                                tokv = e; \
                            } \
                            const uint32_t kind = e & 0x300u; \
                            if (kind > (KIND_BASE << 8)) { \
                                stop = (e & 0x100u) ? 2u : 1u; /* KIND_INVALID (3) / KIND_EOB (2) */ \
                                { ta += 4u * (SLOT); break; } \
                            } \
                            is_match = kind != 0u; \
                        } \
                        if (is_match) { \
                            INF_TAKE_WORD() \
                            const uint32_t xb = (e >> 4) & 15u; \
                            const uint32_t len = (e >> 16) + ((uint32_t)buf & ((1u << xb) - 1u)); \
                            buf >>= xb; \
                            cnt -= (int)xb; \
                            uint32_t d; \
                            asm volatile("{\n\t.reg .b32 a;\n\tmad.lo.u32 a, %1, 4, %2;\n\tld.shared.u32 %0, [a];\n\t}" \
                                         : "=r"(d) : "r"((uint32_t)buf & ((1u << DIST_ROOT_BITS) - 1u)), "r"(dist_s) : "memory"); \
                            if ((d & 0x300u) != (KIND_BASE << 8)) { \
                                if ((d & 15u) == 0) d = slow_decode(TAB_DIST, (uint32_t)buf, DIST_ROOT_BITS, S->dist_sorted, &S->dist); \
                                if ((d & 0x300u) != (KIND_BASE << 8)) { \
                                    stop = 2; \
                                    { ta += 4u * (SLOT); break; } \
                                } \
                            } \
                            buf >>= (d & 15u); \
                            cnt -= (int)(d & 15u); \
                            const uint32_t db = (d >> 4) & 15u; \
                            const uint32_t dist = (d >> 16) + ((uint32_t)buf & ((1u << db) - 1u)); \
                            buf >>= db; \
                            cnt -= (int)db; \
                            tokv = (len << 16) | dist; \
                            if (TAIL) INF_TAKE_WORD() \
                        } \
                    } \
                    asm volatile("st.shared.u32 [%0], %1;" ::"r"(ta + 4u * (SLOT)), "r"(tokv) : "memory"); }
                // Two symbols per trip (the token slots of a batch are an even number): one loop test for both, and the
                // second one does not ask for a word: behind a literal that was read right after that test at least 17
                // bits are left, enough for any code, and a match of the first symbol takes a word when it is done.
                do {
                    INF_SYMBOL(0u, true, true)
                    INF_SYMBOL(1u, false, false)
                    ta += 8u;
                } while (ta != tok_e);
#undef INF_SYMBOL
#undef INF_TAKE_WORD
                ntok = (ta - tok_s) >> 2;
                __syncwarp();
                if (lane < ntok) asm volatile("ld.shared.u32 %0, [%1];" : "=r"(mytok) : "r"(tok_s + 4u * lane) : "memory");
                br.buf = buf;
                br.cnt = cnt;
                br.rd += ((ra - ra0) & (4u * INF_RING_WORDS - 1u)) >> 2;  // (fewer than INF_RING_WORDS words per batch)
            }
            if (stop == 1) eob = true;
            if (stop == 2) status = ZLB_ST_BAD_CODE;
            if (br_bits_used(br) > in_bits) {
                // the batch ran past the end of the input: nothing of it is trusted; which error it is -- a code or
                // extra bits cut short -- is found by replaying the batch
                status = inf_classify_symbols(S, src, in_len, batch_pos);
                break;
            }
            // -- output positions: exclusive prefix sum of the token lengths
            const bool mine = lane < ntok;
            const uint32_t dist = mytok & 0xFFFFu;  // (of a match)
            const bool is_match = mine && (mytok & INF_TOK_MATCH);
            const uint32_t len = !mine ? 0u : (is_match ? (mytok >> 16) & 0x7FFFu : 1u);
            uint32_t inc = len;
#pragma unroll
            for (int sft = 1; sft < 32; sft <<= 1) {
                const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, sft);
                if (lane >= (unsigned)sft) inc += t;
            }
            // Everything below works with 32-bit offsets from the batch's first byte (a batch is at most 32 x 258 bytes):
            // `rel` = where this token's bytes start; the output written so far and the room left are clamped to
            // values that decide the same (a distance is at most 32768, a batch at most 8256 bytes).
            const uint32_t rel = inc - len;
            T* const bdst = dst + op;  // first byte of the batch
            const uint32_t behind = op > 0x00FFFFFFull ? 0x00FFFFFFu : (uint32_t)op;         // bytes in front of the batch
            const uint32_t room = cap - op > 0x00FFFFFFull ? 0x00FFFFFFu : (uint32_t)(cap - op);  // (op <= cap always)
            // a distance beyond the start of the output (the reference would copy `undefined` -> 0) or an
            // output slot that is too small ends the batch before the offending token
            const bool bad_dist = is_match && dist > behind + rel + reach;
            // (INF_RANGE: a token that starts at or behind the cap is not wanted, one that crosses it is clamped)
            const bool over = MODE != INF_SIZE && mine && (MODE == INF_RANGE ? rel >= room : rel + len > room);
            const uint32_t wlen = MODE == INF_RANGE ? min(len, room - min(rel, room)) : len;  // bytes the token writes
            const unsigned bad_mask = __ballot_sync(0xFFFFFFFFu, bad_dist || over);
            uint32_t nvalid = ntok;
            if (bad_mask) {
                nvalid = (uint32_t)__ffs((int)bad_mask) - 1u;
                const bool first_is_dist = __shfl_sync(0xFFFFFFFFu, (int)bad_dist, (int)nvalid) != 0;
                if (MODE == INF_RANGE && __shfl_sync(0xFFFFFFFFu, (int)over, (int)nvalid))
                    full = true;  // (a bad distance behind the cap is not looked at)
                else
                    status = first_is_dist ? ZLB_ST_BAD_CODE : ZLB_ST_OUT_OVERFLOW;
            }
            const bool live = lane < nvalid;
            if constexpr (MODE == INF_SIZE) {
                // nothing is written: the batch moves the cursor and tells how far its matches reached
                if (live && is_match && dist > behind + rel) reached = max(reached, dist - (behind + rel));
                op += nvalid ? __shfl_sync(0xFFFFFFFFu, inc, (int)nvalid - 1) : 0u;
                __syncwarp();
                continue;
            }
            // -- literals: one store
            ZTS_ASSERT(!live || (op + rel + wlen <= cap && (!is_match || dist <= op + rel + reach)));
            if (live && !is_match) bdst[rel] = (uint8_t)(mytok >> 16);
            __syncwarp();  // (a match may read the literals of its own batch)
            // -- matches, sub-batch by sub-batch: a sub-batch ends in front of the first match that reads what a match
            //    of the same sub-batch writes
            uint32_t start = 0;
            unsigned match_mask = __ballot_sync(0xFFFFFFFFu, live && is_match);
            // where this match's source ends (exclusive), as an offset from the batch's first byte: negative when it
            // lies in front of the batch
            const int src_end = (int)rel - (int)dist + (int)(len < dist ? len : dist);
            while (match_mask) {
                // first byte the matches of this sub-batch write (its first match's: match_mask holds lanes >= start)
                const int sub_start = (int)__shfl_sync(0xFFFFFFFFu, rel, __ffs((int)match_mask) - 1);
                // reads bytes written by this very sub-batch? (source end beyond that byte)
                const bool dep = live && is_match && lane >= start && src_end > sub_start;
                const unsigned dep_mask = __ballot_sync(0xFFFFFFFFu, dep);
                const uint32_t cut = dep_mask ? (uint32_t)__ffs((int)dep_mask) - 1u : 32u;  // behind the first match always
                const bool in_sub = live && is_match && lane >= start && lane < cut;
                const bool small = in_sub && len <= 8u && dist >= len && (!DICT || dist <= behind + rel);
                if (__any_sync(0xFFFFFFFFu, small)) {
                    // short non-overlapping matches: every lane copies its own, loads first, then stores
                    T v[8];
                    T* dp = bdst + rel;
                    const T* sp = dp - dist;
#pragma unroll
                    for (int k = 0; k < 8; ++k) v[k] = (small && (uint32_t)k < wlen) ? sp[k] : (T)0;
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                        if (small && (uint32_t)k < wlen) dp[k] = v[k];
                }
                unsigned big_mask = __ballot_sync(0xFFFFFFFFu, in_sub && !small);
                while (big_mask) {
                    const int j = __ffs((int)big_mask) - 1;
                    big_mask &= big_mask - 1;
                    const uint32_t jl = __shfl_sync(0xFFFFFFFFu, wlen, j);
                    const uint32_t jd = __shfl_sync(0xFFFFFFFFu, dist, j);
                    const uint32_t jr = __shfl_sync(0xFFFFFFFFu, rel, j);
                    T* o = bdst + jr;
                    const T* s0 = o - jd;
                    if (DICT && jd > behind + jr) {
                        // the source starts in the dictionary (then behind == op): byte k is byte
                        // op + jr - jd + (k mod jd) of dictionary || output, which lies in front of the match
                        const int x0 = (int)(behind + jr) - (int)jd;
                        uint32_t r = lane % jd;
                        const uint32_t step = 32u % jd;
                        for (uint32_t k = lane; k < jl; k += 32) {
                            const int x = x0 + (int)r;
                            o[k] = x < 0 ? dtail[(int)reach + x] : dst[x];
                            r += step;
                            if (r >= jd) r -= jd;
                        }
                    } else if (jd >= jl) {
                        for (uint32_t k = lane; k < jl; k += 32) o[k] = s0[k];
                    } else {
                        // periodic source: byte k comes from s0[k mod dist]
                        uint32_t r = lane % jd;
                        const uint32_t step = 32u % jd;
                        for (uint32_t k = lane; k < jl; k += 32) {
                            o[k] = s0[r];
                            r += step;
                            if (r >= jd) r -= jd;
                        }
                    }
                }
                __syncwarp();  // the next sub-batch reads what this one wrote
                start = cut;
                match_mask = cut < 32u ? (match_mask >> cut) << cut : 0u;
            }
            // bytes of the tokens that were written (all of them unless the batch was cut short)
            op += nvalid ? __shfl_sync(0xFFFFFFFFu, inc, (int)nvalid - 1) : 0u;
            if (MODE == INF_RANGE && op >= cap) {
                op = cap;
                full = true;
            }
            __syncwarp();
        }
        if (status == ZLB_ST_OK && br_bits_used(br) > in_bits) status = ZLB_ST_INPUT_BROKEN;
    }

    if constexpr (MODE == INF_SIZE) reached = __reduce_max_sync(0xFFFFFFFFu, reached);
    if constexpr (MODE == INF_POINTS)
        if (lane == 0) sink.count[item] = pt_next < pt_end ? pt_next - sink.first[item] : pt_end - sink.first[item];
    if (lane == 0) {
        zlb_result r = results[item];
        if (MODE == INF_SIZE && (flags & ZLB_INFLATE_SEGMENT)) r.crc32 = reached;
        r.status = status;
        r.blocks = blocks | ((flags & ZLB_INFLATE_SEGMENT) && bfinal ? 0x80000000u : 0u);  // segment mode: saw BFINAL
        r.out_len = op;
        r.in_used = bits ? br_bits_used(br) - sb : (br_bits_used(br) + 7) >> 3;  // whole unread bytes are given back (:511-514)
        results[item] = r;
    }
}

template <int MODE>
static int inflate_launch_mode(zlb_ctx* ctx, cudaStream_t st, const uint8_t* d_in, uint8_t* d_out, const zlb_item* d_items,
                               zlb_result* d_results, size_t n, uint32_t flags, const zlb_dict* d_dicts,
                               const uint8_t* d_dict, ZtsPointSink sink = ZtsPointSink{})
{
    const size_t smem = sizeof(InfWarpSmem) * INF_WARPS_PER_CTA;
    ZTS_CUDA(ctx, cudaFuncSetAttribute(inflate_warp_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    unsigned grid = (unsigned)((n + INF_WARPS_PER_CTA - 1) / INF_WARPS_PER_CTA);
    ZTS_LAUNCH(ctx,
               MODE == INF_WINDOW ? ZK_INFLATE_WINDOW : MODE == INF_DICT ? ZK_INFLATE_DICT : MODE == INF_SIZE ? ZK_INFLATE_SIZE
               : MODE == INF_POINTS ? ZK_INFLATE_POINTS : MODE == INF_RANGE ? ZK_INFLATE_RANGE : ZK_INFLATE,
               inflate_warp_kernel<MODE><<<grid, INF_WARPS_PER_CTA * 32, smem, st>>>(d_in, d_out, d_items, d_results,
                                                                                    (uint32_t)n, flags, d_dicts, d_dict, sink));
    return ZLB_OK;
}
// the decoder: with a dictionary table (d_dicts[i] belongs to d_items[i]) the dictionary instantiation; without an
// output (d_out == NULL, a size call) the size instantiation, which reads the table's lengths only
static int inflate_launch(zlb_ctx* ctx, cudaStream_t st, const uint8_t* d_in, uint8_t* d_out, const zlb_item* d_items,
                          zlb_result* d_results, size_t n, uint32_t flags, const zlb_dict* d_dicts = nullptr,
                          const uint8_t* d_dict = nullptr)
{
    if (!d_out) return inflate_launch_mode<INF_SIZE>(ctx, st, d_in, nullptr, d_items, d_results, n, flags, d_dicts, nullptr);
    if (d_dicts) return inflate_launch_mode<INF_DICT>(ctx, st, d_in, d_out, d_items, d_results, n, flags, d_dicts, d_dict);
    return inflate_launch_mode<INF_BYTES>(ctx, st, d_in, d_out, d_items, d_results, n, flags, nullptr, nullptr);
}

// ---- marker split (ZLB_INFLATE_SPLIT) ------------------------------------------------------------------------
// A stream written by zlb_deflate_batch is a sequence of pieces joined by empty stored blocks, `00 00 FF FF` after
// byte alignment. One warp per piece decodes a 1 GiB stream in the time of a 64 KiB one. Nothing is assumed about the
// input: the pieces are decoded into scratch slots in segment mode, and only if every piece (a) ends exactly where the
// next one starts, (b) never reaches before its own first byte and (c) fits its slot is the result gathered. Items
// that fail (b) alone -- primed streams, zlib's Z_SYNC_FLUSH, whose matches reach across the markers -- are decoded
// once more in window mode (below); a false marker, a reference before the start of the stream or anything else that
// fails a check sends the item to the one-warp decoder.
#define SPLIT_MIN_BYTES (256u << 10)   // items at least this large are worth splitting
#define SPLIT_SLOT (128u << 10)        // scratch bytes per piece (pieces of this engine's streams are <= 64 KiB)
#define SPLIT_MAX_MARKS (1u << 22)
#define SPLIT_MIN_PIECE 64u            // compressed bytes a piece has at least (64 KiB of zeros deflate to 78 + the marker)

__global__ void __launch_bounds__(256)
marker_scan_kernel(const uint8_t* __restrict__ in, unsigned long long n, unsigned long long* __restrict__ marks,
                   uint32_t* __restrict__ count, uint32_t cap, unsigned long long tag)
{
    // thread t looks at 16 consecutive start offsets
    const unsigned long long base = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) * 16ull;
    if (base + 4 > n) return;
    uint8_t b[19];
#pragma unroll
    for (int k = 0; k < 19; ++k) b[k] = (base + k < n) ? in[base + k] : (uint8_t)0x55;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        if (b[k] == 0 && b[k + 1] == 0 && b[k + 2] == 0xFF && b[k + 3] == 0xFF && base + k + 4 <= n) {
            const uint32_t slot = atomicAdd(count, 1u);
            if (slot < cap) marks[slot] = tag | (base + k + 4);  // first byte after the marker (+ the item's tag)
        }
    }
}

// ---- block finder: where a stream without markers may be cut ----------------------------------------------------
// An ordinary zlib / gzip stream has no markers; its blocks start at arbitrary bit offsets. block_find_kernel tests
// the bit offsets of a span, one warp per span and one offset per lane, for a block header that an encoder would
// write: BFINAL = 0 and a dynamic header whose three codes are ones an encoder writes (zlib's own rules, stricter than
// the decoder), or a stored block whose LEN / NLEN agree. A span's answer is the first offset that passes. Nothing
// depends on it being right: the split uses a cut only once the piece in front of it decoded cleanly and ended exactly
// there (split_chain), so a false candidate costs time, never a result. A stored block is proposed by where it ends:
// the block behind it starts exactly there, while its own header may be preceded by zero bits that pass the same test.
struct ZtsFindCut {
    unsigned long long first, last, end;  // bits of the input: offsets [first, last) are tested; a block ends by `end`
};
#define FIND_WARPS 4
#define FIND_NONE (~0ull)

// 32 bits of the input at bit `pos` (aligned word loads of words that overlap [.., end_byte); zero behind)
__device__ __forceinline__ uint32_t find_peek(const uint8_t* in, unsigned long long pos, const uint8_t* end)
{
    const uintptr_t a = (uintptr_t)(in + (pos >> 3));
    const uint32_t* p = (const uint32_t*)(a & ~(uintptr_t)3);
    const uint32_t w0 = (const uint8_t*)p < end ? __ldg(p) : 0u;
    const uint32_t w1 = (const uint8_t*)(p + 1) < end ? __ldg(p + 1) : 0u;
    return (uint32_t)((((unsigned long long)w1 << 32) | w0) >> ((a & 3u) * 8u + (uint32_t)(pos & 7u)));
}

// the dynamic block header at bit b (its first 17 bits passed the prefilter): the code-length code is complete, the
// HLIT + HDIST lengths decode without a leading repeat and without overrunning, the literal / length code is complete
// and codes symbol 256, the distance code is complete, one code of length 1 or empty, and all of it ends by `end`.
// tab: this lane's 128-entry table of the code-length code (symbol | length << 5).
__device__ bool find_dynamic(const uint8_t* in, unsigned long long b, unsigned long long end, const uint8_t* in_end,
                             uint8_t* tab)
{
    const uint32_t h = find_peek(in, b, in_end);
    const uint32_t hlit = ((h >> 3) & 31u) + 257u, hdist = ((h >> 8) & 31u) + 1u, hclen = ((h >> 13) & 15u) + 4u;
    unsigned long long pos = b + 17;
    if (pos + 3 * hclen > end) return false;
    const unsigned long long lo = find_peek(in, pos, in_end), hi = find_peek(in, pos + 32, in_end);
    const unsigned long long v = lo | (hi << 32);
    unsigned long long lens = 0;  // 3 bits per code-length symbol
    uint32_t kraft = 0;
    for (uint32_t i = 0; i < hclen; ++i) {
        const uint32_t l = (uint32_t)(v >> (3 * i)) & 7u;
        lens |= (unsigned long long)l << (3 * c_huff_order[i]);
        kraft += l ? 128u >> l : 0u;
    }
    if (kraft != 128u) return false;
    pos += 3 * hclen;
    uint32_t code = 0;
    for (uint32_t L = 1; L <= 7; ++L) {
        for (uint32_t s = 0; s < 19; ++s) {
            if (((lens >> (3 * s)) & 7u) != L) continue;
            for (uint32_t j = __brev(code) >> (32 - L); j < 128u; j += 1u << L) tab[j] = (uint8_t)(s | (L << 5));
            ++code;
        }
        code <<= 1;
    }
    const uint32_t total = hlit + hdist;
    uint32_t i = 0, prev = 0, lit_k = 0, dist_k = 0, dist_n = 0;
    bool has_eob = false;
    while (i < total) {
        uint32_t x = find_peek(in, pos, in_end);
        const uint32_t e = tab[x & 127u], L = e >> 5, sym = e & 31u;
        pos += L;
        x >>= L;
        uint32_t rep = 1, val = sym;
        if (sym == 16) {
            if (i == 0) return false;
            rep = 3 + (x & 3u);
            pos += 2;
            val = prev;
        } else if (sym == 17) {
            rep = 3 + (x & 7u);
            pos += 3;
            val = 0;
        } else if (sym == 18) {
            rep = 11 + (x & 127u);
            pos += 7;
            val = 0;
        }
        if (i + rep > total || pos > end) return false;
        const uint32_t nl = i < hlit ? min(rep, hlit - i) : 0u, nd = rep - nl;
        if (val) {
            lit_k += nl << (15 - val);
            dist_k += nd << (15 - val);
            dist_n += nd;
        }
        if (i <= 256u && 256u < i + nl) has_eob = val != 0;
        prev = val;
        i += rep;
    }
    return lit_k == (1u << 15) && has_eob && (dist_k == (1u << 15) || dist_n == 0 || (dist_n == 1 && dist_k == (1u << 14)));
}

// the stored block at bit b (its 3 header bits are zero): zero padding, LEN == ~NLEN, the block ends before `end`,
// and the block behind it is a stored one (LEN == ~NLEN) or passes the dynamic test (BFINAL either): 3 zero bits and
// two 16-bit fields that agree turn up in compressed data every few hundred KB, this second header makes such a
// chance hit rare. Returns the bit where it ends, FIND_NONE if it is not one.
__device__ unsigned long long find_stored(const uint8_t* in, unsigned long long b, uint32_t h, unsigned long long end,
                                          const uint8_t* in_end, uint8_t* tab)
{
    const unsigned long long a = (b + 3 + 7) & ~7ull;  // the byte boundary LEN starts at
    const uint32_t pad = (uint32_t)(a - b - 3);
    if (((h >> 3) & ((1u << pad) - 1u)) != 0) return FIND_NONE;
    if (a + 32 > end) return FIND_NONE;
    const uint32_t w = find_peek(in, a, in_end);
    if (((w & 0xFFFFu) ^ (w >> 16)) != 0xFFFFu) return FIND_NONE;
    const unsigned long long stop = a + 32 + 8ull * (w & 0xFFFFu);
    if (stop + 40 > end) return FIND_NONE;
    const uint32_t h2 = find_peek(in, stop, in_end);
    if ((h2 & 0xFEu) == 0u) {  // stored, starting on the byte boundary
        const uint32_t w2 = find_peek(in, stop + 8, in_end);
        return ((w2 & 0xFFFFu) ^ (w2 >> 16)) == 0xFFFFu ? stop : FIND_NONE;
    }
    if ((h2 & 6u) == 4u && ((h2 >> 3) & 31u) <= 29u && ((h2 >> 8) & 31u) <= 29u && find_dynamic(in, stop, end, in_end, tab))
        return stop;
    return FIND_NONE;
}

// out[c] = the first candidate of span c (a stored block: where it ends), FIND_NONE if there is none
__global__ void __launch_bounds__(FIND_WARPS * 32)
block_find_kernel(const uint8_t* __restrict__ in, const ZtsFindCut* __restrict__ cuts, uint32_t n,
                  unsigned long long* __restrict__ out)
{
    __shared__ uint8_t tabs[FIND_WARPS * 32][128];
    const unsigned lane = zts_lane();
    const uint32_t c = blockIdx.x * FIND_WARPS + (threadIdx.x >> 5);
    if (c >= n) return;
    const ZtsFindCut cut = cuts[c];
    const uint8_t* in_end = in + ((cut.end + 7) >> 3);
    unsigned long long found = FIND_NONE;
    for (unsigned long long base = cut.first; base < cut.last; base += 32) {
        const unsigned long long b = base + lane;
        unsigned long long prop = FIND_NONE;
        if (b < cut.last && b + 17 <= cut.end) {
            const uint32_t h = find_peek(in, b, in_end);
            // prefilter on 17 bits: BFINAL = 0, BTYPE = 2, HLIT <= 286, HDIST <= 30 (or BTYPE = 0)
            if ((h & 7u) == 4u) {
                if (((h >> 3) & 31u) <= 29u && ((h >> 8) & 31u) <= 29u && find_dynamic(in, b, cut.end, in_end, tabs[threadIdx.x]))
                    prop = b;
            } else if ((h & 7u) == 0u) {
                prop = find_stored(in, b, h, cut.end, in_end, tabs[threadIdx.x]);
            }
        }
        const unsigned m = __ballot_sync(0xFFFFFFFFu, prop != FIND_NONE);
        if (m) {
            found = __shfl_sync(0xFFFFFFFFu, prop, __ffs((int)m) - 1);
            break;
        }
    }
    if (lane == 0) out[c] = found;
}

// one launch of the finder over h_cuts; results in h_out. The tables go to ctx->d_misc.
static int block_find(zlb_ctx* ctx, const uint8_t* d_in, const std::vector<ZtsFindCut>& h_cuts, unsigned long long* h_out)
{
    const size_t n = h_cuts.size();
    if (!n) return ZLB_OK;
    cudaStream_t st = ctx->stream;
    int rc = zts_reserve(ctx, &ctx->d_misc, n * (sizeof(ZtsFindCut) + 8) + 256);
    if (rc) return rc;
    ZtsFindCut* d_cuts = (ZtsFindCut*)ctx->d_misc.p;
    unsigned long long* d_found = (unsigned long long*)(d_cuts + n);
    ZTS_CUDA(ctx, cudaMemcpyAsync(d_cuts, h_cuts.data(), n * sizeof(ZtsFindCut), cudaMemcpyHostToDevice, st));
    ZTS_LAUNCH(ctx, ZK_BLOCK_FIND,
               block_find_kernel<<<(unsigned)((n + FIND_WARPS - 1) / FIND_WARPS), FIND_WARPS * 32, 0, st>>>(d_in, d_cuts,
                                                                                                         (uint32_t)n, d_found));
    ZTS_CUDA(ctx, cudaMemcpyAsync(h_out, d_found, n * 8, cudaMemcpyDeviceToHost, st));
    ZTS_CUDA(ctx, cudaStreamSynchronize(st));
    return ZLB_OK;
}

struct ZtsGather {
    unsigned long long src, dst, len;
};

__global__ void __launch_bounds__(256)
segment_gather_kernel(const uint8_t* __restrict__ scratch, uint8_t* __restrict__ out, const ZtsGather* __restrict__ g)
{
    const ZtsGather e = g[blockIdx.x];
    const uint8_t* s = scratch + e.src;
    uint8_t* d = out + e.dst;
    // 16-byte copies where both sides allow it (slots are 16-byte aligned; the destination decides)
    const uint32_t head = (uint32_t)min((unsigned long long)((16u - ((uintptr_t)d & 15u)) & 15u), e.len);
    for (uint32_t i = threadIdx.x; i < head; i += 256) d[i] = s[i];
    const unsigned long long body = (e.len - head) & ~15ull;
    if ((((uintptr_t)(s + head)) & 15u) == 0) {
        const uint4* s4 = reinterpret_cast<const uint4*>(s + head);
        uint4* d4 = reinterpret_cast<uint4*>(d + head);
        for (unsigned long long i = threadIdx.x; i < body / 16; i += 256) d4[i] = s4[i];
    } else {
        for (unsigned long long i = threadIdx.x; i < body; i += 256) d[head + i] = s[head + i];
    }
    for (unsigned long long i = head + body + threadIdx.x; i < e.len; i += 256) d[i] = s[i];
}

// ---- window mode: pieces that reach up to 32 KiB in front of their first byte -----------------------------------
// Every piece of such an item is decoded again by inflate_warp_kernel<true>, into 16-bit words: a byte (< 0x100), or
// 0x8000 | w, "byte w of the piece's window" (the 32768 output bytes in front of its first byte). The last 32768
// words of window ++ piece are the piece's tail map T_j: W_{j+1} in terms of W_j (a piece shorter than a window
// shifts the older part of W_j along, so a window may span many short pieces). Composition
// (A;B)[i] = B[i] < 0x100 ? B[i] : A[B[i] & 0x7FFF] is associative, so W_j in terms of W_0 -- the window in front of
// the stream, of which no byte exists -- is an exclusive scan of the tail maps over the pieces of the item, starting
// from the identity. A byte of a piece that still names W_0 after that reaches before the start of the stream: the
// item fails and goes to the one-warp decoder. The scan has a fixed depth and no CTA ever waits for another: a CTA
// composes a run of about sqrt(n) consecutive pieces (window_run_kernel), one per item composes the runs
// (window_scan_kernel), and a CTA per run applies its prefix piece by piece while it turns the words into bytes in
// the pieces' byte slots (window_resolve_kernel), which are gathered like those of independent pieces.
struct ZtsWinPiece {
    unsigned long long words;  // byte offset in the window arena of the piece's first output word
    unsigned long long bytes;  // byte offset in the split scratch of its resolved bytes
    uint32_t len, cap;         // output words, slot words
};
struct ZtsWinRun {
    uint32_t first, count;  // pieces [first, first + count)
    uint32_t item;          // index of its item among those resolved
    uint32_t pad;
};
struct ZtsWinItem {
    uint32_t first_run, runs;
    const uint8_t* dict;  // W_0: the last dict_len (<= 32768) bytes of the item's preset dictionary (none: 0)
    uint32_t dict_len, pad;
};
#define WIN_THREADS 1024
#define WIN_SMEM (2u * WIN_WORDS * 2u)  // the map being composed and the next one

__device__ __forceinline__ void win_identity(uint16_t* E)
{
    uint32_t* e = reinterpret_cast<uint32_t*>(E);
    for (uint32_t i = threadIdx.x; i < WIN_WORDS / 2; i += WIN_THREADS) e[i] = 0x80008000u | (2u * i) | ((2u * i + 1u) << 16);
    __syncthreads();
}
// 64 KiB, both sides 16-byte aligned
__device__ __forceinline__ void win_copy(uint16_t* dst, const uint16_t* src)
{
    uint4* d = reinterpret_cast<uint4*>(dst);
    const uint4* s = reinterpret_cast<const uint4*>(src);
    for (uint32_t i = threadIdx.x; i < WIN_WORDS / 8; i += WIN_THREADS) d[i] = s[i];
    __syncthreads();
}
// En = E;tail
__device__ __forceinline__ void win_compose(const uint16_t* E, uint16_t* En, const uint16_t* __restrict__ tail)
{
    for (uint32_t i = threadIdx.x; i < WIN_WORDS; i += WIN_THREADS) {
        const uint32_t t = tail[i];
        En[i] = (t & 0x8000u) ? E[t & 0x7FFFu] : (uint16_t)t;
    }
    __syncthreads();
}
// T_j: the last 32768 words of window ++ piece
__device__ __forceinline__ const uint16_t* win_tail(const uint8_t* arena, const ZtsWinPiece& p)
{
    ZTS_ASSERT(p.len <= p.cap && p.words >= 2ull * WIN_WORDS && p.words % 16 == 0);  // (the window words in front)
    return reinterpret_cast<const uint16_t*>(arena + p.words) + ((long long)p.len - (long long)WIN_WORDS);
}

// aggregate of run r: W_{last + 1} in terms of W_first
__global__ void __launch_bounds__(WIN_THREADS)
window_run_kernel(const uint8_t* __restrict__ arena, const ZtsWinPiece* __restrict__ pieces,
                  const ZtsWinRun* __restrict__ runs, uint16_t* __restrict__ agg)
{
    extern __shared__ __align__(16) uint16_t wmap[];
    uint16_t *E = wmap, *En = wmap + WIN_WORDS;
    const ZtsWinRun r = runs[blockIdx.x];
    win_identity(E);
    for (uint32_t j = r.first; j < r.first + r.count; ++j) {
        win_compose(E, En, win_tail(arena, pieces[j]));
        uint16_t* t = E;
        E = En;
        En = t;
    }
    win_copy(agg + (size_t)blockIdx.x * WIN_WORDS, E);
}

// prefix of every run of item i: the window in front of the run's first piece in terms of W_0. With a preset
// dictionary W_0 is known in part: its last dict_len words are the dictionary's bytes, the scan starts from that map.
__global__ void __launch_bounds__(WIN_THREADS)
window_scan_kernel(const ZtsWinItem* __restrict__ items, const uint16_t* __restrict__ agg, uint16_t* __restrict__ prefix)
{
    extern __shared__ __align__(16) uint16_t wmap[];
    uint16_t *E = wmap, *En = wmap + WIN_WORDS;
    const ZtsWinItem it = items[blockIdx.x];
    win_identity(E);
    if (it.dict_len) {
        for (uint32_t i = threadIdx.x; i < it.dict_len; i += WIN_THREADS) E[WIN_WORDS - it.dict_len + i] = it.dict[i];
        __syncthreads();
    }
    for (uint32_t r = it.first_run; r < it.first_run + it.runs; ++r) {
        win_copy(prefix + (size_t)r * WIN_WORDS, E);
        if (r + 1 < it.first_run + it.runs) {
            win_compose(E, En, agg + (size_t)r * WIN_WORDS);
            uint16_t* t = E;
            E = En;
            En = t;
        }
    }
}

__device__ __forceinline__ uint32_t win_resolve(const uint16_t* E, uint32_t w)
{
    return (w & 0x8000u) ? E[w & 0x7FFFu] : w;
}

// the bytes of every piece of run r; fail[item] = 1 when one of them lies before the start of the stream
__global__ void __launch_bounds__(WIN_THREADS)
window_resolve_kernel(const uint8_t* __restrict__ arena, uint8_t* __restrict__ scratch, const ZtsWinPiece* __restrict__ pieces,
                      const ZtsWinRun* __restrict__ runs, const uint16_t* __restrict__ prefix, uint32_t* __restrict__ fail)
{
    extern __shared__ __align__(16) uint16_t wmap[];
    uint16_t *E = wmap, *En = wmap + WIN_WORDS;
    const ZtsWinRun r = runs[blockIdx.x];
    win_copy(E, prefix + (size_t)blockIdx.x * WIN_WORDS);
    uint32_t seen = 0;  // or of the resolved words: bit 15 = a byte before the stream
    for (uint32_t j = r.first; j < r.first + r.count; ++j) {
        const ZtsWinPiece p = pieces[j];
        ZTS_ASSERT(p.len <= p.cap);
        const uint16_t* w = reinterpret_cast<const uint16_t*>(arena + p.words);
        uint8_t* o = scratch + p.bytes;
        // four words at a time (both slots are 256-byte aligned)
        const uint32_t n4 = p.len / 4u;
        for (uint32_t q = threadIdx.x; q < n4; q += WIN_THREADS) {
            const uint2 v = reinterpret_cast<const uint2*>(w)[q];
            const uint32_t b0 = win_resolve(E, v.x & 0xFFFFu), b1 = win_resolve(E, v.x >> 16);
            const uint32_t b2 = win_resolve(E, v.y & 0xFFFFu), b3 = win_resolve(E, v.y >> 16);
            seen |= b0 | b1 | b2 | b3;
            reinterpret_cast<uint32_t*>(o)[q] = (b0 & 0xFFu) | ((b1 & 0xFFu) << 8) | ((b2 & 0xFFu) << 16) | (b3 << 24);
        }
        for (uint32_t k = 4u * n4 + threadIdx.x; k < p.len; k += WIN_THREADS) {
            const uint32_t b = win_resolve(E, w[k]);
            seen |= b;
            o[k] = (uint8_t)b;
        }
        if (j + 1 < r.first + r.count) {
            win_compose(E, En, win_tail(arena, p));
            uint16_t* t = E;
            E = En;
            En = t;
        }
    }
    if (__syncthreads_or((int)(seen & 0x8000u)) && threadIdx.x == 0) fail[r.item] = 1u;
}

// The access points a zlb_inflate_index call collects (inflate_device with a sink): the caller's host tables. The
// split's routes offer the starts of an item's pieces, the one-warp route (INF_POINTS) its block headers; both take
// them by the same greedy rule (ZtsPointSink).
struct ZtsIndexSink {
    unsigned long long spacing;
    zlb_point* points;
    const uint64_t* first;  // n + 1 entries
    uint64_t* count;
};

// window of a point: the min(out_pos, 32768) output bytes in front of it, in the item's output slot
static unsigned long long index_win_off(const zlb_item& it, unsigned long long out_pos)
{
    return it.out_off + out_pos - std::min(out_pos, (unsigned long long)WIN_WORDS);
}

// the greedy choice over the ascending candidates c[0 .. n) of item i, into its slots
static void index_select(const ZtsIndexSink& s, size_t i, const zlb_item& it, const zlb_point* c, size_t n)
{
    const uint64_t slots = s.first[i + 1] - s.first[i];
    uint64_t taken = 0;
    unsigned long long due = 0;
    for (size_t j = 0; j < n && taken < slots; ++j) {
        if (c[j].out_pos < due) continue;
        s.points[s.first[i] + taken++] = {c[j].in_bit, c[j].out_pos, index_win_off(it, c[j].out_pos)};
        due = c[j].out_pos + s.spacing;
    }
    s.count[i] = taken;
}

// One call's split: the caller's items and preset dictionaries (dicts == NULL: none), the indices of its large items,
// and the pieces of item big[k], seg[first[k] .. first[k + 1]) (split_layout). seg[j] is piece j's input span, in bytes
// or, with `bits` (the searched split), in bits of the input; the decode split gives it a byte slot of its scratch
// (out_off / out_cap).
struct SplitJob {
    const zlb_item* items;
    const zlb_dict* dicts;
    std::vector<size_t> big;
    std::vector<size_t> first;
    std::vector<zlb_item> seg;
    bool bits = false;
    ZtsIndexSink* sink = nullptr;  // zlb_inflate_index: where the piece starts of a decoded item go
    size_t pieces(size_t k) const { return first[k + 1] - first[k]; }
    // where the last piece of big[k] starts, from the item's first input byte (bit)
    unsigned long long last_start(size_t k) const
    {
        return seg[first[k + 1] - 1].in_off - items[big[k]].in_off * (bits ? 8u : 1u);
    }
};

// The chain checks of the pieces r[0 .. n) of an item: each one decoded cleanly, ended exactly where the next one
// starts, and only the last one saw BFINAL. With `window`, a piece behind the first (or the first too, when the item
// has a preset dictionary: `dict`) that stopped at an undefined code or distance may have reached before its first
// byte: SPLIT_WINDOW says window mode may still decode the item.
enum { SPLIT_BAD = 0, SPLIT_OK = 1, SPLIT_WINDOW = 2 };
static int split_chain(const zlb_result* r, const zlb_item* seg, size_t n, bool window, bool dict)
{
    bool reaches = false;
    for (size_t j = 0; j < n; ++j) {
        const bool last = j + 1 == n;
        const bool fin = (r[j].blocks & 0x80000000u) != 0;
        if (window && (j > 0 || dict) && r[j].status == ZLB_ST_BAD_CODE) {
            reaches = true;
            continue;
        }
        if (r[j].status != ZLB_ST_OK) return SPLIT_BAD;
        if (last ? !fin : (fin || r[j].in_used != seg[j].in_len)) return SPLIT_BAD;
    }
    return reaches ? SPLIT_WINDOW : SPLIT_OK;
}

// result of item big[k], whose pieces' results r[0 .. job.pieces(k)) passed the checks
static zlb_result split_result(const SplitJob& job, size_t k, const zlb_result* r)
{
    const size_t n = job.pieces(k);
    zlb_result o;
    memset(&o, 0, sizeof o);
    unsigned long long blocks = 0;
    for (size_t j = 0; j < n; ++j) {
        o.out_len += r[j].out_len;
        blocks += r[j].blocks & 0x7FFFFFFFu;
    }
    o.status = ZLB_ST_OK;
    o.in_used = job.bits ? (job.last_start(k) + r[n - 1].in_used + 7) >> 3 : job.last_start(k) + r[n - 1].in_used;
    o.blocks = (uint32_t)blocks;
    return o;
}

// split_result, checked against the item's slot; the pieces' bytes (r[j].out_len at scratch offset seg[j].out_off)
// are queued for the gather when they fit
static zlb_result split_finish(const SplitJob& job, size_t k, const zlb_result* r, std::vector<ZtsGather>& gath)
{
    const zlb_item& it = job.items[job.big[k]];
    const zlb_item* seg = &job.seg[job.first[k]];
    zlb_result o = split_result(job, k, r);
    const unsigned long long total = o.out_len;
    if (total > it.out_cap) {
        o.status = ZLB_ST_OUT_OVERFLOW;
        o.out_len = 0;
    }
    if (total <= it.out_cap && total) {
        unsigned long long at = 0;
        for (size_t j = 0; j < job.pieces(k); ++j) {
            if (r[j].out_len) gath.push_back({seg[j].out_off, it.out_off + at, r[j].out_len});
            at += r[j].out_len;
        }
    }
    if (job.sink && o.status == ZLB_ST_OK) {  // the pieces' starts, in bits from the item's first byte
        std::vector<zlb_point> cand(job.pieces(k));
        unsigned long long at = 0;
        for (size_t j = 0; j < cand.size(); ++j) {
            cand[j] = {job.bits ? seg[j].in_off - 8 * it.in_off : 8 * (seg[j].in_off - it.in_off), at, 0};
            at += r[j].out_len;
        }
        index_select(*job.sink, job.big[k], it, cand.data(), cand.size());
    }
    return o;
}

// Scratch budget of an arena of the split stage: a quarter of what the device has free plus what the arena already
// holds, at most 16 GiB, and at most k times what `in_bytes` of input could legitimately inflate to (2048 x, at least
// 64 MiB). Items whose scratch does not fit are not split: the one-warp decoder gives the same result.
struct SplitBudget {
    size_t device;
    explicit SplitBudget(const ZtsDevBuf& arena)
    {
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) free_b = 0;
        device = std::min((free_b + arena.cap) / 4, (size_t)16 << 30);
    }
    size_t operator()(size_t in_bytes, size_t k) const
    {
        return std::min(device, k * std::max(in_bytes * 2048u, (size_t)64 << 20));
    }
};

// Reserves scratch of the split stage; *got = false, and no error left behind, when the device cannot give it (the
// items then go to the one-warp decoder).
static int split_reserve(zlb_ctx* ctx, ZtsDevBuf* arena, size_t bytes, bool* got)
{
    const int rc = zts_reserve(ctx, arena, bytes);
    *got = rc == ZLB_OK;
    if (rc != ZLB_E_NOMEM) return rc;
    ctx->err[0] = 0;
    return ZLB_OK;
}

// One segment-mode launch of the decoder over the piece table seg, whose copy and results go to d_seg / d_res in the
// caller's arena; res = the pieces' results. MODE INF_BYTES writes byte slots at d_out, INF_WINDOW word slots at
// d_out, INF_SIZE nothing (d_out NULL). bits: the table's spans count bits (ZLB_INFLATE_BITS).
template <int MODE>
static int split_segments(zlb_ctx* ctx, const uint8_t* d_in, uint8_t* d_out, const std::vector<zlb_item>& seg,
                          zlb_item* d_seg, zlb_result* d_res, uint32_t flags, std::vector<zlb_result>& res,
                          bool bits = false)
{
    cudaStream_t st = ctx->stream;
    const size_t np = seg.size();
    ZTS_CUDA(ctx, cudaMemcpyAsync(d_seg, seg.data(), np * sizeof(zlb_item), cudaMemcpyHostToDevice, st));
    ZTS_CUDA(ctx, cudaMemsetAsync(d_res, 0, np * sizeof(zlb_result), st));
    const int rc = inflate_launch_mode<MODE>(ctx, st, d_in, d_out, d_seg, d_res, np,
                                             (flags & ZLB_INFLATE_CHECK_NLEN) | ZLB_INFLATE_SEGMENT |
                                                 (bits ? ZLB_INFLATE_BITS : 0u), nullptr, nullptr);
    if (rc) return rc;
    res.assign(np, zlb_result());
    ZTS_CUDA(ctx, cudaMemcpyAsync(res.data(), d_res, np * sizeof(zlb_result), cudaMemcpyDeviceToHost, st));
    ZTS_CUDA(ctx, cudaStreamSynchronize(st));
    return ZLB_OK;
}

// The window arena, as byte offsets: word slots (each behind its window, `words` bytes in all) | a map per run: the
// aggregates, the prefixes | per piece: the decode's item and result | the resolve's pieces, runs and items | a fail
// flag per item
struct WinLayout {
    size_t agg, prefix, seg, res, pieces, runs, items, fail, total;
};
static WinLayout win_layout(size_t words, size_t np, size_t nr, size_t ni)
{
    WinLayout l;
    l.agg = words;
    l.prefix = l.agg + nr * WIN_WORDS * 2;
    l.seg = l.prefix + nr * WIN_WORDS * 2;
    l.res = l.seg + np * sizeof(zlb_item);
    l.pieces = l.res + np * sizeof(zlb_result);
    l.runs = l.pieces + np * sizeof(ZtsWinPiece);
    l.items = l.runs + nr * sizeof(ZtsWinRun);
    l.fail = l.items + ni * sizeof(ZtsWinItem);
    l.total = l.fail + ni * 4 + 256;
    return l;
}

// Window mode for the items big[cand[*]] (byte slots at seg[j].out_off of d_scratch, as inflate_split_batch laid them
// out): all of them in one decode launch and one scan; h_results / done / gath as there. d_dict: the blob of the
// job's preset dictionaries.
static int inflate_split_window(zlb_ctx* ctx, const uint8_t* d_in, uint8_t* d_scratch, const uint8_t* d_dict,
                                const SplitJob& job, uint32_t flags, const std::vector<size_t>& cand,
                                zlb_result* h_results, std::vector<char>& done, std::vector<ZtsGather>& gath)
{
    cudaStream_t st = ctx->stream;
    // runs of about sqrt(n) pieces: the scan's depth is then about 3 sqrt(n) compositions
    auto run_len = [](size_t n) {
        size_t g = 8;
        while (g * g < n) ++g;
        return g;
    };
    const size_t map_b = (size_t)WIN_WORDS * 2;
    // The scratch is bounded like the byte slots', with three times their bound by input (two bytes per word, the
    // windows, the maps).
    const SplitBudget budget(ctx->d_window);
    std::vector<size_t> take;
    size_t words = 0, np = 0, nr = 0, in_b = 0;
    for (size_t k : cand) {
        const size_t a = job.first[k], n = job.pieces(k), in_k = job.items[job.big[k]].in_len;
        size_t w = 0;
        for (size_t j = a; j < a + n; ++j) w += map_b + 2 * (size_t)job.seg[j].out_cap;  // (out_cap: a multiple of 256)
        const size_t g = run_len(n);
        if (win_layout(words + w, np + n, nr + (n + g - 1) / g, take.size() + 1).total > budget(in_b + in_k, 3)) continue;
        take.push_back(k);
        words += w;
        np += n;
        nr += (n + g - 1) / g;
        in_b += in_k;
    }
    if (take.empty()) return ZLB_OK;
    const WinLayout lay = win_layout(words, np, nr, take.size());
    bool got = false;
    int rc = split_reserve(ctx, &ctx->d_window, lay.total, &got);
    if (rc || !got) return rc;
    uint8_t* arena = (uint8_t*)ctx->d_window.p;
    uint16_t* d_agg = (uint16_t*)(arena + lay.agg);
    uint16_t* d_prefix = (uint16_t*)(arena + lay.prefix);
    ZtsWinPiece* d_pieces = (ZtsWinPiece*)(arena + lay.pieces);
    ZtsWinRun* d_runs = (ZtsWinRun*)(arena + lay.runs);
    ZtsWinItem* d_witems = (ZtsWinItem*)(arena + lay.items);
    uint32_t* d_fail = (uint32_t*)(arena + lay.fail);
    // 1. every piece of those items in window mode, one launch
    std::vector<zlb_item> wseg;
    wseg.reserve(np);
    size_t at = 0;
    for (size_t k : take)
        for (size_t j = job.first[k]; j < job.first[k + 1]; ++j) {
            zlb_item w = job.seg[j];
            w.out_off = at + map_b;  // the window's words in front
            at += map_b + 2 * (size_t)w.out_cap;
            wseg.push_back(w);
        }
    std::vector<zlb_result> wres;
    rc = split_segments<INF_WINDOW>(ctx, d_in, arena, wseg, (zlb_item*)(arena + lay.seg), (zlb_result*)(arena + lay.res),
                                    flags, wres, job.bits);
    if (rc) return rc;
    // 2. the chain checks; the items that pass are resolved
    std::vector<ZtsWinPiece> wp;
    std::vector<ZtsWinRun> runs;
    std::vector<ZtsWinItem> witems;
    std::vector<size_t> wk, wfirst;  // per resolved item: its k, its first piece in wseg / wres
    for (size_t t = 0, wj = 0; t < take.size(); ++t) {
        const size_t k = take[t], a = job.first[k], n = job.pieces(k);
        const size_t w0 = wj;
        wj += n;
        if (split_chain(&wres[w0], &job.seg[a], n, false, false) != SPLIT_OK) continue;
        const size_t g = run_len(n);
        const zlb_dict d = job.dicts ? job.dicts[job.big[k]] : zlb_dict{0, 0};
        const uint32_t dl = d.len < WIN_WORDS ? (uint32_t)d.len : WIN_WORDS;
        witems.push_back({(uint32_t)runs.size(), (uint32_t)((n + g - 1) / g), dl ? d_dict + d.off + d.len - dl : nullptr, dl, 0u});
        for (size_t s = 0; s < n; s += g)
            runs.push_back({(uint32_t)(wp.size() + s), (uint32_t)std::min(g, n - s), (uint32_t)wk.size(), 0u});
        for (size_t j = 0; j < n; ++j)
            wp.push_back({wseg[w0 + j].out_off, job.seg[a + j].out_off, (uint32_t)wres[w0 + j].out_len, (uint32_t)job.seg[a + j].out_cap});
        wk.push_back(k);
        wfirst.push_back(w0);
    }
    if (wk.empty()) return ZLB_OK;
    // 3. tail maps, scan, resolve
    ZTS_CUDA(ctx, cudaMemcpyAsync(d_pieces, wp.data(), wp.size() * sizeof(ZtsWinPiece), cudaMemcpyHostToDevice, st));
    ZTS_CUDA(ctx, cudaMemcpyAsync(d_runs, runs.data(), runs.size() * sizeof(ZtsWinRun), cudaMemcpyHostToDevice, st));
    ZTS_CUDA(ctx, cudaMemcpyAsync(d_witems, witems.data(), witems.size() * sizeof(ZtsWinItem), cudaMemcpyHostToDevice, st));
    ZTS_CUDA(ctx, cudaMemsetAsync(d_fail, 0, wk.size() * 4, st));
    ZTS_CUDA(ctx, cudaFuncSetAttribute(window_run_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)WIN_SMEM));
    ZTS_CUDA(ctx, cudaFuncSetAttribute(window_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)WIN_SMEM));
    ZTS_CUDA(ctx, cudaFuncSetAttribute(window_resolve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)WIN_SMEM));
    ZTS_LAUNCH(ctx, ZK_WINDOW_RUN,
               window_run_kernel<<<(unsigned)runs.size(), WIN_THREADS, WIN_SMEM, st>>>(arena, d_pieces, d_runs, d_agg));
    ZTS_LAUNCH(ctx, ZK_WINDOW_SCAN,
               window_scan_kernel<<<(unsigned)witems.size(), WIN_THREADS, WIN_SMEM, st>>>(d_witems, d_agg, d_prefix));
    ZTS_LAUNCH(ctx, ZK_WINDOW_RESOLVE,
               window_resolve_kernel<<<(unsigned)runs.size(), WIN_THREADS, WIN_SMEM, st>>>(arena, d_scratch, d_pieces, d_runs,
                                                                                            d_prefix, d_fail));
    std::vector<uint32_t> fail(wk.size());
    ZTS_CUDA(ctx, cudaMemcpyAsync(fail.data(), d_fail, wk.size() * 4, cudaMemcpyDeviceToHost, st));
    ZTS_CUDA(ctx, cudaStreamSynchronize(st));
    for (size_t i = 0; i < wk.size(); ++i) {
        if (fail[i]) continue;  // a byte before the start of the stream
        h_results[job.big[wk[i]]] = split_finish(job, wk[i], &wres[wfirst[i]], gath);
        done[job.big[wk[i]]] = 1;
    }
    return ZLB_OK;
}

// The pieces of the job's large items (job.first / job.seg): one marker scan per item (queued back to back, one
// read-back for all), a piece starting at 0 and behind every marker that leaves at least one byte. An item with a
// stretch longer than SPLIT_SEARCH_GAP between its start, markers and end is searched instead (sjob, in bits): every
// such stretch gets a nominal cut every SPLIT_SEARCH_STEP bytes, the block finder runs on all of them in one launch,
// and its proposals join the markers as cuts. Items whose pieces are all shorter keep the marker route (no finder
// launch when no item is searched). An item goes to one of the two jobs or to neither (no cut inside); the other job
// lists no pieces for it. A piece's out_off / out_cap are 0. < 0 on API errors.
#define SPLIT_TAG_SHIFT 40  // marks carry the item's index above the byte offset (offsets < 1 TiB, < 16 M large items)
// Far above the longest piece this engine's own streams have (a 64 KiB chunk, at most 64 KiB + 5 bytes compressed),
// and above the pieces of streams flushed at least every 1 MiB of input (zlib Z_SYNC_FLUSH / Z_FULL_FLUSH, pigz): all
// of those keep the marker route, which already decodes their pieces side by side. A stretch this long holds dozens
// of blocks of any encoder.
#define SPLIT_SEARCH_GAP (1u << 20)
// Nominal cut spacing of a searched stretch, about one cut per zlib block (16 K symbols at its default memLevel,
// ~15-30 KB compressed). Chosen on a B200 at 1000 W (profiles/r03d_split_step.json, both builds in one session, 256 MiB
// through zlib -6, decompressed GB/s): 32 KiB against 16 KiB gave mixed 9.4 / 9.2, text 9.2 / 7.8, random data
// 15.7 / 9.3. A finer step finds more block starts (mixed: 6338 against 3863), but each costs the finder a search up
// to the next block, many cuts of text land on the same block (3118 starts from 5826 cuts), and every piece costs the
// size and window passes a table build and a 64 KiB map. 64 KiB was measured with the finder alone (finder_step in
// profiles/r03d_split_search.json): it halves the block starts found again (1931 on mixed), which lengthens the
// longest piece. (-DSPLIT_SEARCH_STEP=... builds another step for such a comparison.)
#ifndef SPLIT_SEARCH_STEP
#define SPLIT_SEARCH_STEP (32u << 10)
#endif
static int split_layout(zlb_ctx* ctx, const uint8_t* d_in, SplitJob& job, SplitJob& sjob)
{
    const size_t nb = job.big.size();
    if (nb >= (1ull << 24)) return ZLB_OK;
    cudaStream_t st = ctx->stream;
    int rc = zts_reserve(ctx, &ctx->d_misc, (size_t)SPLIT_MAX_MARKS * 8 + 256);
    if (rc) return rc;
    unsigned long long* d_marks = (unsigned long long*)((uint8_t*)ctx->d_misc.p + 256);
    uint32_t* d_count = (uint32_t*)ctx->d_misc.p;
    ZTS_CUDA(ctx, cudaMemsetAsync(d_count, 0, 4, st));
    for (size_t k = 0; k < nb; ++k) {
        const zlb_item& it = job.items[job.big[k]];
        if (it.in_len >= (1ull << SPLIT_TAG_SHIFT)) continue;
        const unsigned grid = (unsigned)((it.in_len / 16 + 255) / 256 + 1);
        ZTS_LAUNCH(ctx, ZK_MARKER_SCAN,
                   marker_scan_kernel<<<grid, 256, 0, st>>>(d_in + it.in_off, it.in_len, d_marks, d_count, SPLIT_MAX_MARKS,
                                                           (unsigned long long)k << SPLIT_TAG_SHIFT));
    }
    uint32_t count = 0;
    ZTS_CUDA(ctx, cudaMemcpyAsync(&count, d_count, 4, cudaMemcpyDeviceToHost, st));
    ZTS_CUDA(ctx, cudaStreamSynchronize(st));
    if (count > SPLIT_MAX_MARKS) return ZLB_OK;
    std::vector<unsigned long long> marks(count);
    if (count) {
        ZTS_CUDA(ctx, cudaMemcpyAsync(marks.data(), d_marks, (size_t)count * 8, cudaMemcpyDeviceToHost, st));
        ZTS_CUDA(ctx, cudaStreamSynchronize(st));
    }
    std::sort(marks.begin(), marks.end());  // by item, then by offset
    // marker cuts of every item (byte offsets from its start, 0 first); the searched items get nominal cuts
    std::vector<std::vector<unsigned long long>> cuts(nb);
    std::vector<char> searched(nb, 0);
    std::vector<ZtsFindCut> find;
    std::vector<size_t> find_first(nb + 1, 0);
    size_t mi = 0;
    for (size_t k = 0; k < nb; ++k) {
        const zlb_item& it = job.items[job.big[k]];
        std::vector<unsigned long long>& c = cuts[k];
        find_first[k] = find.size();
        if (it.in_len >= (1ull << SPLIT_TAG_SHIFT)) continue;
        c.push_back(0);
        for (; mi < marks.size() && (marks[mi] >> SPLIT_TAG_SHIFT) == k; ++mi) {
            const unsigned long long m = marks[mi] & ((1ull << SPLIT_TAG_SHIFT) - 1);
            // a piece of this engine's streams holds a whole block: never closer than SPLIT_MIN_PIECE bytes to the
            // previous cut (a hostile stream of empty stored blocks would otherwise ask for a slot per 5 bytes)
            if (m < it.in_len && m >= c.back() + SPLIT_MIN_PIECE) c.push_back(m);
        }
        for (size_t j = 0; j < c.size(); ++j) {
            const unsigned long long g0 = c[j], g1 = j + 1 < c.size() ? c[j + 1] : it.in_len;
            if (g1 - g0 <= SPLIT_SEARCH_GAP) continue;
            searched[k] = 1;
            const unsigned long long base = 8ull * it.in_off;
            for (unsigned long long p = g0 + SPLIT_SEARCH_STEP; p < g1; p += SPLIT_SEARCH_STEP)
                find.push_back({base + 8 * p, base + 8 * std::min(p + SPLIT_SEARCH_STEP, g1), base + 8 * it.in_len});
        }
    }
    find_first[nb] = find.size();
    std::vector<unsigned long long> found(find.size());
    if ((rc = block_find(ctx, d_in, find, found.data()))) return rc;
    job.first.assign(nb + 1, 0);
    sjob.first.assign(nb + 1, 0);
    for (size_t k = 0; k < nb; ++k) {
        const zlb_item& it = job.items[job.big[k]];
        job.first[k] = job.seg.size();
        sjob.first[k] = sjob.seg.size();
        if (cuts[k].size() < (searched[k] ? 1u : 2u)) continue;  // no marker inside: nothing to gain
        if (!searched[k]) {
            for (unsigned long long m : cuts[k]) job.seg.push_back({it.in_off + m, 0, 0, 0});
            job.seg.back().in_len = it.in_len - cuts[k].back();
            for (size_t j = job.first[k]; j + 1 < job.seg.size(); ++j) job.seg[j].in_len = job.seg[j + 1].in_off - job.seg[j].in_off;
            continue;
        }
        // bit offsets: the markers' and the finder's proposals, in order, each at least SPLIT_MIN_PIECE bytes behind
        // the one in front
        const unsigned long long b0 = 8ull * it.in_off, b1 = 8ull * (it.in_off + it.in_len);
        std::vector<unsigned long long> bc;
        for (unsigned long long m : cuts[k]) bc.push_back(b0 + 8 * m);
        for (size_t f = find_first[k]; f < find_first[k + 1]; ++f)
            if (found[f] != FIND_NONE && found[f] > b0 && found[f] < b1) bc.push_back(found[f]);
        std::sort(bc.begin(), bc.end());
        std::vector<zlb_item>& seg = sjob.seg;
        const size_t a = seg.size();
        for (unsigned long long x : bc)
            if (seg.size() == a || x >= seg.back().in_off + 8ull * SPLIT_MIN_PIECE) seg.push_back({x, 0, 0, 0});
        if (seg.size() - a < 2) {
            seg.resize(a);
            continue;
        }
        for (size_t j = a; j < seg.size(); ++j) seg[j].in_len = (j + 1 < seg.size() ? seg[j + 1].in_off : b1) - seg[j].in_off;
    }
    job.first[nb] = job.seg.size();
    sjob.first[nb] = sjob.seg.size();
    return ZLB_OK;
}

// Decodes the job's large items piecewise, all of them in one pass: one segment-mode launch over the pieces of every
// item, one window-mode pass for the items whose pieces reach into their predecessors, one gather. An item that
// worked gets its result in h_results and done set; the others have to go through the serial decoder. < 0 on API
// errors.
static int inflate_split_batch(zlb_ctx* ctx, const uint8_t* d_in, uint8_t* d_out, const uint8_t* d_dict, SplitJob& job,
                               uint32_t flags, zlb_result* h_results, std::vector<char>& done)
{
    const size_t nb = job.big.size(), np = job.seg.size();
    cudaStream_t st = ctx->stream;
    // slots: a piece of L compressed bytes cannot inflate to more than ~1032 L (258 bytes per 2 bits at best), and a
    // piece of this engine's streams holds at most one 64 KiB chunk
    size_t scratch = 0, big_in = 0;
    for (size_t k = 0; k < nb; ++k)
        if (job.pieces(k)) big_in += job.items[job.big[k]].in_len;
    for (zlb_item& s : job.seg) {
        size_t slot = (size_t)s.in_len * 1032u + 512u;
        if (slot > SPLIT_SLOT) slot = SPLIT_SLOT;
        slot = (slot + 255) & ~(size_t)255;
        s.out_off = scratch;
        s.out_cap = slot;
        scratch += slot;
    }
    const size_t need = ((scratch + 255) & ~(size_t)255) + np * (sizeof(zlb_item) + sizeof(zlb_result) + sizeof(ZtsGather)) + 1024;
    if (need > SplitBudget(ctx->d_split)(big_in, 1)) return ZLB_OK;
    bool got = false;
    int rc = split_reserve(ctx, &ctx->d_split, need, &got);
    if (rc || !got) return rc;
    uint8_t* d_scratch = (uint8_t*)ctx->d_split.p;
    zlb_item* d_seg = (zlb_item*)(d_scratch + ((scratch + 255) & ~(size_t)255));
    zlb_result* d_segres = (zlb_result*)(d_seg + np);
    ZtsGather* d_gather = (ZtsGather*)(d_segres + np);
    std::vector<zlb_result> sres;
    if ((rc = split_segments<INF_BYTES>(ctx, d_in, d_scratch, job.seg, d_seg, d_segres, flags, sres))) return rc;
    // validate every item's chain of pieces; the valid ones are gathered in one launch, together with those that
    // window mode decodes
    std::vector<ZtsGather> gath;
    std::vector<size_t> window;
    for (size_t k = 0; k < nb; ++k) {
        const size_t a = job.first[k], n = job.pieces(k);
        if (n < 2) continue;
        const int chain = split_chain(&sres[a], &job.seg[a], n, true, job.dicts && job.dicts[job.big[k]].len);
        if (chain == SPLIT_WINDOW) window.push_back(k);
        if (chain != SPLIT_OK) continue;
        h_results[job.big[k]] = split_finish(job, k, &sres[a], gath);
        done[job.big[k]] = 1;
    }
    if (!window.empty()) {
        rc = inflate_split_window(ctx, d_in, d_scratch, d_dict, job, flags, window, h_results, done, gath);
        if (rc) return rc;
    }
    if (!gath.empty()) {
        ZTS_CUDA(ctx, cudaMemcpyAsync(d_gather, gath.data(), gath.size() * sizeof(ZtsGather), cudaMemcpyHostToDevice, st));  // <= np entries
        ZTS_LAUNCH(ctx, ZK_GATHER, segment_gather_kernel<<<(unsigned)gath.size(), 256, 0, st>>>(d_scratch, d_out, d_gather));
        ZTS_CUDA(ctx, cudaStreamSynchronize(st));  // gath goes out of scope
    }
    return ZLB_OK;
}

// Whether the segment-mode size results sres of item big[k]'s pieces reach no further than the output of the pieces
// in front of each plus the dictionary's reachable bytes (crc32: how far a piece reached in front of its first byte):
// the one-warp decoder's own condition, so it then fails no distance either.
static bool split_reach_ok(const SplitJob& job, size_t k, const std::vector<zlb_result>& sres)
{
    const size_t a = job.first[k], n = job.pieces(k);
    const unsigned long long dl = job.dicts ? std::min(job.dicts[job.big[k]].len, (uint64_t)WIN_WORDS) : 0;
    unsigned long long before = 0;  // output of the pieces in front
    for (size_t j = a; j < a + n; ++j) {
        if (sres[j].crc32 > before + dl) return false;
        before += sres[j].out_len;
    }
    return true;
}

// An item of a size call is settled when its chain passes and no piece reaches too far (split_reach_ok); it then gets
// the one-warp decoder's result by construction.
static void split_settle_sizes(const SplitJob& job, const std::vector<zlb_result>& sres, zlb_result* h_results,
                               std::vector<char>& done)
{
    for (size_t k = 0; k < job.big.size(); ++k) {
        const size_t a = job.first[k], n = job.pieces(k);
        if (n < 2 || split_chain(&sres[a], &job.seg[a], n, false, false) != SPLIT_OK) continue;
        if (!split_reach_ok(job, k, sres)) continue;
        h_results[job.big[k]] = split_result(job, k, &sres[a]);
        done[job.big[k]] = 1;
    }
}

// The marker split of a size call: the job's pieces are sized by one segment-mode launch of the size decoder. A
// piece's size does not depend on the bytes in front of it, only whether a distance reaches before the stream (or
// before its dictionary) does, and a piece tells how far in front of its first byte it reached (crc32). No byte slots
// and no window scratch: the piece tables take the place of the marks. h_results / done as for inflate_split_batch.
static int inflate_split_sizes(zlb_ctx* ctx, const uint8_t* d_in, const SplitJob& job, uint32_t flags,
                               zlb_result* h_results, std::vector<char>& done)
{
    const size_t np = job.seg.size();
    int rc = zts_reserve(ctx, &ctx->d_misc, np * (sizeof(zlb_item) + sizeof(zlb_result)) + 256);
    if (rc) return rc;
    zlb_item* d_seg = (zlb_item*)ctx->d_misc.p;
    std::vector<zlb_result> sres;
    if ((rc = split_segments<INF_SIZE>(ctx, d_in, nullptr, job.seg, d_seg, (zlb_result*)(d_seg + np), flags, sres))) return rc;
    split_settle_sizes(job, sres, h_results, done);
    return ZLB_OK;
}

// ---- the searched split: size first, then window ----------------------------------------------------------------
// Almost every piece of a searched item reaches into its predecessor, so there is no byte-slot pass: the size decoder
// runs over the pieces in segment mode (the chain check, and each piece's exact output size), broken chains are
// repaired, and the window pass decodes the pieces into exact slots.
#define SPLIT_REPAIR_ROUNDS 3

// Sizes the pieces of sjob; res = their results. Where a chain breaks, each maximal run of broken pieces is merged with
// the piece behind it (a cut the piece in front did not end at is dropped) and only the merged pieces are sized again,
// for at most SPLIT_REPAIR_ROUNDS rounds. A chain that reaches a clean BFINAL before its last piece is kept up to that
// piece: the one-warp decoder stops there too. On return every item left with pieces passes split_chain; the others
// have none (the one-warp decoder takes them).
static int split_search_size(zlb_ctx* ctx, const uint8_t* d_in, SplitJob& job, uint32_t flags, std::vector<zlb_result>& res)
{
    const size_t nb = job.big.size();
    res.assign(job.seg.size(), zlb_result());
    std::vector<size_t> todo(job.seg.size());
    for (size_t j = 0; j < todo.size(); ++j) todo[j] = j;
    for (int round = 0;; ++round) {
        if (!todo.empty()) {
            std::vector<zlb_item> part(todo.size());
            for (size_t t = 0; t < todo.size(); ++t) part[t] = job.seg[todo[t]];
            int rc = zts_reserve(ctx, &ctx->d_misc, part.size() * (sizeof(zlb_item) + sizeof(zlb_result)) + 256);
            if (rc) return rc;
            zlb_item* d_seg = (zlb_item*)ctx->d_misc.p;
            std::vector<zlb_result> pres;
            rc = split_segments<INF_SIZE>(ctx, d_in, nullptr, part, d_seg, (zlb_result*)(d_seg + part.size()), flags, pres,
                                          true);
            if (rc) return rc;
            for (size_t t = 0; t < todo.size(); ++t) res[todo[t]] = pres[t];
        }
        todo.clear();
        std::vector<zlb_item> nseg;
        std::vector<zlb_result> nres;
        std::vector<size_t> nfirst(nb + 1, 0);
        for (size_t k = 0; k < nb; ++k) {
            const size_t a = job.first[k], n = job.pieces(k);
            nfirst[k] = nseg.size();
            if (n < 2) continue;
            const zlb_item* g = &job.seg[a];
            const zlb_result* r = &res[a];
            auto fin = [&](size_t j) { return r[j].status == ZLB_ST_OK && (r[j].blocks & 0x80000000u); };
            auto good = [&](size_t j) {
                return r[j].status == ZLB_ST_OK && (j + 1 == n ? fin(j) : !fin(j) && r[j].in_used == g[j].in_len);
            };
            size_t ok = 0;  // pieces in front that are good
            while (ok < n && good(ok)) ++ok;
            if (ok == n || (ok < n && fin(ok))) {  // the whole chain, or up to a clean BFINAL
                const size_t keep = ok == n ? n : ok + 1;
                nseg.insert(nseg.end(), g, g + keep);
                nres.insert(nres.end(), r, r + keep);
                continue;
            }
            if (round == SPLIT_REPAIR_ROUNDS) continue;
            bool progress = false;
            const size_t b0 = nseg.size();
            for (size_t j = 0; j < n;) {
                if (good(j)) {
                    nseg.push_back(g[j]);
                    nres.push_back(r[j]);
                    ++j;
                    continue;
                }
                size_t e = j;
                while (e + 1 < n && !good(e + 1)) ++e;
                const size_t last = std::min(e + 1, n - 1);  // the run and the piece behind it
                progress |= last > j;
                nseg.push_back({g[j].in_off, g[last].in_off + g[last].in_len - g[j].in_off, 0, 0});
                nres.push_back(zlb_result());
                todo.push_back(nseg.size() - 1);
                j = last + 1;
            }
            if (!progress || nseg.size() - b0 < 2) {  // nothing left to merge, or one piece: the one-warp decoder
                while (!todo.empty() && todo.back() >= b0) todo.pop_back();
                nseg.resize(b0);
                nres.resize(b0);
            }
        }
        nfirst[nb] = nseg.size();
        job.seg.swap(nseg);
        job.first.swap(nfirst);
        res.swap(nres);
        if (todo.empty()) return ZLB_OK;
    }
}

// The decode of the searched items, sized by split_search_size (res): exact byte slots, the window pass, one gather.
// An item whose pieces do not fit ZtsWinPiece's 32-bit sizes, or whose scratch exceeds the budget, is left to the
// one-warp decoder; one whose output exceeds its slot gets ZLB_ST_OUT_OVERFLOW without a decode, but only when no
// distance reaches before the stream or its dictionary (split_reach_ok) -- the one-warp decoder would stop at such a
// distance with ZLB_ST_BAD_CODE if it came before the slot filled, so such an item is left to it.
static int inflate_split_search(zlb_ctx* ctx, const uint8_t* d_in, uint8_t* d_out, const uint8_t* d_dict, SplitJob& job,
                                const std::vector<zlb_result>& res, uint32_t flags, zlb_result* h_results,
                                std::vector<char>& done)
{
    cudaStream_t st = ctx->stream;
    std::vector<ZtsGather> gath;
    std::vector<size_t> cand;
    size_t scratch = 0, big_in = 0;
    for (size_t k = 0; k < job.big.size(); ++k) {
        const size_t a = job.first[k], n = job.pieces(k);
        if (n < 2) continue;
        unsigned long long total = 0;
        bool fits = true;
        for (size_t j = a; j < a + n; ++j) {
            total += res[j].out_len;
            fits &= res[j].out_len <= 0xFFFFFF00ull;
        }
        if (!fits) continue;
        if (total > job.items[job.big[k]].out_cap) {
            if (!split_reach_ok(job, k, res)) continue;
            std::vector<ZtsGather> none;
            h_results[job.big[k]] = split_finish(job, k, &res[a], none);
            done[job.big[k]] = 1;
            continue;
        }
        for (size_t j = a; j < a + n; ++j) {
            job.seg[j].out_off = scratch;
            job.seg[j].out_cap = (res[j].out_len + 255) & ~255ull;
            scratch += job.seg[j].out_cap;
        }
        big_in += job.items[job.big[k]].in_len;
        cand.push_back(k);
    }
    if (cand.empty()) return ZLB_OK;
    const size_t np = job.seg.size();
    const size_t need = scratch + np * sizeof(ZtsGather) + 256;
    if (need > SplitBudget(ctx->d_split)(big_in, 1)) return ZLB_OK;
    bool got = false;
    int rc = split_reserve(ctx, &ctx->d_split, need, &got);
    if (rc || !got) return rc;
    uint8_t* d_scratch = (uint8_t*)ctx->d_split.p;
    ZtsGather* d_gather = (ZtsGather*)(d_scratch + scratch);
    if ((rc = inflate_split_window(ctx, d_in, d_scratch, d_dict, job, flags, cand, h_results, done, gath))) return rc;
    if (!gath.empty()) {
        ZTS_CUDA(ctx, cudaMemcpyAsync(d_gather, gath.data(), gath.size() * sizeof(ZtsGather), cudaMemcpyHostToDevice, st));
        ZTS_LAUNCH(ctx, ZK_GATHER, segment_gather_kernel<<<(unsigned)gath.size(), 256, 0, st>>>(d_scratch, d_out, d_gather));
        ZTS_CUDA(ctx, cudaStreamSynchronize(st));  // gath goes out of scope
    }
    return ZLB_OK;
}

// A "_host" call without a split, in waves; the tables are queued on ctx->stream already. The input of wave k+1 travels
// on a copy stream while wave k is decoded, and as soon as the sizes of wave k are known (its results are read back
// behind it, wave k+1 is already queued) what it wrote travels back on the other copy stream. The waves are launched
// on up to four compute streams in turn: a stream is decoded by one warp from start to end (milliseconds, whatever the
// batch size), so waves that do not fill the device by themselves run side by side, staggered by their input copies,
// and their outputs leave as each one finishes; waves that do fill it simply take over the SMs as their predecessor
// drains.
static int inflate_waves(zlb_ctx* ctx, const uint8_t* d_in, uint8_t* d_out, const uint8_t* d_dict, const zlb_item* d_items,
                         const zlb_dict* d_dicts, zlb_result* d_results, const zlb_item* h_items, zlb_result* h_results,
                         size_t n, uint32_t flags, uint32_t kinds, const ZtsHostIO& hio)
{
    // waves only pay when the items are laid out in order on both sides (then a wave is one contiguous copy each way)
    size_t n_waves = 1;
    if (n >= 1024) {
        n_waves = n >= 32768 ? 16 : n >= 16384 ? 8 : 4;  // (the last wave's output travels alone: keep it small)
        for (size_t i = 1; i < n && n_waves > 1; ++i)
            if (h_items[i].in_off < h_items[i - 1].in_off + h_items[i - 1].in_len ||
                h_items[i].out_off < h_items[i - 1].out_off + h_items[i - 1].out_cap)
                n_waves = 1;
    }
    int rc = zts_host_streams(ctx);
    if (rc) return rc;
    rc = zts_reserve_pinned(ctx, &ctx->h_pin2, n * sizeof(zlb_result));
    if (rc) return rc;
    zlb_result* pin_res = (zlb_result*)ctx->h_pin2.p;
    const size_t per = (n + n_waves - 1) / n_waves;
    // events: 0 = item table on the device; 1 + 2k = input of wave k arrived; 2 + 2k = wave k decoded, results read back
    cudaEvent_t ev_tab = zts_sync_event(ctx, 0);
    ZTS_CUDA(ctx, cudaEventRecord(ev_tab, ctx->stream));
    auto wave_range = [&](size_t k, size_t& a, size_t& b) {
        a = k * per;
        b = a + per < n ? a + per : n;
        if (a > n) a = n;
    };
    auto wave_in = [&](size_t k) -> int {
        size_t a, b;
        wave_range(k, a, b);
        if (a < b) {
            uint64_t ilo, ihi;
            if (n_waves == 1) {  // items in any order: the whole blob
                ilo = 0;
                ihi = hio.in_bytes;
            } else {
                ilo = h_items[a].in_off;
                ihi = h_items[b - 1].in_off + h_items[b - 1].in_len;
            }
            if (ihi > ilo) {
                zts_stage_wait_in(hio.stage, ilo, ihi);
                ZTS_CUDA(ctx, cudaMemcpyAsync((void*)(d_in + ilo), hio.h_in + ilo, ihi - ilo, cudaMemcpyHostToDevice, ctx->s_in));
            }
        }
        ZTS_CUDA(ctx, cudaEventRecord(zts_sync_event(ctx, 1 + 2 * k), ctx->s_in));
        return ZLB_OK;
    };
    const bool trace = getenv("ZTS_TRACE_WAVES") != nullptr;  // development aid: when does the host see each wave
    const auto t_begin = std::chrono::steady_clock::now();
    auto wave_out = [&](size_t k) -> int {
        size_t a, b;
        wave_range(k, a, b);
        ZTS_CUDA(ctx, cudaEventSynchronize(zts_sync_event(ctx, 2 + 2 * k)));
        if (trace)
            fprintf(stderr, "inflate wave %zu of %zu decoded at %.2f ms\n", k, n_waves,
                    std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count());
        if (a >= b) return ZLB_OK;
        // The results are read back only now, on a stream of their own: a copy queued behind a kernel that is still
        // running holds up every later copy of its direction (the copy engine serves its queue in order), and the
        // outputs of the earlier waves would wait for the last wave's kernel.
        ZTS_CUDA(ctx, cudaMemcpyAsync(pin_res + a, d_results + a, (b - a) * sizeof(zlb_result), cudaMemcpyDeviceToHost, ctx->s_res));
        ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->s_res));
        memcpy(h_results + a, pin_res + a, (b - a) * sizeof(zlb_result));
        return zts_copy_back(ctx, hio.stage, ctx->s_out, d_out, hio.h_out, h_items, h_results, d_items, d_results, a, b);
    };
    if ((rc = wave_in(0))) return rc;
    for (size_t k = 0; k < n_waves; ++k) {
        size_t a, b;
        wave_range(k, a, b);
        // checksums are computed on the context's stream (their tables are staged there): then every wave runs on it
        cudaStream_t st = (kinds || k % 4 == 0) ? ctx->stream : ctx->s_aux[k % 4 - 1];
        if (st != ctx->stream && k < 4) ZTS_CUDA(ctx, cudaStreamWaitEvent(st, ev_tab, 0));  // the item table
        ZTS_CUDA(ctx, cudaStreamWaitEvent(st, zts_sync_event(ctx, 1 + 2 * k), 0));
        if (a < b) {
            ctx->work = st;
            rc = inflate_launch(ctx, st, d_in, d_out, d_items + a, d_results + a, b - a, flags, d_dicts ? d_dicts + a : nullptr,
                                d_dict);
            ctx->work = ctx->stream;
            if (rc) return rc;
            if (kinds) {
                rc = zts_checksum_device(ctx, d_out, d_items + a, d_results + a, h_items + a, b - a, kinds, 1);
                if (rc) return rc;
            }
        }
        ZTS_CUDA(ctx, cudaEventRecord(zts_sync_event(ctx, 2 + 2 * k), st));
        if (k + 1 < n_waves && (rc = wave_in(k + 1))) return rc;  // behind the launches: may wait for the copy threads
    }
    // the call ends on ctx->stream -- joined only here: a join inside the loop would make the next wave queued on
    // ctx->stream wait for the waves in flight on the other streams
    for (size_t k = 0; k < n_waves; ++k)
        if (!(kinds || k % 4 == 0)) ZTS_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, zts_sync_event(ctx, 2 + 2 * k), 0));
    // every wave is queued (none waits for the host): their outputs leave in order, each as soon as its wave is done
    for (size_t k = 0; k < n_waves; ++k)
        if ((rc = wave_out(k))) return rc;
    ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->s_out));
    if (trace)
        fprintf(stderr, "inflate outputs back at %.2f ms\n",
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count());
    return ZLB_OK;
}

// Decodes n items on device buffers; results land in h_results after the final synchronise. The item table goes to the
// device with the dictionary table beside it. With ZLB_INFLATE_SPLIT the large items are cut at markers (split_layout)
// and tried piecewise first (inflate_split_batch), which settles some of them in h_results and in the mask `done`;
// the items left go through one decoder launch, over a compacted table when the split settled any.
// Then one tail: checksums, the result read-back and, on a "_host" call, the copy-back of the outputs. A "_host" call
// without a split runs in waves instead (inflate_waves).
// d_dict / h_dicts: the preset dictionaries (h_dicts == NULL: none; checked by the caller)
// d_out == NULL: a size call (zlb_inflate_size_batch). The same route with the size decoder, the split's sizing stage
// (inflate_split_sizes) and no checksums (refused by the caller); nothing is written, d_dict is not read, a "_host"
// call copies its input over in one piece and nothing back.
// sink (zlb_inflate_index, no dictionaries): the split's routes report the piece starts of the items they decode,
// and the items left go through INF_POINTS instead of the plain decoder (never in waves); without a sink the call
// launches what it launched before.
static int inflate_device(zlb_ctx* ctx, const uint8_t* d_in, uint8_t* d_out, const uint8_t* d_dict,
                          const zlb_dict* h_dicts, const zlb_item* h_items, zlb_result* h_results, size_t n, uint32_t flags,
                          const ZtsHostIO* hio, ZtsIndexSink* sink = nullptr)
{
    // large items that may be cut at sync-flush markers (each is massively parallel by itself)
    flags &= ~ZLB_INFLATE_BITS;  // (internal)
    SplitJob job{h_items, h_dicts, {}, {}, {}};
    job.sink = sink;
    if (sink)
        for (size_t i = 0; i < n; ++i) sink->count[i] = 0;
    if ((flags & ZLB_INFLATE_SPLIT) && !(flags & ZLB_INFLATE_SEGMENT))
        for (size_t i = 0; i < n; ++i)
            if (h_items[i].in_len >= SPLIT_MIN_BYTES) job.big.push_back(i);
    // d_items holds the call's per-item tables: items | dictionaries, and with a split the same for the items left
    const size_t row = sizeof(zlb_item) + (h_dicts ? sizeof(zlb_dict) : 0);
    int rc = zts_reserve(ctx, &ctx->d_items, (job.big.empty() ? 1 : 2) * n * row + 64);
    if (rc) return rc;
    rc = zts_reserve(ctx, &ctx->d_results, n * sizeof(zlb_result) + 64);
    if (rc) return rc;
    auto upload = [&](size_t at, const zlb_item* items, const zlb_dict* dicts, size_t m, zlb_item*& d_it,
                      zlb_dict*& d_di) -> int {
        d_it = (zlb_item*)((uint8_t*)ctx->d_items.p + at);
        d_di = dicts ? (zlb_dict*)(d_it + m) : nullptr;
        ZTS_CUDA(ctx, cudaMemcpyAsync(d_it, items, m * sizeof(zlb_item), cudaMemcpyHostToDevice, ctx->stream));
        if (dicts) ZTS_CUDA(ctx, cudaMemcpyAsync(d_di, dicts, m * sizeof(zlb_dict), cudaMemcpyHostToDevice, ctx->stream));
        return ZLB_OK;
    };
    zlb_item* d_items;
    zlb_dict* d_dicts;
    if ((rc = upload(0, h_items, h_dicts, n, d_items, d_dicts))) return rc;
    zlb_result* d_results = (zlb_result*)ctx->d_results.p;
    ZTS_CUDA(ctx, cudaMemsetAsync(d_results, 0, n * sizeof(zlb_result), ctx->stream));
    uint32_t kinds = 0;
    if (flags & ZLB_INFLATE_WANT_CRC32) kinds |= ZLB_SUM_CRC32;
    if (flags & ZLB_INFLATE_WANT_ADLER32) kinds |= ZLB_SUM_ADLER32;
    const bool sizes = d_out == nullptr;
    if (hio && job.big.empty() && !sizes && !sink)
        return inflate_waves(ctx, d_in, d_out, d_dict, d_items, d_dicts, d_results, h_items, h_results, n, flags, kinds, *hio);

    // the split: the items it decodes get their results in h_results; when it decoded any, rest lists the others
    zlb_item* d_rest = d_items;
    zlb_dict* d_rest_dicts = d_dicts;
    size_t m = n;
    bool split_any = false;
    std::vector<size_t> rest;
    std::vector<zlb_item> rest_items;
    std::vector<zlb_dict> rest_dicts;
    if (hio) {  // (a "_host" call that does not run in waves: its whole input first)
        zts_stage_wait_in(hio->stage, 0, hio->in_bytes);
        ZTS_CUDA(ctx, cudaMemcpyAsync((void*)d_in, hio->h_in, hio->in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    if (!job.big.empty()) {
        std::vector<char> done(n, 0);
        SplitJob sjob{h_items, h_dicts, job.big, {}, {}, true, sink};  // the searched items
        rc = split_layout(ctx, d_in, job, sjob);
        if (!rc && !job.seg.empty())
            rc = sizes ? inflate_split_sizes(ctx, d_in, job, flags, h_results, done)
                       : inflate_split_batch(ctx, d_in, d_out, d_dict, job, flags, h_results, done);
        if (!rc && !sjob.seg.empty()) {
            std::vector<zlb_result> sres;
            rc = split_search_size(ctx, d_in, sjob, flags, sres);
            if (!rc && sizes) split_settle_sizes(sjob, sres, h_results, done);
            if (!rc && !sizes) rc = inflate_split_search(ctx, d_in, d_out, d_dict, sjob, sres, flags, h_results, done);
        }
        if (rc) return rc;
        split_any = std::find(done.begin(), done.end(), 1) != done.end();
        if (split_any) {
            for (size_t i = 0; i < n; ++i)
                if (!done[i]) {
                    rest.push_back(i);
                    rest_items.push_back(h_items[i]);
                    if (h_dicts) rest_dicts.push_back(h_dicts[i]);
                }
            m = rest.size();
            if ((rc = upload(n * row, rest_items.data(), h_dicts ? rest_dicts.data() : nullptr, m, d_rest, d_rest_dicts)))
                return rc;
        }
    }
    // the items left, in one launch; after a split their results come back to the host, join the split's there, and
    // the whole table goes to d_results in one copy (the checksums read out_len from it)
    // (with a sink: the launched items' slots, compacted, in ctx->d_misc; read back behind the results)
    std::vector<unsigned long long> pt_first, pt_count;
    std::vector<zlb_point> pts;
    if (m && sink) {
        pt_first.assign(m + 1, 0);
        for (size_t j = 0; j < m; ++j) {
            const size_t i = split_any ? rest[j] : j;
            pt_first[j + 1] = pt_first[j] + (sink->first[i + 1] - sink->first[i]);
        }
        pts.resize(pt_first[m]);
        pt_count.resize(m);
        rc = zts_reserve(ctx, &ctx->d_misc, (2 * m + 1) * 8 + pts.size() * sizeof(zlb_point) + 256);
        if (rc) return rc;
        ZtsPointSink ds;
        ds.first = (const unsigned long long*)ctx->d_misc.p;
        ds.count = (unsigned long long*)ctx->d_misc.p + m + 1;
        ds.points = (zlb_point*)(ds.count + m);
        ds.spacing = sink->spacing;
        ZTS_CUDA(ctx, cudaMemcpyAsync((void*)ds.first, pt_first.data(), (m + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
        rc = inflate_launch_mode<INF_POINTS>(ctx, ctx->stream, d_in, d_out, d_rest, d_results, m, flags, nullptr, nullptr, ds);
        if (rc) return rc;
        ZTS_CUDA(ctx, cudaMemcpyAsync(pt_count.data(), ds.count, m * 8, cudaMemcpyDeviceToHost, ctx->stream));
        if (!pts.empty())
            ZTS_CUDA(ctx, cudaMemcpyAsync(pts.data(), ds.points, pts.size() * sizeof(zlb_point), cudaMemcpyDeviceToHost, ctx->stream));
    } else if (m) {
        rc = inflate_launch(ctx, ctx->stream, d_in, d_out, d_rest, d_results, m, flags, d_rest_dicts, d_dict);
        if (rc) return rc;
    }
    if (split_any) {
        std::vector<zlb_result> rr(m);
        ZTS_CUDA(ctx, cudaMemcpyAsync(rr.data(), d_results, m * sizeof(zlb_result), cudaMemcpyDeviceToHost, ctx->stream));
        ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        for (size_t j = 0; j < m; ++j) h_results[rest[j]] = rr[j];
        ZTS_CUDA(ctx, cudaMemcpyAsync(d_results, h_results, n * sizeof(zlb_result), cudaMemcpyHostToDevice, ctx->stream));
    }
    if (kinds) {
        rc = zts_checksum_device(ctx, d_out, d_items, d_results, h_items, n, kinds, 1);
        if (rc) return rc;
    }
    ZTS_CUDA(ctx, cudaMemcpyAsync(h_results, d_results, n * sizeof(zlb_result), cudaMemcpyDeviceToHost, ctx->stream));
    if (!pt_first.empty()) {  // the one-warp items' points, for those that decoded
        ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        for (size_t j = 0; j < m; ++j) {
            const size_t i = split_any ? rest[j] : j;
            if (h_results[i].status != ZLB_ST_OK) continue;
            for (unsigned long long c = 0; c < pt_count[j]; ++c) {
                zlb_point p = pts[pt_first[j] + c];
                p.win_off = index_win_off(h_items[i], p.out_pos);
                sink->points[sink->first[i] + c] = p;
            }
            sink->count[i] = pt_count[j];
        }
    }
    if (hio && !sizes) {
        ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // the sizes decide what travels
        rc = zts_copy_back(ctx, hio->stage, ctx->stream, d_out, hio->h_out, h_items, h_results, d_items, d_results, 0, n);
        if (rc) return rc;
    }
    return ZLB_OK;
}

extern "C" int zlb_inflate_batch_dict(zlb_ctx* ctx, const void* d_in, void* d_out, const void* d_dict,
                                      const zlb_dict* dicts, const zlb_item* items, zlb_result* results, size_t n,
                                      uint32_t flags)
{
    bool any = false;
    int rc = zts_entry_begin(ctx, (d_in && d_out) || !n, items, results, n, 0x7FFFFFFFull, d_dict, SIZE_MAX, dicts, &any);
    if (rc) return rc > 0 ? ZLB_OK : rc;
    rc = inflate_device(ctx, (const uint8_t*)d_in, (uint8_t*)d_out, (const uint8_t*)d_dict, any ? dicts : nullptr, items,
                        results, n, flags, nullptr);
    if (rc) return rc;
    ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ZLB_OK;
}

extern "C" int zlb_inflate_batch(zlb_ctx* ctx, const void* d_in, void* d_out, const zlb_item* items,
                                 zlb_result* results, size_t n, uint32_t flags)
{
    return zlb_inflate_batch_dict(ctx, d_in, d_out, nullptr, nullptr, items, results, n, flags);
}

extern "C" int zlb_inflate_batch_dict_host(zlb_ctx* ctx, const void* h_in, size_t in_bytes, void* h_out,
                                           size_t out_bytes, const void* h_dict, size_t dict_bytes,
                                           const zlb_dict* dicts, const zlb_item* items, zlb_result* results, size_t n,
                                           uint32_t flags)
{
    return zts_host_call(ctx, h_in, in_bytes, h_out, out_bytes, h_dict, dict_bytes, dicts, items, results, n,
                         0x7FFFFFFFull, [&](ZtsHostIO& io, const zlb_dict* d) {
        return inflate_device(ctx, (const uint8_t*)ctx->d_stage_in.p, (uint8_t*)ctx->d_stage_out.p,
                              (const uint8_t*)ctx->d_dict.p, d, items, results, n, flags, &io);
    });
}

extern "C" int zlb_inflate_batch_host(zlb_ctx* ctx, const void* h_in, size_t in_bytes, void* h_out, size_t out_bytes,
                                      const zlb_item* items, zlb_result* results, size_t n, uint32_t flags)
{
    return zlb_inflate_batch_dict_host(ctx, h_in, in_bytes, h_out, out_bytes, nullptr, 0, nullptr, items, results, n,
                                       flags);
}

// the refusals of a size call, with a text: an input buffer is needed whenever there are items, checksums cannot be
// computed without the bytes
static int size_flags_check(zlb_ctx* ctx, bool in_ok, uint32_t flags)
{
    if (!ctx) return ZLB_E_ARG;
    if (!in_ok) return zts_fail(ctx, ZLB_E_ARG, "the input buffer is NULL");
    if (flags & (ZLB_INFLATE_WANT_CRC32 | ZLB_INFLATE_WANT_ADLER32))
        return zts_fail(ctx, ZLB_E_ARG, "a size call computes no checksums (ZLB_INFLATE_WANT_CRC32 / _ADLER32)");
    return ZLB_OK;
}

extern "C" int zlb_inflate_size_batch(zlb_ctx* ctx, const void* d_in, const zlb_dict* dicts, const zlb_item* items,
                                      zlb_result* results, size_t n, uint32_t flags)
{
    int rc = size_flags_check(ctx, d_in || !n, flags);
    if (rc) return rc;
    bool any = false;
    rc = zts_entry_begin(ctx, true, items, results, n, 0x7FFFFFFFull, nullptr, SIZE_MAX, dicts, &any, true);
    if (rc) return rc > 0 ? ZLB_OK : rc;
    rc = inflate_device(ctx, (const uint8_t*)d_in, nullptr, nullptr, any ? dicts : nullptr, items, results, n, flags,
                        nullptr);
    if (rc) return rc;
    ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ZLB_OK;
}

extern "C" int zlb_inflate_size_batch_host(zlb_ctx* ctx, const void* h_in, size_t in_bytes, const zlb_dict* dicts,
                                           const zlb_item* items, zlb_result* results, size_t n, uint32_t flags)
{
    const int rc = size_flags_check(ctx, h_in || !n, flags);
    if (rc) return rc;
    return zts_host_call(ctx, h_in, in_bytes, nullptr, 0, nullptr, 0, dicts, items, results, n, 0x7FFFFFFFull,
                         [&](ZtsHostIO& io, const zlb_dict* d) {
        return inflate_device(ctx, (const uint8_t*)ctx->d_stage_in.p, nullptr, nullptr, d, items, results, n, flags, &io);
    }, ZTS_HOST_SIZES);
}

extern "C" int zlb_debug_block_starts(zlb_ctx* ctx, const void* d_in, uint64_t n, const uint64_t* h_cuts, size_t n_cuts,
                                      uint64_t span, uint64_t* h_bits_out)
{
    if (!ctx || (n_cuts && (!d_in || !h_cuts || !h_bits_out)) || n_cuts >= (1ull << 32)) return ZLB_E_ARG;
    ZTS_CUDA(ctx, cudaSetDevice(ctx->device));
    std::vector<ZtsFindCut> cuts(n_cuts);
    for (size_t c = 0; c < n_cuts; ++c) {
        if (h_cuts[c] >= n) return zts_fail(ctx, ZLB_E_ARG, "cut %zu lies behind the input", c);
        cuts[c] = {8 * h_cuts[c], std::min(8 * h_cuts[c] + span, 8 * n), 8 * n};
    }
    static_assert(sizeof(unsigned long long) == sizeof(uint64_t), "");
    return block_find(ctx, (const uint8_t*)d_in, cuts, (unsigned long long*)h_bits_out);
}

// ---- random access: an index of access points ------------------------------------------------------------------
#define ZTS_INDEX_FLAGS (ZLB_INFLATE_WANT_CRC32 | ZLB_INFLATE_WANT_ADLER32 | ZLB_INFLATE_CHECK_NLEN)

static int index_check(zlb_ctx* ctx, uint32_t flags, const zlb_point* points, const uint64_t* first, const uint64_t* count,
                       size_t n)
{
    if (!ctx) return ZLB_E_ARG;
    if (flags & ~ZTS_INDEX_FLAGS)
        return zts_fail(ctx, ZLB_E_ARG, "an index build takes ZLB_INFLATE_WANT_CRC32 / _ADLER32 / _CHECK_NLEN only");
    if (!n) return ZLB_OK;
    if (!first || !count) return zts_fail(ctx, ZLB_E_ARG, "point_first / point_count is NULL");
    for (size_t i = 0; i < n; ++i)
        if (first[i + 1] < first[i]) return zts_fail(ctx, ZLB_E_ARG, "point_first decreases at item %zu", i);
    if (first[n] > first[0] && !points) return zts_fail(ctx, ZLB_E_ARG, "the point table is NULL");
    return ZLB_OK;
}

extern "C" int zlb_inflate_index(zlb_ctx* ctx, const void* d_in, void* d_out, const zlb_item* items, zlb_result* results,
                                 size_t n, uint32_t flags, uint64_t spacing, zlb_point* points, const uint64_t* point_first,
                                 uint64_t* point_count)
{
    int rc = index_check(ctx, flags, points, point_first, point_count, n);
    if (rc) return rc;
    bool any = false;
    rc = zts_entry_begin(ctx, (d_in && d_out) || !n, items, results, n, 0x7FFFFFFFull, nullptr, SIZE_MAX, nullptr, &any);
    if (rc) return rc > 0 ? ZLB_OK : rc;
    ZtsIndexSink sink{spacing ? spacing : ZLB_INDEX_DEFAULT_SPACING, points, point_first, point_count};
    rc = inflate_device(ctx, (const uint8_t*)d_in, (uint8_t*)d_out, nullptr, nullptr, items, results, n,
                        flags | ZLB_INFLATE_SPLIT, nullptr, &sink);
    if (rc) return rc;
    ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ZLB_OK;
}

extern "C" int zlb_inflate_index_host(zlb_ctx* ctx, const void* h_in, size_t in_bytes, void* h_out, size_t out_bytes,
                                      const zlb_item* items, zlb_result* results, size_t n, uint32_t flags, uint64_t spacing,
                                      zlb_point* points, const uint64_t* point_first, uint64_t* point_count)
{
    const int rc = index_check(ctx, flags, points, point_first, point_count, n);
    if (rc) return rc;
    ZtsIndexSink sink{spacing ? spacing : ZLB_INDEX_DEFAULT_SPACING, points, point_first, point_count};
    return zts_host_call(ctx, h_in, in_bytes, h_out, out_bytes, nullptr, 0, nullptr, items, results, n, 0x7FFFFFFFull,
                         [&](ZtsHostIO& io, const zlb_dict*) {
        return inflate_device(ctx, (const uint8_t*)ctx->d_stage_in.p, (uint8_t*)ctx->d_stage_out.p, nullptr, nullptr, items,
                              results, n, flags | ZLB_INFLATE_SPLIT, &io, &sink);
    });
}

// The checks of a ranges call, with a text. in_bytes / win_bytes / out_bytes == SIZE_MAX: device buffers, whose sizes
// are not known; win_given: the window blob is not NULL. A stream's points (pt_first, pt_count, in_len) are checked
// once per call however many ranges name them.
static int ranges_check(zlb_ctx* ctx, const zlb_point* points, size_t n_points, const zlb_range* ranges, size_t n,
                        uint32_t flags, size_t in_bytes, size_t win_bytes, size_t out_bytes, bool win_given)
{
    if (flags & ~ZTS_INDEX_FLAGS)
        return zts_fail(ctx, ZLB_E_ARG, "a ranges call takes ZLB_INFLATE_WANT_CRC32 / _ADLER32 / _CHECK_NLEN only");
    if (n && !points) return zts_fail(ctx, ZLB_E_ARG, "the point table is NULL");
    std::set<std::array<uint64_t, 3>> checked;
    for (size_t i = 0; i < n; ++i) {
        const zlb_range& r = ranges[i];
        if (in_bytes != SIZE_MAX && (r.in_off > in_bytes || r.in_len > in_bytes - r.in_off))
            return zts_fail(ctx, ZLB_E_ARG, "range %zu: its stream lies outside the input", i);
        if (r.in_len >= (1ull << 60) || r.in_off >= (1ull << 60))
            return zts_fail(ctx, ZLB_E_ARG, "range %zu: its stream lies beyond 2^60 bytes", i);  // (bit offsets fit)
        if (out_bytes != SIZE_MAX && (r.out_off > out_bytes || r.out_cap > out_bytes - r.out_off))
            return zts_fail(ctx, ZLB_E_ARG, "range %zu: its slot lies outside the output", i);
        if (r.pos > UINT64_MAX - r.out_cap) return zts_fail(ctx, ZLB_E_ARG, "range %zu: pos + out_cap overflows", i);
        if (!checked.insert({r.pt_first, r.pt_count, r.in_len}).second) continue;
        if (r.pt_count == 0) return zts_fail(ctx, ZLB_E_ARG, "range %zu has no access points", i);
        if (r.pt_first > n_points || r.pt_count > n_points - r.pt_first)
            return zts_fail(ctx, ZLB_E_ARG, "range %zu: its points lie outside the point table", i);
        const zlb_point* p = points + r.pt_first;
        if (p[0].in_bit || p[0].out_pos) return zts_fail(ctx, ZLB_E_ARG, "range %zu: its first point is not {0, 0}", i);
        for (uint64_t k = 0; k < r.pt_count; ++k) {
            if (k && (p[k].in_bit <= p[k - 1].in_bit || p[k].out_pos <= p[k - 1].out_pos))
                return zts_fail(ctx, ZLB_E_ARG, "range %zu: its points do not ascend (point %llu)", i, (unsigned long long)k);
            if (p[k].in_bit >= 8 * r.in_len)
                return zts_fail(ctx, ZLB_E_ARG, "range %zu: point %llu lies behind the stream", i, (unsigned long long)k);
            const uint64_t wl = std::min(p[k].out_pos, (uint64_t)WIN_WORDS);
            if (wl && !win_given)
                return zts_fail(ctx, ZLB_E_ARG, "range %zu: point %llu has a window but the window blob is NULL", i,
                                (unsigned long long)k);
            if (win_bytes != SIZE_MAX && (p[k].win_off > win_bytes || wl > win_bytes - p[k].win_off))
                return zts_fail(ctx, ZLB_E_ARG, "range %zu: the window of point %llu lies outside the window blob", i,
                                (unsigned long long)k);
        }
    }
    return ZLB_OK;
}

// A piece of a range: one warp from one point. The first piece of a range that starts behind its point decodes the
// `skip` bytes in front of pos as well, into scratch; the others decode into the range's slot.
struct ZtsRangePiece {
    size_t range;
    unsigned long long skip, want;  // bytes in front of pos; bytes of the range it is to give
    zlb_item item;                  // bits from the input's first byte; out_off: a device address
    zlb_dict win;
};

// Output bytes a stream can still give from bit `in_bit` of its `in_len` bytes on: a match of at most 258 bytes takes
// at least two bits (a length and a distance code), a literal one, a stored byte eight; saturates.
static unsigned long long range_reach(const zlb_range& r, const zlb_point& p)
{
    const unsigned long long bits = 8 * r.in_len - p.in_bit;
    return bits > ULLONG_MAX / 258 ? ULLONG_MAX : 258 * bits;
}

// The reads of zlb_inflate_ranges[_host] on device buffers: pieces planned here, INF_RANGE over a wave of them per
// launch (a wave's scratch within SplitBudget), the gather of the first pieces, then the results, the checksum tail and
// on a "_host" call the copy-back. h_results is final on return. A range whose pos lies beyond what the stream can give
// from the point in front of it gets no piece (out_len 0); a first piece whose scratch -- the bytes in front of pos
// plus its part, at most what the stream can give -- exceeds the budget by itself fails the call with ZLB_E_NOMEM.
static int ranges_device(zlb_ctx* ctx, const uint8_t* d_in, const uint8_t* d_win, uint8_t* d_out, const zlb_point* points,
                         const zlb_range* ranges, zlb_result* h_results, size_t n, uint32_t flags, const ZtsHostIO* hio)
{
    cudaStream_t st = ctx->stream;
    const size_t budget = SplitBudget(ctx->d_split).device;
    std::vector<ZtsRangePiece> pieces;
    for (size_t i = 0; i < n; ++i) {
        const zlb_range& r = ranges[i];
        const zlb_point* p = points + r.pt_first;
        const unsigned long long end = r.pos + r.out_cap;  // (no overflow: ranges_check)
        // the last point at or before pos, then every point inside [pos, end)
        size_t j = std::upper_bound(p, p + r.pt_count, r.pos, [](unsigned long long v, const zlb_point& q) { return v < q.out_pos; }) - p - 1;
        if (r.pos - p[j].out_pos >= range_reach(r, p[j])) continue;  // past the end of the stream: no byte to give
        for (bool first = true; r.out_cap && j < r.pt_count && (first || p[j].out_pos < end); ++j, first = false) {
            const unsigned long long from = std::max((unsigned long long)r.pos, (unsigned long long)p[j].out_pos);
            const unsigned long long to = j + 1 < r.pt_count ? std::min(end, (unsigned long long)p[j + 1].out_pos) : end;
            ZtsRangePiece q;
            q.range = i;
            q.skip = from - p[j].out_pos;
            q.want = to - from;
            q.item = {8 * r.in_off + p[j].in_bit, 8 * r.in_len - p[j].in_bit, (uintptr_t)(d_out + r.out_off + (from - r.pos)),
                      std::min(q.skip + q.want, range_reach(r, p[j]))};
            q.win = {p[j].win_off, std::min(p[j].out_pos, (uint64_t)WIN_WORDS)};
            if (q.skip && q.item.out_cap > budget)
                return zts_fail(ctx, ZLB_E_NOMEM,
                                "range %zu: %llu bytes in front of pos would be decoded into scratch, more than the %zu a "
                                "call may take: pass the access points between",
                                i, q.skip, budget);
            pieces.push_back(q);
        }
    }
    const size_t np = pieces.size();
    int rc = zts_reserve(ctx, &ctx->d_items, (n + np) * sizeof(zlb_item) + np * (sizeof(zlb_dict) + sizeof(ZtsGather)) + 256);
    if (rc) return rc;
    rc = zts_reserve(ctx, &ctx->d_results, std::max(n, np) * sizeof(zlb_result) + 64);
    if (rc) return rc;
    zlb_item* d_slots = (zlb_item*)ctx->d_items.p;
    zlb_item* d_pitems = d_slots + n;
    zlb_dict* d_pwin = (zlb_dict*)(d_pitems + np);
    ZtsGather* d_gather = (ZtsGather*)(d_pwin + np);
    zlb_result* d_results = (zlb_result*)ctx->d_results.p;
    std::vector<zlb_result> pres(np);
    // waves: pieces in order, a new wave where the first pieces' scratch would exceed the budget (a piece's scratch is
    // at most the budget, so the rounding below cannot wrap)
    std::vector<unsigned long long> soff(np, 0);
    for (size_t a = 0; a < np;) {
        size_t b = a, scratch = 0;
        for (; b < np; ++b) {
            if (!pieces[b].skip) continue;
            const size_t s = (pieces[b].item.out_cap + 255) & ~(size_t)255;
            if (scratch && scratch + s > budget) break;
            soff[b] = scratch;
            scratch += s;
        }
        if (scratch) {
            bool got = false;
            if ((rc = split_reserve(ctx, &ctx->d_split, scratch, &got))) return rc;
            if (!got) return zts_fail(ctx, ZLB_E_NOMEM, "no device memory for %zu bytes of range scratch", scratch);
        }
        std::vector<zlb_item> it(b - a);
        std::vector<zlb_dict> win(b - a);
        for (size_t k = a; k < b; ++k) {
            it[k - a] = pieces[k].item;
            if (pieces[k].skip) it[k - a].out_off = (uintptr_t)ctx->d_split.p + soff[k];
            win[k - a] = pieces[k].win;
        }
        ZTS_CUDA(ctx, cudaMemcpyAsync(d_pitems + a, it.data(), (b - a) * sizeof(zlb_item), cudaMemcpyHostToDevice, st));
        ZTS_CUDA(ctx, cudaMemcpyAsync(d_pwin + a, win.data(), (b - a) * sizeof(zlb_dict), cudaMemcpyHostToDevice, st));
        ZTS_CUDA(ctx, cudaMemsetAsync(d_results, 0, (b - a) * sizeof(zlb_result), st));
        // (the slots' out_off are device addresses: the output base is NULL)
        rc = inflate_launch_mode<INF_RANGE>(ctx, st, d_in, nullptr, d_pitems + a, d_results, b - a,
                                            (flags & ZLB_INFLATE_CHECK_NLEN) | ZLB_INFLATE_BITS, d_pwin + a, d_win);
        if (rc) return rc;
        ZTS_CUDA(ctx, cudaMemcpyAsync(pres.data() + a, d_results, (b - a) * sizeof(zlb_result), cudaMemcpyDeviceToHost, st));
        ZTS_CUDA(ctx, cudaStreamSynchronize(st));
        std::vector<ZtsGather> gath;
        for (size_t k = a; k < b; ++k) {
            const ZtsRangePiece& q = pieces[k];
            if (q.skip && pres[k].out_len > q.skip)
                gath.push_back({soff[k] + q.skip, ranges[q.range].out_off, pres[k].out_len - q.skip});
        }
        if (!gath.empty()) {
            ZTS_CUDA(ctx, cudaMemcpyAsync(d_gather, gath.data(), gath.size() * sizeof(ZtsGather), cudaMemcpyHostToDevice, st));
            ZTS_LAUNCH(ctx, ZK_GATHER, segment_gather_kernel<<<(unsigned)gath.size(), 256, 0, st>>>(
                                           (const uint8_t*)ctx->d_split.p, d_out, d_gather));
            ZTS_CUDA(ctx, cudaStreamSynchronize(st));  // gath goes out of scope, the next wave reuses the scratch
        }
        a = b;
    }
    // a range's result: its pieces in order, up to the first that failed or came short (the stream ended there)
    for (size_t i = 0; i < n; ++i) memset(&h_results[i], 0, sizeof(zlb_result));
    std::vector<char> closed(n, 0);
    for (size_t k = 0; k < np; ++k) {
        const ZtsRangePiece& q = pieces[k];
        if (closed[q.range]) continue;
        zlb_result& o = h_results[q.range];
        const unsigned long long got = pres[k].out_len > q.skip ? pres[k].out_len - q.skip : 0;
        o.out_len += std::min(got, q.want);
        if (pres[k].status != ZLB_ST_OK) o.status = pres[k].status;
        if (pres[k].status != ZLB_ST_OK || got < q.want) closed[q.range] = 1;
    }
    std::vector<zlb_item> slots(n);
    for (size_t i = 0; i < n; ++i) slots[i] = {ranges[i].in_off, ranges[i].in_len, ranges[i].out_off, ranges[i].out_cap};
    ZTS_CUDA(ctx, cudaMemcpyAsync(d_slots, slots.data(), n * sizeof(zlb_item), cudaMemcpyHostToDevice, st));
    ZTS_CUDA(ctx, cudaMemcpyAsync(d_results, h_results, n * sizeof(zlb_result), cudaMemcpyHostToDevice, st));
    uint32_t kinds = 0;
    if (flags & ZLB_INFLATE_WANT_CRC32) kinds |= ZLB_SUM_CRC32;
    if (flags & ZLB_INFLATE_WANT_ADLER32) kinds |= ZLB_SUM_ADLER32;
    if (kinds) {
        rc = zts_checksum_device(ctx, d_out, d_slots, d_results, slots.data(), n, kinds, 1);
        if (rc) return rc;
        ZTS_CUDA(ctx, cudaMemcpyAsync(h_results, d_results, n * sizeof(zlb_result), cudaMemcpyDeviceToHost, st));
    }
    ZTS_CUDA(ctx, cudaStreamSynchronize(st));  // (slots goes out of scope; the copy-back needs the sizes)
    if (hio) return zts_copy_back(ctx, hio->stage, st, d_out, hio->h_out, slots.data(), h_results, d_slots, d_results, 0, n);
    return ZLB_OK;
}

extern "C" int zlb_inflate_ranges(zlb_ctx* ctx, const void* d_in, const void* d_win, void* d_out, const zlb_point* points,
                                  size_t n_points, const zlb_range* ranges, zlb_result* results, size_t n, uint32_t flags)
{
    if (!ctx || (n && (!d_in || !d_out || !ranges || !results))) return ZLB_E_ARG;
    int rc = ranges_check(ctx, points, n_points, ranges, n, flags, SIZE_MAX, SIZE_MAX, SIZE_MAX, d_win != nullptr);
    if (rc || !n) return rc;
    ZTS_CUDA(ctx, cudaSetDevice(ctx->device));
    return ranges_device(ctx, (const uint8_t*)d_in, (const uint8_t*)d_win, (uint8_t*)d_out, points, ranges, results, n, flags,
                         nullptr);
}

extern "C" int zlb_inflate_ranges_host(zlb_ctx* ctx, const void* h_in, size_t in_bytes, const void* h_win, size_t win_bytes,
                                       void* h_out, size_t out_bytes, const zlb_point* points, size_t n_points,
                                       const zlb_range* ranges, zlb_result* results, size_t n, uint32_t flags)
{
    if (!ctx || (n && (!ranges || !results))) return ZLB_E_ARG;
    int rc = ranges_check(ctx, points, n_points, ranges, n, flags, in_bytes, win_bytes, out_bytes, h_win != nullptr);
    if (rc || !n) return rc;
    // the window blob travels the way a dictionary blob does (one table entry naming all of it)
    std::vector<zlb_item> slots(n);
    for (size_t i = 0; i < n; ++i) slots[i] = {ranges[i].in_off, ranges[i].in_len, ranges[i].out_off, ranges[i].out_cap};
    const std::vector<zlb_dict> whole(n, zlb_dict{0, win_bytes});
    return zts_host_call(ctx, h_in, in_bytes, h_out, out_bytes, h_win, win_bytes, whole.data(), slots.data(), results, n,
                         SIZE_MAX, [&](ZtsHostIO& io, const zlb_dict*) {
        zts_stage_wait_in(io.stage, 0, io.in_bytes);
        ZTS_CUDA(ctx, cudaMemcpyAsync(ctx->d_stage_in.p, io.h_in, io.in_bytes, cudaMemcpyHostToDevice, ctx->stream));
        return ranges_device(ctx, (const uint8_t*)ctx->d_stage_in.p, (const uint8_t*)ctx->d_dict.p,
                             (uint8_t*)ctx->d_stage_out.p, points, ranges, results, n, flags, &io);
    });
}
