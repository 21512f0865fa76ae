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
#include <cstddef>
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
// The dictionary arguments are read by INF_DICT only.
#define WIN_WORDS 32768u
enum { INF_BYTES = 0, INF_WINDOW = 1, INF_DICT = 2 };
template <int MODE>
__global__ void __launch_bounds__(INF_WARPS_PER_CTA * 32, INF_MIN_CTAS)
inflate_warp_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, const zlb_item* __restrict__ items,
                    zlb_result* __restrict__ results, uint32_t n_items, uint32_t flags,
                    const zlb_dict* __restrict__ dicts, const uint8_t* __restrict__ dict)
{
    using T = typename std::conditional<MODE == INF_WINDOW, uint16_t, uint8_t>::type;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const unsigned lane = zts_lane();
    const unsigned warp = threadIdx.x >> 5;
    InfWarpSmem* S = reinterpret_cast<InfWarpSmem*>(smem_raw) + warp;
    const uint32_t item = blockIdx.x * INF_WARPS_PER_CTA + warp;
    if (item >= n_items) return;

    const zlb_item it = items[item];
    const uint8_t* src = in + it.in_off;
    T* dst = reinterpret_cast<T*>(out + it.out_off);
    uint32_t reach = MODE == INF_WINDOW ? WIN_WORDS : 0u;  // how far a distance may reach in front of the output
    const uint8_t* dtail = nullptr;                       // INF_DICT: the `reach` bytes in front of the output
    if constexpr (MODE == INF_DICT) {
        const zlb_dict d = dicts[item];
        reach = d.len < WIN_WORDS ? (uint32_t)d.len : WIN_WORDS;
        dtail = dict + d.off + d.len - reach;
    }
    if constexpr (MODE == INF_WINDOW) {
        uint4* w = reinterpret_cast<uint4*>(dst - WIN_WORDS);  // (slots are 256-byte aligned)
        for (uint32_t i = lane; i < WIN_WORDS / 8; i += 32) {
            const uint32_t a = 0x80008000u | (8u * i) | ((8u * i + 1u) << 16);
            w[i] = make_uint4(a, a + 0x00020002u, a + 0x00040004u, a + 0x00060006u);
        }
        __syncwarp();
    }
    const unsigned long long in_bits = it.in_len * 8ull;
    const unsigned long long cap = it.out_cap;

    BitReader br;
    br.ring_s = (uint32_t)__cvta_generic_to_shared(S->ring);
    br_init(br, src, src + it.in_len, 0);

    unsigned long long op = 0;
    uint32_t status = ZLB_ST_OK;
    uint32_t blocks = 0;
    int have_fixed = 0;
    bool bfinal = false;

    while (!bfinal && status == ZLB_ST_OK) {
        // segment mode: a piece of a larger stream ends cleanly where a block ends and its input is used up
        if ((flags & ZLB_INFLATE_SEGMENT) && blocks > 0 && br_bits_used(br) == in_bits) break;
        br_refill(br);
        if (br_bits_used(br) + 3 > in_bits) {
            status = ZLB_ST_INPUT_BROKEN;
            break;
        }
        uint32_t hdr = br_take(br, 3);  // src/RawInflate.ts:146-152
        bfinal = hdr & 1u;
        uint32_t btype = hdr >> 1;
        blocks++;

        if (btype == 0) {
            // ---- stored block (src/RawInflate.ts:251-318): drop to the byte boundary, LEN, NLEN
            unsigned long long used = br_bits_used(br);
            unsigned long long byte_pos = (used + 7) >> 3;
            if (byte_pos + 4 > it.in_len) {
                // src/RawInflate.ts:266 (LEN) / :272 (NLEN): which of the two 16-bit fields is cut short
                status = byte_pos + 2 > it.in_len ? ZLB_ST_STORED_LEN : (ZLB_ST_STORED_LEN | (1u << 8));
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
            if (byte_pos + len > it.in_len) {
                status = ZLB_ST_INPUT_BROKEN;
                break;
            }
            if (op + len > cap) {
                status = ZLB_ST_OUT_OVERFLOW;
                break;
            }
            for (uint32_t k = lane; k < len; k += 32) dst[op + k] = src[byte_pos + k];
            op += len;
            br_init(br, src + byte_pos + len, src + it.in_len, (byte_pos + len) * 8ull);
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
                if (br_bits_used(br) > in_bits) status = inf_classify_cl(S, src, it.in_len, cl_pos);
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
        while (!eob && status == ZLB_ST_OK) {
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
                status = inf_classify_symbols(S, src, it.in_len, batch_pos);
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
            const bool over = mine && rel + len > room;
            const unsigned bad_mask = __ballot_sync(0xFFFFFFFFu, bad_dist || over);
            uint32_t nvalid = ntok;
            if (bad_mask) {
                nvalid = (uint32_t)__ffs((int)bad_mask) - 1u;
                const bool first_is_dist = __shfl_sync(0xFFFFFFFFu, (int)bad_dist, (int)nvalid) != 0;
                status = first_is_dist ? ZLB_ST_BAD_CODE : ZLB_ST_OUT_OVERFLOW;
            }
            const bool live = lane < nvalid;
            // -- literals: one store
            ZTS_ASSERT(!live || (op + rel + len <= cap && (!is_match || dist <= op + rel + reach)));
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
                const bool small = in_sub && len <= 8u && dist >= len && (MODE != INF_DICT || dist <= behind + rel);
                if (__any_sync(0xFFFFFFFFu, small)) {
                    // short non-overlapping matches: every lane copies its own, loads first, then stores
                    T v[8];
                    T* dp = bdst + rel;
                    const T* sp = dp - dist;
#pragma unroll
                    for (int k = 0; k < 8; ++k) v[k] = (small && (uint32_t)k < len) ? sp[k] : (T)0;
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                        if (small && (uint32_t)k < len) dp[k] = v[k];
                }
                unsigned big_mask = __ballot_sync(0xFFFFFFFFu, in_sub && !small);
                while (big_mask) {
                    const int j = __ffs((int)big_mask) - 1;
                    big_mask &= big_mask - 1;
                    const uint32_t jl = __shfl_sync(0xFFFFFFFFu, len, j);
                    const uint32_t jd = __shfl_sync(0xFFFFFFFFu, dist, j);
                    const uint32_t jr = __shfl_sync(0xFFFFFFFFu, rel, j);
                    T* o = bdst + jr;
                    const T* s0 = o - jd;
                    if (MODE == INF_DICT && jd > behind + jr) {
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
            __syncwarp();
        }
        if (status == ZLB_ST_OK && br_bits_used(br) > in_bits) status = ZLB_ST_INPUT_BROKEN;
    }

    if (lane == 0) {
        zlb_result r = results[item];
        r.status = status;
        r.blocks = blocks | ((flags & ZLB_INFLATE_SEGMENT) && bfinal ? 0x80000000u : 0u);  // segment mode: saw BFINAL
        r.out_len = op;
        r.in_used = (br_bits_used(br) + 7) >> 3;  // whole unread bytes are given back (:511-514)
        results[item] = r;
    }
}

template <int MODE>
static int inflate_launch_mode(zlb_ctx* ctx, cudaStream_t st, const uint8_t* d_in, uint8_t* d_out, const zlb_item* d_items,
                               zlb_result* d_results, size_t n, uint32_t flags, const zlb_dict* d_dicts,
                               const uint8_t* d_dict)
{
    const size_t smem = sizeof(InfWarpSmem) * INF_WARPS_PER_CTA;
    ZTS_CUDA(ctx, cudaFuncSetAttribute(inflate_warp_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    unsigned grid = (unsigned)((n + INF_WARPS_PER_CTA - 1) / INF_WARPS_PER_CTA);
    ZTS_LAUNCH(ctx, MODE == INF_WINDOW ? ZK_INFLATE_WINDOW : MODE == INF_DICT ? ZK_INFLATE_DICT : ZK_INFLATE,
               inflate_warp_kernel<MODE><<<grid, INF_WARPS_PER_CTA * 32, smem, st>>>(d_in, d_out, d_items, d_results,
                                                                                    (uint32_t)n, flags, d_dicts, d_dict));
    return ZLB_OK;
}
// the decoder: with a dictionary table (d_dicts[i] belongs to d_items[i]) the dictionary instantiation
static int inflate_launch(zlb_ctx* ctx, cudaStream_t st, const uint8_t* d_in, uint8_t* d_out, const zlb_item* d_items,
                          zlb_result* d_results, size_t n, uint32_t flags, const zlb_dict* d_dicts = nullptr,
                          const uint8_t* d_dict = nullptr)
{
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

struct SplitPiece {
    uint32_t item;  // index into big
    unsigned long long start;
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

// result of an item whose n pieces passed the checks; their bytes (r[j].out_len at scratch offset seg[j].out_off)
// are queued for the gather when they fit
static void split_finish(const zlb_item& it, const zlb_result* r, const zlb_item* seg, size_t n, unsigned long long last_start,
                         zlb_result& o, std::vector<ZtsGather>& gath)
{
    unsigned long long total = 0, blocks = 0;
    for (size_t j = 0; j < n; ++j) {
        total += r[j].out_len;
        blocks += r[j].blocks & 0x7FFFFFFFu;
    }
    o.status = total > it.out_cap ? ZLB_ST_OUT_OVERFLOW : ZLB_ST_OK;
    o.out_len = total > it.out_cap ? 0 : total;
    o.in_used = last_start + r[n - 1].in_used;
    o.blocks = (uint32_t)blocks;
    if (total <= it.out_cap && total) {
        unsigned long long at = 0;
        for (size_t j = 0; j < n; ++j) {
            if (r[j].out_len) gath.push_back({seg[j].out_off, it.out_off + at, r[j].out_len});
            at += r[j].out_len;
        }
    }
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

// Window mode for the items big[cand[*]] (pieces as laid out by inflate_split_batch, byte slots at seg[j].out_off of
// d_scratch): all of them in one decode launch and one scan; done[k] / res[k] / gath as there. h_dicts / d_dict: the
// preset dictionaries of h_items (NULL: none).
static int inflate_split_window(zlb_ctx* ctx, const uint8_t* d_in, uint8_t* d_scratch, const zlb_item* h_items,
                                const zlb_dict* h_dicts, const uint8_t* d_dict,
                                const std::vector<size_t>& big, uint32_t flags, const std::vector<SplitPiece>& pieces,
                                const std::vector<size_t>& first, const std::vector<zlb_item>& seg,
                                const std::vector<size_t>& cand, std::vector<zlb_result>& res, std::vector<char>& done,
                                std::vector<ZtsGather>& gath)
{
    cudaStream_t st = ctx->stream;
    // runs of about sqrt(n) pieces: the scan's depth is then about 3 sqrt(n) compositions
    auto run_len = [](size_t n) {
        size_t g = 8;
        while (g * g < n) ++g;
        return g;
    };
    const size_t map_b = (size_t)WIN_WORDS * 2;
    // arena: word slots (each behind its window) | aggregates | prefixes | items | results | pieces | runs | items | fail
    auto layout = [&](size_t words, size_t np, size_t nr, size_t ni, size_t* off) {
        off[0] = words;
        off[1] = off[0] + nr * map_b;
        off[2] = off[1] + nr * map_b;
        off[3] = off[2] + np * sizeof(zlb_item);
        off[4] = off[3] + np * sizeof(zlb_result);
        off[5] = off[4] + np * sizeof(ZtsWinPiece);
        off[6] = off[5] + nr * sizeof(ZtsWinRun);
        off[7] = off[6] + ni * sizeof(ZtsWinItem);
        return off[7] + ni * 4 + 256;
    };
    // The scratch is bounded like the byte slots', with three times their bound by input (two bytes per word, the
    // windows, the maps).
    const SplitBudget budget(ctx->d_window);
    std::vector<size_t> take;
    size_t words = 0, np = 0, nr = 0, in_b = 0, need = 0, off[8];
    for (size_t k : cand) {
        const size_t a = first[k], b = first[k + 1], n = b - a;
        size_t w = 0;
        for (size_t j = a; j < b; ++j) w += map_b + 2 * (size_t)seg[j].out_cap;  // (out_cap: a multiple of 256)
        const size_t g = run_len(n);
        const size_t need_k = layout(words + w, np + n, nr + (n + g - 1) / g, take.size() + 1, off);
        if (need_k > budget(in_b + h_items[big[k]].in_len, 3)) continue;
        take.push_back(k);
        words += w;
        np += n;
        nr += (n + g - 1) / g;
        in_b += h_items[big[k]].in_len;
        need = need_k;
    }
    if (take.empty()) return ZLB_OK;
    bool got = false;
    int rc = split_reserve(ctx, &ctx->d_window, need, &got);
    if (rc || !got) return rc;
    layout(words, np, nr, take.size(), off);
    uint8_t* arena = (uint8_t*)ctx->d_window.p;
    uint16_t* d_agg = (uint16_t*)(arena + off[0]);
    uint16_t* d_prefix = (uint16_t*)(arena + off[1]);
    zlb_item* d_wseg = (zlb_item*)(arena + off[2]);
    zlb_result* d_wres = (zlb_result*)(arena + off[3]);
    ZtsWinPiece* d_pieces = (ZtsWinPiece*)(arena + off[4]);
    ZtsWinRun* d_runs = (ZtsWinRun*)(arena + off[5]);
    ZtsWinItem* d_witems = (ZtsWinItem*)(arena + off[6]);
    uint32_t* d_fail = (uint32_t*)(arena + off[7]);
    // 1. every piece of those items in window mode, one launch
    std::vector<zlb_item> wseg;
    wseg.reserve(np);
    size_t at = 0;
    for (size_t k : take)
        for (size_t j = first[k]; j < first[k + 1]; ++j) {
            zlb_item w = seg[j];
            w.out_off = at + map_b;  // the window's words in front
            at += map_b + 2 * (size_t)seg[j].out_cap;
            wseg.push_back(w);
        }
    ZTS_CUDA(ctx, cudaMemcpyAsync(d_wseg, wseg.data(), np * sizeof(zlb_item), cudaMemcpyHostToDevice, st));
    ZTS_CUDA(ctx, cudaMemsetAsync(d_wres, 0, np * sizeof(zlb_result), st));
    rc = inflate_launch_mode<INF_WINDOW>(ctx, st, d_in, arena, d_wseg, d_wres, np,
                                         (flags & ZLB_INFLATE_CHECK_NLEN) | ZLB_INFLATE_SEGMENT, nullptr, nullptr);
    if (rc) return rc;
    std::vector<zlb_result> wres(np);
    ZTS_CUDA(ctx, cudaMemcpyAsync(wres.data(), d_wres, np * sizeof(zlb_result), cudaMemcpyDeviceToHost, st));
    ZTS_CUDA(ctx, cudaStreamSynchronize(st));
    // 2. the chain checks; the items that pass are resolved
    std::vector<ZtsWinPiece> wp;
    std::vector<ZtsWinRun> runs;
    std::vector<ZtsWinItem> witems;
    std::vector<size_t> wk, wfirst;  // per resolved item: its k, its first piece in wseg / wres
    for (size_t t = 0, wj = 0; t < take.size(); ++t) {
        const size_t k = take[t], a = first[k], n = first[k + 1] - a;
        const size_t w0 = wj;
        wj += n;
        if (split_chain(&wres[w0], &seg[a], n, false, false) != SPLIT_OK) continue;
        const size_t g = run_len(n);
        const zlb_dict d = h_dicts ? h_dicts[big[k]] : zlb_dict{0, 0};
        const uint32_t dl = d.len < WIN_WORDS ? (uint32_t)d.len : WIN_WORDS;
        witems.push_back({(uint32_t)runs.size(), (uint32_t)((n + g - 1) / g), dl ? d_dict + d.off + d.len - dl : nullptr, dl, 0u});
        for (size_t s = 0; s < n; s += g)
            runs.push_back({(uint32_t)(wp.size() + s), (uint32_t)std::min(g, n - s), (uint32_t)wk.size(), 0u});
        for (size_t j = 0; j < n; ++j)
            wp.push_back({wseg[w0 + j].out_off, seg[a + j].out_off, (uint32_t)wres[w0 + j].out_len, (uint32_t)seg[a + j].out_cap});
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
        const size_t k = wk[i], a = first[k], n = first[k + 1] - a;
        split_finish(h_items[big[k]], &wres[wfirst[i]], &seg[a], n, pieces[a + n - 1].start, res[k], gath);
        done[k] = 1;
    }
    return ZLB_OK;
}

// Tries to decode the items h_items[big[*]] piecewise, all of them in one pass: one marker scan per item (queued back
// to back, one read-back for all), one segment-mode launch over the pieces of every item, one window-mode pass for
// the items whose pieces reach into their predecessors, one gather. done[k] tells whether big[k] worked (then res[k]
// is filled); the others have to go through the serial decoder. < 0 on API errors.
#define SPLIT_TAG_SHIFT 40  // marks carry the item's index above the byte offset (offsets < 1 TiB, < 16 M large items)
static int inflate_split_batch(zlb_ctx* ctx, const uint8_t* d_in, uint8_t* d_out, const zlb_item* h_items,
                               const zlb_dict* h_dicts, const uint8_t* d_dict, const std::vector<size_t>& big,
                               uint32_t flags, std::vector<zlb_result>& res, std::vector<char>& done)
{
    const size_t nb = big.size();
    res.assign(nb, zlb_result());
    done.assign(nb, 0);
    for (size_t k = 0; k < nb; ++k) memset(&res[k], 0, sizeof(zlb_result));
    if (nb >= (1ull << 24)) return ZLB_OK;
    cudaStream_t st = ctx->stream;
    int rc = zts_reserve(ctx, &ctx->d_misc, (size_t)SPLIT_MAX_MARKS * 8 + 256);
    if (rc) return rc;
    unsigned long long* d_marks = (unsigned long long*)((uint8_t*)ctx->d_misc.p + 256);
    uint32_t* d_count = (uint32_t*)ctx->d_misc.p;
    ZTS_CUDA(ctx, cudaMemsetAsync(d_count, 0, 4, st));
    for (size_t k = 0; k < nb; ++k) {
        const zlb_item& it = h_items[big[k]];
        if (it.in_len >= (1ull << SPLIT_TAG_SHIFT)) continue;
        const unsigned grid = (unsigned)((it.in_len / 16 + 255) / 256 + 1);
        ZTS_LAUNCH(ctx, ZK_MARKER_SCAN,
                   marker_scan_kernel<<<grid, 256, 0, st>>>(d_in + it.in_off, it.in_len, d_marks, d_count, SPLIT_MAX_MARKS,
                                                           (unsigned long long)k << SPLIT_TAG_SHIFT));
    }
    uint32_t count = 0;
    ZTS_CUDA(ctx, cudaMemcpyAsync(&count, d_count, 4, cudaMemcpyDeviceToHost, st));
    ZTS_CUDA(ctx, cudaStreamSynchronize(st));
    if (count == 0 || count > SPLIT_MAX_MARKS) return ZLB_OK;
    std::vector<unsigned long long> marks(count);
    ZTS_CUDA(ctx, cudaMemcpyAsync(marks.data(), d_marks, (size_t)count * 8, cudaMemcpyDeviceToHost, st));
    ZTS_CUDA(ctx, cudaStreamSynchronize(st));
    std::sort(marks.begin(), marks.end());  // by item, then by offset
    // pieces of every item: it starts at 0 and behind every marker that leaves at least one byte
    std::vector<SplitPiece> pieces;
    std::vector<size_t> first(nb + 1, 0);  // pieces of item k: [first[k], first[k + 1])
    {
        size_t mi = 0;
        for (size_t k = 0; k < nb; ++k) {
            first[k] = pieces.size();
            const unsigned long long n = h_items[big[k]].in_len;
            pieces.push_back({(uint32_t)k, 0ull});
            for (; mi < marks.size() && (marks[mi] >> SPLIT_TAG_SHIFT) == k; ++mi) {
                const unsigned long long m = marks[mi] & ((1ull << SPLIT_TAG_SHIFT) - 1);
                // a piece of this engine's streams holds a whole block: never closer than SPLIT_MIN_PIECE bytes to the
                // previous cut (a hostile stream of empty stored blocks would otherwise ask for a slot per 5 bytes)
                if (m < n && m >= pieces.back().start + SPLIT_MIN_PIECE) pieces.push_back({(uint32_t)k, m});
            }
            if (pieces.size() - first[k] < 2) pieces.resize(first[k]);  // no marker inside: nothing to gain
        }
        first[nb] = pieces.size();
    }
    const size_t np = pieces.size();
    if (np == 0) return ZLB_OK;
    // slots: a piece of L compressed bytes cannot inflate to more than ~1032 L (258 bytes per 2 bits at best), and a
    // piece of this engine's streams holds at most one 64 KiB chunk
    std::vector<zlb_item> seg(np);
    size_t scratch = 0, big_in = 0;
    for (size_t k = 0; k < nb; ++k) {
        const zlb_item& it = h_items[big[k]];
        if (first[k + 1] > first[k]) big_in += it.in_len;
        for (size_t j = first[k]; j < first[k + 1]; ++j) {
            seg[j].in_off = it.in_off + pieces[j].start;
            seg[j].in_len = (j + 1 < first[k + 1] ? pieces[j + 1].start : it.in_len) - pieces[j].start;
            size_t slot = (size_t)seg[j].in_len * 1032u + 512u;
            if (slot > SPLIT_SLOT) slot = SPLIT_SLOT;
            slot = (slot + 255) & ~(size_t)255;
            seg[j].out_off = scratch;
            seg[j].out_cap = slot;
            scratch += slot;
        }
    }
    const size_t need = ((scratch + 255) & ~(size_t)255) + np * (sizeof(zlb_item) + sizeof(zlb_result) + sizeof(ZtsGather)) + 1024;
    if (need > SplitBudget(ctx->d_split)(big_in, 1)) return ZLB_OK;
    bool got = false;
    if ((rc = split_reserve(ctx, &ctx->d_split, need, &got)) || !got) return rc;
    uint8_t* d_scratch = (uint8_t*)ctx->d_split.p;
    zlb_item* d_seg = (zlb_item*)(d_scratch + ((scratch + 255) & ~(size_t)255));
    zlb_result* d_segres = (zlb_result*)(d_seg + np);
    ZtsGather* d_gather = (ZtsGather*)(d_segres + np);
    ZTS_CUDA(ctx, cudaMemcpyAsync(d_seg, seg.data(), np * sizeof(zlb_item), cudaMemcpyHostToDevice, st));
    ZTS_CUDA(ctx, cudaMemsetAsync(d_segres, 0, np * sizeof(zlb_result), st));
    rc = inflate_launch(ctx, st, d_in, d_scratch, d_seg, d_segres, np,
                        (flags & ZLB_INFLATE_CHECK_NLEN) | ZLB_INFLATE_SEGMENT);
    if (rc) return rc;
    std::vector<zlb_result> sres(np);
    ZTS_CUDA(ctx, cudaMemcpyAsync(sres.data(), d_segres, np * sizeof(zlb_result), cudaMemcpyDeviceToHost, st));
    ZTS_CUDA(ctx, cudaStreamSynchronize(st));
    // validate every item's chain of pieces; the valid ones are gathered in one launch, together with those that
    // window mode decodes
    std::vector<ZtsGather> gath;
    std::vector<size_t> window;
    for (size_t k = 0; k < nb; ++k) {
        const size_t a = first[k], b = first[k + 1];
        if (b - a < 2) continue;
        const int chain = split_chain(&sres[a], &seg[a], b - a, true, h_dicts && h_dicts[big[k]].len);
        if (chain == SPLIT_WINDOW) window.push_back(k);
        if (chain != SPLIT_OK) continue;
        split_finish(h_items[big[k]], &sres[a], &seg[a], b - a, pieces[b - 1].start, res[k], gath);
        done[k] = 1;
    }
    if (!window.empty()) {
        rc = inflate_split_window(ctx, d_in, d_scratch, h_items, h_dicts, d_dict, big, flags, pieces, first, seg, window, res,
                                  done, gath);
        if (rc) return rc;
    }
    if (!gath.empty()) {
        ZTS_CUDA(ctx, cudaMemcpyAsync(d_gather, gath.data(), gath.size() * sizeof(ZtsGather), cudaMemcpyHostToDevice, st));  // <= np entries
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
    rc = zts_reserve_pinned2(ctx, n * sizeof(zlb_result));
    if (rc) return rc;
    zlb_result* pin_res = (zlb_result*)ctx->h_pin2;
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
// device with the dictionary table beside it. With ZLB_INFLATE_SPLIT the large items are tried piecewise first
// (inflate_split_batch); the items left go through one decoder launch, over a compacted table when the split did some.
// Then one tail: checksums, the result read-back and, on a "_host" call, the copy-back of the outputs. A "_host" call
// without a split runs in waves instead (inflate_waves).
// d_dict / h_dicts: the preset dictionaries (h_dicts == NULL: none; checked by the caller)
static int inflate_device(zlb_ctx* ctx, const uint8_t* d_in, uint8_t* d_out, const uint8_t* d_dict,
                          const zlb_dict* h_dicts, const zlb_item* h_items, zlb_result* h_results, size_t n, uint32_t flags,
                          const ZtsHostIO* hio)
{
    // large items that may be cut at sync-flush markers (each is massively parallel by itself)
    std::vector<size_t> big;
    if ((flags & ZLB_INFLATE_SPLIT) && !(flags & ZLB_INFLATE_SEGMENT))
        for (size_t i = 0; i < n; ++i)
            if (h_items[i].in_len >= SPLIT_MIN_BYTES) big.push_back(i);
    // d_items holds the call's per-item tables: items | dictionaries, and with a split the same for the items left
    const size_t row = sizeof(zlb_item) + (h_dicts ? sizeof(zlb_dict) : 0);
    int rc = zts_reserve(ctx, &ctx->d_items, (big.empty() ? 1 : 2) * n * row + 64);
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
    if (hio && big.empty())
        return inflate_waves(ctx, d_in, d_out, d_dict, d_items, d_dicts, d_results, h_items, h_results, n, flags, kinds, *hio);

    // the split: the items it decodes get their results in h_results; when it decoded any, rest lists the others
    zlb_item* d_rest = d_items;
    zlb_dict* d_rest_dicts = d_dicts;
    size_t m = n;
    bool split_any = false;
    std::vector<size_t> rest;
    std::vector<zlb_item> rest_items;
    std::vector<zlb_dict> rest_dicts;
    if (!big.empty()) {
        if (hio) {
            zts_stage_wait_in(hio->stage, 0, hio->in_bytes);
            ZTS_CUDA(ctx, cudaMemcpyAsync((void*)d_in, hio->h_in, hio->in_bytes, cudaMemcpyHostToDevice, ctx->stream));
        }
        std::vector<zlb_result> bres;
        std::vector<char> bdone, done(n, 0);
        rc = inflate_split_batch(ctx, d_in, d_out, h_items, h_dicts, d_dict, big, flags, bres, bdone);
        if (rc) return rc;
        for (size_t k = 0; k < big.size(); ++k)
            if (bdone[k]) {
                done[big[k]] = 1;
                h_results[big[k]] = bres[k];
                split_any = true;
            }
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
    if (m) {
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
    if (hio) {
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
