// zts_checksum.cu -- parallel slice-and-combine CRC-32 / Adler-32 (replaces src/CRC32.ts:25-47 and
// src/Adler32.ts:28-48 at the container call sites listed in include/zlibts_b200.h).
//
// Both checksums are affine in the message, so an item is cut into slices (one CTA each), a slice
// into 256 right-aligned runs (one thread each, 16-byte vector loads), and the pieces are folded:
//   CRC register  state(A||B) = state(A) * x^(8|B|) mod P  xor  state(B)        (raw: init 0, no xorout)
//   Adler (a,b)   a = a_A + a_B ;  b = b_A + |B| * a_A + b_B                     (raw: s1 starts at 0)
// The init / xorout (CRC) and the initial s1 = 1 (Adler) are applied once per item at the end.
//
// HBM-bound: algorithmic bytes = N (each input byte read once), 12 bytes written per slice.
#include "zts_common.cuh"

#define ZTS_SUM_THREADS 256
#define ZTS_SUM_SLICE (256u * 1024u)  // bytes per CTA; run per thread = 1 KiB (<= 4 KiB keeps Adler in u32)
#define ADLER_MOD 65521u

struct ZtsSlice {
    uint32_t item;
    uint32_t index;  // slice number within the item
};

struct ZtsSlicePartial {
    uint32_t crc_raw;
    uint32_t a, b;  // Adler raw sums mod 65521
};

__host__ __device__ static inline uint32_t zts_gf2_mulmod(uint32_t a, uint32_t b)
{
    uint32_t p = 0;
    for (uint32_t m = 0x80000000u; m; m >>= 1) {
        if (a & m) p ^= b;
        b = (b & 1u) ? (b >> 1) ^ 0xEDB88320u : (b >> 1);
    }
    return p;
}

// x^(8*nbytes) mod P (reflected representation: x^0 = 0x80000000)
__host__ __device__ static inline uint32_t zts_xpow_bytes(uint64_t nbytes)
{
    uint32_t xp = 0x80000000u, sq = 0x00800000u;
    for (uint64_t n = nbytes; n; n >>= 1) {
        if (n & 1) xp = zts_gf2_mulmod(sq, xp);
        sq = zts_gf2_mulmod(sq, sq);
    }
    return xp;
}

// x^(-8*p) mod P for p = 0..15: the CRC-32 polynomial is primitive, ord(x) = 2^32 - 1.
__constant__ uint32_t c_xinv_bytes[16];
static uint32_t h_xinv_bytes[16];
static bool h_xinv_ready = false;

static uint32_t host_xpow_bits(uint64_t nbits)
{
    uint32_t xp = 0x80000000u, sq = 0x40000000u;  // x^1
    for (uint64_t n = nbits; n; n >>= 1) {
        if (n & 1) xp = zts_gf2_mulmod(sq, xp);
        sq = zts_gf2_mulmod(sq, sq);
    }
    return xp;
}

__device__ __forceinline__ uint32_t crc_step_word(uint32_t crc, uint32_t w, const uint32_t* __restrict__ tab)
{
    crc ^= w;
    crc = (crc >> 8) ^ tab[crc & 0xFF];
    crc = (crc >> 8) ^ tab[crc & 0xFF];
    crc = (crc >> 8) ^ tab[crc & 0xFF];
    crc = (crc >> 8) ^ tab[crc & 0xFF];
    return crc;
}

// One CTA per slice. Thread t owns the run [E-(T-t)R, E-(T-t-1)R) of the 16-byte-aligned envelope
// [.., E) of the slice; bytes outside the slice read as zero (leading zeros do not change a raw
// state; the <= 15 trailing pad bytes are divided out at the end).
__global__ void __launch_bounds__(ZTS_SUM_THREADS)
checksum_slices_kernel(const uint8_t* __restrict__ in, const zlb_item* __restrict__ items,
                       const zlb_result* __restrict__ results, int use_out_len,
                       const ZtsSlice* __restrict__ slices, ZtsSlicePartial* __restrict__ partials,
                       uint32_t kinds)
{
    __shared__ uint32_t s_tab[256];
    __shared__ uint32_t s_lvl[8];  // x^(8*R*2^k)
    __shared__ uint32_t s_wcrc[8], s_wa[8];
    __shared__ unsigned long long s_wb[8];

    const unsigned t = threadIdx.x;
    {  // CRC table, src/CRC32.ts:61-69
        uint32_t c = t;
#pragma unroll
        for (int j = 0; j < 8; ++j) c = (c & 1u) ? (0xEDB88320u ^ (c >> 1)) : (c >> 1);
        s_tab[t] = c;
    }
    const ZtsSlice sl = slices[blockIdx.x];
    const zlb_item it = items[sl.item];
    const uint64_t item_len = use_out_len ? results[sl.item].out_len : it.in_len;
    const uint64_t item_off = use_out_len ? it.out_off : it.in_off;
    const uint64_t s_begin = (uint64_t)sl.index * ZTS_SUM_SLICE;
    uint64_t s_len = item_len > s_begin ? item_len - s_begin : 0;
    if (s_len > ZTS_SUM_SLICE) s_len = ZTS_SUM_SLICE;

    const uint64_t abs_begin = (uint64_t)(uintptr_t)in + item_off + s_begin;
    const uint64_t abs_end = abs_begin + s_len;
    const uint64_t env_end = (abs_end + 15) & ~(uint64_t)15;
    const uint32_t pad = (uint32_t)(env_end - abs_end);
    // run length: multiple of 16 covering the slice with 256 runs
    uint32_t R = (uint32_t)((s_len + pad + ZTS_SUM_THREADS - 1) / ZTS_SUM_THREADS);
    R = (R + 15u) & ~15u;
    if (R == 0) R = 16;
    if (t == 0) {
        uint32_t c = zts_xpow_bytes(R);
        for (int k = 0; k < 8; ++k) {
            s_lvl[k] = c;
            c = zts_gf2_mulmod(c, c);
        }
    }
    __syncthreads();

    // my run, clipped to the slice
    const int64_t run_lo = (int64_t)env_end - (int64_t)(ZTS_SUM_THREADS - t) * R;
    const int64_t run_hi = run_lo + R;
    uint32_t crc = 0, a = 0, b = 0;
    if (run_hi > (int64_t)abs_begin) {
        // 16-byte vectors; [run_lo, run_hi) is 16-aligned at both ends
        for (int64_t p = run_lo; p < run_hi; p += 16) {
            if (p + 16 <= (int64_t)abs_begin) continue;  // entirely before the slice
            uint4 v = *reinterpret_cast<const uint4*>((uintptr_t)p);
            uint32_t w[4] = {v.x, v.y, v.z, v.w};
            if (p < (int64_t)abs_begin || p + 16 > (int64_t)abs_end) {
                // mask bytes outside [abs_begin, abs_end)
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    uint32_t m = 0;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        int64_t q = p + 4 * k + j;
                        if (q >= (int64_t)abs_begin && q < (int64_t)abs_end) m |= 0xFFu << (8 * j);
                    }
                    w[k] &= m;
                }
            }
            if (kinds & ZLB_SUM_CRC32) {
#pragma unroll
                for (int k = 0; k < 4; ++k) crc = crc_step_word(crc, w[k], s_tab);
            }
            if (kinds & ZLB_SUM_ADLER32) {
                // 16 bytes: b += 16*a + sum (16-j)*byte_j ; a += sum byte_j
                uint32_t sum = 0, wsum = 0;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    uint32_t x = w[k];
                    uint32_t b0 = x & 0xFF, b1 = (x >> 8) & 0xFF, b2 = (x >> 16) & 0xFF, b3 = x >> 24;
                    sum += b0 + b1 + b2 + b3;
                    wsum += (16 - 4 * k) * b0 + (15 - 4 * k) * b1 + (14 - 4 * k) * b2 + (13 - 4 * k) * b3;
                }
                b += 16u * a + wsum;
                a += sum;
            }
        }
    }
    // R <= 4096 keeps a < 2^21 and b < 2^32 before this reduction
    a %= ADLER_MOD;
    unsigned long long bb = b % ADLER_MOD;

    // warp tree: lower lane is the LEFT operand, right operand spans R * 2^k bytes
    const unsigned lane = t & 31u, warp = t >> 5;
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        uint32_t rc = __shfl_down_sync(0xFFFFFFFFu, crc, 1u << k);
        uint32_t ra = __shfl_down_sync(0xFFFFFFFFu, a, 1u << k);
        unsigned long long rb = __shfl_down_sync(0xFFFFFFFFu, bb, 1u << k);
        if ((lane & ((2u << k) - 1u)) == 0) {
            if (kinds & ZLB_SUM_CRC32) crc = zts_gf2_mulmod(crc, s_lvl[k]) ^ rc;
            unsigned long long nr = ((unsigned long long)R << k) % ADLER_MOD;
            bb = (bb + nr * a + rb) % ADLER_MOD;
            a = (a + ra) % ADLER_MOD;
        }
    }
    if (lane == 0) {
        s_wcrc[warp] = crc;
        s_wa[warp] = a;
        s_wb[warp] = bb;
    }
    __syncthreads();
    if (t == 0) {
        // fold the 8 warp results left to right; each right operand spans 32*R bytes
        uint32_t c = s_wcrc[0], ta = s_wa[0];
        unsigned long long tb = s_wb[0];
        const unsigned long long nr = (32ull * R) % ADLER_MOD;
        for (int w = 1; w < ZTS_SUM_THREADS / 32; ++w) {
            if (kinds & ZLB_SUM_CRC32) c = zts_gf2_mulmod(c, s_lvl[5]) ^ s_wcrc[w];
            tb = (tb + nr * ta + s_wb[w]) % ADLER_MOD;
            ta = (ta + s_wa[w]) % ADLER_MOD;
        }
        // remove the trailing zero padding
        if (pad) {
            c = zts_gf2_mulmod(c, c_xinv_bytes[pad]);
            tb = (tb + (unsigned long long)ADLER_MOD * pad - (unsigned long long)pad * ta) % ADLER_MOD;
        }
        ZtsSlicePartial out;
        out.crc_raw = c;
        out.a = ta;
        out.b = (uint32_t)tb;
        partials[blockIdx.x] = out;
    }
}

// One warp per item: every slice's partial is advanced past the bytes that follow it, then summed.
__global__ void __launch_bounds__(128)
checksum_combine_kernel(const zlb_item* __restrict__ items, zlb_result* __restrict__ results, int use_out_len,
                        const uint32_t* __restrict__ slice_begin, const ZtsSlicePartial* __restrict__ partials,
                        uint32_t n_items, uint32_t kinds)
{
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t item = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (item >= n_items) return;
    const uint64_t len = use_out_len ? results[item].out_len : items[item].in_len;
    const uint32_t s0 = slice_begin[item], s1 = slice_begin[item + 1];
    uint32_t crc = 0;
    unsigned long long a = 0, b = 0;
    for (uint32_t s = s0 + lane; s < s1; s += 32) {
        const uint64_t end = (uint64_t)(s - s0 + 1) * ZTS_SUM_SLICE;
        const uint64_t after = len > end ? len - end : 0;
        const ZtsSlicePartial p = partials[s];
        if (kinds & ZLB_SUM_CRC32) crc ^= zts_gf2_mulmod(p.crc_raw, zts_xpow_bytes(after));
        a = (a + p.a) % ADLER_MOD;
        b = (b + p.b + (after % ADLER_MOD) * p.a) % ADLER_MOD;
    }
    crc = __reduce_xor_sync(0xFFFFFFFFu, crc);
    uint32_t a32 = (uint32_t)a, b32 = (uint32_t)b;
    a32 = __reduce_add_sync(0xFFFFFFFFu, a32) % ADLER_MOD;
    b32 = __reduce_add_sync(0xFFFFFFFFu, b32) % ADLER_MOD;
    if (lane == 0) {
        if (kinds & ZLB_SUM_CRC32) {
            // init 0xFFFFFFFF travels through len bytes; xorout 0xFFFFFFFF  (src/CRC32.ts:29,46)
            results[item].crc32 = (zts_gf2_mulmod(0xFFFFFFFFu, zts_xpow_bytes(len)) ^ crc) ^ 0xFFFFFFFFu;
        }
        if (kinds & ZLB_SUM_ADLER32) {
            // s1 starts at 1 (src/Adler32.ts:19): s1 = 1 + a, s2 = len + b
            uint32_t s1v = (1u + a32) % ADLER_MOD;
            uint32_t s2v = (uint32_t)((len % ADLER_MOD + b32) % ADLER_MOD);
            results[item].adler32 = (s2v << 16) | s1v;
        }
    }
}

// d_items / d_results already hold the items (and, when use_out_len, the out_len of each result).
int zts_checksum_device(zlb_ctx* ctx, const uint8_t* d_in, const zlb_item* d_items, zlb_result* d_results,
                        const zlb_item* h_items, size_t n, uint32_t kinds, int use_out_len)
{
    if (n == 0 || (kinds & (ZLB_SUM_CRC32 | ZLB_SUM_ADLER32)) == 0) return ZLB_OK;
    if (!h_xinv_ready) {
        for (int p = 0; p < 16; ++p) h_xinv_bytes[p] = host_xpow_bits(0xFFFFFFFFull - 8ull * p);
        h_xinv_ready = true;
    }
    ZTS_CUDA(ctx, cudaMemcpyToSymbolAsync(c_xinv_bytes, h_xinv_bytes, sizeof h_xinv_bytes, 0,
                                          cudaMemcpyHostToDevice, ctx->stream));
    // the pinned staging area is shared with other tables that may still be in flight on the stream
    ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    // slice table from the host copy of the items. With use_out_len the true lengths are only on
    // the device; out_cap bounds them, empty trailing slices contribute nothing.
    size_t n_slices = 0;
    for (size_t i = 0; i < n; ++i) {
        uint64_t len = use_out_len ? h_items[i].out_cap : h_items[i].in_len;
        uint64_t s = (len + ZTS_SUM_SLICE - 1) / ZTS_SUM_SLICE;
        n_slices += s ? s : 1;
    }
    if (n_slices > 0x7FFFFFFFull) return zts_fail(ctx, ZLB_E_ARG, "too many checksum slices");
    size_t tab_bytes = n_slices * sizeof(ZtsSlice) + (n + 1) * sizeof(uint32_t);
    int rc = zts_reserve_pinned(ctx, &ctx->h_pin, tab_bytes);
    if (rc) return rc;
    ZtsSlice* h_sl = (ZtsSlice*)ctx->h_pin.p;
    uint32_t* h_begin = (uint32_t*)(h_sl + n_slices);
    size_t k = 0;
    for (size_t i = 0; i < n; ++i) {
        uint64_t len = use_out_len ? h_items[i].out_cap : h_items[i].in_len;
        uint64_t s = (len + ZTS_SUM_SLICE - 1) / ZTS_SUM_SLICE;
        if (!s) s = 1;
        h_begin[i] = (uint32_t)k;
        for (uint64_t j = 0; j < s; ++j) {
            h_sl[k].item = (uint32_t)i;
            h_sl[k].index = (uint32_t)j;
            ++k;
        }
    }
    h_begin[n] = (uint32_t)k;
    rc = zts_reserve(ctx, &ctx->d_sums, tab_bytes + n_slices * sizeof(ZtsSlicePartial) + 64);
    if (rc) return rc;
    uint8_t* base = (uint8_t*)ctx->d_sums.p;
    ZtsSlice* d_sl = (ZtsSlice*)base;
    uint32_t* d_begin = (uint32_t*)(d_sl + n_slices);
    size_t poff = (tab_bytes + 15) & ~(size_t)15;
    ZtsSlicePartial* d_part = (ZtsSlicePartial*)(base + poff);
    ZTS_CUDA(ctx, cudaMemcpyAsync(d_sl, h_sl, tab_bytes, cudaMemcpyHostToDevice, ctx->stream));
    ZTS_LAUNCH(ctx, ZK_CHECKSUM_SLICES,
               checksum_slices_kernel<<<(unsigned)n_slices, ZTS_SUM_THREADS, 0, ctx->stream>>>(
                   d_in, d_items, d_results, use_out_len, d_sl, d_part, kinds));
    unsigned wpb = 4;
    ZTS_LAUNCH(ctx, ZK_CHECKSUM_COMBINE,
               checksum_combine_kernel<<<(unsigned)((n + wpb - 1) / wpb), wpb * 32, 0, ctx->stream>>>(
                   d_items, d_results, use_out_len, d_begin, d_part, (uint32_t)n, kinds));
    // the pinned table must stay untouched until the copy has been consumed
    ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ZLB_OK;
}

static int checksum_common(zlb_ctx* ctx, const void* d_in, const zlb_item* items, zlb_result* results, size_t n,
                           uint32_t kinds)
{
    int rc = zts_reserve(ctx, &ctx->d_items, n * sizeof(zlb_item) + 64);
    if (rc) return rc;
    rc = zts_reserve(ctx, &ctx->d_results, n * sizeof(zlb_result) + 64);
    if (rc) return rc;
    ZTS_CUDA(ctx, cudaMemcpyAsync(ctx->d_items.p, items, n * sizeof(zlb_item), cudaMemcpyHostToDevice, ctx->stream));
    ZTS_CUDA(ctx, cudaMemsetAsync(ctx->d_results.p, 0, n * sizeof(zlb_result), ctx->stream));
    rc = zts_checksum_device(ctx, (const uint8_t*)d_in, (const zlb_item*)ctx->d_items.p,
                             (zlb_result*)ctx->d_results.p, items, n, kinds, 0);
    if (rc) return rc;
    ZTS_CUDA(ctx, cudaMemcpyAsync(results, ctx->d_results.p, n * sizeof(zlb_result), cudaMemcpyDeviceToHost,
                                  ctx->stream));
    ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (size_t i = 0; i < n; ++i) results[i].out_len = 0;
    return ZLB_OK;
}

extern "C" int zlb_checksum_batch(zlb_ctx* ctx, const void* d_in, const zlb_item* items, zlb_result* results,
                                  size_t n, uint32_t kinds)
{
    if (!ctx || (!d_in && n) || (!items && n) || (!results && n)) return ZLB_E_ARG;
    if (n == 0) return ZLB_OK;
    ZTS_CUDA(ctx, cudaSetDevice(ctx->device));
    return checksum_common(ctx, d_in, items, results, n, kinds);
}

extern "C" int zlb_checksum_batch_host(zlb_ctx* ctx, const void* h_in, size_t in_bytes, const zlb_item* items,
                                       zlb_result* results, size_t n, uint32_t kinds)
{
    if (!ctx || (!h_in && in_bytes) || (!items && n) || (!results && n)) return ZLB_E_ARG;
    if (n == 0) return ZLB_OK;
    ZTS_CUDA(ctx, cudaSetDevice(ctx->device));
    for (size_t i = 0; i < n; ++i)
        if (items[i].in_off + items[i].in_len > in_bytes) return zts_fail(ctx, ZLB_E_ARG, "item %zu out of range", i);
    int rc = zts_reserve(ctx, &ctx->d_stage_in, in_bytes + 64);
    if (rc) return rc;
    ZTS_CUDA(ctx, cudaMemcpyAsync(ctx->d_stage_in.p, h_in, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    return checksum_common(ctx, ctx->d_stage_in.p, items, results, n, kinds);
}
