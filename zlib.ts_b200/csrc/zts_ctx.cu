// zts_ctx.cu -- context, arenas, per-kernel event timers, checksum combine (host side).
#include <stdarg.h>

#include "zts_common.cuh"

int zts_fail(zlb_ctx* ctx, int code, const char* fmt, ...)
{
    if (ctx) {
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(ctx->err, sizeof ctx->err, fmt, ap);
        va_end(ap);
    }
    return code;
}

int zts_reserve(zlb_ctx* ctx, ZtsDevBuf* b, size_t bytes)
{
    if (bytes <= b->cap) return ZLB_OK;
    size_t want = bytes + bytes / 4 + 256;
    // the buffer may still be in use by work queued on the stream
    ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (b->p) {
        cudaFree(b->p);
        b->p = nullptr;
        b->cap = 0;
    }
    cudaError_t e = cudaMalloc(&b->p, want);
    if (e != cudaSuccess) {
        b->p = nullptr;
        return zts_fail(ctx, ZLB_E_NOMEM, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
    }
    b->cap = want;
    return ZLB_OK;
}

int zts_check_dicts(zlb_ctx* ctx, const void* blob, size_t blob_bytes, const zlb_dict* dicts, size_t n, bool* any)
{
    *any = false;
    if (!dicts) return ZLB_OK;
    for (size_t i = 0; i < n; ++i) {
        const zlb_dict d = dicts[i];
        if (d.len == 0) continue;
        if (!blob) return zts_fail(ctx, ZLB_E_ARG, "item %zu has a dictionary but the dictionary blob is NULL", i);
        if (d.off > blob_bytes || d.len > blob_bytes - d.off)
            return zts_fail(ctx, ZLB_E_ARG, "dictionary of item %zu out of range", i);
        *any = true;
    }
    return ZLB_OK;
}

int zts_reserve_pinned(zlb_ctx* ctx, size_t bytes)
{
    if (bytes <= ctx->h_pin_cap) return ZLB_OK;
    size_t want = bytes + bytes / 4 + 4096;
    ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->h_pin) cudaFreeHost(ctx->h_pin);
    ctx->h_pin = nullptr;
    ctx->h_pin_cap = 0;
    cudaError_t e = cudaMallocHost(&ctx->h_pin, want);
    if (e != cudaSuccess) return zts_fail(ctx, ZLB_E_NOMEM, "cudaMallocHost(%zu) failed: %s", want, cudaGetErrorString(e));
    ctx->h_pin_cap = want;
    return ZLB_OK;
}

int zts_reserve_pinned2(zlb_ctx* ctx, size_t bytes)
{
    if (bytes <= ctx->h_pin2_cap) return ZLB_OK;
    size_t want = bytes + bytes / 4 + 4096;
    ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->h_pin2) cudaFreeHost(ctx->h_pin2);
    ctx->h_pin2 = nullptr;
    ctx->h_pin2_cap = 0;
    cudaError_t e = cudaMallocHost(&ctx->h_pin2, want);
    if (e != cudaSuccess) return zts_fail(ctx, ZLB_E_NOMEM, "cudaMallocHost(%zu) failed: %s", want, cudaGetErrorString(e));
    ctx->h_pin2_cap = want;
    return ZLB_OK;
}

int zts_host_streams(zlb_ctx* ctx)
{
    if (ctx->s_in) return ZLB_OK;
    ZTS_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->s_in, cudaStreamNonBlocking));
    ZTS_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->s_out, cudaStreamNonBlocking));
    for (int i = 0; i < 3; ++i) ZTS_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->s_aux[i], cudaStreamNonBlocking));
    ZTS_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->s_res, cudaStreamNonBlocking));
    return ZLB_OK;
}

cudaEvent_t zts_sync_event(zlb_ctx* ctx, size_t k)
{
    while (ctx->sync_events.size() <= k) {
        cudaEvent_t e = nullptr;
        if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return nullptr;
        ctx->sync_events.push_back(e);
    }
    return ctx->sync_events[k];
}

static cudaEvent_t prof_event(zlb_ctx* ctx)
{
    if (!ctx->ev_pool.empty()) {
        cudaEvent_t e = ctx->ev_pool.back();
        ctx->ev_pool.pop_back();
        return e;
    }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}

void zts_prof_begin(zlb_ctx* ctx, int slot)
{
    ctx->launches++;
    ctx->slot_launches[slot]++;
    if (!ctx->prof) return;
    ZtsProfRec r;
    r.slot = slot;
    r.a = prof_event(ctx);
    r.b = prof_event(ctx);
    cudaEventRecord(r.a, ctx->work);
    ctx->pending.push_back(r);
}

void zts_prof_end(zlb_ctx* ctx, int slot)
{
    (void)slot;
    if (!ctx->prof) return;
    cudaEventRecord(ctx->pending.back().b, ctx->work);
}

static void prof_resolve(zlb_ctx* ctx)
{
    if (ctx->pending.empty()) return;
    cudaStreamSynchronize(ctx->stream);
    for (const ZtsProfRec& r : ctx->pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) ctx->slot_ms[r.slot] += ms;
        ctx->ev_pool.push_back(r.a);
        ctx->ev_pool.push_back(r.b);
    }
    ctx->pending.clear();
}

// ---- reading results back to the host: only what was written ------------------------------------------------------
// The "_host" entry points stage the output blob in a device buffer that is reused from call to call. Copying whole
// slots (or one span over all of them) back would put stale bytes of earlier calls between the items' outputs, so
// only [out_off, out_off + out_len) of every item travels; adjacent ranges are merged into one copy (a batch of
// streams that fill their slots is one copy). Should that still take more than ZTS_COPYBACK_MAX copies, the slack
// behind every item is zeroed on the device and one span is copied instead.
#define ZTS_COPYBACK_MAX 2048u

__global__ void __launch_bounds__(256)
zero_slack_kernel(uint8_t* __restrict__ out, const zlb_item* __restrict__ items, const zlb_result* __restrict__ res)
{
    const zlb_item it = items[blockIdx.x];
    const zlb_result r = res[blockIdx.x];
    const unsigned long long len = r.out_len <= it.out_cap ? r.out_len : 0ull;
    uint8_t* p = out + it.out_off;
    for (unsigned long long i = len + threadIdx.x; i < it.out_cap; i += 256) p[i] = 0;
}

int zts_copy_back(zlb_ctx* ctx, ZtsHostStage* st, cudaStream_t s, const uint8_t* d_out, uint8_t* h_out,
                  const zlb_item* h_items, const zlb_result* h_res, const zlb_item* d_items, const zlb_result* d_res,
                  size_t a, size_t b)
{
    struct Run {
        uint64_t off, len;
    };
    std::vector<Run> runs;
    uint64_t lo = ~0ull, hi = 0;
    for (size_t i = a; i < b; ++i) {
        const uint64_t len = h_res[i].out_len <= h_items[i].out_cap ? h_res[i].out_len : 0;  // an overflowed item wrote nothing usable
        const uint64_t off = h_items[i].out_off;
        if (off < lo) lo = off;
        if (off + h_items[i].out_cap > hi) hi = off + h_items[i].out_cap;
        if (!len) continue;
        if (!runs.empty() && runs.back().off + runs.back().len == off)
            runs.back().len += len;
        else
            runs.push_back({off, len});
    }
    if (runs.size() > ZTS_COPYBACK_MAX && d_items && d_res) {
        zero_slack_kernel<<<(unsigned)(b - a), 256, 0, s>>>(const_cast<uint8_t*>(d_out), d_items + a, d_res + a);
        ZTS_CUDA(ctx, cudaGetLastError());
        runs.clear();
        runs.push_back({lo, hi - lo});
    }
    for (const Run& r : runs) {
        ZTS_CUDA(ctx, cudaMemcpyAsync(h_out + r.off, d_out + r.off, r.len, cudaMemcpyDeviceToHost, s));
        int rc = zts_stage_out_ready(ctx, st, s, r.off, r.len);
        if (rc) return rc;
    }
    return ZLB_OK;
}

extern "C" {

int zlb_abi_version(void) { return ZLB_ABI_VERSION; }

int zlb_create(int device, void* stream, zlb_ctx** out)
{
    if (!out) return ZLB_E_ARG;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count <= 0 || device < 0 || device >= count) return ZLB_E_CUDA;  // no CPU fallback
    if (cudaSetDevice(device) != cudaSuccess) return ZLB_E_CUDA;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return ZLB_E_CUDA;
    if (prop.major < 10) return ZLB_E_UNSUPPORTED;  // kernels are built for sm_100a only
    zlb_ctx* ctx = new zlb_ctx();
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    if (stream) {
        ctx->stream = (cudaStream_t)stream;
        ctx->own_stream = false;
    } else {
        if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
            delete ctx;
            return ZLB_E_CUDA;
        }
        ctx->own_stream = true;
    }
    ctx->work = ctx->stream;
    *out = ctx;
    return ZLB_OK;
}

void zlb_destroy(zlb_ctx* ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->s_in) cudaStreamSynchronize(ctx->s_in);
    if (ctx->s_out) cudaStreamSynchronize(ctx->s_out);
    for (int i = 0; i < 3; ++i)
        if (ctx->s_aux[i]) cudaStreamSynchronize(ctx->s_aux[i]);
    ZtsDevBuf* bufs[] = {&ctx->d_items, &ctx->d_results, &ctx->d_chunks, &ctx->d_chunk_info, &ctx->d_tokens,
                         &ctx->d_spec,  &ctx->d_hist,    &ctx->d_codes,  &ctx->d_sortT,      &ctx->d_sums,
                         &ctx->d_misc,  &ctx->d_stage_in, &ctx->d_stage_out, &ctx->d_split, &ctx->d_window,
                         &ctx->d_body,  &ctx->d_frames, &ctx->d_dict, &ctx->d_dict_stage};
    for (ZtsDevBuf* b : bufs)
        if (b->p) cudaFree(b->p);
    zts_stage_destroy_ctx(ctx);
    if (ctx->h_pin) cudaFreeHost(ctx->h_pin);
    if (ctx->h_pin2) cudaFreeHost(ctx->h_pin2);
    for (cudaEvent_t e : ctx->sync_events) cudaEventDestroy(e);
    if (ctx->s_in) cudaStreamDestroy(ctx->s_in);
    if (ctx->s_out) cudaStreamDestroy(ctx->s_out);
    if (ctx->s_res) cudaStreamDestroy(ctx->s_res);
    for (int i = 0; i < 3; ++i)
        if (ctx->s_aux[i]) cudaStreamDestroy(ctx->s_aux[i]);
    for (const ZtsProfRec& r : ctx->pending) {
        cudaEventDestroy(r.a);
        cudaEventDestroy(r.b);
    }
    for (cudaEvent_t e : ctx->ev_pool) cudaEventDestroy(e);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char* zlb_last_error(const zlb_ctx* ctx) { return ctx ? ctx->err : "null ctx"; }
void* zlb_stream(const zlb_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
uint64_t zlb_launch_count(const zlb_ctx* ctx) { return ctx ? ctx->launches : 0; }

int zlb_profile_enable(zlb_ctx* ctx, int on)
{
    if (!ctx) return ZLB_E_ARG;
    prof_resolve(ctx);
    ctx->prof = on != 0;
    return ZLB_OK;
}

int zlb_profile_reset(zlb_ctx* ctx)
{
    if (!ctx) return ZLB_E_ARG;
    prof_resolve(ctx);
    for (int i = 0; i < ZK_COUNT; ++i) {
        ctx->slot_ms[i] = 0;
        ctx->slot_launches[i] = 0;
    }
    return ZLB_OK;
}

int zlb_profile_read(zlb_ctx* ctx, int* n, const char** names, double* total_ms, uint64_t* launches)
{
    if (!ctx || !n) return ZLB_E_ARG;
    prof_resolve(ctx);
    if (names && total_ms && launches) {
        int m = *n < ZK_COUNT ? *n : ZK_COUNT;
        for (int i = 0; i < m; ++i) {
            names[i] = kZtsKernelNames[i];
            total_ms[i] = ctx->slot_ms[i];
            launches[i] = ctx->slot_launches[i];
        }
    }
    *n = ZK_COUNT;
    return ZLB_OK;
}

// ---- checksum combine -------------------------------------------------------------------------
// CRC-32 of A||B = crc(A) * x^(8*len_B) mod P  xor  crc(B), polynomials in the reflected
// representation used by src/CRC32.ts (0xEDB88320).
static uint32_t gf2_mulmod(uint32_t a, uint32_t b)
{
    uint32_t p = 0;
    for (uint32_t m = 0x80000000u; m; m >>= 1) {
        if (a & m) p ^= b;
        b = (b & 1u) ? (b >> 1) ^ 0xEDB88320u : (b >> 1);
    }
    return p;
}

uint32_t zlb_crc32_combine(uint32_t crc_a, uint32_t crc_b, uint64_t len_b)
{
    uint32_t xp = 0x80000000u;  // x^0
    uint32_t sq = 0x00800000u;  // x^8 : one byte
    for (uint64_t n = len_b; n; n >>= 1) {
        if (n & 1) xp = gf2_mulmod(sq, xp);
        sq = gf2_mulmod(sq, sq);
    }
    return gf2_mulmod(xp, crc_a) ^ crc_b;
}

// Adler-32 (src/Adler32.ts:28-48): s1 = 1 + sum b_i, s2 = sum of the running s1 values (mod 65521).
uint32_t zlb_adler32_combine(uint32_t adler_a, uint32_t adler_b, uint64_t len_b)
{
    const uint64_t M = 65521;
    uint64_t a1 = adler_a & 0xFFFF, a2 = (adler_a >> 16) & 0xFFFF;
    uint64_t b1 = adler_b & 0xFFFF, b2 = (adler_b >> 16) & 0xFFFF;
    uint64_t rem = len_b % M;
    // B alone started from s1 = 1; appended after A it starts from s1 = a1
    uint64_t s1 = (a1 + b1 + M - 1) % M;
    uint64_t s2 = (a2 + b2 + rem * ((a1 + M - 1) % M)) % M;
    return (uint32_t)((s2 << 16) | s1);
}

}  // extern "C"
