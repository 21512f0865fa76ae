// zts_hoststage.cu -- host-side plumbing of the "_host" entry points for callers whose buffers are NOT page-locked
// (a plain malloc'ed / JS-heap buffer), the prologue and epilogue the batch entry points share, plus zlb_host_alloc /
// zlb_host_free for callers that can do better.
//
// cudaMemcpyAsync from pageable memory is staged by the driver through a small bounce buffer and serialises with
// the caller's thread; the wave pipelines of the host paths (input of wave k+1 and output of wave k-1 travelling while
// wave k is computed) would lose their overlap. Instead the library keeps page-locked SHADOWS of the two blobs per
// context (grow-only) and a small pool of copy threads:
//   input   the pool copies the caller's bytes into the shadow in 2 MiB pieces, in order, ahead of the pipeline; the
//           pipeline asks for a byte range right before it queues that range's H2D copy (zts_stage_wait_in);
//   output  every D2H copy lands in the shadow and is followed by an event; the pool waits for the event and moves the
//           range to the caller's buffer (zts_stage_out_ready); the entry point returns when the pool has drained.
// One cudaMemcpyAsync per piece, no batched-memcpy APIs. Blobs beyond ZTS_STAGE_MAX bytes are not shadowed (plain
// copies from pageable memory: correct, slower).
#include <atomic>
#include <condition_variable>
#include <deque>
#include <memory>
#include <mutex>
#include <thread>

#include "zts_common.cuh"

#define ZTS_STAGE_PIECE ((size_t)2 << 20)
#define ZTS_STAGE_MAX ((size_t)4 << 30)

struct ZtsCopyTask {
    const uint8_t* src;
    uint8_t* dst;
    size_t len;
    cudaEvent_t ev;                  // wait for it first (output side), or nullptr
    std::atomic<uint8_t>* flag;      // set when done (input side), or nullptr
};

struct ZtsCopyPool {
    int device;
    std::vector<std::thread> threads;
    std::mutex m;
    std::condition_variable cv, cv_idle;
    std::deque<ZtsCopyTask> q;
    size_t in_flight = 0;
    bool stop = false;

    explicit ZtsCopyPool(int dev) : device(dev)
    {
        unsigned hc = std::thread::hardware_concurrency();
        unsigned n = hc / 2;  // (measured on a 16-thread host: 4 threads reach 80 % of the page-locked rate, 8 reach 88 %)
        if (n < 2) n = 2;
        if (n > 8) n = 8;
        if (const char* e = getenv("ZLB_COPY_THREADS")) {
            int v = atoi(e);
            if (v >= 1 && v <= 64) n = (unsigned)v;
        }
        for (unsigned i = 0; i < n; ++i) threads.emplace_back([this] { run(); });
    }
    ~ZtsCopyPool()
    {
        {
            std::lock_guard<std::mutex> l(m);
            stop = true;
        }
        cv.notify_all();
        for (auto& t : threads) t.join();
    }
    void run()
    {
        cudaSetDevice(device);
        for (;;) {
            ZtsCopyTask t;
            {
                std::unique_lock<std::mutex> l(m);
                cv.wait(l, [this] { return stop || !q.empty(); });
                if (q.empty()) return;
                t = q.front();
                q.pop_front();
            }
            if (t.ev) cudaEventSynchronize(t.ev);
            memcpy(t.dst, t.src, t.len);
            if (t.flag) t.flag->store(1, std::memory_order_release);
            {
                std::lock_guard<std::mutex> l(m);
                --in_flight;
            }
            cv_idle.notify_all();
        }
    }
    void push(const ZtsCopyTask& t)
    {
        {
            std::lock_guard<std::mutex> l(m);
            q.push_back(t);
            ++in_flight;
        }
        cv.notify_one();
    }
    void drain()
    {
        std::unique_lock<std::mutex> l(m);
        cv_idle.wait(l, [this] { return in_flight == 0; });
    }
};

struct ZtsHostStage {
    zlb_ctx* ctx = nullptr;
    // input
    const uint8_t* user_in = nullptr;
    const uint8_t* eff_in = nullptr;
    size_t in_bytes = 0;
    std::unique_ptr<std::atomic<uint8_t>[]> in_flags;  // one per piece of the shadow
    // output
    uint8_t* user_out = nullptr;
    uint8_t* eff_out = nullptr;
    size_t out_bytes = 0;
    bool stage_in = false, stage_out = false;
    std::vector<cudaEvent_t> events;  // taken from the ctx pool for this call
};

static bool is_pinned(const void* p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

static int reserve_shadow(zlb_ctx* ctx, void** p, size_t* cap, size_t bytes)
{
    if (bytes <= *cap) return ZLB_OK;
    const size_t want = bytes + bytes / 8 + 4096;
    ZTS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (*p) cudaFreeHost(*p);
    *p = nullptr;
    *cap = 0;
    cudaError_t e = cudaHostAlloc(p, want, cudaHostAllocDefault);
    if (e != cudaSuccess) {
        *p = nullptr;
        return zts_fail(ctx, ZLB_E_NOMEM, "cudaHostAlloc(%zu) failed: %s", want, cudaGetErrorString(e));
    }
    *cap = want;
    return ZLB_OK;
}

int zts_stage_begin(zlb_ctx* ctx, const void* h_in, size_t in_bytes, void* h_out, size_t out_bytes, ZtsHostStage** out)
{
    ZtsHostStage* st = new ZtsHostStage();
    st->ctx = ctx;
    st->user_in = st->eff_in = (const uint8_t*)h_in;
    st->user_out = st->eff_out = (uint8_t*)h_out;
    st->in_bytes = in_bytes;
    st->out_bytes = out_bytes;
    *out = st;
    const bool off = getenv("ZLB_NO_STAGING") != nullptr;
    st->stage_in = !off && h_in && in_bytes >= (64u << 10) && in_bytes <= ZTS_STAGE_MAX && !is_pinned(h_in);
    st->stage_out = !off && h_out && out_bytes >= (64u << 10) && out_bytes <= ZTS_STAGE_MAX && !is_pinned(h_out);
    if (!st->stage_in && !st->stage_out) return ZLB_OK;
    if (!ctx->copy_pool) ctx->copy_pool = new ZtsCopyPool(ctx->device);
    ZtsCopyPool* pool = (ZtsCopyPool*)ctx->copy_pool;
    int rc;
    if (st->stage_in) {
        if ((rc = reserve_shadow(ctx, &ctx->h_shadow_in, &ctx->h_shadow_in_cap, in_bytes))) return rc;
        st->eff_in = (const uint8_t*)ctx->h_shadow_in;
        const size_t np = (in_bytes + ZTS_STAGE_PIECE - 1) / ZTS_STAGE_PIECE;
        st->in_flags.reset(new std::atomic<uint8_t>[np]);
        for (size_t i = 0; i < np; ++i) st->in_flags[i].store(0, std::memory_order_relaxed);
        for (size_t i = 0; i < np; ++i) {  // in order: the pipeline asks for the front of the blob first
            const size_t o = i * ZTS_STAGE_PIECE;
            const size_t len = in_bytes - o < ZTS_STAGE_PIECE ? in_bytes - o : ZTS_STAGE_PIECE;
            pool->push({st->user_in + o, (uint8_t*)ctx->h_shadow_in + o, len, nullptr, &st->in_flags[i]});
        }
    }
    if (st->stage_out) {
        if ((rc = reserve_shadow(ctx, &ctx->h_shadow_out, &ctx->h_shadow_out_cap, out_bytes))) return rc;
        st->eff_out = (uint8_t*)ctx->h_shadow_out;
    }
    return ZLB_OK;
}

const uint8_t* zts_stage_in_ptr(const ZtsHostStage* st) { return st->eff_in; }
uint8_t* zts_stage_out_ptr(const ZtsHostStage* st) { return st->eff_out; }

void zts_stage_wait_in(ZtsHostStage* st, size_t lo, size_t hi)
{
    if (!st || !st->stage_in || hi <= lo) return;
    if (hi > st->in_bytes) hi = st->in_bytes;
    for (size_t i = lo / ZTS_STAGE_PIECE; i <= (hi - 1) / ZTS_STAGE_PIECE; ++i)
        while (!st->in_flags[i].load(std::memory_order_acquire)) std::this_thread::yield();
}

// [off, off + len) of the output has been queued for its D2H copy on `s` (into the shadow when the output is staged):
// hand the range to the copy threads, which wait for the copy to land first
int zts_stage_out_ready(zlb_ctx* ctx, ZtsHostStage* st, cudaStream_t s, size_t off, size_t len)
{
    if (!st || !st->stage_out || len == 0) return ZLB_OK;
    cudaEvent_t ev = nullptr;
    if (!ctx->stage_ev_pool.empty()) {
        ev = ctx->stage_ev_pool.back();
        ctx->stage_ev_pool.pop_back();
    } else {
        ZTS_CUDA(ctx, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    }
    st->events.push_back(ev);
    ZTS_CUDA(ctx, cudaEventRecord(ev, s));
    ZtsCopyPool* pool = (ZtsCopyPool*)ctx->copy_pool;
    for (size_t o = 0; o < len; o += ZTS_STAGE_PIECE) {
        const size_t l = len - o < ZTS_STAGE_PIECE ? len - o : ZTS_STAGE_PIECE;
        pool->push({st->eff_out + off + o, st->user_out + off + o, l, ev, nullptr});
    }
    return ZLB_OK;
}

// waits until every queued copy has been done (also on error paths: the threads hold pointers into this call's buffers)
int zts_stage_end(zlb_ctx* ctx, ZtsHostStage* st)
{
    if (!st) return ZLB_OK;
    if (ctx->copy_pool && (st->stage_in || st->stage_out)) ((ZtsCopyPool*)ctx->copy_pool)->drain();
    for (cudaEvent_t e : st->events) ctx->stage_ev_pool.push_back(e);
    delete st;
    return ZLB_OK;
}

void zts_stage_destroy_ctx(zlb_ctx* ctx)
{
    if (ctx->copy_pool) delete (ZtsCopyPool*)ctx->copy_pool;
    ctx->copy_pool = nullptr;
    if (ctx->h_shadow_in) cudaFreeHost(ctx->h_shadow_in);
    if (ctx->h_shadow_out) cudaFreeHost(ctx->h_shadow_out);
    for (cudaEvent_t e : ctx->stage_ev_pool) cudaEventDestroy(e);
    ctx->stage_ev_pool.clear();
}

// ---- what the batch entry points share ------------------------------------------------------------------------------
int zts_entry_begin(zlb_ctx* ctx, bool bufs_ok, const zlb_item* items, const zlb_result* results, size_t n,
                    size_t max_items, const void* dict_blob, size_t dict_bytes, const zlb_dict* dicts, bool* any,
                    bool dict_lens_only)
{
    if (!ctx || !bufs_ok || (!items && n) || (!results && n)) return ZLB_E_ARG;
    if (n == 0) return 1;
    if (n > max_items) return zts_fail(ctx, ZLB_E_ARG, "too many items");
    int rc = zts_check_dicts(ctx, dict_blob, dict_bytes, dicts, n, any, dict_lens_only);
    if (rc) return rc;
    ZTS_CUDA(ctx, cudaSetDevice(ctx->device));
    return ZLB_OK;
}

int zts_host_call(zlb_ctx* ctx, const void* h_in, size_t in_bytes, void* h_out, size_t out_bytes, const void* h_dict,
                  size_t dict_bytes, const zlb_dict* dicts, const zlb_item* items, const zlb_result* results, size_t n,
                  size_t max_items, const std::function<int(ZtsHostIO& io, const zlb_dict* dicts)>& body,
                  ZtsHostKind kind)
{
    const bool sizes = kind == ZTS_HOST_SIZES;
    if (sizes) {
        h_out = nullptr;
        out_bytes = 0;
    }
    bool any = false;
    int rc = zts_entry_begin(ctx, (h_in || !in_bytes) && (h_out || !out_bytes), items, results, n, max_items, h_dict,
                             dict_bytes, dicts, &any, sizes);
    if (rc) return rc > 0 ? ZLB_OK : rc;
    for (size_t i = 0; i < n; ++i) {
        if (items[i].in_off + items[i].in_len > in_bytes || (!sizes && items[i].out_off + items[i].out_cap > out_bytes))
            return zts_fail(ctx, ZLB_E_ARG, "item %zu out of range", i);
    }
    // the dictionaries go over first, on the context's stream (everything of the call is ordered behind it)
    if (any && !sizes) {
        if ((rc = zts_reserve(ctx, &ctx->d_dict, dict_bytes + 256))) return rc;
        ZTS_CUDA(ctx, cudaMemcpyAsync(ctx->d_dict.p, h_dict, dict_bytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    rc = zts_reserve(ctx, &ctx->d_stage_in, in_bytes + 256);
    if (rc) return rc;
    if (!sizes && (rc = zts_reserve(ctx, &ctx->d_stage_out, out_bytes + 256))) return rc;
    ZtsHostStage* stage = nullptr;
    rc = zts_stage_begin(ctx, h_in, in_bytes, h_out, out_bytes, &stage);
    if (!rc) {
        ZtsHostIO io = {zts_stage_in_ptr(stage), zts_stage_out_ptr(stage), in_bytes, stage};
        rc = body(io, any ? dicts : nullptr);
        if (!rc && cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = zts_fail(ctx, ZLB_E_CUDA, "synchronize failed");
    }
    zts_stage_end(ctx, stage);  // also on errors: the copy threads hold pointers into the caller's buffers
    return rc;
}

// ---- page-locked memory for callers (an N-API addon hands it out as external ArrayBuffers) -------------------------
extern "C" int zlb_host_alloc(size_t bytes, void** out)
{
    if (!out) return ZLB_E_ARG;
    *out = nullptr;
    cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable);
    if (e != cudaSuccess) {
        *out = nullptr;
        return e == cudaErrorMemoryAllocation ? ZLB_E_NOMEM : ZLB_E_CUDA;
    }
    return ZLB_OK;
}

extern "C" void zlb_host_free(void* p)
{
    if (p) cudaFreeHost(p);
}

extern "C" int zlb_host_is_pinned(const void* p) { return p && is_pinned(p) ? 1 : 0; }
