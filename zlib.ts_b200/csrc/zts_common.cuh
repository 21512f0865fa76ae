// zts_common.cuh -- shared host/device plumbing for libzlibts_b200.so (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <functional>
#include <vector>

#include "../../include/zlibts_b200.h"

// ---- kernel slots for the per-kernel event timers (zlb_profile_*) ---------------------------
enum ZtsKernelSlot {
    ZK_INFLATE = 0,
    ZK_CHECKSUM_SLICES,
    ZK_CHECKSUM_COMBINE,
    ZK_LZ77,
    ZK_HUFFMAN,
    ZK_SCAN,
    ZK_BITPACK,
    ZK_STORED,
    ZK_FINALIZE,
    ZK_MARKER_SCAN,
    ZK_GATHER,
    ZK_FRAME_BODY,
    ZK_FRAME_HEADER,
    ZK_INFLATE_WINDOW,  // marker split, window mode (zts_inflate.cu)
    ZK_WINDOW_RUN,
    ZK_WINDOW_SCAN,
    ZK_WINDOW_RESOLVE,
    ZK_DICT_STAGE,      // preset dictionaries (zts_deflate.cu, zts_inflate.cu)
    ZK_INFLATE_DICT,
    ZK_COUNT
};

static const char* const kZtsKernelNames[ZK_COUNT] = {
    "inflate_warp_kernel", "checksum_slices_kernel", "checksum_combine_kernel",
    "lz77_chunk_kernel",   "huffman_build_kernel",   "chunk_scan_kernel",
    "bitpack_kernel",      "stored_block_kernel",    "deflate_finalize_kernel",
    "marker_scan_kernel",  "segment_gather_kernel",
    "frame_body_kernel",   "frame_header_kernel",
    "inflate_warp_kernel_window", "window_run_kernel", "window_scan_kernel", "window_resolve_kernel",
    "dict_stage_kernel", "inflate_warp_kernel_dict"};

struct ZtsDevBuf {
    void* p = nullptr;
    size_t cap = 0;
};

struct ZtsProfRec {
    int slot;
    cudaEvent_t a, b;
};

struct zlb_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t work = nullptr;  // the stream kernels are launched on right now (== stream unless waves overlap)
    bool own_stream = false;
    int sm_count = 148;
    char err[512] = {0};

    // device arenas (grow-only, freed in zlb_destroy)
    ZtsDevBuf d_items, d_results, d_chunks, d_chunk_info, d_tokens, d_spec, d_hist, d_codes, d_sortT,
        d_sums, d_misc, d_stage_in, d_stage_out, d_split, d_window, d_body, d_frames, d_dict, d_dict_stage;
    // pinned host staging for the small tables
    void* h_pin = nullptr;
    size_t h_pin_cap = 0;
    void* h_pin2 = nullptr;  // read-back area of the pipelined host paths
    size_t h_pin2_cap = 0;
    // copy / second compute streams of the pipelined host paths (created on first use)
    cudaStream_t s_in = nullptr, s_out = nullptr, s_aux[3] = {nullptr, nullptr, nullptr};
    cudaStream_t s_res = nullptr;  // small read-backs that must not queue behind (or in front of) anything else
    std::vector<cudaEvent_t> sync_events;  // disable-timing events, reused across calls

    // "_host" entry points with pageable caller buffers: page-locked shadows + copy threads (zts_hoststage.cu)
    void* copy_pool = nullptr;
    void* h_shadow_in = nullptr;
    size_t h_shadow_in_cap = 0;
    void* h_shadow_out = nullptr;
    size_t h_shadow_out_cap = 0;
    std::vector<cudaEvent_t> stage_ev_pool;

    // profiling
    bool prof = false;
    std::vector<ZtsProfRec> pending;
    std::vector<cudaEvent_t> ev_pool;
    double slot_ms[ZK_COUNT] = {0};
    uint64_t slot_launches[ZK_COUNT] = {0};
    uint64_t launches = 0;
};

int zts_fail(zlb_ctx* ctx, int code, const char* fmt, ...);
int zts_reserve(zlb_ctx* ctx, ZtsDevBuf* b, size_t bytes);
int zts_reserve_pinned(zlb_ctx* ctx, size_t bytes);
int zts_reserve_pinned2(zlb_ctx* ctx, size_t bytes);
int zts_host_streams(zlb_ctx* ctx);                 // creates s_in / s_out / s_aux
cudaEvent_t zts_sync_event(zlb_ctx* ctx, size_t k);  // k-th reusable ordering event (nullptr on failure)
// host staging for pageable caller buffers (zts_hoststage.cu); every function accepts st == nullptr / unstaged sides
struct ZtsHostStage;
int zts_stage_begin(zlb_ctx* ctx, const void* h_in, size_t in_bytes, void* h_out, size_t out_bytes, ZtsHostStage** out);
const uint8_t* zts_stage_in_ptr(const ZtsHostStage* st);   // where H2D copies read from (shadow or the caller's buffer)
uint8_t* zts_stage_out_ptr(const ZtsHostStage* st);        // where D2H copies write to
void zts_stage_wait_in(ZtsHostStage* st, size_t lo, size_t hi);  // blocks until [lo, hi) of the input may be copied from
int zts_stage_out_ready(zlb_ctx* ctx, ZtsHostStage* st, cudaStream_t s, size_t off, size_t len);
int zts_stage_end(zlb_ctx* ctx, ZtsHostStage* st);
void zts_stage_destroy_ctx(zlb_ctx* ctx);
// The checks every batch entry point makes first, in this order: the pointers (bufs_ok: the caller's data buffers are
// given where they are needed), n == 0 (returns 1: nothing to do), at most max_items items, the dictionary table
// (zts_check_dicts); then the context's device is selected.
int zts_entry_begin(zlb_ctx* ctx, bool bufs_ok, const zlb_item* items, const zlb_result* results, size_t n,
                    size_t max_items, const void* dict_blob, size_t dict_bytes, const zlb_dict* dicts, bool* any);
// Host buffers of a "_host" entry point, as its device path sees them. Their bytes travel through the staging arenas
// ctx->d_stage_in / d_stage_out, the dictionary blob through ctx->d_dict.
struct ZtsHostIO {
    const uint8_t* h_in;   // where H2D copies read from: the caller's page-locked buffer, or the library's shadow
    uint8_t* h_out;        // where D2H copies write to
    size_t in_bytes;
    bool out_done;         // set by a device path that has already copied the output back, wave by wave
    ZtsHostStage* stage;   // copy threads behind the shadows (pageable caller buffers), see zts_hoststage.cu
};
// A "_host" entry point: zts_entry_begin, every item inside the blobs, the dictionary blob to the device, the staging
// arenas and the copy threads; then body(io, dictionary table or NULL when no item has one) and a synchronise.
// The copy threads are drained on every path, errors included.
int zts_host_call(zlb_ctx* ctx, const void* h_in, size_t in_bytes, void* h_out, size_t out_bytes, const void* h_dict,
                  size_t dict_bytes, const zlb_dict* dicts, const zlb_item* items, const zlb_result* results, size_t n,
                  size_t max_items, const std::function<int(ZtsHostIO& io, const zlb_dict* dicts)>& body);
// D2H of what items [a, b) wrote (adjacent ranges merged; see zts_ctx.cu); h_out = zts_stage_out_ptr() when staged
int zts_copy_back(zlb_ctx* ctx, ZtsHostStage* st, cudaStream_t s, const uint8_t* d_out, uint8_t* h_out,
                  const zlb_item* h_items, const zlb_result* h_res, const zlb_item* d_items, const zlb_result* d_res,
                  size_t a, size_t b);
// preset dictionaries: checks a table (NULL = none; blob_bytes = SIZE_MAX when the blob's size is not known, i.e. a
// device blob) and tells whether any item has one
int zts_check_dicts(zlb_ctx* ctx, const void* blob, size_t blob_bytes, const zlb_dict* dicts, size_t n, bool* any);
void zts_prof_begin(zlb_ctx* ctx, int slot);
void zts_prof_end(zlb_ctx* ctx, int slot);

// -DZTS_CHECK: bounds asserts on the kernels' table / token / bitmap indices (compute-sanitizer is not available on
// the GPU pool; the checked build runs the GPU test suite once per round, see profiles/). Off in the product build.
#ifdef ZTS_CHECK
#include <stdio.h>
#define ZTS_ASSERT(c)                                                        \
    do {                                                                     \
        if (!(c)) {                                                          \
            printf("ZTS_ASSERT %s:%d %s\n", __FILE__, __LINE__, #c);         \
            __trap();                                                        \
        }                                                                    \
    } while (0)
#else
#define ZTS_ASSERT(c) ((void)0)
#endif

#define ZTS_CUDA(ctx, call)                                                                       \
    do {                                                                                          \
        cudaError_t _e = (call);                                                                  \
        if (_e != cudaSuccess)                                                                    \
            return zts_fail((ctx), ZLB_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), \
                            __FILE__, __LINE__);                                                  \
    } while (0)

// Launch wrapper: counts the launch, brackets it with events when profiling, checks the launch.
#define ZTS_LAUNCH(ctx, slot, ...)                                                                \
    do {                                                                                          \
        zts_prof_begin((ctx), (slot));                                                            \
        __VA_ARGS__;                                                                              \
        zts_prof_end((ctx), (slot));                                                              \
        cudaError_t _e = cudaGetLastError();                                                      \
        if (_e != cudaSuccess)                                                                    \
            return zts_fail((ctx), ZLB_E_CUDA, "launch %s failed: %s", kZtsKernelNames[(slot)],   \
                            cudaGetErrorString(_e));                                              \
    } while (0)

// ---- cross-file entry points (device buffers, async on ctx->stream) ---------------------------
// checksums of n items; writes crc32/adler32 into d_results[i] (fields selected by kinds)
int zts_checksum_device(zlb_ctx* ctx, const uint8_t* d_in, const zlb_item* d_items, zlb_result* d_results,
                        const zlb_item* h_items, size_t n, uint32_t kinds, int use_out_len);

// ---- small device helpers ----------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ unsigned zts_lane() { return threadIdx.x & 31u; }
// block-wide copy of len bytes, any alignment on either side: aligned 4-byte stores, the source read as aligned
// words and shifted into place (all threads of the block call it)
__device__ __forceinline__ void zts_block_copy(uint8_t* dst, const uint8_t* src, uint32_t len, uint32_t tid, uint32_t nthr)
{
    const uint32_t head = min(len, (uint32_t)((4u - ((uintptr_t)dst & 3u)) & 3u));
    if (tid < head) dst[tid] = src[tid];
    const uint32_t words = (len - head) >> 2;
    const uint8_t* s0 = src + head;
    const uint32_t mis = (uint32_t)((uintptr_t)s0 & 3u);
    const uint32_t* sw = reinterpret_cast<const uint32_t*>(s0 - mis);
    uint32_t* dw = reinterpret_cast<uint32_t*>(dst + head);
    if (mis == 0) {
        for (uint32_t i = tid; i < words; i += nthr) dw[i] = sw[i];
    } else {
        // sw[i + 1] holds the upper bytes of word i, so it lies inside the source whenever it is read
        for (uint32_t i = tid; i < words; i += nthr) dw[i] = __funnelshift_r(sw[i], sw[i + 1], mis * 8);
    }
    const uint32_t done = head + (words << 2);
    if (tid < len - done) dst[done + tid] = src[done + tid];
}
__device__ __forceinline__ unsigned zts_lanemask_lt()
{
    unsigned m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}
#endif
