// addon.cc -- Node.js N-API binding of libzlibts_b200.so (include/zlibts_b200.h).
//
// NOT RUN IN THIS IMAGE: there is no Node binary and no node_api.h here or on the GPU boxes (SURVEY.md section 0.6);
// tests/test_abi.py type-checks this file against a stub of the N-API declarations it uses (tests/napi_stub/). It is
// the binding a maintainer adds to the reference: pure marshalling, no algorithm. The tested equivalent of this layer
// is zlib.ts_b200/api.py over the same C ABI.
//
// Memory: everything the GPU copies from or to is page-locked (zlb_host_alloc). Outputs are handed to JS as views into
// ONE external ArrayBuffer over the page-locked result buffer (no copy; freed when the last view is collected). Inputs
// that live in the JS heap are gathered into a page-locked blob (one memcpy); an input that already lives in memory
// from hostAlloc() (exported below) is passed as it is.
//
// Exports (all synchronous, like the reference's API):
//   deflateBatch(inputs: Uint8Array[], compressionType, chunkBytes, flags, mode?) -> {outputs: Uint8Array[], crc32: number[], adler32: number[]}
//   inflateBatch(input: Uint8Array, offsets: number[], lengths: number[], caps: number[], flags)
//                                                          -> {outputs, status: number[], inUsed: number[], crc32, adler32}
//   checksumBatch(inputs: Uint8Array[], kinds)             -> {crc32: number[], adler32: number[]}
//   crc32Combine(a, b, lenB), adler32Combine(a, b, lenB)
//   hostAlloc(bytes) -> Uint8Array over page-locked memory (build inputs in it: they then travel without a copy)
//   archive(kind, inputs: Uint8Array[], heads: Uint8Array[], cdirs: Uint8Array[] | null, methods: number[] | null,
//           tail: Uint8Array, compressionType, chunkBytes, mode)
//                                   -> {output: Uint8Array, crc32, adler32, offsets: number[], lengths: number[]}
//     the whole container (zlib streams / gzip members / zip archive) framed and packed on the device
#include <node_api.h>

#include <cstring>
#include <vector>

#include "../include/zlibts_b200.h"

static zlb_ctx* g_ctx = nullptr;

static bool ensure_ctx(napi_env env)
{
    if (g_ctx) return true;
    if (zlb_create(0, nullptr, &g_ctx) != ZLB_OK) {
        napi_throw_error(env, nullptr, "zlib.ts-b200: no usable B200 device (there is no CPU fallback)");
        return false;
    }
    return true;
}

struct Bytes {
    uint8_t* p;
    size_t n;
};

static bool get_u8(napi_env env, napi_value v, Bytes* out)
{
    bool is_ta = false;
    napi_is_typedarray(env, v, &is_ta);
    if (!is_ta) return false;
    napi_typedarray_type t;
    size_t len, off;
    void* data;
    napi_value ab;
    napi_get_typedarray_info(env, v, &t, &len, &data, &ab, &off);
    if (t != napi_uint8_array) return false;
    out->p = (uint8_t*)data;
    out->n = len;
    return true;
}

// page-locked host memory for the duration of a call
struct HostBuf {
    uint8_t* p = nullptr;
    size_t n = 0;
    explicit HostBuf(size_t bytes) : n(bytes ? bytes : 1)
    {
        void* q = nullptr;
        if (zlb_host_alloc(n, &q) == ZLB_OK) p = (uint8_t*)q;
    }
    ~HostBuf()
    {
        if (p) zlb_host_free(p);
    }
    uint8_t* release()
    {
        uint8_t* q = p;
        p = nullptr;
        return q;
    }
    HostBuf(const HostBuf&) = delete;
    HostBuf& operator=(const HostBuf&) = delete;
};

static void free_host(napi_env, void* data, void*) { zlb_host_free(data); }

// An external ArrayBuffer that takes over a page-locked buffer (freed by the finalizer), and views into it
static napi_value adopt_buffer(napi_env env, uint8_t* p, size_t n)
{
    napi_value ab;
    if (napi_create_external_arraybuffer(env, p, n, free_host, nullptr, &ab) != napi_ok) {
        zlb_host_free(p);  // (runtimes that forbid external buffers: the caller falls back to a copy)
        return nullptr;
    }
    return ab;
}
static napi_value view_u8(napi_env env, napi_value ab, size_t off, size_t n)
{
    napi_value ta;
    napi_create_typedarray(env, napi_uint8_array, n, ab, off, &ta);
    return ta;
}
static napi_value copy_u8(napi_env env, const uint8_t* src, size_t n)
{
    void* data;
    napi_value ab, ta;
    napi_create_arraybuffer(env, n, &data, &ab);
    if (n) memcpy(data, src, n);
    napi_create_typedarray(env, napi_uint8_array, n, ab, 0, &ta);
    return ta;
}
// the outputs of a batch: views into the adopted result buffer, or copies where that is not possible
struct Outputs {
    napi_env env;
    napi_value ab = nullptr;
    uint8_t* base;
    Outputs(napi_env e, HostBuf& out) : env(e), base(out.p)
    {
        const size_t n = out.n;
        ab = adopt_buffer(env, out.release(), n);
        if (!ab) base = nullptr;
    }
    napi_value at(const uint8_t* fallback_base, size_t off, size_t n) const
    {
        return ab ? view_u8(env, ab, off, n) : copy_u8(env, fallback_base + off, n);
    }
};

static napi_value num_array(napi_env env, const std::vector<double>& v)
{
    napi_value a;
    napi_create_array_with_length(env, v.size(), &a);
    for (size_t i = 0; i < v.size(); ++i) {
        napi_value x;
        napi_create_double(env, v[i], &x);
        napi_set_element(env, a, (uint32_t)i, x);
    }
    return a;
}

static std::vector<double> get_numbers(napi_env env, napi_value arr)
{
    uint32_t n = 0;
    napi_get_array_length(env, arr, &n);
    std::vector<double> v(n);
    for (uint32_t i = 0; i < n; ++i) {
        napi_value e;
        napi_get_element(env, arr, i, &e);
        napi_get_value_double(env, e, &v[i]);
    }
    return v;
}

// an optional preset dictionary argument (Uint8Array, shared by every item; undefined / empty = none): the zlb_dict
// table of n items that all name it
static bool get_dict(napi_env env, size_t argc, napi_value* argv, size_t k, size_t n, Bytes* dict,
                     std::vector<zlb_dict>* dicts)
{
    dict->p = nullptr;
    dict->n = 0;
    if (argc <= k) return true;
    napi_valuetype t;
    napi_typeof(env, argv[k], &t);
    if (t == napi_undefined || t == napi_null) return true;
    if (!get_u8(env, argv[k], dict)) {
        napi_throw_type_error(env, nullptr, "dictionary must be Uint8Array");
        return false;
    }
    if (dict->n) dicts->assign(n, zlb_dict{0, (uint64_t)dict->n});
    return true;
}

// deflateBatch(inputs, compressionType, chunkBytes, flags, mode = 0, dictionary?)  <- new RawDeflate(input, opts).compress()
static napi_value DeflateBatch(napi_env env, napi_callback_info info)
{
    size_t argc = 6;
    napi_value argv[6];
    napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr);
    if (!ensure_ctx(env)) return nullptr;
    uint32_t n = 0, ctype = 2, chunk = 0, flags = 0, mode = ZLB_MODE_COMPAT;
    napi_get_array_length(env, argv[0], &n);
    napi_get_value_uint32(env, argv[1], &ctype);
    napi_get_value_uint32(env, argv[2], &chunk);
    napi_get_value_uint32(env, argv[3], &flags);
    if (argc > 4) napi_get_value_uint32(env, argv[4], &mode);   // ZLB_MODE_FAST | ZLB_MODE_PRIMED | ZLB_MODE_SMALLEST
    Bytes dict;
    std::vector<zlb_dict> dicts;
    if (!get_dict(env, argc, argv, 5, n, &dict, &dicts)) return nullptr;
    // primed mode and dictionaries: chunks of at most 32 KiB (the slots are sized with the chunk size used)
    if ((mode & ZLB_MODE_PRIMED || !dicts.empty()) && (chunk == 0 || chunk > ZLB_PRIMED_CHUNK)) chunk = ZLB_PRIMED_CHUNK;
    std::vector<zlb_item> items(n);
    std::vector<zlb_result> res(n);
    std::vector<Bytes> in(n);
    uint64_t in_total = 0, out_total = 0;
    for (uint32_t i = 0; i < n; ++i) {
        napi_value e;
        napi_get_element(env, argv[0], i, &e);
        if (!get_u8(env, e, &in[i])) {
            napi_throw_type_error(env, nullptr, "inputs must be Uint8Array");
            return nullptr;
        }
        items[i].in_off = in_total;
        items[i].in_len = in[i].n;
        items[i].out_off = out_total;
        items[i].out_cap = zlb_deflate_bound(in[i].n, chunk, (int)ctype);
        in_total += in[i].n;
        out_total += items[i].out_cap;
    }
    // one input that already lives in page-locked memory (hostAlloc) travels as it is; anything else is gathered
    const bool direct = n == 1 && in[0].n && zlb_host_is_pinned(in[0].p);
    HostBuf blob(direct ? 1 : in_total), out(out_total);
    if (!blob.p || !out.p) {
        napi_throw_error(env, nullptr, "zlib.ts-b200: out of host memory");
        return nullptr;
    }
    if (!direct)
        for (uint32_t i = 0; i < n; ++i)
            if (in[i].n) memcpy(blob.p + items[i].in_off, in[i].p, in[i].n);
    int rc = zlb_deflate_batch_dict_host(g_ctx, direct ? in[0].p : blob.p, in_total, out.p, out_total, dict.p, dict.n,
                                         dicts.empty() ? nullptr : dicts.data(), items.data(), res.data(), n, (int)mode,
                                         (int)ctype, chunk, flags);
    if (rc != ZLB_OK) {
        napi_throw_error(env, nullptr, zlb_last_error(g_ctx));
        return nullptr;
    }
    napi_value result, outs;
    napi_create_object(env, &result);
    napi_create_array_with_length(env, n, &outs);
    std::vector<double> crc(n), adler(n);
    const uint8_t* out_base = out.p;
    Outputs views(env, out);  // the result buffer now belongs to the ArrayBuffer the outputs are views of
    for (uint32_t i = 0; i < n; ++i) {
        napi_set_element(env, outs, i, views.at(out_base, items[i].out_off, (size_t)res[i].out_len));
        crc[i] = res[i].crc32;
        adler[i] = res[i].adler32;
    }
    napi_set_named_property(env, result, "outputs", outs);
    napi_set_named_property(env, result, "crc32", num_array(env, crc));
    napi_set_named_property(env, result, "adler32", num_array(env, adler));
    return result;
}

// inflateBatch(input, offsets, lengths, caps, flags, dictionary?)  <- new RawInflate(input, {index}).decompress()
static napi_value InflateBatch(napi_env env, napi_callback_info info)
{
    size_t argc = 6;
    napi_value argv[6];
    napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr);
    if (!ensure_ctx(env)) return nullptr;
    Bytes in;
    if (!get_u8(env, argv[0], &in)) {
        napi_throw_type_error(env, nullptr, "input must be Uint8Array");
        return nullptr;
    }
    std::vector<double> offs = get_numbers(env, argv[1]), lens = get_numbers(env, argv[2]), caps = get_numbers(env, argv[3]);
    uint32_t flags = 0;
    napi_get_value_uint32(env, argv[4], &flags);
    const size_t n = offs.size();
    Bytes dict;
    std::vector<zlb_dict> dicts;
    if (!get_dict(env, argc, argv, 5, n, &dict, &dicts)) return nullptr;
    std::vector<zlb_item> items(n);
    std::vector<zlb_result> res(n);
    uint64_t out_total = 0;
    for (size_t i = 0; i < n; ++i) {
        items[i].in_off = (uint64_t)offs[i];
        items[i].in_len = (uint64_t)lens[i];
        items[i].out_off = out_total;
        items[i].out_cap = (uint64_t)caps[i];
        out_total += items[i].out_cap;
    }
    // the input is one Uint8Array already: page-locked if it came from hostAlloc(), otherwise the library stages it
    // through its own page-locked shadow (copy threads, overlapped with the transfers)
    HostBuf out(out_total);
    if (!out.p) {
        napi_throw_error(env, nullptr, "zlib.ts-b200: out of host memory");
        return nullptr;
    }
    int rc = zlb_inflate_batch_dict_host(g_ctx, in.p, in.n, out.p, out_total, dict.p, dict.n,
                                         dicts.empty() ? nullptr : dicts.data(), items.data(), res.data(), n, flags);
    if (rc != ZLB_OK) {
        napi_throw_error(env, nullptr, zlb_last_error(g_ctx));
        return nullptr;
    }
    napi_value result, outs;
    napi_create_object(env, &result);
    napi_create_array_with_length(env, n, &outs);
    std::vector<double> st(n), used(n), crc(n), adler(n);
    const uint8_t* out_base = out.p;
    Outputs views(env, out);
    for (size_t i = 0; i < n; ++i) {
        napi_set_element(env, outs, (uint32_t)i, views.at(out_base, items[i].out_off, (size_t)res[i].out_len));
        st[i] = res[i].status;
        used[i] = (double)res[i].in_used;
        crc[i] = res[i].crc32;
        adler[i] = res[i].adler32;
    }
    napi_set_named_property(env, result, "outputs", outs);
    napi_set_named_property(env, result, "status", num_array(env, st));
    napi_set_named_property(env, result, "inUsed", num_array(env, used));
    napi_set_named_property(env, result, "crc32", num_array(env, crc));
    napi_set_named_property(env, result, "adler32", num_array(env, adler));
    return result;
}

// checksumBatch(inputs, kinds)  <- CRC32.create / Adler32.create
static napi_value ChecksumBatch(napi_env env, napi_callback_info info)
{
    size_t argc = 2;
    napi_value argv[2];
    napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr);
    if (!ensure_ctx(env)) return nullptr;
    uint32_t n = 0, kinds = 3;
    napi_get_array_length(env, argv[0], &n);
    napi_get_value_uint32(env, argv[1], &kinds);
    std::vector<zlb_item> items(n);
    std::vector<zlb_result> res(n);
    std::vector<Bytes> in(n);
    uint64_t total = 0;
    for (uint32_t i = 0; i < n; ++i) {
        napi_value e;
        napi_get_element(env, argv[0], i, &e);
        if (!get_u8(env, e, &in[i])) {
            napi_throw_type_error(env, nullptr, "inputs must be Uint8Array");
            return nullptr;
        }
        items[i].in_off = total;
        items[i].in_len = in[i].n;
        total += in[i].n;
    }
    const bool direct = n == 1 && in[0].n && zlb_host_is_pinned(in[0].p);
    HostBuf blob(direct ? 1 : total);
    if (!blob.p) {
        napi_throw_error(env, nullptr, "zlib.ts-b200: out of host memory");
        return nullptr;
    }
    if (!direct)
        for (uint32_t i = 0; i < n; ++i)
            if (in[i].n) memcpy(blob.p + items[i].in_off, in[i].p, in[i].n);
    if (zlb_checksum_batch_host(g_ctx, direct ? in[0].p : blob.p, total, items.data(), res.data(), n, kinds) != ZLB_OK) {
        napi_throw_error(env, nullptr, zlb_last_error(g_ctx));
        return nullptr;
    }
    std::vector<double> crc(n), adler(n);
    for (uint32_t i = 0; i < n; ++i) {
        crc[i] = res[i].crc32;
        adler[i] = res[i].adler32;
    }
    napi_value result;
    napi_create_object(env, &result);
    napi_set_named_property(env, result, "crc32", num_array(env, crc));
    napi_set_named_property(env, result, "adler32", num_array(env, adler));
    return result;
}

// archive(kind, inputs, heads, cdirs, methods, tail, compressionType, chunkBytes, mode)
//   <- Deflate.compress (src/Deflate.ts:60-99), GZip.compress (src/GZip.ts:96-194), Zip.compress (src/Zip.ts:117-372)
static napi_value Archive(napi_env env, napi_callback_info info)
{
    size_t argc = 9;
    napi_value argv[9];
    napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr);
    if (!ensure_ctx(env)) return nullptr;
    uint32_t kind = 0, n = 0, ctype = 2, chunk = 0, mode = 0;
    napi_get_value_uint32(env, argv[0], &kind);
    napi_get_array_length(env, argv[1], &n);
    napi_get_value_uint32(env, argv[6], &ctype);
    napi_get_value_uint32(env, argv[7], &chunk);
    napi_get_value_uint32(env, argv[8], &mode);
    napi_valuetype cd_t, me_t;
    napi_typeof(env, argv[3], &cd_t);
    napi_typeof(env, argv[4], &me_t);
    const bool has_cdir = cd_t == napi_object, has_methods = me_t == napi_object;
    std::vector<double> methods = has_methods ? get_numbers(env, argv[4]) : std::vector<double>();
    std::vector<zlb_entry> ent(n);
    std::vector<zlb_result> res(n);
    std::vector<Bytes> in(n), head(n), cdir(n);
    Bytes tail = {nullptr, 0};
    get_u8(env, argv[5], &tail);
    uint64_t in_total = 0, meta_total = 0;
    for (uint32_t i = 0; i < n; ++i) {
        napi_value e;
        napi_get_element(env, argv[1], i, &e);
        bool ok = get_u8(env, e, &in[i]);
        napi_get_element(env, argv[2], i, &e);
        ok = ok && get_u8(env, e, &head[i]);
        if (has_cdir) {
            napi_get_element(env, argv[3], i, &e);
            ok = ok && get_u8(env, e, &cdir[i]);
        } else {
            cdir[i] = {nullptr, 0};
        }
        if (!ok) {
            napi_throw_type_error(env, nullptr, "inputs, heads and cdirs must be Uint8Array");
            return nullptr;
        }
        memset(&ent[i], 0, sizeof ent[i]);
        ent[i].in_off = in_total;
        ent[i].in_len = in[i].n;
        ent[i].head_off = meta_total;
        ent[i].head_len = (uint32_t)head[i].n;
        ent[i].cdir_off = meta_total + head[i].n;
        ent[i].cdir_len = (uint32_t)cdir[i].n;
        ent[i].method = has_methods ? (uint32_t)methods[i] : 8u;
        in_total += in[i].n;
        meta_total += head[i].n + cdir[i].n;
    }
    const uint64_t tail_off = meta_total;
    meta_total += tail.n;
    const uint32_t cb = (mode & ZLB_MODE_PRIMED) && (chunk == 0 || chunk > ZLB_PRIMED_CHUNK) ? ZLB_PRIMED_CHUNK : chunk;
    HostBuf blob(in_total), meta(meta_total), out(zlb_archive_bound((int)kind, ent.data(), n, tail.n, cb, (int)ctype) + 1);
    if (!blob.p || !meta.p || !out.p) {
        napi_throw_error(env, nullptr, "zlib.ts-b200: out of host memory");
        return nullptr;
    }
    for (uint32_t i = 0; i < n; ++i) {
        if (in[i].n) memcpy(blob.p + ent[i].in_off, in[i].p, in[i].n);
        if (head[i].n) memcpy(meta.p + ent[i].head_off, head[i].p, head[i].n);
        if (cdir[i].n) memcpy(meta.p + ent[i].cdir_off, cdir[i].p, cdir[i].n);
    }
    if (tail.n) memcpy(meta.p + tail_off, tail.p, tail.n);
    uint64_t total = 0;
    int rc = zlb_archive_host(g_ctx, (int)kind, blob.p, in_total, meta.p, meta_total, ent.data(), n, tail_off,
                              tail.n, out.p, out.n, &total, res.data(), (int)mode, (int)ctype, chunk);
    if (rc != ZLB_OK) {
        napi_throw_error(env, nullptr, zlb_last_error(g_ctx));
        return nullptr;
    }
    std::vector<double> crc(n), adler(n), offs(n), lens(n);
    for (uint32_t i = 0; i < n; ++i) {
        crc[i] = res[i].crc32;
        adler[i] = res[i].adler32;
        offs[i] = (double)res[i].in_used;
        lens[i] = (double)res[i].out_len;
    }
    napi_value result;
    napi_create_object(env, &result);
    const uint8_t* out_base = out.p;
    Outputs views(env, out);  // the archive is a view of the page-locked result buffer: no copy
    napi_set_named_property(env, result, "output", views.at(out_base, 0, (size_t)total));
    napi_set_named_property(env, result, "crc32", num_array(env, crc));
    napi_set_named_property(env, result, "adler32", num_array(env, adler));
    napi_set_named_property(env, result, "offsets", num_array(env, offs));
    napi_set_named_property(env, result, "lengths", num_array(env, lens));
    return result;
}

static napi_value Combine(napi_env env, napi_callback_info info, bool crc)
{
    size_t argc = 3;
    napi_value argv[3];
    napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr);
    double a, b, n;
    napi_get_value_double(env, argv[0], &a);
    napi_get_value_double(env, argv[1], &b);
    napi_get_value_double(env, argv[2], &n);
    uint32_t r = crc ? zlb_crc32_combine((uint32_t)a, (uint32_t)b, (uint64_t)n)
                     : zlb_adler32_combine((uint32_t)a, (uint32_t)b, (uint64_t)n);
    napi_value v;
    napi_create_uint32(env, r, &v);
    return v;
}
static napi_value Crc32Combine(napi_env env, napi_callback_info info) { return Combine(env, info, true); }
static napi_value Adler32Combine(napi_env env, napi_callback_info info) { return Combine(env, info, false); }

// hostAlloc(bytes) -> Uint8Array over page-locked memory (zlb_host_alloc): what a caller fills instead of
// `new Uint8Array(n)` (src/RawDeflate.ts:58) when the data should travel without a staging copy
static napi_value HostAlloc(napi_env env, napi_callback_info info)
{
    size_t argc = 1;
    napi_value argv[1];
    napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr);
    double bytes = 0;
    napi_get_value_double(env, argv[0], &bytes);
    const size_t n = bytes > 0 ? (size_t)bytes : 0;
    void* p = nullptr;
    if (zlb_host_alloc(n ? n : 1, &p) != ZLB_OK) {
        napi_throw_error(env, nullptr, "zlib.ts-b200: out of host memory");
        return nullptr;
    }
    napi_value ab = adopt_buffer(env, (uint8_t*)p, n ? n : 1);
    if (!ab) {
        napi_throw_error(env, nullptr, "zlib.ts-b200: this runtime does not allow external ArrayBuffers");
        return nullptr;
    }
    return view_u8(env, ab, 0, n);
}

static napi_value Init(napi_env env, napi_value exports)
{
    napi_property_descriptor d[] = {
        {"deflateBatch", nullptr, DeflateBatch, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"inflateBatch", nullptr, InflateBatch, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"checksumBatch", nullptr, ChecksumBatch, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"archive", nullptr, Archive, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"crc32Combine", nullptr, Crc32Combine, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"adler32Combine", nullptr, Adler32Combine, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"hostAlloc", nullptr, HostAlloc, nullptr, nullptr, nullptr, napi_default, nullptr},
    };
    napi_define_properties(env, exports, sizeof d / sizeof d[0], d);
    return exports;
}
NAPI_MODULE(NODE_GYP_MODULE_NAME, Init)
