// zsgpu_addon.cc -- Node-API addon: pure marshalling between JavaScript typed arrays and the C ABI of
// include/zsgpu.h.  NOT compiled in this repository's image (no node, no node_api.h); it is the
// binding a zlib-streams-ts maintainer adds (see INTEGRATION.md).  Build:
//   g++ -O2 -shared -fPIC -I<node headers> -I../../include zsgpu_addon.cc
//       -L../../zlib-streams-ts_b200 -lzsgpu -Wl,-rpath,'$ORIGIN' -o zsgpu.node
#include <node_api.h>

#include <cstdint>
#include <cstdio>
#include <cstring>
#include <vector>

#include "zsgpu.h"

namespace {

zs_ctx* g_ctx = nullptr;

napi_value throw_code(napi_env env, int rc, const char* where) {
    char msg[320];
    snprintf(msg, sizeof msg, "%s failed: %d (%s)", where, rc, g_ctx ? zs_last_error(g_ctx) : "no context");
    napi_throw_error(env, nullptr, msg);
    return nullptr;
}

bool u8(napi_env env, napi_value v, uint8_t** p, size_t* n) {
    napi_typedarray_type t; napi_value ab; size_t off;
    return napi_get_typedarray_info(env, v, &t, n, (void**)p, &ab, &off) == napi_ok && t == napi_uint8_array;
}
int32_t i32(napi_env env, napi_value v) { int32_t x = 0; napi_get_value_int32(env, v, &x); return x; }
napi_value num(napi_env env, double x) { napi_value v; napi_create_double(env, x, &v); return v; }

// init(device) -> void                                                zs_ctx_create
napi_value Init(napi_env env, napi_callback_info info) {
    size_t argc = 1; napi_value a[1];
    napi_get_cb_info(env, info, &argc, a, nullptr, nullptr);
    if (g_ctx) return nullptr;
    int rc = zs_ctx_create(argc ? i32(env, a[0]) : 0, nullptr, &g_ctx);
    return rc == ZS_OK ? nullptr : throw_code(env, rc, "zs_ctx_create");   // no CPU fallback: it throws
}

// createDeflateDictionary(dict: Uint8Array) -> {handle, id}            zs_deflate_dict_create
// (the handle is destroyed when it is garbage collected)
void FreeDict(napi_env, void* data, void*) { zs_deflate_dict_destroy((zs_deflate_dict*)data); }
napi_value CreateDeflateDictionary(napi_env env, napi_callback_info info) {
    size_t argc = 1; napi_value a[1];
    napi_get_cb_info(env, info, &argc, a, nullptr, nullptr);
    uint8_t* p; size_t n;
    if (argc < 1 || !u8(env, a[0], &p, &n)) return throw_code(env, ZS_STREAM_ERROR, "createDeflateDictionary");
    zs_deflate_dict* d = nullptr;
    int rc = zs_deflate_dict_create(g_ctx, p, n, &d);
    if (rc != ZS_OK) return throw_code(env, rc, "zs_deflate_dict_create");
    napi_value h, o;
    napi_create_external(env, d, FreeDict, nullptr, &h);
    napi_create_object(env, &o);
    napi_set_named_property(env, o, "handle", h);
    napi_set_named_property(env, o, "id", num(env, (double)zs_deflate_dict_id(d)));
    return o;
}

// ---- random access into one stream (zs_inflate_index_*); an index handle is destroyed when it is garbage collected ----
void FreeIndex(napi_env, void* data, void*) { zs_inflate_index_destroy((zs_inflate_index*)data); }
bool u64s(napi_env env, napi_value v, uint64_t** p, size_t* n) {
    napi_typedarray_type t; napi_value ab; size_t off;
    return napi_get_typedarray_info(env, v, &t, n, (void**)p, &ab, &off) == napi_ok && t == napi_biguint64_array;
}
napi_value index_object(napi_env env, zs_inflate_index* x) {
    zs_inflate_index_info inf;
    zs_inflate_index_info_get(x, &inf);
    napi_value h, o;
    napi_create_external(env, x, FreeIndex, nullptr, &h);
    napi_create_object(env, &o);
    napi_set_named_property(env, o, "handle", h);
    napi_set_named_property(env, o, "points", num(env, (double)inf.n_points));
    napi_set_named_property(env, o, "outLen", num(env, (double)inf.out_len));
    return o;
}

// inflateIndexBuild(input: Uint8Array, windowBits, span, out: Uint8Array[, dict: Uint8Array])
//   -> {index: {handle, points, outLen} | null, outLen, inUsed, check, status, msg: Buffer}      zs_inflate_index_build
napi_value InflateIndexBuild(napi_env env, napi_callback_info info) {
    size_t argc = 5; napi_value a[5];
    napi_get_cb_info(env, info, &argc, a, nullptr, nullptr);
    uint8_t *in, *out, *dict = nullptr; size_t n_in, n_out, n_dict = 0;
    if (argc < 4 || !u8(env, a[0], &in, &n_in) || !u8(env, a[3], &out, &n_out)) return throw_code(env, ZS_STREAM_ERROR, "inflateIndexBuild");
    if (argc >= 5 && !u8(env, a[4], &dict, &n_dict)) n_dict = 0;
    uint32_t span = 0;
    napi_get_value_uint32(env, a[2], &span);
    zs_inflate_index_result r;
    zs_inflate_index* x = nullptr;
    int rc = zs_inflate_index_build(g_ctx, in, n_in, i32(env, a[1]), span, out, n_out, n_dict ? dict : nullptr, n_dict, &r, &x);
    if (rc != ZS_OK) return throw_code(env, rc, "zs_inflate_index_build");
    const char* msg = r.status == ZS_STREAM_END ? "" : zs_inflate_message(r.detail);
    napi_value o, m, ix; void* dst = nullptr;
    napi_create_object(env, &o);
    if (x) ix = index_object(env, x);
    else napi_create_object(env, &ix);   // (no index: an object without a handle)
    napi_set_named_property(env, o, "index", ix);
    napi_set_named_property(env, o, "outLen", num(env, (double)r.out_len));
    napi_set_named_property(env, o, "inUsed", num(env, (double)r.in_used));
    napi_set_named_property(env, o, "check", num(env, (double)r.check));
    napi_set_named_property(env, o, "status", num(env, (double)r.status));
    napi_create_buffer_copy(env, strlen(msg), msg, &dst, &m);
    napi_set_named_property(env, o, "msg", m);
    return o;
}

// inflateIndexExtract(handle, input: Uint8Array, off: BigUint64Array, len: BigUint64Array, out: Uint8Array,
//                     outOff: BigUint64Array, got: BigUint64Array, status: Int32Array) -> void   zs_inflate_index_extract
// (status is read as an Int32Array, like inflateBatch's)
napi_value InflateIndexExtract(napi_env env, napi_callback_info info) {
    size_t argc = 8; napi_value a[8];
    napi_get_cb_info(env, info, &argc, a, nullptr, nullptr);
    void* x = nullptr;
    uint8_t *in, *out; size_t n_in, n_out;
    uint64_t *off, *len, *out_off, *got; size_t n1, n2, n3, n4;
    void* status; size_t n5; napi_typedarray_type t; napi_value ab; size_t bo;
    if (argc < 8 || napi_get_value_external(env, a[0], &x) != napi_ok || !u8(env, a[1], &in, &n_in) || !u64s(env, a[2], &off, &n1) ||
        !u64s(env, a[3], &len, &n2) || !u8(env, a[4], &out, &n_out) || !u64s(env, a[5], &out_off, &n3) ||
        !u64s(env, a[6], &got, &n4) || napi_get_typedarray_info(env, a[7], &t, &n5, &status, &ab, &bo) != napi_ok ||
        n2 < n1 || n3 < n1 || n4 < n1 || n5 < n1)
        return throw_code(env, ZS_STREAM_ERROR, "inflateIndexExtract");
    int rc = zs_inflate_index_extract(g_ctx, (const zs_inflate_index*)x, in, n_in, off, len, (uint32_t)n1, out, n_out, out_off, got,
                                      (int32_t*)status);
    return rc == ZS_OK ? nullptr : throw_code(env, rc, "zs_inflate_index_extract");
}

// inflateIndexExport(handle) -> Buffer (the format of zsgpu.h)                   zs_inflate_index_export
napi_value InflateIndexExport(napi_env env, napi_callback_info info) {
    size_t argc = 1; napi_value a[1];
    napi_get_cb_info(env, info, &argc, a, nullptr, nullptr);
    void* x = nullptr;
    if (argc < 1 || napi_get_value_external(env, a[0], &x) != napi_ok) return throw_code(env, ZS_STREAM_ERROR, "inflateIndexExport");
    uint64_t n = 0;
    int rc = zs_inflate_index_export((const zs_inflate_index*)x, nullptr, 0, &n);
    std::vector<uint8_t> blob(n);
    if (rc == ZS_OK) rc = zs_inflate_index_export((const zs_inflate_index*)x, blob.data(), n, &n);
    if (rc != ZS_OK) return throw_code(env, rc, "zs_inflate_index_export");
    napi_value b; void* dst = nullptr;
    napi_create_buffer_copy(env, blob.size(), blob.data(), &dst, &b);
    return b;
}

// inflateIndexImport(blob: Uint8Array) -> {handle, points, outLen}                zs_inflate_index_import
napi_value InflateIndexImport(napi_env env, napi_callback_info info) {
    size_t argc = 1; napi_value a[1];
    napi_get_cb_info(env, info, &argc, a, nullptr, nullptr);
    uint8_t* p; size_t n;
    if (argc < 1 || !u8(env, a[0], &p, &n)) return throw_code(env, ZS_STREAM_ERROR, "inflateIndexImport");
    zs_inflate_index* x = nullptr;
    int rc = zs_inflate_index_import(g_ctx, p, n, &x);
    if (rc != ZS_OK) return throw_code(env, rc, "zs_inflate_index_import");
    return index_object(env, x);
}

// deflateBatch(input: Uint8Array, chunkSize, level, wrap, mode, flags, out: Uint8Array, outOff: BigUint64Array
//              [, dictionary handle]) -> {bytes, bits, check, blocks}   zs_deflate_batch / zs_deflate_batch_dict
napi_value DeflateBatch(napi_env env, napi_callback_info info) {
    size_t argc = 9; napi_value a[9];
    napi_get_cb_info(env, info, &argc, a, nullptr, nullptr);
    uint8_t *in, *out; size_t n, cap;
    if (!u8(env, a[0], &in, &n) || !u8(env, a[6], &out, &cap)) return throw_code(env, ZS_STREAM_ERROR, "deflateBatch");
    uint32_t chunk = (uint32_t)i32(env, a[1]);
    uint32_t n_chunks = n ? (uint32_t)((n + chunk - 1) / chunk) : 1;
    uint64_t* off = nullptr; size_t off_n = 0; napi_typedarray_type t; napi_value ab; size_t bo;
    napi_get_typedarray_info(env, a[7], &t, &off_n, (void**)&off, &ab, &bo);
    zs_deflate_result r;
    void* dict = nullptr;
    if (argc >= 9 && napi_get_value_external(env, a[8], &dict) != napi_ok) dict = nullptr;
    int rc = dict ? zs_deflate_batch_dict(g_ctx, (const zs_deflate_dict*)dict, in, n, nullptr, n_chunks, chunk, i32(env, a[2]),
                                          i32(env, a[3]), (uint32_t)i32(env, a[5]), out, cap,
                                          off_n >= n_chunks + 1 ? off : nullptr, nullptr, nullptr, &r)
                  : zs_deflate_batch(g_ctx, in, n, nullptr, n_chunks, chunk, i32(env, a[2]), i32(env, a[3]), i32(env, a[4]),
                                     (uint32_t)i32(env, a[5]), out, cap, off_n >= n_chunks + 1 ? off : nullptr, nullptr, nullptr, &r);
    if (rc != ZS_OK) return throw_code(env, rc, "zs_deflate_batch");
    napi_value o; napi_create_object(env, &o);
    napi_set_named_property(env, o, "bytes", num(env, (double)r.total_out_bytes));
    napi_set_named_property(env, o, "bits", num(env, (double)r.total_out_bits));
    napi_set_named_property(env, o, "check", num(env, (double)r.check));
    napi_set_named_property(env, o, "blocks", num(env, (double)r.n_blocks));
    return o;
}

// deflateIndexed(input: Uint8Array, chunkSize, level, wrap, flags, span, out: Uint8Array[, outOff: BigUint64Array])
//   -> {outLen, check, index: {handle, points, outLen}}                zs_deflate_indexed
// One stitched stream and its index for `span`, made from the encoder's block layout (no decode).
napi_value DeflateIndexed(napi_env env, napi_callback_info info) {
    size_t argc = 8; napi_value a[8];
    napi_get_cb_info(env, info, &argc, a, nullptr, nullptr);
    uint8_t *in, *out; size_t n, cap;
    if (argc < 7 || !u8(env, a[0], &in, &n) || !u8(env, a[6], &out, &cap)) return throw_code(env, ZS_STREAM_ERROR, "deflateIndexed");
    uint32_t chunk = (uint32_t)i32(env, a[1]);
    if (chunk == 0) return throw_code(env, ZS_STREAM_ERROR, "deflateIndexed");
    uint32_t n_chunks = n ? (uint32_t)((n + chunk - 1) / chunk) : 1;
    uint32_t span = 0;
    napi_get_value_uint32(env, a[5], &span);
    uint64_t* off = nullptr; size_t off_n = 0;
    if (argc >= 8 && !u64s(env, a[7], &off, &off_n)) off_n = 0;
    zs_deflate_result r;
    zs_inflate_index* x = nullptr;
    int rc = zs_deflate_indexed(g_ctx, in, n, nullptr, n_chunks, chunk, i32(env, a[2]), i32(env, a[3]), (uint32_t)i32(env, a[4]),
                                span, out, cap, off_n >= n_chunks + 1 ? off : nullptr, nullptr, nullptr, &r, &x);
    if (rc != ZS_OK) return throw_code(env, rc, "zs_deflate_indexed");
    napi_value o; napi_create_object(env, &o);
    napi_set_named_property(env, o, "outLen", num(env, (double)r.total_out_bytes));
    napi_set_named_property(env, o, "check", num(env, (double)r.check));
    napi_set_named_property(env, o, "index", index_object(env, x));
    return o;
}

// inflateBatch(input, inOff: BigUint64Array, windowBits, out, outOff: BigUint64Array, outLen: BigUint64Array,
//              checks: Uint32Array, status: Int32Array[, dicts: Uint8Array, dictRng: BigUint64Array (2 per stream)])
//   -> void                                                            zs_inflate_batch
napi_value InflateBatch(napi_env env, napi_callback_info info) {
    size_t argc = 10; napi_value a[10];
    napi_get_cb_info(env, info, &argc, a, nullptr, nullptr);
    uint8_t *in, *out; size_t n_in, n_out;
    if (!u8(env, a[0], &in, &n_in) || !u8(env, a[3], &out, &n_out)) return throw_code(env, ZS_STREAM_ERROR, "inflateBatch");
    void *in_off, *out_off, *out_len, *checks, *status; size_t n1, n2, n3, n4, n5;
    napi_typedarray_type t; napi_value ab; size_t bo;
    napi_get_typedarray_info(env, a[1], &t, &n1, &in_off, &ab, &bo);
    napi_get_typedarray_info(env, a[4], &t, &n2, &out_off, &ab, &bo);
    napi_get_typedarray_info(env, a[5], &t, &n3, &out_len, &ab, &bo);
    napi_get_typedarray_info(env, a[6], &t, &n4, &checks, &ab, &bo);
    napi_get_typedarray_info(env, a[7], &t, &n5, &status, &ab, &bo);
    uint8_t* dict = nullptr; size_t n_dict = 0; void* dict_rng = nullptr; size_t n6 = 0;
    if (argc >= 10 && u8(env, a[8], &dict, &n_dict)) {
        napi_get_typedarray_info(env, a[9], &t, &n6, &dict_rng, &ab, &bo);
        if (n6 < 2 * (n1 - 1)) return throw_code(env, ZS_STREAM_ERROR, "inflateBatch: dictRng needs 2 entries per stream");
    }
    int rc = zs_inflate_batch(g_ctx, in, (const uint64_t*)in_off, (uint32_t)(n1 - 1), i32(env, a[2]), out,
                              (const uint64_t*)out_off, (uint64_t*)out_len, nullptr, (uint32_t*)checks, (int32_t*)status,
                              dict_rng ? dict : nullptr, (const uint64_t*)dict_rng, dict_rng ? n_dict : 0);
    return rc == ZS_OK ? nullptr : throw_code(env, rc, "zs_inflate_batch");
}

// gunzip(input: Uint8Array, out: Uint8Array[, members: BigUint64Array, 5 per member: inOff, inLen, outOff, outLen,
//        crc32]) -> {outLen, inUsed, members, status, msg: Buffer}        zs_gunzip
napi_value Gunzip(napi_env env, napi_callback_info info) {
    size_t argc = 3; napi_value a[3];
    napi_get_cb_info(env, info, &argc, a, nullptr, nullptr);
    uint8_t *in, *out; size_t n_in, n_out;
    if (argc < 2 || !u8(env, a[0], &in, &n_in) || !u8(env, a[1], &out, &n_out)) return throw_code(env, ZS_STREAM_ERROR, "gunzip");
    uint64_t* tab = nullptr; size_t n_tab = 0;
    napi_typedarray_type t; napi_value ab; size_t bo;
    if (argc >= 3 && (napi_get_typedarray_info(env, a[2], &t, &n_tab, (void**)&tab, &ab, &bo) != napi_ok || t != napi_biguint64_array))
        n_tab = 0;
    std::vector<zs_gz_member> table(n_tab / 5);
    zs_gunzip_result r;
    int rc = zs_gunzip(g_ctx, in, n_in, out, n_out, &r, table.empty() ? nullptr : table.data(), table.size());
    if (rc != ZS_OK) return throw_code(env, rc, "zs_gunzip");
    for (size_t i = 0; i < table.size() && i < r.n_members; ++i) {
        const zs_gz_member& e = table[i];
        const uint64_t f[5] = {e.in_off, e.in_len, e.out_off, e.out_len, e.crc32};
        memcpy(tab + 5 * i, f, sizeof f);
    }
    const char* msg = r.status == ZS_STREAM_END ? "" : zs_inflate_message(r.detail);
    napi_value o, m; void* dst = nullptr;
    napi_create_object(env, &o);
    napi_set_named_property(env, o, "outLen", num(env, (double)r.out_len));
    napi_set_named_property(env, o, "inUsed", num(env, (double)r.in_used));
    napi_set_named_property(env, o, "members", num(env, (double)r.n_members));
    napi_set_named_property(env, o, "status", num(env, (double)r.status));
    napi_create_buffer_copy(env, msg ? strlen(msg) : 0, msg ? msg : "", &dst, &m);
    napi_set_named_property(env, o, "msg", m);
    return o;
}

// checksum(kind, init, buf) -> number                                  zs_checksum
napi_value Checksum(napi_env env, napi_callback_info info) {
    size_t argc = 3; napi_value a[3];
    napi_get_cb_info(env, info, &argc, a, nullptr, nullptr);
    uint8_t* p; size_t n; uint32_t init = 0, res = 0;
    napi_get_value_uint32(env, a[1], &init);
    if (!u8(env, a[2], &p, &n)) return throw_code(env, ZS_STREAM_ERROR, "checksum");
    int rc = zs_checksum(g_ctx, i32(env, a[0]), p, n, init, &res);
    return rc == ZS_OK ? num(env, res) : throw_code(env, rc, "zs_checksum");
}

// ---- streaming shim: one external zs_stream per JS Stream object -------------------------------------
// The holder owns what the C ABI only borrows: the gzip header record inflateGetHeader registers and
// the buffers its extra / name / comment fields point at.
struct Holder {
    zs_stream s;
    zs_gz_header gz;
    std::vector<uint8_t> extra, name, comment;
};
void FreeStream(napi_env, void* data, void*) { delete (Holder*)data; }
Holder* holder_of(napi_env env, napi_value v) { void* p = nullptr; napi_get_value_external(env, v, &p); return (Holder*)p; }
zs_stream* strm_of(napi_env env, napi_value v) { Holder* h = holder_of(env, v); return h ? &h->s : nullptr; }

// streamNew() -> external
napi_value StreamNew(napi_env env, napi_callback_info) {
    Holder* h = new Holder(); memset(&h->s, 0, sizeof h->s); memset(&h->gz, 0, sizeof h->gz);
    napi_value v; napi_create_external(env, h, FreeStream, nullptr, &v); return v;
}
// deflateInit2(h, level, method, windowBits, memLevel, strategy) -> rc  zs_stream_deflate_init
napi_value DeflateInit2(napi_env env, napi_callback_info info) {
    size_t argc = 6; napi_value a[6]; napi_get_cb_info(env, info, &argc, a, nullptr, nullptr);
    return num(env, zs_stream_deflate_init(g_ctx, strm_of(env, a[0]), i32(env, a[1]), i32(env, a[2]), i32(env, a[3]),
                                           i32(env, a[4]), i32(env, a[5])));
}
// inflateInit2(h, windowBits) -> rc                                     zs_stream_inflate_init
napi_value InflateInit2(napi_env env, napi_callback_info info) {
    size_t argc = 2; napi_value a[2]; napi_get_cb_info(env, info, &argc, a, nullptr, nullptr);
    return num(env, zs_stream_inflate_init(g_ctx, strm_of(env, a[0]), i32(env, a[1])));
}
// process(h, which, flush, next_in, in_index, avail_in, next_out, out_index, avail_out)
//   -> [rc, used_in, made_out, total_in, total_out, adler]              zs_stream_deflate / zs_stream_inflate
napi_value Process(napi_env env, napi_callback_info info) {
    size_t argc = 9; napi_value a[9]; napi_get_cb_info(env, info, &argc, a, nullptr, nullptr);
    zs_stream* s = strm_of(env, a[0]);
    uint8_t *in = nullptr, *out = nullptr; size_t n_in = 0, n_out = 0;
    u8(env, a[3], &in, &n_in); u8(env, a[6], &out, &n_out);
    uint32_t ii = (uint32_t)i32(env, a[4]), ai = (uint32_t)i32(env, a[5]), oi = (uint32_t)i32(env, a[7]), ao = (uint32_t)i32(env, a[8]);
    s->next_in = in ? in + ii : nullptr; s->avail_in = ai;
    s->next_out = out ? out + oi : nullptr; s->avail_out = ao;
    // which: 0 deflate, 1 inflate, 2 deflateParams (flush carries level + 1 | strategy << 8; it may have to
    // flush pending input through the same buffers, deflate.ts:572-579)
    const int which = i32(env, a[1]), f = i32(env, a[2]);
    int rc = which == 0 ? zs_stream_deflate(s, f) : which == 1 ? zs_stream_inflate(s, f)
                        : zs_stream_deflate_params(s, (f & 0xff) - 1, f >> 8);
    napi_value arr; napi_create_array_with_length(env, 6, &arr);
    double vals[6] = {(double)rc, (double)(ai - s->avail_in), (double)(ao - s->avail_out), (double)s->total_in,
                      (double)s->total_out, (double)s->adler};
    for (uint32_t i = 0; i < 6; i++) napi_set_element(env, arr, i, num(env, vals[i]));
    return arr;
}
// end(h, which) -> rc                                                   zs_stream_deflate_end / zs_stream_inflate_end
napi_value End(napi_env env, napi_callback_info info) {
    size_t argc = 2; napi_value a[2]; napi_get_cb_info(env, info, &argc, a, nullptr, nullptr);
    zs_stream* s = strm_of(env, a[0]);
    return num(env, i32(env, a[1]) == 0 ? zs_stream_deflate_end(s) : zs_stream_inflate_end(s));
}
// setDictionary(h, which, dict) -> rc
napi_value SetDictionary(napi_env env, napi_callback_info info) {
    size_t argc = 3; napi_value a[3]; napi_get_cb_info(env, info, &argc, a, nullptr, nullptr);
    uint8_t* d; size_t n;
    if (!u8(env, a[2], &d, &n)) return num(env, ZS_STREAM_ERROR);
    zs_stream* s = strm_of(env, a[0]);
    return num(env, i32(env, a[1]) == 0 ? zs_stream_deflate_set_dictionary(s, d, (uint32_t)n)
                                        : zs_stream_inflate_set_dictionary(s, d, (uint32_t)n));
}
// inflateReset(h) -> rc
napi_value InflateReset(napi_env env, napi_callback_info info) {
    size_t argc = 1; napi_value a[1]; napi_get_cb_info(env, info, &argc, a, nullptr, nullptr);
    return num(env, zs_stream_inflate_reset(strm_of(env, a[0])));
}

// control(h, op, a) -> rc      op 0 deflateReset, 2 inflateReset2(windowBits)
napi_value Control(napi_env env, napi_callback_info info) {
    size_t argc = 3; napi_value a[3]; napi_get_cb_info(env, info, &argc, a, nullptr, nullptr);
    zs_stream* s = strm_of(env, a[0]);
    switch (i32(env, a[1])) {
        case 0: return num(env, zs_stream_deflate_reset(s));
        case 2: return num(env, zs_stream_inflate_reset2(s, i32(env, a[2])));
    }
    return num(env, ZS_STREAM_ERROR);
}
// deflatePending(h) -> [rc, pending, bits]                               zs_stream_deflate_pending
napi_value DeflatePending(napi_env env, napi_callback_info info) {
    size_t argc = 1; napi_value a[1]; napi_get_cb_info(env, info, &argc, a, nullptr, nullptr);
    uint32_t pending = 0; int bits = 0;
    int rc = zs_stream_deflate_pending(strm_of(env, a[0]), &pending, &bits);
    napi_value arr; napi_create_array_with_length(env, 3, &arr);
    napi_set_element(env, arr, 0, num(env, rc)); napi_set_element(env, arr, 1, num(env, pending)); napi_set_element(env, arr, 2, num(env, bits));
    return arr;
}
// deflateSetHeader(h, text, time, os, hcrc, extra|null, name|null, comment|null) -> rc   zs_stream_deflate_set_header
// (name and comment arrive zero-terminated from the facade)
napi_value DeflateSetHeader(napi_env env, napi_callback_info info) {
    size_t argc = 8; napi_value a[8]; napi_get_cb_info(env, info, &argc, a, nullptr, nullptr);
    zs_gz_header g; memset(&g, 0, sizeof g);
    g.text = i32(env, a[1]); g.time = (uint32_t)i32(env, a[2]); g.os = i32(env, a[3]); g.hcrc = i32(env, a[4]);
    size_t n = 0;
    if (u8(env, a[5], &g.extra, &n)) g.extra_len = (uint32_t)n;
    u8(env, a[6], &g.name, &n);
    u8(env, a[7], &g.comment, &n);
    return num(env, zs_stream_deflate_set_header(strm_of(env, a[0]), &g));
}

// inflateGetHeader(h, extraMax, nameMax, commMax) -> rc                   zs_stream_inflate_get_header
napi_value InflateGetHeader(napi_env env, napi_callback_info info) {
    size_t argc = 4; napi_value a[4]; napi_get_cb_info(env, info, &argc, a, nullptr, nullptr);
    Holder* h = holder_of(env, a[0]);
    if (!h) return num(env, -2);
    memset(&h->gz, 0, sizeof h->gz);
    h->extra.assign((size_t)i32(env, a[1]), 0); h->name.assign((size_t)i32(env, a[2]), 0); h->comment.assign((size_t)i32(env, a[3]), 0);
    if (!h->extra.empty()) { h->gz.extra = h->extra.data(); h->gz.extra_max = (uint32_t)h->extra.size(); }
    if (!h->name.empty()) { h->gz.name = h->name.data(); h->gz.name_max = (uint32_t)h->name.size(); }
    if (!h->comment.empty()) { h->gz.comment = h->comment.data(); h->gz.comm_max = (uint32_t)h->comment.size(); }
    return num(env, zs_stream_inflate_get_header(&h->s, &h->gz));
}
// inflateHeaderState(h) -> [done, text, time, xflags, os, hcrc, extraLen, extra, name, comment]
// (read by the facade after inflate() while head._done is still 0)
napi_value InflateHeaderState(napi_env env, napi_callback_info info) {
    size_t argc = 1; napi_value a[1]; napi_get_cb_info(env, info, &argc, a, nullptr, nullptr);
    Holder* h = holder_of(env, a[0]);
    napi_value arr; napi_create_array_with_length(env, 10, &arr);
    if (!h) return arr;
    const zs_gz_header& g = h->gz;
    const double f[7] = {(double)g.done, (double)g.text, (double)g.time, (double)g.xflags, (double)g.os, (double)g.hcrc, (double)g.extra_len};
    for (uint32_t i = 0; i < 7; ++i) napi_set_element(env, arr, i, num(env, f[i]));
    const std::vector<uint8_t>* b[3] = {&h->extra, &h->name, &h->comment};
    for (uint32_t i = 0; i < 3; ++i) {
        void* dst = nullptr; napi_value buf;
        napi_create_buffer_copy(env, b[i]->size(), b[i]->data(), &dst, &buf);
        napi_set_element(env, arr, 7 + i, buf);
    }
    return arr;
}

napi_value Register(napi_env env, napi_value exports) {
    const struct { const char* name; napi_callback fn; } fns[] = {
        {"init", Init}, {"deflateBatch", DeflateBatch}, {"inflateBatch", InflateBatch}, {"gunzip", Gunzip}, {"checksum", Checksum},
        {"createDeflateDictionary", CreateDeflateDictionary},
        {"deflateIndexed", DeflateIndexed}, {"inflateIndexBuild", InflateIndexBuild}, {"inflateIndexExtract", InflateIndexExtract},
        {"inflateIndexExport", InflateIndexExport}, {"inflateIndexImport", InflateIndexImport},
        {"streamNew", StreamNew}, {"deflateInit2", DeflateInit2}, {"inflateInit2", InflateInit2}, {"process", Process},
        {"end", End}, {"setDictionary", SetDictionary}, {"inflateReset", InflateReset}, {"control", Control},
        {"deflatePending", DeflatePending}, {"deflateSetHeader", DeflateSetHeader},
        {"inflateGetHeader", InflateGetHeader}, {"inflateHeaderState", InflateHeaderState}};
    for (auto& f : fns) {
        napi_value v; napi_create_function(env, f.name, NAPI_AUTO_LENGTH, f.fn, nullptr, &v);
        napi_set_named_property(env, exports, f.name, v);
    }
    return exports;
}

}  // namespace

NAPI_MODULE(zsgpu, Register)
