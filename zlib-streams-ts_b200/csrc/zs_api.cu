// zs_api.cu -- the C ABI of include/zsgpu.h: context, batch deflate / inflate / checksum entry points
// (device-pointer and host-buffer variants).  The streaming shim lives in zs_stream.cu.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "zs_common.cuh"

constexpr uint64_t kParMinInput = 128u << 10;   // shorter streams are decoded by one warp

// ---- scratch (slots: zs_common.cuh) -----------------------------------------------------------------
void* zs_scratch_get(zs_ctx* ctx, zs_scratch_slot slot, size_t bytes) {
    zs_scratch& s = ctx->scr[slot];
    s.gen++;
    if (bytes == 0) bytes = 16;
    if (s.cap >= bytes) return s.p;
    if (s.p) {
        cudaStreamSynchronize(ctx->stream);
        cudaFree(s.p);
        s.p = nullptr;
        s.cap = 0;
    }
    size_t want = bytes + (bytes >> 3) + 256;  // a little head-room so that growing inputs do not realloc every call
    want = (want + 255) & ~(size_t)255;
    cudaError_t e = cudaMalloc(&s.p, want);
    if (e != cudaSuccess) {
        want = (bytes + 255) & ~(size_t)255;
        e = cudaMalloc(&s.p, want);
    }
    if (e != cudaSuccess) {
        snprintf(ctx->err, sizeof(ctx->err), "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
        cudaGetLastError();
        s.p = nullptr;
        return nullptr;
    }
    s.cap = want;
    return s.p;
}

// ---- per-kernel timing -------------------------------------------------------------------------------
struct zs_prof_rec {
    const char* name;
    cudaEvent_t a, b;
};
struct zs_profile {
    std::vector<zs_prof_rec> recs;      // one per launch since the last read
    std::vector<cudaEvent_t> pool;      // recycled events
    cudaEvent_t get() {
        if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
        cudaEvent_t e = nullptr;
        cudaEventCreate(&e);
        return e;
    }
};

void zs_prof_begin(zs_ctx* ctx, const char* name) {
    if (!ctx->prof_on) return;
    zs_profile* pr = (zs_profile*)ctx->prof;
    zs_prof_rec r = {name, pr->get(), pr->get()};
    cudaEventRecord(r.a, ctx->stream);
    pr->recs.push_back(r);
}

void zs_prof_end(zs_ctx* ctx) {
    if (!ctx->prof_on) return;
    zs_profile* pr = (zs_profile*)ctx->prof;
    cudaEventRecord(pr->recs.back().b, ctx->stream);
}

int zs_set_cuda_error(zs_ctx* ctx, cudaError_t e, const char* where) {
    snprintf(ctx->err, sizeof(ctx->err), "CUDA error at %s: %s", where, cudaGetErrorString(e));
    return ZS_E_CUDA;
}

namespace {

// dictionary ranges [begin, end) -> (begin, length) for the checksum kernels
__global__ void dict_ranges_kernel(const uint64_t* rng, uint64_t* off, uint64_t* len, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { off[i] = rng[2 * i]; len[i] = rng[2 * i + 1] - rng[2 * i]; }
}

__global__ void make_chunk_offsets_kernel(uint64_t* off, uint64_t len, uint64_t chunk, uint32_t n) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= n) {
        uint64_t v = i * chunk;
        off[i] = (v < len && i < n) ? v : len;
    }
}

// Every entry point works on the context's device, whatever the caller's current device is.
inline void bind_device(zs_ctx* ctx) { cudaSetDevice(ctx->device); }

int bad_arg(zs_ctx* ctx, const char* msg) {
    if (ctx) snprintf(ctx->err, sizeof(ctx->err), "%s", msg);
    return ZS_STREAM_ERROR;
}

// The copy streams and events of the pipelined host-buffer paths, created by the first such call.
int ensure_copy_streams(zs_ctx* ctx) {
    if (ctx->s_in) return ZS_OK;
    ZS_CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->s_in, cudaStreamNonBlocking));
    ZS_CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->s_out, cudaStreamNonBlocking));
    ZS_CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->s_res, cudaStreamNonBlocking));
    for (int s = 0; s < kMaxPipeSlices; s++)
        for (cudaEvent_t* e : {&ctx->ev_in[s], &ctx->ev_kern[s], &ctx->ev_res[s]})
            ZS_CUDA_TRY(ctx, cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    ZS_CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->ev_fence, cudaEventDisableTiming));
    return ZS_OK;
}

// Everything issued so far on the context stream (the caller's producers, this call's uploads) comes before
// whatever the copy streams do next.
int fence_copy_streams(zs_ctx* ctx) {
    ZS_CUDA_TRY(ctx, cudaEventRecord(ctx->ev_fence, ctx->stream));
    for (cudaStream_t s : {ctx->s_in, ctx->s_out, ctx->s_res}) ZS_CUDA_TRY(ctx, cudaStreamWaitEvent(s, ctx->ev_fence, 0));
    return ZS_OK;
}

}  // namespace

extern "C" {

const char* zs_version(void) { return "zsgpu 0.1.0 (sm_100a)"; }

int zs_ctx_create(int device, void* cuda_stream, zs_ctx** out) {
    if (!out) return ZS_STREAM_ERROR;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0 || device < 0 || device >= count) {
        cudaGetLastError();
        return ZS_E_CUDA;  // no CPU fallback: without a usable CUDA device there is no engine
    }
    if (cudaSetDevice(device) != cudaSuccess) return ZS_E_CUDA;
    zs_ctx* ctx = new zs_ctx();
    ctx->device = device;
    if (cuda_stream) {
        ctx->stream = (cudaStream_t)cuda_stream;
    } else {
        if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
            delete ctx;
            return ZS_E_CUDA;
        }
        ctx->own_stream = true;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->sm_count = prop.multiProcessorCount;
    *out = ctx;
    return ZS_OK;
}

void zs_ctx_destroy(zs_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (auto& s : ctx->scr)
        if (s.p) cudaFree(s.p);
    if (ctx->h_pin) cudaFreeHost(ctx->h_pin);
    if (ctx->s_in) cudaStreamDestroy(ctx->s_in);
    if (ctx->s_out) cudaStreamDestroy(ctx->s_out);
    if (ctx->s_res) cudaStreamDestroy(ctx->s_res);
    for (int s = 0; s < kMaxPipeSlices; s++)
        for (cudaEvent_t e : {ctx->ev_in[s], ctx->ev_kern[s], ctx->ev_res[s]})
            if (e) cudaEventDestroy(e);
    if (ctx->ev_fence) cudaEventDestroy(ctx->ev_fence);
    if (ctx->prof) {
        zs_profile* pr = (zs_profile*)ctx->prof;
        for (auto& r : pr->recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
        for (auto e : pr->pool) cudaEventDestroy(e);
        delete pr;
    }
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

int zs_ctx_profile(zs_ctx* ctx, int enable) {
    if (!ctx) return ZS_STREAM_ERROR;
    if (!ctx->prof) ctx->prof = new zs_profile();
    ctx->prof_on = enable != 0;
    return ZS_OK;
}

int zs_ctx_profile_read(zs_ctx* ctx, char* buf, uint64_t cap) {
    if (!ctx || !buf || cap == 0) return ZS_STREAM_ERROR;
    buf[0] = 0;
    zs_profile* pr = (zs_profile*)ctx->prof;
    if (!pr) return ZS_OK;
    ZS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    struct Agg { const char* name; double ms; uint64_t n; };
    std::vector<Agg> agg;
    for (auto& r : pr->recs) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, r.a, r.b);
        if (getenv("ZS_PROF_LIST")) fprintf(stderr, "[zs prof] %s %.3f ms\n", r.name, ms);   // every launch, in order
        bool found = false;
        for (auto& g : agg)
            if (!strcmp(g.name, r.name)) { g.ms += ms; g.n++; found = true; break; }
        if (!found) agg.push_back({r.name, (double)ms, 1});
        pr->pool.push_back(r.a);
        pr->pool.push_back(r.b);
    }
    pr->recs.clear();
    uint64_t pos = 0;
    for (auto& g : agg) {
        int w = snprintf(buf + pos, (size_t)(cap - pos), "%s %llu %.6f\n", g.name, (unsigned long long)g.n, g.ms);
        if (w < 0 || pos + (uint64_t)w >= cap) break;
        pos += (uint64_t)w;
    }
    return ZS_OK;
}

const char* zs_last_error(const zs_ctx* ctx) { return ctx ? ctx->err : "no context"; }
uint64_t zs_ctx_launch_count(const zs_ctx* ctx) { return ctx ? ctx->launches : 0; }

int zs_ctx_synchronize(zs_ctx* ctx) {
    if (ctx) bind_device(ctx);
    if (!ctx) return ZS_STREAM_ERROR;
    ZS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return ZS_OK;
}

uint64_t zs_deflate_bound(uint64_t n, int wrap) {
    uint64_t wraplen = wrap == ZS_WRAP_RAW ? 0 : wrap == ZS_WRAP_ZLIB ? 6 : 18;
    return n + (n >> 12) + (n >> 14) + (n >> 25) + 13 - 6 + wraplen;
}

uint64_t zs_deflate_batch_bound(uint64_t total_len, uint32_t n_chunks, uint32_t max_chunk, int wrap, int mode) {
    // every block is at worst stored: 5 bytes (+1 alignment) per <= 16 K symbols, plus per-chunk
    // framing (wrapper or sync marker) and slack for the word-granular encoder
    uint64_t blocks = (uint64_t)n_chunks * ((uint64_t)max_chunk / 16351u + 2u);
    (void)mode;
    return total_len + 6 * blocks + (uint64_t)n_chunks * (18 + 8) + 64;
}

uint32_t zs_crc32_combine(uint32_t c1, uint32_t c2, uint64_t len2) { return zs_host_crc32_combine(c1, c2, len2); }
uint32_t zs_adler32_combine(uint32_t a1, uint32_t a2, uint64_t len2) { return zs_host_adler32_combine(a1, a2, len2); }

// ---- checksums ---------------------------------------------------------------------------------------
int zs_checksum_batch_dev(zs_ctx* ctx, int kind, const uint8_t* d_buf, const uint64_t* d_off, uint32_t n,
                          uint32_t* d_out) {
    if (ctx) bind_device(ctx);
    if (!ctx || (kind != 0 && kind != 1) || (n && (!d_buf || !d_off || !d_out))) return bad_arg(ctx, "checksum: bad arguments");
    return zs_launch_checksum_segments(ctx, kind, d_buf, d_off, nullptr, n, d_out);
}

int zs_checksum_dev(zs_ctx* ctx, int kind, const uint8_t* d_buf, uint64_t len, uint32_t init, uint32_t* result) {
    if (ctx) bind_device(ctx);
    if (!ctx || (kind != 0 && kind != 1) || !result || (len && !d_buf)) return bad_arg(ctx, "checksum: bad arguments");
    uint32_t* d_res = (uint32_t*)zs_scratch_get(ctx, SCR_SMALL, 256);
    if (!d_res) return ZS_MEM_ERROR;
    int rc = zs_launch_checksum_whole(ctx, kind, d_buf, len, init, d_res);
    if (rc != ZS_OK) return rc;
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(result, d_res, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return ZS_OK;
}

int zs_checksum(zs_ctx* ctx, int kind, const uint8_t* buf, uint64_t len, uint32_t init, uint32_t* result) {
    if (ctx) bind_device(ctx);
    if (!ctx || !result || (len && !buf)) return bad_arg(ctx, "checksum: bad arguments");
    uint8_t* d_in = (uint8_t*)zs_scratch_get(ctx, SCR_H_IN, len + 64);
    if (!d_in) return ZS_MEM_ERROR;
    if (len) ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_in, buf, len, cudaMemcpyHostToDevice, ctx->stream));
    return zs_checksum_dev(ctx, kind, d_in, len, init, result);
}

}  // extern "C"

// ---- deflate ------------------------------------------------------------------------------------------
// zs_deflate_batch_dev, and zs_deflate_batch_dict_dev with `dict` (INDEPENDENT, no history, checked by the caller).
// seg_hint: 0, or the LZ77 segment size (chunks) of the whole batch when this call compresses a slice of it.
static int deflate_batch_dev(zs_ctx* ctx, const zs_deflate_dict* dict, const uint8_t* d_in, uint64_t in_len,
                             const uint64_t* d_in_off, uint32_t n_chunks, uint32_t chunk_size, uint32_t max_chunk,
                             uint32_t history, int level, int wrap, int mode, uint32_t flags, uint8_t* d_out,
                             uint64_t out_cap, uint64_t* d_out_off, uint64_t* d_out_bits, uint32_t* d_checks,
                             zs_deflate_result* d_result, uint32_t seg_hint) {
    if (level == -1) level = 6;
    // argument rules of deflateInit2_ (deflate.ts:263-297) that apply to the batch form
    if (level < 0 || level > 9) return bad_arg(ctx, "deflate: level must be 0..9");
    const int strategy = (int)((flags >> 8) & 7u);
    if (strategy > ZS_STRATEGY_FIXED) return bad_arg(ctx, "deflate: unknown strategy");
    if (wrap < 0 || wrap > 2 || (mode != ZS_MODE_INDEPENDENT && mode != ZS_MODE_STITCHED))
        return bad_arg(ctx, "deflate: bad wrap or mode");
    if (!d_out || !d_result || (in_len && !d_in) || n_chunks == 0) return bad_arg(ctx, "deflate: null buffer or zero chunks");
    if ((reinterpret_cast<uintptr_t>(d_out) & 15u) != 0) return bad_arg(ctx, "deflate: d_out must be 16-byte aligned");
    if ((flags & ZS_FLAG_PRIME) && (mode != ZS_MODE_INDEPENDENT || wrap != ZS_WRAP_RAW))
        return bad_arg(ctx, "deflate: ZS_FLAG_PRIME needs INDEPENDENT mode and the raw wrapper (deflate.ts:373)");
    if (history > 32768) history = 32768;
    // an empty part still names its position (its history lies before it): a null pointer with history is
    // a caller error, never a device fault
    if (!d_in && history) return bad_arg(ctx, "deflate: history given without an input pointer");
    if (mode == ZS_MODE_INDEPENDENT && !(flags & ZS_FLAG_PRIME)) history = 0;
    if (!d_in_off) {
        if (chunk_size == 0) return bad_arg(ctx, "deflate: chunk_size is zero");
        uint64_t want = in_len ? (in_len + chunk_size - 1) / chunk_size : 1;
        if (want != n_chunks) return bad_arg(ctx, "deflate: n_chunks does not match in_len / chunk_size");
        max_chunk = chunk_size;
    }
    if (max_chunk == 0) max_chunk = 1;
    if (in_len > 0xffffffff00ull) return bad_arg(ctx, "deflate: input too large for one call");

    zs_deflate_plan p;
    memset(&p, 0, sizeof(p));
    p.d_in = d_in; p.in_len = in_len; p.history = history; p.n_chunks = n_chunks; p.max_chunk = max_chunk;
    p.max_bpc = max_chunk / 16351u + 2u;
    p.level = level; p.wrap = wrap; p.mode = mode; p.flags = flags; p.strategy = strategy;
    p.seg_hint = seg_hint;
    p.dict = dict;
    const size_t slots = (size_t)n_chunks * p.max_bpc;

    uint64_t* off = (uint64_t*)zs_scratch_get(ctx, SCR_D_OFF, (size_t)(n_chunks + 1) * 8);
    p.d_sym = (uint32_t*)zs_scratch_get(ctx, SCR_D_SYM, (size_t)in_len * 4 + 64);
    p.d_chunk_nblk = (uint32_t*)zs_scratch_get(ctx, SCR_D_NBLK, (size_t)n_chunks * 4);
    p.d_blk_desc = (uint32_t*)zs_scratch_get(ctx, SCR_D_DESC, slots * 16);
    p.d_blk_freq = (uint32_t*)zs_scratch_get(ctx, SCR_D_FREQ, slots * 320 * 4);
    p.d_blk_code = (uint32_t*)zs_scratch_get(ctx, SCR_D_CODE, slots * 320 * 4);
    p.d_blk_hdr = (uint32_t*)zs_scratch_get(ctx, SCR_D_HDR, slots * 160 * 4);
    p.d_blk_bits = (uint64_t*)zs_scratch_get(ctx, SCR_D_BITS, slots * 8);
    p.d_chunk_pr = (uint64_t*)zs_scratch_get(ctx, SCR_D_PR, (size_t)n_chunks * 16);
    uint32_t* small = (uint32_t*)zs_scratch_get(ctx, SCR_SMALL, 256);
    uint32_t* checks_scr = (uint32_t*)zs_scratch_get(ctx, SCR_D_CHECKS, (size_t)n_chunks * 4);
    uint64_t* outoff_scr = (uint64_t*)zs_scratch_get(ctx, SCR_D_OUTOFF, (size_t)(n_chunks + 1) * 8);
    uint64_t* outbits_scr = (uint64_t*)zs_scratch_get(ctx, SCR_D_OUTBITS, (size_t)n_chunks * 8);
    if (!off || !p.d_sym || !p.d_chunk_nblk || !p.d_blk_desc || !p.d_blk_freq || !p.d_blk_code || !p.d_blk_hdr ||
        !p.d_blk_bits || !p.d_chunk_pr || !small || !checks_scr || !outoff_scr || !outbits_scr)
        return ZS_MEM_ERROR;
    p.d_seg_counter = small + 8;
    p.d_check_total = small + 9;
    p.d_error = (int32_t*)(small + 10);
    ZS_CUDA_TRY(ctx, cudaMemsetAsync(small + 8, 0, 3 * sizeof(uint32_t), ctx->stream));

    if (d_in_off) {
        p.d_in_off = d_in_off;
    } else {
        ZS_KERNEL(ctx, "make_chunk_offsets_kernel", make_chunk_offsets_kernel<<<(n_chunks + 1 + 255) / 256, 256, 0, ctx->stream>>>(off, in_len, chunk_size, n_chunks));
        p.d_in_off = off;
    }
    p.d_out = d_out; p.out_cap = out_cap;
    p.d_out_off = d_out_off ? d_out_off : outoff_scr;
    p.d_out_bits = d_out_bits ? d_out_bits : outbits_scr;
    p.d_result = d_result;

    // checksums of the uncompressed data (read_buf, deflate.ts:155-159): adler32 for the zlib
    // wrapper, crc32 for gzip; for raw streams only when the caller asks for per-chunk values
    const bool need_check = wrap != ZS_WRAP_RAW || d_checks != nullptr;
    p.d_checks = nullptr;
    if (need_check) {
        const int kind = wrap == ZS_WRAP_ZLIB ? 0 : 1;
        p.d_checks = d_checks ? d_checks : checks_scr;
        int rc = zs_launch_checksum_segments(ctx, kind, d_in, p.d_in_off, nullptr, n_chunks, p.d_checks);
        if (rc != ZS_OK) return rc;
        rc = zs_launch_checksum_fold(ctx, kind, p.d_checks, p.d_in_off, n_chunks, kind ? 0u : 1u, p.d_check_total);
        if (rc != ZS_OK) return rc;
    }
    int rc = zs_launch_lz77(ctx, p);
    if (rc != ZS_OK) return rc;
#ifdef ZS_DEBUG_HOOKS   // the match finder's raw output (block counts, descriptors, symbols), for diffing two runs: tools/dbg_ragged2.py
    if (const char* dump = getenv("ZS_DUMP_LZ")) {
        std::vector<uint32_t> sym(in_len), desc(slots * 4), nblk(n_chunks);
        cudaStreamSynchronize(ctx->stream);
        cudaMemcpy(sym.data(), p.d_sym, in_len * 4, cudaMemcpyDeviceToHost);
        cudaMemcpy(desc.data(), p.d_blk_desc, slots * 16, cudaMemcpyDeviceToHost);
        cudaMemcpy(nblk.data(), p.d_chunk_nblk, (size_t)n_chunks * 4, cudaMemcpyDeviceToHost);
        if (FILE* f = fopen(dump, "wb")) {
            fwrite(nblk.data(), 4, nblk.size(), f); fwrite(desc.data(), 4, desc.size(), f); fwrite(sym.data(), 4, sym.size(), f);
            fclose(f);
        }
    }
#endif
    return zs_launch_huffman(ctx, p);
}

extern "C" {

int zs_deflate_batch_dev(zs_ctx* ctx, const uint8_t* d_in, uint64_t in_len, const uint64_t* d_in_off,
                         uint32_t n_chunks, uint32_t chunk_size, uint32_t max_chunk, uint32_t history, int level,
                         int wrap, int mode, uint32_t flags, uint8_t* d_out, uint64_t out_cap, uint64_t* d_out_off,
                         uint64_t* d_out_bits, uint32_t* d_checks, zs_deflate_result* d_result) {
    if (ctx) bind_device(ctx);
    if (!ctx) return ZS_STREAM_ERROR;
    return deflate_batch_dev(ctx, nullptr, d_in, in_len, d_in_off, n_chunks, chunk_size, max_chunk, history, level, wrap,
                             mode, flags, d_out, out_cap, d_out_off, d_out_bits, d_checks, d_result, 0);
}

// ---- preset dictionaries ------------------------------------------------------------------------------
int zs_deflate_dict_create(zs_ctx* ctx, const uint8_t* dict, uint64_t dict_len, zs_deflate_dict** out) {
    if (ctx) bind_device(ctx);
    if (!ctx || !out || (dict_len && !dict)) return bad_arg(ctx, "deflate_dict_create: bad arguments");
    *out = nullptr;
    // deflateSetDictionary (deflate.ts:367-424): only the last w_size bytes are used; DICTID covers them all
    const uint64_t used = dict_len < 32768 ? dict_len : 32768;
    zs_deflate_dict* d = new zs_deflate_dict();
    d->device = ctx->device;
    d->len = (uint32_t)used;
    // the whole dictionary (for DICTID) and its used tail (16-byte aligned, for the build) are needed only here
    uint8_t *d_whole = nullptr, *d_tail = nullptr;
    auto fail = [&](int rc) {
        cudaFree(d_whole); cudaFree(d_tail); cudaFree(d->d_img);
        delete d;
        return rc;
    };
    cudaError_t e = cudaMalloc(&d_tail, 32768 + 64);
    if (e == cudaSuccess) e = cudaMalloc(&d->d_img, zs_lz77_dict_image_bytes());
    if (e == cudaSuccess && dict_len) e = cudaMalloc(&d_whole, dict_len);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_tail, 0, 32768 + 64, ctx->stream);
    if (e == cudaSuccess && dict_len) e = cudaMemcpyAsync(d_whole, dict, dict_len, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess && used)
        e = cudaMemcpyAsync(d_tail, d_whole + (dict_len - used), used, cudaMemcpyDeviceToDevice, ctx->stream);
    if (e != cudaSuccess) return fail(zs_set_cuda_error(ctx, e, "deflate_dict_create"));
    // DICTID on the device with the checksum kernels
    uint32_t* d_id = (uint32_t*)zs_scratch_get(ctx, SCR_SMALL, 256);
    if (!d_id) return fail(ZS_MEM_ERROR);
    int rc = zs_launch_checksum_whole(ctx, 0, d_whole, dict_len, 1u, d_id);
    if (rc != ZS_OK) return fail(rc);
    e = cudaMemcpyAsync(&d->id, d_id, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) return fail(zs_set_cuda_error(ctx, e, "deflate_dict_create"));
    rc = zs_lz77_dict_build(ctx, d_tail, d->len, d->d_img);   // synchronises
    if (rc != ZS_OK) return fail(rc);
    cudaFree(d_whole);
    cudaFree(d_tail);
    *out = d;
    return ZS_OK;
}

uint32_t zs_deflate_dict_id(const zs_deflate_dict* d) { return d ? d->id : 1u; }

void zs_deflate_dict_destroy(zs_deflate_dict* d) {
    if (!d) return;
    // called from garbage collectors at any time: the caller's current device is left as it was
    int prev = -1;
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    cudaSetDevice(d->device);
    cudaDeviceSynchronize();   // a call that uses the tables may still be queued on any stream of the device
    cudaFree(d->d_img);
    if (prev >= 0 && prev != d->device) cudaSetDevice(prev);
    delete d;
}

// the arguments zlib refuses with a dictionary (deflateSetDictionary, deflate.ts:372) and those the batch form
// has no meaning for: every chunk is one whole independent stream
static int check_dict_call(zs_ctx* ctx, const zs_deflate_dict* dict, int wrap, uint32_t flags) {
    if (!dict) return bad_arg(ctx, "deflate_batch_dict: no dictionary");
    if (dict->device != ctx->device) return bad_arg(ctx, "deflate_batch_dict: dictionary prepared for another device");
    if (wrap != ZS_WRAP_RAW && wrap != ZS_WRAP_ZLIB) return bad_arg(ctx, "deflate_batch_dict: gzip streams take no dictionary (deflate.ts:372)");
    if (flags & ~(7u << 8)) return bad_arg(ctx, "deflate_batch_dict: flags carry the strategy only");
    return ZS_OK;
}

int zs_deflate_batch_dict_dev(zs_ctx* ctx, const zs_deflate_dict* dict, const uint8_t* d_in, uint64_t in_len,
                              const uint64_t* d_in_off, uint32_t n_chunks, uint32_t chunk_size, uint32_t max_chunk, int level,
                              int wrap, uint32_t flags, uint8_t* d_out, uint64_t out_cap, uint64_t* d_out_off,
                              uint64_t* d_out_bits, uint32_t* d_checks, zs_deflate_result* d_result) {
    if (ctx) bind_device(ctx);
    if (!ctx) return ZS_STREAM_ERROR;
    const int rc = check_dict_call(ctx, dict, wrap, flags);
    if (rc != ZS_OK) return rc;
    return deflate_batch_dev(ctx, dict, d_in, in_len, d_in_off, n_chunks, chunk_size, max_chunk, 0, level, wrap,
                             ZS_MODE_INDEPENDENT, flags, d_out, out_cap, d_out_off, d_out_bits, d_checks, d_result, 0);
}

// Host-buffer deflate of a large batch, software-pipelined: the batch is cut into slices of whole waves of
// LZ77 segments, and the H2D copy of slice s+1, the kernels of slice s and the D2H copy of slice s-1 run
// concurrently on three streams.
//  INDEPENDENT: the bytes produced are those of the single-shot path.
//  STITCHED: every slice is one *part* of the stream (ZS_FLAG_NOT_FIRST / NOT_LAST), primed with the 32 KiB
//  before it; a part that is not the last ends with the reference's Z_SYNC_FLUSH marker (deflate.ts:945-946),
//  so slices concatenate byte-wise (5 bytes per slice more than the single-shot stream).  `history` bytes
//  before `in` are readable and primed against; the trailer of a whole stream (deflate.ts:964-988) is
//  written here from the combined checksums.
static int deflate_batch_pipelined(zs_ctx* ctx, const zs_deflate_dict* dict, const uint8_t* in, uint64_t in_len,
                                   uint32_t history, uint32_t n_chunks, uint32_t chunk_size, int level, int wrap, int mode,
                                   uint32_t flags, uint8_t* out, uint64_t out_cap, uint64_t* out_off, uint64_t* out_bits,
                                   uint32_t* checks, zs_deflate_result* result) {
    constexpr int kMaxSlices = 16;
    static_assert(kMaxSlices <= kMaxPipeSlices, "one event per slice");
    const bool stitched = mode == ZS_MODE_STITCHED;
    // Same LZ77 segmentation as the single-shot call over the whole batch; a slice is a whole number
    // of waves of segments (one segment per SM and wave), so that no SM idles inside a slice.
    uint32_t seg = n_chunks / (4u * (uint32_t)ctx->sm_count);
    seg = seg < 1 ? 1 : seg > 16 ? 16 : seg;
    const uint32_t n_seg = (n_chunks + seg - 1) / seg;
    const uint32_t wave = (uint32_t)ctx->sm_count;
    uint32_t waves_per_slice = (n_seg + wave * kMaxSlices - 1) / (wave * kMaxSlices);
    if (waves_per_slice < 1) waves_per_slice = 1;
    if (const char* e = getenv("ZS_SLICE_WAVES")) {   // A/B hook: at least this many waves per slice
        const uint32_t w = (uint32_t)atoi(e);
        if (w > waves_per_slice) waves_per_slice = w;
    }
    // Slice s covers chunks [cb[s], cb[s + 1]).  Greedy levels: equal slices of whole waves (measured on configs[1]:
    // one wave per slice 45.8 ms, two 47.2, three 49.5 -- the searches are even, so a one-wave launch loses little and
    // the first copy is short).  Lazy levels: the search time of a segment varies, a one-wave launch is as slow as its
    // slowest segment (configs[2] shape, 1 GiB: device 68.9 ms, five one-wave slices 95 ms), so the slices GROW -- one
    // wave first, so that the kernels start as soon as a sixteenth of the input is there, then two, four, ... waves,
    // by which time the copies (three times as fast as the kernels) are far ahead.
    uint32_t cb[kMaxSlices + 1];
    int n_slices = 0;
    cb[0] = 0;
    {
        const bool grow = level >= 4 && !getenv("ZS_SLICE_WAVES");
        uint32_t w = waves_per_slice;
        while (cb[n_slices] < n_chunks) {
            if (n_slices >= kMaxSlices) return bad_arg(ctx, "deflate: internal slicing error");
            uint64_t next = (uint64_t)cb[n_slices] + (uint64_t)seg * wave * w;
            if (next > n_chunks || n_slices + 1 == kMaxSlices) next = n_chunks;
            cb[++n_slices] = (uint32_t)next;
            if (grow) w *= 2;
        }
    }
    uint32_t slice_chunks = 0;   // the largest slice: sizes the per-slice output regions
    for (int i = 0; i < n_slices; i++) slice_chunks = cb[i + 1] - cb[i] > slice_chunks ? cb[i + 1] - cb[i] : slice_chunks;
    int rc = ensure_copy_streams(ctx);
    if (rc != ZS_OK) return rc;
    if (!ctx->h_pin) {
        ZS_CUDA_TRY(ctx, cudaMallocHost(&ctx->h_pin, 4096));
        ctx->h_pin_cap = 4096;
    }
    zs_deflate_result* h_res = (zs_deflate_result*)ctx->h_pin;
    const uint64_t slice_bytes = (uint64_t)slice_chunks * chunk_size;
    const uint64_t region = zs_deflate_batch_bound(slice_bytes, slice_chunks, chunk_size, wrap, mode) + (dict ? 4ull * slice_chunks : 0);
    const uint64_t region_al = (region + 255) & ~255ull;
    if (!stitched) history = 0;
    if (history > 32768) history = 32768;
    uint8_t* d_in_base = (uint8_t*)zs_scratch_get(ctx, SCR_H_IN, 32768 + in_len + 64);
    uint8_t* d_out = (uint8_t*)zs_scratch_get(ctx, SCR_H_OUT, region_al * n_slices + 64);
    uint64_t* d_ooff = (uint64_t*)zs_scratch_get(ctx, SCR_H_OFF2, ((size_t)n_chunks + n_slices) * 8);
    uint64_t* d_obits = (uint64_t*)zs_scratch_get(ctx, SCR_H_OFF, (size_t)n_chunks * 8);
    uint32_t* d_cks = (uint32_t*)zs_scratch_get(ctx, SCR_H_CHECKS, (size_t)n_chunks * 4);
    zs_deflate_result* d_res = (zs_deflate_result*)zs_scratch_get(ctx, SCR_H_RES, sizeof(zs_deflate_result) * kMaxSlices);
    if (!d_in_base || !d_out || !d_ooff || !d_obits || !d_cks || !d_res) return ZS_MEM_ERROR;
    uint8_t* d_in = d_in_base + 32768;   // the history of the first slice lies before it
    const bool want_checks = checks != nullptr || wrap != ZS_WRAP_RAW;
    rc = fence_copy_streams(ctx);
    if (rc != ZS_OK) return rc;
    if (history) ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_in - history, in - history, history, cudaMemcpyHostToDevice, ctx->s_in));
    const uint32_t part_mask = ZS_FLAG_NOT_FIRST | ZS_FLAG_NOT_LAST;
    for (int s = 0; s < n_slices; s++) {
        const uint32_t c0 = cb[s];
        const uint32_t nc = cb[s + 1] - cb[s];
        const uint64_t b0 = (uint64_t)c0 * chunk_size;
        const uint64_t len = (b0 + (uint64_t)nc * chunk_size <= in_len) ? (uint64_t)nc * chunk_size : in_len - b0;
        if (len) ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_in + b0, in + b0, len, cudaMemcpyHostToDevice, ctx->s_in));
        ZS_CUDA_TRY(ctx, cudaEventRecord(ctx->ev_in[s], ctx->s_in));
        ZS_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_in[s], 0));
        uint32_t hist = 0, sflags = flags;
        if (stitched) {
            hist = (uint32_t)(b0 + history < 32768 ? b0 + history : 32768);
            sflags = flags & ~part_mask;
            if (s > 0 || (flags & ZS_FLAG_NOT_FIRST)) sflags |= ZS_FLAG_NOT_FIRST;
            if (s + 1 < n_slices || (flags & ZS_FLAG_NOT_LAST)) sflags |= ZS_FLAG_NOT_LAST;
        } else if (flags & ZS_FLAG_PRIME) {
            hist = (uint32_t)(b0 < 32768 ? b0 : 32768);
        }
        rc = deflate_batch_dev(ctx, dict, d_in + b0, len, nullptr, nc, chunk_size, chunk_size, hist, level, wrap, mode, sflags,
                               d_out + region_al * s, region, d_ooff + c0 + s, d_obits + c0,
                               want_checks ? d_cks + c0 : nullptr, d_res + s, seg);
        if (rc != ZS_OK) return rc;
        ZS_CUDA_TRY(ctx, cudaEventRecord(ctx->ev_kern[s], ctx->stream));
        // The 24-byte results come back on their own stream: the bulk D2H copies below are issued as
        // each result arrives and must not queue behind the waits for later slices.
        ZS_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->s_res, ctx->ev_kern[s], 0));
        ZS_CUDA_TRY(ctx, cudaMemcpyAsync(h_res + s, d_res + s, sizeof(zs_deflate_result), cudaMemcpyDeviceToHost, ctx->s_res));
        ZS_CUDA_TRY(ctx, cudaEventRecord(ctx->ev_res[s], ctx->s_res));
    }
    uint64_t host_off = 0;
    uint64_t base[kMaxSlices];
    uint32_t blocks = 0, check = 0;
    bool have_check = false;
    int rc_final = ZS_OK;
    for (int s = 0; s < n_slices; s++) {
        const uint32_t c0 = cb[s];
        const uint32_t nc = cb[s + 1] - cb[s];
        const uint64_t b0 = (uint64_t)c0 * chunk_size;
        const uint64_t len = (b0 + (uint64_t)nc * chunk_size <= in_len) ? (uint64_t)nc * chunk_size : in_len - b0;
        ZS_CUDA_TRY(ctx, cudaEventSynchronize(ctx->ev_res[s]));
        const uint64_t total = h_res[s].total_out_bytes;
        base[s] = host_off;
        if (total > region || host_off + total > out_cap) { rc_final = ZS_BUF_ERROR; break; }
        ZS_CUDA_TRY(ctx, cudaMemcpyAsync(out + host_off, d_out + region_al * s, total, cudaMemcpyDeviceToHost, ctx->s_out));
        if (out_off)
            ZS_CUDA_TRY(ctx, cudaMemcpyAsync(out_off + c0, d_ooff + c0 + s, (size_t)nc * 8, cudaMemcpyDeviceToHost, ctx->s_out));
        if (out_bits)
            ZS_CUDA_TRY(ctx, cudaMemcpyAsync(out_bits + c0, d_obits + c0, (size_t)nc * 8, cudaMemcpyDeviceToHost, ctx->s_out));
        if (checks)
            ZS_CUDA_TRY(ctx, cudaMemcpyAsync(checks + c0, d_cks + c0, (size_t)nc * 4, cudaMemcpyDeviceToHost, ctx->s_out));
        host_off += total;
        blocks += h_res[s].n_blocks;
        if (want_checks) {
            if (!have_check) { check = h_res[s].check; have_check = true; }
            else check = zs_host_check_combine(wrap, check, h_res[s].check, len);
        }
    }
    ZS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->s_out));
    ZS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    // the trailer of a whole stitched stream that went through more than one slice (the device writes it
    // only when one call holds the whole stream)
    if (rc_final == ZS_OK && stitched && n_slices > 1 && !(flags & part_mask) && wrap != ZS_WRAP_RAW) {
        const uint64_t T = wrap == ZS_WRAP_ZLIB ? 4 : 8;
        if (host_off + T > out_cap) {
            rc_final = ZS_BUF_ERROR;
        } else {
            host_off += zs_put_trailer(out + host_off, wrap, check, in_len);
        }
    }
    if (rc_final != ZS_OK) {
        snprintf(ctx->err, sizeof(ctx->err), "deflate: output capacity %llu too small", (unsigned long long)out_cap);
        return rc_final;
    }
    if (out_off) {
        const uint64_t unit = stitched ? 8 : 1;   // STITCHED reports bit offsets
        for (int s = 0; s < n_slices; s++) {
            const uint32_t c0 = cb[s];
            const uint32_t nc = cb[s + 1] - cb[s];
            for (uint32_t i = 0; i < nc; i++) out_off[c0 + i] += base[s] * unit;
        }
        out_off[n_chunks] = host_off * unit;
    }
    result->total_out_bytes = host_off;
    result->total_out_bits = host_off * 8;
    result->check = check;
    result->n_blocks = blocks;
    return ZS_OK;
}

// Shared body of zs_deflate_batch / zs_deflate_part: `history` readable bytes lie before `in`.
static int deflate_batch_host(zs_ctx* ctx, const zs_deflate_dict* dict, const uint8_t* in, uint64_t in_len,
                              uint32_t history, const uint64_t* in_off, uint32_t n_chunks, uint32_t chunk_size, int level,
                              int wrap, int mode, uint32_t flags, uint8_t* out, uint64_t out_cap, uint64_t* out_off,
                              uint64_t* out_bits, uint32_t* checks, zs_deflate_result* result) {
    if (!out || !result || (in_len && !in) || n_chunks == 0) return bad_arg(ctx, "deflate: null buffer or zero chunks");
    if (history && !in) return bad_arg(ctx, "deflate: history without an input pointer");
    if (history > 32768) history = 32768;
    uint32_t max_chunk = chunk_size;
    if (in_off) {
        max_chunk = 1;
        if (in_off[0] != 0 || in_off[n_chunks] != in_len) return bad_arg(ctx, "deflate: in_off must span [0, in_len]");
        for (uint32_t i = 0; i < n_chunks; i++) {
            if (in_off[i + 1] < in_off[i]) return bad_arg(ctx, "deflate: in_off must be non-decreasing");
            uint64_t l = in_off[i + 1] - in_off[i];
            if (l > 0xffffffffull) return bad_arg(ctx, "deflate: chunk too large");
            if (l > max_chunk) max_chunk = (uint32_t)l;
        }
    }
    // Large batches with fixed chunking are software-pipelined (see deflate_batch_pipelined).
    if (!in_off && n_chunks >= 512 && chunk_size >= 4096 && !(mode == ZS_MODE_STITCHED && (flags & ZS_FLAG_PRIME)))
        return deflate_batch_pipelined(ctx, dict, in, in_len, history, n_chunks, chunk_size, level, wrap, mode, flags, out,
                                       out_cap, out_off, out_bits, checks, result);
    if (mode != ZS_MODE_STITCHED) history = 0;
    uint8_t* d_in_base = (uint8_t*)zs_scratch_get(ctx, SCR_H_IN, 32768 + in_len + 64);
    uint8_t* d_out = (uint8_t*)zs_scratch_get(ctx, SCR_H_OUT, out_cap + 64);
    uint64_t* d_off = (uint64_t*)zs_scratch_get(ctx, SCR_H_OFF, (size_t)(n_chunks + 1) * 8);
    uint64_t* d_ooff = (uint64_t*)zs_scratch_get(ctx, SCR_H_OFF2, (size_t)(2 * (size_t)n_chunks + 1) * 8);
    uint8_t* d_res = (uint8_t*)zs_scratch_get(ctx, SCR_H_RES, sizeof(zs_deflate_result) + (size_t)n_chunks * 4 + 64);
    if (!d_in_base || !d_out || !d_off || !d_ooff || !d_res) return ZS_MEM_ERROR;
    uint8_t* d_in = d_in_base + 32768;
    zs_deflate_result* d_result = (zs_deflate_result*)d_res;
    uint32_t* d_checks = checks ? (uint32_t*)(d_res + 64) : nullptr;
    if (in_len + history)
        ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_in - history, in - history, in_len + history, cudaMemcpyHostToDevice, ctx->stream));
    if (in_off)
        ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_off, in_off, (size_t)(n_chunks + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    int rc = deflate_batch_dev(ctx, dict, d_in, in_len, in_off ? d_off : nullptr, n_chunks, chunk_size, max_chunk, history,
                               level, wrap, mode, flags, d_out, out_cap, d_ooff, d_ooff + n_chunks + 1, d_checks, d_result, 0);
    if (rc != ZS_OK) return rc;
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(result, d_result, sizeof(zs_deflate_result), cudaMemcpyDeviceToHost, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (result->total_out_bytes > out_cap) {
        snprintf(ctx->err, sizeof(ctx->err), "deflate: output needs %llu bytes, capacity %llu",
                 (unsigned long long)result->total_out_bytes, (unsigned long long)out_cap);
        return ZS_BUF_ERROR;
    }
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(out, d_out, result->total_out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (out_off)
        ZS_CUDA_TRY(ctx, cudaMemcpyAsync(out_off, d_ooff, (size_t)(n_chunks + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (out_bits)
        ZS_CUDA_TRY(ctx, cudaMemcpyAsync(out_bits, d_ooff + n_chunks + 1, (size_t)n_chunks * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (checks)
        ZS_CUDA_TRY(ctx, cudaMemcpyAsync(checks, d_checks, (size_t)n_chunks * 4, cudaMemcpyDeviceToHost, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return ZS_OK;
}

int zs_deflate_batch(zs_ctx* ctx, const uint8_t* in, uint64_t in_len, const uint64_t* in_off, uint32_t n_chunks,
                     uint32_t chunk_size, int level, int wrap, int mode, uint32_t flags, uint8_t* out, uint64_t out_cap,
                     uint64_t* out_off, uint64_t* out_bits, uint32_t* checks, zs_deflate_result* result) {
    if (ctx) bind_device(ctx);
    if (!ctx) return ZS_STREAM_ERROR;
    return deflate_batch_host(ctx, nullptr, in, in_len, 0, in_off, n_chunks, chunk_size, level, wrap, mode, flags, out, out_cap,
                              out_off, out_bits, checks, result);
}

int zs_deflate_batch_dict(zs_ctx* ctx, const zs_deflate_dict* dict, const uint8_t* in, uint64_t in_len, const uint64_t* in_off,
                          uint32_t n_chunks, uint32_t chunk_size, int level, int wrap, uint32_t flags, uint8_t* out,
                          uint64_t out_cap, uint64_t* out_off, uint64_t* out_bits, uint32_t* checks, zs_deflate_result* result) {
    if (ctx) bind_device(ctx);
    if (!ctx) return ZS_STREAM_ERROR;
    const int rc = check_dict_call(ctx, dict, wrap, flags);
    if (rc != ZS_OK) return rc;
    // every chunk is its own segment in a dictionary call, so slicing a large batch cannot change the output
    return deflate_batch_host(ctx, dict, in, in_len, 0, in_off, n_chunks, chunk_size, level, wrap, ZS_MODE_INDEPENDENT, flags,
                              out, out_cap, out_off, out_bits, checks, result);
}

int zs_deflate_part(zs_ctx* ctx, const uint8_t* in, uint64_t in_len, uint32_t history, uint32_t chunk_size, int level,
                    int wrap, uint32_t flags, uint8_t* out, uint64_t out_cap, uint64_t* out_bits, zs_deflate_result* result) {
    if (ctx) bind_device(ctx);
    if (!ctx) return ZS_STREAM_ERROR;
    if (chunk_size == 0) return bad_arg(ctx, "deflate: chunk_size is zero");
    if (flags & ZS_FLAG_PRIME) return bad_arg(ctx, "deflate: ZS_FLAG_PRIME does not apply to a part of a stream");
    const uint64_t nc = in_len ? (in_len + chunk_size - 1) / chunk_size : 1;
    if (nc > 0xffffffffull) return bad_arg(ctx, "deflate: too many chunks");
    return deflate_batch_host(ctx, nullptr, in, in_len, history, nullptr, (uint32_t)nc, chunk_size, level, wrap, ZS_MODE_STITCHED,
                              flags, out, out_cap, nullptr, out_bits, nullptr, result);
}

int zs_bit_concat_dev(zs_ctx* ctx, uint8_t* d_dst, uint64_t dst_bit_off, const uint8_t* d_src, uint64_t n_bits) {
    if (ctx) bind_device(ctx);
    if (!ctx || !d_dst || (n_bits && !d_src)) return bad_arg(ctx, "bit_concat: bad arguments");
    return zs_launch_bit_concat(ctx, d_dst, dst_bit_off, d_src, n_bits);
}

}  // extern "C"

// ---- inflate ------------------------------------------------------------------------------------------
// zs_inflate_batch_dev with options.  o.resume: res->mark receives the block mark (copied on the context stream);
// `res` may be null otherwise.
static int inflate_batch_dev_impl(zs_ctx* ctx, const uint8_t* d_in, const uint64_t* d_in_off, uint32_t n, int window_bits,
                                  uint8_t* d_out, const uint64_t* d_out_off, uint64_t* d_out_len, uint64_t* d_in_used,
                                  uint32_t* d_checks, int32_t* d_status, const uint8_t* d_dict, const uint64_t* d_dict_rng,
                                  const InflateOpts& o, InflateOut* res) {
    if (n == 0) return ZS_OK;
    if (!d_in || !d_in_off || !d_out || !d_out_off || !d_out_len || !d_status) return bad_arg(ctx, "inflate: null buffer");
    if ((reinterpret_cast<uintptr_t>(d_in) & 7u) != 0) return bad_arg(ctx, "inflate: d_in must be 8-byte aligned");
    int wrap, d64;
    if (!zs_inflate_window_bits(window_bits, &wrap, &d64)) return bad_arg(ctx, "inflate: windowBits out of range");

    // misc scratch: detail[n] trailer[2n] flags[n] adler[n] crc[n] dict_adler[n] | dict off[n] len[n] (u64)
    uint32_t* misc = (uint32_t*)zs_scratch_get(ctx, SCR_I_MISC, (size_t)n * 7 * 4 + 16 + (size_t)n * 16);
    if (!misc) return ZS_MEM_ERROR;
    zs_inflate_args a;
    a.d_in = d_in; a.d_in_off = d_in_off; a.n = n; a.wrap = wrap; a.deflate64 = d64;
    a.d_out = d_out; a.d_out_off = d_out_off; a.d_out_len = d_out_len; a.d_in_used = d_in_used;
    a.d_status = d_status;
    a.d_detail = (int32_t*)misc;
    a.d_trailer = misc + n;
    a.d_flags = misc + 3 * (size_t)n;
    a.d_dict = d_dict; a.d_dict_rng = d_dict_rng;
    a.d_dict_adler = nullptr;
    if ((wrap & 1) && d_dict && d_dict_rng) {
        // zlib streams with FDICT are decoded when their DICTID is the adler32 of the dictionary they were given
        uint32_t* d_da = misc + 6 * (size_t)n;
        uint64_t* d_doff = (uint64_t*)(((uintptr_t)(misc + 7 * (size_t)n) + 15) & ~(uintptr_t)15);
        ZS_KERNEL(ctx, "dict_ranges_kernel", dict_ranges_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(d_dict_rng, d_doff, d_doff + n, n));
        const int rc0 = zs_launch_checksum_segments(ctx, 0, d_dict, d_doff, d_doff + n, n, d_da);
        if (rc0 != ZS_OK) return rc0;
        a.d_dict_adler = d_da;
    }
    a.d_start_bit = nullptr; a.d_block_mark = nullptr;
    const bool resume = o.resume && n == 1;
    if (resume) {
        // one stream of the streaming shim: [0] start bit (in), [1..2] block mark (out)
        uint64_t* d_rs = (uint64_t*)zs_scratch_get(ctx, SCR_I_RESUME, 64);
        if (!d_rs) return ZS_MEM_ERROR;
        ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_rs, &o.start_bit, 8, cudaMemcpyHostToDevice, ctx->stream));
        if (o.start_bit != ~0ull) a.d_start_bit = d_rs;
        a.d_block_mark = d_rs + 1;
    }
    // test hooks: force the thread-per-stream (1) or the warp-per-stream (-1) kernel
    a.force_tps = getenv("ZS_INFLATE_TPS") ? 1 : getenv("ZS_INFLATE_WARP") ? -1 : 0;
    a.d_hdr_state = nullptr; a.d_resume = nullptr;
    uint32_t* d_adler = misc + 4 * (size_t)n;
    uint32_t* d_crc = misc + 5 * (size_t)n;
    int rc;
    // One long stream whose sizes the caller knows on the host: cut it at its flush points and decode the
    // segments in parallel (zs_inflate_par.cu); inflate_kernel then continues behind them -- the trailer
    // and the final status, or whatever the parallel part had to leave.
    const bool par = o.par.on && n == 1 && !d64 && o.par.in_len >= kParMinInput && ((o.par.in_off & 7u) == 0) &&
                     !getenv("ZS_INFLATE_SERIAL");
    const uint32_t n_choice = o.batch_n > n ? o.batch_n : n;
    if (par) {
        uint64_t* d_ps = (uint64_t*)zs_scratch_get(ctx, SCR_P_STATE, 16 * 8);
        if (!d_ps) return ZS_MEM_ERROR;
        zs_inflate_args h = a;
        h.d_hdr_state = d_ps;
        h.d_block_mark = nullptr;
        rc = zs_launch_inflate(ctx, h, n_choice);
        if (rc != ZS_OK) return rc;
        rc = zs_launch_inflate_parallel(ctx, d_in + o.par.in_off, o.par.in_len, d_out + o.par.out_off, o.par.out_cap,
                                        d_dict ? d_dict + o.par.dict_off : nullptr, d_dict ? o.par.dict_len : 0, d_ps, d_ps + 8);
        if (rc != ZS_OK) return rc;
        a.d_resume = d_ps + 8;
    }
    rc = zs_launch_inflate(ctx, a, n_choice);
    if (rc != ZS_OK) return rc;
    ctx->d_last_detail = a.d_detail;
    ctx->last_detail_n = n;
    // checksum of what was produced (inf_leave / CHECK, inflate.ts:1012-1015,1079-1085)
    const bool want_adler = (wrap & 1) != 0;
    const bool want_crc = (wrap & 2) != 0 || (wrap == 0 && d_checks != nullptr);
    if (par) {
        // one long stream: its output is cut into pieces for the checksum too (a warp per stream would take
        // 0.5 s per GiB)
        if (want_adler) rc = zs_launch_checksum_stream(ctx, 0, d_out, d_out_off, d_out_len, o.par.out_cap, d_adler);
        if (rc == ZS_OK && want_crc) rc = zs_launch_checksum_stream(ctx, 1, d_out, d_out_off, d_out_len, o.par.out_cap, d_crc);
        if (rc != ZS_OK) return rc;
    } else {
        if (want_adler) {
            rc = zs_launch_checksum_segments(ctx, 0, d_out, d_out_off, d_out_len, n, d_adler);
            if (rc != ZS_OK) return rc;
        }
        if (want_crc) {
            rc = zs_launch_checksum_segments(ctx, 1, d_out, d_out_off, d_out_len, n, d_crc);
            if (rc != ZS_OK) return rc;
        }
    }
    rc = zs_launch_inflate_verify(ctx, n, want_adler ? d_adler : nullptr, want_crc ? d_crc : nullptr, a.d_trailer, a.d_flags,
                                  d_out_len, d_checks, d_status, a.d_detail);
    if (rc == ZS_OK && resume)
        ZS_CUDA_TRY(ctx, cudaMemcpyAsync(res->mark, a.d_block_mark, 16, cudaMemcpyDeviceToHost, ctx->stream));
    return rc;
}

// Host-buffer inflate of a large batch, pipelined like deflate_batch_pipelined: the streams are cut into slices
// of about equal input + output bytes; slice s+1 is copied in while the kernels of slice s run and the output of
// slice s-1 is copied out (three streams, events between them).  Every slice is decoded by the kernel the
// whole batch would have used (InflateOpts::batch_n), so the results are those of the unsliced call.
static int inflate_batch_pipelined(zs_ctx* ctx, const uint8_t* in, const uint64_t* in_off, uint32_t n, int window_bits,
                                   uint8_t* out, const uint64_t* out_off, uint64_t* out_len, uint64_t* in_used,
                                   uint32_t* checks, int32_t* status, uint8_t* d_in, uint8_t* d_out, uint64_t* d_ioff,
                                   uint64_t* d_ooff, uint8_t* d_res, const uint8_t* d_dict, const uint64_t* d_rng) {
    // a slice must still fill the GPU: 32768 streams for the thread-per-stream kernel, one warp per stream and
    // 32 resident warps per SM otherwise
    constexpr int kMaxSlices = 8;
    static_assert(kMaxSlices <= kMaxPipeSlices, "one event per slice");
    const uint32_t fill = n >= 32768 ? 32768u : (uint32_t)ctx->sm_count * 32u;
    int kSlices = (int)(n / fill);
    kSlices = kSlices < 2 ? 2 : kSlices > kMaxSlices ? kMaxSlices : kSlices;
    int rc = ensure_copy_streams(ctx);
    if (rc != ZS_OK) return rc;
    // slice boundaries: stream index at which the running input + output bytes pass s/kSlices of the total
    uint32_t b[kMaxSlices + 1];
    const uint64_t total = in_off[n] + out_off[n];
    b[0] = 0;
    for (int s = 1; s < kSlices; s++) {
        const uint64_t want = total / kSlices * s;
        uint32_t lo = b[s - 1], hi = n;
        while (lo < hi) {
            const uint32_t mid = lo + (hi - lo) / 2;
            if (in_off[mid] + out_off[mid] < want) lo = mid + 1; else hi = mid;
        }
        b[s] = lo;
    }
    b[kSlices] = n;
    uint64_t* d_olen = (uint64_t*)d_res;
    uint64_t* d_used = d_olen + n;
    uint32_t* d_checks = (uint32_t*)(d_used + n);
    int32_t* d_status = (int32_t*)(d_checks + n);
    int32_t* d_det = (int32_t*)zs_scratch_get(ctx, SCR_H_DETAIL, (size_t)n * 4);
    if (!d_det) return ZS_MEM_ERROR;
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_ioff, in_off, (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_ooff, out_off, (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    rc = fence_copy_streams(ctx);
    if (rc != ZS_OK) return rc;
    InflateOpts o;
    o.batch_n = n;
    for (int s = 0; s < kSlices; s++) {
        const uint32_t lo = b[s], ns = b[s + 1] - b[s];
        if (ns == 0) continue;
        // whole 8-byte words around the slice's input (the decoders read aligned words)
        const uint64_t i0 = in_off[lo] & ~7ull, i1 = in_off[lo + ns];
        if (i1 > i0) ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_in + i0, in + i0, i1 - i0, cudaMemcpyHostToDevice, ctx->s_in));
        ZS_CUDA_TRY(ctx, cudaEventRecord(ctx->ev_in[s], ctx->s_in));
        ZS_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_in[s], 0));
        rc = inflate_batch_dev_impl(ctx, d_in, d_ioff + lo, ns, window_bits, d_out, d_ooff + lo, d_olen + lo, d_used + lo,
                                    d_checks + lo, d_status + lo, d_dict, d_rng ? d_rng + 2 * (size_t)lo : nullptr, o, nullptr);
        if (rc != ZS_OK) return rc;
        ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_det + lo, ctx->d_last_detail, (size_t)ns * 4, cudaMemcpyDeviceToDevice, ctx->stream));
        ZS_CUDA_TRY(ctx, cudaEventRecord(ctx->ev_kern[s], ctx->stream));
        ZS_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->s_out, ctx->ev_kern[s], 0));
        const uint64_t o0 = out_off[lo], o1 = out_off[lo + ns];
        if (o1 > o0) ZS_CUDA_TRY(ctx, cudaMemcpyAsync(out + o0, d_out + o0, o1 - o0, cudaMemcpyDeviceToHost, ctx->s_out));
    }
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(out_len, d_olen, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (in_used) ZS_CUDA_TRY(ctx, cudaMemcpyAsync(in_used, d_used, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (checks) ZS_CUDA_TRY(ctx, cudaMemcpyAsync(checks, d_checks, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(status, d_status, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->s_out));
    ZS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->d_last_detail = d_det;
    ctx->last_detail_n = n;
    return ZS_OK;
}

int inflate_batch_host_impl(zs_ctx* ctx, const uint8_t* in, const uint64_t* in_off, uint32_t n, int window_bits, uint8_t* out,
                            const uint64_t* out_off, uint64_t* out_len, uint64_t* in_used, uint32_t* checks, int32_t* status,
                            const uint8_t* dict, const uint64_t* dict_rng, uint64_t dict_total, const InflateOpts& opts,
                            InflateOut* res) {
    if (n == 0) return ZS_OK;
    if (!in_off || !out_off || !out_len || !status) return bad_arg(ctx, "inflate: null buffer");
    const uint64_t in_total = in_off[n], out_total = out_off[n];
    if ((in_total && !in) || (out_total && !out)) return bad_arg(ctx, "inflate: null buffer");
    uint8_t* d_in = (uint8_t*)zs_scratch_get(ctx, SCR_H_IN, in_total + 64);
    uint8_t* d_out = (uint8_t*)zs_scratch_get(ctx, SCR_H_OUT, out_total + 64);
    uint64_t* d_ioff = (uint64_t*)zs_scratch_get(ctx, SCR_H_OFF, (size_t)(n + 1) * 8);
    uint64_t* d_ooff = (uint64_t*)zs_scratch_get(ctx, SCR_H_OFF2, (size_t)(n + 1) * 8);
    // results: out_len[n] in_used[n] (u64) | checks[n] status[n] (u32)
    uint8_t* d_res = (uint8_t*)zs_scratch_get(ctx, SCR_H_RES, (size_t)n * 24 + 64);
    if (!d_in || !d_out || !d_ioff || !d_ooff || !d_res) return ZS_MEM_ERROR;
    uint64_t* d_olen = (uint64_t*)d_res;
    uint64_t* d_used = d_olen + n;
    uint32_t* d_checks = (uint32_t*)(d_used + n);
    int32_t* d_status = (int32_t*)(d_checks + n);
    uint8_t* d_dict = nullptr;
    uint64_t* d_rng = nullptr;
    if (dict && dict_rng && dict_total) {
        d_dict = (uint8_t*)zs_scratch_get(ctx, SCR_H_DICT, dict_total + 64);
        d_rng = (uint64_t*)zs_scratch_get(ctx, SCR_H_RNG, (size_t)n * 16);
        if (!d_dict || !d_rng) return ZS_MEM_ERROR;
        ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_dict, dict, dict_total, cudaMemcpyHostToDevice, ctx->stream));
        ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_rng, dict_rng, (size_t)n * 16, cudaMemcpyHostToDevice, ctx->stream));
    }
    // large batches: copies and kernels overlap slice by slice
    if (n >= 2u * (uint32_t)ctx->sm_count * 32u && in_total + out_total >= (64ull << 20) && !opts.resume && !getenv("ZS_INFLATE_UNPIPELINED"))
        return inflate_batch_pipelined(ctx, in, in_off, n, window_bits, out, out_off, out_len, in_used, checks, status, d_in,
                                       d_out, d_ioff, d_ooff, d_res, d_dict, d_rng);
    if (in_total) ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_in, in, in_total, cudaMemcpyHostToDevice, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_ioff, in_off, (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_ooff, out_off, (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    InflateOpts o = opts;
    if (n == 1) {
        o.par.on = true;
        o.par.in_off = in_off[0]; o.par.in_len = in_off[1] - in_off[0];
        o.par.out_off = out_off[0]; o.par.out_cap = out_off[1] - out_off[0];
        o.par.dict_off = d_rng ? dict_rng[0] : 0; o.par.dict_len = d_rng ? dict_rng[1] - dict_rng[0] : 0;
        if (res) {
            res->d_out = d_out + out_off[0];
            res->out_gen = ctx->scr[SCR_H_OUT].gen;
        }
    }
    int rc = inflate_batch_dev_impl(ctx, d_in, d_ioff, n, window_bits, d_out, d_ooff, d_olen, d_used, d_checks, d_status,
                                    d_dict, d_rng, o, res);
    if (rc != ZS_OK) return rc;
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(out_len, d_olen, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (n == 1 && out_total > (1u << 20)) {
        // one stream with a generous capacity (the streaming shim asks for 4x its input): bring back what was produced
        ZS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
        const uint64_t made = out_len[0] < out_total ? out_len[0] : out_total;
        if (made) ZS_CUDA_TRY(ctx, cudaMemcpyAsync(out + out_off[0], d_out + out_off[0], made, cudaMemcpyDeviceToHost, ctx->stream));
    } else if (out_total) {
        ZS_CUDA_TRY(ctx, cudaMemcpyAsync(out, d_out, out_total, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (in_used) ZS_CUDA_TRY(ctx, cudaMemcpyAsync(in_used, d_used, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (checks) ZS_CUDA_TRY(ctx, cudaMemcpyAsync(checks, d_checks, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(status, d_status, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return ZS_OK;
}

extern "C" {

int zs_inflate_batch_dev(zs_ctx* ctx, const uint8_t* d_in, const uint64_t* d_in_off, uint32_t n, int window_bits,
                         uint8_t* d_out, const uint64_t* d_out_off, uint64_t* d_out_len, uint64_t* d_in_used,
                         uint32_t* d_checks, int32_t* d_status, const uint8_t* d_dict, const uint64_t* d_dict_rng) {
    if (ctx) bind_device(ctx);
    if (!ctx) return ZS_STREAM_ERROR;
    // (no segment-parallel decode here, even for one stream: its sizes are on the device)
    return inflate_batch_dev_impl(ctx, d_in, d_in_off, n, window_bits, d_out, d_out_off, d_out_len, d_in_used, d_checks,
                                  d_status, d_dict, d_dict_rng, InflateOpts(), nullptr);
}

int zs_inflate_batch(zs_ctx* ctx, const uint8_t* in, const uint64_t* in_off, uint32_t n, int window_bits, uint8_t* out,
                     const uint64_t* out_off, uint64_t* out_len, uint64_t* in_used, uint32_t* checks, int32_t* status,
                     const uint8_t* dict, const uint64_t* dict_rng, uint64_t dict_total) {
    if (ctx) bind_device(ctx);
    if (!ctx) return ZS_STREAM_ERROR;
    return inflate_batch_host_impl(ctx, in, in_off, n, window_bits, out, out_off, out_len, in_used, checks, status, dict,
                                   dict_rng, dict_total, InflateOpts(), nullptr);
}

int zs_inflate_stream_dev(zs_ctx* ctx, const uint8_t* d_in, uint64_t in_len, int window_bits, uint8_t* d_out, uint64_t out_cap,
                          uint64_t* d_out_len, uint64_t* d_in_used, uint32_t* d_check, int32_t* d_status, const uint8_t* d_dict,
                          uint64_t dict_len) {
    if (ctx) bind_device(ctx);
    if (!ctx) return ZS_STREAM_ERROR;
    if (!d_in || !d_out || !d_out_len || !d_status) return bad_arg(ctx, "inflate: null buffer");
    uint64_t* d_o = (uint64_t*)zs_scratch_get(ctx, SCR_I_STREAM, 8 * 8);
    if (!d_o) return ZS_MEM_ERROR;
    const uint64_t h[6] = {0, in_len, 0, out_cap, 0, dict_len};
    // (pageable source: the copy is staged before the call returns)
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_o, h, sizeof(h), cudaMemcpyHostToDevice, ctx->stream));
    InflateOpts o;
    o.par.on = true;
    o.par.in_len = in_len; o.par.out_cap = out_cap; o.par.dict_len = d_dict ? dict_len : 0;
    return inflate_batch_dev_impl(ctx, d_in, d_o, 1, window_bits, d_out, d_o + 2, d_out_len, d_in_used, d_check, d_status,
                                  d_dict && dict_len ? d_dict : nullptr, d_dict && dict_len ? d_o + 4 : nullptr, o, nullptr);
}

int zs_inflate_last_details(zs_ctx* ctx, int32_t* detail, uint32_t n) {
    if (ctx) bind_device(ctx);
    if (!ctx || !detail) return ZS_STREAM_ERROR;
    if (!ctx->d_last_detail || n > ctx->last_detail_n) return bad_arg(ctx, "inflate: no details available");
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(detail, ctx->d_last_detail, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return ZS_OK;
}

}  // extern "C"
