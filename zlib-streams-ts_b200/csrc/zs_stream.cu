// zs_stream.cu -- the z_stream protocol of the reference's deflate()/inflate() on top of the batch engine.
//
// Mirrors, call for call: createDeflateStream/deflateInit2_ (src/mod/deflate/deflate.ts:80,253),
// deflate (:716, argument and progress rules :720-748, flush handling :936-961, trailers :964-988),
// deflateSetDictionary (:367), deflateEnd (:991); createInflateStream/inflateInit2_
// (src/mod/inflate/inflate.ts:68,174), inflate (:332, return rules of inf_leave :1059-1100),
// inflateSetDictionary (:1220), inflateReset (:124), inflateEnd (:1187).
//
// The GPU needs whole chunks, so the shim is framing + buffering only (no codec work on the host):
//  * deflate: input is buffered; a flush, Z_FINISH or 16 MiB of pending input sends one *part* to
//    zs_deflate_batch_dev as a STITCHED + SYNC run of chunks whose first chunk is primed with the
//    last 32 KiB of the previous part.  Every non-final part therefore ends with the reference's
//    own Z_SYNC_FLUSH marker (empty stored block) and is byte aligned; the wrapper trailer of a
//    multi-part stream is assembled from the per-part checksums with *_combine.
//  * inflate: input is buffered and decoded incrementally at block granularity: every attempt reports
//    where the last block it began starts; the blocks before that point are final (their input is
//    dropped, their output joins the running checksum and the 64 KiB window) and the next attempt
//    resumes there in raw mode.  Bytes decoded so far are handed out immediately, Z_STREAM_END gives
//    back the unused input; the wrapper trailer of a stream decoded in several attempts is checked here.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <mutex>
#include <utility>
#include <vector>

#include "zs_common.cuh"

namespace {

// Host byte buffer of the shim (grows without initialising what it grows by): ordinary memory while it is small,
// page-locked once it holds more than kPinAbove.  A pageable cudaMemcpy is staged through the driver's bounce
// buffers at a few GB/s, and a fresh 64 MiB of ordinary memory costs 16 384 page faults on first touch: together
// most of a stream's time (CompressionStream, 64 MiB of text: 47 ms, of which the kernels took 4.3).  Page-locking
// costs about as much as one such copy, so the large buffers are handed from stream to stream through a small
// pool: the first long stream of a process pays for them, the following ones do not.
constexpr size_t kPinAbove = 1u << 20;

// Large host buffers handed from stream to stream: take() hands out the best fit for `want` (or, with
// `else_largest`, the largest buffer there is when none fits), give() keeps at most max_items buffers of max_bytes in
// all and releases the rest.
struct BufPool {
    const size_t max_items, max_bytes;
    void (*const release)(void*);
    std::mutex mu;
    struct Item { uint8_t* p; size_t cap; };
    std::vector<Item> free_list;
    BufPool(size_t items, size_t bytes, void (*rel)(void*)) : max_items(items), max_bytes(bytes), release(rel) {}
    uint8_t* take(size_t want, bool else_largest, size_t* cap) {
        std::lock_guard<std::mutex> g(mu);
        if (free_list.empty()) return nullptr;
        size_t best = free_list.size(), largest = 0;
        for (size_t i = 0; i < free_list.size(); i++) {
            if (free_list[i].cap >= want && (best == free_list.size() || free_list[i].cap < free_list[best].cap)) best = i;
            if (free_list[i].cap > free_list[largest].cap) largest = i;
        }
        if (best == free_list.size()) {
            if (!else_largest) return nullptr;
            best = largest;
        }
        Item it = free_list[best];
        free_list.erase(free_list.begin() + best);
        *cap = it.cap;
        return it.p;
    }
    void give(uint8_t* p, size_t cap) {
        {
            std::lock_guard<std::mutex> g(mu);
            size_t held = 0;
            for (const Item& it : free_list) held += it.cap;
            if (free_list.size() < max_items && held + cap <= max_bytes) { free_list.push_back({p, cap}); return; }
        }
        release(p);
    }
};
// Both pools are never destroyed: they outlive the CUDA runtime's teardown.
// Page-locked buffers: what the pool keeps page-locked between streams.
BufPool& pin_pool() { static BufPool* pool = new BufPool(8, 768u << 20, [](void* p) { cudaFreeHost(p); }); return *pool; }
// The same for large buffers in ORDINARY memory (the inflate side): what is expensive about them is the first touch --
// a device-to-host copy of 64 MiB into freshly mapped pages takes 41 ms on the B200 box, 3.7 ms into pages that have
// been touched (profiles/pincost_r2.txt) -- so a stream's large buffers go to the next stream instead of back to the
// allocator.
BufPool& page_pool() { static BufPool* pool = new BufPool(4, 512u << 20, free); return *pool; }

struct HostBuf {
    uint8_t* p = nullptr;
    size_t n = 0, cap = 0;
    bool pinned = false;
    bool may_pin = true;            // false: stays in ordinary memory whatever its size
    HostBuf() = default;
    HostBuf(const HostBuf&) = delete;
    HostBuf& operator=(const HostBuf&) = delete;
    ~HostBuf() { release(); }
    void release() {
        if (p) {
            if (pinned) pin_pool().give(p, cap);
            else if (cap > kPinAbove) page_pool().give(p, cap);
            else free(p);
        }
        p = nullptr; n = cap = 0; pinned = false;
    }
    uint8_t* data() { return p; }
    const uint8_t* data() const { return p; }
    size_t size() const { return n; }
    bool empty() const { return n == 0; }
    void clear() { n = 0; }
    uint8_t operator[](size_t i) const { return p[i]; }
    // `part_hint`: the size a large buffer is expected to reach (one part of input / its bound of output)
    bool reserve(size_t want, size_t part_hint) {
        if (want <= cap) return true;
        size_t c = cap + (cap >> 1);
        if (c < want) c = want;
        if (may_pin && c > kPinAbove) {
            if (c < part_hint) c = part_hint;
            size_t got = c;
            uint8_t* q = pin_pool().take(c, false, &got);
            if (!q) {   // none in the pool fits: page-lock a new one
                void* h = nullptr;
                if (cudaHostAlloc(&h, c, cudaHostAllocPortable) == cudaSuccess) q = (uint8_t*)h;
                else cudaGetLastError();
            }
            if (q) {
                if (n) memcpy(q, p, n);
                if (p) { if (pinned) pin_pool().give(p, cap); else free(p); }
                p = q; cap = got; pinned = true;
                return true;
            }
        }
        if (pinned) {   // no more page-locked memory: carry on in ordinary memory
            uint8_t* q = (uint8_t*)malloc(c);
            if (!q) return false;
            if (n) memcpy(q, p, n);
            pin_pool().give(p, cap);
            p = q; cap = c; pinned = false;
            return true;
        }
        if (cap <= kPinAbove && c > kPinAbove) {   // becoming large: a buffer whose pages have been touched, if there is one
            size_t got = 0;   // (the largest one when none holds c: growing it with realloc keeps the touched pages)
            uint8_t* q = page_pool().take(c, true, &got);
            if (q) {
                if (n) memcpy(q, p, n);
                free(p);
                p = q; cap = got;
                if (cap >= want) return true;
            }
        }
        uint8_t* q = (uint8_t*)realloc(p, c ? c : 1);
        if (!q) return false;
        p = q; cap = c;
        return true;
    }
    bool append(const uint8_t* src, size_t k, size_t part_hint) {
        if (!reserve(n + k, part_hint)) return false;
        if (k) memcpy(p + n, src, k);
        n += k;
        return true;
    }
    bool push_back(uint8_t b) { return append(&b, 1, 0); }
    bool resize(size_t want) {   // grows without initialising what it grows by
        if (!reserve(want, 0)) return false;
        n = want;
        return true;
    }
    void erase_front(size_t k) {
        if (k >= n) { n = 0; return; }
        memmove(p, p + k, n - k);
        n -= k;
    }
    void swap(HostBuf& o) {
        std::swap(p, o.p); std::swap(n, o.n); std::swap(cap, o.cap); std::swap(pinned, o.pinned); std::swap(may_pin, o.may_pin);
    }
    bool grow(size_t k, size_t part_hint) {   // k more bytes, left uninitialised
        if (!reserve(n + k, part_hint)) return false;
        n += k;
        return true;
    }
};

double now_s() {
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

enum { ST_INIT = 1, ST_BUSY = 2, ST_FINISH = 3 };
constexpr size_t kPartThreshold = 16u << 20;
constexpr size_t kPartOutHint = 2 * kPartThreshold;   // a part's output (the stored-block bound and change) behind what is still waiting
// inflate: while a stream has brought less input than this it is decoded on EVERY call, so the call that brings the
// last byte of a short stream returns Z_STREAM_END and hands back what follows it through avail_in, exactly like the
// reference, however fast the calls arrive.  Longer streams are paced (see zs_stream_inflate): the end may be found in
// a later call, when input that arrived earlier can only be accounted for in total_in (INTEGRATION.md, "Streaming inflate").
// (An attempt on a 32 KiB slice is ~5 ms of one warp decoding serially: with the limit at 256 KiB the first eight
// calls of EVERY stream cost 43 ms -- a third of a 64 MiB DecompressionStream -- so the limit is two slices.)
constexpr size_t kEveryCallBelow = 64u << 10;

struct DeflateState {
    uint32_t magic = 0x44464c54;  // 'DFLT'
    zs_ctx* ctx = nullptr;
    int level = 6, strategy = 0, wrap = 1;
    HostBuf in;                     // buffered, not yet compressed: at most one part (kPartThreshold)
    HostBuf out;                    // compressed, not yet delivered
    // A part that was started because a whole part of input had piled up runs in the BACKGROUND: its copies and
    // kernels are queued on the context's stream and the call returns, so the caller buffers the next part while the
    // GPU compresses this one (the zlib contract lets deflate(Z_NO_FLUSH) hold output back).  Its input stays in
    // `in_flight`, its output lands in `out` behind the bytes that are waiting there, followed by the result record;
    // harvest() -- before the next part, on any flush, on a call without input, at deflateEnd -- waits for it.
    HostBuf in_flight;
    // What deflateReset starts afresh (the buffers above keep their memory)
    struct Progress {
        int status = ST_INIT, last_flush = -2;
        std::vector<uint8_t> hist;      // last <= 32 KiB already compressed (or the preset dictionary)
        size_t out_pos = 0;
        bool pending = false;           // a part is in flight: p_old, p_cap, p_cap_al, p_n describe it
        size_t p_old = 0, p_cap = 0, p_cap_al = 0, p_n = 0;
        bool header_done = false, any_part = false, trailer_done = false, have_dict = false;
        uint32_t check = 0, dict_id = 0;
        uint64_t total_in_len = 0;
    } prog;
    // deflateSetHeader: a copy of the caller's gzip header fields
    bool gz_custom = false, gz_has_extra = false, gz_has_name = false, gz_has_comment = false;
    int gz_text = 0, gz_os = 0, gz_hcrc = 0;
    uint32_t gz_time = 0;
    std::vector<uint8_t> gz_extra, gz_name, gz_comment;
    // ZS_STREAM_PROF=1: where a stream's time went (seconds), printed by deflateEnd
    double t_append = 0, t_part = 0, t_drain = 0, t_alloc = 0, t_d2h = 0, t_created = 0;
    unsigned n_parts = 0, n_calls = 0;
};

struct InflateState {
    uint32_t magic = 0x494e464c;  // 'INFL'
    zs_ctx* ctx = nullptr;
    int window_bits = 15;
    // Decoding is incremental at block granularity: every attempt reports where the last block it began
    // starts; the blocks before that point are final, their input is dropped and the next attempt
    // resumes there in raw mode with the last 64 KiB of output as its window.
    HostBuf in;                     // input not yet consumed: from the byte that holds the next block header on
    HostBuf out;                    // output of the latest attempt (from the resume point); page-locked once it is large
    HostBuf ready;                  // decoded, not yet delivered
    std::vector<uint8_t> leftover;  // input after the end of the stream that could not be handed back (inflateReset keeps it)
    size_t out_cap_hint = 1 << 20;  // (a capacity hint: inflateReset keeps it, a smaller one would cost a re-decode)
    // What inflateReset starts afresh (the buffers above keep their memory)
    struct Progress {
        bool out_on_device = false;     // `out` is byte for byte what the last attempt left on the device at out_dev ...
        const uint8_t* out_dev = nullptr;
        uint64_t out_gen = 0;           // ... as long as the context has not handed that scratch out again (InflateOut)
        std::vector<uint8_t> hist;      // window: the last <= 64 KiB of final output, or the preset dictionary
        size_t ready_pos = 0;           // delivered part of `ready`
        size_t out_pushed = 0;          // bytes of `out` already copied to `ready`
        size_t next_attempt = 0;
        bool fresh_input = false;       // input has arrived since the last attempt
        uint32_t in_tail = 1;           // the last 4 input bytes received, across calls (big endian; 1 = none yet)
        double attempt_end = 0.0;       // monotonic clock at the end of the last attempt ...
        double attempt_cost = 0.0;      // ... and how long it took (seconds): the pacing of a long stream's attempts
        bool body = false;              // the wrapper header is behind us: raw blocks from start_bit
        uint64_t start_bit = 0;         // of the next block header inside `in`
        int trailer = 0;                // 0 none (raw), 1 zlib (adler32), 2 gzip (crc32 + isize)
        uint32_t run_check = 0;         // checksum of the final output so far (adler32 for zlib, crc32 otherwise)
        uint64_t run_len = 0;           // its length
        bool await_trailer = false;     // the last block is decoded, the trailer bytes are not all here yet
        size_t trailer_pos = 0;         // where they start inside `in`
        bool done = false, failed = false, need_dict = false, have_dict = false;
        int fail_code = 0;
        const char* fail_msg = "";
        uint32_t check = 0;
        zs_gz_header* gzhead = nullptr;   // inflateGetHeader (inflateReset drops the request)
    } prog;
    // The inflate buffers stay in ordinary memory: their sizes follow the stream (four times the buffered input, what
    // is waiting for delivery), so page-locked ones would rarely be reusable from stream to stream, and page-locking
    // 100 MiB anew costs more than the pageable copy it replaces (measured through the stream API: 0.39-0.91 GB/s,
    // erratic, and the pool's churn slowed the deflate streams between them from 3 to 0.5-1.2 GB/s).
    InflateState() { in.may_pin = false; out.may_pin = false; ready.may_pin = false; t_created = now_s(); }
    // ZS_STREAM_PROF=1: where a stream's time went (seconds), printed by inflateEnd
    double t_created = 0, t_insert = 0, t_attempts = 0, t_engine = 0, t_deliver = 0;
    unsigned n_attempts = 0, n_calls = 0;
};

int rank_of(int f) { return f * 2 - (f > 4 ? 9 : 0); }  // RANK, deflate.ts:105

// inflate: a long stream whose calls arrive faster than attempts complete waits kPaceFactor x the duration of its
// last attempt before the next one, or until this much undecoded input is buffered
constexpr double kPaceFactor = 2.0;
constexpr size_t kAttemptAtLeastEvery = 64u << 20;

DeflateState* dstate(zs_stream* s) {
    if (!s || !s->state) return nullptr;
    DeflateState* st = (DeflateState*)s->state;
    return st->magic == 0x44464c54 ? st : nullptr;
}
InflateState* istate(zs_stream* s) {
    if (!s || !s->state) return nullptr;
    InflateState* st = (InflateState*)s->state;
    return st->magic == 0x494e464c ? st : nullptr;
}


// crc32 of a few header bytes on the host (framing only; payload checksums are computed on the GPU)
uint32_t host_crc32(const uint8_t* p, size_t n) {
    uint32_t c = 0xffffffffu;
    for (size_t i = 0; i < n; i++) {
        c ^= p[i];
        for (int k = 0; k < 8; k++) c = (c >> 1) ^ (0xedb88320u & (0u - (c & 1u)));
    }
    return c ^ 0xffffffffu;
}

// The gzip header with the caller's fields, deflate.ts:803-921.
void put_gzip_header(DeflateState* st) {
    std::vector<uint8_t> h;
    h.push_back(0x1f); h.push_back(0x8b); h.push_back(8);
    h.push_back((uint8_t)((st->gz_text ? 1 : 0) + (st->gz_hcrc ? 2 : 0) + (st->gz_has_extra ? 4 : 0) +
                          (st->gz_has_name ? 8 : 0) + (st->gz_has_comment ? 16 : 0)));
    for (int k = 0; k < 4; k++) h.push_back((uint8_t)(st->gz_time >> (8 * k)));
    h.push_back(zs_gzip_xfl(st->level, st->strategy));
    h.push_back((uint8_t)st->gz_os);
    if (st->gz_has_extra) {
        const uint32_t n = (uint32_t)st->gz_extra.size() & 0xffffu;
        h.push_back((uint8_t)n); h.push_back((uint8_t)(n >> 8));
        h.insert(h.end(), st->gz_extra.begin(), st->gz_extra.begin() + n);
    }
    if (st->gz_has_name) h.insert(h.end(), st->gz_name.begin(), st->gz_name.end());        // with the terminator
    if (st->gz_has_comment) h.insert(h.end(), st->gz_comment.begin(), st->gz_comment.end());
    if (st->gz_hcrc) {
        const uint32_t c = host_crc32(h.data(), h.size());
        h.push_back((uint8_t)c); h.push_back((uint8_t)(c >> 8));
    }
    st->out.append(h.data(), h.size(), 0);
}

// A part is done and `res` is its result: fold its check into the stream's running check (read_buf,
// deflate.ts:155-159) and count its n bytes of input.
int end_part(zs_stream* strm, DeflateState* st, const zs_deflate_result& res, uint64_t cap, size_t n) {
    DeflateState::Progress& p = st->prog;
    if (res.total_out_bytes > cap) return ZS_BUF_ERROR;
    if (st->wrap != ZS_WRAP_RAW) {
        p.check = p.total_in_len || p.any_part ? zs_host_check_combine(st->wrap, p.check, res.check, n) : res.check;
        strm->adler = p.check;
    }
    p.total_in_len += n;
    p.header_done = true;
    p.any_part = true;
    return ZS_OK;
}

// History for the next part: the last 32 KiB of (history + the part's input).
void keep_history(std::vector<uint8_t>& hist, const HostBuf& in) {
    const size_t hist_len = hist.size(), total = hist_len + in.size(), keep = total < 32768 ? total : 32768;
    std::vector<uint8_t> h(keep);
    for (size_t i = 0; i < keep; i++) {
        size_t idx = total - keep + i;
        h[i] = idx < hist_len ? hist[idx] : in[idx - hist_len];
    }
    hist.swap(h);
}

// Wait for the part in flight (if any) and take its output and checksum.
int harvest(zs_stream* strm, DeflateState* st) {
    DeflateState::Progress& p = st->prog;
    if (!p.pending) return ZS_OK;
    zs_ctx* ctx = st->ctx;
    p.pending = false;
    const double t0 = now_s();
    ZS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    st->t_part += now_s() - t0;
    zs_deflate_result res;
    memcpy(&res, st->out.data() + p.p_old + p.p_cap_al, sizeof(res));
    const int rc = end_part(strm, st, res, p.p_cap, p.p_n);
    if (rc != ZS_OK) return rc;
    st->out.n = p.p_old + (size_t)res.total_out_bytes;
    st->in_flight.clear();
    return ZS_OK;
}

// Wait for the part in flight (if any) without taking its output: before its buffers are cleared or released.
void wait_part(DeflateState* st) {
    if (!st->prog.pending) return;
    cudaSetDevice(st->ctx->device);
    cudaStreamSynchronize(st->ctx->stream);
    st->prog.pending = false;
}

// Compress everything buffered as one part.  `finish` makes it the last part of the stream; `background`: queue it
// and return (see DeflateState::in_flight).
int run_part(zs_stream* strm, DeflateState* st, bool finish, bool full_flush, bool background = false) {
    zs_ctx* ctx = st->ctx;
    DeflateState::Progress& p = st->prog;
    cudaSetDevice(ctx->device);
    {
        const int rc = harvest(strm, st);
        if (rc != ZS_OK) return rc;
    }
    const double t_part0 = now_s();
    struct PartTimer { DeflateState* s; double t0; ~PartTimer() { s->t_part += now_s() - t0; s->n_parts++; } } part_timer{st, t_part0};
    const size_t hist_len = p.hist.size(), n = st->in.size();
    // zlib header with a preset dictionary carries FDICT + DICTID: host framing (deflate.ts:754-777)
    if (!p.header_done && st->wrap == ZS_WRAP_ZLIB && p.have_dict) {
        uint8_t h[6];
        st->out.append(h, zs_put_zlib_header(h, st->level, st->strategy, true, p.dict_id), 0);
        p.header_done = true;
    }
    if (!p.header_done && st->wrap == ZS_WRAP_GZIP && st->gz_custom) {
        put_gzip_header(st);
        p.header_done = true;
    }
    const bool whole = !p.any_part && finish && !p.header_done;  // the GPU frames a single-part stream completely
    uint32_t flags = ZS_FLAG_SYNC | ZS_FLAG_STRATEGY(st->strategy);
    if (p.header_done || p.any_part) flags |= ZS_FLAG_NOT_FIRST;
    if (!finish) flags |= ZS_FLAG_NOT_LAST;
    const uint32_t chunk = n >= (148u * 4u * 262144u) ? 262144u : 65536u;
    const uint32_t n_chunks = n ? (uint32_t)((n + chunk - 1) / chunk) : 1u;
    const uint64_t cap = zs_deflate_batch_bound(n, n_chunks, chunk, st->wrap, ZS_MODE_STITCHED);
    // Device buffers of a part: the context's grow-only scratch (the slots of the host-buffer batch calls, which are
    // free while a part runs: zs_deflate_batch_dev uses the SCR_D_* slots only).  They used to belong to the stream --
    // cudaMalloc at its first part, cudaFree at deflateEnd -- and the driver took up to 19 ms for the one and 17 ms for
    // the other: as much as the whole 64 MiB stream (ZS_STREAM_PROF).
    const double t_alloc0 = now_s();
    uint8_t* d_in_buf = (uint8_t*)zs_scratch_get(ctx, SCR_H_IN, hist_len + n + 64 + 16);
    uint8_t* d_out_buf = (uint8_t*)zs_scratch_get(ctx, SCR_H_OUT, cap + 64);
    uint8_t* d_res_buf = (uint8_t*)zs_scratch_get(ctx, SCR_H_RES, 256);
    st->t_alloc += now_s() - t_alloc0;
    if (!d_in_buf || !d_out_buf || !d_res_buf) return ZS_MEM_ERROR;
    // history and input are contiguous on the device; keep the input 16-byte aligned
    const size_t pad = (16 - (hist_len & 15)) & 15;
    uint8_t* d_hist = d_in_buf + pad;
    if (hist_len) ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_hist, p.hist.data(), hist_len, cudaMemcpyHostToDevice, ctx->stream));
    if (n) ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_hist + hist_len, st->in.data(), n, cudaMemcpyHostToDevice, ctx->stream));
    zs_deflate_result* d_result = (zs_deflate_result*)d_res_buf;
    int rc = zs_deflate_batch_dev(ctx, d_hist + hist_len, n, nullptr, n_chunks, chunk, chunk, (uint32_t)hist_len, st->level,
                                  st->wrap, ZS_MODE_STITCHED, flags, d_out_buf, cap, nullptr, nullptr, nullptr, d_result);
    if (rc != ZS_OK) return rc;
    if (background && !finish && !full_flush) {
        // what is still waiting in `out` moves to its front, the part's output (as much as it can be: its size is
        // known only when the kernels are done) and the result record are copied behind it; harvest() ends the part
        if (p.out_pos == st->out.size()) st->out.clear();
        else if (p.out_pos) st->out.erase_front(p.out_pos);
        p.out_pos = 0;
        const size_t old = st->out.size(), cap_al = ((size_t)cap + 15) & ~(size_t)15;
        if (!st->out.reserve(old + cap_al + 64, kPartOutHint)) return ZS_MEM_ERROR;
        ZS_CUDA_TRY(ctx, cudaMemcpyAsync(st->out.data() + old + cap_al, d_result, sizeof(zs_deflate_result), cudaMemcpyDeviceToHost, ctx->stream));
        ZS_CUDA_TRY(ctx, cudaMemcpyAsync(st->out.data() + old, d_out_buf, cap, cudaMemcpyDeviceToHost, ctx->stream));
        p.pending = true;
        p.p_old = old; p.p_cap = (size_t)cap; p.p_cap_al = cap_al; p.p_n = n;
        keep_history(p.hist, st->in);
        st->in.swap(st->in_flight);   // the copy engine is still reading it
        st->in.clear();
        return ZS_OK;
    }
    zs_deflate_result res;
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(&res, d_result, sizeof(res), cudaMemcpyDeviceToHost, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    rc = end_part(strm, st, res, cap, n);
    if (rc != ZS_OK) return rc;
    const size_t old = st->out.size();
    const double t_d2h0 = now_s();
    if (!st->out.grow(res.total_out_bytes, kPartOutHint)) return ZS_MEM_ERROR;
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(st->out.data() + old, d_out_buf, res.total_out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    st->t_d2h += now_s() - t_d2h0;
    if (finish && !whole && !p.trailer_done) {   // trailer of a multi-part stream (deflate.ts:964-988)
        uint8_t t[8];
        st->out.append(t, zs_put_trailer(t, st->wrap, p.check, p.total_in_len), 0);
    }
    if (finish) p.trailer_done = true;
    // none after Z_FULL_FLUSH
    if (full_flush || finish) p.hist.clear();
    else keep_history(p.hist, st->in);
    st->in.clear();
    return ZS_OK;
}

void drain(zs_stream* strm, HostBuf& out, size_t& pos, bool pending = false) {
    size_t avail = out.size() - pos;
    size_t c = avail < strm->avail_out ? avail : (size_t)strm->avail_out;
    if (c) {
        memcpy(strm->next_out, out.data() + pos, c);
        strm->next_out += c;
        strm->avail_out -= c;
        strm->total_out += c;
        pos += c;
    }
    if (pos == out.size() && !pending) { out.clear(); pos = 0; }   // (a part in flight is writing behind out.size())
}

}  // namespace

extern "C" {

int zs_stream_deflate_init(zs_ctx* ctx, zs_stream* strm, int level, int method, int window_bits, int mem_level,
                           int strategy) {
    if (!strm || !ctx) return ZS_STREAM_ERROR;
    strm->msg = "";
    // deflateInit2_, deflate.ts:263-297
    int wrap = 1;
    if (level == -1) level = 6;
    if (window_bits < 0) {
        wrap = 0;
        if (window_bits < -15) return ZS_STREAM_ERROR;
        window_bits = -window_bits;
    } else if (window_bits > 15) {
        wrap = 2;
        window_bits -= 16;
    }
    if (mem_level < 1 || mem_level > 9 || method != 8 || window_bits < 8 || window_bits > 15 || level < 0 || level > 9 ||
        strategy < 0 || strategy > 4 || (window_bits == 8 && wrap != 1))
        return ZS_STREAM_ERROR;
    DeflateState* st = new DeflateState();
    st->ctx = ctx;
    st->level = level;
    st->strategy = strategy;
    st->wrap = wrap;
    st->prog.status = ST_INIT;
    st->t_created = now_s();
    strm->state = st;
    strm->total_in = strm->total_out = 0;
    strm->adler = wrap == 2 ? 0u : 1u;
    strm->data_type = 2;  // Z_UNKNOWN
    return ZS_OK;
}

int zs_stream_deflate_set_dictionary(zs_stream* strm, const uint8_t* dict, uint32_t dict_len) {
    DeflateState* st = dstate(strm);
    if (!st || !dict) return ZS_STREAM_ERROR;
    // deflate.ts:372-375: not for gzip, for zlib only before the first deflate call, never mid-block
    if (st->wrap == 2 || (st->wrap == 1 && st->prog.status != ST_INIT) || !st->in.empty()) return ZS_STREAM_ERROR;
    if (st->wrap == 1) {
        uint32_t id = 0;
        int rc = zs_checksum(st->ctx, 0, dict, dict_len, strm->adler, &id);
        if (rc != ZS_OK) return rc;
        strm->adler = id;
        st->prog.dict_id = id;
        st->prog.have_dict = true;
    }
    const uint32_t keep = dict_len < 32768 ? dict_len : 32768;
    st->prog.hist.assign(dict + (dict_len - keep), dict + dict_len);
    return ZS_OK;
}

int zs_stream_deflate(zs_stream* strm, int flush) {
    DeflateState* st = dstate(strm);
    if (!st || flush > ZS_BLOCK || flush < 0) return ZS_STREAM_ERROR;
    if (!strm->next_out || (strm->avail_in != 0 && !strm->next_in) || (st->prog.status == ST_FINISH && flush != ZS_FINISH)) {
        strm->msg = "stream error";
        return ZS_STREAM_ERROR;
    }
    if (strm->avail_out == 0) { strm->msg = "buffer error"; return ZS_BUF_ERROR; }
    cudaSetDevice(st->ctx->device);   // (the buffers below may be page-locked: on this context's device, not on device 0)
    st->n_calls++;
    // a part in flight is waited for when the caller asks for output (a call without input, any flush request)
    if (st->prog.pending && (strm->avail_in == 0 || flush != ZS_NO_FLUSH)) {
        const int rc = harvest(strm, st);
        if (rc != ZS_OK) { strm->msg = zs_last_error(st->ctx); return rc; }
    }
    const int old_flush = st->prog.last_flush;
    st->prog.last_flush = flush;
    if (st->prog.out_pos < st->out.size()) {
        drain(strm, st->out, st->prog.out_pos, st->prog.pending);
        if (strm->avail_out == 0) { st->prog.last_flush = -1; return ZS_OK; }
    } else if (strm->avail_in == 0 && rank_of(flush) <= rank_of(old_flush) && flush != ZS_FINISH) {
        strm->msg = "buffer error";
        return ZS_BUF_ERROR;
    }
    if (st->prog.status == ST_FINISH && strm->avail_in != 0) { strm->msg = "buffer error"; return ZS_BUF_ERROR; }
    if (st->prog.status == ST_INIT) {
        if (st->wrap == 1 && !st->prog.have_dict) strm->adler = 1u;
        st->prog.status = ST_BUSY;
    }
    // Input is buffered one part at a time: a call that brings more than a part compresses full parts as it goes
    // and comes back for output room when a part's output does not fit (Z_OK with avail_in > 0, as in the reference).
    while (strm->avail_in) {
        const size_t room = kPartThreshold > st->in.size() ? kPartThreshold - st->in.size() : 0;
        const size_t take = strm->avail_in < room ? (size_t)strm->avail_in : room;
        const double t_app0 = now_s();
        if (!st->in.append(strm->next_in, take, kPartThreshold)) { strm->msg = "insufficient memory"; return ZS_MEM_ERROR; }
        st->t_append += now_s() - t_app0;
        strm->next_in += take;
        strm->total_in += take;
        strm->avail_in -= take;
        if (strm->avail_in == 0 || st->prog.status != ST_BUSY) break;
        const int rc = run_part(strm, st, false, false, true);
        if (rc != ZS_OK) {
            strm->msg = zs_last_error(st->ctx);
            return rc;
        }
        drain(strm, st->out, st->prog.out_pos, st->prog.pending);
        if (st->prog.out_pos < st->out.size()) { st->prog.last_flush = -1; return ZS_OK; }
    }
    if (st->prog.status == ST_BUSY) {
        int rc = ZS_OK;
        if (flush == ZS_FINISH) {
            rc = run_part(strm, st, true, false);
            if (rc == ZS_OK) st->prog.status = ST_FINISH;
        } else if (flush != ZS_NO_FLUSH) {
            if (!st->in.empty() || !st->prog.any_part) {
                rc = run_part(strm, st, false, flush == ZS_FULL_FLUSH);
            } else {
                // nothing new since the last flush point: just the marker (deflate.ts:945-946)
                static const uint8_t marker[5] = {0, 0, 0, 0xff, 0xff};
                st->out.append(marker, 5, 0);
                if (flush == ZS_FULL_FLUSH) st->prog.hist.clear();
            }
        } else if (st->in.size() >= kPartThreshold) {
            rc = run_part(strm, st, false, false, true);
        }
        if (rc != ZS_OK) {
            strm->msg = zs_last_error(st->ctx);
            return rc;
        }
    }
    {
        const double t0 = now_s();
        drain(strm, st->out, st->prog.out_pos, st->prog.pending);
        st->t_drain += now_s() - t0;
    }
    if (flush == ZS_FINISH && st->prog.status == ST_FINISH && st->prog.out_pos >= st->out.size()) return ZS_STREAM_END;
    return ZS_OK;
}

// deflateResetKeep / deflateReset, deflate.ts:444-495: same parameters, fresh stream
int zs_stream_deflate_reset(zs_stream* strm) {
    DeflateState* st = dstate(strm);
    if (!st) return ZS_STREAM_ERROR;
    wait_part(st);
    st->in.clear(); st->in_flight.clear(); st->out.clear();
    st->prog = {};
    strm->total_in = strm->total_out = 0;
    strm->msg = "";
    strm->data_type = 2;
    strm->adler = st->wrap == 2 ? 0u : 1u;
    return ZS_OK;
}

// deflateParams, deflate.ts:553-595.  What has been buffered is compressed with the old parameters
// first (the reference does this with deflate(strm, Z_BLOCK)); like there, Z_BUF_ERROR means that the
// output buffer could not take everything and the call must be repeated after draining.
int zs_stream_deflate_params(zs_stream* strm, int level, int strategy) {
    DeflateState* st = dstate(strm);
    if (!st) return ZS_STREAM_ERROR;
    if (level == -1) level = 6;
    if (level < 0 || level > 9 || strategy < 0 || strategy > 4) return ZS_STREAM_ERROR;
    const bool lazy_old = st->level >= 4, lazy_new = level >= 4;
    const bool func_changes = (st->level == 0) != (level == 0) || lazy_old != lazy_new;
    if ((strategy != st->strategy || func_changes) && st->prog.last_flush != -2) {
        const int err = zs_stream_deflate(strm, ZS_BLOCK);
        if (err == ZS_STREAM_ERROR) return err;
        if (strm->avail_in || !st->in.empty() || st->prog.out_pos < st->out.size()) return ZS_BUF_ERROR;
    }
    st->level = level;
    st->strategy = strategy;
    return ZS_OK;
}

// deflatePending (deflate.ts:505-516): bytes produced but not yet delivered; the engine never holds a
// partial byte back between calls (every part ends byte aligned), so `bits` is always 0, as is
// deflateUsed's answer (deflate.ts:518-526) for the last byte.
int zs_stream_deflate_pending(zs_stream* strm, uint32_t* pending, int* bits) {
    DeflateState* st = dstate(strm);
    if (!st) return ZS_STREAM_ERROR;
    if (pending) {
        const size_t n = st->out.size() - st->prog.out_pos;
        *pending = n > 0xffffffffull ? 0xffffffffu : (uint32_t)n;
    }
    if (bits) *bits = 0;
    return ZS_OK;
}

// deflateSetHeader, deflate.ts:497-503
int zs_stream_deflate_set_header(zs_stream* strm, const zs_gz_header* head) {
    DeflateState* st = dstate(strm);
    if (!st || st->wrap != 2 || !head) return ZS_STREAM_ERROR;
    st->gz_custom = true;
    st->gz_text = head->text; st->gz_time = head->time; st->gz_os = head->os; st->gz_hcrc = head->hcrc;
    st->gz_has_extra = head->extra != nullptr;
    st->gz_has_name = head->name != nullptr;
    st->gz_has_comment = head->comment != nullptr;
    st->gz_extra.clear(); st->gz_name.clear(); st->gz_comment.clear();
    if (head->extra) st->gz_extra.assign(head->extra, head->extra + (head->extra_len & 0xffffu));
    auto zstr = [](const uint8_t* p, std::vector<uint8_t>& v) { size_t n = 0; while (p[n]) n++; v.assign(p, p + n + 1); };
    if (head->name) zstr(head->name, st->gz_name);
    if (head->comment) zstr(head->comment, st->gz_comment);
    return ZS_OK;
}

int zs_stream_deflate_end(zs_stream* strm) {
    DeflateState* st = dstate(strm);
    if (!st) return ZS_STREAM_ERROR;
    const int status = st->prog.status;
    wait_part(st);   // before the buffers go back to the pool
    if (getenv("ZS_STREAM_PROF")) {
        const double t0 = now_s();
        const unsigned long long tin = strm->total_in;
        const double life = t0 - st->t_created, app = st->t_append, part = st->t_part, alloc = st->t_alloc, d2h = st->t_d2h, dr = st->t_drain;
        const unsigned np = st->n_parts, nc = st->n_calls;
        delete st;
        fprintf(stderr, "[stream prof] deflate: %llu bytes in %.1f ms: %u calls, append %.1f ms, %u parts %.1f ms (device alloc %.1f, copy out %.1f), drain %.1f, end %.1f\n",
                tin, 1e3 * life, nc, 1e3 * app, np, 1e3 * part, 1e3 * alloc, 1e3 * d2h, 1e3 * dr, 1e3 * (now_s() - t0));
    } else {
        delete st;
    }
    strm->state = nullptr;
    return status == ST_BUSY ? ZS_DATA_ERROR : ZS_OK;  // deflate.ts:1012
}

// ---- inflate ----------------------------------------------------------------------------------------
int zs_stream_inflate_init(zs_ctx* ctx, zs_stream* strm, int window_bits) {
    if (!strm || !ctx) return ZS_STREAM_ERROR;
    strm->msg = "";
    if (!zs_inflate_window_bits(window_bits, nullptr, nullptr)) return ZS_STREAM_ERROR;
    InflateState* st = new InflateState();
    st->ctx = ctx;
    st->window_bits = window_bits;
    strm->state = st;
    strm->total_in = strm->total_out = 0;
    strm->adler = zs_inflate_initial_adler(window_bits);
    strm->data_type = 0;
    return ZS_OK;
}

// DICTID of a zlib stream that asks for a dictionary: bytes 2..5 of the buffered stream (0 while they are not all here)
static uint32_t dict_id(const InflateState* st) {
    const HostBuf& b = st->in;
    return b.size() >= 6 ? ((uint32_t)b[2] << 24 | (uint32_t)b[3] << 16 | (uint32_t)b[4] << 8 | b[5]) : 0u;
}

int zs_stream_inflate_set_dictionary(zs_stream* strm, const uint8_t* dict, uint32_t dict_len) {
    InflateState* st = istate(strm);
    if (!st || !dict) return ZS_STREAM_ERROR;
    // inflate.ts:1229: raw streams any time before data, wrapped streams only when Z_NEED_DICT was returned
    if (st->window_bits >= 0 && !st->prog.need_dict) return ZS_STREAM_ERROR;
    if (st->prog.need_dict) {
        // DICTID check (inflate.ts:1233-1238)
        uint32_t id = 0;
        int rc = zs_checksum(st->ctx, 0, dict, dict_len, 1u, &id);
        if (rc != ZS_OK) return rc;
        if (id != dict_id(st)) return ZS_DATA_ERROR;
        st->prog.need_dict = false;
        // the 2-byte header and the DICTID are behind us: raw blocks from byte 6, adler32 trailer
        st->prog.body = true;
        st->prog.start_bit = 48;
        st->prog.trailer = 1;
        st->prog.run_check = 1u;
        st->prog.run_len = 0;
    }
    const uint32_t keep = dict_len < 65536 ? dict_len : 65536;
    st->prog.hist.assign(dict + (dict_len - keep), dict + dict_len);
    st->prog.have_dict = true;
    st->prog.next_attempt = 0;
    return ZS_OK;
}

// inflateGetHeader: fill the caller's struct from the buffered start of the stream (host framing; the
// kernel parses and checks the header on its own, inflate.ts:423-580).
static void fill_gz_header(InflateState* st) {
    zs_gz_header* g = st->prog.gzhead;
    if (!g || g->done != 0 || st->prog.body) return;   // `in` starts at the stream start only until the first resume
    const HostBuf& b = st->in;
    if (b.size() < 2) return;
    if (!(b[0] == 0x1f && b[1] == 0x8b)) { g->done = -1; return; }   // a zlib stream (windowBits 32+), inflate.ts:404
    if (b.size() < 10) return;
    const unsigned flg = b[3];
    size_t p = 10;
    size_t xoff = 0, xlen = 0, noff = 0, nlen = 0, coff = 0, clen = 0;
    if (flg & 4) {
        if (b.size() < p + 2) return;
        xlen = b[p] | (b[p + 1] << 8);
        p += 2;
        if (b.size() < p + xlen) return;
        xoff = p; p += xlen;
    }
    if (flg & 8) {
        noff = p;
        while (p < b.size() && b[p]) p++;
        if (p >= b.size()) return;
        nlen = ++p - noff;
    }
    if (flg & 16) {
        coff = p;
        while (p < b.size() && b[p]) p++;
        if (p >= b.size()) return;
        clen = ++p - coff;
    }
    if (flg & 2) { if (b.size() < p + 2) return; }
    g->text = (flg >> 0) & 1;
    g->time = b[4] | (b[5] << 8) | (b[6] << 16) | ((uint32_t)b[7] << 24);
    g->xflags = b[8];
    g->os = b[9];
    g->hcrc = (flg >> 1) & 1;
    g->extra_len = (uint32_t)xlen;
    if ((flg & 4) && g->extra) memcpy(g->extra, b.data() + xoff, xlen < g->extra_max ? xlen : g->extra_max);
    if (g->name) { if (flg & 8) memcpy(g->name, b.data() + noff, nlen < g->name_max ? nlen : g->name_max); else if (g->name_max) g->name[0] = 0; }
    if (g->comment) { if (flg & 16) memcpy(g->comment, b.data() + coff, clen < g->comm_max ? clen : g->comm_max); else if (g->comm_max) g->comment[0] = 0; }
    g->done = 1;
}

// Everything of `out` below `upto` that has not been queued for delivery yet goes to `ready`.
static void push_ready(InflateState* st, size_t upto) {
    if (upto > st->prog.out_pushed) {
        st->ready.append(st->out.data() + st->prog.out_pushed, upto - st->prog.out_pushed, 0);
        st->prog.out_pushed = upto;
    }
}

// Running checksum continued over the first n bytes of `out`.  While the output of the attempt that produced them is
// still on the device (out_dev), the bytes are not uploaded a second time.
static int out_checksum(InflateState* st, size_t n, uint32_t* result) {
    const int kind = st->prog.trailer == 1 ? 0 : 1;
    if (st->prog.out_on_device && st->prog.out_gen == st->ctx->scr[SCR_H_OUT].gen && st->prog.out_dev) return zs_checksum_dev(st->ctx, kind, st->prog.out_dev, n, st->prog.run_check, result);
    return zs_checksum(st->ctx, kind, st->out.data(), n, st->prog.run_check, result);
}

// The blocks before (mark_bit, mark_out) are final: fold their output into the running checksum and
// the window, drop their input, and make the mark the next resume point.
static int advance_to_mark(InflateState* st, uint64_t mark_bit, uint64_t mark_out) {
    if (mark_out) {
        push_ready(st, (size_t)mark_out);
        int rc = out_checksum(st, (size_t)mark_out, &st->prog.run_check);
        if (rc != ZS_OK) return rc;
        st->prog.run_len += mark_out;
        // the window: the last 64 KiB of final output (only those are copied: mark_out is the whole batch of a paced stream)
        if (mark_out >= 65536) {
            st->prog.hist.assign(st->out.data() + (size_t)mark_out - 65536, st->out.data() + (size_t)mark_out);
        } else {
            st->prog.hist.insert(st->prog.hist.end(), st->out.data(), st->out.data() + (size_t)mark_out);
            if (st->prog.hist.size() > 65536) st->prog.hist.erase(st->prog.hist.begin(), st->prog.hist.end() - 65536);
        }
        st->out.erase_front((size_t)mark_out);
        st->prog.out_on_device = false;
        st->prog.out_pushed -= (size_t)mark_out;
    }
    const size_t bytes = (size_t)(mark_bit >> 3);
    st->in.erase_front(bytes);
    st->prog.start_bit = mark_bit & 7u;
    st->prog.body = true;
    return ZS_OK;
}

// The last block is decoded and `out` holds its output: check the trailer (CHECK / LENGTH,
// inflate.ts:1006-1037) if its bytes are here.
static int finish_stream(InflateState* st) {
    const size_t T = st->prog.trailer == 1 ? 4 : st->prog.trailer == 2 ? 8 : 0;
    if (st->in.size() < st->prog.trailer_pos + T) { st->prog.await_trailer = true; return ZS_OK; }
    st->prog.await_trailer = false;
    uint32_t total = st->prog.run_check;
    int rc = out_checksum(st, st->out.size(), &total);
    if (rc != ZS_OK) return rc;
    const uint64_t total_len = st->prog.run_len + st->out.size();
    const uint8_t* t = st->in.data() + st->prog.trailer_pos;
    if (st->prog.trailer == 1) {
        const uint32_t want = (uint32_t)t[0] << 24 | (uint32_t)t[1] << 16 | (uint32_t)t[2] << 8 | t[3];
        if (want != total) { st->prog.failed = true; st->prog.fail_code = ZS_DATA_ERROR; st->prog.fail_msg = "incorrect data check"; return ZS_OK; }
    } else if (st->prog.trailer == 2) {
        const uint32_t want = (uint32_t)t[0] | (uint32_t)t[1] << 8 | (uint32_t)t[2] << 16 | (uint32_t)t[3] << 24;
        const uint32_t isize = (uint32_t)t[4] | (uint32_t)t[5] << 8 | (uint32_t)t[6] << 16 | (uint32_t)t[7] << 24;
        if (want != total) { st->prog.failed = true; st->prog.fail_code = ZS_DATA_ERROR; st->prog.fail_msg = "incorrect data check"; return ZS_OK; }
        if (isize != (uint32_t)total_len) { st->prog.failed = true; st->prog.fail_code = ZS_DATA_ERROR; st->prog.fail_msg = "incorrect length check"; return ZS_OK; }
    }
    st->prog.check = total;
    st->prog.done = true;
    const size_t used = st->prog.trailer_pos + T;
    if (st->in.size() > used) st->leftover.assign(st->in.data() + used, st->in.data() + st->in.size());
    st->in.clear();
    return ZS_OK;
}

static int inflate_attempt(zs_stream* strm, InflateState* st) {
    zs_ctx* ctx = st->ctx;
    if (st->prog.await_trailer) return finish_stream(st);
    const int raw_wb = st->window_bits == -16 ? -16 : -15;
    for (;;) {
        // `out` is rebuilt by every attempt; what was queued from it stays in `ready`
        if (st->out_cap_hint < 4 * st->in.size()) st->out_cap_hint = 4 * st->in.size();   // a typical ratio: fewer re-decodes
        // (the capacity handed to the decoder must be the one the "output full" test below compares with: taken before
        // the line above, a large attempt stopped at the old capacity and was mistaken for "input ran dry")
        const uint64_t in_off[2] = {0, st->in.size()}, out_off[2] = {0, st->out_cap_hint};
        if (!st->out.resize(st->out_cap_hint)) return ZS_MEM_ERROR;
        uint64_t out_len = 0, in_used = 0, rng[2] = {0, st->prog.hist.size()};
        uint32_t check = 0;
        int32_t status = 0, detail = 0;
        InflateOpts opts;
        opts.resume = true;
        opts.start_bit = st->prog.body ? st->prog.start_bit : ~0ull;
        InflateOut io;
        const double t_eng0 = now_s();
        int rc = inflate_batch_host_impl(ctx, st->in.data(), in_off, 1, st->prog.body ? raw_wb : st->window_bits, st->out.data(),
                                         out_off, &out_len, &in_used, &check, &status, st->prog.hist.empty() ? nullptr : st->prog.hist.data(),
                                         st->prog.hist.empty() ? nullptr : rng, st->prog.hist.size(), opts, &io);
        st->t_engine += now_s() - t_eng0;
        if (rc != ZS_OK) { strm->msg = zs_last_error(ctx); return rc; }
        if (status == ZS_BUF_ERROR && out_len == st->out_cap_hint) {  // output full: grow and decode again
            st->out_cap_hint *= 4;
            continue;
        }
        const uint64_t mark_bit = io.mark[0], mark_out = io.mark[1];
        st->out.resize(out_len);
        st->prog.out_on_device = true;
        st->prog.out_dev = io.d_out;
        st->prog.out_gen = io.out_gen;
        if (status == ZS_STREAM_END) {
            if (!st->prog.body) {
                // the whole stream in one attempt: wrapper and trailer were checked on the device
                push_ready(st, out_len);
                st->prog.check = check;
                st->prog.done = true;
                if (st->in.size() > (size_t)in_used) st->leftover.assign(st->in.data() + (size_t)in_used, st->in.data() + st->in.size());
                st->in.clear();
                return ZS_OK;
            }
            push_ready(st, out_len);
            st->prog.trailer_pos = (size_t)in_used;
            return finish_stream(st);
        }
        if (status == ZS_NEED_DICT) { st->prog.need_dict = true; return ZS_OK; }
        if (status == ZS_DATA_ERROR) {
            zs_inflate_last_details(ctx, &detail, 1);
            push_ready(st, out_len);   // what was decoded before the error is delivered first, like the reference
            st->prog.failed = true;
            st->prog.fail_code = ZS_DATA_ERROR;
            st->prog.fail_msg = zs_inflate_message(detail);
            return ZS_OK;
        }
        // the input ran dry (Z_BUF_ERROR / Z_OK): everything decoded so far is final output
        push_ready(st, out_len);
        if (!st->prog.body) {
            // mark_bit > 0 means the wrapper header is complete and the block loop was entered
            if (mark_bit == 0 && st->window_bits >= 0) return ZS_OK;
            const bool gz = st->window_bits > 15 && st->in.size() >= 2 && st->in[0] == 0x1f && st->in[1] == 0x8b;
            st->prog.trailer = st->window_bits < 0 ? 0 : gz ? 2 : 1;
            st->prog.run_check = st->prog.trailer == 1 ? 1u : 0u;
            st->prog.run_len = 0;
        }
        if (mark_bit > st->prog.start_bit || !st->prog.body) return advance_to_mark(st, mark_bit, mark_out);
        return ZS_OK;
    }
}

int zs_stream_inflate(zs_stream* strm, int flush) {
    InflateState* st = istate(strm);
    if (!st || !strm->next_out || (!strm->next_in && strm->avail_in != 0)) return ZS_STREAM_ERROR;
    const uint64_t in0 = strm->avail_in, out0 = strm->avail_out;
    cudaSetDevice(st->ctx->device);   // (large buffers are page-locked: on this context's device, not on device 0)
    // Like inflate(), which stops consuming input when the output buffer is full: while more decoded bytes
    // are waiting than this call can deliver, no new input is taken (the reference's driver loop,
    // streams.ts:86 `while (strm.avail_in > 0)`, then keeps calling with fresh output buffers).
    const bool backlog = st->ready.size() - st->prog.ready_pos > strm->avail_out;
    if (!st->prog.done && !st->prog.failed && !backlog) {
        // input left over from the previous member is consumed first (inflateReset flow)
        if (!st->leftover.empty() && st->in.empty()) {
            st->in.clear();
            st->in.append(st->leftover.data(), st->leftover.size(), 0);
            st->leftover.clear();
            st->prog.next_attempt = 0;
        }
        if (strm->avail_in) {
            const double t_ins0 = now_s();
            if (!st->in.append(strm->next_in, (size_t)strm->avail_in, 0)) { strm->msg = "insufficient memory"; return ZS_MEM_ERROR; }
            for (size_t i = strm->avail_in > 4 ? (size_t)strm->avail_in - 4 : 0; i < strm->avail_in; i++)
                st->prog.in_tail = st->prog.in_tail << 8 | strm->next_in[i];
            st->t_insert += now_s() - t_ins0;
            strm->next_in += strm->avail_in;
            strm->total_in += strm->avail_in;
            strm->avail_in = 0;
        }
        if (st->prog.need_dict) return ZS_NEED_DICT;
        fill_gz_header(st);
        // `in` holds only what follows the last resume point, so an attempt costs the current block plus the new
        // input (a single huge block is decoded from its start each time).  When is one due?
        //  * on every call while the stream is short (kEveryCallBelow), on any flush request, and on a call that
        //    brings no new input while some of what is buffered has not been through an attempt yet (a caller that
        //    never sends Z_FINISH must still reach Z_STREAM_END);
        //  * otherwise attempts are PACED by what they cost: the next one runs once kPaceFactor x the duration of
        //    the last one has passed since it ended (or 64 MiB of undecoded input have piled up).  An attempt costs
        //    the latency of one warp decoding one segment twice (count pass, decode pass: ~13 ms) plus the serial
        //    decoder on what follows the last flush point however little input it holds, while a large one goes
        //    through the segment-parallel decoder (zs_inflate_par.cu) at GB/s.  A caller that is slower than the
        //    decoder -- a socket, an interactive protocol, anything that waits for output -- therefore gets an
        //    attempt on EVERY call, exactly like the reference: progress, Z_STREAM_END and the hand-back of trailing
        //    bytes through avail_in happen in the call that brings the bytes.  A caller that feeds from memory, calls
        //    microseconds apart, gets a few large attempts; between them inflate(Z_NO_FLUSH) consumes input without
        //    producing output, which the zlib contract allows.
        //    (Round 2 first doubled the batches of a long stream -- an attempt when as much input as had been seen had
        //    arrived again: 0.22-0.26 GB/s for a 64 MiB stream fed in 32 KiB slices, nine attempts of ~20 ms.)
        //  * whatever the pace, on a call that brings input which ends with a sync / full flush marker (00 00 ff ff,
        //    possibly split across calls): a request/response peer hands over one flushed message per call and waits
        //    for its reply, so the message must be decoded now.  A memory-fed caller's slice almost never ends on a
        //    marker, so bulk input keeps its pacing;
        //  * and on a call that brings input while the last block is decoded and only the trailer is missing: finishing
        //    the stream is host work plus one checksum, and Z_STREAM_END with the hand-back of what follows the
        //    trailer through avail_in belongs to the call that brings its last byte.
        if (in0) st->prog.fresh_input = true;
        bool due = flush != ZS_NO_FLUSH || st->in.size() >= st->prog.next_attempt || (in0 == 0 && st->prog.fresh_input) ||
                   (in0 && (st->prog.in_tail == 0x0000ffffu || st->prog.await_trailer));
        if (!due && st->prog.fresh_input && now_s() - st->prog.attempt_end >= kPaceFactor * st->prog.attempt_cost) due = true;
        if (due && !st->in.empty()) {
            const double t_begin = now_s();
            int rc = inflate_attempt(strm, st);
            if (rc != ZS_OK) return rc;
            st->prog.fresh_input = false;
            st->prog.attempt_end = now_s();
            st->prog.attempt_cost = st->prog.attempt_end - t_begin;
            st->t_attempts += st->prog.attempt_cost;
            st->n_attempts++;
            st->prog.next_attempt = st->in.size() + ((size_t)strm->total_in < kEveryCallBelow ? 1 : kAttemptAtLeastEvery);
            if (st->prog.need_dict) {
                strm->adler = dict_id(st);
                return ZS_NEED_DICT;
            }
            if (st->prog.done && !st->leftover.empty()) {
                // hand back what the caller gave us in this call and we did not need
                const size_t give = st->leftover.size() <= in0 ? st->leftover.size() : (size_t)in0;
                strm->next_in -= give;
                strm->avail_in += give;
                strm->total_in -= give;
                // Bytes behind the end that arrived in EARLIER calls (a long stream is decoded in batches) cannot
                // be handed back through avail_in any more; total_in stays exact -- it is what the reference's
                // multi-member flow positions the next member with (test/inflate/test-multistream.ts:50-53).
                strm->total_in -= st->leftover.size() - give;
                st->leftover.clear();
            }
        }
    }
    // deliver what has been decoded
    st->n_calls++;
    const double t_del0 = now_s();
    struct DeliverTimer { InflateState* s; double t0; ~DeliverTimer() { s->t_deliver += now_s() - t0; } } deliver_timer{st, t_del0};
    if (st->prog.ready_pos < st->ready.size()) {
        size_t c = st->ready.size() - st->prog.ready_pos;
        if (c > strm->avail_out) c = (size_t)strm->avail_out;
        memcpy(strm->next_out, st->ready.data() + st->prog.ready_pos, c);
        strm->next_out += c;
        strm->avail_out -= c;
        strm->total_out += c;
        st->prog.ready_pos += c;
        if (st->prog.ready_pos == st->ready.size()) { st->ready.clear(); st->prog.ready_pos = 0; }
        else if (st->prog.ready_pos > (8u << 20) && st->prog.ready_pos >= st->ready.size() / 2) {   // (amortised: the delivered half goes, the rest moves once)
            st->ready.erase_front(st->prog.ready_pos);
            st->prog.ready_pos = 0;
        }
    }
    const bool all_out = st->prog.ready_pos >= st->ready.size();
    if (st->prog.failed && all_out) {
        strm->msg = st->prog.fail_msg;
        return st->prog.fail_code;
    }
    if (st->prog.done && all_out) {
        strm->adler = st->prog.check;
        return ZS_STREAM_END;
    }
    // inf_leave, inflate.ts:1092-1098: no progress, or Z_FINISH without reaching the end
    const bool progress = (in0 != strm->avail_in) || (out0 != strm->avail_out);
    // Decoded bytes still waiting for output room: Z_OK = "call again with more room", also under Z_FINISH
    // (the reference never holds decoded bytes back, so it has no such state; streams.ts:139-170 drains with
    // repeated Z_FINISH calls and treats anything but Z_OK / Z_STREAM_END as fatal).
    if (!all_out && progress) return ZS_OK;
    if (!progress || flush == ZS_FINISH) return ZS_BUF_ERROR;
    return ZS_OK;
}

// inflateGetHeader, inflate.ts (state._gzhead = head; head.done = 0)
int zs_stream_inflate_get_header(zs_stream* strm, zs_gz_header* head) {
    InflateState* st = istate(strm);
    if (!st || !head) return ZS_STREAM_ERROR;
    const int wb = st->window_bits;
    if (wb < 16) return ZS_STREAM_ERROR;   // (state._wrap & 2) == 0: raw or zlib-only
    st->prog.gzhead = head;
    head->done = 0;
    return ZS_OK;
}

int zs_stream_inflate_reset(zs_stream* strm) {
    InflateState* st = istate(strm);
    if (!st) return ZS_STREAM_ERROR;
    st->in.clear();
    st->out.clear();
    st->ready.clear();
    st->prog = {};   // (inflateResetKeep drops the header request too)
    strm->total_in = strm->total_out = 0;
    strm->msg = "";
    return ZS_OK;
}

// inflateReset2, inflate.ts:138-172: new windowBits, then inflateReset
int zs_stream_inflate_reset2(zs_stream* strm, int window_bits) {
    InflateState* st = istate(strm);
    if (!st) return ZS_STREAM_ERROR;
    if (!zs_inflate_window_bits(window_bits, nullptr, nullptr)) return ZS_STREAM_ERROR;
    st->window_bits = window_bits;
    st->leftover.clear();
    const int rc = zs_stream_inflate_reset(strm);
    strm->adler = zs_inflate_initial_adler(window_bits);
    return rc;
}

int zs_stream_inflate_end(zs_stream* strm) {
    InflateState* st = istate(strm);
    if (!st) return ZS_STREAM_ERROR;
    if (getenv("ZS_STREAM_PROF"))
        fprintf(stderr, "[stream prof] inflate: %llu bytes out in %.1f ms: %u calls, buffering input %.1f ms, %u attempts %.1f ms (engine incl. copies %.1f), "
                "delivery %.1f ms\n", (unsigned long long)strm->total_out, 1e3 * (now_s() - st->t_created), st->n_calls, 1e3 * st->t_insert,
                st->n_attempts, 1e3 * st->t_attempts, 1e3 * st->t_engine, 1e3 * st->t_deliver);
    delete st;
    strm->state = nullptr;
    return ZS_OK;
}

}  // extern "C"
