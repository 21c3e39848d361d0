// zs_common.cuh -- device helpers shared by the sm_100a kernels of libzsgpu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/zsgpu.h"

#define ZS_FULL_MASK 0xffffffffu

// ---- context (host side) -------------------------------------------------------------------------
// Device scratch of a context: one grow-only buffer per slot (zs_scratch_get).  Every user of a slot works in
// order on the context stream, and a slot that has to grow synchronises that stream before it frees its old
// buffer, so users that share a slot never see each other's work in flight.
enum zs_scratch_slot {
    // zs_launch_checksum_whole and zs_launch_checksum_stream (offsets, partial sums of the pieces): shared by both
    SCR_CK_OFF = 0, SCR_CK_PART,
    // 256 bytes shared by zs_checksum_dev (the result), deflate_batch_dev (segment counter, total check, error
    // flag) and zs_deflate_dict_create (DICTID): each reads its values back or consumes them in its own kernels
    SCR_SMALL,
    // deflate_batch_dev
    SCR_D_SYM, SCR_D_NBLK, SCR_D_DESC, SCR_D_FREQ, SCR_D_CODE, SCR_D_HDR, SCR_D_BITS, SCR_D_PR, SCR_D_OFF,
    SCR_D_CHECKS, SCR_D_OUTOFF, SCR_D_OUTBITS,
    // staged input, output and results of the host-buffer calls (zs_checksum, zs_deflate_batch*, zs_inflate_batch),
    // shared with the deflate stream's parts (zs_stream.cu: run_part), around a zs_deflate_batch_dev that uses none
    SCR_H_IN, SCR_H_OUT, SCR_H_RES,
    // the rest of the host-buffer calls
    SCR_H_OFF, SCR_H_OFF2, SCR_H_DICT, SCR_H_RNG, SCR_H_CHECKS, SCR_H_DETAIL,
    // batch inflate: details / trailers / checksums, the streaming shim's resume record, and zs_inflate_stream_dev's
    // offsets followed by the results inflate_stream_one reads back
    SCR_I_MISC, SCR_I_RESUME, SCR_I_STREAM,
    // one-stream segment-parallel inflate.  SCR_P_STATE is taken by the API layer and shared with the parallel
    // decoder: the header pass writes it, zs_launch_inflate_parallel reads and extends it, inflate_kernel resumes from it
    SCR_P_STATE,
    // zs_inflate_par.cu
    SCR_P_CAND, SCR_P_SEG, SCR_P_PLAN, SCR_P_SYM, SCR_P_WIN, SCR_P_GMAP,
    // zs_gunzip.cu: tile counts, member candidates, one pass's plan and verdict, member-table entries, and the aligned
    // copy of a member decoded alone.  Its own: the batch and one-stream inflate calls it makes use none of them, and
    // zs_gunzip stages its input and output in SCR_H_IN / SCR_H_OUT around them
    SCR_G_TILE, SCR_G_CAND, SCR_G_PASS, SCR_G_MEMB, SCR_G_ALIGN,
    // zs_inflate_index.cu.  Build: the record pass's start record and counters.
    // Extract: per-range plan and verdicts, per-warp history rings, and the staged input of the host-buffer call (its
    // output goes to SCR_H_OUT)
    SCR_X_BUILD, SCR_X_PLAN, SCR_X_RING, SCR_X_IN,
    // zs_deflate_indexed*: the block starts deflate_record_kernel keeps, a counter and a region of pairs per slice.  Its
    // own: the deflate it runs uses the deflate and host-buffer slots above, and the index it makes allocates its memory
    SCR_D_REC,
    ZS_SCR_COUNT
};

struct zs_scratch {
    void* p = nullptr;
    size_t cap = 0;
    uint64_t gen = 0;   // bumped by every zs_scratch_get of the slot: what a call left there is intact while it is unchanged
};

// slices of one pipelined host-buffer call: deflate cuts a batch into at most 16, inflate into at most 8
constexpr int kMaxPipeSlices = 16;

struct zs_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    char err[256] = {0};
    uint64_t launches = 0;
    int sm_count = 148;
    zs_scratch scr[ZS_SCR_COUNT];
    // pinned host staging for small results
    void* h_pin = nullptr;
    size_t h_pin_cap = 0;
    // last inflate details (device ptr into scratch) for zs_inflate_last_details
    int32_t* d_last_detail = nullptr;
    uint32_t last_detail_n = 0;
    // copy streams and events of the pipelined host-buffer paths (ensure_copy_streams, zs_api.cu)
    cudaStream_t s_in = nullptr, s_out = nullptr, s_res = nullptr;   // H2D, bulk D2H, small result readbacks
    cudaEvent_t ev_in[kMaxPipeSlices] = {nullptr};     // [s] slice s is on the device
    cudaEvent_t ev_kern[kMaxPipeSlices] = {nullptr};   // [s] kernels of slice s are done
    cudaEvent_t ev_res[kMaxPipeSlices] = {nullptr};    // [s] result of slice s is on the host
    cudaEvent_t ev_fence = nullptr;                    // the caller's work queued before the call
    // profiling (zs_ctx_profile)
    bool prof_on = false;
    void* prof = nullptr;  // zs_profile*, zs_api.cu
};

void* zs_scratch_get(zs_ctx* ctx, zs_scratch_slot slot, size_t bytes);  // nullptr on failure (err set)
int zs_set_cuda_error(zs_ctx* ctx, cudaError_t e, const char* where);
int zs_bad_arg(zs_ctx* ctx, const char* msg);   // an argument error: msg to ctx->err (ctx may be null), ZS_STREAM_ERROR
#define ZS_CUDA_TRY(ctx, expr)                                                   \
    do {                                                                         \
        cudaError_t _e = (expr);                                                 \
        if (_e != cudaSuccess) return zs_set_cuda_error((ctx), _e, #expr);       \
    } while (0)
#ifdef ZS_DEBUG_HOOKS   // wait for every kernel so that a fault names the kernel that caused it
#define ZS_DEBUG_SYNC(ctx, e) do { if ((e) == cudaSuccess) (e) = cudaStreamSynchronize((ctx)->stream); } while (0)
#else
#define ZS_DEBUG_SYNC(ctx, e) do { } while (0)
#endif
#define ZS_LAUNCH_CHECK(ctx, name)                                               \
    do {                                                                         \
        (ctx)->launches++;                                                       \
        cudaError_t _e = cudaGetLastError();                                     \
        ZS_DEBUG_SYNC(ctx, _e);                                                  \
        if (_e != cudaSuccess) return zs_set_cuda_error((ctx), _e, name);        \
    } while (0)

// per-kernel CUDA-event timing (zs_ctx_profile): begin/end bracket one launch on ctx->stream
void zs_prof_begin(zs_ctx* ctx, const char* name);
void zs_prof_end(zs_ctx* ctx);
#define ZS_KERNEL(ctx, name, ...)        \
    do {                                 \
        zs_prof_begin((ctx), name);      \
        __VA_ARGS__;                     \
        zs_prof_end((ctx));              \
        ZS_LAUNCH_CHECK((ctx), name);    \
    } while (0)

// ---- device helpers --------------------------------------------------------------------------------
#ifdef __CUDACC__

__device__ __forceinline__ unsigned zs_lane() { return threadIdx.x & 31u; }
__device__ __forceinline__ unsigned zs_lanemask_lt() {
    unsigned m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

// Unaligned little-endian loads from a read-only buffer whose base is 8-byte aligned.  `safe_end`
// is the buffer length rounded up to 8: aligned words below it are readable (cudaMalloc and the
// torch caching allocator hand out >= 256-byte granules), words at or above it read as zero.
__device__ __forceinline__ uint64_t zs_ld64(const uint8_t* __restrict__ base, uint64_t pos, uint64_t safe_end) {
    uint64_t a = pos & ~7ull;
    unsigned sh = (unsigned)(pos & 7u) * 8u;
    uint64_t lo = (a < safe_end) ? __ldg(reinterpret_cast<const unsigned long long*>(base + a)) : 0ull;
    if (sh == 0) return lo;
    uint64_t hi = (a + 8 < safe_end) ? __ldg(reinterpret_cast<const unsigned long long*>(base + a + 8)) : 0ull;
    return (lo >> sh) | (hi << (64u - sh));
}

__device__ __forceinline__ uint32_t zs_ld32(const uint8_t* __restrict__ base, uint64_t pos, uint64_t safe_end) {
    uint64_t a = pos & ~3ull;
    unsigned sh = (unsigned)(pos & 3u) * 8u;
    uint32_t lo = (a < safe_end) ? __ldg(reinterpret_cast<const unsigned*>(base + a)) : 0u;
    uint32_t hi = (sh != 0 && a + 4 < safe_end) ? __ldg(reinterpret_cast<const unsigned*>(base + a + 4)) : 0u;
    return __funnelshift_r(lo, hi, sh);
}

// Exclusive scan of n values by one block (<= 1024 threads): out[i] = min(base + sum of val(j) for j < i, clip) for
// i = 0..n.  A thread reads val(i) and writes out[i] for its own [lo, hi) only, and out[n] is never read, so out may
// hold the values themselves (an in-place scan).
template <class Val>
__device__ void block_scan(uint32_t n, const Val& val, uint64_t base, uint64_t clip, uint64_t* out) {
    __shared__ uint64_t s_warp[32];
    const uint32_t per = (n + blockDim.x - 1) / blockDim.x;
    const uint32_t lo = min(n, threadIdx.x * per), hi = min(n, lo + per);
    uint64_t sum = 0;
    for (uint32_t i = lo; i < hi; i++) sum += val(i);
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    uint64_t incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint64_t v = __shfl_up_sync(ZS_FULL_MASK, incl, o);
        if ((int)lane >= o) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const uint64_t w = lane < blockDim.x / 32 ? s_warp[lane] : 0;
        uint64_t wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint64_t v = __shfl_up_sync(ZS_FULL_MASK, wi, o);
            if ((int)lane >= o) wi += v;
        }
        s_warp[lane] = wi - w;
    }
    __syncthreads();
    uint64_t run = base + s_warp[warp] + incl - sum;
    for (uint32_t i = lo; i < hi; i++) {
        const uint64_t v = val(i);
        out[i] = run < clip ? run : clip;
        run += v;
    }
    if (threadIdx.x == blockDim.x - 1) out[n] = run < clip ? run : clip;
}

__device__ __forceinline__ unsigned zs_bitrev(unsigned code, unsigned len) { return __brev(code) >> (32u - len); }

// ---- RFC 1951 symbol geometry (deflate/constants.ts, trees-util.ts; regenerated from the RFC) ----
// length code index 0..28 for (match length - 3)
__device__ __forceinline__ unsigned zs_len_code(unsigned lc) {
    if (lc < 8) return lc;
    if (lc == 255) return 28;
    unsigned hb = 31u - __clz(lc);          // 3..7
    return ((hb - 1u) << 2) + ((lc >> (hb - 2u)) & 3u);
}
__device__ __forceinline__ unsigned zs_len_xbits(unsigned code) { return (code < 8 || code == 28) ? 0u : (code - 4u) >> 2; }
__device__ __forceinline__ unsigned zs_len_base(unsigned code) {  // base of (length - 3)
    if (code < 8) return code;
    if (code == 28) return 255;
    unsigned xb = (code - 4u) >> 2;
    return ((4u + (code & 3u)) << xb);
}
// distance code 0..29 for (distance - 1)
__device__ __forceinline__ unsigned zs_dist_code(unsigned d) {
    if (d < 4) return d;
    unsigned hb = 31u - __clz(d);           // >= 2
    return (hb << 1) + ((d >> (hb - 1u)) & 1u);
}
__device__ __forceinline__ unsigned zs_dist_xbits(unsigned code) { return code < 4 ? 0u : (code - 2u) >> 1; }
__device__ __forceinline__ unsigned zs_dist_base(unsigned code) {  // base of (distance - 1)
    if (code < 4) return code;
    unsigned xb = (code - 2u) >> 1;
    return (2u + (code & 1u)) << xb;
}

#endif  // __CUDACC__

// A prepared preset dictionary (zs_deflate_dict_create): the match finder's tables built from the last
// <= 32 KiB of the caller's dictionary, with those bytes in their ring (layout private to zs_lz77.cu).
struct zs_deflate_dict {
    int device;
    uint32_t len;        // bytes used: the last min(dict_len, 32768)
    uint32_t id;         // adler32 of the whole dictionary (DICTID)
    uint8_t* d_img;      // saved tables
};

// ---- kernel entry points (host wrappers, one per .cu) ---------------------------------------------
// checksum
int zs_launch_checksum_segments(zs_ctx* ctx, int kind, const uint8_t* d_buf, const uint64_t* d_off,
                                const uint64_t* d_len, uint32_t n, uint32_t* d_out);
int zs_launch_checksum_whole(zs_ctx* ctx, int kind, const uint8_t* d_buf, uint64_t len, uint32_t init,
                             uint32_t* d_result);
int zs_launch_checksum_stream(zs_ctx* ctx, int kind, const uint8_t* d_buf, const uint64_t* d_base, const uint64_t* d_len,
                              uint64_t max_len, uint32_t* d_result);
int zs_launch_checksum_fold(zs_ctx* ctx, int kind, const uint32_t* d_part, const uint64_t* d_off, uint32_t n,
                            uint32_t init, uint32_t* d_result);
uint32_t zs_host_crc32_combine(uint32_t c1, uint32_t c2, uint64_t len2);
uint32_t zs_host_adler32_combine(uint32_t a1, uint32_t a2, uint64_t len2);
// The check of a stream continued by len2 bytes whose own check is c2: adler32 for zlib, crc32 for gzip.
inline uint32_t zs_host_check_combine(int wrap, uint32_t c1, uint32_t c2, uint64_t len2) {
    return wrap == ZS_WRAP_ZLIB ? zs_host_adler32_combine(c1, c2, len2) : zs_host_crc32_combine(c1, c2, len2);
}

// ---- wrapper framing (deflate.ts:750-832, 964-988): the device's frame_kernel and the host paths --------
__host__ __device__ inline void zs_put_be32(uint8_t* p, uint32_t x) {
    p[0] = (uint8_t)(x >> 24); p[1] = (uint8_t)(x >> 16); p[2] = (uint8_t)(x >> 8); p[3] = (uint8_t)x;
}
// zlib header: CMF/FLG with FLEVEL from level and strategy (level_flags, deflate.ts:757-765), and with a preset
// dictionary FDICT + DICTID (big-endian, putShortMSB twice).  Returns its length.
__host__ __device__ inline unsigned zs_put_zlib_header(uint8_t* p, int level, int strategy, bool fdict, uint32_t dict_id) {
    unsigned header = (8u + (7u << 4)) << 8;
    const unsigned lf = (strategy >= ZS_STRATEGY_HUFFMAN_ONLY || level < 2) ? 0u : level < 6 ? 1u : level == 6 ? 2u : 3u;
    header |= lf << 6;
    if (fdict) header |= 0x20u;   // PRESET_DICT
    header += 31u - header % 31u;
    p[0] = (uint8_t)(header >> 8); p[1] = (uint8_t)header;
    if (!fdict) return 2;
    zs_put_be32(p + 2, dict_id);
    return 6;
}
// gzip XFL, deflate.ts:796
__host__ __device__ inline uint8_t zs_gzip_xfl(int level, int strategy) {
    return level == 9 ? 2 : (strategy >= ZS_STRATEGY_HUFFMAN_ONLY || level < 2) ? 4 : 0;
}
// The trailer of a `wrap` stream: adler32 big-endian (zlib), crc32 and the input size mod 2^32 little-endian (gzip),
// nothing (raw).  Returns its length.
__host__ __device__ inline unsigned zs_put_trailer(uint8_t* p, int wrap, uint32_t check, uint64_t isize) {
    if (wrap == ZS_WRAP_ZLIB) {
        zs_put_be32(p, check);
        return 4;
    }
    if (wrap != ZS_WRAP_GZIP) return 0;
    p[0] = (uint8_t)check; p[1] = (uint8_t)(check >> 8); p[2] = (uint8_t)(check >> 16); p[3] = (uint8_t)(check >> 24);
    p[4] = (uint8_t)isize; p[5] = (uint8_t)(isize >> 8); p[6] = (uint8_t)(isize >> 16); p[7] = (uint8_t)(isize >> 24);
    return 8;
}

// inflateReset2's windowBits rules (inflate.ts:138-172), and raw deflate64 at -16: false for a value out of range.
// `wrap` (bit0 zlib, bit1 gzip, 0 raw) and `deflate64` may be null.
inline bool zs_inflate_window_bits(int window_bits, int* wrap, int* deflate64) {
    int w, d64 = 0;
    if (window_bits < 0) {
        if (window_bits < -16) return false;
        w = 0;
        d64 = window_bits == -16;
        window_bits = -window_bits;
    } else {
        w = ((window_bits >> 4) + 5) & 3;
        if (window_bits < 48) window_bits &= 15;
    }
    if (window_bits && (window_bits < 8 || window_bits > (d64 ? 16 : 15))) return false;
    if (wrap) *wrap = w;
    if (deflate64) *deflate64 = d64;
    return true;
}
// strm->adler after inflateInit2 / inflateReset2: 1 when a zlib header may come, else 0 (the window size then comes
// from the header, or there is none)
inline uint32_t zs_inflate_initial_adler(int window_bits) {
    return (window_bits >= 0 && (((window_bits >> 4) + 5) & 1)) ? 1u : 0u;
}

// inflate
struct zs_inflate_args {
    const uint8_t* d_in;
    const uint64_t* d_in_off;
    uint32_t n;
    int wrap;       // bit0 zlib, bit1 gzip (both = auto)
    int deflate64;
    uint8_t* d_out;
    const uint64_t* d_out_off;
    uint64_t* d_out_len;
    uint64_t* d_in_used;
    int32_t* d_status;
    int32_t* d_detail;
    uint32_t* d_trailer;  // [2n]: stored check, stored isize (wrapped streams)
    uint32_t* d_flags;    // [n]: 1 = has zlib trailer (adler), 2 = has gzip trailer (crc)
    const uint8_t* d_dict;
    const uint64_t* d_dict_rng;
    const uint32_t* d_dict_adler;   // [n]: adler32 of each stream's dictionary range (zlib streams with FDICT), or nullptr
    int force_tps;        // tests: 1 = thread-per-stream kernel for any batch of >= 32 streams, -1 = never
    // streaming shim (warp kernel only): decode raw blocks from this bit of each stream instead of
    // from its start, and report where the last block that was begun starts: [2n] = (bit offset in the
    // stream, bytes produced before it) -- the point a later call can resume from
    const uint64_t* d_start_bit;
    uint64_t* d_block_mark;
    // segment-parallel decode of one stream (zs_inflate_par.cu):
    //  d_hdr_state != nullptr: parse the wrapper header only and report [5] = bit position of the first block
    //  (~0 if the header does not parse), [6] = trailer kind (1 zlib, 2 gzip)
    //  d_resume != nullptr: [4n] per stream = (start bit or ~0 for "from the beginning", bytes already
    //  produced, trailer kind | 4 = all blocks are decoded, -): continue behind what the parallel part did
    uint64_t* d_hdr_state;
    const uint64_t* d_resume;
};
// n_choice: the stream count that picks the kernel (a slice of a batch decodes like the whole batch)
int zs_launch_inflate(zs_ctx* ctx, const zs_inflate_args& a, uint32_t n_choice);
int zs_launch_inflate_parallel(zs_ctx* ctx, const uint8_t* d_in, uint64_t in_len, uint8_t* d_out, uint64_t out_cap,
                               const uint8_t* d_hist, uint64_t hist_len, uint64_t* d_state, uint64_t* d_resume);
int zs_launch_inflate_record(zs_ctx* ctx, const uint8_t* d_in, uint64_t in_len, uint64_t out_cap, bool planned, uint64_t* d_state,
                             const uint64_t* d_tail, int wrap, uint64_t span, uint64_t* d_rec, uint64_t rec_cap,
                             unsigned long long* d_cnt);
int zs_launch_inflate_verify(zs_ctx* ctx, uint32_t n, const uint32_t* d_adler, const uint32_t* d_crc,
                             const uint32_t* d_trailer, const uint32_t* d_flags, const uint64_t* d_out_len,
                             uint32_t* d_checks, int32_t* d_status, int32_t* d_detail);

// zs_inflate_index.cu: the index of a stream (in_len bytes, out_len bytes of output, its check) from its kept block
// starts -- n_rec (bit, output offset) pairs in any order that include every access point: the points for `span`, and
// their windows gathered from d_src (the output; when hist > 0, preceded by the last hist of dict_len bytes at d_dict).
// Synchronises; *out is set only on success.
int zs_index_from_starts(zs_ctx* ctx, const uint64_t* rec, uint64_t n_rec, uint64_t span, int window_bits, uint32_t check,
                         uint64_t in_len, uint64_t out_len, const uint8_t* d_src, const uint8_t* d_dict, uint64_t dict_len,
                         uint64_t hist, zs_inflate_index** out);

// Options of one batch inflate call (zs_api.cu) that the public entry points do not take.
struct InflateOpts {
    // one stream whose sizes the host knows: it may take the segment-parallel decoder (zs_inflate_par.cu).
    // inflate_batch_host_impl sets it for every one-stream call.
    struct { bool on = false; uint64_t in_off = 0, in_len = 0, out_off = 0, out_cap = 0, dict_off = 0, dict_len = 0; } par;
    // one stream of the streaming shim: decode raw blocks from start_bit (~0: from the wrapper header on) and
    // report the block mark
    bool resume = false;
    uint64_t start_bit = 0;
    uint32_t batch_n = 0;   // streams of the whole batch when this call decodes a slice of it (kernel choice), or 0
};
// What a one-stream call leaves for its caller.
struct InflateOut {
    uint64_t mark[2] = {0, 0};        // resume: (bit offset, bytes produced before it) of the last block begun
    const uint8_t* d_out = nullptr;   // host-buffer call: the stream's output, still on the device ...
    uint64_t out_gen = 0;             // ... while ctx->scr[SCR_H_OUT].gen equals this
};
// What zs_inflate_stream_dev reports for its one stream.
struct InflateOneResult {
    uint64_t out_len, in_used;
    uint32_t check;
    int32_t status, detail;
};
// zs_inflate_stream_dev, then its results and message code read back in one synchronise.
int inflate_stream_one(zs_ctx* ctx, const uint8_t* d_in, uint64_t in_len, int window_bits, uint8_t* d_out, uint64_t out_cap,
                       const uint8_t* d_dict, uint64_t dict_len, InflateOneResult* r);
// zs_inflate_batch with options; `res` may be null.  The caller has bound the context's device.
int inflate_batch_host_impl(zs_ctx* ctx, const uint8_t* in, const uint64_t* in_off, uint32_t n, int window_bits, uint8_t* out,
                            const uint64_t* out_off, uint64_t* out_len, uint64_t* in_used, uint32_t* checks, int32_t* status,
                            const uint8_t* dict, const uint64_t* dict_rng, uint64_t dict_total, const InflateOpts& o,
                            InflateOut* res);

// deflate
// Where deflate_record_kernel (zs_huff.cu) appends the block starts of one deflate call that the access-point rule may
// select: (bit, input offset) pairs local to the call at rec[2i], rec[2i + 1], i taken from *cnt.
struct DeflateRecord {
    uint64_t* rec;
    uint64_t cap;        // pairs
    unsigned long long* cnt;
    uint64_t span;
};
struct zs_deflate_plan {
    const uint8_t* d_in;      // points at the first byte of this call's input
    uint64_t in_len;
    uint32_t history;         // readable bytes before d_in
    const uint64_t* d_in_off; // [n_chunks+1], device (always materialised)
    uint32_t n_chunks;
    uint32_t max_chunk;
    uint32_t max_bpc;         // block descriptor slots per chunk
    uint32_t seg_hint;        // 0 or the LZ77 segment size to use (chunks)
    int level, wrap, mode;
    int strategy;             // ZS_STRATEGY_*
    uint32_t flags;
    // scratch
    uint32_t* d_sym;          // [in_len] packed symbols
    uint32_t* d_chunk_nblk;   // [n_chunks]
    uint32_t* d_blk_desc;     // [n_chunks*max_bpc][4]: sym_begin(rel chunk), sym_count, in_begin(rel chunk), in_len
    uint32_t* d_blk_freq;     // [n_chunks*max_bpc][320]: 286 lit/len + 30 dist (+pad)
    uint32_t* d_blk_code;     // [n_chunks*max_bpc][320]: code | len<<16
    uint32_t* d_blk_hdr;      // [n_chunks*max_bpc][160]: word0 = type | hdr_bits<<8, words 1.. = header bits
    uint64_t* d_blk_bits;     // [n_chunks*max_bpc]: body size in bits (excl. stored padding) / abs bit offset
    uint64_t* d_chunk_pr;     // [n_chunks][2]: P (bits before first stored block, or all), R (rest), packed
    uint32_t* d_seg_counter;  // dynamic segment scheduler
    // outputs
    uint8_t* d_out;
    uint64_t out_cap;
    uint64_t* d_out_off;      // [n_chunks+1]
    uint64_t* d_out_bits;     // [n_chunks]
    uint32_t* d_checks;       // [n_chunks] or nullptr
    uint32_t* d_check_total;  // 1
    zs_deflate_result* d_result;
    int32_t* d_error;         // device flag: ZS_BUF_ERROR if out_cap too small
    const zs_deflate_dict* dict;   // zs_deflate_batch_dict*: every chunk starts from this dictionary, or nullptr
    const DeflateRecord* record;   // zs_deflate_indexed*: keep the block starts an index may select, or nullptr
};
int zs_launch_lz77(zs_ctx* ctx, const zs_deflate_plan& p);
// Runs d_dict[0, len) (len <= 32768, 16-byte aligned, readable to len rounded up to 16) through the match
// finder's insert stages alone and writes the saved tables to d_img (zs_lz77_dict_image_bytes()).
int zs_lz77_dict_build(zs_ctx* ctx, const uint8_t* d_dict, uint32_t len, uint8_t* d_img);
size_t zs_lz77_dict_image_bytes();
int zs_launch_huffman(zs_ctx* ctx, const zs_deflate_plan& p);
int zs_launch_bit_concat(zs_ctx* ctx, uint8_t* d_dst, uint64_t dst_bit_off, const uint8_t* d_src, uint64_t n_bits);
