// zs_inflate_index.cu -- random access into one deflate stream: an index of access points built on the device, and
// many byte ranges extracted from it at once (the method of zlib's examples/zran.c, DESIGN.md 3.3d).
//
// Build (zs_inflate_index_build_dev): the stream is decoded by the one-stream path (zs_inflate_stream_dev), then
//   par_record_kernel   (zs_inflate_par.cu) walks it again, lengths only: a warp per planned segment of the
//                       segment-parallel decode, and one warp over whatever the serial decoder decoded.  Each walk keeps
//                       the block starts the point rule may select (its first one, and any that a multiple of the span
//                       falls on), so the kept starts are a superset of the points;
//   (host)              the rule applied to the kept starts, sorted by bit, gives the points exactly;
//   ix_gather_kernel    copies every point's window (dictionary, then output) out of the decoded output.
// The host rule, the allocation and the gather are zs_index_from_starts, which the indexed deflate calls (zs_api.cu)
// use too: their kept starts come from deflate_record_kernel (zs_huff.cu) and their windows from the input.
// Extract (zs_inflate_index_extract_dev):
//   ix_plan_kernel      per range: the first point at or before its start and the number of intervals it spans;
//   ix_scan_kernel      exclusive scan of those counts (block_scan, zs_common.cuh): work item g belongs to range r with
//                       base[r] <= g < base[r+1];
//   ix_extract_kernel   persistent warps take items from a counter; a warp decodes raw deflate from the item's point
//                       against its window through a private 64 KiB history ring, writing only the item's bytes (the
//                       block walk of zs_inflate_common.cuh, walk_blocks, with ExtractSink);
//   ix_finish_kernel    per range: bytes, status and message code.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "zs_inflate_common.cuh"

struct zs_inflate_index {
    int device;
    int32_t window_bits;
    uint32_t check;
    uint64_t in_len, out_len, span, n;
    std::vector<uint64_t> bit, off;   // host copy of the point table
    std::vector<uint32_t> wlen;
    uint64_t win_total;               // window bytes on the device (each window starts 16-byte aligned)
    void* d_mem;                      // bit[n] | off[n + 1] (off[n] = out_len) | woff[n] | wlen[n] (u64) | - | windows
    const uint64_t* d_bit() const { return (const uint64_t*)d_mem; }
    const uint64_t* d_off() const { return d_bit() + n; }
    const uint64_t* d_woff() const { return d_off() + n + 1; }
    const uint64_t* d_wlen() const { return d_woff() + n; }
    const uint8_t* d_win() const { return (const uint8_t*)(d_wlen() + n + 1); }   // 16-byte aligned
};

namespace {

using namespace zsinf;

constexpr int kWarps = 4;
constexpr uint64_t kRing = 65536;             // per-warp history: a 32 KiB distance plus a 258-byte match never alias
constexpr uint64_t kExportHeader = 56;
constexpr uint64_t kExportPoint = 24;

// ---- build ---------------------------------------------------------------------------------------------------------

__global__ void ix_gather_kernel(const uint64_t* off, const uint64_t* woff, const uint64_t* wlen, uint64_t n, uint8_t* win,
                                 const uint8_t* out, const uint8_t* dict, uint64_t dict_len) {
    for (uint64_t p = blockIdx.x; p < n; p += gridDim.x) {
        const uint64_t o = off[p], wl = wlen[p];
        uint8_t* dst = win + woff[p];
        for (uint64_t i = threadIdx.x; i < wl; i += blockDim.x) {
            const int64_t s = (int64_t)o - (int64_t)wl + (int64_t)i;
            dst[i] = s >= 0 ? out[s] : dict[(int64_t)dict_len + s];
        }
    }
}

// ---- extract -------------------------------------------------------------------------------------------------------

struct IxTables {
    const uint64_t *bit, *off, *woff, *wlen;
    const uint8_t* win;
    uint64_t n, out_len;
};

struct IxRanges {
    const uint64_t *off, *len, *out_off;
    uint64_t* got;
    int32_t* status;
    int32_t* detail;
    uint64_t* p0;     // [n] first point of the range
    uint64_t* base;   // [n + 1] counts, then their exclusive scan (base[n] = items in all)
    uint64_t* fail;   // [n] min over failed items of (byte of the range where it failed << 8 | detail), ~0 = none
    unsigned long long* next;   // item counter of the persistent warps
    uint32_t n;
};

__device__ __forceinline__ uint64_t range_end(uint64_t off, uint64_t len, uint64_t out_len) {
    if (off >= out_len) return off;
    return len > out_len - off ? out_len : off + len;
}

// last point p in [0, n) with off[p] <= x (strict: off[p] < x); off[0] = 0
__device__ __forceinline__ uint64_t last_point(const uint64_t* off, uint64_t n, uint64_t x, bool strict) {
    uint64_t lo = 0, hi = n;
    while (lo < hi) {
        const uint64_t mid = lo + (hi - lo) / 2;
        if (strict ? off[mid] < x : off[mid] <= x) lo = mid + 1; else hi = mid;
    }
    return lo - 1;
}

__global__ void ix_plan_kernel(IxTables t, IxRanges r) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= r.n) return;
    const uint64_t off = r.off[i], e = range_end(off, r.len[i], t.out_len);
    uint64_t p0 = 0, cnt = 0;
    if (e > off) {
        p0 = last_point(t.off, t.n, off, false);
        cnt = last_point(t.off, t.n, e, true) - p0 + 1;
    }
    r.p0[i] = p0;
    r.base[i] = cnt;
    r.fail[i] = ~0ull;
}

// exclusive scan of the counts, in place: base[n] = items in all
__global__ void __launch_bounds__(1024) ix_scan_kernel(uint64_t* base, uint32_t n) {
    block_scan(n, [=](uint32_t i) { return base[i]; }, 0, ~0ull, base);
}

// An item's bytes: every byte decoded from the point goes to the warp's ring, those from `skip` on to dest as well, and
// the walk stops once `want` bytes are out.
struct ExtractSink {
    static constexpr uint64_t M = kRing - 1;
    const uint8_t* in;
    uint8_t* ring;
    uint8_t* dest;
    uint64_t skip, want;
    uint64_t r, h;   // bytes decoded from the point; history bytes in the ring
    __device__ bool at_block(uint64_t, bool) const { return false; }
    __device__ bool full() const { return r >= want; }
    __device__ int stored(uint64_t pos, uint64_t n) {
        const uint64_t c = n < want - r ? n : want - r;
        for (uint64_t j = zs_lane(); j < c; j += 32) {
            const uint8_t b = __ldg(in + pos + j);
            ring[(h + j) & M] = b;
            if (r + j >= skip) dest[r + j - skip] = b;
        }
        __syncwarp();
        r += c; h += c;
        return 0;
    }
    __device__ void literal(unsigned byte) {
        if (zs_lane() == 0) {
            ring[h & M] = (uint8_t)byte;
            if (r >= skip) dest[r - skip] = (uint8_t)byte;
        }
        r++; h++;
    }
    __device__ int match(unsigned len, uint64_t dist) {
        if (dist > h) return D_TOO_FAR;
        const uint64_t c = len < want - r ? len : want - r;
        __syncwarp();
        for (unsigned j = zs_lane(); j < c; j += 32) {
            const uint8_t b = ring[(h - dist + (dist >= c ? j : j % dist)) & M];
            ring[(h + j) & M] = b;
            if (r + j >= skip) dest[r + j - skip] = b;
        }
        __syncwarp();
        r += c; h += c;
        return 0;
    }
};

// One item: raw deflate from bit `bit` against the wl-byte window `win`, through the warp's ring, until `want` bytes
// have been decoded; bytes from `skip` on go to dest.  Returns 0, the detail code of the error, or -1 when the input or
// the stream ended first; *made = bytes decoded.  Warp-uniform.
__device__ int extract_item(const uint8_t* in, uint64_t in_len, uint64_t bit, const uint8_t* win, uint64_t wl, uint8_t* ring,
                            uint64_t skip, uint64_t want, uint8_t* dest, WarpArena& A, const FixedTables& F, uint64_t* made) {
    // windows start 16-byte aligned in the index (and the ring bytes past wl are written before they are read)
    for (uint64_t j = zs_lane(); j < (wl + 15) / 16; j += 32) reinterpret_cast<uint4*>(ring)[j] = reinterpret_cast<const uint4*>(win)[j];
    __syncwarp();
    ExtractSink s{in, ring, dest, skip, want, 0, wl};
    const int rc = walk_blocks_at(in, in_len, bit, A, F, s);
    __syncwarp();
    *made = s.r;
    return rc;
}

__global__ void __launch_bounds__(kWarps * 32, 8) ix_extract_kernel(IxTables t, IxRanges r, const uint8_t* in, uint64_t in_len,
                                                                uint8_t* out, uint8_t* rings) {
    __shared__ WarpArena s_arena[kWarps];
    __shared__ FixedTables s_fixed;
    const unsigned wid = threadIdx.x >> 5, lane = zs_lane();
    if (wid == 0) build_fixed_tables(s_fixed, s_arena[0], false);
    __syncthreads();
    uint8_t* ring = rings + ((uint64_t)blockIdx.x * kWarps + wid) * kRing;
    const uint64_t total = r.base[r.n];
    for (;;) {
        unsigned long long g = 0;
        if (lane == 0) g = atomicAdd(r.next, 1ull);
        g = __shfl_sync(ZS_FULL_MASK, g, 0);
        if (g >= total) break;
        // the range: the last one whose base is <= g
        uint32_t lo = 0, hi = r.n + 1;
        while (lo < hi) {
            const uint32_t mid = lo + (hi - lo) / 2;
            if (r.base[mid] <= g) lo = mid + 1; else hi = mid;
        }
        const uint32_t ri = lo - 1;
        const uint64_t p = r.p0[ri] + (g - r.base[ri]);
        const uint64_t roff = r.off[ri], e = range_end(roff, r.len[ri], t.out_len);
        const uint64_t o = t.off[p], o_next = t.off[p + 1];
        const uint64_t b0 = roff > o ? roff : o, b1 = e < o_next ? e : o_next;
        uint64_t made = 0;
        const int rc = extract_item(in, in_len, t.bit[p], t.win + t.woff[p], t.wlen[p], ring, b0 - o, b1 - o,
                                    out + r.out_off[ri] + (b0 - roff), s_arena[wid], s_fixed, &made);
        if (rc && lane == 0) {
            // the range's bytes before the failure are written; "ended early" has no message of its own (D_NONE)
            const uint64_t at = (b0 - roff) + (made > b0 - o ? made - (b0 - o) : 0);
            atomicMin((unsigned long long*)&r.fail[ri], (unsigned long long)((at << 8) | (unsigned)(rc < 0 ? D_NONE : rc)));
        }
    }
}

__global__ void ix_finish_kernel(IxRanges r, uint64_t out_len) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= r.n) return;
    const uint64_t f = r.fail[i];
    if (f != ~0ull) {
        r.got[i] = f >> 8;
        r.status[i] = ZS_DATA_ERROR;
        r.detail[i] = (int32_t)(f & 255u);
    } else {
        const uint64_t got = range_end(r.off[i], r.len[i], out_len) - r.off[i];
        r.got[i] = got;
        r.status[i] = got < r.len[i] ? ZS_BUF_ERROR : ZS_OK;
        r.detail[i] = D_NONE;
    }
}

// The point rule over the kept block starts (bit, output offset), in stream order: the first start, and every start
// some m = k * span < out_len falls on -- m in (offset of the kept start before it, its offset].  The kept starts
// include every point, so this is the rule over all block starts (DESIGN.md 3.3d).
void select_points(const uint64_t* rec, size_t m, uint64_t span, uint64_t out_len, std::vector<uint64_t>& bit, std::vector<uint64_t>& off) {
    std::vector<size_t> order(m);
    for (size_t i = 0; i < m; i++) order[i] = i;
    std::sort(order.begin(), order.end(), [&](size_t a, size_t b) { return rec[2 * a] < rec[2 * b]; });
    uint64_t prev_bit = ~0ull, prev_off = 0;
    for (size_t k = 0; k < m; k++) {
        const uint64_t b = rec[2 * order[k]], o = rec[2 * order[k] + 1];
        if (b == prev_bit) continue;   // the same start kept by two walks
        bool take = bit.empty();
        if (!take && o > prev_off) {
            const uint64_t mm = (prev_off / span + 1) * span;   // the first multiple above the start before
            take = mm <= o && mm < out_len;
        }
        if (take) { bit.push_back(b); off.push_back(o); }
        prev_bit = b; prev_off = o;
    }
}

// Allocates the index's device memory and uploads its table; the windows are filled by the caller.
int index_alloc(zs_ctx* ctx, zs_inflate_index* x) {
    std::vector<uint64_t> tab(4 * x->n + 2);
    uint64_t* t_off = tab.data() + x->n;
    uint64_t* t_woff = t_off + x->n + 1;
    uint64_t* t_wlen = t_woff + x->n;
    uint64_t w = 0;
    for (uint64_t p = 0; p < x->n; p++) {
        tab[p] = x->bit[p];
        t_off[p] = x->off[p];
        t_woff[p] = w;
        t_wlen[p] = x->wlen[p];
        w += (x->wlen[p] + 15) & ~15ull;
    }
    t_off[x->n] = x->out_len;
    x->win_total = w;
    const size_t bytes = tab.size() * 8 + w + 16;
    cudaError_t e = cudaMalloc(&x->d_mem, bytes);
    if (e == cudaSuccess) e = cudaMemsetAsync(x->d_mem, 0, bytes, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(x->d_mem, tab.data(), tab.size() * 8, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);   // (tab is pageable and goes out of scope)
    if (e != cudaSuccess) return zs_set_cuda_error(ctx, e, "inflate_index: device memory");
    return ZS_OK;
}

void put32(uint8_t* p, uint32_t v) { memcpy(p, &v, 4); }
void put64(uint8_t* p, uint64_t v) { memcpy(p, &v, 8); }
uint32_t get32(const uint8_t* p) { uint32_t v; memcpy(&v, p, 4); return v; }
uint64_t get64(const uint8_t* p) { uint64_t v; memcpy(&v, p, 8); return v; }

}  // namespace

int zs_index_from_starts(zs_ctx* ctx, const uint64_t* rec, uint64_t n_rec, uint64_t span, int window_bits, uint32_t check,
                         uint64_t in_len, uint64_t out_len, const uint8_t* d_src, const uint8_t* d_dict, uint64_t dict_len,
                         uint64_t hist, zs_inflate_index** out) {
    zs_inflate_index* x = new zs_inflate_index();
    x->device = ctx->device;
    x->window_bits = window_bits;
    x->check = check;
    x->in_len = in_len;
    x->out_len = out_len;
    x->span = span;
    x->d_mem = nullptr;
    select_points(rec, n_rec, span, out_len, x->bit, x->off);
    x->n = x->bit.size();
    x->wlen.resize(x->n);
    for (uint64_t p = 0; p < x->n; p++) x->wlen[p] = (uint32_t)(hist + x->off[p] < kWin ? hist + x->off[p] : kWin);
    int rc = index_alloc(ctx, x);
    if (rc == ZS_OK && x->n)
        ZS_KERNEL(ctx, "ix_gather_kernel",
                  ix_gather_kernel<<<(unsigned)(x->n < 4096 ? x->n : 4096), 256, 0, ctx->stream>>>(
                      x->d_off(), x->d_woff(), x->d_wlen(), x->n, (uint8_t*)x->d_win(), d_src, hist ? d_dict : nullptr, dict_len));
    if (rc == ZS_OK) {
        const cudaError_t e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = zs_set_cuda_error(ctx, e, "inflate_index: windows");
    }
    if (rc != ZS_OK) {
        cudaFree(x->d_mem);
        delete x;
        return rc;
    }
    *out = x;
    return ZS_OK;
}

extern "C" {

int zs_inflate_index_build_dev(zs_ctx* ctx, const uint8_t* d_in, uint64_t in_len, int window_bits, uint64_t span, uint8_t* d_out,
                               uint64_t out_cap, const uint8_t* d_dict, uint64_t dict_len, zs_inflate_index_result* res,
                               zs_inflate_index** out) {
    if (out) *out = nullptr;
    if (!ctx) return ZS_STREAM_ERROR;
    cudaSetDevice(ctx->device);
    int wrap = 0, d64 = 0;
    if (!res || !out || !d_in || !d_out) return zs_bad_arg(ctx, "inflate_index_build: null argument");
    if (!zs_inflate_window_bits(window_bits, &wrap, &d64) || d64) return zs_bad_arg(ctx, "inflate_index_build: windowBits out of range (deflate64 has no index)");
    if (span == 0) return zs_bad_arg(ctx, "inflate_index_build: span is zero");
    if (!d_dict) dict_len = 0;
    // the walk's start record [4] | counters [2]
    uint64_t* scr = (uint64_t*)zs_scratch_get(ctx, SCR_X_BUILD, 6 * 8);
    if (!scr) return ZS_MEM_ERROR;
    const uint64_t gen0 = ctx->scr[SCR_P_STATE].gen;
    InflateOneResult one;
    int rc = inflate_stream_one(ctx, d_in, in_len, window_bits, d_out, out_cap, d_dict, dict_len, &one);
    if (rc != ZS_OK) return rc;
    // the segment-parallel path took this stream when it used its state slot in this call
    const bool planned = ctx->scr[SCR_P_STATE].gen != gen0;
    *res = {one.out_len, one.in_used, one.check, one.status, one.detail};
    if (res->status != ZS_STREAM_END) return ZS_OK;
    const uint64_t out_len = one.out_len;

    // the block starts the rule may select
    uint64_t* d_state = planned ? (uint64_t*)ctx->scr[SCR_P_STATE].p : nullptr;
    uint64_t* tail = scr;
    unsigned long long* cnt = (unsigned long long*)(scr + 4);
    const uint64_t tail0[4] = {~0ull, 0, 0, 0};
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(tail, tail0, sizeof(tail0), cudaMemcpyHostToDevice, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaMemsetAsync(cnt, 0, 16, ctx->stream));
    // kept starts: at most one per 10 input bits (the shortest block), and at most the first of every walk plus one per
    // multiple of the span (a planned segment is at least 8 KiB of input)
    const uint64_t by_bits = in_len * 8 / 10 + in_len / 8192 + 4, by_span = out_len / span + in_len / 8192 + 4;
    const uint64_t rec_cap = by_bits < by_span ? by_bits : by_span;
    uint64_t* d_rec = nullptr;
    ZS_CUDA_TRY(ctx, cudaMalloc(&d_rec, rec_cap * 16));
    rc = zs_launch_inflate_record(ctx, d_in, in_len, out_cap, planned, d_state, planned ? d_state + 8 : tail, wrap, span, d_rec,
                                  rec_cap, cnt);
    uint64_t c[2] = {0, 0}, n_planned = 0;
    uint8_t head[2] = {0, 0};
    cudaError_t e = rc == ZS_OK ? cudaMemcpyAsync(c, cnt, 16, cudaMemcpyDeviceToHost, ctx->stream) : cudaSuccess;
    if (rc == ZS_OK && e == cudaSuccess && planned) e = cudaMemcpyAsync(&n_planned, d_state, 8, cudaMemcpyDeviceToHost, ctx->stream);
    if (rc == ZS_OK && e == cudaSuccess && in_len >= 2) e = cudaMemcpyAsync(head, d_in, 2, cudaMemcpyDeviceToHost, ctx->stream);
    if (rc == ZS_OK && e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    std::vector<uint64_t> rec;
    if (rc == ZS_OK && e == cudaSuccess && c[0] <= rec_cap) {
        rec.resize(2 * c[0]);
        if (c[0]) e = cudaMemcpy(rec.data(), d_rec, c[0] * 16, cudaMemcpyDeviceToHost);
    }
    cudaFree(d_rec);
    if (rc != ZS_OK) return rc;
    if (e != cudaSuccess) return zs_set_cuda_error(ctx, e, "inflate_index_build: block starts");
    if (c[0] > rec_cap || c[1] != n_planned + 1) {   // cannot happen: every walk covers part of a stream that decoded
        snprintf(ctx->err, sizeof(ctx->err), "inflate_index_build: the block walk did not complete");
        return ZS_E_CUDA;
    }

    // the dictionary is history only where the decoder used it: raw streams, and zlib streams that name one (FDICT)
    const bool gz = in_len >= 2 && head[0] == 0x1f && head[1] == 0x8b && (wrap & 2);
    const bool fdict = (wrap & 1) && !gz && (head[1] & 0x20);
    const uint64_t hist = (wrap == 0 || fdict) ? (dict_len < kWin ? dict_len : kWin) : 0;
    return zs_index_from_starts(ctx, rec.data(), c[0], span, window_bits, res->check, in_len, out_len, d_out, d_dict, dict_len,
                                hist, out);
}

int zs_inflate_index_build(zs_ctx* ctx, const uint8_t* in, uint64_t in_len, int window_bits, uint64_t span, uint8_t* out,
                           uint64_t out_cap, const uint8_t* dict, uint64_t dict_len, zs_inflate_index_result* res,
                           zs_inflate_index** index) {
    if (index) *index = nullptr;
    if (!ctx) return ZS_STREAM_ERROR;
    cudaSetDevice(ctx->device);
    if ((in_len && !in) || (out_cap && !out) || (dict_len && !dict) || !res) return zs_bad_arg(ctx, "inflate_index_build: null buffer");
    uint8_t* d_in = (uint8_t*)zs_scratch_get(ctx, SCR_X_IN, in_len + 64);
    uint8_t* d_out = (uint8_t*)zs_scratch_get(ctx, SCR_H_OUT, out_cap + 64);
    uint8_t* d_dict = dict_len ? (uint8_t*)zs_scratch_get(ctx, SCR_H_DICT, dict_len + 64) : nullptr;
    if (!d_in || !d_out || (dict_len && !d_dict)) return ZS_MEM_ERROR;
    if (in_len) ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_in, in, in_len, cudaMemcpyHostToDevice, ctx->stream));
    if (dict_len) ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_dict, dict, dict_len, cudaMemcpyHostToDevice, ctx->stream));
    const int rc = zs_inflate_index_build_dev(ctx, d_in, in_len, window_bits, span, d_out, out_cap, d_dict, dict_len, res, index);
    if (rc != ZS_OK) return rc;
    const uint64_t made = res->out_len < out_cap ? res->out_len : out_cap;
    if (made) ZS_CUDA_TRY(ctx, cudaMemcpy(out, d_out, made, cudaMemcpyDeviceToHost));
    return ZS_OK;
}

int zs_inflate_index_info_get(const zs_inflate_index* x, zs_inflate_index_info* info) {
    if (!x || !info) return ZS_STREAM_ERROR;
    info->in_len = x->in_len;
    info->out_len = x->out_len;
    info->span = x->span;
    info->n_points = x->n;
    info->check = x->check;
    info->window_bits = x->window_bits;
    return ZS_OK;
}

int zs_inflate_index_points(const zs_inflate_index* x, uint64_t* in_bit, uint64_t* out_off, uint64_t max) {
    if (!x) return ZS_STREAM_ERROR;
    const uint64_t n = x->n < max ? x->n : max;
    for (uint64_t p = 0; p < n; p++) {
        if (in_bit) in_bit[p] = x->bit[p];
        if (out_off) out_off[p] = x->off[p];
    }
    return ZS_OK;
}

int zs_inflate_index_export(const zs_inflate_index* x, uint8_t* buf, uint64_t cap, uint64_t* len) {
    if (!x || !len) return ZS_STREAM_ERROR;
    uint64_t wsum = 0;
    for (uint64_t p = 0; p < x->n; p++) wsum += x->wlen[p];
    const uint64_t need = kExportHeader + kExportPoint * x->n + wsum;
    *len = need;
    if (cap == 0) return ZS_OK;
    if (!buf || cap < need) return ZS_BUF_ERROR;
    memset(buf, 0, kExportHeader + kExportPoint * x->n);
    memcpy(buf, "ZSIX", 4);
    put32(buf + 4, 1);
    put32(buf + 8, (uint32_t)x->window_bits);
    put64(buf + 16, x->in_len);
    put64(buf + 24, x->out_len);
    put64(buf + 32, x->span);
    put32(buf + 40, x->check);
    put64(buf + 48, x->n);
    // the windows: one copy of the device's 16-byte aligned layout, packed here
    std::vector<uint8_t> dev(x->win_total);
    int prev = -1;
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    cudaSetDevice(x->device);
    const cudaError_t e = x->win_total ? cudaMemcpy(dev.data(), x->d_win(), x->win_total, cudaMemcpyDeviceToHost) : cudaSuccess;
    if (prev >= 0 && prev != x->device) cudaSetDevice(prev);
    if (e != cudaSuccess) return ZS_E_CUDA;
    uint8_t* w = buf + kExportHeader + kExportPoint * x->n;
    uint64_t dw = 0;
    for (uint64_t p = 0; p < x->n; p++) {
        uint8_t* q = buf + kExportHeader + kExportPoint * p;
        put64(q, x->bit[p]);
        put64(q + 8, x->off[p]);
        put32(q + 16, x->wlen[p]);
        memcpy(w, dev.data() + dw, x->wlen[p]);
        w += x->wlen[p];
        dw += (x->wlen[p] + 15) & ~15ull;
    }
    return ZS_OK;
}

int zs_inflate_index_import(zs_ctx* ctx, const uint8_t* buf, uint64_t len, zs_inflate_index** out) {
    if (out) *out = nullptr;
    if (!ctx) return ZS_STREAM_ERROR;
    cudaSetDevice(ctx->device);
    if (!out || (len && !buf)) return zs_bad_arg(ctx, "inflate_index_import: null argument");
    auto bad = [&](const char* msg) {
        snprintf(ctx->err, sizeof(ctx->err), "inflate_index_import: %s", msg);
        return ZS_DATA_ERROR;
    };
    if (len < kExportHeader) return bad("shorter than the header");
    if (memcmp(buf, "ZSIX", 4) != 0) return bad("wrong magic");
    if (get32(buf + 4) != 1) return bad("unknown version");
    const int32_t wb = (int32_t)get32(buf + 8);
    int wrap = 0, d64 = 0;
    if (!zs_inflate_window_bits(wb, &wrap, &d64) || d64) return bad("window_bits out of range");
    if (get32(buf + 12) != 0 || get32(buf + 44) != 0) return bad("reserved field not zero");
    const uint64_t in_len = get64(buf + 16), out_len = get64(buf + 24), span = get64(buf + 32), n = get64(buf + 48);
    if (span == 0) return bad("span is zero");
    if (n == 0 || n > (len - kExportHeader) / kExportPoint) return bad("point count does not fit the length");
    uint64_t wsum = 0, hist = ~0ull;   // hist: dictionary bytes before the stream, from the first window shorter than 32 KiB
    for (uint64_t p = 0; p < n; p++) {
        const uint8_t* q = buf + kExportHeader + kExportPoint * p;
        const uint64_t b = get64(q), o = get64(q + 8);
        const uint32_t wl = get32(q + 16);
        if (get32(q + 20) != 0) return bad("reserved field not zero");
        if (b >= in_len * 8 || o > out_len) return bad("point outside the stream");
        if (p == 0 && o != 0) return bad("first point not at output offset 0");
        if (p > 0 && (b <= get64(q - kExportPoint) || o < get64(q - kExportPoint + 8))) return bad("points not in stream order");
        if (wl > kWin) return bad("window longer than 32 KiB");
        if (wl < kWin) {
            if (wl < o) return bad("window shorter than the output before it");
            if (hist == ~0ull) hist = wl - o;
            else if (wl - o != hist) return bad("windows disagree about the dictionary");
        } else if (hist != ~0ull && o + hist < kWin) {
            return bad("window longer than the output and dictionary before it");
        }
        wsum += wl;
    }
    if (len != kExportHeader + kExportPoint * n + wsum) return bad("length does not match the windows");
    zs_inflate_index* x = new zs_inflate_index();
    x->device = ctx->device;
    x->window_bits = wb;
    x->check = get32(buf + 40);
    x->in_len = in_len; x->out_len = out_len; x->span = span; x->n = n;
    x->d_mem = nullptr;
    x->bit.resize(n); x->off.resize(n); x->wlen.resize(n);
    for (uint64_t p = 0; p < n; p++) {
        const uint8_t* q = buf + kExportHeader + kExportPoint * p;
        x->bit[p] = get64(q); x->off[p] = get64(q + 8); x->wlen[p] = get32(q + 16);
    }
    int rc = index_alloc(ctx, x);
    // the windows in the device's 16-byte aligned layout, then one copy
    std::vector<uint8_t> dev(x->win_total);
    const uint8_t* w = buf + kExportHeader + kExportPoint * n;
    uint64_t dw = 0;
    for (uint64_t p = 0; p < n; p++) {
        memcpy(dev.data() + dw, w, x->wlen[p]);
        w += x->wlen[p];
        dw += (x->wlen[p] + 15) & ~15ull;
    }
    if (rc == ZS_OK && x->win_total) {
        const cudaError_t e = cudaMemcpyAsync((uint8_t*)x->d_win(), dev.data(), x->win_total, cudaMemcpyHostToDevice, ctx->stream);
        if (e != cudaSuccess) rc = zs_set_cuda_error(ctx, e, "inflate_index_import: windows");
    }
    if (rc == ZS_OK) {
        const cudaError_t e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = zs_set_cuda_error(ctx, e, "inflate_index_import: windows");
    }
    if (rc != ZS_OK) {
        cudaFree(x->d_mem);
        delete x;
        return rc;
    }
    *out = x;
    return ZS_OK;
}

void zs_inflate_index_destroy(zs_inflate_index* x) {
    if (!x) return;
    // called from garbage collectors at any time: the caller's current device is left as it was
    int prev = -1;
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    cudaSetDevice(x->device);
    cudaDeviceSynchronize();   // an extraction that reads the index may still be queued on any stream of the device
    cudaFree(x->d_mem);
    if (prev >= 0 && prev != x->device) cudaSetDevice(prev);
    delete x;
}

int zs_inflate_index_extract_dev(zs_ctx* ctx, const zs_inflate_index* x, const uint8_t* d_in, uint64_t in_len, const uint64_t* d_off,
                                 const uint64_t* d_len, uint32_t n, uint8_t* d_out, const uint64_t* d_out_off, uint64_t* d_got,
                                 int32_t* d_status) {
    if (!ctx) return ZS_STREAM_ERROR;
    cudaSetDevice(ctx->device);
    if (!x) return zs_bad_arg(ctx, "inflate_index_extract: no index");
    if (x->device != ctx->device) return zs_bad_arg(ctx, "inflate_index_extract: index built for another device");
    if (in_len != x->in_len) return zs_bad_arg(ctx, "inflate_index_extract: in_len is not the indexed stream's");
    if (n == 0) return ZS_OK;
    if (!d_in || !d_off || !d_len || !d_out || !d_out_off || !d_got || !d_status) return zs_bad_arg(ctx, "inflate_index_extract: null buffer");
    if ((reinterpret_cast<uintptr_t>(d_in) & 7u) != 0) return zs_bad_arg(ctx, "inflate_index_extract: d_in must be 8-byte aligned");
    uint8_t* plan = (uint8_t*)zs_scratch_get(ctx, SCR_X_PLAN, (size_t)n * 28 + 64);
    const unsigned ctas = (unsigned)ctx->sm_count * 8u;
    uint8_t* rings = (uint8_t*)zs_scratch_get(ctx, SCR_X_RING, (size_t)ctas * kWarps * kRing);
    if (!plan || !rings) return ZS_MEM_ERROR;
    IxTables t;
    t.bit = x->d_bit(); t.off = x->d_off(); t.woff = x->d_woff(); t.wlen = x->d_wlen(); t.win = x->d_win();
    t.n = x->n; t.out_len = x->out_len;
    IxRanges r;
    r.off = d_off; r.len = d_len; r.out_off = d_out_off; r.got = d_got; r.status = d_status;
    r.next = (unsigned long long*)plan;
    r.base = (uint64_t*)plan + 1;       // [n + 1]
    r.p0 = r.base + n + 1;              // [n]
    r.fail = r.p0 + n;                  // [n]
    r.detail = (int32_t*)(r.fail + n);  // [n]
    r.n = n;
    ZS_CUDA_TRY(ctx, cudaMemsetAsync(r.next, 0, 8, ctx->stream));
    ZS_KERNEL(ctx, "ix_plan_kernel", ix_plan_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(t, r));
    ZS_KERNEL(ctx, "ix_scan_kernel", ix_scan_kernel<<<1, 1024, 0, ctx->stream>>>(r.base, n));
    ZS_KERNEL(ctx, "ix_extract_kernel", ix_extract_kernel<<<ctas, kWarps * 32, 0, ctx->stream>>>(t, r, d_in, in_len, d_out, rings));
    ZS_KERNEL(ctx, "ix_finish_kernel", ix_finish_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(r, x->out_len));
    ctx->d_last_detail = r.detail;
    ctx->last_detail_n = n;
    return ZS_OK;
}

int zs_inflate_index_extract(zs_ctx* ctx, const zs_inflate_index* x, const uint8_t* in, uint64_t in_len, const uint64_t* off,
                             const uint64_t* len, uint32_t n, uint8_t* out, uint64_t out_cap, const uint64_t* out_off,
                             uint64_t* got, int32_t* status) {
    if (!ctx) return ZS_STREAM_ERROR;
    cudaSetDevice(ctx->device);
    if (!x) return zs_bad_arg(ctx, "inflate_index_extract: no index");
    if (in_len != x->in_len) return zs_bad_arg(ctx, "inflate_index_extract: in_len is not the indexed stream's");
    if (n == 0) return ZS_OK;
    if (!in || !off || !len || !out_off || !got || !status) return zs_bad_arg(ctx, "inflate_index_extract: null buffer");
    // the input each range needs: from its first point's byte to the byte of the point after its last one (or the end),
    // plus the bit reader's read-ahead; output room for every range as clipped to the stream
    std::vector<std::pair<uint64_t, uint64_t>> span;
    span.reserve(n);
    for (uint32_t i = 0; i < n; i++) {
        const uint64_t o = off[i], e = o >= x->out_len ? o : (len[i] > x->out_len - o ? x->out_len : o + len[i]);
        if (e <= o) continue;
        if (!out || out_off[i] > out_cap || e - o > out_cap - out_off[i]) return zs_bad_arg(ctx, "inflate_index_extract: a range does not fit out_cap");
        const uint64_t p0 = (uint64_t)(std::upper_bound(x->off.begin(), x->off.end(), o) - x->off.begin()) - 1;
        const uint64_t p1 = (uint64_t)(std::lower_bound(x->off.begin(), x->off.end(), e) - x->off.begin());   // the point after the last
        const uint64_t lo = (x->bit[p0] >> 3) & ~7ull;
        uint64_t hi = p1 < x->n ? ((x->bit[p1] + 7) >> 3) + 16 : in_len;
        hi = (hi + 7) & ~7ull;
        span.emplace_back(lo, hi < in_len ? hi : in_len);
    }
    std::sort(span.begin(), span.end());
    uint8_t* d_in = (uint8_t*)zs_scratch_get(ctx, SCR_X_IN, in_len + 64);
    uint8_t* d_out = (uint8_t*)zs_scratch_get(ctx, SCR_H_OUT, out_cap + 64);
    uint64_t* d_arr = (uint64_t*)zs_scratch_get(ctx, SCR_H_OFF, (size_t)n * 36 + 64);
    if (!d_in || !d_out || !d_arr) return ZS_MEM_ERROR;
    for (size_t k = 0; k < span.size();) {
        uint64_t lo = span[k].first, hi = span[k].second;
        for (++k; k < span.size() && span[k].first <= hi + 4096; ++k) hi = span[k].second > hi ? span[k].second : hi;
        ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_in + lo, in + lo, hi - lo, cudaMemcpyHostToDevice, ctx->stream));
    }
    uint64_t* d_off = d_arr;
    uint64_t* d_len = d_off + n;
    uint64_t* d_ooff = d_len + n;
    uint64_t* d_got = d_ooff + n;
    int32_t* d_status = (int32_t*)(d_got + n);
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_off, off, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_len, len, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_ooff, out_off, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    int rc = zs_inflate_index_extract_dev(ctx, x, d_in, in_len, d_off, d_len, n, d_out, d_ooff, d_got, d_status);
    if (rc != ZS_OK) return rc;
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(got, d_got, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(status, d_status, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    // the bytes written, back to the caller's buffer (ranges that lie next to each other in one copy)
    std::vector<std::pair<uint64_t, uint64_t>> w;
    for (uint32_t i = 0; i < n; i++)
        if (got[i]) w.emplace_back(out_off[i], out_off[i] + got[i]);
    std::sort(w.begin(), w.end());
    for (size_t k = 0; k < w.size();) {
        uint64_t lo = w[k].first, hi = w[k].second;
        for (++k; k < w.size() && w[k].first <= hi; ++k) hi = w[k].second > hi ? w[k].second : hi;
        ZS_CUDA_TRY(ctx, cudaMemcpyAsync(out + lo, d_out + lo, hi - lo, cudaMemcpyDeviceToHost, ctx->stream));
    }
    ZS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return ZS_OK;
}

}  // extern "C"
