// zs_gunzip.cu -- zs_gunzip_dev / zs_gunzip: every member of a multi-member gzip file (RFC 1952 2.2) in one call.
//
// The result is what the reference's multi-member loop produces (test/inflate/test-multistream.ts:16-79:
// inflate(Z_FINISH) to Z_STREAM_END, inflateReset, continue at total_in).  What is new here is finding the members:
//  1. locate: a byte scan for 1f 8b 08 with FLG's reserved bits clear; every hit must also pass the decoders' own
//     header parser (read_wrapper_header) over its first kHeaderCheck bytes.  Compacted in position order; position 0
//     is always slot 0.
//  2. plan by hypothesis: candidate k spans [c_k, c_k+1) and produces the ISIZE stored in the 4 bytes before c_k+1; an
//     exclusive scan of those sizes places the outputs.
//  3. decode the planned members as one batch (zs_inflate_batch_dev: kernel choice, checksums, trailer verify).
//  4. verify: member i is trusted when it ended with Z_STREAM_END, used exactly c_i+1 - c_i bytes and produced its
//     planned size -- a boundary is trusted only when the decode before it lands on it.  The first untrusted member
//     (one atomicMin) ends the pass.
//  5. the member the pass could not take, and every member of >= kLargeMember planned input bytes, is decoded alone by
//     zs_inflate_stream_dev (the one-stream path: segment-parallel where it is long): over 1, 2, 4, 8, ... candidates
//     while a try runs short of input or of its planned room -- a Z_STREAM_END over a range is final -- and else over
//     the whole rest of the input, which is the reference's loop step itself: its status, message, total_in and
//     output prefix are final.  Planning starts again behind it.
// A pass that takes nothing (a false candidate at its first member) sends the next 1, 2, 4, ... members straight to the
// one-stream path, and a pass after a failed one plans at most twice the members the failed one took (at least
// kMinWindow), so input full of false candidates costs about what the member-by-member loop costs.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "zs_inflate_common.cuh"

namespace {

constexpr unsigned kLocThreads = 256;
constexpr unsigned kLocBytes = 32;                                    // positions per thread
constexpr uint64_t kLocTile = (uint64_t)kLocThreads * kLocBytes;      // 8 KiB per block
constexpr unsigned kScanThreads = 1024;
// Members of at least this many planned input bytes are decoded alone: one warp decodes 25-30 MB/s, so a long member
// would bound the whole batch, and from this size on the one-stream path cuts a stream into segments (kParMinInput of
// zs_api.cu).  Measured on both sides in profiles/gunzip_b200.txt.
constexpr uint64_t kLargeMember = 128u << 10;
constexpr uint64_t kMinWindow = 16;
// Bytes a candidate's header check may read.  Without a bound, input full of `1f 8b 08 08` and no zero byte would make
// every candidate read its file name to the end of the input: quadratic.  A header longer than this (FEXTRA can be 64
// KiB) stays a candidate unchecked; a false one kept and a true one missed are both settled by the trust rule.
constexpr uint64_t kHeaderCheck = 1024;

// A gzip header that does not fail inside [p, min(in_len, p + kHeaderCheck)): it parses, or it goes on past the bound.
__device__ bool header_plausible(const uint8_t* in, uint64_t in_len, uint64_t safe_end, uint64_t p) {
    zsinf::BitReader br;
    br.open(in, p, in_len - p > kHeaderCheck ? p + kHeaderCheck : in_len, safe_end);
    int status = ZS_OK, detail = 0;
    unsigned tflags = 0;
    zsinf::read_wrapper_header(br, 2, status, detail, tflags, nullptr);
    return status == ZS_OK || status == ZS_BUF_ERROR;
}

// Bit i: a member may start at base + i (base a multiple of 32).
__device__ uint32_t member_starts(const uint8_t* in, uint64_t in_len, uint64_t safe_end, uint64_t base) {
    if (base >= in_len) return 0;
    uint32_t w[10];
#pragma unroll
    for (int k = 0; k < 5; k++) {
        const uint64_t q = zs_ld64(in, base + 8 * k, safe_end);
        w[2 * k] = (uint32_t)q;
        w[2 * k + 1] = (uint32_t)(q >> 32);
    }
    uint32_t m = 0;
#pragma unroll
    for (int i = 0; i < 32; i++) {
        const uint32_t v = __funnelshift_r(w[i >> 2], w[(i >> 2) + 1], (i & 3) * 8);
        if ((v & 0xe0ffffffu) == 0x00088b1fu) m |= 1u << i;
    }
    uint32_t ok = base == 0 ? 1u : 0u;   // position 0 is always a candidate: its decode reports what is wrong with it
    while (m) {
        const int i = __ffs(m) - 1;
        m &= m - 1;
        const uint64_t p = base + (uint64_t)i;
        if (p + 10 <= in_len && header_plausible(in, in_len, safe_end, p)) ok |= 1u << i;
    }
    return ok;
}

// The ISIZE field in the 4 bytes before `end`: the planned output size of the member that ends there.
__device__ __forceinline__ uint32_t isize_before(const uint8_t* in, uint64_t end, uint64_t safe_end) {
    return end >= 4 ? zs_ld32(in, end - 4, safe_end) : 0u;
}

__global__ void __launch_bounds__(kLocThreads) gunzip_locate_kernel(const uint8_t* in, uint64_t in_len, uint64_t safe_end,
                                                                    uint64_t* tile_cnt) {
    const uint64_t base = ((uint64_t)blockIdx.x * kLocThreads + threadIdx.x) * kLocBytes;
    const int n = __popc(member_starts(in, in_len, safe_end, base));
    __shared__ unsigned s_cnt;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    if (n) atomicAdd(&s_cnt, (unsigned)n);
    __syncthreads();
    if (threadIdx.x == 0) tile_cnt[blockIdx.x] = s_cnt;
}

// tile counts [n_tiles] -> tile offsets [n_tiles + 1] behind them; the last is the candidate count
__global__ void __launch_bounds__(kScanThreads) gunzip_scan_tiles_kernel(uint64_t* tile, uint32_t n_tiles) {
    block_scan(n_tiles, [=](uint32_t i) { return tile[i]; }, 0, ~0ull, tile + n_tiles + 1);
}

// Candidates in position order: cand[m] = in_len closes the last one; isz[k] = the ISIZE field before cand[k].
__global__ void __launch_bounds__(kLocThreads) gunzip_compact_kernel(const uint8_t* in, uint64_t in_len, uint64_t safe_end,
                                                                     const uint64_t* tile_off, uint32_t n_tiles, uint64_t* cand,
                                                                     uint32_t* isz) {
    const uint64_t base = ((uint64_t)blockIdx.x * kLocThreads + threadIdx.x) * kLocBytes;
    uint32_t ok = member_starts(in, in_len, safe_end, base);
    const unsigned n = __popc(ok);
    __shared__ unsigned s_warp[kLocThreads / 32];
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    unsigned incl = n;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned v = __shfl_up_sync(ZS_FULL_MASK, incl, o);
        if ((int)lane >= o) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    unsigned before = 0;
    for (unsigned k = 0; k < warp; k++) before += s_warp[k];
    uint64_t at = tile_off[blockIdx.x] + before + incl - n;
    while (ok) {
        const int i = __ffs(ok) - 1;
        ok &= ok - 1;
        const uint64_t p = base + (uint64_t)i;
        cand[at] = p;
        isz[at] = isize_before(in, p, safe_end);
        at++;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        const uint64_t m = tile_off[n_tiles];
        cand[m] = in_len;
        isz[m] = isize_before(in, in_len, safe_end);
    }
}

// Planned output offsets of members k0 .. k0+nb-1 (global candidate index), from `produced` on, clipped to out_cap.
__global__ void __launch_bounds__(kScanThreads) gunzip_plan_kernel(const uint32_t* isz, uint32_t nb, uint64_t produced,
                                                                   uint64_t out_cap, uint64_t* out_off, uint32_t* first_bad) {
    if (threadIdx.x == 0) *first_bad = nb;
    block_scan(nb, [=](uint32_t i) { return isz[i + 1]; }, produced, out_cap, out_off);   // the ISIZE that ends member i
}

// The trust rule of a planned member, and its member-table entry.
__global__ void gunzip_verify_kernel(const uint64_t* cand, const uint32_t* isz, uint32_t nb, const uint64_t* out_off,
                                     const uint64_t* out_len, const uint64_t* in_used, const uint32_t* checks,
                                     const int32_t* status, uint32_t* first_bad, zs_gz_member* mem) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nb) return;
    const uint64_t c0 = cand[i], c1 = cand[i + 1];
    const bool ok = status[i] == ZS_STREAM_END && in_used[i] == c1 - c0 && out_len[i] == (uint64_t)isz[i + 1];
    if (!ok) atomicMin(first_bad, i);
    if (mem) {
        zs_gz_member e;
        e.in_off = c0; e.in_len = c1 - c0; e.out_off = out_off[i]; e.out_len = out_len[i]; e.crc32 = checks[i];
        mem[i] = e;
    }
}

// [0] = members trusted (u), [1] = where the output of member u would start
__global__ void gunzip_pass_kernel(const uint32_t* first_bad, const uint64_t* out_off, uint64_t* res) {
    const uint32_t u = *first_bad;
    res[0] = u;
    res[1] = out_off[u];
}

// inflate(Z_FINISH) of d_in[pos, end) into d_out with `room` bytes, by the one-stream path (zs_inflate_stream_dev).
// That path wants an 8-byte aligned start: a member elsewhere is copied to scratch first.
int decode_one(zs_ctx* ctx, const uint8_t* d_in, uint64_t pos, uint64_t end, uint8_t* d_out, uint64_t room, InflateOneResult* r) {
    const uint64_t len = end - pos;
    const uint8_t* src = d_in + pos;
    if (pos & 7u) {
        uint8_t* al = (uint8_t*)zs_scratch_get(ctx, SCR_G_ALIGN, len + 64);
        if (!al) return ZS_MEM_ERROR;
        ZS_CUDA_TRY(ctx, cudaMemcpyAsync(al, src, len, cudaMemcpyDeviceToDevice, ctx->stream));
        src = al;
    }
    return inflate_stream_one(ctx, src, len, 31, d_out, room, nullptr, 0, r);
}

int gunzip_dev(zs_ctx* ctx, const uint8_t* d_in, uint64_t in_len, uint8_t* d_out, uint64_t out_cap, zs_gunzip_result* res,
               zs_gz_member* members, uint64_t max_members) {
    if (!res || (in_len && !d_in) || (out_cap && !d_out) || (max_members && !members)) return zs_bad_arg(ctx, "gunzip: null buffer");
    if ((reinterpret_cast<uintptr_t>(d_in) & 7u) != 0) return zs_bad_arg(ctx, "gunzip: d_in must be 8-byte aligned");
    memset(res, 0, sizeof(*res));
    if (in_len == 0) {   // inflate() without input makes no progress
        res->status = ZS_BUF_ERROR;
        return ZS_OK;
    }
    if (!members) max_members = 0;
    const uint64_t safe_end = (in_len + 7) & ~7ull;

    // 1. locate: candidate count, then the candidates in position order with the ISIZE field before each
    const uint64_t n_tiles64 = (in_len + kLocTile - 1) / kLocTile;
    if (n_tiles64 > 0x7fffffffull) return zs_bad_arg(ctx, "gunzip: input too large for one call");
    const uint32_t n_tiles = (uint32_t)n_tiles64;
    uint64_t* d_tile = (uint64_t*)zs_scratch_get(ctx, SCR_G_TILE, ((size_t)n_tiles * 2 + 2) * 8);
    if (!d_tile) return ZS_MEM_ERROR;
    uint64_t* d_tile_off = d_tile + n_tiles + 1;
    ZS_KERNEL(ctx, "gunzip_locate_kernel",
              gunzip_locate_kernel<<<n_tiles, kLocThreads, 0, ctx->stream>>>(d_in, in_len, safe_end, d_tile));
    ZS_KERNEL(ctx, "gunzip_scan_tiles_kernel", gunzip_scan_tiles_kernel<<<1, kScanThreads, 0, ctx->stream>>>(d_tile, n_tiles));
    uint64_t m = 0;
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(&m, d_tile_off + n_tiles, 8, cudaMemcpyDeviceToHost, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (m > 0xfffffffeull) return zs_bad_arg(ctx, "gunzip: too many member candidates");
    uint8_t* cand_blob = (uint8_t*)zs_scratch_get(ctx, SCR_G_CAND, (size_t)(m + 1) * 12 + 16);
    // one pass: out_off [m+1], out_len [m], in_used [m] (u64) | checks [m], status [m], first untrusted | verdict [2] (u64)
    uint8_t* pass = (uint8_t*)zs_scratch_get(ctx, SCR_G_PASS, (size_t)m * 32 + 128);
    zs_gz_member* d_mem = nullptr;
    if (max_members) d_mem = (zs_gz_member*)zs_scratch_get(ctx, SCR_G_MEMB, (size_t)m * sizeof(zs_gz_member));
    if (!cand_blob || !pass || (max_members && !d_mem)) return ZS_MEM_ERROR;
    uint64_t* d_cand = (uint64_t*)cand_blob;
    uint32_t* d_isz = (uint32_t*)(d_cand + m + 1);
    ZS_KERNEL(ctx, "gunzip_compact_kernel",
              gunzip_compact_kernel<<<n_tiles, kLocThreads, 0, ctx->stream>>>(d_in, in_len, safe_end, d_tile_off, n_tiles,
                                                                              d_cand, d_isz));
    uint64_t* d_ooff = (uint64_t*)pass;
    uint64_t* d_olen = d_ooff + m + 1;
    uint64_t* d_used = d_olen + m;
    uint32_t* d_checks = (uint32_t*)(d_used + m);
    int32_t* d_status = (int32_t*)(d_checks + m);
    uint32_t* d_bad = (uint32_t*)(d_status + m);
    uint64_t* d_res = (uint64_t*)(((uintptr_t)(d_bad + 1) + 15) & ~(uintptr_t)15);
    if (!d_out) d_out = pass;   // no room: the decoders write nothing, but want an address
    uint64_t large = kLargeMember;
    if (const char* e = getenv("ZS_GUNZIP_LARGE")) large = strtoull(e, nullptr, 10);   // A/B hook: the threshold in bytes
    std::vector<uint64_t> cand(m + 1);
    std::vector<uint32_t> isz(m + 1);
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(cand.data(), d_cand, (size_t)(m + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaMemcpyAsync(isz.data(), d_isz, (size_t)(m + 1) * 4, cudaMemcpyDeviceToHost, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));

    uint64_t pos = 0, produced = 0, n_members = 0;
    uint64_t j = 0;                       // first candidate at or after pos
    uint64_t window = ~0ull;              // members the next pass may plan
    uint64_t penalty = 0, alone_due = 0;  // members to decode alone before the next pass
    int32_t status = ZS_STREAM_END, detail = 0;
    for (;;) {
        while (j < m && cand[j] < pos) j++;
        const bool at_cand = j < m && cand[j] == pos;
        uint64_t nb = 0;
        bool tried = false;   // the pass decoded the member at pos over its planned range and could not trust it
        if (at_cand && alone_due == 0)
            while (j + nb < m && nb < window && cand[j + nb + 1] - cand[j + nb] < large) nb++;
        if (nb) {
            // 2-4. plan, decode and verify the members j .. j+nb-1
            ZS_KERNEL(ctx, "gunzip_plan_kernel", gunzip_plan_kernel<<<1, kScanThreads, 0, ctx->stream>>>(
                                                     d_isz + j, (uint32_t)nb, produced, out_cap, d_ooff, d_bad));
            int rc = zs_inflate_batch_dev(ctx, d_in, d_cand + j, (uint32_t)nb, 31, d_out, d_ooff, d_olen, d_used, d_checks,
                                          d_status, nullptr, nullptr);
            if (rc != ZS_OK) return rc;
            ZS_KERNEL(ctx, "gunzip_verify_kernel",
                      gunzip_verify_kernel<<<(unsigned)((nb + 255) / 256), 256, 0, ctx->stream>>>(
                          d_cand + j, d_isz + j, (uint32_t)nb, d_ooff, d_olen, d_used, d_checks, d_status, d_bad, d_mem));
            ZS_KERNEL(ctx, "gunzip_pass_kernel", gunzip_pass_kernel<<<1, 1, 0, ctx->stream>>>(d_bad, d_ooff, d_res));
            uint64_t h[2];
            ZS_CUDA_TRY(ctx, cudaMemcpyAsync(h, d_res, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
            ZS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
            const uint64_t u = h[0];
            if (n_members < max_members && u) {
                const uint64_t take = u < max_members - n_members ? u : max_members - n_members;
                ZS_CUDA_TRY(ctx, cudaMemcpyAsync(members + n_members, d_mem, (size_t)take * sizeof(zs_gz_member),
                                                 cudaMemcpyDeviceToHost, ctx->stream));
                ZS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
            }
            n_members += u;
            produced = h[1];
            j += u;
            pos = cand[j];
            if (u == nb) {
                if (window != ~0ull) window *= 2;
                if (pos == in_len) break;
                continue;
            }
            window = 2 * u > kMinWindow ? 2 * u : kMinWindow;   // a pass after a failed one plans twice what it took
            if (u == 0) {
                penalty = penalty ? 2 * penalty : 1;
                alone_due = penalty;
            } else {
                penalty = 0;
            }
            tried = true;
        } else if (alone_due) {
            alone_due--;
        }
        // 5. the member at pos alone, over a range of candidates: the one behind it (when the pass has not tried that) with
        // room for its planned size, then 2, 4, 8, ... candidates with all the room that is left, for as long as a try
        // stops for want of input or of the planned room (false candidates inside the member, a false ISIZE before one).
        // A Z_STREAM_END over any range is final.  Anything else is decided over the whole rest of the input with all
        // the room: one step of the reference's loop.
        InflateOneResult r;
        bool final_ = false;
        const uint64_t room = out_cap - produced;
        for (uint64_t step = tried ? 2 : 1; at_cand && j + step <= m && cand[j + step] < in_len; step *= 2) {
            const uint64_t end = cand[j + step];
            const uint64_t cap = step == 1 && isz[j + 1] < room ? isz[j + 1] : room;
            const int rc = decode_one(ctx, d_in, pos, end, d_out + produced, cap, &r);
            if (rc != ZS_OK) return rc;
            final_ = r.status == ZS_STREAM_END;
            const bool short_in = r.in_used == end - pos && r.out_len < cap;
            const bool short_room = r.out_len == cap && cap < room;
            if (final_ || r.status != ZS_BUF_ERROR || !(short_in || short_room)) break;
        }
        if (!final_) {
            const int rc = decode_one(ctx, d_in, pos, in_len, d_out + produced, room, &r);
            if (rc != ZS_OK) return rc;
        }
        if (r.status != ZS_STREAM_END) {
            status = r.status;
            detail = r.detail;
            produced += r.out_len;
            pos += r.in_used;
            break;
        }
        if (n_members < max_members) {
            zs_gz_member& e = members[n_members];
            e.in_off = pos; e.in_len = r.in_used; e.out_off = produced; e.out_len = r.out_len; e.crc32 = r.check;
        }
        n_members++;
        produced += r.out_len;
        pos += r.in_used;
        if (pos == in_len) break;
    }
    res->out_len = produced;
    res->in_used = pos;
    res->n_members = n_members;
    res->status = status;
    res->detail = detail;
    return ZS_OK;
}

}  // namespace

extern "C" {

int zs_gunzip_dev(zs_ctx* ctx, const uint8_t* d_in, uint64_t in_len, uint8_t* d_out, uint64_t out_cap, zs_gunzip_result* res,
                  zs_gz_member* members, uint64_t max_members) {
    if (!ctx) return ZS_STREAM_ERROR;
    cudaSetDevice(ctx->device);
    return gunzip_dev(ctx, d_in, in_len, d_out, out_cap, res, members, max_members);
}

int zs_gunzip(zs_ctx* ctx, const uint8_t* in, uint64_t in_len, uint8_t* out, uint64_t out_cap, zs_gunzip_result* res,
              zs_gz_member* members, uint64_t max_members) {
    if (!ctx) return ZS_STREAM_ERROR;
    cudaSetDevice(ctx->device);
    if (!res || (in_len && !in) || (out_cap && !out)) return zs_bad_arg(ctx, "gunzip: null buffer");
    uint8_t* d_in = (uint8_t*)zs_scratch_get(ctx, SCR_H_IN, in_len + 64);
    uint8_t* d_out = (uint8_t*)zs_scratch_get(ctx, SCR_H_OUT, out_cap + 64);
    if (!d_in || !d_out) return ZS_MEM_ERROR;
    if (in_len) ZS_CUDA_TRY(ctx, cudaMemcpyAsync(d_in, in, in_len, cudaMemcpyHostToDevice, ctx->stream));
    const int rc = gunzip_dev(ctx, d_in, in_len, d_out, out_cap, res, members, max_members);
    if (rc != ZS_OK) return rc;
    if (res->out_len) ZS_CUDA_TRY(ctx, cudaMemcpyAsync(out, d_out, res->out_len, cudaMemcpyDeviceToHost, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return ZS_OK;
}

}  // extern "C"
