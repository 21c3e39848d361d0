// zs_inflate.cu -- K6/K7: batch inflate of independent streams (deflate and raw deflate64).
//
// One warp per stream.  Results must be bit-exact with the reference decoder: inflate_fast
// (src/mod/inflate/inffast.ts:5), inflate_table (inftrees.ts:62), the block / header / trailer modes
// of inflate() (inflate.ts:332-1100) when called as inflate(strm, Z_FINISH) on a whole stream: same
// output bytes, same total_in / total_out, same return code and message.  (One known difference: total_in after
// a Z_BUF_ERROR for want of output room, see store_result in zs_inflate_common.cuh.)
//
// Layout: every warp owns a private decode-table arena in shared memory (852 length + 594 distance
// entries of 32 bits, the reference's ENOUGH bounds).  The run-length coded code lengths of a dynamic
// block header are read by lane 0 (a serial chain); the decode tables are built by the whole warp from the
// canonical codes (zs_inflate_common.cuh); symbol decoding is warp-uniform (every lane tracks the same bit buffer, shared
// memory table reads are broadcasts) so that back-reference copies and stored-block copies are
// executed by all 32 lanes without any hand-off.  Output goes straight to HBM; the history window
// of the reference (32/64 KiB ring) is the already written output itself plus the optional preset
// dictionary.
#include <cstdio>

#include "zs_inflate_common.cuh"

namespace {
// ceil(2^16 / d) for d = 1 .. 31 (index 0 unused): lane % d == lane - d * ((lane * c_inv16[d]) >> 16) for lane < 32
__constant__ uint32_t c_inv16[32] = {0, 65536, 32768, 21846, 16384, 13108, 10923, 9363, 8192, 7282, 6554, 5958, 5462, 5042, 4682, 4370, 4096, 3856, 3641, 3450, 3277, 3121, 2979, 2850, 2731, 2622, 2521, 2428, 2341, 2260, 2185, 2115};


using namespace zsinf;

constexpr int kWarps = 4;

__global__ void __launch_bounds__(kWarps * 32) inflate_kernel(zs_inflate_args a) {
    __shared__ WarpArena s_arena[kWarps];
    __shared__ FixedTables s_fixed;
    const unsigned lane = zs_lane();
    const unsigned wid = threadIdx.x >> 5;
    const bool d64 = a.deflate64 != 0;

    // fixedtables (inflate.ts:218-280): built once per CTA
    if (wid == 0) build_fixed_tables(s_fixed, s_arena[0], d64);
    __syncthreads();

    WarpArena& A = s_arena[wid];
    const uint64_t in_total = a.d_in_off[a.n];
    const uint64_t safe_end = (in_total + 7) & ~7ull;

    for (uint64_t sidx = (uint64_t)blockIdx.x * kWarps + wid; sidx < a.n; sidx += (uint64_t)gridDim.x * kWarps) {
        BitReader br;
        uint64_t cap, dict_len;
        const uint8_t* dict;
        open_stream(a, sidx, safe_end, br, cap, dict, dict_len);
        const uint64_t in_start = br.pos;
        uint8_t* out = a.d_out + a.d_out_off[sidx];
        uint64_t op = 0;
        int status = ZS_OK;  // ZS_OK while running
        int detail = D_NONE;
        unsigned tflags = 0;  // 1 zlib trailer, 2 gzip trailer
        uint32_t t_check = 0, t_isize = 0;

        uint64_t mark_bit = 0, mark_out = 0;   // where the last block that was begun starts
        bool skip_header = false, blocks_done = false;
        uint64_t sb = ~0ull;
        if (a.d_start_bit) sb = a.d_start_bit[sidx];   // continuation of a stream whose wrapper and earlier blocks a previous call consumed
        if (a.d_resume && a.d_resume[4 * sidx] != ~0ull) {
            // behind the segments the parallel decoder produced (zs_inflate_par.cu)
            sb = a.d_resume[4 * sidx];
            op = a.d_resume[4 * sidx + 1];
            tflags = (unsigned)(a.d_resume[4 * sidx + 2] & 3u);
            blocks_done = (a.d_resume[4 * sidx + 2] & 4u) != 0;
        }
        if (sb != ~0ull) {
            skip_header = true;
            br.pos = in_start + (sb >> 3);
            if (br.pos > br.end) br.pos = br.end;
            if (sb & 7u) {
                if (!br.need(8)) status = ZS_BUF_ERROR;
                else br.drop((unsigned)(sb & 7u));
            }
        }
        if (a.wrap && !skip_header)
            read_wrapper_header(br, a.wrap, status, detail, tflags, a.d_dict_adler && dict_len ? a.d_dict_adler + sidx : nullptr);

        if (a.d_hdr_state) {
            // header only: where the blocks start, for the segment-parallel decoder
            if (lane == 0) {
                a.d_hdr_state[5] = status == ZS_OK ? (br.pos - in_start) * 8 - br.bits : ~0ull;
                a.d_hdr_state[6] = tflags;
            }
            continue;
        }

        // ---- blocks ----
        bool last = blocks_done;
        while (status == ZS_OK && !last) {
            mark_bit = (br.pos - in_start) * 8 - br.bits;
            mark_out = op;
            if (!br.need(3)) { status = ZS_BUF_ERROR; break; }
            last = br.take(1) != 0;
            unsigned type = br.take(2);
            const uint32_t* lcode;
            const uint32_t* dcode;
            unsigned lenbits, distbits;
            if (type == 0) {
                // STORED / COPY (inflate.ts:631-672)
                br.align_byte();
                if (!br.need(32)) { status = ZS_BUF_ERROR; break; }
                unsigned w = (unsigned)br.hold;
                if ((w & 0xffffu) != ((w >> 16) ^ 0xffffu)) { status = ZS_DATA_ERROR; detail = D_STORED_LEN; break; }
                br.drop(32);
                br.unload();
                uint64_t n = w & 0xffffu, avail_in = br.end - br.pos, avail_out = cap - op;
                uint64_t c = n < avail_in ? n : avail_in;
                if (c > avail_out) c = avail_out;
                for (uint64_t j = lane; j < c; j += 32) out[op + j] = __ldg(a.d_in + br.pos + j);
                br.pos += c;
                op += c;
                if (c < n) { status = ZS_BUF_ERROR; break; }
                continue;
            } else if (type == 1) {
                lcode = s_fixed.len; dcode = s_fixed.dist; lenbits = 9; distbits = 5;
            } else if (type == 2) {
                unsigned dist_at = 0;
                lenbits = distbits = 0;
                const int rc = read_dynamic_header(br, A, d64, lenbits, distbits, dist_at);
                if (rc < 0) { status = ZS_BUF_ERROR; break; }
                if (rc > 0) { status = ZS_DATA_ERROR; detail = rc; break; }
                lcode = A.codes; dcode = A.codes + dist_at;
            } else {
                status = ZS_DATA_ERROR; detail = D_BLOCK_TYPE; break;
            }

            // LEN..MATCH / LIT (inflate.ts:840-1005, inffast.ts:31-214), one symbol per trip
            const unsigned lmask = (1u << lenbits) - 1u, dmask = (1u << distbits) - 1u;
            for (;;) {
                // ---- fast path: the role of inflate_fast (inffast.ts:5-228).  While at least 8 input bytes and
                // some output room remain, symbols are decoded without the per-symbol end-of-buffer tests;
                // anything unusual -- end of block, an invalid code, a distance beyond the dictionary, a match
                // longer than the room left --
                // is left, unconsumed, to the careful loop below, which reproduces the
                // reference's verdicts.  (deflate64: matches of up to 65538 bytes, 16 length extra bits.)
                {
                    uint64_t in_left = br.end - br.pos, out_left = cap - op;
                    uint32_t in_rem = in_left > 0xffffffffull ? 0xffffffffu : (uint32_t)in_left;
                    uint32_t out_rem = out_left > 0xffffffffull ? 0xffffffffu : (uint32_t)out_left;
                    uint8_t* wp = out + op;
                    uint32_t made = 0;     // bytes written by the fast path since `op` was last updated
                    // How far back a match may reach, in 32 bits: what has been produced (own0) plus the dictionary
                    // (back0), both capped far above the largest distance (65538).  `made` stays below 2^32 - 2^21
                    // in any stream shorter than 4 GiB; beyond that a wrapped sum sends the pair to the careful loop,
                    // which decides with 64-bit arithmetic.
                    const uint32_t own0 = op < (1u << 20) ? (uint32_t)op : (1u << 20);
                    const uint32_t back0 = own0 + (dict_len < (1u << 20) ? (uint32_t)dict_len : (1u << 20));
                    // input window: the 128 bytes from the current position, one word per lane (two coalesced
                    // loads and a funnel shift per lane when the position is not word aligned); a refill is a
                    // register shuffle.  woff = offset of the next unread byte inside the window, a multiple of 4.
                    uint64_t win_base = br.pos;
                    uint32_t woff = 0;
                    uint32_t inw = 0;
#define ZS_LOAD_WINDOW()                                                                                   \
    do {                                                                                                   \
        const uint64_t wa_ = (win_base & ~3ull) + 4ull * lane;                                             \
        const uint32_t lo_ = wa_ < br.safe_end ? __ldg(reinterpret_cast<const unsigned*>(br.base + wa_)) : 0u;          \
        const uint32_t hi_ = wa_ + 4 < br.safe_end ? __ldg(reinterpret_cast<const unsigned*>(br.base + wa_ + 4)) : 0u;  \
        inw = __funnelshift_r(lo_, hi_, 8u * (unsigned)(win_base & 3u));                                   \
    } while (0)
#define ZS_FAST_REFILL()                                                                                   \
    do {                                                                                                   \
        if (woff >= 128u) { win_base += 128; woff = 0; ZS_LOAD_WINDOW(); }                                 \
        br.hold |= (uint64_t)__shfl_sync(ZS_FULL_MASK, inw, woff >> 2) << br.bits;                         \
        br.bits += 32; woff += 4; in_rem -= 4;                                                             \
    } while (0)
                    if (in_rem >= 8u && out_rem) ZS_LOAD_WINDOW();
                    // A match of <= 32 bytes is one load and one store per lane; the store is deferred to the next
                    // match (or the end of the fast path), so the load's latency overlaps the symbols in between.
                    unsigned pend_n = 0;
                    uint8_t pend_v = 0;
                    uint8_t* pend_dp = nullptr;
                    // a symbol pulls at most 8 bytes: two refills of 32 bits
                    while (in_rem >= 8u && out_rem) {
                        if (br.bits <= 32) ZS_FAST_REFILL();
                        unsigned used;
                        uint32_t here = table_lookup<true>(lcode, lmask, br.hold, used);
                        const unsigned lop = E_OP(here);
                        if (lop == 0) {  // literal
                            br.drop(used);
                            if (lane == 0) wp[made] = (uint8_t)E_VAL(here);
                            made++; out_rem--;
                            continue;
                        }
                        if (lop & 0x60u) break;   // end of block / invalid code
                        // length + distance: <= 15 + 16 + 15 + 14 bits; the state is restored if the pair is unusual
                        const uint64_t hold0 = br.hold;
                        const unsigned bits0 = br.bits;
                        const uint64_t wb0 = win_base;
                        const uint32_t woff0 = woff;
                        unsigned xb = lop & (d64 ? 31u : 15u);
                        const unsigned len = E_VAL(here) + (((unsigned)(br.hold >> used)) & ((1u << xb) - 1u));
                        br.drop(used + xb);
                        if (br.bits <= 32) ZS_FAST_REFILL();
                        here = table_lookup<false>(dcode, dmask, br.hold, used);
                        xb = E_OP(here) & 15u;
                        const unsigned dist = E_VAL(here) + (((unsigned)(br.hold >> used)) & ((1u << xb) - 1u));
                        if ((E_OP(here) & 64u) || dist > back0 + made || len > out_rem) {
                            // invalid distance code, a distance too far back, or a match that does not fit: undo the pair
                            br.hold = hold0; br.bits = bits0;
                            win_base = wb0; woff = woff0;
                            break;
                        }
                        br.drop(used + xb);
                        // copy: the source is periodic with period dist, so every byte comes from before wp + made
                        if (pend_n) { if (lane < pend_n) pend_dp[lane] = pend_v; pend_n = 0; }
                        __syncwarp();
                        const uint8_t* sp = wp + made - dist;
                        uint8_t* dp = wp + made;
                        if (dist > own0 + made) {
                            // the match starts in the preset dictionary (inflate.ts:951-975)
                            const int64_t s0 = (int64_t)(op + made) - (int64_t)dist;
                            for (unsigned j = lane; j < len; j += 32) {
                                const int64_t si = s0 + (int64_t)(dist >= len ? j : j % dist);
                                dp[j] = si >= 0 ? out[si] : __ldg(dict + dict_len + si);
                            }
                            __syncwarp();
                        } else if (len <= 32u) {
                            // lane % dist for an overlapping copy (dist < len <= 32) without the division: dist is
                            // warp-uniform, so the reciprocal is one constant-memory read (ceil(2^16 / dist), exact for
                            // lane < 32); the generic 32-bit modulo was 9 % of this kernel's instructions
                            if (lane < len) pend_v = sp[dist >= len ? lane : lane - dist * ((lane * c_inv16[dist]) >> 16)];
                            pend_dp = dp;
                            pend_n = len;
                        } else if (dist >= len) {
                            for (unsigned j = lane; j < len; j += 32) dp[j] = sp[j];
                            __syncwarp();
                        } else {
                            for (unsigned j = lane; j < len; j += 32) dp[j] = sp[j % dist];
                            __syncwarp();
                        }
                        made += len; out_rem -= len;
                    }
                    if (pend_n) { if (lane < pend_n) pend_dp[lane] = pend_v; }
                    __syncwarp();
#undef ZS_FAST_REFILL
#undef ZS_LOAD_WINDOW
                    br.pos = win_base + woff;
                    op += made;
                }
                // ---- careful path: one symbol with every test of inflate() (also reached for the tail of a buffer)
                br.refill();
                unsigned used;
                uint32_t here = table_lookup<true>(lcode, lmask, br.hold, used);
                if (used > br.bits) { status = ZS_BUF_ERROR; break; }
                unsigned lop = E_OP(here);
                if (lop == 0) {  // literal
                    if (op >= cap) { status = ZS_BUF_ERROR; break; }
                    br.drop(used);
                    if (lane == 0) out[op] = (uint8_t)E_VAL(here);
                    op++;
                    continue;
                }
                if (lop & 32) { br.drop(used); break; }  // end of block
                if (lop & 64) { status = ZS_DATA_ERROR; detail = D_LITLEN_CODE; break; }
                // length
                unsigned xb = lop & (d64 ? 31u : 15u);
                if (used + xb > br.bits) { status = ZS_BUF_ERROR; break; }
                br.drop(used);
                unsigned len = E_VAL(here) + br.take(xb);
                // distance
                br.refill();
                here = table_lookup<false>(dcode, dmask, br.hold, used);
                if (used > br.bits) { status = ZS_BUF_ERROR; break; }
                if (E_OP(here) & 64) { status = ZS_DATA_ERROR; detail = D_DIST_CODE; break; }
                xb = E_OP(here) & 15u;
                if (used + xb > br.bits) { status = ZS_BUF_ERROR; break; }
                br.drop(used);
                uint64_t dist = E_VAL(here) + br.take(xb);
                if (op >= cap) { status = ZS_BUF_ERROR; break; }  // MATCH with left == 0 (inflate.ts:944)
                if (dist > op + dict_len) { status = ZS_DATA_ERROR; detail = D_TOO_FAR; break; }
                // copy: all lanes, periodic source so that overlapping copies need no ordering
                uint64_t c = len;
                if (c > cap - op) c = cap - op;
                __syncwarp();
                for (uint64_t j = lane; j < c; j += 32) {
                    uint64_t k = (dist >= c) ? j : (j % dist);
                    int64_t src = (int64_t)op - (int64_t)dist + (int64_t)k;
                    out[op + j] = src >= 0 ? out[src] : __ldg(dict + dict_len + src);
                }
                __syncwarp();
                op += c;
                if (c < len) { status = ZS_BUF_ERROR; break; }
            }
        }

        read_trailer(br, tflags, status, t_check, t_isize);
        if (lane == 0) {
            store_result(a, sidx, br, in_start, op, cap, status, detail, tflags, t_check, t_isize);
            if (a.d_block_mark) { a.d_block_mark[2 * sidx] = mark_bit; a.d_block_mark[2 * sidx + 1] = mark_out; }
        }
        __syncwarp();
    }
}

// Compare the checksum of the produced output with the stored trailer ("incorrect data check",
// "incorrect length check", inflate.ts:1012-1033) and publish the per-stream check value.
__global__ void inflate_verify_kernel(uint32_t n, const uint32_t* __restrict__ adler, const uint32_t* __restrict__ crc,
                                      const uint32_t* __restrict__ trailer, const uint32_t* __restrict__ flags,
                                      const uint64_t* __restrict__ out_len, uint32_t* __restrict__ checks,
                                      int32_t* __restrict__ status, int32_t* __restrict__ detail) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    unsigned f = flags[i];
    uint32_t ck = (f == 0 && crc) ? crc[i] : 0u;  // raw streams report the crc32 of what they produced
    if (f == 1) {
        ck = adler[i];
        if (ck != trailer[2 * i]) { status[i] = ZS_DATA_ERROR; detail[i] = D_DATA_CHECK; }
    } else if (f == 2) {
        ck = crc[i];
        if (ck != trailer[2 * i]) { status[i] = ZS_DATA_ERROR; detail[i] = D_DATA_CHECK; }
        else if ((uint32_t)out_len[i] != trailer[2 * i + 1]) { status[i] = ZS_DATA_ERROR; detail[i] = D_LENGTH_CHECK; }
    }
    if (checks) checks[i] = ck;
}

}  // namespace

int zs_launch_inflate_tps(zs_ctx* ctx, const zs_inflate_args& a);  // zs_inflate_tps.cu

// Batches of many streams go to the thread-per-stream kernel (32 streams per warp instruction;
// measured 29 GB/s vs 12.5 GB/s on 128 K x 4 KiB gzip records); fewer / larger streams keep a whole
// warp each (cooperative copies, big lookup tables: 21.6 vs 7.3 GB/s on 8 K x 64 KiB streams).
int zs_launch_inflate(zs_ctx* ctx, const zs_inflate_args& a, uint32_t n_choice) {
    if (a.n == 0) return ZS_OK;
    // thread per stream needs >= 32 k streams to fill the GPU (1024 warps); measured (tools/infmatrix.py):
    // 28-29 GB/s from 32768 streams up whatever the record size, 16-18 GB/s at 16384, where a warp per
    // stream gives 14 (4 KiB records) to 21 GB/s (64 KiB)
    if (!a.d_start_bit && !a.d_block_mark && a.force_tps >= 0 && (n_choice >= 32768 || (a.force_tps > 0 && a.n >= 32)))
        return zs_launch_inflate_tps(ctx, a);
    unsigned ctas = (a.n + kWarps - 1) / kWarps;
    unsigned cap = (unsigned)ctx->sm_count * 8u;
    if (ctas > cap) ctas = cap;
    ZS_KERNEL(ctx, "inflate_kernel", inflate_kernel<<<ctas, kWarps * 32, 0, ctx->stream>>>(a));
    return ZS_OK;
}

int zs_launch_inflate_verify(zs_ctx* ctx, uint32_t n, const uint32_t* d_adler, const uint32_t* d_crc,
                             const uint32_t* d_trailer, const uint32_t* d_flags, const uint64_t* d_out_len,
                             uint32_t* d_checks, int32_t* d_status, int32_t* d_detail) {
    if (n == 0) return ZS_OK;
    ZS_KERNEL(ctx, "inflate_verify_kernel", inflate_verify_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(n, d_adler, d_crc, d_trailer, d_flags, d_out_len,
                                                                    d_checks, d_status, d_detail));
    return ZS_OK;
}

extern "C" const char* zs_inflate_message(int detail) {
    static const char* const msgs[] = {
        "",
        "incorrect header check",
        "unknown compression method",
        "invalid window size",
        "unknown header flags set",
        "header crc mismatch",
        "invalid block type",
        "invalid stored block lengths",
        "too many length or distance symbols",
        "too many length",
        "invalid code lengths set",
        "invalid bit length repeat",
        "invalid code -- missing end-of-block",
        "invalid literal/lengths set",
        "invalid distances set",
        "invalid literal/length code",
        "invalid distance code",
        "invalid distance too far back",
        "incorrect data check",
        "incorrect length check",
    };
    if (detail < 0 || detail > D_LENGTH_CHECK) return "";
    return msgs[detail];
}
