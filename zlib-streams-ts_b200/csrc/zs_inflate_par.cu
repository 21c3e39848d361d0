// zs_inflate_par.cu -- segment-parallel inflate of ONE deflate stream at its flush points.
//
// The reference decodes a stream serially (inflate(), src/mod/inflate/inflate.ts:332; inflate_fast,
// inffast.ts:5); a stream written with Z_SYNC_FLUSH / Z_FULL_FLUSH points (deflate.ts:936-961 -- what this
// engine's own STITCHED + ZS_FLAG_SYNC deflate, pigz and every flushing writer produce) can be cut at the
// byte-aligned block boundaries those points leave behind.  Back-references still cross the cuts (only
// Z_FULL_FLUSH forgets the window), so a segment is decoded against an UNKNOWN 32 KiB window and its
// output is symbolic until the window is known.  Kernels, all on the context's stream, no host round trip:
//
//   par_scan_kernel     candidate cuts: the first byte position in every tile of the input that follows the
//                       marker 00 00 FF FF (the empty stored block of a flush point).  A candidate is only a
//                       guess: the pattern also occurs inside stored data and by chance.
//   par_count_kernel    a warp per candidate decodes from it WITHOUT output (lengths only) until it stands,
//                       at a block boundary, exactly on a later candidate (or ends the stream, or fails, or
//                       runs out of input).  A wrong guess decodes garbage and dies or is never reached.
//   par_plan_kernel     follows the chain from the true start of the stream: segment -> the candidate it
//                       landed on -> ...; exclusive scan of the output lengths = where every segment writes.
//   par_decode_kernel   a warp per planned segment decodes again, now writing 16-bit symbols: a byte, or
//                       256 + w for "byte w of the 32 KiB window before this segment" (copied around like
//                       any other symbol by later matches).
//   par_win*_kernel     the window after segment k is the resolved tail of its symbols: a chain over the
//                       segments, made short by composing it per group of 32 segments (par_wingroup_kernel, all
//                       groups in parallel, symbolic), linking the groups (par_winlink_kernel, the only serial
//                       step: 32 Ki elements per GROUP) and filling in every window (par_window_kernel, parallel).
//   par_resolve_kernel  symbols -> bytes, every segment with its own window, all in parallel.
//   par_finish_kernel   where the serial decoder (inflate_kernel, zs_inflate.cu) takes over: behind the last
//                       planned segment -- for the trailer and the final status only when the chain reached
//                       the end of the stream, or for whatever the parallel part could not prove (an error,
//                       truncated input, output space running out, a distance beyond the start of the
//                       stream), so that status, message and output prefix stay the reference's.
//   par_record_kernel   launched only by the index build (zs_inflate_index.cu), after a decode: the planned segments
//                       and the serial decoder's part walked again, lengths only, keeping the block starts an index
//                       of access points may use.
// The count, decode and record passes are one block walk (walk_blocks, zs_inflate_common.cuh) with three sinks:
// CountSink, SymbolSink and RecordSink.
#include <cstdio>
#include <cstring>

#include "zs_inflate_common.cuh"

namespace {

using namespace zsinf;

constexpr int kWarps = 4;
constexpr unsigned kMaxPassed = 48;         // candidates a count pass may run over before it gives up
constexpr uint64_t kMaxTiles = 64;          // ... and tiles of input it may consume
constexpr uint64_t kMaxSpan = 2u << 20;     // (but not fewer bytes than this: the tiles of a short input are small)
constexpr uint32_t kEndOfInput = 0xffffffffu;   // next_slot of a segment that ends exactly where the input ends

enum { SEG_LANDED = 0, SEG_FINAL = 1, SEG_STOPPED = 2 };   // STOPPED: error, truncated input, gave up

struct SegInfo {
    uint64_t end_bit;     // LANDED: bit position of the candidate reached; FINAL: first bit after the last block
    uint64_t out_len;
    uint32_t status;
    uint32_t next_slot;   // LANDED: slot of the candidate reached
};

struct ParArgs {
    const uint8_t* in;
    uint64_t in_len;
    uint64_t tile;            // bytes per candidate tile
    uint32_t n_slots;         // 1 + number of tiles: slot 0 is the start of the stream
    uint64_t* cand;           // [n_slots] bit position of every candidate (~0 = none)
    uint64_t* spec;           // [n_slots] speculative candidates of par_spec_kernel (~0 = none), merged into cand
    const uint64_t* marker_count;   // = &state[7] as par_scan_kernel left it
    SegInfo* seg;             // [n_slots]
    // plan
    uint32_t* plan_slot;      // [n_slots]
    uint64_t* plan_off;       // [n_slots + 1] output offset of every planned segment
    uint32_t* plan_err;       // [n_slots] set by the decode pass: the segment needs the serial decoder
    uint64_t* state;          // [8]: 0 n_planned, 1 total_out, 2 resume bit, 3 resume out, 4 blocks done, 5 body bit (in), 6 tflags (in), 7 flush-point candidates found
    uint64_t out_cap;
    uint64_t hist_len;        // bytes of preset dictionary / earlier output before the stream's first byte
    const uint8_t* hist;      // the last hist_len (<= 32768) bytes before the stream
    uint16_t* sym;            // [out_cap] symbols
    uint8_t* windows;         // [n_slots + 1][32768]
    uint16_t* gmap;           // [ceil(n_slots / kWinGroup)][32768] symbolic window maps of the segment groups
    uint8_t* out;
    uint64_t* resume;         // [4] record for inflate_kernel: start bit, start out, flags, -
};

__global__ void par_scan_kernel(ParArgs a) {
    // one warp per tile: the first marker whose following byte position lies in the tile
    const unsigned lane = zs_lane();
    const uint64_t t = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (t + 1 >= a.n_slots) return;
    const uint64_t lo = t * a.tile, hi = lo + a.tile < a.in_len ? lo + a.tile : a.in_len;
    const uint64_t body = a.state[5] == ~0ull ? ~0ull : (a.state[5] + 7) >> 3;
    uint64_t found = ~0ull;
    for (uint64_t p0 = lo; p0 < hi && found == ~0ull; p0 += 32) {
        const uint64_t p = p0 + lane;   // candidate start: bytes p-4 .. p-1 are the marker
        bool hit = false;
        if (p < hi && p >= 4 && p - 4 >= body && body != ~0ull)
            hit = a.in[p - 4] == 0 && a.in[p - 3] == 0 && a.in[p - 2] == 0xff && a.in[p - 1] == 0xff;
        const unsigned m = __ballot_sync(ZS_FULL_MASK, hit);
        if (m) found = p0 + (unsigned)(__ffs((int)m) - 1);
    }
    if (lane == 0) a.cand[t + 1] = found == ~0ull ? ~0ull : found * 8;
    if (lane == 0 && found != ~0ull) atomicAdd((unsigned long long*)&a.state[7], 1ull);   // candidates in all
    if (t == 0 && lane == 0) a.cand[0] = a.state[5];
}

// ---- speculative cuts: streams without flush points ---------------------------------------------------
// A stream written in one go (zlib.deflateSync, gzip -- the streams a DecompressionStream usually gets) has no
// markers to cut at, and one warp decodes it at 25-30 MB/s.  Its blocks still end somewhere: par_spec_kernel
// looks, in every tile that has no marker candidate, for the first BIT position at which a non-final dynamic
// block with a well-formed header begins -- HLIT/HDIST in range (inflate.ts:684-690), a complete code-length
// code, run-length coded lengths that neither over-subscribe nor overrun, complete literal/length and distance
// sets (or the reference's one-code / no-code distance sets, inftrees.ts:104-130), an end-of-block code.  Every
// lane tests its own bit position; what a random position survives is the 17-bit test (1 in 9), then the
// completeness of the code-length code (about 1 in 100 of those), then a few dozen decoded lengths before the
// running Kraft sum overflows.  A position that passes everything by chance is harmless: the count pass only
// trusts a candidate that an earlier segment LANDS on, bit exact, at a block boundary of its own decode.
__device__ __forceinline__ uint64_t peek_bits57(const uint8_t* in, uint64_t safe_end, uint64_t bitpos) {   // >= 57 bits from bitpos
    const uint64_t byte = bitpos >> 3;
    const uint64_t lo = zs_ld32(in, byte, safe_end), hi = zs_ld32(in, byte + 4, safe_end);
    return (lo | (hi << 32)) >> (bitpos & 7u);
}

__device__ bool spec_header_ok(const uint8_t* in, uint64_t in_len, uint64_t safe_end, uint64_t p) {
    if ((p >> 3) + 40 > in_len) return false;                 // too close to the end for a whole header
    const uint64_t w = peek_bits57(in, safe_end, p);
    // BFINAL = 0, BTYPE = 2, HLIT <= 29, HDIST <= 29
    if ((w & 7u) != 4u) return false;
    const unsigned hlit = (unsigned)(w >> 3) & 31u, hdist = (unsigned)(w >> 8) & 31u, hclen = (unsigned)(w >> 13) & 15u;
    if (hlit > 29u || hdist > 29u) return false;
    const unsigned ncode = hclen + 4u;
    // the code-length code: ncode 3-bit lengths, complete (inflate_table for CODES refuses anything else)
    const uint64_t c = peek_bits57(in, safe_end, p + 17);     // 57 bits = 19 lengths
    unsigned kraft = 0;
    uint8_t cl[19];
#pragma unroll
    for (int i = 0; i < 19; i++) {
        const unsigned l = i < (int)ncode ? (unsigned)(c >> (3 * i)) & 7u : 0u;
        cl[c_bl_order[i]] = (uint8_t)l;
        kraft += l ? 128u >> l : 0u;
    }
    if (kraft != 128u) return false;
    // canonical code-length code: counts, first codes, symbols sorted by (length, symbol)
    unsigned cnt[8] = {0, 0, 0, 0, 0, 0, 0, 0}, offs[8];
    for (int i = 0; i < 19; i++) cnt[cl[i]]++;
    cnt[0] = 0;
    offs[1] = 0;
    for (int l = 1; l < 7; l++) offs[l + 1] = offs[l] + cnt[l];
    uint8_t sorted[19];
    for (int i = 0; i < 19; i++)
        if (cl[i]) sorted[offs[cl[i]]++] = (uint8_t)i;
    // the run-length coded lengths (inflate.ts:729-790), judged on the fly
    BitReader br;
    br.base = in; br.end = in_len; br.safe_end = safe_end;
    const uint64_t q = p + 17 + 3ull * ncode;
    br.pos = q >> 3; br.hold = 0; br.bits = 0;
    if (!br.need(8)) return false;
    br.drop((unsigned)(q & 7u));
    const unsigned nlen = hlit + 257u, total = nlen + hdist + 1u;
    unsigned have = 0, prev = 0, kl = 0, kd = 0, nd = 0, d1 = 0, eob = 0;   // Kraft sums in units of 2^-15
    while (have < total) {
        br.refill();
        if (br.bits < 14) return false;                      // input ends inside the header
        // one symbol of the code-length code, bit by bit (<= 7 bits)
        unsigned code = 0, first = 0, index = 0, sym = 19, used = 0;
        for (unsigned l = 1; l <= 7; l++) {
            code |= (unsigned)(br.hold >> (l - 1)) & 1u;
            const unsigned n = cnt[l];
            if (code - first < n) { sym = sorted[index + (code - first)]; used = l; break; }
            index += n; first += n; first <<= 1; code <<= 1;
        }
        if (sym > 18) return false;
        br.drop(used);
        unsigned rep = 1, len = sym;
        if (sym == 16) { if (have == 0) return false; len = prev; rep = 3 + br.take(2); }
        else if (sym == 17) { len = 0; rep = 3 + br.take(3); }
        else if (sym == 18) { len = 0; rep = 11 + br.take(7); }
        if (have + rep > total) return false;
        prev = len;
        if (len) {
            const unsigned unit = 32768u >> len;
            for (unsigned r = 0; r < rep; r++) {
                const unsigned i = have + r;
                if (i < nlen) { kl += unit; if (i == 256) eob = 1; }
                else { kd += unit; nd++; d1 = len == 1; }
            }
            if (kl > 32768u || kd > 32768u) return false;     // over-subscribed
        }
        have += rep;
    }
    if (!eob || kl != 32768u) return false;                   // (a one-code literal/length set is legal and useless)
    if (!(kd == 32768u || nd == 0 || (nd == 1 && d1))) return false;
    return true;
}

// The 17-bit test -- BFINAL = 0, BTYPE = 2, HLIT <= 29, HDIST <= 29 -- for 32 consecutive bit positions at once:
// bit i of the result is position i of the window `w` (>= 45 valid bits).  1 position in 9 passes.
__device__ __forceinline__ uint32_t spec_quick_mask(uint64_t w) {
    uint64_t m = ~w & ~(w >> 1) & (w >> 2);                            // 0, 0, 1: not final, dynamic
    m &= ~((w >> 4) & (w >> 5) & (w >> 6) & (w >> 7));                 // HLIT (bits 3..7) is not 30 or 31
    m &= ~((w >> 9) & (w >> 10) & (w >> 11) & (w >> 12));              // HDIST (bits 8..12) is not 30 or 31
    return (uint32_t)m;
}
// The code-length code of the header at p is complete (Kraft sum of its HCLEN + 4 three-bit lengths = 1): what the
// 17-bit test lets through fails here 99 times in 100, so this runs before anything that needs arrays.
__device__ __forceinline__ bool spec_clcode_complete(const uint8_t* in, uint64_t safe_end, uint64_t p) {
    const unsigned ncode = ((unsigned)(peek_bits57(in, safe_end, p + 13) & 15u)) + 4u;
    uint64_t c = peek_bits57(in, safe_end, p + 17);                    // 57 bits = 19 lengths
    if (ncode < 19u) c &= (1ull << (3u * ncode)) - 1ull;
    const uint64_t weights = 0x0102040810204000ull;                    // byte l: 128 >> l (0 for an unused symbol)
    unsigned kraft = 0;
#pragma unroll
    for (int i = 0; i < 19; i++) kraft += (unsigned)(weights >> (8u * ((unsigned)(c >> (3 * i)) & 7u))) & 0xffu;
    return kraft == 128u;
}

constexpr unsigned kSpecWarpsPerTile = 4;
constexpr unsigned kSpecWarpsPerCta = 4;
constexpr unsigned kSpecQueue = 32 + 32 * 11;   // fewer than 32 waiting + at most 11 finds per lane (the pattern is 3 bits long)
__global__ void __launch_bounds__(32 * kSpecWarpsPerCta) par_spec_kernel(ParArgs a) {
    // few markers for the size of the input?  (a stream with flush points needs no guessing)
    if (a.state[5] == ~0ull || a.marker_count[0] * (256ull << 10) >= a.in_len) return;
    // Two stages, so that the expensive one runs on full warps.  Stage 1: a lane takes 32 consecutive bit positions
    // through the 17-bit test with a dozen 64-bit operations (a warp: 128 bytes of input per iteration) and queues
    // the survivors -- 1 in 9 -- in position order.  Stage 2: once 32 are waiting, each lane takes one through the
    // rest of the header test, the Kraft sum of the code-length code first.  (Run straight through with a lane per
    // position, the later stages were executed for 3 or 4 lanes in nearly every iteration: 40 ms per 420 MB of
    // input, the largest kernel of the one-stream decode of a stream without flush points; queued: 18.8 ms.)
    __shared__ uint32_t s_queue[kSpecWarpsPerCta][kSpecQueue];
    const unsigned lane = zs_lane(), wq = threadIdx.x >> 5;
    const uint64_t w = (uint64_t)blockIdx.x * kSpecWarpsPerCta + wq;
    const uint64_t t = w / kSpecWarpsPerTile, part = w % kSpecWarpsPerTile;
    if (t + 1 >= a.n_slots || a.cand[t + 1] != ~0ull) return;   // (markers were found by par_scan_kernel, which ran before)
    const uint64_t tile_bits = a.tile * 8, part_bits = tile_bits / kSpecWarpsPerTile;   // < 2^32: a tile is in_len / 6144 bytes
    uint64_t lo = t * tile_bits + part * part_bits, hi = lo + part_bits;
    const uint64_t body = a.state[5];
    if (lo <= body) lo = body + 1;                            // slot 0 is the true start
    if (a.in_len < 40) return;
    if (hi > (a.in_len - 39) * 8) hi = (a.in_len - 39) * 8;   // a whole header needs 40 bytes from the byte that holds p
    const uint64_t safe_end = (a.in_len + 7) & ~7ull;
    uint32_t* queue = s_queue[wq];
    unsigned qn = 0;                                          // queued positions (relative to lo, increasing), warp-uniform
    uint64_t found = ~0ull;
    for (uint64_t p0 = lo; p0 < hi && found == ~0ull; p0 += 1024) {
        // stage 1
        const uint64_t base = p0 + 32u * lane;
        uint32_t m = 0;
        if (base < hi) {
            m = spec_quick_mask(peek_bits57(a.in, safe_end, base));
            if (hi - base < 32) m &= (1u << (unsigned)(hi - base)) - 1u;
        }
        unsigned cnt = __popc(m), off = cnt;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned v = __shfl_up_sync(ZS_FULL_MASK, off, d);
            if ((int)lane >= d) off += v;
        }
        const unsigned total = __shfl_sync(ZS_FULL_MASK, off, 31);
        off = qn + off - cnt;
        const uint32_t rel = (uint32_t)(base - lo);
        while (m) {
            queue[off++] = rel + (unsigned)(__ffs((int)m) - 1);
            m &= m - 1u;
        }
        qn += total;
        __syncwarp();
        // stage 2
        unsigned head = 0;
        while (qn - head >= 32u) {
            const uint64_t p = lo + queue[head + lane];
            const bool ok = spec_clcode_complete(a.in, safe_end, p) && spec_header_ok(a.in, a.in_len, safe_end, p);
            const unsigned mm = __ballot_sync(ZS_FULL_MASK, ok);
            if (mm) { found = lo + queue[head + (unsigned)(__ffs((int)mm) - 1)]; break; }   // position order: the lowest lane is the first find
            head += 32u;
        }
        if (found == ~0ull && head) {   // the remainder (< 32) moves to the front
            const uint32_t rest = head + lane < qn ? queue[head + lane] : 0u;
            __syncwarp();
            queue[lane] = rest;
            qn -= head;
            __syncwarp();
        }
    }
    if (found == ~0ull && qn) {                               // what is left in the queue (< 32 positions)
        bool ok = false;
        if (lane < qn) {
            const uint64_t p = lo + queue[lane];
            ok = spec_clcode_complete(a.in, safe_end, p) && spec_header_ok(a.in, a.in_len, safe_end, p);
        }
        const unsigned mm = __ballot_sync(ZS_FULL_MASK, ok);
        if (mm) found = lo + queue[__ffs((int)mm) - 1];
    }
    if (found != ~0ull && lane == 0) atomicMin((unsigned long long*)&a.spec[t + 1], (unsigned long long)found);
}
// the speculative finds become candidates (kept apart until every part of a tile has reported its first)
__global__ void par_spec_merge_kernel(ParArgs a) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t + 1 >= a.n_slots) return;
    const uint64_t s = a.spec[t + 1];
    if (s != ~0ull && a.cand[t + 1] == ~0ull) {
        a.cand[t + 1] = s;
        atomicAdd((unsigned long long*)&a.state[7], 1ull);
    }
}

// The count pass: lengths only, until the walk stands at a block boundary exactly on a later candidate (LANDED), ends
// the stream (FINAL), or fails, runs out of input or gives up (STOPPED).
struct CountSink {
    const ParArgs& a;
    uint64_t start_bit;
    uint64_t t_seen;     // candidate slots up to here have been looked at
    unsigned passed;
    SegInfo r;           // r.out_len: the output so far
    __device__ bool at_block(uint64_t bit, bool last) {
        if (bit <= start_bit) return false;
        const uint64_t byte = bit >> 3, t = byte / a.tile + 1;
        if (last) {
            r.status = SEG_FINAL;
        } else if ((bit & 7u) == 0 && byte == a.in_len) {
            r.status = SEG_LANDED; r.next_slot = kEndOfInput;
        } else if (t < a.n_slots && a.cand[t] == bit) {   // a candidate of this tile at exactly this bit (markers are
            r.status = SEG_LANDED; r.next_slot = (uint32_t)t;   // byte aligned, speculative cuts are not)
        }
        if (r.status != SEG_STOPPED) { r.end_bit = bit; return true; }
        // A wrong guess decodes garbage until it fails; bound what it may cost: candidates run over without standing
        // on one, and input consumed.  (A true segment that long is left to the serial decoder, together with what
        // follows it.)
        while (t_seen < t && t_seen + 1 < a.n_slots) {
            ++t_seen;
            const uint64_t c = a.cand[t_seen];
            if (c != ~0ull && c < bit) ++passed;
        }
        return passed > kMaxPassed || byte - (start_bit >> 3) > (kMaxTiles * a.tile > kMaxSpan ? kMaxTiles * a.tile : kMaxSpan);
    }
    __device__ bool full() const { return false; }
    __device__ int stored(uint64_t, uint64_t n) { r.out_len += n; return r.out_len > a.out_cap; }
    __device__ void literal(unsigned) { r.out_len++; }
    __device__ int match(unsigned len, uint64_t) { r.out_len += len; return r.out_len > a.out_cap; }
};

// The decode pass: 16-bit symbols to `sym` until the walk reaches stop_bit (the candidate the count pass landed on) or
// ends the stream.  A reference to byte w of the 32 KiB window before the segment is the symbol 256 + w.
struct SymbolSink {
    const ParArgs& a;
    uint16_t* sym;
    uint64_t stop_bit;
    uint64_t avail_hist;   // bytes of stream, dictionary or earlier output before the segment
    uint64_t op;
    __device__ bool at_block(uint64_t bit, bool last) { return bit >= stop_bit || last; }
    __device__ bool full() const { return false; }
    __device__ int stored(uint64_t pos, uint64_t n) {
        for (uint64_t j = zs_lane(); j < n; j += 32) sym[op + j] = a.in[pos + j];
        op += n;
        return 0;
    }
    __device__ void literal(unsigned byte) {
        if (zs_lane() == 0) sym[op] = (uint16_t)byte;
        op++;
    }
    __device__ int match(unsigned len, uint64_t dist) {
        // a distance that reaches before the start of the stream (and its dictionary) is the reference's "invalid
        // distance too far back": left to the serial decoder
        if (dist > op + avail_hist) return 1;
        __syncwarp();
        const int64_t s0 = (int64_t)op - (int64_t)dist;
        for (unsigned j = zs_lane(); j < len; j += 32) {
            const int64_t si = s0 + (int64_t)(dist >= len ? j : j % dist);
            sym[op + j] = si >= 0 ? sym[si] : (uint16_t)(256 + kWin + si);
        }
        __syncwarp();
        op += len;
        return 0;
    }
};

// Where the index build's pass appends the block starts it keeps: (bit, output offset) pairs at rec[2i], rec[2i + 1],
// i taken from cnt[0]; cnt[1] counts the walks that reached their end.
struct RecordOut {
    uint64_t* rec;
    uint64_t cap;        // pairs
    unsigned long long* cnt;
    uint64_t span;
};

// The index build's pass (zs_inflate_index.cu): lengths only, from a walk's start to stop_bit or the end of the last
// block.  It keeps the first block start and every later one that some multiple of the span falls on -- one whose output
// offset o has a multiple of the span in (o of the block start before it, o].  A block start the access-point rule
// selects is always kept, whichever walk it falls in.
struct RecordSink {
    const RecordOut& out;
    uint64_t stop_bit;
    uint64_t o;          // output offset in the stream
    uint64_t prev;       // o of the block start before this one (none yet: ~0)
    bool landed;         // the walk reached its end (a flag, not the walk's result: that cost a move per symbol here)
    __device__ bool at_block(uint64_t bit, bool last) {
        if (bit >= stop_bit || last) { landed = true; return true; }
        if (prev == ~0ull || o / out.span > prev / out.span) {
            if (zs_lane() == 0) {
                const unsigned long long i = atomicAdd(out.cnt, 1ull);
                if (i < out.cap) { out.rec[2 * i] = bit; out.rec[2 * i + 1] = o; }
            }
        }
        prev = o;
        return false;
    }
    __device__ bool full() const { return false; }
    __device__ int stored(uint64_t, uint64_t n) { o += n; return 0; }
    __device__ void literal(unsigned) { o++; }
    __device__ int match(unsigned len, uint64_t) { o += len; return 0; }
};

__global__ void __launch_bounds__(kWarps * 32) par_count_kernel(ParArgs a) {
    __shared__ WarpArena s_arena[kWarps];
    __shared__ FixedTables s_fixed;
    const unsigned wid = threadIdx.x >> 5;
    if (wid == 0) build_fixed_tables(s_fixed, s_arena[0], false);
    __syncthreads();
    for (uint64_t slot = (uint64_t)blockIdx.x * kWarps + wid; slot < a.n_slots; slot += (uint64_t)gridDim.x * kWarps) {
        const uint64_t start = a.cand[slot];
        // No flush point anywhere (a stream written in one go): nothing to cut.  The count pass from the start of
        // the stream would run through the whole input serially only for the serial decoder to do it again
        // (measured on an 8 MiB C zlib stream through the stream API: 0.5 s of count passes, 0.44 s of decode pass).
        if (start == ~0ull || a.state[7] == 0) {
            if (zs_lane() == 0) { SegInfo r; r.end_bit = 0; r.out_len = 0; r.status = SEG_STOPPED; r.next_slot = 0; a.seg[slot] = r; }
            continue;
        }
        CountSink cs{a, start, (start >> 3) / a.tile + 1, 0, {0, 0, SEG_STOPPED, 0}};
        walk_blocks_at(a.in, a.in_len, start, s_arena[wid], s_fixed, cs);
        if (zs_lane() == 0) a.seg[slot] = cs.r;
        __syncwarp();
    }
}

__global__ void par_plan_kernel(ParArgs a) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    uint64_t off = 0, n = 0;
    uint32_t cur = 0;
    uint64_t resume_bit = a.cand[0], done = 0;
    if (resume_bit != ~0ull) {
        for (;;) {
            const SegInfo s = a.seg[cur];
            if (s.status == SEG_STOPPED) break;
            if (off + s.out_len > a.out_cap) break;          // the serial decoder reports the overflow
            a.plan_slot[n] = cur;
            a.plan_off[n] = off;
            a.plan_err[n] = 0;
            n++;
            off += s.out_len;
            resume_bit = s.end_bit;
            if (s.status == SEG_FINAL) { done = 1; break; }
            if (s.next_slot == kEndOfInput) break;            // more input may follow: the serial decoder says so
            cur = s.next_slot;
        }
    }
    a.plan_off[n] = off;
    a.state[0] = n;
    a.state[1] = off;
    a.state[2] = resume_bit;
    a.state[3] = off;
    a.state[4] = done;
}

__global__ void __launch_bounds__(kWarps * 32) par_decode_kernel(ParArgs a) {
    __shared__ WarpArena s_arena[kWarps];
    __shared__ FixedTables s_fixed;
    const unsigned wid = threadIdx.x >> 5;
    if (wid == 0) build_fixed_tables(s_fixed, s_arena[0], false);
    __syncthreads();
    const uint64_t n = a.state[0];
    for (uint64_t k = (uint64_t)blockIdx.x * kWarps + wid; k < n; k += (uint64_t)gridDim.x * kWarps) {
        const uint32_t slot = a.plan_slot[k];
        const SegInfo s = a.seg[slot];
        const uint64_t off = a.plan_off[k];
        SymbolSink ss{a, a.sym + off, s.end_bit, off + a.hist_len, 0};
        // a walk that does not reach the end the count pass reached: cannot happen, but never trust it
        if (walk_blocks_at(a.in, a.in_len, a.cand[slot], s_arena[wid], s_fixed, ss) != 0) a.plan_err[k] = 1u;
        __syncwarp();
    }
}

// windows[k] = the 32 KiB before planned segment k, right aligned (bytes that do not exist read as 0 and are
// never referenced: the decode pass refused such distances).
//
// The window after segment k is the resolved tail of its symbols -- a chain over the segments, 32 Ki elements per
// link.  One CTA walking all of it was the largest item of a long stream (6.5 us per segment: 29 ms of the 70 ms
// of a 256 MiB stream with 4400 segments).  The chain is a composition of maps ("element j of the next window is a
// literal, or element w of the current one"), and maps compose: the segments are taken in groups of kWinGroup,
//   par_wingroup_kernel  every group, in parallel: the window after its last segment as a SYMBOLIC map of the
//                        window before its first (16-bit entries: a byte, or 256 + index into that window);
//   par_winlink_kernel   one CTA: the window before every group, by applying the groups' maps in order
//                        (n / kWinGroup links instead of n);
//   par_window_kernel    every group, in parallel: the concrete windows of its segments from its first one.
constexpr unsigned kWinGroup = 32;
constexpr int kWinPer = kWin / 1024;   // elements per thread

// element j of the window after a segment of `len` symbols at `sym`: symbol j + len - 32768, or -- where the segment
// is shorter than the window -- element j + len of the window before it (returned as 0x10000 + index).  All loads of
// a thread are issued before the first is used: the chain is latency bound.
__device__ __forceinline__ void window_tail(const uint16_t* sym, uint64_t len, unsigned tid, unsigned (&s)[kWinPer]) {
#pragma unroll
    for (int u = 0; u < kWinPer; u++) {
        const unsigned j = tid + 1024u * u;
        const int64_t t = (int64_t)j + (int64_t)len - (int64_t)kWin;
        s[u] = t >= 0 ? (unsigned)__ldcs(sym + t) : 0x10000u + (unsigned)(j + len);
    }
}

__global__ void __launch_bounds__(1024) par_wingroup_kernel(ParArgs a) {
    extern __shared__ __align__(16) uint8_t s_win_raw[];
    uint16_t (*s_map)[kWin] = reinterpret_cast<uint16_t (*)[kWin]>(s_win_raw);
    const unsigned tid = threadIdx.x;
    const uint64_t n = a.state[0];
    const uint64_t k0 = (uint64_t)blockIdx.x * kWinGroup, k1 = k0 + kWinGroup < n ? k0 + kWinGroup : n;
    if (k0 >= n) return;
    for (unsigned j = tid; j < kWin; j += 1024) s_map[0][j] = (uint16_t)(256u + j);   // the identity: the window before the group
    __syncthreads();
    unsigned cur = 0;
    for (uint64_t k = k0; k < k1; k++) {
        const uint64_t off = a.plan_off[k], len = a.plan_off[k + 1] - off;
        unsigned s[kWinPer];
        window_tail(a.sym + off, len, tid, s);
#pragma unroll
        for (int u = 0; u < kWinPer; u++) {
            const unsigned v = s[u];
            s_map[cur ^ 1][tid + 1024u * u] = v < 256 ? (uint16_t)v : v < 0x10000u ? s_map[cur][v - 256] : s_map[cur][v - 0x10000u];
        }
        __syncthreads();
        cur ^= 1;
    }
    uint16_t* g = a.gmap + (uint64_t)blockIdx.x * kWin;
    for (unsigned j = tid; j < kWin; j += 1024) g[j] = s_map[cur][j];
}

__global__ void __launch_bounds__(1024) par_winlink_kernel(ParArgs a) {
    extern __shared__ __align__(16) uint8_t s_win_raw[];
    uint8_t (*s_win)[kWin] = reinterpret_cast<uint8_t (*)[kWin]>(s_win_raw);
    const unsigned tid = threadIdx.x;
    const uint64_t n = a.state[0];
    for (unsigned j = tid; j < kWin; j += 1024) {
        const uint64_t pad = kWin - a.hist_len;   // hist_len <= 32768
        const uint8_t v = j >= pad ? a.hist[j - pad] : 0;
        s_win[0][j] = v;
        a.windows[j] = v;
    }
    __syncthreads();
    unsigned cur = 0;
    const uint64_t ng = (n + kWinGroup - 1) / kWinGroup;
    for (uint64_t g = 0; g + 1 < ng; g++) {   // the window before group g + 1
        const uint16_t* m = a.gmap + g * kWin;
        uint8_t* next = a.windows + (g + 1) * kWinGroup * (uint64_t)kWin;
        unsigned v[kWinPer];
#pragma unroll
        for (int u = 0; u < kWinPer; u++) v[u] = __ldcs(m + tid + 1024u * u);
#pragma unroll
        for (int u = 0; u < kWinPer; u++) {
            const unsigned j = tid + 1024u * u;
            const uint8_t b = v[u] < 256 ? (uint8_t)v[u] : s_win[cur][v[u] - 256];
            s_win[cur ^ 1][j] = b;
            next[j] = b;
        }
        __syncthreads();
        cur ^= 1;
    }
}

__global__ void __launch_bounds__(1024) par_window_kernel(ParArgs a) {
    extern __shared__ __align__(16) uint8_t s_win_raw[];
    uint8_t (*s_win)[kWin] = reinterpret_cast<uint8_t (*)[kWin]>(s_win_raw);
    const unsigned tid = threadIdx.x;
    const uint64_t n = a.state[0];
    const uint64_t k0 = (uint64_t)blockIdx.x * kWinGroup, k1 = k0 + kWinGroup < n ? k0 + kWinGroup : n;
    if (k0 >= n) return;
    {
        const uint8_t* w0 = a.windows + k0 * (uint64_t)kWin;
        for (unsigned j = tid; j < kWin; j += 1024) s_win[0][j] = w0[j];
    }
    __syncthreads();
    unsigned cur = 0;
    for (uint64_t k = k0; k < k1; k++) {
        const uint64_t off = a.plan_off[k], len = a.plan_off[k + 1] - off;
        uint8_t* next = a.windows + (k + 1) * (uint64_t)kWin;
        unsigned s[kWinPer];
        window_tail(a.sym + off, len, tid, s);
#pragma unroll
        for (int u = 0; u < kWinPer; u++) {
            const unsigned j = tid + 1024u * u;
            const unsigned v = s[u];
            const uint8_t b = v < 256 ? (uint8_t)v : v < 0x10000u ? s_win[cur][v - 256] : s_win[cur][v - 0x10000u];
            s_win[cur ^ 1][j] = b;
            next[j] = b;
        }
        __syncthreads();
        cur ^= 1;
    }
}

__global__ void __launch_bounds__(256) par_resolve_kernel(ParArgs a) {
    const uint64_t n = a.state[0];
    for (uint64_t k = blockIdx.x; k < n; k += gridDim.x) {
        const uint64_t off = a.plan_off[k], len = a.plan_off[k + 1] - off;
        const uint8_t* win = a.windows + k * (uint64_t)kWin;
        const uint16_t* sym = a.sym + off;
        uint8_t* out = a.out + off;
        for (uint64_t i = threadIdx.x; i < len; i += blockDim.x) {
            const unsigned s = sym[i];
            out[i] = s < 256 ? (uint8_t)s : win[s - 256];
        }
    }
}

__global__ void par_finish_kernel(ParArgs a) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const uint64_t n = a.state[0];
    uint64_t bit = a.state[2], out = a.state[3], done = a.state[4];
    for (uint64_t k = 0; k < n; k++) {
        if (a.plan_err[k]) {   // everything from this segment on is the serial decoder's
            bit = a.cand[a.plan_slot[k]];
            out = a.plan_off[k];
            done = 0;
            break;
        }
    }
    if (a.cand[0] == ~0ull) {
        // the wrapper header did not parse: the serial decoder starts over and reports it
        a.resume[0] = ~0ull; a.resume[1] = 0; a.resume[2] = 0;
    } else {
        a.resume[0] = bit; a.resume[1] = out; a.resume[2] = (a.state[6] & 3u) | (done ? 4u : 0u);
    }
}

// The index build's pass (zs_inflate_index.cu).  Warp item 0 walks what the serial decoder decoded: from bit tail[0]
// (~0: the first block, behind the wrapper header) with tail[1] bytes before it -- nothing when tail[2] & 4 says the
// planned segments reached the last block.  Items 1..n are the planned segments of the decode that ran before.  The
// walk goes first: it is the longest item whenever the parallel part gave up early.
__global__ void __launch_bounds__(kWarps * 32) par_record_kernel(ParArgs a, RecordOut ro, const uint64_t* tail, int wrap) {
    __shared__ WarpArena s_arena[kWarps];
    __shared__ FixedTables s_fixed;
    const unsigned wid = threadIdx.x >> 5;
    if (wid == 0) build_fixed_tables(s_fixed, s_arena[0], false);
    __syncthreads();
    const uint64_t n = a.state ? a.state[0] : 0;
    for (uint64_t k = (uint64_t)blockIdx.x * kWarps + wid; k <= n; k += (uint64_t)gridDim.x * kWarps) {
        uint64_t bit, stop = ~0ull, out;
        if (k == 0) {
            if (tail[2] & 4u) {
                if (zs_lane() == 0) atomicAdd(ro.cnt + 1, 1ull);
                continue;
            }
            bit = tail[0]; out = tail[1];
            if (bit == ~0ull) {
                BitReader br;
                br.open(a.in, 0, a.in_len, (a.in_len + 7) & ~7ull);
                int status = ZS_OK, detail = D_NONE;
                unsigned tflags = 0;
                // (a zlib header with FDICT reports Z_NEED_DICT here: the stream decoded with its dictionary already)
                if (wrap) read_wrapper_header(br, wrap, status, detail, tflags, nullptr);
                bit = br.pos * 8 - br.bits;
                out = 0;
            }
        } else {
            const uint32_t slot = a.plan_slot[k - 1];
            bit = a.cand[slot]; stop = a.seg[slot].end_bit; out = a.plan_off[k - 1];
        }
        RecordSink rs{ro, stop, out, ~0ull, false};
        walk_blocks_at(a.in, a.in_len, bit, s_arena[wid], s_fixed, rs);
        if (rs.landed && zs_lane() == 0) atomicAdd(ro.cnt + 1, 1ull);
        __syncwarp();
    }
}

// The decoder's view of its scratch for one stream of in_len bytes and out_cap bytes of output room.  The same sizes
// give the same buffers, so a later call finds there what the decode left.
int par_args(zs_ctx* ctx, const uint8_t* d_in, uint64_t in_len, uint64_t out_cap, uint64_t* d_state, ParArgs& p, unsigned& n_groups) {
    p.in = d_in; p.in_len = in_len;
    // At most 6144 candidates (1.3 waves of warps); for shorter inputs the tiles shrink to 8 KiB so that every flush
    // point of a stream cut every 64 KiB is a candidate: what an attempt costs is the slowest warp, and a warp that
    // has to run over a flush point that is not the first of its tile decodes two or three segments, one after the
    // other (measured through the stream API: 29 ms per pass with 32 KiB tiles; one segment is ~8 ms).
    uint64_t tile = in_len / 6144;
    if (tile < (8u << 10)) tile = 8u << 10;
    tile = (tile + 31) & ~31ull;
    p.tile = tile;
    const uint64_t n_tiles = (in_len + tile - 1) / tile;
    p.n_slots = (uint32_t)(n_tiles + 1);
    p.cand = (uint64_t*)zs_scratch_get(ctx, SCR_P_CAND, (size_t)p.n_slots * 16);   // candidates, then the speculative finds
    p.spec = p.cand ? p.cand + p.n_slots : nullptr;
    p.marker_count = d_state + 7;
    p.seg = (SegInfo*)zs_scratch_get(ctx, SCR_P_SEG, (size_t)p.n_slots * sizeof(SegInfo));
    uint8_t* plan = (uint8_t*)zs_scratch_get(ctx, SCR_P_PLAN, (size_t)p.n_slots * 16 + 64);
    p.sym = (uint16_t*)zs_scratch_get(ctx, SCR_P_SYM, (size_t)out_cap * 2 + 64);
    p.windows = (uint8_t*)zs_scratch_get(ctx, SCR_P_WIN, ((size_t)p.n_slots + 1) * kWin);
    n_groups = (p.n_slots + kWinGroup - 1) / kWinGroup;
    p.gmap = (uint16_t*)zs_scratch_get(ctx, SCR_P_GMAP, (size_t)n_groups * kWin * 2);
    if (!p.cand || !p.seg || !plan || !p.sym || !p.windows || !p.gmap) return ZS_MEM_ERROR;
    p.plan_off = (uint64_t*)plan;                                   // [n_slots + 1]
    p.plan_slot = (uint32_t*)(plan + ((size_t)p.n_slots + 1) * 8);  // [n_slots]
    p.plan_err = p.plan_slot + p.n_slots;                           // [n_slots]  (16 bytes per slot + 8 in all)
    p.state = d_state;
    p.out_cap = out_cap;
    p.hist_len = 0; p.hist = nullptr; p.out = nullptr; p.resume = nullptr;
    return ZS_OK;
}

}  // namespace

// One stream, wrapper header already located: a.d_resume receives where inflate_kernel continues.
int zs_launch_inflate_parallel(zs_ctx* ctx, const uint8_t* d_in, uint64_t in_len, uint8_t* d_out, uint64_t out_cap,
                               const uint8_t* d_hist, uint64_t hist_len, uint64_t* d_state, uint64_t* d_resume) {
    ParArgs p;
    unsigned n_groups = 0;
    const int rc = par_args(ctx, d_in, in_len, out_cap, d_state, p, n_groups);
    if (rc != ZS_OK) return rc;
    p.hist_len = hist_len > kWin ? kWin : hist_len;
    p.hist = d_hist + (hist_len > kWin ? hist_len - kWin : 0);
    p.out = d_out;
    p.resume = d_resume;
    const unsigned sms = (unsigned)ctx->sm_count;
    ZS_CUDA_TRY(ctx, cudaMemsetAsync(d_state + 7, 0, 8, ctx->stream));   // candidate counter
    {
        const unsigned warps = p.n_slots - 1;
        if (warps) ZS_KERNEL(ctx, "par_scan_kernel", par_scan_kernel<<<(warps + 7) / 8, 256, 0, ctx->stream>>>(p));
        else ZS_KERNEL(ctx, "par_scan_kernel", par_scan_kernel<<<1, 32, 0, ctx->stream>>>(p));
    }
    if (p.n_slots > 1 && !getenv("ZS_INFLATE_NO_SPEC")) {
        ZS_CUDA_TRY(ctx, cudaMemsetAsync(p.spec, 0xff, (size_t)p.n_slots * 8, ctx->stream));
        const uint64_t warps = (uint64_t)(p.n_slots - 1) * kSpecWarpsPerTile;
        ZS_KERNEL(ctx, "par_spec_kernel",
                  par_spec_kernel<<<(unsigned)((warps + kSpecWarpsPerCta - 1) / kSpecWarpsPerCta), 32 * kSpecWarpsPerCta, 0, ctx->stream>>>(p));
        ZS_KERNEL(ctx, "par_spec_merge_kernel", par_spec_merge_kernel<<<(p.n_slots + 255) / 256, 256, 0, ctx->stream>>>(p));
    }
    unsigned ctas = (p.n_slots + kWarps - 1) / kWarps;
    if (ctas > sms * 8u) ctas = sms * 8u;
    ZS_KERNEL(ctx, "par_count_kernel", par_count_kernel<<<ctas, kWarps * 32, 0, ctx->stream>>>(p));
    ZS_KERNEL(ctx, "par_plan_kernel", par_plan_kernel<<<1, 32, 0, ctx->stream>>>(p));
    ZS_KERNEL(ctx, "par_decode_kernel", par_decode_kernel<<<ctas, kWarps * 32, 0, ctx->stream>>>(p));
    static bool attr_set[64] = {false};
    const int dev_slot = ctx->device >= 0 && ctx->device < 64 ? ctx->device : 0;
    if (!attr_set[dev_slot] || ctx->device >= 64) {
        ZS_CUDA_TRY(ctx, cudaFuncSetAttribute(par_wingroup_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * (int)kWin));
        ZS_CUDA_TRY(ctx, cudaFuncSetAttribute(par_winlink_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * (int)kWin));
        ZS_CUDA_TRY(ctx, cudaFuncSetAttribute(par_window_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * (int)kWin));
        attr_set[dev_slot] = true;
    }
    ZS_KERNEL(ctx, "par_wingroup_kernel", par_wingroup_kernel<<<n_groups, 1024, 4 * kWin, ctx->stream>>>(p));
    ZS_KERNEL(ctx, "par_winlink_kernel", par_winlink_kernel<<<1, 1024, 2 * kWin, ctx->stream>>>(p));
    ZS_KERNEL(ctx, "par_window_kernel", par_window_kernel<<<n_groups, 1024, 2 * kWin, ctx->stream>>>(p));
    ZS_KERNEL(ctx, "par_resolve_kernel", par_resolve_kernel<<<sms * 8u, 256, 0, ctx->stream>>>(p));
    ZS_KERNEL(ctx, "par_finish_kernel", par_finish_kernel<<<1, 32, 0, ctx->stream>>>(p));
    return ZS_OK;
}

// The index build's record pass (par_record_kernel) over one stream that zs_inflate_stream_dev decoded just before
// with the same in_len and out_cap.  planned: that decode took the segment-parallel path, whose plan is still in its
// scratch and whose state (SCR_P_STATE) is d_state; otherwise the whole stream is walked from its wrapper header.
// d_tail: the walk's start record (see par_record_kernel); d_cnt[2] zeroed by the caller.
int zs_launch_inflate_record(zs_ctx* ctx, const uint8_t* d_in, uint64_t in_len, uint64_t out_cap, bool planned, uint64_t* d_state,
                             const uint64_t* d_tail, int wrap, uint64_t span, uint64_t* d_rec, uint64_t rec_cap,
                             unsigned long long* d_cnt) {
    ParArgs p;
    memset(&p, 0, sizeof(p));
    unsigned ctas = 1;
    if (planned) {
        unsigned n_groups = 0;
        const int rc = par_args(ctx, d_in, in_len, out_cap, d_state, p, n_groups);
        if (rc != ZS_OK) return rc;
        ctas = (p.n_slots + 1 + kWarps - 1) / kWarps;
        if (ctas > (unsigned)ctx->sm_count * 8u) ctas = (unsigned)ctx->sm_count * 8u;
    } else {
        p.in = d_in; p.in_len = in_len; p.tile = 1; p.out_cap = ~0ull;
    }
    RecordOut ro;
    ro.rec = d_rec; ro.cap = rec_cap; ro.cnt = d_cnt; ro.span = span;
    ZS_KERNEL(ctx, "par_record_kernel", par_record_kernel<<<ctas, kWarps * 32, 0, ctx->stream>>>(p, ro, d_tail, wrap));
    return ZS_OK;
}
