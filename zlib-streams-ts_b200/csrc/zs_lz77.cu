// zs_lz77.cu -- K1/K2: LZ77 match finding (greedy levels 1-3, lazy levels 4-9) and parse for
// independent or dictionary-primed chunks.  (K3, the symbol histogram, is histogram_kernel in
// zs_huff.cu.)
//
// Replaces, for whole chunks, the reference's per-byte loop: INSERT_STRING / hash chains
// (src/mod/deflate/deflate.ts:109-141), longest_match (:1053-1115), deflate_fast (:1281-1350),
// deflate_slow incl. the TOO_FAR rule (:1352-1448), _tr_tally_lit/_tr_tally_dist
// (src/mod/deflate/utils.ts:55-81), with CONFIGURATION_TABLE (deflate.ts:86-103) giving
// max_chain / nice_length / max_lazy per level.  The bit stream differs from the reference's (the
// north star allows it); what must hold is: the symbols decode to the input, and the compressed
// size stays within 3 % of the reference at the same level (tests/test_deflate_gpu.py).
//
// Work decomposition (B200: 148 SMs, 227 KB shared memory per CTA):
//   * one persistent CTA (1024 threads) per SM pulls *segments* (runs of consecutive chunks) from
//     an atomic counter.  Everything the per-byte loop touches lives in shared memory: a 64 KiB
//     ring of the window (staged from HBM once: the first look-ahead of a segment with 16-byte
//     loads, every step after that by the copy engine -- 1-D cp.async.bulk on an mbarrier), the
//     hash-chain tables prev[32768] (16-bit hop distances to the previous position with the same
//     hash; the reference stores positions) and head[16384] (one bit less than
//     the reference's hash so that 30 wide warps fit; measured cost: +0.8 % size at level 6), and
//     ~60 KB of rings between the pipeline stages.  Tables and ring are carried from chunk to chunk
//     inside a segment, so dictionary priming costs one 32 KiB insert-only pass per segment.
//   * inside the CTA the serial loop of the reference becomes a 7-stage software pipeline over
//     960-position steps, one __syncthreads per step.  Thirty "wide" warps do everything that is
//     independent per position; two "thin" warps do only the two inherently ordered updates (a
//     single warp retires roughly one dependent instruction per 15-25 cycles when 32 warps are
//     resident, so every instruction moved off the thin warps counts):
//        prep    (wide) : hash 32 positions, find equal hashes inside the batch with ballots
//                         (nearest lower peer / last of its group);
//        insert  (thin) : head[] exchange in position order -- read the old head, publish the
//                         batch's last position of every hash;
//        link    (wide) : turn old head / in-batch peer into the prev[] link of every position;
//        search  (wide) : one lane per position walks that position's chain (<= max_chain
//                         candidates, compares in the shared-memory ring, 16-bit ring indices);
//                         every position is searched speculatively, which is what makes the
//                         chain walk 960-wide.  Greedy levels: compares stop at nice_length inside
//                         the loop, the winners are extended together behind it; each greedy level
//                         has its own kernel, and level 1's walk is four straight-line rounds.  Lazy levels: the
//                         batch walks in lock step with a straggler stop, and a candidate is first
//                         tested on the four bytes that end at index best_len;
//        resolve (wide) : greedy / lazy rule per position, 5 rounds of pointer doubling per batch
//                         (for every possible entry lane: visited positions, exit, symbol count),
//                         then two adjacent batches are composed into one 64-position hop (lazy
//                         levels: resolve and emit pairs are claimed from a counter by the warps
//                         that are done searching);
//        parse   (thin) : chains the 64-position hops, one shared-memory load each (entry of the
//                         next hop = exit of this one), counts symbols, cuts blocks every <= 16383
//                         symbols (lit_bufsize - 1, deflate.ts:323,336);
//        emit    (wide) : writes the packed symbols of every batch at the index the parse gave it.
//     The link stage runs at most 2 steps ahead of a searcher, so restricting matches to
//     32768 - 2*960 bytes keeps every prev[] slot a searcher reads stable: no races, and the output
//     does not depend on scheduling (tables are reset per segment).
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "zs_common.cuh"

namespace {

#ifndef ZS_SEARCH_WARPS
#define ZS_SEARCH_WARPS 30
#endif
#ifndef ZS_HASH_BITS
#define ZS_HASH_BITS 14
#endif
#ifndef ZS_LZ_PREV_POS   // prev[] holds hop distances (chain_hop); -DZS_LZ_PREV_POS: positions, as in the reference
#define ZS_LZ_PREV_DELTA 1
#endif
constexpr int kSearchWarps = ZS_SEARCH_WARPS;
// The two thin roles get the highest warp ids: the SMSP arbiter favours high warp ids and these
// short critical-path warps must never wait behind the wide warps.
constexpr int kWarpParse = kSearchWarps;
constexpr int kWarpInsert = kSearchWarps + 1;
constexpr int kThreads = 32 * (kSearchWarps + 2);
constexpr int kStep = 32 * kSearchWarps;               // positions per pipeline step
constexpr unsigned kMaxDist = 32768u - 2u * kStep;      // see header comment
constexpr unsigned kNoPrev = 0xffffu;                   // ZS_LZ_PREV_DELTA: prev[] entry of a position without predecessor
constexpr unsigned kSymLimit = 16383u;                  // symbols per block, deflate.ts:336
constexpr unsigned kTooFar = 4096u;                     // deflate/constants.ts (TOO_FAR)
constexpr unsigned kHashBits = ZS_HASH_BITS;
constexpr unsigned kRing = 65536;      // window ring: position p lives at ring[p & 0xffff]
constexpr unsigned kRingGuard = 288;   // ring[kRing + i] mirrors ring[i] so that 8-byte reads never wrap
// position-indexed rings between the stages (power-of-two sizes: cheap indexing)
constexpr unsigned pow2_at_least(unsigned v) { unsigned r = 1; while (r < v) r <<= 1; return r; }
constexpr unsigned kResRing = pow2_at_least(4 * kStep + 64);  // written by search, read by resolve and (three steps later) emit
constexpr unsigned kMjRing = pow2_at_least(3 * kStep + 64);   // written by resolve, read by parse (one step later) and emit (two)
constexpr unsigned kPbRing = pow2_at_least(2 * kSearchWarps + 4);
constexpr unsigned kMaxSegChunks = 256;  // chunks per segment (boundary table in shared memory)  // per pair of batches (entry offset, first symbol index): parse -> emit

struct LevelCfg { int lazy_fn, good, lazy, nice, chain; };
// CONFIGURATION_TABLE, deflate.ts:86-103
constexpr LevelCfg kLevels[10] = {
    {0, 0, 0, 0, 0},      {0, 4, 4, 8, 4},      {0, 4, 5, 16, 8},      {0, 4, 6, 32, 32},
    {1, 4, 4, 16, 16},    {1, 8, 16, 32, 32},   {1, 8, 16, 128, 128},  {1, 8, 32, 128, 256},
    {1, 32, 128, 258, 1024}, {1, 32, 258, 258, 4096}};
// A row of the table as a compile-time constant in device code (kernels specialised for one level)
__host__ __device__ constexpr LevelCfg level_cfg(int level) { return kLevels[level]; }

// prep word: hash | nearest lower peer lane << 16 | has peer << 21 | last of its group << 22 | valid << 23
constexpr uint32_t PREP_HAS_PRED = 1u << 21, PREP_LAST = 1u << 22, PREP_VALID = 1u << 23;

struct Smem {
    uint8_t ring[kRing + kRingGuard];
    uint16_t head[1 << kHashBits];
    uint16_t prev[32768];
    uint32_t prep[3 * kStep];  // prep -> insert (next step) -> link (the step after): 3 buffers
    uint16_t oldh[2 * kStep];  // insert -> link: head[] value seen by each position, double buffered
    uint2 pb[kPbRing];         // parse -> emit, per aligned pair of batches: (entry offset or 64 = nothing to emit, index of its first symbol)
    uint32_t res[kResRing];    // stage 3 -> 4,5: dist (15) | match len << 15 (9, 0 = none) | literal << 24
    uint2 mj[kMjRing];         // resolve -> parse, emit: (visited mask, packed exits/counts, see resolve) for a parse entering at this lane
    uint32_t bnd[kMaxSegChunks + 1];  // chunk boundaries of the segment, as range offsets (bnd[0] = first data position)
    uint32_t seg;              // segment being processed
    uint32_t claim[2];         // lazy levels: resolve / emit pairs claimed in this iteration (and the next one's counter, being reset)
    alignas(8) uint64_t stage_bar;   // mbarrier the bulk copies of the window staging complete on
};
static_assert(sizeof(Smem) <= 227 * 1024, "shared memory budget");

struct LzArgs {
    const uint8_t* buf;        // 16-byte aligned; position 0 of all indices below
    uint64_t org;              // index of the call's first input byte (d_in[0]) inside buf
    uint64_t valid_lo;         // first readable index (org - history)
    uint64_t data_end;         // one past the last input byte
    const uint64_t* in_off;    // [n_chunks+1] relative to org
    uint32_t n_chunks, seg_chunks, n_seg, max_bpc;
    uint32_t n_big, seg_small;   // segments [0, n_big) hold seg_chunks chunks, the later ones seg_small (see zs_launch_lz77)
    LevelCfg cfg;              // kLevels[level] (kernels specialised for one level use their own compile-time copy)
    int strategy;              // ZS_STRATEGY_* (FILTERED and RLE act here)
    int cross;                 // 1: matches may reach before the chunk start (PRIME / STITCHED)
    uint32_t* sym;
    uint32_t* chunk_nblk;
    uint32_t* blk_desc;
    uint32_t* seg_counter;
    unsigned stop_after, stop_active;   // lazy levels: straggler stop of the chain walk (search_lazy_endwin)
    // lz77_dict_kernel only (every segment is one chunk, see DictImage): the prepared dictionary's saved
    // tables (nullptr: build them -- the call's one chunk is the dictionary), where a build writes them,
    // and the dictionary's length (<= 32 KiB)
    const uint8_t* dict_img;
    uint8_t* dict_save;
    uint32_t dict_len;
};

// The tables of a prepared dictionary (zs_deflate_dict), as lz77_dict_kernel leaves them after running the
// dictionary alone through prep / insert / link with range offset q = ring index (the dictionary's first
// byte at q = 0): head[] and prev[] as they lie in shared memory, then ring[0, 32 KiB) and its guard mirror.
// Every position whose three hash bytes lie inside the dictionary is inserted; the last two are not (their
// hash needs the chunk's first two bytes: deflateSetDictionary leaves s->insert = 2, deflate.ts:367-424).
constexpr unsigned kImgTables = (1u << kHashBits) * 2u + 32768u * 2u;   // head[] + prev[]
constexpr unsigned kImgRing = kImgTables;                               // ring[0, 32768)
constexpr unsigned kImgGuard = kImgRing + 32768u;                       // ring[kRing, kRing + kRingGuard)
constexpr unsigned kImgBytes = kImgGuard + kRingGuard;

#ifdef ZS_LZ_PROF
// cycle counters: [0] thin insert, [1] thin parse, [2] wide warps (summed), [3] whole step incl.
// barrier (warp 0), [4] steps, [5] slowest wide warp of each step (summed)
__device__ unsigned long long g_prof[16];
#define PROF_T(i) if (lane == 0) atomicAdd(&g_prof[i], (unsigned long long)(clock64() - t_begin))
#else
#define PROF_T(i)
#endif

__device__ __forceinline__ unsigned res_slot(uint32_t q) { return q & (kResRing - 1u); }
__device__ __forceinline__ unsigned mj_slot(uint32_t q) { return q & (kMjRing - 1u); }

// ---- window staging -------------------------------------------------------------------------------
// The match finder reads the window byte-granular and at random (one candidate per lane), which
// through L1 costs one 128-byte line per lane per load and saturates the L1 wavefront queue.  The
// window is therefore staged once, coalesced (16 bytes per lane), into a 64 KiB shared-memory ring
// that always holds the last 32 KiB plus the look-ahead; all compares are shared-memory loads.
__device__ __forceinline__ uint32_t win32(const Smem& S, uint64_t pos) {
    const unsigned idx = (unsigned)pos & (kRing - 1u);
    const unsigned al = idx & ~3u;
    const uint32_t lo = *reinterpret_cast<const uint32_t*>(S.ring + al);
    const uint32_t hi = *reinterpret_cast<const uint32_t*>(S.ring + al + 4);
    return __funnelshift_r(lo, hi, (idx & 3u) * 8u);
}

// Copy input [from, to) (absolute indices, multiples of 16) into the ring; `tid`/`nthr` describe
// the cooperating threads.  Bytes past the end of the input are staged as zeros.
__device__ __forceinline__ void stage_window(Smem& S, const LzArgs& a, uint64_t from, uint64_t to, unsigned tid, unsigned nthr) {
    const uint64_t safe16 = (a.data_end + 15) & ~15ull;
    for (uint64_t pos = from + 16ull * tid; pos < to; pos += 16ull * nthr) {
        uint4 v = make_uint4(0, 0, 0, 0);
        if (pos < safe16) v = __ldg(reinterpret_cast<const uint4*>(a.buf + pos));
        const unsigned idx = (unsigned)pos & (kRing - 1u);
        *reinterpret_cast<uint4*>(S.ring + idx) = v;
        if (idx < kRingGuard) *reinterpret_cast<uint4*>(S.ring + kRing + idx) = v;
    }
}

// Dictionary kernel: the 16 bytes of range offsets [ql, ql + 16) that come from the input, byte q at absolute
// index g0 + q (g0 = the chunk's first absolute index - its range offset, negative for a chunk near the start
// of the buffer).  The chunk starts at any byte, so the ring line is assembled from five aligned words;
// words before index 0 or at / past safe16 (the input's end rounded up to 16) read as zeros.
__device__ __forceinline__ uint4 dict_src_line(const LzArgs& a, int64_t g0, int64_t safe16, uint32_t ql) {
    const int64_t g = g0 + (int64_t)ql;
    const int64_t al = g - (g & 3);
    const unsigned sh = (unsigned)(g & 3) * 8u;
    uint32_t w[5];
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        const int64_t at = al + 4 * k;
        w[k] = (at >= 0 && at < safe16) ? __ldg(reinterpret_cast<const uint32_t*>(a.buf + at)) : 0u;
    }
    return make_uint4(__funnelshift_r(w[0], w[1], sh), __funnelshift_r(w[1], w[2], sh), __funnelshift_r(w[2], w[3], sh),
                      __funnelshift_r(w[3], w[4], sh));
}

// ---- bulk-async staging (Blackwell: the copy engine moves the window, no thread does) ------------
// Steady state: one elected lane of the thin insert warp arms an mbarrier with the byte count and issues
// 1-D cp.async.bulk copies global -> shared (UBLKCP in SASS): the step's ~1 KiB of look-ahead goes into
// the ring without a single LDG/STS on the CTA's critical warp, whose loads used to sit in registers
// across the thirty head exchanges.  The warp waits for the barrier's phase just before the step
// barrier, which publishes the bytes to the wide warps.
#ifndef ZS_LZ_NO_BULK
#define ZS_LZ_BULK 1
#endif
__device__ __forceinline__ unsigned smem_addr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "ZS_MBAR_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra ZS_MBAR_DONE;\n"
        "bra ZS_MBAR_WAIT;\n"
        "ZS_MBAR_DONE:\n"
        "}\n" ::"r"(smem_addr(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_addr(dst)),
                 "l"(src), "r"(bytes), "r"(smem_addr(bar))
                 : "memory");
}
// Issue the copies for input [from, to) (multiples of 16, to - from < kRing, to <= the readable end): the part up to
// the ring's wrap, the part after it, and the mirror of ring[0, kRingGuard) behind the ring.  One thread calls
// this; returns the bytes the barrier has to expect.
__device__ __forceinline__ unsigned bulk_stage(Smem& S, const uint8_t* buf, uint64_t from, uint64_t to) {
    unsigned total = 0;
    while (from < to) {
        const unsigned idx = (unsigned)from & (kRing - 1u);
        unsigned nb = (unsigned)(to - from);
        if (idx + nb > kRing) nb = kRing - idx;
#ifdef ZS_DEBUG_HOOKS   // compute-sanitizer is closed on the pool: the copy engine's targets are checked here
        if (idx + nb > kRing || (nb & 15u) || (idx & 15u) || ((uintptr_t)(buf + from) & 15u)) { printf("[lz77 bulk] bad copy idx %u nb %u\n", idx, nb); __trap(); }
#endif
        bulk_g2s(S.ring + idx, buf + from, nb, &S.stage_bar);
        total += nb;
        if (idx < kRingGuard) {
            const unsigned g = idx + nb < kRingGuard ? nb : kRingGuard - idx;
#ifdef ZS_DEBUG_HOOKS
            if (idx + g > kRingGuard || (g & 15u)) { printf("[lz77 bulk] bad guard copy idx %u g %u\n", idx, g); __trap(); }
#endif
            bulk_g2s(S.ring + kRing + idx, buf + from, g, &S.stage_bar);
            total += g;
        }
        from += nb;
    }
    return total;
}

__device__ __forceinline__ unsigned hash3(uint32_t w) { return ((w & 0xffffffu) * 0x9E3779B1u) >> (32 - kHashBits); }

// Per-range constants, all 32-bit: stages address positions by their offset q inside the range.
// A range is one whole segment: the <= 32 KiB dictionary before its first chunk (inserted only)
// followed by its chunks, back to back.  Chunk boundaries only matter to the search (matches stop
// at the end of their chunk and, without priming, do not reach before its start) and to the parse
// (blocks and symbol counts are per chunk).
struct RangeCtx {
    uint32_t cb;     // low 32 bits of the range's first absolute position: ring index = (cb + q) & 0xffff
    uint32_t n;      // bytes in the range
    uint32_t pre;    // bytes before the range that may be matched, capped at kMaxDist
    uint32_t tail;   // bytes readable from the range start to the end of the input (saturating)
    uint32_t q_data; // first position that is compressed (everything before is dictionary)
    uint32_t nc;     // chunks in the segment
    int cross;       // matches may reach before the chunk start
    unsigned min_len;  // shortest match worth emitting: 3, or 6 with Z_FILTERED at the lazy levels (deflate.ts:1381-1387)
    uint32_t ins_lo;   // dictionary kernel: first position prep inserts
};

// ---- stage 1: prep (wide) -----------------------------------------------------------------------
// 32 consecutive positions starting at offset q0; positions >= limit (end of the step being inserted)
// or without three readable bytes are not inserted.
template <bool kDict = false>
__device__ __forceinline__ uint32_t prep_batch(const Smem& S, const RangeCtx& c, uint32_t q0, uint32_t limit) {
    const unsigned lane = zs_lane();
    const uint32_t q = q0 + lane;
    // (dictionary kernel: the positions below ins_lo are in the restored tables already)
    const bool valid = q < limit && q + 2 < c.tail && (!kDict || q >= c.ins_lo);
    unsigned h = 0;
    if (valid) h = hash3(win32(S, c.cb + q));
    // lanes with the same hash: kHashBits independent ballots (measured faster than one MATCH.ANY,
    // which iterates over the distinct values: 9.2 k vs 9.7 k cycles per step)
#ifndef ZS_PREP_MATCH_ANY
    unsigned peers = __ballot_sync(ZS_FULL_MASK, valid);
#pragma unroll
    for (int bit = 0; bit < (int)kHashBits; ++bit) {
        const bool one = (h >> bit) & 1u;
        const unsigned bal = __ballot_sync(ZS_FULL_MASK, one);
        peers &= one ? bal : ~bal;
    }
#else
    const unsigned peers = __match_any_sync(ZS_FULL_MASK, valid ? h : 0x10000u + lane);
#endif
    if (!valid) return 0u;
    const unsigned lower = peers & zs_lanemask_lt();
    uint32_t w = h | PREP_VALID;
    if (lower) w |= PREP_HAS_PRED | ((31u - __clz(lower)) << 16);
    if ((peers >> lane) == 1u) w |= PREP_LAST;
    return w;
}

// ---- stage 2: insert (thin) + link (wide) -----------------------------------------------------------
// Chains are kept in position order: the predecessor of p is the nearest earlier position with the
// same hash -- inside the batch (from prep) or head[h]; "none" is encoded as a self link.
// Only the head[] accesses are ordered (read the old head, then publish the batch's last position of
// every hash); that is all the thin warp does.  Turning the old head into the prev[] link is
// independent per position and is done by the wide warps one step later.
// The link reads the old head only for a valid position without an in-batch peer, so every lane loads it
// unconditionally (an invalid prep word reads head[0]): per batch that leaves one load of the prep word, the
// head[] load and store, the oldh[] store and the value p + lane.
__device__ __forceinline__ void head_exchange(Smem& S, uint32_t p, uint32_t w, uint16_t* oldh) {
    const unsigned h = w & ((1u << kHashBits) - 1u);
    const uint16_t old = S.head[h];
    if (w & PREP_LAST) S.head[h] = (uint16_t)p;
    oldh[zs_lane()] = old;
    __syncwarp();  // orders this batch's head[] stores before the next batch's loads
}
__device__ __forceinline__ void link_batch(Smem& S, const RangeCtx& c, uint32_t q0, uint32_t w, unsigned old) {
    if (w & PREP_VALID) {
        const uint32_t q = q0 + zs_lane();
        const unsigned p16 = (c.cb + q) & 0xffffu;
#ifdef ZS_LZ_PREV_DELTA
        unsigned hop = kNoPrev;
        if (w & PREP_HAS_PRED) {
            hop = zs_lane() - ((w >> 16) & 31u);
        } else {
            const unsigned delta = (p16 - old) & 0xffffu;
            if (delta != 0 && delta <= kMaxDist && delta <= q + c.pre) hop = delta;
        }
        S.prev[p16 & 32767u] = (uint16_t)hop;
#else
        unsigned pred = p16;
        if (w & PREP_HAS_PRED) {
            pred = (c.cb + q0 + ((w >> 16) & 31u)) & 0xffffu;
        } else {
            const unsigned delta = (p16 - old) & 0xffffu;
            if (delta != 0 && delta <= kMaxDist && delta <= q + c.pre) pred = (p16 - delta) & 0xffffu;
        }
        S.prev[p16 & 32767u] = (uint16_t)pred;
#endif
    }
}

// One hop along the hash chain: from ring index ci to its predecessor, `dist` = distance from the searching position.
// Returns false when the chain ends (no predecessor, or further back than max_back).
#ifdef ZS_LZ_PREV_DELTA
// prev[] holds the hop itself (0xffff = none: no distance survives adding it), so a hop is one load, one add, one test
// (positions as in the reference cost a subtraction, a mask and a second test per candidate: level 1 -2.6 %, level 6
// -4.1 % kernel time on text).
__device__ __forceinline__ bool chain_hop(const Smem& S, unsigned& ci, unsigned& dist, unsigned max_back, unsigned& delta) {
    delta = S.prev[ci & 32767u];
    dist += delta;
    if (dist > max_back) return false;
    ci = (ci - delta) & (kRing - 1u);
    return true;
}
#else
__device__ __forceinline__ bool chain_hop(const Smem& S, unsigned& ci, unsigned& dist, unsigned max_back, unsigned& delta) {
    delta = (ci - S.prev[ci & 32767u]) & 0xffffu;
    if (delta == 0) return false;
    dist += delta;
    if (dist > max_back) return false;
    ci = (ci - delta) & (kRing - 1u);
    return true;
}
#endif

// ---- stage 3: search (wide), one lane per position -----------------------------------------------
// All arithmetic is on 16-bit ring indices and 32-bit distances (the ring is a multiple of the
// 32 KiB prev[] period, so prev[] is indexed by the ring index too).
__device__ __forceinline__ uint32_t ring32(const Smem& S, unsigned idx) {
    idx &= kRing - 1u;
    const unsigned al = idx & ~3u;
    const uint32_t lo = *reinterpret_cast<const uint32_t*>(S.ring + al);
    const uint32_t hi = *reinterpret_cast<const uint32_t*>(S.ring + al + 4);
    return __funnelshift_r(lo, hi, (idx & 3u) * 8u);
}
__device__ __forceinline__ unsigned first_diff_byte(uint32_t x) { return (unsigned)(__ffs((int)x) - 1) >> 3; }

__device__ __forceinline__ uint2 ring64(const Smem& S, unsigned idx) {
    idx &= kRing - 1u;
    const unsigned al = idx & ~3u, sh = (idx & 3u) * 8u;   // al + 11 < kRing + kRingGuard
    const uint32_t w0 = *reinterpret_cast<const uint32_t*>(S.ring + al);
    const uint32_t w1 = *reinterpret_cast<const uint32_t*>(S.ring + al + 4);
    const uint32_t w2 = *reinterpret_cast<const uint32_t*>(S.ring + al + 8);
    return make_uint2(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh));
}
// Bytes [0, len) of the candidate at ring index ci and of the position at pi are equal: compare on from there, eight
// bytes per round (the two streams keep their own word alignment, the last word loaded is carried into the next
// round: 2 + 2 loads per 8 bytes), until a difference or max_len.  The result is not capped at max_len.
__device__ __forceinline__ unsigned extend_match(const Smem& S, unsigned ci, unsigned pi, unsigned len, unsigned max_len) {
    unsigned aa = ((ci + len) & (kRing - 1u)) & ~3u, ab = ((pi + len) & (kRing - 1u)) & ~3u;   // the guard mirrors 288 bytes
    const unsigned sa = ((ci + len) & 3u) * 8u, sb = ((pi + len) & 3u) * 8u;
    uint32_t a0 = *reinterpret_cast<const uint32_t*>(S.ring + aa);
    uint32_t b0 = *reinterpret_cast<const uint32_t*>(S.ring + ab);
    while (len < max_len) {
        const uint32_t a1 = *reinterpret_cast<const uint32_t*>(S.ring + aa + 4);
        const uint32_t a2 = *reinterpret_cast<const uint32_t*>(S.ring + aa + 8);
        const uint32_t b1 = *reinterpret_cast<const uint32_t*>(S.ring + ab + 4);
        const uint32_t b2 = *reinterpret_cast<const uint32_t*>(S.ring + ab + 8);
        const uint32_t yl = __funnelshift_r(a0, a1, sa) ^ __funnelshift_r(b0, b1, sb);
        const uint32_t yh = __funnelshift_r(a1, a2, sa) ^ __funnelshift_r(b1, b2, sb);
        if (yl | yh) return len + (yl ? first_diff_byte(yl) : 4u + first_diff_byte(yh));
        a0 = a2; b0 = b2;
        aa += 8; ab += 8;
        len += 8;
    }
    return len;
}
// Length of the match between the candidate at ring index ci and the position at pi (first eight bytes of the
// position in pw0/pw1), not capped at max_len (the caller clamps); compares stop at max_len rounded up to 8.
__device__ __forceinline__ unsigned match_length(const Smem& S, unsigned ci, unsigned pi, uint32_t pw0, uint32_t pw1, unsigned max_len) {
    const uint2 cw = ring64(S, ci);
    const uint32_t x0 = cw.x ^ pw0, x1 = cw.y ^ pw1;
    if (x0) return first_diff_byte(x0);
    if (x1) return 4u + first_diff_byte(x1);
    return extend_match(S, ci, pi, 8u, max_len);
}

// [cs, ce) is the chunk that holds q.
// kMode: 0 greedy levels (1-3), 2 Z_RLE.  (The lazy levels 4-9 use search_lazy_endwin below.)
// kLevel: 0 = cfg is read at run time, 1-3 = cfg is the compile-time row kLevels[kLevel].
// Work bounds of the lazy levels on periodic data: a chain is "dense" when the hop to the candidate is at most
// kDenseHop positions -- runs and short periods, not ordinary text or DNA-like data, whose ties and good
// matches must not cut the search short (measured: +5.8 % size on a 4-letter alphabet at level 6 when they did).
constexpr unsigned kDenseHop = 8;       // hops this short mark a run / a short period
constexpr int kInteriorChain = 16;      // candidates left once a good match turns out to lie inside a longer one
template <int kMode, int kLevel>
__device__ __forceinline__ uint32_t search_position(const Smem& S, const LevelCfg& cfg, const RangeCtx& c, uint32_t q,
                                                    uint32_t cs, uint32_t ce) {
    static_assert(kMode == 0 || kMode == 2, "levels 4-9 go through search_lazy_endwin");
    const uint32_t room = ce - q;
    const unsigned max_len = room < 258u ? room : 258u;
    const unsigned pi = (c.cb + q) & (kRing - 1u);
    const uint2 pw = ring64(S, pi);
    const uint32_t pw0 = pw.x, pw1 = pw.y;
    const uint32_t lit = (pw0 & 0xffu) << 24;
    if (max_len < 3) return lit;
    if (kMode == 2) {
        // deflate_rle (deflate.ts:1450-1523): the only candidate is the previous byte; the match is the
        // rest of the run it starts
        const uint32_t back = c.cross ? q + c.pre : q - cs;
        if (back == 0) return lit;
        const uint32_t pat = (uint32_t)S.ring[(pi - 1u) & (kRing - 1u)] * 0x01010101u;
        unsigned len = 0;
        while (len < max_len) {
            const uint32_t x = ring32(S, pi + len) ^ pat;
            if (x) { len += first_diff_byte(x); break; }
            len += 4;
        }
        if (len > max_len) len = max_len;
        return len >= 3 ? (lit | (len << 15) | 1u) : lit;
    }
    const unsigned nice = (unsigned)cfg.nice < max_len ? (unsigned)cfg.nice : max_len;
    const uint32_t back = c.cross ? q + c.pre : q - cs;
    const unsigned max_back = back < kMaxDist ? back : kMaxDist;
    unsigned best_len = 2, best_dist = 0, best_ci = pi;
    unsigned ci = pi, dist = 0;
    if constexpr (kLevel != 0 && level_cfg(kLevel).nice <= 8) {
        // Level 1 (chain 4, nice 8): the whole walk fits in the first eight bytes, so it runs as max_chain
        // straight-line rounds, each one hop and one 8-byte compare per lane that is still walking, with no
        // branch for the compiler to stop at: the hop of round r+1 is issued together with the window loads of
        // round r.  There is no collision test: a candidate that differs in its first three bytes has a length
        // below 3 and cannot beat best_len = 2.  A lane stops at the chain's end or once it holds a match of nice.
        // (At level 1 the loop below costs about 10 warp instructions per input byte at 17 of 32 lanes active:
        // profiles/lz77_r2b_l1_summary.md.)
        bool alive = true;
        unsigned delta = S.prev[ci & 32767u];
#pragma unroll
        for (int round = 0; round < level_cfg(kLevel).chain; ++round) {
            dist += delta;
            alive = alive && dist <= max_back;
            ci = (ci - delta) & (kRing - 1u);
            // a lane that is done reads at its own position (consecutive across the batch: no extra bank
            // conflicts) instead of branching around the loads
            const unsigned li = alive ? ci : pi;
            const uint2 cw = ring64(S, li);
            if (round + 1 < level_cfg(kLevel).chain) delta = S.prev[li & 32767u];
            const uint32_t x0 = cw.x ^ pw0, x1 = cw.y ^ pw1;
            // bytes equal from the start: trailing zero bits of the 64-bit xor / 8, without a branch
            // ((x - 1) & ~x has the trailing zeros of x as ones: 32 of them for x = 0, so 8 bytes for equal words)
            const uint32_t xw = x0 ? x0 : x1;
            unsigned len = ((x0 ? 0u : 32u) + __popc((xw - 1u) & ~xw)) >> 3;
            if (len > max_len) len = max_len;
            if (alive && len > best_len) {
                best_len = len;
                best_dist = dist;
                best_ci = ci;
            }
            alive = alive && len < nice;
        }
    } else
    for (int chain = cfg.chain; chain > 0; --chain) {
        unsigned delta;
        if (!chain_hop(S, ci, dist, max_back, delta)) break;
        uint32_t x = ring32(S, ci) ^ pw0;
        if ((x & 0xffffffu) != 0) continue;  // hash collision
        unsigned len;
        if (x) {
            len = 3;
        } else {
            x = ring32(S, ci + 4) ^ pw1;
            if (x) {
                len = 4 + first_diff_byte(x);
            } else {
                // Eight bytes match.  Inside the chain loop the compare goes on as far as nice_length only (not at
                // all at level 1, nice_length 8): a match that long ends the search whatever its full length, and
                // the full length is found after the loop, where the lanes that hold such a match extend them
                // together -- in the loop that path ran for 1.7 of 32 lanes, up to max_chain times per batch
                // (mixed corpus, level 1: 25.5 -> 22.1 ms per 512 MiB).
                len = 8;
                if (nice > 8u) len = extend_match(S, ci, pi, 8u, nice);
            }
        }
        if (len > max_len) len = max_len;
        if (len > best_len) {
            best_len = len;
            best_dist = dist;
            if (len >= nice) { best_ci = ci; break; }
        }
    }
    if (best_len >= nice) {   // bytes [0, nice) are equal: whole 8-byte rounds from there
        best_len = extend_match(S, best_ci, pi, nice & ~7u, max_len);
        if (best_len > max_len) best_len = max_len;
    }
    if (best_len < c.min_len) return lit;
    // A 3-byte match far back costs more bits than three literals (a distance code plus up to 13 extra
    // bits).  deflate_fast has no such rule, but it seldom finds these matches, because it leaves the inside
    // of every match longer than max_insert out of its hash chains (deflate.ts:1310-1322); this search
    // inserts every position and finds them all: JSON-like rows came out 4.1 % / 2.8 % larger than the
    // reference's at levels 1 / 2.  With deflate_slow's TOO_FAR rule (deflate.ts:1381-1387) applied to the
    // greedy levels too they are 3.5 % / 4.8 % smaller, text 2.9 % / 4.2 % smaller, and no data kind of
    // tools/ratiocheck.py is more than 0.04 % larger (modelled with tools/lzmodel.py -- too_far=4096, then
    // measured: profiles/ab_lz_r2.txt).
    if (best_len == 3 && best_dist > kTooFar) return lit;
    return lit | (best_len << 15) | best_dist;
}

// The lazy levels' chain walk is warp-synchronous with a straggler stop.  All 32 lanes of the batch run the
// candidate loop in lock step; once at least `stop.after` candidates have been visited and at most
// `stop.active` lanes are still walking, the batch stops and those lanes keep the best match they have.  A
// lone long chain otherwise holds up its warp and, through the step barrier, the whole CTA.  Modelled first
// (tools/lzmodel.c, `stop_active=K stop_after=M`), then measured (profiles/ab_straggler_r2.txt): mixed corpus
// level 9 5.3 -> 12.9 GB/s, level 6 11.3 -> 13.5 GB/s, text level 6 11.0 -> 13.1 GB/s for +0.4 % size on text
// (worst of eight data kinds: +1.65 % against zlib).  The vote is taken on well defined per-lane state, so the
// result does not depend on scheduling.
struct StopCfg { unsigned after, active; };

// ---- the lazy levels' search: end-window filter in front of the compare ------------------------------
// What the warp pays for is not the candidates a lane visits but the code paths any lane takes: with one
// candidate per lane and iteration, the deep compare used to run in nearly every iteration for the two or
// three lanes whose candidate got past the 3-byte test (ncu, level 6: a third of the kernel's instructions
// at 1.5-6 of 32 lanes).  A candidate can only beat the match in hand if it agrees with the position on
// the four bytes that END at index best_len -- longest_match's scan_end test (deflate.ts:1063-1081) widened
// to a word -- so that window is compared FIRST: one unaligned word of the ring per candidate, and only
// candidates that can improve the match reach the compare.  The compare itself starts with one 8-byte
// round (three aligned words of the ring against the position's first eight bytes in registers).
// Lazy levels (4-9): the lock-step candidate loop with the filter in front of the compare.  The two
// rules that look at candidates which do not improve the match -- "eight bytes match but the byte at best_len
// does not" and "ties with the best match", both on dense chains only -- are now decided on the filtered-out
// candidate's first eight bytes: it agrees with the position on min(best_len, 8) bytes (for best_len < 8 that
// is exactly a tie, since the window said the byte at best_len differs).
__device__ __forceinline__ uint32_t search_lazy_endwin(const Smem& S, const LevelCfg& cfg, const StopCfg stop, const RangeCtx& c,
                                                       uint32_t q, uint32_t cs, uint32_t ce, bool live) {
    const uint32_t room = live ? ce - q : 0u;
    const unsigned max_len = room < 258u ? room : 258u;
    const unsigned pi = (c.cb + q) & (kRing - 1u);
    uint2 pw = make_uint2(0, 0);
    if (live) pw = ring64(S, pi);
    const uint32_t lit = (pw.x & 0xffu) << 24;
    const unsigned nice = (unsigned)cfg.nice < max_len ? (unsigned)cfg.nice : max_len;
    const uint32_t back = c.cross ? q + c.pre : q - cs;
    const unsigned max_back = back < kMaxDist ? back : kMaxDist;
    unsigned best_len = 2, best_dist = 0;
    unsigned ci = pi, dist = 0;
    unsigned woff = 0;
    uint32_t wown = pw.x, wmask = 0xffffffu;
    int chain = (live && max_len >= 3) ? cfg.chain : 0;
    for (unsigned it = 0;; ++it) {
        const unsigned walking = __ballot_sync(ZS_FULL_MASK, chain > 0);
        if (walking == 0) break;
        if (it >= stop.after && (unsigned)__popc(walking) <= stop.active) break;
        if (chain > 0) {
            do {   // one candidate; `break` = next candidate, chain = 0 = this lane is done
                unsigned delta;
                if (!chain_hop(S, ci, dist, max_back, delta)) { chain = 0; break; }
                if ((ring32(S, ci + woff) ^ wown) & wmask) {
                    if (delta <= kDenseHop && best_len >= 3) {   // a run or a short period: is this a tie / an 8-byte match?
                        const uint2 cw = ring64(S, ci);
                        const uint32_t x0 = cw.x ^ pw.x, x1 = cw.y ^ pw.y;
                        const unsigned m = x0 ? first_diff_byte(x0) : x1 ? 4u + first_diff_byte(x1) : 8u;
                        if (m >= (best_len < 8u ? best_len : 8u)) chain -= chain >> 2;
                    }
                    break;
                }
                unsigned len = match_length(S, ci, pi, pw.x, pw.y, max_len);
                if (len > max_len) len = max_len;
                if (len > best_len) {
                    // With a good match in hand the rest of the chain gets a quarter of the budget (the rule longest_match
                    // applies when the previous position's match was good, deflate.ts:1069-1071) -- here only where the
                    // reference would not be searching at all: on a dense chain (a run) or when the match also extends
                    // backwards, i.e. q lies inside a longer match that started earlier (deflate_slow skips the bytes a
                    // match covers; the speculative search cannot, but it stops after kInteriorChain more candidates).
                    if (best_len < (unsigned)cfg.good && len >= (unsigned)cfg.good) {
                        const bool interior = S.ring[(ci - 1u) & (kRing - 1u)] == S.ring[(pi - 1u) & (kRing - 1u)];
                        if (interior || delta <= kDenseHop) chain >>= 2;
                        if (interior && chain > kInteriorChain) chain = kInteriorChain;
                    }
                    best_len = len;
                    best_dist = dist;
                    if (len >= nice) { chain = 0; break; }
                    woff = len - 3u; wmask = 0xffffffffu;
                    wown = ring32(S, pi + woff);
                } else if (len == best_len && delta <= kDenseHop) {
                    chain -= chain >> 2;   // only with best_len == max_len's neighbours: a tie that passed the window
                }
            } while (0);
            --chain;
        }
    }
    if (best_len < c.min_len) return lit;
    if (best_len == 3 && best_dist > kTooFar) return lit;   // deflate.ts:1381-1387
    return lit | (best_len << 15) | best_dist;
}

// ---- stage 4: resolve (wide) -----------------------------------------------------------------------
// mj[].y layout: exit (9 bits) | is_match << 9 | popc(visited) << 10 (6 bits) | pair exit - 32 << 16
// (9 bits) | pair symbol count << 25 (7 bits).  The pair fields are valid for the first batch of an
// aligned pair of batches: a parse entering the pair at this lane leaves it at "pair exit"
// (relative to the pair's first position) after emitting "pair symbol count" symbols.
constexpr unsigned MJ_MATCH = 1u << 9;
__device__ __forceinline__ unsigned mj_exit(unsigned y) { return y & 0x1ffu; }
__device__ __forceinline__ unsigned mj_count(unsigned y) { return (y >> 10) & 0x3fu; }
__device__ __forceinline__ unsigned mj_pair_exit(unsigned y) { return ((y >> 16) & 0x1ffu) + 32u; }
__device__ __forceinline__ unsigned mj_pair_count(unsigned y) { return y >> 25; }

// One batch of 32 positions starting at q0: greedy / lazy rule per position, then 5 rounds of
// pointer doubling.  Needs the search result of position q0+32 (or q0+32 >= n).
template <int kMode>
__device__ __forceinline__ void resolve_one(const Smem& S, const LevelCfg& cfg, uint32_t n, uint32_t q0, unsigned& M,
                                            unsigned& J, bool& is_match) {
    const unsigned lane = zs_lane();
    const uint32_t q = q0 + lane;
    const uint32_t r = q < n ? S.res[res_slot(q)] : 0u;
    const unsigned L = (r >> 15) & 0x1ffu;
    unsigned Ln = __shfl_down_sync(ZS_FULL_MASK, L, 1);
    if (lane == 31) Ln = (q + 1 < n) ? ((S.res[res_slot(q + 1)] >> 15) & 0x1ffu) : 0u;
    // deflate_slow's lazy evaluation (deflate.ts:1372-1426): the match at q is dropped for a
    // literal when the match at q+1 is strictly longer and L < max_lazy
    const bool deferred = kMode == 1 && L >= 3 && L < (unsigned)cfg.lazy && Ln > L;
    is_match = L >= 3 && !deferred;
    // positions past the end of the chunk are terminal and never visited
    J = q < n ? lane + (is_match ? L : 1u) : 32u;
    M = q < n ? 1u << lane : 0u;
#pragma unroll
    for (int round = 0; round < 5; ++round) {
        const unsigned src = J < 32 ? J : lane;
        const unsigned Mj = __shfl_sync(ZS_FULL_MASK, M, src);
        const unsigned Jj = __shfl_sync(ZS_FULL_MASK, J, src);
        if (J < 32) { M |= Mj; J = Jj; }
    }
}

// An aligned pair of batches [q0, q0+64): both are resolved by the same warp and composed, so that
// the thin parse needs one hop per 64 positions.
template <int kMode>
__device__ __forceinline__ void resolve_pair(Smem& S, const LevelCfg& cfg, uint32_t n, uint32_t q0) {
    const unsigned lane = zs_lane();
    unsigned Ma, Ja, Mb, Jb;
    bool ma, mb;
    resolve_one<kMode>(S, cfg, n, q0, Ma, Ja, ma);
    resolve_one<kMode>(S, cfg, n, q0 + 32, Mb, Jb, mb);
    const unsigned ca = __popc(Ma), cb = __popc(Mb);
    // entering the pair at this lane of the first batch: where does the parse enter the second?
    const unsigned xa = Ja - 32u;
    const unsigned src = xa < 32u ? xa : lane;
    const unsigned jb = __shfl_sync(ZS_FULL_MASK, Jb, src), cbx = __shfl_sync(ZS_FULL_MASK, cb, src);
    const unsigned pair_exit = xa < 32u ? 32u + jb : Ja;   // >= 64 unless the chunk ends inside the pair
    const unsigned pair_cnt = xa < 32u ? ca + cbx : ca;
    const unsigned pe = pair_exit >= 32u ? pair_exit - 32u : 0u;
    if (q0 + lane < n)
        S.mj[mj_slot(q0 + lane)] = make_uint2(Ma, Ja | (ma ? MJ_MATCH : 0u) | (ca << 10) | (pe << 16) | (pair_cnt << 25));
    if (q0 + 32 + lane < n)
        S.mj[mj_slot(q0 + 32 + lane)] = make_uint2(Mb, Jb | (mb ? MJ_MATCH : 0u) | (cb << 10));
}

// ---- stage 5: parse (thin) ---------------------------------------------------------------------------
// Positions are range offsets and symbol indices count from the segment's first symbol: the symbols
// of a segment are stored back to back from the slot of its first input byte, so a chunk boundary
// inside a batch costs the emit stage nothing.  Blocks and their descriptors are per chunk.
struct ParseState {
    uint32_t ppos;       // next pair of batches, range offset
    uint32_t skip;       // leading positions of that pair already covered by an emitted match
    uint32_t nsym;       // symbols emitted in the segment
    uint32_t blk;        // blocks closed in the current chunk
    uint32_t blk_sym0;   // first symbol of the open block
    uint32_t blk_pos0;   // first input position of the open block (range offset)
    uint32_t jc;         // current chunk of the segment
    uint32_t cstart;     // its first position
    uint32_t nb;         // its end = the next boundary (0xffffffff after the last chunk)
};

// Block descriptor: first symbol (relative to the slot of the chunk's first byte: negative, as a
// wrapped 32-bit value, when earlier chunks of the segment produced fewer symbols than bytes),
// symbols, first input byte (relative to the chunk), input bytes.
__device__ __forceinline__ void close_block(const LzArgs& a, const RangeCtx& rc, ParseState& ps, uint32_t c0, uint32_t pos_end) {
    if (ps.blk < a.max_bpc && zs_lane() == 0) {  // max_bpc is sized so that the test always holds
        uint32_t* d = a.blk_desc + ((uint64_t)(c0 + ps.jc) * a.max_bpc + ps.blk) * 4;
        d[0] = ps.blk_sym0 - (ps.cstart - rc.q_data);
        d[1] = ps.nsym - ps.blk_sym0;
        d[2] = ps.blk_pos0 - ps.cstart;
        d[3] = pos_end - ps.blk_pos0;
    }
    ps.blk++;
    ps.blk_sym0 = ps.nsym;
    ps.blk_pos0 = pos_end;
}

// The parse stands on the boundary ps.nb: the final (possibly empty) block of the chunk, next chunk.
__device__ __forceinline__ void close_chunk(const Smem& S, const LzArgs& a, const RangeCtx& rc, ParseState& ps, uint32_t c0) {
    close_block(a, rc, ps, c0, ps.nb);
    if (zs_lane() == 0) a.chunk_nblk[c0 + ps.jc] = ps.blk < a.max_bpc ? ps.blk : a.max_bpc;
    ps.jc++;
    ps.cstart = ps.nb;
    ps.nb = ps.jc < rc.nc ? S.bnd[ps.jc + 1] : 0xffffffffu;
    ps.blk = 0;
}

__device__ __forceinline__ unsigned below(unsigned b) { return b >= 32u ? 0xffffffffu : (1u << b) - 1u; }

// Thin parse: the serial chain only, one hop per aligned pair of batches (64 positions).  For a group
// of up to kParseGroup pairs starting at qb the entry offset of every pair (0..63, or 64 = nothing
// to emit) and the index of its first symbol go to the pb ring; the wide warps write the symbols one
// step later (emit_batch).  Matches never cross a chunk boundary, so the chain lands on every
// boundary; a boundary strictly inside a pair splits the hop (rare: once per chunk).
// The chain is the thin warp's whole cost: it shares its SM sub-partition with seven issue-bound wide
// warps, so every instruction of a hop costs 6-7 cycles.  A hop entering pair q0 at offset s needs one
// word, mj[q0 + s].y (the pair fields for s < 32, the batch fields of the second batch for s >= 32),
// loaded on the chain as a broadcast.
// kRare = false: groups that no chunk boundary can touch and that cannot fill the open block (a pair adds
// at most 64 symbols), i.e. nearly all of them: unrolled, without a branch.  kRare = true: every other
// group, a plain loop with the boundary and block-cut tests per hop.
constexpr int kParseGroup = 16;
template <bool kRare>
__device__ __forceinline__ void parse_group(Smem& S, const LzArgs& a, const RangeCtx& rc, ParseState& ps, uint32_t c0,
                                            uint32_t qb, int np) {
    const unsigned lane = zs_lane();
    const uint32_t n = rc.n;
    unsigned pb_entry = 64u, pb_sym = 0;   // lane u: entry offset and first symbol of pair u
    uint32_t pos = qb + ps.skip;           // kRare = false: the position the chain stands on
    constexpr int kUnroll = kRare ? 1 : kParseGroup;
#pragma unroll kUnroll
    for (int u = 0; u < kParseGroup; ++u) {
        if (u >= np) break;
        const uint32_t q0 = qb + 64u * u;
        const uint32_t first_sym = ps.nsym;
        unsigned entry = 64u;
        if constexpr (!kRare) {
            // The group ends more than 258 positions before the next boundary, so pos < n and every exit lies
            // in a later pair.  A pair the previous match covers (pos >= q0 + 64) reads a word it does not use.
            const bool hop = pos < q0 + 64u, first = pos < q0 + 32u;
            const unsigned y = S.mj[mj_slot(pos)].y;
            const unsigned cnt = first ? mj_pair_count(y) : mj_count(y);
            const unsigned e = (y >> (first ? 16u : 0u)) & 0x1ffu;   // exit relative to the pair, - 32
            ps.nsym += hop ? cnt : 0u;
            entry = hop ? pos - q0 : 64u;
            if (hop) pos = q0 + 32u + e;
        } else if (ps.skip >= 64) {
            ps.skip -= 64;
        } else {
            unsigned s = ps.skip;
            entry = s;
            while (ps.nb < q0 + 64u) {
                // sub-hop [s, b): the symbols of the visited positions before the boundary
                const unsigned b = ps.nb - q0;
                unsigned c;
                if (b <= s) {
                    c = 0;   // an empty chunk; position q0 + s may be the end of the range, whose mj[] slot is stale
                } else if (s < 32u) {
                    const uint2 m = S.mj[mj_slot(q0 + s)];
                    c = __popc(m.x & below(b));
                    if (b > 32u) {
                        // the chain enters the second batch at xa <= b - 32; at xa == b - 32 it stands on the
                        // boundary already (and that slot of mj[] is stale when b is the end of the range)
                        const unsigned xa = mj_exit(m.y) - 32u;
                        if (xa < b - 32u) c += __popc(S.mj[mj_slot(q0 + 32u + xa)].x & below(b - 32u));
                    }
                } else {
                    c = __popc(S.mj[mj_slot(q0 + s)].x & below(b - 32u));
                }
                if (ps.nsym - ps.blk_sym0 + c > kSymLimit) close_block(a, rc, ps, c0, q0 + s);
                ps.nsym += c;
                close_chunk(S, a, rc, ps, c0);
                s = b;
            }
            // past the end of the range (it ends inside this pair) nothing is visited: the mj[] slots are stale
            unsigned cnt = 0, exit_rel = 64u;
            if (q0 + s < n) {
                const unsigned y = S.mj[mj_slot(q0 + s)].y;
                if (s < 32) { cnt = mj_pair_count(y); exit_rel = mj_pair_exit(y); }
                else { cnt = mj_count(y); exit_rel = 32u + mj_exit(y); }
            }
            if (ps.nsym - ps.blk_sym0 + cnt > kSymLimit) close_block(a, rc, ps, c0, q0 + s);
            ps.nsym += cnt;
            ps.skip = exit_rel >= 64u ? exit_rel - 64u : 0u;   // < 64 only where the range ends
            while (ps.nb <= q0 + exit_rel) close_chunk(S, a, rc, ps, c0);   // landed on a boundary
        }
        if (lane == (unsigned)u) { pb_entry = entry; pb_sym = first_sym; }
    }
    if constexpr (!kRare) ps.skip = pos - (qb + 64u * np);
    if (lane < (unsigned)np) S.pb[((qb >> 6) + lane) & (kPbRing - 1u)] = make_uint2(pb_entry, pb_sym);
}

// Wide emit: the symbols of one batch.  The pair's entry offset and first symbol index come from
// the thin parse; the second batch of a pair derives its own entry from the first batch's table.
__device__ __forceinline__ void emit_batch(const Smem& S, const LzArgs& a, uint64_t sym_base, uint32_t n, uint32_t q0) {
    const unsigned lane = zs_lane();
    const uint2 e = S.pb[(q0 >> 6) & (kPbRing - 1u)];
    if (e.x >= 64u) return;
    unsigned entry, first = e.y;
    if (!(q0 & 32u)) {                     // first batch of the pair
        if (e.x >= 32u) return;
        entry = e.x;
    } else if (e.x >= 32u) {               // the parse entered the pair in its second batch
        entry = e.x - 32u;
    } else {                               // through the first batch: continue where it left
        const unsigned ya = S.mj[mj_slot(q0 - 32u + e.x)].y;
        const unsigned xa = mj_exit(ya) - 32u;
        if (xa >= 32u) return;
        entry = xa;
        first += mj_count(ya);
    }
    // The chain may have reached the end of the range inside this pair: the mj[] slots from position n on
    // are stale (resolve never writes them), and symbols written from them would land in the slots of
    // the segments that follow.
    if (q0 + entry >= n) return;
    const unsigned visited = S.mj[mj_slot(q0 + entry)].x;  // same address in all lanes: a broadcast
    if (((visited >> lane) & 1u) && q0 + lane < n) {
        const uint32_t q = q0 + lane;
        const uint32_t r = S.res[res_slot(q)];
        const bool is_match = (S.mj[mj_slot(q)].y & MJ_MATCH) != 0;
        // packed symbol: distance << 16 | length, or the literal byte (distance 0)
        a.sym[sym_base + first + __popc(visited & zs_lanemask_lt())] =
            is_match ? (((r & 0x7fffu) << 16) | ((r >> 15) & 0x1ffu)) : (r >> 24);
    }
}

// Pipeline schedule (k = iteration): prep of step k, head exchange of step k-1, link of step k-2,
// search of step k-3; then, by position: resolve up to R(k), thin parse up to R(k-1), emit up to
// R(k-2), where R(k) is the resolved frontier after iteration k: the aligned pairs of batches
// (64 positions) whose successor position was searched before iteration k.
__device__ __forceinline__ uint32_t resolved_frontier(uint32_t searched, uint32_t n) {
    if (searched >= n) return n;
    return searched >= 64 ? (searched - 1) & ~63u : 0;
}

// kMode 1: levels 4-9 (deflate_slow's rules); 0: levels 1-3, greedy; 2: Z_RLE, greedy with distance 1 only.
// kLevel (greedy levels): 0 = the level's parameters come from a.cfg, 1-3 = that level's row at compile time.
// kDict: lz77_dict_kernel -- every segment is one chunk whose range starts with the prepared dictionary.
// The range offset q is the ring index itself (cb = 0): the dictionary's last <= 32 KiB at q = [0, L), the
// chunk at q = [L, L + len).  At segment start the CTA restores the saved tables and the dictionary's ring
// bytes (DictImage) instead of zeroing head[] / prev[], inserts from L - 2 on (the two positions the build
// deferred) and searches from L on, with the 32-position batches on the grid of the PRIME path for a range that
// starts at the dictionary.  The chunk is staged from global memory with plain loads (it starts at any byte,
// so the ring and the input are not congruent modulo 16 as the bulk copies need).  The output equals that of
// the PRIME path on a buffer holding the dictionary followed by the chunk.  With dict_img == nullptr the call
// builds the image instead: its one chunk is the dictionary, inserted and nothing searched.
template <int kMode, int kLevel, bool kDict>
__device__ __forceinline__ void lz77_run(const LzArgs& a) {
    static_assert(kLevel == 0 || (kMode == 0 && kLevel <= 3), "only the greedy levels are specialised");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem& S = *reinterpret_cast<Smem*>(smem_raw);
    const unsigned wid = threadIdx.x >> 5, lane = zs_lane();
    LevelCfg cfg = a.cfg;
    if constexpr (kLevel != 0) {
        constexpr LevelCfg row = level_cfg(kLevel);
        cfg = row;
    }
    const StopCfg stop = {a.stop_after, a.stop_active};
    (void)stop;

#ifdef ZS_LZ_BULK
    if (!kDict && threadIdx.x == 0) mbar_init(&S.stage_bar, 1);   // published by the first __syncthreads of the segment loop
#endif
#ifdef ZS_LZ_PROF
    // slowest wide warp of step k: prof_wmax[k & 1], reset by thread 0 behind the barrier of step k (no
    // warp reaches step k + 2 before that)
    __shared__ unsigned long long prof_wmax[2];
    if (threadIdx.x < 2) prof_wmax[threadIdx.x] = 0;
#endif
    for (;;) {
        if (threadIdx.x == 0) S.seg = atomicAdd(a.seg_counter, 1u);
        __syncthreads();
        const uint32_t seg = S.seg;
        if (seg >= a.n_seg) break;
        const bool big = seg < a.n_big;
        const uint32_t c0 = big ? seg * a.seg_chunks : a.n_big * a.seg_chunks + (seg - a.n_big) * a.seg_small;
        const uint32_t sc = big ? a.seg_chunks : a.seg_small;
        const uint32_t c1 = (c0 + sc < a.n_chunks) ? c0 + sc : a.n_chunks;

        const uint32_t nc = c1 - c0;

        // fresh tables per segment: the output never depends on which CTA ran which segment
        if (threadIdx.x == 0) S.claim[0] = 0;
        if (kDict && a.dict_img) {
            // the dictionary's tables and ring bytes, from L2 (one image for every chunk of the call)
            const uint4* src = reinterpret_cast<const uint4*>(a.dict_img);
            uint4* ht = reinterpret_cast<uint4*>(S.head);   // prev[] follows head[], as in the image
            for (unsigned i = threadIdx.x; i < kImgTables / 16u; i += kThreads) ht[i] = __ldg(src + i);
            const unsigned nring = (a.dict_len + 15u) / 16u;
            for (unsigned i = threadIdx.x; i < nring; i += kThreads) reinterpret_cast<uint4*>(S.ring)[i] = __ldg(src + kImgRing / 16u + i);
            for (unsigned i = threadIdx.x; i < kRingGuard / 16u; i += kThreads)
                reinterpret_cast<uint4*>(S.ring + kRing)[i] = __ldg(src + kImgGuard / 16u + i);
        } else {
            uint4* z = reinterpret_cast<uint4*>(S.head);
            const unsigned nz = (sizeof(S.head) + sizeof(S.prev)) / sizeof(uint4);
#ifdef ZS_LZ_PREV_DELTA
            const unsigned nh = sizeof(S.head) / sizeof(uint4);   // prev[] follows head[]: "no predecessor" is 0xffff there
            for (unsigned i = threadIdx.x; i < nz; i += kThreads) {
                const unsigned v = i < nh ? 0u : 0xffffffffu;
                z[i] = make_uint4(v, v, v, v);
            }
#else
            for (unsigned i = threadIdx.x; i < nz; i += kThreads) z[i] = make_uint4(0, 0, 0, 0);
#endif
        }
        // The range starts with the dictionary (deflateSetDictionary, deflate.ts:367-424): the
        // <= 32 KiB before the first chunk go through prep + insert + link only.
        const uint64_t off0 = a.in_off[c0];
        const uint64_t seg_start = a.org + off0;
        const uint64_t seg_end = a.org + a.in_off[c1];
        uint64_t prime0 = seg_start;
        if (kDict) {
            prime0 = 0;   // unused: the range offset is the ring index
        } else if (a.cross) {
            prime0 = seg_start > a.valid_lo + 32768 ? seg_start - 32768 : a.valid_lo;
            prime0 = (prime0 + 31) & ~31ull;
            if (prime0 > seg_start) prime0 = seg_start;
        }
        RangeCtx rc;
        rc.cb = (uint32_t)prime0;
        rc.n = (uint32_t)(seg_end - prime0);
        rc.q_data = (uint32_t)(seg_start - prime0);
        rc.nc = nc;
        rc.cross = a.cross;
        rc.min_len = (kMode == 1 && a.strategy == ZS_STRATEGY_FILTERED) ? 6u : 3u;
        uint32_t q_src = 0, q_start = 0;   // dictionary kernel: range offset of the chunk's first byte, first step
        if constexpr (kDict) {
            // build: the chunk is the dictionary (q = [0, L), nothing compressed); use: it follows the dictionary
            const uint32_t L = a.dict_len;
            q_src = a.dict_img ? L : 0u;
            rc.q_data = L;
            rc.n = q_src + (uint32_t)(seg_end - seg_start);
            rc.pre = 0;
            rc.tail = rc.n;   // as on the PRIME path with the chunk alone in the call: its last two positions are not inserted
            rc.ins_lo = a.dict_img ? (L >= 2u ? L - 2u : 0u) : 0u;
            q_start = rc.ins_lo & ~63u;   // a whole aligned pair of batches: the PRIME path's grid
            if (threadIdx.x < 2) S.bnd[threadIdx.x] = threadIdx.x ? rc.n : rc.q_data;
        } else {
            const uint64_t pre = a.cross ? prime0 - a.valid_lo : 0;
            rc.pre = pre < kMaxDist ? (uint32_t)pre : kMaxDist;
            const uint64_t tail = a.data_end - prime0;
            rc.tail = tail < 0xffffffffull ? (uint32_t)tail : 0xffffffffu;
            for (unsigned j = threadIdx.x; j <= nc; j += kThreads) S.bnd[j] = (uint32_t)(a.in_off[c0 + j] - off0) + rc.q_data;
        }
        // Staging addresses positions relative to base16 (the 16-byte line that holds the range's first byte):
        // after iteration k the ring holds everything below stage_rel(k + 1) = q_prep + 3 steps + guard, rounded up.
        const uint64_t base16 = prime0 & ~15ull;
        const uint32_t p0lo = (uint32_t)prime0 & 15u;
        const uint32_t safe_rel = [&] {   // first line past the end of the input, saturating
            const uint64_t d = ((a.data_end + 15) & ~15ull) - base16;
            return d < 0xfffffff0ull ? (uint32_t)d : 0xfffffff0u;
        }();
        // look-ahead for the first two steps of the range
        const int64_t g0 = (int64_t)seg_start - (int64_t)q_src;   // dictionary kernel: absolute index of range offset 0
        const int64_t dsafe16 = (int64_t)((a.data_end + 15) & ~15ull);
        if constexpr (kDict) {
            __syncthreads();   // the restored ring line that holds q_src is merged below
            const uint32_t to = (q_start + 2u * kStep + kRingGuard + 15u) & ~15u;
            for (uint32_t ql = (q_src & ~15u) + 16u * threadIdx.x; ql < to; ql += 16u * kThreads) {
                uint4 v = dict_src_line(a, g0, dsafe16, ql);
                const unsigned idx = ql & (kRing - 1u);
                if (ql < q_src) {   // the dictionary's last bytes share this line with the chunk's first ones
                    const uint4 d = *reinterpret_cast<const uint4*>(S.ring + idx);
                    const unsigned keep = q_src - ql;   // 1..15 bytes from the dictionary
                    auto m = [&](unsigned w) { return keep >= 4u * w + 4u ? 0xffffffffu : keep <= 4u * w ? 0u : (1u << (8u * (keep - 4u * w))) - 1u; };
                    v.x = (d.x & m(0)) | (v.x & ~m(0)); v.y = (d.y & m(1)) | (v.y & ~m(1));
                    v.z = (d.z & m(2)) | (v.z & ~m(2)); v.w = (d.w & m(3)) | (v.w & ~m(3));
                }
                *reinterpret_cast<uint4*>(S.ring + idx) = v;
                if (idx < kRingGuard) *reinterpret_cast<uint4*>(S.ring + kRing + idx) = v;
            }
        } else {
            stage_window(S, a, base16, base16 + ((p0lo + 2u * kStep + kRingGuard + 15u) & ~15u), threadIdx.x, kThreads);
        }
        __syncthreads();

        const uint32_t n = rc.n;
        const uint32_t nsteps = (n - q_start + kStep - 1) / kStep;
        const uint32_t n_iter = nsteps + 6;
        // The staging barrier completes one phase per step; a segment uses an even number of them (one empty phase
        // more after an odd number of steps), so the parity to wait for is k & 1 in every segment.  (Re-initialising
        // the barrier per segment -- mbarrier.inval + init -- was tried first: waits of later segments never returned.)
        const uint32_t nwait = (nsteps + 1u) & ~1u;
        (void)nwait;
        const uint32_t qd64 = rc.q_data & ~63u;   // the pair of batches that holds the first data position
        ParseState ps;
        ps.ppos = qd64; ps.skip = rc.q_data - qd64; ps.nsym = 0; ps.blk = 0; ps.blk_sym0 = 0; ps.blk_pos0 = rc.q_data;
        ps.jc = 0; ps.cstart = rc.q_data; ps.nb = S.bnd[1];
        if (wid == kWarpParse)
            while (ps.nb <= rc.q_data) close_chunk(S, a, rc, ps, c0);   // leading empty chunks
        // search: the chunk that holds this warp's batch (only moves forward) and its bounds
        unsigned js = 0;
        uint32_t cs_w = rc.q_data, ce_w = S.bnd[1];
        // per-iteration uniform state, kept incrementally (no multiplies / 64-bit math in the loop)
        uint32_t q_prep = q_start;           // first position of the step being prepped (q_start + k * kStep)
        unsigned s_prep = 0;                 // prep[] buffer of step k (k % 3)
        uint32_t searched = q_start;         // positions searched before this iteration
        uint32_t r0 = qd64, r1 = qd64, r2 = qd64, r3 = qd64;   // resolved frontier after iteration k, k-1, k-2, k-3

        for (uint32_t k = 0; k < n_iter; ++k) {
#ifdef ZS_LZ_PROF
            const long long t_begin = clock64();
#endif
            r3 = r2; r2 = r1; r1 = r0;
            r0 = resolved_frontier(searched, n);
            if (r0 < qd64) r0 = qd64;
            const unsigned s_ins = s_prep == 0 ? 2u : s_prep - 1u;     // (k - 1) % 3
            const unsigned s_link = s_ins == 0 ? 2u : s_ins - 1u;      // (k - 2) % 3
            if (kDict && wid == kWarpInsert) {
                // the same look-ahead as below, from the chunk through registers (range offset = ring index)
                const uint32_t stage_from = (q_prep + 2u * kStep + kRingGuard + 15u) & ~15u;
                const uint32_t stage_to = k < nsteps ? (q_prep + 3u * kStep + kRingGuard + 15u) & ~15u : stage_from;
                constexpr int kStageVec = (kStep + 16 + 511) / 512;   // 16-byte vectors per lane and step (covers a step)
                uint4 sv[kStageVec];
#pragma unroll
                for (int v = 0; v < kStageVec; ++v) {
                    const uint32_t pos = stage_from + 16u * (lane + 32 * v);
                    sv[v] = pos < stage_to ? dict_src_line(a, g0, dsafe16, pos) : make_uint4(0, 0, 0, 0);
                }
                if (k >= 1 && k - 1 < nsteps) {
                    const uint32_t p = q_prep - kStep + lane;
                    const uint32_t* pw = S.prep + s_ins * kStep + lane;
                    uint16_t* oh = S.oldh + ((k - 1) & 1u) * kStep;
#pragma unroll
                    for (int u = 0; u < kSearchWarps; ++u) head_exchange(S, p + 32u * u, pw[32 * u], oh + 32 * u);
                }
#pragma unroll
                for (int v = 0; v < kStageVec; ++v) {
                    const uint32_t pos = stage_from + 16u * (lane + 32 * v);
                    if (pos < stage_to) {
                        const unsigned idx = pos & (kRing - 1u);
                        *reinterpret_cast<uint4*>(S.ring + idx) = sv[v];
                        if (idx < kRingGuard) *reinterpret_cast<uint4*>(S.ring + kRing + idx) = sv[v];
                    }
                }
            } else if (wid == kWarpInsert) {
                // Bytes the next iteration reads (prep of step k+1, look-ahead of the search of step
                // k-2) replace positions 64 KiB older, which nobody reads any more.
                const uint32_t stage_from = (p0lo + q_prep + 2u * kStep + kRingGuard + 15u) & ~15u;
                const uint32_t stage_to = k < nsteps ? (p0lo + q_prep + 3u * kStep + kRingGuard + 15u) & ~15u : stage_from;
#ifdef ZS_LZ_BULK
                // The copy engine stages the readable part; it is started first and awaited last, so the
                // transfer runs behind the table updates.
                const uint32_t bulk_to = stage_to < safe_rel ? stage_to : safe_rel;
                if (k < nwait && lane == 0) {
                    unsigned total = 0;
                    if (stage_from < bulk_to) {
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // the ring slots were last written by ordinary stores
                        // expect_tx is given the total first: a copy may complete before a later arrive
                        const unsigned i0 = ((uint32_t)base16 + stage_from) & (kRing - 1u), nb = bulk_to - stage_from;
                        total = nb;
                        // the mirrored part: ring indices [0, kRingGuard) inside [i0, i0 + nb), before and after the wrap
                        if (i0 < kRingGuard) total += (i0 + nb < kRingGuard ? nb : kRingGuard - i0);
                        if (i0 + nb > kRing) total += (i0 + nb - kRing < kRingGuard ? i0 + nb - kRing : kRingGuard);
                    }
                    mbar_expect_tx(&S.stage_bar, total);
                    if (total) bulk_stage(S, a.buf, base16 + stage_from, base16 + bulk_to);
                }
#else
                // The global loads are issued first and stored last so that their latency hides behind the
                // table updates.
                constexpr int kStageVec = (kStep + 16 + 511) / 512;   // 16-byte vectors per lane and step
                uint4 sv[kStageVec];
#pragma unroll
                for (int v = 0; v < kStageVec; ++v) {
                    const uint32_t pos = stage_from + 16u * (lane + 32 * v);
                    sv[v] = make_uint4(0, 0, 0, 0);
                    if (pos < stage_to && pos < safe_rel) sv[v] = __ldg(reinterpret_cast<const uint4*>(a.buf + base16 + pos));
                }
#endif
                if (k >= 1 && k - 1 < nsteps) {
                    const uint32_t p = rc.cb + q_prep - kStep + lane;
                    const uint32_t* pw = S.prep + s_ins * kStep + lane;
                    uint16_t* oh = S.oldh + ((k - 1) & 1u) * kStep;
#pragma unroll
                    for (int u = 0; u < kSearchWarps; ++u) head_exchange(S, p + 32u * u, pw[32 * u], oh + 32 * u);
                }
#ifdef ZS_LZ_BULK
                // past the end of the input the window reads as zeros (the last steps of the last segment only)
                if (stage_to > safe_rel) {
                    for (uint32_t pos = (stage_from > safe_rel ? stage_from : safe_rel) + 16u * lane; pos < stage_to; pos += 512u) {
                        const unsigned idx = ((uint32_t)base16 + pos) & (kRing - 1u);
                        *reinterpret_cast<uint4*>(S.ring + idx) = make_uint4(0, 0, 0, 0);
                        if (idx < kRingGuard) *reinterpret_cast<uint4*>(S.ring + kRing + idx) = make_uint4(0, 0, 0, 0);
                    }
                }
#ifdef ZS_LZ_BULK_DEBUG   // a wait that does not end reports where it stands and gives up
                if (k < nwait) {
                    unsigned tries = 0, ok = 0;
                    while (!ok && tries < 200000u) {
                        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                                     : "=r"(ok) : "r"(smem_addr(&S.stage_bar)), "r"(k & 1u) : "memory");
                        ++tries;
                    }
                    if (!ok && lane == 0)
                        printf("[lz77 bulk] wait timed out: cta %u seg %u k %u of %u from %u to %u bulk_to %u safe %u p0lo %u base16 %llu\n",
                               blockIdx.x, seg, k, nsteps, stage_from, stage_to, bulk_to, safe_rel, p0lo, (unsigned long long)base16);
                }
#else
                if (k < nwait) mbar_wait(&S.stage_bar, k & 1u);
#endif
#else
#pragma unroll
                for (int v = 0; v < kStageVec; ++v) {
                    const uint32_t pos = stage_from + 16u * (lane + 32 * v);
                    if (pos < stage_to) {
                        const unsigned idx = ((uint32_t)base16 + pos) & (kRing - 1u);
                        *reinterpret_cast<uint4*>(S.ring + idx) = sv[v];
                        if (idx < kRingGuard) *reinterpret_cast<uint4*>(S.ring + kRing + idx) = sv[v];
                    }
                }
                // anything beyond kStageVec vectors per lane (never with the fixed 3-step look-ahead)
                if (stage_to > stage_from + 512u * kStageVec)
                    stage_window(S, a, base16 + stage_from + 512u * kStageVec, base16 + stage_to, lane, 32);
#endif
            } else if (wid == kWarpParse) {
                while (ps.ppos < r1) {
                    int np = (int)((r1 - ps.ppos + 63) / 64);
                    if (np > kParseGroup) np = kParseGroup;
                    // a hop leaves its pair by at most 257 positions and adds at most 64 symbols
                    if (ps.nb > ps.ppos + 64u * (unsigned)np + 258u && ps.nsym - ps.blk_sym0 + 64u * (unsigned)np <= kSymLimit)
                        parse_group<false>(S, a, rc, ps, c0, ps.ppos, np);
                    else
                        parse_group<true>(S, a, rc, ps, c0, ps.ppos, np);
                    ps.ppos += 64u * np;
                }
            } else {
                const unsigned i = wid * 32 + lane;
                // prep of step k
                if (k < nsteps) {
                    const uint32_t se = q_prep + kStep < n ? q_prep + kStep : n;
                    S.prep[s_prep * kStep + i] = prep_batch<kDict>(S, rc, q_prep + 32u * wid, se);
                }
                // link of step k-2 (its head exchange ran in the previous iteration)
                if (k >= 2 && k - 2 < nsteps)
                    link_batch(S, rc, q_prep - 2u * kStep + 32u * wid, S.prep[s_link * kStep + i], S.oldh[(k & 1u) * kStep + i]);
                // search of step k-3: data positions only (the tail of the dictionary inside the first
                // data pair reads as literals nobody visits)
                if (k >= 3 && k - 3 < nsteps) {
                    const uint32_t qw = q_prep - 3u * kStep + 32u * wid;
                    const uint32_t q = qw + lane;
                    if (qw + 32u > qd64 && qw < n) {
                        while (qw >= ce_w) { ++js; cs_w = ce_w; ce_w = S.bnd[js + 1]; }   // qw < n: terminates
                        uint32_t r = 0;
                        if constexpr (kMode == 1) {   // every lane of the batch takes part in the votes
                            const bool live = q >= rc.q_data && q < n;
                            uint32_t cs = cs_w, ce = ce_w;
                            if (live && q >= ce) {
                                unsigned jl = js;
                                do { ++jl; cs = ce; ce = S.bnd[jl + 1]; } while (q >= ce);
                            }
                            const uint32_t rr = search_lazy_endwin(S, cfg, stop, rc, q, cs, ce, live);
                            r = live ? rr : 0u;
                        } else
                        if (q >= rc.q_data && q < n) {
                            uint32_t cs = cs_w, ce = ce_w;
                            if (q >= ce) {   // a boundary inside the batch
                                unsigned jl = js;
                                do { ++jl; cs = ce; ce = S.bnd[jl + 1]; } while (q >= ce);
                            }
                            // (the end-window filter of the lazy levels costs the greedy levels 7 % on text: chains of 4
                            // have nothing to filter)
                            r = search_position<kMode == 1 ? 0 : kMode, kLevel>(S, cfg, rc, q, cs, ce);
                        }
                        if (q < n) S.res[res_slot(q)] = r;
                    }
                }
                // The lower half of the wide warps resolves (one pair of batches each), the upper half
                // emits (one pair each): both are ~150 instructions per pair, so the halves stay balanced.
                // (Claiming the pairs dynamically from a shared counter was measured: slower at level 1.)
                constexpr unsigned kHalf = kSearchWarps / 2;
#ifndef ZS_LZ_NO_CLAIM
                // Lazy levels: the search of a batch takes anything from a few to 128 lock-step candidates, and the step
                // ends with its slowest warp (ncu: the barrier is the first stall reason at level 6).  The resolve and
                // emit pairs are therefore claimed from a counter by whoever is done searching: a warp that is late
                // does none, the early ones share them.  (At the greedy levels the searches are short and even and the
                // static split below is faster.)
                if constexpr (kMode == 1) {
                    const unsigned nr = r0 > r1 ? (r0 - r1 + 63u) >> 6 : 0u, ne = r2 > r3 ? (r2 - r3 + 63u) >> 6 : 0u;
                    if (threadIdx.x == 0) S.claim[(k + 1u) & 1u] = 0;   // next iteration's counter: nobody touches it now
                    for (;;) {
                        unsigned item = 0;
                        if (lane == 0) item = atomicAdd(&S.claim[k & 1u], 1u);
                        item = __shfl_sync(ZS_FULL_MASK, item, 0);
                        if (item >= nr + ne) break;
                        if (item < nr) {
                            resolve_pair<kMode>(S, cfg, n, r1 + 64u * item);
                        } else {
                            const uint32_t q0 = r3 + 64u * (item - nr);
                            emit_batch(S, a, off0, n, q0);
                            if (q0 + 32 < r2) emit_batch(S, a, off0, n, q0 + 32);
                        }
                    }
                } else
#endif
                if (wid < kHalf) {
                    // resolve the pairs whose successor was searched before this iteration
                    for (uint32_t q0 = r1 + 64u * wid; q0 < r0; q0 += 64u * kHalf) resolve_pair<kMode>(S, cfg, n, q0);
                } else {
                    // emit the pairs the thin parse chained in the previous iteration
                    for (uint32_t q0 = r3 + 64u * (wid - kHalf); q0 < r2; q0 += 64u * (kSearchWarps - kHalf)) {
                        emit_batch(S, a, off0, n, q0);
                        if (q0 + 32 < r2) emit_batch(S, a, off0, n, q0 + 32);
                    }
                }
            }
#ifdef ZS_LZ_PROF
            {
                const long long t_work = clock64() - t_begin;
                __syncwarp();
                if (lane == 0) {
                    const int role = wid == kWarpInsert ? 0 : wid == kWarpParse ? 1 : 2;
                    atomicAdd(&g_prof[role], (unsigned long long)t_work);
                    if (role == 2) atomicMax(&prof_wmax[k & 1u], (unsigned long long)t_work);
                    if (wid == 0) atomicAdd(&g_prof[4], 1ull);
                }
            }
#endif
            // the search of step k-3 ran in this iteration
            if (k >= 3) searched = searched + kStep < n ? searched + kStep : n;
            q_prep += kStep;
            s_prep = s_prep == 2 ? 0u : s_prep + 1u;
            __syncthreads();
#ifdef ZS_LZ_PROF
            if (threadIdx.x == 0) {
                atomicAdd(&g_prof[3], (unsigned long long)(clock64() - t_begin));
                atomicAdd(&g_prof[5], prof_wmax[k & 1u]);
                prof_wmax[k & 1u] = 0;
            }
#endif
        }
        if (wid == kWarpParse)
            while (ps.jc < nc) close_chunk(S, a, rc, ps, c0);   // chunks that end with the range (and empty ones after it)
        __syncthreads();
        if (kDict && a.dict_save) {   // build: the tables as the chunks of later calls start from them (DictImage)
            uint4* dst = reinterpret_cast<uint4*>(a.dict_save);
            const uint4* ht = reinterpret_cast<const uint4*>(S.head);
            for (unsigned i = threadIdx.x; i < kImgTables / 16u; i += kThreads) dst[i] = ht[i];
            for (unsigned i = threadIdx.x; i < 32768u / 16u; i += kThreads) dst[kImgRing / 16u + i] = reinterpret_cast<const uint4*>(S.ring)[i];
            for (unsigned i = threadIdx.x; i < kRingGuard / 16u; i += kThreads)
                dst[kImgGuard / 16u + i] = reinterpret_cast<const uint4*>(S.ring + kRing)[i];
        }
    }
}

template <int kMode, int kLevel>
__global__ void __launch_bounds__(kThreads, 1) lz77_kernel(LzArgs a) { lz77_run<kMode, kLevel, false>(a); }
template <int kMode, int kLevel>
__global__ void __launch_bounds__(kThreads, 1) lz77_dict_kernel(LzArgs a) { lz77_run<kMode, kLevel, true>(a); }

// Level 0 (deflate_stored, deflate.ts:1140-1279) and Z_HUFFMAN_ONLY (deflate_huff, :1525-1560) need no
// match finder: the blocks of a chunk are cut at fixed input lengths -- 65535 bytes per stored block,
// kSymLimit literals per Huffman block -- and, for HUFFMAN_ONLY, symbol i of a chunk is its i-th byte.
__global__ void plain_blocks_kernel(LzArgs a, uint32_t per_block, int with_symbols) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= a.n_chunks) return;
    const uint32_t n = (uint32_t)(a.in_off[c + 1] - a.in_off[c]);
    uint32_t nb = (n + per_block - 1) / per_block;
    if (nb == 0) nb = 1;   // an empty chunk still ends with a (final) block
    if (nb > a.max_bpc) nb = a.max_bpc;
    for (uint32_t j = 0; j < nb; j++) {
        uint32_t* d = a.blk_desc + ((uint64_t)c * a.max_bpc + j) * 4;
        const uint32_t b0 = j * per_block, len = n - b0 < per_block ? n - b0 : per_block;
        d[0] = with_symbols ? b0 : 0u;
        d[1] = with_symbols ? len : 0u;
        d[2] = b0;
        d[3] = len;
    }
    a.chunk_nblk[c] = nb;
}
__global__ void literal_symbols_kernel(const uint8_t* in, uint32_t* sym, uint64_t n) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) sym[i] = in[i];
}

}  // namespace

int zs_launch_lz77(zs_ctx* ctx, const zs_deflate_plan& p) {
    // the opt-in to > 48 KB of dynamic shared memory is a per-device function attribute
    static bool attr_set[64] = {false};
    const int dev_slot = ctx->device >= 0 && ctx->device < 64 ? ctx->device : 0;
    // lz77_kernel<0, 0> is the greedy levels with their parameters read at run time, <0, L> level L specialised
    using LzKernel = void (*)(LzArgs);
    static const LzKernel kGreedy[4] = {lz77_kernel<0, 0>, lz77_kernel<0, 1>, lz77_kernel<0, 2>, lz77_kernel<0, 3>};
    static const LzKernel kGreedyDict[4] = {lz77_dict_kernel<0, 0>, lz77_dict_kernel<0, 1>, lz77_dict_kernel<0, 2>,
                                            lz77_dict_kernel<0, 3>};
    if (!attr_set[dev_slot] || ctx->device >= 64) {
        for (LzKernel k : kGreedy)
            ZS_CUDA_TRY(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem)));
        for (LzKernel k : kGreedyDict)
            ZS_CUDA_TRY(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem)));
        ZS_CUDA_TRY(ctx, cudaFuncSetAttribute(lz77_kernel<1, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem)));
        ZS_CUDA_TRY(ctx, cudaFuncSetAttribute(lz77_dict_kernel<1, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem)));
        ZS_CUDA_TRY(ctx, cudaFuncSetAttribute(lz77_kernel<2, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem)));
        attr_set[dev_slot] = true;
    }
    LzArgs a;
    const uintptr_t first = reinterpret_cast<uintptr_t>(p.d_in) - p.history;
    const uintptr_t adj = first & 15u;
    a.buf = reinterpret_cast<const uint8_t*>(first - adj);
    a.valid_lo = adj;
    a.org = adj + p.history;
    a.data_end = a.org + p.in_len;
    a.in_off = p.d_in_off;
    a.n_chunks = p.n_chunks;
    a.max_bpc = p.max_bpc;
    a.cfg = kLevels[p.level];
    a.strategy = p.strategy;
    a.cross = (p.mode == ZS_MODE_STITCHED || (p.flags & ZS_FLAG_PRIME)) ? 1 : 0;
    a.dict_img = nullptr;
    a.dict_save = nullptr;
    a.dict_len = 0;
    // A dictionary call: every chunk is its own segment (it must see the dictionary, not the chunk before it).
    // Z_RLE looks one byte back only and keeps its kernel: there the dictionary changes the framing alone.
    const bool with_dict = p.dict != nullptr && p.strategy != ZS_STRATEGY_RLE;
    if (with_dict) {
        a.cross = 1;
        a.dict_img = p.dict->d_img;
        a.dict_len = p.dict->len;
    }
    // Segments: runs of consecutive chunks that go through the pipeline as one range, sharing one set
    // of hash tables.  A segment pays the pipeline fill/drain (6 steps) and, with cross-chunk
    // matching, one 32 KiB insert-only priming pass.
    uint32_t seg_chunks = 1;
    if (a.cross) {
        // ~4 segments per SM keep the dynamic scheduler balanced; small batches fall back to one chunk
        seg_chunks = p.n_chunks / (4u * (uint32_t)ctx->sm_count);
        if (seg_chunks < 1) seg_chunks = 1;
        if (seg_chunks > 16) seg_chunks = 16;  // fixed for large batches: slicing a batch at multiples of 16 chunks
                                               // (the pipelined host path) then leaves the output unchanged
    } else {
        // Independent chunks: the segmentation cannot change the output (a search never looks before
        // its chunk), so cut a whole number of waves of ~512 KiB segments.
        uint64_t waves = p.in_len / ((uint64_t)ctx->sm_count * (512u << 10));
        if (waves < 1) waves = 1;
        const uint64_t want = waves * (uint64_t)ctx->sm_count;
        uint64_t sc = (p.n_chunks + want - 1) / want;
        if (sc < 1) sc = 1;
        if (sc > kMaxSegChunks) sc = kMaxSegChunks;
        seg_chunks = (uint32_t)sc;
    }
    if (a.cross && p.seg_hint) seg_chunks = p.seg_hint < kMaxSegChunks ? p.seg_hint : kMaxSegChunks;
    if (with_dict) seg_chunks = 1;
    // The CTAs claim segments in index order from an atomic counter, so what the kernel waits for at the end
    // is at most one segment: the last quarter of the chunks is cut into segments a quarter of the size
    // (measured on 8192 x 256 KiB chunks, level 6: 630 equal segments = 4.26 waves over 148 SMs, 14.5 GB/s;
    // the whole 16384-chunk batch, 6.9 waves: 16.8 GB/s).  The output does not depend on the segmentation:
    // every chunk sees the same <= 32 KiB - 2 steps of history whether it is primed or carried.
    a.seg_chunks = seg_chunks;
    a.seg_small = seg_chunks >= 4 ? seg_chunks / 4 : 1;
    a.n_big = (uint32_t)(((uint64_t)p.n_chunks * 3 / 4) / seg_chunks);
    {
        const uint32_t rest = p.n_chunks - a.n_big * seg_chunks;
        a.n_seg = a.n_big + (rest + a.seg_small - 1) / a.seg_small;
    }
    a.sym = p.d_sym;
    a.chunk_nblk = p.d_chunk_nblk;
    a.blk_desc = p.d_blk_desc;
    a.seg_counter = p.d_seg_counter;
    // straggler stop of the lazy levels (policy constants; the environment overrides exist for the A/B tools)
    a.stop_after = 8;
    a.stop_active = 8;
    if (const char* e = getenv("ZS_LZ_STOP_AFTER")) a.stop_after = (unsigned)atoi(e);
    if (const char* e = getenv("ZS_LZ_STOP_ACTIVE")) a.stop_active = (unsigned)atoi(e);
    // ZS_LZ_GREEDY_GENERIC=1: the greedy levels through lz77_kernel<0, 0>, the reference the level-specialised
    // kernels are compared with (same output, byte for byte)
    bool greedy_generic = false;
    if (const char* e = getenv("ZS_LZ_GREEDY_GENERIC")) greedy_generic = atoi(e) != 0;
#ifdef ZS_LZ_PROF
    // chain override in bits 8.. (the specialised kernels have theirs compiled in)
    if (const char* e = getenv("ZS_LZ_DEBUG"); e && (atoi(e) >> 8)) {
        a.cfg.chain = atoi(e) >> 8;
        greedy_generic = true;
    }
#endif
    if (p.level == 0 || p.strategy == ZS_STRATEGY_HUFFMAN_ONLY) {
        const bool stored = p.level == 0;
        ZS_KERNEL(ctx, "plain_blocks_kernel",
                  plain_blocks_kernel<<<(p.n_chunks + 127) / 128, 128, 0, ctx->stream>>>(a, stored ? 65535u : kSymLimit, stored ? 0 : 1));
        if (!stored && p.in_len)
            ZS_KERNEL(ctx, "literal_symbols_kernel",
                      literal_symbols_kernel<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(p.d_in, p.d_sym, p.in_len));
        return ZS_OK;
    }
    ZS_CUDA_TRY(ctx, cudaMemsetAsync(p.d_seg_counter, 0, sizeof(uint32_t), ctx->stream));
    unsigned grid = a.n_seg < (unsigned)ctx->sm_count ? a.n_seg : (unsigned)ctx->sm_count;
    if (grid == 0) return ZS_OK;
#ifdef ZS_DEBUG_HOOKS   // fewer CTAs: segments then run (nearly) in order, which separates scheduling effects from data effects
    if (getenv("ZS_LZ_GRID")) { unsigned g = (unsigned)atoi(getenv("ZS_LZ_GRID")); if (g && g < grid) grid = g; }
#endif
#ifdef ZS_LZ_PROF
    unsigned long long zero[16] = {0};
    cudaMemcpyToSymbol(g_prof, zero, sizeof(zero));
#endif
    if (with_dict) {
        const LzKernel k = p.level >= 4 ? lz77_dict_kernel<1, 0> : kGreedyDict[greedy_generic ? 0 : p.level];
        ZS_KERNEL(ctx, "lz77_dict_kernel", k<<<grid, kThreads, sizeof(Smem), ctx->stream>>>(a));
    } else if (a.strategy == ZS_STRATEGY_RLE) {
        ZS_KERNEL(ctx, "lz77_kernel", lz77_kernel<2, 0><<<grid, kThreads, sizeof(Smem), ctx->stream>>>(a));
    } else if (p.level >= 4) {
        ZS_KERNEL(ctx, "lz77_kernel", lz77_kernel<1, 0><<<grid, kThreads, sizeof(Smem), ctx->stream>>>(a));
    } else {
        const LzKernel k = kGreedy[greedy_generic ? 0 : p.level];
        ZS_KERNEL(ctx, "lz77_kernel", k<<<grid, kThreads, sizeof(Smem), ctx->stream>>>(a));
    }
#ifdef ZS_LZ_PROF
    {
        unsigned long long pr[16];
        cudaStreamSynchronize(ctx->stream);
        cudaMemcpyFromSymbol(pr, g_prof, sizeof(pr));
        double st = pr[4] ? (double)pr[4] : 1.0;
        fprintf(stderr, "[lz77 prof] level %d steps %llu  cycles/step: insert %.0f parse %.0f wide(avg warp) %.0f wide(max warp) %.0f step %.0f | insert: ldg-issued %.0f prep-loaded %.0f inserted %.0f | parse chain done %.0f\n",
                p.level, pr[4], pr[0] / st, pr[1] / st, pr[2] / st / kSearchWarps, pr[5] / st, pr[3] / st, pr[8] / st, pr[9] / st, pr[10] / st, pr[11] / st);
        fprintf(stderr, "[lz77 prof] chain-loop iterations: total %llu max %llu positions>100: %llu (last: best_len %llu at chunk offset %llu)\n",
                pr[12], pr[13], pr[14], pr[15] >> 32, pr[15] & 0xffffffffull);
    }
#endif
    return ZS_OK;
}

size_t zs_lz77_dict_image_bytes() { return kImgBytes; }

int zs_lz77_dict_build(zs_ctx* ctx, const uint8_t* d_dict, uint32_t len, uint8_t* d_img) {
    if (len > 32768u || (reinterpret_cast<uintptr_t>(d_dict) & 15u)) return ZS_STREAM_ERROR;
    // (the use launch sets the shared-memory opt-in of every dictionary kernel; the build runs <1, 0>)
    ZS_CUDA_TRY(ctx, cudaFuncSetAttribute(lz77_dict_kernel<1, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem)));
    // one chunk, the dictionary; nothing is searched, so the symbol and block outputs are a few words of scratch
    uint64_t* work = nullptr;
    ZS_CUDA_TRY(ctx, cudaMalloc(&work, 64 * sizeof(uint64_t)));
    const uint64_t off[2] = {0, len};
    cudaError_t e = cudaMemcpyAsync(work, off, sizeof(off), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(work + 2, 0, 62 * sizeof(uint64_t), ctx->stream);
    if (e != cudaSuccess) { cudaFree(work); return zs_set_cuda_error(ctx, e, "dictionary build"); }
    LzArgs a;
    memset(&a, 0, sizeof(a));
    a.buf = d_dict;
    a.org = 0;
    a.valid_lo = 0;
    a.data_end = len;
    a.in_off = work;
    a.n_chunks = 1; a.seg_chunks = 1; a.n_seg = 1; a.max_bpc = 1;
    a.n_big = 1; a.seg_small = 1;
    a.cfg = kLevels[6];
    a.strategy = ZS_STRATEGY_DEFAULT;
    a.cross = 1;
    a.seg_counter = reinterpret_cast<uint32_t*>(work + 2);
    a.chunk_nblk = reinterpret_cast<uint32_t*>(work + 3);
    a.blk_desc = reinterpret_cast<uint32_t*>(work + 4);
    a.sym = reinterpret_cast<uint32_t*>(work + 8);
    a.stop_after = 8; a.stop_active = 8;
    a.dict_img = nullptr;
    a.dict_save = d_img;
    a.dict_len = len;
    zs_prof_begin(ctx, "lz77_dict_build");
    lz77_dict_kernel<1, 0><<<1, kThreads, sizeof(Smem), ctx->stream>>>(a);
    zs_prof_end(ctx);
    ctx->launches++;
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(work);
    if (e != cudaSuccess) return zs_set_cuda_error(ctx, e, "lz77_dict_build");
    return ZS_OK;
}
