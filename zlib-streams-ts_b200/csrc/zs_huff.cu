// zs_huff.cu -- K4/K5/K9: length-limited Huffman construction, block-type choice, bit-offset layout,
// bit-packing encode, wrapper framing and the bit-granular stitch.
//
// Replaces the reference's trees.ts for whole blocks: build_tree / pqdownheap / gen_bitlen / gen_codes
// (src/mod/deflate/trees.ts:54-76,167-316), scan_tree / send_tree / build_bl_tree / send_all_trees
// (:318-447), compress_block / send_bits (:476-520,78-88), _tr_stored_block (:449-464), the
// stored/static/dynamic choice of _tr_flush_block (:544-590), and the header / trailer bytes that
// deflate() emits (src/mod/deflate/deflate.ts:750-832,964-988).
//
//  * huff_build_kernel: one thread per block runs the reference's heap construction unchanged
//    (same tie-breaks, same overflow repair), so for equal symbol frequencies the code lengths are
//    identical to the reference's -- checked against the oracle's build_tree in the tests.  It
//    also serialises the dynamic header into a per-block bit blob and records the block's size.
//  * layout kernels: stored blocks need byte alignment, so a chunk's bit length depends on the bit
//    offset it starts at; each chunk is summarised as (bits before its first stored block, bits
//    after), chunk starts are resolved by one warp (prefix scan when no chunk of a 32-chunk group
//    holds a stored block, shuffle-serial otherwise), then every block gets its absolute bit offset.
//    This is the "exclusive scan of per-chunk compressed bit lengths" of the north star.
//  * encode_kernel: one CTA per block; per 256-symbol tile a CTA-wide scan of code lengths gives
//    every symbol its bit offset, codes are OR-ed into a shared-memory staging tile and flushed as
//    whole 32-bit words (boundary words with atomicOr, the output having been zeroed).  Blocks
//    land directly at their final bit offset: the stitch is fused into the encode.
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "zs_common.cuh"

namespace {

constexpr int L_CODES = 286, D_CODES = 30, BL_CODES = 19, HEAP_SIZE = 2 * L_CODES + 1;
constexpr int kHdrWords = 160;   // per-block header blob: word0 = control, words 1.. = bits
constexpr uint32_t BT_STORED = 0, BT_STATIC = 1, BT_DYNAMIC = 2;

__constant__ uint8_t c_bl_order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

// ---- Huffman construction: one warp per block, everything in shared memory ----------------------
// The reference's heap (pqdownheap) is not a total order -- ties between equal (frequency, depth)
// pairs are decided by where the entries sit in the heap -- so reproducing its code lengths means
// running the same heap, serially.  Lane 0 does that on a compact layout: a heap entry carries its
// own key (frequency << 16 | depth << 10 | node), so a sift step is one 8-byte shared-memory load of
// the two children and one store, instead of six scattered loads.  Everything around the heap is
// lane-parallel: compaction of the non-zero symbols, leaf depths (every lane climbs dad[] from its
// leaves), bit-length counts, the opt_len / static_len sums, canonical code assignment (one lane per
// code length) and the coalesced stores of the code table.
constexpr int kHuffWarps = 8;
struct HuffWs {
    uint32_t heap[HEAP_SIZE + 3];   // [1 .. heap_len] the heap, [heap_max ..] nodes in extraction order; later: code staging
    uint16_t dad[HEAP_SIZE + 3];
    uint8_t len[HEAP_SIZE + 3];     // serial gen_bitlen only: lengths of all nodes
    uint8_t llen[288], dlen[32], blen[32];   // final code lengths of the three trees
    uint32_t bl_count[16];
    uint32_t bl_freq[20];
    uint16_t lnext[16], dnext[16], bnext[16];
};

__device__ __forceinline__ unsigned static_llen(unsigned n) { return n < 144 ? 8u : n < 256 ? 9u : n < 280 ? 7u : 8u; }
// canonical code of the fixed literal/length tree (RFC 1951 3.2.6), not yet bit-reversed
__device__ __forceinline__ unsigned static_lcode(unsigned n) {
    return n < 144 ? 0x30u + n : n < 256 ? 0x190u + (n - 144u) : n < 280 ? (n - 256u) : 0xC0u + (n - 280u);
}
__device__ __forceinline__ unsigned bl_xbits(unsigned n) { return n == 16 ? 2u : n == 17 ? 3u : n == 18 ? 7u : 0u; }

// kind: 0 literal/length, 1 distance, 2 bit-length
__device__ __forceinline__ unsigned extra_bits(int kind, unsigned n) {
    if (kind == 0) return n >= 257 ? zs_len_xbits(n - 257u) : 0u;
    if (kind == 1) return zs_dist_xbits(n);
    return bl_xbits(n);
}

__device__ __forceinline__ unsigned he_key(uint32_t e) { return e >> 10; }    // (frequency, depth)
__device__ __forceinline__ unsigned he_node(uint32_t e) { return e & 1023u; }

// pqdownheap, trees.ts:167-185.  smaller(n, m) of the reference is key(n) <= key(m).
__device__ __forceinline__ void sift_down(uint32_t* heap, int heap_len, int k) {
    const uint32_t v = heap[k];
    int j = k << 1;
    while (j <= heap_len) {
        const uint2 c = *reinterpret_cast<const uint2*>(heap + j);   // children j, j+1 (j is even; heap[] has a spare slot)
        uint32_t e = c.x;
        if (j < heap_len && he_key(c.y) <= he_key(c.x)) { e = c.y; j++; }
        if (he_key(v) <= he_key(e)) break;
        heap[k] = e;
        k = j;
        j <<= 1;
    }
    heap[k] = v;
}

// build_tree (trees.ts:261-316) + gen_bitlen (:187-259) for one tree, by one warp.  freq_of(n) gives
// the 16-bit frequency of symbol n.  Results: out_len[0 .. elems), w.bl_count, next codes, max_code;
// opt_len / static_len are advanced exactly as the reference does.
template <int KIND, typename FreqFn>
__device__ void build_tree_warp(HuffWs& w, FreqFn freq_of, uint8_t* out_len, uint16_t* next_out, int& max_code_out,
                                uint32_t& opt_len, uint32_t& static_len) {
    constexpr int elems = KIND == 0 ? L_CODES : KIND == 1 ? D_CODES : BL_CODES;
    constexpr int max_length = KIND == 2 ? 7 : 15;
    const unsigned lane = zs_lane();
    // the non-zero symbols, in symbol order, become heap[1 .. heap_len]
    int heap_len = 0, max_code = -1;
    for (int base = 0; base < elems; base += 32) {
        const int n = base + (int)lane;
        const unsigned f = n < elems ? (freq_of(n) & 0xffffu) : 0u;
        const unsigned bal = __ballot_sync(ZS_FULL_MASK, f != 0);
        if (f != 0) w.heap[heap_len + 1 + __popc(bal & zs_lanemask_lt())] = (f << 16) | (unsigned)n;
        if (n < elems) out_len[n] = 0;
        if (bal) max_code = base + 31 - __clz(bal);
        heap_len += __popc(bal);
    }
    if (lane < 16) w.bl_count[lane] = 0;
    // force at least two codes of non-zero frequency (trees.ts:280-288)
    unsigned phantom = 0;   // bit n: symbol n was given frequency 1
    while (heap_len < 2) {
        const int node = max_code < 2 ? ++max_code : 0;
        if (lane == 0) w.heap[heap_len + 1] = (1u << 16) | (unsigned)node;
        heap_len++;
        phantom |= 1u << node;
        opt_len--;
        if (KIND == 0) static_len -= static_llen((unsigned)node);
        else if (KIND == 1) static_len -= 5u;
    }
    __syncwarp();
    int heap_max = HEAP_SIZE;
    if (lane == 0) {
        uint32_t* heap = w.heap;
        for (int n = heap_len / 2; n >= 1; n--) sift_down(heap, heap_len, n);
        int node = elems, hl = heap_len;
        do {
            const uint32_t en = heap[1];
            heap[1] = heap[hl--];
            sift_down(heap, hl, 1);
            const uint32_t em = heap[1];
            heap[--heap_max] = en;
            heap[--heap_max] = em;
            const unsigned f = ((en >> 16) + (em >> 16)) & 0xffffu;   // 16-bit counters like the reference's
            const unsigned dn = (en >> 10) & 63u, dm = (em >> 10) & 63u;
            const unsigned d = (dn >= dm ? dn : dm) + 1u;
            w.dad[he_node(en)] = w.dad[he_node(em)] = (uint16_t)node;
            heap[1] = (f << 16) | (d << 10) | (unsigned)node++;
            sift_down(heap, hl, 1);
        } while (hl >= 2);
        heap[--heap_max] = heap[1];
    }
    heap_max = HEAP_SIZE - (2 * (heap_len - 1) + 1);   // what lane 0 ended with
    __syncwarp();
    const unsigned root = he_node(w.heap[heap_max]);
    // leaf depths: every lane climbs dad[] from its own leaves
    bool overflow = false;
    for (int base = 0; base <= max_code; base += 32) {
        const int n = base + (int)lane;
        if (n <= max_code && ((freq_of(n) & 0xffffu) != 0 || (n < 3 && ((phantom >> n) & 1u)))) {
            unsigned d = 0, x = (unsigned)n;
            while (x != root) { x = w.dad[x]; d++; }
            if (d > (unsigned)max_length) overflow = true;
            else { out_len[n] = (uint8_t)d; atomicAdd(&w.bl_count[d], 1u); }
        }
    }
    overflow = __any_sync(ZS_FULL_MASK, overflow);
    __syncwarp();
    if (overflow) {
        // the reference's clamp-and-repair, serially, in its own order (rare: needs a tree deeper than
        // max_length)
        if (lane == 0) {
            for (int b = 0; b < 16; b++) w.bl_count[b] = 0;
            int over = 0, h;
            w.len[root] = 0;
            for (h = heap_max + 1; h < HEAP_SIZE; h++) {
                const int n = (int)he_node(w.heap[h]);
                int bits = w.len[w.dad[n]] + 1;
                if (bits > max_length) { bits = max_length; over++; }
                w.len[n] = (uint8_t)bits;
                if (n > max_code) continue;
                w.bl_count[bits]++;
            }
            do {
                int bits = max_length - 1;
                while (w.bl_count[bits] == 0) bits--;
                w.bl_count[bits]--;
                w.bl_count[bits + 1] += 2;
                w.bl_count[max_length]--;
                over -= 2;
            } while (over > 0);
            for (int bits = max_length; bits != 0; bits--) {
                int n = (int)w.bl_count[bits];
                while (n != 0) {
                    const int m = (int)he_node(w.heap[--h]);
                    if (m > max_code) continue;
                    w.len[m] = (uint8_t)bits;
                    n--;
                }
            }
            for (int n = 0; n <= max_code; n++) out_len[n] = 0;
            for (h = heap_max; h < HEAP_SIZE; h++) {
                const int n = (int)he_node(w.heap[h]);
                if (n <= max_code) out_len[n] = w.len[n];
            }
        }
        __syncwarp();
    }
    // opt_len / static_len: sums over the leaves (the reference accumulates the same terms while it
    // assigns and repairs the lengths)
    uint32_t so = 0, ss = 0;
    for (int base = 0; base <= max_code; base += 32) {
        const int n = base + (int)lane;
        if (n <= max_code) {
            const unsigned l = out_len[n];
            if (l) {
                const uint32_t f = (n < 3 && ((phantom >> n) & 1u)) ? 1u : (freq_of(n) & 0xffffu);
                const unsigned xb = extra_bits(KIND, (unsigned)n);
                so += f * (l + xb);
                if (KIND == 0) ss += f * (static_llen((unsigned)n) + xb);
                else if (KIND == 1) ss += f * (5u + xb);
            }
        }
    }
    for (int o = 16; o; o >>= 1) { so += __shfl_xor_sync(ZS_FULL_MASK, so, o); ss += __shfl_xor_sync(ZS_FULL_MASK, ss, o); }
    opt_len += so;
    static_len += ss;
    // gen_codes, trees.ts:54-76: next_code per length
    if (lane == 0) {
        unsigned c = 0;
        next_out[0] = 0;
        for (int b = 1; b <= 15; b++) { c = (c + w.bl_count[b - 1]) << 1; next_out[b] = (uint16_t)c; }
    }
    __syncwarp();
    max_code_out = max_code;
}

// Canonical codes in symbol order: lane b owns code length b and walks the symbols.
__device__ __forceinline__ void assign_codes(const uint8_t* len, int max_code, const uint16_t* next, uint32_t* code_out, int elems) {
    const unsigned lane = zs_lane();
    for (int n = (int)lane; n < elems; n += 32) code_out[n] = 0;
    __syncwarp();
    if (lane >= 1 && lane <= 15) {
        unsigned c = next[lane];
        for (int n = 0; n <= max_code; n++)
            if (len[n] == lane) code_out[n] = zs_bitrev(c++, lane) | (lane << 16);
    }
    __syncwarp();
}

// bit blob writer for the dynamic header (lane 0, writes 32-bit words to global memory)
struct BlobWriter {
    uint32_t* w;
    uint64_t acc;
    unsigned nacc, nwords;
    uint32_t total;
    __device__ __forceinline__ void put(unsigned v, unsigned n) {
        acc |= (uint64_t)v << nacc;
        nacc += n;
        total += n;
        if (nacc >= 32) { w[nwords++] = (uint32_t)acc; acc >>= 32; nacc -= 32; }
    }
    __device__ __forceinline__ void finish() { if (nacc) w[nwords++] = (uint32_t)acc; }
};

// scan_tree (count = true, trees.ts:318-363) / send_tree (count = false, trees.ts:365-414)
__device__ void walk_tree(const uint8_t* len, int max_code, bool count, uint32_t* bl_freq,
                          const uint32_t* bl_code, BlobWriter* bw) {
    int prevlen = -1, curlen, nextlen = len[0], cnt = 0, max_count = 7, min_count = 4;
    if (nextlen == 0) { max_count = 138; min_count = 3; }
    for (int n = 0; n <= max_code; n++) {
        curlen = nextlen;
        nextlen = n + 1 <= max_code ? len[n + 1] : 0xffff;  // the reference plants a 0xffff guard
        if (++cnt < max_count && curlen == nextlen) continue;
        if (cnt < min_count) {
            if (count) bl_freq[curlen] += (uint32_t)cnt;
            else do bw->put(bl_code[curlen] & 0xffffu, bl_code[curlen] >> 16); while (--cnt != 0);
        } else if (curlen != 0) {
            if (curlen != prevlen) {
                if (count) bl_freq[curlen]++;
                else { bw->put(bl_code[curlen] & 0xffffu, bl_code[curlen] >> 16); cnt--; }
            }
            if (count) bl_freq[16]++;
            else { bw->put(bl_code[16] & 0xffffu, bl_code[16] >> 16); bw->put((unsigned)(cnt - 3), 2); }
        } else if (cnt <= 10) {
            if (count) bl_freq[17]++;
            else { bw->put(bl_code[17] & 0xffffu, bl_code[17] >> 16); bw->put((unsigned)(cnt - 3), 3); }
        } else {
            if (count) bl_freq[18]++;
            else { bw->put(bl_code[18] & 0xffffu, bl_code[18] >> 16); bw->put((unsigned)(cnt - 11), 7); }
        }
        cnt = 0;
        prevlen = curlen;
        if (nextlen == 0) { max_count = 138; min_count = 3; }
        else if (curlen == nextlen) { max_count = 6; min_count = 3; }
        else { max_count = 7; min_count = 4; }
    }
}

// K3: symbol histogram of every block (_tr_tally_lit/_tr_tally_dist, deflate/utils.ts:55-81): one CTA
// per block, shared-memory atomics, 286 literal/length + 30 distance counters.
struct HistArgs {
    uint32_t n_chunks, max_bpc;
    const uint64_t* in_off;
    const uint32_t* chunk_nblk;
    const uint32_t* blk_desc;
    const uint32_t* sym;
    uint32_t* blk_freq;
};

__global__ void __launch_bounds__(256) histogram_kernel(HistArgs a) {
    const uint64_t gid = blockIdx.x;
    const uint32_t chunk = (uint32_t)(gid / a.max_bpc), j = (uint32_t)(gid % a.max_bpc);
    if (j >= a.chunk_nblk[chunk]) return;
    __shared__ uint32_t h[320];
    for (unsigned i = threadIdx.x; i < 320; i += 256) h[i] = 0;
    __syncthreads();
    const uint32_t sym0 = a.blk_desc[gid * 4 + 0], nsym = a.blk_desc[gid * 4 + 1];
    const uint32_t* sym = a.sym + (int64_t)a.in_off[chunk] + (int32_t)sym0;   // sym0 may be negative, see close_block
    for (uint32_t i = threadIdx.x; i < nsym; i += 256) {
        const uint32_t s = sym[i];
        const unsigned dist = s >> 16, lc = s & 0xffffu;
        if (dist == 0) {
            atomicAdd(&h[lc], 1u);
        } else {
            atomicAdd(&h[257u + zs_len_code(lc - 3u)], 1u);
            atomicAdd(&h[288u + zs_dist_code(dist - 1u)], 1u);
        }
    }
    __syncthreads();
    uint32_t* f = a.blk_freq + gid * 320;
    for (unsigned i = threadIdx.x; i < 320; i += 256) f[i] = h[i];
}

struct HuffArgs {
    uint32_t n_chunks, max_bpc;
    const uint32_t* chunk_nblk;
    const uint32_t* blk_desc;
    const uint32_t* blk_freq;
    uint32_t* blk_code;
    uint32_t* blk_hdr;
    uint64_t* blk_bits;
    int force;   // 0: the reference's choice; 1: stored blocks only (level 0); 2: never dynamic (Z_FIXED, trees.ts:559-568)
};

// _tr_flush_block's decision (trees.ts:544-583) for every block; one warp per block.
__global__ void __launch_bounds__(32 * kHuffWarps) huff_build_kernel(HuffArgs a) {
    __shared__ __align__(16) HuffWs ws[kHuffWarps];
    const unsigned lane = zs_lane(), wid = threadIdx.x >> 5;
    const uint64_t gid = (uint64_t)blockIdx.x * kHuffWarps + wid;
    const uint64_t total = (uint64_t)a.n_chunks * a.max_bpc;
    if (gid >= total) return;
    const uint32_t chunk = (uint32_t)(gid / a.max_bpc), j = (uint32_t)(gid % a.max_bpc);
    if (j >= a.chunk_nblk[chunk]) return;
    HuffWs& w = ws[wid];
    const uint32_t* freq = a.blk_freq + gid * 320;
    const uint32_t in_len = a.blk_desc[gid * 4 + 3];
    if (a.force == 1) {   // deflate_stored: no trees at all
        if (lane == 0) { a.blk_hdr[gid * kHdrWords] = BT_STORED; a.blk_bits[gid] = 3ull + 32ull + 8ull * in_len; }
        return;
    }

    uint32_t opt_len = 0, static_len = 0;
    int l_max, d_max, b_max;
    // END_BLOCK always has frequency 1 (init_block, trees.ts:100)
    build_tree_warp<0>(w, [&](int n) { return n == 256 ? 1u : freq[n]; }, w.llen, w.lnext, l_max, opt_len, static_len);
    build_tree_warp<1>(w, [&](int n) { return freq[288 + n]; }, w.dlen, w.dnext, d_max, opt_len, static_len);
    // build_bl_tree, trees.ts:416-432
    if (lane < 20) w.bl_freq[lane] = 0;
    __syncwarp();
    if (lane == 0) {
        walk_tree(w.llen, l_max, true, w.bl_freq, nullptr, nullptr);
        walk_tree(w.dlen, d_max, true, w.bl_freq, nullptr, nullptr);
    }
    __syncwarp();
    build_tree_warp<2>(w, [&](int n) { return w.bl_freq[n]; }, w.blen, w.bnext, b_max, opt_len, static_len);
    int max_blindex;
    for (max_blindex = BL_CODES - 1; max_blindex >= 3; max_blindex--)
        if (w.blen[c_bl_order[max_blindex]] != 0) break;
    opt_len += 3u * ((uint32_t)max_blindex + 1u) + 5u + 5u + 4u;
    uint32_t opt_lenb = (opt_len + 3u + 7u) >> 3;
    const uint32_t static_lenb = (static_len + 3u + 7u) >> 3;
    if (static_lenb <= opt_lenb || a.force == 2) opt_lenb = static_lenb;

    uint32_t* code = a.blk_code + gid * 320;
    uint32_t* hdr = a.blk_hdr + gid * kHdrWords;
    uint64_t bits;
    if (in_len + 4u <= opt_lenb && in_len <= 65535u) {
        bits = 3ull + 32ull + 8ull * in_len;  // plus alignment padding, resolved by the layout
        if (lane == 0) hdr[0] = BT_STORED;
    } else if (static_lenb == opt_lenb) {
        bits = 3ull + static_len;
        for (unsigned n = lane; n < 320u; n += 32) {
            uint32_t c = 0;
            if (n < (unsigned)L_CODES) { const unsigned l = static_llen(n); c = zs_bitrev(static_lcode(n), l) | (l << 16); }
            else if (n >= 288u && n < 288u + D_CODES) c = zs_bitrev(n - 288u, 5) | (5u << 16);
            code[n] = c;
        }
        if (lane == 0) hdr[0] = BT_STATIC;
    } else {
        bits = 3ull + opt_len;
        uint32_t* stage = w.heap;               // the heap is done: [0, 320) code table, [320, 340) bit-length codes
        assign_codes(w.llen, l_max, w.lnext, stage, 288);
        assign_codes(w.dlen, d_max, w.dnext, stage + 288, 32);
        assign_codes(w.blen, b_max, w.bnext, stage + 320, 20);
        for (unsigned n = lane; n < 320u; n += 32) code[n] = stage[n];
        if (lane == 0) {
            // send_all_trees, trees.ts:434-447
            const uint32_t* bcode = stage + 320;
            BlobWriter bw = {hdr + 1, 0, 0, 0, 0};
            bw.put((unsigned)(l_max + 1 - 257), 5);
            bw.put((unsigned)(d_max + 1 - 1), 5);
            bw.put((unsigned)(max_blindex + 1 - 4), 4);
            for (int r = 0; r <= max_blindex; r++) bw.put(w.blen[c_bl_order[r]], 3);
            walk_tree(w.llen, l_max, false, nullptr, bcode, &bw);
            walk_tree(w.dlen, d_max, false, nullptr, bcode, &bw);
            bw.finish();
            hdr[0] = BT_DYNAMIC | (bw.total << 8);
        }
    }
    if (lane == 0) a.blk_bits[gid] = bits;
}

// ---- Huffman construction, thread per block (batches of very many small blocks) --------------------
// The same algorithm with every array in thread-private local memory.  One warp per block retires
// ~35 k serial instructions per block with one lane, which is issue-bound once a batch holds far
// more blocks than the GPU has warps (4 KiB records: 131 072 blocks); there, 32 blocks per warp in
// lockstep win (measured: 1.8 ms against 4.1 ms), while for 16 384 blocks of incompressible data the
// shared-memory version above is 2.2x faster (1.4 ms against 3.1 ms).
struct TpbTree {
    uint16_t freq[HEAP_SIZE];
    uint16_t dad[HEAP_SIZE];
    uint16_t len[HEAP_SIZE];
    int max_code;
};
struct TpbHeap {
    uint16_t heap[HEAP_SIZE + 1];
    uint8_t depth[HEAP_SIZE];
    int heap_len, heap_max;
    uint16_t bl_count[16];
    uint32_t opt_len, static_len;
};

__device__ __forceinline__ bool tpb_smaller(const TpbTree& t, const TpbHeap& h, int n, int m) {
    return t.freq[n] < t.freq[m] || (t.freq[n] == t.freq[m] && h.depth[n] <= h.depth[m]);
}

// pqdownheap, trees.ts:167-185
__device__ void tpb_sift_down(const TpbTree& t, TpbHeap& h, int k) {
    const int v = h.heap[k];
    int j = k << 1;
    while (j <= h.heap_len) {
        if (j < h.heap_len && tpb_smaller(t, h, h.heap[j + 1], h.heap[j])) j++;
        if (tpb_smaller(t, h, v, h.heap[j])) break;
        h.heap[k] = h.heap[j];
        k = j;
        j <<= 1;
    }
    h.heap[k] = (uint16_t)v;
}

// tpb_gen_bitlen, trees.ts:187-259
__device__ void tpb_gen_bitlen(TpbTree& t, TpbHeap& h, int kind, int max_length) {
    int hh, n, m, bits, overflow = 0;
    for (bits = 0; bits <= 15; bits++) h.bl_count[bits] = 0;
    t.len[h.heap[h.heap_max]] = 0;
    for (hh = h.heap_max + 1; hh < HEAP_SIZE; hh++) {
        n = h.heap[hh];
        bits = t.len[t.dad[n]] + 1;
        if (bits > max_length) { bits = max_length; overflow++; }
        t.len[n] = (uint16_t)bits;
        if (n > t.max_code) continue;
        h.bl_count[bits]++;
        const unsigned xb = extra_bits(kind, (unsigned)n);
        const uint32_t f = t.freq[n];
        h.opt_len += f * ((uint32_t)bits + xb);
        if (kind == 0) h.static_len += f * (static_llen((unsigned)n) + xb);
        else if (kind == 1) h.static_len += f * (5u + xb);
    }
    if (overflow == 0) return;
    do {
        bits = max_length - 1;
        while (h.bl_count[bits] == 0) bits--;
        h.bl_count[bits]--;
        h.bl_count[bits + 1] += 2;
        h.bl_count[max_length]--;
        overflow -= 2;
    } while (overflow > 0);
    for (bits = max_length; bits != 0; bits--) {
        n = h.bl_count[bits];
        while (n != 0) {
            m = h.heap[--hh];
            if (m > t.max_code) continue;
            if (t.len[m] != (unsigned)bits) {
                h.opt_len += (uint32_t)(((int)bits - (int)t.len[m]) * (int)t.freq[m]);
                t.len[m] = (uint16_t)bits;
            }
            n--;
        }
    }
}

// tpb_build_tree, trees.ts:261-316 (gen_codes is applied by the caller, which needs only bl_count)
__device__ void tpb_build_tree(TpbTree& t, TpbHeap& h, int kind) {
    const int elems = kind == 0 ? L_CODES : kind == 1 ? D_CODES : BL_CODES;
    const int max_length = kind == 2 ? 7 : 15;
    int n, m, node, max_code = -1;
    h.heap_len = 0;
    h.heap_max = HEAP_SIZE;
    for (n = 0; n < elems; n++) {
        if (t.freq[n] != 0) { h.heap[++h.heap_len] = (uint16_t)(max_code = n); h.depth[n] = 0; }
        else t.len[n] = 0;
    }
    while (h.heap_len < 2) {
        node = h.heap[++h.heap_len] = (uint16_t)(max_code < 2 ? ++max_code : 0);
        t.freq[node] = 1;
        h.depth[node] = 0;
        h.opt_len--;
        if (kind == 0) h.static_len -= static_llen((unsigned)node);
        else if (kind == 1) h.static_len -= 5u;
    }
    t.max_code = max_code;
    for (n = h.heap_len / 2; n >= 1; n--) tpb_sift_down(t, h, n);
    node = elems;
    do {
        n = h.heap[1];
        h.heap[1] = h.heap[h.heap_len--];
        tpb_sift_down(t, h, 1);
        m = h.heap[1];
        h.heap[--h.heap_max] = (uint16_t)n;
        h.heap[--h.heap_max] = (uint16_t)m;
        t.freq[node] = (uint16_t)(t.freq[n] + t.freq[m]);
        h.depth[node] = (uint8_t)((h.depth[n] >= h.depth[m] ? h.depth[n] : h.depth[m]) + 1);
        t.dad[n] = t.dad[m] = (uint16_t)node;
        h.heap[1] = (uint16_t)node++;
        tpb_sift_down(t, h, 1);
    } while (h.heap_len >= 2);
    h.heap[--h.heap_max] = h.heap[1];
    tpb_gen_bitlen(t, h, kind, max_length);
}

// gen_codes, trees.ts:54-76: next_code per length from bl_count
__device__ __forceinline__ void tpb_next_codes(const uint16_t* bl_count, uint16_t* next) {
    unsigned c = 0;
    next[0] = 0;
    for (int b = 1; b <= 15; b++) { c = (c + bl_count[b - 1]) << 1; next[b] = (uint16_t)c; }
}

// scan_tree (count = true, trees.ts:318-363) / send_tree (count = false, trees.ts:365-414)
__device__ void tpb_walk_tree(const uint16_t* len, int max_code, bool count, uint16_t* bl_freq,
                          const uint16_t* bl_code, const uint16_t* bl_len, BlobWriter* bw) {
    int prevlen = -1, curlen, nextlen = len[0], cnt = 0, max_count = 7, min_count = 4;
    if (nextlen == 0) { max_count = 138; min_count = 3; }
    for (int n = 0; n <= max_code; n++) {
        curlen = nextlen;
        nextlen = n + 1 <= max_code ? len[n + 1] : 0xffff;  // the reference plants a 0xffff guard
        if (++cnt < max_count && curlen == nextlen) continue;
        if (cnt < min_count) {
            if (count) bl_freq[curlen] += (uint16_t)cnt;
            else do bw->put(bl_code[curlen], bl_len[curlen]); while (--cnt != 0);
        } else if (curlen != 0) {
            if (curlen != prevlen) {
                if (count) bl_freq[curlen]++;
                else { bw->put(bl_code[curlen], bl_len[curlen]); cnt--; }
            }
            if (count) bl_freq[16]++;
            else { bw->put(bl_code[16], bl_len[16]); bw->put((unsigned)(cnt - 3), 2); }
        } else if (cnt <= 10) {
            if (count) bl_freq[17]++;
            else { bw->put(bl_code[17], bl_len[17]); bw->put((unsigned)(cnt - 3), 3); }
        } else {
            if (count) bl_freq[18]++;
            else { bw->put(bl_code[18], bl_len[18]); bw->put((unsigned)(cnt - 11), 7); }
        }
        cnt = 0;
        prevlen = curlen;
        if (nextlen == 0) { max_count = 138; min_count = 3; }
        else if (curlen == nextlen) { max_count = 6; min_count = 3; }
        else { max_count = 7; min_count = 4; }
    }
}

// _tr_flush_block's decision (trees.ts:544-583) for every block; one thread per block.
__global__ void __launch_bounds__(64) tpb_huff_build_kernel(HuffArgs a) {
    const uint64_t gid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t total = (uint64_t)a.n_chunks * a.max_bpc;
    if (gid >= total) return;
    const uint32_t chunk = (uint32_t)(gid / a.max_bpc), j = (uint32_t)(gid % a.max_bpc);
    if (j >= a.chunk_nblk[chunk]) return;
    const uint32_t* freq = a.blk_freq + gid * 320;
    const uint32_t in_len = a.blk_desc[gid * 4 + 3];
    if (a.force == 1) {   // deflate_stored: no trees at all
        a.blk_hdr[gid * kHdrWords] = BT_STORED;
        a.blk_bits[gid] = 3ull + 32ull + 8ull * in_len;
        return;
    }

    TpbTree lt, dt, bt;
    TpbHeap h;
    h.opt_len = h.static_len = 0;
    for (int n = 0; n < L_CODES; n++) lt.freq[n] = (uint16_t)freq[n];
    lt.freq[256] = 1;  // END_BLOCK, init_block trees.ts:100
    for (int n = 0; n < D_CODES; n++) dt.freq[n] = (uint16_t)freq[288 + n];
    tpb_build_tree(lt, h, 0);
    uint16_t lnext[16], dnext[16], bnext[16];
    tpb_next_codes(h.bl_count, lnext);
    tpb_build_tree(dt, h, 1);
    tpb_next_codes(h.bl_count, dnext);
    // build_bl_tree, trees.ts:416-432
    for (int n = 0; n < BL_CODES; n++) bt.freq[n] = 0;
    tpb_walk_tree(lt.len, lt.max_code, true, bt.freq, nullptr, nullptr, nullptr);
    tpb_walk_tree(dt.len, dt.max_code, true, bt.freq, nullptr, nullptr, nullptr);
    tpb_build_tree(bt, h, 2);
    tpb_next_codes(h.bl_count, bnext);
    int max_blindex;
    for (max_blindex = BL_CODES - 1; max_blindex >= 3; max_blindex--)
        if (bt.len[c_bl_order[max_blindex]] != 0) break;
    h.opt_len += 3u * ((uint32_t)max_blindex + 1u) + 5u + 5u + 4u;
    uint32_t opt_lenb = (h.opt_len + 3u + 7u) >> 3;
    const uint32_t static_lenb = (h.static_len + 3u + 7u) >> 3;
    if (static_lenb <= opt_lenb || a.force == 2) opt_lenb = static_lenb;

    uint32_t* code = a.blk_code + gid * 320;
    uint32_t* hdr = a.blk_hdr + gid * kHdrWords;
    uint32_t type;
    uint64_t bits;
    if (in_len + 4u <= opt_lenb && in_len <= 65535u) {
        type = BT_STORED;
        bits = 3ull + 32ull + 8ull * in_len;  // plus alignment padding, resolved by the layout
        hdr[0] = type;
    } else if (static_lenb == opt_lenb) {
        type = BT_STATIC;
        bits = 3ull + h.static_len;
        for (unsigned n = 0; n < (unsigned)L_CODES; n++) {
            unsigned l = static_llen(n);
            code[n] = zs_bitrev(static_lcode(n), l) | (l << 16);
        }
        for (unsigned n = 0; n < (unsigned)D_CODES; n++) code[288 + n] = zs_bitrev(n, 5) | (5u << 16);
        hdr[0] = type;
    } else {
        type = BT_DYNAMIC;
        bits = 3ull + h.opt_len;
        for (int n = 0; n < L_CODES; n++) {
            unsigned l = n <= lt.max_code ? lt.len[n] : 0;
            code[n] = l ? (zs_bitrev(lnext[l]++, l) | (l << 16)) : 0u;
        }
        for (int n = 0; n < D_CODES; n++) {
            unsigned l = n <= dt.max_code ? dt.len[n] : 0;
            code[288 + n] = l ? (zs_bitrev(dnext[l]++, l) | (l << 16)) : 0u;
        }
        uint16_t bcode[BL_CODES], blen[BL_CODES];
        for (int n = 0; n < BL_CODES; n++) {
            unsigned l = n <= bt.max_code ? bt.len[n] : 0;
            blen[n] = (uint16_t)l;
            bcode[n] = l ? (uint16_t)zs_bitrev(bnext[l]++, l) : 0;
        }
        // send_all_trees, trees.ts:434-447
        BlobWriter bw = {hdr + 1, 0, 0, 0, 0};
        bw.put((unsigned)(lt.max_code + 1 - 257), 5);
        bw.put((unsigned)(dt.max_code + 1 - 1), 5);
        bw.put((unsigned)(max_blindex + 1 - 4), 4);
        for (int r = 0; r <= max_blindex; r++) bw.put(blen[c_bl_order[r]], 3);
        tpb_walk_tree(lt.len, lt.max_code, false, nullptr, bcode, blen, &bw);
        tpb_walk_tree(dt.len, dt.max_code, false, nullptr, bcode, blen, &bw);
        bw.finish();
        hdr[0] = type | (bw.total << 8);
    }
    a.blk_bits[gid] = bits;
}

// ---- layout --------------------------------------------------------------------------------------
struct LayoutArgs {
    uint32_t n_chunks, max_bpc;
    int wrap, mode;
    uint32_t flags;
    const uint64_t* in_off;
    const uint32_t* chunk_nblk;
    uint32_t* blk_hdr;
    uint64_t* blk_bits;   // in: size; out: absolute bit offset of the block
    uint64_t* chunk_pr;   // [n][2]
    uint64_t* out_off;    // [n+1]
    uint64_t* out_bits;   // [n]
    uint64_t out_cap;
    zs_deflate_result* result;
    int32_t* error;
    const uint32_t* check_total;
    int fdict;            // zlib wrapper with a preset dictionary: FDICT + DICTID, a 6-byte header
};

// bytes of the wrapper header in front of every stream (INDEPENDENT) or of the stream (STITCHED)
__device__ __forceinline__ uint64_t wrap_header_bytes(int wrap, int fdict) {
    return wrap == ZS_WRAP_ZLIB ? (fdict ? 6 : 2) : wrap == ZS_WRAP_GZIP ? 10 : 0;
}

__device__ __forceinline__ unsigned stored_pad(uint64_t bitpos_after_hdr) { return (unsigned)((8u - (bitpos_after_hdr & 7u)) & 7u); }

// chunk summary: P = bits up to (excluding) the first stored block, R = bits from that block's
// LEN field to the end of the chunk (later stored blocks start from a known alignment)
__global__ void layout_chunks_kernel(LayoutArgs a) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= a.n_chunks) return;
    const uint32_t nb = a.chunk_nblk[c];
    // Z_SYNC_FLUSH marker (empty stored block) after the chunk: between chunks when ZS_FLAG_SYNC is
    // set, and always at the end of a part that is not the last one -- the next part must start
    // byte aligned because stored blocks inside it are padded relative to its own first bit
    const bool sync_marker = a.mode == ZS_MODE_STITCHED &&
                             (c + 1 == a.n_chunks ? (a.flags & ZS_FLAG_NOT_LAST) != 0 : (a.flags & ZS_FLAG_SYNC) != 0);
    uint64_t P = 0, R = 0;
    bool seen = false;
    for (uint32_t j = 0; j < nb + (sync_marker ? 1u : 0u); j++) {
        const bool marker = j == nb;
        const uint64_t gid = (uint64_t)c * a.max_bpc + j;
        const uint32_t type = marker ? BT_STORED : (a.blk_hdr[gid * kHdrWords] & 0xffu);
        const uint64_t bits = marker ? 35ull : a.blk_bits[gid];
        if (type == BT_STORED) {
            if (!seen) { seen = true; R = bits - 3; }
            else R += 3 + stored_pad(R + 3) + (bits - 3);  // R counts from a byte boundary
        } else {
            if (seen) R += bits; else P += bits;
        }
    }
    a.chunk_pr[2 * c] = P;
    a.chunk_pr[2 * c + 1] = (R << 1) | (seen ? 1u : 0u);
}

__device__ __forceinline__ uint64_t chunk_len_at(uint64_t start, uint64_t P, uint64_t Rf) {
    if (!(Rf & 1u)) return P;
    return P + 3 + stored_pad(start + P + 3) + (Rf >> 1);
}

// One CTA resolves the start of every chunk.  INDEPENDENT: byte offsets of whole streams (wrapper
// header + body + trailer) -- a plain prefix sum.  STITCHED: bit offsets inside the single stream,
// where a chunk's length depends on the bit its first stored block starts at.  Only the start
// modulo 8 matters, and a chunk that holds a stored block ends at a residue that does not depend on
// where it started (everything after the padding is fixed), so the start residues are a segmented
// scan -- "reset to a constant" for chunks with a stored block, "add P mod 8" for the others --
// followed by an ordinary prefix sum of the lengths.  1024 chunks per round.
constexpr int kScanThreads = 1024;
// residue-scan element: bit 3 = reset, bits 0..2 = value; a then b
__device__ __forceinline__ unsigned res_combine(unsigned a, unsigned b) {
    return (b & 8u) ? b : ((a & 8u) | (((a & 7u) + (b & 7u)) & 7u));
}
__global__ void __launch_bounds__(kScanThreads) layout_scan_kernel(LayoutArgs a) {
    __shared__ unsigned s_res[32];
    __shared__ uint64_t s_len[32];
    __shared__ uint64_t s_tile_len;
    const unsigned lane = zs_lane(), wid = threadIdx.x >> 5;
    const uint64_t H = wrap_header_bytes(a.wrap, a.fdict);
    const uint64_t T = a.wrap == ZS_WRAP_ZLIB ? 4 : a.wrap == ZS_WRAP_GZIP ? 8 : 0;
    const bool stitched = a.mode == ZS_MODE_STITCHED;
    uint64_t pos = 0;  // INDEPENDENT: bytes; STITCHED: bits
    if (stitched && !(a.flags & ZS_FLAG_NOT_FIRST)) pos = 8 * H;
    for (uint32_t base = 0; base < a.n_chunks; base += kScanThreads) {
        const uint32_t c = base + threadIdx.x;
        const bool live = c < a.n_chunks;
        const uint64_t P = live ? a.chunk_pr[2 * c] : 0, Rf = live ? a.chunk_pr[2 * c + 1] : 0;
        unsigned start_res = 0;
        if (stitched) {
            const unsigned e = !live ? 0u : (Rf & 1u) ? (8u | (unsigned)((Rf >> 1) & 7u)) : (unsigned)(P & 7u);
            unsigned x = e;
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned v = __shfl_up_sync(ZS_FULL_MASK, x, o);
                if ((int)lane >= o) x = res_combine(v, x);
            }
            if (lane == 31) s_res[wid] = x;
            unsigned ex = __shfl_up_sync(ZS_FULL_MASK, x, 1);
            if (lane == 0) ex = 0;   // identity
            __syncthreads();
            if (wid == 0) {
                unsigned t = s_res[lane], incl = t;
                for (int o = 1; o < 32; o <<= 1) {
                    const unsigned v = __shfl_up_sync(ZS_FULL_MASK, incl, o);
                    if ((int)lane >= o) incl = res_combine(v, incl);
                }
                unsigned wex = __shfl_up_sync(ZS_FULL_MASK, incl, 1);
                if (lane == 0) wex = 0;
                s_res[lane] = wex;
            }
            __syncthreads();
            const unsigned carry = 8u | (unsigned)(pos & 7u);
            start_res = res_combine(res_combine(carry, s_res[wid]), ex) & 7u;
        }
        const uint64_t my_bits = live ? chunk_len_at(start_res, P, Rf) : 0;
        const uint64_t sz = stitched ? my_bits : (live ? H + ((my_bits + 7) >> 3) + T : 0);
        uint64_t incl = sz;
        for (int o = 1; o < 32; o <<= 1) {
            const uint64_t v = __shfl_up_sync(ZS_FULL_MASK, incl, o);
            if ((int)lane >= o) incl += v;
        }
        if (lane == 31) s_len[wid] = incl;
        __syncthreads();
        if (wid == 0) {
            const uint64_t t = s_len[lane];
            uint64_t wi = t;
            for (int o = 1; o < 32; o <<= 1) {
                const uint64_t v = __shfl_up_sync(ZS_FULL_MASK, wi, o);
                if ((int)lane >= o) wi += v;
            }
            s_len[lane] = wi - t;
            if (lane == 31) s_tile_len = wi;
        }
        __syncthreads();
        const uint64_t my_start = pos + s_len[wid] + incl - sz;
        if (live) { a.out_off[c] = my_start; a.out_bits[c] = my_bits; }
        pos += s_tile_len;
        __syncthreads();   // s_len / s_res are rewritten by the next round
    }
    if (threadIdx.x == 0) {
        uint64_t total_bits, total_bytes;
        if (stitched) {
            total_bits = pos;
            total_bytes = (pos + 7) >> 3;
            if (!(a.flags & ZS_FLAG_NOT_LAST)) {
                // the trailer covers the whole stream, so only a call that holds the whole stream
                // writes it; the last part of a multi-part stream is just padded to a byte
                if (!(a.flags & ZS_FLAG_NOT_FIRST)) total_bytes += T;
                total_bits = total_bytes * 8;
            }
        } else {
            total_bytes = pos;
            total_bits = pos * 8;
        }
        a.out_off[a.n_chunks] = pos;
        a.result->total_out_bytes = total_bytes;
        a.result->total_out_bits = total_bits;
        if (total_bytes > a.out_cap) *a.error = ZS_BUF_ERROR;
    }
}

// absolute bit offset + BFINAL flag for every block
__global__ void layout_blocks_kernel(LayoutArgs a) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= a.n_chunks) return;
    const uint32_t nb = a.chunk_nblk[c];
    const bool stitched = a.mode == ZS_MODE_STITCHED;
    const uint64_t H = wrap_header_bytes(a.wrap, a.fdict);
    uint64_t pos = stitched ? a.out_off[c] : 8 * (a.out_off[c] + H);
    const bool chunk_final = stitched ? (c + 1 == a.n_chunks && !(a.flags & ZS_FLAG_NOT_LAST)) : true;
    for (uint32_t j = 0; j < nb; j++) {
        const uint64_t gid = (uint64_t)c * a.max_bpc + j;
        const uint32_t h0 = a.blk_hdr[gid * kHdrWords];
        const uint64_t bits = a.blk_bits[gid];
        a.blk_bits[gid] = pos;
        if (chunk_final && j + 1 == nb) a.blk_hdr[gid * kHdrWords] = h0 | 0x80000000u;
        if ((h0 & 0xffu) == BT_STORED) pos += 3 + stored_pad(pos + 3) + (bits - 3);
        else pos += bits;
    }
}

// ---- encode --------------------------------------------------------------------------------------
struct EncodeArgs {
    uint32_t n_chunks, max_bpc;
    int wrap, mode;
    uint32_t flags;
    const uint8_t* in;          // d_in
    const uint64_t* in_off;
    const uint32_t* sym;
    const uint32_t* chunk_nblk;
    const uint32_t* blk_desc;
    const uint32_t* blk_code;
    const uint32_t* blk_hdr;
    const uint64_t* blk_abs;    // absolute bit offsets
    const uint64_t* out_off;
    const uint64_t* out_bits;
    const uint32_t* checks;     // per-chunk check values (wrapper trailers), may be null
    const uint32_t* check_total;
    uint8_t* out;
    const zs_deflate_result* result;
    const int32_t* error;
    int level;
    int fdict;            // see LayoutArgs
    uint32_t dict_id;     // DICTID: adler32 of the whole preset dictionary
};

__device__ __forceinline__ void or_bits_global(uint32_t* out32, uint64_t bitpos, uint64_t v, unsigned n) {
    if (n == 0) return;
    uint64_t w = bitpos >> 5;
    unsigned sh = (unsigned)(bitpos & 31u);
    atomicOr(out32 + w, (uint32_t)(v << sh));
    if (sh + n > 32) {
        uint64_t rest = v >> (32 - sh);
        atomicOr(out32 + w + 1, (uint32_t)rest);
        if (sh + n > 64) atomicOr(out32 + w + 2, (uint32_t)(rest >> 32));
    }
}

__global__ void zero_output_kernel(uint8_t* out, const zs_deflate_result* result, const int32_t* error, uint64_t cap) {
    if (*error) return;
    uint64_t nbytes = result->total_out_bytes + 8;  // the encoder ORs whole words near the end
    if (nbytes > cap) nbytes = cap;
    uint64_t nvec = nbytes >> 4;
    uint4* o = reinterpret_cast<uint4*>(out);
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (uint64_t)gridDim.x * blockDim.x)
        o[i] = make_uint4(0, 0, 0, 0);
    if (blockIdx.x == 0 && threadIdx.x < 16) {
        uint64_t i = (nvec << 4) + threadIdx.x;
        if (i < nbytes) out[i] = 0;
    }
}

constexpr int kEncThreads = 256;
constexpr int kSymPerThread = 4;
constexpr unsigned kStageWords = kEncThreads * kSymPerThread * 2 + 4;   // up to 48+ bits per symbol, plus a lead-in word

// compress_block (trees.ts:476-520) for one block per CTA
__global__ void __launch_bounds__(kEncThreads) encode_kernel(EncodeArgs a) {
    if (*a.error) return;
    const uint64_t gid = blockIdx.x;
    const uint32_t chunk = (uint32_t)(gid / a.max_bpc), j = (uint32_t)(gid % a.max_bpc);
    if (j >= a.chunk_nblk[chunk]) return;
    __shared__ uint32_t s_code[320];
    __shared__ uint32_t s_stage[kStageWords];
    __shared__ uint32_t s_warp[kEncThreads / 32];
    const unsigned t = threadIdx.x, lane = t & 31u, wid = t >> 5;
    uint32_t* out32 = reinterpret_cast<uint32_t*>(a.out);
    const uint32_t h0 = a.blk_hdr[gid * kHdrWords];
    const uint32_t type = h0 & 0xffu, final = h0 >> 31, hdr_bits = (h0 >> 8) & 0x7fffffu;
    uint64_t pos = a.blk_abs[gid];
    const uint32_t sym0 = a.blk_desc[gid * 4 + 0], nsym = a.blk_desc[gid * 4 + 1];
    const uint32_t in0 = a.blk_desc[gid * 4 + 2], in_len = a.blk_desc[gid * 4 + 3];
    const uint64_t cbase = a.in_off[chunk];

    if (type == BT_STORED) {
        // _tr_stored_block, trees.ts:449-464
        if (t == 0) or_bits_global(out32, pos, final, 3);
        pos += 3;
        pos += stored_pad(pos);
        uint8_t* o = a.out + (pos >> 3);
        if (t == 0) {
            o[0] = (uint8_t)in_len; o[1] = (uint8_t)(in_len >> 8);
            o[2] = (uint8_t)~in_len; o[3] = (uint8_t)(~in_len >> 8);
        }
        const uint8_t* src = a.in + cbase + in0;
        for (uint32_t i = t; i < in_len; i += kEncThreads) o[4 + i] = __ldg(src + i);
        return;
    }

    for (unsigned i = t; i < 320; i += kEncThreads) s_code[i] = a.blk_code[gid * 320 + i];
    // block header: BFINAL | BTYPE << 1, then the serialised trees of a dynamic block
    if (t == 0) or_bits_global(out32, pos, final | (type << 1), 3);
    pos += 3;
    if (type == BT_DYNAMIC) {
        const uint32_t* hw = a.blk_hdr + gid * kHdrWords + 1;
        const unsigned nw = (hdr_bits + 31) >> 5;
        for (unsigned i = t; i < nw; i += kEncThreads) {
            unsigned nb = (i + 1 == nw && (hdr_bits & 31u)) ? (hdr_bits & 31u) : 32u;
            or_bits_global(out32, pos + 32ull * i, hw[i], nb);
        }
        pos += hdr_bits;
    }
    __syncthreads();

    const uint32_t* sym = a.sym + (int64_t)cbase + (int32_t)sym0;   // sym0 may be negative (zs_lz77.cu, close_block)
    // Tiles of kEncThreads * kSymPerThread symbols; a thread owns kSymPerThread consecutive symbols, so one
    // CTA-wide scan (and three barriers) serves 1024 symbols.
    constexpr uint32_t kTile = kEncThreads * kSymPerThread;
    for (uint32_t tile = 0; tile < nsym; tile += kTile) {
        uint64_t v[kSymPerThread];
        unsigned nb[kSymPerThread];
        unsigned mine = 0;
#pragma unroll
        for (int u = 0; u < kSymPerThread; u++) {
            const uint32_t i = tile + t * kSymPerThread + u;
            v[u] = 0; nb[u] = 0;
            if (i < nsym) {
                const uint32_t s = sym[i];
                const unsigned dist = s >> 16, lc = s & 0xffffu;
                if (dist == 0) {
                    const uint32_t e = s_code[lc];
                    v[u] = e & 0xffffu; nb[u] = e >> 16;
                } else {
                    const unsigned l3 = lc - 3u;
                    const unsigned lcode = zs_len_code(l3);
                    uint32_t e = s_code[257u + lcode];
                    uint64_t vv = e & 0xffffu; unsigned n = e >> 16;
                    unsigned xb = zs_len_xbits(lcode);
                    vv |= (uint64_t)(l3 - zs_len_base(lcode)) << n; n += xb;
                    const unsigned d1 = dist - 1u;
                    const unsigned dcode = zs_dist_code(d1);
                    e = s_code[288u + dcode];
                    vv |= (uint64_t)(e & 0xffffu) << n; n += e >> 16;
                    xb = zs_dist_xbits(dcode);
                    vv |= (uint64_t)(d1 - zs_dist_base(dcode)) << n; n += xb;
                    v[u] = vv; nb[u] = n;
                }
            }
            mine += nb[u];
        }
        // CTA-wide exclusive scan of the per-thread bit counts
        unsigned incl = mine;
        for (int o = 1; o < 32; o <<= 1) {
            unsigned x = __shfl_up_sync(ZS_FULL_MASK, incl, o);
            if ((int)lane >= o) incl += x;
        }
        if (lane == 31) s_warp[wid] = incl;
        for (unsigned k = t; k < kStageWords; k += kEncThreads) s_stage[k] = 0;
        __syncthreads();
        unsigned wbase = 0, tile_bits = 0;
        for (unsigned k = 0; k < kEncThreads / 32; k++) {
            const unsigned x = s_warp[k];
            if (k < wid) wbase += x;
            tile_bits += x;
        }
        const unsigned lead = (unsigned)(pos & 31u);
        unsigned off = lead + wbase + incl - mine;
#pragma unroll
        for (int u = 0; u < kSymPerThread; u++) {
            if (nb[u]) {
                const unsigned w = off >> 5, sh = off & 31u;
                atomicOr(&s_stage[w], (uint32_t)(v[u] << sh));
                if (sh + nb[u] > 32) {
                    const uint64_t rest = v[u] >> (32 - sh);
                    atomicOr(&s_stage[w + 1], (uint32_t)rest);
                    if (sh + nb[u] > 64) atomicOr(&s_stage[w + 2], (uint32_t)(rest >> 32));
                }
                off += nb[u];
            }
        }
        __syncthreads();
        const unsigned nwords = (lead + tile_bits + 31) >> 5;
        const uint64_t w0 = pos >> 5;
        for (unsigned k = t; k < nwords; k += kEncThreads) {
            const uint32_t x = s_stage[k];
            if (k == 0 || k + 1 == nwords) { if (x) atomicOr(out32 + w0 + k, x); }
            else out32[w0 + k] = x;
        }
        pos += tile_bits;
        __syncthreads();
    }
    if (t == 0) {
        const uint32_t e = s_code[256];
        or_bits_global(out32, pos, e & 0xffffu, e >> 16);
    }
}

// wrapper header / trailer bytes (deflate.ts:750-832, 964-988) and the optional sync markers
__global__ void frame_kernel(EncodeArgs a) {
    if (*a.error) return;
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    const bool stitched = a.mode == ZS_MODE_STITCHED;
    uint32_t* out32 = reinterpret_cast<uint32_t*>(a.out);
    if (c >= a.n_chunks) return;
    // Z_SYNC_FLUSH marker after each chunk: empty stored block 000 + pad + 00 00 ff ff
    if (stitched && (c + 1 == a.n_chunks ? (a.flags & ZS_FLAG_NOT_LAST) != 0 : (a.flags & ZS_FLAG_SYNC) != 0)) {
        uint64_t end = a.out_off[c] + a.out_bits[c];  // marker is the tail of the chunk's bits
        uint64_t p = (end >> 3) - 4;                   // marker ends byte aligned
        a.out[p] = 0; a.out[p + 1] = 0; a.out[p + 2] = 0xff; a.out[p + 3] = 0xff;
    }
    const bool first = stitched ? (c == 0 && !(a.flags & ZS_FLAG_NOT_FIRST)) : true;
    const bool last = stitched ? (c + 1 == a.n_chunks && !(a.flags & ZS_FLAG_NOT_LAST)) : true;
    uint8_t* hp = stitched ? a.out : a.out + a.out_off[c];
    if (first) {
        const int strategy = (int)((a.flags >> 8) & 7u);
        if (a.wrap == ZS_WRAP_ZLIB) {
            // FDICT: deflate() sets it when a dictionary was given (strstart != 0)
            zs_put_zlib_header(hp, a.level, strategy, a.fdict, a.dict_id);
        } else if (a.wrap == ZS_WRAP_GZIP) {
            hp[0] = 0x1f; hp[1] = 0x8b; hp[2] = 8;
            for (int k = 3; k < 8; k++) hp[k] = 0;
            hp[8] = zs_gzip_xfl(a.level, strategy);
            hp[9] = 255;  // OS_CODE of the reference, deflate/constants.ts:30
        }
    }
    if (last && a.wrap != ZS_WRAP_RAW && !(stitched && (a.flags & ZS_FLAG_NOT_FIRST))) {
        uint64_t body_end_bits = stitched ? a.out_off[a.n_chunks] : 0;
        uint8_t* tp;
        uint32_t ck;
        uint64_t isize;
        if (stitched) {
            tp = a.out + ((body_end_bits + 7) >> 3);
            ck = *a.check_total;
            isize = a.in_off[a.n_chunks];
        } else {
            const uint64_t H = wrap_header_bytes(a.wrap, a.fdict);
            tp = a.out + a.out_off[c] + H + ((a.out_bits[c] + 7) >> 3);
            ck = a.checks[c];
            isize = a.in_off[c + 1] - a.in_off[c];
        }
        zs_put_trailer(tp, a.wrap, ck, isize);
    }
    (void)out32;
}

__global__ void count_blocks_kernel(const uint32_t* nblk, uint32_t n, zs_deflate_result* result, const uint32_t* check_total) {
    __shared__ uint32_t s[256];
    uint32_t acc = 0;
    for (uint32_t i = threadIdx.x; i < n; i += 256) acc += nblk[i];
    s[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 128; o; o >>= 1) {
        if ((int)threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        result->n_blocks = s[0];
        result->check = check_total ? *check_total : 0u;
    }
}

// K9: OR n_bits of src into dst at bit offset dst_off (dst bits must be zero)
__global__ void bit_concat_kernel(uint32_t* dst32, uint64_t dst_off, const uint8_t* __restrict__ src, uint64_t n_bits) {
    const uint64_t n_words = (n_bits + 31) >> 5;
    const unsigned sh = (unsigned)(dst_off & 31u);
    const uint64_t w0 = dst_off >> 5;
    const uint64_t src_bytes = (n_bits + 7) >> 3;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= n_words; i += (uint64_t)gridDim.x * blockDim.x) {
        // destination word w0+i receives the high part of source word i-1 and the low part of word i
        auto load = [&](uint64_t k) -> uint32_t {
            if (k >= n_words) return 0u;
            uint32_t v = 0;
            uint64_t b = k << 2;
            for (unsigned q = 0; q < 4 && b + q < src_bytes; q++) v |= (uint32_t)__ldg(src + b + q) << (8 * q);
            if (k + 1 == n_words && (n_bits & 31u)) v &= (1u << (n_bits & 31u)) - 1u;
            return v;
        };
        const uint32_t lo = i ? load(i - 1) : 0u, hi = load(i);
        const uint32_t x = sh ? ((hi << sh) | (lo >> (32 - sh))) : hi;
        if (x) {
            if (i == 0 || i + 1 >= n_words) atomicOr(dst32 + w0 + i, x);
            else dst32[w0 + i] |= x;  // interior words belong to this call alone
        }
    }
}

}  // namespace

static int zs_launch_huff_build(zs_ctx* ctx, const HuffArgs& h, uint64_t nblk_slots) {
    // see the comment at tpb_huff_build_kernel; the environment variables are test hooks
    const bool tpb = getenv("ZS_HUFF_TPB") ? true : getenv("ZS_HUFF_WARP") ? false : nblk_slots > 49152;
    if (tpb) {
        ZS_KERNEL(ctx, "huff_build_kernel", tpb_huff_build_kernel<<<(unsigned)((nblk_slots + 63) / 64), 64, 0, ctx->stream>>>(h));
    } else {
        ZS_KERNEL(ctx, "huff_build_kernel",
                  huff_build_kernel<<<(unsigned)((nblk_slots + kHuffWarps - 1) / kHuffWarps), 32 * kHuffWarps, 0, ctx->stream>>>(h));
    }
    return ZS_OK;
}

int zs_launch_huffman(zs_ctx* ctx, const zs_deflate_plan& p) {
    const uint64_t nblk_slots = (uint64_t)p.n_chunks * p.max_bpc;
    if (nblk_slots == 0) return ZS_OK;
    if (nblk_slots > 0x7fffffffull) {
        snprintf(ctx->err, sizeof(ctx->err), "deflate: too many block slots");
        return ZS_STREAM_ERROR;
    }
    HistArgs hs = {p.n_chunks, p.max_bpc, p.d_in_off, p.d_chunk_nblk, p.d_blk_desc, p.d_sym, p.d_blk_freq};
    ZS_KERNEL(ctx, "histogram_kernel", histogram_kernel<<<(unsigned)nblk_slots, 256, 0, ctx->stream>>>(hs));
    HuffArgs h = {p.n_chunks, p.max_bpc, p.d_chunk_nblk, p.d_blk_desc, p.d_blk_freq, p.d_blk_code, p.d_blk_hdr, p.d_blk_bits,
                  p.level == 0 ? 1 : p.strategy == ZS_STRATEGY_FIXED ? 2 : 0};
    {
        const int rc = zs_launch_huff_build(ctx, h, nblk_slots);
        if (rc != ZS_OK) return rc;
    }

    LayoutArgs l;
    l.n_chunks = p.n_chunks; l.max_bpc = p.max_bpc; l.wrap = p.wrap; l.mode = p.mode; l.flags = p.flags;
    l.in_off = p.d_in_off; l.chunk_nblk = p.d_chunk_nblk; l.blk_hdr = p.d_blk_hdr; l.blk_bits = p.d_blk_bits;
    l.chunk_pr = p.d_chunk_pr; l.out_off = p.d_out_off; l.out_bits = p.d_out_bits; l.out_cap = p.out_cap;
    l.result = p.d_result; l.error = p.d_error; l.check_total = p.d_check_total;
    l.fdict = p.dict != nullptr && p.dict->len > 0;
    const unsigned cgrid = (p.n_chunks + 127) / 128;
    ZS_KERNEL(ctx, "layout_chunks_kernel", layout_chunks_kernel<<<cgrid, 128, 0, ctx->stream>>>(l));
    ZS_KERNEL(ctx, "layout_scan_kernel", layout_scan_kernel<<<1, kScanThreads, 0, ctx->stream>>>(l));
    ZS_KERNEL(ctx, "layout_blocks_kernel", layout_blocks_kernel<<<cgrid, 128, 0, ctx->stream>>>(l));

    ZS_KERNEL(ctx, "zero_output_kernel", zero_output_kernel<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(p.d_out, p.d_result, p.d_error, p.out_cap));

    EncodeArgs e;
    e.n_chunks = p.n_chunks; e.max_bpc = p.max_bpc; e.wrap = p.wrap; e.mode = p.mode; e.flags = p.flags;
    e.in = p.d_in; e.in_off = p.d_in_off; e.sym = p.d_sym; e.chunk_nblk = p.d_chunk_nblk; e.blk_desc = p.d_blk_desc;
    e.blk_code = p.d_blk_code; e.blk_hdr = p.d_blk_hdr; e.blk_abs = p.d_blk_bits; e.out_off = p.d_out_off;
    e.out_bits = p.d_out_bits; e.checks = p.d_checks; e.check_total = p.d_check_total; e.out = p.d_out;
    e.result = p.d_result; e.error = p.d_error; e.level = p.level;
    e.fdict = l.fdict; e.dict_id = p.dict ? p.dict->id : 0u;
    ZS_KERNEL(ctx, "encode_kernel", encode_kernel<<<(unsigned)nblk_slots, kEncThreads, 0, ctx->stream>>>(e));
    ZS_KERNEL(ctx, "frame_kernel", frame_kernel<<<cgrid, 128, 0, ctx->stream>>>(e));
    ZS_KERNEL(ctx, "count_blocks_kernel", count_blocks_kernel<<<1, 256, 0, ctx->stream>>>(p.d_chunk_nblk, p.n_chunks, p.d_result, p.d_check_total));
    return ZS_OK;
}

int zs_launch_bit_concat(zs_ctx* ctx, uint8_t* d_dst, uint64_t dst_bit_off, const uint8_t* d_src, uint64_t n_bits) {
    if (n_bits == 0) return ZS_OK;
    const uintptr_t mis = reinterpret_cast<uintptr_t>(d_dst) & 3u;
    uint32_t* dst32 = reinterpret_cast<uint32_t*>(d_dst - mis);
    const uint64_t off = dst_bit_off + 8ull * mis;
    const uint64_t n_words = (n_bits + 31) >> 5;
    uint64_t blocks = (n_words + 1 + 255) / 256;
    const uint64_t cap = (uint64_t)ctx->sm_count * 16;
    if (blocks > cap) blocks = cap;
    ZS_KERNEL(ctx, "bit_concat_kernel", bit_concat_kernel<<<(unsigned)blocks, 256, 0, ctx->stream>>>(dst32, off, d_src, n_bits));
    return ZS_OK;
}

// Host-buffer entry point for the Huffman stage alone (parity tests): every block is its own chunk.
extern "C" int zs_huffman_blocks(zs_ctx* ctx, const uint32_t* freq, const uint32_t* in_len, uint32_t n, uint32_t* code,
                                 uint32_t* type, uint64_t* bits) {
    if (!ctx) return ZS_STREAM_ERROR;
    cudaSetDevice(ctx->device);
    if (n == 0) return ZS_OK;
    if (!freq || !in_len) return ZS_STREAM_ERROR;
    uint32_t *d_freq = nullptr, *d_nblk = nullptr, *d_desc = nullptr, *d_code = nullptr, *d_hdr = nullptr;
    uint64_t* d_bits = nullptr;
    std::vector<uint32_t> ones(n, 1u), desc((size_t)n * 4, 0u), hdr((size_t)n * kHdrWords);
    for (uint32_t i = 0; i < n; i++) desc[(size_t)i * 4 + 3] = in_len[i];
    int rc = ZS_OK;
    auto fail = [&](cudaError_t e) { if (e != cudaSuccess && rc == ZS_OK) { snprintf(ctx->err, sizeof(ctx->err), "huffman_blocks: %s", cudaGetErrorString(e)); rc = ZS_E_CUDA; } };
    fail(cudaMalloc(&d_freq, (size_t)n * 320 * 4));
    fail(cudaMalloc(&d_nblk, (size_t)n * 4));
    fail(cudaMalloc(&d_desc, (size_t)n * 16));
    fail(cudaMalloc(&d_code, (size_t)n * 320 * 4));
    fail(cudaMalloc(&d_hdr, (size_t)n * kHdrWords * 4));
    fail(cudaMalloc(&d_bits, (size_t)n * 8));
    if (rc == ZS_OK) {
        fail(cudaMemcpyAsync(d_freq, freq, (size_t)n * 320 * 4, cudaMemcpyHostToDevice, ctx->stream));
        fail(cudaMemcpyAsync(d_nblk, ones.data(), (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
        fail(cudaMemcpyAsync(d_desc, desc.data(), (size_t)n * 16, cudaMemcpyHostToDevice, ctx->stream));
        fail(cudaMemsetAsync(d_code, 0, (size_t)n * 320 * 4, ctx->stream));
    }
    if (rc == ZS_OK) {
        HuffArgs h = {n, 1u, d_nblk, d_desc, d_freq, d_code, d_hdr, d_bits, 0};
        rc = zs_launch_huff_build(ctx, h, n);
    }
    if (rc == ZS_OK) {
        if (code) fail(cudaMemcpyAsync(code, d_code, (size_t)n * 320 * 4, cudaMemcpyDeviceToHost, ctx->stream));
        if (bits) fail(cudaMemcpyAsync(bits, d_bits, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
        fail(cudaMemcpyAsync(hdr.data(), d_hdr, (size_t)n * kHdrWords * 4, cudaMemcpyDeviceToHost, ctx->stream));
        fail(cudaStreamSynchronize(ctx->stream));
        if (type && rc == ZS_OK) for (uint32_t i = 0; i < n; i++) type[i] = hdr[(size_t)i * kHdrWords] & 0xffu;
    }
    cudaFree(d_freq); cudaFree(d_nblk); cudaFree(d_desc); cudaFree(d_code); cudaFree(d_hdr); cudaFree(d_bits);
    return rc;
}
