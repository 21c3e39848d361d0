// zs_inflate_common.cuh -- pieces shared by the warp-per-stream inflate kernel (zs_inflate.cu), the
// thread-per-stream kernel (zs_inflate_tps.cu), the segment-parallel decoder of one stream (zs_inflate_par.cu)
// and the inflate index (zs_inflate_index.cu): decode-table entries and their lookup, the warp-parallel table
// construction, the bit reader, the dynamic block header, the stream setup, wrapper header, trailer and result
// record of a batch stream, and walk_blocks, the warp-uniform block walk behind the segment-parallel passes and
// the index extract.
//
// The decode tables have the layout of the reference's inflate_table (src/mod/inflate/inftrees.ts:62-307):
// a root table of `root` bits whose entries are symbols (replicated for shorter codes) or pointers to
// sub-tables, entry = op << 24 | bits << 16 | val (src/mod/inflate/utils.ts:51-56).  What is computed is the
// same table; HOW it is computed is not the reference's serial walk over the sorted symbols: a warp builds it
// in parallel from the canonical code of every symbol (see build_table_warp).
#pragma once
#include "zs_common.cuh"

namespace zsinf {

constexpr int kEnoughLens = 852;
constexpr int kEnoughDists = 592;
constexpr int kEnoughDists9 = 594;
constexpr unsigned kWin = 32768;   // the window of a deflate stream (deflate64's is not used by the block walk)

// detail codes -> reference messages (zs_inflate_message, zs_inflate.cu)
enum {
    D_NONE = 0, D_HEADER_CHECK, D_METHOD, D_WINDOW, D_HDR_FLAGS, D_HDR_CRC, D_BLOCK_TYPE, D_STORED_LEN,
    D_TOO_MANY, D_TOO_MANY_9, D_CODE_LENGTHS, D_BIT_REPEAT, D_NO_EOB, D_LITLEN_SET, D_DIST_SET, D_LITLEN_CODE,
    D_DIST_CODE, D_TOO_FAR, D_DATA_CHECK, D_LENGTH_CHECK
};

#define E_OP(e) ((e) >> 24)
#define E_BITS(e) (((e) >> 16) & 0xffu)
#define E_VAL(e) ((e) & 0xffffu)
#define E_PACK(op, bits, val) (((uint32_t)(op) << 24) | ((uint32_t)(bits) << 16) | (uint32_t)(val))

struct WarpArena {
    uint32_t codes[kEnoughLens + kEnoughDists9];
    uint16_t lens[320];
    uint32_t scratch[48];   // table construction: counts / first codes / running ranks per code length
};

struct FixedTables {
    uint32_t len[512];
    uint32_t dist[32];
};

// ---- base / extra tables for length and distance symbols (inflate/constants.ts:8-45) -------------
__device__ __forceinline__ void len_sym(unsigned idx, bool d64, unsigned& base, unsigned& op) {
    // idx = symbol - 257
    if (idx < 28) {
        unsigned eb = idx < 8 ? 0u : (idx - 4u) >> 2;
        base = 3u + (idx < 8 ? idx : ((4u + (idx & 3u)) << eb));
        op = (d64 ? 128u : 16u) + eb;
    } else if (idx == 28) {
        base = d64 ? 3u : 258u;
        op = d64 ? 144u : 16u;
    } else {
        base = 0;
        op = 64u;  // invalid code marker (the reference stores 73/200 resp. 72/78: bit 64 set)
    }
}
__device__ __forceinline__ void dist_sym(unsigned idx, bool d64, unsigned& base, unsigned& op) {
    if (idx < 30) {
        unsigned eb = idx < 4 ? 0u : (idx - 2u) >> 1;
        base = 1u + (idx < 4 ? idx : ((2u + (idx & 1u)) << eb));
        op = (d64 ? 128u : 16u) + eb;
    } else if (d64) {
        base = idx == 30 ? 32769u : 49153u;
        op = 142u;
    } else {
        base = 0;
        op = 64u;
    }
}

// type 0: code-length code, 1: literal/length, 2: distance
__device__ __forceinline__ uint32_t table_entry(unsigned sym, unsigned nbits, int type, bool d64) {
    if (type == 0) return E_PACK(0, nbits, sym);
    if (type == 1) {
        if (sym < 256) return E_PACK(0, nbits, sym);
        if (sym == 256) return E_PACK(96, nbits, 0);
        unsigned base, op;
        len_sym(sym - 257, d64, base, op);
        return E_PACK(op, nbits, base);
    }
    unsigned base, op;
    dist_sym(sym, d64, base, op);
    return E_PACK(op, nbits, base);
}

// Decode table for `codes` symbols with code lengths lens[] (0 = unused), built by the whole warp.
// Returns 0 ok, -1 invalid set (over-subscribed or incomplete, inftrees.ts:104-143), 1 not enough table
// space (the ENOUGH bounds, inftrees.ts:214-217,263-266); *index advances by the space used, *bits receives
// the root bits.  All lanes get the same return value and outputs.
//
// Canonical Huffman: the code of a symbol is first_code[len] + (its rank among the symbols of that length),
// so every symbol can place its own entries.  Steps: (1) length counts with shared-memory atomics; (2) the
// per-length first codes and the validity tests, 15 steps, computed redundantly by every lane; (3) ranks by a
// stable counting pass, 32 symbols at a time (match_any on the length + a running count per length); (4)
// codes longer than `root` first vote the size of their sub-table into the root slot they share (atomicMax of
// len - root: for a complete code the deepest code under a root prefix is what inflate_table's `curr` search
// arrives at), a scan over the root slots in code order hands out the sub-table offsets -- the order in which
// the reference creates them -- and (5) every symbol writes its replicated entries.
static __device__ __noinline__ int build_table_warp(int type, const uint16_t* lens, unsigned codes, uint32_t* table, unsigned* bits,
                                             uint32_t* scratch, unsigned* index, bool d64) {
    const unsigned lane = zs_lane();
    uint32_t* cnt = scratch;          // [16] symbols per code length
    uint32_t* run = scratch + 16;     // [16] symbols of that length ranked so far
    if (lane < 16) { cnt[lane] = 0; run[lane] = 0; }
    __syncwarp();
    for (unsigned s = lane; s < codes; s += 32) atomicAdd(&cnt[lens[s]], 1u);
    __syncwarp();
    uint32_t* first = scratch + 32;   // [16] first canonical code of every length (MSB first)
    unsigned mx = 0, mn = 16;
    int left = 1;
    bool over = false;
    {
        unsigned code = 0;
#pragma unroll
        for (unsigned len = 1; len <= 15; len++) {
            const unsigned c = cnt[len];
            if (c) { mx = len; if (mn == 16) mn = len; }
            left = (left << 1) - (int)c;
            if (left < 0) over = true;
            code <<= 1;
            if (lane == len) first[len] = code;
            code += c;
        }
    }
    __syncwarp();
    unsigned root = *bits;
    if (root > mx) root = mx;
    if (mx == 0) {
        if (d64) return -1;
        // no codes at all: two invalid-code entries (inftrees.ts:113-123)
        if (lane < 2) table[*index + lane] = E_PACK(64, 1, 0);
        __syncwarp();
        *index += 2;
        *bits = 1;
        return 0;
    }
    if (root < mn) root = mn;
    if (over) return -1;
    if (left > 0 && (type == 0 || mx != 1)) return -1;
    const unsigned base = *index;
    const unsigned root_size = 1u << root;
    const unsigned enough = type == 1 ? (unsigned)kEnoughLens : (d64 ? (unsigned)kEnoughDists9 : (unsigned)kEnoughDists);
    // (type 0 never exceeds its 7-bit root table)
    if (type != 0 && (d64 ? root_size >= enough : root_size > enough)) return 1;

    // the root table starts as "invalid code" (what the reference leaves in the unused slot of an
    // incomplete one-code set, inftrees.ts:279-300); slots shared by long codes start at 0 for the vote
    const bool has_long = mx > root;
    for (unsigned e = lane; e < root_size; e += 32) table[base + e] = has_long ? 0u : E_PACK(64, 1, 0);
    __syncwarp();

    // pass A: ranks -> canonical codes; long codes vote their sub-table size
    for (unsigned s0 = 0; has_long && s0 < codes; s0 += 32) {
        const unsigned s = s0 + lane;
        const unsigned len = s < codes ? lens[s] : 0u;
        const unsigned peers = __match_any_sync(ZS_FULL_MASK, len);
        if (len > root) {
            const unsigned code = first[len] + run[len] + __popc(peers & zs_lanemask_lt());
            const unsigned rev = __brev(code) >> (32u - len);
            atomicMax(&table[base + (rev & (root_size - 1u))], len - root);
        }
        __syncwarp();
        if (len && (peers >> lane) == 1u) run[len] += __popc(peers);   // the highest lane of the group
        __syncwarp();
    }
    // sub-table offsets in the order of the codes (MSB-first value of the root prefix)
    unsigned used = root_size;
    if (has_long) {
        for (unsigned p0 = 0; p0 < root_size; p0 += 32) {
            const unsigned p = p0 + lane;
            const unsigned slot = base + (__brev(p) >> (32u - root));
            const unsigned c = p < root_size ? table[slot] : 0u;
            const unsigned size = c ? 1u << c : 0u;
            unsigned incl = size;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned v = __shfl_up_sync(ZS_FULL_MASK, incl, o);
                if ((int)lane >= o) incl += v;
            }
            if (c) table[slot] = E_PACK(c, root, used + incl - size);
            else if (p < root_size) table[slot] = E_PACK(64, 1, 0);
            used += __shfl_sync(ZS_FULL_MASK, incl, 31);
        }
        __syncwarp();
        if (type != 0 && (d64 ? used >= enough : used > enough)) return 1;
    }
    if (lane < 16) run[lane] = 0;
    __syncwarp();
    // pass B: every symbol writes its entries
    for (unsigned s0 = 0; s0 < codes; s0 += 32) {
        const unsigned s = s0 + lane;
        const unsigned len = s < codes ? lens[s] : 0u;
        const unsigned peers = __match_any_sync(ZS_FULL_MASK, len);
        if (len) {
            const unsigned code = first[len] + run[len] + __popc(peers & zs_lanemask_lt());
            const unsigned rev = __brev(code) >> (32u - len);
            if (len <= root) {
                const uint32_t here = table_entry(s, len, type, d64);
                for (unsigned e = rev; e < root_size; e += 1u << len) table[base + e] = here;
            } else {
                const uint32_t ptr = table[base + (rev & (root_size - 1u))];
                const unsigned sub_bits = E_OP(ptr), sub_len = len - root;
                const uint32_t here = table_entry(s, sub_len, type, d64);
                uint32_t* sub = table + base + E_VAL(ptr);
                for (unsigned e = rev >> root; e < (1u << sub_bits); e += 1u << sub_len) sub[e] = here;
            }
        }
        __syncwarp();
        if (len && (peers >> lane) == 1u) run[len] += __popc(peers);
        __syncwarp();
    }
    // (an incomplete set is a single one-bit code here: its other slot keeps the invalid-code marker of the
    // initialisation, with the bit count the reference writes, inftrees.ts:279-300)
    *index = base + used;
    *bits = root;
    return 0;
}

// ---- bit reader over a global buffer ------------------------------------------------------------
struct BitReader {
    const uint8_t* base;
    uint64_t pos, end, safe_end;
    uint64_t hold;
    unsigned bits;
    // empty, at byte p of [b, e); safe_end as for zs_ld32 (the readable words, which may reach past e)
    __device__ __forceinline__ void open(const uint8_t* b, uint64_t p, uint64_t e, uint64_t se) {
        base = b; pos = p; end = e; safe_end = se; hold = 0; bits = 0;
    }
    // drop the first k < 8 bits of a just opened reader; false when the byte that holds them is not there
    __device__ __forceinline__ bool skip(unsigned k) {
        if (k == 0) return true;
        if (!need(8)) return false;
        drop(k);
        return true;
    }
    __device__ __forceinline__ void refill() {
        if (bits <= 32) {
            if (end - pos >= 4) {
                hold |= (uint64_t)zs_ld32(base, pos, safe_end) << bits;
                bits += 32;
                pos += 4;
            } else {
                while (pos < end && bits <= 56) {
                    hold |= (uint64_t)__ldg(base + pos) << bits;
                    bits += 8;
                    pos++;
                }
            }
        }
    }
    __device__ __forceinline__ bool need(unsigned n) {
        if (bits < n) refill();
        return bits >= n;
    }
    __device__ __forceinline__ unsigned peek(unsigned n) const { return (unsigned)hold & ((1u << n) - 1u); }
    __device__ __forceinline__ void drop(unsigned n) { hold >>= n; bits -= n; }
    __device__ __forceinline__ unsigned take(unsigned n) { unsigned v = peek(n); drop(n); return v; }
    __device__ __forceinline__ void align_byte() { drop(bits & 7u); }
    // rewind so that `pos` is the next unread byte and the bit buffer is empty (call when byte aligned)
    __device__ __forceinline__ void unload() { pos -= bits >> 3; hold = 0; bits = 0; }
    // lane 0 read ahead on its own: everybody takes over its state
    __device__ __forceinline__ void from_lane0() {
        pos = __shfl_sync(ZS_FULL_MASK, pos, 0);
        hold = __shfl_sync(ZS_FULL_MASK, hold, 0);
        bits = __shfl_sync(ZS_FULL_MASK, bits, 0);
    }
};

// One symbol's entry of a decode table: the root entry for the low bits of `hold` or, where that points to a
// sub-table, the entry there; `used` receives the bits of the code.  A literal/length root entry is a pointer
// when its op is non-zero with no bit of 0xf0 set; a distance root entry is never op 0, so the test is one
// compare shorter.
template <bool kLitLen>
__device__ __forceinline__ uint32_t table_lookup(const uint32_t* table, unsigned mask, uint64_t hold, unsigned& used) {
    uint32_t here = table[(unsigned)hold & mask];
    used = E_BITS(here);
    if ((!kLitLen || E_OP(here)) && (E_OP(here) & 0xf0u) == 0) {
        const uint32_t first = here;
        here = table[E_VAL(first) + (((unsigned)hold >> E_BITS(first)) & ((1u << E_OP(first)) - 1u))];
        used = E_BITS(first) + E_BITS(here);
    }
    return here;
}

// ---- one stream of a batch (inflate_kernel, inflate_tps_kernel) --------------------------------------

// The reader over stream sidx's input, its output capacity and its preset dictionary (none: dict_len = 0).
// (The output pointer, a.d_out + a.d_out_off[sidx], is formed by the kernel: formed here, it changed how
// inflate_kernel's fast loop computes the addresses of its match copies.)
__device__ __forceinline__ void open_stream(const zs_inflate_args& a, uint64_t sidx, uint64_t safe_end, BitReader& br,
                                            uint64_t& cap, const uint8_t*& dict, uint64_t& dict_len) {
    br.open(a.d_in, a.d_in_off[sidx], a.d_in_off[sidx + 1], safe_end);
    cap = a.d_out_off[sidx + 1] - a.d_out_off[sidx];
    dict = nullptr;
    dict_len = 0;
    if (a.d_dict && a.d_dict_rng) {
        dict = a.d_dict + a.d_dict_rng[2 * sidx];
        dict_len = a.d_dict_rng[2 * sidx + 1] - a.d_dict_rng[2 * sidx];
    }
}

__device__ __forceinline__ uint32_t crc_bitwise(uint32_t crc, unsigned byte) {
    crc ^= byte;
    for (int k = 0; k < 8; k++) crc = (crc & 1u) ? (0xedb88320u ^ (crc >> 1)) : (crc >> 1);
    return crc;
}

// Wrapper header: HEAD..HCRC / DICTID of inflate() (inflate.ts:377-593).  wrap: bit 0 zlib, bit 1 gzip.
// A bad or truncated header sets status (and detail).  FDICT: decoding goes on when the stream's dictionary
// was given (a non-empty range: no deflater sets FDICT for an empty one) and its adler32 (*dict_adler) equals DICTID -- inflateSetDictionary after Z_NEED_DICT,
// inflate.ts:1220-1249 -- and stops with ZS_NEED_DICT otherwise.  tflags: 1 zlib trailer, 2 gzip trailer.
__device__ __forceinline__ void read_wrapper_header(BitReader& br, int wrap, int& status, int& detail, unsigned& tflags,
                                                    const uint32_t* dict_adler) {
    if (!br.need(16)) {
        status = ZS_BUF_ERROR;
    } else {
        unsigned h = br.peek(16);
        if ((wrap & 2) && h == 0x8b1fu) {
            uint32_t hcrc = crc_bitwise(crc_bitwise(0xffffffffu, 0x1f), 0x8b);
            br.drop(16);
            // FLAGS
            if (!br.need(16)) status = ZS_BUF_ERROR;
            unsigned flg = 0;
            if (status == ZS_OK) {
                unsigned w = br.take(16);
                flg = w >> 8;
                if ((w & 0xff) != 8) { status = ZS_DATA_ERROR; detail = D_METHOD; }
                else if (w & 0xe000) { status = ZS_DATA_ERROR; detail = D_HDR_FLAGS; }
                hcrc = crc_bitwise(crc_bitwise(hcrc, w & 0xff), w >> 8);
            }
            // TIME(4) XFL OS
            for (int k = 0; k < 6 && status == ZS_OK; k++) {
                if (!br.need(8)) status = ZS_BUF_ERROR;
                else hcrc = crc_bitwise(hcrc, br.take(8));
            }
            if (status == ZS_OK && (flg & 4)) {  // FEXTRA
                unsigned xlen = 0;
                if (!br.need(16)) status = ZS_BUF_ERROR;
                else {
                    xlen = br.take(16);
                    hcrc = crc_bitwise(crc_bitwise(hcrc, xlen & 0xff), xlen >> 8);
                }
                while (status == ZS_OK && xlen--) {
                    if (!br.need(8)) status = ZS_BUF_ERROR;
                    else hcrc = crc_bitwise(hcrc, br.take(8));
                }
            }
            for (int which = 0; which < 2 && status == ZS_OK; which++) {  // FNAME, FCOMMENT
                if (!(flg & (which ? 16 : 8))) continue;
                for (;;) {
                    if (!br.need(8)) { status = ZS_BUF_ERROR; break; }
                    unsigned c = br.take(8);
                    hcrc = crc_bitwise(hcrc, c);
                    if (c == 0) break;
                }
            }
            if (status == ZS_OK && (flg & 2)) {  // FHCRC
                if (!br.need(16)) status = ZS_BUF_ERROR;
                else if (br.take(16) != ((~hcrc) & 0xffffu)) { status = ZS_DATA_ERROR; detail = D_HDR_CRC; }
            }
            tflags = 2;
        } else if (!(wrap & 1) || (((h & 0xff) << 8) + (h >> 8)) % 31) {
            status = ZS_DATA_ERROR; detail = D_HEADER_CHECK;
        } else if ((h & 0xf) != 8) {
            status = ZS_DATA_ERROR; detail = D_METHOD;
        } else if (((h >> 4) & 0xf) + 8 > 15) {
            status = ZS_DATA_ERROR; detail = D_WINDOW;
        } else {
            br.drop(16);
            tflags = 1;
            if (h & 0x2000) {  // FDICT: DICTID follows (big-endian)
                if (!br.need(32)) status = ZS_BUF_ERROR;
                else {
                    const uint32_t id = __byte_perm((uint32_t)br.hold, 0, 0x0123);
                    br.drop(32);
                    if (!dict_adler || *dict_adler != id) status = ZS_NEED_DICT;
                }
            }
        }
    }
}

// Trailer: CHECK / LENGTH (inflate.ts:1006-1037), read when the blocks ended well (status ZS_OK, which
// becomes ZS_STREAM_END).  check / isize receive the stored values; inflate_verify_kernel compares them.
__device__ __forceinline__ void read_trailer(BitReader& br, unsigned tflags, int& status, uint32_t& check, uint32_t& isize) {
    if (status == ZS_OK) {
        br.align_byte();
        if (tflags) {
            if (!br.need(32)) status = ZS_BUF_ERROR;
            else {
                uint32_t w = (uint32_t)br.hold;
                br.drop(32);
                check = tflags == 1 ? __byte_perm(w, 0, 0x0123) : w;
            }
            if (status == ZS_OK && tflags == 2) {
                if (!br.need(32)) status = ZS_BUF_ERROR;
                else { isize = (uint32_t)br.hold; br.drop(32); }
            }
        }
        if (status == ZS_OK) status = ZS_STREAM_END;
    }
}

// The per-stream result record.  A Z_BUF_ERROR with output space left means the input ran dry: the reference
// has pulled every available byte by then (PULLBYTE, inflate.ts:1147-1158).  A known difference: on a Z_BUF_ERROR
// with the output full, the count leaves out the whole bytes still in the bit buffer, while the reference's total_in
// keeps the bytes it pulled for the symbol that did not fit.
__device__ __forceinline__ void store_result(const zs_inflate_args& a, uint64_t sidx, const BitReader& br, uint64_t in_start,
                                             uint64_t op, uint64_t cap, int status, int detail, unsigned tflags,
                                             uint32_t check, uint32_t isize) {
    a.d_out_len[sidx] = op;
    const uint64_t used_in = (status == ZS_BUF_ERROR && op < cap) ? br.end - in_start : br.pos - (br.bits >> 3) - in_start;
    if (a.d_in_used) a.d_in_used[sidx] = used_in;
    a.d_status[sidx] = status;
    a.d_detail[sidx] = detail;
    a.d_trailer[2 * sidx] = check;
    a.d_trailer[2 * sidx + 1] = isize;
    a.d_flags[sidx] = (status == ZS_STREAM_END) ? tflags : 0u;
}

static __constant__ uint8_t c_bl_order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

// TABLE / LENLENS / CODELENS of inflate() (inflate.ts:673-835), called by the whole warp with a warp-uniform
// bit reader.  The run-length coded code lengths are a serial chain and are read by lane 0; the three tables
// are built by the warp.  Returns 0 ok, >0 detail code (data error), -1 truncated input; on success the
// reader stands behind the header in every lane.
static __device__ __noinline__ int read_dynamic_header(BitReader& br, WarpArena& A, bool d64, unsigned& lenbits, unsigned& distbits,
                                                unsigned& dist_at) {
    const unsigned lane = zs_lane();
    int rc = 0;
    unsigned nlen = 0, ndist = 0;
    if (lane == 0) {
        if (!br.need(14)) {
            rc = -1;
        } else {
            nlen = br.take(5) + 257;
            ndist = br.take(5) + 1;
            const unsigned ncode = br.take(4) + 4;
            if (nlen > 286 || (!d64 && ndist > 30)) {
                rc = d64 ? D_TOO_MANY_9 : D_TOO_MANY;
            } else {
                unsigned have = 0;
                while (have < ncode) {
                    if (!br.need(3)) { rc = -1; break; }
                    A.lens[c_bl_order[have++]] = (uint16_t)br.take(3);
                }
                while (have < 19) A.lens[c_bl_order[have++]] = 0;
            }
        }
    }
    rc = __shfl_sync(ZS_FULL_MASK, rc, 0);
    if (rc) return rc;
    nlen = __shfl_sync(ZS_FULL_MASK, nlen, 0);
    ndist = __shfl_sync(ZS_FULL_MASK, ndist, 0);
    __syncwarp();
    unsigned idx = 0, cbits = 7;
    if (build_table_warp(0, A.lens, 19, A.codes, &cbits, A.scratch, &idx, d64)) return D_CODE_LENGTHS;
    __syncwarp();
    if (lane == 0) {
        unsigned have = 0;
        const unsigned total = nlen + ndist;
        while (have < total) {
            br.refill();
            const uint32_t here = A.codes[br.peek(cbits)];
            if (E_BITS(here) > br.bits) { rc = -1; break; }
            // (a code-length code without codes has only invalid-code entries of 1 bit and value 0; like the
            // reference, which never tests their op here, the loop reads them as lengths of 0)
            const unsigned v = E_VAL(here);
            if (v < 16) {
                br.drop(E_BITS(here));
                A.lens[have++] = (uint16_t)v;
            } else {
                const unsigned xb = v == 16 ? 2u : v == 17 ? 3u : 7u;
                if (E_BITS(here) + xb > br.bits) { rc = -1; break; }
                br.drop(E_BITS(here));
                unsigned rep_len = 0, rep;
                if (v == 16) {
                    if (have == 0) { rc = D_BIT_REPEAT; break; }
                    rep_len = A.lens[have - 1];
                    rep = 3 + br.take(2);
                } else if (v == 17) {
                    rep = 3 + br.take(3);
                } else {
                    rep = 11 + br.take(7);
                }
                if (have + rep > total) { rc = D_BIT_REPEAT; break; }
                while (rep--) A.lens[have++] = (uint16_t)rep_len;
            }
        }
        if (rc == 0 && A.lens[256] == 0) rc = D_NO_EOB;
    }
    rc = __shfl_sync(ZS_FULL_MASK, rc, 0);
    br.from_lane0();
    if (rc) return rc;
    __syncwarp();
    idx = 0;
    lenbits = 9;
    if (build_table_warp(1, A.lens, nlen, A.codes, &lenbits, A.scratch, &idx, d64)) return D_LITLEN_SET;
    dist_at = idx;
    distbits = 6;
    if (build_table_warp(2, A.lens + nlen, ndist, A.codes, &distbits, A.scratch, &idx, d64)) return D_DIST_SET;
    __syncwarp();
    return 0;
}

// fixedtables (inflate.ts:218-280), built once per CTA by warp 0 with `A` as scratch
__device__ __forceinline__ void build_fixed_tables(FixedTables& F, WarpArena& A, bool d64) {
    const unsigned lane = zs_lane();
    for (unsigned s = lane; s < 288; s += 32) A.lens[s] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
    __syncwarp();
    unsigned bits = 9, idx = 0;
    build_table_warp(1, A.lens, 288, F.len, &bits, A.scratch, &idx, d64);
    __syncwarp();
    A.lens[lane] = 5;
    __syncwarp();
    bits = 5; idx = 0;
    build_table_warp(2, A.lens, 32, F.dist, &bits, A.scratch, &idx, d64);
    __syncwarp();
}

// ---- the block walk of the segment-parallel passes (zs_inflate_par.cu) and the index extract (zs_inflate_index.cu) ----
// A warp walks the deflate blocks (32 KiB window) of a positioned reader in lock-step; the dynamic header is built in
// `A`, the fixed tables are `F`.  What it decodes goes to the sink, whose hooks the whole warp calls with warp-uniform
// arguments:
//   bool at_block(bit, last)   a block boundary at input bit `bit`, before the next header (last: the block that ended
//                              there was the final one); true stops the walk
//   bool full()                tested at every boundary and before every symbol; true stops the walk, mid-block too
//   int stored(pos, n)         the n bytes of a stored block at input byte pos: 0, or a code that ends the walk
//   void literal(byte)
//   int match(len, dist)       0, or a code that ends the walk
// The walk synchronises nothing: each sink has the __syncwarp()s its own writes need.  Returns 0 when the sink stopped
// it, a detail code on a data error (or the sink's code), -1 when the input ran out or the last block ended first.
template <class Sink>
__device__ __forceinline__ int walk_blocks(BitReader& br, WarpArena& A, const FixedTables& F, Sink& s) {
    for (bool last = false;;) {
        if (s.at_block(br.pos * 8 - br.bits, last) || s.full()) return 0;
        if (last || !br.need(3)) return -1;
        last = br.take(1) != 0;
        const unsigned type = br.take(2);
        const uint32_t* lcode;
        const uint32_t* dcode;
        unsigned lenbits, distbits;
        if (type == 1) {
            lcode = F.len; dcode = F.dist; lenbits = 9; distbits = 5;
        } else if (type == 2) {
            unsigned dist_at = 0;
            lenbits = distbits = 0;
            if (const int rc = read_dynamic_header(br, A, false, lenbits, distbits, dist_at)) return rc;
            lcode = A.codes; dcode = A.codes + dist_at;
        } else if (type == 0) {
            br.align_byte();
            if (!br.need(32)) return -1;
            const unsigned w = (unsigned)br.hold;
            if ((w & 0xffffu) != ((w >> 16) ^ 0xffffu)) return D_STORED_LEN;
            br.drop(32);
            br.unload();
            const uint64_t n = w & 0xffffu;
            if (n > br.end - br.pos) return -1;
            if (const int rc = s.stored(br.pos, n)) return rc;
            br.pos += n;
            continue;
        } else {
            return D_BLOCK_TYPE;
        }
        const unsigned lmask = (1u << lenbits) - 1u, dmask = (1u << distbits) - 1u;
        for (;;) {
            if (s.full()) return 0;
            br.refill();
            unsigned used;
            uint32_t here = table_lookup<true>(lcode, lmask, br.hold, used);
            if (used > br.bits) return -1;
            const unsigned lop = E_OP(here);
            if (lop == 0) {
                br.drop(used);
                s.literal(E_VAL(here));
                continue;
            }
            if (lop & 32) { br.drop(used); break; }
            if (lop & 64) return D_LITLEN_CODE;
            unsigned xb = lop & 15u;
            if (used + xb > br.bits) return -1;
            br.drop(used);
            const unsigned len = E_VAL(here) + br.take(xb);
            br.refill();
            here = table_lookup<false>(dcode, dmask, br.hold, used);
            if (used > br.bits) return -1;
            if (E_OP(here) & 64) return D_DIST_CODE;
            xb = E_OP(here) & 15u;
            if (used + xb > br.bits) return -1;
            br.drop(used);
            if (const int rc = s.match(len, E_VAL(here) + br.take(xb))) return rc;
        }
    }
}

// walk_blocks from bit `bit` of in[0, in_len) (8-byte aligned, readable to in_len rounded up to 8)
template <class Sink>
__device__ __forceinline__ int walk_blocks_at(const uint8_t* in, uint64_t in_len, uint64_t bit, WarpArena& A, const FixedTables& F,
                                              Sink& s) {
    BitReader br;
    br.open(in, bit >> 3, in_len, (in_len + 7) & ~7ull);
    return br.skip((unsigned)(bit & 7u)) ? walk_blocks(br, A, F, s) : -1;
}

}  // namespace zsinf
