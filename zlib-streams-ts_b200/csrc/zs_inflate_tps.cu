// zs_inflate_tps.cu -- K6/K7 for batches of MANY independent streams: one THREAD per stream.
//
// Same contract as inflate_kernel (zs_inflate.cu): bit-exact with the reference's inflate() called as
// inflate(strm, Z_FINISH) on a whole stream -- inflate_fast (src/mod/inflate/inffast.ts:5),
// inflate_table (inftrees.ts:62), block / header / trailer modes (inflate.ts:332-1100), including
// raw deflate64 -- same output, total_in / total_out, return code and message.
//
// Why a second kernel: symbol decoding is serial inside a stream.  The warp-per-stream kernel spends
// a full warp instruction per scalar decode step (31 of 32 lanes redundant), which bounds it near
// 60 warp instructions per symbol.  With one stream per lane the same instruction decodes 32
// streams (minus divergence), which is what a batch of 1 M x 4 KiB gzip records wants
// (BASELINE.json configs[3]).  The price is table memory: 32 streams per warp cannot each hold the
// reference's 852+594-entry lookup tables, so the tables here are canonical-code tables
// (per code length: left-justified limit and symbol base; symbols sorted by code) -- 640 bytes per
// stream, interleaved by lane in shared memory so that equal indices of different lanes never
// conflict.  The verdicts of inflate_table (over-subscribed / incomplete sets) are reproduced from
// the same length counts; decode results are identical because both describe the same canonical
// code.  The dispatcher (zs_launch_inflate) picks this kernel for >= 32768 streams.
#include <cstdio>

#include "zs_inflate_common.cuh"

namespace {

using namespace zsinf;

// Per-thread table layout.  Shared memory per stream decides how many warps an SM holds (the kernel is
// latency-bound: 7 warps per SM with 928 bytes per stream, 11 with 640), so the sorted symbols are
// bytes: a literal/length symbol is its low byte plus "index >= thr[length]" as bit 8 -- inside one code
// length the symbols are sorted, so those >= 256 sit at the end of the group.
// 16-bit units (index i of lane l lives at w[i * 32 + l]):
constexpr int T_LLIM = 0;        // [16] left-justified exclusive code limit per length (literal/length)
constexpr int T_LBASE = 16;      // [16] symbol index base per length
constexpr int T_DLIM = 32;
constexpr int T_DBASE = 48;
constexpr int T_LTHR = 64;       // [16] first index of each length group whose symbol is >= 256
constexpr int T_LENS = 80;       // 320 code lengths, 4 bits each -> 80 units
constexpr int T_UNITS = 160;
// bytes (index i of lane l lives at b[i * 32 + l]):
constexpr int T_LSYM = 0;        // 288 literal/length symbols sorted by code (low byte)
constexpr int T_DSYM = 288;      // 32 distance symbols sorted by code
constexpr int T_BYTES = 320;
constexpr int kArenaBytes = T_UNITS * 64 + T_BYTES * 32;   // per warp
constexpr int kWarpsPerCta = 1;

struct Tab {
    uint16_t* w;  // warp arena + lane
    uint8_t* b;   // byte region of the warp arena + lane
    __device__ __forceinline__ uint16_t& at(int i) const { return w[i * 32]; }
    __device__ __forceinline__ uint8_t& sym(int i) const { return b[i * 32]; }
    __device__ __forceinline__ unsigned len_get(unsigned i) const { return (w[(T_LENS + (i >> 2)) * 32] >> ((i & 3u) * 4u)) & 15u; }
    __device__ __forceinline__ void len_set(unsigned i, unsigned v) const {
        uint16_t& x = w[(T_LENS + (i >> 2)) * 32];
        const unsigned sh = (i & 3u) * 4u;
        x = (uint16_t)((x & ~(15u << sh)) | (v << sh));
    }
};

// Canonical tables from code lengths lens[first .. first+n): the verdicts of inflate_table
// (inftrees.ts:88-143).  type 0 CODES, 1 LENS, 2 DISTS.  Returns 0 ok, -1 invalid set.
// Output: lim[1..15], base[1..15] (16-bit units at t_lim / t_base), sorted symbols at t_sym, *minlen.
__device__ int build_canon(const Tab& T, unsigned first, unsigned n, int type, bool d64, int t_sym, int t_lim, int t_base,
                           unsigned* minlen) {
    // counts per length (kept in lim[] while building), sort cursors in base[]
    for (int l = 0; l <= 15; l++) T.at(t_lim + l) = 0;
    for (unsigned i = 0; i < n; i++) T.at(t_lim + T.len_get(first + i))++;
    int mx = 15;
    while (mx >= 1 && T.at(t_lim + mx) == 0) mx--;
    if (mx == 0) {
        if (d64) return -1;                       // PARAMS_9._createTableWhenNoCodes = false
        for (int l = 1; l <= 15; l++) { T.at(t_lim + l) = 0; T.at(t_base + l) = 0; }
        *minlen = 1;                              // every code is invalid (inftrees.ts:113-123)
        return 0;
    }
    int left = 1;
    for (int l = 1; l <= 15; l++) {
        left <<= 1;
        left -= (int)T.at(t_lim + l);
        if (left < 0) return -1;                  // over-subscribed
    }
    if (left > 0 && (type == 0 || mx != 1)) return -1;   // incomplete set
    unsigned off = 0;
    for (int l = 1; l <= 15; l++) { T.at(t_base + l) = (uint16_t)off; off += T.at(t_lim + l); if (type == 1) T.at(T_LTHR + l) = 0; }
    for (unsigned i = 0; i < n; i++) {
        const unsigned l = T.len_get(first + i);
        if (l) {
            T.sym(t_sym + T.at(t_base + l)++) = (uint8_t)i;
            if (type == 1 && i < 256) T.at(T_LTHR + l)++;   // literals of this length, for now
        }
    }
    unsigned code = 0;
    off = 0;
    unsigned mn = 0;
    for (int l = 1; l <= 15; l++) {
        const unsigned cnt = T.at(t_lim + l);
        if (cnt && !mn) mn = (unsigned)l;
        T.at(t_lim + l) = (uint16_t)((code + cnt) << (15 - l));   // 0x8000 at most
        T.at(t_base + l) = (uint16_t)(off - code);                 // modulo 2^16, used modulo 2^16
        if (type == 1) T.at(T_LTHR + l) = (uint16_t)(off + T.at(T_LTHR + l));
        off += cnt;
        code = (code + cnt) << 1;
    }
    *minlen = mn ? mn : 1;
    return 0;
}

// The 15 left-justified limits of one code, two per 32-bit register.  They are non-decreasing in the
// code length, so the length of the code at the top of `v` is 1 + #(limits <= v): eight
// SIMD-in-word compares instead of a loop of dependent shared-memory loads.
struct LimSet {
    uint32_t p[8];   // p[k] = limit[2k+1] | limit[2k+2] << 16 ; limit[16] := 0xffff (never <= v)
    __device__ __forceinline__ void load(const Tab& T, int t_lim) {
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const uint32_t lo = T.at(t_lim + 2 * k + 1);
            const uint32_t hi = k < 7 ? (uint32_t)T.at(t_lim + 2 * k + 2) : 0xffffu;
            p[k] = lo | (hi << 16);
        }
    }
    __device__ __forceinline__ unsigned length_of(unsigned v) const {   // 1..16 (16 = invalid code)
        const uint32_t vv = v | (v << 16);
        unsigned m = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) m += __popc(__vcmpleu2(p[k], vv));
        return 1u + (m >> 4);
    }
};

// Decode one symbol: returns its index in the sorted symbol table (or -1 invalid code) and its length.
__device__ __forceinline__ int decode_sym(const Tab& T, uint64_t hold, int t_sym, int t_lim, int t_base, unsigned minlen,
                                          unsigned* nbits) {
    const unsigned v = __brev((unsigned)hold) >> 17;   // 15 bits, first stream bit on top
    unsigned l = minlen;
    while (l <= 15 && v >= T.at(t_lim + (int)l)) l++;
    *nbits = l;
    if (l > 15) return -1;
    const unsigned idx = (unsigned)(uint16_t)(T.at(t_base + (int)l) + (v >> (15 - l)));
    return (int)T.sym(t_sym + (int)idx);   // code-length code: symbols 0..18
}
// the same with the limits held in registers; kLitLen adds bit 8 of a literal/length symbol
template <bool kLitLen>
__device__ __forceinline__ int decode_sym_fast(const Tab& T, const LimSet& L, uint64_t hold, int t_sym, int t_base,
                                               unsigned* nbits) {
    const unsigned v = __brev((unsigned)hold) >> 17;
    const unsigned l = L.length_of(v);
    *nbits = l;
    if (l > 15) return -1;
    const unsigned idx = (unsigned)(uint16_t)(T.at(t_base + (int)l) + (v >> (15 - l)));
    unsigned sym = T.sym(t_sym + (int)idx);
    if (kLitLen && idx >= T.at(T_LTHR + (int)l)) sym |= 256u;
    return (int)sym;
}

// len_sym / dist_sym (zs_inflate_common.cuh) in the form this kernel needs: extra bits and an invalid flag
// instead of a table op, which made the kernel 16 SASS instructions longer when decoded from the op.
__device__ __forceinline__ void len_base(unsigned idx, bool d64, unsigned& base, unsigned& xb, bool& invalid) {
    invalid = false;
    if (idx < 28) {
        xb = idx < 8 ? 0u : (idx - 4u) >> 2;
        base = 3u + (idx < 8 ? idx : ((4u + (idx & 3u)) << xb));
    } else if (idx == 28) {
        base = d64 ? 3u : 258u;
        xb = d64 ? 16u : 0u;
    } else {
        base = 0; xb = 0; invalid = true;
    }
}
__device__ __forceinline__ void dist_base(unsigned idx, bool d64, unsigned& base, unsigned& xb, bool& invalid) {
    invalid = false;
    if (idx < 30) {
        xb = idx < 4 ? 0u : (idx - 2u) >> 1;
        base = 1u + (idx < 4 ? idx : ((2u + (idx & 1u)) << xb));
    } else if (d64) {
        base = idx == 30 ? 32769u : 49153u;
        xb = 14;
    } else {
        base = 0; xb = 0; invalid = true;
    }
}

__global__ void __launch_bounds__(32 * kWarpsPerCta) inflate_tps_kernel(zs_inflate_args a) {
    __shared__ __align__(16) uint8_t s_tab[kWarpsPerCta][kArenaBytes];
    const unsigned lane = zs_lane();
    Tab T;
    T.w = reinterpret_cast<uint16_t*>(s_tab[threadIdx.x >> 5]) + lane;
    T.b = s_tab[threadIdx.x >> 5] + T_UNITS * 64 + lane;
    const bool d64 = a.deflate64 != 0;
    const uint64_t in_total = a.d_in_off[a.n];
    const uint64_t safe_end = (in_total + 7) & ~7ull;

    for (uint64_t sidx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; sidx < a.n; sidx += (uint64_t)gridDim.x * blockDim.x) {
        BitReader br;
        uint64_t cap, dict_len;
        const uint8_t* dict;
        open_stream(a, sidx, safe_end, br, cap, dict, dict_len);
        const uint64_t in_start = br.pos;
        uint8_t* out = a.d_out + a.d_out_off[sidx];
        uint64_t op = 0;
        int status = ZS_OK, detail = D_NONE;
        unsigned tflags = 0;
        uint32_t t_check = 0, t_isize = 0;

        if (a.wrap) read_wrapper_header(br, a.wrap, status, detail, tflags, a.d_dict_adler && dict_len ? a.d_dict_adler + sidx : nullptr);

        // ---- blocks ----
        bool last = false;
        while (status == ZS_OK && !last) {
            if (!br.need(3)) { status = ZS_BUF_ERROR; break; }
            last = br.take(1) != 0;
            const unsigned type = br.take(2);
            unsigned lmin = 1, dmin = 1;
            if (type == 0) {
                br.align_byte();
                if (!br.need(32)) { status = ZS_BUF_ERROR; break; }
                const unsigned w = (unsigned)br.hold;
                if ((w & 0xffffu) != ((w >> 16) ^ 0xffffu)) { status = ZS_DATA_ERROR; detail = D_STORED_LEN; break; }
                br.drop(32);
                br.unload();
                const uint64_t n = w & 0xffffu, avail_in = br.end - br.pos, avail_out = cap - op;
                uint64_t c = n < avail_in ? n : avail_in;
                if (c > avail_out) c = avail_out;
                for (uint64_t j = 0; j < c; j++) out[op + j] = __ldg(a.d_in + br.pos + j);
                br.pos += c;
                op += c;
                if (c < n) { status = ZS_BUF_ERROR; break; }
                continue;
            } else if (type == 1) {
                for (unsigned i = 0; i < 288; i++) T.len_set(i, i < 144 ? 8u : i < 256 ? 9u : i < 280 ? 7u : 8u);
                for (unsigned i = 0; i < 32; i++) T.len_set(288 + i, 5u);
                build_canon(T, 0, 288, 1, d64, T_LSYM, T_LLIM, T_LBASE, &lmin);
                build_canon(T, 288, 32, 2, d64, T_DSYM, T_DLIM, T_DBASE, &dmin);
            } else if (type == 2) {
                // TABLE / LENLENS / CODELENS (inflate.ts:673-835)
                if (!br.need(14)) { status = ZS_BUF_ERROR; break; }
                const unsigned nlen = br.take(5) + 257, ndist = br.take(5) + 1, ncode = br.take(4) + 4;
                if (nlen > 286 || (!d64 && ndist > 30)) { status = ZS_DATA_ERROR; detail = d64 ? D_TOO_MANY_9 : D_TOO_MANY; break; }
                for (unsigned i = 0; i < 19; i++) T.len_set(i, 0);
                bool trunc = false;
                for (unsigned i = 0; i < ncode; i++) {
                    if (!br.need(3)) { trunc = true; break; }
                    T.len_set(c_bl_order[i], br.take(3));
                }
                if (trunc) { status = ZS_BUF_ERROR; break; }
                unsigned cmin = 1;
                // the code-length code uses the literal/length table slots, which are rebuilt below
                if (build_canon(T, 0, 19, 0, d64, T_LSYM, T_LLIM, T_LBASE, &cmin)) { status = ZS_DATA_ERROR; detail = D_CODE_LENGTHS; break; }
                // the 19 lengths are consumed: lens[] can now receive the nlen + ndist lengths
                unsigned have = 0;
                const unsigned total = nlen + ndist;
                unsigned prev_len = 0;
                int err = 0;
                while (have < total) {
                    br.refill();
                    unsigned nb;
                    const int sym = decode_sym(T, br.hold, T_LSYM, T_LLIM, T_LBASE, cmin, &nb);
                    if (sym < 0) { err = nb > br.bits ? -1 : D_CODE_LENGTHS; break; }
                    if (nb > br.bits) { err = -1; break; }
                    if (sym < 16) {
                        br.drop(nb);
                        T.len_set(have++, (unsigned)sym);
                        prev_len = (unsigned)sym;
                    } else {
                        const unsigned xb = sym == 16 ? 2u : sym == 17 ? 3u : 7u;
                        if (nb + xb > br.bits) { err = -1; break; }
                        br.drop(nb);
                        unsigned rep_len = 0, rep;
                        if (sym == 16) {
                            if (have == 0) { err = D_BIT_REPEAT; break; }
                            rep_len = prev_len;
                            rep = 3 + br.take(2);
                        } else if (sym == 17) {
                            rep = 3 + br.take(3);
                        } else {
                            rep = 11 + br.take(7);
                        }
                        if (have + rep > total) { err = D_BIT_REPEAT; break; }
                        while (rep--) T.len_set(have++, rep_len);
                        prev_len = rep_len;
                    }
                }
                if (err < 0) { status = ZS_BUF_ERROR; break; }
                if (err > 0) { status = ZS_DATA_ERROR; detail = err; break; }
                if (T.len_get(256) == 0) { status = ZS_DATA_ERROR; detail = D_NO_EOB; break; }
                if (build_canon(T, 0, nlen, 1, d64, T_LSYM, T_LLIM, T_LBASE, &lmin)) { status = ZS_DATA_ERROR; detail = D_LITLEN_SET; break; }
                if (build_canon(T, nlen, ndist, 2, d64, T_DSYM, T_DLIM, T_DBASE, &dmin)) { status = ZS_DATA_ERROR; detail = D_DIST_SET; break; }
            } else {
                status = ZS_DATA_ERROR; detail = D_BLOCK_TYPE; break;
            }

            // ---- symbols ----
            LimSet LL, DL;
            LL.load(T, T_LLIM);
            DL.load(T, T_DLIM);
            for (;;) {
                br.refill();
                unsigned nb;
                const int sym = decode_sym_fast<true>(T, LL, br.hold, T_LSYM, T_LBASE, &nb);
                if (sym < 0) {
                    if (nb > br.bits && br.bits < 15) status = ZS_BUF_ERROR;
                    else { status = ZS_DATA_ERROR; detail = D_LITLEN_CODE; }
                    break;
                }
                if (nb > br.bits) { status = ZS_BUF_ERROR; break; }
                if (sym < 256) {
                    if (op >= cap) { status = ZS_BUF_ERROR; break; }
                    br.drop(nb);
                    out[op++] = (uint8_t)sym;
                    continue;
                }
                if (sym == 256) { br.drop(nb); break; }
                unsigned base, xb;
                bool invalid;
                len_base((unsigned)sym - 257u, d64, base, xb, invalid);
                if (invalid) { status = ZS_DATA_ERROR; detail = D_LITLEN_CODE; break; }
                if (nb + xb > br.bits) { status = ZS_BUF_ERROR; break; }
                br.drop(nb);
                const unsigned len = base + br.take(xb);
                br.refill();
                const int ds = decode_sym_fast<false>(T, DL, br.hold, T_DSYM, T_DBASE, &nb);
                if (ds < 0) {
                    if (nb > br.bits && br.bits < 15) status = ZS_BUF_ERROR;
                    else { status = ZS_DATA_ERROR; detail = D_DIST_CODE; }
                    break;
                }
                if (nb > br.bits) { status = ZS_BUF_ERROR; break; }
                dist_base((unsigned)ds, d64, base, xb, invalid);
                if (invalid) { status = ZS_DATA_ERROR; detail = D_DIST_CODE; break; }
                if (nb + xb > br.bits) { status = ZS_BUF_ERROR; break; }
                br.drop(nb);
                const uint64_t dist = base + br.take(xb);
                if (op >= cap) { status = ZS_BUF_ERROR; break; }
                if (dist > op + dict_len) { status = ZS_DATA_ERROR; detail = D_TOO_FAR; break; }
                uint64_t c = len;
                if (c > cap - op) c = cap - op;
                // forward copy (overlap-safe like inffast.ts:165-190); the part of the source that lies
                // before the output comes from the preset dictionary.  A byte-by-byte loop would pay
                // one L2 round trip per byte (the loaded byte feeds the next store, and just-written
                // output is not in L1), so bytes move in groups of 8 loads followed by 8 stores when
                // the distance allows, and short periods are replicated from a register.
                uint64_t j = 0;
                if (dist > op) {
                    const uint64_t from_dict = dist - op;
                    const uint64_t nd = from_dict < c ? from_dict : c;
                    for (; j < nd; j++) out[op + j] = __ldg(dict + dict_len - from_dict + j);
                }
                if (dist >= 8) {
                    for (; j + 8 <= c; j += 8) {
                        uint8_t b[8];
#pragma unroll
                        for (int q = 0; q < 8; q++) b[q] = out[op + j + q - dist];
#pragma unroll
                        for (int q = 0; q < 8; q++) out[op + j + q] = b[q];
                    }
                    if (j < c) {
                        uint8_t b[8];
#pragma unroll
                        for (int q = 0; q < 8; q++) b[q] = (j + q < c) ? out[op + j + q - dist] : (uint8_t)0;
#pragma unroll
                        for (int q = 0; q < 8; q++)
                            if (j + q < c) out[op + j + q] = b[q];
                        j = c;
                    }
                } else if (j < c) {
                    // period < 8: load the period once, then store from the register
                    uint64_t pat = 0;
                    const unsigned d = (unsigned)dist;
                    for (unsigned q = 0; q < d; q++) pat |= (uint64_t)out[op + j - dist + q] << (8 * q);
                    unsigned ph = 0;
                    for (; j < c; j++) {
                        out[op + j] = (uint8_t)(pat >> (8 * ph));
                        ph = ph + 1 == d ? 0 : ph + 1;
                    }
                }
                op += c;
                if (c < len) { status = ZS_BUF_ERROR; break; }
            }
        }

        read_trailer(br, tflags, status, t_check, t_isize);
        store_result(a, sidx, br, in_start, op, cap, status, detail, tflags, t_check, t_isize);
    }
}

}  // namespace

int zs_launch_inflate_tps(zs_ctx* ctx, const zs_inflate_args& a) {
    if (a.n == 0) return ZS_OK;
    unsigned ctas = (a.n + 31) / 32;
    const unsigned cap = (unsigned)ctx->sm_count * (227u * 1024u / (unsigned)(kArenaBytes * kWarpsPerCta)) * 4u;
    if (ctas > cap) ctas = cap;
    ZS_KERNEL(ctx, "inflate_tps_kernel", inflate_tps_kernel<<<ctas, 32 * kWarpsPerCta, 0, ctx->stream>>>(a));
    return ZS_OK;
}
