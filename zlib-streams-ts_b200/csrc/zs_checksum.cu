// zs_checksum.cu -- K8: adler32 / crc32 over device buffers with combine-based parallel reduction.
//
// Results must be bit-exact with the reference's adler32 (src/mod/common/adler32.ts:4) and crc32
// (src/mod/common/crc32.ts:26).  The reference walks the buffer serially; here a warp owns one
// segment and reads it in rows of 512 bytes, lane l taking the 16-byte unit l of every row, so that
// each load instruction is one fully coalesced 512-byte access (lane-contiguous slices cost one
// 128-byte line per lane and load, and the L1 wavefront rate -- which the crc tables in shared
// memory share -- capped adler32 at 64 % and crc32 at 27 % of the HBM copy bandwidth).  Both
// checksums are linear enough for that: adler32's b is a position-weighted sum, so a unit at
// position p adds (len - p) * sum(d) - sum(i * d_i); for crc32 a lane's running remainder is
// advanced over the bytes it skips by table lookups (multiplication by a power of x mod P,
// byte-sliced) and the slicing tables are looked up staggered and conflict free (see
// crc32_segments_kernel).  The 32 lane results are merged with the combine algebra (crc: multiply
// by x^(8*bytes_after) mod P).  Algorithmic traffic = 1 read of every input byte.
#include <cstdio>

#include "zs_common.cuh"

namespace {

constexpr uint32_t kPoly = 0xedb88320u;
constexpr uint32_t kAdlerBase = 65521u;

// x^(8 * 2^k) mod P for k = 0..47 (reflected representation), filled by the host at start-up.
__constant__ uint32_t c_xpow[48];
// slicing-by-16 tables [0..15] and the byte-sliced multiplication by x^(8*496) mod P [16..19], built
// on the host once and kept in global memory; [20..22]: x^(8*k), x^(8*256*k), x^(8*65536*k) mod P
// for k = 0..255, which make x^(8*n) two multiplications for n < 2^24.
__device__ uint32_t g_crc_tab[23][256];
// The staggered tables of crc32_segments_kernel: g_crc_tt[e][s] is entry e of the table of byte position s & 31 of a
// 32-byte macro unit (bytes 0-15: a lane's unit of row k, premultiplied by x^(8*512); bytes 16-31: its unit of row
// k + 1), every table stored twice (s and s + 32) so that lane l can address position l + t without wrapping;
// g_crc_s2[j][b]: (b << 8j) * x^(8*1024) mod P, the running remainder carried over two rows.
__device__ uint32_t g_crc_tt[256][64];
__device__ uint32_t g_crc_s2[4][256];

// ---- GF(2)[x] mod P helpers (host + device) -----------------------------------------------------
__host__ __device__ inline uint32_t gf2_mulmod(uint32_t a, uint32_t b) {
    uint32_t p = 0;
    for (;;) {
        if (a & 0x80000000u) p ^= b;
        a <<= 1;
        if (a == 0) break;
        b = (b & 1u) ? ((b >> 1) ^ kPoly) : (b >> 1);
    }
    return p;
}

__device__ inline uint32_t dev_xpow8n(uint64_t nbytes) {
    uint32_t r = 0x80000000u;  // x^0
    for (int k = 0; nbytes != 0 && k < 48; ++k, nbytes >>= 1)
        if (nbytes & 1u) r = gf2_mulmod(r, c_xpow[k]);
    return r;
}

inline uint32_t host_xpow8n(uint64_t nbytes) {
    uint32_t r = 0x80000000u, sq = 0x00800000u;  // x^0, x^8
    while (nbytes) {
        if (nbytes & 1u) r = gf2_mulmod(r, sq);
        sq = gf2_mulmod(sq, sq);
        nbytes >>= 1;
    }
    return r;
}

__device__ inline uint32_t dev_crc_combine(uint32_t c1, uint32_t c2, uint64_t len2) {
    return len2 ? (gf2_mulmod(dev_xpow8n(len2), c1) ^ c2) : c1;
}
__host__ __device__ inline uint32_t adler_combine(uint32_t a1v, uint32_t a2v, uint64_t len2) {
    uint32_t rem = (uint32_t)(len2 % kAdlerBase);
    uint32_t a1 = a1v & 0xffffu, b1 = a1v >> 16, a2 = a2v & 0xffffu, b2 = a2v >> 16;
    uint32_t a = (a1 + a2 + kAdlerBase - 1u) % kAdlerBase;
    uint32_t b = (uint32_t)(((uint64_t)rem * ((a1 + kAdlerBase - 1u) % kAdlerBase) + b1 + b2) % kAdlerBase);
    return (b << 16) | a;
}

// ---- per-segment folds ------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t crc_step16(uint32_t c, const uint4 v, const uint32_t (*T)[256]) {
    const uint32_t a = v.x ^ c;
    return T[15][a & 0xff] ^ T[14][(a >> 8) & 0xff] ^ T[13][(a >> 16) & 0xff] ^ T[12][a >> 24] ^
           T[11][v.y & 0xff] ^ T[10][(v.y >> 8) & 0xff] ^ T[9][(v.y >> 16) & 0xff] ^ T[8][v.y >> 24] ^
           T[7][v.z & 0xff] ^ T[6][(v.z >> 8) & 0xff] ^ T[5][(v.z >> 16) & 0xff] ^ T[4][v.z >> 24] ^
           T[3][v.w & 0xff] ^ T[2][(v.w >> 8) & 0xff] ^ T[1][(v.w >> 16) & 0xff] ^ T[0][v.w >> 24];
}
// remainder * x^(8*496) mod P
__device__ __forceinline__ uint32_t crc_skip496(uint32_t c, const uint32_t (*T)[256]) {
    return T[16][c & 0xff] ^ T[17][(c >> 8) & 0xff] ^ T[18][(c >> 16) & 0xff] ^ T[19][c >> 24];
}
// x^(8*n) mod P
__device__ __forceinline__ uint32_t crc_xpow(uint64_t n, const uint32_t (*T)[256]) {
    if (n >> 24) return dev_xpow8n(n);
    uint32_t r = T[20][n & 0xff];
    if (n >> 8) r = gf2_mulmod(r, T[21][(n >> 8) & 0xff]);
    if (n >> 16) r = gf2_mulmod(r, T[22][n >> 16]);
    return r;
}
__device__ inline uint32_t crc_bytes(const uint8_t* __restrict__ p, unsigned n, const uint32_t (*T)[256]) {
    uint32_t c = 0;
    for (unsigned i = 0; i < n; i++) c = T[0][(c ^ __ldg(p + i)) & 0xffu] ^ (c >> 8);
    return c;
}

// adler32: one warp per segment, grid-stride.
__global__ void __launch_bounds__(256) adler32_segments_kernel(const uint8_t* __restrict__ buf,
                                                                const uint64_t* __restrict__ off,
                                                                const uint64_t* __restrict__ seg_len, uint32_t n,
                                                                uint32_t* __restrict__ out) {
    const unsigned lane = zs_lane();
    const unsigned warps_per_cta = blockDim.x >> 5;
    for (uint64_t seg = (uint64_t)blockIdx.x * warps_per_cta + (threadIdx.x >> 5); seg < n;
         seg += (uint64_t)gridDim.x * warps_per_cta) {
        // segment = [off[seg], off[seg+1]) or, when seg_len is given, seg_len[seg] bytes at off[seg]
        const uint64_t beg = off[seg];
        const uint64_t len = seg_len ? seg_len[seg] : off[seg + 1] - beg;
        const uint8_t* p = buf + beg;
        // head: bytes before the first 16-byte boundary; body: whole 16-byte units; tail: the rest
        uint64_t head = (16u - (unsigned)(reinterpret_cast<uintptr_t>(p) & 15u)) & 15u;
        if (head > len) head = len;
        const uint64_t units = (len - head) >> 4;
        const unsigned tail = (unsigned)(len - head - (units << 4));
        const uint4* q = reinterpret_cast<const uint4*>(p + head);
        // units of this lane: lane, lane + 32, ...; `mine` of them
        const uint64_t mine = units > lane ? (units - lane + 31) >> 5 : 0;
        {
            // A = 1 + sum d_j, B = len + sum (len - j) d_j   (mod 65521)
            uint64_t A = 0, Bq = 0;
            uint32_t w = (uint32_t)((len - head - 16ull * lane) % kAdlerBase);   // (len - position of the unit) mod BASE
            if (units <= lane) w = 0;
            auto unit = [&](const uint4 v) {
                uint32_t s = __dp4a(v.x, 0x01010101u, 0u);
                s = __dp4a(v.y, 0x01010101u, s);
                s = __dp4a(v.z, 0x01010101u, s);
                s = __dp4a(v.w, 0x01010101u, s);
                uint32_t t = __dp4a(v.x, 0x03020100u, 0u);
                t = __dp4a(v.y, 0x07060504u, t);
                t = __dp4a(v.z, 0x0b0a0908u, t);
                t = __dp4a(v.w, 0x0f0e0d0cu, t);
                A += s;
                Bq += (uint64_t)w * s + (kAdlerBase - t);   // t <= 30600 < BASE
                w = w >= 512u ? w - 512u : w + kAdlerBase - 512u;
            };
            uint64_t k = 0;
            for (; k + 4 <= mine; k += 4) {
                const uint4 v0 = __ldg(q + lane + 32 * k), v1 = __ldg(q + lane + 32 * (k + 1));
                const uint4 v2 = __ldg(q + lane + 32 * (k + 2)), v3 = __ldg(q + lane + 32 * (k + 3));
                unit(v0); unit(v1); unit(v2); unit(v3);
            }
            for (; k < mine; k++) unit(__ldg(q + lane + 32 * k));
            if (lane == 0)
                for (uint64_t j = 0; j < head; j++) { const uint32_t d = __ldg(p + j); A += d; Bq += ((len - j) % kAdlerBase) * d; }
            if (lane == 1)
                for (unsigned j = 0; j < tail; j++) { const uint32_t d = __ldg(p + len - tail + j); A += d; Bq += (uint64_t)(tail - j) * d; }
            uint32_t a = (uint32_t)(A % kAdlerBase), b2 = (uint32_t)(Bq % kAdlerBase);
            for (int o = 16; o; o >>= 1) {
                a += __shfl_xor_sync(ZS_FULL_MASK, a, o);
                b2 += __shfl_xor_sync(ZS_FULL_MASK, b2, o);
            }
            if (lane == 0) {
                const uint32_t Av = (1u + a) % kAdlerBase;
                const uint32_t Bv = (uint32_t)(((uint64_t)b2 + len % kAdlerBase) % kAdlerBase);
                out[seg] = (Bv << 16) | Av;
            }
        }
    }
}

// ---- crc32, conflict-free table lookups -------------------------------------------------------------
// Slicing-by-16 costs one table lookup per byte; with every lane of a load instruction indexing the SAME 1 KB
// table at a random entry, a lookup instruction is ~2.8 shared-memory wavefronts (ncu, round 1: L1/TEX 92 %
// busy, 40 % of the HBM copy bandwidth).  Here the lookups of a warp are staggered: a lane takes two units at a
// time (its 16 bytes of row k and of row k + 1, a 32-byte macro unit), rotates them left by `lane` bytes in
// registers, and at step t looks up byte position (t + lane) mod 32 -- so in one instruction the 32 lanes use
// 32 DIFFERENT tables.  The tables are interleaved entry-major (g_crc_tt[e][position]): the table of a position
// lives in one bank, lane l only ever touches bank (l + t) mod 32, and a lookup instruction is exactly one
// wavefront whatever the data is.  crc is linear, so the order in which a lane XORs its 32 contributions does
// not matter; the remainder carried in (two rows = x^(8*1024)) is four more lookups.
constexpr int kCrcThreads = 512;
struct CrcSmem {
    uint32_t TT[256][64];
    uint32_t S2[4][256];
    uint32_t T[23][256];
};

__device__ __forceinline__ uint32_t crc_pair(uint32_t c, const uint4 va, const uint4 vb, const CrcSmem& M, unsigned lane) {
    uint32_t w0 = va.x, w1 = va.y, w2 = va.z, w3 = va.w, w4 = vb.x, w5 = vb.y, w6 = vb.z, w7 = vb.w;
    // rotate the eight words left by lane >> 2 words (barrel: 1, 2, 4) ...
    if (lane & 4u) { const uint32_t t = w0; w0 = w1; w1 = w2; w2 = w3; w3 = w4; w4 = w5; w5 = w6; w6 = w7; w7 = t; }
    if (lane & 8u) { const uint32_t t0 = w0, t1 = w1; w0 = w2; w1 = w3; w2 = w4; w3 = w5; w4 = w6; w5 = w7; w6 = t0; w7 = t1; }
    if (lane & 16u) {
        uint32_t t;
        t = w0; w0 = w4; w4 = t; t = w1; w1 = w5; w5 = t; t = w2; w2 = w6; w6 = t; t = w3; w3 = w7; w7 = t;
    }
    // ... and the bytes by lane & 3
    const unsigned sh = (lane & 3u) * 8u;
    uint32_t d[8];
    d[0] = __funnelshift_r(w0, w1, sh); d[1] = __funnelshift_r(w1, w2, sh); d[2] = __funnelshift_r(w2, w3, sh);
    d[3] = __funnelshift_r(w3, w4, sh); d[4] = __funnelshift_r(w4, w5, sh); d[5] = __funnelshift_r(w5, w6, sh);
    d[6] = __funnelshift_r(w6, w7, sh); d[7] = __funnelshift_r(w7, w0, sh);
    uint32_t acc = M.S2[0][c & 0xffu] ^ M.S2[1][(c >> 8) & 0xffu] ^ M.S2[2][(c >> 16) & 0xffu] ^ M.S2[3][c >> 24];
    const uint32_t* A = &M.TT[0][lane];   // entry e of the table of position lane + t: A[64 * e + t]
#pragma unroll
    for (int t = 0; t < 32; ++t) {
        const unsigned e = (d[t >> 2] >> (8 * (t & 3))) & 0xffu;
#ifdef ZS_DEBUG_HOOKS
        if (64u * e + t + lane >= 256u * 64u) __trap();
#endif
        acc ^= A[64u * e + t];
    }
    return acc;
}

// One warp per segment, grid-stride; same decomposition of a segment as adler32_segments_kernel.
__global__ void __launch_bounds__(kCrcThreads) crc32_segments_kernel(const uint8_t* __restrict__ buf, const uint64_t* __restrict__ off,
                                                                    const uint64_t* __restrict__ seg_len, uint32_t n,
                                                                    uint32_t* __restrict__ out) {
    extern __shared__ __align__(16) unsigned char crc_smem_raw[];
    CrcSmem& M = *reinterpret_cast<CrcSmem*>(crc_smem_raw);
    {
        uint4* dst = reinterpret_cast<uint4*>(&M);
        const uint4* tt = reinterpret_cast<const uint4*>(&g_crc_tt[0][0]);
        const uint4* s2 = reinterpret_cast<const uint4*>(&g_crc_s2[0][0]);
        const uint4* tb = reinterpret_cast<const uint4*>(&g_crc_tab[0][0]);
        constexpr unsigned n_tt = sizeof(M.TT) / 16, n_s2 = sizeof(M.S2) / 16, n_tb = sizeof(M.T) / 16;
        for (unsigned i = threadIdx.x; i < n_tt + n_s2 + n_tb; i += blockDim.x)
            dst[i] = i < n_tt ? tt[i] : i < n_tt + n_s2 ? s2[i - n_tt] : tb[i - n_tt - n_s2];
        __syncthreads();
    }
    const uint32_t (*T)[256] = M.T;
    const unsigned lane = zs_lane();
    const unsigned warps_per_cta = blockDim.x >> 5;
    for (uint64_t seg = (uint64_t)blockIdx.x * warps_per_cta + (threadIdx.x >> 5); seg < n; seg += (uint64_t)gridDim.x * warps_per_cta) {
        const uint64_t beg = off[seg];
        const uint64_t len = seg_len ? seg_len[seg] : off[seg + 1] - beg;
        const uint8_t* p = buf + beg;
        uint64_t head = (16u - (unsigned)(reinterpret_cast<uintptr_t>(p) & 15u)) & 15u;
        if (head > len) head = len;
        const uint64_t units = (len - head) >> 4;
        const unsigned tail = (unsigned)(len - head - (units << 4));
        const uint4* q = reinterpret_cast<const uint4*>(p + head);
        const uint64_t mine = units > lane ? (units - lane + 31) >> 5 : 0;
        uint32_t c = 0;
        uint64_t k = 0;
        // two macro units (four rows) in flight per lane
        for (; k + 4 <= mine; k += 4) {
            const uint4 v0 = __ldg(q + lane + 32 * k), v1 = __ldg(q + lane + 32 * (k + 1));
            const uint4 v2 = __ldg(q + lane + 32 * (k + 2)), v3 = __ldg(q + lane + 32 * (k + 3));
            c = crc_pair(c, v0, v1, M, lane);
            c = crc_pair(c, v2, v3, M, lane);
        }
        if (k + 2 <= mine) {
            const uint4 v0 = __ldg(q + lane + 32 * k), v1 = __ldg(q + lane + 32 * (k + 1));
            c = crc_pair(c, v0, v1, M, lane);
            k += 2;
        }
        if (k < mine) c = crc_step16(crc_skip496(c, T), __ldg(q + lane + 32 * k), T);
        uint32_t r = 0;
        if (mine) {
            const uint64_t end = head + ((lane + 32 * (mine - 1) + 1) << 4);   // end of this lane's last unit
            r = len - end ? gf2_mulmod(crc_xpow(len - end, T), c) : c;
        }
        if (lane == 0 && head) r ^= gf2_mulmod(crc_xpow(len - head, T), crc_bytes(p, (unsigned)head, T));
        if (lane == 1 && tail) r ^= crc_bytes(p + len - tail, tail, T);
        if (lane == 2) r ^= gf2_mulmod(crc_xpow(len, T), 0xffffffffu);   // the 0xffffffff preset: a term in front of the segment
        for (int o = 16; o; o >>= 1) r ^= __shfl_xor_sync(ZS_FULL_MASK, r, o);
        if (lane == 0) out[seg] = ~r;
    }
}

// Fold n per-segment checksums (segment i covers off[i+1]-off[i] bytes) into one value continuing
// from `init`.  Single CTA; each thread folds a contiguous run, then a shared-memory tree.
template <int KIND>
__global__ void __launch_bounds__(1024) checksum_fold_kernel(const uint32_t* __restrict__ part,
                                                             const uint64_t* __restrict__ off, uint32_t n,
                                                             uint32_t init, uint32_t* __restrict__ result) {
    __shared__ uint32_t s_val[1024];
    __shared__ uint64_t s_len[1024];
    const unsigned t = threadIdx.x, nt = blockDim.x;
    const uint32_t per = (n + nt - 1) / nt;
    uint32_t b = t * per, e = b + per;
    if (b > n) b = n;
    if (e > n) e = n;
    uint32_t acc = KIND ? 0u : 1u;
    uint64_t alen = 0;
    for (uint32_t i = b; i < e; ++i) {
        uint64_t l = off[i + 1] - off[i];
        acc = KIND ? dev_crc_combine(acc, part[i], l) : adler_combine(acc, part[i], l);
        alen += l;
    }
    s_val[t] = acc;
    s_len[t] = alen;
    __syncthreads();
    for (unsigned stride = 1; stride < nt; stride <<= 1) {
        if ((t & (2 * stride - 1)) == 0 && t + stride < nt) {
            uint32_t v2 = s_val[t + stride];
            uint64_t l2 = s_len[t + stride];
            s_val[t] = KIND ? dev_crc_combine(s_val[t], v2, l2) : adler_combine(s_val[t], v2, l2);
            s_len[t] += l2;
        }
        __syncthreads();
    }
    if (t == 0) {
        uint32_t v = s_val[0];
        uint64_t l = s_len[0];
        *result = KIND ? dev_crc_combine(init, v, l) : adler_combine(init, v, l);
    }
}

__global__ void make_offsets_kernel(uint64_t* off, uint64_t len, uint64_t piece, uint32_t n) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= n) {
        uint64_t v = i * piece;
        off[i] = v < len ? v : len;
    }
}

// the same for a length that only the device knows (the output of one inflated stream), at most max_len
__global__ void make_offsets_dev_kernel(uint64_t* off, const uint64_t* base, const uint64_t* len, uint64_t piece, uint32_t n) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= n) {
        uint64_t v = i * piece;
        off[i] = *base + (v < *len ? v : *len);
    }
}

bool g_tables_ready[64] = {false};

int ensure_tables(zs_ctx* ctx) {
    if (ctx->device < 64 && g_tables_ready[ctx->device]) return ZS_OK;
    static uint32_t tab[23][256];
    for (unsigned n = 0; n < 256; n++) {
        uint32_t c = n;
        for (int k = 0; k < 8; k++) c = (c & 1u) ? (kPoly ^ (c >> 1)) : (c >> 1);
        tab[0][n] = c;
    }
    for (unsigned n = 0; n < 256; n++)
        for (int k = 1; k < 16; k++) {
            uint32_t p = tab[k - 1][n];
            tab[k][n] = (p >> 8) ^ tab[0][p & 0xffu];
        }
    // multiplication by x^(8*496) mod P, one table per byte of the remainder
    const uint32_t x496 = host_xpow8n(496);
    for (int j = 0; j < 4; j++)
        for (unsigned n = 0; n < 256; n++) tab[16 + j][n] = gf2_mulmod((uint32_t)n << (8 * j), x496);
    for (unsigned n = 0; n < 256; n++) {
        tab[20][n] = host_xpow8n(n);
        tab[21][n] = host_xpow8n((uint64_t)n << 8);
        tab[22][n] = host_xpow8n((uint64_t)n << 16);
    }
    uint32_t xp[48];
    uint32_t sq = 0x00800000u;
    for (int k = 0; k < 48; k++) {
        xp[k] = sq;
        sq = gf2_mulmod(sq, sq);
    }
    static uint32_t tt[256][64], s2[4][256];
    const uint32_t x512 = host_xpow8n(512), x1024 = host_xpow8n(1024);
    for (unsigned e = 0; e < 256; e++)
        for (unsigned sl = 0; sl < 64; sl++) {
            const unsigned pos = sl & 31u;   // byte position inside the macro unit
            tt[e][sl] = pos < 16 ? gf2_mulmod(tab[15 - pos][e], x512) : tab[15 - (pos - 16)][e];
        }
    for (int j = 0; j < 4; j++)
        for (unsigned b = 0; b < 256; b++) s2[j][b] = gf2_mulmod((uint32_t)b << (8 * j), x1024);
    ZS_CUDA_TRY(ctx, cudaMemcpyToSymbolAsync(g_crc_tt, tt, sizeof(tt), 0, cudaMemcpyHostToDevice, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaMemcpyToSymbolAsync(g_crc_s2, s2, sizeof(s2), 0, cudaMemcpyHostToDevice, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaFuncSetAttribute(crc32_segments_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(CrcSmem)));
    ZS_CUDA_TRY(ctx, cudaMemcpyToSymbolAsync(g_crc_tab, tab, sizeof(tab), 0, cudaMemcpyHostToDevice, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaMemcpyToSymbolAsync(c_xpow, xp, sizeof(xp), 0, cudaMemcpyHostToDevice, ctx->stream));
    ZS_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));  // `tab`/`xp` are host temporaries
    if (ctx->device < 64) g_tables_ready[ctx->device] = true;
    return ZS_OK;
}

}  // namespace

uint32_t zs_host_crc32_combine(uint32_t c1, uint32_t c2, uint64_t len2) {
    return len2 ? (gf2_mulmod(host_xpow8n(len2), c1) ^ c2) : c1;
}
uint32_t zs_host_adler32_combine(uint32_t a1, uint32_t a2, uint64_t len2) { return adler_combine(a1, a2, len2); }

int zs_launch_checksum_segments(zs_ctx* ctx, int kind, const uint8_t* d_buf, const uint64_t* d_off,
                                const uint64_t* d_len, uint32_t n, uint32_t* d_out) {
    if (n == 0) return ZS_OK;
    int rc = ensure_tables(ctx);
    if (rc != ZS_OK) return rc;
    unsigned ctas = (n + 7) / 8;
    unsigned cap = (unsigned)ctx->sm_count * 8u;
    if (ctas > cap) ctas = cap;
    if (kind) {
        // 16 warps per CTA share one copy of the tables (91 KB: two CTAs per SM)
        unsigned g = (n + 15) / 16;
        if (g > (unsigned)ctx->sm_count * 2u) g = (unsigned)ctx->sm_count * 2u;
        ZS_KERNEL(ctx, "checksum_segments_kernel",
                  crc32_segments_kernel<<<g, kCrcThreads, sizeof(CrcSmem), ctx->stream>>>(d_buf, d_off, d_len, n, d_out));
    } else {
        ZS_KERNEL(ctx, "checksum_segments_kernel", adler32_segments_kernel<<<ctas, 256, 0, ctx->stream>>>(d_buf, d_off, d_len, n, d_out));
    }
    return ZS_OK;
}

int zs_launch_checksum_fold(zs_ctx* ctx, int kind, const uint32_t* d_part, const uint64_t* d_off, uint32_t n,
                            uint32_t init, uint32_t* d_result) {
    int rc = ensure_tables(ctx);
    if (rc != ZS_OK) return rc;
    if (kind)
        ZS_KERNEL(ctx, "checksum_fold_kernel", checksum_fold_kernel<1><<<1, 1024, 0, ctx->stream>>>(d_part, d_off, n, init, d_result));
    else
        ZS_KERNEL(ctx, "checksum_fold_kernel", checksum_fold_kernel<0><<<1, 1024, 0, ctx->stream>>>(d_part, d_off, n, init, d_result));
    return ZS_OK;
}

// Whole-buffer checksum: cut into 64 KiB pieces (one warp each), then fold.
// Checksum of d_buf[*d_base .. *d_base + *d_len), *d_len <= max_len: 64 KiB pieces in parallel, then the fold.
int zs_launch_checksum_stream(zs_ctx* ctx, int kind, const uint8_t* d_buf, const uint64_t* d_base, const uint64_t* d_len,
                              uint64_t max_len, uint32_t* d_result) {
    const uint64_t piece = 65536;
    uint64_t n64 = (max_len + piece - 1) / piece;
    if (n64 == 0) n64 = 1;
    if (n64 > 0xfffffff0ull) {
        snprintf(ctx->err, sizeof(ctx->err), "checksum: buffer too large");
        return ZS_STREAM_ERROR;
    }
    const uint32_t n = (uint32_t)n64;
    uint64_t* d_off = (uint64_t*)zs_scratch_get(ctx, SCR_CK_OFF, (size_t)(n + 1) * sizeof(uint64_t));
    uint32_t* d_part = (uint32_t*)zs_scratch_get(ctx, SCR_CK_PART, (size_t)n * sizeof(uint32_t));
    if (!d_off || !d_part) return ZS_MEM_ERROR;
    ZS_KERNEL(ctx, "make_offsets_dev_kernel", make_offsets_dev_kernel<<<(n + 1 + 255) / 256, 256, 0, ctx->stream>>>(d_off, d_base, d_len, piece, n));
    int rc = zs_launch_checksum_segments(ctx, kind, d_buf, d_off, nullptr, n, d_part);
    if (rc != ZS_OK) return rc;
    return zs_launch_checksum_fold(ctx, kind, d_part, d_off, n, kind ? 0u : 1u, d_result);
}

int zs_launch_checksum_whole(zs_ctx* ctx, int kind, const uint8_t* d_buf, uint64_t len, uint32_t init,
                             uint32_t* d_result) {
    const uint64_t piece = 65536;
    uint64_t n64 = (len + piece - 1) / piece;
    if (n64 == 0) n64 = 1;
    if (n64 > 0xfffffff0ull) {
        snprintf(ctx->err, sizeof(ctx->err), "checksum: buffer too large");
        return ZS_STREAM_ERROR;
    }
    uint32_t n = (uint32_t)n64;
    uint64_t* d_off = (uint64_t*)zs_scratch_get(ctx, SCR_CK_OFF, (size_t)(n + 1) * sizeof(uint64_t));
    uint32_t* d_part = (uint32_t*)zs_scratch_get(ctx, SCR_CK_PART, (size_t)n * sizeof(uint32_t));
    if (!d_off || !d_part) return ZS_MEM_ERROR;
    ZS_KERNEL(ctx, "make_offsets_kernel", make_offsets_kernel<<<(n + 1 + 255) / 256, 256, 0, ctx->stream>>>(d_off, len, piece, n));
    int rc = zs_launch_checksum_segments(ctx, kind, d_buf, d_off, nullptr, n, d_part);
    if (rc != ZS_OK) return rc;
    return zs_launch_checksum_fold(ctx, kind, d_part, d_off, n, init, d_result);
}
