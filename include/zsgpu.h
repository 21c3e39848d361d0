/*
 * zsgpu.h -- C ABI of libzsgpu, the B200-native (sm_100a) deflate / inflate / checksum engine that
 * sits behind the zlib-streams-ts API.
 *
 * The reference (zlib-streams-ts, pure TypeScript) has no FFI seam; this header IS the seam a
 * maintainer binds from a Node-API addon (see INTEGRATION.md).  Every entry point names the
 * reference interface it replaces (paths relative to the reference tree).  Plain C types only:
 * no CUDA or torch types appear in the signatures (a CUDA stream is passed as void*).
 *
 * There is no CPU fallback: every data-path call runs CUDA kernels and fails with ZS_E_CUDA if no
 * device is usable.
 *
 * Conventions
 *  - "_dev" entry points take DEVICE pointers, enqueue work on the context's stream and do not
 *    synchronise; results (offsets, lengths, statuses) are device arrays.
 *  - the un-suffixed batch entry points take HOST pointers, copy in, run the same kernels, copy
 *    out and synchronise.
 *  - status codes are the reference's Z_* values (src/mod/common/constants.ts:21-29).
 */
#ifndef ZSGPU_H
#define ZSGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- return / status codes: src/mod/common/constants.ts:21-29 ---- */
#define ZS_OK 0
#define ZS_STREAM_END 1
#define ZS_NEED_DICT 2
#define ZS_ERRNO (-1)
#define ZS_STREAM_ERROR (-2)
#define ZS_DATA_ERROR (-3)
#define ZS_MEM_ERROR (-4)
#define ZS_BUF_ERROR (-5)
#define ZS_VERSION_ERROR (-6)
#define ZS_E_CUDA (-100) /* not a zlib code: CUDA runtime failure, see zs_last_error() */

/* ---- flush values: src/mod/common/constants.ts:13-19 ---- */
#define ZS_NO_FLUSH 0
#define ZS_PARTIAL_FLUSH 1
#define ZS_SYNC_FLUSH 2
#define ZS_FULL_FLUSH 3
#define ZS_FINISH 4
#define ZS_BLOCK 5

/* ---- wrappers: the formats of src/mod/streams.ts:220,233 ---- */
#define ZS_WRAP_RAW 0  /* "deflate-raw"  windowBits -15 */
#define ZS_WRAP_ZLIB 1 /* "deflate"      windowBits  15 */
#define ZS_WRAP_GZIP 2 /* "gzip"         windowBits  31 */

/* ---- deflate batch modes ---- */
#define ZS_MODE_INDEPENDENT 0 /* every chunk becomes a complete stream with the wrapper */
#define ZS_MODE_STITCHED 1    /* one stream: chunk bit-streams concatenated at bit granularity */

/* ---- deflate batch flags ---- */
#define ZS_FLAG_PRIME 1u     /* INDEPENDENT: prime each chunk with the <=32 KiB that precede it in the
                                input (deflateSetDictionary, deflate.ts:367); raw wrapper only */
#define ZS_FLAG_NOT_FIRST 2u /* STITCHED: this call is not the first part (no wrapper header) */
#define ZS_FLAG_NOT_LAST 4u  /* STITCHED: not the last part: no BFINAL, no trailer; the part ends with an
                                empty stored block (Z_SYNC_FLUSH marker) so that the next part starts
                                byte aligned (stored blocks are padded relative to the part's first bit) */
#define ZS_FLAG_SYNC 8u      /* STITCHED: end every chunk with an empty stored block (Z_SYNC_FLUSH
                                marker, deflate.ts:945-946) so chunks start byte aligned */

/* strategy (last argument of deflateInit2_, src/mod/common/constants.ts): bits 8..10 of the flags.
 * FILTERED drops matches of length <= 5 at the lazy levels (deflate.ts:1381-1387), HUFFMAN_ONLY emits
 * literals only (deflate_huff, :1525), RLE matches at distance 1 only (deflate_rle, :1450), FIXED never
 * builds dynamic trees (trees.ts:559). */
#define ZS_STRATEGY_DEFAULT 0
#define ZS_STRATEGY_FILTERED 1
#define ZS_STRATEGY_HUFFMAN_ONLY 2
#define ZS_STRATEGY_RLE 3
#define ZS_STRATEGY_FIXED 4
#define ZS_FLAG_STRATEGY(s) (((uint32_t)(s) & 7u) << 8)

typedef struct zs_ctx zs_ctx;
typedef struct zs_inflate_index zs_inflate_index;   /* random access into one stream: see zs_inflate_index_build */

#if defined(__GNUC__)
#define ZS_API __attribute__((visibility("default")))
#else
#define ZS_API
#endif

ZS_API const char* zs_version(void);

/* Create / destroy an engine context bound to CUDA device `device`.  `cuda_stream` is a
 * cudaStream_t (or NULL for a stream owned by the context). */
ZS_API int zs_ctx_create(int device, void* cuda_stream, zs_ctx** out);
ZS_API void zs_ctx_destroy(zs_ctx* ctx);
ZS_API const char* zs_last_error(const zs_ctx* ctx);
ZS_API int zs_ctx_synchronize(zs_ctx* ctx);
/* number of kernel launches issued through this context so far */
ZS_API uint64_t zs_ctx_launch_count(const zs_ctx* ctx);
/* Per-kernel device timing: while enabled every kernel launch is bracketed by CUDA events on the
 * context's stream.  zs_ctx_profile_read synchronises, writes one line "name launches total_ms" per
 * kernel into buf and clears the records. */
ZS_API int zs_ctx_profile(zs_ctx* ctx, int enable);
ZS_API int zs_ctx_profile_read(zs_ctx* ctx, char* buf, uint64_t cap);

/* deflateBound, src/mod/deflate/deflate.ts:615-674 (windowBits 15, memLevel 8) */
ZS_API uint64_t zs_deflate_bound(uint64_t source_len, int wrap);
/* Capacity the batch calls need for `n_chunks` chunks of at most `max_chunk` bytes. */
ZS_API uint64_t zs_deflate_batch_bound(uint64_t total_len, uint32_t n_chunks, uint32_t max_chunk, int wrap, int mode);

/* ---- checksums: src/mod/common/adler32.ts:4, src/mod/common/crc32.ts:26 ---- */
/* kind 0 = adler32, 1 = crc32.  Host-side scalar combine (C zlib semantics; the reference has none). */
ZS_API uint32_t zs_crc32_combine(uint32_t crc1, uint32_t crc2, uint64_t len2);
ZS_API uint32_t zs_adler32_combine(uint32_t adler1, uint32_t adler2, uint64_t len2);
/* Per-segment checksums of n segments [off[i], off[i+1]) of a device buffer; d_out[i] receives the
 * checksum of segment i started from the reference's initial value (adler 1 / crc 0). */
ZS_API int zs_checksum_batch_dev(zs_ctx* ctx, int kind, const uint8_t* d_buf, const uint64_t* d_off, uint32_t n,
                          uint32_t* d_out);
/* Checksum of one device buffer, continuing from `init`; the result is returned to the host. */
ZS_API int zs_checksum_dev(zs_ctx* ctx, int kind, const uint8_t* d_buf, uint64_t len, uint32_t init, uint32_t* result);
/* Host buffer variant: adler32(adler, buf, len) / crc32(crc, buf, len). */
ZS_API int zs_checksum(zs_ctx* ctx, int kind, const uint8_t* buf, uint64_t len, uint32_t init, uint32_t* result);

/* ---- deflate: replaces deflate_fast/deflate_slow/longest_match (deflate.ts:1053-1448), _tr_tally*
 *      (deflate/utils.ts:55-81), build_tree/gen_bitlen/gen_codes/compress_block/_tr_flush_block
 *      (trees.ts) and the header/trailer emission of deflate() (deflate.ts:750-832,964-988) ---- */
typedef struct zs_deflate_result {
    uint64_t total_out_bytes; /* bytes valid in `out` */
    uint64_t total_out_bits;  /* STITCHED: exact bit length of this part (a multiple of 8) */
    uint32_t check;           /* adler32 (zlib) / crc32 (gzip, raw) of this call's whole input */
    uint32_t n_blocks;        /* deflate blocks emitted */
} zs_deflate_result;

/*
 * Chunk i is d_in[d_in_off[i] .. d_in_off[i+1]).  If d_in_off is NULL the input is cut into
 * `chunk_size`-byte chunks (the last one short) and n_chunks must equal ceil(in_len/chunk_size)
 * (or 1 when in_len == 0).  `history` bytes before d_in[0] are readable and may be matched against
 * (STITCHED continuation parts / PRIME).  level 0..9 (-1 = 6), CONFIGURATION_TABLE deflate.ts:86;
 * level 0 stores every chunk as stored blocks (deflate_stored, deflate.ts:1140).
 * Outputs (device): d_out, d_out_off[n_chunks+1] = byte offsets of the streams (INDEPENDENT) or
 * bit offsets of the chunk bit-streams (STITCHED); d_out_bits[n_chunks] = compressed bit length of
 * each chunk; d_checks[n_chunks] (may be NULL) = per-chunk adler32/crc32; d_result = summary.
 */
ZS_API int zs_deflate_batch_dev(zs_ctx* ctx, const uint8_t* d_in, uint64_t in_len, const uint64_t* d_in_off,
                         uint32_t n_chunks, uint32_t chunk_size, uint32_t max_chunk, uint32_t history,
                         int level, int wrap, int mode, uint32_t flags, uint8_t* d_out, uint64_t out_cap,
                         uint64_t* d_out_off, uint64_t* d_out_bits, uint32_t* d_checks,
                         zs_deflate_result* d_result);

/* Host-buffer variant (what the Node-API addon binds for deflateBatch).  in_off may be NULL as
 * above; out_off / out_bits / checks may be NULL.  Returns ZS_OK, ZS_BUF_ERROR (out_cap too
 * small), ZS_STREAM_ERROR (bad arguments) or ZS_E_CUDA. */
ZS_API int zs_deflate_batch(zs_ctx* ctx, const uint8_t* in, uint64_t in_len, const uint64_t* in_off, uint32_t n_chunks,
                     uint32_t chunk_size, int level, int wrap, int mode, uint32_t flags, uint8_t* out,
                     uint64_t out_cap, uint64_t* out_off, uint64_t* out_bits, uint32_t* checks,
                     zs_deflate_result* result);

/* One *part* of a STITCHED stream from HOST buffers (no reference analogue: this is the entry a rank of the
 * multi-GPU split, or a caller feeding a stream piecewise, binds).  The part is cut into `chunk_size`
 * chunks; `history` (<= 32768) bytes before in[0] are readable and matched against, like the window
 * deflate() carries from call to call (deflate.ts:166-236).  flags: ZS_FLAG_NOT_FIRST / ZS_FLAG_NOT_LAST /
 * ZS_FLAG_SYNC / strategy.  A part that is not the last ends with the Z_SYNC_FLUSH marker
 * (deflate.ts:945-946), so parts concatenate byte-wise; the wrapper header comes with the first part, the
 * trailer (deflate.ts:964-988) only when one call holds the whole stream -- otherwise the caller appends
 * it from the combined result->check values (zs_adler32_combine / zs_crc32_combine).  Large parts are
 * pipelined in slices (H2D, kernels and D2H overlap); out_bits[n_chunks] may be NULL. */
ZS_API int zs_deflate_part(zs_ctx* ctx, const uint8_t* in, uint64_t in_len, uint32_t history, uint32_t chunk_size,
                    int level, int wrap, uint32_t flags, uint8_t* out, uint64_t out_cap, uint64_t* out_bits,
                    zs_deflate_result* result);

/* ---- deflate one stream and index it in the same call ----
 * The arguments of zs_deflate_batch_dev / zs_deflate_batch without mode (always ZS_MODE_STITCHED: one stream) and
 * history, with the span of an index (zs_inflate_index_*, below) and the index itself.  The compressed bytes, out_off,
 * out_bits, checks and the result are those zs_deflate_batch_dev / zs_deflate_batch write with ZS_MODE_STITCHED and the
 * same arguments (the host call's slices and their sync markers included): indexing does not change the stream.
 * *index receives the index zs_inflate_index_build makes from that output with window_bits 15 / 31 / -15 (zlib / gzip /
 * raw) and the same span -- header, points and windows alike, with crc32 as the check of a raw stream -- without
 * decoding it: the encoder's block layout gives every block start (DESIGN.md 3.3e), the input is the output before it.
 * flags: the strategy and ZS_FLAG_SYNC.  ZS_FLAG_PRIME, ZS_FLAG_NOT_FIRST, ZS_FLAG_NOT_LAST (a part is not a whole
 * stream), span 0, a null index pointer and whatever the batch call refuses are ZS_STREAM_ERROR; an out_cap too small
 * for the stream is ZS_BUF_ERROR.  *index is NULL unless the call returns ZS_OK.  The calls make host decisions, so they
 * SYNCHRONISE.  The device call writes d_result (device memory) as zs_deflate_batch_dev does; d_in must stay valid and
 * unchanged until it returns (the windows are read from it). */
ZS_API int zs_deflate_indexed_dev(zs_ctx* ctx, const uint8_t* d_in, uint64_t in_len, const uint64_t* d_in_off,
                                  uint32_t n_chunks, uint32_t chunk_size, uint32_t max_chunk, int level, int wrap,
                                  uint32_t flags, uint64_t span, uint8_t* d_out, uint64_t out_cap, uint64_t* d_out_off,
                                  uint64_t* d_out_bits, uint32_t* d_checks, zs_deflate_result* d_result,
                                  zs_inflate_index** index);
/* Host-buffer variant: `result` is host memory, as in zs_deflate_batch. */
ZS_API int zs_deflate_indexed(zs_ctx* ctx, const uint8_t* in, uint64_t in_len, const uint64_t* in_off, uint32_t n_chunks,
                              uint32_t chunk_size, int level, int wrap, uint32_t flags, uint64_t span, uint8_t* out,
                              uint64_t out_cap, uint64_t* out_off, uint64_t* out_bits, uint32_t* checks,
                              zs_deflate_result* result, zs_inflate_index** index);

/* ---- preset dictionary for batch deflate (deflateSetDictionary, deflate.ts:367-424, once for many
 *      records).  Many small records compress far better against a shared dictionary; the batch calls
 *      below compress every chunk as one whole stream that starts from it. ---- */
typedef struct zs_deflate_dict zs_deflate_dict;

/* Copies the dictionary to the context's device and builds the match finder's tables from it once (about
 * 128 KiB of device memory).  Like deflateSetDictionary, only the last 32 KiB of a longer dictionary are
 * used; an empty one is allowed.  Synchronises.  The handle may be used by any context on the same device. */
ZS_API int zs_deflate_dict_create(zs_ctx* ctx, const uint8_t* dict, uint64_t dict_len, zs_deflate_dict** out);
/* DICTID: adler32 of the WHOLE dictionary (what a zlib stream made with it names, and what an inflater
 * compares with the dictionary it is given). */
ZS_API uint32_t zs_deflate_dict_id(const zs_deflate_dict* d);
/* Frees the dictionary (waits for the device).  Destroy it before the context it was created with. */
ZS_API void zs_deflate_dict_destroy(zs_deflate_dict* d);

/* Batch deflate against a prepared dictionary: the arguments of zs_deflate_batch_dev without history and
 * mode.  Every chunk becomes an independent stream compressed as deflateSetDictionary + deflate(Z_FINISH)
 * would: matches reach back into the dictionary's last 32 KiB (in this engine at most 32768 - 1920 bytes
 * before the matching position, as everywhere: DESIGN.md 3.1), and the output of a chunk is byte-identical to
 * zs_deflate_batch_dev with ZS_FLAG_PRIME on a buffer holding the dictionary's last <= 32 KiB followed by the
 * chunk alone.  wrap: ZS_WRAP_RAW, or ZS_WRAP_ZLIB with FDICT set and the 4-byte DICTID after the 2-byte
 * header when the dictionary is not empty (6 + body + 4 bytes per stream; the adler32 trailer covers the
 * chunk alone).  ZS_WRAP_GZIP returns ZS_STREAM_ERROR (deflate.ts:372), as does any flag other than the
 * strategy (PRIME, SYNC, part flags).  Level 0, Z_HUFFMAN_ONLY and Z_RLE produce the same blocks as without
 * the dictionary (only the framing changes).  out_cap: zs_deflate_batch_bound(in_len, n_chunks, max_chunk,
 * wrap, ZS_MODE_INDEPENDENT) + 4 * n_chunks is always enough. */
ZS_API int zs_deflate_batch_dict_dev(zs_ctx* ctx, const zs_deflate_dict* dict, const uint8_t* d_in, uint64_t in_len,
                                     const uint64_t* d_in_off, uint32_t n_chunks, uint32_t chunk_size, uint32_t max_chunk,
                                     int level, int wrap, uint32_t flags, uint8_t* d_out, uint64_t out_cap,
                                     uint64_t* d_out_off, uint64_t* d_out_bits, uint32_t* d_checks,
                                     zs_deflate_result* d_result);
/* Host-buffer variant, sliced and pipelined like zs_deflate_batch (slicing cannot change the output). */
ZS_API int zs_deflate_batch_dict(zs_ctx* ctx, const zs_deflate_dict* dict, const uint8_t* in, uint64_t in_len,
                                 const uint64_t* in_off, uint32_t n_chunks, uint32_t chunk_size, int level, int wrap,
                                 uint32_t flags, uint8_t* out, uint64_t out_cap, uint64_t* out_off, uint64_t* out_bits,
                                 uint32_t* checks, zs_deflate_result* result);

/* Bit-granular stitch (no reference analogue; deflatePrime, deflate.ts:528, is the reference's
 * "insert bits at a bit offset" primitive): OR `n_bits` bits of d_src into d_dst starting at bit
 * `dst_bit_off`.  The destination bits must be zero beforehand. */
ZS_API int zs_bit_concat_dev(zs_ctx* ctx, uint8_t* d_dst, uint64_t dst_bit_off, const uint8_t* d_src, uint64_t n_bits);

/* The Huffman stage alone, for n blocks given by their symbol frequencies: build_tree / gen_bitlen /
 * gen_codes (trees.ts:54-76,167-316), build_bl_tree (:416-432) and the stored / static / dynamic
 * choice of _tr_flush_block (:544-583).  freq[n][320]: 286 literal/length counters at 0.., 30
 * distance counters at 288.. (END_BLOCK is added by the engine); in_len[n]: input bytes of each
 * block, for the stored-block test.  Outputs (each may be NULL): code[n][320] = code | length << 16
 * of the chosen trees, type[n] (0 stored, 1 static, 2 dynamic), bits[n] = block size in bits
 * without alignment padding.  Host buffers; this is what the parity tests compare with the oracle's
 * build_tree. */
ZS_API int zs_huffman_blocks(zs_ctx* ctx, const uint32_t* freq, const uint32_t* in_len, uint32_t n, uint32_t* code,
                      uint32_t* type, uint64_t* bits);

/* ---- inflate: replaces inflate_fast (inffast.ts:5), inflate_table (inftrees.ts:62) and the
 *      block/header/trailer modes of inflate() (inflate.ts:332-1100) for whole streams ---- */
/*
 * Stream i is d_in[d_in_off[i] .. d_in_off[i+1]); its output goes to d_out[d_out_off[i] ..
 * d_out_off[i+1]) (capacity).  window_bits as inflateInit2_ (inflate.ts:174): 15 zlib, -15 raw,
 * 31 gzip, 47 auto-detect zlib/gzip, -16 raw deflate64.  Optional per-stream preset dictionary
 * (inflateSetDictionary inflate.ts:1220-1249): stream i uses d_dict[d_dict_rng[2i] .. d_dict_rng[2i+1]).
 * A raw stream decodes against it directly.  A zlib stream whose header has FDICT decodes against it when
 * the adler32 of the whole range equals the stream's DICTID (inflate -> Z_NEED_DICT -> inflateSetDictionary
 * -> inflate(Z_FINISH)); without a dictionary, or with another one, its status is Z_NEED_DICT.  An empty range
 * is no dictionary (a deflater sets FDICT only for a non-empty one).  Per stream: d_out_len = bytes produced, d_in_used = bytes consumed
 * (total_in), d_checks = adler32/crc32 of the output, d_status = what inflate(strm, Z_FINISH)
 * returns (Z_STREAM_END, Z_DATA_ERROR, Z_BUF_ERROR, Z_NEED_DICT).  d_in_used / d_checks may be NULL.
 */
ZS_API int zs_inflate_batch_dev(zs_ctx* ctx, const uint8_t* d_in, const uint64_t* d_in_off, uint32_t n, int window_bits,
                         uint8_t* d_out, const uint64_t* d_out_off, uint64_t* d_out_len, uint64_t* d_in_used,
                         uint32_t* d_checks, int32_t* d_status, const uint8_t* d_dict,
                         const uint64_t* d_dict_rng);

/* Host-buffer variant (what the addon binds for inflateBatch). `in_total` = in_off[n],
 * out capacity = out_off[n].  dict / dict_rng may be NULL.  A large batch (thousands of streams, >= 64 MiB of
 * input + output) is cut into slices of streams whose copies overlap the kernels of their neighbours; the
 * results are those of the unsliced call.  Pinned host buffers make the copies asynchronous. */
ZS_API int zs_inflate_batch(zs_ctx* ctx, const uint8_t* in, const uint64_t* in_off, uint32_t n, int window_bits,
                     uint8_t* out, const uint64_t* out_off, uint64_t* out_len, uint64_t* in_used, uint32_t* checks,
                     int32_t* status, const uint8_t* dict, const uint64_t* dict_rng, uint64_t dict_total);

/* ONE stream of any length in device memory (d_in 8-byte aligned), sizes given by the host; results stay on
 * the device (asynchronous like the other _dev calls).  This is inflate(strm, Z_FINISH) of
 * src/mod/inflate/inflate.ts:332 for a whole stream -- same output, status, message -- decoded in parallel
 * where the stream has flush points (Z_SYNC_FLUSH / Z_FULL_FLUSH markers, deflate.ts:936-961): the stream is
 * cut at the byte-aligned block boundaries behind the markers, the segments are decoded concurrently against
 * a symbolic 32 KiB window and resolved in order (csrc/zs_inflate_par.cu).  A stream without flush points is
 * cut at dynamic block headers located by search (trusted only when the segment before lands on them bit
 * exact); raw deflate64 (-16) is decoded by one warp.  The host-buffer call zs_inflate_batch with n = 1 and the
 * streaming shim take the same path.  d_dict: optional preset dictionary / earlier output (raw streams, and
 * zlib streams with FDICT as in zs_inflate_batch_dev). */
ZS_API int zs_inflate_stream_dev(zs_ctx* ctx, const uint8_t* d_in, uint64_t in_len, int window_bits, uint8_t* d_out,
                          uint64_t out_cap, uint64_t* d_out_len, uint64_t* d_in_used, uint32_t* d_check,
                          int32_t* d_status, const uint8_t* d_dict, uint64_t dict_len);

/* Message the reference would leave in strm.msg for a detail code (see zs_inflate_last_details). */
ZS_API const char* zs_inflate_message(int detail);
/* Optional: per-stream detail code (index into the reference's message strings) of the last
 * zs_inflate_batch[_dev] call on this context, copied to the host array `detail[n]`. */
ZS_API int zs_inflate_last_details(zs_ctx* ctx, int32_t* detail, uint32_t n);

/* ---- random access into one stream: an index of access points (the method of zlib's examples/zran.c) ----
 * Reading bytes from the middle of a long zlib, gzip or raw deflate stream otherwise means decoding everything before
 * them.  An index records ACCESS POINTS: deflate block starts, each with its input bit, its output offset and the
 * 32 KiB window before it.  A read then decodes from the nearest point at or before it.
 *
 * Block starts are every point where a deflate block begins (what inflate(Z_BLOCK) stops at: data_type & 128 set, the
 * last block not yet seen): input bit total_in * 8 - (bits held) and output offset total_out.  The first is right after
 * the wrapper header.  For a span S >= 1, the access points are, without duplicates, "the first block start, in stream
 * order, whose output offset is >= m" for m = 0, S, 2S, ... with m < out_len; the first block start is always a point.
 * This depends on the stream's block structure and S alone.  Any byte is then at most S plus one block's output after
 * its point.  The window of a point at output offset o is the last min(32768, dict_len + o) bytes of the preset
 * dictionary (when the stream uses one: raw, or zlib with FDICT) followed by out[0, o).
 *
 * The index lives on the device of the context that made it: its point table and n_points windows of up to 32 KiB,
 * with a host copy of the table.  Any context on that device may use it; destroy it before that context.  Only the first
 * gzip member is indexed (zs_gunzip's member table serves multi-member files).  Deflate64 has no index. */
typedef struct zs_inflate_index_info {
    uint64_t in_len, out_len, span, n_points;
    uint32_t check;      /* adler32 (zlib) / crc32 (gzip, raw) of the whole output */
    int32_t window_bits;
} zs_inflate_index_info;
typedef struct zs_inflate_index_result {
    uint64_t out_len;    /* total_out */
    uint64_t in_used;    /* total_in */
    uint32_t check;
    int32_t status;      /* what zs_inflate_stream_dev reports */
    int32_t detail;      /* message code: zs_inflate_message(detail) */
} zs_inflate_index_result;
/* inflate(Z_FINISH) of one stream, exactly as zs_inflate_stream_dev: same output, out_len, in_used, check, status and
 * detail.  When the status is Z_STREAM_END, *out also receives an index of the points above for span `span`; otherwise
 * *out is NULL.  window_bits 15 / -15 / 31 / 47; -16 (deflate64) and span 0 are ZS_STREAM_ERROR.  d_in 8-byte aligned,
 * d_dict optional as in zs_inflate_stream_dev.  Makes host decisions, so it SYNCHRONISES; res is host memory.  After the
 * decode, the stream is walked once more for its block starts: in parallel over the segments the one-stream decoder
 * cut it into, by one warp over the part it decoded serially (DESIGN.md 3.3d). */
ZS_API int zs_inflate_index_build_dev(zs_ctx* ctx, const uint8_t* d_in, uint64_t in_len, int window_bits, uint64_t span,
                                      uint8_t* d_out, uint64_t out_cap, const uint8_t* d_dict, uint64_t dict_len,
                                      zs_inflate_index_result* res, zs_inflate_index** out);
/* Host-buffer variant: copies in, runs zs_inflate_index_build_dev, copies res->out_len bytes out. */
ZS_API int zs_inflate_index_build(zs_ctx* ctx, const uint8_t* in, uint64_t in_len, int window_bits, uint64_t span, uint8_t* out,
                                  uint64_t out_cap, const uint8_t* dict, uint64_t dict_len, zs_inflate_index_result* res,
                                  zs_inflate_index** index);
ZS_API int zs_inflate_index_info_get(const zs_inflate_index* index, zs_inflate_index_info* info);
/* The first min(n_points, max) points into host arrays (either may be NULL), in stream order. */
ZS_API int zs_inflate_index_points(const zs_inflate_index* index, uint64_t* in_bit, uint64_t* out_off, uint64_t max);
/* Serialised index, format version 1, little-endian (synchronises):
 *   offset  0  "ZSIX"
 *           4  u32 version (1)
 *           8  i32 window_bits
 *          12  u32 reserved (0)
 *          16  u64 in_len        24  u64 out_len        32  u64 span
 *          40  u32 check         44  u32 reserved (0)   48  u64 n_points
 *          56  n_points x { u64 in_bit, u64 out_off, u32 win_len, u32 reserved (0) }
 *          then the windows back to back, win_len bytes each, in point order.
 * cap 0: *len receives the size only.  A smaller non-zero cap is ZS_BUF_ERROR. */
ZS_API int zs_inflate_index_export(const zs_inflate_index* index, uint8_t* buf, uint64_t cap, uint64_t* len);
/* Rebuilds an index on the context's device from an export.  Everything is validated before the device is touched:
 * magic, version, window_bits, reserved fields, a length that is exactly header + points + windows, a first point at
 * output offset 0, points strictly increasing in bit and non-decreasing in output, in_bit < 8 * in_len,
 * out_off <= out_len, win_len <= 32768 and consistent with out_off and one dictionary length.  Anything else is
 * ZS_DATA_ERROR (zs_last_error names the check). */
ZS_API int zs_inflate_index_import(zs_ctx* ctx, const uint8_t* buf, uint64_t len, zs_inflate_index** out);
/* Frees the index (waits for the device). */
ZS_API void zs_inflate_index_destroy(zs_inflate_index* index);
/* Range i is the uncompressed bytes [off[i], off[i] + len[i]) of the indexed stream, written to d_out + d_out_off[i].
 * d_got[i] = bytes written; d_status[i] = Z_OK (the whole range), Z_BUF_ERROR (clipped at out_len: got < len) or
 * Z_DATA_ERROR (the input does not decode from a point: a wrong or damaged stream).  On Z_DATA_ERROR got counts the
 * range's bytes before the failure, and zs_inflate_last_details gives the message code per range (0 when the input
 * or the stream ended first).  A range spanning k intervals between points is k work items decoded in parallel.
 * d_in must hold the same stream (8-byte aligned); in_len must equal the index's, else ZS_STREAM_ERROR.  Device
 * arrays; asynchronous like the other _dev calls. */
ZS_API int zs_inflate_index_extract_dev(zs_ctx* ctx, const zs_inflate_index* index, const uint8_t* d_in, uint64_t in_len,
                                        const uint64_t* d_off, const uint64_t* d_len, uint32_t n, uint8_t* d_out,
                                        const uint64_t* d_out_off, uint64_t* d_got, int32_t* d_status);
/* Host-buffer variant (synchronises).  It copies in only the input the ranges need -- from the byte of each range's
 * first point to the byte of the point after its last one, or to in_len, plus the bit reader's read-ahead -- not the
 * whole stream, and copies back only the bytes written.  Every range as clipped must fit: out_off[i] + its bytes <=
 * out_cap, else ZS_STREAM_ERROR. */
ZS_API int zs_inflate_index_extract(zs_ctx* ctx, const zs_inflate_index* index, const uint8_t* in, uint64_t in_len,
                                    const uint64_t* off, const uint64_t* len, uint32_t n, uint8_t* out, uint64_t out_cap,
                                    const uint64_t* out_off, uint64_t* got, int32_t* status);

/* ---- multi-member gzip (RFC 1952 2.2: bgzip / BGZF, `cat a.gz b.gz`, appended archives, this engine's own
 *      INDEPENDENT gzip output): every member in one call ----
 * The result is what the reference's multi-member loop produces (test/inflate/test-multistream.ts:16-79):
 * inflateInit2(31), then inflate(Z_FINISH) on the rest of the input; on Z_STREAM_END inflateReset and go on behind
 * total_in, until the input is used up.  So the call is as strict as that loop: bytes after the last member that do
 * not form a member -- garbage, and zero padding too -- end it with that member's header error ("incorrect header
 * check"), and empty input is Z_BUF_ERROR.  On an error the output holds the members before the failing one and that
 * member's prefix; status / detail / in_used are what inflate() reports for it (in_used counted from the file start).
 * Only gzip members are read; concatenated zlib or raw streams are not members.
 * The members are found on the device (candidate headers, an output plan from their ISIZE fields, a batch decode that
 * must land exactly on the next candidate; DESIGN.md 3.3c); a member that does not, and any member of 128 KiB or more,
 * is decoded alone by the one-stream path of zs_inflate_stream_dev.  The calls make host decisions as they go, so
 * they SYNCHRONISE; `res` and `members` are host memory. */
typedef struct zs_gunzip_result {
    uint64_t out_len;   /* bytes written to out */
    uint64_t in_used;   /* bytes consumed (total_in of the loop) */
    uint64_t n_members; /* members that ended with Z_STREAM_END (always the true count) */
    int32_t status;     /* Z_STREAM_END when every byte belonged to a member, else the failing member's status */
    int32_t detail;     /* message code of the failing member: zs_inflate_message(detail) */
} zs_gunzip_result;
/* One decoded member: where it lies in the input and in the output, and the crc32 of its output.  A BGZF reader
 * builds its .gzi random-access index from these. */
typedef struct zs_gz_member {
    uint64_t in_off, in_len;
    uint64_t out_off, out_len;
    uint32_t crc32;
} zs_gz_member;
/* d_in (8-byte aligned) and d_out are device memory; d_out may be NULL when out_cap is 0.  At most max_members entries go to `members` (may be NULL with
 * max_members 0), in file order.  Returns ZS_OK when the input was processed (its verdict is res->status),
 * ZS_STREAM_ERROR for bad arguments, ZS_MEM_ERROR or ZS_E_CUDA. */
ZS_API int zs_gunzip_dev(zs_ctx* ctx, const uint8_t* d_in, uint64_t in_len, uint8_t* d_out, uint64_t out_cap,
                         zs_gunzip_result* res, zs_gz_member* members, uint64_t max_members);
/* Host-buffer variant: copies in, runs zs_gunzip_dev, copies res->out_len bytes out. */
ZS_API int zs_gunzip(zs_ctx* ctx, const uint8_t* in, uint64_t in_len, uint8_t* out, uint64_t out_cap, zs_gunzip_result* res,
                     zs_gz_member* members, uint64_t max_members);

/* ---- streaming shim: the z_stream protocol of deflate()/inflate() over the batch engine ----
 * Mirrors createDeflateStream/deflateInit2_/deflate/deflateEnd (deflate.ts:80,253,716,991),
 * deflateSetDictionary (:367) and createInflateStream/inflateInit2_/inflate/inflateEnd/
 * inflateSetDictionary/inflateReset (inflate.ts:68,174,332,1187,1220,124).  The counters are the
 * Stream fields of src/mod/common/types.ts:1-15.
 * Scheduling (INTEGRATION.md, section 4): deflate buffers one part (16 MiB) of input; a part that is complete under
 * Z_NO_FLUSH is compressed in the background while the caller feeds the next one, and its output is handed out by
 * later calls, by any flush request or by a call without input.  inflate decodes on every call while a stream has
 * brought less than 64 KiB, on any flush request and on a call without new input; beyond that its decode attempts
 * are paced by what they cost, so a caller that is slower than the decoder still gets one per call and a caller that
 * feeds from memory gets a few large ones.  Both are what the zlib contract allows a Z_NO_FLUSH call to do. */
typedef struct zs_stream {
    const uint8_t* next_in;
    uint64_t avail_in;
    uint64_t total_in;
    uint8_t* next_out;
    uint64_t avail_out;
    uint64_t total_out;
    const char* msg;
    uint32_t adler;
    int32_t data_type;
    void* state; /* opaque */
} zs_stream;

ZS_API int zs_stream_deflate_init(zs_ctx* ctx, zs_stream* strm, int level, int method, int window_bits, int mem_level,
                           int strategy);
ZS_API int zs_stream_deflate_set_dictionary(zs_stream* strm, const uint8_t* dict, uint32_t dict_len);
ZS_API int zs_stream_deflate(zs_stream* strm, int flush);
ZS_API int zs_stream_deflate_end(zs_stream* strm);
/* deflateReset / deflateResetKeep (deflate.ts:444-495), deflateParams (:553-595), deflatePending /
 * deflateUsed (:505-526; the engine never keeps a partial byte between calls: bits = 0). */
ZS_API int zs_stream_deflate_reset(zs_stream* strm);
ZS_API int zs_stream_deflate_params(zs_stream* strm, int level, int strategy);
ZS_API int zs_stream_deflate_pending(zs_stream* strm, uint32_t* pending, int* bits);
/* gzip header fields: GzipHeader of src/mod/common/types.ts:137-151 (zlib's gz_header).
 * deflate side (deflateSetHeader, deflate.ts:497; written by deflate(), :803-921): extra / name /
 * comment are present when their pointer is not NULL (name and comment zero-terminated, extra_len
 * bytes of extra); hcrc != 0 adds the header CRC16; the fields are copied by the call.
 * inflate side (inflateGetHeader, inflate.ts; filled by inflate(), :423-580): the caller's struct is
 * filled while the header is parsed -- up to extra_max / name_max / comm_max bytes into the buffers
 * that are not NULL -- and done becomes 1 (header complete) or -1 (not a gzip stream).  The struct
 * must stay valid until then. */
typedef struct zs_gz_header {
    int32_t text;
    uint32_t time;
    int32_t xflags;
    int32_t os;
    uint8_t* extra;
    uint32_t extra_max;
    uint32_t extra_len;
    uint8_t* name;
    uint32_t name_max;
    uint8_t* comment;
    uint32_t comm_max;
    int32_t hcrc;
    int32_t done;
} zs_gz_header;
ZS_API int zs_stream_deflate_set_header(zs_stream* strm, const zs_gz_header* head);
ZS_API int zs_stream_inflate_get_header(zs_stream* strm, zs_gz_header* head);
ZS_API int zs_stream_inflate_init(zs_ctx* ctx, zs_stream* strm, int window_bits);
ZS_API int zs_stream_inflate_set_dictionary(zs_stream* strm, const uint8_t* dict, uint32_t dict_len);
ZS_API int zs_stream_inflate(zs_stream* strm, int flush);
ZS_API int zs_stream_inflate_reset(zs_stream* strm);
/* inflateReset2, inflate.ts:138-172 */
ZS_API int zs_stream_inflate_reset2(zs_stream* strm, int window_bits);
ZS_API int zs_stream_inflate_end(zs_stream* strm);

#ifdef __cplusplus
}
#endif
#endif /* ZSGPU_H */
