// zlib-streams-gpu.ts -- TypeScript facade: the reference's API names over the Node-API addon.
// NOT compiled in this repository's image (no node / tsc).  A zlib-streams-ts maintainer drops this
// next to src/index.ts (or re-points the exports of src/mod/deflate/index.ts and
// src/mod/inflate/index.ts at it); src/mod/streams.ts then works unchanged because it only talks to
// the four callbacks _createStream/_init/_process/_end (streams.ts:40-45).
/* eslint-disable @typescript-eslint/no-var-requires */
const addon = require("./zsgpu.node");
addon.init(0);

export const Z_OK = 0, Z_STREAM_END = 1, Z_NEED_DICT = 2, Z_STREAM_ERROR = -2, Z_DATA_ERROR = -3, Z_BUF_ERROR = -5;
export const Z_NO_FLUSH = 0, Z_SYNC_FLUSH = 2, Z_FULL_FLUSH = 3, Z_FINISH = 4;

// the reference's Stream carrier, src/mod/common/types.ts:1-15
export interface Stream {
  next_in: Uint8Array; next_in_index: number; avail_in: number; total_in: number;
  next_out: Uint8Array; next_out_index: number; avail_out: number; total_out: number;
  msg: string; _data_type: number; _adler: number; _state: unknown;
}
const EMPTY = new Uint8Array(0);
function createStream(): Stream {
  return { next_in: EMPTY, next_in_index: 0, avail_in: 0, total_in: 0, next_out: EMPTY, next_out_index: 0,
           avail_out: 0, total_out: 0, msg: "", _data_type: 0, _adler: 0, _state: undefined };
}
// the reference's GzipHeader record, src/mod/common/types.ts
export interface GzipHeader {
  _text: number; _time: number; _xflags: number; _os: number; _hcrc: number; _done: number;
  _extra: Uint8Array | null; _extra_max: number; _extra_len: number;
  _name: Uint8Array | null; _name_max: number; _comment: Uint8Array | null; _comm_max: number;
}
type Handle = { h: unknown; which: 0 | 1; gzhead?: GzipHeader };

export const createDeflateStream = createStream;   // deflate.ts:80
export const createInflateStream = createStream;   // inflate.ts:68

export function deflateInit(strm: Stream, level: number): number { return deflateInit2_(strm, level); }   // deflate.ts:238
export function deflateInit2_(strm: Stream, level: number, method = 8, windowBits = 15, memLevel = 8, strategy = 0): number {
  if (!strm) return Z_STREAM_ERROR;                                                                      // deflate.ts:263
  const h = addon.streamNew();
  const rc = addon.deflateInit2(h, level, method, windowBits, memLevel, strategy);
  if (rc === Z_OK) strm._state = { h, which: 0 } as Handle;
  return rc;
}
export function inflateInit(strm: Stream): number { return inflateInit2_(strm, 15); }                    // inflate.ts:74
export function inflateInit2_(strm: Stream, windowBits: number): number {                                // inflate.ts:174
  if (!strm) return Z_STREAM_ERROR;
  const h = addon.streamNew();
  const rc = addon.inflateInit2(h, windowBits);
  if (rc === Z_OK) strm._state = { h, which: 1 } as Handle;
  return rc;
}
function process(strm: Stream, flush: number, which: 0 | 1 | 2): number {
  const st = strm && (strm._state as Handle);
  if (!st || st.which !== (which === 2 ? 0 : which)) return Z_STREAM_ERROR;
  const [rc, used, made, tin, tout, adler] = addon.process(st.h, which, flush, strm.next_in, strm.next_in_index,
    strm.avail_in, strm.next_out, strm.next_out_index, strm.avail_out);
  strm.next_in_index += used; strm.avail_in -= used; strm.next_out_index += made; strm.avail_out -= made;
  strm.total_in = tin; strm.total_out = tout; strm._adler = adler;
  if (st.gzhead && st.gzhead._done === 0) syncGzipHeader(st);
  return rc;
}
function syncGzipHeader(st: Handle): void {
  const head = st.gzhead as GzipHeader;
  const [done, text, time, xflags, os, hcrc, extraLen, extra, name, comment] = addon.inflateHeaderState(st.h);
  if (!done) return;
  head._done = done;              // 1 = header read, -1 = the stream is not gzip
  if (done !== 1) return;
  head._text = text; head._time = time; head._xflags = xflags; head._os = os; head._hcrc = hcrc; head._extra_len = extraLen;
  if (head._extra_max) head._extra = (extra as Uint8Array).subarray(0, Math.min(extraLen, head._extra_max));
  const cstr = (b: Uint8Array) => { const i = b.indexOf(0); return i < 0 ? b : b.subarray(0, i + 1); };
  if (head._name_max) head._name = cstr(name as Uint8Array);
  if (head._comm_max) head._comment = cstr(comment as Uint8Array);
}
export function deflate(strm: Stream, flush: number): number { return process(strm, flush, 0); }         // deflate.ts:716
export function inflate(strm: Stream, flush: number): number { return process(strm, flush, 1); }         // inflate.ts:332
function end(strm: Stream, which: 0 | 1): number {
  const st = strm && (strm._state as Handle);
  if (!st || st.which !== which) return Z_STREAM_ERROR;
  strm._state = undefined;
  return addon.end(st.h, which);
}
export function deflateEnd(strm: Stream): number { return end(strm, 0); }                                // deflate.ts:991
export function inflateEnd(strm: Stream): number { return end(strm, 1); }                                // inflate.ts:1187
export function deflateSetDictionary(strm: Stream, dict: Uint8Array, n: number): number {               // deflate.ts:367
  const st = strm && (strm._state as Handle);
  return st && st.which === 0 ? addon.setDictionary(st.h, 0, dict.subarray(0, n)) : Z_STREAM_ERROR;
}
export function inflateSetDictionary(strm: Stream, dict: Uint8Array, n: number): number {               // inflate.ts:1220
  const st = strm && (strm._state as Handle);
  return st && st.which === 1 ? addon.setDictionary(st.h, 1, dict.subarray(0, n)) : Z_STREAM_ERROR;
}
export function inflateReset(strm: Stream): number {                                                    // inflate.ts:124
  const st = strm && (strm._state as Handle);
  return st && st.which === 1 ? addon.inflateReset(st.h) : Z_STREAM_ERROR;
}
export function deflateReset(strm: Stream): number {                                                    // deflate.ts:489
  const st = strm && (strm._state as Handle);
  if (!st || st.which !== 0) return Z_STREAM_ERROR;
  strm.total_in = strm.total_out = 0; strm.msg = "";
  return addon.control(st.h, 0, 0);
}
export const deflateResetKeep = deflateReset;                                                           // deflate.ts:444
export function deflateParams(strm: Stream, level: number, strategy: number): number {                  // deflate.ts:553
  // pending input is flushed with the old parameters inside the call: same buffer handling as deflate()
  return process(strm, ((level + 1) & 0xff) | (strategy << 8), 2);
}
export function deflatePending(strm: Stream, pending?: { _value: number }, bits?: { _value: number }): number {   // deflate.ts:505
  const st = strm && (strm._state as Handle);
  if (!st || st.which !== 0) return Z_STREAM_ERROR;
  const [rc, p, b] = addon.deflatePending(st.h);
  if (pending) pending._value = p;
  if (bits) bits._value = b;
  return rc;
}
export function deflateUsed(strm: Stream, bits?: { _value: number }): number {                           // deflate.ts:518
  const st = strm && (strm._state as Handle);
  if (!st || st.which !== 0) return Z_STREAM_ERROR;
  if (bits) bits._value = 0;   // every part the engine emits ends byte aligned
  return Z_OK;
}
export function deflateSetHeader(strm: Stream, head: { _text: number; _time: number; _os: number; _hcrc: number;
    _extra?: Uint8Array | null; _extra_len?: number; _name?: Uint8Array | null; _comment?: Uint8Array | null }): number {   // deflate.ts:497
  const st = strm && (strm._state as Handle);
  if (!st || st.which !== 0) return Z_STREAM_ERROR;
  const z = (b?: Uint8Array | null) => { if (!b) return null; const i = b.indexOf(0); const r = new Uint8Array((i < 0 ? b.length : i) + 1); r.set(b.subarray(0, r.length - 1)); return r; };
  return addon.deflateSetHeader(st.h, head._text ? 1 : 0, head._time >>> 0, head._os & 0xff, head._hcrc ? 1 : 0,
    head._extra ? head._extra.subarray(0, head._extra_len ?? head._extra.length) : null, z(head._name), z(head._comment));
}
export function inflateGetHeader(strm: Stream, head: GzipHeader): number {                               // inflate.ts:1251
  const st = strm && (strm._state as Handle);
  if (!st || st.which !== 1 || !head) return Z_STREAM_ERROR;
  const rc = addon.inflateGetHeader(st.h, head._extra_max | 0, head._name_max | 0, head._comm_max | 0);
  if (rc === Z_OK) { head._done = 0; st.gzhead = head; }
  return rc;
}
export function inflateReset2(strm: Stream, windowBits: number): number {                                // inflate.ts:138
  const st = strm && (strm._state as Handle);
  if (!st || st.which !== 1) return Z_STREAM_ERROR;
  strm.total_in = strm.total_out = 0; strm.msg = "";
  return addon.control(st.h, 2, windowBits);
}
export const Z_FILTERED = 1, Z_HUFFMAN_ONLY = 2, Z_RLE = 3, Z_FIXED = 4, Z_DEFAULT_STRATEGY = 0;
export function adler32(adler: number, buf?: Uint8Array, len?: number): number {                         // adler32.ts:4
  return buf === undefined || len === undefined ? 1 : addon.checksum(0, adler, buf.subarray(0, len));
}
export function crc32(crc = 0, buf?: Uint8Array, len?: number): number {                                 // crc32.ts:26
  return !buf ? 0 : addon.checksum(1, crc, buf.subarray(0, len ?? buf.length));
}

// ---- new batch entry points (no reference analogue) ----
// A preset dictionary prepared once for many deflateBatch calls (deflateSetDictionary for every chunk); `id` is
// the DICTID zlib streams made with it carry (adler32 of the whole dictionary).
export interface DeflateDictionary { handle: unknown; id: number }
export function createDeflateDictionary(dict: Uint8Array): DeflateDictionary {
  return addon.createDeflateDictionary(dict);
}
// With `dictionary` every chunk is an independent stream that starts from it (raw or zlib, not stitched or primed).
export function deflateBatch(input: Uint8Array, opts: { chunkSize: number; level?: number; wrap?: 0 | 1 | 2; stitched?: boolean; prime?: boolean;
                                                       strategy?: number; dictionary?: DeflateDictionary }) {
  const nChunks = Math.max(1, Math.ceil(input.length / opts.chunkSize));
  const out = new Uint8Array(input.length + 6 * nChunks * (Math.floor(opts.chunkSize / 16351) + 2) + 26 * nChunks + 64 +
    (opts.dictionary ? 4 * nChunks : 0));
  const off = new BigUint64Array(nChunks + 1);
  if (opts.dictionary && (opts.stitched || opts.prime))
    throw new Error("deflateBatch: a dictionary call compresses every chunk as its own stream (not stitched, not primed)");
  const flags = (opts.prime ? 1 : 0) | ((opts.strategy ?? 0) << 8);
  const r = opts.dictionary
    ? addon.deflateBatch(input, opts.chunkSize, opts.level ?? 6, opts.wrap ?? 0, 0, flags, out, off, opts.dictionary.handle)
    : addon.deflateBatch(input, opts.chunkSize, opts.level ?? 6, opts.wrap ?? 0, opts.stitched ? 1 : 0, flags, out, off);
  return { data: out.subarray(0, r.bytes), offsets: off, check: r.check, bits: r.bits };
}
// dictionaries[i]: preset dictionary of stream i (raw streams, and zlib streams whose DICTID names it)
export function inflateBatch(streams: Uint8Array[], windowBits: number, outCaps: number[], dictionaries?: (Uint8Array | undefined)[]) {
  const n = streams.length;
  const inOff = new BigUint64Array(n + 1), outOff = new BigUint64Array(n + 1);
  streams.forEach((s, i) => { inOff[i + 1] = inOff[i] + BigInt(s.length); outOff[i + 1] = outOff[i] + BigInt(outCaps[i]); });
  const input = new Uint8Array(Number(inOff[n]));
  streams.forEach((s, i) => input.set(s, Number(inOff[i])));
  const out = new Uint8Array(Number(outOff[n]) + 16), outLen = new BigUint64Array(n);
  const checks = new Uint32Array(n), status = new Int32Array(n);
  if (dictionaries) {
    const rng = new BigUint64Array(2 * n);
    let total = 0;
    for (let i = 0; i < n; i++) { rng[2 * i] = BigInt(total); total += dictionaries[i]?.length ?? 0; rng[2 * i + 1] = BigInt(total); }
    const blob = new Uint8Array(total + 1);
    for (let i = 0; i < n; i++) if (dictionaries[i]) blob.set(dictionaries[i]!, Number(rng[2 * i]));
    addon.inflateBatch(input, inOff, windowBits, out, outOff, outLen, checks, status, blob, rng);
  } else {
    addon.inflateBatch(input, inOff, windowBits, out, outOff, outLen, checks, status);
  }
  return { out, outOff, outLen, checks, status };
}
// Every member of a multi-member gzip file (bgzip / BGZF, `cat a.gz b.gz`, deflateBatch's independent gzip output) in
// one call: what inflate(Z_FINISH) / inflateReset repeated until the input is used up produces
// (test/inflate/test-multistream.ts:16-79), strict about trailing bytes like that loop.  Without outCap the room
// starts at four times the input (at least 64 KiB) and doubles while the call ends with Z_BUF_ERROR on a full output.
// With `members`, `table` holds inOff, inLen, outOff, outLen, crc32 per member (the makings of a .gzi index).
export function gunzip(input: Uint8Array, opts: { outCap?: number; members?: boolean } = {}) {
  const grow = opts.outCap === undefined;
  let cap = grow ? Math.max(4 * input.length, 65536) : opts.outCap!;
  let nTab = opts.members ? Math.floor(input.length / 1024) + 1024 : 0;
  for (;;) {
    const out = new Uint8Array(cap + 16), table = new BigUint64Array(5 * nTab);
    const r = addon.gunzip(input, out.subarray(0, cap), table);
    if (grow && r.status === -5 && r.outLen === cap) { cap *= 2; continue; }
    if (opts.members && r.members > nTab) { nTab = r.members; continue; }
    return { data: out.subarray(0, r.outLen), inUsed: r.inUsed, members: r.members, status: r.status,
             msg: Buffer.from(r.msg).toString(), table: opts.members ? table.subarray(0, 5 * Math.min(r.members, nTab)) : undefined };
  }
}
// Random access into one zlib / gzip / raw deflate stream (zs_inflate_index_*): access points about every `span` bytes of
// output, each with the 32 KiB window before it, kept on the GPU.  build() decodes the whole stream once (as inflate with
// Z_FINISH would) and returns the index with the output; extract() then reads any byte ranges of the stream without
// decoding what comes before them.  toBytes() / fromBytes() carry an index across processes (the format of zsgpu.h).
export class InflateIndex {
  constructor(private readonly h: { handle: unknown; points: number; outLen: number }) {}
  get points(): number { return this.h.points; }
  get outLen(): number { return this.h.outLen; }
  static build(input: Uint8Array, opts: { windowBits?: number; span?: number; dictionary?: Uint8Array; outCap?: number } = {}) {
    const grow = opts.outCap === undefined;
    let cap = grow ? Math.max(4 * input.length, 65536) : opts.outCap!;
    for (;;) {
      const out = new Uint8Array(cap + 16);
      const args = [input, opts.windowBits ?? 15, opts.span ?? (1 << 20), out.subarray(0, cap)];
      const r = opts.dictionary ? addon.inflateIndexBuild(...args, opts.dictionary) : addon.inflateIndexBuild(...args);
      if (grow && r.status === -5 && r.outLen === cap) { cap *= 2; continue; }
      return { index: r.index.handle ? new InflateIndex(r.index) : undefined, data: out.subarray(0, r.outLen),
               inUsed: r.inUsed, check: r.check, status: r.status, msg: Buffer.from(r.msg).toString() };
    }
  }
  static fromBytes(blob: Uint8Array): InflateIndex { return new InflateIndex(addon.inflateIndexImport(blob)); }
  toBytes(): Uint8Array { return addon.inflateIndexExport(this.h.handle); }
  // ranges: [offset, length] in the uncompressed stream; `input` is the indexed stream.  A range past the end comes back
  // short with status Z_BUF_ERROR; one the input does not decode for has status Z_DATA_ERROR.
  extract(input: Uint8Array, ranges: [number, number][]) {
    const n = ranges.length;
    const off = new BigUint64Array(n), len = new BigUint64Array(n), outOff = new BigUint64Array(n);
    let total = 0;
    ranges.forEach(([o, l], i) => {
      off[i] = BigInt(o); len[i] = BigInt(l); outOff[i] = BigInt(total);
      total += Math.max(0, Math.min(l, this.h.outLen - o));
    });
    const out = new Uint8Array(total + 16), got = new BigUint64Array(n), status = new Int32Array(n);
    addon.inflateIndexExtract(this.h.handle, input, off, len, out.subarray(0, total), outOff, got, status);
    return ranges.map((_, i) => ({ data: out.subarray(Number(outOff[i]), Number(outOff[i]) + Number(got[i])), status: status[i] }));
  }
}
// One stitched stream (deflateBatch with stitched: true) and its InflateIndex, made in the same call from the encoder's
// block layout without decoding the stream: the index equals InflateIndex.build(data, {windowBits, span}).index.
// flags: the strategy (bits 8..10) and 8 (a sync marker after every chunk).
export function deflateIndexed(input: Uint8Array, opts: { chunkSize?: number; level?: number; wrap?: 0 | 1 | 2; flags?: number;
                                                         span?: number } = {}) {
  const chunkSize = opts.chunkSize ?? 65536;
  const nChunks = Math.max(1, Math.ceil(input.length / chunkSize));
  const out = new Uint8Array(input.length + 6 * nChunks * (Math.floor(chunkSize / 16351) + 2) + 26 * nChunks + 64);
  const r = addon.deflateIndexed(input, chunkSize, opts.level ?? 6, opts.wrap ?? 1, opts.flags ?? 0, opts.span ?? (1 << 20), out);
  return { data: out.subarray(0, r.outLen), check: r.check, index: new InflateIndex(r.index) };
}
