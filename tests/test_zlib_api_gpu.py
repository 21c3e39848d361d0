"""GPU: the reference-facing API (createDeflateStream/deflateInit/deflate/deflateEnd, inflateInit2_/
inflate/inflateEnd, CompressionStream/DecompressionStream) -- the parity tests read like the
reference's own (test/deflate/test-main-roundtrip.ts, test-small-buffers.ts,
test-avail-out-guard.ts, test-errors.ts, test/inflate/test-multistream.ts,
test/round-trip/test-streams-roundtrip.ts, test-streams-empty-input.ts)."""
import zlib

import pytest

from conftest import make_text, pkg, rand_bytes

pytestmark = pytest.mark.gpu


def _Z():
    return pkg("zlib_api")


def chunked_deflate(data, level, wbits, in_chunk, out_chunk):
    Z = _Z()
    s = Z.createDeflateStream()
    assert Z.deflateInit2_(s, level, Z.Z_DEFLATED, wbits, 8, 0) == Z.Z_OK
    out = bytearray()
    pos = 0
    while pos < len(data):
        piece = data[pos: pos + in_chunk]
        s.next_in, s.next_in_index, s.avail_in = piece, 0, len(piece)
        while s.avail_in > 0:
            buf = bytearray(out_chunk)
            s.next_out, s.next_out_index, s.avail_out = buf, 0, out_chunk
            assert Z.deflate(s, Z.Z_NO_FLUSH) == Z.Z_OK
            out += buf[: s.next_out_index]
        pos += len(piece)
    while True:
        buf = bytearray(out_chunk)
        s.next_in, s.next_in_index, s.avail_in = b"", 0, 0
        s.next_out, s.next_out_index, s.avail_out = buf, 0, out_chunk
        r = Z.deflate(s, Z.Z_FINISH)
        out += buf[: s.next_out_index]
        if r == Z.Z_STREAM_END:
            break
        assert r == Z.Z_OK
    assert s.total_in == len(data) and s.total_out == len(out)
    adler = s._adler
    assert Z.deflateEnd(s) == Z.Z_OK
    return bytes(out), adler


def chunked_inflate(stream, wbits, in_chunk, out_chunk):
    Z = _Z()
    s = Z.createInflateStream()
    assert Z.inflateInit2_(s, wbits) == Z.Z_OK
    out = bytearray()
    pos = 0
    r = Z.Z_OK
    while r != Z.Z_STREAM_END:
        piece = stream[pos: pos + in_chunk]
        s.next_in, s.next_in_index, s.avail_in = piece, 0, len(piece)
        buf = bytearray(out_chunk)
        s.next_out, s.next_out_index, s.avail_out = buf, 0, out_chunk
        r = Z.inflate(s, Z.Z_NO_FLUSH)
        assert r in (Z.Z_OK, Z.Z_STREAM_END, Z.Z_BUF_ERROR), (r, s.msg)
        out += buf[: s.next_out_index]
        pos += len(piece) - s.avail_in
        if r == Z.Z_BUF_ERROR and pos >= len(stream) and s.next_out_index == 0:
            break
    total_in = s.total_in
    assert Z.inflateEnd(s) == Z.Z_OK
    return bytes(out), r, total_in


@pytest.mark.parametrize("wbits", [15, 31, -15])
def test_main_roundtrip(gpu_ctx, oracle, wbits):
    # test/deflate/test-main-roundtrip.ts:9-43 -- C zlib (and the oracle) inflate what we deflate
    for data in (make_text(300000, 1), rand_bytes(100000, 2), bytes(j % 251 for j in range(1 << 20)), b"", b"x"):
        out, adler = chunked_deflate(data, 6, wbits, 65536, 65536)
        d = zlib.decompressobj(wbits)
        assert d.decompress(out) + d.flush() == data and d.eof
        ret, o2, used, _ = oracle.inflate(out, wbits, len(data) + 64)
        assert ret == 1 and o2 == data and used == len(out)
        if wbits == 15:
            assert adler == zlib.adler32(data)
        if wbits == 31:
            assert adler == zlib.crc32(data) and out[9] == 255
        # and our own inflate gives it back through the same API
        back, r, total_in = chunked_inflate(out, wbits, 65536, 65536)
        assert back == data and r == 1 and total_in == len(out)


def test_small_buffers(gpu_ctx, oracle):
    # test/deflate/test-small-buffers.ts:7-35, test/common/utils.ts:21-71
    data = make_text(5000, 3)
    for in_chunk, out_chunk in ((1, 64), (31, 7), (4096, 1)):
        out, _ = chunked_deflate(data, 9, 15, in_chunk, out_chunk)
        assert zlib.decompress(out) == data
    z = zlib.compress(data, 6)
    for in_chunk, out_chunk in ((3, 8), (1, 4096), (4096, 1)):
        back, r, _ = chunked_inflate(z, 15, in_chunk, out_chunk)
        assert back == data and r == 1


def test_protocol_pins(gpu_ctx):
    Z = _Z()
    # null stream -> Z_STREAM_ERROR for every entry point except deflateBound (test-errors.ts)
    assert Z.deflateInit(None, 6) == Z.Z_STREAM_ERROR and Z.deflate(None, 0) == Z.Z_STREAM_ERROR
    assert Z.deflateEnd(None) == Z.Z_STREAM_ERROR and Z.inflateInit(None) == Z.Z_STREAM_ERROR
    assert Z.inflate(None, 0) == Z.Z_STREAM_ERROR and Z.inflateEnd(None) == Z.Z_STREAM_ERROR
    assert Z.deflateBound(None, 1000) > 1000
    s = Z.createDeflateStream()
    for bad in (dict(level=10), dict(level=6, method=7), dict(level=6, windowBits=16 + 16), dict(level=6, memLevel=0),
                dict(level=6, strategy=5), dict(level=6, windowBits=-8)):
        args = dict(level=6, method=8, windowBits=15, memLevel=8, strategy=0)
        args.update(bad)
        assert Z.deflateInit2_(s, args["level"], args["method"], args["windowBits"], args["memLevel"], args["strategy"]) == Z.Z_STREAM_ERROR
    # Z_FINISH with avail_out == 0 -> Z_BUF_ERROR, stream still usable (test-avail-out-guard.ts:20-50)
    assert Z.deflateInit(s, 6) == Z.Z_OK
    s.next_in, s.next_in_index, s.avail_in = b"hello", 0, 5
    s.next_out, s.next_out_index, s.avail_out = bytearray(0), 0, 0
    assert Z.deflate(s, Z.Z_FINISH) == Z.Z_BUF_ERROR
    buf = bytearray(64)
    s.next_out, s.next_out_index, s.avail_out = buf, 0, 64
    assert Z.deflate(s, Z.Z_FINISH) == Z.Z_STREAM_END
    assert zlib.decompress(bytes(buf[: s.next_out_index])) == b"hello"
    assert Z.deflateEnd(s) == Z.Z_OK                       # finished stream -> Z_OK
    assert Z.deflate(s, Z.Z_FINISH) == Z.Z_STREAM_ERROR    # ended stream
    # deflateEnd in the middle of a stream -> Z_DATA_ERROR (deflate.ts:1012)
    s = Z.createDeflateStream()
    Z.deflateInit(s, 1)
    s.next_in, s.next_in_index, s.avail_in = b"abc", 0, 3
    s.next_out, s.next_out_index, s.avail_out = bytearray(64), 0, 64
    assert Z.deflate(s, Z.Z_NO_FLUSH) == Z.Z_OK
    assert Z.deflateEnd(s) == Z.Z_DATA_ERROR
    # inflate: bad windowBits, empty input -> Z_BUF_ERROR (test-inflate9-needmore.spec.ts)
    i = Z.createInflateStream()
    assert Z.inflateInit2_(i, -17) == Z.Z_STREAM_ERROR
    assert Z.inflateInit2_(i, -16) == Z.Z_OK
    i.next_in, i.next_in_index, i.avail_in = b"", 0, 0
    i.next_out, i.next_out_index, i.avail_out = bytearray(16), 0, 16
    assert Z.inflate(i, Z.Z_NO_FLUSH) == Z.Z_BUF_ERROR
    assert Z.inflateEnd(i) == Z.Z_OK


def test_flush_modes_and_dictionary(gpu_ctx, oracle):
    Z = _Z()
    data = make_text(200000, 4)
    # sync / full flush points: everything fed so far must be decodable (test-flush-modes.ts)
    s = Z.createDeflateStream()
    assert Z.deflateInit2_(s, 6, 8, -15, 8, 0) == Z.Z_OK
    out = bytearray()
    d = zlib.decompressobj(-15)
    got = b""
    for k, flush in enumerate((Z.Z_SYNC_FLUSH, Z.Z_FULL_FLUSH, Z.Z_SYNC_FLUSH, Z.Z_FINISH)):
        piece = data[k * 50000: (k + 1) * 50000]
        s.next_in, s.next_in_index, s.avail_in = piece, 0, len(piece)
        while True:
            buf = bytearray(1 << 16)
            s.next_out, s.next_out_index, s.avail_out = buf, 0, len(buf)
            r = Z.deflate(s, flush)
            out += buf[: s.next_out_index]
            got += d.decompress(bytes(buf[: s.next_out_index]))
            if s.avail_out != 0:
                break
        assert got == data[: (k + 1) * 50000], k
        assert r == (Z.Z_STREAM_END if flush == Z.Z_FINISH else Z.Z_OK)
    assert Z.deflateEnd(s) == Z.Z_OK
    # preset dictionary, zlib wrapper: FDICT + DICTID framing, C zlib decodes with zdict
    dic = data[:20000]
    s = Z.createDeflateStream()
    Z.deflateInit(s, 6)
    assert Z.deflateSetDictionary(s, dic, len(dic)) == Z.Z_OK
    body = data[20000:90000]
    s.next_in, s.next_in_index, s.avail_in = body, 0, len(body)
    buf = bytearray(1 << 17)
    s.next_out, s.next_out_index, s.avail_out = buf, 0, len(buf)
    assert Z.deflate(s, Z.Z_FINISH) == Z.Z_STREAM_END
    stream = bytes(buf[: s.next_out_index])
    assert stream[1] & 0x20
    assert zlib.decompressobj(15, zdict=dic).decompress(stream) == body
    ret, o2, _, _ = oracle.inflate(stream, 15, len(body) + 64, dic)
    assert ret == 1 and o2 == body
    assert len(stream) < len(zlib.compress(body, 6))          # the dictionary helped
    # ... and our inflate asks for it (Z_NEED_DICT, inflate.ts:587-590)
    i = Z.createInflateStream()
    Z.inflateInit(i)
    i.next_in, i.next_in_index, i.avail_in = stream, 0, len(stream)
    ob = bytearray(len(body) + 64)
    i.next_out, i.next_out_index, i.avail_out = ob, 0, len(ob)
    assert Z.inflate(i, Z.Z_NO_FLUSH) == Z.Z_NEED_DICT
    assert i._adler == zlib.adler32(dic)
    assert Z.inflateSetDictionary(i, b"wrong", 5) == Z.Z_DATA_ERROR
    assert Z.inflateSetDictionary(i, dic, len(dic)) == Z.Z_OK
    assert Z.inflate(i, Z.Z_FINISH) == Z.Z_STREAM_END
    assert bytes(ob[: i.next_out_index]) == body


def test_multi_member_gzip(gpu_ctx):
    # test/inflate/test-multistream.ts:16-79
    Z = _Z()
    a, b = make_text(30000, 1), make_text(20000, 2)
    blob = zlib.compress(a, 6, 31) + zlib.compress(b, 9, 31)
    s = Z.createInflateStream()
    Z.inflateInit2_(s, 31)
    s.next_in, s.next_in_index, s.avail_in = blob, 0, len(blob)
    ob = bytearray(1 << 16)
    s.next_out, s.next_out_index, s.avail_out = ob, 0, len(ob)
    assert Z.inflate(s, Z.Z_NO_FLUSH) == Z.Z_STREAM_END
    first = s.total_in
    assert bytes(ob[: s.next_out_index]) == a and 0 < first < len(blob) and s.avail_in == len(blob) - first
    assert Z.inflateReset(s) == Z.Z_OK
    s.next_out, s.next_out_index, s.avail_out = ob, 0, len(ob)
    assert Z.inflate(s, Z.Z_NO_FLUSH) == Z.Z_STREAM_END
    assert bytes(ob[: s.next_out_index]) == b and first + s.total_in == len(blob)
    Z.inflateEnd(s)


@pytest.mark.parametrize("fmt", ["deflate", "gzip", "deflate-raw"])
def test_streams_roundtrip(gpu_ctx, fmt):
    # test/round-trip/test-streams-roundtrip.ts, test-streams-options.ts, test-streams-empty-input.ts
    S = pkg("streams")
    wb = {"deflate": 15, "gzip": 31, "deflate-raw": -15}[fmt]
    for level in (None, 1, 9):
        for data in (make_text(1 << 20, 5), rand_bytes(70000, 6), b""):
            cs = S.CompressionStream(fmt, {"level": level} if level is not None else None)
            comp = b"".join(cs.write(data[: len(data) // 2]) + cs.write(data[len(data) // 2:]) + cs.close())
            d = zlib.decompressobj(wb)
            assert d.decompress(comp) + d.flush() == data
            assert S.DecompressionStream(fmt).transform(comp) == data
    assert S.CompressionStream("deflate-raw").transform(b"") == bytes([3, 0])
    with pytest.raises(RuntimeError):
        S.DecompressionStream(fmt).transform(b"")               # truncated stream rejects
    with pytest.raises(TypeError):
        S.CompressionStream("deflate64-raw")


def test_decompression_stream_deflate64(gpu_ctx, fixtures64):
    S = pkg("streams")
    f = next(x for x in fixtures64 if x["name"] == "10k_lines.deflate64")
    out = S.DecompressionStream("deflate64-raw").transform(f["data"])
    assert len(out) == f["out_len"] and zlib.crc32(out) == f["crc32"]


@pytest.mark.parametrize("wbits", [15, 31, -15])
def test_incremental_inflate_of_a_long_stream(gpu_ctx, wbits):
    """A multi-megabyte stream fed in 32 KiB pieces (the slicing of src/mod/streams.ts:7): decoding resumes
    at block boundaries, the trailer is checked after the last attempt, input behind the end is handed back."""
    import time
    from conftest import make_mixed
    Z = _Z()
    data = make_mixed(6 << 20, 77) + make_text(1 << 20, 78)
    co = zlib.compressobj(6, zlib.DEFLATED, wbits)
    stream = co.compress(data) + co.flush()
    tail = b"TRAILING-GARBAGE"
    t0 = time.time()
    for corrupt in (False, True):
        src = bytearray(stream)
        if corrupt and wbits > 0:
            src[-1] ^= 0x55                      # last trailer byte: ISIZE (gzip) / adler32 (zlib)
        src += tail
        s = Z.createInflateStream()
        assert Z.inflateInit2_(s, wbits) == Z.Z_OK
        out = bytearray()
        pos, r = 0, Z.Z_OK
        while r == Z.Z_OK:
            piece = bytes(src[pos: pos + 32768])
            s.next_in, s.next_in_index, s.avail_in = piece, 0, len(piece)
            while True:
                buf = bytearray(65536)
                s.next_out, s.next_out_index, s.avail_out = buf, 0, len(buf)
                r = Z.inflate(s, Z.Z_NO_FLUSH)
                out += buf[: s.next_out_index]
                if r != Z.Z_OK or (s.avail_in == 0 and s.avail_out != 0):
                    break
            pos += len(piece) - s.avail_in
            if pos >= len(src) and r == Z.Z_OK:
                # drain like the reference's flush() (streams.ts:139-170): Z_FINISH until Z_STREAM_END; a long
                # stream is decoded in batches, so more than one output buffer may still be waiting
                while r == Z.Z_OK:
                    buf = bytearray(65536)
                    s.next_out, s.next_out_index, s.avail_out = buf, 0, len(buf)
                    r = Z.inflate(s, Z.Z_FINISH)
                    out += buf[: s.next_out_index]
                break
        if corrupt and wbits > 0:
            assert r == Z.Z_DATA_ERROR and s.msg in ("incorrect data check", "incorrect length check"), (r, s.msg)
            assert bytes(out) == data            # everything decoded before the check is still delivered
        else:
            assert r == Z.Z_STREAM_END, (r, s.msg)
            assert bytes(out) == data
            # total_in is exact; the garbage is handed back through avail_in when it arrived in the call that
            # found the end of the stream (a long stream is decoded in batches: it may have arrived earlier)
            assert s.total_in == len(stream) and pos in (len(stream), len(src)), (s.total_in, pos, len(stream))
            if wbits == 15:
                assert s._adler == zlib.adler32(data)
            if wbits == 31:
                assert s._adler == zlib.crc32(data)
        assert Z.inflateEnd(s) == Z.Z_OK
    assert time.time() - t0 < 60                 # linear: a restart-from-scratch decoder needs minutes here


def test_inflate_without_finish_reaches_stream_end(gpu_ctx):
    """A caller that never sends Z_FINISH (the classic zlib loop: refill, inflate(Z_NO_FLUSH), until
    Z_STREAM_END): a long stream is decoded in batches, so after the last piece some input is still waiting for
    its attempt -- a call that brings no new input must decode it instead of answering Z_BUF_ERROR for ever."""
    Z = _Z()
    data = make_text(3 << 20, 91)
    for wbits in (15, 31, -15):
        co = zlib.compressobj(6, zlib.DEFLATED, wbits)
        stream = co.compress(data) + co.flush()
        assert len(stream) > (512 << 10)          # far beyond the shim's every-call threshold (64 KiB, kEveryCallBelow)
        s = Z.createInflateStream()
        assert Z.inflateInit2_(s, wbits) == Z.Z_OK
        out = bytearray()
        pos, r, idle = 0, Z.Z_OK, 0
        while r != Z.Z_STREAM_END:
            piece = stream[pos: pos + 32768]      # empty once the input is exhausted
            s.next_in, s.next_in_index, s.avail_in = piece, 0, len(piece)
            buf = bytearray(1 << 16)
            s.next_out, s.next_out_index, s.avail_out = buf, 0, len(buf)
            r = Z.inflate(s, Z.Z_NO_FLUSH)
            assert r in (Z.Z_OK, Z.Z_STREAM_END, Z.Z_BUF_ERROR), (r, s.msg)
            out += buf[: s.next_out_index]
            pos += len(piece) - s.avail_in
            idle = idle + 1 if (not piece and s.next_out_index == 0) else 0
            assert idle < 4, "no progress although undecoded input is buffered"
        assert bytes(out) == data and s.total_in == len(stream)
        assert Z.inflateEnd(s) == Z.Z_OK


def test_incremental_inflate_truncated(gpu_ctx):
    Z = _Z()
    data = make_text(900000, 79)
    stream = zlib.compress(data, 6)[:-300000 // 100]     # cut inside the last blocks
    s = Z.createInflateStream()
    assert Z.inflateInit(s) == Z.Z_OK
    out = bytearray()
    for pos in range(0, len(stream), 10000):
        piece = stream[pos: pos + 10000]
        s.next_in, s.next_in_index, s.avail_in = piece, 0, len(piece)
        buf = bytearray(1 << 20)
        s.next_out, s.next_out_index, s.avail_out = buf, 0, len(buf)
        assert Z.inflate(s, Z.Z_NO_FLUSH) == Z.Z_OK
        out += buf[: s.next_out_index]
    buf = bytearray(1 << 20)
    s.next_in, s.next_in_index, s.avail_in = b"", 0, 0
    s.next_out, s.next_out_index, s.avail_out = buf, 0, len(buf)
    assert Z.inflate(s, Z.Z_FINISH) == Z.Z_BUF_ERROR     # inflate.ts:1092-1098
    out += buf[: s.next_out_index]
    d = zlib.decompressobj()
    assert bytes(out) == d.decompress(stream)            # exactly what C zlib can decode from the same bytes
    assert Z.inflateEnd(s) == Z.Z_OK


def test_window_bits_zero_is_a_zlib_stream(gpu_ctx):
    """inflateInit2_(strm, 0): zlib wrapper with the window size taken from the header
    (inflateReset2, inflate.ts:138-172; CINFO check :396-415).  Fed in 7-byte pieces so that the first
    call sees less than the 2-byte header + first block."""
    Z = _Z()
    s = Z.createInflateStream()
    assert Z.inflateInit2_(s, 0) == Z.Z_OK
    assert s._adler == 1
    assert Z.inflateEnd(s) == Z.Z_OK
    data = make_text(30000, 83)
    stream = zlib.compress(data, 6)
    out, r, total_in = chunked_inflate(stream[:1] , 0, 1, 4096)      # one byte only: no progress beyond buffering
    assert out == b"" and r != Z.Z_STREAM_END
    out, r, total_in = chunked_inflate(stream, 0, 7, 4096)
    assert r == Z.Z_STREAM_END and out == data and total_in == len(stream)


def test_stream_loop_in_c(gpu_ctx):
    """The driver loop of src/mod/streams.ts:78-93,139-170 in C (bindings/c/stream_pump.c: 32 KiB slices with
    Z_NO_FLUSH, the last one with Z_FINISH, 64 KiB output buffers) -- what bench.py measures the stream API with.
    Calls arrive within microseconds of each other here, so a long stream's decode attempts are paced by the shim
    (zs_stream.cu): the results must not depend on when the attempts run."""
    import ctypes as C
    import numpy as np
    from tools import streampump
    capi = pkg("capi")
    lib = capi.load()
    data = np.frombuffer(make_text(5 << 20, 123), dtype=np.uint8)
    big = np.empty(data.size + (1 << 20), dtype=np.uint8)
    for level, wbits in ((1, 31), (6, 15), (6, -15)):
        zs = capi.ZStream()
        assert lib.zs_stream_deflate_init(gpu_ctx.handle, C.byref(zs), level, 8, wbits, 8, 0) == 0
        rc, made, calls = streampump.pump(lib.zs_stream_deflate, zs, data, big)
        assert rc == 1 and zs.total_in == data.size and zs.total_out == made and calls >= data.size // 32768
        assert lib.zs_stream_deflate_end(C.byref(zs)) == 0
        comp = big[:made].copy()
        assert zlib.decompress(comp.tobytes(), wbits) == data.tobytes()
        co = zlib.compressobj(6, zlib.DEFLATED, wbits)
        czlib = np.frombuffer(co.compress(data.tobytes()) + co.flush(), dtype=np.uint8)   # no flush points inside
        for src in (comp, czlib):
            zs = capi.ZStream()
            assert lib.zs_stream_inflate_init(gpu_ctx.handle, C.byref(zs), wbits) == 0
            rc, made, calls = streampump.pump(lib.zs_stream_inflate, zs, src, big)
            assert rc == 1, (rc, zs.msg)
            assert made == data.size and zs.total_in == src.size and zs.total_out == made
            assert np.array_equal(big[:made], data)
            if wbits == 31:
                assert zs.adler == zlib.crc32(data.tobytes())
            if wbits == 15:
                assert zs.adler == zlib.adler32(data.tobytes())
            assert lib.zs_stream_inflate_end(C.byref(zs)) == 0
    # parts that run in the background: 40 MiB is two full parts (16 MiB each, started when their input is complete and
    # compressed while the next one is buffered) and a final one; fed in 32 KiB slices, in one giant call (the call
    # compresses part by part and comes back for output room: Z_OK with avail_in > 0), and through a 1000-byte output buffer
    long_data = np.frombuffer(make_text(40 << 20, 321), dtype=np.uint8)
    big2 = np.empty(long_data.size + (1 << 20), dtype=np.uint8)
    outs = []
    for in_slice, out_slice, level, wbits in ((32768, 65536, 1, 31), (48 << 20, 65536, 6, 15), (1 << 20, 1000, 1, -15)):
        zs = capi.ZStream()
        assert lib.zs_stream_deflate_init(gpu_ctx.handle, C.byref(zs), level, 8, wbits, 8, 0) == 0
        rc, made, calls = streampump.pump(lib.zs_stream_deflate, zs, long_data, big2, in_slice, out_slice)
        assert rc == 1 and zs.total_in == long_data.size and zs.total_out == made, (rc, in_slice, out_slice)
        if wbits == 31:
            assert zs.adler == zlib.crc32(long_data.tobytes())
        if wbits == 15:
            assert zs.adler == zlib.adler32(long_data.tobytes())
        assert lib.zs_stream_deflate_end(C.byref(zs)) == 0
        d = zlib.decompressobj(wbits)
        assert d.decompress(big2[:made].tobytes()) + d.flush() == long_data.tobytes() and d.eof and d.unused_data == b""
        outs.append(made)
    # a stream abandoned with a part in flight: deflateEnd waits for it (Z_DATA_ERROR: mid-stream, deflate.ts:1012)
    zs = capi.ZStream()
    assert lib.zs_stream_deflate_init(gpu_ctx.handle, C.byref(zs), 1, 8, 15, 8, 0) == 0
    obuf = np.empty(65536, dtype=np.uint8)
    zs.next_in, zs.avail_in = long_data.ctypes.data, 17 << 20
    zs.next_out, zs.avail_out = obuf.ctypes.data, obuf.size
    assert lib.zs_stream_deflate(C.byref(zs), 0) == 0 and zs.avail_in == 0
    assert lib.zs_stream_deflate_end(C.byref(zs)) == capi.Z_DATA_ERROR
    # a truncated stream: Z_BUF_ERROR under Z_FINISH, everything decodable delivered
    co = zlib.compressobj(6)
    whole = co.compress(data.tobytes()) + co.flush()
    cut = np.frombuffer(whole[: len(whole) * 2 // 3], dtype=np.uint8)
    zs = capi.ZStream()
    assert lib.zs_stream_inflate_init(gpu_ctx.handle, C.byref(zs), 15) == 0
    rc, made, calls = streampump.pump(lib.zs_stream_inflate, zs, cut, big)
    assert rc == capi.Z_BUF_ERROR
    assert big[:made].tobytes() == zlib.decompressobj().decompress(cut.tobytes())
    assert lib.zs_stream_inflate_end(C.byref(zs)) == 0
