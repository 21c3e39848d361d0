"""zlib's examples/zran.c method with C zlib itself, through ctypes (test infrastructure: no engine code is involved).

block_starts finds every block start of a stream as zran.c does, with inflate(Z_BLOCK).  decode_from reads from an
access point as zran.c does: inflateInit2(-15), inflatePrime with the unused high bits of the point's byte,
inflateSetDictionary with the window, then inflate from the next byte.  (Python's zlib module has neither Z_BLOCK stops
nor inflatePrime, and shifting the input instead would move the byte boundaries that stored blocks pad to.)"""
import ctypes as C
import ctypes.util
import zlib

Z_OK, Z_STREAM_END, Z_NEED_DICT, Z_BUF_ERROR, Z_BLOCK = 0, 1, 2, -5, 5


class _ZStream(C.Structure):
    _fields_ = [("next_in", C.c_void_p), ("avail_in", C.c_uint), ("total_in", C.c_ulong),
                ("next_out", C.c_void_p), ("avail_out", C.c_uint), ("total_out", C.c_ulong),
                ("msg", C.c_char_p), ("state", C.c_void_p), ("zalloc", C.c_void_p), ("zfree", C.c_void_p),
                ("opaque", C.c_void_p), ("data_type", C.c_int), ("adler", C.c_ulong), ("reserved", C.c_ulong)]


_z = None


def _lib():
    global _z
    if _z is None:
        _z = C.CDLL(ctypes.util.find_library("z") or "libz.so.1")
        _z.zlibVersion.restype = C.c_char_p
        _z.inflateInit2_.argtypes = [C.POINTER(_ZStream), C.c_int, C.c_char_p, C.c_int]
        _z.inflatePrime.argtypes = [C.POINTER(_ZStream), C.c_int, C.c_int]
        _z.inflateSetDictionary.argtypes = [C.POINTER(_ZStream), C.c_void_p, C.c_uint]
        _z.inflate.argtypes = [C.POINTER(_ZStream), C.c_int]
        _z.inflateEnd.argtypes = [C.POINTER(_ZStream)]
    return _z


def decode_from(stream: bytes, bit: int, window: bytes, want: int, max_in: int = 1 << 20) -> bytes:
    """Up to `want` bytes of raw deflate decoded from bit `bit` of `stream` with `window` as the history before it."""
    z = _lib()
    s = _ZStream()
    assert z.inflateInit2_(C.byref(s), -15, z.zlibVersion(), C.sizeof(_ZStream)) == 0
    try:
        byte, k = bit >> 3, bit & 7
        if k:
            assert z.inflatePrime(C.byref(s), 8 - k, stream[byte] >> k) == 0
            byte += 1
        if window:
            wbuf = C.create_string_buffer(window, len(window))
            assert z.inflateSetDictionary(C.byref(s), wbuf, len(window)) == 0
        src = stream[byte: byte + max_in]
        ibuf = C.create_string_buffer(src, max(len(src), 1))
        obuf = C.create_string_buffer(max(want, 1))
        s.next_in, s.avail_in = C.addressof(ibuf), len(src)
        s.next_out, s.avail_out = C.addressof(obuf), want
        ret = z.inflate(C.byref(s), 0)
        assert ret in (0, 1, -5), (ret, s.msg)
        return obuf.raw[: want - s.avail_out]
    finally:
        z.inflateEnd(C.byref(s))


def block_starts(stream: bytes, window_bits: int = 15, dictionary=None) -> list:
    """Every block start of a whole stream as [(input bit, output offset), ...].  inflate(Z_BLOCK) stops at each block
    boundary; a stop with data_type & 128 set before the last block was seen (data_type & 64) is a block start at bit
    (input used) * 8 - (bits held), output offset total_out.  zran takes the bits held as data_type & 7; the field holds
    their whole count below 64, so data_type & 63 reads it exactly.  Input used is counted from avail_in: total_in leaves
    out the header bytes read before a Z_NEED_DICT return.  A raw stream has no header to stop behind: inflate goes
    straight into its first block, which starts at bit 0."""
    d = zlib.decompressobj(window_bits, zdict=dictionary) if dictionary else zlib.decompressobj(window_bits)
    out_len = len(d.decompress(stream))
    if not d.eof:
        raise ValueError("the stream does not decode")
    z = _lib()
    s = _ZStream()
    assert z.inflateInit2_(C.byref(s), window_bits, z.zlibVersion(), C.sizeof(_ZStream)) == Z_OK
    try:
        dbuf = C.create_string_buffer(bytes(dictionary), len(dictionary)) if dictionary else None
        if dictionary and window_bits < 0:
            assert z.inflateSetDictionary(C.byref(s), dbuf, len(dictionary)) == Z_OK
        ibuf = C.create_string_buffer(stream, max(len(stream), 1))
        obuf = C.create_string_buffer(max(out_len, 1))
        s.next_in, s.avail_in = C.addressof(ibuf), len(stream)
        s.next_out, s.avail_out = C.addressof(obuf), out_len
        starts = [(0, 0)] if window_bits < 0 else []
        while True:
            ret = z.inflate(C.byref(s), Z_BLOCK)
            if ret == Z_NEED_DICT:
                assert dictionary and z.inflateSetDictionary(C.byref(s), dbuf, len(dictionary)) == Z_OK
                continue
            if ret == Z_STREAM_END:
                return starts
            assert ret in (Z_OK, Z_BUF_ERROR), (ret, s.msg)
            dt = s.data_type
            if (dt & 128) and not (dt & 64):
                pos = ((len(stream) - s.avail_in) * 8 - (dt & 63), s.total_out)
                if not starts or starts[-1] != pos:
                    starts.append(pos)
    finally:
        z.inflateEnd(C.byref(s))
