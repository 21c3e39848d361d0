"""Pinned call traces of the streaming shim (zs_stream_deflate* / zs_stream_inflate* through the C ABI) under seeded
call schedules.  Each case records, for every call, the return code, the bytes consumed and produced, adler,
total_in and total_out, and the produced bytes themselves; tests/golden/stream_shim_digests.json keeps one sha256
of that trace per case.  The deflate cases reach every way a part of a stream ends: raw / zlib / gzip at levels 0,
1, 6 and 9 and with every strategy, interleaved flush values (a flush without new input included), deflateParams
through a small output buffer, preset dictionaries (the FDICT header), deflateSetHeader, streams of more than two
parts that run in the background (fed in slices, in one call, through a 1000-byte buffer), a stream abandoned or
reset with a part in flight.  Every deflate output must also decode with C zlib to its input.  The inflate cases
cover inflateReset / inflateReset2 between the members of a multi-member input, inflateSetDictionary and
inflateGetHeader; every call there asks for Z_SYNC_FLUSH or Z_FINISH, so every call runs a decode attempt and the
trace does not depend on the clock.

Regenerate the digests (only when the output is meant to change): python tests/test_stream_shim_golden_gpu.py --write"""
import ctypes as C
import hashlib
import json
import os
import random
import struct
import sys
import zlib

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from conftest import GOLDEN, make_mixed, make_text, pkg  # noqa: E402

pytestmark = pytest.mark.gpu

DIGESTS = os.path.join(GOLDEN, "stream_shim_digests.json")
Z_NO_FLUSH, Z_PARTIAL_FLUSH, Z_SYNC_FLUSH, Z_FULL_FLUSH, Z_FINISH, Z_BLOCK = 0, 1, 2, 3, 4, 5
Z_OK, Z_STREAM_END, Z_NEED_DICT, Z_STREAM_ERROR, Z_DATA_ERROR, Z_BUF_ERROR = 0, 1, 2, -2, -3, -5
WRAPS = [("raw", -15), ("zlib", 15), ("gzip", 31)]
STRATEGIES = [("filtered", 1), ("huffman", 2), ("rle", 3), ("fixed", 4)]


class _Trace:
    """sha256 over (operation, return code, consumed, produced, adler, total_in, total_out, produced bytes) per call."""

    def __init__(self):
        self.h = hashlib.sha256()
        self.calls = 0

    def add(self, op, rc, used, made, zs, produced=b""):
        self.h.update(struct.pack("<8siqqIQQ", op.encode(), rc, used, made, zs.adler, zs.total_in, zs.total_out))
        self.h.update(produced)
        self.calls += 1

    def digest(self):
        return self.h.hexdigest()


class _Stream:
    """One zs_stream driven through ctypes; `src` is the whole input, calls point into it."""

    def __init__(self, kind, src, trace):
        self.capi = pkg("capi")
        self.lib = self.capi.load()
        self.ctx = pkg("batch").default_context(0)
        self.zs = self.capi.ZStream()
        self.kind = kind
        self.src = np.frombuffer(src, dtype=np.uint8) if len(src) else np.zeros(1, dtype=np.uint8)
        self.obuf = np.empty(1 << 20, dtype=np.uint8)
        self.trace = trace
        self.out = bytearray()

    def _io(self, pos, n, room):
        zs = self.zs
        zs.next_in, zs.avail_in = self.src.ctypes.data + pos, n
        zs.next_out, zs.avail_out = self.obuf.ctypes.data, room

    def _done(self, op, rc, n, room):
        used, made = n - self.zs.avail_in, room - self.zs.avail_out
        produced = self.obuf[:made].tobytes()
        self.trace.add(op, rc, used, made, self.zs, produced)
        self.out += produced
        return rc, used, made

    def call(self, pos, n, room, flush):
        self._io(pos, n, room)
        fn = self.lib.zs_stream_deflate if self.kind == "deflate" else self.lib.zs_stream_inflate
        return self._done("call", fn(C.byref(self.zs), flush), n, room)

    def params(self, level, strategy, room):
        self._io(0, 0, room)
        return self._done("params", self.lib.zs_stream_deflate_params(C.byref(self.zs), level, strategy), 0, room)

    def op(self, name, rc):
        self.trace.add(name, rc, 0, 0, self.zs)
        return rc


N_MIXED, N_BIG = 700_000, 33 << 20
_DATA = {}


def _data(name):
    """Inputs are made when a case runs (collecting the tests makes none)."""
    if name not in _DATA:
        _DATA[name] = {"mixed": lambda: make_mixed(N_MIXED, 41), "big": lambda: make_text(N_BIG, 321),
                       "small": lambda: make_text(50_000, 42), "dict": lambda: make_text(40_000, 43)}[name]()
    return _DATA[name]


# ---- deflate ---------------------------------------------------------------------------------------

def _deflate_init(src, trace, level, wbits, strategy=0):
    s = _Stream("deflate", src, trace)
    s.op("init", s.lib.zs_stream_deflate_init(s.ctx.handle, C.byref(s.zs), level, 8, wbits, 8, strategy))
    return s


def _feed(s, lo, hi, room, flush):
    """zlib's deflate loop for one slice: call until the slice is consumed and the output buffer is not filled, or
    Z_STREAM_END; any other return code ends the slice."""
    pos = lo
    for _ in range(200000):
        rc, used, made = s.call(pos, hi - pos, room, flush)
        pos += used
        if rc != Z_OK or (pos == hi and made < room):
            return rc
    raise AssertionError("deflate loop does not end")


def _schedule(n, seed, max_slice, flushes=(Z_NO_FLUSH, Z_NO_FLUSH, Z_NO_FLUSH, Z_SYNC_FLUSH, Z_FULL_FLUSH,
                                         Z_PARTIAL_FLUSH, Z_BLOCK), rooms=(1000, 65536, 1 << 20)):
    """(slice end, output room, flush) per slice; the third slice is followed by a Z_PARTIAL_FLUSH slice and two
    flushes without new input (Z_SYNC_FLUSH: the empty marker alone; Z_FULL_FLUSH after it), the last is Z_FINISH."""
    rng = random.Random(seed)
    out, pos = [], 0
    while pos < n:
        pos = min(n, pos + rng.randint(1, max_slice))
        out.append((pos, rng.choice(rooms), rng.choice(flushes)))
        if len(out) == 3 and pos < n:
            pos = min(n, pos + rng.randint(1, max_slice))
            out += [(pos, 65536, Z_PARTIAL_FLUSH), (pos, 65536, Z_SYNC_FLUSH), (pos, 65536, Z_FULL_FLUSH)]
    out.append((n, rng.choice(rooms), Z_FINISH))
    return out


def _run(s, sched, base=0):
    """Feeds the slices of a schedule whose offsets count from src[base]."""
    prev = 0
    for end, room, flush in sched:
        rc = _feed(s, base + prev, base + end, room, flush)
        prev = end
    return rc


def _decodes(comp, data, wbits, zdict=None):
    d = zlib.decompressobj(wbits, zdict=zdict) if zdict is not None else zlib.decompressobj(wbits)
    return d.decompress(bytes(comp)) + d.flush() == data and d.eof and d.unused_data == b""


def _deflate_cases():
    """Yields (case id, thunk -> digest) for every deflate case; each thunk asserts that its output decodes."""

    def flushes(wbits, level, strategy, seed):
        def run():
            mixed = _data("mixed")
            t = _Trace()
            s = _deflate_init(mixed, t, level, wbits, strategy)
            assert _run(s, _schedule(N_MIXED, seed, 150_000)) == Z_STREAM_END
            s.op("end", s.lib.zs_stream_deflate_end(C.byref(s.zs)))
            assert _decodes(s.out, mixed, wbits)
            return t.digest()
        return run

    def whole(wbits, level, strategy):
        def run():
            data = _data("small")
            t = _Trace()
            s = _deflate_init(data, t, level, wbits, strategy)
            assert _feed(s, 0, len(data), 1 << 20, Z_FINISH) == Z_STREAM_END
            s.op("end", s.lib.zs_stream_deflate_end(C.byref(s.zs)))
            assert _decodes(s.out, data, wbits)
            return t.digest()
        return run

    def params(wbits):
        """deflateParams through a 100-byte output buffer: Z_BUF_ERROR until what it compressed is delivered."""
        def run():
            mixed = _data("mixed")
            t = _Trace()
            s = _deflate_init(mixed, t, 1, wbits)
            s.params(1, 0, 100)                     # before any data: nothing to compress
            cuts = [0, 200_000, 350_000, 500_000, 600_000]
            assert _feed(s, 0, cuts[1], 1 << 20, Z_NO_FLUSH) == Z_OK
            for i, (level, strategy) in enumerate(((6, 0), (9, 3), (2, 2))):
                for _ in range(100000):
                    rc, _, _ = s.params(level, strategy, 100)
                    if rc != Z_BUF_ERROR:
                        break
                assert rc == Z_OK
                assert _feed(s, cuts[i + 1], cuts[i + 2], 65536, Z_NO_FLUSH) == Z_OK
            assert _feed(s, cuts[-1], N_MIXED, 65536, Z_FINISH) == Z_STREAM_END
            s.op("end", s.lib.zs_stream_deflate_end(C.byref(s.zs)))
            assert _decodes(s.out, mixed, wbits)
            return t.digest()
        return run

    def with_dict(wbits, sched):
        def run():
            mixed, dictionary = _data("mixed"), _data("dict")
            t = _Trace()
            s = _deflate_init(mixed, t, 6, wbits)
            d = np.frombuffer(dictionary, dtype=np.uint8)
            rc = s.op("setdict", s.lib.zs_stream_deflate_set_dictionary(C.byref(s.zs), d.ctypes.data, d.size))
            if wbits == 31:
                assert rc == Z_STREAM_ERROR     # not for gzip
            else:
                assert rc == Z_OK
                assert _run(s, sched) == Z_STREAM_END
            s.op("end", s.lib.zs_stream_deflate_end(C.byref(s.zs)))
            assert wbits == 31 or _decodes(s.out, mixed, wbits, dictionary)
            return t.digest()
        return run

    def gz_header(level, strategy, sched):
        def run():
            mixed = _data("mixed")
            t = _Trace()
            s = _deflate_init(mixed, t, level, 31, strategy)
            extra, name, comment = b"AB\x04\x00xyz!", b"stream-shim.txt\0", b"pinned by a golden trace\0"
            keep = [C.create_string_buffer(x, len(x)) for x in (extra, name, comment)]
            h = s.capi.GzHeader(text=1, time=0x5f3759df, xflags=0, os=3, extra=C.addressof(keep[0]), extra_max=0,
                                extra_len=len(extra), name=C.addressof(keep[1]), name_max=0,
                                comment=C.addressof(keep[2]), comm_max=0, hcrc=1, done=0)
            s.op("sethead", s.lib.zs_stream_deflate_set_header(C.byref(s.zs), C.byref(h)))
            assert _run(s, sched) == Z_STREAM_END
            s.op("end", s.lib.zs_stream_deflate_end(C.byref(s.zs)))
            assert _decodes(s.out, mixed, 31)
            # FLG: FTEXT, FHCRC, FEXTRA, FNAME, FCOMMENT; XFL from level and strategy
            assert s.out[3] == 0x1f and s.out[8] == (2 if level == 9 else 4 if strategy >= 2 or level < 2 else 0)
            return t.digest()
        return run

    def long_stream(wbits, level, in_slice, room):
        """More than two parts of 16 MiB: the full ones run in the background."""
        def run():
            big = _data("big")
            t = _Trace()
            s = _deflate_init(big, t, level, wbits)
            sched = [(min(N_BIG, p + in_slice), room, Z_NO_FLUSH) for p in range(0, N_BIG, in_slice)]
            sched[-1] = (N_BIG, room, Z_FINISH)
            assert _run(s, sched) == Z_STREAM_END
            s.op("end", s.lib.zs_stream_deflate_end(C.byref(s.zs)))
            assert _decodes(s.out, big, wbits)
            return t.digest()
        return run

    def in_flight(then):
        """deflateEnd or deflateReset while a part runs in the background; the reset stream is used again."""
        def run():
            big = _data("big")
            t = _Trace()
            s = _deflate_init(big, t, 1, 15)
            assert _feed(s, 0, 17 << 20, 65536, Z_NO_FLUSH) == Z_OK
            if then == "end":
                assert s.op("end", s.lib.zs_stream_deflate_end(C.byref(s.zs))) == Z_DATA_ERROR
                return t.digest()
            assert s.op("reset", s.lib.zs_stream_deflate_reset(C.byref(s.zs))) == Z_OK
            s.out = bytearray()
            assert _run(s, _schedule(300_000, 47, 60_000), 17 << 20) == Z_STREAM_END
            s.op("end", s.lib.zs_stream_deflate_end(C.byref(s.zs)))
            assert _decodes(s.out, big[17 << 20: (17 << 20) + 300_000], 15)
            return t.digest()
        return run

    for wname, wbits in WRAPS:
        for level in (0, 1, 6, 9):
            yield f"flush/{wname}/L{level}", flushes(wbits, level, 0, 100 + level)
        for sname, strategy in STRATEGIES:
            yield f"flush/{wname}/{sname}", flushes(wbits, 6, strategy, 200 + strategy)
        for level in (0, 1, 2, 5, 6, 7, 9):
            yield f"whole/{wname}/L{level}", whole(wbits, level, 0)
        for sname, strategy in STRATEGIES:
            yield f"whole/{wname}/{sname}", whole(wbits, 6, strategy)
        yield f"params/{wname}", params(wbits)
        yield f"dict/{wname}/flushes", with_dict(wbits, _schedule(N_MIXED, 300, 150_000))
        yield f"dict/{wname}/whole", with_dict(wbits, [(N_MIXED, 1 << 20, Z_FINISH)])
    for level, strategy in ((0, 0), (1, 0), (6, 0), (9, 0), (6, 2)):
        yield f"gzhead/L{level}/s{strategy}/flushes", gz_header(level, strategy, _schedule(N_MIXED, 400, 150_000))
        yield f"gzhead/L{level}/s{strategy}/whole", gz_header(level, strategy, [(N_MIXED, 1 << 20, Z_FINISH)])
    yield "long/gzip/L1/slices32k/out64k", long_stream(31, 1, 32768, 65536)
    yield "long/zlib/L6/onecall/out64k", long_stream(15, 6, N_BIG, 65536)
    yield "long/raw/L1/slices1m/out1000", long_stream(-15, 1, 1 << 20, 1000)
    yield "inflight/end", in_flight("end")
    yield "inflight/reset", in_flight("reset")


# ---- inflate ---------------------------------------------------------------------------------------

def _inflate_init(src, trace, wbits):
    s = _Stream("inflate", src, trace)
    s.op("init", s.lib.zs_stream_inflate_init(s.ctx.handle, C.byref(s.zs), wbits))
    return s


def _inflate_member(s, pos, n, rng, max_slice):
    """Feeds src[pos:n] in seeded slices with Z_SYNC_FLUSH / Z_FINISH until Z_STREAM_END or an error; returns
    (return code, position after what was consumed)."""
    for _ in range(100000):
        k = min(n - pos, rng.randint(1, max_slice))
        rc, used, made = s.call(pos, k, rng.choice((1000, 65536, 1 << 20)), rng.choice((Z_SYNC_FLUSH, Z_FINISH)))
        pos += used
        if rc not in (Z_OK, Z_BUF_ERROR) or (rc == Z_BUF_ERROR and pos == n and made == 0):
            return rc, pos
    raise AssertionError("inflate loop does not end")


def _compress(data, level, wbits, zdict=None, flush_every=0):
    co = zlib.compressobj(level, zlib.DEFLATED, wbits, zdict=zdict) if zdict else zlib.compressobj(level, zlib.DEFLATED, wbits)
    step = flush_every or len(data) or 1
    out = b""
    for p in range(0, len(data), step):
        out += co.compress(data[p: p + step])
        if flush_every:
            out += co.flush(zlib.Z_SYNC_FLUSH)
    return out + co.flush()


def _gzip_with_header(data):
    """A gzip member whose header has FTEXT, FEXTRA, FNAME, FCOMMENT and FHCRC."""
    extra = b"AB\x04\x00xyz!"
    h = b"\x1f\x8b\x08\x1f" + struct.pack("<I", 0x5f3759df) + b"\x00\x03" + struct.pack("<H", len(extra)) + extra
    h += b"member.txt\0a comment\0"
    h += struct.pack("<H", zlib.crc32(h) & 0xffff)
    return h + _compress(data, 6, -15) + struct.pack("<II", zlib.crc32(data), len(data))


def _texts():
    if "texts" not in _DATA:
        _DATA["texts"] = [make_text(30_000, 51), make_mixed(200_000, 52), make_text(5_000, 53), make_mixed(2_500_000, 54)]
    return _DATA["texts"]


def _inflate_cases():
    """Yields (case id, thunk -> digest) for every inflate case; each thunk asserts what it decodes."""

    def members(seed, max_slice, reset2):
        """Members back to back, with inflateReset (all gzip) or inflateReset2 to a new windowBits between them;
        the input after the last member is handed back."""
        def run():
            texts = _texts()
            rng = random.Random(seed)
            # (windowBits of the inflate, windowBits of the compressor, level)
            fmts = ([(31, 31, 6), (15, 15, 1), (-15, -15, 9), (47, 31, 6), (47, 15, 6), (0, 15, 1)] if reset2 else
                    [(31, 31, 6), (31, 31, 1), (31, 31, 9), (31, 31, 0)])
            parts = [_compress(texts[i % 3], lv, cw, flush_every=7000 if i == 1 else 0) for i, (_, cw, lv) in enumerate(fmts)]
            src = b"".join(parts) + b"trailing bytes"
            t = _Trace()
            s = _inflate_init(src, t, fmts[0][0])
            pos = 0
            for i, (wb, _, _) in enumerate(fmts):
                if i and reset2:
                    s.op("reset2", s.lib.zs_stream_inflate_reset2(C.byref(s.zs), wb))
                elif i:
                    s.op("reset", s.lib.zs_stream_inflate_reset(C.byref(s.zs)))
                s.out = bytearray()
                rc, pos = _inflate_member(s, pos, len(src), rng, max_slice)
                assert rc == Z_STREAM_END and bytes(s.out) == texts[i % 3], (i, rc)
            assert pos == len(src) - len(b"trailing bytes")
            s.op("end", s.lib.zs_stream_inflate_end(C.byref(s.zs)))
            return t.digest()
        return run

    def long_member(wbits, seed):
        """A stream decoded in many attempts: block marks, the window, the trailer checked on the host."""
        def run():
            data = _texts()[3]
            src = _compress(data, 6, wbits, flush_every=300_000)
            t = _Trace()
            s = _inflate_init(src, t, wbits)
            rc, pos = _inflate_member(s, 0, len(src), random.Random(seed), 65536)
            assert rc == Z_STREAM_END and pos == len(src) and bytes(s.out) == data
            s.op("end", s.lib.zs_stream_inflate_end(C.byref(s.zs)))
            return t.digest()
        return run

    def with_dict(wbits):
        def run():
            data, dictionary = _texts()[1], make_text(70_000, 55)
            src = _compress(data, 6, wbits, zdict=dictionary)
            t = _Trace()
            s = _inflate_init(src, t, wbits)
            rng = random.Random(61)

            def setdict(d):
                b = np.frombuffer(d, dtype=np.uint8)
                return s.op("setdict", s.lib.zs_stream_inflate_set_dictionary(C.byref(s.zs), b.ctypes.data, b.size))

            pos = 0
            if wbits < 0:
                assert setdict(dictionary) == Z_OK
            else:
                rc, pos = _inflate_member(s, 0, len(src), rng, 20_000)
                assert rc == Z_NEED_DICT and s.zs.adler == zlib.adler32(dictionary)
                assert setdict(dictionary[1:]) == Z_DATA_ERROR
                assert setdict(dictionary) == Z_OK
            rc, pos = _inflate_member(s, pos, len(src), rng, 20_000)
            assert rc == Z_STREAM_END and pos == len(src) and bytes(s.out) == data
            s.op("end", s.lib.zs_stream_inflate_end(C.byref(s.zs)))
            return t.digest()
        return run

    def get_header():
        """inflateGetHeader fills the caller's struct; inflateReset drops the request."""
        def run():
            texts = _texts()
            src = _gzip_with_header(texts[0]) + _compress(texts[2], 6, 31)
            t = _Trace()
            s = _inflate_init(src, t, 31)
            bufs = [C.create_string_buffer(64) for _ in range(3)]
            h = s.capi.GzHeader(extra=C.addressof(bufs[0]), extra_max=64, name=C.addressof(bufs[1]), name_max=64,
                                comment=C.addressof(bufs[2]), comm_max=64)
            s.op("gethead", s.lib.zs_stream_inflate_get_header(C.byref(s.zs), C.byref(h)))
            rng = random.Random(71)
            rc, pos = _inflate_member(s, 0, len(src), rng, 3000)
            assert rc == Z_STREAM_END and h.done == 1 and bytes(s.out) == texts[0]
            t.h.update(struct.pack("<iIiiIii", h.text, h.time, h.xflags, h.os, h.extra_len, h.hcrc, h.done))
            t.h.update(b"".join(bytes(b) for b in bufs))
            s.op("reset", s.lib.zs_stream_inflate_reset(C.byref(s.zs)))
            h.done = 7
            s.out = bytearray()
            rc, pos = _inflate_member(s, pos, len(src), rng, 3000)
            assert rc == Z_STREAM_END and pos == len(src) and h.done == 7 and bytes(s.out) == texts[2]
            s.op("end", s.lib.zs_stream_inflate_end(C.byref(s.zs)))
            return t.digest()
        return run

    yield "members/reset/slices4k", members(81, 4000, False)
    yield "members/reset/slices64k", members(82, 65536, False)
    yield "members/reset2/slices4k", members(83, 4000, True)
    yield "members/reset2/slices64k", members(84, 65536, True)
    for wname, wbits in WRAPS:
        yield f"long/{wname}", long_member(wbits, 90 + wbits)
    yield "dict/zlib", with_dict(15)
    yield "dict/raw", with_dict(-15)
    yield "gethead", get_header()


def _golden():
    return json.load(open(DIGESTS))


def _ids(gen):
    return [cid for cid, _ in gen()]


@pytest.mark.parametrize("cid", _ids(_deflate_cases))
def test_deflate_trace_is_pinned(gpu_ctx, cid):
    got = dict(_deflate_cases())[cid]()
    assert got == _golden()[cid], cid


@pytest.mark.parametrize("cid", _ids(_inflate_cases))
def test_inflate_trace_is_pinned(gpu_ctx, cid):
    got = dict(_inflate_cases())[cid]()
    assert got == _golden()[cid], cid


# ---- windowBits --------------------------------------------------------------------------------------

WINDOW_BITS = [-17, -16, -15, -8, -7, -1, 0, 7, 8, 15, 16, 31, 32, 47, 48]


def _accepted(wb):
    """inflateReset2's rules (zlib: raw -8..-15, 0 or 8..15 for zlib, +16 gzip, +32 auto below 48), and this engine
    reads raw deflate64 at -16."""
    if wb < 0:
        return wb == -16 or 8 <= -wb <= 15
    if wb < 48:
        wb &= 15
    return wb == 0 or 8 <= wb <= 15


def _initial_adler(wb):
    """What strm->adler holds after inflateInit2 / inflateReset2: 1 while a zlib header may come (wrap & 1), else 0."""
    return 1 if wb >= 0 and ((wb >> 4) + 5) & 1 else 0


@pytest.mark.parametrize("wb", WINDOW_BITS)
def test_window_bits_table(gpu_ctx, wb):
    capi = pkg("capi")
    lib = capi.load()
    want = Z_OK if _accepted(wb) else Z_STREAM_ERROR
    src = np.frombuffer(zlib.compress(b"window bits" * 50), dtype=np.uint8)
    in_off = np.array([0, src.size], dtype=np.uint64)
    out = np.zeros(4096, dtype=np.uint8)
    out_off = np.array([0, out.size], dtype=np.uint64)
    out_len, in_used = np.zeros(1, dtype=np.uint64), np.zeros(1, dtype=np.uint64)
    checks, status = np.zeros(1, dtype=np.uint32), np.zeros(1, dtype=np.int32)
    ptr = lambda a: a.ctypes.data  # noqa: E731
    rc = lib.zs_inflate_batch(gpu_ctx.handle, ptr(src), ptr(in_off), 1, wb, ptr(out), ptr(out_off), ptr(out_len),
                              ptr(in_used), ptr(checks), ptr(status), None, None, 0)
    assert rc == want, ("zs_inflate_batch", wb, rc)

    zs = capi.ZStream()
    rc = lib.zs_stream_inflate_init(gpu_ctx.handle, C.byref(zs), wb)
    assert rc == want, ("zs_stream_inflate_init", wb, rc)
    if rc == Z_OK:
        assert zs.adler == _initial_adler(wb)
        assert lib.zs_stream_inflate_end(C.byref(zs)) == Z_OK

    zs = capi.ZStream()
    assert lib.zs_stream_inflate_init(gpu_ctx.handle, C.byref(zs), 15) == Z_OK
    zs.adler = 12345
    rc = lib.zs_stream_inflate_reset2(C.byref(zs), wb)
    assert rc == want, ("zs_stream_inflate_reset2", wb, rc)
    assert zs.adler == (_initial_adler(wb) if rc == Z_OK else 12345)
    assert lib.zs_stream_inflate_end(C.byref(zs)) == Z_OK


if __name__ == "__main__" and "--write" in sys.argv:
    out = {}
    for gen in (_deflate_cases, _inflate_cases):
        for cid, run in gen():
            out[cid] = run()
            print(cid, out[cid], flush=True)
    with open(DIGESTS, "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
        f.write("\n")
    print(f"{len(out)} digests -> {DIGESTS}")
