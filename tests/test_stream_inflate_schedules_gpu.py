"""GPU: the streaming inflate shim (zs_stream_inflate behind zlib_api.inflate) under call schedules.

The shim decodes in attempts that resume at a block boundary with a 64 KiB window, trims input and
output at the block mark, carries the running checksum and checks the trailer on the host.  Whether a
call runs an attempt depends on the stream's length, the flush value and the wall clock, so a wrong
mark, window or trailer would show only for some schedules.  Every stream here is fed through an
explicit schedule -- (end offset of the slice, output room, flush) per call, seeded -- and compared
with two references driven the same way: the oracle's streaming inflate (the reference's inflate.ts
restated in C) for return codes, msg, totals, adler and the avail_in hand-back, and C zlib for the bytes.

A call with Z_SYNC_FLUSH always runs an attempt, so what is asserted about such a "forced" call does not
depend on timing; of Z_NO_FLUSH calls only schedule-independent results are asserted.
"""
import ctypes as C
import math
import random
import zlib

import pytest

from conftest import make_mixed, make_text, pkg, rand_bytes

pytestmark = pytest.mark.gpu

Z_NO_FLUSH, Z_SYNC_FLUSH, Z_FULL_FLUSH, Z_FINISH = 0, 2, 3, 4
Z_OK, Z_STREAM_END, Z_NEED_DICT, Z_DATA_ERROR, Z_BUF_ERROR = 0, 1, 2, -3, -5
EMPTY_FLUSH = b"\x00\x00\x00\xff\xff"    # an empty non-final stored block: a bare flush point
EVERY_CALL_BELOW = 64 << 10              # the shim runs an attempt on every call while total_in is below this


# ---- the three parties ---------------------------------------------------------------------------

class _Facade:
    """zlib_api: the Python facade over the C ABI."""

    def __init__(self, wbits, head=None):
        self.Z = pkg("zlib_api")
        self.s = self.Z.createInflateStream()
        assert self.Z.inflateInit2_(self.s, wbits) == Z_OK
        if head is not None:
            assert self.Z.inflateGetHeader(self.s, head) == Z_OK

    def call(self, data, room, flush):
        s = self.s
        s.next_in, s.next_in_index, s.avail_in = data, 0, len(data)
        buf = bytearray(room)
        s.next_out, s.next_out_index, s.avail_out = buf, 0, room
        rc = self.Z.inflate(s, flush)
        return rc, s.next_in_index, bytes(buf[: s.next_out_index])

    def set_dictionary(self, d):
        return self.Z.inflateSetDictionary(self.s, d, len(d))

    def reset(self):
        assert self.Z.inflateReset(self.s) == Z_OK

    def end(self):
        assert self.Z.inflateEnd(self.s) == Z_OK

    total_in = property(lambda self: self.s.total_in)
    total_out = property(lambda self: self.s.total_out)
    adler = property(lambda self: self.s._adler)
    msg = property(lambda self: self.s.msg)


class _CAbi:
    """zs_stream_inflate called through ctypes, as a C caller does."""

    def __init__(self, wbits, head=None):
        capi = pkg("capi")
        self.lib = capi.load()
        self.zs = capi.ZStream()
        ctx = pkg("batch").default_context(0)
        assert self.lib.zs_stream_inflate_init(ctx.handle, C.byref(self.zs), wbits) == Z_OK
        assert head is None

    def call(self, data, room, flush):
        zs = self.zs
        ib = (C.c_ubyte * max(len(data), 1)).from_buffer_copy(data or b"\0")
        ob = (C.c_ubyte * max(room, 1))()
        zs.next_in, zs.avail_in, zs.next_out, zs.avail_out = C.addressof(ib), len(data), C.addressof(ob), room
        rc = self.lib.zs_stream_inflate(C.byref(zs), flush)
        return rc, len(data) - zs.avail_in, C.string_at(C.addressof(ob), room - zs.avail_out)

    def set_dictionary(self, d):
        b = (C.c_ubyte * max(len(d), 1)).from_buffer_copy(d or b"\0")
        return self.lib.zs_stream_inflate_set_dictionary(C.byref(self.zs), b, len(d))

    def end(self):
        assert self.lib.zs_stream_inflate_end(C.byref(self.zs)) == Z_OK

    total_in = property(lambda self: self.zs.total_in)
    total_out = property(lambda self: self.zs.total_out)
    adler = property(lambda self: self.zs.adler)
    msg = property(lambda self: (self.zs.msg or b"").decode())


class _Oracle:
    def __init__(self, oracle, wbits):
        self.o = oracle.InflateStream(wbits)
        assert self.o.ret == Z_OK

    def call(self, data, room, flush):
        rc, made, used = self.o.step(data, room, flush)
        return rc, used, made

    def set_dictionary(self, d):
        return self.o.set_dictionary(d)

    def end(self):
        self.o.close()

    total_in = property(lambda self: self.o.total_in)
    total_out = property(lambda self: self.o.total_out)
    adler = property(lambda self: self.o.adler)
    msg = property(lambda self: self.o.msg)


# ---- schedules and the driver ----------------------------------------------------------------------

def random_schedule(rng, n, *, lo=1, hi=65536, forced=0.3, rooms=(1 << 16,), cuts=()):
    """Slices covering [0, n) as (end offset, output room, flush).  Sizes are log-uniform in [lo, hi];
    every offset in `cuts` is a slice end too, and the call that ends there is forced."""
    ends = {c for c in cuts if 0 < c < n}
    forced_at = set(ends)
    pos = 0
    while pos < n:
        pos += max(1, int(math.exp(rng.uniform(math.log(lo), math.log(hi)))))
        if pos < n:
            ends.add(pos)
    ends.add(n)
    return [(e, rng.choice(rooms), Z_SYNC_FLUSH if e in forced_at or rng.random() < forced else Z_NO_FLUSH)
            for e in sorted(ends)]


TERMINAL = (Z_STREAM_END, Z_DATA_ERROR, Z_NEED_DICT, -2, -4)


def drive(party, data, schedule, dictionary=None):
    """Feed `data` through `schedule`; output that does not fit is drained by calls that bring the rest of
    the slice (none once the party holds it).  After the schedule, Z_FINISH calls without input drain and
    end the stream.  Returns a record of the run; `events` holds one entry per schedule step:
    (flush, input offset after the step, bytes delivered after the step, last code)."""
    out = bytearray()
    pos, rc, events, dict_ids, hand_back = 0, Z_OK, [], [], None
    for end, room, flush in schedule:
        piece = data[pos:end]
        while True:
            rc, used, made = party.call(piece, room, flush)
            piece = piece[used:]
            pos += used
            out += made
            if rc == Z_NEED_DICT and dictionary is not None:
                dict_ids.append(party.adler)
                assert party.set_dictionary(dictionary) == Z_OK
                continue
            if rc in TERMINAL or (not piece and len(made) < room) or rc == Z_BUF_ERROR:
                break
        if rc == Z_STREAM_END:
            hand_back = (len(piece), flush)
        events.append((flush, pos, len(out), rc))
        if rc in TERMINAL:
            break
    else:
        for _ in range(1000):
            rc, _, made = party.call(b"", 1 << 20, Z_FINISH)
            out += made
            if rc != Z_OK or not made:
                break
        events.append((Z_FINISH, pos, len(out), rc))
        if rc == Z_STREAM_END:
            hand_back = (0, Z_FINISH)
    r = dict(out=bytes(out), rc=rc, msg=party.msg if rc == Z_DATA_ERROR else "", total_in=party.total_in,
             total_out=party.total_out, adler=party.adler, pos=pos, events=events, dict_ids=dict_ids, hand_back=hand_back)
    party.end()
    return r


def _show(schedule):
    names = {Z_NO_FLUSH: "-", Z_SYNC_FLUSH: "S", Z_FINISH: "F"}
    return " ".join(f"{e}/{room}{names.get(f, f)}" for e, room, f in schedule)


def check_schedule(oracle, data, wbits, schedule, *, seed, expect=None, marks=(), dictionary=None, party=_Facade, head=None):
    """Run `data` through the shim and the oracle with the same schedule and compare everything that does
    not depend on when the shim's attempts run.  `expect` is C zlib's output (None: the oracle's);
    `marks` are the input offsets just behind flush points."""
    why = f"seed {seed}, wbits {wbits}, {len(data)} bytes, schedule [{_show(schedule)}]"
    g = drive(party(wbits, head), data, schedule, dictionary)
    o = drive(_Oracle(oracle, wbits), data, schedule, dictionary)
    assert g["rc"] == o["rc"], (g["rc"], g["msg"], o["rc"], o["msg"], why)
    assert g["msg"] == o["msg"], why
    if expect is not None and g["rc"] != Z_DATA_ERROR:
        assert o["out"] == expect, "the oracle disagrees with C zlib: " + why
    assert len(g["out"]) == len(o["out"]) and g["out"] == o["out"], (len(g["out"]), len(o["out"]), why)
    assert g["total_out"] == o["total_out"] == len(o["out"]), why
    assert g["dict_ids"] == o["dict_ids"], why
    if g["rc"] in (Z_STREAM_END, Z_BUF_ERROR):
        # (the reference, like C zlib, leaves the bytes read by the call that returned Z_NEED_DICT out of total_in;
        # the shim counts every byte it consumed)
        want = o["pos"] if o["dict_ids"] else o["total_in"]
        assert g["total_in"] == want, (g["total_in"], want, why)
    if g["rc"] == Z_STREAM_END:
        if wbits >= 0:
            assert g["adler"] == o["adler"], (hex(g["adler"]), hex(o["adler"]), why)
        # the avail_in hand-back is exact on a forced call, and on every call while the stream is short
        if g["hand_back"][1] != Z_NO_FLUSH or len(data) < EVERY_CALL_BELOW:
            assert g["hand_back"][0] == o["hand_back"][0] and g["pos"] == o["pos"], (g["hand_back"], o["hand_back"], why)
    # flush-point floor: what precedes a flush point is final once a call has consumed it -- a forced call, or one
    # whose input ends with the flush marker, which the shim decodes whatever the pace
    marks = set(marks)
    for flush, pos, delivered, rc in g["events"]:
        if pos in marks and rc in (Z_OK, Z_BUF_ERROR):
            floor = len(zlib.decompressobj(wbits).decompress(data[:pos]))
            assert delivered == floor, (pos, delivered, floor, why)
    return g


# ---- streams ---------------------------------------------------------------------------------------

def flushed_stream(data, wbits, rng, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, n_flush=6):
    """C zlib's stream of `data` with sync and full flush points at random places, some followed by a bare
    empty flush.  Returns (stream, offsets just behind each flush point)."""
    co = zlib.compressobj(level, zlib.DEFLATED, wbits, 8, strategy)
    out, marks, prev = bytearray(), [], 0
    for cut in sorted(rng.sample(range(1, len(data)), n_flush)):
        out += co.compress(data[prev:cut]) + co.flush(rng.choice((zlib.Z_SYNC_FLUSH, zlib.Z_FULL_FLUSH)))
        marks.append(len(out))
        if rng.random() < 0.4:
            out += EMPTY_FLUSH
            marks.append(len(out))
        prev = cut
    out += co.compress(data[prev:]) + co.flush()
    return bytes(out), marks


def _wrap_of(wbits):
    return "raw" if wbits < 0 else "gzip" if wbits & 16 else "zlib"


MATRIX = ([(w, lvl, zlib.Z_DEFAULT_STRATEGY) for w in (15, 31, -15) for lvl in (0, 1, 6, 9)]
          + [(15, 6, s) for s in (zlib.Z_FIXED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE)])


@pytest.mark.parametrize("wbits,level,strategy", MATRIX, ids=[f"{_wrap_of(w)}-L{l}-s{s}" for w, l, s in MATRIX])
def test_formats_levels_strategies(gpu_ctx, oracle, wbits, level, strategy):
    for seed in range(level * 10 + strategy, 400, 100):
        rng = random.Random(seed)
        data = make_text(rng.randrange(120000, 260000), seed) + rand_bytes(rng.randrange(1, 5000), seed)
        stream, marks = flushed_stream(data, wbits, rng, level, strategy)
        sched = random_schedule(rng, len(stream), lo=64, hi=40000, forced=0.3, rooms=(1 << 16, 4096, 1 << 20),
                                cuts=marks + [len(stream) - 3, len(stream) - 9])
        check_schedule(oracle, stream, wbits, sched, seed=seed, expect=data, marks=marks)


WBITS = [(0, 15), (9, 9), (10, 10), (11, 11), (12, 12), (13, 13), (14, 14), (15, 15), (31, 31), (47, 15), (47, 31)] + \
        [(-w, -w) for w in range(9, 16)]


@pytest.mark.parametrize("wbits,enc", WBITS, ids=[f"{w}<-{e}" for w, e in WBITS])
def test_inflate_init2_window_bits(gpu_ctx, oracle, wbits, enc):
    """inflateInit2_ windowBits 0, 9-15, 31, 47 and -9 ... -15, each fed a stream written with a matching window."""
    seed = 1000 + wbits * 7 + enc
    rng = random.Random(seed)
    data = make_text(90000, seed)
    stream, marks = flushed_stream(data, enc, rng, 6, n_flush=3)
    sched = random_schedule(rng, len(stream), lo=16, hi=20000, forced=0.4, cuts=marks + [2, 10])
    check_schedule(oracle, stream, wbits, sched, seed=seed, expect=data, marks=marks)


def test_flush_points_every_call_forced_and_through_the_c_abi(gpu_ctx, oracle):
    """Many flush points, each ended exactly by a forced call: everything before it must be delivered.  The same
    schedules run through the C ABI."""
    for seed, wbits in ((7, 15), (8, 31), (9, -15)):
        rng = random.Random(seed)
        data = make_text(400000, seed)
        stream, marks = flushed_stream(data, wbits, rng, 6, n_flush=40)
        sched = [(m, 1 << 20, Z_SYNC_FLUSH) for m in marks] + [(len(stream), 1 << 20, Z_SYNC_FLUSH)]
        check_schedule(oracle, stream, wbits, sched, seed=seed, expect=data, marks=marks)
        sched = random_schedule(rng, len(stream), lo=1000, hi=50000, forced=0.5, cuts=marks[::3])
        check_schedule(oracle, stream, wbits, sched, seed=seed, expect=data, marks=marks, party=_CAbi)


class _Bits:
    """Deflate bit writer, enough for fixed-Huffman and stored blocks."""

    def __init__(self):
        self.out, self.acc, self.n = bytearray(), 0, 0

    def put(self, v, n):
        self.acc |= v << self.n
        self.n += n
        while self.n >= 8:
            self.out.append(self.acc & 255)
            self.acc >>= 8
            self.n -= 8

    def code(self, c, n):                     # Huffman codes go most significant bit first
        self.put(int(format(c, f"0{n}b")[::-1], 2), n)

    def literal(self, b):
        if b < 144:
            self.code(0x30 + b, 8)
        else:
            self.code(0x190 + b - 144, 9)

    def fixed(self, lits, final=False, matches=()):
        self.put(int(final), 1)
        self.put(1, 2)
        for b in lits:
            self.literal(b)
        for (lsym, lextra, lxbits, dcode, dextra, dxbits) in matches:
            self.code(0xC0 + lsym - 280, 8) if lsym >= 280 else self.code(lsym - 256, 7)
            self.put(lextra, lxbits)
            self.code(dcode, 5)
            self.put(dextra, dxbits)
        self.code(0, 7)

    def stored(self, data, final=False):
        """Returns the offset of the byte holding the block header."""
        at = len(self.out)
        self.put(int(final), 1)
        self.put(0, 2)
        if self.n:
            self.put(0, 8 - self.n)
        self.out += len(data).to_bytes(2, "little") + (len(data) ^ 0xFFFF).to_bytes(2, "little") + data
        return at

    def done(self):
        if self.n:
            self.put(0, 8 - self.n)
        return bytes(self.out)


def test_stored_block_length_field_and_header_bits(gpu_ctx, oracle):
    """A 65 535-byte stored block whose header starts at each of the 8 bit positions of a byte, behind a fixed
    block, followed by a fixed block and a final block that copies 258 bytes from 32 768 back, into the stored
    data.  Slices end at every byte of the stored header and its LEN/NLEN field, and at every byte of the next
    block's header."""
    rng = random.Random(65535)
    payload = rng.randbytes(65535)
    for high in range(8):                       # literals of 9 bits move the stored header's bit position
        w = _Bits()
        w.fixed(b"abc" + bytes([200] * high))
        hdr = w.stored(payload)
        next_hdr = len(w.out)
        w.fixed(b"xyz" + bytes([150, 250]))
        w.fixed(b"!", final=True, matches=[(285, 0, 0, 29, 32768 - 24577, 13), (265, 0, 1, 13, 100 - 97, 5)])
        stream = w.done()
        expect = zlib.decompressobj(-15).decompress(stream)
        assert len(expect) == 3 + high + 65535 + 5 + 1 + 258 + 11
        cuts = list(range(hdr, hdr + 7)) + list(range(next_hdr - 1, next_hdr + 4))
        seed = 500 + high
        for c in cuts:
            sched = [(c, 1 << 17, Z_SYNC_FLUSH), (c + 1 + (c * 7) % 300, 1 << 17, Z_SYNC_FLUSH), (len(stream), 1 << 17, Z_SYNC_FLUSH)]
            check_schedule(oracle, stream, -15, sorted(set(sched)), seed=seed, expect=expect)
        sched = [(c, 1 << 17, Z_SYNC_FLUSH) for c in cuts] + [(len(stream), 1 << 17, Z_SYNC_FLUSH)]
        check_schedule(oracle, stream, -15, sched, seed=seed, expect=expect)
        sched = random_schedule(rng, len(stream), lo=1, hi=30000, forced=0.5)
        check_schedule(oracle, stream, -15, sched, seed=seed, expect=expect)


def _gzip_member(body, flg, level=6):
    h = bytes([0x1F, 0x8B, 8, flg]) + (123456789).to_bytes(4, "little") + b"\x00\x03"
    if flg & 4:
        h += (5).to_bytes(2, "little") + b"ab\x00cd"
    if flg & 8:
        h += b"name.txt\x00"
    if flg & 16:
        h += b"a comment\x00"
    if flg & 2:
        h += (zlib.crc32(h) & 0xFFFF).to_bytes(2, "little")
    co = zlib.compressobj(level, zlib.DEFLATED, -15)
    return h, h + co.compress(body) + co.flush() + zlib.crc32(body).to_bytes(4, "little") + len(body).to_bytes(4, "little")


@pytest.mark.parametrize("flg", [0, 2, 4, 8, 16, 30])
def test_gzip_header_fields_one_byte_at_a_time(gpu_ctx, oracle, flg):
    """FEXTRA / FNAME / FCOMMENT / FHCRC headers fed one byte per call, read back with inflateGetHeader."""
    Z = pkg("zlib_api")
    seed = 300 + flg
    rng = random.Random(seed)
    body = make_text(150000, seed)
    h, member = _gzip_member(body, flg)
    for wbits in (31, 47):
        head = Z.GzipHeader(extra_max=16, name_max=32, comm_max=32)
        sched = [(i, 1 << 16, Z_NO_FLUSH) for i in range(1, len(h) + 3)]
        sched += [s for s in random_schedule(rng, len(member), lo=100, hi=30000, forced=0.3, cuts=[len(member) - 5])
                  if s[0] > len(h) + 2]
        check_schedule(oracle, member, wbits, sched, seed=seed, expect=body, head=head)
        assert head._done == 1
        assert (head._time, head._os, head._hcrc, head._text) == (123456789, 3, (flg >> 1) & 1, 0)
        assert head._extra == (b"ab\x00cd" if flg & 4 else b"") and head._extra_len == (5 if flg & 4 else 0)
        assert head._name == (b"name.txt" if flg & 8 else b"") and head._comment == (b"a comment" if flg & 16 else b"")


@pytest.mark.parametrize("wbits", [15, -15])
def test_preset_dictionary_across_resume_points(gpu_ctx, oracle, wbits):
    """A zlib stream with FDICT (Z_NEED_DICT, adler = DICTID, then inflateSetDictionary), and a raw stream whose
    dictionary is set before any data.  The body is cut by sync flushes and keeps copying from the dictionary,
    so matches into it are decoded after resume points."""
    seed = 77 + wbits
    rng = random.Random(seed)
    dic = make_text(20000, 5)
    body = b"".join(rng.randbytes(rng.randrange(50, 400)) + dic[-rng.randrange(600, 8000):][:300] for _ in range(40))
    assert len(body) < 24000
    co = zlib.compressobj(6, zlib.DEFLATED, wbits, 8, 0, zdict=dic)
    stream, marks = bytearray(), []
    for i in range(0, len(body), 2000):
        stream += co.compress(body[i: i + 2000]) + co.flush(zlib.Z_SYNC_FLUSH)
        marks.append(len(stream))
    stream = bytes(stream + co.flush())
    assert len(stream) < len(zlib.compress(body, 6)) - 2000          # the dictionary is used
    for trial in range(6):
        sched = random_schedule(rng, len(stream), lo=1, hi=3000, forced=0.5, cuts=marks[trial::3] + [1, 3, 6])
        for party in (_Facade, _CAbi):
            if wbits < 0:
                g = party(wbits)
                assert g.set_dictionary(dic) == Z_OK
                o = _Oracle(oracle, wbits)
                assert o.set_dictionary(dic) == Z_OK
                gr, orr = drive(g, stream, sched), drive(o, stream, sched)
                assert gr["rc"] == orr["rc"] == Z_STREAM_END and gr["out"] == orr["out"] == body, (seed, trial, _show(sched))
                continue
            g = check_schedule(oracle, stream, wbits, sched, seed=seed, expect=body, dictionary=dic, party=party)
            assert g["dict_ids"] == [zlib.adler32(dic)]


def test_deflate64_window_across_resume_points(gpu_ctx, oracle):
    """deflate64 (windowBits -16): matches reach 40-60 KiB back, across resume points, into the 64 KiB window."""
    for seed in (64, 65):
        rng = random.Random(seed)
        again = rng.randbytes(6000)
        data = b"".join(again + rng.randbytes(rng.randrange(36000, 54000)) for i in range(9))
        stream = oracle.deflate64_encode(data)
        assert len(stream) < len(data) - 20000                    # the far copies are used (random bytes alone grow)
        ret, ref, used, _ = oracle.inflate(stream, -16, len(data) + 64)
        assert ret == Z_STREAM_END and ref == data and used == len(stream)
        for trial in range(3):
            sched = random_schedule(rng, len(stream), lo=500, hi=60000, forced=0.6, rooms=(1 << 16, 1 << 20))
            check_schedule(oracle, stream, -16, sched, seed=seed)


LONG = [("mixed-zlib", 15, 0, 0), ("text-gzip", 31, 0, 0), ("mixed-raw-flushed", -15, 1, 0), ("text-zlib-flushed", 15, 1, 0),
        ("mixed-zlib", 15, 0, 1), ("mixed-raw-flushed", -15, 1, 1)]


@pytest.mark.parametrize("name,wbits,flushed,serial", LONG, ids=[x[0] + ("-serial" if x[3] else "") for x in LONG])
def test_multi_mib_streams(gpu_ctx, oracle, monkeypatch, name, wbits, flushed, serial):
    """Multi-MiB streams: attempts above 128 KiB go through the segment-parallel decoder, inflate_kernel continues
    behind it.  With ZS_INFLATE_SERIAL=1 the same schedules, one stream with and one without flush points, take the
    serial decoder only: both paths are held to the same reference."""
    if serial:
        monkeypatch.setenv("ZS_INFLATE_SERIAL", "1")
    seed = sum(map(ord, name))
    rng = random.Random(seed)
    data = (make_mixed if name.startswith("mixed") else make_text)(rng.randrange(3 << 20, 4 << 20), seed)
    if flushed:
        stream, marks = flushed_stream(data, wbits, rng, 6, n_flush=12)
    else:
        co = zlib.compressobj(6, zlib.DEFLATED, wbits)
        stream, marks = co.compress(data) + co.flush(), []
    for trial in range(4):
        sched = random_schedule(rng, len(stream), lo=16 << 10, hi=1 << 20, forced=0.25, rooms=(1 << 20, 4 << 20),
                                cuts=marks[trial::4] + [len(stream) - 2])
        check_schedule(oracle, stream, wbits, sched, seed=seed, expect=data, marks=marks)


@pytest.mark.parametrize("wbits", [15, 31, -15])
def test_corrupt_and_truncated_streams_under_schedules(gpu_ctx, oracle, wbits):
    """1-3 MiB streams with a flipped bit in the body, stomped header and trailer bytes, or cut at random points and
    inside the trailer, each fed with random slicing: verdict, message and the bytes before the error are the
    oracle's whatever the schedule."""
    seed = 4000 + wbits
    rng = random.Random(seed)
    data = make_mixed(rng.randrange(3 << 20, 5 << 20), seed)
    co = zlib.compressobj(6, zlib.DEFLATED, wbits)
    stream = co.compress(data) + co.flush()
    assert (1 << 20) < len(stream) < (3 << 20)
    T = {15: 4, 31: 8, -15: 0}[wbits]
    H = {15: 2, 31: 10, -15: 0}[wbits]
    cases = []
    for _ in range(6):
        b = bytearray(stream)
        b[rng.randrange(H + 1000, len(stream) - T - 10)] ^= 1 << rng.randrange(8)
        cases.append(("bit flip", bytes(b)))
    for at in ([0, 1, 2, 3] if H else [0])[:2] + ([len(stream) - 1, len(stream) - T] if T else []):
        b = bytearray(stream)
        b[at] ^= 0x5A
        cases.append((f"byte {at} stomped", bytes(b)))
    for cut in [rng.randrange(H + 1, len(stream)) for _ in range(2)] + ([len(stream) - 1, len(stream) - T + 1] if T else [len(stream) - 1]):
        cases.append((f"cut at {cut}", stream[:cut]))
    for what, src in cases:
        sched = random_schedule(rng, len(src), lo=8 << 10, hi=1 << 20, forced=0.3, rooms=(1 << 20,))
        check_schedule(oracle, src, wbits, sched, seed=f"{seed} ({what})")


def test_multi_member_gzip_under_both_continuation_idioms(gpu_ctx):
    """Three gzip members -- over 1 MiB compressed, empty, 20 KB -- back to back.  Fed in 32 KiB Z_NO_FLUSH slices
    and continued by total_in (test-multistream.ts, INTEGRATION.md), and with every call forced, continued by
    next_in / avail_in after inflateReset (C zlib's idiom)."""
    bodies = [make_mixed(3 << 20, 9), b"", make_text(20000, 10)]
    members = [zlib.compress(b, 6, 31) for b in bodies]
    assert len(members[0]) > (1 << 20)
    blob = b"".join(members)
    # by total_in
    g = _Facade(31)
    base, totals = 0, []
    for body in bodies:
        out, pos, rc = bytearray(), base, Z_OK
        while rc != Z_STREAM_END:
            piece = blob[pos: pos + 32768]
            rc, used, made = g.call(piece, 1 << 16, Z_NO_FLUSH if piece else Z_FINISH)
            out += made
            pos += used
            assert rc in (Z_OK, Z_STREAM_END), (rc, g.msg)
        totals.append(g.total_in)
        assert bytes(out) == body
        base += g.total_in
        g.reset()
    assert totals == [len(m) for m in members] and sum(totals) == len(blob)
    g.end()
    # by next_in / avail_in, every call forced
    rng = random.Random(3)
    g = _Facade(31)
    sched = random_schedule(rng, len(blob), lo=1000, hi=200000, forced=1.0, cuts=[len(members[0]) - 2, len(members[0]) + 10])
    pos, k, out = 0, 0, bytearray()
    for end, room, flush in sched:
        piece = blob[pos:end]
        while True:
            rc, used, made = g.call(piece, room, flush)
            piece, pos, out = piece[used:], pos + used, out + made
            assert rc in (Z_OK, Z_STREAM_END, Z_BUF_ERROR), (rc, g.msg)
            if rc == Z_STREAM_END:
                assert bytes(out) == bodies[k] and pos == sum(map(len, members[: k + 1])), (k, pos, _show(sched))
                k, out = k + 1, bytearray()
                g.reset()
                if not piece:
                    break
                continue
            if not piece and len(made) < room:
                break
    assert k == 3 and pos == len(blob)
    g.end()


# ---- request/response peers and the trailer ----------------------------------------------------------

@pytest.mark.parametrize("variant", ["whole", "marker-alone", "marker-split", "full-flush"])
@pytest.mark.parametrize("wbits", [15, -15])
def test_sync_flushed_messages_are_delivered_by_the_call_that_completes_them(gpu_ctx, wbits, variant):
    """A permessage-deflate style peer: 300 messages of 1-6 KiB, each ended by a sync (or full) flush, one
    inflate(Z_NO_FLUSH) call per message, back to back.  Each call that completes a message must deliver it --
    the peer waits for the reply before it sends more -- also when the 4-byte marker comes in a call of its own
    or split 2 + 2 across two calls, and long after the stream passed the every-call threshold."""
    rng = random.Random(11 if wbits > 0 else 12)
    text = make_text(2 << 20, 13)
    co = zlib.compressobj(6, zlib.DEFLATED, wbits)
    mode = zlib.Z_FULL_FLUSH if variant == "full-flush" else zlib.Z_SYNC_FLUSH
    msgs, wires, at = [], [], 0
    for _ in range(300):
        n = rng.randrange(1024, 6 * 1024 + 1)
        msgs.append(text[at: at + n])
        at += n
        w = co.compress(msgs[-1]) + co.flush(mode)
        assert w.endswith(b"\x00\x00\xff\xff")
        wires.append(w)
    assert sum(map(len, wires)) > (3 << 16)
    g = _Facade(wbits)
    got, want = bytearray(), bytearray()
    for i, w in enumerate(wires):
        calls = {"marker-alone": [w[:-4], w[-4:]], "marker-split": [w[:-2], w[-2:]]}.get(variant, [w])
        for c in calls:
            rc, used, made = g.call(c, 1 << 16, Z_NO_FLUSH)
            assert rc == Z_OK and used == len(c), (i, rc, g.msg)
            got += made
        want += msgs[i]
        assert len(got) == len(want), f"message {i} ({len(msgs[i])} bytes): {len(got) - len(want) + len(msgs[i])} delivered by its call"
        assert got == want, i
    g.end()


@pytest.mark.parametrize("wbits,corrupt", [(15, None), (15, "check"), (31, None), (31, "check"), (31, "length")])
def test_call_that_completes_the_trailer_ends_the_stream(gpu_ctx, wbits, corrupt):
    """The last block is decoded by a forced call that lacks the last 3 trailer bytes; the next, immediate
    Z_NO_FLUSH call brings them and 16 bytes of what follows.  It must end the stream -- Z_STREAM_END, the
    16 bytes handed back through avail_in, total_in and adler exact -- or give the trailer's verdict.  (A wrong
    gzip CRC is held back with the ISIZE behind it: C zlib judges the CRC as soon as its 4 bytes are in.)  The
    calls go through the C ABI, back to back as a C caller makes them."""
    data = make_mixed(3 << 20, 21)
    co = zlib.compressobj(6, zlib.DEFLATED, wbits)
    stream = bytearray(co.compress(data) + co.flush())
    assert len(stream) >= (1 << 20)
    if corrupt == "check":
        stream[-8 if wbits == 31 else -1] ^= 0x10
    elif corrupt == "length":
        stream[-1] ^= 0x10
    stream = bytes(stream)
    g = _CAbi(wbits)
    out = []
    head = len(stream) - (7 if corrupt == "check" and wbits == 31 else 3)
    tail = stream[head:] + b"G" * 16
    ends = list(range(32768, head - (512 << 10), 32768)) + [head]
    for pos, end in zip([0] + ends, ends):
        # the last 512 KiB come in one forced call with room for all of the output: no drain call follows it
        rc, used, made = g.call(stream[pos:end], 4 << 20, Z_SYNC_FLUSH if end == head else Z_NO_FLUSH)
        assert rc == Z_OK and used == end - pos, (rc, g.msg)
        out.append(made)
    rc, used, made = g.call(tail, 1 << 16, Z_NO_FLUSH)
    assert b"".join(out) == data and made == b""   # the forced call decoded the last block
    if corrupt:
        assert rc == Z_DATA_ERROR, f"{rc} instead of Z_DATA_ERROR"
        assert g.msg == ("incorrect length check" if corrupt == "length" else "incorrect data check")
    else:
        assert rc == Z_STREAM_END, f"{rc} instead of Z_STREAM_END"
        assert len(tail) - used == 16 and g.total_in == len(stream)
        assert g.adler == (zlib.adler32(data) if wbits == 15 else zlib.crc32(data))
    g.end()
