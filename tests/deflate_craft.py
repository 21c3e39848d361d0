"""A deflate writer for tests (RFC 1951), and the hand-built streams the inflate tests share.

C zlib writes a narrow set of code shapes: its distance tree always has two codes or more, it writes length 258
as code 285, its code-length repeats never cross from the literal/length lengths into the distance lengths,
and its code-length code stays below 7 bits.  The writer here lets a test choose every one of those things:
block types and BFINAL, the literal/length and distance code lengths (incomplete sets included), the
run-length coded length sequence with HLIT / HDIST / HCLEN and the code-length code, the length code of a
match, and raw code words.

splice() joins byte-aligned pieces into one stream.  A piece is C zlib bulk data (its own compressobj(-15)
ended by Z_SYNC_FLUSH) or a crafted group of blocks ended by an empty stored block, so crafted blocks can sit
behind 32 KiB of history, deep inside a multi-MiB stream, and still be written in a fraction of a second.
"""
from __future__ import annotations

import heapq
import random
import struct
import zlib
from dataclasses import dataclass

CL_ORDER = (16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15)
LEN_BASE = (3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195,
            227, 258)
LEN_EXTRA = (0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0)
DIST_BASE = (1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073,
             4097, 6145, 8193, 12289, 16385, 24577)
DIST_EXTRA = (0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13)
FIXED_LIT = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
FIXED_DIST = [5] * 32
EOB = 256


# ---- bits and codes ---------------------------------------------------------------------------------

class BitWriter:
    """LSB-first fields, MSB-first Huffman codes."""

    def __init__(self):
        self.out, self.acc, self.k = bytearray(), 0, 0

    @property
    def n(self) -> int:
        """Bits written so far."""
        return len(self.out) * 8 + self.k

    def bits(self, val: int, k: int):
        assert 0 <= val < (1 << k) or k == 0 and val == 0, (val, k)
        self.acc |= val << self.k
        self.k += k
        while self.k >= 8:
            self.out.append(self.acc & 255)
            self.acc >>= 8
            self.k -= 8

    def code(self, c: int, k: int):
        self.bits(int(format(c, f"0{k}b")[::-1], 2) if k else 0, k)

    def align(self):
        if self.k:
            self.bits(0, 8 - self.k)

    def raw(self, data: bytes):
        """Whole bytes at a byte boundary."""
        assert self.k == 0
        self.out += data

    def data(self, fill: int = 0) -> bytes:
        """The bytes written so far; the unused high bits of the last byte are `fill` (0 or 1 each)."""
        if not self.k:
            return bytes(self.out)
        pad = (((1 << (8 - self.k)) - 1) << self.k) if fill else 0
        return bytes(self.out) + bytes([(self.acc | pad) & 255])


def canonical(lens) -> list:
    """Canonical codes (RFC 1951 3.2.2) of a length list; None for length 0.  Incomplete sets are allowed; an
    over-subscribed set gives codes that do not fit their length, which the caller can still write."""
    count = [0] * 16
    for l in lens:
        count[l] += 1
    count[0] = 0
    nxt, code = [0] * 16, 0
    for b in range(1, 16):
        code = (code + count[b - 1]) << 1
        nxt[b] = code
    out = []
    for l in lens:
        if l:
            out.append(nxt[l])
            nxt[l] += 1
        else:
            out.append(None)
    return out


def huffman_lengths(freqs, limit: int) -> list:
    """Huffman code lengths of `freqs` no longer than `limit` (frequencies are flattened until they fit).  A set
    with one used symbol gets a second one, so the code is complete."""
    f = list(freqs)
    used = [i for i, x in enumerate(f) if x]
    if len(used) == 1:
        f[0 if used[0] else 1] = 1
    while True:
        heap = [(x, i, (i,)) for i, x in enumerate(f) if x]
        heapq.heapify(heap)
        lens = [0] * len(f)
        k = len(f)
        while len(heap) > 1:
            a, b = heapq.heappop(heap), heapq.heappop(heap)
            for s in a[2] + b[2]:
                lens[s] += 1
            heapq.heappush(heap, (a[0] + b[0], k, a[2] + b[2]))
            k += 1
        if max(lens) <= limit:
            return lens
        f = [(x >> 1) + 1 if x else 0 for x in f]


def length_code(n: int) -> tuple:
    """(symbol, extra value, extra bits) of match length n; 258 is code 285."""
    if n == 258:
        return 285, 0, 0
    i = max(k for k in range(28) if LEN_BASE[k] <= n)
    return 257 + i, n - LEN_BASE[i], LEN_EXTRA[i]


def dist_code(d: int) -> tuple:
    i = max(k for k in range(30) if DIST_BASE[k] <= d)
    assert d - DIST_BASE[i] < (1 << DIST_EXTRA[i]), d
    return i, d - DIST_BASE[i], DIST_EXTRA[i]


# ---- symbols ----------------------------------------------------------------------------------------

@dataclass
class Match:
    length: int
    dist: int
    lsym: int | None = None          # force the length code (284 + 31 extra bits for 258)


@dataclass
class Sym:
    """A literal/length code word with nothing after it (e.g. symbol 286 of a fixed block)."""
    sym: int


@dataclass
class DSym:
    """A distance code word with `extra` on `xbits` bits after it."""
    sym: int
    extra: int = 0
    xbits: int = 0


@dataclass
class Bits:
    """Raw bits (LSB first): the unused slot of a one-code set, a code word of an empty set."""
    val: int
    n: int


def rle(lens, cross: bool = True, split: int | None = None) -> list:
    """Run-length code (16/17/18) for a length sequence as [(symbol, extra value)].  cross=False codes the first
    `split` lengths and the rest separately, as C zlib does; cross=True lets runs run over that boundary."""
    if not cross:
        return rle(lens[:split]) + rle(lens[split:])
    out, i, n = [], 0, len(lens)
    while i < n:
        v, j = lens[i], i
        while j < n and lens[j] == v:
            j += 1
        run = j - i
        if v == 0:
            while run >= 11:
                k = min(run, 138)
                out.append((18, k - 11)); run -= k
            if run >= 3:
                out.append((17, run - 3)); run = 0
            out += [(0, 0)] * run
        else:
            out.append((v, 0)); run -= 1
            while run >= 3:
                k = min(run, 6)
                out.append((16, k - 3)); run -= k
            out += [(v, 0)] * run
        i = j
    return out


def rle_expand(seq, total: int) -> list:
    """The lengths an RLE sequence stands for (for a valid sequence)."""
    out = []
    for s, x in seq:
        if s < 16:
            out.append(s)
        elif s == 16:
            out += [out[-1]] * (3 + x)
        else:
            out += [0] * ((3 if s == 17 else 11) + x)
    assert len(out) == total, (len(out), total)
    return out


# ---- blocks -----------------------------------------------------------------------------------------

class Deflate:
    """Raw deflate, block by block.  Every block's BFINAL is explicit."""

    def __init__(self):
        self.w = BitWriter()

    def _symbols(self, symbols, lcodes, llens, dcodes, dlens):
        w = self.w
        for s in symbols:
            if isinstance(s, int):
                w.code(lcodes[s], llens[s])
            elif isinstance(s, Match):
                sym, x, xb = length_code(s.length)
                if s.lsym is not None:
                    sym = s.lsym
                    x, xb = s.length - LEN_BASE[sym - 257], LEN_EXTRA[sym - 257]
                w.code(lcodes[sym], llens[sym])
                w.bits(x, xb)
                ds, dx, dxb = dist_code(s.dist)
                w.code(dcodes[ds], dlens[ds])
                w.bits(dx, dxb)
            elif isinstance(s, Sym):
                w.code(lcodes[s.sym], llens[s.sym])
            elif isinstance(s, DSym):
                w.code(dcodes[s.sym], dlens[s.sym])
                w.bits(s.extra, s.xbits)
            elif isinstance(s, Bits):
                w.bits(s.val, s.n)
            else:
                raise TypeError(s)

    def stored(self, data: bytes, final: bool = False, nlen: int | None = None):
        self.w.bits(int(final), 1)
        self.w.bits(0, 2)
        self.w.align()
        n = len(data)
        self.w.bits(n, 16)
        self.w.bits((n ^ 0xFFFF) if nlen is None else nlen, 16)
        self.w.raw(data)
        return self

    def sync(self):
        """An empty non-final stored block: a flush point that leaves the writer byte aligned."""
        return self.stored(b"")

    def fixed(self, symbols, final: bool = False, eob: bool = True):
        self.w.bits(int(final), 1)
        self.w.bits(1, 2)
        self._symbols(list(symbols) + ([EOB] if eob else []), canonical(FIXED_LIT), FIXED_LIT,
                      canonical(FIXED_DIST), FIXED_DIST)
        return self

    def dynamic(self, lit_lens, dist_lens, symbols, final: bool = False, eob: bool = True, seq=None, cl_lens=None,
                hlit: int | None = None, hdist: int | None = None, hclen: int | None = None, cross: bool = True,
                btype: int = 2):
        """A dynamic block.  lit_lens / dist_lens are padded with zeros to HLIT / HDIST (default: just past the last
        used symbol, at least 257 / 1).  seq is the run-length coded sequence [(symbol, extra)] (default rle());
        cl_lens the 19 code-length code lengths by symbol (default: a Huffman code of seq, at most 7 bits); hclen
        the count of lengths written in CL_ORDER (default: the fewest that cover cl_lens)."""
        lit = list(lit_lens)
        dist = list(dist_lens)
        if hlit is None:
            hlit = max(257, max((i + 1 for i, l in enumerate(lit) if l), default=0))
        if hdist is None:
            hdist = max(1, max((i + 1 for i, l in enumerate(dist) if l), default=0))
        lit = (lit + [0] * 288)[:max(hlit, 288)]
        dist = (dist + [0] * 32)[:max(hdist, 32)]
        if seq is None:
            seq = rle(lit[:hlit] + dist[:hdist], cross, hlit)
        if cl_lens is None:
            freq = [0] * 19
            for s, _ in seq:
                freq[s] += 1
            cl_lens = huffman_lengths(freq, 7)
        if hclen is None:
            hclen = max(4, max((k + 1 for k, s in enumerate(CL_ORDER) if cl_lens[s]), default=0))
        w = self.w
        w.bits(int(final), 1)
        w.bits(btype, 2)
        w.bits(hlit - 257, 5)
        w.bits(hdist - 1, 5)
        w.bits(hclen - 4, 4)
        for k in range(hclen):
            w.bits(cl_lens[CL_ORDER[k]], 3)
        ccodes = canonical(cl_lens)
        for s, x in seq:
            w.code(ccodes[s], cl_lens[s])
            if s >= 16:
                w.bits(x, {16: 2, 17: 3, 18: 7}[s])
        self._symbols(list(symbols) + ([EOB] if eob else []), canonical(lit), lit, canonical(dist), dist)
        return self

    def bits(self, val: int, n: int):
        self.w.bits(val, n)
        return self

    def data(self, fill: int = 0) -> bytes:
        return self.w.data(fill)


# ---- wrappers and splicing ---------------------------------------------------------------------------

def _decoded(body: bytes, dictionary=None) -> bytes:
    d = zlib.decompressobj(-15, zdict=dictionary) if dictionary else zlib.decompressobj(-15)
    try:
        return d.decompress(body)
    except zlib.error:
        return b""


def zlib_wrap(body: bytes) -> bytes:
    return b"\x78\x9c" + body + struct.pack(">I", zlib.adler32(_decoded(body)))


def gzip_wrap(body: bytes) -> bytes:
    out = _decoded(body)
    return b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x00\x03" + body + struct.pack("<II", zlib.crc32(out), len(out) & 0xFFFFFFFF)


def wrap(body: bytes, wbits: int) -> bytes:
    """The stream as windowBits `wbits` reads it: raw (< 0), zlib (8..15), gzip (31) or gzip for auto (47)."""
    return body if wbits < 0 else zlib_wrap(body) if wbits <= 15 else gzip_wrap(body)


def bulk(data: bytes, level: int = 6, sync_every: int = 0, final: bool = False) -> bytes:
    """C zlib raw deflate of `data` ending in Z_SYNC_FLUSH: non-final and byte aligned (final: ending in the final
    block instead).  sync_every adds flush points inside it."""
    co = zlib.compressobj(level, zlib.DEFLATED, -15)
    step = sync_every or len(data) or 1
    parts = [co.compress(data[i: i + step]) + (co.flush(zlib.Z_SYNC_FLUSH) if i + step < len(data) or not final else b"")
             for i in range(0, len(data), step)]
    return b"".join(parts) + (co.flush() if final else b"")


def splice(pieces) -> bytes:
    """One stream of byte-aligned pieces, each ending on a block boundary (the last one with the final block)."""
    return b"".join(pieces)


def crafted(case, final: bool) -> bytes:
    """The blocks of `case` (a function of (Deflate, final)) as a piece: ending in the final block, or in an empty
    stored block when more pieces follow."""
    d = Deflate()
    fill = case(d, final) or 0          # a case returns 1 to fill the last byte's unused bits with ones
    if not final:
        d.sync()
    return d.data(fill if final else 0)


def end_piece() -> bytes:
    """An empty final fixed block: ends a spliced stream."""
    return Deflate().fixed([], final=True).data()


def text(n: int, seed: int) -> bytes:
    """Compressible filler: words from a small seeded vocabulary."""
    rng = random.Random(seed)
    words = [bytes(rng.choice(b"abcdefghijklmnopqrstuvwxyz") for _ in range(rng.randrange(2, 9))) for _ in range(300)]
    out = bytearray()
    while len(out) < n:
        out += rng.choice(words) + (b"\n" if rng.random() < 0.08 else b" ")
    return bytes(out[:n])


def deep_stream(case, final: bool, seed: int, *, before: int = 3, piece: int = 700 << 10, sync_every: int = 0,
                after: int = 2) -> bytes:
    """`before` bulk pieces of `piece` bytes of output, the crafted blocks, `after` more bulk pieces and an empty
    final block (or the crafted blocks' own final block when `final`).  With sync_every = 0 the stream has no flush
    point but the two around the crafted blocks: the bulk data ahead of them is one piece, and the bulk data behind
    them one C zlib stream that ends the whole stream."""
    if sync_every:
        pieces = [bulk(text(piece, seed * 31 + k), 6, sync_every) for k in range(before)]
    else:
        pieces = [bulk(b"".join(text(piece, seed * 31 + k) for k in range(before)))] if before else []
    pieces.append(crafted(case, final))
    if not final:
        if sync_every:
            pieces += [bulk(text(piece, seed * 37 + k), 6, sync_every) for k in range(after)] + [end_piece()]
        else:
            pieces.append(bulk(b"".join(text(piece, seed * 37 + k) for k in range(after)), final=True) if after
                          else end_piece())
    return splice(pieces)


# ---- table-filling code length sets -------------------------------------------------------------------

def random_complete_lengths(rng, n: int, deep: float) -> list:
    """Lengths (1..15) of a complete code of n symbols, grown from two 1-bit leaves by splitting a leaf in two: with
    chance `deep` a longest leaf below 15 bits, otherwise one of a random length.  Shuffled over the symbols."""
    count = [0] * 16
    count[1] = 2
    for _ in range(n - 2):
        ls = [l for l in range(1, 15) if count[l]]
        l = ls[-1] if rng.random() < deep else rng.choice(ls)
        count[l] -= 1
        count[l + 1] += 2
    lens = [l for l in range(16) for _ in range(count[l])]
    rng.shuffle(lens)
    return lens


def table_used(oracle, ctype: int, lens, root: int) -> tuple:
    """inflate_table (the oracle's restatement) of lens with `root` bits: (return code, table entries used)."""
    import ctypes as C
    import numpy as np
    a = np.asarray(lens, dtype=np.uint16)
    table = np.zeros(2048, dtype=np.uint32)
    work = np.zeros(max(288, a.size), dtype=np.uint16)
    bits, index = C.c_uint(root), C.c_uint(0)
    ret = oracle.lib().zo_inflate_table(ctype, a.ctypes.data, a.size, table.ctypes.data, C.addressof(bits),
                                        work.ctypes.data, C.addressof(index), 0)
    return ret, index.value


def table_filling_sets(oracle, trials: int = 300, seed: int = 852):
    """The seeded search for literal/length (286 symbols, 9 root bits) and distance (30 symbols, 6 root bits)
    length sets that use as many decode-table entries as possible.  Returns (lit lens, lit used, dist lens, dist
    used)."""
    rng = random.Random(seed)
    best = {}
    for ctype, n, root in ((1, 286, 9), (2, 30, 6)):
        top = (0, None)
        for _ in range(trials):
            lens = random_complete_lengths(rng, n, rng.random())
            ret, used = table_used(oracle, ctype, lens, root)
            assert ret == 0, (ret, lens)
            if used > top[0]:
                top = (used, lens)
        best[ctype] = top
    return best[1][1], best[1][0], best[2][1], best[2][0]


# ---- the corpus ---------------------------------------------------------------------------------------
# A case is a function of (Deflate, final) that writes its blocks, the last one with BFINAL = final.

HIST = random.Random(32768).randbytes(32768)      # 32 KiB of history ahead of the far copies
DICT = text(1000, 5)                               # the preset dictionary of the dictionary case


def lens_of(n: int, pairs: dict) -> list:
    out = [0] * n
    for s, v in pairs.items():
        out[s] = v
    return out


def zero16(seq) -> list:
    """The same lengths with 16 repeating a zero: the last three zeros of every long enough 17 or 18 run."""
    out = []
    for s, x in seq:
        out += [(s, x - 3), (16, 0)] if s in (17, 18) and x >= 3 else [(s, x)]
    return out


def chain_cl(seq) -> list:
    """A code-length code of lengths 1, 2, ..., 7, 7 over the symbols of seq (at most 8) and unused fillers.  The
    fillers take the short codes and the used symbols the long ones, the rarest the two 7-bit codes, so the code
    words written include 7-bit ones."""
    freq = [0] * 19
    for s, _ in seq:
        freq[s] += 1
    used = sorted((s for s in range(19) if freq[s]), key=lambda s: (-freq[s], s))
    assert 2 <= len(used) <= 8
    order = [s for s in range(19) if not freq[s]][: 8 - len(used)] + used
    cl = [0] * 19
    for k, s in enumerate(order):
        cl[s] = min(k + 1, 7)
    return cl


def all_codes(lit, dist):
    """32 KiB of stored history, then one dynamic block that uses every literal/length and distance code of the
    given sets."""
    def case(d, final):
        d.stored(HIST)
        syms = [s for s in range(256) if lit[s]]
        ls = [s for s in range(257, 286) if lit[s]]
        ds = [s for s in range(30) if dist[s]]
        for i in range(max(len(ls), len(ds))):
            L, D = ls[i % len(ls)], ds[i % len(ds)]
            syms.append(Match(LEN_BASE[L - 257], DIST_BASE[D], lsym=L))
        d.dynamic(lit, dist, syms, final)
    return case


_ONE = lens_of(258, {97: 1, 256: 2, 257: 2})          # 'a', EOB, length 3
# literals a-d and k-n (a gap of six zeros: a 17 run), lengths 3-9, and 16 distance codes, all 4 bits
_X8 = lens_of(264, {**{s: 4 for s in b"abcdklmn"}, **{s: 4 for s in range(256, 264)}})
_X8_SYMS = list(b"abcdklmn") + [Match(9, 8), Match(3, 1), Match(5, 17), 98, Match(7, 25)]
_X8_SEQ = rle(_X8 + [4] * 16)


def _many_blocks(d, final):
    d.fixed(list(b"many blocks: ") * 4)
    for i in range(2000):
        d.fixed([Match(258, 1 + i % 50)] if i % 3 else [])
        d.dynamic(lens_of(257, {256: 1, 97: 1}), [0], [97] if i % 2 else [], final and i == 1999)


def _stored_phases(d, final):
    rng = random.Random(7)
    d.stored(b"")
    for j in range(8):
        d.fixed([0x90] * j)                   # 10 + 9j bits: the stored header that follows starts at bit (2 + j) % 8
        d.stored(rng.randbytes(j * 37 + 1))
        d.stored(b"")
    d.stored(rng.randbytes(65535), final)


VALID = [
    ("one_code_dist", lambda d, f: d.dynamic(_ONE, [1], [97, Match(3, 1), 97, Match(3, 1)], f)),
    ("no_code_dist", lambda d, f: d.dynamic(lens_of(257, {97: 1, 98: 2, 256: 2}), [0], [97, 98, 97], f)),
    ("eob_only", lambda d, f: (d.fixed(b"xyz"), d.dynamic(lens_of(257, {256: 1}), [0], [], f))),
    ("far_fixed", lambda d, f: (d.stored(HIST), d.fixed([Match(258, 32768), Match(3, 32767), Match(258, 32768, lsym=284),
                                                         65, Match(3, 1), Match(4, 2), Match(5, 3)], f))),
    ("far_dynamic", lambda d, f: (d.stored(HIST), d.dynamic(lens_of(286, {65: 2, 256: 2, 284: 2, 285: 2}),
                                                            lens_of(30, {0: 2, 1: 2, 2: 2, 29: 2}),
                                                            [Match(258, 32768), Match(258, 32767, lsym=284), 65,
                                                             Match(258, 1), Match(258, 2, lsym=284), Match(258, 3),
                                                             Match(258, 24577)], f))),
    ("dist_is_produced", lambda d, f: d.fixed(list(b"abcdefgh") + [Match(8, 8), Match(16, 16), 120, Match(33, 33)], f)),
    ("len258_code284", lambda d, f: d.fixed([120, Match(258, 1, lsym=284), 121, Match(258, 260, lsym=284)], f)),
    ("repeat_across_trees", lambda d, f: d.dynamic(_X8, [4] * 16, _X8_SYMS, f)),
    ("repeat_zero_with_16", lambda d, f: d.dynamic(_X8, [4] * 16, _X8_SYMS, f, seq=zero16(_X8_SEQ))),
    ("cl_code_7_bits", lambda d, f: d.dynamic(_X8, [4] * 16, _X8_SYMS, f, cl_lens=chain_cl(_X8_SEQ), hclen=19)),
    ("all_286_and_30", all_codes(huffman_lengths([random.Random(1).randrange(1, 50) for _ in range(286)], 15),
                                 huffman_lengths([random.Random(2).randrange(1, 50) for _ in range(30)], 15))),
    ("stored_phases", _stored_phases),
    ("many_blocks", _many_blocks),
    ("junk_tail", lambda d, f: (d.fixed(list(b"junk bits follow"), f), 1)[1]),
]


def valid_cases(oracle=None) -> list:
    """VALID, and with the oracle at hand the table-filling sets of table_filling_sets() too."""
    if oracle is None:
        return list(VALID)
    lit, _, dist, _ = table_filling_sets(oracle)
    return VALID + [("table_filling", all_codes(lit, dist))]


def dict_case(d, final):
    """Copies that reach exactly to the start of a 1000-byte preset dictionary (DICT)."""
    d.fixed([Match(10, 1000), 97, Match(20, 1011)], final)


_OK_LIT = lens_of(257, {97: 1, 256: 1})


def _header_only(lit, dist, **kw):
    return lambda d, f: d.dynamic(lit, dist, [], f, eob=False, **kw)


# (name, case, message, only at the start of a stream)
ERRORS = [
    ("block_type", lambda d, f: d.bits(int(f), 1).bits(3, 2), "invalid block type", False),
    ("stored_nlen", lambda d, f: d.stored(b"abc", f, nlen=0x1234), "invalid stored block lengths", False),
    ("too_many_lit", _header_only(_OK_LIT, [1], seq=[], hlit=287), "too many length or distance symbols", False),
    ("too_many_dist", _header_only(_OK_LIT, [1], seq=[], hdist=31), "too many length or distance symbols", False),
    ("cl_oversubscribed", _header_only(_OK_LIT, [1], seq=[], cl_lens=lens_of(19, {0: 1, 8: 1, 18: 1})),
     "invalid code lengths set", False),
    ("cl_incomplete", _header_only(_OK_LIT, [1], seq=[], cl_lens=lens_of(19, {0: 1, 18: 2})),
     "invalid code lengths set", False),
    ("repeat_first", _header_only(_OK_LIT, [1], seq=[(16, 0)], cl_lens=lens_of(19, {16: 1, 0: 2, 1: 2})),
     "invalid bit length repeat", False),
    ("repeat_past_end", _header_only(_OK_LIT, [1], seq=[(1, 0), (1, 0)] + [(18, 127)] * 2,
                                     cl_lens=lens_of(19, {1: 1, 18: 1})), "invalid bit length repeat", False),
    ("hclen4_no_eob", _header_only(_OK_LIT, [1], seq=[(18, 127), (18, 109)], cl_lens=lens_of(19, {0: 1, 18: 1}),
                                   hclen=4), "invalid code -- missing end-of-block", False),
    ("cl_code_empty", lambda d, f: d.dynamic(_OK_LIT, [1], [Bits(0, 258)], f, eob=False, seq=[], cl_lens=[0] * 19,
                                             hclen=4), "invalid code -- missing end-of-block", False),
    ("eob_length_0", _header_only(lens_of(257, {97: 1, 98: 1}), [1]), "invalid code -- missing end-of-block", False),
    ("lit_oversubscribed", _header_only(lens_of(257, {97: 1, 98: 1, 256: 1}), [1]), "invalid literal/lengths set", False),
    ("lit_incomplete", _header_only(lens_of(257, {97: 2, 98: 2, 256: 2}), [1]), "invalid literal/lengths set", False),
    ("dist_oversubscribed", _header_only(_OK_LIT, [1, 1, 1]), "invalid distances set", False),
    ("dist_incomplete", _header_only(_OK_LIT, [2, 2, 2]), "invalid distances set", False),
    ("fixed_286", lambda d, f: d.fixed([97, Sym(286)], f, eob=False), "invalid literal/length code", False),
    ("fixed_287", lambda d, f: d.fixed([97, Sym(287)], f, eob=False), "invalid literal/length code", False),
    ("fixed_dist_30", lambda d, f: d.fixed([97, Sym(257), DSym(30)], f, eob=False), "invalid distance code", False),
    ("fixed_dist_31", lambda d, f: d.fixed([97, Sym(257), DSym(31)], f, eob=False), "invalid distance code", False),
    ("lit_unused_slot", lambda d, f: d.dynamic(lens_of(257, {256: 1}), [0], [Bits(1, 1)], f, eob=False),
     "invalid literal/length code", False),
    ("dist_unused_slot", lambda d, f: d.dynamic(_ONE, [1], [97, Sym(257), Bits(1, 1)], f, eob=False),
     "invalid distance code", False),
    ("dist_empty_set", lambda d, f: d.dynamic(_ONE, [0], [97, Sym(257), Bits(0, 1)], f, eob=False),
     "invalid distance code", False),
    ("too_far", lambda d, f: d.fixed([97, 98, Match(3, 3)], f), "invalid distance too far back", True),
]


# invalid-code triggers that can end a stream: (name, lit lens, dist lens, symbols before the trigger, trigger bit)
TAIL_TRIGGERS = [
    ("lit_unused_slot", lens_of(257, {256: 1}), [0], [], 1, "invalid literal/length code"),
    ("dist_unused_slot", _ONE, [1], [97, Sym(257)], 1, "invalid distance code"),
    ("dist_empty_set", _ONE, [0], [97, Sym(257)], 0, "invalid distance code"),
]


def tail_trigger(lit, dist, before, bit: int, r: int) -> bytes:
    """A raw stream whose invalid code word starts r bits before its end (1 <= r <= 14): a fixed block of 9-bit
    literals sets the bit phase, then the dynamic block with the trigger, then r - 1 zero bits."""
    for j in range(8):
        d = Deflate()
        d.fixed([0x90] * j)
        d.dynamic(lit, dist, list(before), True, eob=False)
        if (d.w.n + r) % 8 == 0:
            d.bits(bit, 1)
            for _ in range(r - 1):
                d.bits(0, 1)
            out = d.data()
            assert len(out) * 8 == d.w.n
            return out
    raise AssertionError("no phase fits")
