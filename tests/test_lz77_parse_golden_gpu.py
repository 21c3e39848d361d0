"""Pinned output of the LZ77 parse (the thin parse warp of lz77_kernel) on shapes that take its rare paths: a
block cut every 16383 literals at every hop offset of a parse group, matches of 258 that carry the skip across
hops and groups, chunk boundaries inside pairs (empty chunks, chunks of 1-63 bytes), segments of up to 256
chunks and ranges that end inside a pair, in independent, primed and stitched mode, at levels 1, 2, 3, 6, 9 and
with Z_RLE and Z_FILTERED.  Every kernel instantiation shares the parse, so comparing two kernels cannot catch a
parse bug; the digests in tests/golden/lz77_parse_digests.json pin the compressed bytes, the chunk offsets and
bit lengths and the totals instead.  Every stream also has to decode with C zlib to its input.

Regenerate the digests (only when the output is meant to change): python tests/test_lz77_parse_golden_gpu.py --write"""
import hashlib
import json
import os
import sys
import zlib

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from conftest import GOLDEN, make_text, pkg  # noqa: E402

pytestmark = pytest.mark.gpu

DIGESTS = os.path.join(GOLDEN, "lz77_parse_digests.json")
N = 3 << 20
Z_FILTERED, Z_RLE = 1, 3
# (name, level, strategy)
LEVELS = [("L1", 1, 0), ("L2", 2, 0), ("L3", 3, 0), ("L6", 6, 0), ("L9", 9, 0), ("rle", 6, Z_RLE), ("filtered", 6, Z_FILTERED)]
KINDS = ["random", "sparse", "runs", "text"]


def _random(n, seed):
    return np.random.default_rng(seed).integers(0, 256, n, dtype=np.uint8).tobytes()


def _sparse(n, seed):
    """Incompressible bytes with a few short copies: the blocks are still cut by the symbol limit, but the parse
    enters the hops at every offset."""
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 256, n, dtype=np.uint8)
    for p in rng.integers(300, n - 64, n // 700):
        ln = int(rng.integers(3, 40))
        d = int(rng.integers(1, 300))
        a[p: p + ln] = a[p - d: p - d + ln]
    return a.tobytes()


def _runs(n, seed):
    """Runs of one byte up to 3000 long and short periods repeated: matches of 258, skips across group edges."""
    rng = np.random.default_rng(seed)
    out = bytearray()
    while len(out) < n:
        k = rng.integers(0, 3)
        if k == 0:
            out += bytes([int(rng.integers(0, 256))]) * int(rng.integers(1, 3000))
        elif k == 1:
            out += rng.integers(0, 256, int(rng.integers(1, 10)), dtype=np.uint8).tobytes() * int(rng.integers(1, 600))
        else:
            out += rng.integers(0, 256, int(rng.integers(1, 64)), dtype=np.uint8).tobytes()
    return bytes(out[:n])


_DATA = {}


def _data(kind):
    if kind not in _DATA:
        _DATA[kind] = {"random": lambda: _random(N, 11), "sparse": lambda: _sparse(N, 12), "runs": lambda: _runs(N, 13),
                       "text": lambda: make_text(N, 14)}[kind]()
    return _DATA[kind]


def _ragged(n, seed):
    """Chunk offsets over n bytes: empty chunks, chunks of 1-63 bytes, and longer ones up to 70000 bytes."""
    rng = np.random.default_rng(seed)
    lens = []
    while sum(lens) < n:
        k = rng.integers(0, 4)
        lens.append(0 if k == 0 else int(rng.integers(1, 64)) if k == 1 else int(rng.integers(64, 3000)) if k == 2
                    else int(rng.integers(3000, 70000)))
    off = np.zeros(len(lens) + 1, dtype=np.uint64)
    np.cumsum(lens, out=off[1:])
    off[-1] = n
    return np.minimum(off, n)


# (name, chunk size, chunk offsets or None): 1 MiB chunks hold 64 block cuts of incompressible data each
LAYOUTS = [("c1m", 1 << 20), ("c64k", 65536), ("c1000", 1000), ("ragged", 0)]


def _modes(B):
    return [("indep", B.MODE_INDEPENDENT, 0), ("primed", B.MODE_INDEPENDENT, B.FLAG_PRIME), ("stitched", B.MODE_STITCHED, 0)]


def _digest(r):
    h = hashlib.sha256()
    h.update(r.data)
    h.update(np.asarray(r.out_off, dtype=np.uint64).tobytes())
    h.update(np.asarray(r.out_bits, dtype=np.uint64).tobytes())
    h.update(np.array([r.total_out_bytes, r.total_out_bits, r.check, r.n_blocks], dtype=np.uint64).tobytes())
    return h.hexdigest()


def _decodes(B, r, data, mode, flags, off):
    if mode == B.MODE_STITCHED:
        return zlib.decompress(r.data, -15) == data
    for i in range(off.size - 1):
        lo, hi = int(off[i]), int(off[i + 1])
        d = zlib.decompressobj(-15, zdict=data[max(0, lo - 32768): lo]) if flags & B.FLAG_PRIME and lo else zlib.decompressobj(-15)
        if d.decompress(r.stream(i)) + d.flush() != data[lo:hi]:
            return False
    return True


def _cases(kind, lname, level, strategy):
    """Yields (case id, digest) for every layout and mode of one data kind and level; asserts that every stream
    decodes to its input."""
    B = pkg("batch")
    data = _data(kind)
    for layout, chunk in LAYOUTS:
        off = _ragged(len(data), 21) if chunk == 0 else np.minimum(np.arange(0, len(data) + chunk, chunk, dtype=np.uint64), len(data))
        off = np.unique(off) if chunk else off
        for mname, mode, flags in _modes(B):
            r = B.deflate_batch(data, chunk, level, B.WRAP_RAW, mode, flags | B.flag_strategy(strategy),
                                in_off=off if chunk == 0 else None)
            cid = f"{kind}/{lname}/{layout}/{mname}"
            assert _decodes(B, r, data, mode, flags, off), cid
            yield cid, _digest(r)


def _segments_of_256(B):
    """1000-byte chunks, independent: a batch of more than 148 * 255 chunks is cut into segments of 256 chunks
    (256000 bytes: the range ends inside a pair)."""
    rng = np.random.default_rng(31)
    n = 38_000_000
    parts = [make_text(n // 2, 32), _runs(n // 4, 33), rng.integers(0, 256, n - n // 2 - n // 4, dtype=np.uint8).tobytes()]
    data = b"".join(parts)
    off = np.minimum(np.arange(0, n + 1000, 1000, dtype=np.uint64), n)
    for lname, level, strategy in [("L1", 1, 0), ("L6", 6, 0)]:
        r = B.deflate_batch(data, 1000, level, B.WRAP_RAW, B.MODE_INDEPENDENT, B.flag_strategy(strategy))
        cid = f"seg256/{lname}/c1000/indep"
        assert _decodes(B, r, data, B.MODE_INDEPENDENT, 0, off), cid
        yield cid, _digest(r)


def _golden():
    return json.load(open(DIGESTS))


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("lname,level,strategy", LEVELS, ids=[x[0] for x in LEVELS])
def test_parse_output_is_pinned(gpu_ctx, kind, lname, level, strategy):
    want = _golden()
    for cid, got in _cases(kind, lname, level, strategy):
        assert got == want[cid], cid


def test_segments_of_256_chunks_are_pinned(gpu_ctx):
    want = _golden()
    for cid, got in _segments_of_256(pkg("batch")):
        assert got == want[cid], cid


if __name__ == "__main__" and "--write" in sys.argv:
    out = {}
    for kind in KINDS:
        for lname, level, strategy in LEVELS:
            out.update(_cases(kind, lname, level, strategy))
    out.update(_segments_of_256(pkg("batch")))
    with open(DIGESTS, "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
        f.write("\n")
    print(f"{len(out)} digests -> {DIGESTS}")
