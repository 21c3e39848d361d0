"""The greedy levels run through kernels specialised for their level (lz77_kernel<0, L>: level 1 walks its chain
of four as straight-line rounds).  ZS_LZ_GREEDY_GENERIC=1 sends them through lz77_kernel<0, 0>, which reads the
level's parameters at run time.  Both must produce the same compressed bytes, chunk offsets and bit lengths."""
import glob
import os
import zlib

import numpy as np
import pytest

from conftest import ROOT, make_text, pkg
from test_deflate_gpu import _kinds

pytestmark = pytest.mark.gpu

N = (1 << 20) + 12345   # the last chunk is ragged at every chunk size
CHUNKS = [4096, 65536, 262144]


def _runs(n, seed):
    """Runs of one byte (up to 3000 long), short periods repeated, and random stretches between them."""
    rng = np.random.default_rng(seed)
    out = bytearray()
    while len(out) < n:
        k = rng.integers(0, 3)
        if k == 0:
            out += bytes([int(rng.integers(0, 256))]) * int(rng.integers(1, 3000))
        elif k == 1:
            out += rng.integers(0, 256, int(rng.integers(2, 10)), dtype=np.uint8).tobytes() * int(rng.integers(1, 400))
        else:
            out += rng.integers(0, 256, int(rng.integers(1, 64)), dtype=np.uint8).tobytes()
    return bytes(out[:n])


def _source(n):
    files = sorted(glob.glob(os.path.join(ROOT, "zlib-streams-ts_b200", "csrc", "*"))) + [os.path.join(ROOT, "DESIGN.md")]
    txt = b"".join(open(f, "rb").read() for f in files)
    return (txt * (n // len(txt) + 1))[:n]


_DATA = {}


def _data(kind):
    if not _DATA:
        _DATA.update(_kinds(N))
        _DATA["source"] = _source(N)
        _DATA["runs"] = _runs(N, 31)
    return _DATA[kind]


def _both(monkeypatch, data, chunk, level, wrap, mode, flags=0, in_off=None):
    B = pkg("batch")
    monkeypatch.setenv("ZS_LZ_GREEDY_GENERIC", "1")
    ref = B.deflate_batch(data, chunk, level, wrap, mode, flags, in_off=in_off)
    monkeypatch.delenv("ZS_LZ_GREEDY_GENERIC")
    got = B.deflate_batch(data, chunk, level, wrap, mode, flags, in_off=in_off)
    what = (level, chunk, wrap, mode, flags)
    assert got.total_out_bits == ref.total_out_bits, what
    assert np.array_equal(got.out_off, ref.out_off), what
    assert np.array_equal(got.out_bits, ref.out_bits), what
    assert got.data == ref.data, what
    return got


KINDS = ["text", "mixed", "dna", "short_repeats", "counters", "floats", "json", "source", "runs"]


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("level", [1, 2, 3])
def test_same_output_as_generic_kernel(gpu_ctx, monkeypatch, kind, level):
    B = pkg("batch")
    data = _data(kind)
    for chunk in CHUNKS:
        for flags in (0, B.FLAG_PRIME):
            _both(monkeypatch, data, chunk, level, B.WRAP_RAW, B.MODE_INDEPENDENT, flags)
    r = _both(monkeypatch, data, 65536, level, B.WRAP_ZLIB, B.MODE_STITCHED)
    assert zlib.decompress(r.data) == data


@pytest.mark.parametrize("level", [1, 2, 3])
def test_same_output_on_ragged_and_tiny_chunks(gpu_ctx, monkeypatch, level):
    """Empty chunks, chunks shorter than 8 and than 258 bytes (the nice and maximum lengths clipped at the chunk
    end), boundaries inside long runs, and a few long chunks between them."""
    B = pkg("batch")
    rng = np.random.default_rng(50 + level)
    fixed = [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 0, 0, 15, 16, 17, 200, 257, 258, 259, 260, 515, 516, 4096, 65536, 70000, 0]
    lens = np.concatenate([fixed, rng.integers(0, 600, size=3000), rng.integers(0, 9, size=500), [0, 1, 7]])
    lens[rng.integers(0, lens.size, 300)] = 0
    rng.shuffle(lens)
    off = np.zeros(lens.size + 1, dtype=np.uint64)
    np.cumsum(lens, out=off[1:])
    n = int(off[-1])
    half = _runs(n // 2, 77)
    data = half + make_text(n - len(half), 78)
    for mode, flags in ((B.MODE_INDEPENDENT, 0), (B.MODE_INDEPENDENT, B.FLAG_PRIME), (B.MODE_STITCHED, 0)):
        _both(monkeypatch, data, 0, level, B.WRAP_RAW, mode, flags, in_off=off)
