"""GPU tests of the inflate index (zs_inflate_index_*): random access into one deflate stream.

The build must decode exactly as zs_inflate_stream_dev; its access points must be the point rule applied to the block
starts C zlib's inflate(Z_BLOCK) reports (zran_check.block_starts, the zran.c method); every window must let C zlib decode
from its point with no engine code involved; extracted ranges must be slices of the whole output."""
import gzip
import io
import random
import zlib

import numpy as np
import pytest

from conftest import make_mixed, make_text, pkg
from zran_check import block_starts, decode_from

pytestmark = pytest.mark.gpu

SPANS = (1, 4096, 65536, 1 << 20)
DICT = make_text(40000, 9)[-20000:]


def _sync_flushed(data, every, mode, wbits=15, level=6):
    c = zlib.compressobj(level, zlib.DEFLATED, wbits)
    parts = []
    for i in range(0, len(data), every):
        parts.append(c.compress(data[i: i + every]))
        parts.append(c.flush(mode))
    parts.append(c.flush())
    return b"".join(parts)


def _strategy(data, strategy, wbits=15, level=6):
    c = zlib.compressobj(level, zlib.DEFLATED, wbits, 8, strategy)
    return c.compress(data) + c.flush()


def _gives_up(data):
    """Raw stream: a part with sync flush points, then 3 MiB of fixed-code blocks (no marker, no dynamic header to cut
    at), so the parallel decoder stops at the last marker and the serial decoder does the rest."""
    a = zlib.compressobj(6, zlib.DEFLATED, -15)
    head = b"".join(a.compress(data[i: i + 65536]) + a.flush(zlib.Z_SYNC_FLUSH) for i in range(0, 1 << 20, 65536))
    return head + _strategy(data[1 << 20:], zlib.Z_FIXED, -15)


def _gzip_named(data):
    buf = io.BytesIO()
    with gzip.GzipFile(filename="sample.txt", mode="wb", fileobj=buf, mtime=12345) as f:
        f.write(data)
    return buf.getvalue()


def _engine_sync(data):
    B = pkg("batch")
    return B.deflate_batch(data, 65536, 6, B.WRAP_ZLIB, B.MODE_STITCHED, B.FLAG_SYNC).data


def _cases():
    text, mixed = make_text(3 << 20, 21), make_mixed(3 << 20, 22)
    small = make_text(50000, 23)
    return [
        ("engine_sync", lambda: _engine_sync(text), 15, None),
        ("zlib_l1", lambda: zlib.compress(mixed, 1), 15, None),
        ("zlib_l6", lambda: zlib.compress(text, 6), 15, None),
        ("zlib_l9", lambda: zlib.compress(mixed, 9), 15, None),
        ("zlib_sync", lambda: _sync_flushed(text, 200000, zlib.Z_SYNC_FLUSH), 15, None),
        ("zlib_full", lambda: _sync_flushed(mixed, 300000, zlib.Z_FULL_FLUSH), 15, None),
        ("stored", lambda: zlib.compress(text[: 1 << 20], 0), 15, None),
        ("fixed", lambda: _strategy(text, zlib.Z_FIXED), 15, None),
        ("huffman_only", lambda: _strategy(mixed, zlib.Z_HUFFMAN_ONLY), 15, None),
        ("rle", lambda: _strategy(mixed, zlib.Z_RLE), 15, None),
        ("gives_up_raw", lambda: _gives_up(text + mixed[: 1 << 20]), -15, None),
        ("gzip_named", lambda: _gzip_named(mixed), 31, None),
        ("auto_gzip", lambda: _gzip_named(small), 47, None),
        ("auto_zlib", lambda: zlib.compress(text, 6), 47, None),
        ("raw_dict", lambda: _dict_stream(text[: 1 << 20], -15), -15, DICT),
        ("zlib_fdict", lambda: _dict_stream(small, 15), 15, DICT),
        ("empty", lambda: zlib.compress(b""), 15, None),
        ("small", lambda: zlib.compress(small, 6), 15, None),
    ]


def _dict_stream(data, wbits):
    c = zlib.compressobj(6, zlib.DEFLATED, wbits, 8, zlib.Z_DEFAULT_STRATEGY, DICT)
    return c.compress(data) + c.flush()


CASES = _cases()
IDS = [c[0] for c in CASES]
_streams = {}


def _stream(i):
    if i not in _streams:
        _streams[i] = CASES[i][1]()
    return _streams[i]


def _rule(starts, span, out_len):
    """The access points: per m = 0, S, 2S, ... < out_len the first block start with offset >= m; the first start always."""
    pts = [starts[0]]
    m, k = span, 1
    while m < out_len:
        while k < len(starts) and starts[k][1] < m:
            k += 1
        if k == len(starts):
            break
        if starts[k] != pts[-1]:
            pts.append(starts[k])
        m = (starts[k][1] // span + 1) * span
    return pts


def _stream_dev(data, wbits, dictionary, out_cap):
    """zs_inflate_stream_dev of the same stream: (status, out bytes, out_len, in_used, check, detail)."""
    import torch
    B, capi = pkg("batch"), pkg("capi")
    ctx = B.default_context(0)
    d_in = torch.frombuffer(bytearray(data) or bytearray(8), dtype=torch.uint8)[: len(data)].cuda()
    out = torch.zeros(out_cap + 16, dtype=torch.uint8, device="cuda")
    r = torch.zeros(4, dtype=torch.int64, device="cuda")
    d_dict = torch.frombuffer(bytearray(dictionary), dtype=torch.uint8).cuda() if dictionary else None
    lib = capi.load()
    rc = lib.zs_inflate_stream_dev(ctx.handle, B._ptr(d_in), len(data), wbits, B._ptr(out), out_cap, B._ptr(r[0:1]),
                                   B._ptr(r[1:2]), B._ptr(r[2:3]), B._ptr(r[3:4]), B._ptr(d_dict),
                                   len(dictionary) if dictionary else 0)
    ctx.check(rc, "zs_inflate_stream_dev")
    det = np.zeros(1, dtype=np.int32)
    ctx.check(lib.zs_inflate_last_details(ctx.handle, det.ctypes.data, 1), "details")
    h = r.cpu().numpy()
    n = int(h[0])
    return int(np.int32(h[3] & 0xffffffff)), out[:n].cpu().numpy().tobytes(), n, int(h[1]), int(h[2]) & 0xffffffff, int(det[0])


def _check_windows(ix, data, out, limit=40):
    """C zlib, given a point's window as its dictionary, decodes raw deflate from the point's bit to out[o:] (the first
    64 KiB of it)."""
    pts = ix.points
    blob = ix.to_bytes()
    n = len(pts)
    wl = np.frombuffer(blob[56: 56 + 24 * n], dtype=np.uint64).reshape(n, 3)[:, 2] & 0xffffffff
    starts = np.concatenate([[0], np.cumsum(wl)]).astype(np.int64) + 56 + 24 * n
    sel = sorted(set(np.linspace(0, n - 1, min(n, limit)).astype(int)))
    for p in sel:
        bit, o = int(pts[p][0]), int(pts[p][1])
        window = blob[starts[p]: starts[p + 1]]
        want = min(len(out) - o, 1 << 16)
        got = decode_from(data, bit, window, want) if want else b""
        assert got == out[o: o + want], (p, bit, o)


def _random_ranges(rng, out_len, n):
    r = [(0, 0), (0, min(out_len, 1000)), (max(out_len - 500, 0), 500), (max(out_len - 100, 0), 1000), (0, out_len),
         (out_len, 10), (out_len + 5, 0)]
    for _ in range(n):
        o = rng.randrange(0, out_len + 1) if out_len else 0
        r.append((o, rng.choice([0, 1, 17, 4096, 70000, 1 << 20])))
    return r


def _check_extract(ix, data, out, ranges):
    off = [o for o, _ in ranges]
    ln = [n for _, n in ranges]
    host = ix.extract_ranges(off, ln, data)
    import torch
    d_in = torch.frombuffer(bytearray(data) or bytearray(8), dtype=torch.uint8)[: len(data)].cuda()
    dev = ix.extract_ranges(off, ln, d_in)
    for r in (host, dev):
        for i, (o, n) in enumerate(ranges):
            want = out[o: o + n] if o < len(out) else b""
            assert r.range(i) == want, (i, o, n)
            assert int(r.got[i]) == len(want)
            assert int(r.status[i]) == (0 if len(want) == n else -5), (i, o, n, int(r.status[i]))
    assert host.data == dev.data


@pytest.mark.parametrize("i", range(len(CASES)), ids=IDS)
def test_build_points_windows_extract(gpu_ctx, oracle, i):
    B = pkg("batch")
    name, _, wbits, dictionary = CASES[i]
    data = _stream(i)
    ref_ret, ref_out, _, _ = oracle.inflate(data, wbits, dictionary=dictionary)
    assert ref_ret == oracle.Z_STREAM_END
    cap = len(ref_out) + 64
    want = _stream_dev(data, wbits, dictionary, cap)
    starts = block_starts(data, wbits, dictionary)
    rng = random.Random(i)
    for span in SPANS:
        ix, built = B.InflateIndex.build(data, wbits, span, dictionary=dictionary, out_cap=cap)
        got = (built.status, built.data[: built.out_len].cpu().numpy().tobytes(), built.out_len, built.in_used,
               built.check & 0xffffffff, built.detail)
        assert got == want
        assert built.status == 1 and ix is not None
        pts = [tuple(int(v) for v in p) for p in ix.points]
        assert pts == _rule(starts, span, len(ref_out)), span
        info = ix.info
        assert (info.in_len, info.out_len, info.span, info.n_points) == (len(data), len(ref_out), span, len(pts))
        if span == 65536:
            _check_windows(ix, data, ref_out)
        if span in (4096, 1 << 20):
            _check_extract(ix, data, ref_out, _random_ranges(rng, len(ref_out), 40))
        ix.close()


@pytest.mark.parametrize("i", [IDS.index(n) for n in ("engine_sync", "zlib_l6", "gives_up_raw")],
                         ids=["engine_sync", "zlib_l6", "gives_up_raw"])
def test_index_independent_of_decode_path(gpu_ctx, monkeypatch, i):
    B = pkg("batch")
    _, _, wbits, dictionary = CASES[i]
    data = _stream(i)
    base = B.InflateIndex.build(data, wbits, 65536, dictionary=dictionary)[0].to_bytes()
    for hook in ("ZS_INFLATE_SERIAL", "ZS_INFLATE_NO_SPEC"):
        monkeypatch.setenv(hook, "1")
        assert B.InflateIndex.build(data, wbits, 65536, dictionary=dictionary)[0].to_bytes() == base, hook
        monkeypatch.delenv(hook)


def test_large_stream_64mib(gpu_ctx, oracle):
    B = pkg("batch")
    src = make_mixed(64 << 20, 31)
    data = zlib.compress(src, 1)
    starts = block_starts(data, 15)
    for span in (65536, 1 << 20):
        ix, built = B.InflateIndex.build(data, 15, span, out_cap=len(src) + 64)
        assert built.status == 1 and built.out_len == len(src)
        assert [tuple(int(v) for v in p) for p in ix.points] == _rule(starts, span, len(src))
    _check_windows(ix, data, src, limit=16)
    rng = random.Random(5)
    _check_extract(ix, data, src, _random_ranges(rng, len(src), 200))
    # 10 000 ranges in one call
    ranges = [(rng.randrange(0, len(src)), 4096) for _ in range(10000)]
    r = ix.extract_ranges([o for o, _ in ranges], [n for _, n in ranges])
    for k in range(0, 10000, 97):
        o, n = ranges[k]
        assert r.range(k) == src[o: o + n]
    assert int((r.status == -3).sum()) == 0


@pytest.mark.parametrize("kind", ["truncated", "corrupt", "bad_header"])
def test_failed_build_matches_stream_dev(gpu_ctx, kind):
    B = pkg("batch")
    src = make_text(1 << 20, 41)
    data = bytearray(zlib.compress(src, 6))
    if kind == "truncated":
        data = data[: len(data) * 2 // 3]
    elif kind == "corrupt":
        data[len(data) // 2] ^= 0x55
        data[len(data) // 2 + 1] ^= 0xff
    else:
        data[0] ^= 0x10
    data = bytes(data)
    cap = len(src) + 64
    want = _stream_dev(data, 15, None, cap)
    ix, built = B.InflateIndex.build(data, 15, 65536, out_cap=cap)
    assert ix is None and built.status != 1
    got = (built.status, built.data[: built.out_len].cpu().numpy().tobytes(), built.out_len, built.in_used,
           built.check & 0xffffffff, built.detail)
    assert got == want


def test_bad_arguments(gpu_ctx):
    B, capi = pkg("batch"), pkg("capi")
    data = zlib.compress(make_text(100000, 3))
    with pytest.raises(capi.ZsError) as e:
        B.InflateIndex.build(data, 15, 0)
    assert e.value.code == capi.Z_STREAM_ERROR
    with pytest.raises(capi.ZsError) as e:
        B.InflateIndex.build(data, -16, 4096)
    assert e.value.code == capi.Z_STREAM_ERROR
    ix, _ = B.InflateIndex.build(data, 15, 4096)
    with pytest.raises(capi.ZsError) as e:
        ix.extract_ranges([0], [10], data[:-1])
    assert e.value.code == capi.Z_STREAM_ERROR


def test_damaged_input_gives_data_error(gpu_ctx, oracle):
    """Zeroing the input from a byte-aligned point on: ranges before it still read, ranges that need it fail with the
    reference's message for the damaged stream, and got counts the bytes before the point."""
    B = pkg("batch")
    src = make_text(2 << 20, 51)
    data = _engine_sync(src)
    ix, _ = B.InflateIndex.build(data, 15, 1 << 18)
    pts = ix.points
    k = next(p for p in range(len(pts) // 2, len(pts)) if int(pts[p][0]) % 8 == 0 and int(pts[p][1]) > 0)
    byte, o = int(pts[k][0]) >> 3, int(pts[k][1])
    bad = data[:byte] + bytes(len(data) - byte)
    ret, _, _, _ = oracle.inflate(bad, 15, len(src) + 64)
    assert ret == oracle.Z_DATA_ERROR
    s = oracle.InflateStream(15)
    s.step(bad, len(src) + 64, oracle.Z_FINISH)
    msg = s.msg
    ranges = [(0, 1000), (o - 5000, 10000), (o, 10), (len(src) - 10, 10)]
    for d in (bad, None):
        import torch
        src_in = bad if d is not None else torch.frombuffer(bytearray(bad), dtype=torch.uint8).cuda()
        r = ix.extract_ranges([a for a, _ in ranges], [n for _, n in ranges], src_in)
        assert int(r.status[0]) == 0 and r.range(0) == src[:1000]
        for i in (1, 2, 3):
            assert int(r.status[i]) == -3 and r.message(i) == msg, (i, r.message(i), msg)
        assert int(r.got[1]) == 5000 and r.range(1) == src[o - 5000: o]
        assert int(r.got[2]) == 0


def test_export_import_roundtrip(gpu_ctx):
    B = pkg("batch")
    src = make_mixed(3 << 20, 61)
    data = _sync_flushed(src, 100000, zlib.Z_SYNC_FLUSH, wbits=31)
    ix, _ = B.InflateIndex.build(data, 31, 1 << 18)
    blob = ix.to_bytes()
    assert blob[:4] == b"ZSIX"
    ix2 = B.InflateIndex.from_bytes(blob, source=data)
    assert ix2.to_bytes() == blob
    assert np.array_equal(ix2.points, ix.points)
    rng = random.Random(7)
    ranges = _random_ranges(rng, len(src), 50)
    a = ix.extract_ranges([o for o, _ in ranges], [n for _, n in ranges], data)
    b = ix2.extract_ranges([o for o, _ in ranges], [n for _, n in ranges])
    assert a.data == b.data and np.array_equal(a.got, b.got) and np.array_equal(a.status, b.status)


def test_import_rejects_malformed(gpu_ctx):
    B, capi = pkg("batch"), pkg("capi")
    src = make_text(1 << 20, 71)
    data = zlib.compress(src, 6)
    ix, _ = B.InflateIndex.build(data, 15, 1 << 17)
    blob = bytearray(ix.to_bytes())
    n = int.from_bytes(blob[48:56], "little")
    assert n >= 3

    def rejected(b):
        with pytest.raises(capi.ZsError) as e:
            B.InflateIndex.from_bytes(bytes(b))
        assert e.value.code == capi.Z_DATA_ERROR

    def edit(pos, val, size=8):
        b = bytearray(blob)
        b[pos: pos + size] = int(val).to_bytes(size, "little", signed=val < 0)
        return b

    rejected(b"XSIX" + blob[4:])                          # magic
    rejected(edit(4, 2, 4))                                # version
    rejected(edit(8, -16, 4))                              # window_bits (deflate64)
    rejected(edit(48, n + 1))                              # count disagrees with the length
    rejected(edit(48, n - 1))
    p1 = 56 + 24
    rejected(edit(p1, int.from_bytes(blob[56:64], "little")))        # bits not increasing
    rejected(edit(p1 + 24 + 8, 0))                                   # output offsets going back
    rejected(edit(p1 + 16, 32769, 4))                                # win_len > 32768
    rejected(edit(p1, len(data) * 8))                                # bit beyond the input
    for cut in sorted({0, 3, 4, 8, 12, 16, 24, 32, 40, 44, 48, 55, 56, 60, 79, 80, 56 + 24 * n, len(blob) - 1}):
        rejected(blob[:cut])                                          # truncation at every field
    rejected(blob + b"\0")
    assert B.InflateIndex.from_bytes(bytes(blob)).to_bytes() == bytes(blob)
